/*
 * dgr_b200.h — C ABI of the B200-native differentiable Gaussian-splat rasterizer (libdgr_b200.so).
 *
 * This is the drop-in boundary for the ONE native call DreamGaussian makes on its hot path:
 *   GaussianRasterizer(raster_settings)(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
 *   cov3D_precomp) -> (color, radii, depth, alpha)          /root/reference/gs_renderer.py:745-809
 * The reference binds that through the pybind module `diff_gaussian_rasterization._C` of an un-vendored package
 * (readme.md:30-32): `rasterize_gaussians`, `rasterize_gaussians_backward`, `mark_visible`  [EXT, SURVEY.md §8b].
 * The entry points below are what those three bindings would call; everything is plain pointers and sizes, no
 * torch types.  All pointers are DEVICE pointers unless named *_host.  All work is enqueued on `stream`
 * (a cudaStream_t passed as void*); nothing here synchronises the device unless stated.
 *
 * Return value: 0 on success, otherwise a cudaError_t / negative dgr error code; dgr_last_error() has the text.
 */
#ifndef DGR_B200_H
#define DGR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGR_ABI_VERSION 4

/* == GaussianRasterizationSettings, the 12-field NamedTuple built at gs_renderer.py:745-758 == */
typedef struct DgrSettings {
    int32_t image_height;
    int32_t image_width;
    float   tanfovx;
    float   tanfovy;
    float   scale_modifier;
    int32_t sh_degree;       /* active degree, 0..3 */
    int32_t prefiltered;     /* accepted, unused (always False in the reference, gs_renderer.py:756) */
    int32_t debug;           /* !=0: synchronise and check after every kernel */
    const float *bg;         /* [3]   */
    const float *viewmatrix; /* [4,4] row-major, p_view = [p,1] @ V   (gs_renderer.py:656-662) */
    const float *projmatrix; /* [4,4] row-major, full projection      (gs_renderer.py:663-670) */
    const float *campos;     /* [3]   as given by the caller (= -c2w[:3,3], gs_renderer.py:671) */
} DgrSettings;

/* == the per-Gaussian inputs of GaussianRasterizer.forward (gs_renderer.py:800-809); float32, contiguous ==
 * Alignment: `rotations`, and `shs` / `shs_rest` when their rows are a multiple of 16 bytes (M % 4 == 0, (M - 1) % 4 == 0), are read
 * with 128-bit loads and must be 16-byte aligned — what every device allocation is; the two host layers of this repository
 * re-allocate a view that is not (rasterizer.py::_dev_f32, dgr_torch.cpp::dev_f32).  When ALL of means3D / scales / rotations /
 * opacities / shs (/ shs_rest) are 16-byte aligned the per-Gaussian kernels stage them with bulk TMA (see dgr_set_tuning). */
typedef struct DgrGaussians {
    int32_t P;                   /* number of Gaussians */
    int32_t M;                   /* SH coefficients per channel in `shs` (= shs.shape[1]); 0 if shs == NULL */
    const float *means3D;        /* [P,3]   */
    const float *shs;            /* [P,M,3] or NULL (then colors_precomp) */
    const float *colors_precomp; /* [P,3]   or NULL */
    const float *opacities;      /* [P,1]   */
    const float *scales;         /* [P,3]   or NULL (then cov3D_precomp) */
    const float *rotations;      /* [P,4]   (w,x,y,z), consumed un-normalised */
    const float *cov3D_precomp;  /* [P,6]   xx,xy,xz,yy,yz,zz or NULL */
    /* SURVEY.md §8 row f1 — GaussianModel's RAW parameters with the activations fused into the kernels
     * (gs_renderer.py:196-216): when activations != 0, `opacities` is _opacity (sigmoid applied here), `scales` is _scaling
     * (exp), `rotations` is _rotation (F.normalize, eps 1e-12), `shs` is _features_dc [P,1,3] and `shs_rest` is
     * _features_rest [P,M-1,3] (NULL when M == 1) — no torch.cat copy; M stays the TOTAL coefficient count.  Requires
     * shs != NULL and cov3D_precomp == NULL.  The gradients come back with respect to the raw tensors. */
    const float *shs_rest;
    int32_t activations;
} DgrGaussians;

/* == outputs of the forward (gs_renderer.py:800) == */
typedef struct DgrImages {
    float   *color;  /* [3,H,W] */
    float   *depth;  /* [1,H,W] sum depth*alpha*T (not normalised) */
    float   *alpha;  /* [1,H,W] sum alpha*T */
    int32_t *radii;  /* [P]     0 = not rendered */
} DgrImages;

/* == upstream gradients into the backward; any pointer may be NULL (= zeros) == */
typedef struct DgrImageGrads {
    const float *dL_dcolor; /* [3,H,W] */
    const float *dL_ddepth; /* [1,H,W] */
    const float *dL_dalpha; /* [1,H,W] */
} DgrImageGrads;

/* Multi-GPU, view-sharded (SURVEY.md §8e): lets the per-Gaussian backward deliver gradient rows straight to the rank that OWNS
 * them.  Gaussian g belongs to rank g / gaussians_per_owner (a positive multiple of 256 with gaussians_per_owner * world >= P).
 * All the gradient pointers of the call must then lie in ONE local flat buffer, and delta_floats[o] is the distance, in
 * floats, from any address in that buffer to the same element of THIS rank's slot in rank o's staging area (peer-mapped
 * symmetric memory); delta_floats[rank] = 0.  With it the backward writes, for every Gaussian of another owner,
 * (accumulate ? what the local buffer holds : 0) + this view's gradient to the owner instead of to the local buffer — the
 * reduce-scatter half of the all-reduce rides on the kernel; dgr_peer_reduce_staged() finishes the sum. */
typedef struct DgrPeerPush {
    int32_t world, rank;
    int64_t gaussians_per_owner;
    int64_t delta_floats[16];
} DgrPeerPush;

/* == gradients w.r.t. the inputs; any pointer may be NULL (= not wanted) == */
typedef struct DgrGaussianGrads {
    float *dL_dmeans3D;        /* [P,3]   */
    float *dL_dmeans2D;        /* [P,3]   NDC units, z = 0 (gs_renderer.py:626 reads [:, :2]) */
    float *dL_dshs;            /* [P,M,3] */
    float *dL_dcolors_precomp; /* [P,3]   */
    float *dL_dopacities;      /* [P,1]   */
    float *dL_dscales;         /* [P,3]   */
    float *dL_drotations;      /* [P,4]   */
    float *dL_dcov3D_precomp;  /* [P,6]   */
    int32_t accumulate;        /* 0: overwrite; 1: add into the buffers (several views -> one flat gradient) */
    float *dL_dshs_rest;       /* [P,M-1,3] with DgrGaussians.activations (then dL_dshs is [P,1,3]); else unused */
    /* Densification bookkeeping fused into the per-Gaussian backward (gs_renderer.py:625-627, main.py:279-281); each may
     * be NULL.  For every Gaussian with radii > 0 in this render: xyz_gradient_accum += |dL/dmeans2D[:, :2]| (this
     * render's gradient), denom += 1, max_radii2D = max(max_radii2D, radii).  All float32 [P] (the reference's [P,1]). */
    float *xyz_gradient_accum;
    float *denom;
    float *max_radii2D;
    const DgrPeerPush *push;   /* NULL: everything goes to the local buffers */
} DgrGaussianGrads;

/* Scratch sizes.  The caller owns the three scratch buffers (upstream: geomBuffer / binningBuffer / imgBuffer),
 * must keep them alive and untouched between a forward and its backward, and aligns them to 256 bytes. */
size_t dgr_geom_bytes(int32_t P, int32_t image_height, int32_t image_width);
size_t dgr_image_bytes(int32_t image_height, int32_t image_width);
size_t dgr_binning_bytes(uint64_t capacity_instances, int32_t image_height, int32_t image_width);

/* Forward, stage 1: per-Gaussian preprocess (cull, EWA cov2D, conic, radius, SH->RGB, opacity-aware pixel AABB)
 * fused with the per-tile instance histogram (kept in `image` scratch).  Writes radii. */
int dgr_forward_preprocess(const DgrSettings *s, const DgrGaussians *g, void *geom, void *image, int32_t *radii,
                           void *stream);

/* Forward, stage 2: tile ranges (device-side scans), instance emission, per-tile depth sort + record gather, and the
 * per-tile front-to-back compositing.  Nothing here waits for the host.  Two things are guessed by the caller:
 *   - `capacity_instances`, the instance capacity `binning` was sized for;
 *   - DGR_FLAG_BIG_TILES in `flags`: whether to also launch the sorter for tiles with more than 4096 instances.
 * The truth is written to geom scratch and, if counts_host != NULL (pinned host memory, 4 x uint64), made available to
 * the host right after the scan: counts_host[0] = instance count, counts_host[1] = number of big tiles.  Two protocols:
 *   ticket == 0: an asynchronous copy, then count_ready_event (from dgr_event_create, may be NULL) is recorded — the caller
 *                keeps enqueuing work and checks the guesses once that event has fired;
 *   ticket != 0: the scan kernel stores the two counts and then counts_host[2] = ticket straight into the caller's memory
 *                (which must therefore be device-mapped pinned memory — under unified addressing every cudaHostAlloc /
 *                torch pin_memory buffer is); the caller polls counts_host[2] for the ticket value it chose for THIS call.
 *                No copy or event sits between the kernels then, so the whole forward chains with programmatic dependent
 *                launches (each kernel's prologue overlaps its predecessor's tail); count_ready_event is ignored.  If counts_host[0] > capacity_instances, or counts_host[1] > 0 without
 * DGR_FLAG_BIG_TILES, the call produced a memory-safe but wrong image: re-run stage 2 with corrected guesses and
 * DGR_FLAG_RERUN set. */
#define DGR_FLAG_BIG_TILES 1
#define DGR_FLAG_RERUN 2      /* set when stage 2 is repeated for the same stage 1 (corrected guesses) */
int dgr_forward_render(const DgrSettings *s, const DgrGaussians *g, void *geom, void *binning,
                       uint64_t capacity_instances, void *image, const DgrImages *out, int32_t flags,
                       uint64_t *counts_host, uint64_t ticket, void *count_ready_event, void *stream);

/* Tuning knobs (process-wide atomics; results do not depend on them beyond the summation order of the gradient atomics):
 * pixels per lane of the forward / backward render kernels (1, 2 or 4; the backward has 1 and 2) and a bit field:
 *   bit 3        programmatic dependent launches OFF (the environment variable DGR_PDL=0 does the same)
 *   bits 4-6     hits the forward evaluates together (1, 2, 4; 0 = default)      bits 8-10   the same for the backward
 *   bits 12-15   persistent CTAs per SM of the forward render kernel (0 = as many as fit)     bits 16-19   backward
 *   bit 20       render work queue consumed from both ends (experiment, measured slower)
 *   bit 21       backward work in tile-population order instead of the cost the forward measured
 *   bits 22-23   record staging of the render kernels: 0 = automatic (by Gaussian id when the sorted copy would exceed twice
 *                the L2 size), 1 = always the sorted copy, 2 = always by id
 *   bit 24 / 25  the per-Gaussian forward / backward kernel reads its inputs with per-thread global loads instead of staging
 *                each warp's 32 contiguous Gaussians through shared memory with bulk TMA (A/B switch; the staged path needs
 *                SH + scale / rotation inputs and 16-byte aligned base pointers and is otherwise not taken anyway)
 *   bit 26       step 2 of the backward render kernel in its per-pixel form (A/B switch; default sub-tile shape only)
 * the other bits are accepted and ignored. */
int dgr_set_tuning(int ppl_fwd, int ppl_bwd, int tile_order);

/* Thin cudaEvent wrappers so a host without the CUDA runtime headers (ctypes, cgo ...) can use the protocol above. */
void *dgr_event_create(void);
int dgr_event_synchronize(void *event);
void dgr_event_destroy(void *event);

/* Backward of both stages.  geom / binning / image are the scratch buffers of the matching forward
 * (`capacity_instances` = the value stage 2 ran with); geom is also used as scratch for the per-Gaussian
 * reduction.  `out_alpha` is the alpha image the forward produced (accepted for signature parity with the
 * reference binding; the final transmittance is kept in `image` at full precision instead of 1 - alpha). */
int dgr_backward(const DgrSettings *s, const DgrGaussians *g, void *geom, const void *binning,
                 uint64_t capacity_instances, const void *image, const int32_t *radii, const float *out_alpha,
                 const DgrImageGrads *gin, const DgrGaussianGrads *gout, void *stream);

/* == Batched views: V cameras (1 <= V <= 16) of ONE cloud at ONE resolution ==
 * A batch gives what V single-view calls give when their backwards accumulate into the same gradient buffers, but the
 * per-Gaussian stages read the inputs once for all views and write the summed gradient once.
 *   - s is a HOST array of V DgrSettings.  image_height / image_width, sh_degree, scale_modifier, prefiltered and debug must be
 *     equal in all of them; tanfovx / tanfovy, bg, viewmatrix, projmatrix and campos may differ.
 *   - g: SHs (plain or raw, DgrGaussians.activations) and scales / rotations; colors_precomp / cov3D_precomp are rejected.
 *     Every per-Gaussian input pointer must be 16-byte aligned (misaligned input is rejected).
 *   - Scratch: ONE geom allocation of dgr_batch_geom_bytes(V, P, H, W) and ONE image allocation of dgr_batch_image_bytes(V, H, W);
 *     view v's geom scratch starts at geom + v * dgr_geom_bytes(P, H, W) and its image scratch at image + v * dgr_image_bytes(H, W)
 *     (both strides are multiples of 256 bytes; the base pointers are 256-byte aligned).  Each view has its own binning buffer.
 *   - radii is [V, P] int32 (view v at radii + v * P).
 * dgr_forward_preprocess_batch leaves in every view's scratch exactly what dgr_forward_preprocess leaves there for that view; stage
 * 2 of view v is then dgr_forward_render(&s[v], g, view v's geom, view v's binning, ..., view v's image, ...) as for one view.
 * dgr_backward_batch runs the backward render of every view (binning[v] / capacity[v]: HOST arrays, the buffers and capacities
 * stage 2 of view v ran with) and then ONE per-Gaussian backward over all views.  gin is a HOST array of V DgrImageGrads.  gout:
 * means3D / shs (/ shs_rest) / opacities / scales / rotations gradients summed over the views (written, or added with accumulate);
 * dL_dmeans2D is [V, P, 3], per view; xyz_gradient_accum / denom / max_radii2D are updated once per view with radii > 0, as V
 * single-view backwards do; dL_dcolors_precomp / dL_dcov3D_precomp are unused and push must be NULL. */
size_t dgr_batch_geom_bytes(int32_t num_views, int32_t P, int32_t image_height, int32_t image_width);
size_t dgr_batch_image_bytes(int32_t num_views, int32_t image_height, int32_t image_width);
int dgr_forward_preprocess_batch(const DgrSettings *s, int32_t num_views, const DgrGaussians *g, void *geom, void *image,
                                 int32_t *radii, void *stream);
int dgr_backward_batch(const DgrSettings *s, int32_t num_views, const DgrGaussians *g, void *geom, void *const *binning,
                       const uint64_t *capacity_instances, const void *image, const int32_t *radii, const DgrImageGrads *gin,
                       const DgrGaussianGrads *gout, void *stream);

/* Multi-GPU (view-sharded data parallelism, SURVEY.md §8e): all-reduce(sum) of the flat float32 gradient buffer over
 * NVLink with this library's own kernel.  The buffer lives in symmetric memory: peer_ptrs[w] (HOST array of `world` device
 * addresses) is rank w's copy mapped into this process; multicast_ptr, if non-zero, is the NVSwitch multicast address of
 * the same buffer (then multimem.ld_reduce / multimem.st are used and peer_ptrs may be NULL).  n_floats % 4 == 0.
 * peer_flag_ptrs (HOST array of `world` device addresses, or NULL): rank w's flag area of dgr_peer_flag_bytes() bytes in
 * the same symmetric allocation, zero-initialised once; with it the kernel carries its own two cross-rank barriers and
 * `epoch` must be 1, 2, 3, ... over successive calls (the same value on every rank).  With NULL the caller synchronises the
 * ranks (device-side barrier) before and after the call. */
size_t dgr_peer_flag_bytes(void);
int dgr_peer_allreduce(const uint64_t *peer_ptrs, int32_t world, int32_t rank, uint64_t n_floats, uint64_t multicast_ptr,
                       const uint64_t *peer_flag_ptrs, uint32_t epoch, void *stream);

/* The all-reduce split in two, its first half fused into the backward (DgrPeerPush): every rank has pushed the rows it does not own;
 * this call makes rank `push->rank` add the `world` staged copies of ITS rows (stage_ptr: local address of its staging area,
 * slot s at stage_ptr + s * padded_floats floats; its own contribution is read from its flat buffer peer_ptrs[rank]) in rank order
 * and publish the sums to every rank's flat buffer (multicast_ptr != 0: multimem.st; else stores to peer_ptrs[w]).  The flat buffer is
 * n_seg (<= 8) segments [P, seg_stride[k]] starting at float seg_off[k].  peer_flag_ptrs / epoch as for dgr_peer_allreduce (NULL: the
 * caller synchronises the ranks before and after).  dgr_peer_push_flat does the push for a rank that has no backward to ride on
 * (no view this iteration): it copies the rows of other owners from `local` (its flat buffer) to their owners. */
int dgr_peer_reduce_staged(const uint64_t *peer_ptrs, const DgrPeerPush *push, int64_t P, int32_t n_seg, const int64_t *seg_off,
                           const int32_t *seg_stride, uint64_t stage_ptr, uint64_t padded_floats, uint64_t multicast_ptr,
                           const uint64_t *peer_flag_ptrs, uint32_t epoch, void *stream);
int dgr_peer_push_flat(const float *local, const DgrPeerPush *push, int64_t P, int32_t n_seg, const int64_t *seg_off,
                       const int32_t *seg_stride, void *stream);

/* SURVEY.md §8 row f3 — replaces simple_knn._C.distCUDA2 (/root/reference/simple-knn/spatial.cu:15-26 -> SimpleKNN::knn,
 * simple_knn.cu:185-221; caller gs_renderer.py:341): mean_dists[i] = mean of the squared distances from point i to its 3
 * nearest OTHER points (exact; a point set smaller than 4 yields the reference's FLT_MAX arithmetic).  points [P,3] float32.
 * scratch: dgr_knn_scratch_bytes(P) bytes of device memory.  Stream-ordered, no host synchronisation, no library sort. */
size_t dgr_knn_scratch_bytes(int32_t P);
int dgr_dist_cuda2(int32_t P, const float *points, float *mean_dists, void *scratch, void *stream);

/* SURVEY.md §8 row f4 — GaussianModel.extract_fields (/root/reference/gs_renderer.py:218-294; gaussian_3d_coeff :64-83):
 * occ[resolution^3] (x-major, z fastest) = per-voxel sum of opacity * exp(-1/2 d^T Sigma^-1 d) over the Gaussians with
 * sigmoid(opacity) > 0.005 whose normalised centre lies strictly inside the voxel's block's bounding box grown by
 * relax_ratio * 2/num_blocks.  Inputs are the RAW model tensors (_xyz [P,3], _opacity [P,1], _scaling [P,3], _rotation
 * [P,4]); center_scale (device, 4 floats, may be NULL) receives the model's `center` and `scale` (:237-238).
 * resolution % num_blocks == 0, num_blocks <= 64, (resolution/num_blocks)^3 <= 4096.  Stream-ordered, no host read-back. */
size_t dgr_fields_scratch_bytes(int32_t P, int32_t num_blocks);
int dgr_extract_fields(int32_t P, const float *xyz, const float *opacity_raw, const float *scaling_raw, const float *rotation_raw,
                       int32_t resolution, int32_t num_blocks, float relax_ratio, float *occ, float *center_scale, void *scratch,
                       void *stream);

/* SURVEY.md §8 row f2 — the optimiser step of the stage-1 loop: torch.optim.Adam(lr per group, eps) over the model's six
 * parameter tensors (/root/reference/gs_renderer.py:361-370, stepped at main.py:274-276) as ONE launch.  bias correction 1 - beta^step per tensor; no weight decay, no amsgrad.  betas / eps are doubles because torch derives 1 - beta and
 * the bias corrections in double before rounding to float32.  Updates param / exp_avg / exp_avg_sq in place. */
typedef struct DgrAdamGroup {
    float *param;
    const float *grad;
    float *exp_avg;
    float *exp_avg_sq;
    uint64_t n;       /* elements */
    float lr;
    int32_t step;     /* this tensor's own step count after the update, from 1 (torch keeps state['step'] per tensor: a tensor
                       * whose .grad was None in some iteration lags behind) */
} DgrAdamGroup;
int dgr_adam_step(const DgrAdamGroup *groups, int32_t n_groups, double beta1, double beta2, double eps, void *stream);

/* SURVEY.md §8 row f2 — the reference's densify_and_prune (/root/reference/gs_renderer.py:586-609 = densify_and_clone
 * :582-600 + densify_and_split :555-580 + prune_points :509-513, with the optimizer-state surgery of :464-552) as stream
 * compaction.  Two calls with ONE host read-back between them (the new point count sizes the output tensors):
 *   dgr_densify_plan   classifies every point (grad = xyz_gradient_accum / denom, NaN -> 0; clone if |grad| >= grad_threshold
 *                      and max(exp(scaling)) <= dense_extent; split if grad >= grad_threshold and max > dense_extent; pruned
 *                      if sigmoid(opacity) < min_opacity or — when use_world != 0, the reference's `if max_screen_size:` —
 *                      max(exp(scaling)) > max_world; max_radii2D never matters: densification_postfix has zeroed it, :551)
 *                      and copies counts_host[4] = { kept originals, surviving clones, points selected for the split,
 *                      surviving children per copy } (pinned host memory) — new point count = [0] + [1] + 2 * [3].
 *   dgr_densify_apply  writes the new tensors in the reference's order (kept originals, clones, first children, second
 *                      children): the six parameter tensors and both Adam moments (zero for new points).  A child's position is
 *                      xyz + R(q/|q|) (noise[child * counts[2] + rank] * exp(scaling)), its scaling log(exp(scaling) / 1.6);
 *                      noise = standard normals [2 * counts[2], 3] (device), rank = the point's rank among the selected.
 * Tensor order in DgrDensifyTensors: xyz, f_dc, f_rest, opacity, scaling, rotation; width = floats per point (f_rest may be 0). */
typedef struct DgrDensifyTensors {
    const float *in[6], *exp_avg_in[6], *exp_avg_sq_in[6];
    float *out[6], *exp_avg_out[6], *exp_avg_sq_out[6];
    int32_t width[6];
} DgrDensifyTensors;
size_t dgr_densify_scratch_bytes(int32_t P);
int dgr_densify_plan(int32_t P, const float *xyz_gradient_accum, const float *denom, const float *opacity_raw, const float *scaling_raw,
                     float grad_threshold, float dense_extent, float min_opacity, float max_world, int32_t use_world,
                     void *scratch, uint32_t *counts_host, void *stream);
int dgr_densify_apply(int32_t P, const DgrDensifyTensors *t, const float *noise, const void *scratch, void *stream);

/* GaussianRasterizer.markVisible: present[i] = 1 if Gaussian i passes the near-plane test. */
int dgr_mark_visible(int32_t P, const float *means3D, const float *viewmatrix, const float *projmatrix,
                     uint8_t *present, void *stream);

/* Introspection for tests: copies per-Gaussian forward state out of geom scratch (any pointer may be NULL):
 * mean_px [P,2], depth [P], conic [P,3] (natural units), rgb [P,3], opacity-aware pixel AABB [P,4] int32. */
int dgr_debug_geom(int32_t P, int32_t image_height, int32_t image_width, const void *geom, float *mean_px, float *depth, float *conic, float *rgb,
                   int32_t *aabb, uint32_t *tiles_touched, void *stream);

/* How many kernels of THIS library were launched by the calling thread since the last reset (for bench.py). */
uint64_t dgr_launch_count(void);
void dgr_reset_launch_count(void);

/* Per-kernel CUDA-event timing (tracing hook): when enabled, every kernel this thread launches is bracketed by
 * events on its stream; dgr_profile_collect waits for them and returns (name, ms) pairs, names '\n'-joined. */
void dgr_profile_enable(int on);
int dgr_profile_collect(char *names, size_t names_bytes, float *ms, int max);

int dgr_abi_version(void);
const char *dgr_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* DGR_B200_H */
