// dgr_lib.cu — the translation unit of libdgr_b200.so: the single-view C ABI (dgr_api.cu, included as it is) followed by the
// batched multi-view entry points (include/dgr_b200.h, "Batched views"), which reuse its launch helpers, tuning knobs and
// per-device state.
#include "dgr_api.cu"
#include "dgr_multiview.cuh"

namespace {

// dynamic shared memory of one forward CTA: 2 CTAs per SM (228 KB per SM; per CTA 1 KB is reserved and 2.7 KB are static)
constexpr size_t kMvFwdSmemBudget = 110 * 1024;

int check_batch(const DgrSettings *s, int32_t V, const DgrGaussians *g) {
    if (!s) return fail(-1, "settings is NULL");
    if (V < 1 || V > kMaxBatchViews) return fail(-1, "batch: 1 to 16 views");
    for (int v = 0; v < V; v++) {
        if (int e = check_settings(s + v)) return e;
        const DgrSettings &a = s[0], &b = s[v];
        if (a.image_height != b.image_height || a.image_width != b.image_width || a.sh_degree != b.sh_degree ||
            a.scale_modifier != b.scale_modifier || (a.prefiltered != 0) != (b.prefiltered != 0) || (a.debug != 0) != (b.debug != 0))
            return fail(-1, "batch: image size, sh_degree, scale_modifier, prefiltered and debug must be the same for every view");
        if (!b.campos) return fail(-1, "campos must not be NULL with SHs");
    }
    if (int e = check_gaussians(s, g)) return e;
    if (g->colors_precomp || g->cov3D_precomp)
        return fail(-2, "batch: colors_precomp / cov3D_precomp are not supported; pass SHs and scales / rotations");
    if (g->P == 0) return 0;
    if (!g->shs || !g->scales || !g->rotations) return fail(-2, "batch: SHs and scales / rotations are required");
    uintptr_t bits = (uintptr_t)g->means3D | (uintptr_t)g->scales | (uintptr_t)g->rotations | (uintptr_t)g->opacities | (uintptr_t)g->shs;
    if (g->activations && g->M > 1) bits |= (uintptr_t)g->shs_rest;
    if (bits & 15u) return fail(-1, "batch: every per-Gaussian input pointer must be 16-byte aligned");
    return 0;
}

MvViews make_views(const DgrSettings *s, int V) {
    MvViews w;
    memset(&w, 0, sizeof(w));
    for (int v = 0; v < V; v++) w.v[v] = MvView{ s[v].viewmatrix, s[v].projmatrix, s[v].campos, s[v].tanfovx, s[v].tanfovy };
    return w;
}

MvScratch make_scratch(char *geom, char *image, const GeomLayout &GL, const ImageLayout &IL) {
    MvScratch sc;
    sc.geom = geom; sc.geom_stride = GL.total; sc.image = image; sc.image_stride = IL.total;
    sc.off_rec = GL.off_rec; sc.off_touched = GL.off_touched; sc.off_gradrec = GL.off_gradrec; sc.off_runs = GL.off_runs;
    sc.off_count = IL.off_count;
    return sc;
}

// views per launch of the forward kernel: as many tile histograms as fit next to the staging slices in the 2-CTA budget (at least 1)
int mv_fwd_group(int tiles, int M) {
    const size_t stage = (size_t)(kPreThreads / 32) * stage_warp_floats(M) * 4;
    const size_t per_view = (size_t)tiles * 4;
    const size_t room = kMvFwdSmemBudget > stage + 128 ? kMvFwdSmemBudget - stage - 128 : 0;
    const size_t n = room / per_view;
    return n < 1 ? 1 : (n > (size_t)kMaxBatchViews ? kMaxBatchViews : (int)n);
}

template <int DEG, bool RAW>
int launch_mv_fwd(const DgrSettings *s, int V, const DgrGaussians *g, const MvViews &views, const MvScratch &sc, const GeomLayout &L,
                  int32_t *radii, cudaStream_t st) {
    const int G = mv_fwd_group(L.tiles, g->M);
    for (int v0 = 0; v0 < V; v0 += G) {
        const int nv = min(G, V - v0);
        const size_t stage_off = align_up((size_t)nv * L.tiles * 4, 128);
        const size_t smem = stage_off + (size_t)(kPreThreads / 32) * stage_warp_floats(g->M) * 4;
        if (smem + 1024 > kMaxKernelSmem) return fail(-3, "batch: image has too many tiles for the batched preprocess");
        auto kernel = preprocess_fwd_multiview_kernel<DEG, RAW>;
        if (smem > 48 * 1024) DGR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        DGR_KERNEL("preprocess_fwd_multiview", st, s->debug,
                   launch_k(kernel, dim3(L.nblocks), dim3(kPreThreads), smem, st, false, g->P, g->M, s->image_height, s->image_width,
                            s->scale_modifier, views, v0, nv, g->means3D, g->shs, g->shs_rest, g->opacities, g->scales, g->rotations,
                            radii, sc, L.tiles, L.iters, (int)stage_off));
    }
    return 0;
}

template <int DEG, bool RAW>
int launch_mv_bwd(const DgrSettings *s, int V, const DgrGaussians *g, const MvViews &views, const MvScratch &sc, const int32_t *radii,
                  const MvGrads &out, int accumulate, bool pdl, cudaStream_t st) {
    const int wfl = mv_bwd_warp_floats(g->M, RAW);
    const size_t smem = (size_t)(kPreThreads / 32) * wfl * 4;
    auto kernel = preprocess_bwd_multiview_kernel<DEG, RAW>;
    if (smem > 48 * 1024) DGR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int nb = (g->P + kPreThreads - 1) / kPreThreads;
    DGR_KERNEL("preprocess_bwd_multiview", st, s->debug,
               launch_k(kernel, dim3(nb), dim3(kPreThreads), smem, st, pdl, g->P, g->M, s->image_height, s->image_width, s->scale_modifier,
                        views, V, g->means3D, g->shs, g->shs_rest, g->opacities, g->scales, g->rotations, radii, sc, out, accumulate, wfl));
    return 0;
}

#define DGR_MV_DISPATCH(FN, ...)                                                                          \
    (g->activations ? (s->sh_degree == 0 ? FN<0, true>(__VA_ARGS__) : s->sh_degree == 1 ? FN<1, true>(__VA_ARGS__)     \
                                          : s->sh_degree == 2 ? FN<2, true>(__VA_ARGS__) : FN<3, true>(__VA_ARGS__))   \
                    : (s->sh_degree == 0 ? FN<0, false>(__VA_ARGS__) : s->sh_degree == 1 ? FN<1, false>(__VA_ARGS__)   \
                                          : s->sh_degree == 2 ? FN<2, false>(__VA_ARGS__) : FN<3, false>(__VA_ARGS__)))

// The backward render kernel of one view into that view's moment records: the launch dgr_backward makes, with the same
// variant selection (tuning knobs) and the same record staging rule.
int render_bwd_view(const DgrSettings *s, char *geom, const char *binning, uint64_t capacity, const char *image, const DgrImageGrads *gin,
                    int P, cudaStream_t st) {
    const int H = s->image_height, W = s->image_width;
    GeomLayout GL(P, H, W);
    ImageLayout IL(H, W);
    BinningLayout BL(capacity);
    const int tiles = IL.gx * IL.gy;
    float *grad_rec = reinterpret_cast<float *>(geom + GL.off_gradrec);
    DevInfo *dv = dev_info();
    if (!dv) return -1;
    const TileWork *work = reinterpret_cast<const TileWork *>(image + IL.off_work);
    unsigned long long *bwd_next = reinterpret_cast<unsigned long long *>(geom + GL.off_bwdwork);
    const int ppl = g_ppl_bwd.load(), ub = g_u_bwd.load();
    CostOrder co{};
    if (g_cost_order.load()) {
        TileWork *wk = const_cast<TileWork *>(work);
        co.cost_acc = const_cast<unsigned *>(reinterpret_cast<const unsigned *>(image + IL.off_cost)); co.cls_count = wk->cls_count;
        co.cls_items = const_cast<unsigned *>(reinterpret_cast<const unsigned *>(image + IL.off_clsitems)); co.cost_bpt = &wk->cost_bpt;
        co.tiles = tiles; co.bwd_ppl = ppl == 1 ? 1 : 2;
    }
    const int lz = g_lazy.load();
    const bool lazy = lz == 2 || (lz == 0 && (size_t)capacity * sizeof(Rec) > 2 * dv->l2_bytes);
#define DGR_MV_RENDER_BWD_K(KERNEL_, PPL_)                                                                               \
    do {                                                                                                                 \
        const size_t smem_ = sizeof(BwdSmem<PPL_>) * kRenderWarps;                                                       \
        int grid_ = min(persistent_grid(dv, KERNEL_, kRenderThreads, smem_), (tiles * SubTile<PPL_>::kPerTile + kRenderWarps - 1) / kRenderWarps); \
        if (g_cta_bwd.load() > 0) grid_ = min(grid_, g_cta_bwd.load() * dv->sms);                                        \
        DGR_KERNEL("render_bwd", st, s->debug,                                                                           \
                   launch_k(KERNEL_, dim3((unsigned)grid_), dim3(kRenderThreads), smem_, st, false, H, W, IL.gx,         \
                            reinterpret_cast<const unsigned *>(image + IL.off_order), &work->n_nonempty, bwd_next, g_two_ended.load(), dv->sms, co, \
                            reinterpret_cast<const uint2 *>(image + IL.off_oranges),                                     \
                            reinterpret_cast<const Rec *>(binning + BL.off_rec), reinterpret_cast<const Rec *>(geom + GL.off_rec), \
                            (const unsigned *)&work->lazy, reinterpret_cast<const unsigned *>(binning + BL.off_ids),        \
                            s->bg, reinterpret_cast<const float *>(image + IL.off_finalT),                               \
                            reinterpret_cast<const unsigned *>(image + IL.off_ncontrib), gin->dL_dcolor, gin->dL_ddepth, gin->dL_dalpha, grad_rec)); \
    } while (0)
#define DGR_MV_RENDER_BWD(PPL_, U_) do { if (lazy) DGR_MV_RENDER_BWD_K((render_bwd_kernel<PPL_, U_, true>), PPL_); \
                                         else DGR_MV_RENDER_BWD_K((render_bwd_kernel<PPL_, U_, false>), PPL_); } while (0)
    if (ppl == 1 && ub != 1 && !lazy && !g_rowsum.load()) DGR_MV_RENDER_BWD_K((render_bwd_kernel<1, 2, false, false>), 1);
    else if (ppl == 1) { if (ub == 1) DGR_MV_RENDER_BWD(1, 1); else DGR_MV_RENDER_BWD(1, 2); }
    else { if (ub == 2) DGR_MV_RENDER_BWD(2, 2); else DGR_MV_RENDER_BWD(2, 1); }
#undef DGR_MV_RENDER_BWD
#undef DGR_MV_RENDER_BWD_K
    return 0;
}

}  // namespace

extern "C" {

size_t dgr_batch_geom_bytes(int32_t V, int32_t P, int32_t H, int32_t W) { return (size_t)(V > 0 ? V : 0) * GeomLayout(P, H, W).total; }
size_t dgr_batch_image_bytes(int32_t V, int32_t H, int32_t W) { return (size_t)(V > 0 ? V : 0) * ImageLayout(H, W).total; }

int dgr_forward_preprocess_batch(const DgrSettings *s, int32_t V, const DgrGaussians *g, void *geom_v, void *image_v, int32_t *radii,
                                 void *stream) {
    NvtxRange nvtx_("dgr_forward_preprocess_batch");
    if (int e = check_batch(s, V, g)) return e;
    cudaStream_t st = (cudaStream_t)stream;
    char *geom = (char *)geom_v, *image = (char *)image_v;
    if (!geom || !image) return fail(-1, "geom / image scratch is NULL");
    GeomLayout L(g->P, s->image_height, s->image_width);
    ImageLayout IL(s->image_height, s->image_width);
    if ((size_t)L.tiles * 4 > kMaxTileSmem) return fail(-3, "image has more than 51200 tiles (16x16): not supported");
    // every view's work block + per-tile totals + backward cost accumulators (what dgr_forward_preprocess zeroes): one 2-D memset
    DGR_CUDA(cudaMemset2DAsync(image + IL.off_work, IL.total, 0, (IL.off_cost - IL.off_work) + (size_t)L.tiles * 8 * 4, (size_t)V, st));
    if (g->P == 0) return 0;
    if (!radii) return fail(-1, "radii is NULL");
    const MvViews views = make_views(s, V);
    const MvScratch sc = make_scratch(geom, image, L, IL);
    return DGR_MV_DISPATCH(launch_mv_fwd, s, V, g, views, sc, L, radii, st);
}

int dgr_backward_batch(const DgrSettings *s, int32_t V, const DgrGaussians *g, void *geom_v, void *const *binning, const uint64_t *capacity,
                       const void *image_v, const int32_t *radii, const DgrImageGrads *gin, const DgrGaussianGrads *gout, void *stream) {
    NvtxRange nvtx_("dgr_backward_batch");
    if (int e = check_batch(s, V, g)) return e;
    if (!geom_v || !image_v || !gin || !gout || !binning || !capacity) return fail(-1, "NULL argument");
    if (gout->push) return fail(-2, "batch: DgrGaussianGrads.push is not supported");
    if (g->P == 0) return 0;
    if (!radii) return fail(-1, "radii is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    char *geom = (char *)geom_v;
    const char *image = (const char *)image_v;
    GeomLayout GL(g->P, s->image_height, s->image_width);
    ImageLayout IL(s->image_height, s->image_width);
    // every view's work counter + moment accumulators: one 2-D memset
    DGR_CUDA(cudaMemset2DAsync(geom + GL.off_bwdwork, GL.total, 0, (GL.off_gradrec - GL.off_bwdwork) + (size_t)g->P * kGradRecFloats * 4,
                               (size_t)V, st));
    bool last_kernel = false;        // the launch right before the per-Gaussian kernel was a kernel: it may chain with PDL
    for (int v = 0; v < V; v++) {
        last_kernel = false;
        if (binning[v] && capacity[v] > 0) {
            if (int e = render_bwd_view(s + v, geom + (size_t)v * GL.total, (const char *)binning[v], capacity[v], image + (size_t)v * IL.total,
                                        gin + v, g->P, st))
                return e;
            last_kernel = true;
        }
    }
    const MvViews views = make_views(s, V);
    const MvScratch sc = make_scratch(geom, const_cast<char *>(image), GL, IL);
    MvGrads out;
    out.dL_dmeans3D = gout->dL_dmeans3D; out.dL_dmeans2D = gout->dL_dmeans2D; out.dL_dshs = gout->dL_dshs;
    out.dL_dopacities = gout->dL_dopacities; out.dL_dscales = gout->dL_dscales; out.dL_drotations = gout->dL_drotations;
    out.dL_dshs_rest = (g->activations && g->M > 1) ? gout->dL_dshs_rest : nullptr;
    out.xyz_gradient_accum = gout->xyz_gradient_accum; out.denom = gout->denom; out.max_radii2D = gout->max_radii2D;
    return DGR_MV_DISPATCH(launch_mv_bwd, s, V, g, views, sc, radii, out, gout->accumulate, last_kernel, st);
}

}  // extern "C"
