// dgr_multiview.cuh — the per-Gaussian kernels of a BATCH of V views of one cloud (1 <= V <= 16, one resolution).
//
// A loop of V single-view calls reads every Gaussian's inputs (44 + 12 M bytes) V times in the forward preprocess and again V
// times in the backward preprocess, and read-modify-writes the whole gradient V times (accumulate).  Here a warp stages its 32
// Gaussians' inputs ONCE with the bulk-TMA helpers of dgr_preprocess.cuh, applies the activations and builds what does not
// depend on the view once, and then produces every view from registers:
//   forward:  view v's records / touched / radii / per-tile totals / run-matrix rows, exactly where dgr_forward_preprocess
//             leaves them in view v's scratch (so stage 2 of view v is the unchanged dgr_forward_render);
//   backward: view v's chain rule from view v's moment records, summed over the views in the warp's shared-memory output image,
//             which leaves ONCE with 16-byte stores; means2D gradients and densification statistics per view.
// The per-view arithmetic is the single-view kernels' (same __device__ functions, same expressions in the same order): results
// differ from them only where ptxas fuses a multiply-add pair differently in this instantiation.
//
// Tile histograms of the forward: every view needs its own per-block histogram for the whole block range (the run-matrix row of
// a block covers all its Gaussians).  They live in shared memory next to the staging slices; when V x tiles counters do not fit
// the budget of two CTAs per SM the host launches the kernel once per GROUP of views that does (inputs then read once per group).
#pragma once
#include "dgr_backward.cuh"

namespace dgr {

constexpr int kMaxBatchViews = 16;

struct MvView { const float *V, *PM, *cam; float tanfovx, tanfovy; };
struct MvViews { MvView v[kMaxBatchViews]; };

// view v's scratch: geom at geom + v * geom_stride, image at image + v * image_stride (GeomLayout / ImageLayout of (P, H, W))
struct MvScratch {
    char *geom; size_t geom_stride;
    char *image; size_t image_stride;
    size_t off_rec, off_touched, off_gradrec, off_runs, off_count;
};

struct MvFrame { FrameConsts fc; float tanfovx, tanfovy, pad[2]; };

__device__ __forceinline__ void load_frames(MvFrame *fr, const MvViews &vw, int v0, int nv) {
    for (int i = threadIdx.x; i < nv * 37; i += blockDim.x) {
        const int v = i / 37, j = i - v * 37;
        const MvView &x = vw.v[v0 + v];
        if (j < 16) fr[v].fc.V[j] = __ldg(x.V + j);
        else if (j < 32) fr[v].fc.PM[j - 16] = __ldg(x.PM + j - 16);
        else if (j < 35) fr[v].fc.cam[j - 32] = __ldg(x.cam + j - 32);
        else if (j == 35) fr[v].tanfovx = x.tanfovx;
        else fr[v].tanfovy = x.tanfovy;
    }
}

// One warp's inputs into registers: staged (full warp, already in flight on wbar) or per-thread loads (partial last warp).
template <int DEG, bool RAW>
__device__ __forceinline__ void mv_load_inputs(bool staged, const float *ws, int g, int M, const float *means3D, const float *shs,
                                               const float *shs_rest, const float *opacities, const float *scales, const float *rotations,
                                               float3 &p, float3 &s_in, float4 &q_in, float &o_in, float &dc0, float &dc1, float &dc2,
                                               float (&shc)[48]) {
    const int lane = threadIdx.x & 31;
    if (staged) {
        p = make_float3(ws[kStgMean + 3 * lane], ws[kStgMean + 3 * lane + 1], ws[kStgMean + 3 * lane + 2]);
        s_in = make_float3(ws[kStgScale + 3 * lane], ws[kStgScale + 3 * lane + 1], ws[kStgScale + 3 * lane + 2]);
        q_in = *reinterpret_cast<const float4 *>(ws + kStgRot + 4 * lane);
        o_in = ws[kStgOp + lane];
        if (RAW) {
            dc0 = ws[kStgSh + 3 * lane]; dc1 = ws[kStgSh + 3 * lane + 1]; dc2 = ws[kStgSh + 3 * lane + 2];
            if (DEG > 0) lds_sh_row<DEG, 1>(ws + kStgSh + 96 + lane * (M - 1) * 3, ((M - 1) & 3) == 0, shc);
        } else lds_sh_row<DEG>(ws + kStgSh + lane * M * 3, (M & 3) == 0, shc);
    } else {
        p = make_float3(__ldg(means3D + 3 * (size_t)g), __ldg(means3D + 3 * (size_t)g + 1), __ldg(means3D + 3 * (size_t)g + 2));
        s_in = make_float3(__ldg(scales + 3 * (size_t)g), __ldg(scales + 3 * (size_t)g + 1), __ldg(scales + 3 * (size_t)g + 2));
        q_in = ldg_f4(rotations + 4 * (size_t)g);
        o_in = __ldg(opacities + g);
        if (RAW) {
            dc0 = __ldg(shs + 3 * (size_t)g); dc1 = __ldg(shs + 3 * (size_t)g + 1); dc2 = __ldg(shs + 3 * (size_t)g + 2);
            if (DEG > 0) load_sh_row<DEG, 1>(shs_rest + (size_t)g * (M - 1) * 3, ((M - 1) & 3) == 0, shc);
        } else load_sh_row<DEG>(shs + (size_t)g * M * 3, (M & 3) == 0, shc);
    }
}

// Shared memory of the forward: [nv x tiles histogram counters | 8 warps x staging slice]; 2 CTAs per SM (the host sizes the
// view groups so that the dynamic part fits 110 KB).
template <int DEG, bool RAW>
__global__ void __launch_bounds__(kPreThreads, 2)
preprocess_fwd_multiview_kernel(int P, int M, int H, int W, float scale_modifier, const __grid_constant__ MvViews views, int v0, int nv,
                                const float *__restrict__ means3D, const float *__restrict__ shs, const float *__restrict__ shs_rest,
                                const float *__restrict__ opacities, const float *__restrict__ scales, const float *__restrict__ rotations,
                                int *__restrict__ radii, const MvScratch sc, int tiles, int gpb_iters, int stage_off) {
    extern __shared__ __align__(128) unsigned s_hist[];
    __shared__ MvFrame s_fr[kMaxBatchViews];
    __shared__ uint64_t s_stage_bar[kPreThreads / 32];
    const int lane = threadIdx.x & 31;
    float *wstage = reinterpret_cast<float *>(reinterpret_cast<unsigned char *>(s_hist) + stage_off) + (threadIdx.x >> 5) * stage_warp_floats(M);
    uint64_t *wbar = &s_stage_bar[threadIdx.x >> 5];
    unsigned stage_phase = 0;
    bool stage_inflight;                 // warp-uniform: the copies of the NEXT block iteration have been started
    if (lane == 0) { mbar_init(wbar, 1); mbar_fence_init(); }
    __syncwarp();
    {
        const int g0 = (int)(blockIdx.x * gpb_iters * kPreThreads + (threadIdx.x & ~31u));
        stage_inflight = g0 + 32 <= P;
        if (stage_inflight && lane == 0) stage_issue<RAW>(wstage, wbar, g0, M, means3D, scales, rotations, opacities, shs, shs_rest);
    }
    load_frames(s_fr, views, v0, nv);
    for (int t = threadIdx.x; t < nv * tiles; t += kPreThreads) s_hist[t] = 0u;
    __syncthreads();
    const int gx = (W + kTile - 1) / kTile, gy = (H + kTile - 1) / kTile;
    for (int it = 0; it < gpb_iters; it++) {
        const int g = (int)((blockIdx.x * gpb_iters + it) * kPreThreads + threadIdx.x);
        float3 p = make_float3(0.f, 0.f, 0.f), s_in = p;
        float4 q_in = make_float4(1.f, 0.f, 0.f, 0.f);
        float o_in = 0.f, dc0 = 0.f, dc1 = 0.f, dc2 = 0.f, shc[48];
        const bool staged = stage_inflight;
        if (staged) {
            mbar_wait(wbar, stage_phase); stage_phase ^= 1u;
            mv_load_inputs<DEG, RAW>(true, wstage, g, M, means3D, shs, shs_rest, opacities, scales, rotations, p, s_in, q_in, o_in, dc0, dc1, dc2, shc);
        }
        __syncwarp();                    // every lane has its values in registers: the staging slice is free for the next iteration
        stage_inflight = false;
        if (it + 1 < gpb_iters) {
            const int g0 = (int)((blockIdx.x * gpb_iters + it + 1) * kPreThreads + (threadIdx.x & ~31u));
            stage_inflight = g0 + 32 <= P;
            if (stage_inflight && lane == 0) stage_issue<RAW>(wstage, wbar, g0, M, means3D, scales, rotations, opacities, shs, shs_rest);
        }
        if (g >= P) continue;
        if (!staged)
            mv_load_inputs<DEG, RAW>(false, wstage, g, M, means3D, shs, shs_rest, opacities, scales, rotations, p, s_in, q_in, o_in, dc0, dc1, dc2, shc);
        // view-independent: activations, 3D covariance, opacity
        float S6[6];
        {
            float3 s = s_in;
            if (RAW) s = make_float3(expf(s.x), expf(s.y), expf(s.z));
            s = make_float3(scale_modifier * s.x, scale_modifier * s.y, scale_modifier * s.z);
            float4 q = q_in;
            if (RAW) { float inv; q = act_normalize(q, inv); }
            float R[9]; quat_to_R(q, R);
            cov3d_from_scale_rot(s, R, S6);
        }
        const float o = RAW ? act_sigmoid(o_in) : o_in;
        for (int v = 0; v < nv; v++) {
            const FrameConsts &fc = s_fr[v].fc;
            const float tanfovx = s_fr[v].tanfovx, tanfovy = s_fr[v].tanfovy;
            char *geom = sc.geom + (size_t)(v0 + v) * sc.geom_stride;
            unsigned touched = 0, clamp_flags = 0;
            int radius_out = 0;
            Rec r;
            r.q0 = make_float4(0.f, 0.f, 0.f, 0.f); r.q1 = r.q0; r.q2 = r.q0;
            const float tzc = p.x * fc.V[2] + p.y * fc.V[6] + p.z * fc.V[10] + fc.V[14];
            if (tzc > DGR_NEAR_CULL_Z) {
                const float fx = (float)W / (2.f * tanfovx), fy = (float)H / (2.f * tanfovy);
                Geo geo;
                project_geo(fc, p, S6, fx, fy, DGR_FOV_CLAMP * tanfovx, DGR_FOV_CLAMP * tanfovy, geo);
                const float det = geo.cxx * geo.cyy - geo.cxy * geo.cxy;
                const float mid = 0.5f * (geo.cxx + geo.cyy);
                const float lam = mid + sqrtf(fmaxf(DGR_EIG_FLOOR, mid * mid - det));
                const float rad_f = ceilf(DGR_RADIUS_SIGMAS * sqrtf(lam));
                const float mx = ((geo.ndcx + 1.f) * (float)W - 1.f) * 0.5f;
                const float my = ((geo.ndcy + 1.f) * (float)H - 1.f) * 0.5f;
                const bool finite_ok = (det > 0.f) && (fabsf(mx) < 1e9f) && (fabsf(my) < 1e9f) && (rad_f < 1e9f);
                if (finite_ok) {
                    const int rminx = min(gx, max(0, (int)((mx - rad_f) / kTile)));
                    const int rminy = min(gy, max(0, (int)((my - rad_f) / kTile)));
                    const int rmaxx = min(gx, max(0, (int)((mx + rad_f + (kTile - 1)) / kTile)));
                    const int rmaxy = min(gy, max(0, (int)((my + rad_f + (kTile - 1)) / kTile)));
                    if (rmaxx > rminx && rmaxy > rminy) {
                        radius_out = (int)rad_f;
                        float cr, cg, cb;
                        {
                            float dx = p.x - fc.cam[0], dy = p.y - fc.cam[1], dz = p.z - fc.cam[2];
                            const float il = 1.f / sqrtf(dx * dx + dy * dy + dz * dz);
                            dx *= il; dy *= il; dz *= il;
                            float b[16]; sh_basis<DEG>(dx, dy, dz, b);
                            constexpr int NB = (DEG + 1) * (DEG + 1);
                            if (RAW) {
                                cr = b[0] * dc0; cg = b[0] * dc1; cb = b[0] * dc2;
#pragma unroll
                                for (int k = 1; k < NB; k++) { cr += b[k] * shc[3 * (k - 1)]; cg += b[k] * shc[3 * (k - 1) + 1]; cb += b[k] * shc[3 * (k - 1) + 2]; }
                            } else {
                                cr = 0.f; cg = 0.f; cb = 0.f;
#pragma unroll
                                for (int k = 0; k < NB; k++) { cr += b[k] * shc[3 * k]; cg += b[k] * shc[3 * k + 1]; cb += b[k] * shc[3 * k + 2]; }
                            }
                            cr += DGR_SH_OFFSET; cg += DGR_SH_OFFSET; cb += DGR_SH_OFFSET;
                            clamp_flags = (cr < 0.f ? 1u : 0u) | (cg < 0.f ? 2u : 0u) | (cb < 0.f ? 4u : 0u);
                            cr = fmaxf(cr, 0.f); cg = fmaxf(cg, 0.f); cb = fmaxf(cb, 0.f);
                        }
                        const float di = 1.f / det;
                        const float cA = geo.cyy * di, cB = -geo.cxy * di, cC = geo.cxx * di;
                        int bx0 = 1, bx1 = 0, by0 = 1, by1 = 0;
                        const float o255 = o * 255.f;
                        if (o255 > 1.f) {
                            const float tau = 2.f * logf(o255);
                            const float ex = sqrtf(tau * geo.cxx) * 1.0005f + 0.02f;
                            const float ey = sqrtf(tau * geo.cyy) * 1.0005f + 0.02f;
                            const float lim = 1e9f;
                            bx0 = max(rminx * kTile, (int)ceilf(fmaxf(mx - ex, -lim)));
                            by0 = max(rminy * kTile, (int)ceilf(fmaxf(my - ey, -lim)));
                            bx1 = min(min(rmaxx * kTile, W) - 1, (int)floorf(fminf(mx + ex, lim)));
                            by1 = min(min(rmaxy * kTile, H) - 1, (int)floorf(fminf(my + ey, lim)));
                        }
                        if (!(bx0 <= bx1 && by0 <= by1)) { bx0 = 1; bx1 = 0; by0 = 1; by1 = 0; }
                        r.q0 = make_float4(mx, my, cA * (-0.5f * kLog2e), cB * (-kLog2e));
                        r.q1 = make_float4(cC * (-0.5f * kLog2e), o, geo.t[2], __uint_as_float((unsigned)bx0 | ((unsigned)bx1 << 16)));
                        r.q2 = make_float4(cr, cg, cb, __uint_as_float((unsigned)by0 | ((unsigned)by1 << 16)));
                        unsigned *hist = s_hist + v * tiles;
                        for_each_touched_tile(__float_as_uint(r.q1.w), __float_as_uint(r.q2.w), gx,
                                              [&](int t) { atomicAdd(&hist[t], 1u); touched++; });
                    }
                }
            }
            radii[(size_t)(v0 + v) * P + g] = radius_out;
            reinterpret_cast<Rec *>(geom + sc.off_rec)[g] = r;
            reinterpret_cast<unsigned *>(geom + sc.off_touched)[g] = touched | (clamp_flags << 29);
        }
    }
    __syncthreads();
    // every view's histogram: one global atomic per (block, view, tile), 12 in flight per thread; the returned start goes into the
    // block's row of that view's run matrix
    constexpr int kB = 12;
    const int n = nv * tiles;
    for (int i0 = threadIdx.x; i0 < n; i0 += kPreThreads * kB) {
        unsigned c[kB], got[kB];
#pragma unroll
        for (int j = 0; j < kB; j++) { const int i = i0 + j * kPreThreads; c[j] = i < n ? s_hist[i] : 0u; }
#pragma unroll
        for (int j = 0; j < kB; j++) {
            const int i = i0 + j * kPreThreads, v = i / tiles, t = i - v * tiles;
            unsigned *tile_count = reinterpret_cast<unsigned *>(sc.image + (size_t)(v0 + v) * sc.image_stride + sc.off_count);
            got[j] = c[j] ? atomicAdd(tile_count + t, c[j]) : 0u;
        }
#pragma unroll
        for (int j = 0; j < kB; j++) {
            const int i = i0 + j * kPreThreads, v = i / tiles, t = i - v * tiles;
            if (i < n) reinterpret_cast<unsigned *>(sc.geom + (size_t)(v0 + v) * sc.geom_stride + sc.off_runs)[(size_t)blockIdx.x * tiles + t] = got[j];
        }
    }
}

// ---- backward --------------------------------------------------------------------------------------------------------------------
// Output image of a warp (floats), summed over the views: [0,96) means3D | [96,192) means2D of the current view (flushed per view) |
// [192,224) opacities | [224,320) scales | [320,448) rotations | [448,544) _features_dc (raw) | [544,800) each lane's activated scale
// and rotation (8 floats: kept here rather than in registers, which the SH row and the chain rule fill) | [800, 800 + 32 R) SH rows,
// R = the row length 3 M' (M' = M, or M - 1 for _features_rest) rounded up to an odd number of words (conflict-free per-lane adds).
constexpr int kMvO3D = 0, kMvO2D = 96, kMvOOp = 192, kMvOScale = 224, kMvORot = 320, kMvODc = 448, kMvOAct = 544, kMvOSh = 800;
__host__ __device__ inline int mv_sh_row_stride(int M, bool raw) { return (3 * (raw ? M - 1 : M)) | 1; }
__host__ __device__ inline int mv_bwd_warp_floats(int M, bool raw) {
    const int out = kMvOSh + 32 * mv_sh_row_stride(M, raw);
    const int stg = stage_warp_floats(M);
    return out > stg ? out : stg;
}

struct MvGrads {
    float *dL_dmeans3D, *dL_dmeans2D /* [V,P,3] */, *dL_dshs, *dL_dopacities, *dL_dscales, *dL_drotations, *dL_dshs_rest;
    float *xyz_gradient_accum, *denom, *max_radii2D;
};

// rows of K floats kept at a padded stride in shared memory -> one contiguous run of nrows x K floats in global memory
__device__ __forceinline__ void warp_flush_strided(float *seg, int K, int stride, int row_base, int nrows, bool acc, const float *ws) {
    if (!seg || K <= 0) return;
    const int lane = threadIdx.x & 31;
    float *dst = seg + (size_t)row_base * K;
    const int n = nrows * K;
    for (int i = lane; i < n; i += 32) {
        const int row = i / K, col = i - row * K;
        float x = ws[row * stride + col];
        if (acc) x += dst[i];
        dst[i] = x;
    }
}

template <int DEG, bool RAW>
__global__ void __launch_bounds__(kPreThreads, 2)
preprocess_bwd_multiview_kernel(int P, int M, int H, int W, float scale_modifier, const __grid_constant__ MvViews views, int nv,
                                const float *__restrict__ means3D, const float *__restrict__ shs, const float *__restrict__ shs_rest,
                                const float *__restrict__ opacities, const float *__restrict__ scales, const float *__restrict__ rotations,
                                const int *__restrict__ radii, const MvScratch sc, const MvGrads out, int accumulate, int warp_floats) {
    __shared__ MvFrame s_fr[kMaxBatchViews];
    __shared__ uint64_t s_stage_bar[kPreThreads / 32];
    extern __shared__ __align__(128) float s_dyn[];
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int row_base = (int)(blockIdx.x * blockDim.x) + (int)(threadIdx.x & ~31u);
    const int nrows = min(32, P - row_base);
    float *ws = s_dyn + (threadIdx.x >> 5) * warp_floats;
    uint64_t *wbar = &s_stage_bar[threadIdx.x >> 5];
    const bool staged = row_base + 32 <= P;                     // warp-uniform
    if (lane == 0) {
        mbar_init(wbar, 1); mbar_fence_init();
        if (staged) stage_issue<RAW>(ws, wbar, row_base, M, means3D, scales, rotations, opacities, shs, shs_rest);
    }
    __syncwarp();
    load_frames(s_fr, views, 0, nv);
    __syncthreads();
    const bool acc = accumulate != 0;
    const bool in_range = g < P;
    float3 p = make_float3(0.f, 0.f, 0.f), s_in = p;
    float4 q_in = make_float4(1.f, 0.f, 0.f, 0.f);
    float o_in = 0.f, dc0, dc1, dc2, shc[48];
    if (staged) {
        mbar_wait(wbar, 0u);
        mv_load_inputs<DEG, RAW>(true, ws, g, M, means3D, shs, shs_rest, opacities, scales, rotations, p, s_in, q_in, o_in, dc0, dc1, dc2, shc);
    }
    __syncwarp();                        // every lane has its inputs in registers: from here on the slice is the warp's output image
    if (in_range && !staged)
        mv_load_inputs<DEG, RAW>(false, ws, g, M, means3D, shs, shs_rest, opacities, scales, rotations, p, s_in, q_in, o_in, dc0, dc1, dc2, shc);
    (void)dc0; (void)dc1; (void)dc2;
    const int shw = 3 * (RAW ? M - 1 : M), shstride = mv_sh_row_stride(M, RAW);
    float *shrow = ws + kMvOSh + lane * shstride;
#pragma unroll
    for (int k = 0; k < 3; k++) { ws[kMvO3D + 3 * lane + k] = 0.f; ws[kMvOScale + 3 * lane + k] = 0.f; ws[kMvODc + 3 * lane + k] = 0.f; }
    ws[kMvOOp + lane] = 0.f;
    *reinterpret_cast<float4 *>(ws + kMvORot + 4 * lane) = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < shw; j++) shrow[j] = 0.f;
    // view-independent: activations
    {
        float3 s = s_in;
        if (RAW) s = make_float3(expf(s.x), expf(s.y), expf(s.z));
        s = make_float3(scale_modifier * s.x, scale_modifier * s.y, scale_modifier * s.z);
        float4 q = q_in;
        float inv_qnorm = 1.f;
        if (RAW) q = act_normalize(q, inv_qnorm);
        reinterpret_cast<float4 *>(ws + kMvOAct + 8 * lane)[0] = make_float4(s.x, s.y, s.z, inv_qnorm);
        reinterpret_cast<float4 *>(ws + kMvOAct + 8 * lane)[1] = q;
    }
    const float o = RAW ? act_sigmoid(o_in) : o_in;
    // Everything above reads only the op's inputs: under a programmatic dependent launch it overlaps the tail of the last backward
    // render kernel.  The moments are complete after this point.
    pdl_wait();
    for (int v = 0; v < nv; v++) {
        const FrameConsts &fc = s_fr[v].fc;
        const float tanfovx = s_fr[v].tanfovx, tanfovy = s_fr[v].tanfovy;
        const char *geom = sc.geom + (size_t)v * sc.geom_stride;
        const int radius_in = in_range ? __ldg(radii + (size_t)v * P + g) : 0;
        float gndx = 0.f, gndy = 0.f;
        if (radius_in > 0) {
            const unsigned touched_in = __ldg(reinterpret_cast<const unsigned *>(geom + sc.off_touched) + g);
            const float *grad_rec = reinterpret_cast<const float *>(geom + sc.off_gradrec);
            const float4 sa = reinterpret_cast<const float4 *>(ws + kMvOAct + 8 * lane)[0];
            const float4 q = reinterpret_cast<const float4 *>(ws + kMvOAct + 8 * lane)[1];
            const float3 s = make_float3(sa.x, sa.y, sa.z);
            const float inv_qnorm = sa.w;
            float R[9], S6[6];
            quat_to_R(q, R);
            cov3d_from_scale_rot(s, R, S6);
            const float fx = (float)W / (2.f * tanfovx), fy = (float)H / (2.f * tanfovy);
            Geo geo;
            project_geo(fc, p, S6, fx, fy, DGR_FOV_CLAMP * tanfovx, DGR_FOV_CLAMP * tanfovy, geo);
            const float a = geo.cxx, b = geo.cxy, c = geo.cyy;
            const float det = a * c - b * b, di = 1.f / det;
            const float cA = c * di, cB = -b * di, cC = a * di;
            const float4 m0 = ldg_f4(grad_rec + (size_t)g * kGradRecFloats);
            const float4 m1 = ldg_f4(grad_rec + (size_t)g * kGradRecFloats + 4);
            const float4 m2 = ldg_f4(grad_rec + (size_t)g * kGradRecFloats + 8);
            const float gpx = -(cA * m0.y + cB * m0.z), gpy = -(cC * m0.z + cB * m0.y);
            const float gA = -0.5f * m0.w, gB = -m1.x, gC = -0.5f * m1.y;
            const float g_op = (o != 0.f) ? m0.x / o : 0.f;
            const float g_rgb[3] = { m1.z, m1.w, m2.x };
            const float g_depth = m2.y;
            float dmean[3] = { 0.f, 0.f, 0.f };
            gndx = gpx * 0.5f * (float)W; gndy = gpy * 0.5f * (float)H;
            if (out.xyz_gradient_accum) out.xyz_gradient_accum[g] += sqrtf(gndx * gndx + gndy * gndy);
            if (out.denom) out.denom[g] += 1.f;
            if (out.max_radii2D) out.max_radii2D[g] = fmaxf(out.max_radii2D[g], (float)radius_in);
            {
                const float *PM = fc.PM;
                const float mul1 = geo.ndcx * geo.pw, mul2 = geo.ndcy * geo.pw;
#pragma unroll
                for (int k = 0; k < 3; k++)
                    dmean[k] += (PM[4 * k] * geo.pw - PM[4 * k + 3] * mul1) * gndx + (PM[4 * k + 1] * geo.pw - PM[4 * k + 3] * mul2) * gndy;
            }
#pragma unroll
            for (int k = 0; k < 3; k++) dmean[k] += fc.V[4 * k + 2] * g_depth;
            {
                float dx = p.x - fc.cam[0], dy = p.y - fc.cam[1], dz = p.z - fc.cam[2];
                const float il = 1.f / sqrtf(dx * dx + dy * dy + dz * dz);
                dx *= il; dy *= il; dz *= il;
                float bs[16];
                sh_basis<DEG>(dx, dy, dz, bs);
                const unsigned flags = touched_in >> 29;
                float gr[3];
#pragma unroll
                for (int ch = 0; ch < 3; ch++) gr[ch] = ((flags >> ch) & 1u) ? 0.f : g_rgb[ch];
                float ddx = 0.f, ddy = 0.f, ddz = 0.f;
                constexpr int NB = (DEG + 1) * (DEG + 1);
#pragma unroll
                for (int k = 1; k < NB; k++) {
                    const int off = RAW ? 3 * (k - 1) : 3 * k;
                    const float dotc = shc[off] * gr[0] + shc[off + 1] * gr[1] + shc[off + 2] * gr[2];
                    float bx, by, bz;
                    sh_dbasis(k, dx, dy, dz, bx, by, bz);
                    ddx += bx * dotc; ddy += by * dotc; ddz += bz * dotc;
                }
                const float dot = dx * ddx + dy * ddy + dz * ddz;
                dmean[0] += (ddx - dx * dot) * il; dmean[1] += (ddy - dy * dot) * il; dmean[2] += (ddz - dz * dot) * il;
                // SH gradient of this view, added into the warp's rows
                if (RAW) {
#pragma unroll
                    for (int ch = 0; ch < 3; ch++) ws[kMvODc + 3 * lane + ch] += bs[0] * gr[ch];
#pragma unroll
                    for (int k = 1; k < NB; k++)
#pragma unroll
                        for (int ch = 0; ch < 3; ch++) shrow[3 * (k - 1) + ch] += bs[k] * gr[ch];
                } else {
#pragma unroll
                    for (int k = 0; k < NB; k++)
#pragma unroll
                        for (int ch = 0; ch < 3; ch++) shrow[3 * k + ch] += bs[k] * gr[ch];
                }
            }
            ws[kMvOOp + lane] += RAW ? g_op * o * (1.f - o) : g_op;
            const float d2 = di * di;
            const float ga = d2 * (-c * c * gA + b * c * gB - b * b * gC);
            const float gc = d2 * (-b * b * gA + a * b * gB - a * a * gC);
            const float gb = d2 * (2.f * b * c * gA - (det + 2.f * b * b) * gB + 2.f * a * b * gC);
            const float G00 = ga, G01 = 0.5f * gb, G11 = gc;
            const float *T0 = geo.T0, *T1 = geo.T1;
            float dS[9];
#pragma unroll
            for (int k = 0; k < 3; k++)
#pragma unroll
                for (int l = 0; l < 3; l++)
                    dS[3 * k + l] = T0[k] * (G00 * T0[l] + G01 * T1[l]) + T1[k] * (G01 * T0[l] + G11 * T1[l]);
            const float Sg[9] = { S6[0], S6[1], S6[2], S6[1], S6[3], S6[4], S6[2], S6[4], S6[5] };
            float TS0[3], TS1[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                TS0[k] = T0[0] * Sg[k] + T0[1] * Sg[3 + k] + T0[2] * Sg[6 + k];
                TS1[k] = T1[0] * Sg[k] + T1[1] * Sg[3 + k] + T1[2] * Sg[6 + k];
            }
            float dT0[3], dT1[3];
#pragma unroll
            for (int k = 0; k < 3; k++) { dT0[k] = 2.f * (G00 * TS0[k] + G01 * TS1[k]); dT1[k] = 2.f * (G01 * TS0[k] + G11 * TS1[k]); }
            float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                dJ00 += dT0[k] * fc.V[4 * k]; dJ02 += dT0[k] * fc.V[4 * k + 2];
                dJ11 += dT1[k] * fc.V[4 * k + 1]; dJ12 += dT1[k] * fc.V[4 * k + 2];
            }
            const float tz = geo.t[2];
            const float tz2 = 1.f / (tz * tz), tz3 = tz2 / tz;
            const float dtx = geo.clx ? 0.f : -fx * tz2 * dJ02;
            const float dty = geo.cly ? 0.f : -fy * tz2 * dJ12;
            const float dtz = -fx * tz2 * dJ00 - fy * tz2 * dJ11 + 2.f * fx * geo.tx * tz3 * dJ02 + 2.f * fy * geo.ty * tz3 * dJ12;
#pragma unroll
            for (int k = 0; k < 3; k++) dmean[k] += fc.V[4 * k] * dtx + fc.V[4 * k + 1] * dty + fc.V[4 * k + 2] * dtz;
#pragma unroll
            for (int k = 0; k < 3; k++) ws[kMvO3D + 3 * lane + k] += dmean[k];
            float Mx[9];
#pragma unroll
            for (int i = 0; i < 3; i++) { Mx[3 * i] = R[3 * i] * s.x; Mx[3 * i + 1] = R[3 * i + 1] * s.y; Mx[3 * i + 2] = R[3 * i + 2] * s.z; }
            float dM[9];
#pragma unroll
            for (int i = 0; i < 3; i++)
#pragma unroll
                for (int k = 0; k < 3; k++)
                    dM[3 * i + k] = 2.f * (dS[3 * i] * Mx[k] + dS[3 * i + 1] * Mx[3 + k] + dS[3 * i + 2] * Mx[6 + k]);
            const float sv[3] = { s.x, s.y, s.z };
            float dR[9];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                float vv = 0.f;
#pragma unroll
                for (int i = 0; i < 3; i++) { vv += dM[3 * i + k] * R[3 * i + k]; dR[3 * i + k] = dM[3 * i + k] * sv[k]; }
                ws[kMvOScale + 3 * lane + k] += RAW ? vv * sv[k] : vv * scale_modifier;
            }
            {
                const float r = q.x, x = q.y, y = q.z, z = q.w;
                float dq[4];
                dq[0] = 2.f * (-z * dR[1] + y * dR[2] + z * dR[3] - x * dR[5] - y * dR[6] + x * dR[7]);
                dq[1] = 2.f * (y * dR[1] + z * dR[2] + y * dR[3] - 2.f * x * dR[4] - r * dR[5] + z * dR[6] + r * dR[7] - 2.f * x * dR[8]);
                dq[2] = 2.f * (-2.f * y * dR[0] + x * dR[1] + r * dR[2] + x * dR[3] + z * dR[5] - r * dR[6] + z * dR[7] - 2.f * y * dR[8]);
                dq[3] = 2.f * (-2.f * z * dR[0] - r * dR[1] + x * dR[2] + r * dR[3] - 2.f * z * dR[4] + y * dR[5] + x * dR[6] + y * dR[7]);
                if (RAW) {
                    const float qd = r * dq[0] + x * dq[1] + y * dq[2] + z * dq[3];
                    dq[0] = (dq[0] - r * qd) * inv_qnorm; dq[1] = (dq[1] - x * qd) * inv_qnorm;
                    dq[2] = (dq[2] - y * qd) * inv_qnorm; dq[3] = (dq[3] - z * qd) * inv_qnorm;
                }
                float4 *rot = reinterpret_cast<float4 *>(ws + kMvORot + 4 * lane);
                float4 acc4 = *rot;
                acc4.x += dq[0]; acc4.y += dq[1]; acc4.z += dq[2]; acc4.w += dq[3];
                *rot = acc4;
            }
        }
        // this view's means2D gradient (NDC units, z = 0; zero rows for Gaussians it culled) leaves now
        ws[kMvO2D + 3 * lane] = gndx; ws[kMvO2D + 3 * lane + 1] = gndy; ws[kMvO2D + 3 * lane + 2] = 0.f;
        __syncwarp();
        if (nrows > 0 && out.dL_dmeans2D) warp_flush(out.dL_dmeans2D + (size_t)v * P * 3, 3, 0, row_base, nrows, acc, ws + kMvO2D);
        __syncwarp();
    }
    // ---- the sums over the views leave together (rows past the end of the arrays are not written)
    if (nrows > 0) {
        warp_flush(out.dL_dmeans3D, 3, 0, row_base, nrows, acc, ws + kMvO3D);
        warp_flush(out.dL_dopacities, 1, 0, row_base, nrows, acc, ws + kMvOOp);
        warp_flush(out.dL_dscales, 3, 0, row_base, nrows, acc, ws + kMvOScale);
        warp_flush(out.dL_drotations, 4, 0, row_base, nrows, acc, ws + kMvORot);
        if (RAW) {
            warp_flush(out.dL_dshs, 3, 0, row_base, nrows, acc, ws + kMvODc);
            warp_flush_strided(out.dL_dshs_rest, shw, shstride, row_base, nrows, acc, ws + kMvOSh);
        } else warp_flush_strided(out.dL_dshs, shw, shstride, row_base, nrows, acc, ws + kMvOSh);
    }
}

}  // namespace dgr
