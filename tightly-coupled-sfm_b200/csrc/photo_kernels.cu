// The `return_errors` photometric block of solve_pose_iteratively (reference
// train_mono.py:84-92; the same arithmetic is compute_photometric_error,
// optimization_experiments/helpers.py:12-18), fused: for a stack of pairs
//
//   auto_mask_error = mean_c(0.15 * clamp|tgt - src| + 0.85 * SSIM(tgt, src))
//   diff_img        = mean_c(0.15 * clamp|rec - tgt| + 0.85 * SSIM(tgt, rec))
//   auto_mask       = diff_img < auto_mask_error
//   weight_mask     = 1 - clamp(|cd - pd| / (cd + pd), 0, 1)
//
// and the backward w.r.t. the reconstructed image `rec` and the two depths.  Same tiling
// and register-window SSIM as the pair kernels (csrc/pair_kernels.cu), minus the geometry:
// the reconstructed image is an input here because the pose network consumes it too.
#include "tile.cuh"

namespace tcsfm {

constexpr int kPhotoCoefPlanes = 9;

struct PhotoArgs {
    const float* tgt; int64_t tgt_sb, tgt_sc;
    const float* src; int64_t src_sb, src_sc;
    const float* rec;                 // [N,3,H,W] contiguous
    const float* pd; const float* cd; // [N,1,H,W]
    const float* valid;               // [N,1,H,W] or NULL: folded into auto_mask (helpers.py:18)
    float* auto_err; float* diff; float* auto_mask; float* weight;
    float* coef;                      // [N,9,H,W] workspace (fwd writes, bwd reads) or NULL
    const float* g_diff; const float* g_weight;
    float* g_rec; float* g_pd; float* g_cd;
    Arith A;
    float w_l1, w_ssim, C1, C2;
};

// d E / d w of one channel's reconstructed value w at a cell with target t, from the 3x3 sums V0, V1, V2 of the
// SSIM adjoint coefficients (Ay, B, Cc) of the windows that read the cell: V0 + 2 w V1 + t V2, plus the sign term of
// the L1 adjoint `gl1` where |t - w| <= 1 (0 at cells that are no own pixel).
__device__ __forceinline__ float rec_adjoint(float V0, float V1, float V2, float t, float w, float gl1) {
    const float dlt = t - w;
    float g = V0 + 2.0f * w * V1 + t * V2;
    if (fabsf(dlt) <= 1.0f) g += (dlt > 0.f) ? -gl1 : ((dlt < 0.f) ? gl1 : 0.f);
    return g;
}

template <int F>
__global__ void __launch_bounds__(kTileThreads, 3)
photo_fwd_kernel(const __grid_constant__ PhotoArgs P) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float2, tr);                                  // [3][cells] (target, rec)
    float2* tsrc = tr + 3 * T1::kCells;                          // [3][cells] (target, src)
    const Arith& A = P.A;
    const int H = A.H, W = A.W, n = H * W;
    const int b = blockIdx.y;
    int x0, y0;
    tile_origin(blockIdx.x, W, x0, y0);
    const float* tgt = P.tgt + b * P.tgt_sb;
    const float* src = P.src + b * P.src_sb;
    const float* rec = P.rec + (int64_t)b * 3 * n;
    // two cells per sweep: their eighteen loads are in flight before the first shared-memory store
    for (int cell0 = threadIdx.x; cell0 < T1::kCells; cell0 += 2 * kTileThreads) {
        int pix[2];
        bool ok[2];
        float t[2][3], r[2][3], sv[2][3];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int cell = cell0 + u * kTileThreads;
            int ry = 0, rx = 0;
            ok[u] = cell < T1::kCells && T1::cell_to_reflected(cell, x0, y0, H, W, ry, rx);
            pix[u] = ok[u] ? ry * W + rx : 0;
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                t[u][ch] = ok[u] ? __ldg(tgt + ch * P.tgt_sc + pix[u]) : 0.f;
                r[u][ch] = ok[u] ? __ldg(rec + (int64_t)ch * n + pix[u]) : 0.f;
                sv[u][ch] = ok[u] ? __ldg(src + ch * P.src_sc + pix[u]) : 0.f;
            }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int cell = cell0 + u * kTileThreads;
            if (cell < T1::kCells) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    tr[ch * T1::kCells + cell] = make_float2(t[u][ch], r[u][ch]);
                    tsrc[ch * T1::kCells + cell] = make_float2(t[u][ch], sv[u][ch]);
                }
            }
        }
    }
    __syncthreads();
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx, gy0 = y0 + ty0;
    float e_rec[kPixPerThread], e_src[kPixPerThread];
    float* coef_b = P.coef ? P.coef + (int64_t)b * kPhotoCoefPlanes * n : nullptr;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        // coef_ch captured by value and the bounds read from P: in this form the kernel keeps the SASS of its former
        // own strip loop (other forms were scheduled differently, one of them measured 1 % slower)
        ssim_l1_strip(tr + ch * T1::kCells, tx, ty0, P, ch == 0, e_rec,
                      [&, coef_ch = coef_b ? coef_b + (int64_t)3 * ch * n : nullptr](int k, const SsimStats& s, const SsimTerms& t) {
            const int gy = gy0 + k;
            if (coef_ch && gx < P.A.W && gy < P.A.H) {
                const SsimCoef kf = ssim_coef(s, t, P.A.third * P.w_ssim);     // x = target, y = reconstruction
                float* cp = coef_ch + gy * P.A.W + gx;
                cp[0] = kf.Ay; cp[n] = kf.B; cp[2 * (int64_t)n] = kf.Cc;
            }
        });
        ssim_l1_strip(tsrc + ch * T1::kCells, tx, ty0, P, ch == 0, e_src, NoSsimSink());
    }
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = gy0 + k;
        if (gx < W && gy < H) {
            const int64_t o = (int64_t)b * n + gy * W + gx;
            const float diff = mean3_of_sum<F>(e_rec[k], A);
            const float aerr = mean3_of_sum<F>(e_src[k], A);
            if (P.diff) P.diff[o] = diff;
            if (P.auto_err) P.auto_err[o] = aerr;
            if (P.auto_mask) P.auto_mask[o] = (diff < aerr) ? (P.valid ? __ldg(P.valid + o) : 1.f) : 0.f;
            if (P.weight) P.weight[o] = __fsub_rn(1.0f, depth_inconsistency(__ldg(P.cd + o), __ldg(P.pd + o)));
        }
    }
}

__global__ void __launch_bounds__(kTileThreads, 3)
photo_bwd_kernel(const __grid_constant__ PhotoArgs P) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float, cs);                     // [9][cells] upstream-scaled coefficients
    const Arith& A = P.A;
    const int H = A.H, W = A.W, n = H * W;
    const int b = blockIdx.y;
    int x0, y0;
    tile_origin(blockIdx.x, W, x0, y0);
    const float* gdiff = P.g_diff ? P.g_diff + (int64_t)b * n : nullptr;
    const float* coef = P.coef + (int64_t)b * kPhotoCoefPlanes * n;
    // two cells per sweep: the twenty loads of both are in flight before the first product is stored
    for (int cell0 = threadIdx.x; cell0 < T1::kCells; cell0 += 2 * kTileThreads) {
        int pix[2];
        bool inside[2];
        float Gd[2], v[2][9];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int cell = cell0 + u * kTileThreads;
            int cx, cy;
            T1::cell_xy(cell < T1::kCells ? cell : 0, cx, cy);
            const int qx = x0 + cx, qy = y0 + cy;
            inside[u] = cell < T1::kCells && gdiff && qx >= 0 && qx < W && qy >= 0 && qy < H;
            pix[u] = inside[u] ? qy * W + qx : 0;
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            Gd[u] = inside[u] ? __ldg(gdiff + pix[u]) : 0.f;
#pragma unroll
            for (int j = 0; j < 9; ++j) v[u][j] = inside[u] ? __ldg(coef + (int64_t)j * n + pix[u]) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int cell = cell0 + u * kTileThreads;
            if (cell < T1::kCells) {
#pragma unroll
                for (int j = 0; j < 9; ++j) cs[j * T1::kCells + cell] = Gd[u] * v[u][j];
            }
        }
    }
    __syncthreads();
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;
    const float* tgt = P.tgt + b * P.tgt_sb;
    const float* rec = P.rec + (int64_t)b * 3 * n;
    // the own pixels' target / reconstruction values and upstream: requested before the window sums
    float tq[kPixPerThread][3], wq[kPixPerThread][3], gq[kPixPerThread];
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        const bool own = gx < W && gy < H;
        const int pix = own ? gy * W + gx : 0;
        gq[k] = (own && gdiff) ? __ldg(gdiff + pix) : 0.f;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            tq[k][ch] = own ? __ldg(tgt + ch * P.tgt_sc + pix) : 0.f;
            wq[k][ch] = own ? __ldg(rec + (int64_t)ch * n + pix) : 0.f;
        }
    }
    float h[3][9];
    const bool dup_l = (gx == 1), dup_r = (gx == W - 2);
    auto hsum = [&](int r, float (&out)[9]) {
        const int c1 = T1::cell(tx, ty0 - 1 + r);
#pragma unroll
        for (int j = 0; j < 9; ++j) {
            const float* pl = cs + j * T1::kCells + c1;
            const float l = pl[-1], m = pl[0], rr = pl[1];
            float s = (l + m) + rr;
            if (dup_l) s += l;
            if (dup_r) s += rr;
            out[j] = s;
        }
    };
    hsum(0, h[0]);
    hsum(1, h[1]);
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        hsum(k + 2, h[(k + 2) % 3]);
        const int gy = y0 + ty0 + k;
        if (gx < W && gy < H) {
            const bool dup_u = (gy == 1), dup_d = (gy == H - 2);
            const int pix = gy * W + gx;
            const int64_t o = (int64_t)b * n + pix;
            const float Gd = gq[k];
            const float gl1 = Gd * A.third * P.w_l1;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                float V[3];
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int q = 3 * ch + j;
                    float s = (h[k % 3][q] + h[(k + 1) % 3][q]) + h[(k + 2) % 3][q];
                    if (dup_u) s += h[k % 3][q];
                    if (dup_d) s += h[(k + 2) % 3][q];
                    V[j] = s;
                }
                const float gw = rec_adjoint(V[0], V[1], V[2], tq[k][ch], wq[k][ch], gl1);
                if (P.g_rec) P.g_rec[((int64_t)b * 3 + ch) * n + pix] = gw;
            }
            if (P.g_pd || P.g_cd) {
                float g_Z = 0.f, g_p = 0.f;
                if (P.g_weight) depth_inconsistency_adjoint(__ldg(P.cd + o), __ldg(P.pd + o), -__ldg(P.g_weight + o), g_Z, g_p);
                if (P.g_cd) P.g_cd[o] = g_Z;
                if (P.g_pd) P.g_pd[o] = g_p;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// compute_photometric_error for `per` pose hypotheses of each of B frame pairs (the loss-surface sweeps of
// plot_loss_surface.py:11-87): per hypothesis the warp of inverse_warp2, the maps above and the masked sums
//   error_sum = sum((diff * auto_mask * valid) * weight)      valid_sum = sum(auto_mask * valid)
// Three launches: the pose-independent auto-mask error once per pair, one CTA per (hypothesis, tile), and a
// fixed-order reduction of the per-CTA partials (no float atomics: the sums are deterministic).  Hypotheses are
// pair-major: global hypothesis hyp is start hyp % per of pair hyp / per.
// ---------------------------------------------------------------------------
struct SweepArgs {
    PhotoArgs P;                          // tgt / src views of pair 0 and their batch strides, auto_err scratch [B,H,W],
                                          // weights, SSIM constants, arithmetic
    const float* tdep; const float* sdep; // [B,H,W]
    const float* kinv; const float* proj; // [B,9], [N,12]
    float* partials;                      // [tiles][N][2]: per-CTA (sum of products, sum of the mask)
    float* rec; float* diff; float* mask; float* weight;   // optional maps [N,3,H,W], [N,1,H,W] x 3
    int N, tiles, per;                    // N = B * per hypotheses in all, per of them for each pair
};

// The inputs of pair b: 64-bit bases, from which the per-pixel code keeps its 32-bit channel and pixel offsets.  The
// kernels form them where they read them: held in registers across the tile fill, they cost photo_sweep_kernel<F, false>
// a spill.
struct SweepPair {
    const float* tgt; const float* src; const float* tdep; const float* sdep;
};

__device__ __forceinline__ SweepPair sweep_pair(const SweepArgs& S, int b) {
    const int64_t n = (int64_t)S.P.A.H * S.P.A.W;
    return SweepPair{S.P.tgt + b * S.P.tgt_sb, S.P.src + b * S.P.src_sb, S.tdep + b * n, S.sdep + b * n};
}

// auto_err = mean_c(w_l1 * clamp|tgt - src| + w_ssim * SSIM(tgt, src)) of pair blockIdx.y: photo_fwd_kernel's e_src.
// kPairs = false: one pair, read without any pair arithmetic (this kernel and photo_sweep_kernel then keep the
// instructions they had before B pairs; the pair arithmetic measured 5-12 % slower on one pair).
template <int F, bool kPairs>
__global__ void __launch_bounds__(kTileThreads)
photo_auto_err_kernel(const __grid_constant__ PhotoArgs P) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float2, ts);                                  // [3][cells] (target, src)
    const int H = P.A.H, W = P.A.W;
    // tile_origin spelled out: with the call, ptxas schedules this kernel differently (measured 0.6 % slower)
    const int tiles_x = (W + kTileW - 1) / kTileW;
    const int tile_y = blockIdx.x / tiles_x, tile_x = blockIdx.x - tile_y * tiles_x;
    const int x0 = tile_x * kTileW, y0 = tile_y * kTileH;
    const int64_t b = kPairs ? blockIdx.y : 0;
    for (int cell = threadIdx.x; cell < T1::kCells; cell += kTileThreads) {
        int ry = 0, rx = 0;
        const bool ok = T1::cell_to_reflected(cell, x0, y0, H, W, ry, rx);
        const int pix = ok ? ry * W + rx : 0;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch)
            ts[ch * T1::kCells + cell] = ok ? make_float2(__ldg(P.tgt + b * P.tgt_sb + ch * P.tgt_sc + pix),
                                                          __ldg(P.src + b * P.src_sb + ch * P.src_sc + pix))
                                            : make_float2(0.f, 0.f);
    }
    __syncthreads();
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;
    float e[kPixPerThread];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) ssim_l1_strip(ts + ch * T1::kCells, tx, ty0, P, ch == 0, e, NoSsimSink());
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        if (gx < W && gy < H) (P.auto_err + b * H * W)[gy * W + gx] = mean3_of_sum<F>(e[k], P.A);
    }
}

// ---------------------------------------------------------------------------
// d loss_n / d proj_n of the loss surface, loss_n = E_n / V_n with E_n = sum((diff * mask) * weight), V_n = sum(mask):
// the mask is a comparison (no gradient) and V_n a constant, so the gradient is dE_n / d proj_n over V_n.  One CTA per
// (hypothesis, tile) recomputes the tile's forward (photo_sweep_kernel<F, true>), then runs the adjoint in cell space over the
// tile and its ring: a cell's warped value is read by the 3x3 SSIM windows of the own pixels around it, so its gradient
// is the gather of their coefficients (the form of photo_bwd_kernel).  Ring cells at the image border hold the
// reflected pixel itself, so the reflection needs no duplicate taps here.  Each cell then runs the bilinear and
// projective adjoints of its own warp; own pixels add the weight term through the sampled source depth and Z.
// ---------------------------------------------------------------------------
constexpr int kSweepGradParts = 14;       // per CTA: E, V, d E / d proj [12]

// g[ch] = d E / d (warped value of channel ch) of the image pixel (rx, ry); g_weight = d E / d weight at that pixel
// (own pixels only).  Adds d E / d proj through this pixel's warp into acc (row-major K[R|t]).
template <int F>
__device__ __forceinline__ void sweep_cell_adjoint(const SweepArgs& S, int b, const Cam& cam, int rx, int ry,
                                                   const float (&g)[3], float g_weight, float (&acc)[12]) {
    const Arith& A = S.P.A;
    const SweepPair pr = sweep_pair(S, b);
    const int pix = ry * A.W + rx;
    WarpPt p;
    warp_point<F>(cam, A, rx, ry, __ldg(pr.tdep + pix), p);
    const TapIdx ti = make_taps(p, A.H, A.W);
    Taps tc[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) tc[ch] = load_taps(pr.src, (int)(ch * S.P.src_sc), ti, A.W);
    float g_ix = 0.f, g_iy = 0.f, g_Z = 0.f;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) bilinear_grad(tc[ch], p, g[ch], g_ix, g_iy);
    if (g_weight != 0.f) {
        // weight = 1 - depth_inconsistency(Z, sampled source depth)
        const Taps td = load_taps(pr.sdep, 0, ti, A.W);
        float g_pd = 0.f;
        depth_inconsistency_adjoint(p.Z, blend(td, ti), -g_weight, g_Z, g_pd);
        bilinear_grad(td, p, g_pd, g_ix, g_iy);
    }
    const GeomGrad gg = geom_adjoint(cam, A, p, g_ix, g_iy, g_Z);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        acc[i * 4 + 0] += gg.gp[i] * p.cam[0];
        acc[i * 4 + 1] += gg.gp[i] * p.cam[1];
        acc[i * 4 + 2] += gg.gp[i] * p.cam[2];
        acc[i * 4 + 3] += gg.gp[i];
    }
}

// The adjoint of one tile for photo_sweep_kernel<F, true>, after its forward: scales the raw coefficients the strips left
// in `cs` by the upstream, then accumulates d E / d proj of the tile's cells into acc.  Contains __syncthreads().
template <int F>
__device__ __forceinline__ void sweep_tile_adjoint(const SweepArgs& S, int b, const Cam& cam, const float2* tw, float* cs,
                                                   int x0, int y0,
                                                   const float (&diff)[kPixPerThread], const float (&m)[kPixPerThread],
                                                   const float (&wgt)[kPixPerThread], float (&acc)[12]) {
    using T1 = Tile<1>;
    const Arith& A = S.P.A;
    const int H = A.H, W = A.W;
    // coefficients: d E / d diff = mask * weight at each own pixel, zero for the filler cells of partial tiles and the ring
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const float u = m[k] * wgt[k];
        const int c = T1::cell(tx, ty0 + k);
#pragma unroll
        for (int j = 0; j < kPhotoCoefPlanes; ++j) cs[j * T1::kCells + c] = (m[k] != 0.f) ? cs[j * T1::kCells + c] * u : 0.f;
    }
    if (threadIdx.x < kRingCells) {
        int cx, cy;
        ring_cell(threadIdx.x, cx, cy);
#pragma unroll
        for (int j = 0; j < kPhotoCoefPlanes; ++j) cs[j * T1::kCells + T1::cell(cx, cy)] = 0.f;
    }
    __syncthreads();

#pragma unroll
    for (int i = 0; i < 12; ++i) acc[i] = 0.f;
    const float l1_scale = A.third * S.P.w_l1;
    // own cells: the 3x3 coefficient sums slide down the strip, three row sums of the nine planes live at a time
    float h[3][kPhotoCoefPlanes];
    auto hsum = [&](int r, float (&out)[kPhotoCoefPlanes]) {
        const int c1 = T1::cell(tx, ty0 - 1 + r);
#pragma unroll
        for (int j = 0; j < kPhotoCoefPlanes; ++j) {
            const float* pl = cs + j * T1::kCells + c1;
            out[j] = (pl[-1] + pl[0]) + pl[1];
        }
    };
    hsum(0, h[0]);
    hsum(1, h[1]);
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        hsum(k + 2, h[(k + 2) % 3]);
        const int gy = y0 + ty0 + k;
        if (gx > W || gy > H) continue;         // filler cells that no pixel's window reaches
        const bool own = gx < W && gy < H;
        const int c = T1::cell(tx, ty0 + k);
        const float gl1 = own ? m[k] * wgt[k] * l1_scale : 0.f;
        float g[3];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            float V[3];
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int q = 3 * ch + j;
                V[j] = (h[k % 3][q] + h[(k + 1) % 3][q]) + h[(k + 2) % 3][q];
            }
            const float2 tv = tw[ch * T1::kCells + c];
            g[ch] = rec_adjoint(V[0], V[1], V[2], tv.x, tv.y, gl1);
        }
        // a filler cell one past the last row / column holds the reflection of the one before the last
        sweep_cell_adjoint<F>(S, b, cam, gx < W ? gx : 2 * W - 2 - gx, gy < H ? gy : 2 * H - 2 - gy, g,
                              own ? diff[k] * m[k] : 0.f, acc);
    }
    // ring cells: the coefficients of the own pixels among their 3x3 neighbours
    if (threadIdx.x < kRingCells) {
        int cx, cy, ry = 0, rx = 0;
        ring_cell(threadIdx.x, cx, cy);
        const int c = T1::cell(cx, cy);
        if (T1::cell_to_reflected(c, x0, y0, H, W, ry, rx)) {
            float V[kPhotoCoefPlanes];
#pragma unroll
            for (int j = 0; j < kPhotoCoefPlanes; ++j) V[j] = 0.f;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const int nx = cx + dx, ny = cy + dy;
                    if (nx < 0 || nx >= kTileW || ny < 0 || ny >= kTileH) continue;
#pragma unroll
                    for (int j = 0; j < kPhotoCoefPlanes; ++j) V[j] += cs[j * T1::kCells + T1::cell(nx, ny)];
                }
            float g[3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float2 tv = tw[ch * T1::kCells + c];
                g[ch] = rec_adjoint(V[3 * ch], V[3 * ch + 1], V[3 * ch + 2], tv.x, tv.y, 0.f);
            }
            sweep_cell_adjoint<F>(S, b, cam, rx, ry, g, 0.f, acc);
        }
    }
}

// One CTA per (hypothesis, tile).  kGrad = false: the sums and optional maps of tcsfm_photo_sweep.  kGrad = true: the
// same forward, instruction for instruction (so E and V keep their bits), whose strips also leave their SSIM adjoint
// coefficients in shared memory; then the adjoint of the tile (sweep_tile_adjoint), and a partial (E, V, dE/dproj[12]).
// kPairs as in photo_auto_err_kernel.
template <int F, bool kGrad, bool kPairs>
__global__ void __launch_bounds__(kTileThreads, kGrad ? 2 : 3)
photo_sweep_kernel(const __grid_constant__ SweepArgs S) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float2, tw);                                  // [3][cells] (target, warped source)
    TCSFM_SHARED float red[(kGrad ? kSweepGradParts : 2) * (kTileThreads / 32)];
    const Arith& A = S.P.A;
    const int H = A.H, W = A.W, n = H * W;
    const int hyp = blockIdx.x / S.tiles, tile = blockIdx.x - hyp * S.tiles;
    const int b = kPairs ? hyp / S.per : 0;
    int x0, y0;
    tile_origin(tile, W, x0, y0);
    const Cam cam = load_cam(S.kinv + 9 * (int64_t)b, S.proj + (int64_t)hyp * 12, 0);
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;
    float* cs = kGrad ? reinterpret_cast<float*>(tw + 3 * T1::kCells) : nullptr;   // kGrad: [9][cells] coefficients
    auto fill = [&](int rx, int ry, int cell, WarpPt& p) {
        const SweepPair pr = sweep_pair(S, b);
        return fill_warped_cell<F>(cam, A, pr.tgt, (int)S.P.tgt_sc, pr.src, (int)S.P.src_sc, rx, ry, __ldg(pr.tdep + ry * W + rx), tw,
                                   cell, p);
    };
    // own pixels: the cell, plus valid and weight = 1 - depth_inconsistency(computed, projected depth) of the warp.
    // Own cells that no consumer reads (partial tiles) are filled from a clamped pixel, as in the pair forward.
    bool valid[kPixPerThread];
    float wgt[kPixPerThread];
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        const int sx = min(max(gx < W ? gx : 2 * W - 2 - gx, 0), W - 1);
        const int sy = min(max(gy < H ? gy : 2 * H - 2 - gy, 0), H - 1);
        WarpPt p;
        const TapIdx ti = fill(sx, sy, T1::cell(tx, ty0 + k), p);
        valid[k] = p.valid;
        wgt[k] = __fsub_rn(1.0f, depth_inconsistency(p.Z, blend(load_taps(sweep_pair(S, b).sdep, 0, ti, W), ti)));
    }
    if (threadIdx.x < kRingCells) {
        int cx, cy, ry = 0, rx = 0;
        ring_cell(threadIdx.x, cx, cy);
        const int cell = T1::cell(cx, cy);
        WarpPt p;
        if (T1::cell_to_reflected(cell, x0, y0, H, W, ry, rx)) fill(rx, ry, cell, p);
        else zero_cell(tw, cell);
    }
    __syncthreads();
    float esum[kPixPerThread];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
        ssim_l1_strip(tw + ch * T1::kCells, tx, ty0, S.P, ch == 0, esum,
                      [&](int k, const SsimStats& s, const SsimTerms& t) {
            if constexpr (kGrad) {
                // the raw coefficients of every own cell, filler cells included: sweep_tile_adjoint scales them
                const SsimCoef kf = ssim_coef(s, t, A.third * S.P.w_ssim);
                float* cp = cs + 3 * ch * T1::kCells + T1::cell(tx, ty0 + k);
                cp[0] = kf.Ay; cp[T1::kCells] = kf.B; cp[2 * T1::kCells] = kf.Cc;
            }
        });
    float part_e = 0.f, part_m = 0.f;
    float diff_k[kPixPerThread], m_k[kPixPerThread];             // kGrad: per own pixel, 0 for filler pixels
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        if constexpr (kGrad) { diff_k[k] = 0.f; m_k[k] = 0.f; }
        if (gx < W && gy < H) {
            const int pix = gy * W + gx;
            const float diff = mean3_of_sum<F>(esum[k], A);
            const float m = (diff < __ldg(S.P.auto_err + (int64_t)b * n + pix)) ? (valid[k] ? 1.f : 0.f) : 0.f;
            if constexpr (kGrad) { diff_k[k] = diff; m_k[k] = m; }
            // (diff_img * valid_mask) * weight_mask, each product rounded like the eager expression
            part_e = __fadd_rn(part_e, __fmul_rn(__fmul_rn(diff, m), wgt[k]));
            part_m = __fadd_rn(part_m, m);
            const int64_t o = (int64_t)hyp * n + pix;
            if (S.diff) S.diff[o] = diff;
            if (S.mask) S.mask[o] = m;
            if (S.weight) S.weight[o] = wgt[k];
            if (S.rec) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) S.rec[((int64_t)hyp * 3 + ch) * n + pix] = tw[ch * T1::kCells + T1::cell(tx, ty0 + k)].y;
            }
        }
    }
    if constexpr (kGrad) {
        float acc[12];
        sweep_tile_adjoint<F>(S, b, cam, tw, cs, x0, y0, diff_k, m_k, wgt, acc);
        float part[kSweepGradParts];
        part[0] = part_e;
        part[1] = part_m;
#pragma unroll
        for (int i = 0; i < 12; ++i) part[2 + i] = acc[i];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        // fixed-order block sum: for every value the butterfly of warp_sum (so E and V get the forward's bits), then
        // the warps in index order
        const float s = warp_sum_transposed<kSweepGradParts>(part, lane);
        const int idx = (lane >> 1) & 15;
        if (!(lane & 1) && idx < kSweepGradParts) red[idx * (kTileThreads / 32) + warp] = s;
        __syncthreads();
        if (threadIdx.x < kSweepGradParts) {
            const float* r = red + threadIdx.x * (kTileThreads / 32);
            float v = r[0];
            for (int w = 1; w < kTileThreads / 32; ++w) v = __fadd_rn(v, r[w]);
            S.partials[((int64_t)tile * S.N + hyp) * kSweepGradParts + threadIdx.x] = v;
        }
    } else {
        // fixed-order block sum: butterfly within each warp, then the warps in index order
        part_e = warp_sum(part_e);
        part_m = warp_sum(part_m);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) { red[warp] = part_e; red[kTileThreads / 32 + warp] = part_m; }
        __syncthreads();
        if (threadIdx.x == 0) {
            float se = red[0], sm = red[kTileThreads / 32];
            for (int w = 1; w < kTileThreads / 32; ++w) { se = __fadd_rn(se, red[w]); sm = __fadd_rn(sm, red[kTileThreads / 32 + w]); }
            float* dst = S.partials + ((int64_t)tile * S.N + hyp) * 2;
            dst[0] = se;
            dst[1] = sm;
        }
    }
}

// Hypothesis hyp's per-CTA partials ([tiles][N][kParts]) added in tile order: the products E in double (the caller
// rounds to fp32 once), the mask counts V in fp32 (exact: integers below 2^24) and, for kParts = kSweepGradParts,
// d E / d proj in double.
template <int kParts>
__device__ __forceinline__ void sweep_partials_sum(const float* __restrict__ partials, int tiles, int N, int hyp, double& e,
                                                   float& m, double (&g)[12]) {
    e = 0.0;
    m = 0.f;
#pragma unroll
    for (int i = 0; i < kParts - 2; ++i) g[i] = 0.0;
    for (int t = 0; t < tiles; ++t) {
        const float* p = partials + ((int64_t)t * N + hyp) * kParts;
        e += (double)__ldg(p);
        m = __fadd_rn(m, __ldg(p + 1));
#pragma unroll
        for (int i = 0; i < kParts - 2; ++i) g[i] += (double)__ldg(p + 2 + i);
    }
}

// sums[n] = (error_sum, valid_sum) of hypothesis n from its per-CTA partials.
constexpr int kSweepFinishThreads = 128;
__global__ void __launch_bounds__(kSweepFinishThreads)
photo_sweep_finish_kernel(const float* __restrict__ partials, int tiles, int N, float* __restrict__ sums) {
    const int hyp = blockIdx.x * kSweepFinishThreads + threadIdx.x;
    if (hyp >= N) return;
    double e, g[12];
    float m;
    sweep_partials_sum<2>(partials, tiles, N, hyp, e, m, g);
    sums[2 * hyp] = (float)e;
    sums[2 * hyp + 1] = m;
}

// sums[n] exactly as photo_sweep_finish_kernel forms them; g_proj[n] = (d E / d proj, its partials added in tile
// order in double) / valid_sum, NaN where no pixel is valid.
__global__ void __launch_bounds__(kSweepFinishThreads)
photo_sweep_grad_finish_kernel(const float* __restrict__ partials, int tiles, int N, float* __restrict__ sums,
                               float* __restrict__ g_proj) {
    const int hyp = blockIdx.x * kSweepFinishThreads + threadIdx.x;
    if (hyp >= N) return;
    double e, g[12];
    float m;
    sweep_partials_sum<kSweepGradParts>(partials, tiles, N, hyp, e, m, g);
    sums[2 * hyp] = (float)e;
    sums[2 * hyp + 1] = m;
#pragma unroll
    for (int i = 0; i < 12; ++i) g_proj[12 * hyp + i] = (float)(g[i] / (double)m);
}

// ---------------------------------------------------------------------------
// Multi-start refinement: Adam on each hypothesis's pose, descending its loss surface value.  Per step the fused
// forward + adjoint (photo_sweep_kernel<F, true>) and photo_refine_step_kernel, one thread per hypothesis, which
// finishes the sums and the gradient like photo_sweep_grad_finish_kernel, keeps the loss history and the best
// pose seen, maps the gradient to the pose (pose_proj_bwd_body), updates the pose and forms its next K[R|t]
// (pose_proj_fwd_body) with the K of its pair.  Every operation of the update is a separately rounded fp32 operation,
// so a loop of torch operators on fp32 tensors reproduces its bits.
// ---------------------------------------------------------------------------
struct RefineArgs {
    const float* partials;     // [tiles][N][kSweepGradParts] (update) or [tiles][N][2] (last evaluation)
    const float* K;            // [B,9]
    float* poses;              // [N,6], updated in place
    float* m; float* v;        // [N,6] Adam moments
    float* proj;               // [N,12] K[R|t] of the poses, rewritten after the update
    float* loss;               // [N]: the row of this evaluation
    float* best_loss; int* best_step; float* best_pose;   // [N], [N], [N,6]
    int tiles, N, per, step;   // N = B * per pair-major hypotheses; step: the number of updates behind this evaluation
    int project;               // instead of an evaluation: K[R|t] of the starting poses into proj
};

// The step's scalars, each rounded to fp32 once from double on the host.  first: the first evaluation of the call
// (m = v = 0 and no best pose yet).
struct AdamStep {
    float b1, a1, b2, a2, c1, c2, e;
    int first;
};

constexpr float kRefineSign = -1.f;       // inverse_warp2 takes -pose (compute_photometric_error, helpers.py:9)

template <bool kUpdate, bool kNoFma>
__global__ void __launch_bounds__(kSweepFinishThreads)
photo_refine_step_kernel(const RefineArgs R, const AdamStep s) {
    const int hyp = blockIdx.x * kSweepFinishThreads + threadIdx.x;
    if (hyp >= R.N) return;
    const float* K = R.K + 9 * (hyp / R.per);
    if (R.project) {
        pose_proj_fwd_body<kNoFma>(R.poses + hyp * 6, kRefineSign, K, 1, R.proj, hyp);
        return;
    }
    double e, g[12];
    float V;
    sweep_partials_sum<kUpdate ? kSweepGradParts : 2>(R.partials, R.tiles, R.N, hyp, e, V, g);
    const float loss = __fdiv_rn((float)e, V);
    R.loss[hyp] = loss;
    float p[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) p[j] = R.poses[hyp * 6 + j];
    // best so far: the smallest finite loss, the first evaluation that reaches it
    const int best = s.first ? -1 : R.best_step[hyp];
    if (fabsf(loss) < INFINITY && (best < 0 || loss < R.best_loss[hyp])) {
        R.best_loss[hyp] = loss;
        R.best_step[hyp] = R.step;
#pragma unroll
        for (int j = 0; j < 6; ++j) R.best_pose[hyp * 6 + j] = p[j];
    } else if (s.first) {
        R.best_loss[hyp] = __int_as_float(0x7fffffff);
        R.best_step[hyp] = -1;
#pragma unroll
        for (int j = 0; j < 6; ++j) R.best_pose[hyp * 6 + j] = p[j];
    }
    if constexpr (kUpdate) {
        float* m = R.m + hyp * 6;
        float* v = R.v + hyp * 6;
        if (V > 0.f) {
            float g_proj[12], gp[6];
#pragma unroll
            for (int i = 0; i < 12; ++i) g_proj[i] = (float)(g[i] / (double)V);
            pose_proj_bwd_body(p, kRefineSign, K, 1, g_proj, gp, 0);
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const float mj = __fadd_rn(__fmul_rn(s.b1, s.first ? 0.f : m[j]), __fmul_rn(s.a1, gp[j]));
                const float vj = __fadd_rn(__fmul_rn(s.b2, s.first ? 0.f : v[j]), __fmul_rn(s.a2, __fmul_rn(gp[j], gp[j])));
                const float den = __fadd_rn(__fdiv_rn(sqrtf(vj), s.c2), s.e);
                p[j] = __fsub_rn(p[j], __fmul_rn(s.c1, __fdiv_rn(mj, den)));
                m[j] = mj;
                v[j] = vj;
                R.poses[hyp * 6 + j] = p[j];
            }
            pose_proj_fwd_body<kNoFma>(p, kRefineSign, K, 1, R.proj, hyp);
        } else if (s.first) {
            // frozen: no valid pixel, so no gradient; the pose (and its K[R|t]) stays, the moments start at 0
#pragma unroll
            for (int j = 0; j < 6; ++j) { m[j] = 0.f; v[j] = 0.f; }
        }
    }
}

// The shape check and the launch arguments that every photometric entry point shares.
static int fill_photo_common(PhotoArgs& P, const char* who, int N, int H, int W, float w_l1, float w_ssim, int flags) {
    if (N <= 0 || H < 2 || W < 2) { set_error("%s: bad shape N=%d H=%d W=%d", who, N, H, W); return 1; }
    P.A = make_arith(H, W, flags);
    P.w_l1 = w_l1; P.w_ssim = w_ssim;
    P.C1 = kSsimC1; P.C2 = kSsimC2;
    return 0;
}

static int fill_photo(PhotoArgs& P, int N, int H, int W, float w_l1, float w_ssim, int flags, const char* who) {
    if (int rc = fill_photo_common(P, who, N, H, W, w_l1, w_ssim, flags)) return rc;
    if (N > 65535) { set_error("%s: N=%d exceeds 65535", who, N); return 1; }
    if (!P.tgt || !P.rec || !P.pd || !P.cd) { set_error("%s: null input pointer", who); return 1; }
    return 0;
}

}  // namespace tcsfm

using namespace tcsfm;

extern "C" int tcsfm_photo_coef_planes(void) { return kPhotoCoefPlanes; }

extern "C" int tcsfm_photo_fwd(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb, int64_t src_sc,
                               const float* rec, const float* proj_depth, const float* comp_depth,
                               float* auto_err, float* diff, float* auto_mask, float* weight, float* coef,
                               const float* valid,
                               int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    PhotoArgs P;
    memset(&P, 0, sizeof(P));
    P.tgt = tgt; P.tgt_sb = tgt_sb; P.tgt_sc = tgt_sc; P.src = src; P.src_sb = src_sb; P.src_sc = src_sc;
    P.rec = rec; P.pd = proj_depth; P.cd = comp_depth;
    P.auto_err = auto_err; P.diff = diff; P.auto_mask = auto_mask; P.weight = weight; P.coef = coef; P.valid = valid;
    if (int rc = fill_photo(P, N, H, W, w_l1, w_ssim, flags, "tcsfm_photo_fwd")) return rc;
    if (!src) { set_error("tcsfm_photo_fwd: null src"); return 1; }
    const size_t smem = 6 * Tile<1>::kCells * sizeof(float2);
#ifndef TCSFM_HOST_EMU
    cudaError_t e = cudaSuccess;
    TCSFM_DISPATCH_FLAVOUR(flags, e = cudaFuncSetAttribute(photo_fwd_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (e != cudaSuccess) { set_error("tcsfm_photo_fwd: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return 2; }
#endif
    dim3 grid(tile_count(H, W), N), block(kTileThreads);
    TCSFM_DISPATCH_FLAVOUR(flags, TCSFM_LAUNCH(photo_fwd_kernel<F>, grid, block, smem, stream, P));
    return check_launch("tcsfm_photo_fwd");
}

extern "C" int tcsfm_photo_bwd(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* rec,
                               const float* proj_depth, const float* comp_depth, const float* coef,
                               const float* g_diff, const float* g_weight, float* g_rec, float* g_pd, float* g_cd,
                               int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    PhotoArgs P;
    memset(&P, 0, sizeof(P));
    P.tgt = tgt; P.tgt_sb = tgt_sb; P.tgt_sc = tgt_sc; P.rec = rec; P.pd = proj_depth; P.cd = comp_depth;
    P.coef = const_cast<float*>(coef); P.g_diff = g_diff; P.g_weight = g_weight; P.g_rec = g_rec; P.g_pd = g_pd; P.g_cd = g_cd;
    if (int rc = fill_photo(P, N, H, W, w_l1, w_ssim, flags, "tcsfm_photo_bwd")) return rc;
    if (!coef) { set_error("tcsfm_photo_bwd: the forward's coef workspace is required"); return 1; }
    const size_t smem = 9 * Tile<1>::kCells * sizeof(float);
    dim3 grid(tile_count(H, W), N), block(kTileThreads);
    TCSFM_LAUNCH(photo_bwd_kernel, grid, block, smem, stream, P);
    return check_launch("tcsfm_photo_bwd");
}

extern "C" int64_t tcsfm_photo_sweep_partial_floats(int N, int H, int W) {
    if (N <= 0 || H <= 0 || W <= 0) return 0;
    return 2 * (int64_t)N * tile_count(H, W);
}

// The argument checks and launch arguments shared by the sweep, sweep_grad and refine entry points: B pairs of N
// hypotheses each, whose images are `*_sb` floats apart.
static int fill_sweep(SweepArgs& S, const char* who, int B, const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src,
                      int64_t src_sb, int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                      const float* proj, float* scratch, float* partials, float* sums, int N, int H, int W, float w_l1,
                      float w_ssim, int flags) {
    memset(&S, 0, sizeof(S));
    if (int rc = fill_photo_common(S.P, who, N, H, W, w_l1, w_ssim, flags)) return rc;
    if (B < 1) { set_error("%s: bad pair count B=%d", who, B); return 1; }
    if ((int64_t)B * N > 0x7fffffff) { set_error("%s: B=%d pairs x N=%d hypotheses exceed 2^31 - 1", who, B, N); return 1; }
    if (!tgt || !src || !tgt_depth || !src_depth || !kinv || !proj) { set_error("%s: null input pointer", who); return 1; }
    if (!scratch || !partials || !sums) { set_error("%s: null scratch, partials or sums", who); return 1; }
    const int tiles = tile_count(H, W), total = B * N;
    if ((int64_t)tiles * total > 0x7fffffff) {
        set_error("%s: %s%d hypotheses of %d tiles exceed the grid", who, B > 1 ? "B x N = " : "N=", total, tiles); return 1;
    }
    // the kernels address a channel plane with 32-bit offsets from the pair's base
    const int64_t n = (int64_t)H * W;
    if (tgt_sc < 0 || src_sc < 0 || 2 * tgt_sc + n > 0x7fffffff || 2 * src_sc + n > 0x7fffffff) {
        set_error("%s: channel strides %lld / %lld out of range", who, (long long)tgt_sc, (long long)src_sc); return 1;
    }
    if (tgt_sb < 0 || src_sb < 0) {
        set_error("%s: batch strides %lld / %lld are negative", who, (long long)tgt_sb, (long long)src_sb); return 1;
    }
    S.P.tgt = tgt; S.P.tgt_sb = tgt_sb; S.P.tgt_sc = tgt_sc; S.P.src = src; S.P.src_sb = src_sb; S.P.src_sc = src_sc;
    S.P.auto_err = scratch;
    S.tdep = tgt_depth; S.sdep = src_depth; S.kinv = kinv; S.proj = proj; S.partials = partials;
    S.N = total; S.tiles = tiles; S.per = N;
    return 0;
}

// dynamic shared memory of photo_auto_err_kernel and photo_sweep_kernel<F, false>, and of photo_sweep_kernel<F, true>
constexpr size_t kSweepSmem = 3 * Tile<1>::kCells * sizeof(float2);
constexpr size_t kSweepGradSmem = kSweepSmem + kPhotoCoefPlanes * Tile<1>::kCells * sizeof(float);

// The kernels for B pairs: B = 1 takes the instantiations without pair arithmetic.
template <int F>
static auto auto_err_kernel(int B) { return B > 1 ? photo_auto_err_kernel<F, true> : photo_auto_err_kernel<F, false>; }
template <int F, bool kGrad>
static auto sweep_kernel(int B) { return B > 1 ? photo_sweep_kernel<F, kGrad, true> : photo_sweep_kernel<F, kGrad, false>; }

// The auto-mask error of every pair into the scratch: tiles x B CTAs.
static int sweep_auto_err(const SweepArgs& S, const char* who, int B, int flags, void* stream) {
    TCSFM_DISPATCH_FLAVOUR(flags, auto* auto_err = auto_err_kernel<F>(B);
                                  TCSFM_LAUNCH(auto_err, dim3(S.tiles, B), dim3(kTileThreads), kSweepSmem, stream, S.P));
    return check_launch(who);
}

// What the sweep_grad and refine entry points do before their first photo_sweep_kernel<F, true>: raise that kernel's
// dynamic shared-memory limit and launch the pairs' auto-mask error into the scratch.
static int sweep_grad_prologue(const SweepArgs& S, const char* who, int B, int flags, void* stream) {
#ifndef TCSFM_HOST_EMU
    cudaError_t e = cudaSuccess;
    TCSFM_DISPATCH_FLAVOUR(flags, e = cudaFuncSetAttribute(sweep_kernel<F, true>(B), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSweepGradSmem));
    if (e != cudaSuccess) { set_error("%s: cannot raise dynamic smem: %s", who, cudaGetErrorString(e)); return 2; }
#endif
    return sweep_auto_err(S, who, B, flags, stream);
}

static int photo_sweep(const char* who, int B, const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src,
                       int64_t src_sb, int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                       const float* proj, float* scratch, float* partials, float* sums,
                       float* rec, float* diff, float* mask, float* weight,
                       int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    SweepArgs S;
    if (int rc = fill_sweep(S, who, B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth, kinv, proj, scratch,
                            partials, sums, N, H, W, w_l1, w_ssim, flags)) return rc;
    S.rec = rec; S.diff = diff; S.mask = mask; S.weight = weight;
    const int tiles = S.tiles, total = S.N;
    if (int rc = sweep_auto_err(S, who, B, flags, stream)) return rc;
    TCSFM_DISPATCH_FLAVOUR(flags, auto* sweep = sweep_kernel<F, false>(B);
                                  TCSFM_LAUNCH(sweep, dim3((unsigned)(tiles * total)), dim3(kTileThreads), kSweepSmem, stream, S));
    if (int rc = check_launch(who)) return rc;
    TCSFM_LAUNCH(photo_sweep_finish_kernel, dim3((total + kSweepFinishThreads - 1) / kSweepFinishThreads), dim3(kSweepFinishThreads),
                 0, stream, partials, tiles, total, sums);
    return check_launch(who);
}

static int photo_sweep_grad(const char* who, int B, const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src,
                            int64_t src_sb, int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                            const float* proj, float* scratch, float* partials, float* sums, float* g_proj,
                            int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    SweepArgs S;
    if (int rc = fill_sweep(S, who, B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth, kinv, proj, scratch,
                            partials, sums, N, H, W, w_l1, w_ssim, flags)) return rc;
    if (!g_proj) { set_error("%s: null g_proj", who); return 1; }
    const int tiles = S.tiles, total = S.N;
    if (int rc = sweep_grad_prologue(S, who, B, flags, stream)) return rc;
    TCSFM_DISPATCH_FLAVOUR(flags, auto* sweep = sweep_kernel<F, true>(B);
                                  TCSFM_LAUNCH(sweep, dim3((unsigned)(tiles * total)), dim3(kTileThreads), kSweepGradSmem, stream, S));
    if (int rc = check_launch(who)) return rc;
    TCSFM_LAUNCH(photo_sweep_grad_finish_kernel, dim3((total + kSweepFinishThreads - 1) / kSweepFinishThreads),
                 dim3(kSweepFinishThreads), 0, stream, partials, tiles, total, sums, g_proj);
    return check_launch(who);
}

static int photo_refine(const char* who, int B, const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src,
                        int64_t src_sb, int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                        const float* K, float* poses, float* m, float* v, float* proj, float* scratch, float* partials,
                        float* loss, float* best_loss, int* best_step, float* best_pose,
                        int N, int H, int W, int steps, double lr, double beta1, double beta2, double eps,
                        float w_l1, float w_ssim, int flags, int pose_flags, void* stream) {
    if (!K || !poses || !m || !v || !best_loss || !best_step || !best_pose) { set_error("%s: null pointer", who); return 1; }
    if (steps < 0) { set_error("%s: steps=%d is negative", who, steps); return 1; }
    if (B > 0 && N > 0 && ((int64_t)steps + 1) * B * N > 0x7fffffff) {
        set_error("%s: the loss history of %d steps x %lld hypotheses exceeds 2^31 - 1 entries", who, steps,
                  (long long)B * N);
        return 1;
    }
    if (!(lr > 0.0 && lr < INFINITY) || !(eps > 0.0 && eps < INFINITY) || !(beta1 >= 0.0 && beta1 < 1.0) ||
        !(beta2 >= 0.0 && beta2 < 1.0)) {
        set_error("%s: bad optimizer arguments lr=%g betas=(%g, %g) eps=%g", who, lr, beta1, beta2, eps); return 1;
    }
    // `loss` stands in for the sums of fill_sweep's checks: each row of it is written from the partials here
    SweepArgs S;
    if (int rc = fill_sweep(S, who, B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth, kinv, proj, scratch,
                            partials, loss, N, H, W, w_l1, w_ssim, flags)) return rc;
    const int tiles = S.tiles, total = S.N;
    if (int rc = sweep_grad_prologue(S, who, B, flags, stream)) return rc;
    auto* step = (pose_flags & TCSFM_ARITH_BMM_NOFMA) ? photo_refine_step_kernel<true, true> : photo_refine_step_kernel<true, false>;
    const dim3 step_grid((total + kSweepFinishThreads - 1) / kSweepFinishThreads), step_block(kSweepFinishThreads);
    RefineArgs R;
    memset(&R, 0, sizeof(R));
    R.partials = partials; R.K = K; R.poses = poses; R.m = m; R.v = v; R.proj = proj;
    R.best_loss = best_loss; R.best_step = best_step; R.best_pose = best_pose;
    R.tiles = tiles; R.N = total; R.per = N;
    AdamStep s;
    s.b1 = (float)beta1; s.a1 = (float)(1.0 - beta1); s.b2 = (float)beta2; s.a2 = (float)(1.0 - beta2); s.e = (float)eps;
    s.c1 = s.c2 = 0.f;
    s.first = 1;
    // K[R|t] of the starting poses: one pair reads K[i % 1] in the pose kernel, B pairs their own K in the step kernel
    if (B == 1) {
        if (int rc = tcsfm_pose_proj_fwd(poses, kRefineSign, K, 1, proj, N, pose_flags, stream)) return rc;
    } else {
        R.project = 1;
        TCSFM_LAUNCH(step, step_grid, step_block, 0, stream, R, s);
        if (int rc = check_launch(who)) return rc;
        R.project = 0;
    }
    for (int t = 1; t <= steps; ++t) {
        TCSFM_DISPATCH_FLAVOUR(flags, auto* sweep = sweep_kernel<F, true>(B);
                                      TCSFM_LAUNCH(sweep, dim3((unsigned)(tiles * total)), dim3(kTileThreads), kSweepGradSmem, stream, S));
        if (int rc = check_launch(who)) return rc;
        s.c1 = (float)(lr / (1.0 - pow(beta1, (double)t)));
        s.c2 = (float)sqrt(1.0 - pow(beta2, (double)t));
        s.first = t == 1;
        R.loss = loss + (int64_t)(t - 1) * total;
        R.step = t - 1;
        TCSFM_LAUNCH(step, step_grid, step_block, 0, stream, R, s);
        if (int rc = check_launch(who)) return rc;
    }
    // the poses after the last update: their loss and the last chance to be the best
    TCSFM_DISPATCH_FLAVOUR(flags, auto* sweep = sweep_kernel<F, false>(B);
                                  TCSFM_LAUNCH(sweep, dim3((unsigned)(tiles * total)), dim3(kTileThreads), kSweepSmem, stream, S));
    if (int rc = check_launch(who)) return rc;
    s.first = steps == 0;
    R.loss = loss + (int64_t)steps * total;
    R.step = steps;
    auto* last = photo_refine_step_kernel<false, false>;
    TCSFM_LAUNCH(last, step_grid, step_block, 0, stream, R, s);
    return check_launch(who);
}

extern "C" int64_t tcsfm_photo_sweep_grad_partial_floats(int N, int H, int W) {
    if (N <= 0 || H <= 0 || W <= 0) return 0;
    return kSweepGradParts * (int64_t)N * tile_count(H, W);
}

extern "C" int tcsfm_photo_sweep(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                                 const float* tgt_depth, const float* src_depth, const float* kinv, const float* proj,
                                 float* scratch, float* partials, float* sums,
                                 float* rec, float* diff, float* mask, float* weight,
                                 int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    return photo_sweep("tcsfm_photo_sweep", 1, tgt, 0, tgt_sc, src, 0, src_sc, tgt_depth, src_depth, kinv, proj, scratch,
                       partials, sums, rec, diff, mask, weight, N, H, W, w_l1, w_ssim, flags, stream);
}

extern "C" int tcsfm_photo_sweep_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb,
                                       int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                                       const float* proj, float* scratch, float* partials, float* sums,
                                       float* rec, float* diff, float* mask, float* weight,
                                       int B, int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    return photo_sweep("tcsfm_photo_sweep_pairs", B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth, kinv,
                       proj, scratch, partials, sums, rec, diff, mask, weight, N, H, W, w_l1, w_ssim, flags, stream);
}

extern "C" int tcsfm_photo_sweep_grad(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                                      const float* tgt_depth, const float* src_depth, const float* kinv, const float* proj,
                                      float* scratch, float* partials, float* sums, float* g_proj,
                                      int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    return photo_sweep_grad("tcsfm_photo_sweep_grad", 1, tgt, 0, tgt_sc, src, 0, src_sc, tgt_depth, src_depth, kinv, proj,
                            scratch, partials, sums, g_proj, N, H, W, w_l1, w_ssim, flags, stream);
}

extern "C" int tcsfm_photo_sweep_grad_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src,
                                            int64_t src_sb, int64_t src_sc, const float* tgt_depth, const float* src_depth,
                                            const float* kinv, const float* proj, float* scratch, float* partials,
                                            float* sums, float* g_proj,
                                            int B, int N, int H, int W, float w_l1, float w_ssim, int flags, void* stream) {
    return photo_sweep_grad("tcsfm_photo_sweep_grad_pairs", B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth,
                            kinv, proj, scratch, partials, sums, g_proj, N, H, W, w_l1, w_ssim, flags, stream);
}

extern "C" int tcsfm_photo_refine(const float* tgt, int64_t tgt_sc, const float* src, int64_t src_sc,
                                  const float* tgt_depth, const float* src_depth, const float* kinv, const float* K,
                                  float* poses, float* m, float* v, float* proj, float* scratch, float* partials,
                                  float* loss, float* best_loss, int* best_step, float* best_pose,
                                  int N, int H, int W, int steps, double lr, double beta1, double beta2, double eps,
                                  float w_l1, float w_ssim, int flags, int pose_flags, void* stream) {
    return photo_refine("tcsfm_photo_refine", 1, tgt, 0, tgt_sc, src, 0, src_sc, tgt_depth, src_depth, kinv, K, poses, m, v,
                        proj, scratch, partials, loss, best_loss, best_step, best_pose, N, H, W, steps, lr, beta1, beta2,
                        eps, w_l1, w_ssim, flags, pose_flags, stream);
}

extern "C" int tcsfm_photo_refine_pairs(const float* tgt, int64_t tgt_sb, int64_t tgt_sc, const float* src, int64_t src_sb,
                                        int64_t src_sc, const float* tgt_depth, const float* src_depth, const float* kinv,
                                        const float* K, float* poses, float* m, float* v, float* proj, float* scratch,
                                        float* partials, float* loss, float* best_loss, int* best_step, float* best_pose,
                                        int B, int N, int H, int W, int steps, double lr, double beta1, double beta2,
                                        double eps, float w_l1, float w_ssim, int flags, int pose_flags, void* stream) {
    return photo_refine("tcsfm_photo_refine_pairs", B, tgt, tgt_sb, tgt_sc, src, src_sb, src_sc, tgt_depth, src_depth, kinv,
                        K, poses, m, v, proj, scratch, partials, loss, best_loss, best_step, best_pose, N, H, W, steps, lr,
                        beta1, beta2, eps, w_l1, w_ssim, flags, pose_flags, stream);
}
