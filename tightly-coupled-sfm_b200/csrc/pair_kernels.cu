// Fused pair loss: Compute_Loss.compute_pairwise_loss (reference losses.py:151-183)
// + the sums of mean_on_mask (losses.py:142-149), forward and backward.
//
// Both kernels are instruction-issue bound (hundreds of fp32 operations per pixel for
// 40-44 algorithmic bytes), so the design minimises issued instructions while keeping
// every rounding step of eager PyTorch:
//
// Forward (64x16 tile, 256 threads, a vertical strip of 4 pixels per thread):
//   A. each thread back-projects / projects its pixels (the CTA also the 1-pixel halo
//      ring), gathers the 4 bilinear taps of the 3 source channels and stores
//      (target, warped) as one float2 per cell of a shared-memory tile.  Two strip pixels
//      are staged together (geometry of both, every gather of both, then the blends) so
//      that their load latencies overlap;
//   C. per channel a thread slides a 3x3 register window down its strip: one LDS.64 per
//      tap, squares/products once per tap, and the five avg_pool2d-ordered running sums
//      as packed fp32x2 adds; /9 is an exact 3-instruction sequence.  L1, auto-mask,
//      SSIM, depth-consistency weight, block-reduced masked sums (3 atomics per CTA).
//   When a backward pass will follow, the SSIM adjoint coefficients (3 per channel) are
//   written next to diff_img/mask (40 B/px of workspace) so that the backward neither
//   re-warps a 2-pixel halo nor recomputes window statistics.
//
// Backward (same tiling), three phases with disjoint register working sets:
//   B. cp.async the nine coefficient planes of the tile + 1 ring into shared memory next
//      to the per-cell upstream gradient (explicit grad + masked-mean term + per-pixel min
//      routing); cells with a zero upstream are zero-filled without reading HBM;
//   C. separable rolling 3x3 sums of coefficient x upstream (reflection = two conditional
//      extra terms) reduce to the line g_w = P + w * Q per channel; (P, Q) and the own
//      depth replace the coefficients of the thread's own cells;
//   D. per own pixel: L1 / depth-consistency adjoints, then the bilinear + projective
//      adjoint: grad(target depth) is a direct store, grad(source depth) a 4-tap atomic
//      scatter, grad(K[R|t]) 12 block-reduced accumulators per batch element.
#include "tile.cuh"
#ifndef TCSFM_HOST_EMU
#include <cuda.h>                  // CUtensorMap (the encoder itself is fetched through cudaGetDriverEntryPoint: no libcuda link)
#endif

namespace tcsfm {

// resident CTAs per SM the register allocation targets (256 threads each)
#ifndef TCSFM_FWD_MIN_BLOCKS
#define TCSFM_FWD_MIN_BLOCKS 3
#endif
#ifndef TCSFM_BWD_MIN_BLOCKS
#define TCSFM_BWD_MIN_BLOCKS 4      // measured: 4 CTAs/SM (64 registers, 24 B of spills) beats 3 CTAs/SM without spills by 9 %
#endif
#ifndef TCSFM_BWD_D_UNROLL
#define TCSFM_BWD_D_UNROLL 2      // measured: 2 overlaps two pixels' gather chains (-3%), 4 spills
#endif
constexpr int kBwdDUnroll = TCSFM_BWD_D_UNROLL;

constexpr int kMaxGroups = 8;
constexpr int kCoefPlanes = 10;      // 3 channels x (A, B, C) + the un-weighted photometric error

struct PairLaunch {
    tcsfm_pair_group g[kMaxGroups];
    Arith A;
    float w_l1, w_ssim, C1, C2;
    int flags;
    int vec16;                       // backward: every coefficient row start is 16-byte aligned (W % 4 == 0, aligned base)
#ifndef TCSFM_HOST_EMU
    alignas(64) CUtensorMap coef_map[kMaxGroups];   // backward, TMA staging: the group's workspace as a [B][10][H][W] tensor
#endif
};

struct PairCtx {
    const float* tgt; const float* ref; const float* tdep; const float* rdep;
    int tgt_sc, ref_sc;              // channel strides; fill_launch checks that 3 planes stay below 2^31 elements
};

__device__ __forceinline__ PairCtx make_ctx(const tcsfm_pair_group& g, int b, int n) {
    PairCtx c;
    c.tgt = pin_pointer(g.tgt_img + b * g.tgt_sb);
    c.ref = pin_pointer(g.ref_img + b * g.ref_sb);
    c.tdep = pin_pointer(g.tgt_depth + (int64_t)b * n);
    c.rdep = pin_pointer(g.ref_depth ? g.ref_depth + (int64_t)b * n : nullptr);
    c.tgt_sc = (int)g.tgt_sc;
    c.ref_sc = (int)g.ref_sc;
    return c;
}

template <int F>
__global__ void __launch_bounds__(kTileThreads, TCSFM_FWD_MIN_BLOCKS)
pair_fwd_kernel(const __grid_constant__ PairLaunch L) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float2, tw);                       // [3][T1::kCells] (target, warped)
    TCSFM_SHARED float red[3 * (kTileThreads / 32)];

    const tcsfm_pair_group& g = L.g[blockIdx.z];
    const Arith& A = L.A;
    const int H = A.H, W = A.W, n = H * W;
    const int b = blockIdx.y;
    int x0, y0;
    tile_origin(blockIdx.x, W, x0, y0);
    const Cam cam = load_cam(g.kinv, g.proj, b);
    const PairCtx c = make_ctx(g, b, n);
    const bool auto_mask = (L.flags & TCSFM_AUTO_MASK) != 0;
    const bool depth_mask = (L.flags & TCSFM_DEPTH_MASK) != 0;
    const bool depth_consist = (L.flags & TCSFM_DEPTH_CONSIST) != 0;
    const bool need_depth = depth_mask || depth_consist;
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;

    float own_mask[kPixPerThread], own_dd[kPixPerThread];
    // ---- phase A: own pixels.  The target depths head the longest dependent chain (depth ->
    //      projection -> tap addresses -> gathers), so all of a thread's are requested first. ----
    // Own cells that no consumer reads (more than a pixel outside the image, partial tiles only) are
    // filled like the others, from a clamped source pixel: the fills carry no control flow.
    auto own_src = [&](int k, int& sx, int& sy) {
        const int gy = y0 + ty0 + k;
        sx = min(max(gx < W ? gx : 2 * W - 2 - gx, 0), W - 1);      // reflect1 for the one column / row past the edge
        sy = min(max(gy < H ? gy : 2 * H - 2 - gy, 0), H - 1);
    };
    float src_depth[kPixPerThread];
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        int sx, sy;
        own_src(k, sx, sy);
        src_depth[k] = __ldg(c.tdep + sy * W + sx);
    }
    int ring_x = 0, ring_y = 0, ring_at = 0;          // the thread's halo-ring cell, if it has one
    bool ring_ok = false;
    float ring_depth = 1.0f;
    if (threadIdx.x < kRingCells) {
        int cx, cy;
        ring_cell(threadIdx.x, cx, cy);
        ring_at = T1::cell(cx, cy);
        ring_ok = T1::cell_to_reflected(ring_at, x0, y0, H, W, ring_y, ring_x);
        if (ring_ok) ring_depth = __ldg(c.tdep + ring_y * W + ring_x);
    }
    // Two strip pixels at a time, staged by hand (geometry of both, then every gather of both, then
    // the blends): ptxas keeps the cells strictly serial otherwise, because the IEEE-division slow
    // paths are calls.  Cells no consumer reads are filled from a clamped source pixel (no branches).
#pragma unroll
    for (int k0 = 0; k0 < kPixPerThread; k0 += 2) {
        WarpPt p[2];
        TapIdx ti[2];
        int pix[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            int sx, sy;
            own_src(k0 + j, sx, sy);
            pix[j] = sy * W + sx;
            warp_point<F>(cam, A, sx, sy, src_depth[k0 + j], p[j]);
            ti[j] = make_taps(p[j], H, W);
        }
        Taps tv[2][3], td[2];
        float tg[2][3], rf[2][3];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                tv[j][ch] = load_taps(c.ref, ch * c.ref_sc, ti[j], W);
                tg[j][ch] = __ldg(c.tgt + (ch * c.tgt_sc + pix[j]));
                rf[j][ch] = auto_mask ? __ldg(c.ref + (ch * c.ref_sc + pix[j])) : 0.f;
            }
            if (need_depth) td[j] = load_taps(c.rdep, 0, ti[j], W);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int k = k0 + j, gy = y0 + ty0 + k;
            const int cell = T1::cell(tx, ty0 + k);
            const bool own = gx < W && gy < H;
            float wv[3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                wv[ch] = blend(tv[j][ch], ti[j]);
                tw[ch * T1::kCells + cell] = make_float2(tg[j][ch], wv[ch]);
            }
            float m = (p[j].valid && own) ? 1.f : 0.f;
            if (auto_mask) {
                float l1[3], ar[3];
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    l1[ch] = clamp01_nan(fabsf(__fsub_rn(tg[j][ch], wv[ch])));
                    ar[ch] = fabsf(__fsub_rn(tg[j][ch], rf[j][ch]));
                }
                if (!(mean3<F>(l1[0], l1[1], l1[2], A) < mean3<F>(ar[0], ar[1], ar[2], A))) m = 0.f;
            }
            own_mask[k] = m;
            own_dd[k] = (need_depth && own) ? depth_inconsistency(p[j].Z, blend(td[j], ti[j])) : 0.f;
        }
    }
    // ---- phase A': the halo ring (one cell per thread) ----
    if (threadIdx.x < kRingCells) {
        WarpPt p;
        if (ring_ok) fill_warped_cell<F>(cam, A, c.tgt, c.tgt_sc, c.ref, c.ref_sc, ring_x, ring_y, ring_depth, tw, ring_at, p);
        else zero_cell(tw, ring_at);
    }
    __syncthreads();

    // ---- phase C: 3x3 statistics down the strip, one channel at a time ----
    float esum[kPixPerThread];
    float* coef_base = pin_pointer(g.coef ? g.coef + (int64_t)b * kCoefPlanes * n : nullptr);   // offsets below: < 2^31 (fill_launch)
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        ssim_l1_strip(tw + ch * T1::kCells, tx, ty0, L, ch == 0, esum,
                      [&](int k, const SsimStats& s, const SsimTerms& t) {
            const int gy = y0 + ty0 + k;
            if (coef_base && gx < W && gy < H) {
                // d diff / d ssim_c = (1 - dd) * (1/3) * w_ssim ; the backward multiplies by its upstream
                const float gq = (depth_mask ? (1.0f - own_dd[k]) : 1.0f) * A.third * L.w_ssim;
                const SsimCoef kf = ssim_coef(s, t, gq);            // x = target, y = warped
                const int o = (3 * ch) * n + gy * W + gx;
                store_streaming(coef_base + o, kf.Ay);
                store_streaming(coef_base + (o + n), kf.B);
                store_streaming(coef_base + (o + 2 * n), kf.Cc);
            }
        });
    }
    float part[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        if (gx < W && gy < H) {
            const float s = esum[k];
            const float diff0 = mean3_of_sum<F>(s, A);
            float diff = diff0;
            if (depth_mask) diff = __fmul_rn(diff0, __fsub_rn(1.0f, own_dd[k]));
            const int64_t o = (int64_t)b * n + gy * W + gx;
            if (g.diff_img) g.diff_img[o] = diff;
            if (g.mask) g.mask[o] = own_mask[k];
            if (coef_base) store_streaming(coef_base + (9 * n + gy * W + gx), diff0);
            part[0] += diff * own_mask[k];
            part[1] += own_mask[k];
            if (depth_consist) part[2] += own_dd[k] * own_mask[k];
        }
    }
    block_atomic_accumulate<3>(part, red, g.sums, threadIdx.x, kTileThreads);
}

// ---------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------
struct BwdScalars {
    float c_rep, c_dep, g_min;
    const float* min_self;          // this group's plane of the min-reprojection candidates (batch element b)
    const float* min_other;         // the other candidate's plane when there are exactly two
};

__device__ __forceinline__ BwdScalars bwd_scalars(const tcsfm_pair_group& g, bool depth_consist, int64_t bn) {
    BwdScalars s;
    s.c_rep = 0.f; s.c_dep = 0.f;
    s.g_min = g.min_base ? __ldg(g.g_min) : 0.f;
    s.min_self = pin_pointer(g.min_base ? g.min_base + bn + (int64_t)g.min_index * g.min_stride : nullptr);
    s.min_other = pin_pointer((g.min_base && g.min_count == 2) ? g.min_base + bn + (int64_t)(1 - g.min_index) * g.min_stride : nullptr);
    if (g.g_scalars) {
        const float s1 = __ldg(g.sums + 1);
        if (s1 > 10000.0f) {                        // mean_on_mask, losses.py:144
            s.c_rep = __ldg(g.g_scalars + 0) / s1;
            if (depth_consist) s.c_dep = __ldg(g.g_scalars + 1) / s1;
        }
    }
    return s;
}

// Upstream gradient of diff_img at pixel `pix` of batch element b: the explicit per-pixel
// gradient, the masked-mean term and the per-pixel min routing (losses.py:129-132).
__device__ __forceinline__ float upstream_diff(const tcsfm_pair_group& g, const BwdScalars& sc, const float* gdiff,
                                               int64_t bn, int pix, float m) {
    float Gd = sc.c_rep * m;
    if (gdiff) Gd += __ldg(gdiff + pix);
    if (sc.min_self) {
        const float v = __ldg(sc.min_self + pix);
        bool win = true;
        // torch.min(dim): the first index holding the minimum wins; a NaN is the minimum
        if (sc.min_other) {                          // the usual two sources: branch-free, both loads in flight
            const float o = __ldg(sc.min_other + pix);
            win = (g.min_index == 1) ? !(o <= v || o != o) : !(o < v || (o != o && v == v));
        } else {
            const float* mine = g.min_base + bn + pix;
            for (int j = 0; j < g.min_count; ++j) {
                if (j == g.min_index) continue;
                const float o = __ldg(mine + (int64_t)j * g.min_stride);
                if (j < g.min_index) win = win && !(o <= v || o != o);
                else win = win && !(o < v || (o != o && v == v));
            }
        }
        if (win) Gd += sc.g_min;
    }
    return Gd;
}

// Out-of-line copy for the rare layouts (more than two min-reprojection candidates): keeps the
// staging code of the common case small.
__device__ __noinline__ float upstream_diff_generic(const tcsfm_pair_group& g, const BwdScalars& sc, const float* gdiff,
                                                    int64_t bn, int pix, float m) {
    return upstream_diff(g, sc, gdiff, bn, pix, m);
}

// Backward tile: row pitch 68 floats with the interior starting at column 4, so that the 64 interior
// cells of a row are 16-byte aligned in shared memory and go global -> shared as 16 cp.async of 16
// bytes instead of 64 of 4.  The left halo sits at column 3, the right halo of row r in the (otherwise
// unused) column 0 of row r + 1; hence the 4 trailing floats.
struct BwdTile {
    static constexpr int kPitch = kTileW + 4;
    static constexpr int kRows = kTileH + 2;
    static constexpr int kCells = kPitch * kRows + 4;                 // floats per plane
    static constexpr int kLogical = (kTileW + 2) * kRows;             // cells that exist
    __device__ __forceinline__ static int cell(int cx, int cy) { return (cy + 1) * kPitch + cx + 4; }
};
constexpr size_t kBwdSmemBytes = 10 * BwdTile::kCells * sizeof(float);
static_assert(4 * (kBwdSmemBytes + 1024) <= 196 * 1024, "four backward CTAs must fit the 196 KB shared-memory carve-out");

// TMA staging (kTma): one cp.async.bulk.tensor brings the nine coefficient planes of the tile + its left halo and the
// rows above / below -- a 68 x 18 x 9 box of the group's [B][10][H][W] workspace starting at (x0 - 4, y0 - 1, plane 0);
// the innermost start coordinate must be a multiple of 16 bytes (measured: x0 - 3 raises an illegal-instruction fault)
// -- into shared memory; rows / columns outside the image arrive as zeros (the tensor map's out-of-bounds fill), so
// the staging needs no per-thread address arithmetic, predicates or cp.async instructions.  The dense box has exactly
// the layout above (pitch 68, interior at column 4, left halo at column 3) with plane stride 68 * 18; the right halo
// column (one value per row and plane) is loaded by 162 threads into registers before the wait and stored, like
// above, into column 0 of the next row (which the box filled with an unused value).
struct TmaTile {
    static constexpr int kBoxW = kTileW + 4, kBoxH = kTileH + 2, kPlanes = 9;
    static constexpr int kPlane = kBoxW * kBoxH;                                   // floats per plane
    static constexpr unsigned kBytes = kPlane * kPlanes * sizeof(float);
};
static_assert(TmaTile::kBoxW == BwdTile::kPitch && TmaTile::kBoxH == BwdTile::kRows, "the TMA box is the backward tile");
constexpr size_t kBwdTmaSmemBytes = (TmaTile::kPlane * 9 + BwdTile::kCells) * sizeof(float) + 16;      // + the mbarrier
static_assert(4 * (kBwdTmaSmemBytes + 1024) <= 196 * 1024, "four backward CTAs must fit the 196 KB shared-memory carve-out");
static_assert((TmaTile::kPlane * 9 + BwdTile::kCells) * sizeof(float) % 8 == 0, "mbarrier alignment");

#ifndef TCSFM_HOST_EMU
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbarrier_init(void* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // make the init visible to the async proxy
}
__device__ __forceinline__ void mbarrier_expect_tx(void* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, void* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 :: "r"(smem_addr(dst)), "l"(map), "r"(smem_addr(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// waits for phase `parity`; a transfer that never completes (bad descriptor) traps instead of hanging the GPU
__device__ __forceinline__ void mbarrier_wait(void* bar, unsigned parity) {
    for (unsigned spin = 0;; ++spin) {
        unsigned done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_addr(bar)), "r"(parity) : "memory");
        if (done) return;
        if (spin > (1u << 24)) __trap();
    }
}
#endif

template <int F, bool kTma>
__global__ void __launch_bounds__(kTileThreads, TCSFM_BWD_MIN_BLOCKS)
pair_bwd_kernel(const __grid_constant__ PairLaunch L) {
    using BT = BwdTile;
#ifndef TCSFM_HOST_EMU
    extern __shared__ __align__(128) unsigned char cs_raw_[];
    float* cs = reinterpret_cast<float*>(cs_raw_);  // [9][plane] coefficients, [BT::kCells] upstream gradient (, mbarrier)
#else
    TCSFM_DYN_SMEM(float, cs);
#endif
    constexpr int kPlane = kTma ? TmaTile::kPlane : BT::kCells;       // floats per coefficient plane in shared memory
    auto pcell = [](int cx, int cy) { return BT::cell(cx, cy); };

    const tcsfm_pair_group& g = L.g[blockIdx.z];
    const Arith& A = L.A;
    const int H = A.H, W = A.W, n = H * W;
    const int b = blockIdx.y;
    int x0, y0;
    tile_origin(blockIdx.x, W, x0, y0);
    const Cam cam = load_cam(g.kinv, g.proj, b);
    const PairCtx c = make_ctx(g, b, n);
    const bool depth_mask = (L.flags & TCSFM_DEPTH_MASK) != 0;
    const bool depth_consist = (L.flags & TCSFM_DEPTH_CONSIST) != 0;
    const bool need_depth = depth_mask || depth_consist;
    const bool shared_grads = (L.flags & TCSFM_SHARED_GRADS) != 0;
    const BwdScalars sc = bwd_scalars(g, depth_consist, (int64_t)b * n);
    const float* gdiff = pin_pointer(g.g_diff ? g.g_diff + (int64_t)b * n : nullptr);
    const float* mask = pin_pointer(g.mask + (int64_t)b * n);
    const float* coef = pin_pointer(g.coef + (int64_t)b * kCoefPlanes * n);      // offsets below: < 2^31 (fill_launch)
    const int tx = threadIdx.x & (kTileW - 1);
    const int ty0 = (threadIdx.x >> 6) * kPixPerThread;
    const int gx = x0 + tx;

    // ---- phase B: the nine coefficient planes of the tile + 1 ring go global -> shared with
    //      cp.async (no register staging, all loads in flight at once; zero fill outside the
    //      image), next to the upstream gradient of diff_img at each ring pixel ----
    float* Gs = cs + 9 * kPlane;                   // [BT::kCells] upstream gradient (0 outside the image)
#ifndef TCSFM_HOST_EMU
    void* bar = Gs + BT::kCells;
    if (kTma) {
        if (threadIdx.x == 0) mbarrier_init(bar, 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            mbarrier_expect_tx(bar, TmaTile::kBytes);
            tma_load_4d(cs, &L.coef_map[blockIdx.z], bar, x0 - 4, y0 - 1, 0, b);
        }
    }
#endif
    // the right halo column of the TMA path: plane j, tile row r (one value per thread, zero outside the image)
    float rh_val = 0.f;
    int rh_at = -1;
    if (kTma && threadIdx.x < TmaTile::kPlanes * BT::kRows) {
        const int j = threadIdx.x / BT::kRows, r = threadIdx.x - j * BT::kRows;
        const int qy = y0 + r - 1, qx = x0 + kTileW;
        rh_at = j * kPlane + BT::cell(kTileW, r - 1);
        if (qy >= 0 && qy < H && qx < W) rh_val = __ldg(coef + (j * n + qy * W + qx));
    }
    const bool two_way = sc.min_other != nullptr;                    // per-pixel min over exactly two sources
    // Upstream gradient of one pixel from its loaded ingredients (mask, explicit grad, own / other
    // min-reprojection candidate); torch.min(dim): the first index holding the minimum wins, a NaN is the minimum.
    const bool many_way = sc.min_self && g.min_count > 2;            // rare: out of line
    const bool one_way = sc.min_self && g.min_count == 1;            // a single source always holds the minimum
    auto combine = [&](int pix, float m, float gd, float v, float o) {
        if (many_way) return upstream_diff_generic(g, sc, gdiff, (int64_t)b * n, pix, m);
        float Gd = sc.c_rep * m + gd;
        const bool win = (g.min_index == 1) ? !(o <= v || o != o) : !(o < v || (o != o && v == v));
        if (one_way || (two_way && win)) Gd += sc.g_min;
        return Gd;
    };
    if (L.vec16) {
        // Rows are 16-byte aligned: a task is four interior cells of one row (288 tasks) or one halo
        // cell (36 tasks).  Its thread loads mask / gradient / candidates as float4, forms the four
        // upstream values and issues one 16-byte cp.async per coefficient plane.  A chunk is read
        // when any of its cells has a non-zero upstream (dead cells multiply by zero later); masked-out
        // pixels of the inverse groups and the losing source of the per-pixel min skip their 36 B/px.
        constexpr int kChunkTasks = BT::kRows * (kTileW / 4), kTasks = kChunkTasks + 2 * BT::kRows;
        auto stage_task = [&](int task) {
            if (task < kChunkTasks) {
                const int row = task / (kTileW / 4), chunk = task - row * (kTileW / 4);
                const int qy = y0 + row - 1, qx = x0 + 4 * chunk;
                const bool inside = qy >= 0 && qy < H && qx < W;
                const int pix = inside ? qy * W + qx : 0;                // pixel 0 stands in: always a valid address
                const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
                const float4 m4 = __ldg(reinterpret_cast<const float4*>(mask + pix));
                const float4 g4 = gdiff ? __ldg(reinterpret_cast<const float4*>(gdiff + pix)) : zero4;
                const float4 v4 = two_way ? __ldg(reinterpret_cast<const float4*>(sc.min_self + pix)) : zero4;
                const float4 o4 = two_way ? __ldg(reinterpret_cast<const float4*>(sc.min_other + pix)) : zero4;
                float4 G4 = zero4;
                if (inside) {
                    G4.x = combine(pix, m4.x, g4.x, v4.x, o4.x);
                    G4.y = combine(pix + 1, m4.y, g4.y, v4.y, o4.y);
                    G4.z = combine(pix + 2, m4.z, g4.z, v4.z, o4.z);
                    G4.w = combine(pix + 3, m4.w, g4.w, v4.w, o4.w);
                }
                const int at = row * BT::kPitch + 4 + 4 * chunk;
                *reinterpret_cast<float4*>(Gs + at) = G4;
                const bool live = (G4.x != 0.f) || (G4.y != 0.f) || (G4.z != 0.f) || (G4.w != 0.f);
                if (!kTma) {
#pragma unroll
                    for (int j = 0; j < 9; ++j) async_copy16(cs + j * BT::kCells + at, coef + (j * n + pix), live);
                }
            } else {
                const int h2 = task - kChunkTasks;
                const int row = h2 >> 1, cx = (h2 & 1) ? kTileW : -1;
                const int qy = y0 + row - 1, qx = x0 + cx;
                const bool inside = qy >= 0 && qy < H && qx >= 0 && qx < W;
                const int pix = inside ? qy * W + qx : 0;
                float Gd = 0.f;
                if (inside) Gd = combine(pix, __ldg(mask + pix), gdiff ? __ldg(gdiff + pix) : 0.f,
                                         two_way ? __ldg(sc.min_self + pix) : 0.f, two_way ? __ldg(sc.min_other + pix) : 0.f);
                const int at = BT::cell(cx, row - 1);
                Gs[at] = Gd;
                const bool live = Gd != 0.f;
                if (!kTma) {
#pragma unroll
                    for (int j = 0; j < 9; ++j) async_copy4(cs + j * BT::kCells + at, coef + (j * n + pix), live);
                }
            }
        };
        stage_task(threadIdx.x);
        if (threadIdx.x + kTileThreads < kTasks) stage_task(threadIdx.x + kTileThreads);
    } else {
        // unaligned rows (W % 4 != 0): one cell at a time, all loads of a thread's cells requested first
        constexpr int kStageIters = (BT::kLogical + kTileThreads - 1) / kTileThreads;
        int st_pix[kStageIters];
        float st_m[kStageIters], st_g[kStageIters], st_v[kStageIters], st_o[kStageIters];
        auto logical_xy = [&](int l, int& cx, int& cy) { cy = l / (kTileW + 2); cx = l - cy * (kTileW + 2) - 1; cy -= 1; };
#pragma unroll
        for (int it = 0; it < kStageIters; ++it) {
            const int l = threadIdx.x + it * kTileThreads;
            int cx, cy;
            logical_xy(l < BT::kLogical ? l : 0, cx, cy);
            const int qx = x0 + cx, qy = y0 + cy;
            const bool inside = l < BT::kLogical && qx >= 0 && qx < W && qy >= 0 && qy < H;
            const int pix = inside ? qy * W + qx : 0;
            st_pix[it] = inside ? pix : -1;
            st_m[it] = __ldg(mask + pix);
            st_g[it] = gdiff ? __ldg(gdiff + pix) : 0.f;
            st_v[it] = two_way ? __ldg(sc.min_self + pix) : 0.f;
            st_o[it] = two_way ? __ldg(sc.min_other + pix) : 0.f;
        }
#pragma unroll
        for (int it = 0; it < kStageIters; ++it) {
            const int l = threadIdx.x + it * kTileThreads;
            if (l >= BT::kLogical) break;
            int cx, cy;
            logical_xy(l, cx, cy);
            const int cell = BT::cell(cx, cy);
            const bool inside = st_pix[it] >= 0;
            const int pix = inside ? st_pix[it] : 0;
            const float Gd = inside ? combine(pix, st_m[it], st_g[it], st_v[it], st_o[it]) : 0.f;
            Gs[cell] = Gd;
            const bool live = Gd != 0.f;
#pragma unroll
            for (int j = 0; j < 9; ++j) async_copy4(cs + j * BT::kCells + cell, coef + (j * n + pix), live);
        }
    }
    __pipeline_commit();
    __pipeline_wait_prior(0);
#ifndef TCSFM_HOST_EMU
    if (kTma) {
        mbarrier_wait(bar, 0);
        if (rh_at >= 0) cs[rh_at] = rh_val;             // after the box has landed: it wrote an unused value there
    }
#endif
    __syncthreads();

    // ---- phase C: separable 3x3 sums of the nine coefficient planes down the strip with a
    //      rolling window of horizontal 3-sums.  Reflection padding folds window taps that fall
    //      outside the image back onto row/column 1 and H-2/W-2: those receive the border
    //      neighbour twice.  Per channel the result is the gradient wrt the warped value as a
    //      line in that value, g_w = P + w * Q; (P, Q) replace the coefficients of the own cells
    //      in shared memory so that phase D starts with an empty register file. ----
    float dep_own[kPixPerThread];                  // heads phase D's longest chain: requested before phase C
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        dep_own[k] = (gx < W && gy < H) ? __ldg(c.tdep + gy * W + gx) : 1.0f;
    }
    {
        float pq[kPixPerThread][6];
        float h[3][9];
        // The three cells (c-1, c, c+1) of a row are read as one aligned 8-byte pair and one single:
        // even columns pair (c, c+1) and take c-1 alone, odd columns pair (c-1, c) and take c+1 alone
        // (two shared-memory wavefronts per warp instead of three).  The upstream weights are permuted
        // to match; a border neighbour that reflection folds back counts twice.
        const int par = tx & 1;
        const float dup_l = (gx == 1) ? 2.f : 1.f, dup_r = (gx == W - 2) ? 2.f : 1.f;
        const float f_a = par ? dup_l : 1.f, f_b = par ? 1.f : dup_r, f_c = par ? dup_r : dup_l;
        const int single_at = par ? 2 : -1;                  // offset of the single cell from the pair
        auto hsum = [&](int r, float (&out)[9]) {          // horizontal 3-sums of tile row ty0 - 1 + r
            const int c0 = BT::cell(tx, ty0 - 1 + r) - par;  // even: the pair starts at the centre cell
            const float2 gp = *reinterpret_cast<const float2*>(Gs + c0);
            const float wa = gp.x * f_a, wb = gp.y * f_b, wc = Gs[c0 + single_at] * f_c;
#pragma unroll
            for (int j = 0; j < 9; ++j) {
                const float* pl = cs + j * kPlane + c0;
                const float2 pr = *reinterpret_cast<const float2*>(pl);
                out[j] = pr.x * wa + pr.y * wb + pl[single_at] * wc;
            }
        };
        hsum(0, h[1]);
        hsum(1, h[2]);
#pragma unroll
        for (int k = 0; k < kPixPerThread; ++k) {
#pragma unroll
            for (int j = 0; j < 9; ++j) { h[0][j] = h[1][j]; h[1][j] = h[2][j]; }
            hsum(k + 2, h[2]);
            const int gy = y0 + ty0 + k;
            const bool own = gx < W && gy < H;
            const bool dup_u = (gy == 1), dup_d = (gy == H - 2);
            float V[9];
#pragma unroll
            for (int j = 0; j < 9; ++j) {
                float s = (h[0][j] + h[1][j]) + h[2][j];
                if (dup_u) s += h[0][j];
                if (dup_d) s += h[2][j];
                V[j] = s;
            }
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                // d/dw of the SSIM terms around this pixel: V0 + 2 w V1 + t V2  (t = target)
                const float t = own ? __ldg(c.tgt + (ch * c.tgt_sc + gy * W + gx)) : 0.f;
                pq[k][2 * ch] = V[3 * ch] + t * V[3 * ch + 2];
                pq[k][2 * ch + 1] = 2.0f * V[3 * ch + 1];
            }
        }
        __syncthreads();                                    // every neighbour has read the coefficients
#pragma unroll
        for (int k = 0; k < kPixPerThread; ++k)
#pragma unroll
            for (int j = 0; j < 6; ++j) cs[j * kPlane + pcell(tx, ty0 + k)] = pq[k][j];
#pragma unroll
        for (int k = 0; k < kPixPerThread; ++k) cs[6 * kPlane + pcell(tx, ty0 + k)] = dep_own[k];
    }

    // ---- phase D, one own pixel at a time: L1 / depth adjoints and the geometry adjoint ----
    float acc[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) acc[i] = 0.f;
#pragma unroll kBwdDUnroll
    for (int k = 0; k < kPixPerThread; ++k) {
        const int gy = y0 + ty0 + k;
        if (gx < W && gy < H) {
            const int pix = gy * W + gx;
            const int cell = pcell(tx, ty0 + k);
            const float dep = cs[6 * kPlane + cell], m = __ldg(mask + pix);
            const float d0 = depth_mask ? __ldg(coef + (9 * n + pix)) : 0.f;
            WarpPt p;
            warp_point<F>(cam, A, gx, gy, dep, p);
            const TapIdx ti = make_taps(p, H, W);
            const float Gd = Gs[cell];
            // d loss / d dd = c_dep * mask - Gd * diff0   (diff = diff0 * (1 - dd), losses.py:176-177)
            const float Gdd = sc.c_dep * m - Gd * d0;
            float pd = 0.f, dd = 0.f;
            Taps td;
            if (need_depth) {
                td = load_taps(c.rdep, 0, ti, W);
                pd = blend(td, ti);
                dd = depth_inconsistency(p.Z, pd);
            }
            const float G0 = depth_mask ? Gd * (1.0f - dd) : Gd;
            float g_ix = 0.f, g_iy = 0.f;
            const float gl1 = G0 * A.third * L.w_l1;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const Taps tv = load_taps(c.ref, ch * c.ref_sc, ti, W);
                const float t = __ldg(c.tgt + (ch * c.tgt_sc + pix));
                const float w = blend(tv, ti);
                const float dlt = t - w;
                float gwc = cs[(2 * ch) * kPlane + cell] + w * cs[(2 * ch + 1) * kPlane + cell];
                if (fabsf(dlt) <= 1.0f) gwc += (dlt > 0.f) ? -gl1 : ((dlt < 0.f) ? gl1 : 0.f);
                bilinear_grad(tv, p, gwc, g_ix, g_iy);
            }
            float g_Z = 0.f, g_pd = 0.f;
            if (need_depth && Gdd != 0.f) {
                depth_inconsistency_adjoint(p.Z, pd, Gdd, g_Z, g_pd);
                bilinear_grad(td, p, g_pd, g_ix, g_iy);
                if (g.g_ref_depth && g_pd != 0.f) scatter_taps(g.g_ref_depth + (int64_t)b * n, 0, ti, g_pd, W);
            }
            const GeomGrad gg = geom_adjoint(cam, A, p, g_ix, g_iy, g_Z);
            if (g.g_tgt_depth) {
                if (shared_grads) atomicAdd(g.g_tgt_depth + (int64_t)b * n + pix, gg.g_depth);
                else g.g_tgt_depth[(int64_t)b * n + pix] = gg.g_depth;
            }
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                acc[i * 4 + 0] += gg.gp[i] * p.cam[0];
                acc[i * 4 + 1] += gg.gp[i] * p.cam[1];
                acc[i * 4 + 2] += gg.gp[i] * p.cam[2];
                acc[i * 4 + 3] += gg.gp[i];
            }
        }
    }
    __syncthreads();                                   // phase D is over everywhere: the tile doubles as reduction scratch
    if (g.g_proj) block_atomic_accumulate<12>(acc, cs, g.g_proj + b * 12, threadIdx.x, kTileThreads);
}

// ---------------------------------------------------------------------------
// exact re-evaluation of single pixels (the near-ties of the min-reprojection under the "fast" arithmetic)
// ---------------------------------------------------------------------------
// diff_img of single pixels exactly as pair_fwd_kernel computes it (every rounding step of eager PyTorch): the 3x3
// window of (target, warped) per channel, avg_pool2d-ordered statistics, IEEE SSIM ratio, L1 blend, channel mean,
// depth-consistency weight.  Sixteen lanes share one (near-tie pixel, competing group) task: lanes 0..8 warp one window
// position each (one round of dependent gathers instead of nine), then every lane accumulates the window in
// avg_pool2d's row-major order from the shuffled values and lane 0 overwrites the group's diff_img entry.

// One (pixel, group) task on the 16 lanes [seg, seg + 16) of a warp; every lane of the warp must call it (full-mask
// shuffles), dead tasks (live = false) compute on pixel 0 and write nothing.
template <int F>
__device__ __forceinline__ void resolve_tie(const PairLaunch& L, int j, int pix, int sub, bool live) {
    const Arith& A = L.A;
    const int H = A.H, W = A.W, n = H * W;
    const int b = pix / n, r = pix - b * n;
    const int y = r / W, x = r - y * W;
    const tcsfm_pair_group& g = L.g[j];
    const Cam cam = load_cam(g.kinv, g.proj, b);
    const PairCtx c = make_ctx(g, b, n);
    const bool need_depth = (L.flags & TCSFM_DEPTH_MASK) != 0;
    const int i = sub < 9 ? sub : 4;                       // this lane's window position (idle lanes redo the centre)
    const int ry = reflect1(y + i / 3 - 1, H), rx = reflect1(x + i % 3 - 1, W);
    WarpPt p;
    warp_point<F>(cam, A, rx, ry, __ldg(c.tdep + (ry * W + rx)), p);
    const TapIdx ti = make_taps(p, H, W);
    float t[3], w[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        w[ch] = blend(load_taps(c.ref, ch * c.ref_sc, ti, W), ti);
        t[ch] = __ldg(c.tgt + (ch * c.tgt_sc + ry * W + rx));
    }
    float dd = need_depth ? depth_inconsistency(p.Z, blend(load_taps(c.rdep, 0, ti, W), ti)) : 0.f;
    const int seg = threadIdx.x & 16;                      // first lane of this task inside the warp
    dd = __shfl_sync(0xffffffffu, dd, seg + 4);
    float esum = 0.f;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;        // like ssim_stats: row-major from zero
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            const float tk = __shfl_sync(0xffffffffu, t[ch], seg + k), wk = __shfl_sync(0xffffffffu, w[ch], seg + k);
            sx = __fadd_rn(sx, tk);
            sy = __fadd_rn(sy, wk);
            sxx = __fadd_rn(sxx, __fmul_rn(tk, tk));
            syy = __fadd_rn(syy, __fmul_rn(wk, wk));
            sxy = __fadd_rn(sxy, __fmul_rn(tk, wk));
        }
        const float tc = __shfl_sync(0xffffffffu, t[ch], seg + 4), wc = __shfl_sync(0xffffffffu, w[ch], seg + 4);
        SsimStats s;
        s.mu_x = div9_exact(sx);
        s.mu_y = div9_exact(sy);
        s.sig_x = __fsub_rn(div9_exact(sxx), __fmul_rn(s.mu_x, s.mu_x));
        s.sig_y = __fsub_rn(div9_exact(syy), __fmul_rn(s.mu_y, s.mu_y));
        s.sig_xy = __fsub_rn(div9_exact(sxy), __fmul_rn(s.mu_x, s.mu_y));
        const SsimTerms tt = ssim_terms(s, L.C1, L.C2);
        const float l1 = clamp01_nan(fabsf(__fsub_rn(tc, wc)));
        const float ev = __fadd_rn(__fmul_rn(l1, L.w_l1), __fmul_rn(clamp01_nan(tt.raw), L.w_ssim));
        esum = (ch == 0) ? ev : __fadd_rn(esum, ev);
    }
    const float diff0 = mean3_of_sum<F>(esum, A);
    if (live && sub == 0) g.diff_img[pix] = need_depth ? __fmul_rn(diff0, __fsub_rn(1.0f, dd)) : diff0;
}

// Per-pixel min over the competing forward groups (losses.py:129-132) and the exact re-evaluation of its near-ties in
// ONE launch: a block takes the min of its 2048 pixels (sum -> out_sum), collects the pixels whose two best
// candidates are closer than `band` (or involve a NaN) in shared memory and then re-evaluates exactly those with
// the exact arithmetic, sixteen lanes per (pixel, group), overwriting the groups' diff_img entries before any
// backward pass reads the routing.  The sum is the one of the values as the forward produced them.
constexpr int kMinResolveThreads = 256, kMinResolvePix = 8;      // 2048 pixels per block: config 2 is one wave of 480 blocks

template <int F>
__global__ void __launch_bounds__(kMinResolveThreads)
min_resolve_kernel(const __grid_constant__ PairLaunch L, int n_groups, int64_t n_total, float band,
                   float* __restrict__ out_sum, int* __restrict__ tie_count, FrameFinalize fin) {
    TCSFM_SHARED float red[kMinResolveThreads / 32];
    TCSFM_SHARED int buf[kMinResolveThreads * kMinResolvePix];
    TCSFM_SHARED int n_buf;
    if (threadIdx.x == 0) n_buf = 0;
    __syncthreads();
    // every load of a candidate map is in flight before the first comparison (a thread's eight pixels per map)
    float part[1] = {0.f};
    // Pixels are dealt to the blocks in 32-pixel segments, round robin: near-ties come in runs (image borders, rows
    // that leave the view), and a block that owned such a run alone re-evaluated thousands of them one round of sixteen
    // at a time while the rest of the grid idled (measured: 267 us instead of 13 at 376x1242).
    const int64_t lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    constexpr int kWarps = kMinResolveThreads / 32;
    auto pixel = [&](int k) { return (((int64_t)k * kWarps + wrp) * gridDim.x + blockIdx.x) * 32 + lane; };
    float m[kMinResolvePix], second[kMinResolvePix];
    bool odd[kMinResolvePix];
    {
        const float* first = L.g[0].diff_img;
#pragma unroll
        for (int k = 0; k < kMinResolvePix; ++k) {
            const int64_t i = pixel(k);
            m[k] = i < n_total ? __ldg(first + i) : 0.f;
            second[k] = INFINITY;
        }
#pragma unroll
        for (int k = 0; k < kMinResolvePix; ++k) odd[k] = m[k] != m[k];
    }
    for (int j = 1; j < n_groups; ++j) {
        const float* cand = L.g[j].diff_img;
        float v[kMinResolvePix];
#pragma unroll
        for (int k = 0; k < kMinResolvePix; ++k) {
            const int64_t i = pixel(k);
            v[k] = i < n_total ? __ldg(cand + i) : INFINITY;
        }
#pragma unroll
        for (int k = 0; k < kMinResolvePix; ++k) {
            odd[k] = odd[k] || v[k] != v[k];
            if (v[k] < m[k]) { second[k] = m[k]; m[k] = v[k]; }
            else if (v[k] < second[k]) second[k] = v[k];
        }
    }
#pragma unroll
    for (int k = 0; k < kMinResolvePix; ++k) {
        const int64_t i = pixel(k);
        if (i < n_total) {
            part[0] += m[k];
            if (n_groups > 1 && (odd[k] || !(second[k] - m[k] >= band))) buf[atomicAdd(&n_buf, 1)] = (int)i;
        }
    }
    __syncthreads();
    const int ties = n_buf;
    if (threadIdx.x == 0 && ties) atomicAdd(tie_count, ties);
    const int n_tasks = ties * n_groups, sub = threadIdx.x & 15;
    for (int t0 = 0; t0 < n_tasks; t0 += kMinResolveThreads / 16) {
        if (t0 + (threadIdx.x >> 5) * 2 >= n_tasks) continue;      // both tasks of this warp are past the end (warp-uniform)
        const int task = t0 + (threadIdx.x >> 4);
        const bool live = task < n_tasks;
        const int e = live ? task / n_groups : 0, j = live ? task - e * n_groups : 0;
        resolve_tie<F>(L, j, live ? buf[e] : 0, sub, live);
    }
    block_atomic_accumulate<1>(part, red, out_sum, threadIdx.x, kMinResolveThreads);
    finalize_by_last_block(fin, out_sum);          // (optional) the loss terms, by the last block to arrive
}

#ifndef TCSFM_HOST_EMU
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        if (getenv("TCSFM_NO_TMA")) return nullptr;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
    }
    return fn;
}
// The workspace of one group as a rank-4 fp32 tensor [B][10][H][W] with a 68 x 18 x 9 x 1 box; out-of-bounds elements
// (the halo outside the image) are filled with zeros.
static bool encode_coef_map(CUtensorMap* map, const float* coef, int B, int H, int W) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc || W % 4 != 0 || reinterpret_cast<uintptr_t>(coef) % 16 != 0) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)kCoefPlanes, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)kCoefPlanes * H * W * 4};
    const cuuint32_t box[4] = {(cuuint32_t)TmaTile::kBoxW, (cuuint32_t)TmaTile::kBoxH, (cuuint32_t)TmaTile::kPlanes, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(coef), dims, strides, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
#endif

static int fill_launch(PairLaunch& L, const tcsfm_pair_group* groups, int n, int B, int H, int W,
                       float w_l1, float w_ssim, int flags, const char* who, bool bwd) {
    if (B <= 0 || H < 2 || W < 2) { set_error("%s: bad shape B=%d H=%d W=%d", who, B, H, W); return 1; }
    if (B > 65535) { set_error("%s: B=%d exceeds 65535", who, B); return 1; }
    if ((int64_t)H * W * kCoefPlanes >= (int64_t)1 << 31) { set_error("%s: image too large", who); return 1; }
    if (!(flags & TCSFM_SSIM)) { set_error("%s: the fused pair loss requires TCSFM_SSIM (l_ssim)", who); return 1; }
    const bool need_depth = (flags & (TCSFM_DEPTH_MASK | TCSFM_DEPTH_CONSIST)) != 0;
    for (int i = 0; i < n; ++i) {
        const tcsfm_pair_group& g = groups[i];
        if (!g.tgt_img || !g.ref_img || !g.tgt_depth || !g.kinv || !g.proj || !g.sums) {
            set_error("%s: group %d has a null input pointer", who, i); return 1;
        }
        // in-kernel offsets inside one batch element are 32-bit
        const int64_t lim = ((int64_t)1 << 31) - 1 - (int64_t)H * W;
        if (g.tgt_sc < 0 || g.ref_sc < 0 || 2 * g.tgt_sc > lim || 2 * g.ref_sc > lim) {
            set_error("%s: group %d: channel stride out of range", who, i); return 1;
        }
        if (need_depth && !g.ref_depth) { set_error("%s: group %d needs ref_depth for the depth terms", who, i); return 1; }
        if (bwd && (!g.mask || !g.coef)) { set_error("%s: group %d: backward needs the forward's mask and coef workspace", who, i); return 1; }
        L.g[i] = g;
    }
    L.A = make_arith(H, W, flags);
    L.w_l1 = w_l1; L.w_ssim = w_ssim;
    L.C1 = kSsimC1; L.C2 = kSsimC2;
    L.flags = flags;
    return 0;
}

}  // namespace tcsfm

using namespace tcsfm;

extern "C" int tcsfm_pair_coef_planes(void) { return kCoefPlanes; }

// the tolerance-level SSIM arithmetic: csrc/pair_fast_kernels.cu
int tcsfm_pair_fast_fwd(const tcsfm_pair_group* groups, int n_groups, int B, int H, int W,
                        float w_l1, float w_ssim, int flags, void* stream);

extern "C" int tcsfm_pair_loss_fwd(const tcsfm_pair_group* groups, int n_groups, int B, int H, int W,
                                   float w_l1, float w_ssim, int flags, void* stream) {
    if (!groups || n_groups <= 0) { set_error("tcsfm_pair_loss_fwd: no groups"); return 1; }
    if (flags & TCSFM_ARITH_FAST) return tcsfm_pair_fast_fwd(groups, n_groups, B, H, W, w_l1, w_ssim, flags, stream);
    const size_t smem = 3 * Tile<1>::kCells * sizeof(float2);
    const int tiles = tile_count(H, W);
    for (int base = 0; base < n_groups; base += kMaxGroups) {
        const int n = (n_groups - base < kMaxGroups) ? n_groups - base : kMaxGroups;
        PairLaunch L;
        memset(&L, 0, sizeof(L));
        if (int rc = fill_launch(L, groups + base, n, B, H, W, w_l1, w_ssim, flags, "tcsfm_pair_loss_fwd", false)) return rc;
        // zero the accumulated sums; groups whose buffers are adjacent share one memset
        for (int i = 0; i < n;) {
            int j = i + 1;
            while (j < n && L.g[j].sums == L.g[j - 1].sums + 4) ++j;
            cudaMemsetAsync(L.g[i].sums, 0, (size_t)(j - i) * 4 * sizeof(float), (cudaStream_t)stream);
            i = j;
        }
        dim3 grid(tiles, B, n), block(kTileThreads);
        TCSFM_DISPATCH_FLAVOUR(flags, TCSFM_LAUNCH(pair_fwd_kernel<F>, grid, block, smem, stream, L));
        if (int rc = check_launch("tcsfm_pair_loss_fwd")) return rc;
    }
    return 0;
}

extern "C" int tcsfm_pair_loss_bwd(const tcsfm_pair_group* groups, int n_groups, int B, int H, int W,
                                   float w_l1, float w_ssim, int flags, void* stream) {
    if (!groups || n_groups <= 0) { set_error("tcsfm_pair_loss_bwd: no groups"); return 1; }
    const size_t smem = kBwdSmemBytes;
    const int tiles = tile_count(H, W);
    for (int base = 0; base < n_groups; base += kMaxGroups) {
        const int n = (n_groups - base < kMaxGroups) ? n_groups - base : kMaxGroups;
        PairLaunch L;
        memset(&L, 0, sizeof(L));
        if (int rc = fill_launch(L, groups + base, n, B, H, W, w_l1, w_ssim, flags, "tcsfm_pair_loss_bwd", true)) return rc;
        for (int i = 0; i < n; ++i) {
            if (L.g[i].min_base && (!L.g[i].g_min || L.g[i].min_count < 1 || L.g[i].min_index >= L.g[i].min_count)) {
                set_error("tcsfm_pair_loss_bwd: group %d: inconsistent min-reprojection fields", base + i); return 1;
            }
            if (L.g[i].g_ref_depth && !(flags & TCSFM_SHARED_GRADS)) cudaMemsetAsync(L.g[i].g_ref_depth, 0, (size_t)B * H * W * sizeof(float), (cudaStream_t)stream);
        }
        for (int i = 0; i < n;) {                     // adjacent g_proj buffers share one memset
            if (!L.g[i].g_proj) { ++i; continue; }
            int j = i + 1;
            while (j < n && L.g[j].g_proj == L.g[j - 1].g_proj + (size_t)B * 12) ++j;
            cudaMemsetAsync(L.g[i].g_proj, 0, (size_t)(j - i) * B * 12 * sizeof(float), (cudaStream_t)stream);
            i = j;
        }
        // 16-byte staging needs every row start of the planes it reads aligned
        auto aligned16 = [](const void* ptr) { return reinterpret_cast<uintptr_t>(ptr) % 16 == 0; };
        L.vec16 = (W % 4 == 0);
        for (int i = 0; i < n; ++i)
            L.vec16 = L.vec16 && aligned16(L.g[i].coef) && aligned16(L.g[i].mask) && aligned16(L.g[i].g_diff) &&
                      aligned16(L.g[i].min_base) && L.g[i].min_stride % 4 == 0;
        dim3 grid(tiles, B, n), block(kTileThreads);
        bool tma = false;
#ifndef TCSFM_HOST_EMU
        // TMA staging of the coefficient planes when every group's workspace can be described by a tensor map
        // (16-byte aligned rows); otherwise the cp.async staging
        tma = L.vec16 != 0;
        for (int i = 0; i < n && tma; ++i) tma = encode_coef_map(&L.coef_map[i], L.g[i].coef, B, H, W);
        if (tma) {
            cudaError_t e = cudaSuccess;
            TCSFM_DISPATCH_FLAVOUR(flags, e = cudaFuncSetAttribute(pair_bwd_kernel<F, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdTmaSmemBytes));
            if (e != cudaSuccess) { set_error("tcsfm_pair_loss_bwd: cannot raise dynamic smem: %s", cudaGetErrorString(e)); return 2; }
            TCSFM_DISPATCH_FLAVOUR(flags, TCSFM_LAUNCH((pair_bwd_kernel<F, true>), grid, block, kBwdTmaSmemBytes, stream, L));
        }
#endif
        if (!tma) { TCSFM_DISPATCH_FLAVOUR(flags, TCSFM_LAUNCH((pair_bwd_kernel<F, false>), grid, block, smem, stream, L)); }
        if (int rc = check_launch("tcsfm_pair_loss_bwd")) return rc;
    }
    return 0;
}

/* Per-pixel min over the groups' diff_img and the exact re-evaluation of its near-ties (+ tcsfm_frame_finalize when
 * `cfg` is given) as one launch: out_sum [1] = the sum over the B*H*W pixels of that min, counters [2] = (number of
 * pixels re-evaluated, scratch ticket). */
extern "C" int tcsfm_pair_min_resolve(const tcsfm_pair_group* groups, int n_groups, int B, int H, int W,
                                      float w_l1, float w_ssim, int flags, float band, float* out_sum, int* counters,
                                      const float* sums, const tcsfm_frame_cfg* cfg, float* out_terms, float* out_total,
                                      void* stream) {
    if (!groups || n_groups <= 0 || n_groups > kMaxGroups) { set_error("tcsfm_pair_min_resolve: 1..%d groups", kMaxGroups); return 1; }
    if (!out_sum || !counters) { set_error("tcsfm_pair_min_resolve: null output"); return 1; }
    if (cfg && (!sums || !out_terms || cfg->n_groups <= 0 || cfg->n_groups > 8)) { set_error("tcsfm_pair_min_resolve: bad finalize arguments"); return 1; }
    PairLaunch L;
    memset(&L, 0, sizeof(L));
    if (int rc = fill_launch(L, groups, n_groups, B, H, W, w_l1, w_ssim, flags & ~TCSFM_ARITH_FAST, "tcsfm_pair_min_resolve", false)) return rc;
    for (int i = 0; i < n_groups; ++i)
        if (!L.g[i].diff_img) { set_error("tcsfm_pair_min_resolve: group %d has no diff_img", i); return 1; }
    const int64_t n_total = (int64_t)B * H * W;
    if (n_total >= ((int64_t)1 << 31)) { set_error("tcsfm_pair_min_resolve: more than 2^31 pixels"); return 1; }
    cudaMemsetAsync(out_sum, 0, sizeof(float), (cudaStream_t)stream);
    cudaMemsetAsync(counters, 0, 2 * sizeof(int), (cudaStream_t)stream);
    FrameFinalize fin;
    memset(&fin, 0, sizeof(fin));
    if (cfg) { fin.sums = sums; fin.cfg = *cfg; fin.out = out_terms; fin.total = out_total; fin.ticket = counters + 1; }
    const int per_block = kMinResolveThreads * kMinResolvePix;
    dim3 grid((unsigned)((n_total + per_block - 1) / per_block)), block(kMinResolveThreads);
    TCSFM_DISPATCH_FLAVOUR(flags, TCSFM_LAUNCH(min_resolve_kernel<F>, grid, block, 0, stream, L, n_groups, n_total, band, out_sum, counters, fin));
    return check_launch("tcsfm_pair_min_resolve");
}
