// SSIM_Loss.forward (reference losses.py:27-41) and its backward as shared-memory
// stencils.  A CTA of 256 threads owns a 64x16 output tile of one [H,W] plane,
// stages the reflect-padded x / y tiles (+1 halo forward, +2 halo backward) in
// shared memory with coalesced row loads, and each thread produces 4 pixels.
#include "tile.cuh"

namespace tcsfm {

// kMean: instead of the map, accumulate mean(map) into out[0] (`scale` = 1 / element count): the
// `.mean()` that follows SSIM_Loss in the PFT depth-initialisation term (optimizer.py:89-90)
template <bool kMean>
__global__ void __launch_bounds__(kTileThreads)
ssim_fwd_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ out,
                int H, int W, float C1, float C2, float scale) {
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float, smem);
    TCSFM_SHARED float red[kTileThreads / 32];
    float* xs = smem;
    float* ys = smem + T1::kCells;
    const int x0 = blockIdx.x * kTileW, y0 = blockIdx.y * kTileH;
    const int64_t plane = (int64_t)blockIdx.z * H * W;
    for (int cell = threadIdx.x; cell < T1::kCells; cell += kTileThreads) {
        int ry, rx;
        const bool ok = T1::cell_to_reflected(cell, x0, y0, H, W, ry, rx);
        xs[cell] = ok ? __ldg(x + plane + (int64_t)ry * W + rx) : 0.f;
        ys[cell] = ok ? __ldg(y + plane + (int64_t)ry * W + rx) : 0.f;
    }
    __syncthreads();
    float part[1] = {0.f};
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        int tx, ty;
        own_pixel(threadIdx.x, k, tx, ty);
        const int gx = x0 + tx, gy = y0 + ty;
        if (gx < W && gy < H) {
            const int c = T1::cell(tx, ty);
            const float v = ssim_value(xs + c, ys + c, T1::kPitch, C1, C2);
            if (kMean) part[0] += v * scale;
            else out[plane + (int64_t)gy * W + gx] = v;
        }
    }
    if (kMean) block_atomic_accumulate<1>(part, red, out, threadIdx.x, kTileThreads);
}

__global__ void __launch_bounds__(kTileThreads)
ssim_bwd_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ g_out,
                const float* __restrict__ g_mean, float scale,
                float* __restrict__ g_x, float* __restrict__ g_y, int H, int W, float C1, float C2) {
    using T2 = Tile<2>;
    using T1 = Tile<1>;
    TCSFM_DYN_SMEM(float, smem);
    float* xs = smem;
    float* ys = xs + T2::kCells;
    float* cAx = ys + T2::kCells;
    float* cAy = cAx + T1::kCells;
    float* cB = cAy + T1::kCells;
    float* cC = cB + T1::kCells;
    const int x0 = blockIdx.x * kTileW, y0 = blockIdx.y * kTileH;
    const int64_t plane = (int64_t)blockIdx.z * H * W;
    for (int cell = threadIdx.x; cell < T2::kCells; cell += kTileThreads) {
        int ry, rx;
        const bool ok = T2::cell_to_reflected(cell, x0, y0, H, W, ry, rx);
        xs[cell] = ok ? __ldg(x + plane + (int64_t)ry * W + rx) : 0.f;
        ys[cell] = ok ? __ldg(y + plane + (int64_t)ry * W + rx) : 0.f;
    }
    __syncthreads();
    // adjoint coefficients of every output pixel q in the +1 ring (zero outside the image)
    for (int cell = threadIdx.x; cell < T1::kCells; cell += kTileThreads) {
        int cx, cy;
        T1::cell_xy(cell, cx, cy);
        const int gx = x0 + cx, gy = y0 + cy;
        SsimCoef k;
        k.Ax = k.Ay = k.B = k.Cc = 0.f;
        if (gx >= 0 && gx < W && gy >= 0 && gy < H) {
            // upstream: a per-pixel map, or the gradient of the map's mean (one device scalar / count)
            const float g = g_out ? __ldg(g_out + plane + (int64_t)gy * W + gx) : __ldg(g_mean) * scale;
            const int c2 = T2::cell(cx, cy);
            const SsimStats s = ssim_stats(xs + c2, ys + c2, T2::kPitch);
            k = ssim_coef(s, ssim_terms(s, C1, C2), g);
        }
        cAx[cell] = k.Ax; cAy[cell] = k.Ay; cB[cell] = k.B; cC[cell] = k.Cc;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
        int tx, ty;
        own_pixel(threadIdx.x, k, tx, ty);
        const int gx = x0 + tx, gy = y0 + ty;
        if (gx < W && gy < H) {
            float sAx = 0.f, sAy = 0.f, sB = 0.f, sC = 0.f;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy) {
                const int my = reflect_mult(gy + dy, gy, H);
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) {
                    const float m = (float)(my * reflect_mult(gx + dx, gx, W));
                    const int c1 = T1::cell(tx + dx, ty + dy);
                    sAx += m * cAx[c1]; sAy += m * cAy[c1]; sB += m * cB[c1]; sC += m * cC[c1];
                }
            }
            const int c2 = T2::cell(tx, ty);
            const float xp = xs[c2], yp = ys[c2];
            const int64_t o = plane + (int64_t)gy * W + gx;
            if (g_x) g_x[o] = sAx + 2.0f * xp * sB + yp * sC;
            if (g_y) g_y[o] = sAy + 2.0f * yp * sB + xp * sC;
        }
    }
}

}  // namespace tcsfm

using namespace tcsfm;

extern "C" int tcsfm_ssim_fwd(const float* x, const float* y, float* out, int N, int H, int W, int flags, void* stream) {
    (void)flags;
    if (N <= 0 || H < 2 || W < 2) { set_error("tcsfm_ssim_fwd: bad shape N=%d H=%d W=%d", N, H, W); return 1; }
    if (!x || !y || !out) { set_error("tcsfm_ssim_fwd: null pointer"); return 1; }
    if (N > 65535) { set_error("tcsfm_ssim_fwd: N=%d exceeds 65535 planes", N); return 1; }
    dim3 grid(tiles_x(W), tiles_y(H), N), block(kTileThreads);
    const size_t smem = 2 * Tile<1>::kCells * sizeof(float);
    TCSFM_LAUNCH(ssim_fwd_kernel<false>, grid, block, smem, stream, x, y, out, H, W, kSsimC1, kSsimC2, 0.f);
    return check_launch("tcsfm_ssim_fwd");
}

extern "C" int tcsfm_ssim_mean_fwd(const float* x, const float* y, float* out_mean, int N, int H, int W, int flags, void* stream) {
    (void)flags;
    if (N <= 0 || H < 2 || W < 2) { set_error("tcsfm_ssim_mean_fwd: bad shape N=%d H=%d W=%d", N, H, W); return 1; }
    if (!x || !y || !out_mean) { set_error("tcsfm_ssim_mean_fwd: null pointer"); return 1; }
    if (N > 65535) { set_error("tcsfm_ssim_mean_fwd: N=%d exceeds 65535 planes", N); return 1; }
    dim3 grid(tiles_x(W), tiles_y(H), N), block(kTileThreads);
    const size_t smem = 2 * Tile<1>::kCells * sizeof(float);
    cudaMemsetAsync(out_mean, 0, sizeof(float), (cudaStream_t)stream);
    const float scale = (float)(1.0 / ((double)N * H * W));
    TCSFM_LAUNCH(ssim_fwd_kernel<true>, grid, block, smem, stream, x, y, out_mean, H, W, kSsimC1, kSsimC2, scale);
    return check_launch("tcsfm_ssim_mean_fwd");
}

extern "C" int tcsfm_ssim_bwd(const float* x, const float* y, const float* g_out, float* g_x, float* g_y,
                              int N, int H, int W, int flags, void* stream) {
    (void)flags;
    if (N <= 0 || H < 2 || W < 2) { set_error("tcsfm_ssim_bwd: bad shape N=%d H=%d W=%d", N, H, W); return 1; }
    if (!x || !y || !g_out) { set_error("tcsfm_ssim_bwd: null pointer"); return 1; }
    if (N > 65535) { set_error("tcsfm_ssim_bwd: N=%d exceeds 65535 planes", N); return 1; }
    dim3 grid(tiles_x(W), tiles_y(H), N), block(kTileThreads);
    const size_t smem = (2 * Tile<2>::kCells + 4 * Tile<1>::kCells) * sizeof(float);
    TCSFM_LAUNCH(ssim_bwd_kernel, grid, block, smem, stream, x, y, g_out, (const float*)nullptr, 0.f, g_x, g_y, H, W, kSsimC1, kSsimC2);
    return check_launch("tcsfm_ssim_bwd");
}

extern "C" int tcsfm_ssim_mean_bwd(const float* x, const float* y, const float* g_mean, float* g_x, float* g_y,
                                   int N, int H, int W, int flags, void* stream) {
    (void)flags;
    if (N <= 0 || H < 2 || W < 2) { set_error("tcsfm_ssim_mean_bwd: bad shape N=%d H=%d W=%d", N, H, W); return 1; }
    if (!x || !y || !g_mean) { set_error("tcsfm_ssim_mean_bwd: null pointer"); return 1; }
    if (N > 65535) { set_error("tcsfm_ssim_mean_bwd: N=%d exceeds 65535 planes", N); return 1; }
    dim3 grid(tiles_x(W), tiles_y(H), N), block(kTileThreads);
    const size_t smem = (2 * Tile<2>::kCells + 4 * Tile<1>::kCells) * sizeof(float);
    const float scale = (float)(1.0 / ((double)N * H * W));
    TCSFM_LAUNCH(ssim_bwd_kernel, grid, block, smem, stream, x, y, (const float*)nullptr, g_mean, scale, g_x, g_y, H, W, kSsimC1, kSsimC2);
    return check_launch("tcsfm_ssim_mean_bwd");
}
