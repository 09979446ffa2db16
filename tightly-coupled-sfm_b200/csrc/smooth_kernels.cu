// get_smooth_loss (reference losses.py:43-61): edge-aware smoothness of the mean-normalised
// disparity, forward and backward, as four small kernels instead of ~45 eager launches.
//
//   m_b   = mean over the image of disp[b]                       (mean(2).mean(3))
//   n     = disp / (m_b + 1e-7)
//   loss  = mean_{x<W-1} |n(x) - n(x+1)| * exp(-mean_c |I(x) - I(x+1)|)
//         + mean_{y<H-1} |n(y) - n(y+1)| * exp(-mean_c |I(y) - I(y+1)|)
//
// The value is a reduction (no masks depend on it), so sums use block reductions + atomics.
#include "tcsfm_math.cuh"

namespace tcsfm {

constexpr int kSmoothThreads = 256;

// sums[b] = sum over the image of disp[b]
__global__ void __launch_bounds__(kSmoothThreads)
smooth_mean_kernel(const float* __restrict__ disp, int n, float* __restrict__ sums) {
    TCSFM_SHARED float red[kSmoothThreads / 32];
    const int b = blockIdx.y;
    float part[1] = {0.f};
    for (int i = blockIdx.x * kSmoothThreads + threadIdx.x; i < n; i += gridDim.x * kSmoothThreads)
        part[0] += __ldg(disp + (int64_t)b * n + i);
    block_atomic_accumulate<1>(part, red, sums + b, threadIdx.x, kSmoothThreads);
}

__device__ __forceinline__ float edge_weight(const float* __restrict__ img, int64_t sc, int p, int q) {
    float s = 0.f;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) s += fabsf(__ldg(img + ch * sc + p) - __ldg(img + ch * sc + q));
    return expf(-s * (1.0f / 3.0f));
}

// acc[0] += sum |n(x)-n(x+1)| w_x,  acc[1] += sum |n(y)-n(y+1)| w_y
__global__ void __launch_bounds__(kSmoothThreads)
smooth_fwd_kernel(const float* __restrict__ disp, const float* __restrict__ img, int64_t img_sb, int64_t img_sc,
                  const float* __restrict__ sums, int H, int W, float* __restrict__ acc) {
    TCSFM_SHARED float red[2 * (kSmoothThreads / 32)];
    const int b = blockIdx.y, n = H * W;
    const float inv = 1.0f / (__ldg(sums + b) / (float)n + 1e-7f);
    const float* d = disp + (int64_t)b * n;
    const float* im = img + b * img_sb;
    float part[2] = {0.f, 0.f};
    for (int p = blockIdx.x * kSmoothThreads + threadIdx.x; p < n; p += gridDim.x * kSmoothThreads) {
        const int y = p / W, x = p - y * W;
        const float c = __fmul_rn(__ldg(d + p), inv);
        if (x + 1 < W) part[0] += fabsf(c - __fmul_rn(__ldg(d + p + 1), inv)) * edge_weight(im, img_sc, p, p + 1);
        if (y + 1 < H) part[1] += fabsf(c - __fmul_rn(__ldg(d + p + W), inv)) * edge_weight(im, img_sc, p, p + W);
    }
    block_atomic_accumulate<2>(part, red, acc, threadIdx.x, kSmoothThreads);
}

__device__ __forceinline__ float sgn(float a) { return (a > 0.f) ? 1.f : ((a < 0.f) ? -1.f : 0.f); }

// g_norm[p] = d loss / d n[p]  (scaled by the upstream gradient), dots[b] += sum_p g_norm[p] * disp[p]
__global__ void __launch_bounds__(kSmoothThreads)
smooth_bwd_kernel(const float* __restrict__ disp, const float* __restrict__ img, int64_t img_sb, int64_t img_sc,
                  const float* __restrict__ sums, const float* __restrict__ g_out, int H, int W, float cx, float cy,
                  float* __restrict__ g_norm, float* __restrict__ dots) {
    TCSFM_SHARED float red[kSmoothThreads / 32];
    const int b = blockIdx.y, n = H * W;
    const float inv = 1.0f / (__ldg(sums + b) / (float)n + 1e-7f);
    const float go = __ldg(g_out);
    const float gx = go * cx, gy = go * cy;              // 1 / (B*H*(W-1)), 1 / (B*(H-1)*W)
    const float* d = disp + (int64_t)b * n;
    const float* im = img + b * img_sb;
    float part[1] = {0.f};
    for (int p = blockIdx.x * kSmoothThreads + threadIdx.x; p < n; p += gridDim.x * kSmoothThreads) {
        const int y = p / W, x = p - y * W;
        const float dc = __ldg(d + p);
        // every normalised value rounded on its own (__fmul_rn: no FMA contraction into the difference), so equal
        // neighbours differ by exactly 0 and get no gradient, like abs at 0 in eager PyTorch
        const float c = __fmul_rn(dc, inv);
        float g = 0.f;
        if (x + 1 < W) g += gx * sgn(c - __fmul_rn(__ldg(d + p + 1), inv)) * edge_weight(im, img_sc, p, p + 1);
        if (x > 0) g -= gx * sgn(__fmul_rn(__ldg(d + p - 1), inv) - c) * edge_weight(im, img_sc, p - 1, p);
        if (y + 1 < H) g += gy * sgn(c - __fmul_rn(__ldg(d + p + W), inv)) * edge_weight(im, img_sc, p, p + W);
        if (y > 0) g -= gy * sgn(__fmul_rn(__ldg(d + p - W), inv) - c) * edge_weight(im, img_sc, p - W, p);
        g_norm[(int64_t)b * n + p] = g;
        part[0] += g * dc;
    }
    block_atomic_accumulate<1>(part, red, dots + b, threadIdx.x, kSmoothThreads);
}

// g_disp = g_norm / (m+eps) - dot_b / ((m+eps)^2 * n)      (in place on g_norm)
__global__ void __launch_bounds__(kSmoothThreads)
smooth_bwd_finish_kernel(const float* __restrict__ sums, const float* __restrict__ dots, int n, float* __restrict__ g) {
    const int b = blockIdx.y;
    const float inv = 1.0f / (__ldg(sums + b) / (float)n + 1e-7f);
    const float corr = __ldg(dots + b) * inv * inv / (float)n;
    for (int p = blockIdx.x * kSmoothThreads + threadIdx.x; p < n; p += gridDim.x * kSmoothThreads)
        g[(int64_t)b * n + p] = g[(int64_t)b * n + p] * inv - corr;
}

// loss = acc[0] / (B*H*(W-1)) + acc[1] / (B*(H-1)*W)
__global__ void smooth_finalize_kernel(const float* __restrict__ acc, float cx, float cy, float* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) out[0] = acc[0] * cx + acc[1] * cy;
}

static inline int smooth_blocks(int n) {
    int blocks = (n + kSmoothThreads * 4 - 1) / (kSmoothThreads * 4);
    return blocks < 1 ? 1 : (blocks > 592 ? 592 : blocks);
}

}  // namespace tcsfm

using namespace tcsfm;

// workspace: [2*B + 2] floats (sums[B], dots[B], acc[2]); zeroed here
extern "C" int tcsfm_smooth_fwd(const float* disp, const float* img, int64_t img_sb, int64_t img_sc,
                                float* workspace, float* out, int B, int H, int W, void* stream) {
    if (!disp || !img || !workspace || !out || B <= 0 || B > 65535 || H < 2 || W < 2) { set_error("tcsfm_smooth_fwd: bad arguments"); return 1; }
    const int n = H * W;
    cudaMemsetAsync(workspace, 0, (size_t)(2 * B + 2) * sizeof(float), (cudaStream_t)stream);
    float* sums = workspace; float* acc = workspace + 2 * B;
    dim3 grid(smooth_blocks(n), B), block(kSmoothThreads);
    TCSFM_LAUNCH(smooth_mean_kernel, grid, block, 0, stream, disp, n, sums);
    TCSFM_LAUNCH(smooth_fwd_kernel, grid, block, 0, stream, disp, img, img_sb, img_sc, sums, H, W, acc);
    const float cx = 1.0f / ((float)B * H * (W - 1)), cy = 1.0f / ((float)B * (H - 1) * W);
    TCSFM_LAUNCH(smooth_finalize_kernel, dim3(1), dim3(32), 0, stream, acc, cx, cy, out);
    return check_launch("tcsfm_smooth_fwd");
}

extern "C" int tcsfm_smooth_bwd(const float* disp, const float* img, int64_t img_sb, int64_t img_sc,
                                float* workspace, const float* g_out, float* g_disp, int B, int H, int W, void* stream) {
    if (!disp || !img || !workspace || !g_out || !g_disp || B <= 0 || B > 65535 || H < 2 || W < 2) { set_error("tcsfm_smooth_bwd: bad arguments"); return 1; }
    const int n = H * W;
    float* sums = workspace; float* dots = workspace + B;
    cudaMemsetAsync(dots, 0, (size_t)B * sizeof(float), (cudaStream_t)stream);
    dim3 grid(smooth_blocks(n), B), block(kSmoothThreads);
    const float cx = 1.0f / ((float)B * H * (W - 1)), cy = 1.0f / ((float)B * (H - 1) * W);
    TCSFM_LAUNCH(smooth_bwd_kernel, grid, block, 0, stream, disp, img, img_sb, img_sc, sums, g_out, H, W, cx, cy, g_disp, dots);
    TCSFM_LAUNCH(smooth_bwd_finish_kernel, grid, block, 0, stream, sums, dots, n, g_disp);
    return check_launch("tcsfm_smooth_bwd");
}
