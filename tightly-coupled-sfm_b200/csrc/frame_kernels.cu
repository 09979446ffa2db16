// Small kernels that replace the eager-PyTorch glue around the pair kernels inside
// Compute_Loss.forward (reference losses.py:75-140) so that a whole loss step is a
// dozen launches instead of ~200:
//
//   pose_proj_fwd/bwd   6-DoF pose -> K[R|t] (models/stn.py:81-116,143-158,262) and the
//                       chain rule back from grad(K[R|t]) to the pose;
//   min_reduce          sum over pixels of the per-pixel minimum over the source images'
//                       error maps (losses.py:129-132);
//   frame_finalize      mean_on_mask thresholds + the 0.3 / depth-consistency weights
//                       (losses.py:112-127,142-149) from the pair kernels' sums;
//   frame_bwd_prepare   the per-group upstream scalars the backward pair kernel consumes.
#include "tcsfm_math.cuh"

namespace tcsfm {

template <bool kNoFma>
__global__ void pose_proj_fwd_kernel(const float* __restrict__ pose, float sign, const float* __restrict__ K, int Bk,
                                     float* __restrict__ proj, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) pose_proj_fwd_body<kNoFma>(pose + i * 6, sign, K, Bk, proj, i);
}

__global__ void pose_proj_bwd_kernel(const float* __restrict__ pose, float sign, const float* __restrict__ K, int Bk,
                                     const float* __restrict__ g_proj, float* __restrict__ g_pose, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) pose_proj_bwd_body(pose + i * 6, sign, K, Bk, g_proj, g_pose, i);
}

// K^-1 of [B,3,3] fp32 matrices with the bits of torch.inverse / torch.linalg.inv_ex on CUDA (models/stn.py:257), which
// run cuBLAS' batched LU (getrf) and two triangular solves on the permuted identity (getrs): ten small launches.  The
// ordering of that arithmetic was identified by matching 20 000 probed inverses bit for bit (tools/probe_kinv.py,
// tools/match_kinv.py; camera intrinsics, skewed, lower-triangular and dense matrices, signs of zeros included):
//   getrf: partial pivoting on the first maximal |a| of the column; multipliers l = a * RN(1 / pivot); Schur update
//          a_ij = fma(-l_i, u_j, a_ij);
//   getrs: forward substitution y_i = fma(-l_ik, y_k, y_i); backward substitution column by column from the last
//          (x_2 first, then b_0 takes u_02 x_2 before u_01 x_1), fma updates, IEEE division by the diagonal.
// One thread per matrix; the output is row-major [B,9], which is what the warp kernels read.
__device__ __forceinline__ void intrinsics_inverse_body(const float* __restrict__ K, float* __restrict__ kinv, int b) {
    float a[3][3];
    int perm[3] = {0, 1, 2};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) a[i][j] = __ldg(K + b * 9 + i * 3 + j);
#pragma unroll
    for (int col = 0; col < 2; ++col) {
        int piv = col;
#pragma unroll
        for (int i = col + 1; i < 3; ++i)
            if (fabsf(a[i][col]) > fabsf(a[piv][col])) piv = i;
#pragma unroll
        for (int i = col + 1; i < 3; ++i)
            if (piv == i) {
#pragma unroll
                for (int j = 0; j < 3; ++j) { const float t = a[col][j]; a[col][j] = a[i][j]; a[i][j] = t; }
                const int t = perm[col]; perm[col] = perm[i]; perm[i] = t;
            }
        const float r = __frcp_rn(a[col][col]);
#pragma unroll
        for (int i = col + 1; i < 3; ++i) {
            a[i][col] = __fmul_rn(a[i][col], r);
#pragma unroll
            for (int j = col + 1; j < 3; ++j) a[i][j] = __fmaf_rn(-a[i][col], a[col][j], a[i][j]);
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {                       // column c of the inverse: solve L U x = P e_c
        float y0 = perm[0] == c ? 1.f : 0.f, y1 = perm[1] == c ? 1.f : 0.f, y2 = perm[2] == c ? 1.f : 0.f;
        y1 = __fmaf_rn(-a[1][0], y0, y1);
        y2 = __fmaf_rn(-a[2][0], y0, y2);
        y2 = __fmaf_rn(-a[2][1], y1, y2);
        const float x2 = __fdiv_rn(y2, a[2][2]);
        y1 = __fmaf_rn(-a[1][2], x2, y1);
        y0 = __fmaf_rn(-a[0][2], x2, y0);
        const float x1 = __fdiv_rn(y1, a[1][1]);
        y0 = __fmaf_rn(-a[0][1], x1, y0);
        const float x0 = __fdiv_rn(y0, a[0][0]);
        kinv[b * 9 + 0 * 3 + c] = x0;
        kinv[b * 9 + 1 * 3 + c] = x1;
        kinv[b * 9 + 2 * 3 + c] = x2;
    }
}

__global__ void intrinsics_inverse_kernel(const float* __restrict__ K, float* __restrict__ kinv, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) intrinsics_inverse_body(K, kinv, b);
}

// disp_to_depth (utils/learning_helpers.py:77-86) for up to 4 equally sized maps in one launch:
// depth = 1 / (min_disp + (max_disp - min_disp) * disp), each step rounded like the eager operators
// (mul by scalar, add scalar, reciprocal).  Backward: g_disp = -g_depth * depth^2 * (max_disp - min_disp).
struct MapPtrs { const float* in[4]; const float* aux[4]; float* out[4]; int count; };

// kVec = 4: 16-byte accesses (n % 4 == 0 and every pointer 16-byte aligned, checked by the launcher); the loads of all
// maps of a thread are in flight before the first store.
template <int kVec>
__device__ __forceinline__ void disp_to_depth_fwd_body(const MapPtrs& M, int64_t n, float min_disp, float range, int block) {
    const int64_t i = ((int64_t)block * 256 + threadIdx.x) * kVec;
    if (i >= n) return;
    float v[4][kVec];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < M.count) {
            if (kVec == 4) {
                const float4 q = __ldg(reinterpret_cast<const float4*>(M.in[k] + i));
                v[k][0] = q.x; v[k][1 % kVec] = q.y; v[k][2 % kVec] = q.z; v[k][3 % kVec] = q.w;
            } else {
                v[k][0] = __ldg(M.in[k] + i);
            }
        }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < M.count) {
#pragma unroll
            for (int j = 0; j < kVec; ++j) v[k][j] = __frcp_rn(__fadd_rn(__fmul_rn(v[k][j], range), min_disp));
            if (kVec == 4) *reinterpret_cast<float4*>(M.out[k] + i) = make_float4(v[k][0], v[k][1 % kVec], v[k][2 % kVec], v[k][3 % kVec]);
            else M.out[k][i] = v[k][0];
        }
}

template <int kVec>
__global__ void __launch_bounds__(256)
disp_to_depth_fwd_kernel(const __grid_constant__ MapPtrs M, int64_t n, float min_disp, float range) {
    disp_to_depth_fwd_body<kVec>(M, n, min_disp, range, blockIdx.x);
}

template <int kVec>
__device__ __forceinline__ void disp_to_depth_bwd_body(const MapPtrs& M, int64_t n, float range, int block) {
    const int64_t i = ((int64_t)block * 256 + threadIdx.x) * kVec;
    if (i >= n) return;
    float g[4][kVec], d[4][kVec];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < M.count) {
            if (kVec == 4) {
                const float4 q = __ldg(reinterpret_cast<const float4*>(M.in[k] + i));
                const float4 r = __ldg(reinterpret_cast<const float4*>(M.aux[k] + i));       // the depth computed by the forward
                g[k][0] = q.x; g[k][1 % kVec] = q.y; g[k][2 % kVec] = q.z; g[k][3 % kVec] = q.w;
                d[k][0] = r.x; d[k][1 % kVec] = r.y; d[k][2 % kVec] = r.z; d[k][3 % kVec] = r.w;
            } else {
                g[k][0] = __ldg(M.in[k] + i);
                d[k][0] = __ldg(M.aux[k] + i);
            }
        }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < M.count) {
#pragma unroll
            for (int j = 0; j < kVec; ++j) g[k][j] = -g[k][j] * d[k][j] * d[k][j] * range;
            if (kVec == 4) *reinterpret_cast<float4*>(M.out[k] + i) = make_float4(g[k][0], g[k][1 % kVec], g[k][2 % kVec], g[k][3 % kVec]);
            else M.out[k][i] = g[k][0];
        }
}

template <int kVec>
__global__ void __launch_bounds__(256)
disp_to_depth_bwd_kernel(const __grid_constant__ MapPtrs M, int64_t n, float range) {
    disp_to_depth_bwd_body<kVec>(M, n, range, blockIdx.x);
}

// The glue on either side of the pair kernels as ONE launch each (a small kernel costs ~3 us of a 0.3 ms step whatever
// it does): prologue = disp -> depth of up to four maps + pose -> K[R|t] of every group, the poses read through a
// pointer table so that no concatenated copy is needed; epilogue = their two chain rules.  Blocks [0, nb_maps) work
// on the maps, the blocks behind them on the poses (item i = group i / per, row i % per).
struct FrameGlue {
    MapPtrs M;
    int64_t n;
    float min_disp, range, sign;
    int nb_maps, pose_stride, per, N, Bk;
    const float* pose[8];
    const float* K;
    float* proj;
    float* kinv;             // prologue: K^-1 [Bk,9] out (nullable)
    const float* g_proj;
    float* g_pose;
};

template <int kVec, bool kNoFma>
__global__ void __launch_bounds__(256) frame_prologue_kernel(const __grid_constant__ FrameGlue G) {
    if ((int)blockIdx.x < G.nb_maps) { disp_to_depth_fwd_body<kVec>(G.M, G.n, G.min_disp, G.range, blockIdx.x); return; }
    const int i = ((int)blockIdx.x - G.nb_maps) * 256 + threadIdx.x;
    if (i < G.N) pose_proj_fwd_body<kNoFma>(G.pose[i / G.per] + (i % G.per) * G.pose_stride, G.sign, G.K, G.Bk, G.proj, i);
    // K^-1 by the last threads of the pose blocks (the first ones hold a pose each), hidden behind the map blocks
    const int j = (int)(gridDim.x - G.nb_maps) * 256 - 1 - i;
    if (G.kinv && j < G.Bk) intrinsics_inverse_body(G.K, G.kinv, j);
}

template <int kVec>
__global__ void __launch_bounds__(256) frame_epilogue_kernel(const __grid_constant__ FrameGlue G) {
    if ((int)blockIdx.x < G.nb_maps) { disp_to_depth_bwd_body<kVec>(G.M, G.n, G.range, blockIdx.x); return; }
    const int i = ((int)blockIdx.x - G.nb_maps) * 256 + threadIdx.x;
    if (i < G.N) pose_proj_bwd_body(G.pose[i / G.per] + (i % G.per) * G.pose_stride, G.sign, G.K, G.Bk, G.g_proj, G.g_pose, i);
}

static bool maps_vectorisable(const MapPtrs& M, int64_t n) {
    if (n % 4) return false;
    for (int k = 0; k < M.count; ++k)
        if (((uintptr_t)M.in[k] | (uintptr_t)M.out[k] | (uintptr_t)M.aux[k]) & 15) return false;
    return true;
}

// The same with the nearest-neighbour upsample of the lower pyramid scales folded in
// (Compute_Loss.forward, losses.py:86-88,102-104: F.interpolate(disp, (H, W), mode='nearest') then
// disp_to_depth).  ATen's rule: src = min(int(floorf(dst * scale)), in - 1), scale = float(in) / out.
struct UpShape { int B, h, w, H, W; float sh, sw; };

__device__ __forceinline__ int nearest_src(int dst, float scale, int in_size) {
    const int s = (int)floorf(__fmul_rn((float)dst, scale));
    return s < in_size - 1 ? s : in_size - 1;
}

__global__ void __launch_bounds__(256)
disp_up_to_depth_fwd_kernel(const __grid_constant__ MapPtrs M, UpShape U, float min_disp, float range) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t plane = (int64_t)U.H * U.W;
    if (i >= U.B * plane) return;
    const int b = (int)(i / plane);
    const int r = (int)(i - b * plane);
    const int Y = r / U.W, X = r - Y * U.W;
    const int64_t src = ((int64_t)b * U.h + nearest_src(Y, U.sh, U.h)) * U.w + nearest_src(X, U.sw, U.w);
    for (int k = 0; k < M.count; ++k) {
        const float scaled = __fadd_rn(__fmul_rn(__ldg(M.in[k] + src), range), min_disp);
        M.out[k][i] = __frcp_rn(scaled);
    }
}

// One thread per low-resolution pixel gathers the gradients of the full-resolution pixels that read it.
__global__ void __launch_bounds__(256)
disp_up_to_depth_bwd_kernel(const __grid_constant__ MapPtrs M, UpShape U, float range) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t plane = (int64_t)U.h * U.w;
    if (i >= U.B * plane) return;
    const int b = (int)(i / plane);
    const int r = (int)(i - b * plane);
    const int y = r / U.w, x = r - y * U.w;
    // candidate destination ranges (one extra on each side), filtered with the forward's own rule
    int Y0 = (int)floorf((float)y / U.sh) - 1, Y1 = (int)ceilf((float)(y + 1) / U.sh) + 1;
    int X0 = (int)floorf((float)x / U.sw) - 1, X1 = (int)ceilf((float)(x + 1) / U.sw) + 1;
    Y0 = Y0 < 0 ? 0 : Y0; X0 = X0 < 0 ? 0 : X0;
    Y1 = Y1 > U.H - 1 ? U.H - 1 : Y1; X1 = X1 > U.W - 1 ? U.W - 1 : X1;
    for (int k = 0; k < M.count; ++k) {
        float acc = 0.f;
        for (int Y = Y0; Y <= Y1; ++Y) {
            if (nearest_src(Y, U.sh, U.h) != y) continue;
            const int64_t row = ((int64_t)b * U.H + Y) * U.W;
            for (int X = X0; X <= X1; ++X) {
                if (nearest_src(X, U.sw, U.w) != x) continue;
                const float d = __ldg(M.aux[k] + row + X);
                acc += -__ldg(M.in[k] + row + X) * d * d * range;
            }
        }
        M.out[k][i] = acc;
    }
}

// uint8 image -> float in [0, 1] exactly like the reference's loader does on the host
// (utils/custom_transforms.py:74: torch.from_numpy(im).float() / 255, a true IEEE division), four pixels per thread:
// the images can then cross the host link as bytes (a quarter of the fp32 traffic).
__global__ void __launch_bounds__(256)
u8_to_float_kernel(const unsigned char* __restrict__ src, float* __restrict__ dst, int64_t n) {
    const int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 4;
    if (i + 3 < n && (reinterpret_cast<uintptr_t>(src + i) & 3) == 0 && (reinterpret_cast<uintptr_t>(dst + i) & 15) == 0) {
        const unsigned v = *reinterpret_cast<const unsigned*>(src + i);
        float4 o;
        o.x = __fdiv_rn((float)(v & 255u), 255.0f);
        o.y = __fdiv_rn((float)((v >> 8) & 255u), 255.0f);
        o.z = __fdiv_rn((float)((v >> 16) & 255u), 255.0f);
        o.w = __fdiv_rn((float)(v >> 24), 255.0f);
        *reinterpret_cast<float4*>(dst + i) = o;
    } else {
        for (int64_t k = i; k < n && k < i + 4; ++k) dst[k] = __fdiv_rn((float)src[k], 255.0f);
    }
}

constexpr int kReduceThreads = 256;

// `fin.out` != nullptr: the last block to arrive also turns the sums into the loss terms (frame_finalize_body), so the
// min-reprojection reduce and the finalize are one launch.
constexpr int kReducePix = 8;       // pixels per thread and sweep: their loads of one candidate map are issued together

__global__ void __launch_bounds__(kReduceThreads)
min_reduce_kernel(const float* __restrict__ base, int64_t stride, int count, int64_t n, float* __restrict__ out, FrameFinalize fin) {
    TCSFM_SHARED float red[kReduceThreads / 32];
    float part[1] = {0.f};
    const int64_t sweep = (int64_t)gridDim.x * kReduceThreads * kReducePix;
    for (int64_t i0 = (int64_t)blockIdx.x * kReduceThreads * kReducePix + threadIdx.x; i0 < n; i0 += sweep) {
        float m[kReducePix];
#pragma unroll
        for (int k = 0; k < kReducePix; ++k) {
            const int64_t i = i0 + k * kReduceThreads;
            m[k] = i < n ? __ldg(base + i) : 0.f;
        }
        for (int j = 1; j < count; ++j) {
            float v[kReducePix];
#pragma unroll
            for (int k = 0; k < kReducePix; ++k) {
                const int64_t i = i0 + k * kReduceThreads;
                v[k] = i < n ? __ldg(base + j * stride + i) : 0.f;
            }
#pragma unroll
            for (int k = 0; k < kReducePix; ++k) m[k] = (v[k] < m[k] || v[k] != v[k]) ? v[k] : m[k];   // torch.min: lowest index on ties, NaN propagates
        }
#pragma unroll
        for (int k = 0; k < kReducePix; ++k) part[0] += m[k];         // (pixels past the end contributed min(0, 0) = 0)
    }
    block_atomic_accumulate<1>(part, red, out, threadIdx.x, kReduceThreads);
    finalize_by_last_block(fin, out);
}

__global__ void frame_finalize_kernel(const float* __restrict__ sums, const float* __restrict__ min_sum, tcsfm_frame_cfg cfg,
                                      float* __restrict__ out, float* __restrict__ total) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    frame_finalize_body(sums, min_sum, cfg, out, total);
}

// The upstream of the three terms / of their sum -> per-group scalars, by one thread; the other threads of the grid zero
// the accumulated gradient buffer of the backward pair launch (`zero`, n4 float4 elements; nullable), so that the
// backward needs no separate fill.
__global__ void __launch_bounds__(256)
frame_bwd_prepare_kernel(const float* __restrict__ g_out, const float* __restrict__ g_total, tcsfm_frame_cfg cfg,
                         float* __restrict__ g_scalars, float* __restrict__ g_min, float4* __restrict__ zero, int64_t n4) {
    for (int64_t i0 = (int64_t)blockIdx.x * 1024 + threadIdx.x; i0 < n4; i0 += (int64_t)gridDim.x * 1024) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (i0 + k * 256 < n4) zero[i0 + k * 256] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const float gt = g_total ? g_total[0] : 0.f;
    const float g_inv = (g_out ? g_out[0] : 0.f) + gt, g_fwd = (g_out ? g_out[1] : 0.f) + gt, g_dep = (g_out ? g_out[2] : 0.f) + gt;
    for (int g = 0; g < cfg.n_groups; ++g) {
        g_scalars[g * 2 + 0] = (cfg.role[g] == 0) ? cfg.w_inverse * g_inv : 0.f;
        g_scalars[g * 2 + 1] = cfg.w_depth * g_dep;
    }
    g_min[0] = g_fwd / (float)cfg.n_min_pixels;
}

}  // namespace tcsfm

using namespace tcsfm;

extern "C" int tcsfm_intrinsics_inverse(const float* K, float* kinv, int B, void* stream) {
    if (!K || !kinv || B <= 0) { set_error("tcsfm_intrinsics_inverse: bad arguments"); return 1; }
    TCSFM_LAUNCH(intrinsics_inverse_kernel, dim3((B + 63) / 64), dim3(64), 0, stream, K, kinv, B);
    return check_launch("tcsfm_intrinsics_inverse");
}

extern "C" int tcsfm_u8_to_float(const unsigned char* src, float* dst, int64_t n, void* stream) {
    if (!src || !dst || n <= 0) { set_error("tcsfm_u8_to_float: bad arguments"); return 1; }
    const int64_t blocks = (n + 1023) / 1024;
    if (blocks >= ((int64_t)1 << 31)) { set_error("tcsfm_u8_to_float: too many elements"); return 1; }
    TCSFM_LAUNCH(u8_to_float_kernel, dim3((unsigned)blocks), dim3(256), 0, stream, src, dst, n);
    return check_launch("tcsfm_u8_to_float");
}

extern "C" int tcsfm_pose_proj_fwd(const float* pose, float sign, const float* K, int Bk, float* proj, int N, int flags,
                                   void* stream) {
    if (!pose || !K || !proj || N <= 0 || Bk <= 0) { set_error("tcsfm_pose_proj_fwd: bad arguments"); return 1; }
    if (flags & TCSFM_ARITH_BMM_NOFMA) {
        TCSFM_LAUNCH(pose_proj_fwd_kernel<true>, dim3((N + 63) / 64), dim3(64), 0, stream, pose, sign, K, Bk, proj, N);
    } else {
        TCSFM_LAUNCH(pose_proj_fwd_kernel<false>, dim3((N + 63) / 64), dim3(64), 0, stream, pose, sign, K, Bk, proj, N);
    }
    return check_launch("tcsfm_pose_proj_fwd");
}

extern "C" int tcsfm_pose_proj_bwd(const float* pose, float sign, const float* K, int Bk, const float* g_proj,
                                   float* g_pose, int N, void* stream) {
    if (!pose || !K || !g_proj || !g_pose || N <= 0 || Bk <= 0) { set_error("tcsfm_pose_proj_bwd: bad arguments"); return 1; }
    TCSFM_LAUNCH(pose_proj_bwd_kernel, dim3((N + 63) / 64), dim3(64), 0, stream, pose, sign, K, Bk, g_proj, g_pose, N);
    return check_launch("tcsfm_pose_proj_bwd");
}

extern "C" int tcsfm_disp_to_depth_fwd(const float* const* disp, float* const* depth, int count, int64_t n,
                                       float min_disp, float range, void* stream) {
    if (!disp || !depth || count < 1 || count > 4 || n <= 0) { set_error("tcsfm_disp_to_depth_fwd: bad arguments"); return 1; }
    MapPtrs M;
    memset(&M, 0, sizeof(M));
    M.count = count;
    for (int k = 0; k < count; ++k) { M.in[k] = disp[k]; M.out[k] = depth[k]; }
    if (maps_vectorisable(M, n))
        TCSFM_LAUNCH(disp_to_depth_fwd_kernel<4>, dim3((unsigned)((n / 4 + 255) / 256)), dim3(256), 0, stream, M, n, min_disp, range);
    else
        TCSFM_LAUNCH(disp_to_depth_fwd_kernel<1>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, M, n, min_disp, range);
    return check_launch("tcsfm_disp_to_depth_fwd");
}

extern "C" int tcsfm_disp_to_depth_bwd(const float* const* g_depth, const float* const* depth, float* const* g_disp, int count,
                                       int64_t n, float range, void* stream) {
    if (!g_depth || !depth || !g_disp || count < 1 || count > 4 || n <= 0) { set_error("tcsfm_disp_to_depth_bwd: bad arguments"); return 1; }
    MapPtrs M;
    memset(&M, 0, sizeof(M));
    M.count = count;
    for (int k = 0; k < count; ++k) { M.in[k] = g_depth[k]; M.aux[k] = depth[k]; M.out[k] = g_disp[k]; }
    if (maps_vectorisable(M, n))
        TCSFM_LAUNCH(disp_to_depth_bwd_kernel<4>, dim3((unsigned)((n / 4 + 255) / 256)), dim3(256), 0, stream, M, n, range);
    else
        TCSFM_LAUNCH(disp_to_depth_bwd_kernel<1>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, M, n, range);
    return check_launch("tcsfm_disp_to_depth_bwd");
}

static bool up_shape(UpShape& U, int B, int h, int w, int H, int W) {
    if (B <= 0 || h <= 0 || w <= 0 || H < h || W < w) return false;
    U.B = B; U.h = h; U.w = w; U.H = H; U.W = W;
    U.sh = (float)h / (float)H; U.sw = (float)w / (float)W;          // ATen compute_scales_value<float>
    return true;
}

extern "C" int tcsfm_disp_upsample_to_depth_fwd(const float* const* disp, float* const* depth, int count, int B, int h, int w,
                                                int H, int W, float min_disp, float range, void* stream) {
    UpShape U;
    if (!disp || !depth || count < 1 || count > 4 || !up_shape(U, B, h, w, H, W)) { set_error("tcsfm_disp_upsample_to_depth_fwd: bad arguments"); return 1; }
    MapPtrs M;
    memset(&M, 0, sizeof(M));
    M.count = count;
    for (int k = 0; k < count; ++k) { M.in[k] = disp[k]; M.out[k] = depth[k]; }
    const int64_t n = (int64_t)B * H * W;
    TCSFM_LAUNCH(disp_up_to_depth_fwd_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, M, U, min_disp, range);
    return check_launch("tcsfm_disp_upsample_to_depth_fwd");
}

extern "C" int tcsfm_disp_upsample_to_depth_bwd(const float* const* g_depth, const float* const* depth, float* const* g_disp,
                                                int count, int B, int h, int w, int H, int W, float range, void* stream) {
    UpShape U;
    if (!g_depth || !depth || !g_disp || count < 1 || count > 4 || !up_shape(U, B, h, w, H, W)) { set_error("tcsfm_disp_upsample_to_depth_bwd: bad arguments"); return 1; }
    MapPtrs M;
    memset(&M, 0, sizeof(M));
    M.count = count;
    for (int k = 0; k < count; ++k) { M.in[k] = g_depth[k]; M.aux[k] = depth[k]; M.out[k] = g_disp[k]; }
    const int64_t n = (int64_t)B * h * w;
    TCSFM_LAUNCH(disp_up_to_depth_bwd_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, M, U, range);
    return check_launch("tcsfm_disp_upsample_to_depth_bwd");
}

extern "C" int tcsfm_min_reduce(const float* base, int64_t stride, int count, int64_t n, float* out_sum, int* ticket,
                                const float* sums, const tcsfm_frame_cfg* cfg, float* out, float* total, void* stream) {
    if (!base || !out_sum || count <= 0 || n <= 0) { set_error("tcsfm_min_reduce: bad arguments"); return 1; }
    if (cfg && (!ticket || !sums || !out || cfg->n_groups <= 0 || cfg->n_groups > 8)) { set_error("tcsfm_min_reduce: bad finalize arguments"); return 1; }
    cudaMemsetAsync(out_sum, 0, sizeof(float), (cudaStream_t)stream);
    FrameFinalize fin;
    memset(&fin, 0, sizeof(fin));
    if (cfg) {
        cudaMemsetAsync(ticket, 0, sizeof(int), (cudaStream_t)stream);
        fin.sums = sums; fin.cfg = *cfg; fin.out = out; fin.total = total; fin.ticket = ticket;
    }
    int64_t blocks = (n + kReduceThreads * 8 - 1) / (kReduceThreads * 8);
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    TCSFM_LAUNCH(min_reduce_kernel, dim3((unsigned)blocks), dim3(kReduceThreads), 0, stream, base, stride, count, n, out_sum, fin);
    return check_launch("tcsfm_min_reduce");
}

extern "C" int tcsfm_frame_finalize(const float* sums, const float* min_sum, const tcsfm_frame_cfg* cfg, float* out, float* total,
                                    void* stream) {
    if (!sums || !cfg || !out || cfg->n_groups <= 0 || cfg->n_groups > 8) { set_error("tcsfm_frame_finalize: bad arguments"); return 1; }
    TCSFM_LAUNCH(frame_finalize_kernel, dim3(1), dim3(32), 0, stream, sums, min_sum, *cfg, out, total);
    return check_launch("tcsfm_frame_finalize");
}

extern "C" int tcsfm_frame_bwd_prepare(const float* g_out, const float* g_total, const tcsfm_frame_cfg* cfg, float* g_scalars,
                                       float* g_min, float* zero, int64_t n_zero, void* stream) {
    if ((!g_out && !g_total) || !cfg || !g_scalars || !g_min || cfg->n_groups <= 0 || cfg->n_groups > 8) { set_error("tcsfm_frame_bwd_prepare: bad arguments"); return 1; }
    if (zero && (n_zero <= 0 || n_zero % 4 || ((uintptr_t)zero & 15))) { set_error("tcsfm_frame_bwd_prepare: the buffer must be 16-byte aligned with a multiple of 4 elements"); return 1; }
    const int64_t n4 = zero ? n_zero / 4 : 0;
    int64_t blocks = (n4 + 1023) / 1024;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks < 1) blocks = 1;
    TCSFM_LAUNCH(frame_bwd_prepare_kernel, dim3((unsigned)blocks), dim3(256), 0, stream, g_out, g_total, *cfg, g_scalars, g_min,
                 reinterpret_cast<float4*>(zero), n4);
    return check_launch("tcsfm_frame_bwd_prepare");
}


static int fill_glue(FrameGlue& G, int count, int64_t n, const float* const* pose, int n_groups, int pose_stride, float sign,
                     const float* K, int B, const char* who) {
    if (count < 1 || count > 4 || n <= 0 || !pose || n_groups < 1 || n_groups > 8 || pose_stride < 6 || !K || B <= 0) {
        set_error("%s: bad arguments", who); return 1;
    }
    G.M.count = count;
    G.n = n;
    G.sign = sign;
    G.pose_stride = pose_stride; G.per = B; G.N = n_groups * B; G.Bk = B;
    for (int g = 0; g < n_groups; ++g) {
        if (!pose[g]) { set_error("%s: null pose pointer", who); return 1; }
        G.pose[g] = pose[g];
    }
    G.K = K;
    return 0;
}

extern "C" int tcsfm_frame_prologue(const float* const* disp, float* const* depth, int count, int64_t n, float min_disp, float range,
                                    const float* const* pose, int n_groups, int pose_stride, float sign, const float* K, int B,
                                    float* proj, float* kinv, int flags, void* stream) {
    FrameGlue G;
    memset(&G, 0, sizeof(G));
    if (!disp || !depth || !proj) { set_error("tcsfm_frame_prologue: null pointer"); return 1; }
    if (int rc = fill_glue(G, count, n, pose, n_groups, pose_stride, sign, K, B, "tcsfm_frame_prologue")) return rc;
    for (int k = 0; k < count; ++k) { G.M.in[k] = disp[k]; G.M.out[k] = depth[k]; }
    G.min_disp = min_disp; G.range = range; G.proj = proj; G.kinv = kinv;
    const bool vec = maps_vectorisable(G.M, n);
    G.nb_maps = (int)(((vec ? n / 4 : n) + 255) / 256);
    dim3 grid(G.nb_maps + (G.N + 255) / 256), block(256);
    const bool nofma = (flags & TCSFM_ARITH_BMM_NOFMA) != 0;
    if (vec) { if (nofma) TCSFM_LAUNCH((frame_prologue_kernel<4, true>), grid, block, 0, stream, G); else TCSFM_LAUNCH((frame_prologue_kernel<4, false>), grid, block, 0, stream, G); }
    else { if (nofma) TCSFM_LAUNCH((frame_prologue_kernel<1, true>), grid, block, 0, stream, G); else TCSFM_LAUNCH((frame_prologue_kernel<1, false>), grid, block, 0, stream, G); }
    return check_launch("tcsfm_frame_prologue");
}

extern "C" int tcsfm_frame_epilogue(const float* const* g_depth, const float* const* depth, float* const* g_disp, int count, int64_t n,
                                    float range, const float* const* pose, int n_groups, int pose_stride, float sign,
                                    const float* K, int B, const float* g_proj, float* g_pose, void* stream) {
    FrameGlue G;
    memset(&G, 0, sizeof(G));
    if (!g_depth || !depth || !g_disp || !g_proj || !g_pose) { set_error("tcsfm_frame_epilogue: null pointer"); return 1; }
    if (int rc = fill_glue(G, count, n, pose, n_groups, pose_stride, sign, K, B, "tcsfm_frame_epilogue")) return rc;
    for (int k = 0; k < count; ++k) { G.M.in[k] = g_depth[k]; G.M.aux[k] = depth[k]; G.M.out[k] = g_disp[k]; }
    G.range = range; G.g_proj = g_proj; G.g_pose = g_pose;
    const bool vec = maps_vectorisable(G.M, n);
    G.nb_maps = (int)(((vec ? n / 4 : n) + 255) / 256);
    dim3 grid(G.nb_maps + (G.N + 255) / 256), block(256);
    if (vec) TCSFM_LAUNCH(frame_epilogue_kernel<4>, grid, block, 0, stream, G);
    else TCSFM_LAUNCH(frame_epilogue_kernel<1>, grid, block, 0, stream, G);
    return check_launch("tcsfm_frame_epilogue");
}
