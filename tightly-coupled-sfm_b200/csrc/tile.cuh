// 64x16-pixel output tiles with a halo ring, 256 threads, 4 pixels per thread.
//
// Shared-memory tiles are indexed in *padded-image* coordinates: cell (cx, cy),
// cx in [-R, 64+R), cy in [-R, 16+R), holds the value at image position
// (reflect1(y0+cy), reflect1(x0+cx)) -- i.e. ReflectionPad2d(1) is applied when
// the tile is filled, so a 3x3 window is a plain neighbourhood read.  Only one
// pixel of padding exists; cells further outside the image are never read by a
// consumer and are filled with zeros.
#pragma once
#include "tcsfm_math.cuh"

namespace tcsfm {

constexpr int kTileW = 64;
constexpr int kTileH = 16;
constexpr int kTileThreads = 256;
constexpr int kPixPerThread = 4;    // a vertical strip of 4 rows at one column

// thread `tid`'s k-th own pixel inside the tile: warps span 32 consecutive columns
__device__ __forceinline__ void own_pixel(int tid, int k, int& tx, int& ty) {
    tx = tid & (kTileW - 1);
    ty = (tid >> 6) * kPixPerThread + k;
}

// The tiles covering an H x W image, numbered row-major; partial tiles at the right and bottom edges.
__host__ __device__ __forceinline__ int tiles_x(int W) { return (W + kTileW - 1) / kTileW; }
__host__ __device__ __forceinline__ int tiles_y(int H) { return (H + kTileH - 1) / kTileH; }
inline int tile_count(int H, int W) { return tiles_x(W) * tiles_y(H); }

// image position (x0, y0) of tile `t`'s cell (0, 0); `t` is unsigned like blockIdx.x (an unsigned division is the shorter)
__device__ __forceinline__ void tile_origin(unsigned t, int W, int& x0, int& y0) {
    const int tx = tiles_x(W);
    const int ty = t / tx;
    const int tile_x = t - ty * tx;
    x0 = tile_x * kTileW;
    y0 = ty * kTileH;
}

template <int R>
struct Tile {
    static constexpr int kPitch = kTileW + 2 * R;
    static constexpr int kRows = kTileH + 2 * R;
    static constexpr int kCells = kPitch * kRows;
    // linear cell index of tile-relative coordinates (may be negative down to -R)
    __device__ __forceinline__ static int cell(int cx, int cy) { return (cy + R) * kPitch + (cx + R); }
    __device__ __forceinline__ static void cell_xy(int cell, int& cx, int& cy) {
        cy = cell / kPitch;
        cx = cell - cy * kPitch - R;
        cy -= R;
    }
    // Maps a cell to the image pixel whose value it holds.  Returns false for
    // cells that no consumer reads (more than one pixel outside the image).
    __device__ __forceinline__ static bool cell_to_reflected(int cell, int x0, int y0, int H, int W, int& ry, int& rx) {
        int cx, cy;
        cell_xy(cell, cx, cy);
        const int gx = x0 + cx, gy = y0 + cy;
        if (gx < -1 || gx > W || gy < -1 || gy > H) return false;
        rx = reflect1(gx, W);
        ry = reflect1(gy, H);
        return true;
    }
};

// The halo ring of a Tile<1>, enumerated 0 .. kRingCells - 1 (top row, bottom row, left column, right column).
constexpr int kRingCells = 2 * (kTileW + 2) + 2 * kTileH;
__device__ __forceinline__ void ring_cell(int r, int& cx, int& cy) {
    if (r < kTileW + 2) { cx = r - 1; cy = -1; }
    else if (r < 2 * (kTileW + 2)) { cx = r - (kTileW + 2) - 1; cy = kTileH; }
    else if (r < 2 * (kTileW + 2) + kTileH) { cx = -1; cy = r - 2 * (kTileW + 2); }
    else { cx = kTileW; cy = r - 2 * (kTileW + 2) - kTileH; }
}

// Zeroes one cell of the three channel planes of a float2 Tile<1>.
__device__ __forceinline__ void zero_cell(float2* tw, int cell) {
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) tw[ch * Tile<1>::kCells + cell] = make_float2(0.f, 0.f);
}

// Fills one cell of a (target, warped source) tile with the image pixel (rx, ry), whose target depth is `depth`, warped
// under `cam` exactly as warp_fwd_kernel forms projected_img there; returns the warp in p and its taps.  Channel
// planes are tgt_sc / src_sc elements apart (32-bit offsets).
template <int F>
__device__ __forceinline__ TapIdx fill_warped_cell(const Cam& cam, const Arith& A, const float* tgt, int tgt_sc, const float* src,
                                                   int src_sc, int rx, int ry, float depth, float2* tw, int cell, WarpPt& p) {
    const int pix = ry * A.W + rx;
    warp_point<F>(cam, A, rx, ry, depth, p);
    const TapIdx ti = make_taps(p, A.H, A.W);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const float w = blend(load_taps(src, ch * src_sc, ti, A.W), ti);
        tw[ch * Tile<1>::kCells + cell] = make_float2(__ldg(tgt + (ch * tgt_sc + pix)), w);
    }
    return ti;
}

// One channel of  w_l1 * clamp|x - y| + w_ssim * SSIM(x, y)  down the strip of own pixels (tx, ty0 .. ty0 + 3) of a
// Tile<1> plane of (x, y) pairs: a rolling 3-row register window of taps whose squares / products are formed per use
// (cheaper than keeping 27 more registers live across the strip), the five statistics as packed fp32x2 sums in
// avg_pool2d order, exact /9.  esum[k] = the value of pixel k (`first` channel) or esum[k] + it.  Every pixel's window
// statistics go to sink(k, stats, terms): the callers that keep SSIM adjoint coefficients store them from there.
// `a` is the kernel's argument struct, whose w_l1, w_ssim, C1 and C2 are read through the reference (passed as
// values, they changed the kernels' register allocation and scheduling).
template <class Args, class Sink>
__device__ __forceinline__ void ssim_l1_strip(const float2* plane, int tx, int ty0, const Args& a, bool first,
                                              float (&esum)[kPixPerThread], Sink&& sink) {
    using T1 = Tile<1>;
    float2 v[3][3];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) v[r][cc] = plane[T1::cell(tx - 1 + cc, ty0 - 1 + r)];
#pragma unroll
    for (int k = 0; k < kPixPerThread; ++k) {
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) v[(k + 2) % 3][cc] = plane[T1::cell(tx - 1 + cc, ty0 + 1 + k)];
        float2 wv[9], wsq[9];
        float wab[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            wv[i] = v[(k + i / 3) % 3][i % 3];
            wsq[i] = square2_rn(wv[i]);
            wab[i] = __fmul_rn(wv[i].x, wv[i].y);
        }
        const SsimStats s = ssim_stats_packed(wv, wsq, wab);
        const SsimTerms t = ssim_terms(s, a.C1, a.C2);
        const float l1 = clamp01_nan(fabsf(__fsub_rn(wv[4].x, wv[4].y)));
        const float e = __fadd_rn(__fmul_rn(l1, a.w_l1), __fmul_rn(clamp01_nan(t.raw), a.w_ssim));
        esum[k] = first ? e : __fadd_rn(esum[k], e);
        sink(k, s, t);
    }
}

// the sink of ssim_l1_strip for callers that keep no coefficients
struct NoSsimSink {
    __device__ __forceinline__ void operator()(int, const SsimStats&, const SsimTerms&) const {}
};

}  // namespace tcsfm
