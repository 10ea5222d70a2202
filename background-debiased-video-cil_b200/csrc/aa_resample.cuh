// Device side of torchvision's antialiased bilinear resize (ATen's separable CPU kernel, UpSampleKernel.cpp) on uint8
// planes, shared by the ragged BG-mix blend (raggedmix.cu) and the batched RandomResizedCrop (resized_crop.cu).
//
// A source is a window of a channel plane: `org` points at the window's top-left pixel and `stride` is the plane's row
// stride in bytes, so a resize of a whole image is the window at origin 0 with stride = width, and a crop is the window
// at (top, left).  Per axis, a table built on the host by bgd_aa_resize_table (in = window size, out = output size) holds
// one entry per output index: {first source index relative to the window, tap count, K float weights}; an axis whose
// size does not change has no table and its pass is skipped.  The arithmetic (stated in full in raggedmix.cu):
// horizontal pass first, then vertical; each output acc = v_0 * w_0, then acc += v_j * w_j for j = 1 .. size-1, where
// the first 4 * floor((size - 1) / 4) steps round the product and the sum separately and the rest are fused
// multiply-adds.
#pragma once

#include <cstdint>

namespace bgd {

// one accumulation step of ATen's tap loop: step j (1-based) of n = size - 1 steps
__device__ __forceinline__ float aa_step(float acc, float v, float w, int j, int n_unfused)
{
    return j <= n_unfused ? __fadd_rn(acc, __fmul_rn(v, w)) : __fmaf_rn(v, w, acc);
}

// horizontal pass at one output column of one source row: `row` points at the window's column 0 of that row
__device__ __forceinline__ float aa_row(const uint8_t *row, const int32_t *ent)
{
    const int mn = ent[0], size = ent[1];
    const float *w = reinterpret_cast<const float *>(ent + 2);
    float acc = __fmul_rn((float)__ldg(row + mn), __ldg(w));
    const int n_unfused = ((size - 1) >> 2) << 2;
    for (int j = 1; j < size; ++j) acc = aa_step(acc, (float)__ldg(row + mn + j), __ldg(w + j), j, n_unfused);
    return acc;
}

// value of the resized window at output (Y, X): window origin `org` in a plane of row stride `stride` bytes; column /
// row tables at word offsets xtab / ytab of `tables` with kx / ky taps per entry (-1 = that axis keeps its size)
__device__ __forceinline__ float aa_sample(const uint8_t *org, int64_t stride, const int32_t *tables, int xtab, int kx,
                                           int ytab, int ky, int Y, int X)
{
    const int32_t *xe = xtab >= 0 ? tables + xtab + (int64_t)X * (2 + kx) : nullptr;
    if (ytab < 0) {
        const uint8_t *row = org + (int64_t)Y * stride;
        return xe ? aa_row(row, xe) : (float)__ldg(row + X);
    }
    const int32_t *ye = tables + ytab + (int64_t)Y * (2 + ky);
    const int mn = ye[0], size = ye[1];
    const float *w = reinterpret_cast<const float *>(ye + 2);
    const int n_unfused = ((size - 1) >> 2) << 2;
    float acc = 0.f;
    for (int r = 0; r < size; ++r) {
        const uint8_t *row = org + (int64_t)(mn + r) * stride;
        const float hv = xe ? aa_row(row, xe) : (float)__ldg(row + X);
        acc = r == 0 ? __fmul_rn(hv, __ldg(w)) : aa_step(acc, hv, __ldg(w + r), r, n_unfused);
    }
    return acc;
}

// ---- tiled form: the horizontal pass of a tile's source rows into shared memory, then the vertical pass from there ----
// Window rows rmin .. rend-1 feed output rows Y0 .. Ylast of a tile (the rows themselves when the axis keeps its size).
__device__ __forceinline__ void aa_tile_rows(const int32_t *tables, int ytab, int ky, int Y0, int Ylast, int &rmin, int &rend)
{
    rmin = Y0;
    rend = Ylast + 1;
    if (ytab >= 0) {
        rmin = tables[ytab + (int64_t)Y0 * (2 + ky)];
        const int32_t *last = tables + ytab + (int64_t)Ylast * (2 + ky);
        rend = last[0] + last[1];
    }
}

// Horizontal pass of one output column (table entry `xe`, or the pixel column X itself when xe is null) of window rows
// rmin + r for r = r_first, r_first + kRowStep, ... < nrows, all three channel planes (`plane` bytes apart), into
// s_h[c][r][x].  The caller's threads split the columns and the row phases among themselves.
template <int kRowStep, int kRows, int kCols>
__device__ __forceinline__ void aa_tile_hpass(float (&s_h)[3][kRows][kCols], const uint8_t *org, int64_t plane, int stride,
                                              const int32_t *xe, int X, int x, int rmin, int r_first, int nrows)
{
    const int xmin = xe ? xe[0] : X, xsize = xe ? xe[1] : 1;
    const int step = kRowStep * stride;                                 // bytes between this thread's source rows
    if (xsize <= 3) {
        // up to 3 taps (any up-scaling): v0 w0, then fused multiply-adds -- ATen's order for fewer than 5 taps.
        // An absent tap has weight 0 and re-reads the pixel before it, which leaves the sum unchanged.
        const float *w = reinterpret_cast<const float *>(xe + 2);
        const float w0 = xe ? __ldg(w) : 1.f, w1 = xsize > 1 ? __ldg(w + 1) : 0.f, w2 = xsize > 2 ? __ldg(w + 2) : 0.f;
        const int o1 = xsize > 1 ? 1 : 0, o2 = xsize > 2 ? 2 : o1;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint8_t *q = org + c * plane + (int64_t)(rmin + r_first) * stride + xmin;
            float *dst = &s_h[c][r_first][x];
#pragma unroll 4
            for (int r = r_first; r < nrows; r += kRowStep) {
                const float v0 = (float)__ldg(q), v1 = (float)__ldg(q + o1), v2 = (float)__ldg(q + o2);
                *dst = __fmaf_rn(v2, w2, __fmaf_rn(v1, w1, __fmul_rn(v0, w0)));
                q += step;
                dst += kRowStep * kCols;
            }
        }
    } else {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint8_t *q = org + c * plane + (int64_t)(rmin + r_first) * stride;
            for (int r = r_first; r < nrows; r += kRowStep, q += step) s_h[c][r][x] = aa_row(q, xe);
        }
    }
}

// Vertical pass for 4 adjacent output columns tx .. tx+3 of the tile at output row Y (table entry `ye`, or window row
// Y itself when ye is null) from the horizontal results in s_h: g[c][i].
template <int kRows, int kCols>
__device__ __forceinline__ void aa_tile_vpass4(const float (&s_h)[3][kRows][kCols], const int32_t *ye, int Y, int rmin, int tx,
                                               float (&g)[3][4])
{
    if (!ye) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float4 v = *reinterpret_cast<const float4 *>(&s_h[c][Y - rmin][tx]);
            g[c][0] = v.x; g[c][1] = v.y; g[c][2] = v.z; g[c][3] = v.w;
        }
        return;
    }
    const int r0 = ye[0] - rmin, size = ye[1];
    const float *w = reinterpret_cast<const float *>(ye + 2);
    const int n_unfused = ((size - 1) >> 2) << 2;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float4 v = *reinterpret_cast<const float4 *>(&s_h[c][r0][tx]);
        const float wy0 = __ldg(w);
        float a0 = __fmul_rn(v.x, wy0), a1 = __fmul_rn(v.y, wy0), a2 = __fmul_rn(v.z, wy0), a3 = __fmul_rn(v.w, wy0);
        for (int r = 1; r < size; ++r) {
            v = *reinterpret_cast<const float4 *>(&s_h[c][r0 + r][tx]);
            const float wr = __ldg(w + r);
            a0 = aa_step(a0, v.x, wr, r, n_unfused); a1 = aa_step(a1, v.y, wr, r, n_unfused);
            a2 = aa_step(a2, v.z, wr, r, n_unfused); a3 = aa_step(a3, v.w, wr, r, n_unfused);
        }
        g[c][0] = a0; g[c][1] = a1; g[c][2] = a2; g[c][3] = a3;
    }
}

}  // namespace bgd
