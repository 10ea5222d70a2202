// BG-mix over a RAGGED uint8 background pool: Resize(bg_resize) + RandomCrop + Normalize + blend in one launch.
//
// Replaces, for a whole batch,
//   libs/loader/comix_loader.py:72-75    bg_pipeline = Compose([Resize(bg_resize), RandomCrop(bg_crop_size), Normalize])
//   libs/loader/comix_loader.py:126-136  _get_bg_image: a pool image (:129-131) OR a random frame of a random video (:133-136)
//   libs/loader/comix_loader.py:138-145  _mix_background
// for pools whose images differ in size (HMDB51 / Sth-Sth-v2 backgrounds have mixed widths, the reference resizes and
// crops every background at its own size), for pools too large to keep resized in fp32 (Sth-Sth-v2: ~68 GB as uint8,
// ~308 GB as resized fp32), and for the random-frame mode, whose "pool" is the handful of frames a batch drew.
//
// The pool is one byte buffer; image s is planar uint8 [3][h][w] (what torchvision.io.read_image returns) at
// slots[s].offset.  Resize is torchvision's: float CHW tensor -> torch.nn.functional.interpolate(mode="bilinear",
// antialias=True, align_corners=False) -> ATen's separable CPU kernel (aten/src/ATen/native/cpu/UpSampleKernel.cpp,
// third-party, not in the reference tree).  Its arithmetic, restated here and pinned bit for bit against the installed
// torch 2.11 / torchvision 0.26 by the tests:
//   per axis and output index i (all in float unless noted):
//     scale   = float(in) / out;  support = scale >= 1 ? scale : 1;  invscale = scale >= 1 ? 1 / scale : 1
//     center  = float(scale * (i + 0.5))                                  (product in double)
//     min     = max(int64(center - support + 0.5), 0);  size = min(int64(center + support + 0.5), in) - min
//     w_j     = tri((j + min - center + 0.5) * invscale) / sum_j tri(..),   tri(x) = |x| < 1 ? 1 - |x| : 0
//   horizontal pass first, then vertical, each output  acc = v_0 * w_0;  acc += v_j * w_j  for j = 1 .. size-1  where the
//   first 4 * floor((size - 1) / 4) of those steps round the product and the sum separately and the remaining
//   (size - 1) % 4 steps are fused multiply-adds -- what GCC 13 makes of that loop in the AVX-512 build of ATen (4-wide
//   in-order vector part + scalar epilogue with contraction); an axis whose size does not change is skipped.
// The weights depend on (in, out, i) only; bgd_aa_resize_table evaluates them on the host, once per distinct size.
//
// Blend arithmetic as in bgmix.cu (each operation rounded, no contraction):
//   fg = lut[c][x];  bg = (resized - mean[c]) / std[c];  out = fg * f32(1 - alpha) + bg * f32(alpha)
#include "aa_resample.cuh"
#include "bgd_common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace bgd {
namespace {

constexpr int kThreads = 256;

struct RaggedParams {
    const uint8_t *fg;
    const float *fgn;                 // normalised foreground instead of fg + lut (may be null)
    const uint8_t *pool;
    const bgd_ragged_slot *slots;
    const int32_t *tables;
    const int32_t *bg_idx, *top, *left;
    const uint8_t *apply;
    const float *lut;
    void *out;                        // float, or OutT of the uint8-foreground kernels
    int64_t T, H, W, P;
    float mean[3], std[3];
    float w_fg, w_bg;
    int64_t out_stride_t, out_stride_c;   // in elements (NTHWC: 3 * H * W, 1)
};

__device__ __forceinline__ bgd_ragged_slot load_slot(const RaggedParams &prm, int64_t b, int &top, int &left)
{
    int64_t idx = prm.bg_idx[b];
    idx = idx < 0 ? 0 : (idx >= prm.P ? prm.P - 1 : idx);                    // host validates; clamp = no OOB
    const bgd_ragged_slot s = prm.slots[idx];
    top = min(max(prm.top[b], 0), max(s.Hb - (int)prm.H, 0));
    left = min(max(prm.left[b], 0), max(s.Wb - (int)prm.W, 0));
    return s;
}

// uint8 foreground [B][T][H][W][3]: one thread owns PX adjacent pixels of one sample for all T frames (as bgmix_kernel,
// whose OutT / IL this kernel and the tile kernel share)
template <int PX, typename OutT, bool IL>
__global__ void __launch_bounds__(kThreads) bgmix_ragged_kernel(const RaggedParams prm)
{
    __shared__ float s_lut[3 * 256];
    for (int i = threadIdx.x; i < 3 * 256; i += kThreads) s_lut[i] = __ldg(prm.lut + i);
    __syncthreads();

    const int64_t b = blockIdx.y;
    const int64_t HW = prm.H * prm.W;
    const int64_t p0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * PX;
    if (p0 >= HW) return;

    const bool apply = prm.apply[b] != 0;
    float g[3][PX];
    if (apply) {
        int top, left;
        const bgd_ragged_slot s = load_slot(prm, b, top, left);
        const int y = (int)(p0 / prm.W), x = (int)(p0 - (int64_t)y * prm.W);
        const uint8_t *img = prm.pool + s.offset;
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int i = 0; i < PX; ++i) {
                const float raw = aa_sample(img + (int64_t)c * s.h * s.w, s.w, prm.tables, s.xtab, s.kx, s.ytab, s.ky, top + y,
                                            left + x + i);
                g[c][i] = __fmul_rn(__fdiv_rn(__fsub_rn(raw, prm.mean[c]), prm.std[c]), prm.w_bg);
            }
    }

    const uint8_t *fg = prm.fg + (b * prm.T * HW + p0) * 3;
    OutT *out = static_cast<OutT *>(prm.out) + b * prm.T * 3 * HW + (IL ? 3 * p0 : p0);
#pragma unroll 2
    for (int64_t t = 0; t < prm.T; ++t) {
        uint8_t px[3 * PX];
        if (PX == 4) {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(fg + t * HW * 3);
            const uint32_t w0 = __ldcs(src), w1 = __ldcs(src + 1), w2 = __ldcs(src + 2);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                px[k] = (w0 >> (8 * k)) & 0xFF;
                px[4 + k] = (w1 >> (8 * k)) & 0xFF;
                px[8 + k] = (w2 >> (8 * k)) & 0xFF;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 3 * PX; ++k) px[k] = __ldcs(fg + t * HW * 3 + k);
        }
        float r[3][PX];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
            for (int i = 0; i < PX; ++i) {
                const float f = s_lut[c * 256 + px[i * 3 + c]];
                r[c][i] = apply ? __fadd_rn(__fmul_rn(f, prm.w_fg), g[c][i]) : f;
            }
            OutT *dst = out + t * prm.out_stride_t + c * prm.out_stride_c;
            if constexpr (PX == 4 && !IL) store_out4(dst, r[c]);
            else if constexpr (PX == 1) store_out(dst, r[c][0]);
        }
        if constexpr (PX == 4 && IL) store_out12(out + t * prm.out_stride_t, r);
    }
}

// ---- tiled form of the same blend (the product path when W % 4 == 0) -------------------------------------------------
// A CTA owns a 32 x 32 tile of output pixels of one sample.  The separable Resize is done the way ATen does it, once per
// tile instead of once per output value: the horizontal pass of every source row the tile's 32 output rows touch (32 rows
// when up-scaling 240 -> 256) goes to shared memory -- a thread keeps ONE output column, so its column entry (first tap,
// weights) is read once -- then every thread runs the vertical pass for its own 4 adjacent pixels, normalises, scales and
// walks the T frames like bgmix_kernel.  About half the instructions of the per-value form (1.55 k against 3.0 k per thread
// for 240x320 / 240x427 backgrounds).  Tiles whose source-row span does not fit the buffer (strong down-scaling) fall back
// to the per-value evaluation, tile by tile.
constexpr int kTile = 32;                 // output rows and columns per CTA
constexpr int kMaxSrcRows = 48;           // source rows of one tile kept in shared memory
#ifndef BGD_RAGGED_MINBLOCKS
#define BGD_RAGGED_MINBLOCKS 6
#endif

template <typename OutT, bool IL>
__global__ void __launch_bounds__(kThreads, BGD_RAGGED_MINBLOCKS) bgmix_ragged_tile_kernel(const RaggedParams prm)
{
    __shared__ float s_lut[3 * 256];
    __shared__ __align__(16) float s_h[3][kMaxSrcRows][kTile];
    for (int i = threadIdx.x; i < 3 * 256; i += kThreads) s_lut[i] = __ldg(prm.lut + i);

    const int64_t b = blockIdx.z;
    const int tx0 = blockIdx.x * kTile, ty0 = blockIdx.y * kTile;
    const int ty = threadIdx.x >> 3, tx = (threadIdx.x & 7) << 2;      // this thread's row and first column inside the tile
    const int W = (int)prm.W, H = (int)prm.H;
    const bool inside = ty0 + ty < H && tx0 + tx < W;                  // W % 4 == 0: a group of 4 is inside or outside as a whole
    const bool apply = prm.apply[b] != 0;                              // uniform over the CTA

    float g[3][4];
    if (apply) {
        int top, left;
        const bgd_ragged_slot s = load_slot(prm, b, top, left);
        const uint8_t *img = prm.pool + s.offset;
        const int Y0 = top + ty0, Ylast = top + min(ty0 + kTile, H) - 1;
        int rmin, rend;
        aa_tile_rows(prm.tables, s.ytab, s.ky, Y0, Ylast, rmin, rend);
        const int nrows = rend - rmin;
        if (nrows <= kMaxSrcRows) {
            // horizontal pass: thread -> output column x of the tile, source rows r = warp, warp + 8, ...
            const int x = threadIdx.x & 31, X = left + tx0 + x, r_first = threadIdx.x >> 5;
            if (tx0 + x < W) {
                const int32_t *xe = s.xtab >= 0 ? prm.tables + s.xtab + (int64_t)X * (2 + s.kx) : nullptr;
                aa_tile_hpass<kThreads / 32>(s_h, img, (int64_t)s.h * s.w, s.w, xe, X, x, rmin, r_first, nrows);
            }
            __syncthreads();
            if (inside) {
                const int Y = top + ty0 + ty;
                const int32_t *ye = s.ytab >= 0 ? prm.tables + s.ytab + (int64_t)Y * (2 + s.ky) : nullptr;
                aa_tile_vpass4(s_h, ye, Y, rmin, tx, g);
            }
        } else {
            __syncthreads();
            if (inside) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        g[c][i] = aa_sample(img + (int64_t)c * s.h * s.w, s.w, prm.tables, s.xtab, s.kx, s.ytab, s.ky,
                                            top + ty0 + ty, left + tx0 + tx + i);
            }
        }
        if (inside) {
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    g[c][i] = __fmul_rn(__fdiv_rn(__fsub_rn(g[c][i], prm.mean[c]), prm.std[c]), prm.w_bg);
        }
    } else {
        __syncthreads();                                               // the table load above
    }
    if (!inside) return;

    const int64_t HW = prm.H * prm.W;
    const int64_t p0 = (int64_t)(ty0 + ty) * W + tx0 + tx;
    const uint8_t *fg = prm.fg + (b * prm.T * HW + p0) * 3;
    OutT *out = static_cast<OutT *>(prm.out) + b * prm.T * 3 * HW + (IL ? 3 * p0 : p0);
#pragma unroll 4
    for (int64_t t = 0; t < prm.T; ++t) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(fg + t * HW * 3);
        const uint32_t w0 = __ldcs(src), w1 = __ldcs(src + 1), w2 = __ldcs(src + 2);
        uint8_t px[12];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            px[k] = (w0 >> (8 * k)) & 0xFF;
            px[4 + k] = (w1 >> (8 * k)) & 0xFF;
            px[8 + k] = (w2 >> (8 * k)) & 0xFF;
        }
        float r[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float f = s_lut[c * 256 + px[i * 3 + c]];
                r[c][i] = apply ? __fadd_rn(__fmul_rn(f, prm.w_fg), g[c][i]) : f;
            }
            if constexpr (!IL) store_out4(out + t * prm.out_stride_t + c * prm.out_stride_c, r[c]);
        }
        if constexpr (IL) store_out12(out + t * prm.out_stride_t, r);
    }
}

// normalised fp32 foreground [B][T][3][H][W] (the reference's `imgs`): one thread = one pixel of one (sample, channel)
__global__ void __launch_bounds__(kThreads) bgmix_ragged_normfg_kernel(const RaggedParams prm)
{
    const int64_t b = blockIdx.z, c = blockIdx.y;
    const int64_t HW = prm.H * prm.W;
    const int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= HW) return;
    const bool apply = prm.apply[b] != 0;
    float g = 0.f;
    if (apply) {
        int top, left;
        const bgd_ragged_slot s = load_slot(prm, b, top, left);
        const int y = (int)(p / prm.W), x = (int)(p - (int64_t)y * prm.W);
        const float raw = aa_sample(prm.pool + s.offset + c * (int64_t)s.h * s.w, s.w, prm.tables, s.xtab, s.kx, s.ytab, s.ky,
                                    top + y, left + x);
        g = __fmul_rn(__fdiv_rn(__fsub_rn(raw, prm.mean[c]), prm.std[c]), prm.w_bg);
    }
    const float *src = prm.fgn + (b * prm.T * 3 + c) * HW + p;
    float *out = static_cast<float *>(prm.out) + b * prm.T * 3 * HW + c * prm.out_stride_c + p;
    for (int64_t t = 0; t < prm.T; ++t) {
        const float f = __ldcs(src + t * 3 * HW);
        __stcs(out + t * prm.out_stride_t, apply ? __fadd_rn(__fmul_rn(f, prm.w_fg), g) : f);
    }
}

// Resize alone: planar uint8 [3][h][w] -> fp32 [3][Hb][Wb]
__global__ void __launch_bounds__(kThreads) aa_resize_kernel(const uint8_t *__restrict__ img, bgd_ragged_slot s,
                                                             const int32_t *__restrict__ tables, float *__restrict__ out)
{
    const int64_t n = (int64_t)s.Hb * s.Wb;
    const int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= n) return;
    const int c = blockIdx.y, Y = (int)(p / s.Wb), X = (int)(p - (int64_t)Y * s.Wb);
    out[c * n + p] = aa_sample(img + (int64_t)c * s.h * s.w, s.w, tables, s.xtab, s.kx, s.ytab, s.ky, Y, X);
}

}  // namespace

// ---- host: ATen's weight computation (see the header of this file) ---------------------------------------------------
// Expression types follow UpSampleKernel.cpp (HelperInterpBase::_compute_indices_min_size_weights_aa with scalar_t = float)
// operation by operation: what is float there is float here, what is promoted to double there is double here.
static int aa_taps(int64_t in_size, int64_t out_size, float *scale_out, float *support_out)
{
    const float scale = static_cast<float>(in_size) / out_size;
    const int interp_size = 2;
    const float support = (scale >= 1.0) ? (interp_size * 0.5) * scale : interp_size * 0.5;
    *scale_out = scale;
    *support_out = support;
    return (int)std::ceil(support) * 2 + 1;
}

int aa_resize_table(int64_t in_size, int64_t out_size, int32_t *K_out, int32_t *words, int64_t cap_words)
{
    if (in_size <= 0 || out_size <= 0 || in_size >= (1 << 24) || out_size >= (1 << 24))
        return fail(BGD_ERR_INVALID, "aa_resize_table: sizes must be in 1 .. 2^24 (in %lld, out %lld)", (long long)in_size, (long long)out_size);
    float scale, support;
    const int K = aa_taps(in_size, out_size, &scale, &support);
    if (K_out) *K_out = K;
    if (!words) return BGD_OK;
    if (cap_words < out_size * (2 + K)) return fail(BGD_ERR_INVALID, "aa_resize_table: buffer of %lld words, %lld needed", (long long)cap_words, (long long)(out_size * (2 + K)));
    const int64_t max_interp_size = K;
    for (int64_t i = 0; i < out_size; ++i) {
        int32_t *ent = words + i * (2 + K);
        float *wt = reinterpret_cast<float *>(ent + 2);
        float center = scale * (i + 0.5);
        float total_w = 0.0;
        float invscale = (scale >= 1.0) ? 1.0 / scale : 1.0;
        int64_t xmin = std::max(static_cast<int64_t>(center - support + 0.5), static_cast<int64_t>(0));
        int64_t xsize = std::min(static_cast<int64_t>(center + support + 0.5), in_size) - xmin;
        xsize = std::min(std::max(xsize, static_cast<int64_t>(0)), max_interp_size);
        int64_t j = 0;
        for (; j < xsize; j++) {
            float x = (j + xmin - center + 0.5) * invscale;
            x = std::abs(x);
            float w = (x < 1.0) ? (float)(1.0 - x) : 0.0f;
            wt[j] = w;
            total_w += w;
        }
        if (total_w != 0.0) {
            for (j = 0; j < xsize; j++) wt[j] /= total_w;
        }
        for (; j < max_interp_size; j++) wt[j] = 0.0f;
        ent[0] = (int32_t)xmin;
        ent[1] = (int32_t)xsize;
    }
    return BGD_OK;
}

static int fill_params(RaggedParams &prm, int64_t B, int64_t T, int64_t H, int64_t W, const uint8_t *d_pool,
                       const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables, const int32_t *d_bg_idx,
                       const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply, const float *h_mean,
                       const float *h_std, double alpha, int layout, int out_dtype, void *d_out)
{
    if (B < 0 || T < 0 || H < 0 || W < 0 || P < 0) return fail(BGD_ERR_INVALID, "bgmix (ragged): negative size");
    if (!d_out || !d_apply) return fail(BGD_ERR_INVALID, "bgmix (ragged): null pointer");
    if (!h_mean || !h_std) return fail(BGD_ERR_INVALID, "bgmix (ragged): null mean/std");
    if (P > 0 && (!d_pool || !d_slots || !d_bg_idx || !d_top || !d_left)) return fail(BGD_ERR_INVALID, "bgmix (ragged): null pool argument");
    if (layout != BGD_LAYOUT_NTCHW && layout != BGD_LAYOUT_NCTHW && layout != BGD_LAYOUT_NTHWC)
        return fail(BGD_ERR_INVALID, "bgmix (ragged): unknown layout %d", layout);
    if (!out_elem_bytes(out_dtype)) return fail(BGD_ERR_INVALID, "bgmix (ragged): unknown output type %d", out_dtype);
    if (B > 65535) return fail(BGD_ERR_INVALID, "bgmix (ragged): batch larger than 65535");
    if (H >= (1 << 24) || W >= (1 << 24)) return fail(BGD_ERR_INVALID, "bgmix (ragged): crop too large");
    prm.pool = d_pool; prm.slots = d_slots; prm.tables = d_tables; prm.bg_idx = d_bg_idx; prm.top = d_top; prm.left = d_left;
    prm.apply = d_apply; prm.out = d_out;
    prm.T = T; prm.H = H; prm.W = W; prm.P = P > 0 ? P : 1;
    for (int c = 0; c < 3; ++c) { prm.mean[c] = h_mean[c]; prm.std[c] = h_std[c]; }
    prm.w_fg = (float)(1.0 - alpha);
    prm.w_bg = (float)alpha;
    const int64_t HW = H * W;
    if (layout == BGD_LAYOUT_NTCHW)      { prm.out_stride_t = 3 * HW; prm.out_stride_c = HW; }
    else if (layout == BGD_LAYOUT_NCTHW) { prm.out_stride_t = HW;     prm.out_stride_c = T * HW; }
    else                                 { prm.out_stride_t = 3 * HW; prm.out_stride_c = 1; }
    return BGD_OK;
}

int launch_bgmix_ragged(const uint8_t *d_fg, const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W,
                        const uint8_t *d_pool, const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                        const float *d_lut, const float *h_mean, const float *h_std, double alpha, int layout, int out_dtype,
                        void *d_out, cudaStream_t stream)
{
    RaggedParams prm{};
    if (int rc = fill_params(prm, B, T, H, W, d_pool, d_slots, P, d_tables, d_bg_idx, d_top, d_left, d_apply, h_mean, h_std, alpha,
                             layout, out_dtype, d_out))
        return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_fg && !d_fg_norm) return fail(BGD_ERR_INVALID, "bgmix (ragged): null foreground");
    if (d_fg && !d_lut) return fail(BGD_ERR_INVALID, "bgmix (ragged): null table");
    prm.fg = d_fg; prm.fgn = d_fg_norm; prm.lut = d_lut;
    const int64_t HW = H * W;
    if (d_fg_norm) {
        if (layout == BGD_LAYOUT_NTHWC || out_dtype != BGD_OUT_F32)
            return fail(BGD_ERR_INVALID, "bgmix (ragged): a normalised foreground blends to fp32 NTCHW / NCTHW only");
        dim3 grid((unsigned)((HW + kThreads - 1) / kThreads), 3u, (unsigned)B);
        bgmix_ragged_normfg_kernel<<<grid, kThreads, 0, stream>>>(prm);
    } else {
        const bool vec = (W % 4 == 0) && (reinterpret_cast<uintptr_t>(d_fg) % 4 == 0) &&
                         (reinterpret_cast<uintptr_t>(d_out) % (4 * out_elem_bytes(out_dtype)) == 0);
        const int px = vec ? 4 : 1;
        dim3 grid((unsigned)((HW / px + kThreads - 1) / kThreads), (unsigned)B);
        static const bool per_value = getenv("BGD_RAGGED_PER_VALUE") != nullptr;     // differential testing of the two forms
        dim3 tgrid((unsigned)((W + kTile - 1) / kTile), (unsigned)((H + kTile - 1) / kTile), (unsigned)B);
        if (vec && !per_value && tgrid.y > 65535) return fail(BGD_ERR_INVALID, "bgmix (ragged): crop too tall");
        dispatch_out(out_dtype, layout, [&](auto o, auto il) {
            using OutT = typename decltype(o)::type;
            constexpr bool IL = decltype(il)::value;
            if (vec && !per_value) bgmix_ragged_tile_kernel<OutT, IL><<<tgrid, kThreads, 0, stream>>>(prm);
            else if (vec)          bgmix_ragged_kernel<4, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
            else                   bgmix_ragged_kernel<1, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
        });
    }
    count_launch();
    BGD_CUDA_TRY(cudaGetLastError());
    return BGD_OK;
}

int launch_aa_resize(const uint8_t *d_img, const bgd_ragged_slot *h_slot, const int32_t *d_tables, float *d_out, cudaStream_t stream)
{
    if (!d_img || !h_slot || !d_out) return fail(BGD_ERR_INVALID, "aa_resize: null pointer");
    const bgd_ragged_slot s = *h_slot;
    if (s.h <= 0 || s.w <= 0 || s.Hb <= 0 || s.Wb <= 0) return fail(BGD_ERR_INVALID, "aa_resize: empty image");
    if ((s.xtab >= 0 || s.ytab >= 0) && !d_tables) return fail(BGD_ERR_INVALID, "aa_resize: null tables");
    if ((s.xtab < 0 && s.Wb != s.w) || (s.ytab < 0 && s.Hb != s.h)) return fail(BGD_ERR_INVALID, "aa_resize: an axis without a table must keep its size");
    const int64_t n = (int64_t)s.Hb * s.Wb;
    dim3 grid((unsigned)((n + kThreads - 1) / kThreads), 3u);
    aa_resize_kernel<<<grid, kThreads, 0, stream>>>(d_img + s.offset, s, d_tables, d_out);
    count_launch();
    BGD_CUDA_TRY(cudaGetLastError());
    return BGD_OK;
}

}  // namespace bgd
