// The BG-mix blend epilogue shared by the dense (bgmix.cu), ragged (raggedmix.cu) and fused-resize (resize.cu) kernels.
//
// The three families differ in how they get a foreground value and a raw background value; from there on the arithmetic is
// the reference's, operation by operation, each rounded to fp32 and never contracted into an FMA:
//     fg  = lut[c][x]                       (table = cv2.subtract/cv2.multiply result per level)
//     bg  = (raw - mean[c]) / std[c]        (torchvision Normalize)
//     out = fg * f32(1 - alpha) + bg * f32(alpha)
// stored as fp32, bf16 or fp16 in NTCHW, NCTHW or NTHWC.  Those steps, the checks of their arguments and the output strides
// live here, once.  The clamps of the draws stay in the kernels: each family bounds its crop offsets differently, and a
// shared clamp of bg_idx moved ptxas's register allocation (more spills in the ragged kernels).
#pragma once

#include "bgd_common.cuh"

namespace bgd {

// The part of a blend launch's parameters every family carries; each family's struct holds one plus its own geometry.
struct BlendParams {
    const int32_t *bg_idx, *top, *left;
    const uint8_t *apply;
    const float *lut;
    void *out;                            // float, or the OutT of the kernel
    float mean[3], std[3];
    float w_fg, w_bg;
    int64_t out_stride_t, out_stride_c;   // in elements; NTCHW / NCTHW folded into strides (NTHWC: 3 * H * W, 1)
};

// Validates the output half of a blend launch (sizes, layout, output type, batch within the grid) and fills the table,
// output and strides.  An empty launch is valid with null pointers; the caller returns before launching.
inline int fill_blend_out(const char *who, int64_t B, int64_t T, int64_t H, int64_t W, const float *d_lut, int layout,
                          int out_dtype, void *d_out, BlendParams *bp)
{
    if (B < 0 || T < 0 || H < 0 || W < 0) return fail(BGD_ERR_INVALID, "%s: negative size", who);
    if (layout != BGD_LAYOUT_NTCHW && layout != BGD_LAYOUT_NCTHW && layout != BGD_LAYOUT_NTHWC)
        return fail(BGD_ERR_INVALID, "%s: unknown layout %d", who, layout);
    if (!out_elem_bytes(out_dtype)) return fail(BGD_ERR_INVALID, "%s: unknown output type %d", who, out_dtype);
    if (B > 65535) return fail(BGD_ERR_INVALID, "%s: batch larger than 65535", who);
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_out) return fail(BGD_ERR_INVALID, "%s: null pointer", who);
    bp->lut = d_lut;
    bp->out = d_out;
    const int64_t HW = H * W;
    if (layout == BGD_LAYOUT_NTCHW)      { bp->out_stride_t = 3 * HW; bp->out_stride_c = HW; }
    else if (layout == BGD_LAYOUT_NCTHW) { bp->out_stride_t = HW;     bp->out_stride_c = T * HW; }
    else                                 { bp->out_stride_t = 3 * HW; bp->out_stride_c = 1; }
    return BGD_OK;
}

// fill_blend_out, then the draws (read when P > 0) and the background's normalisation and weights.
inline int fill_blend(const char *who, int64_t B, int64_t T, int64_t H, int64_t W, int64_t P, const int32_t *d_bg_idx,
                      const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply, const float *d_lut,
                      const float *h_mean, const float *h_std, double alpha, int layout, int out_dtype, void *d_out,
                      BlendParams *bp)
{
    if (P < 0) return fail(BGD_ERR_INVALID, "%s: negative size", who);
    if (int rc = fill_blend_out(who, B, T, H, W, d_lut, layout, out_dtype, d_out, bp)) return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_apply) return fail(BGD_ERR_INVALID, "%s: null pointer", who);
    if (!h_mean || !h_std) return fail(BGD_ERR_INVALID, "%s: null mean/std", who);
    if (P > 0 && (!d_bg_idx || !d_top || !d_left)) return fail(BGD_ERR_INVALID, "%s: null pool argument", who);
    bp->bg_idx = d_bg_idx; bp->top = d_top; bp->left = d_left; bp->apply = d_apply;
    for (int c = 0; c < 3; ++c) { bp->mean[c] = h_mean[c]; bp->std[c] = h_std[c]; }
    bp->w_fg = (float)(1.0 - alpha);      // python: (1 - alpha) in double, then tensor * scalar rounds to fp32
    bp->w_bg = (float)alpha;
    return BGD_OK;
}

// The normalisation table into shared memory, NTHREADS threads numbered tid; the caller synchronises before reading it.
template <int NTHREADS>
__device__ __forceinline__ void stage_lut(float *s_lut, const float *lut, int tid)
{
    for (int i = tid; i < 3 * 256; i += NTHREADS) s_lut[i] = __ldg(lut + i);
}

// bg * f32(alpha) for a raw background value of channel c
__device__ __forceinline__ float scaled_bg(const BlendParams &bp, int64_t c, float raw)
{
    return __fmul_rn(__fdiv_rn(__fsub_rn(raw, bp.mean[c]), bp.std[c]), bp.w_bg);
}

// the blend of one value: f is the normalised foreground, g = scaled_bg(..); a sample that is not mixed keeps f
__device__ __forceinline__ float mix(float f, float g, bool apply, float w_fg)
{
    return apply ? __fadd_rn(__fmul_rn(f, w_fg), g) : f;
}

// One frame of PX (1 or 4) adjacent pixels of a uint8 foreground [..][H][W][3]: fg is the first pixel's byte, out its first
// output value in this frame.  PX = 4 reads the 12 bytes as 3 streaming 32-bit loads (fg 4-byte aligned) and stores three
// 4-value runs, one per channel plane, or with IL (BGD_LAYOUT_NTHWC) 12 consecutive values (store_out12).
template <int PX, bool IL, typename OutT>
__device__ __forceinline__ void blend_frame(const uint8_t *fg, const float *s_lut, bool apply, const float (&g)[3][PX],
                                            const BlendParams &bp, OutT *out)
{
    uint8_t px[3 * PX];
    if (PX == 4) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(fg);
        const uint32_t w0 = __ldcs(src), w1 = __ldcs(src + 1), w2 = __ldcs(src + 2);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            px[k] = (w0 >> (8 * k)) & 0xFF;
            px[4 + k] = (w1 >> (8 * k)) & 0xFF;
            px[8 + k] = (w2 >> (8 * k)) & 0xFF;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 3 * PX; ++k) px[k] = __ldcs(fg + k);
    }
    float r[3][PX];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int i = 0; i < PX; ++i) r[c][i] = mix(s_lut[c * 256 + px[i * 3 + c]], g[c][i], apply, bp.w_fg);
        OutT *dst = out + c * bp.out_stride_c;
        if constexpr (PX == 4 && !IL) store_out4(dst, r[c]);
        else if constexpr (PX == 1) store_out(dst, r[c][0]);
    }
    if constexpr (PX == 4 && IL) store_out12(out, r);
}

}  // namespace bgd
