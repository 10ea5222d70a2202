// BG-mix blend: fused uint8 -> fp32 normalise / crop / blend / layout kernel.
//
// Replaces BackgroundMixDataset._mix_background (libs/loader/comix_loader.py:138-145) together
// with the bg_pipeline's RandomCrop + Normalize (:72-75) and the foreground's mmaction
// Normalize + FormatShape (config ..._bgmix_plus_randAug.py:137-138) for a whole batch.
//
// Arithmetic: blend.cuh.
//
// HBM-bound elementwise work: per clip T*H*W*3 bytes in (uint8), H*W*3 floats of background,
// T*H*W*3 floats out.  One thread owns 4 adjacent pixels of one sample: it keeps the 12
// pre-scaled background values in registers and walks the T frames, reading 12 foreground bytes
// (3 x 32-bit, coalesced) and writing three 16-byte vectors (one per channel plane) per frame.
#include "blend.cuh"

namespace bgd {
namespace {

constexpr int kThreads = 256;
// 8 CTAs per SM (32 registers) and 4 frames of loads in flight per thread: the kernel waits on memory
// (long-scoreboard stalls), so occupancy beats registers here (profiles/r1_bgmix_unroll_occupancy.txt)
constexpr int kMixUnroll = 4;
constexpr int kMixMinBlocks = 8;

struct MixParams {
    const uint8_t *fg;
    const void *pool;
    int64_t T, H, W, P, Hb, Wb;
    BlendParams blend;
};

template <typename PoolT>
__device__ __forceinline__ float load_bg(const PoolT *p) { return (float)__ldg(p); }

// OutT: float, __nv_bfloat16 or __half.  IL (BGD_LAYOUT_NTHWC): a pixel's 3 channels are adjacent in the output, so the
// 4 pixels of a thread make 12 consecutive values (store_out12) instead of three 4-value runs, one per channel plane.
template <typename PoolT, int PX, typename OutT, bool IL>
__global__ void __launch_bounds__(kThreads, kMixMinBlocks) bgmix_kernel(const MixParams prm)
{
    const BlendParams &bp = prm.blend;
    __shared__ float s_lut[3 * 256];
    stage_lut<kThreads>(s_lut, bp.lut, threadIdx.x);
    __syncthreads();

    const int64_t b = blockIdx.y;
    const int64_t HW = prm.H * prm.W;
    const int64_t p0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * PX;   // first pixel
    if (p0 >= HW) return;

    const bool apply = bp.apply[b] != 0;
    float g[3][PX];                                  // bg * alpha, per channel / pixel
    if (apply) {
        const int64_t y = p0 / prm.W, x = p0 - y * prm.W;
        int64_t idx = bp.bg_idx[b];
        idx = idx < 0 ? 0 : (idx >= prm.P ? prm.P - 1 : idx);               // host validates; clamp = no OOB
        const int64_t top = min(max((int64_t)bp.top[b], (int64_t)0), prm.Hb - prm.H);     // host validates; clamp = no OOB
        const int64_t left = min(max((int64_t)bp.left[b], (int64_t)0), prm.Wb - prm.W);
        const PoolT *pb = static_cast<const PoolT *>(prm.pool) + ((idx * 3) * prm.Hb + (top + y)) * prm.Wb + left + x;
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int i = 0; i < PX; ++i) g[c][i] = scaled_bg(bp, c, load_bg(pb + (int64_t)c * prm.Hb * prm.Wb + i));
    }

    const uint8_t *fg = prm.fg + (b * prm.T * HW + p0) * 3;
    OutT *out = static_cast<OutT *>(bp.out) + b * prm.T * 3 * HW + (IL ? 3 * p0 : p0);

#pragma unroll kMixUnroll
    for (int64_t t = 0; t < prm.T; ++t) blend_frame<PX, IL>(fg + t * HW * 3, s_lut, apply, g, bp, out + t * bp.out_stride_t);
}

// Foreground already normalised (fp32 [B][T][3][H][W], what the reference's pipeline hands to
// _mix_background): out = fg * f32(1 - alpha) + bg_norm * f32(alpha), or a plain copy when the
// sample is not mixed.  One thread: VEC adjacent pixels of one (sample, channel), all T frames.
template <typename PoolT, int VEC>
__global__ void __launch_bounds__(kThreads) bgmix_normfg_kernel(const MixParams prm, const float *__restrict__ fgn)
{
    const BlendParams &bp = prm.blend;
    const int64_t b = blockIdx.z, c = blockIdx.y;
    const int64_t HW = prm.H * prm.W;
    const int64_t p0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
    if (p0 >= HW) return;
    const bool apply = bp.apply[b] != 0;
    float g[VEC];
    if (apply) {
        const int64_t y = p0 / prm.W, x = p0 - y * prm.W;
        int64_t idx = bp.bg_idx[b];
        idx = idx < 0 ? 0 : (idx >= prm.P ? prm.P - 1 : idx);               // host validates; clamp = no OOB
        const int64_t top = min(max((int64_t)bp.top[b], (int64_t)0), prm.Hb - prm.H);
        const int64_t left = min(max((int64_t)bp.left[b], (int64_t)0), prm.Wb - prm.W);
        const PoolT *pb = static_cast<const PoolT *>(prm.pool) + ((idx * 3 + c) * prm.Hb + (top + y)) * prm.Wb + left + x;
#pragma unroll
        for (int i = 0; i < VEC; ++i) g[i] = scaled_bg(bp, c, load_bg(pb + i));
    }
    const float *src = fgn + (b * prm.T * 3 + c) * HW + p0;
    float *out = static_cast<float *>(bp.out) + b * prm.T * 3 * HW + c * bp.out_stride_c + p0;
    for (int64_t t = 0; t < prm.T; ++t) {
        float f[VEC];
        if (VEC == 4) {
            const float4 v = __ldcs(reinterpret_cast<const float4 *>(src + t * 3 * HW));
            f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
        } else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) f[i] = __ldcs(src + t * 3 * HW + i);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) f[i] = mix(f[i], g[i], apply, bp.w_fg);
        float *dst = out + t * bp.out_stride_t;
        if (VEC == 4) __stcs(reinterpret_cast<float4 *>(dst), make_float4(f[0], f[1], f[2], f[3]));
        else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) __stcs(dst + i, f[i]);
        }
    }
}

__global__ void sum_f32_kernel(const float *__restrict__ x, int64_t n, double *__restrict__ out)
{
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        acc += (double)x[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double s[32];
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        acc = threadIdx.x < (blockDim.x >> 5) ? s[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (threadIdx.x == 0) atomicAdd(out, acc);
    }
}

}  // namespace

int launch_bgmix(const uint8_t *d_fg, const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W, const void *d_pool,
                 bool pool_is_u8, int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                 const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                 const float *d_lut, const float *h_mean, const float *h_std, double alpha, int layout,
                 int out_dtype, void *d_out, cudaStream_t stream)
{
    MixParams prm{};
    if (int rc = fill_blend("bgmix", B, T, H, W, P, d_bg_idx, d_top, d_left, d_apply, d_lut, h_mean, h_std, alpha, layout,
                            out_dtype, d_out, &prm.blend))
        return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_fg_norm && (!d_fg || !d_lut)) return fail(BGD_ERR_INVALID, "bgmix: null pointer");
    if (P > 0 && !d_pool) return fail(BGD_ERR_INVALID, "bgmix: null pool argument");
    if (P > 0 && (Hb < H || Wb < W))
        return fail(BGD_ERR_INVALID, "bgmix: crop %lldx%lld larger than pool image %lldx%lld",
                    (long long)H, (long long)W, (long long)Hb, (long long)Wb);
    if (d_fg_norm && (layout == BGD_LAYOUT_NTHWC || out_dtype != BGD_OUT_F32))
        return fail(BGD_ERR_INVALID, "bgmix: a normalised foreground blends to fp32 NTCHW / NCTHW only");
    prm.fg = d_fg; prm.pool = d_pool;
    prm.T = T; prm.H = H; prm.W = W; prm.P = P > 0 ? P : 1; prm.Hb = Hb; prm.Wb = Wb;
    const int64_t HW = H * W;

    if (d_fg_norm) {
        const bool v4 = (W % 4 == 0) && reinterpret_cast<uintptr_t>(d_fg_norm) % 16 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0;
        const int vw = v4 ? 4 : 1;
        dim3 grid((unsigned)((HW / vw + kThreads - 1) / kThreads), 3u, (unsigned)B);
        if (pool_is_u8) {
            if (v4) bgmix_normfg_kernel<uint8_t, 4><<<grid, kThreads, 0, stream>>>(prm, d_fg_norm);
            else    bgmix_normfg_kernel<uint8_t, 1><<<grid, kThreads, 0, stream>>>(prm, d_fg_norm);
        } else {
            if (v4) bgmix_normfg_kernel<float, 4><<<grid, kThreads, 0, stream>>>(prm, d_fg_norm);
            else    bgmix_normfg_kernel<float, 1><<<grid, kThreads, 0, stream>>>(prm, d_fg_norm);
        }
        count_launch();
        BGD_CUDA_TRY(cudaGetLastError());
        return BGD_OK;
    }
    // 4-pixel vectors: W % 4 == 0 keeps every thread's first pixel a multiple of 4, so its stores stay aligned
    const bool vec = (W % 4 == 0) && (reinterpret_cast<uintptr_t>(d_fg) % 4 == 0) &&
                     (reinterpret_cast<uintptr_t>(d_out) % (4 * out_elem_bytes(out_dtype)) == 0);
    const int px = vec ? 4 : 1;
    dim3 grid((unsigned)((HW / px + kThreads - 1) / kThreads), (unsigned)B);
    dispatch_out(out_dtype, layout, [&](auto o, auto il) {
        using OutT = typename decltype(o)::type;
        constexpr bool IL = decltype(il)::value;
        if (pool_is_u8) {
            if (vec) bgmix_kernel<uint8_t, 4, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
            else     bgmix_kernel<uint8_t, 1, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
        } else {
            if (vec) bgmix_kernel<float, 4, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
            else     bgmix_kernel<float, 1, OutT, IL><<<grid, kThreads, 0, stream>>>(prm);
        }
    });
    count_launch();
    BGD_CUDA_TRY(cudaGetLastError());
    return BGD_OK;
}

int launch_sum_f32(const float *d_x, int64_t n, double *d_sum, cudaStream_t stream)
{
    BGD_CUDA_TRY(cudaMemsetAsync(d_sum, 0, sizeof(double), stream));
    if (n > 0) {
        int blocks = (int)((n + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        sum_f32_kernel<<<blocks, 256, 0, stream>>>(d_x, n, d_sum);
        count_launch();
        BGD_CUDA_TRY(cudaGetLastError());
    }
    return BGD_OK;
}

}  // namespace bgd
