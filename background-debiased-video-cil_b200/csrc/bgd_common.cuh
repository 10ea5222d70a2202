// Shared helpers for libbgdebias_b200.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <type_traits>

#include "bgdebias.h"

namespace bgd {

// ---- output element types of the batch blends (BGD_OUT_*) --------------------------------
// The blend is computed in fp32 exactly as before; a 16-bit output is that value converted once, round to nearest even
// (what torch's .to(torch.bfloat16) / .to(torch.float16) does).  Stores stream past L2 (st.global.cs) like the fp32 ones.
template <typename OutT> struct OutElem;
template <> struct OutElem<__nv_bfloat16> {
    static __device__ __forceinline__ unsigned short one(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
    static __device__ __forceinline__ uint32_t two(float lo, float hi)
    {
        const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
        return (uint32_t)__bfloat16_as_ushort(p.x) | ((uint32_t)__bfloat16_as_ushort(p.y) << 16);
    }
};
template <> struct OutElem<__half> {
    static __device__ __forceinline__ unsigned short one(float v) { return __half_as_ushort(__float2half_rn(v)); }
    static __device__ __forceinline__ uint32_t two(float lo, float hi)
    {
        const __half2 p = __floats2half2_rn(lo, hi);
        return (uint32_t)__half_as_ushort(p.x) | ((uint32_t)__half_as_ushort(p.y) << 16);
    }
};

// one value
__device__ __forceinline__ void store_out(float *p, float v) { __stcs(p, v); }
template <typename OutT> __device__ __forceinline__ void store_out(OutT *p, float v)
{
    __stcs(reinterpret_cast<unsigned short *>(p), OutElem<OutT>::one(v));
}

// 4 consecutive values of one channel plane (p 16-byte aligned for fp32, 8-byte for 16-bit)
__device__ __forceinline__ void store_out4(float *p, const float (&r)[4])
{
    __stcs(reinterpret_cast<float4 *>(p), make_float4(r[0], r[1], r[2], r[3]));
}
template <typename OutT> __device__ __forceinline__ void store_out4(OutT *p, const float (&r)[4])
{
    __stcs(reinterpret_cast<uint2 *>(p), make_uint2(OutElem<OutT>::two(r[0], r[1]), OutElem<OutT>::two(r[2], r[3])));
}

// 4 pixels x 3 channels, channel innermost (BGD_LAYOUT_NTHWC): the 12 values r[c][i] go to p[3 * i + c], as three 16-byte
// (fp32) or 8-byte (16-bit) stores; p is aligned like store_out4's when the first pixel's index is a multiple of 4
__device__ __forceinline__ void store_out12(float *p, const float (&r)[3][4])
{
    __stcs(reinterpret_cast<float4 *>(p), make_float4(r[0][0], r[1][0], r[2][0], r[0][1]));
    __stcs(reinterpret_cast<float4 *>(p + 4), make_float4(r[1][1], r[2][1], r[0][2], r[1][2]));
    __stcs(reinterpret_cast<float4 *>(p + 8), make_float4(r[2][2], r[0][3], r[1][3], r[2][3]));
}
template <typename OutT> __device__ __forceinline__ void store_out12(OutT *p, const float (&r)[3][4])
{
    using E = OutElem<OutT>;
    uint2 *q = reinterpret_cast<uint2 *>(p);
    __stcs(q, make_uint2(E::two(r[0][0], r[1][0]), E::two(r[2][0], r[0][1])));
    __stcs(q + 1, make_uint2(E::two(r[1][1], r[2][1]), E::two(r[0][2], r[1][2])));
    __stcs(q + 2, make_uint2(E::two(r[2][2], r[0][3]), E::two(r[1][3], r[2][3])));
}

inline int out_elem_bytes(int out_dtype)           // 0 = not a BGD_OUT_* value
{
    return out_dtype == BGD_OUT_F32 ? 4 : (out_dtype == BGD_OUT_BF16 || out_dtype == BGD_OUT_F16) ? 2 : 0;
}

// Calls f(Tag<OutT>{}, std::integral_constant<bool, INTERLEAVED>{}) for the output type and layout of a launch, so that a
// launcher instantiates its kernel once per (type, planar / interleaved); NTCHW and NCTHW are both planar (strides).
// The caller has validated both arguments.
template <typename T> struct Tag { using type = T; };
template <typename F> void dispatch_out(int out_dtype, int layout, F &&f)
{
    const bool il = layout == BGD_LAYOUT_NTHWC;
    if (out_dtype == BGD_OUT_BF16) {
        if (il) f(Tag<__nv_bfloat16>{}, std::true_type{}); else f(Tag<__nv_bfloat16>{}, std::false_type{});
    } else if (out_dtype == BGD_OUT_F16) {
        if (il) f(Tag<__half>{}, std::true_type{}); else f(Tag<__half>{}, std::false_type{});
    } else {
        if (il) f(Tag<float>{}, std::true_type{}); else f(Tag<float>{}, std::false_type{});
    }
}

// ---- error state (per host thread) -------------------------------------------------------
std::string &last_error_ref();
int fail(int code, const char *fmt, ...);

#define BGD_CUDA_TRY(expr)                                                                  \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return ::bgd::fail(BGD_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                \
                               cudaGetErrorString(_e), __FILE__, __LINE__);                 \
    } while (0)

// ---- launch accounting -------------------------------------------------------------------
extern std::atomic<int64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- device properties, cached per device ------------------------------------------------
struct DeviceProps {
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    int64_t smem_optin = 0;
    int64_t smem_per_sm = 0;
    int64_t total_mem = 0;
    bool ok = false;
};
int get_device_props(int device, DeviceProps *out);   // returns bgd_status
int current_device_props(DeviceProps *out);

// ---- kernels' host launchers (defined in the .cu files) ----------------------------------
int launch_median_swar(const uint8_t *d_frames, const int64_t *d_row0, const int32_t *d_T,
                       int64_t V, int64_t N, uint8_t *d_out, int T_max, cudaStream_t stream);

struct MedianWork;  // planner output, see median_bitsliced.cu
int median_bitsliced_varlen(const uint8_t *d_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                            uint8_t *d_out, cudaStream_t stream);
bool median_bitsliced_supports(int64_t T_max, int64_t N);
// `subset` (may be null = all V videos): the n_subset video indices this call reduces; the others are left alone
int median_tma_varlen(const uint8_t *d_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                           uint8_t *d_out, bool use_ldsm, const int64_t *subset, int64_t n_subset, cudaStream_t stream);
bool median_tma_supports(int64_t T_max, int64_t N);

int launch_bgmix(const uint8_t *d_fg, const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W, const void *d_pool,
                 bool pool_is_u8, int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                 const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                 const float *d_lut, const float *h_mean, const float *h_std, double alpha,
                 int layout, int out_dtype, void *d_out, cudaStream_t stream);
int launch_resize_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H, int64_t W,
                     uint8_t *d_out, cudaStream_t stream);
int launch_resize_blend(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H,
                        int64_t W, const void *d_pool, bool pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                        const float *d_lut, const float *h_mean, const float *h_std, double alpha, int layout, int out_dtype,
                        void *d_out, cudaStream_t stream);
int aa_resize_table(int64_t in_size, int64_t out_size, int32_t *K_out, int32_t *words, int64_t cap_words);
int launch_bgmix_ragged(const uint8_t *d_fg, const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W,
                        const uint8_t *d_pool, const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                        const float *d_lut, const float *h_mean, const float *h_std, double alpha, int layout, int out_dtype,
                        void *d_out, cudaStream_t stream);
int launch_aa_resize(const uint8_t *d_img, const bgd_ragged_slot *h_slot, const int32_t *d_tables, float *d_out, cudaStream_t stream);
int launch_resized_crop_aa(const uint8_t *d_src, int64_t src_bytes, const bgd_crop_desc *h_desc, int64_t n,
                           const int32_t *d_tables, int64_t table_words, int64_t out_h, int64_t out_w, float *d_out,
                           cudaStream_t stream);
int launch_sum_f32(const float *d_x, int64_t n, double *d_sum, cudaStream_t stream);
int launch_nan_reduce(const float *d_frames, int64_t T, int64_t N, int avg_method, int zero_is_missing, uint8_t *d_out_u8,
                      float *d_out_f32, cudaStream_t stream);
int launch_cutmix(const uint8_t *d_actor, const uint8_t *d_mask, const uint8_t *d_scene, int64_t n, uint8_t *d_out,
                  unsigned long long *d_mask_sum, cudaStream_t stream);
int launch_ragged_pack(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_segments, int64_t n, uint8_t *d_out,
                       int64_t out_bytes, cudaStream_t stream);
int launch_ragged_gather(const uint8_t *const *d_bases, const int64_t *h_base_bytes, int64_t n_bases, const int64_t *h_segments,
                         int64_t n, uint8_t *d_out, int64_t out_bytes, cudaStream_t stream);
int launch_nan_reduce_varlen(const float *d_frames, const int64_t *h_offsets, int64_t V, int64_t N, int avg_method,
                             int zero_is_missing, uint8_t *d_out_u8, float *d_out_f32, cudaStream_t stream);

// ---- small device workspace that survives across calls (per device, per host thread) -----
// Used for the per-launch tables (row offsets, frame counts, tile lists).  Stream-ordered use:
// `acquire` hands out the next of kRing slots (pinned mirror + device buffer + event), the caller
// uploads with cudaMemcpyAsync from the mirror, launches on the same stream and calls `release`,
// which records the slot's event there.  A slot is reused kRing calls later, so a call never waits
// for the kernels of the calls just before it: the host only blocks when kRing calls are in flight.
struct Workspace {
    static constexpr int kRing = 16;
    struct Slot {
        void *d_ptr = nullptr;
        void *h_pinned = nullptr;
        size_t bytes = 0;
        cudaEvent_t ready = nullptr;
        bool in_flight = false;
    };
    Slot ring[kRing];
    int next = 0, cur = 0;
    int device = -1;
    // the slot handed out by the last acquire()
    void *d_ptr = nullptr;
    void *h_pinned = nullptr;
    size_t bytes = 0;
    int acquire(size_t need);                 // ensures capacity and that the slot's previous user is done
    int release(cudaStream_t stream);         // records the slot's event on the stream that used it
    void free_all();
    ~Workspace() { free_all(); }
};
Workspace &thread_workspace();

}  // namespace bgd
