// Foreground pipeline tail on the GPU: mmaction Resize((W,H), keep_ratio=False) -> Normalize -> FormatShape -> BG-mix blend.
//
// Replaces, for a whole batch in one launch, the tail of the training pipeline
// (configs/ucf101/bgmix_plus_randAug/..._bgmix_plus_randAug.py:136-138) that produces the `imgs` handed to
// BackgroundMixDataset._mix_background (libs/loader/comix_loader.py:138-145), and that blend.  The Resize itself lives in
// third-party code absent from the reference tree: mmaction2 0.x `Resize` -> mmcv 1.x `imresize` -> `cv2.resize(img, (W, H),
// interpolation=cv2.INTER_LINEAR)` (no versions pinned by the reference).  The arithmetic below restates OpenCV's 8-bit
// linear resize (fixed-point, 11-bit coefficients) and is checked bit for bit against cv2.resize by the tests:
//     scale   = 1 / (double(dst) / src)
//     f       = float((d + 0.5) * scale - 0.5);  s = floor(f);  f -= s
//     columns: s < 0 -> (s, f) = (0, 0);  s >= src-1 -> (s, f) = (src-1, 0);  rows: no change to f, both taps clamped into the image
//     c0, c1  = round_half_even((1 - f) * 2048), round_half_even(f * 2048)
//     row     = p[s] * c0 + p[s+1] * c1                                         (horizontal pass, 32-bit)
//     out     = (((b0 * (row0 >> 4)) >> 16) + ((b1 * (row1 >> 4)) >> 16) + 2) >> 2
//
// Source clips are ragged (MultiScaleCrop yields a different crop size per sample, config :129-135): one packed uint8 buffer
// plus a per-clip table (byte offset of the crop's first pixel, crop height/width, row and frame strides), so a crop can also
// be addressed inside a full decoded frame without a host-side copy.
//
// The coefficients depend on (source size, destination size, index) only: the host evaluates them once per distinct size
// (float/double arithmetic exactly as above) into small tables that travel with the per-clip table.  A CTA owns a 32x8 tile of
// output pixels of one clip, one thread per pixel: it reads its column entry and its row entry, then walks the T frames of the
// clip.  Per frame it reads the two 6-byte tap pairs (RGB of two adjacent source pixels) with aligned 32-bit loads and a
// funnel shift, so neighbouring lanes share cache lines, pairs left/right bytes with byte permutes and multiplies with dp2a;
// the 3 results go through the normalisation table and the blend of bgmix.cu and are stored as one coalesced 128-byte row
// per warp and channel plane.
#include "bgd_common.cuh"

#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

namespace bgd {
namespace {

#ifndef BGD_RESIZE_TILEH
#define BGD_RESIZE_TILEH 8
#endif
constexpr int kTileW = 32, kTileH = BGD_RESIZE_TILEH, kThreads = kTileW * kTileH;
#ifndef BGD_RESIZE_UNROLL
#define BGD_RESIZE_UNROLL 1
#endif
#ifndef BGD_RESIZE_MINBLOCKS
#define BGD_RESIZE_MINBLOCKS 8
#endif
constexpr int kFrameUnroll = BGD_RESIZE_UNROLL, kBlendMinBlocks = BGD_RESIZE_MINBLOCKS;

struct Coef {                  // one per destination column / row, built on the host
    int32_t i0, i1;            // columns: byte offset of the left tap in its row, -;  rows: the two source rows (clamped)
    int32_t c0, c1;            // 11-bit weights of the two taps
};

struct ClipGeom {              // one per clip, built on the host
    int64_t offset;            // bytes from d_src to the crop's first pixel of frame 0
    int64_t row_stride, frame_stride;
    int32_t xtab, ytab;        // first entry of the clip's column / row coefficients in the Coef array
};

struct TailParams {
    const uint8_t *src;
    const ClipGeom *geom;
    const Coef *coef;
    // blend half (unused by the uint8 resize kernel)
    const void *pool;
    const int32_t *bg_idx, *top, *left;
    const uint8_t *apply;
    const float *lut;
    void *out;                 // OutT of resize_blend_kernel
    uint8_t *out_u8;
    int64_t T, H, W, P, Hb, Wb;
    float mean[3], std[3];
    float w_fg, w_bg;
    int64_t out_stride_t, out_stride_c;
};

struct Taps {
    int64_t row0, row1;        // byte offsets (from src) of the left tap in the two source rows, frame 0
    uint32_t a01;              // column weights, a0 | a1 << 16
    uint32_t b0, b1;           // row weights
};

__device__ __forceinline__ Taps make_taps(const TailParams &prm, const ClipGeom &g, int x, int y)
{
    const int4 cx = __ldg(reinterpret_cast<const int4 *>(prm.coef + g.xtab + x));
    const int4 cy = __ldg(reinterpret_cast<const int4 *>(prm.coef + g.ytab + y));
    Taps t;
    t.a01 = (uint32_t)cx.z | ((uint32_t)cx.w << 16);
    t.b0 = (uint32_t)cy.z; t.b1 = (uint32_t)cy.w;
    t.row0 = g.offset + (int64_t)cy.x * g.row_stride + cx.x;
    t.row1 = g.offset + (int64_t)cy.y * g.row_stride + cx.x;
    return t;
}

// Horizontal pass of one source row for the three channels: h[c] = left[c] * a0 + right[c] * a1 (x2048).
// The six tap bytes (RGB of the left pixel, RGB of the right pixel) start `sh` bits into the aligned word *w:
// aligned 32-bit loads + funnel shift bring them to (lo, hi), two byte permutes pair left/right per channel and a 16x8-bit
// dot product (dp2a) does multiply and add.
__device__ __forceinline__ void hpass(const uint32_t *w, uint32_t sh, uint32_t a01, uint32_t (&h)[3])
{
    const uint32_t q0 = __ldg(w), q1 = __ldg(w + 1);
    const uint32_t q2 = sh == 24u ? __ldg(w + 2) : 0u;          // bytes 4..5 reach the third word only at offset 3
    const uint32_t lo = __funnelshift_r(q0, q1, sh);            // l0 l1 l2 r0
    const uint32_t hi = __funnelshift_r(q1, q2, sh);            // r1 r2 .  .
    const uint32_t p01 = __byte_perm(lo, hi, 0x4130);           // l0 r0 l1 r1
    const uint32_t p2 = __byte_perm(lo, hi, 0x0052);            // l2 r2 .  .
    h[0] = __dp2a_lo(a01, p01, 0u);
    h[1] = __dp2a_hi(a01, p01, 0u);
    h[2] = __dp2a_lo(a01, p2, 0u);
}

// Vertical pass + rounding: (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, always within 0..255
// (weights sum to at most 2049/2048 and every shift truncates).  The +2 rides on the first product as 2 << 16.
__device__ __forceinline__ uint32_t vpass(uint32_t h0, uint32_t h1, const Taps &t)
{
    const uint32_t v = ((t.b0 * (h0 >> 4) + 0x20000u) >> 16) + ((t.b1 * (h1 >> 4)) >> 16);
    return v >> 2;
}

// Walks the T frames of one output pixel: emit(f, c, value) receives the resized uint8 value of channel c in frame f.
// ALIGNED (frame stride a multiple of 4 bytes, every clip packed by ops.pack_clips with even sizes is): the word pointers
// advance by a constant and the funnel-shift counts never change; otherwise both are recomputed per frame.
template <bool ALIGNED, typename Emit>
__device__ __forceinline__ void for_each_frame(const TailParams &prm, const ClipGeom &g, const Taps &t, Emit emit)
{
    const uint32_t *base = reinterpret_cast<const uint32_t *>(prm.src);
    if (ALIGNED) {
        const uint32_t *w0 = base + (t.row0 >> 2), *w1 = base + (t.row1 >> 2);
        const uint32_t s0 = ((uint32_t)t.row0 & 3u) * 8u, s1 = ((uint32_t)t.row1 & 3u) * 8u;
        const int64_t step = g.frame_stride >> 2;
#pragma unroll kFrameUnroll
        for (int64_t f = 0; f < prm.T; ++f, w0 += step, w1 += step) {
            uint32_t h0[3], h1[3];
            hpass(w0, s0, t.a01, h0);
            hpass(w1, s1, t.a01, h1);
#pragma unroll
            for (int c = 0; c < 3; ++c) emit(f, c, vpass(h0[c], h1[c], t));
        }
    } else {
        int64_t at0 = t.row0, at1 = t.row1;
        for (int64_t f = 0; f < prm.T; ++f, at0 += g.frame_stride, at1 += g.frame_stride) {
            uint32_t h0[3], h1[3];
            hpass(base + (at0 >> 2), ((uint32_t)at0 & 3u) * 8u, t.a01, h0);
            hpass(base + (at1 >> 2), ((uint32_t)at1 & 3u) * 8u, t.a01, h1);
#pragma unroll
            for (int c = 0; c < 3; ++c) emit(f, c, vpass(h0[c], h1[c], t));
        }
    }
}

__global__ void __launch_bounds__(kThreads) resize_u8_kernel(const TailParams prm)
{
    const int64_t b = blockIdx.z;
    const int x = blockIdx.x * kTileW + threadIdx.x, y = blockIdx.y * kTileH + threadIdx.y;
    if (x >= prm.W || y >= prm.H) return;
    const ClipGeom g = prm.geom[b];
    const Taps t = make_taps(prm, g, x, y);
    const int64_t HW = prm.H * prm.W, frame = HW * 3;
    uint8_t *out = prm.out_u8 + (b * prm.T * HW + (int64_t)y * prm.W + x) * 3;
    auto emit = [&](int64_t f, int c, uint32_t v) { out[f * frame + c] = (uint8_t)v; };
    if ((g.frame_stride & 3) == 0) for_each_frame<true>(prm, g, t, emit);
    else                           for_each_frame<false>(prm, g, t, emit);
}

// OutT: float, __nv_bfloat16 or __half.  IL (BGD_LAYOUT_NTHWC): the pixel's 3 channels are adjacent in the output; a
// lane then stores 3 consecutive values per frame and a warp still covers whole 32-byte sectors (scalar stores).
template <typename PoolT, typename OutT, bool IL>
__global__ void __launch_bounds__(kThreads, kBlendMinBlocks) resize_blend_kernel(const TailParams prm)
{
    __shared__ float s_lut[3 * 256];
    for (int i = threadIdx.y * kTileW + threadIdx.x; i < 3 * 256; i += kThreads) s_lut[i] = __ldg(prm.lut + i);
    __syncthreads();

    const int64_t b = blockIdx.z;
    const int x = blockIdx.x * kTileW + threadIdx.x, y = blockIdx.y * kTileH + threadIdx.y;
    if (x >= prm.W || y >= prm.H) return;
    const ClipGeom g = prm.geom[b];
    const Taps t = make_taps(prm, g, x, y);

    const bool apply = prm.apply[b] != 0;
    float bgw[3] = {0.f, 0.f, 0.f};                  // normalised background * alpha
    if (apply) {
        // one pool image has fewer than 2^31 elements (checked on the host): only the image index needs 64 bits
        const int Hb = (int)prm.Hb, Wb = (int)prm.Wb, plane = Hb * Wb;
        int64_t idx = prm.bg_idx[b];
        idx = idx < 0 ? 0 : (idx >= prm.P ? prm.P - 1 : idx);               // host validates; clamp = no OOB
        const int top = min(max(prm.top[b], 0), Hb - (int)prm.H);
        const int left = min(max(prm.left[b], 0), Wb - (int)prm.W);
        const PoolT *pb = static_cast<const PoolT *>(prm.pool) + idx * (3 * plane) + ((top + y) * Wb + left + x);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float raw = (float)__ldg(pb + c * plane);
            bgw[c] = __fmul_rn(__fdiv_rn(__fsub_rn(raw, prm.mean[c]), prm.std[c]), prm.w_bg);
        }
    }

    const int64_t HW = prm.H * prm.W;
    OutT *out = IL ? static_cast<OutT *>(prm.out) + b * prm.T * 3 * HW + 3 * ((int64_t)y * prm.W + x)
                   : static_cast<OutT *>(prm.out) + b * prm.T * 3 * HW + (int64_t)y * prm.W + x;
    const int64_t st = prm.out_stride_t, sc = prm.out_stride_c;
    const float w_fg = prm.w_fg;
    auto emit = [&](int64_t f, int c, uint32_t v) {
        const float n = s_lut[c * 256 + v];
        store_out(out + f * st + c * sc, apply ? __fadd_rn(__fmul_rn(n, w_fg), bgw[c]) : n);
    };
    if ((g.frame_stride & 3) == 0) for_each_frame<true>(prm, g, t, emit);
    else                           for_each_frame<false>(prm, g, t, emit);
}

// ---- host: coefficient tables ------------------------------------------------------------------------------------------------
// cv::resize (INTER_LINEAR, 8-bit): inv_scale = dst / src, scale = 1 / inv_scale (doubles); per destination index d:
// f = float((d + 0.5) * scale - 0.5), s = floor(f), f -= s.  Columns snap taps outside the image onto the border pixel with
// weights (1, 0); rows keep their fraction and clamp the two tap rows.  Weights: saturate_cast<short>(c * 2048), i.e. the
// float product (exact, a power of two) rounded half to even.  volatile keeps the compiler from fusing or reassociating.
void fill_coefs(int src, int dst, bool columns, Coef *out)
{
    const volatile double inv_scale = (double)dst / (double)src;
    const volatile double scale = 1.0 / inv_scale;
    for (int d = 0; d < dst; ++d) {
        const volatile double scaled = ((double)d + 0.5) * scale;
        volatile float f = (float)(scaled - 0.5);
        int s = (int)std::floor(f);
        f = f - (float)s;
        Coef c;
        if (columns) {
            if (s < 0) { s = 0; f = 0.f; }
            if (s >= src - 1) { s = src - 1; f = 0.f; }
        }
        const volatile float one_minus = 1.f - f;
        c.c0 = (int32_t)std::nearbyint(one_minus * 2048.f);
        c.c1 = (int32_t)std::nearbyint(f * 2048.f);
        if (columns) {
            // the right tap of the last column has weight 0: read the pair one pixel to the left and swap the weights
            if (s >= src - 1 && src >= 2) { s = src - 2; c.c1 = c.c0; c.c0 = 0; }
            c.i0 = s * 3; c.i1 = 0;
        } else {
            c.i0 = std::max(0, std::min(s, src - 1));
            c.i1 = std::max(0, std::min(s + 1, src - 1));
        }
        out[d] = c;
    }
}

struct TableKey { int64_t src; bool columns; int32_t at; };

// Validates the host geometry table [B][5] = {offset, h, w, row stride, frame stride} against the buffer, builds the
// coefficient tables (one per distinct source size and axis) and uploads both: [ClipGeom x B][Coef x n].
int upload_geom(const int64_t *h_geom, int64_t B, int64_t T, int64_t H, int64_t W, int64_t src_bytes, Workspace &ws,
                TailParams *prm, cudaStream_t stream)
{
    std::vector<TableKey> tables;
    std::unordered_map<int64_t, int32_t> index;            // 2 * source size + axis -> first entry
    std::vector<int32_t> xt(B), yt(B);
    int64_t n_coef = 0;
    auto table_of = [&](int64_t src, bool columns) {
        auto it = index.find(2 * src + (columns ? 1 : 0));
        if (it != index.end()) return it->second;
        tables.push_back({src, columns, (int32_t)n_coef});
        index.emplace(2 * src + (columns ? 1 : 0), (int32_t)n_coef);
        n_coef += columns ? W : H;
        return tables.back().at;
    };
    for (int64_t b = 0; b < B; ++b) {
        const int64_t *q = h_geom + b * 5;
        const int64_t off = q[0], h = q[1], w = q[2], rs = q[3], fs = q[4];
        if (h < 1 || w < 1 || h > INT32_MAX / 4 || w > INT32_MAX / 4)
            return fail(BGD_ERR_INVALID, "resize: clip %lld has size %lldx%lld", (long long)b, (long long)h, (long long)w);
        if (off < 0 || rs < w * 3 || fs < 0)
            return fail(BGD_ERR_INVALID, "resize: clip %lld has a negative offset or a row stride below 3*w", (long long)b);
        // the kernel reads tap PAIRS: a one-pixel-wide crop reads 6 bytes per row as well
        const int64_t end = off + (T - 1) * fs + (h - 1) * rs + std::max<int64_t>(w, 2) * 3;
        if (end > src_bytes)
            return fail(BGD_ERR_INVALID, "resize: clip %lld ends at byte %lld of a %lld-byte buffer", (long long)b,
                        (long long)end, (long long)src_bytes);
        if (n_coef + H + W > INT32_MAX) return fail(BGD_ERR_INVALID, "resize: too many distinct clip sizes");
        xt[b] = table_of(w, true);
        yt[b] = table_of(h, false);
    }
    const size_t geom_bytes = (size_t)B * sizeof(ClipGeom), bytes = geom_bytes + (size_t)n_coef * sizeof(Coef);
    if (int rc = ws.acquire(bytes)) return rc;
    ClipGeom *hg = static_cast<ClipGeom *>(ws.h_pinned);
    Coef *hc = reinterpret_cast<Coef *>(static_cast<char *>(ws.h_pinned) + geom_bytes);
    for (int64_t b = 0; b < B; ++b) {
        const int64_t *q = h_geom + b * 5;
        hg[b].offset = q[0]; hg[b].row_stride = q[3]; hg[b].frame_stride = q[4];
        hg[b].xtab = xt[b]; hg[b].ytab = yt[b];
    }
    for (const TableKey &k : tables) fill_coefs((int)k.src, (int)(k.columns ? W : H), k.columns, hc + k.at);
    BGD_CUDA_TRY(cudaMemcpyAsync(ws.d_ptr, ws.h_pinned, bytes, cudaMemcpyHostToDevice, stream));
    prm->geom = static_cast<const ClipGeom *>(ws.d_ptr);
    prm->coef = reinterpret_cast<const Coef *>(static_cast<const char *>(ws.d_ptr) + geom_bytes);
    return BGD_OK;
}

int check_common(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H, int64_t W)
{
    if (B < 0 || T < 0 || H < 0 || W < 0 || src_bytes < 0) return fail(BGD_ERR_INVALID, "resize: negative size");
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;          // nothing to do: pointers may be null
    if (!d_src || !h_geom) return fail(BGD_ERR_INVALID, "resize: null pointer");
    if (reinterpret_cast<uintptr_t>(d_src) % 4 != 0 || src_bytes % 4 != 0)
        return fail(BGD_ERR_INVALID, "resize: the source buffer must be 4-byte aligned and a multiple of 4 bytes long "
                                     "(it is read with aligned 32-bit loads)");
    if (B > 65535) return fail(BGD_ERR_INVALID, "resize: batch larger than 65535");
    if (H > 65535 * kTileH || W > INT32_MAX / 4) return fail(BGD_ERR_INVALID, "resize: output size too large");
    return BGD_OK;
}

dim3 tile_grid(int64_t B, int64_t H, int64_t W)
{
    return dim3((unsigned)((W + kTileW - 1) / kTileW), (unsigned)((H + kTileH - 1) / kTileH), (unsigned)B);
}

}  // namespace

int launch_resize_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H, int64_t W,
                     uint8_t *d_out, cudaStream_t stream)
{
    if (int rc = check_common(d_src, src_bytes, h_geom, B, T, H, W)) return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_out) return fail(BGD_ERR_INVALID, "resize: null output");
    Workspace &ws = thread_workspace();
    TailParams prm{};
    if (int rc = upload_geom(h_geom, B, T, H, W, src_bytes, ws, &prm, stream)) return rc;
    prm.src = d_src; prm.out_u8 = d_out;
    prm.T = T; prm.H = H; prm.W = W;
    resize_u8_kernel<<<tile_grid(B, H, W), dim3(kTileW, kTileH), 0, stream>>>(prm);
    count_launch();
    cudaError_t e = cudaGetLastError();
    const int rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "resize_u8_kernel launch failed: %s", cudaGetErrorString(e));
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
}

int launch_resize_blend(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H,
                        int64_t W, const void *d_pool, bool pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                        const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                        const float *d_lut, const float *h_mean, const float *h_std, double alpha, int layout, int out_dtype,
                        void *d_out, cudaStream_t stream)
{
    if (int rc = check_common(d_src, src_bytes, h_geom, B, T, H, W)) return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) return BGD_OK;
    if (!d_out || !d_lut || !d_apply) return fail(BGD_ERR_INVALID, "bgmix_resize: null pointer");
    if (!h_mean || !h_std) return fail(BGD_ERR_INVALID, "bgmix_resize: null mean/std");
    if (P > 0 && (!d_pool || !d_bg_idx || !d_top || !d_left)) return fail(BGD_ERR_INVALID, "bgmix_resize: null pool argument");
    if (P > 0 && (Hb < H || Wb < W))
        return fail(BGD_ERR_INVALID, "bgmix_resize: crop %lldx%lld larger than pool image %lldx%lld", (long long)H, (long long)W,
                    (long long)Hb, (long long)Wb);
    if (P > 0 && (Hb > INT32_MAX / 4 || Wb > INT32_MAX / 4 || 3 * Hb * Wb > INT32_MAX))
        return fail(BGD_ERR_INVALID, "bgmix_resize: pool images larger than 2^31 elements");
    if (layout != BGD_LAYOUT_NTCHW && layout != BGD_LAYOUT_NCTHW && layout != BGD_LAYOUT_NTHWC)
        return fail(BGD_ERR_INVALID, "bgmix_resize: unknown layout %d", layout);
    if (!out_elem_bytes(out_dtype)) return fail(BGD_ERR_INVALID, "bgmix_resize: unknown output type %d", out_dtype);

    Workspace &ws = thread_workspace();
    TailParams prm{};
    if (int rc = upload_geom(h_geom, B, T, H, W, src_bytes, ws, &prm, stream)) return rc;
    prm.src = d_src;
    prm.pool = d_pool; prm.bg_idx = d_bg_idx; prm.top = d_top; prm.left = d_left; prm.apply = d_apply; prm.lut = d_lut;
    prm.out = d_out;
    prm.T = T; prm.H = H; prm.W = W; prm.P = P > 0 ? P : 1; prm.Hb = Hb; prm.Wb = Wb;
    for (int c = 0; c < 3; ++c) { prm.mean[c] = h_mean[c]; prm.std[c] = h_std[c]; }
    prm.w_fg = (float)(1.0 - alpha);
    prm.w_bg = (float)alpha;
    const int64_t HW = H * W;
    if (layout == BGD_LAYOUT_NTCHW)      { prm.out_stride_t = 3 * HW; prm.out_stride_c = HW; }
    else if (layout == BGD_LAYOUT_NCTHW) { prm.out_stride_t = HW;     prm.out_stride_c = T * HW; }
    else                                 { prm.out_stride_t = 3 * HW; prm.out_stride_c = 1; }
    dispatch_out(out_dtype, layout, [&](auto o, auto il) {
        using OutT = typename decltype(o)::type;
        constexpr bool IL = decltype(il)::value;
        if (pool_is_u8) resize_blend_kernel<uint8_t, OutT, IL><<<tile_grid(B, H, W), dim3(kTileW, kTileH), 0, stream>>>(prm);
        else            resize_blend_kernel<float, OutT, IL><<<tile_grid(B, H, W), dim3(kTileW, kTileH), 0, stream>>>(prm);
    });
    count_launch();
    cudaError_t e = cudaGetLastError();
    const int rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "resize_blend_kernel launch failed: %s", cudaGetErrorString(e));
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
}

}  // namespace bgd
