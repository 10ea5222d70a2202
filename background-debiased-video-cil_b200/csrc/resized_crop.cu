// RandomResizedCrop(size) of many frames in one launch (the simulated-camera-motion background extraction).
//
// Replaces, for every frame of a batch of frame folders,
//   cil_tools/extract_background.py:81     cam_motion_pipeline = Compose([RandomResizedCrop(size=100)])
//   cil_tools/extract_background.py:89-90  frame = cam_motion_pipeline(read_image(f).float()).permute(1, 2, 0)
// RandomResizedCrop draws (top, left, h, w) from the torch RNG (replayed on the host, extract_background.crop_draws) and
// returns torchvision.transforms.functional.resized_crop(img, top, left, h, w, size, bilinear, antialias=True): the
// window img[:, top:top+h, left:left+w] through the antialiased bilinear resize of ATen's separable CPU kernel, whose
// arithmetic aa_resample.cuh restates (horizontal pass, then vertical; per-axis host tables from bgd_aa_resize_table;
// an axis whose crop size equals the output size is skipped).  Cropping a uint8 frame and converting the window to
// float is the same as converting the frame first: the conversion is exact.
//
// Input: frames planar uint8 [3][H][W] (torchvision.io.read_image's layout) anywhere in one byte buffer, any sizes.
// Output: float32 [n][out_h][out_w][3], channels last -- the `.permute(1, 2, 0)` of the reference and the layout the
// NaN-masked temporal reduction reads.
//
// Form: a CTA owns a 32 x 32 tile of one frame's output (as bgmix_ragged_tile_kernel).  The horizontal pass runs once
// per source row and output column of the tile into shared memory, then every thread runs the vertical pass for its 4
// adjacent output columns.  Tiles whose source-row span does not fit the buffer (down-scaling by more than ~2.9x, i.e.
// large crops of 480p / 720p frames) evaluate each value on its own.
#include "aa_resample.cuh"
#include "bgd_common.cuh"

#include <climits>
#include <cstdlib>
#include <cstring>

namespace bgd {
namespace {

constexpr int kThreads = 256;
constexpr int kTile = 32;                 // output rows and columns per CTA
constexpr int kMaxSrcRows = 96;           // source rows of one tile in shared memory (36 KB): every crop of frames up
                                          // to ~280 rows (down-scaling up to ~2.9x) takes the tiled form
constexpr int kMinBlocks = 4;             // 64 registers: no spills (ptxas left alone picks 48 and spills)

struct CropParams {
    const uint8_t *src;
    const bgd_crop_desc *desc;            // device copy of the descriptors
    const int32_t *tables;
    float *out;
    int out_h, out_w;
    int tiles_x;
    bool vec;                             // out_w % 4 == 0 and d_out 16-byte aligned: float4 stores
};

__global__ void __launch_bounds__(kThreads, kMinBlocks) resized_crop_aa_tile_kernel(const CropParams prm)
{
    __shared__ __align__(16) float s_h[3][kMaxSrcRows][kTile];
    const int64_t f = blockIdx.x;
    const bgd_crop_desc d = prm.desc[f];
    const int tx0 = (blockIdx.y % prm.tiles_x) * kTile, ty0 = (blockIdx.y / prm.tiles_x) * kTile;
    const int ty = threadIdx.x >> 3, tx = (threadIdx.x & 7) << 2;      // this thread's row and first column inside the tile
    const int OH = prm.out_h, OW = prm.out_w;
    const bool inside = ty0 + ty < OH && tx0 + tx < OW;                // at least the first of the 4 columns is an output
    const int64_t plane = (int64_t)d.H * d.W;
    const uint8_t *org = prm.src + d.offset + (int64_t)d.top * d.W + d.left;      // crop origin in channel 0

    float g[3][4];
    const int Y0 = ty0, Ylast = min(ty0 + kTile, OH) - 1;
    int rmin, rend;
    aa_tile_rows(prm.tables, d.ytab, d.ky, Y0, Ylast, rmin, rend);
    const int nrows = rend - rmin;
    if (nrows <= kMaxSrcRows) {
        // horizontal pass: thread -> output column x of the tile, source rows r = warp, warp + 8, ...
        const int x = threadIdx.x & 31, X = tx0 + x, r_first = threadIdx.x >> 5;
        if (X < OW) {
            const int32_t *xe = d.xtab >= 0 ? prm.tables + d.xtab + (int64_t)X * (2 + d.kx) : nullptr;
            aa_tile_hpass<kThreads / 32>(s_h, org, plane, d.W, xe, X, x, rmin, r_first, nrows);
        }
        __syncthreads();
        if (!inside) return;
        const int Y = ty0 + ty;
        const int32_t *ye = d.ytab >= 0 ? prm.tables + d.ytab + (int64_t)Y * (2 + d.ky) : nullptr;
        aa_tile_vpass4(s_h, ye, Y, rmin, tx, g);                       // columns past out_w read unused shared memory
    } else {
        if (!inside) return;
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int i = 0; i < 4; ++i)
                g[c][i] = tx0 + tx + i < OW ? aa_sample(org + c * plane, d.W, prm.tables, d.xtab, d.kx, d.ytab, d.ky, ty0 + ty,
                                                        tx0 + tx + i)
                                            : 0.f;
    }

    float *dst = prm.out + ((f * OH + ty0 + ty) * OW + tx0 + tx) * 3;
    if (prm.vec) {
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        __stcs(d4 + 0, make_float4(g[0][0], g[1][0], g[2][0], g[0][1]));
        __stcs(d4 + 1, make_float4(g[1][1], g[2][1], g[0][2], g[1][2]));
        __stcs(d4 + 2, make_float4(g[2][2], g[0][3], g[1][3], g[2][3]));
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (tx0 + tx + i < OW) {
#pragma unroll
                for (int c = 0; c < 3; ++c) __stcs(dst + i * 3 + c, g[c][i]);
            }
    }
}

int check_desc(const bgd_crop_desc &d, int64_t i, int64_t src_bytes, int64_t table_words, int64_t out_h, int64_t out_w)
{
    if (d.H < 1 || d.W < 1) return fail(BGD_ERR_INVALID, "resized_crop: frame %lld has size %dx%d", (long long)i, d.H, d.W);
    if (d.offset < 0 || d.offset > src_bytes || 3 * (int64_t)d.H * d.W > src_bytes - d.offset)
        return fail(BGD_ERR_INVALID, "resized_crop: frame %lld (%d x %d x 3 bytes at offset %lld) is not inside the %lld-byte buffer",
                    (long long)i, d.H, d.W, (long long)d.offset, (long long)src_bytes);
    if (d.top < 0 || d.left < 0 || d.h < 1 || d.w < 1 || d.h > d.H - d.top || d.w > d.W - d.left)
        return fail(BGD_ERR_INVALID, "resized_crop: crop (top %d, left %d, %d x %d) of frame %lld is not inside its %d x %d frame",
                    d.top, d.left, d.h, d.w, (long long)i, d.H, d.W);
    const struct { int32_t tab, taps, in; int64_t out; const char *axis; } ax[2] = {{d.xtab, d.kx, d.w, out_w, "x"},
                                                                                    {d.ytab, d.ky, d.h, out_h, "y"}};
    for (const auto &a : ax) {
        if (a.tab < 0) {
            if (a.tab != -1 || a.in != a.out)
                return fail(BGD_ERR_INVALID, "resized_crop: frame %lld: the %s axis has no table but its crop size %d differs from "
                            "the output size %lld", (long long)i, a.axis, a.in, (long long)a.out);
            continue;
        }
        int32_t taps = 0;
        if (int rc = aa_resize_table(a.in, a.out, &taps, nullptr, 0)) return rc;
        if (a.taps != taps)
            return fail(BGD_ERR_INVALID, "resized_crop: frame %lld: %s table has %d taps, bgd_aa_resize_table(%d, %lld) has %d",
                        (long long)i, a.axis, a.taps, a.in, (long long)a.out, taps);
        if ((int64_t)a.tab + a.out * (2 + a.taps) > table_words)
            return fail(BGD_ERR_INVALID, "resized_crop: frame %lld: %s table at word %d runs past the %lld-word table buffer",
                        (long long)i, a.axis, a.tab, (long long)table_words);
    }
    return BGD_OK;
}

}  // namespace

int launch_resized_crop_aa(const uint8_t *d_src, int64_t src_bytes, const bgd_crop_desc *h_desc, int64_t n,
                           const int32_t *d_tables, int64_t table_words, int64_t out_h, int64_t out_w, float *d_out,
                           cudaStream_t stream)
{
    if (n < 0 || src_bytes < 0 || table_words < 0 || out_h < 0 || out_w < 0)
        return fail(BGD_ERR_INVALID, "resized_crop: negative size");
    if (out_h == 0 || out_w == 0 || out_h > 65535 * kTile || out_w > 65535 * kTile)
        return fail(BGD_ERR_INVALID, "resized_crop: output size %lld x %lld out of range", (long long)out_h, (long long)out_w);
    const int64_t tiles_x = (out_w + kTile - 1) / kTile, tiles = tiles_x * ((out_h + kTile - 1) / kTile);
    if (tiles > 65535) return fail(BGD_ERR_INVALID, "resized_crop: output of %lld tiles, at most 65535", (long long)tiles);
    if (n > INT32_MAX) return fail(BGD_ERR_INVALID, "resized_crop: %lld frames in one launch, at most 2^31 - 1", (long long)n);
    if (n == 0) return BGD_OK;
    if (!d_src || !h_desc || !d_out) return fail(BGD_ERR_INVALID, "resized_crop: null pointer");
    bool any_table = false;
    for (int64_t i = 0; i < n; ++i) {
        if (int rc = check_desc(h_desc[i], i, src_bytes, table_words, out_h, out_w)) return rc;
        any_table |= h_desc[i].xtab >= 0 || h_desc[i].ytab >= 0;
    }
    if (any_table && !d_tables) return fail(BGD_ERR_INVALID, "resized_crop: null tables");

    Workspace &ws = thread_workspace();
    const size_t bytes = (size_t)n * sizeof(bgd_crop_desc);
    if (int rc = ws.acquire(bytes)) return rc;
    std::memcpy(ws.h_pinned, h_desc, bytes);
    cudaError_t e = cudaMemcpyAsync(ws.d_ptr, ws.h_pinned, bytes, cudaMemcpyHostToDevice, stream);
    int rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "resized_crop: descriptor upload failed: %s", cudaGetErrorString(e));
    if (!rc) {
        CropParams prm{};
        prm.src = d_src; prm.desc = static_cast<const bgd_crop_desc *>(ws.d_ptr); prm.tables = d_tables; prm.out = d_out;
        prm.out_h = (int)out_h; prm.out_w = (int)out_w; prm.tiles_x = (int)tiles_x;
        prm.vec = out_w % 4 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0;
        resized_crop_aa_tile_kernel<<<dim3((unsigned)n, (unsigned)tiles), kThreads, 0, stream>>>(prm);
        count_launch();
        e = cudaGetLastError();
        rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "resized_crop_aa_tile_kernel launch failed: %s", cudaGetErrorString(e));
    }
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
}

}  // namespace bgd
