// Batched ragged gather: the owner side of the sharded-pool exchange (pool.ShardedPool.fetch).
//
// A rank that owns a shard of the background pool packs, for every peer, the whole native images that peer's batch drew into
// one send buffer, ordered by destination rank and then by the peer's request order; one all_to_all_single then delivers each
// peer its chunk.  This replaces, for the owned images of a whole batch, the per-sample background read of the reference
// (libs/loader/comix_loader.py:126-131: bg_files[bg_idx] -> read_image), which there happens once per mixed sample.
//
// The copy is a table of segments {src_offset, dst_offset, bytes}.  One CTA copies one chunk of kChunk bytes of one segment:
// grid = (chunks of the largest segment) x segments, so a batch of ~128 images of ~300 KB puts ~640 CTAs on the 148 SMs.
// Both ends of every segment are 16-byte aligned (RaggedPool.append starts every image on a 16-byte boundary, the pack
// layout pads every image to 16 bytes), so the body moves uint4 vectors: kUnroll loads in flight per thread, then streaming
// stores (the send buffer is read once, by the network, never by this SM again).  The last 0..15 bytes of a segment whose
// size is not a multiple of 16 are copied byte by byte.
#include "bgd_common.cuh"

#include <algorithm>

namespace bgd {
namespace {

constexpr int kThreads = 256, kUnroll = 4;
constexpr int64_t kChunk = (int64_t)kThreads * kUnroll * 16 * 4;       // 64 KB of one segment per CTA

struct PackSeg { int64_t src, dst, bytes; };

__global__ void __launch_bounds__(kThreads) ragged_pack_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                               const PackSeg *__restrict__ segs)
{
    const PackSeg s = segs[blockIdx.y];
    const int64_t begin = (int64_t)blockIdx.x * kChunk;
    if (begin >= s.bytes) return;
    const int64_t end = min(begin + kChunk, s.bytes);
    const int64_t n_vec = (end - begin) >> 4;
    const uint4 *in = reinterpret_cast<const uint4 *>(src + s.src + begin) + threadIdx.x;
    uint4 *out = reinterpret_cast<uint4 *>(dst + s.dst + begin) + threadIdx.x;
    int i = threadIdx.x;                                       // < kChunk / 16 vectors: 32 bits suffice
    const int nv = (int)n_vec;
    for (; i + (kUnroll - 1) * kThreads < nv; i += kUnroll * kThreads, in += kUnroll * kThreads, out += kUnroll * kThreads) {
        uint4 v[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) v[u] = __ldcs(in + u * kThreads);
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) __stcs(out + u * kThreads, v[u]);
    }
    for (; i < nv; i += kThreads, in += kThreads, out += kThreads) __stcs(out, __ldcs(in));
    const int64_t tail = begin + (n_vec << 4);                 // only the segment's last chunk has one
    if (threadIdx.x < end - tail) dst[s.dst + tail + threadIdx.x] = src[s.src + tail + threadIdx.x];
}

}  // namespace

int launch_ragged_pack(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_segments, int64_t n, uint8_t *d_out,
                       int64_t out_bytes, cudaStream_t stream)
{
    if (n < 0 || src_bytes < 0 || out_bytes < 0) return fail(BGD_ERR_INVALID, "ragged_pack: negative size");
    if (n == 0) return BGD_OK;                                          // nothing to copy: no launch
    if (!h_segments) return fail(BGD_ERR_INVALID, "ragged_pack: null segment table");
    if (n > 65535) return fail(BGD_ERR_INVALID, "ragged_pack: %lld segments, at most 65535 per call", (long long)n);
    int64_t max_bytes = 0;
    for (int64_t k = 0; k < n; ++k) {
        const int64_t so = h_segments[3 * k], d = h_segments[3 * k + 1], b = h_segments[3 * k + 2];
        if (so < 0 || d < 0 || b < 0)
            return fail(BGD_ERR_INVALID, "ragged_pack: segment %lld has a negative offset or size", (long long)k);
        if ((so | d) & 15)
            return fail(BGD_ERR_INVALID, "ragged_pack: segment %lld is not 16-byte aligned (src %lld, dst %lld)", (long long)k,
                        (long long)so, (long long)d);
        if (b > src_bytes - so)
            return fail(BGD_ERR_INVALID, "ragged_pack: segment %lld reads bytes %lld..%lld of a %lld-byte pool", (long long)k,
                        (long long)so, (long long)(so + b), (long long)src_bytes);
        if (b > out_bytes - d)
            return fail(BGD_ERR_INVALID, "ragged_pack: segment %lld writes bytes %lld..%lld of a %lld-byte output", (long long)k,
                        (long long)d, (long long)(d + b), (long long)out_bytes);
        max_bytes = std::max(max_bytes, b);
    }
    if (max_bytes == 0) return BGD_OK;                                  // only empty segments
    if (!d_src || !d_out) return fail(BGD_ERR_INVALID, "ragged_pack: null buffer");
    if ((reinterpret_cast<uintptr_t>(d_src) | reinterpret_cast<uintptr_t>(d_out)) & 15)
        return fail(BGD_ERR_INVALID, "ragged_pack: the pool and the output must be 16-byte aligned");

    Workspace &ws = thread_workspace();
    const size_t bytes = (size_t)n * sizeof(PackSeg);
    if (int rc = ws.acquire(bytes)) return rc;
    PackSeg *hs = static_cast<PackSeg *>(ws.h_pinned);
    for (int64_t k = 0; k < n; ++k) hs[k] = PackSeg{h_segments[3 * k], h_segments[3 * k + 1], h_segments[3 * k + 2]};
    BGD_CUDA_TRY(cudaMemcpyAsync(ws.d_ptr, ws.h_pinned, bytes, cudaMemcpyHostToDevice, stream));
    const dim3 grid((unsigned)((max_bytes + kChunk - 1) / kChunk), (unsigned)n);
    ragged_pack_kernel<<<grid, kThreads, 0, stream>>>(d_src, d_out, static_cast<const PackSeg *>(ws.d_ptr));
    count_launch();
    cudaError_t e = cudaGetLastError();
    const int rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "ragged_pack_kernel launch failed: %s", cudaGetErrorString(e));
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
}

}  // namespace bgd
