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
//
// ragged_gather_kernel is the same copy with many sources: the receiving side of pool.PeerPool.gather.  Each rank's shard is
// mapped into every other rank once (cudaIpcOpenMemHandle), so a rank reads the images its batch drew straight from their
// owners' HBM over NVLink into its per-batch pool; a segment {source, src_offset, dst_offset, bytes} names the owner by its
// row of a device table of base pointers.  Both kernels instantiate one body, templated on how a segment's source is found.
#include "bgd_common.cuh"

#include <algorithm>

namespace bgd {
namespace {

constexpr int kThreads = 256, kUnroll = 4;
constexpr int64_t kChunk = (int64_t)kThreads * kUnroll * 16 * 4;       // 64 KB of one segment per CTA

struct PackSeg { int64_t src, dst, bytes; };
struct GatherSeg { int64_t src, dst, bytes, source; };

// where a segment's bytes come from: one pool (ragged_pack) or a row of a table of (peer-mapped) base pointers
struct OnePool {
    const uint8_t *base;
    using Seg = PackSeg;
    __device__ const uint8_t *from(const Seg &s) const { return base + s.src; }
};
struct BaseTable {
    const uint8_t *const *bases;
    using Seg = GatherSeg;
    __device__ const uint8_t *from(const Seg &s) const { return bases[s.source] + s.src; }
};

template <class Source>
__device__ __forceinline__ void ragged_copy(Source source, uint8_t *__restrict__ dst, const typename Source::Seg *__restrict__ segs)
{
    const typename Source::Seg s = segs[blockIdx.y];
    const int64_t begin = (int64_t)blockIdx.x * kChunk;
    if (begin >= s.bytes) return;
    const uint8_t *src = source.from(s);
    const int64_t end = min(begin + kChunk, s.bytes);
    const int64_t n_vec = (end - begin) >> 4;
    const uint4 *in = reinterpret_cast<const uint4 *>(src + begin) + threadIdx.x;
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
    if (threadIdx.x < end - tail) dst[s.dst + tail + threadIdx.x] = src[tail + threadIdx.x];
}

__global__ void __launch_bounds__(kThreads) ragged_pack_kernel(OnePool source, uint8_t *__restrict__ dst,
                                                               const PackSeg *__restrict__ segs)
{
    ragged_copy(source, dst, segs);
}

__global__ void __launch_bounds__(kThreads) ragged_gather_kernel(BaseTable source, uint8_t *__restrict__ dst,
                                                                 const GatherSeg *__restrict__ segs)
{
    ragged_copy(source, dst, segs);
}

// Fills the validated table (`fill(Seg *)`) in the per-thread workspace ring, uploads it on `stream` and launches
// grid = chunks of the largest segment x segments.
template <class Source, class Fill>
int launch_ragged_copy(const char *name, void (*kernel)(Source, uint8_t *, const typename Source::Seg *), Source source,
                       Fill fill, int64_t n, int64_t max_bytes, uint8_t *d_out, cudaStream_t stream)
{
    using Seg = typename Source::Seg;
    Workspace &ws = thread_workspace();
    const size_t bytes = (size_t)n * sizeof(Seg);
    if (int rc = ws.acquire(bytes)) return rc;
    fill(static_cast<Seg *>(ws.h_pinned));
    BGD_CUDA_TRY(cudaMemcpyAsync(ws.d_ptr, ws.h_pinned, bytes, cudaMemcpyHostToDevice, stream));
    const dim3 grid((unsigned)((max_bytes + kChunk - 1) / kChunk), (unsigned)n);
    kernel<<<grid, kThreads, 0, stream>>>(source, d_out, static_cast<const Seg *>(ws.d_ptr));
    count_launch();
    cudaError_t e = cudaGetLastError();
    const int rc = e == cudaSuccess ? BGD_OK : fail(BGD_ERR_CUDA, "%s launch failed: %s", name, cudaGetErrorString(e));
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
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
    auto fill = [&](PackSeg *t) {
        for (int64_t k = 0; k < n; ++k) t[k] = PackSeg{h_segments[3 * k], h_segments[3 * k + 1], h_segments[3 * k + 2]};
    };
    return launch_ragged_copy("ragged_pack_kernel", ragged_pack_kernel, OnePool{d_src}, fill, n, max_bytes, d_out, stream);
}

int launch_ragged_gather(const uint8_t *const *d_bases, const int64_t *h_base_bytes, int64_t n_bases, const int64_t *h_segments,
                         int64_t n, uint8_t *d_out, int64_t out_bytes, cudaStream_t stream)
{
    if (n < 0 || n_bases < 0 || out_bytes < 0) return fail(BGD_ERR_INVALID, "ragged_gather: negative size");
    if (n == 0) return BGD_OK;                                          // nothing to copy: no launch
    if (!h_segments) return fail(BGD_ERR_INVALID, "ragged_gather: null segment table");
    if (n_bases > 0 && !h_base_bytes) return fail(BGD_ERR_INVALID, "ragged_gather: null table of source sizes");
    if (n > 65535) return fail(BGD_ERR_INVALID, "ragged_gather: %lld segments, at most 65535 per call", (long long)n);
    int64_t max_bytes = 0;
    for (int64_t k = 0; k < n; ++k) {
        const int64_t r = h_segments[4 * k], so = h_segments[4 * k + 1], d = h_segments[4 * k + 2], b = h_segments[4 * k + 3];
        if (r < 0 || r >= n_bases)
            return fail(BGD_ERR_INVALID, "ragged_gather: segment %lld reads source %lld of %lld", (long long)k, (long long)r,
                        (long long)n_bases);
        if (so < 0 || d < 0 || b < 0)
            return fail(BGD_ERR_INVALID, "ragged_gather: segment %lld has a negative offset or size", (long long)k);
        if ((so | d) & 15)
            return fail(BGD_ERR_INVALID, "ragged_gather: segment %lld is not 16-byte aligned (src %lld, dst %lld)",
                        (long long)k, (long long)so, (long long)d);
        if (b > h_base_bytes[r] - so)
            return fail(BGD_ERR_INVALID, "ragged_gather: segment %lld reads bytes %lld..%lld of the %lld-byte source %lld",
                        (long long)k, (long long)so, (long long)(so + b), (long long)h_base_bytes[r], (long long)r);
        if (b > out_bytes - d)
            return fail(BGD_ERR_INVALID, "ragged_gather: segment %lld writes bytes %lld..%lld of a %lld-byte output",
                        (long long)k, (long long)d, (long long)(d + b), (long long)out_bytes);
        max_bytes = std::max(max_bytes, b);
    }
    if (max_bytes == 0) return BGD_OK;                                  // only empty segments
    if (!d_bases || !d_out) return fail(BGD_ERR_INVALID, "ragged_gather: null base table or output");
    if (reinterpret_cast<uintptr_t>(d_out) & 15) return fail(BGD_ERR_INVALID, "ragged_gather: the output must be 16-byte aligned");
    auto fill = [&](GatherSeg *t) {
        for (int64_t k = 0; k < n; ++k)
            t[k] = GatherSeg{h_segments[4 * k + 1], h_segments[4 * k + 2], h_segments[4 * k + 3], h_segments[4 * k]};
    };
    return launch_ragged_copy("ragged_gather_kernel", ragged_gather_kernel, BaseTable{d_bases}, fill, n, max_bytes, d_out,
                              stream);
}

}  // namespace bgd
