// extern "C" entry points of libbgdebias_b200.so (see include/bgdebias.h) and the host-side
// plumbing they share: error state, device properties, the per-thread workspace, and the pinned
// staging pipeline behind the host-buffer calls.
#include <algorithm>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include <cudaTypedefs.h>

#include "bgd_common.cuh"

namespace bgd {

// ---- error state / accounting ----------------------------------------------------------------
std::string &last_error_ref()
{
    static thread_local std::string s;
    return s;
}

int fail(int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    return code;
}

std::atomic<int64_t> g_launches{0};
static std::atomic<int> g_variant{BGD_MEDIAN_AUTO};

// ---- device properties ------------------------------------------------------------------------
int get_device_props(int device, DeviceProps *out)
{
    static std::mutex mu;
    static DeviceProps cache[64];
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(BGD_ERR_NO_DEVICE, "no CUDA device available (%s)", e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(BGD_ERR_INVALID, "device %d out of range (0..%d)", device, count - 1);
    std::lock_guard<std::mutex> lock(mu);
    if (device < 64 && cache[device].ok) { *out = cache[device]; return BGD_OK; }
    cudaDeviceProp p;
    BGD_CUDA_TRY(cudaGetDeviceProperties(&p, device));
    DeviceProps d;
    d.sm_count = p.multiProcessorCount;
    d.cc_major = p.major;
    d.cc_minor = p.minor;
    d.smem_optin = (int64_t)p.sharedMemPerBlockOptin;
    d.smem_per_sm = (int64_t)p.sharedMemPerMultiprocessor;
    d.total_mem = (int64_t)p.totalGlobalMem;
    d.ok = true;
    if (device < 64) cache[device] = d;
    *out = d;
    return BGD_OK;
}

int current_device_props(DeviceProps *out)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(BGD_ERR_NO_DEVICE, "no CUDA device available (%s)", cudaGetErrorString(e));
    }
    if (int rc = get_device_props(dev, out)) return rc;
    if (out->cc_major != 10)
        return fail(BGD_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", dev,
                    out->cc_major, out->cc_minor);
    return BGD_OK;
}

// ---- workspace --------------------------------------------------------------------------------
void Workspace::free_all()
{
    // at thread exit the context may already be gone (process teardown): errors are ignored, nothing is reported
    for (Slot &s : ring) {
        if (s.d_ptr) cudaFree(s.d_ptr);
        if (s.h_pinned) cudaFreeHost(s.h_pinned);
        if (s.ready) cudaEventDestroy(s.ready);
        s = Slot{};
    }
    cudaGetLastError();
    d_ptr = h_pinned = nullptr;
    bytes = 0;
}

int Workspace::acquire(size_t need)
{
    int dev = 0;
    BGD_CUDA_TRY(cudaGetDevice(&dev));
    if (dev != device) {                       // buffers AND events belong to the device they were created on
        if (device >= 0) {
            int back = dev;
            cudaSetDevice(device);
            free_all();
            cudaSetDevice(back);
        }
        device = dev;
    }
    cur = next;
    next = (next + 1) % kRing;
    Slot &s = ring[cur];
    if (s.in_flight) {
        BGD_CUDA_TRY(cudaEventSynchronize(s.ready));   // the call kRing calls ago has consumed its tables
        s.in_flight = false;
    }
    if (need > s.bytes) {
        if (s.d_ptr) cudaFree(s.d_ptr);
        if (s.h_pinned) cudaFreeHost(s.h_pinned);
        s.d_ptr = s.h_pinned = nullptr;
        s.bytes = 0;
        size_t cap = std::max<size_t>(need, 1 << 16);
        cap = (cap + 4095) & ~(size_t)4095;
        BGD_CUDA_TRY(cudaMalloc(&s.d_ptr, cap));
        BGD_CUDA_TRY(cudaMallocHost(&s.h_pinned, cap));
        s.bytes = cap;
    }
    if (!s.ready) BGD_CUDA_TRY(cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming));
    d_ptr = s.d_ptr;
    h_pinned = s.h_pinned;
    bytes = s.bytes;
    return BGD_OK;
}

int Workspace::release(cudaStream_t stream)
{
    Slot &s = ring[cur];
    if (s.ready) {
        BGD_CUDA_TRY(cudaEventRecord(s.ready, stream));
        s.in_flight = true;
    }
    return BGD_OK;
}

Workspace &thread_workspace()
{
    static thread_local Workspace ws;
    return ws;
}

// ---- median dispatch -------------------------------------------------------------------------
static int median_varlen_dispatch(const uint8_t *d_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                                  uint8_t *d_out, cudaStream_t stream)
{
    if (V < 0 || N < 0) return fail(BGD_ERR_INVALID, "median: negative size");
    if (V == 0) return BGD_OK;
    if (!h_offsets) return fail(BGD_ERR_INVALID, "median: null offsets");
    int64_t T_max = 0;
    for (int64_t v = 0; v < V; ++v) {
        const int64_t T = h_offsets[v + 1] - h_offsets[v];
        // reference: np.median([]) is nan and the JPEG write raises (extract_background.py:73-74)
        if (T <= 0) return fail(BGD_ERR_INVALID, "median: video %lld has no frames", (long long)v);
        T_max = std::max(T_max, T);
    }
    if (N == 0) return BGD_OK;
    if (!d_frames || !d_out) return fail(BGD_ERR_INVALID, "median: null pointer");
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;

    const int variant = g_variant.load();
    const bool aligned = reinterpret_cast<uintptr_t>(d_frames) % 16 == 0 && reinterpret_cast<uintptr_t>(d_out) % 16 == 0;
    const bool can_col = aligned && median_tma_supports(T_max, N);
    const bool can_bit = aligned && median_bitsliced_supports(T_max, N);
    if (((variant == BGD_MEDIAN_COLPLANE || variant == BGD_MEDIAN_LDSM) && !can_col) || (variant == BGD_MEDIAN_BITSLICED && !can_bit))
        return fail(BGD_ERR_UNSUPPORTED,
                    "median: the TMA variants need N %% 16 == 0, 16-byte aligned buffers and at most ~500 frames per video (T=%lld N=%lld)",
                    (long long)T_max, (long long)N);
    // AUTO / LDSM: videos of up to 512 frames take the transposing-load kernel, longer ones the column-plane kernel
    if (variant == BGD_MEDIAN_COLPLANE || variant == BGD_MEDIAN_LDSM || (variant == BGD_MEDIAN_AUTO && can_col))
        return median_tma_varlen(d_frames, h_offsets, V, N, d_out, variant != BGD_MEDIAN_COLPLANE, nullptr, 0, stream);
    // AUTO with SOME videos beyond the TMA kernels' frame limit (the rawframes variant has no frame cap,
    // comix_loader.py:157-161): those videos alone take the generic kernel, the rest of the batch keeps the fast path
    std::vector<int64_t> fast, slow;
    if (variant == BGD_MEDIAN_AUTO && aligned && median_tma_supports(1, N)) {
        for (int64_t v = 0; v < V; ++v)
            (median_tma_supports(h_offsets[v + 1] - h_offsets[v], N) ? fast : slow).push_back(v);
    }
    if (!fast.empty()) {
        if (int rc = median_tma_varlen(d_frames, h_offsets, V, N, d_out, true, fast.data(), (int64_t)fast.size(), stream)) return rc;
        if (slow.empty()) return BGD_OK;
    } else if (variant == BGD_MEDIAN_BITSLICED || (variant == BGD_MEDIAN_AUTO && can_bit)) {
        return median_bitsliced_varlen(d_frames, h_offsets, V, N, d_out, stream);
    } else {
        slow.resize((size_t)V);
        for (int64_t v = 0; v < V; ++v) slow[(size_t)v] = v;
    }

    // generic variant: tables row0[n] | T[n] for the videos in `slow`; grid.y carries the position in a run of
    // consecutive videos, 65535 per launch
    const int64_t n = (int64_t)slow.size();
    Workspace &ws = thread_workspace();
    if (int rc = ws.acquire((size_t)n * 12)) return rc;
    int64_t *h_row0 = static_cast<int64_t *>(ws.h_pinned);
    int32_t *h_T = reinterpret_cast<int32_t *>(h_row0 + n);
    for (int64_t i = 0; i < n; ++i) {
        const int64_t v = slow[(size_t)i];
        h_row0[i] = h_offsets[v];
        h_T[i] = (int32_t)(h_offsets[v + 1] - h_offsets[v]);
    }
    BGD_CUDA_TRY(cudaMemcpyAsync(ws.d_ptr, ws.h_pinned, (size_t)n * 12, cudaMemcpyHostToDevice, stream));
    const int64_t *d_row0 = static_cast<const int64_t *>(ws.d_ptr);
    const int32_t *d_T = reinterpret_cast<const int32_t *>(d_row0 + n);
    int rc = BGD_OK;
    for (int64_t i0 = 0; i0 < n && rc == BGD_OK;) {
        int64_t i1 = i0 + 1;                                   // a run of consecutive videos shares a launch
        int32_t run_T = h_T[i0];
        while (i1 < n && i1 - i0 < 65535 && slow[(size_t)i1] == slow[(size_t)i1 - 1] + 1) run_T = std::max(run_T, h_T[i1++]);
        rc = launch_median_swar(d_frames, d_row0 + i0, d_T + i0, i1 - i0, N, d_out + slow[(size_t)i0] * N, (int)run_T, stream);
        i0 = i1;
    }
    const int rc2 = ws.release(stream);
    return rc ? rc : rc2;
}

// ---- pinned staging for the host-buffer calls --------------------------------------------------
// Two pinned slabs + two device slabs per host thread; a chunk of whole videos is packed into a
// pinned slab by the CPU while the previous chunk's copy and kernel run on the other slab.
struct Stager {
    static constexpr int kSlots = 2;
    uint8_t *h_in[kSlots] = {nullptr, nullptr};
    uint8_t *d_in[kSlots] = {nullptr, nullptr};
    uint8_t *h_out[kSlots] = {nullptr, nullptr};
    uint8_t *d_out[kSlots] = {nullptr, nullptr};
    size_t in_cap = 0, out_cap = 0;
    cudaStream_t stream[kSlots] = {nullptr, nullptr};
    cudaEvent_t done[kSlots] = {nullptr, nullptr};
    int device = -1;

    size_t h_in_cap = 0, h_out_cap = 0;

    ~Stager()
    {
        release_all();                       // at thread exit; errors (context already gone) are ignored
        cudaGetLastError();
    }

    // device slabs of in_bytes / out_bytes; pinned mirrors only as large as asked (0 = caller's memory is pinned)
    int ensure(int dev, size_t in_bytes, size_t out_bytes, size_t h_in_bytes = (size_t)-1, size_t h_out_bytes = (size_t)-1)
    {
        if (h_in_bytes == (size_t)-1) h_in_bytes = in_bytes;
        if (h_out_bytes == (size_t)-1) h_out_bytes = out_bytes;
        BGD_CUDA_TRY(cudaSetDevice(dev));
        if (dev != device) {
            release_all();
            device = dev;
            for (int s = 0; s < kSlots; ++s) {
                BGD_CUDA_TRY(cudaStreamCreateWithFlags(&stream[s], cudaStreamNonBlocking));
                BGD_CUDA_TRY(cudaEventCreateWithFlags(&done[s], cudaEventDisableTiming));
            }
        }
        if (in_bytes > in_cap) {
            for (int s = 0; s < kSlots; ++s) { if (d_in[s]) cudaFree(d_in[s]); d_in[s] = nullptr; }
            in_cap = 0;
            for (int s = 0; s < kSlots; ++s) BGD_CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_in[s]), in_bytes));
            in_cap = in_bytes;
        }
        if (h_in_bytes > h_in_cap) {
            for (int s = 0; s < kSlots; ++s) { if (h_in[s]) cudaFreeHost(h_in[s]); h_in[s] = nullptr; }
            h_in_cap = 0;
            for (int s = 0; s < kSlots; ++s) BGD_CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&h_in[s]), h_in_bytes));
            h_in_cap = h_in_bytes;
        }
        if (out_bytes > out_cap) {
            for (int s = 0; s < kSlots; ++s) { if (d_out[s]) cudaFree(d_out[s]); d_out[s] = nullptr; }
            out_cap = 0;
            for (int s = 0; s < kSlots; ++s) BGD_CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_out[s]), out_bytes));
            out_cap = out_bytes;
        }
        if (h_out_bytes > h_out_cap) {
            for (int s = 0; s < kSlots; ++s) { if (h_out[s]) cudaFreeHost(h_out[s]); h_out[s] = nullptr; }
            h_out_cap = 0;
            for (int s = 0; s < kSlots; ++s) BGD_CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&h_out[s]), h_out_bytes));
            h_out_cap = h_out_bytes;
        }
        return BGD_OK;
    }
    void release_all()
    {
        for (int s = 0; s < kSlots; ++s) {
            if (h_in[s]) cudaFreeHost(h_in[s]);
            if (d_in[s]) cudaFree(d_in[s]);
            if (h_out[s]) cudaFreeHost(h_out[s]);
            if (d_out[s]) cudaFree(d_out[s]);
            if (stream[s]) cudaStreamDestroy(stream[s]);
            if (done[s]) cudaEventDestroy(done[s]);
            h_in[s] = d_in[s] = h_out[s] = d_out[s] = nullptr;
            stream[s] = nullptr;
            done[s] = nullptr;
        }
        in_cap = out_cap = h_in_cap = h_out_cap = 0;
    }
};

static Stager &thread_stager()
{
    static thread_local Stager st;
    return st;
}

static bool is_pinned_host(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

static int pack_threads()
{
    static const int n = [] {
        if (const char *s = getenv("BGD_PACK_THREADS")) return std::max(1, std::min(32, atoi(s)));
        const unsigned hc = std::thread::hardware_concurrency();
        return (int)std::max(1u, std::min(8u, hc / 2));
    }();
    return n;
}

static size_t staging_slab_bytes()
{
    size_t mb = 256;
    if (const char *s = getenv("BGD_STAGING_SLAB_MB")) mb = (size_t)std::max(1, atoi(s));
    return mb << 20;
}

// frames given as per-frame pointers (frame_ptrs[row]) or as one block (frames + row * N)
static int median_host_pipeline(const uint8_t *const *frame_ptrs, const uint8_t *frames, const int64_t *h_offsets,
                                int64_t V, int64_t N, uint8_t *h_out, int device)
{
    if (V < 0 || N < 0) return fail(BGD_ERR_INVALID, "median: negative size");
    if (V == 0) return BGD_OK;
    if (!h_offsets || (!frame_ptrs && !frames) || !h_out) return fail(BGD_ERR_INVALID, "median: null pointer");
    int64_t T_max = 0;
    for (int64_t v = 0; v < V; ++v) {
        const int64_t T = h_offsets[v + 1] - h_offsets[v];
        if (T <= 0) return fail(BGD_ERR_INVALID, "median: video %lld has no frames", (long long)v);
        T_max = std::max(T_max, T);
    }
    if (N == 0) return BGD_OK;
    DeviceProps dp;
    if (int rc = get_device_props(device, &dp)) return rc;
    BGD_CUDA_TRY(cudaSetDevice(device));

    const size_t slab = std::max<size_t>(staging_slab_bytes(), (size_t)T_max * N);
    // chunks of whole videos that fit a slab
    std::vector<std::pair<int64_t, int64_t>> chunks;
    for (int64_t v = 0; v < V;) {
        int64_t e = v;
        size_t bytes = 0;
        while (e < V && bytes + (size_t)(h_offsets[e + 1] - h_offsets[e]) * N <= slab) {
            bytes += (size_t)(h_offsets[e + 1] - h_offsets[e]) * N;
            ++e;
        }
        chunks.emplace_back(v, e);
        v = e;
    }
    int64_t max_videos = 0;
    for (auto &c : chunks) max_videos = std::max(max_videos, c.second - c.first);
    // page-locked caller buffers are copied from / into directly; pageable ones go through pinned mirrors
    const bool in_pinned = frames && is_pinned_host(frames);
    const bool out_pinned = is_pinned_host(h_out);
    Stager &st = thread_stager();
    if (int rc = st.ensure(device, slab, (size_t)max_videos * N, in_pinned ? 0 : slab,
                           out_pinned ? 64 : (size_t)max_videos * N))
        return rc;

    std::vector<int64_t> local;
    int pending_slot_chunk[Stager::kSlots] = {-1, -1};
    auto drain = [&](int slot) -> int {
        if (pending_slot_chunk[slot] < 0) return BGD_OK;
        BGD_CUDA_TRY(cudaEventSynchronize(st.done[slot]));
        const auto &c = chunks[pending_slot_chunk[slot]];
        if (!out_pinned) std::memcpy(h_out + c.first * N, st.h_out[slot], (size_t)(c.second - c.first) * N);
        pending_slot_chunk[slot] = -1;
        return BGD_OK;
    };
    for (size_t ci = 0; ci < chunks.size(); ++ci) {
        const int slot = (int)(ci % Stager::kSlots);
        if (int rc = drain(slot)) return rc;
        const int64_t v0 = chunks[ci].first, v1 = chunks[ci].second;
        const int64_t r0 = h_offsets[v0], r1 = h_offsets[v1];
        cudaStream_t s = st.stream[slot];
        if (in_pinned) {
            BGD_CUDA_TRY(cudaMemcpyAsync(st.d_in[slot], frames + (size_t)r0 * N, (size_t)(r1 - r0) * N, cudaMemcpyHostToDevice, s));
        } else {
            // pack the chunk into the pinned slab (gathers separately allocated frames) with a few threads, and
            // send each part as soon as it is packed: the DMA of part i overlaps the packing of part i + 1
            const int64_t rows = r1 - r0;
            const size_t bytes = (size_t)rows * N;
            int parts = bytes >= ((size_t)8 << 20) ? (int)std::min<int64_t>(pack_threads(), rows) : 1;
            std::vector<std::thread> workers;
            auto pack = [&](int64_t a, int64_t b) {
                if (frame_ptrs) {
                    for (int64_t r = a; r < b; ++r) std::memcpy(st.h_in[slot] + (size_t)(r - r0) * N, frame_ptrs[r], (size_t)N);
                } else {
                    std::memcpy(st.h_in[slot] + (size_t)(a - r0) * N, frames + (size_t)a * N, (size_t)(b - a) * N);
                }
            };
            std::vector<int64_t> cut((size_t)parts + 1);
            for (int p = 0; p <= parts; ++p) cut[(size_t)p] = r0 + rows * p / parts;
            for (int p = 1; p < parts; ++p) workers.emplace_back(pack, cut[(size_t)p], cut[(size_t)p + 1]);
            pack(cut[0], cut[1]);
            cudaError_t err = cudaSuccess;
            for (int p = 0; p < parts; ++p) {
                if (p > 0) workers[(size_t)p - 1].join();
                const size_t off = (size_t)(cut[(size_t)p] - r0) * N, len = (size_t)(cut[(size_t)p + 1] - cut[(size_t)p]) * N;
                if (err == cudaSuccess && len) err = cudaMemcpyAsync(st.d_in[slot] + off, st.h_in[slot] + off, len, cudaMemcpyHostToDevice, s);
            }
            if (err != cudaSuccess) return fail(BGD_ERR_CUDA, "cudaMemcpyAsync (frames to device) failed: %s", cudaGetErrorString(err));
        }
        local.resize((size_t)(v1 - v0 + 1));
        for (int64_t v = v0; v <= v1; ++v) local[(size_t)(v - v0)] = h_offsets[v] - r0;
        if (int rc = median_varlen_dispatch(st.d_in[slot], local.data(), v1 - v0, N, st.d_out[slot], s)) return rc;
        uint8_t *dst = out_pinned ? h_out + (size_t)v0 * N : st.h_out[slot];
        BGD_CUDA_TRY(cudaMemcpyAsync(dst, st.d_out[slot], (size_t)(v1 - v0) * N, cudaMemcpyDeviceToHost, s));
        BGD_CUDA_TRY(cudaEventRecord(st.done[slot], s));
        pending_slot_chunk[slot] = (int)ci;
    }
    for (int slot = 0; slot < Stager::kSlots; ++slot)
        if (int rc = drain(slot)) return rc;
    return BGD_OK;
}

// The *_f32 blend entry points keep their contract: fp32 out in NTCHW or NCTHW; NTHWC is for the *_out entry points.
static int f32_layout(const char *who, int layout)
{
    return layout == BGD_LAYOUT_NTHWC ? fail(BGD_ERR_INVALID, "%s: unknown layout %d", who, layout) : BGD_OK;
}

}  // namespace bgd

// =================================================================================================
using namespace bgd;

extern "C" {

int bgd_abi_version(void) { return BGD_ABI_VERSION; }

const char *bgd_last_error(void) { return last_error_ref().c_str(); }

int bgd_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, int64_t *smem_optin_bytes,
                    int64_t *total_mem_bytes)
{
    DeviceProps d;
    if (int rc = get_device_props(device, &d)) return rc;
    if (sm_count) *sm_count = d.sm_count;
    if (cc_major) *cc_major = d.cc_major;
    if (cc_minor) *cc_minor = d.cc_minor;
    if (smem_optin_bytes) *smem_optin_bytes = d.smem_optin;
    if (total_mem_bytes) *total_mem_bytes = d.total_mem;
    return BGD_OK;
}

int64_t bgd_kernel_launch_count(void) { return g_launches.load(); }

int bgd_median_set_variant(int variant)
{
    if (variant < BGD_MEDIAN_AUTO || variant > BGD_MEDIAN_LDSM)
        return fail(BGD_ERR_INVALID, "unknown median variant %d", variant);
    g_variant.store(variant);
    return BGD_OK;
}

int bgd_median_get_variant(void) { return g_variant.load(); }

int bgd_temporal_median_u8(const uint8_t *d_frames, int64_t T, int64_t N, uint8_t *d_out, void *stream)
{
    const int64_t offs[2] = {0, T};
    return median_varlen_dispatch(d_frames, offs, 1, N, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_temporal_median_varlen_u8(const uint8_t *d_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                                  uint8_t *d_out, void *stream)
{
    if (V > 0 && h_offsets) {
        for (int64_t v = 0; v < V; ++v)
            if (h_offsets[v + 1] < h_offsets[v]) return fail(BGD_ERR_INVALID, "median: offsets must be non-decreasing");
    }
    return median_varlen_dispatch(d_frames, h_offsets, V, N, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_temporal_median_u8_host(const uint8_t *const *h_frame_ptrs, int64_t T, int64_t N, uint8_t *h_out, int device)
{
    if (!h_frame_ptrs) return fail(BGD_ERR_INVALID, "median: null frame pointer list");
    const int64_t offs[2] = {0, T};
    return median_host_pipeline(h_frame_ptrs, nullptr, offs, 1, N, h_out, device);
}

int bgd_temporal_median_varlen_u8_host(const uint8_t *h_frames, const int64_t *h_offsets, int64_t V, int64_t N,
                                       uint8_t *h_out, int device)
{
    if (V > 0 && h_offsets) {
        for (int64_t v = 0; v < V; ++v)
            if (h_offsets[v + 1] < h_offsets[v]) return fail(BGD_ERR_INVALID, "median: offsets must be non-decreasing");
        if (h_offsets[0] != 0 && !h_frames) return fail(BGD_ERR_INVALID, "median: null pointer");
    }
    return median_host_pipeline(nullptr, h_frames, h_offsets, V, N, h_out, device);
}

int bgd_nan_temporal_reduce_f32(const float *d_frames, int64_t T, int64_t N, int avg_method, int zero_is_missing,
                                uint8_t *d_out_u8, float *d_out_f32, void *stream)
{
    return launch_nan_reduce(d_frames, T, N, avg_method, zero_is_missing, d_out_u8, d_out_f32,
                             static_cast<cudaStream_t>(stream));
}

int bgd_actor_cut_mix_u8(const uint8_t *d_actor, const uint8_t *d_mask, const uint8_t *d_scene, int64_t n, uint8_t *d_out,
                         uint64_t *d_mask_sum, void *stream)
{
    return launch_cutmix(d_actor, d_mask, d_scene, n, d_out, reinterpret_cast<unsigned long long *>(d_mask_sum),
                         static_cast<cudaStream_t>(stream));
}

int bgd_nan_temporal_reduce_varlen_f32(const float *d_frames, const int64_t *h_offsets, int64_t V, int64_t N, int avg_method,
                                       int zero_is_missing, uint8_t *d_out_u8, float *d_out_f32, void *stream)
{
    return launch_nan_reduce_varlen(d_frames, h_offsets, V, N, avg_method, zero_is_missing, d_out_u8, d_out_f32,
                                    static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_f32(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W, const float *d_bg_pool,
                        int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx, const int32_t *d_top,
                        const int32_t *d_left, const uint8_t *d_apply, const float *d_fg_lut, const float *h_bg_mean,
                        const float *h_bg_std, double alpha, int layout, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (int rc = f32_layout("bgmix", layout)) return rc;
    return launch_bgmix(d_fg, nullptr, B, T, H, W, d_bg_pool, false, P, Hb, Wb, d_bg_idx, d_top, d_left, d_apply, d_fg_lut,
                        h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_u8pool_f32(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W,
                               const uint8_t *d_bg_pool, int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx,
                               const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                               const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std, double alpha,
                               int layout, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (int rc = f32_layout("bgmix", layout)) return rc;
    return launch_bgmix(d_fg, nullptr, B, T, H, W, d_bg_pool, true, P, Hb, Wb, d_bg_idx, d_top, d_left, d_apply, d_fg_lut,
                        h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_out(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W, const void *d_bg_pool, int pool_is_u8,
                        int64_t P, int64_t Hb, int64_t Wb, const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left,
                        const uint8_t *d_apply, const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std,
                        double alpha, int layout, int out_dtype, void *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (!d_fg) return fail(BGD_ERR_INVALID, "bgmix: null foreground");
    return launch_bgmix(d_fg, nullptr, B, T, H, W, d_bg_pool, pool_is_u8 != 0, P, Hb, Wb, d_bg_idx, d_top, d_left, d_apply,
                        d_fg_lut, h_bg_mean, h_bg_std, alpha, layout, out_dtype, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_normfg_f32(const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W,
                               const void *d_bg_pool, int pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                               const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left,
                               const uint8_t *d_apply, const float *h_bg_mean, const float *h_bg_std, double alpha,
                               int layout, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (!d_fg_norm) return fail(BGD_ERR_INVALID, "bgmix: null foreground");
    if (int rc = f32_layout("bgmix", layout)) return rc;
    return launch_bgmix(nullptr, d_fg_norm, B, T, H, W, d_bg_pool, pool_is_u8 != 0, P, Hb, Wb, d_bg_idx, d_top, d_left,
                        d_apply, nullptr, h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out,
                        static_cast<cudaStream_t>(stream));
}

int bgd_aa_resize_table(int64_t in_size, int64_t out_size, int32_t *taps, int32_t *h_words, int64_t cap_words)
{
    return aa_resize_table(in_size, out_size, taps, h_words, cap_words);
}

int bgd_aa_resize_u8_f32(const uint8_t *d_pool, const bgd_ragged_slot *h_slot, const int32_t *d_tables, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_aa_resize(d_pool, h_slot, d_tables, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_ragged_f32(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W, const uint8_t *d_pool,
                               const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables, const int32_t *d_bg_idx,
                               const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply, const float *d_fg_lut,
                               const float *h_bg_mean, const float *h_bg_std, double alpha, int layout, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (!d_fg) return fail(BGD_ERR_INVALID, "bgmix (ragged): null foreground");
    if (int rc = f32_layout("bgmix (ragged)", layout)) return rc;
    return launch_bgmix_ragged(d_fg, nullptr, B, T, H, W, d_pool, d_slots, P, d_tables, d_bg_idx, d_top, d_left, d_apply, d_fg_lut,
                               h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_ragged_out(const uint8_t *d_fg, int64_t B, int64_t T, int64_t H, int64_t W, const uint8_t *d_pool,
                               const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables, const int32_t *d_bg_idx,
                               const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply, const float *d_fg_lut,
                               const float *h_bg_mean, const float *h_bg_std, double alpha, int layout, int out_dtype,
                               void *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (!d_fg) return fail(BGD_ERR_INVALID, "bgmix (ragged): null foreground");
    return launch_bgmix_ragged(d_fg, nullptr, B, T, H, W, d_pool, d_slots, P, d_tables, d_bg_idx, d_top, d_left, d_apply, d_fg_lut,
                               h_bg_mean, h_bg_std, alpha, layout, out_dtype, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_ragged_normfg_f32(const float *d_fg_norm, int64_t B, int64_t T, int64_t H, int64_t W, const uint8_t *d_pool,
                                      const bgd_ragged_slot *d_slots, int64_t P, const int32_t *d_tables,
                                      const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left,
                                      const uint8_t *d_apply, const float *h_bg_mean, const float *h_bg_std, double alpha,
                                      int layout, float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (!d_fg_norm) return fail(BGD_ERR_INVALID, "bgmix (ragged): null foreground");
    if (int rc = f32_layout("bgmix (ragged)", layout)) return rc;
    return launch_bgmix_ragged(nullptr, d_fg_norm, B, T, H, W, d_pool, d_slots, P, d_tables, d_bg_idx, d_top, d_left, d_apply,
                               nullptr, h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_resized_crop_aa_u8_f32(const uint8_t *d_src, int64_t src_bytes, const bgd_crop_desc *h_desc, int64_t n,
                               const int32_t *d_tables, int64_t table_words, int64_t out_h, int64_t out_w, float *d_out,
                               void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_resized_crop_aa(d_src, src_bytes, h_desc, n, d_tables, table_words, out_h, out_w, d_out,
                                  static_cast<cudaStream_t>(stream));
}

int bgd_resize_bilinear_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H,
                           int64_t W, uint8_t *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_resize_u8(d_src, src_bytes, h_geom, B, T, H, W, d_out, static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_resize_blend_f32(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H,
                               int64_t W, const void *d_bg_pool, int pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                               const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                               const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std, double alpha, int layout,
                               float *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    if (int rc = f32_layout("bgmix_resize", layout)) return rc;
    return launch_resize_blend(d_src, src_bytes, h_geom, B, T, H, W, d_bg_pool, pool_is_u8 != 0, P, Hb, Wb, d_bg_idx, d_top,
                               d_left, d_apply, d_fg_lut, h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out,
                               static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_resize_blend_out(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T, int64_t H,
                               int64_t W, const void *d_bg_pool, int pool_is_u8, int64_t P, int64_t Hb, int64_t Wb,
                               const int32_t *d_bg_idx, const int32_t *d_top, const int32_t *d_left, const uint8_t *d_apply,
                               const float *d_fg_lut, const float *h_bg_mean, const float *h_bg_std, double alpha, int layout,
                               int out_dtype, void *d_out, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_resize_blend(d_src, src_bytes, h_geom, B, T, H, W, d_bg_pool, pool_is_u8 != 0, P, Hb, Wb, d_bg_idx, d_top,
                               d_left, d_apply, d_fg_lut, h_bg_mean, h_bg_std, alpha, layout, out_dtype, d_out,
                               static_cast<cudaStream_t>(stream));
}

int bgd_bgmix_blend_f32_host(const uint8_t *h_fg, int64_t B, int64_t T, int64_t H, int64_t W, const float *d_bg_pool,
                             int64_t P, int64_t Hb, int64_t Wb, const int32_t *h_bg_idx, const int32_t *h_top,
                             const int32_t *h_left, const uint8_t *h_apply, const float *d_fg_lut,
                             const float *h_bg_mean, const float *h_bg_std, double alpha, int layout, float *d_out,
                             double *h_checksum, int device)
{
    if (B < 0 || T < 0 || H < 0 || W < 0) return fail(BGD_ERR_INVALID, "bgmix: negative size");
    if (int rc = f32_layout("bgmix", layout)) return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) { if (h_checksum) *h_checksum = 0.0; return BGD_OK; }
    if (!h_fg || !h_bg_idx || !h_top || !h_left || !h_apply) return fail(BGD_ERR_INVALID, "bgmix: null host pointer");
    // the reference's RandomCrop raises when the crop does not fit; validate here, on host values
    for (int64_t b = 0; b < B; ++b) {
        if (!h_apply[b]) continue;
        if (h_bg_idx[b] < 0 || h_bg_idx[b] >= P) return fail(BGD_ERR_INVALID, "bgmix: bg_idx[%lld]=%d outside pool of %lld", (long long)b, h_bg_idx[b], (long long)P);
        if (h_top[b] < 0 || h_top[b] + H > Hb || h_left[b] < 0 || h_left[b] + W > Wb)
            return fail(BGD_ERR_INVALID, "bgmix: crop of sample %lld leaves the pool image", (long long)b);
    }
    DeviceProps dp;
    if (int rc = get_device_props(device, &dp)) return rc;
    BGD_CUDA_TRY(cudaSetDevice(device));
    const size_t fg_bytes = (size_t)B * T * H * W * 3;
    const size_t par_bytes = (size_t)B * 13 + 64;
    const bool fg_pinned = is_pinned_host(h_fg);      // page-locked clips are copied straight from the caller's buffer
    Stager &st = thread_stager();
    if (int rc = st.ensure(device, fg_bytes + par_bytes + 64, 64, (fg_pinned ? 0 : fg_bytes) + par_bytes + 64, 64)) return rc;
    cudaStream_t s = st.stream[0];
    uint8_t *hp = st.h_in[0], *dp_ = st.d_in[0];
    const size_t o = (fg_bytes + 15) & ~(size_t)15;     // device layout: clips | bg_idx | top | left | apply
    uint8_t *hpar = fg_pinned ? hp : hp + o;
    if (!fg_pinned) std::memcpy(hp, h_fg, fg_bytes);
    std::memcpy(hpar, h_bg_idx, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 4, h_top, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 8, h_left, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 12, h_apply, (size_t)B);
    if (fg_pinned) {
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_, h_fg, fg_bytes, cudaMemcpyHostToDevice, s));
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_ + o, hpar, (size_t)B * 13, cudaMemcpyHostToDevice, s));
    } else {
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_, hp, o + (size_t)B * 13, cudaMemcpyHostToDevice, s));
    }
    const int32_t *d_idx = reinterpret_cast<const int32_t *>(dp_ + o);
    if (int rc = launch_bgmix(dp_, nullptr, B, T, H, W, d_bg_pool, false, P, Hb, Wb, d_idx, d_idx + B, d_idx + 2 * B,
                              dp_ + o + (size_t)B * 12, d_fg_lut, h_bg_mean, h_bg_std, alpha, layout, BGD_OUT_F32, d_out, s))
        return rc;
    if (h_checksum) {
        double *d_sum = reinterpret_cast<double *>(st.d_out[0]);
        if (int rc = launch_sum_f32(d_out, (int64_t)B * T * 3 * H * W, d_sum, s)) return rc;
        BGD_CUDA_TRY(cudaMemcpyAsync(st.h_out[0], d_sum, sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    BGD_CUDA_TRY(cudaStreamSynchronize(s));
    if (h_checksum) std::memcpy(h_checksum, st.h_out[0], sizeof(double));
    return BGD_OK;
}

int bgd_bgmix_resize_blend_f32_host(const uint8_t *h_src, int64_t src_bytes, const int64_t *h_geom, int64_t B, int64_t T,
                                    int64_t H, int64_t W, const float *d_bg_pool, int64_t P, int64_t Hb, int64_t Wb,
                                    const int32_t *h_bg_idx, const int32_t *h_top, const int32_t *h_left,
                                    const uint8_t *h_apply, const float *d_fg_lut, const float *h_bg_mean,
                                    const float *h_bg_std, double alpha, int layout, float *d_out, double *h_checksum,
                                    int device)
{
    if (B < 0 || T < 0 || H < 0 || W < 0 || src_bytes < 0) return fail(BGD_ERR_INVALID, "bgmix_resize: negative size");
    if (int rc = f32_layout("bgmix_resize", layout)) return rc;
    if (B == 0 || T == 0 || H == 0 || W == 0) { if (h_checksum) *h_checksum = 0.0; return BGD_OK; }
    if (!h_src || !h_geom || !h_bg_idx || !h_top || !h_left || !h_apply) return fail(BGD_ERR_INVALID, "bgmix_resize: null host pointer");
    if (src_bytes % 4) return fail(BGD_ERR_INVALID, "bgmix_resize: the source buffer must be a multiple of 4 bytes long");
    for (int64_t b = 0; b < B; ++b) {
        if (!h_apply[b]) continue;
        if (h_bg_idx[b] < 0 || h_bg_idx[b] >= P) return fail(BGD_ERR_INVALID, "bgmix_resize: bg_idx[%lld]=%d outside pool of %lld", (long long)b, h_bg_idx[b], (long long)P);
        if (h_top[b] < 0 || h_top[b] + H > Hb || h_left[b] < 0 || h_left[b] + W > Wb)
            return fail(BGD_ERR_INVALID, "bgmix_resize: crop of sample %lld leaves the pool image", (long long)b);
    }
    DeviceProps dp;
    if (int rc = get_device_props(device, &dp)) return rc;
    BGD_CUDA_TRY(cudaSetDevice(device));
    const size_t fg_bytes = (size_t)src_bytes;
    const size_t par_bytes = (size_t)B * 13 + 64;
    const bool fg_pinned = is_pinned_host(h_src);     // page-locked crops are copied straight from the caller's buffer
    Stager &st = thread_stager();
    if (int rc = st.ensure(device, fg_bytes + par_bytes + 64, 64, (fg_pinned ? 0 : fg_bytes) + par_bytes + 64, 64)) return rc;
    cudaStream_t s = st.stream[0];
    uint8_t *hp = st.h_in[0], *dp_ = st.d_in[0];
    const size_t o = (fg_bytes + 15) & ~(size_t)15;     // device layout: crops | bg_idx | top | left | apply
    uint8_t *hpar = fg_pinned ? hp : hp + o;
    if (!fg_pinned) std::memcpy(hp, h_src, fg_bytes);
    std::memcpy(hpar, h_bg_idx, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 4, h_top, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 8, h_left, (size_t)B * 4);
    std::memcpy(hpar + (size_t)B * 12, h_apply, (size_t)B);
    if (fg_pinned) {
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_, h_src, fg_bytes, cudaMemcpyHostToDevice, s));
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_ + o, hpar, (size_t)B * 13, cudaMemcpyHostToDevice, s));
    } else {
        BGD_CUDA_TRY(cudaMemcpyAsync(dp_, hp, o + (size_t)B * 13, cudaMemcpyHostToDevice, s));
    }
    const int32_t *d_idx = reinterpret_cast<const int32_t *>(dp_ + o);
    if (int rc = launch_resize_blend(dp_, src_bytes, h_geom, B, T, H, W, d_bg_pool, false, P, Hb, Wb, d_idx, d_idx + B,
                                     d_idx + 2 * B, dp_ + o + (size_t)B * 12, d_fg_lut, h_bg_mean, h_bg_std, alpha, layout,
                                     BGD_OUT_F32, d_out, s))
        return rc;
    if (h_checksum) {
        double *d_sum = reinterpret_cast<double *>(st.d_out[0]);
        if (int rc = launch_sum_f32(d_out, (int64_t)B * T * 3 * H * W, d_sum, s)) return rc;
        BGD_CUDA_TRY(cudaMemcpyAsync(st.h_out[0], d_sum, sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    BGD_CUDA_TRY(cudaStreamSynchronize(s));
    if (h_checksum) std::memcpy(h_checksum, st.h_out[0], sizeof(double));
    return BGD_OK;
}

int bgd_ragged_pack_u8(const uint8_t *d_src, int64_t src_bytes, const int64_t *h_segments, int64_t n, uint8_t *d_out,
                       int64_t out_bytes, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_ragged_pack(d_src, src_bytes, h_segments, n, d_out, out_bytes, static_cast<cudaStream_t>(stream));
}

int bgd_ragged_gather_u8(const uint8_t *const *d_bases, const int64_t *h_base_bytes, int64_t n_bases, const int64_t *h_segments,
                         int64_t n, uint8_t *d_out, int64_t out_bytes, void *stream)
{
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    return launch_ragged_gather(d_bases, h_base_bytes, n_bases, h_segments, n, d_out, out_bytes,
                                static_cast<cudaStream_t>(stream));
}

int bgd_ipc_export(const void *d_ptr, uint8_t *handle, int64_t *offset)
{
    if (!d_ptr || !handle || !offset) return fail(BGD_ERR_INVALID, "ipc_export: null argument");
    DeviceProps dp;
    if (int rc = current_device_props(&dp)) return rc;
    cudaPointerAttributes attr;
    BGD_CUDA_TRY(cudaPointerGetAttributes(&attr, d_ptr));
    int dev = 0;
    BGD_CUDA_TRY(cudaGetDevice(&dev));
    if (attr.type != cudaMemoryTypeDevice || attr.device != dev)
        return fail(BGD_ERR_INVALID, "ipc_export: %p is not device memory of the current device %d", d_ptr, dev);
    // the allocation that holds d_ptr: torch's caching allocator hands out pieces of larger cudaMalloc segments, and only a
    // segment's base can be exported.  cuMemGetAddressRange is reached through the runtime, so the library links no libcuda.
    static const PFN_cuMemGetAddressRange_v3020 get_range = [] {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuMemGetAddressRange", &fn, 12000, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            fn = nullptr;
        cudaGetLastError();
        return reinterpret_cast<PFN_cuMemGetAddressRange_v3020>(fn);
    }();
    if (!get_range) return fail(BGD_ERR_UNSUPPORTED, "ipc_export: the driver does not provide cuMemGetAddressRange");
    CUdeviceptr base = 0;
    size_t size = 0;
    if (CUresult r = get_range(&base, &size, reinterpret_cast<CUdeviceptr>(d_ptr)))
        return fail(BGD_ERR_UNSUPPORTED, "ipc_export: cuMemGetAddressRange failed on %p (CUresult %d)", d_ptr, (int)r);
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, reinterpret_cast<void *>(base));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(BGD_ERR_UNSUPPORTED,
                    "ipc_export: the allocation at %p cannot be exported with cudaIpcGetMemHandle (%s); peer mapping needs "
                    "memory from cudaMalloc -- torch's native caching allocator without expandable_segments, not the "
                    "cudaMallocAsync backend",
                    reinterpret_cast<void *>(base), cudaGetErrorString(e));
    }
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(handle, &h, sizeof(h));
    *offset = (int64_t)(reinterpret_cast<CUdeviceptr>(d_ptr) - base);
    return BGD_OK;
}

int bgd_ipc_open(const uint8_t *handle, int device, void **d_base)
{
    if (!handle || !d_base) return fail(BGD_ERR_INVALID, "ipc_open: null argument");
    DeviceProps dp;
    if (int rc = get_device_props(device, &dp)) return rc;
    int back = 0;
    BGD_CUDA_TRY(cudaGetDevice(&back));
    BGD_CUDA_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    cudaSetDevice(back);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(BGD_ERR_UNSUPPORTED, "ipc_open: cudaIpcOpenMemHandle failed on device %d: %s", device, cudaGetErrorString(e));
    }
    *d_base = p;
    return BGD_OK;
}

int bgd_ipc_close(void *d_base)
{
    if (!d_base) return fail(BGD_ERR_INVALID, "ipc_close: null pointer");
    BGD_CUDA_TRY(cudaIpcCloseMemHandle(d_base));
    return BGD_OK;
}

}  // extern "C"
