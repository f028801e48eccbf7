// Runtime plumbing of oflib_b200: error reporting, device/stream/memory wrappers for the ctypes shim, and the
// host-buffer entry points (ofh_*) that stream frames through a small ring of device buffers so host<->device copies
// overlap the kernels.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <mutex>

#include "ofk_common.cuh"

namespace ofk {

static thread_local char t_error[512] = "";
std::atomic<unsigned long long> g_launches{0};
std::atomic<unsigned long long> g_paths[4];
std::atomic<unsigned long long> g_consistency_paths[2];

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_error, sizeof(t_error), fmt, ap);
    va_end(ap);
}

int sm_count() {
    static std::atomic<int> cached[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cached[dev] = v;
    }
    return cached[dev];
}

}  // namespace ofk

using namespace ofk;

extern "C" const char* ofk_last_error(void) { return t_error; }
extern "C" int ofk_version(void) { return OFK_VERSION; }
extern "C" unsigned long long ofk_rt_launch_count(void) { return g_launches.load(); }
extern "C" unsigned long long ofk_rt_path_count(int which) {
    if (which >= 0 && which < 4) return g_paths[which].load();
    if (which == 4) return c3_ws_mixed_count();      // synchronous reads of device counters (current device)
    if (which == 5) return warp_ws_mixed_count();
    if (which == 12 || which == 13) return g_consistency_paths[which - 12].load();
    if (which >= 6 && which <= 21) return forward_s_stat(which - 6);
    return 0ull;
}

// ------------------------------------------------------------------------------------------------------- runtime
extern "C" int ofk_rt_device_count(int* count) {
    OFK_CHECK_ARG(count, "ofk_rt_device_count: NULL");
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) {
        *count = 0;
        set_error("cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return OFK_ECUDA;
    }
    return OFK_OK;
}
extern "C" int ofk_rt_set_device(int device) {
    OFK_CUDA(cudaSetDevice(device));
    return OFK_OK;
}
extern "C" int ofk_rt_get_device(int* device) {
    OFK_CHECK_ARG(device, "ofk_rt_get_device: NULL");
    OFK_CUDA(cudaGetDevice(device));
    return OFK_OK;
}
extern "C" int ofk_rt_device_info(int device, int* sm, int* cc_major, int* cc_minor, size_t* l2_bytes,
                                  size_t* total_mem) {
    cudaDeviceProp p;
    OFK_CUDA(cudaGetDeviceProperties(&p, device));
    if (sm) *sm = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (l2_bytes) *l2_bytes = (size_t)p.l2CacheSize;
    if (total_mem) *total_mem = p.totalGlobalMem;
    return OFK_OK;
}

// stream-ordered pool allocation: freed blocks stay cached in the device's default mempool (release threshold
// raised to "never"), so the per-call allocations of the Python shim cost microseconds, not cudaMalloc round trips.
static int ensure_pool(int dev) {
    static std::mutex mu;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lk(mu);
    if (dev < 0 || dev >= 64 || done[dev]) return OFK_OK;
    cudaMemPool_t pool;
    OFK_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    unsigned long long thr = ~0ull;
    OFK_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    done[dev] = true;
    return OFK_OK;
}
extern "C" int ofk_rt_malloc(void** dptr, size_t bytes, ofk_stream_t stream) {
    OFK_CHECK_ARG(dptr, "ofk_rt_malloc: NULL");
    int dev = 0;
    OFK_CUDA(cudaGetDevice(&dev));
    int rc = ensure_pool(dev);
    if (rc != OFK_OK) return rc;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMallocAsync(dptr, bytes, as_stream(stream));
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        set_error("device allocation of %zu bytes failed", bytes);
        return OFK_ENOMEM;
    }
    OFK_CUDA(e);
    return OFK_OK;
}
extern "C" int ofk_rt_free(void* dptr, ofk_stream_t stream) {
    if (dptr == nullptr) return OFK_OK;
    OFK_CUDA(cudaFreeAsync(dptr, as_stream(stream)));
    return OFK_OK;
}
extern "C" int ofk_rt_host_alloc(void** hptr, size_t bytes) {
    OFK_CHECK_ARG(hptr, "ofk_rt_host_alloc: NULL");
    OFK_CUDA(cudaHostAlloc(hptr, bytes ? bytes : 16, cudaHostAllocPortable));
    return OFK_OK;
}
extern "C" int ofk_rt_host_free(void* hptr) {
    if (hptr) OFK_CUDA(cudaFreeHost(hptr));
    return OFK_OK;
}
extern "C" int ofk_rt_host_register(void* hptr, size_t bytes) {
    OFK_CUDA(cudaHostRegister(hptr, bytes, cudaHostRegisterPortable));
    return OFK_OK;
}
extern "C" int ofk_rt_host_unregister(void* hptr) {
    OFK_CUDA(cudaHostUnregister(hptr));
    return OFK_OK;
}
// Large copies from / to pageable memory go through staging.cu (worker threads + pinned pieces); everything else is a
// plain cudaMemcpyAsync.
extern "C" int ofk_rt_memcpy_h2d(void* dst, const void* src, size_t bytes, ofk_stream_t s) {
    if (bytes == 0) return OFK_OK;
    const int staged = staged_copy(dst, src, bytes, true, as_stream(s));
    if (staged < 0) return staged;
    if (staged == 0) OFK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_memcpy_d2h(void* dst, const void* src, size_t bytes, ofk_stream_t s) {
    if (bytes == 0) return OFK_OK;
    const int staged = staged_copy(dst, src, bytes, false, as_stream(s));
    if (staged < 0) return staged;
    if (staged == 0) OFK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_memcpy_d2d(void* dst, const void* src, size_t bytes, ofk_stream_t s) {
    if (bytes) OFK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_memset(void* dst, int value, size_t bytes, ofk_stream_t s) {
    if (bytes) OFK_CUDA(cudaMemsetAsync(dst, value, bytes, as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_stream_create(ofk_stream_t* s) {
    OFK_CHECK_ARG(s, "ofk_rt_stream_create: NULL");
    cudaStream_t st;
    OFK_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    *s = (ofk_stream_t)st;
    return OFK_OK;
}
extern "C" int ofk_rt_stream_destroy(ofk_stream_t s) {
    if (s) OFK_CUDA(cudaStreamDestroy(as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_stream_sync(ofk_stream_t s) {
    OFK_CUDA(cudaStreamSynchronize(as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_device_sync(void) {
    OFK_CUDA(cudaDeviceSynchronize());
    return OFK_OK;
}
extern "C" int ofk_rt_event_create(void** ev) {
    OFK_CHECK_ARG(ev, "ofk_rt_event_create: NULL");
    cudaEvent_t e;
    OFK_CUDA(cudaEventCreate(&e));
    *ev = (void*)e;
    return OFK_OK;
}
extern "C" int ofk_rt_event_destroy(void* ev) {
    if (ev) OFK_CUDA(cudaEventDestroy((cudaEvent_t)ev));
    return OFK_OK;
}
extern "C" int ofk_rt_event_record(void* ev, ofk_stream_t s) {
    OFK_CUDA(cudaEventRecord((cudaEvent_t)ev, as_stream(s)));
    return OFK_OK;
}
extern "C" int ofk_rt_stream_wait_event(ofk_stream_t s, void* ev) {
    OFK_CUDA(cudaStreamWaitEvent(as_stream(s), (cudaEvent_t)ev, 0));
    return OFK_OK;
}
extern "C" int ofk_rt_event_sync(void* ev) {
    OFK_CUDA(cudaEventSynchronize((cudaEvent_t)ev));
    return OFK_OK;
}
extern "C" int ofk_rt_event_elapsed_ms(void* a, void* b, float* ms) {
    OFK_CHECK_ARG(ms, "ofk_rt_event_elapsed_ms: NULL");
    OFK_CUDA(cudaEventElapsedTime(ms, (cudaEvent_t)a, (cudaEvent_t)b));
    return OFK_OK;
}

// ------------------------------------------------------------------------------------------------ host-buffer API
namespace {

constexpr int kSlots = 3;
constexpr size_t kChunkTarget = 48u << 20;  // ~48 MiB of traffic per chunk keeps PCIe busy without hoarding HBM
constexpr size_t kFlagBytes = 2 * sizeof(int);  // per frame: the zero flags of ofk_combine3
constexpr int kMaxBuffers = 11;             // device buffers of one chunk (ofh_apply_combine3 has the most)
constexpr int kMaxPieces = 2;               // staged results of one call (ofh_evaluate: counts and sums)

// Small per-frame results (the zero flags of ofh_combine3, the rows of ofh_evaluate) that come back through the slot's
// pinned staging buffer: a device-to-host copy into the caller's pageable array would block the host until the chunk
// has finished and serialise the ring. The last device buffer of a chunk holds the pieces one after another, each
// frame_bytes[i] for every frame of the chunk; piece i belongs at dst[i] + n0 * frame_bytes[i].
struct Staged {
    void* dst[kMaxPieces] = {};
    size_t frame_bytes[kMaxPieces] = {};
    size_t total() const {
        size_t t = 0;
        for (int i = 0; i < kMaxPieces; ++i) t += dst[i] ? frame_bytes[i] : 0;
        return t;
    }
};

struct Slot {
    cudaStream_t st = nullptr;
    char* dev = nullptr;
    size_t cap = 0;
    char* hstage = nullptr;      // pinned
    size_t hstage_cap = 0;       // bytes
    char* pending_dst[kMaxPieces] = {};   // where the staged pieces of the chunk in flight belong
    size_t pending_bytes[kMaxPieces] = {};
    void deliver() {             // call after the slot's stream has drained
        size_t off = 0;
        for (int i = 0; i < kMaxPieces; ++i) {
            if (pending_dst[i] != nullptr && pending_bytes[i]) memcpy(pending_dst[i], hstage + off, pending_bytes[i]);
            off += pending_bytes[i];
            pending_dst[i] = nullptr;
            pending_bytes[i] = 0;
        }
    }
};
struct Ring {
    int device = -1;
    Slot slot[kSlots];
    std::mutex mu;
};
Ring g_ring;

void ring_free() {
    if (g_ring.device < 0) return;
    cudaSetDevice(g_ring.device);
    for (auto& s : g_ring.slot) {
        if (s.st) cudaStreamSynchronize(s.st);
        if (s.dev) cudaFree(s.dev);
        if (s.hstage) cudaFreeHost(s.hstage);
        if (s.st) cudaStreamDestroy(s.st);
        s = Slot();
    }
    g_ring.device = -1;
}

int ring_prepare(int device, size_t bytes_per_slot, size_t stage_bytes) {
    if (g_ring.device != device) {
        ring_free();
        g_ring.device = device;
    }
    OFK_CUDA(cudaSetDevice(device));
    for (auto& s : g_ring.slot) {
        for (int i = 0; i < kMaxPieces; ++i) {   // nothing is pending between calls (a call that failed half-way
            s.pending_dst[i] = nullptr;          // drops its staged results)
            s.pending_bytes[i] = 0;
        }
        if (!s.st) OFK_CUDA(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
        if (s.cap < bytes_per_slot) {
            if (s.dev) {
                OFK_CUDA(cudaStreamSynchronize(s.st));
                OFK_CUDA(cudaFree(s.dev));
                s.dev = nullptr;
                s.cap = 0;
            }
            cudaError_t e = cudaMalloc((void**)&s.dev, bytes_per_slot);
            if (e != cudaSuccess) {
                cudaGetLastError();
                set_error("ring allocation of %zu bytes failed: %s", bytes_per_slot, cudaGetErrorString(e));
                return OFK_ENOMEM;
            }
            s.cap = bytes_per_slot;
        }
        if (s.hstage_cap < stage_bytes) {
            if (s.hstage) OFK_CUDA(cudaFreeHost(s.hstage));
            s.hstage = nullptr;
            s.hstage_cap = 0;
            OFK_CUDA(cudaHostAlloc((void**)&s.hstage, stage_bytes, cudaHostAllocDefault));
            s.hstage_cap = stage_bytes;
        }
    }
    return OFK_OK;
}

// ofh_* calls run on the device they are given and leave the caller's current device as they found it.
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            cudaGetLastError();
            prev = -1;
        }
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Leaves no transfer in flight when an ofh_* call returns, on the error paths too: the copies read and write the
// caller's buffers, which may be freed as soon as the call is over.
struct DrainRing {
    ~DrainRing() {
        for (auto& s : g_ring.slot)
            if (s.st) cudaStreamSynchronize(s.st);
    }
};

size_t esize(int dtype) {
    switch (dtype) {
        case OFK_U8: return 1;
        case OFK_I16:
        case OFK_U16: return 2;
        case OFK_F32: return 4;
        default: return 8;
    }
}
size_t pad256(size_t b) { return (b + 255) & ~size_t(255); }

// Copies of the ring: pinned / registered user buffers -> plain asynchronous copies on the slot's stream (they overlap
// with the other slots); pageable buffers (plain numpy arrays) -> staging.cu (worker threads + pinned pieces), where the
// upload returns once the source has been read and the download once the destination is complete.
int ring_copy(void* dst, const void* src, size_t bytes, bool to_device, cudaStream_t st) {
    if (bytes == 0) return OFK_OK;
    const int staged = staged_copy(dst, src, bytes, to_device, st);
    if (staged < 0) return staged;
    if (staged == 0)
        OFK_CUDA(cudaMemcpyAsync(dst, src, bytes, to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost, st));
    return OFK_OK;
}
#define OFH_TRY(call)                                                                  \
    do {                                                                               \
        const int rc_ = (call);                                                        \
        if (rc_ != OFK_OK) return rc_;                                                 \
    } while (0)

// Frames [n0, n0 + cn) of a ring pass on one slot: cn frames of each buffer the call listed, packed into the slot (a
// buffer of 0 bytes per frame is absent: nullptr, and its copies do nothing).
struct Chunk {
    Slot* slot = nullptr;
    int n0 = 0, cn = 0;
    const size_t* frame_bytes = nullptr;
    char* buf[kMaxBuffers] = {};

    Chunk() = default;
    Chunk(Slot& s, int n0_, int cn_, const size_t* frame_bytes_, int nbuf)
        : slot(&s), n0(n0_), cn(cn_), frame_bytes(frame_bytes_) {
        size_t off = 0;
        for (int i = 0; i < nbuf; ++i) {
            buf[i] = frame_bytes[i] ? s.dev + off : nullptr;
            off += pad256(frame_bytes[i] * cn);
        }
    }
    template <class T = void>
    T* at(int i) const { return (T*)buf[i]; }
    ofk_stream_t stream() const { return (ofk_stream_t)slot->st; }
    // buffer i from / to the caller's array of all N frames
    int in(int i, const void* host) const {
        return ring_copy(buf[i], (const char*)host + n0 * frame_bytes[i], frame_bytes[i] * cn, true, slot->st);
    }
    int out(void* host, int i) const {
        return ring_copy((char*)host + n0 * frame_bytes[i], buf[i], frame_bytes[i] * cn, false, slot->st);
    }
};

// One pass of N frames through the ring, in chunks of as many frames as kChunkTarget holds, the slots taken in turn.
// frame_bytes lists the device buffers of a chunk in bytes per frame. launch(chunk) queues the chunk's uploads and
// kernels on its slot's stream; download(chunk) queues its downloads, after the NEXT chunk has been launched: with
// pageable user buffers a download blocks the host, and this order keeps the device busy meanwhile (with pinned buffers
// the order is irrelevant, every copy is asynchronous). The pieces of `staged` come back through the slot's pinned
// staging from the last buffer (see Staged).
template <int NB, class Launch, class Download>
int run_ring(int device, int N, const size_t (&frame_bytes)[NB], const Staged& staged, Launch&& launch,
             Download&& download) {
    static_assert(NB <= kMaxBuffers, "raise kMaxBuffers");
    if (N == 0) return OFK_OK;
    std::lock_guard<std::mutex> lk(g_ring.mu);
    DeviceGuard restore_device;
    size_t per_frame = 0;
    for (size_t b : frame_bytes) per_frame += b;
    const int cf = (int)std::min<size_t>(N, std::max<size_t>(1, kChunkTarget / per_frame));
    size_t per_slot = 0;
    for (size_t b : frame_bytes) per_slot += pad256(b * cf);
    OFH_TRY(ring_prepare(device, per_slot, staged.total() * cf));
    DrainRing drain_on_exit;
    auto finish = [&](const Chunk& c) -> int {
        OFH_TRY(download(c));
        if (staged.total()) {
            Slot& s = *c.slot;
            OFK_CUDA(cudaMemcpyAsync(s.hstage, c.buf[NB - 1], staged.total() * c.cn, cudaMemcpyDeviceToHost, s.st));
            for (int i = 0; i < kMaxPieces; ++i) {
                char* dst = (char*)staged.dst[i];
                s.pending_dst[i] = dst ? dst + (size_t)c.n0 * staged.frame_bytes[i] : nullptr;
                s.pending_bytes[i] = dst ? staged.frame_bytes[i] * c.cn : 0;
            }
        }
        return OFK_OK;
    };
    Chunk prev;
    for (int n0 = 0, k = 0; n0 < N; n0 += cf, ++k) {
        Slot& s = g_ring.slot[k % kSlots];
        // a slot is reused only after everything queued on its stream has drained (keeps device buffers private)
        OFK_CUDA(cudaStreamSynchronize(s.st));
        s.deliver();
        const Chunk c(s, n0, std::min(cf, N - n0), frame_bytes, NB);
        OFH_TRY(launch(c));
        if (prev.cn) OFH_TRY(finish(prev));
        prev = c;
    }
    OFH_TRY(finish(prev));
    for (auto& s : g_ring.slot) {
        OFK_CUDA(cudaStreamSynchronize(s.st));
        s.deliver();
    }
    return OFK_OK;
}

}  // namespace

extern "C" int ofh_warp_t(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
                          const uint8_t* payload_mask, const uint8_t* flow_mask, void* out, uint8_t* out_mask,
                          int mask_rule, int N, int H, int W, int device) {
    OFK_CHECK_ARG(flow != nullptr && N >= 0 && H > 0 && W > 0 && C >= 0, "ofh_warp_t: bad arguments");
    OFK_CHECK_ARG(dtype >= OFK_U8 && dtype <= OFK_F64, "ofh_warp_t: unknown dtype %d", dtype);
    const size_t px = (size_t)H * W, b_pay = px * C * esize(dtype);
    // float payloads need apply_flow's pass-through of zero flows (ofk_warp_t_ex); integer payloads come out of the
    // identity taps unchanged
    const bool pass = C > 0 && (dtype == OFK_F32 || dtype == OFK_F64);
    enum { kFlow, kPay, kOut, kPm, kFm, kOm, kNz };
    return run_ring(
        device, N,
        {px * 8, b_pay, b_pay, payload_mask ? px : 0, flow_mask ? px : 0, out_mask ? px : 0, pass ? sizeof(int) : 0},
        Staged(),
        [&](const Chunk& c) {
            OFH_TRY(c.in(kFlow, flow));
            OFH_TRY(c.in(kPay, payload));
            OFH_TRY(c.in(kPm, payload_mask));
            OFH_TRY(c.in(kFm, flow_mask));
            if (pass) OFH_TRY(ofk_nonzero_flags(c.at<float>(kFlow), nullptr, 1e-3f, c.at<int>(kNz), c.cn, H, W,
                                                c.stream()));
            return ofk_warp_t_ex(c.at(kPay), dtype, C, arith, c.at<float>(kFlow), flow_sign, c.at<uint8_t>(kPm),
                                 c.at<uint8_t>(kFm), c.at<int>(kNz), c.at(kOut), c.at<uint8_t>(kOm), mask_rule, c.cn,
                                 H, W, H, W, 0, 0, 1, c.stream());
        },
        [&](const Chunk& c) {
            OFH_TRY(c.out(out, kOut));
            return c.out(out_mask, kOm);
        });
}

extern "C" int ofh_combine3(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, int ref, float thr,
                            float* out, uint8_t* out_mask, int* flags, int N, int H, int W, int device) {
    OFK_CHECK_ARG(A && B && out && out_mask && N >= 0 && H > 0 && W > 0, "ofh_combine3: bad arguments");
    const size_t px = (size_t)H * W, b_flow = px * 8;
    enum { kA, kB, kO, kAm, kBm, kOm, kF };
    return run_ring(
        device, N, {b_flow, b_flow, b_flow, Am ? px : 0, Bm ? px : 0, px, kFlagBytes}, Staged{{flags}, {kFlagBytes}},
        [&](const Chunk& c) {
            OFH_TRY(c.in(kA, A));
            OFH_TRY(c.in(kB, B));
            OFH_TRY(c.in(kAm, Am));
            OFH_TRY(c.in(kBm, Bm));
            return ofk_combine3(c.at<float>(kA), c.at<uint8_t>(kAm), c.at<float>(kB), c.at<uint8_t>(kBm), ref, thr,
                                c.at<float>(kO), c.at<uint8_t>(kOm), c.at<int>(kF), c.cn, H, W, c.stream());
        },
        [&](const Chunk& c) {
            OFH_TRY(c.out(out, kO));
            return c.out(out_mask, kOm);
        });
}

// The pair of calls a frame pipeline makes per batch -- `A.apply(image, return_valid_area=True)` and
// `A.combine_with(B, 3)` -- on host buffers in one pass of the ring: A and its mask are uploaded ONCE and feed both
// kernels of a chunk (two separate calls upload them twice: 30 bytes per pixel in, this 21).
extern "C" int ofh_apply_combine3(const void* image, int dtype, int C, int arith, int mask_rule, const float* A,
                                  const uint8_t* Am, const float* B, const uint8_t* Bm, int ref, float thr,
                                  void* out_image, uint8_t* out_valid, float* out, uint8_t* out_mask, int* flags, int N,
                                  int H, int W, int device) {
    OFK_CHECK_ARG(image && A && B && out_image && out && out_mask && N >= 0 && H > 0 && W > 0 && C > 0,
                  "ofh_apply_combine3: bad arguments");
    OFK_CHECK_ARG(dtype >= OFK_U8 && dtype <= OFK_F64, "ofh_apply_combine3: unknown dtype %d", dtype);
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofh_apply_combine3: ref must be 's' or 't'");
    const size_t px = (size_t)H * W, b_flow = px * 8, b_img = px * C * esize(dtype);
    const bool pass = dtype == OFK_F32 || dtype == OFK_F64;    // zero-flow pass-through, as in ofh_warp_t
    enum { kA, kB, kO, kI, kOi, kAm, kBm, kOm, kOv, kNz, kF };
    return run_ring(
        device, N,
        {b_flow, b_flow, b_flow, b_img, b_img, Am ? px : 0, Bm ? px : 0, px, out_valid ? px : 0,
         pass ? sizeof(int) : 0, kFlagBytes},
        Staged{{flags}, {kFlagBytes}},
        [&](const Chunk& c) {
            OFH_TRY(c.in(kA, A));
            OFH_TRY(c.in(kAm, Am));
            OFH_TRY(c.in(kI, image));
            if (pass) OFH_TRY(ofk_nonzero_flags(c.at<float>(kA), nullptr, 1e-3f, c.at<int>(kNz), c.cn, H, W,
                                                c.stream()));
            // the image warp starts while B is still on its way
            OFH_TRY(ofk_warp_t_ex(c.at(kI), dtype, C, arith, c.at<float>(kA), ref == 't' ? -1.0f : 1.0f, nullptr,
                                  out_valid ? c.at<uint8_t>(kAm) : nullptr, c.at<int>(kNz), c.at(kOi),
                                  c.at<uint8_t>(kOv), mask_rule, c.cn, H, W, H, W, 0, 0, 1, c.stream()));
            OFH_TRY(c.in(kB, B));
            OFH_TRY(c.in(kBm, Bm));
            return ofk_combine3(c.at<float>(kA), c.at<uint8_t>(kAm), c.at<float>(kB), c.at<uint8_t>(kBm), ref, thr,
                                c.at<float>(kO), c.at<uint8_t>(kOm), c.at<int>(kF), c.cn, H, W, c.stream());
        },
        [&](const Chunk& c) {
            OFH_TRY(c.out(out_image, kOi));
            OFH_TRY(c.out(out_valid, kOv));
            OFH_TRY(c.out(out, kO));
            return c.out(out_mask, kOm);
        });
}

// Flow.visualise of N host frames: with the default range (range_max == 0) each chunk carries the magnitudes and
// selection records of ofk_visualise_batch as a per-frame buffer that is never copied.
extern "C" int ofh_visualise(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask,
                             int show_mask_borders, float range_max, uint8_t* out, int N, int H, int W, int device) {
    OFK_CHECK_ARG(flow && out && N >= 0 && H > 0 && W > 0, "ofh_visualise: bad arguments");
    OFK_CHECK_ARG((size_t)H * W < (1ull << 31), "ofh_visualise: a frame needs fewer than 2^31 pixels");
    OFK_CHECK_ARG(mode >= 0 && mode <= 2, "ofh_visualise: mode must be 0 (hsv), 1 (rgb) or 2 (bgr)");
    OFK_CHECK_ARG(range_max >= 0.f, "ofh_visualise: range_max must be positive, or 0 for the default range");
    const size_t px = (size_t)H * W, b_ws = range_max > 0.f ? 0 : ofk_visualise_batch_workspace(1, H, W);
    enum { kFlow, kMask, kOut, kWs };
    return run_ring(
        device, N, {px * 8, mask ? px : 0, px * 3, b_ws}, Staged(),
        [&](const Chunk& c) {
            OFH_TRY(c.in(kFlow, flow));
            OFH_TRY(c.in(kMask, mask));
            return ofk_visualise_batch(c.at<float>(kFlow), c.at<uint8_t>(kMask), thr, mode, show_mask,
                                       show_mask_borders, range_max, c.at<uint8_t>(kOut), c.cn, H, W, c.at(kWs),
                                       b_ws * c.cn, c.stream());
        },
        [&](const Chunk& c) { return c.out(out, kOut); });
}

// Error metrics of N host frames: the partials of ofk_evaluate are a per-frame buffer that is never copied, and the
// rows (counts, then sums, of the chunk's frames) come back through the pinned staging.
extern "C" int ofh_evaluate(const float* est, const uint8_t* est_mask, const float* truth, const uint8_t* truth_mask,
                            const uint8_t* region, float* epe, long long* counts, double* sums, int N, int H, int W,
                            int device) {
    OFK_CHECK_ARG(est && truth && counts && sums && N >= 0 && H > 0 && W > 0, "ofh_evaluate: bad arguments");
    OFK_CHECK_ARG(N <= 65535, "ofh_evaluate: N = %d exceeds 65535 frames", N);
    OFK_CHECK_ARG((size_t)H * W < (1ull << 31), "ofh_evaluate: a frame needs fewer than 2^31 pixels");
    const size_t px = (size_t)H * W, b_ws = ofk_evaluate_workspace(1, H, W);
    const size_t b_counts = 8 * sizeof(long long), b_sums = 5 * sizeof(double);
    enum { kEst, kTruth, kEm, kTm, kRg, kEpe, kWs, kRows };
    return run_ring(
        device, N,
        {px * 8, px * 8, est_mask ? px : 0, truth_mask ? px : 0, region ? px : 0, epe ? px * 4 : 0, b_ws,
         b_counts + b_sums},
        Staged{{counts, sums}, {b_counts, b_sums}},
        [&](const Chunk& c) {
            OFH_TRY(c.in(kEst, est));
            OFH_TRY(c.in(kTruth, truth));
            OFH_TRY(c.in(kEm, est_mask));
            OFH_TRY(c.in(kTm, truth_mask));
            OFH_TRY(c.in(kRg, region));
            char* rows = c.at<char>(kRows);
            return ofk_evaluate(c.at<float>(kEst), c.at<uint8_t>(kEm), c.at<float>(kTruth), c.at<uint8_t>(kTm),
                                c.at<uint8_t>(kRg), c.at<float>(kEpe), (long long*)rows,
                                (double*)(rows + b_counts * c.cn), c.cn, H, W, c.at(kWs), b_ws * c.cn, c.stream());
        },
        [&](const Chunk& c) { return c.out(epe, kEpe); });
}

extern "C" int ofh_release(void) {
    std::lock_guard<std::mutex> lk(g_ring.mu);
    DeviceGuard restore_device;
    ring_free();
    return OFK_OK;
}
