// hc_stage.cu -- see hc_stage.h
#include "hc_stage.h"
#include "../../include/hc_b200.h"

#include <omp.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <unistd.h>
#include <stdio.h>
#include <time.h>

namespace {

constexpr size_t kChunkMax = 8u << 20;     // bytes per pinned staging buffer
constexpr int kRing = 4;                   // buffers in flight
constexpr size_t kBlock = 256u << 10;      // bytes per host thread task

size_t env_size(const char* name, size_t dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    const unsigned long long x = strtoull(v, nullptr, 0);
    return x ? (size_t)x : dflt;
}
// HC_STAGE_MIN: copies below this many bytes take the driver's own path (default 2 MB); HC_STAGE_CHUNK: bytes per
// ring buffer (default and maximum 8 MB).  The tests set both to small values to run small inputs through the ring.
const size_t kDirectBelow = env_size("HC_STAGE_MIN", 2u << 20);
const size_t kChunk = [] { size_t c = env_size("HC_STAGE_CHUNK", kChunkMax); return c > kChunkMax ? kChunkMax : c; }();

struct Ring {
    unsigned char* buf[kRing] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev[kRing];
    cudaStream_t stream = nullptr;         // blocking stream: ordered with the legacy default stream
    bool ok = false;
    bool used[kRing] = {false, false, false, false};   // ev[b] has been recorded at least once
    int next = 0;                          // the buffers are handed out round robin, whichever call comes next
};

std::mutex g_mu;            // one staged copy at a time per process (the ring is shared)

// HC_STAGE_TIMING=1: where the staged copies spend their time (host memcpy / waiting for a ring buffer's DMA), on stderr at exit
struct StageTimes {
    bool on = getenv("HC_STAGE_TIMING") != nullptr;
    double copy_s[2] = {0, 0}, wait_s[2] = {0, 0}, bytes[2] = {0, 0};
    long calls[2] = {0, 0};
    static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; }
    ~StageTimes() {
        if (!on) return;
        for (int d = 0; d < 2; d++)
            fprintf(stderr, "[hc_stage] %s: %ld calls, %.1f MB, host memcpy %.1f ms, waiting for DMAs %.1f ms\n", d ? "device->host" : "host->device",
                    calls[d], bytes[d] / 1e6, copy_s[d] * 1e3, wait_s[d] * 1e3);
    }
} g_times;
Ring g_ring[16];            // per device

cudaError_t ring_for(int dev, Ring** out) {
    Ring& r = g_ring[dev & 15];
    if (!r.ok) {
        cudaError_t e = cudaStreamCreate(&r.stream);
        if (e != cudaSuccess) return e;
        for (int i = 0; i < kRing; i++) {
            e = cudaHostAlloc(reinterpret_cast<void**>(&r.buf[i]), kChunkMax, cudaHostAllocPortable);
            if (e != cudaSuccess) return e;
            e = cudaEventCreateWithFlags(&r.ev[i], cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
        }
        r.ok = true;
    }
    *out = &r;
    return cudaSuccess;
}

bool is_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

int host_threads() {      // HC_STAGE_THREADS: host threads that copy between the caller's buffer and the pinned ring (default: up to 16)
    static const int cap = (int)env_size("HC_STAGE_THREADS", 16);
    int t = omp_get_max_threads();
    if (t > cap) t = cap;
    return t < 1 ? 1 : t;
}

void par_memcpy(void* dst, const void* src, size_t bytes, int threads) {
    const long nb = (long)((bytes + kBlock - 1) / kBlock);
    if (threads <= 1 || nb <= 1 || omp_in_parallel()) { memcpy(dst, src, bytes); return; }
#pragma omp parallel for schedule(static) num_threads(threads)
    for (long b = 0; b < nb; b++) {
        const size_t o = (size_t)b * kBlock;
        memcpy(static_cast<char*>(dst) + o, static_cast<const char*>(src) + o, bytes - o < kBlock ? bytes - o : kBlock);
    }
}

}  // namespace

cudaError_t hc_copy_h2d(void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < kDirectBelow || is_pinned(src)) return cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    Ring* r;
    if ((e = ring_for(dev, &r)) != cudaSuccess) return e;
    const int T = host_threads();
    size_t done = 0;
    for (int i = 0; done < bytes; i++) {
        const int b = r->next;
        r->next = (r->next + 1) % kRing;
        const size_t n = bytes - done < kChunk ? bytes - done : kChunk;
        if (r->used[b] && (e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;   // the DMA that read this buffer
        par_memcpy(r->buf[b], static_cast<const char*>(src) + done, n, T);
        if ((e = cudaMemcpyAsync(static_cast<char*>(dst) + done, r->buf[b], n, cudaMemcpyHostToDevice, r->stream)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(r->ev[b], r->stream)) != cudaSuccess) return e;
        r->used[b] = true;
        done += n;
    }
    return cudaStreamSynchronize(r->stream);
}

cudaError_t hc_copy_d2h(void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < kDirectBelow || is_pinned(dst)) return cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    Ring* r;
    if ((e = ring_for(dev, &r)) != cudaSuccess) return e;
    const int T = host_threads();
    const size_t nchunks = (bytes + kChunk - 1) / kChunk;
    size_t issued = 0, drained = 0;
    int slot[kRing];
    while (drained < nchunks) {
        while (issued < nchunks && issued < drained + kRing) {   // keep the ring full of DMAs
            const int b = r->next;
            r->next = (r->next + 1) % kRing;
            slot[issued % kRing] = b;
            const size_t o = issued * kChunk, n = bytes - o < kChunk ? bytes - o : kChunk;
            if (r->used[b] && (e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;   // a DMA of an earlier call may still use it
            if ((e = cudaMemcpyAsync(r->buf[b], static_cast<const char*>(src) + o, n, cudaMemcpyDeviceToHost, r->stream)) != cudaSuccess) return e;
            if ((e = cudaEventRecord(r->ev[b], r->stream)) != cudaSuccess) return e;
            r->used[b] = true;
            issued++;
        }
        const int b = slot[drained % kRing];
        const size_t o = drained * kChunk, n = bytes - o < kChunk ? bytes - o : kChunk;
        if ((e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;
        par_memcpy(static_cast<char*>(dst) + o, r->buf[b], n, T);
        drained++;
    }
    return cudaSuccess;
}

cudaError_t hc_copy_file_h2d(void* dst, int fd, size_t bytes, size_t* got) {
    if (got) *got = 0;
    if (bytes == 0) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    Ring* r;
    if ((e = ring_for(dev, &r)) != cudaSuccess) return e;
    const int T = host_threads();
    size_t done = 0;
    bool eof = false;
    while (done < bytes && !eof) {
        const int b = r->next;
        r->next = (r->next + 1) % kRing;
        const size_t n = bytes - done < kChunk ? bytes - done : kChunk;
        if (r->used[b] && (e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;
        const long nb = (long)((n + kBlock - 1) / kBlock);
        long short_at = nb;                      // first block that came back short (end of file before `bytes`)
        size_t short_len = 0;
#pragma omp parallel for schedule(static) num_threads(T)
        for (long q = 0; q < nb; q++) {
            const size_t o = (size_t)q * kBlock, want = n - o < kBlock ? n - o : kBlock;
            size_t have = 0;
            while (have < want) {
                const ssize_t k = pread(fd, r->buf[b] + o + have, want - have, (off_t)(done + o + have));
                if (k <= 0) break;
                have += (size_t)k;
            }
            if (have < want) {
#pragma omp critical
                if (q < short_at) { short_at = q; short_len = have; }
            }
        }
        size_t valid = n;
        if (short_at < nb) { valid = (size_t)short_at * kBlock + short_len; eof = true; }
        if (valid) {
            if ((e = cudaMemcpyAsync(static_cast<char*>(dst) + done, r->buf[b], valid, cudaMemcpyHostToDevice, r->stream)) != cudaSuccess) return e;
            if ((e = cudaEventRecord(r->ev[b], r->stream)) != cudaSuccess) return e;
            r->used[b] = true;
        }
        done += valid;
    }
    if (got) *got = done;
    return cudaStreamSynchronize(r->stream);
}

cudaError_t hc_copy_h2d_on(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < (256u << 10) || is_pinned(src)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    Ring* r;
    if ((e = ring_for(dev, &r)) != cudaSuccess) return e;
    const int T = host_threads();
    // a buffer is free again when the DMA that read it -- on whichever stream it was issued last -- has completed: the
    // events are recorded on that stream, so waiting on them is enough whatever stream comes next
    size_t done = 0;
    for (int i = 0; done < bytes; i++) {
        const int b = r->next;
        r->next = (r->next + 1) % kRing;
        const size_t n = bytes - done < kChunk ? bytes - done : kChunk;
        const double ta = g_times.on ? StageTimes::now() : 0;
        if (r->used[b] && (e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;
        const double tb = g_times.on ? StageTimes::now() : 0;
        par_memcpy(r->buf[b], static_cast<const char*>(src) + done, n, T);
        if (g_times.on) { const double tc = StageTimes::now(); g_times.wait_s[0] += tb - ta; g_times.copy_s[0] += tc - tb; g_times.bytes[0] += n; g_times.calls[0] += i == 0; }
        if ((e = cudaMemcpyAsync(static_cast<char*>(dst) + done, r->buf[b], n, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(r->ev[b], st)) != cudaSuccess) return e;
        r->used[b] = true;
        done += n;
    }
    return cudaSuccess;
}

cudaError_t hc_copy_d2h_on(void* dst, const void* src, size_t bytes, cudaStream_t st, bool* completed) {
    if (completed) *completed = false;
    if (bytes == 0) return cudaSuccess;
    if (bytes < (256u << 10) || is_pinned(dst)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_mu);
    Ring* r;
    if ((e = ring_for(dev, &r)) != cudaSuccess) return e;
    const int T = host_threads();
    const size_t nchunks = (bytes + kChunk - 1) / kChunk;
    size_t issued = 0, drained = 0;
    int slot[kRing];
    while (drained < nchunks) {
        while (issued < nchunks && issued < drained + kRing) {   // keep the ring full of DMAs
            const int b = r->next;
            r->next = (r->next + 1) % kRing;
            slot[issued % kRing] = b;
            const size_t o = issued * kChunk, n = bytes - o < kChunk ? bytes - o : kChunk;
            if (r->used[b] && (e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;   // a host->device DMA may still read it
            if ((e = cudaMemcpyAsync(r->buf[b], static_cast<const char*>(src) + o, n, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
            if ((e = cudaEventRecord(r->ev[b], st)) != cudaSuccess) return e;
            r->used[b] = true;
            issued++;
        }
        const int b = slot[drained % kRing];
        const size_t o = drained * kChunk, n = bytes - o < kChunk ? bytes - o : kChunk;
        const double ta = g_times.on ? StageTimes::now() : 0;
        if ((e = cudaEventSynchronize(r->ev[b])) != cudaSuccess) return e;
        const double tb = g_times.on ? StageTimes::now() : 0;
        par_memcpy(static_cast<char*>(dst) + o, r->buf[b], n, T);
        if (g_times.on) { const double tc = StageTimes::now(); g_times.wait_s[1] += tb - ta; g_times.copy_s[1] += tc - tb; g_times.bytes[1] += n; g_times.calls[1] += drained == 0; }
        drained++;
    }
    if (completed) *completed = true;
    return cudaSuccess;
}

cudaError_t hc_scratch_alloc(void** p, size_t bytes) { return hc_scratch_alloc_on(p, bytes, 0); }

void hc_scratch_free(void* p) { hc_scratch_free_on(p, 0); }

cudaError_t hc_scratch_alloc_on(void** p, size_t bytes, cudaStream_t st) {
    static std::mutex mu;
    static bool tuned[16] = {false};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!tuned[dev & 15]) {
            cudaMemPool_t pool;
            if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                unsigned long long keep = 16ull << 30;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            cudaGetLastError();
            tuned[dev & 15] = true;
        }
    }
    return cudaMallocAsync(p, bytes ? bytes : 1, st);
}

void hc_scratch_free_on(void* p, cudaStream_t st) {
    if (p) cudaFreeAsync(p, st);
}

int hc_cuda_fail(const char* who, const char* call, cudaError_t e) {
    hc_set_last_error((std::string(who) + ": " + call + ": " + cudaGetErrorString(e)).c_str());
    if (e != cudaErrorMemoryAllocation) return HC_ERR_CUDA;
    cudaGetLastError();
    return HC_ERR_NOMEM;
}

double hc_now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

// ---- pinned host memory for callers of the host-buffer entry points (include/hc_b200.h) -----------------------------------
extern "C" void* hc_host_alloc(uint64_t bytes, int write_combined) {
    void* p = nullptr;
    const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
    if (cudaHostAlloc(&p, bytes ? (size_t)bytes : 1, flags) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void hc_host_free(void* p) {
    if (p) cudaFreeHost(p);
}
