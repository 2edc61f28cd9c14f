// hc_stage.h -- host<->device copies of large PAGEABLE buffers and stream-ordered device scratch for the
// host-buffer entry points (hc_fno1/3, hc_dedup_edges, hc_store_create*).  cudaMemcpy on pageable memory moves
// ~10 GB/s (one driver thread staging through one pinned buffer); the callers of the reference-facing ABI hold
// std::vector / numpy memory, so the library stages itself: several host threads copy into a ring of pinned
// buffers while the copy engine drains the previous one.  Pinned or registered buffers go straight to cudaMemcpy.
// Also what those entry points share: the scratch owner, the CUDA error path, the grid size and the clock.
#ifndef HC_STAGE_H_
#define HC_STAGE_H_
#include <cuda_runtime.h>
#include <stddef.h>

// Synchronous like cudaMemcpy: ordered after all earlier work of the device, complete on return.
cudaError_t hc_copy_h2d(void* dst_dev, const void* src_host, size_t bytes);
cudaError_t hc_copy_d2h(void* dst_host, const void* src_dev, size_t bytes);

// The same through the ring, but with the device side of the copy on a stream of the caller's (the pipelines of
// hc_ingest_overlaps and hc_score_batch*): pinned / registered host memory is handed to cudaMemcpyAsync as it is.
//   hc_copy_h2d_on returns when the last piece has been handed to the copy engine: `src` may be reused, the copies
//                  complete in stream order on `st` (the caller orders its kernels behind them with an event);
//   hc_copy_d2h_on returns when `dst` holds the data if `dst` is pageable; for pinned memory it only enqueues
//                  (cudaMemcpyAsync semantics) -- *completed says which.
cudaError_t hc_copy_h2d_on(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st);
cudaError_t hc_copy_d2h_on(void* dst_host, const void* src_dev, size_t bytes, cudaStream_t st, bool* completed);

// A file straight to the device: several host threads pread pieces of it into the pinned ring, the copy engine drains
// them -- the host never holds more than the ring (32 MB) of the file.  Reads `bytes` from offset 0 of `fd`; *got = bytes
// that arrived (less if the file is shorter).  Synchronous: the data is on the device on return.
cudaError_t hc_copy_file_h2d(void* dst_dev, int fd, size_t bytes, size_t* got);

// Device scratch from the device's default memory pool, ordered on the legacy default stream (the stream the
// host-buffer entry points launch on); freed memory stays in the pool (up to 16 GB), so that a call does not pay
// cudaMalloc / cudaFree for each of its dozen temporaries.
cudaError_t hc_scratch_alloc(void** p, size_t bytes);
void hc_scratch_free(void* p);
// the same on a stream of the caller's (the store's streams are non-blocking: they do not order with the default stream)
cudaError_t hc_scratch_alloc_on(void** p, size_t bytes, cudaStream_t st);
void hc_scratch_free_on(void* p, cudaStream_t st);

// One hc_scratch_alloc buffer of T, freed when the owner goes out of scope (or earlier, by reset()).
template <class T>
class ScratchBuf {
public:
    ScratchBuf() = default;
    ScratchBuf(const ScratchBuf&) = delete;
    ScratchBuf& operator=(const ScratchBuf&) = delete;
    ScratchBuf(ScratchBuf&& o) noexcept : p_(o.release()) {}
    ScratchBuf& operator=(ScratchBuf&& o) noexcept { if (this != &o) { reset(); p_ = o.release(); } return *this; }
    ~ScratchBuf() { reset(); }
    cudaError_t alloc(size_t count) { reset(); return hc_scratch_alloc(reinterpret_cast<void**>(&p_), count * sizeof(T)); }
    void reset() { hc_scratch_free(p_); p_ = nullptr; }
    T* release() { T* p = p_; p_ = nullptr; return p; }
    T* get() const { return p_; }
    operator T*() const { return p_; }
private:
    T* p_ = nullptr;
};

// The error path of the host-buffer entry points: sets "<who>: <call>: <CUDA's message>" as the last error and returns
// HC_ERR_NOMEM for a failed allocation (cleared, so that later calls do not report it), HC_ERR_CUDA for anything else.
void hc_set_last_error(const char* msg);   // hc_api.cu
int hc_cuda_fail(const char* who, const char* call, cudaError_t e);
// Evaluates `call`; on failure sets rc and jumps to `done` (both, and `who`, in the caller's scope).
#define HC_CU(call)                                                      \
    do {                                                                 \
        const cudaError_t _e = (call);                                   \
        if (_e != cudaSuccess) { rc = hc_cuda_fail(who, #call, _e); goto done; } \
    } while (0)

// Blocks of a grid-stride launch over n items: one per `threads` items, at least 1, at most 16 per SM of a B200.
inline int grid_for(unsigned long long n, int threads) {
    const unsigned long long b = (n + threads - 1) / threads;
    return (int)(b < 148 * 16 ? (b ? b : 1) : 148 * 16);
}

// CLOCK_MONOTONIC in milliseconds (the phase timers of the entry points)
double hc_now_ms();

#endif
