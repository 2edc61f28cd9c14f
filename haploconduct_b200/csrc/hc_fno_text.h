// hc_fno_text.h -- what hc_fno.cu and hc_fno_text.cu share: the phase timer, the CUDA error macro, and the text stage
// that turns the compacted FNO records (still in HBM) into the bytes of overlaps.txt.
#ifndef HC_FNO_TEXT_H_
#define HC_FNO_TEXT_H_
#include <cstdio>
#include <cstdlib>
#include <string>
#include <time.h>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"

void hc_set_last_error(const char* msg);   // hc_api.cu

#define FCU(call)                                                                         \
    do {                                                                                  \
        cudaError_t _e = (call);                                                          \
        if (_e != cudaSuccess) {                                                          \
            hc_set_last_error((std::string(#call) + ": " + cudaGetErrorString(_e)).c_str()); \
            rc = HC_ERR_CUDA;                                                             \
            goto done;                                                                    \
        }                                                                                 \
    } while (0)

// HC_FNO_TIMING=1: phase times on stderr (synchronises the device at every mark)
struct FnoPhase {
    bool on;
    double t0;
    const char* who;
    static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
    explicit FnoPhase(const char* w) : on(getenv("HC_FNO_TIMING") != nullptr), t0(0), who(w) { if (on) t0 = now(); }
    void mark(const char* what) {
        if (!on) return;
        cudaDeviceSynchronize();
        const double t = now();
        fprintf(stderr, "[%s] %-28s %8.2f ms\n", who, what, t - t0);
        t0 = t;
    }
};

// Where the text goes and how it is ordered: FNO1 sorts the lines in byte order and drops repeats (the reference's
// std::set<std::string>), FNO3 keeps every line in record order.
struct FnoText {
    char* text;
    uint64_t cap;
    uint64_t *n_bytes, *n_lines;
    bool sort_unique;
};

// d_rec: n device records in output order, R = hc_fno_overlap_small or hc_fno_overlap.  Writes *n_bytes / *n_lines;
// HC_ERR_CAPACITY (sizes written, nothing copied) if t.cap < *n_bytes, HC_ERR_ARG if n >= 2^32.
template <class R>
int fno_text(const R* d_rec, uint64_t n, const FnoText& t, FnoPhase& ph, const char* who);

#endif
