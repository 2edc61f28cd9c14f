// hc_prims_shim.cu -- test-only C entry points over the header-only primitives (hc_scan.cuh, hc_radix.cuh, hc_text.cuh),
// which have internal linkage and so cannot be reached through libhc_b200.so.  Every wrapper takes host arrays, copies
// them to the device, runs the primitive once on the legacy default stream and copies the device buffers back whole, so
// that the caller sees what the primitive wrote, and every guard entry behind it.  Built by haploconduct_b200/build.py
// into lib/libhc_prims_shim.so, linked against libhc_b200.so (hc_scratch_alloc / hc_scratch_free of hc_radix.cuh).
#include <cstdint>
#include <cuda_runtime.h>

#include "hc_radix.cuh"
#include "hc_scan.cuh"
#include "hc_text.cuh"

#define SCU(call)                                       \
    do {                                                \
        e = (call);                                     \
        if (e != cudaSuccess) goto done;                \
    } while (0)

namespace {
struct KeyLess {
    const uint64_t* key;
    __device__ bool operator()(uint32_t a, uint32_t b) const { return key[a] < key[b]; }
};

__global__ void sort_run_kernel(const uint64_t* key, uint32_t* idx, uint32_t m) { hc_radix::sort_run(idx, m, KeyLess{key}); }
}  // namespace

extern "C" {

// The sizes the primitives are built for: [hc_scan::THREADS, hc_scan::PER_BLOCK, hc_radix::THREADS, hc_radix::TILE,
// newline TILE of hc_text.cuh, scan_counts' block, hc_radix::RUN_INSERTION_MAX].  The tests derive their boundary sizes
// from these.
void hcp_constants(uint64_t* out) {
    out[0] = hc_scan::THREADS;
    out[1] = hc_scan::PER_BLOCK;
    out[2] = hc_radix::THREADS;
    out[3] = hc_radix::TILE;
    out[4] = TILE;
    out[5] = 1024;
    out[6] = hc_radix::RUN_INSERTION_MAX;
}

uint64_t hcp_blocks_for(uint64_t n) { return hc_scan::blocks_for(n); }

// hc_scan::exclusive_u32 over in[0, n).  out (out_len >= n entries) and bsum (bsum_len entries, at least the
// (n + PER_BLOCK - 1) / PER_BLOCK the scan uses) go to the device as the caller filled them and come back whole.
int hcp_exclusive_u32(const uint32_t* in, uint64_t n, uint64_t* out, uint64_t out_len, uint64_t* total, uint64_t* bsum,
                      uint64_t bsum_len) {
    uint32_t* d_in = nullptr;
    uint64_t *d_out = nullptr, *d_total = nullptr, *d_bsum = nullptr;
    cudaError_t e = cudaSuccess;
    if (out_len < n || bsum_len < (n + hc_scan::PER_BLOCK - 1) / hc_scan::PER_BLOCK) return (int)cudaErrorInvalidValue;
    SCU(cudaMalloc(&d_in, (n ? n : 1) * sizeof(uint32_t)));
    SCU(cudaMalloc(&d_out, (out_len ? out_len : 1) * sizeof(uint64_t)));
    SCU(cudaMalloc(&d_bsum, (bsum_len ? bsum_len : 1) * sizeof(uint64_t)));
    SCU(cudaMalloc(&d_total, sizeof(uint64_t)));
    SCU(cudaMemcpy(d_in, in, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    SCU(cudaMemcpy(d_out, out, out_len * sizeof(uint64_t), cudaMemcpyHostToDevice));
    SCU(cudaMemcpy(d_bsum, bsum, bsum_len * sizeof(uint64_t), cudaMemcpyHostToDevice));
    SCU(cudaMemcpy(d_total, total, sizeof(uint64_t), cudaMemcpyHostToDevice));
    hc_scan::exclusive_u32(d_in, n, (hc_scan::u64*)d_out, (hc_scan::u64*)d_total, (hc_scan::u64*)d_bsum, 0);
    SCU(cudaGetLastError());
    SCU(cudaDeviceSynchronize());
    SCU(cudaMemcpy(out, d_out, out_len * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(bsum, d_bsum, bsum_len * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(total, d_total, sizeof(uint64_t), cudaMemcpyDeviceToHost));
done:
    cudaFree(d_in); cudaFree(d_out); cudaFree(d_bsum); cudaFree(d_total);
    return (int)e;
}

// hc_radix::sort_pairs of n (key, value) pairs; keys are [n][2] uint64 (low 64 bits, high 64 bits).  The sorted pairs are
// copied back into keys / vals; *in_tmp = 1 when the result was in the temporary buffers, 0 when in the input ones.
int hcp_sort_pairs(uint64_t* keys, uint32_t* vals, uint64_t n, int* in_tmp) {
    ulonglong2 *d_k = nullptr, *d_kt = nullptr, *kres = nullptr;
    uint32_t *d_v = nullptr, *d_vt = nullptr, *vres = nullptr;
    const uint64_t m = n ? n : 1;
    cudaError_t e = cudaSuccess;
    *in_tmp = -1;
    SCU(cudaMalloc(&d_k, m * sizeof(ulonglong2)));
    SCU(cudaMalloc(&d_kt, m * sizeof(ulonglong2)));
    SCU(cudaMalloc(&d_v, m * sizeof(uint32_t)));
    SCU(cudaMalloc(&d_vt, m * sizeof(uint32_t)));
    SCU(cudaMemcpy(d_k, keys, n * sizeof(ulonglong2), cudaMemcpyHostToDevice));
    SCU(cudaMemcpy(d_v, vals, n * sizeof(uint32_t), cudaMemcpyHostToDevice));
    SCU(hc_radix::sort_pairs(d_k, d_v, d_kt, d_vt, n, &kres, &vres));
    SCU(cudaDeviceSynchronize());
    if (kres == d_k && vres == d_v) *in_tmp = 0;
    else if (kres == d_kt && vres == d_vt) *in_tmp = 1;
    else { e = cudaErrorUnknown; goto done; }       // keys and values in different buffers
    SCU(cudaMemcpy(keys, kres, n * sizeof(ulonglong2), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(vals, vres, n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
done:
    cudaFree(d_k); cudaFree(d_kt); cudaFree(d_v); cudaFree(d_vt);
    return (int)e;
}

// hc_radix::sort_run of the indices 0..m-1 of one run, ordered by key[index], on one thread; idx gets the permutation.
int hcp_sort_run(const uint64_t* keys, uint32_t m, uint32_t* idx) {
    uint64_t* d_k = nullptr;
    uint32_t* d_i = nullptr;
    cudaError_t e = cudaSuccess;
    for (uint32_t i = 0; i < m; i++) idx[i] = i;
    SCU(cudaMalloc(&d_k, (m ? m : 1) * sizeof(uint64_t)));
    SCU(cudaMalloc(&d_i, (m ? m : 1) * sizeof(uint32_t)));
    SCU(cudaMemcpy(d_k, keys, m * sizeof(uint64_t), cudaMemcpyHostToDevice));
    SCU(cudaMemcpy(d_i, idx, m * sizeof(uint32_t), cudaMemcpyHostToDevice));
    sort_run_kernel<<<1, 1>>>(d_k, d_i, m);
    SCU(cudaGetLastError());
    SCU(cudaDeviceSynchronize());
    SCU(cudaMemcpy(idx, d_i, m * sizeof(uint32_t), cudaMemcpyDeviceToHost));
done:
    cudaFree(d_k); cudaFree(d_i);
    return (int)e;
}

// hc_line_index of text[0, n) placed `offset` bytes past a 256-byte aligned device address, with newlines on both sides
// of it (a read outside the text would show up as extra lines).  line_start gets the n_newlines + 1 offsets if cap
// allows (else cudaErrorInvalidValue, with the counts set).
int hcp_line_index(const char* text, uint64_t n, uint64_t offset, uint64_t* line_start, uint64_t cap, uint64_t* n_newlines,
                   uint64_t* n_lines) {
    char* d_buf = nullptr;
    u64* d_ls = nullptr;
    u64 nl = 0, lines = 0;
    cudaError_t e = cudaSuccess;
    SCU(cudaMalloc(&d_buf, offset + n + 64));
    SCU(cudaMemset(d_buf, '\n', offset + n + 64));
    SCU(cudaMemcpy(d_buf + offset, text, n, cudaMemcpyHostToDevice));
    SCU(hc_line_index(d_buf + offset, n, &d_ls, &nl, &lines, 0));
    *n_newlines = nl;
    *n_lines = lines;
    if (n && nl + 1 > cap) { e = cudaErrorInvalidValue; goto done; }
    if (n) SCU(cudaMemcpy(line_start, d_ls, (nl + 1) * sizeof(u64), cudaMemcpyDeviceToHost));
done:
    cudaFree(d_buf); cudaFree(d_ls);
    return (int)e;
}

}  // extern "C"
