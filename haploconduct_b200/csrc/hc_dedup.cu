// hc_dedup.cu -- duplicate-edge resolution of the graph insert on the device
// (EdgeCalculator::process_overlaps, serial section, src/EdgeCalculator.cpp:429-545); see hc_b200.h.
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_stage.h"

namespace {

typedef unsigned long long u64;

// murmur3 finaliser.  (The slot used to be the LOW bits of key * odd constant, which depend on the low bits of the key only:
// all edges of one vertex fell on one slot and probed the same chain -- 535 ms for 5e6 edges instead of 15.)
__device__ __forceinline__ unsigned long long dd_hash(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

__device__ __forceinline__ u64 dd_key(const hc_dedup_edge& e) {
    const u64 lo = min(e.vertex1, e.vertex2), hi = max(e.vertex1, e.vertex2);
    return (lo << 33) | (hi << 1) | (u64)(e.ori1 == e.ori2);     // checkEdgeWithOri's key, :453-454
}

// true iff edge a (index ia) wins against edge b (index ib): :470-521, full ties go to the later one
__device__ __forceinline__ bool dd_beats(const hc_dedup_edge& a, u64 ia, const hc_dedup_edge& b, u64 ib) {
    if (a.score != b.score) return a.score > b.score;                         // :470
    if (a.overlap_len != b.overlap_len) return a.overlap_len > b.overlap_len;  // :476-481
    if (a.mismatch_rate != b.mismatch_rate) return a.mismatch_rate < b.mismatch_rate;   // :482-487
    if (a.vertex1 != b.vertex1) return a.vertex1 < b.vertex1;                  // :488-493
    if (a.ori1 != b.ori1) return a.ori1 != 0;                                  // :494-499
    if (a.ori2 != b.ori2) return a.ori2 != 0;                                  // :500-505
    if (a.pos1 != b.pos1) return a.pos1 < b.pos1;                              // :506-511
    if (a.pos2 != b.pos2) return a.pos2 < b.pos2;                              // :512-517
    return ia > ib;                                                            // :518-520: replace
}

__device__ __forceinline__ u64 dd_slot(u64* keys, u64 key, u64 mask) {
    u64 h = dd_hash(key) & mask;
    while (true) {
        const u64 prev = atomicCAS(&keys[h], ~0ull, key);
        if (prev == ~0ull || prev == key) return h;
        h = (h + 1) & mask;
    }
}

__global__ void dd_claim(const hc_dedup_edge* e, u64 n, u64* keys, u64* best, u64* first, u64 mask, u64* counts) {
    u64 incl = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const hc_dedup_edge me = e[i];
        if (me.perc == 100) incl++;                                            // :449-451
        const u64 h = dd_slot(keys, dd_key(me), mask);
        atomicMin(&first[h], i);
        u64 cur = best[h];
        while (cur == ~0ull || dd_beats(me, i, e[cur], cur)) {
            const u64 prev = atomicCAS(&best[h], cur, i);
            if (prev == cur) break;
            cur = prev;
        }
    }
    if (incl) atomicAdd(&counts[1], incl);
}

__global__ void dd_resolve(const hc_dedup_edge* e, u64 n, const u64* keys, const u64* best, const u64* first, u64 mask,
                           int ignore_inclusions, uint8_t* winner, uint8_t* inclusions, u64* counts) {
    u64 dups = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const hc_dedup_edge me = e[i];
        const u64 key = dd_key(me);
        u64 h = dd_hash(key) & mask;
        while (keys[h] != key) h = (h + 1) & mask;
        winner[i] = best[h] == i;
        if (first[h] != i) dups++;                                             // found an existing edge: doubles++ (:472,:537)
        else if (ignore_inclusions && inclusions && me.perc == 100 && me.mismatch_rate < 0.000001 && me.mismatch_rate >= 0) {   // :459-468
            if (me.pos3 < 0) { if (me.pos1 == 0) inclusions[me.vertex1] = 1; }
            else inclusions[me.vertex2] = 1;
        }
    }
    if (dups) atomicAdd(&counts[0], dups);
}

}  // namespace

extern "C" int hc_dedup_edges(const hc_dedup_edge* edges, uint64_t n, int ignore_inclusions, uint8_t* winner,
                              uint8_t* inclusions, uint64_t n_vertices, uint64_t counts[2], int device) {
    if ((n && (!edges || !winner)) || !counts) { hc_set_last_error("hc_dedup_edges: NULL argument"); return HC_ERR_ARG; }
    counts[0] = counts[1] = 0;
    if (n == 0) return HC_OK;
    for (u64 i = 0; i < n; i++)
        if (edges[i].vertex1 >= n_vertices || edges[i].vertex2 >= n_vertices || edges[i].vertex1 >= (1u << 31) || edges[i].vertex2 >= (1u << 31)) {
            hc_set_last_error("hc_dedup_edges: vertex out of range");
            return HC_ERR_ARG;
        }
    int rc = HC_OK;
    const char* who = "hc_dedup_edges";
    ScratchBuf<hc_dedup_edge> d_e;
    ScratchBuf<u64> d_keys, d_best, d_first, d_counts;
    ScratchBuf<uint8_t> d_win, d_inc;
    u64 cap = 64;
    const int threads = 256, blocks = grid_for(n, threads);
    while (cap < 2 * n + 2) cap <<= 1;
    HC_CU(cudaSetDevice(device));
    HC_CU(d_e.alloc(n));
    HC_CU(d_keys.alloc(cap)); HC_CU(d_best.alloc(cap)); HC_CU(d_first.alloc(cap));
    HC_CU(d_counts.alloc(2)); HC_CU(d_win.alloc(n));
    HC_CU(cudaMemset(d_keys, 0xff, cap * sizeof(u64))); HC_CU(cudaMemset(d_best, 0xff, cap * sizeof(u64)));
    HC_CU(cudaMemset(d_first, 0xff, cap * sizeof(u64))); HC_CU(cudaMemset(d_counts, 0, 2 * sizeof(u64)));
    if (inclusions && n_vertices) { HC_CU(d_inc.alloc(n_vertices)); HC_CU(cudaMemcpy(d_inc, inclusions, n_vertices, cudaMemcpyHostToDevice)); }
    HC_CU(hc_copy_h2d(d_e, edges, n * sizeof(hc_dedup_edge)));
    dd_claim<<<blocks, threads>>>(d_e, n, d_keys, d_best, d_first, cap - 1, d_counts);
    dd_resolve<<<blocks, threads>>>(d_e, n, d_keys, d_best, d_first, cap - 1, ignore_inclusions, d_win, d_inc, d_counts);
    HC_CU(cudaGetLastError());
    HC_CU(hc_copy_d2h(winner, d_win, n));
    HC_CU(cudaMemcpy(counts, d_counts, 2 * sizeof(u64), cudaMemcpyDeviceToHost));
    if (d_inc) HC_CU(cudaMemcpy(inclusions, d_inc, n_vertices, cudaMemcpyDeviceToHost));
done:
    return rc;
}
