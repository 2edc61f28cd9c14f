// hc_radix.cuh -- stable LSD radix sort of (128-bit key, uint32 value) pairs, 8-bit digits.  Per digit position: a count
// of every tile's digits (digit-major matrix), an exclusive scan of that matrix with hc_scan (the start of every
// (digit, tile) range), and a scatter that ranks each element among the equal digits of its tile in index order (warp
// match + per-warp counts), which keeps the sort stable.  Digit positions that every key shares are skipped: one
// reduction of the keys' AND and OR tells which they are (a position is shared iff AND and OR agree on its 8 bits).
#ifndef HC_RADIX_CUH_
#define HC_RADIX_CUH_
#include <cstdint>
#include <cuda_runtime.h>
#include "hc_scan.cuh"
#include "hc_stage.h"

namespace hc_radix {
namespace {     // internal linkage: the header may be included by several translation units

typedef unsigned long long u64;
constexpr int THREADS = 256;                   // = number of digit values: thread d owns digit d in the per-tile tables
constexpr int WARPS = THREADS / 32;
constexpr int ITEMS = 8;
constexpr int TILE = THREADS * ITEMS;

// digit p (0..15) of a key: x holds the low 64 bits, y the high 64 bits
__device__ __forceinline__ uint32_t digit_of(const ulonglong2& k, int p) {
    return (uint32_t)(((p < 8 ? k.x : k.y) >> (8 * (p & 7))) & 0xffu);
}

__global__ void __launch_bounds__(THREADS) and_or(const ulonglong2* __restrict__ keys, u64 n, u64* __restrict__ acc /* and.x, and.y, or.x, or.y */) {
    u64 ax = ~0ull, ay = ~0ull, ox = 0, oy = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const ulonglong2 k = keys[i];
        ax &= k.x; ay &= k.y; ox |= k.x; oy |= k.y;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        ax &= __shfl_xor_sync(0xffffffffu, ax, d); ay &= __shfl_xor_sync(0xffffffffu, ay, d);
        ox |= __shfl_xor_sync(0xffffffffu, ox, d); oy |= __shfl_xor_sync(0xffffffffu, oy, d);
    }
    if ((threadIdx.x & 31) == 0) { atomicAnd(&acc[0], ax); atomicAnd(&acc[1], ay); atomicOr(&acc[2], ox); atomicOr(&acc[3], oy); }
}

__global__ void __launch_bounds__(THREADS) tile_counts(const ulonglong2* __restrict__ keys, u64 n, int p, uint32_t nb, uint32_t* __restrict__ counts) {
    __shared__ uint32_t h[THREADS];
    h[threadIdx.x] = 0;
    __syncthreads();
    const u64 t0 = (u64)blockIdx.x * TILE;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
        const u64 i = t0 + (u64)j * THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[digit_of(keys[i], p)], 1u);
    }
    __syncthreads();
    counts[(u64)threadIdx.x * nb + blockIdx.x] = h[threadIdx.x];
}

// Element i of the tile goes to start[digit][tile] + (elements of the tile before i with the same digit).  Segment j of the
// tile (one element per thread) is ranked after segments < j, warp w after warps < w, lane l after lanes < l: index order.
__global__ void __launch_bounds__(THREADS) tile_scatter(const ulonglong2* __restrict__ kin, const uint32_t* __restrict__ vin, u64 n, int p,
                                                        uint32_t nb, const u64* __restrict__ start, ulonglong2* __restrict__ kout,
                                                        uint32_t* __restrict__ vout) {
    __shared__ uint32_t wcnt[WARPS][THREADS];
    __shared__ u64 base[THREADS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    base[threadIdx.x] = start[(u64)threadIdx.x * nb + blockIdx.x];
    const u64 t0 = (u64)blockIdx.x * TILE;
    for (int j = 0; j < ITEMS; j++) {
        const u64 i = t0 + (u64)j * THREADS + threadIdx.x;
        const bool valid = i < n;
        ulonglong2 k = make_ulonglong2(0, 0);
        uint32_t v = 0, d = THREADS;                       // THREADS: no digit (past the end)
        if (valid) { k = kin[i]; v = vin[i]; d = digit_of(k, p); }
#pragma unroll
        for (int w = 0; w < WARPS; w++) wcnt[w][threadIdx.x] = 0;
        __syncthreads();
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t rank = __popc(peers & lt);
        if (valid && rank == 0) wcnt[warp][d] = __popc(peers);
        __syncthreads();
        uint32_t seg = 0;                                  // thread = digit: exclusive prefix over the warps
#pragma unroll
        for (int w = 0; w < WARPS; w++) { const uint32_t c = wcnt[w][threadIdx.x]; wcnt[w][threadIdx.x] = seg; seg += c; }
        __syncthreads();
        if (valid) {
            const u64 pos = base[d] + wcnt[warp][d] + rank;
            kout[pos] = k;
            vout[pos] = v;
        }
        __syncthreads();
        base[threadIdx.x] += seg;
    }
}

// Sorts n pairs by key, stably.  The result is in (*kres, *vres): (keys, vals) or (ktmp, vtmp), each holding n entries.
// Enqueued on the legacy default stream; synchronises once (to read which digit positions vary).
inline cudaError_t sort_pairs(ulonglong2* keys, uint32_t* vals, ulonglong2* ktmp, uint32_t* vtmp, u64 n,
                              ulonglong2** kres, uint32_t** vres) {
    *kres = keys; *vres = vals;
    if (n == 0) return cudaSuccess;
    const uint32_t nb = (uint32_t)((n + TILE - 1) / TILE);
    const u64 cells = (u64)THREADS * nb;
    u64 *d_acc = nullptr, *d_start = nullptr, *d_total = nullptr, *d_bsum = nullptr;
    uint32_t* d_counts = nullptr;
    u64 acc[4] = {~0ull, ~0ull, 0, 0};
    cudaError_t e;
    ulonglong2 *ki = keys, *ko = ktmp;
    uint32_t *vi = vals, *vo = vtmp;
    if ((e = hc_scratch_alloc((void**)&d_acc, sizeof(acc))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_counts, cells * sizeof(uint32_t))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_start, cells * sizeof(u64))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_total, sizeof(u64))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(cells) * sizeof(u64))) != cudaSuccess) goto done;
    if ((e = cudaMemcpyAsync(d_acc, acc, sizeof(acc), cudaMemcpyHostToDevice)) != cudaSuccess) goto done;
    and_or<<<(unsigned)(nb < 148 * 8 ? nb : 148 * 8), THREADS>>>(keys, n, d_acc);
    if ((e = cudaMemcpy(acc, d_acc, sizeof(acc), cudaMemcpyDeviceToHost)) != cudaSuccess) goto done;
    for (int p = 0; p < 16; p++) {
        const u64 diff = p < 8 ? acc[0] ^ acc[2] : acc[1] ^ acc[3];
        if (((diff >> (8 * (p & 7))) & 0xffu) == 0) continue;       // every key has the same digit here
        tile_counts<<<nb, THREADS>>>(ki, n, p, nb, d_counts);
        hc_scan::exclusive_u32(d_counts, cells, d_start, d_total, d_bsum, 0);
        tile_scatter<<<nb, THREADS>>>(ki, vi, n, p, nb, d_start, ko, vo);
        ulonglong2* tk = ki; ki = ko; ko = tk;
        uint32_t* tv = vi; vi = vo; vo = tv;
        if ((e = cudaGetLastError()) != cudaSuccess) goto done;
    }
    *kres = ki; *vres = vi;
done:
    hc_scratch_free(d_acc); hc_scratch_free(d_counts); hc_scratch_free(d_start); hc_scratch_free(d_total); hc_scratch_free(d_bsum);
    return e;
}

}  // namespace
}  // namespace hc_radix
#endif
