// hc_fno.cu -- FindNextOverlaps on the device: SRBuilder::findNextOverlaps (FNO1), src/FindNextOverlaps.cpp:890-958
// (updateOverlap :25-327, findCliqueIndex :331-347, computeOverlapData :351-565) and SRBuilder::findNextOverlaps3,
// src/FindNextOverlaps3.cpp:20-406.
//
// The reference walks the edge stream sequentially; for every edge (u, v) it tries every pair (new read of u) x (new read
// of v) and keeps, per unordered pair of new reads, the FIRST attempt in processing order -- whether or not that attempt
// then succeeds (:84-97 precede :115-118).  Here every attempt gets its sequence number from an exclusive scan of the
// per-edge attempt counts, the holder of the smallest sequence number per pair is found with atomicMin in a hash table,
// and only those holders are evaluated: the same winners without the sequential walk.
//
// Round-2 layout (the first version spent its time in random DRAM gathers: ~1 KB of traffic per attempt, 30 ms of kernels
// for 2.6e7 attempts):
//   * what a thread needs of a vertex (list range, visited / label / paired flags, id and lengths of the unmerged read) is
//     packed into ONE 32-byte record per vertex, what it needs of a list entry (super-read id and lengths, the two clique
//     indices of findCliqueIndex already resolved) into one 32-byte record per entry -- one sector per lookup instead of
//     five resp. three, and both tables stay in L2 (32 + 51 MB for 1e6 vertices);
//   * pair keys are written once, in attempt order (8 bytes each); the first-found-wins table is then filled PARTITION BY
//     PARTITION (key hash -> partition), each partition's table small enough (<= 32 MB) to live in L2 while the keys stream
//     past it with evict-first loads: atomics hit L2 instead of a 1 GB table in DRAM.  Pass p claims partition p and, in the
//     same sweep, reads the winners of partition p-1 out of the other table;
//   * results are staged as 24-byte records (ids < 2^32, positions / lengths < 2^24, flags in bytes) and an order-preserving
//     compaction writes either those (hc_fno1_small / hc_fno3_small) or the 48-byte hc_fno_overlap; inputs whose values do not
//     fit 24 bytes take a 48-byte staging path.
// All integer / float32 arithmetic, bit-identical to the reference (perc uses IEEE float division, max, multiplication and
// floor, :375,:429,:487,:549).
#include <cstdio>
#include <cstdlib>
#include <time.h>
#include <cstring>
#include <string>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_fno_text.h"
#include "hc_ingest.h"
#include "hc_scan.cuh"
#include "hc_stage.h"

namespace {

typedef unsigned long long u64;

// one 32-byte sector per vertex
struct __align__(16) VDesc {
    uint32_t off, cnt;       // range of the vertex' list entries (EDesc); cnt is the reference's nodes_to_SR[v].size()
    u64 id;                  // new id of the unmerged read (meaningful when !visited)
    uint32_t len1, len2;     // lengths of the original read
    uint32_t flags;          // bit 0 visited, bit 1 label, bit 2 paired
    uint32_t pad;
};
#define VD_VISITED 1u
#define VD_LABEL 2u
#define VD_PAIRED 4u

// one 32-byte sector per (vertex, super-read) list entry
struct __align__(16) EDesc {
    uint32_t id, len1, len2; // the super-read (ids of new reads are below 2^32, checked by the host part)
    int32_t il;              // findCliqueIndex :331-347: index1 - startpos1
    int32_t ir;              //                           index2 - startpos2 if the super-read or the vertex is paired, else il
    uint32_t pad[3];
};

// staged result, 24 bytes: == hc_fno_overlap_small (include/hc_b200.h)
struct Rec24 { uint32_t id1, id2, p1, p2, l1, l2; };

struct DevIn {
    const VDesc* vd;
    const EDesc* en;
    uint32_t resolve_orientations, no_inclusions;
};

__device__ __forceinline__ int perc_of(int t, int la, int lb) {
    const float a = __fdiv_rn((float)t, (float)la), b = __fdiv_rn((float)t, (float)lb);
    return (int)floorf(__fmul_rn(fmaxf(a, b), 100.0f));
}

struct Derived {
    int pos1, pos2, perc, ol1, ol2;
    char ord1, ord2, t1, t2;
};

// src/FindNextOverlaps.cpp:351-565
__device__ bool compute_overlap_data(const hc_fno_read& r1, const hc_fno_read& r2, int idx1l, int idx1r, int idx2l, int idx2r,
                                     const hc_fno_edge& e, Derived& d) {
    const int pos1 = e.pos1, pos2 = e.pos2;
    const bool p1 = r1.len2 > 0, p2 = r2.len2 > 0;
    const int l11 = (int)r1.len1, l12 = (int)r1.len2, l21 = (int)r2.len1, l22 = (int)r2.len2;
    d.pos2 = 0;
    d.pos1 = (pos1 + idx1l) - idx2l;
    if (!p1 && !p2) {                                              // S-S :357-385
        d.t1 = 's'; d.t2 = 's';
        int len;
        if (d.pos1 < 0) { d.ord1 = '2'; d.pos1 = -d.pos1; len = l21; }
        else { d.ord1 = '1'; len = l11; }
        d.ol1 = min(min(len - d.pos1, l11), l21);
        d.ol2 = 0;
        d.perc = perc_of(d.ol1, l11, l21);
        d.ord2 = '-';
        return d.pos1 < len;
    }
    if (p1 && !p2) {                                               // P-S :387-443
        d.t1 = 'p'; d.t2 = 's';
        if (d.pos1 < 0) {
            d.ord1 = '2'; d.pos1 = -d.pos1;
            if (d.pos1 >= l21) return false;
            d.ol1 = l11;
        } else {
            d.ord1 = '1';
            if (d.pos1 >= l11) return false;
            d.ol1 = l11 - d.pos1;
        }
        d.pos2 = e.ord == '1' ? idx2r - (idx1r + pos2) : (pos2 + idx2r) - idx1r;
        if (d.pos2 >= l21 || d.pos2 < 0) return false;
        d.ord2 = '-';
        d.ol2 = min(l21 - d.pos2, l12);
        d.perc = min(perc_of(d.ol1 + d.ol2, l11 + l12, l21), 100);
        return true;
    }
    if (!p1 && p2) {                                               // S-P :445-489
        d.t1 = 's'; d.t2 = 'p';
        if (d.pos1 < 0) {
            d.ord1 = '2'; d.pos1 = -d.pos1;
            if (d.pos1 >= l21) return false;
            d.ol1 = l21 - d.pos1;
        } else {
            d.ord1 = '1';
            if (d.pos1 >= l11) return false;
            d.ol1 = l21;
        }
        d.pos2 = e.ord == '2' ? idx1r - (pos2 + idx2r) : idx1r + pos2 - idx2r;
        if (d.pos2 >= l11 || d.pos2 < 0) return false;
        d.ord2 = '-';
        d.ol2 = min(l11 - d.pos2, l22);
        d.perc = min(perc_of(d.ol1 + d.ol2, l11, l21 + l22), 100);
        return true;
    }
    d.t1 = 'p'; d.t2 = 'p';                                        // P-P :491-551
    if (d.pos1 < 0) {
        d.ord1 = '2'; d.pos1 = -d.pos1;
        if (d.pos1 >= l21) return false;
        d.ol1 = min(l11, l21 - d.pos1);
    } else {
        d.ord1 = '1';
        if (d.pos1 >= l11) return false;
        d.ol1 = min(l11 - d.pos1, l21);
    }
    d.pos2 = e.ord == '1' ? (pos2 + idx1r) - idx2r : idx1r - (pos2 + idx2r);
    if (d.pos2 < 0) {
        d.ord2 = d.ord1 == '1' ? '2' : '1';
        d.pos2 = -d.pos2;
        if (d.pos2 >= l22) return false;
        d.ol2 = min(l12, l22 - d.pos2);
    } else {
        d.ord2 = d.ord1 == '1' ? '1' : '2';
        if (d.pos2 >= l12) return false;
        d.ol2 = min(l12 - d.pos2, l22);
    }
    d.perc = min(perc_of(d.ol1 + d.ol2, l11 + l12, l21 + l22), 100);
    return true;
}


// ---- first found wins: per pair key the smallest sequence number -----------------------------------------------------
struct __align__(16) Cell { u64 key, min; };      // empty: key == ~0, min == ~0

__device__ __forceinline__ u64 mix64(u64 k) {     // murmur3 finaliser: partitions and slots must not follow the structure of the ids
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}
__device__ __forceinline__ uint32_t key_part(u64 h, uint32_t P) { return (uint32_t)(((h >> 32) * (u64)P) >> 32); }
__device__ __forceinline__ uint32_t key_slot(u64 h, uint32_t mask) { return (uint32_t)h & mask; }
__device__ __forceinline__ u64 pair_key(u64 id1, u64 id2) { return (min(id1, id2) << 32) | max(id1, id2); }

// keys per partition (sizes the tables: a partition must never fill its table)
__global__ void ffw_histogram(const u64* __restrict__ keys, u64 n, uint32_t P, unsigned long long* __restrict__ hist) {
    extern __shared__ uint32_t sh[];
    for (uint32_t k = threadIdx.x; k < P; k += blockDim.x) sh[k] = 0;
    __syncthreads();
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        const u64 key = __ldcs(keys + t);
        if (key != ~0ull) atomicAdd(&sh[key_part(mix64(key), P)], 1u);
    }
    __syncthreads();
    for (uint32_t k = threadIdx.x; k < P; k += blockDim.x) if (sh[k]) atomicAdd(&hist[k], (unsigned long long)sh[k]);
}

// Multisplit: the keyed attempts of partition k go to [start_k, start_k + hist_k) of pkey / pseq (cursor[k] starts at start_k).
// A block counts its tile per partition in shared memory, reserves one range per partition with a single atomicAdd and
// places its elements there; the order inside a partition is arbitrary (only the minimum of the sequence numbers matters).
#define FFW_SPLIT_ITEMS 8
__global__ void __launch_bounds__(256) ffw_split(const u64* __restrict__ keys, u64 n, uint32_t P, unsigned long long* __restrict__ cursor,
                                                 u64* __restrict__ pkey, u64* __restrict__ pseq) {
    extern __shared__ unsigned long long shb[];                 // [P] reserved base, then [P] uint32 counts
    uint32_t* cnt = reinterpret_cast<uint32_t*>(shb + P);
    const u64 tile = (u64)blockDim.x * FFW_SPLIT_ITEMS;
    for (u64 base = (u64)blockIdx.x * tile; base < n; base += (u64)gridDim.x * tile) {
        for (uint32_t k = threadIdx.x; k < P; k += blockDim.x) cnt[k] = 0;
        __syncthreads();
        u64 key[FFW_SPLIT_ITEMS];
        uint32_t part[FFW_SPLIT_ITEMS], rank[FFW_SPLIT_ITEMS];
#pragma unroll
        for (int j = 0; j < FFW_SPLIT_ITEMS; j++) {
            const u64 t = base + (u64)j * blockDim.x + threadIdx.x;
            key[j] = t < n ? __ldcs(keys + t) : ~0ull;
        }
#pragma unroll
        for (int j = 0; j < FFW_SPLIT_ITEMS; j++) {
            part[j] = 0xffffffffu;
            if (key[j] != ~0ull) {
                part[j] = key_part(mix64(key[j]), P);
                rank[j] = atomicAdd(&cnt[part[j]], 1u);
            }
        }
        __syncthreads();
        for (uint32_t k = threadIdx.x; k < P; k += blockDim.x) if (cnt[k]) shb[k] = atomicAdd(&cursor[k], (unsigned long long)cnt[k]);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < FFW_SPLIT_ITEMS; j++) {
            if (part[j] != 0xffffffffu) {
                const u64 pos = shb[part[j]] + rank[j];
                pkey[pos] = key[j];
                pseq[pos] = base + (u64)j * blockDim.x + threadIdx.x;
            }
        }
        __syncthreads();
    }
}

// every attempt of one partition claims its pair: smallest sequence number per key
__global__ void ffw_claim(const u64* __restrict__ pkey, const u64* __restrict__ pseq, u64 n, Cell* __restrict__ tab, uint32_t mask) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        const u64 key = __ldcs(pkey + t);
        uint32_t s = key_slot(mix64(key), mask);
        while (true) {
            const u64 prev = atomicCAS(&tab[s].key, ~0ull, key);
            if (prev == ~0ull || prev == key) break;
            s = (s + 1) & mask;
        }
        atomicMin(&tab[s].min, __ldcs(pseq + t));
    }
}

// win[seq] = 1 for the holders of the minimum
__global__ void ffw_check(const u64* __restrict__ pkey, const u64* __restrict__ pseq, u64 n, const Cell* __restrict__ tab, uint32_t mask,
                          uint8_t* __restrict__ win) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        const u64 key = __ldcs(pkey + t), seq = __ldcs(pseq + t);
        uint32_t s = key_slot(mix64(key), mask);
        while (tab[s].key != key) s = (s + 1) & mask;
        if (tab[s].min == seq) win[seq] = 1;
    }
}

// win[t] = 1 for the attempts that hold the smallest sequence number of their key (win must be zero on entry)
cudaError_t ffw_winners(const u64* d_keys, u64 n, uint8_t* d_win) {
    cudaError_t e = cudaSuccess;
    const char* env = getenv("HC_FNO_PART");                 // keys per partition (tests: small values exercise many partitions)
    const u64 per = env && atoll(env) > 0 ? (u64)atoll(env) : 900000ull;
    u64 P = (n + per - 1) / per;
    if (P < 1) P = 1;
    if (P > 2048) P = 2048;                                    // beyond 1.8e9 attempts the tables simply grow
    const int threads = 256, blocks = 148 * 8;
    unsigned long long *h_hist = (unsigned long long*)malloc(2 * P * sizeof(unsigned long long)), *d_hist = nullptr, *d_cursor = nullptr;
    u64 *d_pkey = nullptr, *d_pseq = nullptr, mx = 0, total = 0, slots = 1024;
    Cell* d_tab = nullptr;
    uint32_t mask;
    if (!h_hist) return cudaErrorMemoryAllocation;
    unsigned long long* h_start = h_hist + P;
    if ((e = hc_scratch_alloc((void**)&d_hist, P * sizeof(unsigned long long))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_cursor, P * sizeof(unsigned long long))) != cudaSuccess) goto done;
    if ((e = cudaMemsetAsync(d_hist, 0, P * sizeof(unsigned long long))) != cudaSuccess) goto done;
    ffw_histogram<<<blocks, threads, P * sizeof(uint32_t)>>>(d_keys, n, (uint32_t)P, d_hist);
    if ((e = cudaMemcpy(h_hist, d_hist, P * sizeof(unsigned long long), cudaMemcpyDeviceToHost)) != cudaSuccess) goto done;
    for (u64 k = 0; k < P; k++) { h_start[k] = total; total += h_hist[k]; mx = h_hist[k] > mx ? h_hist[k] : mx; }
    if (total == 0) goto done;                                 // no keyed attempt at all
    while (slots < 2 * mx + 2) slots <<= 1;                    // load <= 0.5: a partition can never fill its table
    mask = (uint32_t)(slots - 1);
    if ((e = hc_scratch_alloc((void**)&d_pkey, total * sizeof(u64))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_pseq, total * sizeof(u64))) != cudaSuccess) goto done;
    if ((e = hc_scratch_alloc((void**)&d_tab, slots * sizeof(Cell))) != cudaSuccess) goto done;
    if ((e = cudaMemcpyAsync(d_cursor, h_start, P * sizeof(unsigned long long), cudaMemcpyHostToDevice)) != cudaSuccess) goto done;
    ffw_split<<<blocks, threads, P * (sizeof(unsigned long long) + sizeof(uint32_t))>>>(d_keys, n, (uint32_t)P, d_cursor, d_pkey, d_pseq);
    for (u64 p = 0; p < P; p++) {
        const u64 c = h_hist[p];
        if (c == 0) continue;
        const int pb = (int)((c + threads - 1) / threads < (u64)(148 * 16) ? (c + threads - 1) / threads : 148 * 16);
        if ((e = cudaMemsetAsync(d_tab, 0xff, slots * sizeof(Cell))) != cudaSuccess) goto done;
        ffw_claim<<<pb, threads>>>(d_pkey + h_start[p], d_pseq + h_start[p], c, d_tab, mask);
        ffw_check<<<pb, threads>>>(d_pkey + h_start[p], d_pseq + h_start[p], c, d_tab, mask, d_win);
    }
    e = cudaGetLastError();
done:
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);        // h_start / h_hist are read by the copies above
    free(h_hist);
    hc_scratch_free(d_hist); hc_scratch_free(d_cursor); hc_scratch_free(d_pkey); hc_scratch_free(d_pseq); hc_scratch_free(d_tab);
    return e;
}

// ---- staged records ----------------------------------------------------------------------------------------------------
// flags byte of l1: bits 0-1 ord (0 '-', 1 '1', 2 '2'), bit 2 ori1 == '+', bit 3 ori2 == '+', bit 4 type1 == 'p', bit 5 type2 == 'p'
__device__ __forceinline__ bool pack24(const hc_fno_overlap& o, Rec24& r) {
    const uint32_t big = ((uint32_t)o.pos1 | (uint32_t)o.pos2 | (uint32_t)o.len1 | (uint32_t)o.len2) >> 24;
    const uint32_t bigp = ((uint32_t)o.perc | (uint32_t)o.perc2) >> 8;
    if (big | bigp | (uint32_t)(o.id1 >> 32) | (uint32_t)(o.id2 >> 32)) return false;
    if (o.ord != '1' && o.ord != '2' && o.ord != '-') return false;
    const uint32_t fl = (o.ord == '1' ? 1u : (o.ord == '2' ? 2u : 0u)) | (o.ori1 == '+' ? 4u : 0u) | (o.ori2 == '+' ? 8u : 0u) |
                        (o.type1 == 'p' ? 16u : 0u) | (o.type2 == 'p' ? 32u : 0u);
    r.id1 = (uint32_t)o.id1; r.id2 = (uint32_t)o.id2;
    r.p1 = (uint32_t)o.pos1 | ((uint32_t)o.perc << 24);
    r.p2 = (uint32_t)o.pos2 | ((uint32_t)o.perc2 << 24);
    r.l1 = (uint32_t)o.len1 | (fl << 24);
    r.l2 = (uint32_t)o.len2;
    return true;
}

__device__ __forceinline__ hc_fno_overlap unpack24(const Rec24& r) {
    hc_fno_overlap o;
    memset(&o, 0, sizeof(o));
    const uint32_t fl = r.l1 >> 24;
    o.id1 = r.id1; o.id2 = r.id2;
    o.pos1 = (int32_t)(r.p1 & 0xffffffu); o.perc = (int32_t)(r.p1 >> 24);
    o.pos2 = (int32_t)(r.p2 & 0xffffffu); o.perc2 = (int32_t)(r.p2 >> 24);
    o.len1 = (int32_t)(r.l1 & 0xffffffu); o.len2 = (int32_t)(r.l2 & 0xffffffu);
    o.ord = (fl & 3u) == 1u ? '1' : ((fl & 3u) == 2u ? '2' : '-');
    o.ori1 = (fl & 4u) ? '+' : '-'; o.ori2 = (fl & 8u) ? '+' : '-';
    o.type1 = (fl & 16u) ? 'p' : 's'; o.type2 = (fl & 32u) ? 'p' : 's';
    return o;
}

// SMALL staging: rec is Rec24[attempts]; a value that does not fit raises *overflow (the host then repeats with 48-byte staging)
template <bool SMALL>
__device__ __forceinline__ void stage(void* rec, u64 seq, const hc_fno_overlap& o, uint32_t* overflow) {
    if (SMALL) {
        Rec24 r;
        if (pack24(o, r)) static_cast<Rec24*>(rec)[seq] = r;
        else *overflow = 1u;
    } else {
        static_cast<hc_fno_overlap*>(rec)[seq] = o;
    }
}

// records of the successful attempts, attempt order -> output order (ranks from the scan of the flags)
template <bool SMALL_IN, bool SMALL_OUT>
__global__ void fno_compact(const uint32_t* __restrict__ flags, const u64* __restrict__ outpos, const void* __restrict__ rec,
                            u64 attempts, void* __restrict__ out, u64 out_cap) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < attempts; t += (u64)gridDim.x * blockDim.x) {
        if (!flags[t]) continue;
        const u64 p = outpos[t];
        if (p >= out_cap) continue;
        if (SMALL_IN && SMALL_OUT) static_cast<Rec24*>(out)[p] = static_cast<const Rec24*>(rec)[t];
        else if (SMALL_IN) static_cast<hc_fno_overlap*>(out)[p] = unpack24(static_cast<const Rec24*>(rec)[t]);
        else static_cast<hc_fno_overlap*>(out)[p] = static_cast<const hc_fno_overlap*>(rec)[t];
    }
}

// ---- FNO1 ----------------------------------------------------------------------------------------------------------------
__global__ void fno_prep_vertices(u64 V, const uint8_t* __restrict__ visited, const uint8_t* __restrict__ label,
                                  const hc_fno_read* __restrict__ vr, const u64* __restrict__ sr_off, VDesc* __restrict__ vd) {
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (u64)gridDim.x * blockDim.x) {
        const hc_fno_read r = vr[v];
        VDesc d;
        d.off = (uint32_t)sr_off[v];
        d.cnt = (uint32_t)(sr_off[v + 1] - sr_off[v]);
        d.id = r.id; d.len1 = r.len1; d.len2 = r.len2;
        d.flags = (visited[v] ? VD_VISITED : 0u) | (label[v] ? VD_LABEL : 0u) | (r.len2 > 0 ? VD_PAIRED : 0u);
        d.pad = 0;
        vd[v] = d;
    }
}

__global__ void fno_prep_entries(u64 V, const hc_fno_read* __restrict__ vr, const u64* __restrict__ sr_off,
                                 const uint32_t* __restrict__ sr_idx, const hc_fno_subread* __restrict__ sr_sub,
                                 const hc_fno_read* __restrict__ superread, EDesc* __restrict__ en) {
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (u64)gridDim.x * blockDim.x) {
        const bool pv = vr[v].len2 > 0;
        for (u64 a = sr_off[v]; a < sr_off[v + 1]; a++) {
            const hc_fno_read s = superread[sr_idx[a]];
            const hc_fno_subread sub = sr_sub[a];
            EDesc d;
            d.id = (uint32_t)s.id; d.len1 = s.len1; d.len2 = s.len2;
            d.il = sub.index1 - sub.startpos1;
            d.ir = (s.len2 > 0 || pv) ? sub.index2 - sub.startpos2 : d.il;
            d.pad[0] = d.pad[1] = d.pad[2] = 0;
            en[a] = d;
        }
    }
}

__device__ __forceinline__ VDesc load_vd(const VDesc* p) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    VDesc d;
    d.off = a.x; d.cnt = a.y; d.id = ((u64)a.w << 32) | a.z; d.len1 = b.x; d.len2 = b.y; d.flags = b.z; d.pad = 0;
    return d;
}

// what an attempt uses of one side: the super-read of a list entry, or the unmerged read itself
struct Side { u64 id; uint32_t len1, len2; int32_t il, ir; };
__device__ __forceinline__ Side side_of_entry(const EDesc* p) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
    Side s;
    s.id = a.x; s.len1 = a.y; s.len2 = a.z; s.il = (int32_t)a.w; s.ir = __ldg(&p->ir);
    return s;
}
__device__ __forceinline__ Side side_of_vertex(const VDesc& d) {
    Side s;
    s.id = d.id; s.len1 = d.len1; s.len2 = d.len2; s.il = 0; s.ir = 0;
    return s;
}

__global__ void fno_count(DevIn D, const hc_fno_edge* __restrict__ edges, u64 n, uint32_t* __restrict__ cnt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const uint2 uv = __ldg(reinterpret_cast<const uint2*>(edges + i));
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(D.vd + uv.x));          // off, cnt
        const uint2 b = __ldg(reinterpret_cast<const uint2*>(D.vd + uv.y));
        const uint32_t fa = __ldg(&D.vd[uv.x].flags), fb = __ldg(&D.vd[uv.y].flags);
        cnt[i] = ((fa & VD_VISITED) ? a.y : 1u) * ((fb & VD_VISITED) ? b.y : 1u);
    }
}

// pair keys in attempt order; ~0 for attempts without first-found bookkeeping (plain copies :46-72, id1 == id2 :241-243)
__global__ void fno_keys(DevIn D, const hc_fno_edge* __restrict__ edges, u64 n, const u64* __restrict__ off, u64* __restrict__ keys) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const uint2 uv = __ldg(reinterpret_cast<const uint2*>(edges + i));
        const VDesc du = load_vd(D.vd + uv.x), dv = load_vd(D.vd + uv.y);
        const bool vu = du.flags & VD_VISITED, vv = dv.flags & VD_VISITED;
        u64 seq = off[i];
        if (!vu && !vv) { keys[seq] = ~0ull; continue; }
        const uint32_t na = vu ? du.cnt : 1u, nb = vv ? dv.cnt : 1u;
        for (uint32_t a = 0; a < na; a++) {
            const u64 id1 = vu ? (u64)__ldg(&D.en[du.off + a].id) : du.id;
            for (uint32_t b = 0; b < nb; b++, seq++) {
                const u64 id2 = vv ? (u64)__ldg(&D.en[dv.off + b].id) : dv.id;
                keys[seq] = id1 == id2 ? ~0ull : pair_key(id1, id2);
            }
        }
    }
}

// flags[seq] = "attempt seq yields an overlap" and, when it does, its record at rec[seq] (attempt order); fno_compact then
// moves the records to their ranks.
template <bool SMALL>
__global__ void fno_resolve(DevIn D, const hc_fno_edge* __restrict__ edges, u64 n, const u64* __restrict__ off,
                            const uint8_t* __restrict__ win, uint32_t* __restrict__ flags, void* __restrict__ rec, uint32_t* overflow) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const uint4 e0 = __ldg(reinterpret_cast<const uint4*>(edges + i)), e1 = __ldg(reinterpret_cast<const uint4*>(edges + i) + 1);
        hc_fno_edge e;
        e.u = e0.x; e.v = e0.y; e.pos1 = (int32_t)e0.z; e.pos2 = (int32_t)e0.w; e.perc = (int32_t)e1.x; e.len1 = (int32_t)e1.y;
        e.len2 = (int32_t)e1.z; e.ord = e1.w & 0xffu; e.ori1 = (e1.w >> 8) & 0xffu; e.ori2 = (e1.w >> 16) & 0xffu; e.nonedge = e1.w >> 24;
        const VDesc du = load_vd(D.vd + e.u), dv = load_vd(D.vd + e.v);
        const bool vu = du.flags & VD_VISITED, vv = dv.flags & VD_VISITED;
        char ori1 = '+', ori2 = '+';
        if (D.resolve_orientations && e.nonedge) {                  // :34-37
            ori1 = (e.ori1 == ((du.flags & VD_LABEL) ? 1u : 0u)) ? '+' : '-';
            ori2 = (e.ori2 == ((dv.flags & VD_LABEL) ? 1u : 0u)) ? '+' : '-';
        }
        u64 seq = off[i];
        if (!vu && !vv) {                                           // :46-72
            const bool ok = !(D.no_inclusions && e.perc == 100);
            flags[seq] = ok;
            if (ok) {
                hc_fno_overlap o;
                memset(&o, 0, sizeof(o));
                o.id1 = du.id; o.id2 = dv.id; o.pos1 = e.pos1; o.pos2 = e.pos2; o.ord = e.ord; o.ori1 = ori1; o.ori2 = ori2;
                o.perc = e.perc; o.len1 = e.len1; o.len2 = e.len2;
                o.type1 = (du.flags & VD_PAIRED) ? 'p' : 's'; o.type2 = (dv.flags & VD_PAIRED) ? 'p' : 's';
                stage<SMALL>(rec, seq, o, overflow);
            }
            continue;
        }
        const uint32_t na = vu ? du.cnt : 1u, nb = vv ? dv.cnt : 1u;
        for (uint32_t a = 0; a < na; a++) {
            for (uint32_t b = 0; b < nb; b++, seq++) {
                bool ok = win[seq] != 0;                            // first found wins, even if it fails below; id1 == id2 never wins
                if (ok) {
                    const Side s1 = vu ? side_of_entry(D.en + du.off + a) : side_of_vertex(du);
                    const Side s2 = vv ? side_of_entry(D.en + dv.off + b) : side_of_vertex(dv);
                    hc_fno_read r1, r2;
                    r1.id = s1.id; r1.len1 = s1.len1; r1.len2 = s1.len2;
                    r2.id = s2.id; r2.len1 = s2.len1; r2.len2 = s2.len2;
                    Derived d;
                    ok = compute_overlap_data(r1, r2, s1.il, s1.ir, s2.il, s2.ir, e, d);
                    if (ok && D.no_inclusions && d.perc == 100) ok = false;
                    if (ok) {
                        hc_fno_overlap o;
                        memset(&o, 0, sizeof(o));
                        if (d.ord1 == '1') { o.id1 = s1.id; o.id2 = s2.id; o.type1 = d.t1; o.type2 = d.t2; }
                        else { o.id1 = s2.id; o.id2 = s1.id; o.type1 = d.t2; o.type2 = d.t1; }
                        o.pos1 = d.pos1; o.pos2 = d.pos2; o.ord = d.ord2; o.ori1 = ori1; o.ori2 = ori2;
                        o.perc = d.perc; o.len1 = d.ol1; o.len2 = d.ol2;
                        stage<SMALL>(rec, seq, o, overflow);
                    }
                }
                flags[seq] = ok;
            }
        }
    }
}

// ---- FindNextOverlaps3 (src/FindNextOverlaps3.cpp:90-406) ------------------------------------------------
__device__ __forceinline__ int perc_one(int l, int a) { return (int)floorf(__fmul_rn(__fdiv_rn((float)l, (float)a), 100.0f)); }

// deduceOverlap :176-406; false = "this overlap will be ignored"
__device__ bool deduce_overlap(const hc_fno_read& A, const hc_fno_read& B, const hc_fno3_pos& pa, const hc_fno3_pos& pb,
                               hc_fno_overlap& o) {
    const bool pA = A.len2 > 0, pB = B.len2 > 0;
    memset(&o, 0, sizeof(o));
    o.ori1 = '+'; o.ori2 = '+'; o.ord = '-';
    const int i1l = pa.index1, i1r = pa.index2, i2l = pb.index1, i2r = pb.index2;
    const bool a_first = i1l - i2l >= 0;
    o.id1 = a_first ? A.id : B.id;
    o.id2 = a_first ? B.id : A.id;
    o.pos1 = a_first ? i1l - i2l : i2l - i1l;
    if (!pA && !pB) {                                                       // S-S :202-243
        const int lenA = (int)A.len1, lenB = (int)B.len1;
        if (o.pos1 > (a_first ? lenA : lenB)) return false;
        o.len1 = a_first ? min(lenA - o.pos1, lenB) : min(lenA, lenB - o.pos1);
        o.perc = perc_of(o.len1, lenA, lenB);
        o.type1 = 's'; o.type2 = 's';
        return true;
    }
    if (pA && !pB) {                                                        // P-S :244-287
        const int lenA1 = (int)A.len1, lenA2 = (int)A.len2, lenB = (int)B.len1;
        o.len1 = a_first ? lenA1 - o.pos1 : min(lenA1, lenB - o.pos1);
        if (o.len1 <= 0) return false;
        o.type1 = a_first ? 'p' : 's'; o.type2 = a_first ? 's' : 'p';
        o.perc = perc_one(o.len1, lenA1);
        o.pos2 = i2r - i1r;
        o.len2 = min(lenA2, lenB - o.pos2);
        if (o.len2 <= 0 || o.pos2 < 0) return false;
        o.perc2 = perc_one(o.len2, lenA2);
        return true;
    }
    if (!pA && pB) {                                                        // S-P :288-331
        const int lenA = (int)A.len1, lenB1 = (int)B.len1, lenB2 = (int)B.len2;
        o.len1 = a_first ? min(lenB1, lenA - o.pos1) : lenB1 - o.pos1;
        if (o.len1 <= 0) return false;
        o.type1 = a_first ? 's' : 'p'; o.type2 = a_first ? 'p' : 's';
        o.perc = perc_one(o.len1, lenB1);
        o.pos2 = i1r - i2r;
        o.len2 = min(lenB2, lenA - o.pos2);
        if (o.len2 <= 0 || o.pos2 < 0) return false;
        o.perc2 = perc_one(o.len2, lenB2);
        return true;
    }
    const int lenA = (int)A.len1, lenB = (int)B.len1, lenC = (int)A.len2, lenD = (int)B.len2;   // P-P :332-401
    o.len1 = a_first ? min(lenA - o.pos1, lenB) : min(lenA, lenB - o.pos1);
    const bool back = i1r - i2r >= 0;
    o.pos2 = back ? i1r - i2r : i2r - i1r;
    o.len2 = back ? min(lenC - o.pos2, lenD) : min(lenC, lenD - o.pos2);
    if (o.len1 <= 0 || o.len2 <= 0) return false;
    o.perc = perc_of(o.len1, lenA, lenB);
    o.perc2 = perc_of(o.len2, lenC, lenD);
    o.ord = (a_first == back) ? '1' : '2';
    o.type1 = 'p'; o.type2 = 'p';
    return true;
}

__global__ void fno3_count(const u64* off, u64 n, uint32_t* cnt) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) {
        const u64 c = off[k + 1] - off[k];
        cnt[k] = (uint32_t)(c * (c - 1) / 2);
    }
}

// pair keys of the attempts of every original read, attempt order (all pairs i < j of its list, :104-131)
__global__ void fno3_keys(const u64* __restrict__ off, u64 n, const uint32_t* __restrict__ sr_idx, const hc_fno_read* __restrict__ reads,
                          const u64* __restrict__ seq0, u64* __restrict__ keys) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) {
        u64 seq = seq0[k];
        const u64 b = off[k], e = off[k + 1];
        for (u64 i = b; i < e; i++) {
            const u64 idA = reads[sr_idx[i]].id;
            for (u64 j = i + 1; j < e; j++, seq++) keys[seq] = pair_key(idA, reads[sr_idx[j]].id);
        }
    }
}

template <bool SMALL>
__global__ void fno3_resolve(const u64* __restrict__ off, u64 n, const uint32_t* __restrict__ sr_idx, const hc_fno3_pos* __restrict__ sr_pos,
                             const hc_fno_read* __restrict__ reads, uint32_t no_inclusions, const u64* __restrict__ seq0,
                             const uint8_t* __restrict__ win, uint32_t* __restrict__ flags, void* __restrict__ rec, uint32_t* overflow) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) {
        u64 seq = seq0[k];
        const u64 b = off[k], e = off[k + 1];
        for (u64 i = b; i < e; i++) {
            for (u64 j = i + 1; j < e; j++, seq++) {
                bool ok = win[seq] != 0;                                       // first original wins, :116-121
                if (ok) {
                    const hc_fno_read A = reads[sr_idx[i]], B = reads[sr_idx[j]];
                    hc_fno_overlap o;
                    ok = deduce_overlap(A, B, sr_pos[i], sr_pos[j], o);
                    if (ok) {
                        const unsigned perc = o.perc2 > 0 ? (unsigned)(0.5 * (o.perc + o.perc2)) : (unsigned)o.perc;   // Overlap::get_perc
                        ok = !(no_inclusions && perc == 100) && o.len1 > 0;      // :157-165
                    }
                    if (ok) stage<SMALL>(rec, seq, o, overflow);
                }
                flags[seq] = ok;
            }
        }
    }
}

// ---- the non-edge segment of the FNO1 stream (hc_fno1_text_nonedges) -----------------------------------------------------
// First position of every ordered vertex pair (u, v) of the adjacency segment: the claim of ffw_claim, keyed by u << 32 | v.
__global__ void adj_claim(const hc_fno_edge* __restrict__ adj, u64 n, Cell* __restrict__ tab, uint32_t mask) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        const uint2 uv = __ldg(reinterpret_cast<const uint2*>(adj + t));
        const u64 key = ((u64)uv.x << 32) | uv.y;
        uint32_t s = key_slot(mix64(key), mask);
        while (true) {
            const u64 prev = atomicCAS(&tab[s].key, ~0ull, key);
            if (prev == ~0ull || prev == key) break;
            s = (s + 1) & mask;
        }
        atomicMin(&tab[s].min, t);
    }
}

__device__ __forceinline__ u64 adj_first(const Cell* __restrict__ tab, uint32_t mask, u64 key) {   // ~0: no such pair
    uint32_t s = key_slot(mix64(key), mask);
    while (true) {
        const u64 k = tab[s].key;
        if (k == key) return tab[s].min;
        if (k == ~0ull) return ~0ull;
        s = (s + 1) & mask;
    }
}

// keep[i] = !(checkEdge(v1, v2, true) > 0), src/FindNextOverlaps.cpp:694-696 with OverlapGraph::checkEdge
// (src/OverlapGraph.cpp:233-259): the first adjacency entry v1 -> v2 decides, and only if there is none the first
// v2 -> v1; its score is > 0 exactly when it is not a non-edge overlap (adjacency scores are never negative).
__global__ void nonedge_probe(const hc_candidate* __restrict__ c, u64 n, const Cell* __restrict__ tab, uint32_t mask,
                              const hc_fno_edge* __restrict__ adj, uint32_t* __restrict__ keep) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const uint2 uv = __ldg(reinterpret_cast<const uint2*>(c + i));
        u64 p = adj_first(tab, mask, ((u64)uv.x << 32) | uv.y);
        if (p == ~0ull) p = adj_first(tab, mask, ((u64)uv.y << 32) | uv.x);
        keep[i] = p == ~0ull || __ldg(&adj[p].nonedge) != 0;
    }
}

// the kept lines as stream edges, in file order: the Edge of :640-690 (score 0, fields of the Overlap) as to_fno_edge
// of hcb_fno.cpp makes it
__global__ void nonedge_scatter(const hc_candidate* __restrict__ c, const uint32_t* __restrict__ keep, const u64* __restrict__ pos,
                                u64 n, hc_fno_edge* __restrict__ out) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (!keep[i]) continue;
        const hc_candidate a = c[i];
        hc_fno_edge e;
        e.u = a.idx1; e.v = a.idx2;
        e.pos1 = (int32_t)a.pos1; e.pos2 = (int32_t)a.pos2;
        e.perc = a.perc2 > 0 ? (int32_t)(uint32_t)(0.5 * (double)((uint32_t)a.perc1 + (uint32_t)a.perc2)) : (int32_t)a.perc1;   // Overlap::get_perc
        e.len1 = (int32_t)a.len1; e.len2 = (int32_t)a.len2;
        e.ord = a.ord; e.ori1 = a.ori1; e.ori2 = a.ori2; e.nonedge = 1;
        out[pos[i]] = e;
    }
}

thread_local std::string g_fno_err;

}  // namespace

static bool fno_force_big() { const char* v = getenv("HC_FNO_STAGE48"); return v && *v && *v != '0'; }

// Winners are known (d_win); stage the successful attempts, rank them, move them to the output.  `resolve(small)` launches
// the resolve kernel with the given staging format.  Exactly one of out48 / out24 / txt is non-null; with txt the compacted
// records stay on the device (24-byte ones unless a value needed 48-byte staging) and fno_text turns them into the file.
template <class Resolve>
static int fno_finish(Resolve resolve, u64 attempts, hc_fno_overlap* out48, hc_fno_overlap_small* out24, const FnoText* txt,
                      u64 out_cap, uint64_t* n_out, FnoPhase& ph, const char* who) {
    int rc = HC_OK;
    uint32_t *d_flags = nullptr, *d_ovf = nullptr, ovf = 0;
    u64 *d_outpos = nullptr, *d_total = nullptr, *d_bsum = nullptr, produced = 0;
    void *d_rec = nullptr, *d_out = nullptr;
    bool small = !fno_force_big(), out_small;
    FCU(hc_scratch_alloc((void**)&d_flags, attempts * sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_outpos, attempts * sizeof(u64)));
    FCU(hc_scratch_alloc((void**)&d_ovf, sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_total, sizeof(u64)));
    FCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(attempts) * sizeof(u64)));
    for (int attempt = 0; attempt < 2; attempt++) {
        FCU(cudaMemsetAsync(d_ovf, 0, sizeof(uint32_t)));
        FCU(hc_scratch_alloc(&d_rec, attempts * (small ? sizeof(Rec24) : sizeof(hc_fno_overlap))));
        resolve(small, d_flags, d_rec, d_ovf);
        FCU(cudaGetLastError());
        ph.mark(small ? "resolve (24-byte staging)" : "resolve (48-byte staging)");
        if (!small) break;
        FCU(cudaMemcpy(&ovf, d_ovf, sizeof(uint32_t), cudaMemcpyDeviceToHost));
        if (!ovf) break;
        if (out24) {
            hc_set_last_error((std::string(who) + ": a value does not fit the 24-byte record (ids below 2^32, positions and lengths "
                               "below 2^24, ord in '1','2','-'); use the 48-byte entry point").c_str());
            rc = HC_ERR_ARG;
            goto done;
        }
        hc_scratch_free(d_rec); d_rec = nullptr;
        small = false;
    }
    hc_scan::exclusive_u32(d_flags, attempts, d_outpos, d_total, d_bsum, 0);
    FCU(cudaMemcpy(&produced, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
    *n_out = produced;
    if (!txt && produced > out_cap) {
        hc_set_last_error((std::string(who) + ": output buffer too small (required size returned in n_out)").c_str());
        rc = HC_ERR_CAPACITY;
        goto done;
    }
    if (produced == 0) {
        if (txt) rc = fno_text((const hc_fno_overlap_small*)nullptr, 0, *txt, ph, who);
        goto done;
    }
    out_small = out24 || (txt && small);
    FCU(hc_scratch_alloc(&d_out, produced * (out_small ? sizeof(Rec24) : sizeof(hc_fno_overlap))));
    ph.mark("scan of flags");
    if (out_small) fno_compact<true, true><<<148 * 16, 256>>>(d_flags, d_outpos, d_rec, attempts, d_out, produced);
    else if (small) fno_compact<true, false><<<148 * 16, 256>>>(d_flags, d_outpos, d_rec, attempts, d_out, produced);
    else fno_compact<false, false><<<148 * 16, 256>>>(d_flags, d_outpos, d_rec, attempts, d_out, produced);
    FCU(cudaGetLastError());
    ph.mark("fno_compact");
    if (txt) {
        hc_scratch_free(d_flags); hc_scratch_free(d_outpos); hc_scratch_free(d_rec);   // the text stage needs the room
        d_flags = nullptr; d_outpos = nullptr; d_rec = nullptr;
        if (out_small) rc = fno_text(static_cast<const hc_fno_overlap_small*>(d_out), produced, *txt, ph, who);
        else rc = fno_text(static_cast<const hc_fno_overlap*>(d_out), produced, *txt, ph, who);
        goto done;
    }
    if (out24) FCU(hc_copy_d2h(out24, d_out, produced * sizeof(Rec24)));
    else FCU(hc_copy_d2h(out48, d_out, produced * sizeof(hc_fno_overlap)));
    ph.mark("copy out");
done:
    hc_scratch_free(d_flags); hc_scratch_free(d_outpos); hc_scratch_free(d_ovf); hc_scratch_free(d_total); hc_scratch_free(d_bsum);
    hc_scratch_free(d_rec); hc_scratch_free(d_out);
    return rc;
}

static bool fno_edges_in_range(const hc_fno_edge* edges, uint64_t n_edges, u64 V, const char* who) {
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)n_edges; i++) bad |= (edges[i].u >= V || edges[i].v >= V);
    if (bad) hc_set_last_error((std::string(who) + ": edge vertex out of range").c_str());
    return !bad;
}

// The checks of hc_fno_input (the edges are checked by the caller)
static int fno1_check_input(const hc_fno_input* in, const char* who) {
    const u64 V = in->n_vertices, NS = in->n_superreads;
    int bad = 0;
    const u64 nsr = V ? in->sr_off[V] : 0;
    if (nsr >> 32) { hc_set_last_error((std::string(who) + ": more than 2^32 super-read list entries").c_str()); return HC_ERR_ARG; }
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)nsr; i++) bad |= (in->sr_idx[i] >= NS);
    if (bad) { hc_set_last_error((std::string(who) + ": super-read index out of range").c_str()); return HC_ERR_ARG; }
    // the first-found-wins table keys a pair of new reads as (min id << 32 | max id): every id that can appear in a key
    // -- a super-read's, an unmerged vertex' -- must fit 32 bits (rename_fas.py numbers reads from 0), else distinct
    // pairs would collide and overlaps the reference finds would be dropped silently
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)NS; i++) bad |= (in->superread[i].id >> 32) != 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long v = 0; v < (long long)V; v++) bad |= (!in->visited[v] && in->vertex_read[v].id != ~0ull && (in->vertex_read[v].id >> 32) != 0);
    if (bad) { hc_set_last_error((std::string(who) + ": a new read id does not fit 32 bits (ids of new reads must be below 2^32)").c_str()); return HC_ERR_ARG; }
    return HC_OK;
}

// FNO1 on `device`.  The edge stream is either the host array `edges` (checked, with `in`, and copied here) or, with
// d_edges_in, already in HBM -- then the caller has checked the edges and `in` (fno1_check_input).
static int fno1_impl(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges, const hc_fno_edge* d_edges_in,
                     hc_fno_overlap* out48, hc_fno_overlap_small* out24, const FnoText* txt, uint64_t out_cap, uint64_t* n_out,
                     int device, const char* who = nullptr) {
    if (!who) who = txt ? "hc_fno1_text" : (out24 ? "hc_fno1_small" : "hc_fno1");
    if (!in || !n_out || (n_edges && !edges && !d_edges_in) || (out_cap && !out48 && !out24)) { hc_set_last_error((std::string(who) + ": NULL argument").c_str()); return HC_ERR_ARG; }
    *n_out = 0;
    const u64 V = in->n_vertices, NS = in->n_superreads;
    int rc = HC_OK;
    if (!d_edges_in) {                                          // device edges: the caller has checked them and `in`
        if (!fno_edges_in_range(edges, n_edges, V, who)) return HC_ERR_ARG;
        if ((rc = fno1_check_input(in, who)) != HC_OK) return rc;
    }
    const u64 nsr = V ? in->sr_off[V] : 0;
    FnoPhase ph(who);
    ph.mark("argument checks");
    uint8_t *d_vis = nullptr, *d_lab = nullptr, *d_win = nullptr;
    hc_fno_read *d_vr = nullptr, *d_sr = nullptr;
    u64 *d_sroff = nullptr, *d_off = nullptr, *d_total = nullptr, *d_keys = nullptr, *d_bsum = nullptr;
    uint32_t *d_sridx = nullptr, *d_cnt = nullptr;
    hc_fno_subread* d_sub = nullptr;
    hc_fno_edge* d_edges_own = nullptr;
    const hc_fno_edge* d_edges = d_edges_in;
    VDesc* d_vd = nullptr;
    EDesc* d_en = nullptr;
    u64 attempts = 0;
    DevIn D;
    const int threads = 256;
    int blocks, vblocks;
    FCU(cudaSetDevice(device));
    if (n_edges == 0) goto done;
    blocks = (int)((n_edges + threads - 1) / threads < 8192 ? (n_edges + threads - 1) / threads : 8192);
    vblocks = (int)((V + threads - 1) / threads < 4096 ? (V + threads - 1) / threads : 4096);
    FCU(hc_scratch_alloc((void**)&d_vis, V ? V : 1)); FCU(hc_scratch_alloc((void**)&d_lab, V ? V : 1));
    FCU(hc_scratch_alloc((void**)&d_vr, (V ? V : 1) * sizeof(hc_fno_read))); FCU(hc_scratch_alloc((void**)&d_sr, (NS ? NS : 1) * sizeof(hc_fno_read)));
    FCU(hc_scratch_alloc((void**)&d_sroff, (V + 1) * sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_sridx, (nsr ? nsr : 1) * sizeof(uint32_t)));
    FCU(hc_scratch_alloc((void**)&d_sub, (nsr ? nsr : 1) * sizeof(hc_fno_subread)));
    FCU(hc_scratch_alloc((void**)&d_vd, (V ? V : 1) * sizeof(VDesc))); FCU(hc_scratch_alloc((void**)&d_en, (nsr ? nsr : 1) * sizeof(EDesc)));
    if (!d_edges_in) FCU(hc_scratch_alloc((void**)&d_edges_own, n_edges * sizeof(hc_fno_edge)));
    FCU(hc_scratch_alloc((void**)&d_cnt, n_edges * sizeof(uint32_t)));
    FCU(hc_scratch_alloc((void**)&d_off, n_edges * sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_total, sizeof(u64)));
    FCU(hc_copy_h2d(d_vis, in->visited, V)); FCU(hc_copy_h2d(d_lab, in->label, V));
    FCU(hc_copy_h2d(d_vr, in->vertex_read, V * sizeof(hc_fno_read)));
    FCU(hc_copy_h2d(d_sr, in->superread, NS * sizeof(hc_fno_read)));
    FCU(hc_copy_h2d(d_sroff, in->sr_off, (V + 1) * sizeof(u64)));
    FCU(hc_copy_h2d(d_sridx, in->sr_idx, nsr * sizeof(uint32_t)));
    FCU(hc_copy_h2d(d_sub, in->sr_sub, nsr * sizeof(hc_fno_subread)));
    // the packed per-vertex / per-entry records are built while the edges (the bulk of the input) are still being copied
    fno_prep_vertices<<<vblocks, threads>>>(V, d_vis, d_lab, d_vr, d_sroff, d_vd);
    fno_prep_entries<<<vblocks, threads>>>(V, d_vr, d_sroff, d_sridx, d_sub, d_sr, d_en);
    if (!d_edges_in) {
        FCU(hc_copy_h2d(d_edges_own, edges, n_edges * sizeof(hc_fno_edge)));
        d_edges = d_edges_own;
    }
    ph.mark("allocations + copies in");
    D.vd = d_vd; D.en = d_en; D.resolve_orientations = in->resolve_orientations; D.no_inclusions = in->no_inclusions;
    fno_count<<<blocks, threads>>>(D, d_edges, n_edges, d_cnt);
    FCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(n_edges) * sizeof(u64)));
    hc_scan::exclusive_u32(d_cnt, n_edges, d_off, d_total, d_bsum, 0);
    FCU(cudaMemcpy(&attempts, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
    ph.mark("count + scan");
    if (attempts == 0) goto done;
    FCU(hc_scratch_alloc((void**)&d_keys, attempts * sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_win, attempts));
    FCU(cudaMemsetAsync(d_win, 0, attempts));
    fno_keys<<<blocks, threads>>>(D, d_edges, n_edges, d_off, d_keys);
    ph.mark("fno_keys");
    FCU(ffw_winners(d_keys, attempts, d_win));
    ph.mark("first-found-wins passes");
    hc_scratch_free(d_keys); d_keys = nullptr;
    rc = fno_finish([&](bool small, uint32_t* d_flags, void* d_rec, uint32_t* d_ovf) {
        if (small) fno_resolve<true><<<blocks, threads>>>(D, d_edges, n_edges, d_off, d_win, d_flags, d_rec, d_ovf);
        else fno_resolve<false><<<blocks, threads>>>(D, d_edges, n_edges, d_off, d_win, d_flags, d_rec, d_ovf);
    }, attempts, out48, out24, txt, out_cap, n_out, ph, who);
done:
    hc_scratch_free(d_vis); hc_scratch_free(d_lab); hc_scratch_free(d_vr); hc_scratch_free(d_sr); hc_scratch_free(d_sroff); hc_scratch_free(d_sridx); hc_scratch_free(d_sub);
    hc_scratch_free(d_edges_own); hc_scratch_free(d_cnt); hc_scratch_free(d_off); hc_scratch_free(d_total); hc_scratch_free(d_keys);
    hc_scratch_free(d_bsum); hc_scratch_free(d_win); hc_scratch_free(d_vd); hc_scratch_free(d_en);
    return rc;
}

extern "C" int hc_fno1(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges, hc_fno_overlap* out, uint64_t out_cap,
                       uint64_t* n_out, int device) {
    return fno1_impl(in, edges, n_edges, nullptr, out, nullptr, nullptr, out_cap, n_out, device);
}

extern "C" int hc_fno1_small(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges, hc_fno_overlap_small* out,
                             uint64_t out_cap, uint64_t* n_out, int device) {
    return fno1_impl(in, edges, n_edges, nullptr, nullptr, out, nullptr, out_cap, n_out, device);
}

static int fno3_impl(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos, uint64_t n_reads,
                     const hc_fno_read* reads, int no_inclusions, hc_fno_overlap* out48, hc_fno_overlap_small* out24, const FnoText* txt,
                     uint64_t out_cap, uint64_t* n_out, int device) {
    const char* who = txt ? "hc_fno3_text" : (out24 ? "hc_fno3_small" : "hc_fno3");
    if (!n_out || (n_originals && (!off || !sr_idx || !sr_pos || !reads)) || (out_cap && !out48 && !out24)) {
        hc_set_last_error((std::string(who) + ": NULL argument").c_str());
        return HC_ERR_ARG;
    }
    *n_out = 0;
    if (n_originals == 0) return HC_OK;
    const u64 nent = off[n_originals];
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)nent; i++) bad |= (sr_idx[i] >= n_reads);
    if (bad) { hc_set_last_error((std::string(who) + ": read index out of range").c_str()); return HC_ERR_ARG; }
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)n_reads; i++) bad |= (reads[i].id >> 32) != 0;      // pair keys are (min id << 32 | max id)
    if (bad) { hc_set_last_error((std::string(who) + ": a new read id does not fit 32 bits (ids of new reads must be below 2^32)").c_str()); return HC_ERR_ARG; }
    int rc = HC_OK;
    FnoPhase ph(who);
    u64 *d_off = nullptr, *d_seq = nullptr, *d_total = nullptr, *d_keys = nullptr, *d_bsum = nullptr;
    uint32_t *d_idx = nullptr, *d_cnt = nullptr;
    uint8_t* d_win = nullptr;
    hc_fno3_pos* d_pos = nullptr;
    hc_fno_read* d_reads = nullptr;
    u64 attempts = 0;
    const int threads = 128;
    const int blocks = (int)((n_originals + threads - 1) / threads < 8192 ? (n_originals + threads - 1) / threads : 8192);
    FCU(cudaSetDevice(device));
    FCU(hc_scratch_alloc((void**)&d_off, (n_originals + 1) * sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_idx, (nent ? nent : 1) * sizeof(uint32_t)));
    FCU(hc_scratch_alloc((void**)&d_pos, (nent ? nent : 1) * sizeof(hc_fno3_pos))); FCU(hc_scratch_alloc((void**)&d_reads, (n_reads ? n_reads : 1) * sizeof(hc_fno_read)));
    FCU(hc_scratch_alloc((void**)&d_cnt, n_originals * sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_seq, n_originals * sizeof(u64)));
    FCU(hc_scratch_alloc((void**)&d_total, sizeof(u64)));
    FCU(hc_copy_h2d(d_off, off, (n_originals + 1) * sizeof(u64)));
    FCU(hc_copy_h2d(d_idx, sr_idx, nent * sizeof(uint32_t)));
    FCU(hc_copy_h2d(d_pos, sr_pos, nent * sizeof(hc_fno3_pos)));
    FCU(hc_copy_h2d(d_reads, reads, n_reads * sizeof(hc_fno_read)));
    ph.mark("allocations + copies in");
    fno3_count<<<blocks, threads>>>(d_off, n_originals, d_cnt);
    FCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(n_originals) * sizeof(u64)));
    hc_scan::exclusive_u32(d_cnt, n_originals, d_seq, d_total, d_bsum, 0);
    FCU(cudaMemcpy(&attempts, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
    if (attempts == 0) goto done;
    FCU(hc_scratch_alloc((void**)&d_keys, attempts * sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_win, attempts));
    FCU(cudaMemsetAsync(d_win, 0, attempts));
    fno3_keys<<<blocks, threads>>>(d_off, n_originals, d_idx, d_reads, d_seq, d_keys);
    ph.mark("count + scan + keys");
    FCU(ffw_winners(d_keys, attempts, d_win));
    ph.mark("first-found-wins passes");
    hc_scratch_free(d_keys); d_keys = nullptr;
    rc = fno_finish([&](bool small, uint32_t* d_flags, void* d_rec, uint32_t* d_ovf) {
        if (small) fno3_resolve<true><<<blocks, threads>>>(d_off, n_originals, d_idx, d_pos, d_reads, (uint32_t)no_inclusions, d_seq, d_win, d_flags, d_rec, d_ovf);
        else fno3_resolve<false><<<blocks, threads>>>(d_off, n_originals, d_idx, d_pos, d_reads, (uint32_t)no_inclusions, d_seq, d_win, d_flags, d_rec, d_ovf);
    }, attempts, out48, out24, txt, out_cap, n_out, ph, who);
done:
    hc_scratch_free(d_off); hc_scratch_free(d_idx); hc_scratch_free(d_pos); hc_scratch_free(d_reads); hc_scratch_free(d_cnt); hc_scratch_free(d_seq); hc_scratch_free(d_total);
    hc_scratch_free(d_keys); hc_scratch_free(d_bsum); hc_scratch_free(d_win);
    return rc;
}

extern "C" int hc_fno3(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos, uint64_t n_reads,
                       const hc_fno_read* reads, int no_inclusions, hc_fno_overlap* out, uint64_t out_cap, uint64_t* n_out,
                       int device) {
    return fno3_impl(n_originals, off, sr_idx, sr_pos, n_reads, reads, no_inclusions, out, nullptr, nullptr, out_cap, n_out, device);
}

extern "C" int hc_fno3_small(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos, uint64_t n_reads,
                             const hc_fno_read* reads, int no_inclusions, hc_fno_overlap_small* out, uint64_t out_cap, uint64_t* n_out,
                             int device) {
    return fno3_impl(n_originals, off, sr_idx, sr_pos, n_reads, reads, no_inclusions, nullptr, out, nullptr, out_cap, n_out, device);
}

// ---- overlaps.txt itself (hc_fno_text.cu) --------------------------------------------------------------------------------
static bool text_args_ok(const char* who, const char* text, uint64_t text_cap, uint64_t* n_bytes, uint64_t* n_lines) {
    if (!n_bytes || !n_lines || (text_cap && !text)) { hc_set_last_error((std::string(who) + ": NULL argument").c_str()); return false; }
    *n_bytes = 0;
    *n_lines = 0;
    return true;
}

extern "C" int hc_fno1_text(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges, char* text, uint64_t text_cap,
                            uint64_t* n_bytes, uint64_t* n_lines, uint64_t* n_records, int device) {
    if (!text_args_ok("hc_fno1_text", text, text_cap, n_bytes, n_lines)) return HC_ERR_ARG;
    const FnoText t = {text, text_cap, n_bytes, n_lines, true};
    uint64_t records = 0;
    const int rc = fno1_impl(in, edges, n_edges, nullptr, nullptr, nullptr, &t, 0, &records, device);
    if (n_records) *n_records = records;
    return rc;
}

// head ++ (the lines of nonedge_text that are not an edge of the adjacency segment) ++ tail, built in HBM.  The text goes
// through the pieces of hc_ingest_cuts (two device buffers, the copy of piece i + 1 overlapping the work on piece i); every
// piece is parsed by the ingestion parser in all-lines mode, probed against the adjacency pairs and compacted in file order
// behind what the earlier pieces kept.  No line is kept past an error line: on HC_ERR_INPUT the stream is discarded.
static int fno1_nonedge_stream(const hc_idmap* m, const hc_fno_edge* head, uint64_t n_head, uint64_t n_adjacency,
                               const char* text, uint64_t n_bytes, const hc_fno_edge* tail, uint64_t n_tail,
                               hc_fno_edge** d_stream_out, hc_fno_nonedge_stats* stats, const char* who) {
    int rc = HC_OK;
    const std::vector<uint64_t> cut = hc_ingest_cuts(text, n_bytes, hc_ingest_piece_bytes());
    const size_t n_pieces = cut.size() - 1;
    u64 max_piece = 0, bound = n_head + n_tail;
    for (size_t i = 0; i < n_pieces; i++) {
        max_piece = std::max<u64>(max_piece, cut[i + 1] - cut[i]);
        bound += hc_ingest_all_cap(cut[i + 1] - cut[i]);
    }
    const u64 tbytes = (max_piece + 16 + 255) & ~255ull, cap = hc_ingest_all_cap(max_piece);
    u64 slots = 1024, kept = 0, lines = 0, total = 0;
    while (slots < 2 * n_adjacency + 2) slots <<= 1;
    hc_fno_edge* d_stream = nullptr;
    char* d_text = nullptr;
    hc_candidate* d_cand = nullptr;
    uint32_t* d_keep = nullptr;
    u64 *d_pos = nullptr, *d_total = nullptr, *d_bsum = nullptr;
    Cell* d_tab = nullptr;
    cudaStream_t s_copy = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, t0 = nullptr, t1 = nullptr;
    hc_ingest_params ip;
    memset(&ip, 0, sizeof(ip));
    ip.max_overlaps = ~0ull;                                     // the loop reads the whole file; ORD / ORI / TYPE split on tabs only
    FCU(cudaStreamCreateWithFlags(&s_copy, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) FCU(cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
    FCU(cudaEventCreate(&t0)); FCU(cudaEventCreate(&t1));
    FCU(cudaEventRecord(t0, 0));
    FCU(hc_scratch_alloc((void**)&d_stream, (bound ? bound : 1) * sizeof(hc_fno_edge)));
    FCU(hc_copy_h2d(d_stream, head, n_head * sizeof(hc_fno_edge)));
    if (n_pieces) {
        FCU(hc_scratch_alloc((void**)&d_text, 2 * tbytes));
        FCU(hc_scratch_alloc((void**)&d_cand, cap * sizeof(hc_candidate)));
        FCU(hc_scratch_alloc((void**)&d_keep, cap * sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_pos, cap * sizeof(u64)));
        FCU(hc_scratch_alloc((void**)&d_total, sizeof(u64))); FCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(cap) * sizeof(u64)));
        FCU(hc_scratch_alloc((void**)&d_tab, slots * sizeof(Cell)));
        FCU(cudaMemsetAsync(d_tab, 0xff, slots * sizeof(Cell)));
        if (n_adjacency) {
            const int ab = (int)std::min<u64>((n_adjacency + 255) / 256, 148 * 16);
            adj_claim<<<ab, 256>>>(d_stream, n_adjacency, d_tab, (uint32_t)(slots - 1));
            FCU(cudaGetLastError());
        }
        FCU(hc_copy_h2d_on(d_text, text, cut[1] - cut[0], s_copy));
        FCU(cudaEventRecord(ev_in[0], s_copy));
    }
    for (size_t i = 0; i < n_pieces; i++) {
        const int b = (int)(i & 1);
        if (i + 1 < n_pieces) {   // buffer b ^ 1 held piece i - 1, whose work has completed (the kept count below is read back)
            FCU(hc_copy_h2d_on(d_text + (size_t)(b ^ 1) * tbytes, text + cut[i + 1], cut[i + 2] - cut[i + 1], s_copy));
            FCU(cudaEventRecord(ev_in[b ^ 1], s_copy));
        }
        FCU(cudaStreamWaitEvent(0, ev_in[b], 0));
        hc_ingest_stats st;
        rc = hc_ingest_device(m, d_text + (size_t)b * tbytes, cut[i + 1] - cut[i], &ip, d_cand, nullptr, cap, nullptr, nullptr, 0,
                              &st, 0, 0, true);
        if (rc != HC_OK) goto done;
        if (st.first_error_line != ~0ull) {
            stats->first_error_line = lines + st.first_error_line;
            stats->first_error_offset = cut[i] + st.first_error_offset;
            stats->first_error_length = st.first_error_length;
            stats->first_error_status = st.first_error_status;
            const char* what = st.first_error_status == HC_LINE_SKIPPED ? "not 13 tab-separated fields"
                               : st.first_error_status == HC_LINE_UNKNOWN_ID ? "a read id that is not in the id map"
                                                                             : "fields the Overlap constructor rejects";
            hc_set_last_error((std::string(who) + ": line " + std::to_string(stats->first_error_line) + " of the non-edge text has " + what).c_str());
            rc = HC_ERR_INPUT;
            goto done;
        }
        lines += st.n_lines;
        if (st.n_scored) {
            const int pb = (int)std::min<u64>((st.n_scored + 255) / 256, 148 * 16);
            nonedge_probe<<<pb, 256>>>(d_cand, st.n_scored, d_tab, (uint32_t)(slots - 1), d_stream, d_keep);
            hc_scan::exclusive_u32(d_keep, st.n_scored, d_pos, d_total, d_bsum, 0);
            nonedge_scatter<<<pb, 256>>>(d_cand, d_keep, d_pos, st.n_scored, d_stream + n_head + kept);
            FCU(cudaGetLastError());
            FCU(cudaMemcpy(&total, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
            kept += total;
        }
    }
    FCU(hc_copy_h2d(d_stream + n_head + kept, tail, n_tail * sizeof(hc_fno_edge)));
    FCU(cudaEventRecord(t1, 0));
    FCU(cudaEventSynchronize(t1));
    FCU(cudaEventElapsedTime(&stats->device_ms, t0, t1));
    stats->n_lines = lines;
    stats->n_nonedges = kept;
    stats->n_stream = n_head + kept + n_tail;
    *d_stream_out = d_stream;
    d_stream = nullptr;
done:
    if (s_copy) { cudaStreamSynchronize(s_copy); cudaStreamDestroy(s_copy); }
    for (int k = 0; k < 2; k++) if (ev_in[k]) cudaEventDestroy(ev_in[k]);
    if (t0) cudaEventDestroy(t0);
    if (t1) cudaEventDestroy(t1);
    hc_scratch_free(d_stream); hc_scratch_free(d_text); hc_scratch_free(d_cand); hc_scratch_free(d_keep); hc_scratch_free(d_pos);
    hc_scratch_free(d_total); hc_scratch_free(d_bsum); hc_scratch_free(d_tab);
    return rc;
}

extern "C" int hc_fno1_text_nonedges(const hc_fno_input* in, const hc_idmap* m, const hc_fno_edge* head, uint64_t n_head,
                                     uint64_t n_adjacency, const char* nonedge_text, uint64_t nonedge_bytes, const hc_fno_edge* tail,
                                     uint64_t n_tail, char* text, uint64_t text_cap, uint64_t* n_bytes, uint64_t* n_lines,
                                     uint64_t* n_records, hc_fno_nonedge_stats* stats, int device) {
    const char* who = "hc_fno1_text_nonedges";
    if (!text_args_ok(who, text, text_cap, n_bytes, n_lines)) return HC_ERR_ARG;
    if (!in || !m || !stats || (n_head && !head) || (n_tail && !tail) || (nonedge_bytes && !nonedge_text)) {
        hc_set_last_error((std::string(who) + ": NULL argument").c_str());
        return HC_ERR_ARG;
    }
    memset(stats, 0, sizeof(*stats));
    stats->first_error_line = ~0ull;
    if (n_records) *n_records = 0;
    const u64 V = in->n_vertices;
    if (m->device != device) { hc_set_last_error((std::string(who) + ": the id map is on another device").c_str()); return HC_ERR_ARG; }
    if (m->n != V) { hc_set_last_error((std::string(who) + ": the id map does not hold one read per vertex (vertex i is read i)").c_str()); return HC_ERR_ARG; }
    if (n_adjacency > n_head) { hc_set_last_error((std::string(who) + ": n_adjacency > n_head").c_str()); return HC_ERR_ARG; }
    for (u64 i = 1; i < n_adjacency; i++)
        if (head[i].u < head[i - 1].u) { hc_set_last_error((std::string(who) + ": the adjacency lists are not in vertex order").c_str()); return HC_ERR_ARG; }
    if (!fno_edges_in_range(head, n_head, V, who) || !fno_edges_in_range(tail, n_tail, V, who)) return HC_ERR_ARG;
    int rc = fno1_check_input(in, who);
    if (rc != HC_OK) return rc;
    hc_fno_edge* d_stream = nullptr;
    FCU(cudaSetDevice(device));
    {
        FnoPhase ph(who);
        rc = fno1_nonedge_stream(m, head, n_head, n_adjacency, nonedge_text, nonedge_bytes, tail, n_tail, &d_stream, stats, who);
        if (rc != HC_OK) goto done;
        ph.mark("stream with non-edge lines");
    }
    {
        const FnoText t = {text, text_cap, n_bytes, n_lines, true};
        uint64_t records = 0;
        rc = fno1_impl(in, nullptr, stats->n_stream, d_stream, nullptr, nullptr, &t, 0, &records, device, who);
        if (n_records) *n_records = records;
    }
done:
    hc_scratch_free(d_stream);
    return rc;
}

extern "C" int hc_fno3_text(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos, uint64_t n_reads,
                            const hc_fno_read* reads, int no_inclusions, char* text, uint64_t text_cap, uint64_t* n_bytes,
                            uint64_t* n_lines, int device) {
    if (!text_args_ok("hc_fno3_text", text, text_cap, n_bytes, n_lines)) return HC_ERR_ARG;
    const FnoText t = {text, text_cap, n_bytes, n_lines, false};
    uint64_t records = 0;
    return fno3_impl(n_originals, off, sr_idx, sr_pos, n_reads, reads, no_inclusions, nullptr, nullptr, &t, 0, &records, device);
}
