// hc_adjacency.cu -- the adjacency lists of the overlap graph on the device: OverlapGraph::addEdge in insertion order
// (src/OverlapGraph.cpp:94-101) and OverlapGraph::sortEdges (:722-764: every list ordered by non-overlap length, then
// vertex2; adj_in rebuilt by walking the sorted lists).  SURVEY 8f rank 1, second half (the first half -- which edges
// survive the insert -- is hc_dedup_edges).
//
// One primitive, used twice: "group items by bucket and order every group by a 64-bit key, ties by item index":
//   count per bucket (atomicAdd) -> exclusive scan -> scatter with a per-bucket cursor (arbitrary order inside a group)
//   -> one thread per bucket sorts its group in place (hc_radix::sort_run; the order is total, so any sorting algorithm
//   gives the same list).
// adj_out: bucket = vertex1, key = item index (insertion order) or non-overlap length << 32 | vertex2 (sortEdges);
// adj_in:  bucket = vertex2, key = position of the edge in the adj_out order.
#include <cstring>
#include <string>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_radix.cuh"
#include "hc_scan.cuh"
#include "hc_stage.h"

namespace {

typedef unsigned long long u64;

struct Item { u64 key; uint32_t idx; uint32_t pad; };     // 16 bytes

struct ItemLess {
    __device__ bool operator()(const Item& a, const Item& b) const { return a.key != b.key ? a.key < b.key : a.idx < b.idx; }
};

__global__ void adj_count(const hc_adj_edge* __restrict__ e, const uint8_t* __restrict__ keep, u64 n, int by_v2, uint32_t* cnt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (!keep || keep[i]) atomicAdd(&cnt[by_v2 ? e[i].vertex2 : e[i].vertex1], 1u);
}

// adj_out: the kept edges, bucket = vertex1
__global__ void adj_scatter_out(const hc_adj_edge* __restrict__ e, const uint8_t* __restrict__ keep, u64 n, int sort,
                                const u64* __restrict__ off, uint32_t* cursor, Item* items) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (keep && !keep[i]) continue;
        const hc_adj_edge x = e[i];
        const u64 p = off[x.vertex1] + atomicAdd(&cursor[x.vertex1], 1u);
        Item it;
        it.key = sort ? ((u64)x.nonoverlap_len << 32) | x.vertex2 : 0ull;
        it.idx = (uint32_t)i;
        it.pad = 0;
        items[p] = it;
    }
}

// adj_in: the edges in adj_out order (perm), bucket = vertex2, key = position in that order
__global__ void adj_scatter_in(const hc_adj_edge* __restrict__ e, const uint32_t* __restrict__ perm, u64 kept,
                               const u64* __restrict__ off, uint32_t* cursor, Item* items) {
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < kept; p += (u64)gridDim.x * blockDim.x) {
        const hc_adj_edge x = e[perm[p]];
        const u64 q = off[x.vertex2] + atomicAdd(&cursor[x.vertex2], 1u);
        Item it;
        it.key = p;
        it.idx = x.vertex1;          // what the in-list holds: the source vertex
        it.pad = 0;
        items[q] = it;
    }
}

// one thread per bucket; out[p] = idx of the p-th item; tie[v] = 1 if two items of a group of more than 16 share a key
// (std::sort leaves their order to its implementation: the host part settles those lists with std::sort itself)
__global__ void adj_sort_groups(u64 V, const u64* __restrict__ off, Item* items, uint32_t* __restrict__ out, uint8_t* __restrict__ tie) {
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (u64)gridDim.x * blockDim.x) {
        const u64 a = off[v], b = off[v + 1];
        const uint32_t m = (uint32_t)(b - a);
        Item* g = items + a;
        hc_radix::sort_run(g, m, ItemLess());
        bool t = false;
        for (uint32_t i = 0; i < m; i++) {
            out[a + i] = g[i].idx;
            if (i && g[i].key == g[i - 1].key) t = true;
        }
        if (tie) tie[v] = (t && m > 16) ? 1 : 0;
    }
}

}  // namespace

extern "C" int hc_build_adjacency(const hc_adj_edge* edges, uint64_t n, const uint8_t* keep, uint64_t n_vertices, int sort,
                                  uint64_t* out_off, uint32_t* out_perm, uint64_t* in_off, uint32_t* in_src, uint8_t* ties,
                                  uint64_t* n_kept, int device) {
    if (!out_off || !n_kept || (n && (!edges || !out_perm)) || (in_off && n && !in_src)) { hc_set_last_error("hc_build_adjacency: NULL argument"); return HC_ERR_ARG; }
    if (n >> 32) { hc_set_last_error("hc_build_adjacency: more than 2^32 edges"); return HC_ERR_ARG; }
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (long long i = 0; i < (long long)n; i++) bad |= (edges[i].vertex1 >= n_vertices || edges[i].vertex2 >= n_vertices);
    if (bad) { hc_set_last_error("hc_build_adjacency: vertex out of range"); return HC_ERR_ARG; }
    *n_kept = 0;
    const u64 V = n_vertices;
    int rc = HC_OK;
    const char* who = "hc_build_adjacency";
    ScratchBuf<hc_adj_edge> d_e;
    ScratchBuf<uint8_t> d_keep, d_tie;
    ScratchBuf<uint32_t> d_cnt, d_perm, d_src;
    ScratchBuf<u64> d_off, d_total, d_bsum;
    ScratchBuf<Item> d_items;
    u64 kept = 0;
    const int threads = 256, eb = grid_for(n, threads), vb = grid_for(V, threads);
    HC_CU(cudaSetDevice(device));
    if (V == 0) goto done;
    HC_CU(d_cnt.alloc(V + 1)); HC_CU(d_off.alloc(V + 1));
    HC_CU(d_total.alloc(1)); HC_CU(d_bsum.alloc(hc_scan::blocks_for(V + 1)));
    HC_CU(cudaMemsetAsync(d_cnt, 0, (V + 1) * sizeof(uint32_t)));
    if (n) {
        HC_CU(d_e.alloc(n));
        HC_CU(hc_copy_h2d(d_e, edges, n * sizeof(hc_adj_edge)));
        if (keep) { HC_CU(d_keep.alloc(n)); HC_CU(hc_copy_h2d(d_keep, keep, n)); }
        adj_count<<<eb, threads>>>(d_e, d_keep, n, 0, d_cnt);
    }
    hc_scan::exclusive_u32(d_cnt, V + 1, d_off, d_total, d_bsum, 0);
    HC_CU(cudaMemcpy(&kept, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
    *n_kept = kept;
    HC_CU(hc_copy_d2h(out_off, d_off, (V + 1) * sizeof(u64)));
    if (kept) {
        HC_CU(d_items.alloc(kept)); HC_CU(d_perm.alloc(kept));
        if (ties) HC_CU(d_tie.alloc(V));
        HC_CU(cudaMemsetAsync(d_cnt, 0, (V + 1) * sizeof(uint32_t)));
        adj_scatter_out<<<eb, threads>>>(d_e, d_keep, n, sort, d_off, d_cnt, d_items);
        adj_sort_groups<<<vb, threads>>>(V, d_off, d_items, d_perm, sort ? d_tie.get() : nullptr);
        HC_CU(cudaGetLastError());
        HC_CU(hc_copy_d2h(out_perm, d_perm, kept * sizeof(uint32_t)));
        if (ties) { if (sort) HC_CU(hc_copy_d2h(ties, d_tie, V)); else memset(ties, 0, V); }
    } else if (ties) {
        memset(ties, 0, V);
    }
    if (in_off) {
        HC_CU(cudaMemsetAsync(d_cnt, 0, (V + 1) * sizeof(uint32_t)));
        if (n) adj_count<<<eb, threads>>>(d_e, d_keep, n, 1, d_cnt);
        hc_scan::exclusive_u32(d_cnt, V + 1, d_off, d_total, d_bsum, 0);
        HC_CU(hc_copy_d2h(in_off, d_off, (V + 1) * sizeof(u64)));
        if (kept) {
            HC_CU(d_src.alloc(kept));
            HC_CU(cudaMemsetAsync(d_cnt, 0, (V + 1) * sizeof(uint32_t)));
            adj_scatter_in<<<grid_for(kept, threads), threads>>>(d_e, d_perm, kept, d_off, d_cnt, d_items);
            adj_sort_groups<<<vb, threads>>>(V, d_off, d_items, d_src, nullptr);
            HC_CU(cudaGetLastError());
            HC_CU(hc_copy_d2h(in_src, d_src, kept * sizeof(uint32_t)));
        }
    }
done:
    return rc;
}

// ---- SRBuilder::calcSubreadInfo (src/SRBuilder.cpp:536-595) for many super-reads at once -------------------------------
// A super-read is built from a clique whose vertices were ordered left to right (sort_vertices) with their start columns
// (pos_list); consensus() says where the consensus sequence starts (trim_pos).  Per vertex the reference records where the
// vertex' read lies in the trimmed consensus: index = pos - trim_pos (startpos = 0) or, for a read that starts in the
// trimmed-away part, startpos = trim_pos - pos (index = 0) -- for the /1 sequence from list 1, for the /2 sequence from
// list 2 (paired-end super-read, trim_pos2 >= 0) or from a LATER entry of the same vertex in list 1 (single-end super-read
// built from a paired read: both mates are in list 1).  These records are the sr_sub input of hc_fno1.
// One thread per list-1 entry: the first entry of a vertex owns the record; it takes index2 / startpos2 from the last later
// entry of its vertex in list 1, then from the last entry of its vertex in list 2.
namespace {
__global__ void subread_info_kernel(const hc_subread_problem* __restrict__ prob, const uint32_t* __restrict__ entry_problem, u64 n_entries,
                                    const int32_t* __restrict__ pos, const uint32_t* __restrict__ vertex, hc_fno_subread* __restrict__ info,
                                    uint8_t* __restrict__ first) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n_entries; k += (u64)gridDim.x * blockDim.x) {
        const uint32_t pi = entry_problem[k];
        hc_fno_subread r;
        r.index1 = r.index2 = r.startpos1 = r.startpos2 = 0;
        if (pi == 0xffffffffu) { first[k] = 0; info[k] = r; continue; }            // an entry of a list 2
        const hc_subread_problem P = prob[pi];
        const uint32_t v = vertex[k];
        bool own = true;
        for (u64 j = P.begin1; j < k; j++) if (vertex[j] == v) { own = false; break; }
        first[k] = own ? 1 : 0;
        if (!own) { info[k] = r; continue; }
        const int32_t p = pos[k];
        if (P.trim_pos1 > p) { r.startpos1 = P.trim_pos1 - p; r.index1 = 0; }
        else { r.startpos1 = 0; r.index1 = p - P.trim_pos1; }
        r.index2 = -1;
        r.startpos2 = -1;
        for (u64 j = k + 1; j < P.end1; j++) {                                    // :543-556, a later entry of the same vertex: last one wins
            if (vertex[j] != v) continue;
            const int32_t q = pos[j];
            if (P.trim_pos1 > q) { r.startpos2 = P.trim_pos1 - q; r.index2 = 0; }
            else { r.startpos2 = 0; r.index2 = q - P.trim_pos1; }
        }
        if (P.trim_pos2 >= 0) {                                                    // :574-592
            for (u64 j = P.begin2; j < P.end2; j++) {
                if (vertex[j] != v) continue;
                const int32_t q = pos[j];
                if (P.trim_pos2 > q) { r.startpos2 = P.trim_pos2 - q; r.index2 = 0; }
                else { r.startpos2 = 0; r.index2 = q - P.trim_pos2; }
            }
        }
        info[k] = r;
    }
}
}  // namespace

extern "C" int hc_subread_info(const hc_subread_problem* problems, uint64_t n_problems, const int32_t* pos, const uint32_t* vertex,
                               uint64_t n_entries, hc_fno_subread* info, uint8_t* first, int device) {
    if ((n_problems && !problems) || (n_entries && (!pos || !vertex || !info || !first))) { hc_set_last_error("hc_subread_info: NULL argument"); return HC_ERR_ARG; }
    if (n_entries == 0) return HC_OK;
    if (n_problems >= 0xffffffffull) { hc_set_last_error("hc_subread_info: too many problems"); return HC_ERR_ARG; }
    // which problem an entry belongs to (list 1) -- also the range check: lists inside [0, n_entries), list 1 ranges disjoint
    std::string err;
    uint32_t* h_ep = (uint32_t*)malloc(n_entries * sizeof(uint32_t));
    if (!h_ep) { hc_set_last_error("hc_subread_info: out of memory"); return HC_ERR_NOMEM; }
    memset(h_ep, 0xff, n_entries * sizeof(uint32_t));
    for (u64 p = 0; p < n_problems && err.empty(); p++) {
        const hc_subread_problem& P = problems[p];
        if (P.begin1 > P.end1 || P.end1 > n_entries || P.begin2 > P.end2 || P.end2 > n_entries) { err = "hc_subread_info: problem " + std::to_string(p) + ": list out of range"; break; }
        if (P.trim_pos2 >= 0 && P.end2 - P.begin2 != P.end1 - P.begin1) { err = "hc_subread_info: problem " + std::to_string(p) + ": the two lists of a paired-end super-read differ in length (the reference asserts, :575)"; break; }
        for (u64 k = P.begin1; k < P.end1; k++) {
            if (h_ep[k] != 0xffffffffu) { err = "hc_subread_info: problem " + std::to_string(p) + ": list 1 overlaps another problem's"; break; }
            h_ep[k] = (uint32_t)p;
        }
    }
    int rc = HC_OK;
    const char* who = "hc_subread_info";
    ScratchBuf<hc_subread_problem> d_prob;
    ScratchBuf<uint32_t> d_ep, d_v;
    ScratchBuf<int32_t> d_pos;
    ScratchBuf<hc_fno_subread> d_info;
    ScratchBuf<uint8_t> d_first;
    if (!err.empty()) { hc_set_last_error(err.c_str()); free(h_ep); return HC_ERR_ARG; }
    HC_CU(cudaSetDevice(device));
    HC_CU(d_prob.alloc(n_problems ? n_problems : 1)); HC_CU(d_ep.alloc(n_entries));
    HC_CU(d_v.alloc(n_entries)); HC_CU(d_pos.alloc(n_entries));
    HC_CU(d_info.alloc(n_entries)); HC_CU(d_first.alloc(n_entries));
    HC_CU(hc_copy_h2d(d_prob, problems, n_problems * sizeof(hc_subread_problem)));
    HC_CU(hc_copy_h2d(d_ep, h_ep, n_entries * sizeof(uint32_t)));
    HC_CU(hc_copy_h2d(d_v, vertex, n_entries * sizeof(uint32_t)));
    HC_CU(hc_copy_h2d(d_pos, pos, n_entries * sizeof(int32_t)));
    subread_info_kernel<<<grid_for(n_entries, 256), 256>>>(d_prob, d_ep, n_entries, d_pos, d_v, d_info, d_first);
    HC_CU(cudaGetLastError());
    HC_CU(hc_copy_d2h(info, d_info, n_entries * sizeof(hc_fno_subread)));
    HC_CU(hc_copy_d2h(first, d_first, n_entries));
done:
    free(h_ep);
    return rc;
}
