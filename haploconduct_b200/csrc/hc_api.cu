// hc_api.cu -- the C ABI of include/hc_b200.h: read-store packing / replication, workspace
// management and the batch entry points.  Host code here is plumbing; the arithmetic lives in
// hc_kernels.cu (device) and hc_tables.cpp (score tables, host libm).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <memory>
#include <mutex>
#include <new>
#include <algorithm>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_layout.h"
#include "hc_tables.h"
#include "hc_stage.h"
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include "hc_kernels.cuh"
#include "hc_pack.cuh"
#include "hc_consensus.cuh"
#include "hc_cons_final.h"
#include "hc_ingest.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (call);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            return fail(HC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));               \
        }                                                                                                \
    } while (0)

struct DevCtx {
    int device = -1;
    int sm_count = 0;
    size_t smem_per_sm = 0;
    // store planes
    uint8_t* pk = nullptr;       // packed layout (code | base << 6), or
    uint8_t* qual = nullptr;     // planar layout: quality codes, 2-bit bases, N mask
    uint32_t* base2 = nullptr;
    uint32_t* nmask = nullptr;
    hc_rdesc* rdesc = nullptr;
    // tables
    uint32_t* fx_table = nullptr;
    double* dbl_table = nullptr;
    bool tables_valid = false;
    double tables_mismatch = 0.0;
    bool has_void = false;
    bool void_exact = false;
    // workspace (grown on demand)
    uint64_t ws_cap = 0;
    hc_tmp32* tmp = nullptr;
    uint8_t* cls = nullptr;
    uint32_t* flagged = nullptr;
    uint32_t* blockcounts = nullptr;
    unsigned long long* counters = nullptr;
    // host-buffer path: two chunk slots (copy-in of chunk k+1 overlaps the kernels of chunk k), device-side
    // accumulation of the ordered outputs, running totals on the device
    uint64_t slot_cap = 0;                 // candidates per slot
    void* d_cand[2] = {nullptr, nullptr};
    uint64_t pc_cap = 0;
    hc_result* d_per_cand[2] = {nullptr, nullptr};
    // whole-shard mode: the shard's records in one device buffer, copied in step by step ahead of the kernels
    size_t whole_cap = 0;                  // bytes
    unsigned char* d_whole = nullptr;
    std::vector<cudaEvent_t> ev_step;      // one "copied in" event per pipeline step
    uint64_t runs_all_cap = 0;             // 32-bit words: every step's [anchors][starts] one after the other
    uint32_t* d_runs_all = nullptr;
    uint32_t* h_runs_all = nullptr;        // pinned
    // run-encoded candidates (hc_score_batch_runs): per slot the chunk's run anchors + relative run starts
    // ([anchor x cap][start x (cap + 1)], host copy pinned) and the tile -> run table
    uint64_t runs_cap = 0, tile_cap = 0;
    uint32_t* d_runs[2] = {nullptr, nullptr};
    uint32_t* h_runs[2] = {nullptr, nullptr};
    uint32_t* d_tile_run[2] = {nullptr, nullptr};
    uint64_t acc_e_cap = 0, acc_n_cap = 0;
    hc_edge* d_acc_edges = nullptr;
    uint64_t* d_acc_nonedge = nullptr;
    uint64_t acc_b_cap = 0;                // small outputs: one bit per candidate of the shard (32-bit words)
    uint32_t* d_acc_bits = nullptr;
    unsigned long long* d_run = nullptr;   // {edges, non-edges} emitted so far in this call
    // hc_ingest_score_overlaps: per slot the kept outputs of a piece ([cand][line][edge records][edge_kept][class], kept_cap each)
    uint64_t kept_cap = 0;
    unsigned char* d_kept[2] = {nullptr, nullptr};
    unsigned long long* h_cnt = nullptr;   // pinned: [2][HC_CNT_N] counter snapshots per slot
    uint64_t* d_counts = nullptr;
    cudaStream_t stream = nullptr, s_copy = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // recorded at the end of every enqueue_batch: the next call waits for it (on its own stream, or on the host before it
    // frees the workspace or rewrites the tables), so calls on different streams do not share the workspace at once
    cudaEvent_t ws_event = nullptr;
    hc_launch_cfg cfg{};
};

}  // namespace

void hc_set_last_error(const char* msg) { g_err = msg ? msg : ""; }   // used by hc_fno.cu

struct hc_store {
    uint64_t n_reads = 0, n_single = 0;
    uint64_t total_positions = 0;
    int ncodes = 0;
    bool packed = false;          // one byte per position (<= 63 quality codes); else three planes
    int code_to_q[HC_MAX_CODES + 1];
    int q_to_code[256];
    std::vector<DevCtx> devs;
    std::vector<uint64_t> ids;        // hc_store_create_fastq only: read ids and mate lengths parsed from the files
    std::vector<uint32_t> lens;
    hc_tables tables;
    bool tables_built = false;
    double tables_mismatch = 0.0;
    std::mutex mu;
};

namespace {

void free_ctx(DevCtx& d) {
    if (d.device < 0) return;
    cudaSetDevice(d.device);
    cudaFree(d.pk); cudaFree(d.qual); cudaFree(d.base2); cudaFree(d.nmask); cudaFree(d.rdesc);
    cudaFree(d.fx_table); cudaFree(d.dbl_table);
    cudaFree(d.tmp); cudaFree(d.cls); cudaFree(d.flagged); cudaFree(d.blockcounts); cudaFree(d.counters);
    for (int k = 0; k < 2; k++) {
        cudaFree(d.d_cand[k]); cudaFree(d.d_per_cand[k]);
        cudaFree(d.d_runs[k]); cudaFree(d.d_tile_run[k]);
        if (d.h_runs[k]) cudaFreeHost(d.h_runs[k]);
        if (d.ev_in[k]) cudaEventDestroy(d.ev_in[k]);
        if (d.ev_done[k]) cudaEventDestroy(d.ev_done[k]);
        if (d.ev_out[k]) cudaEventDestroy(d.ev_out[k]);
    }
    cudaFree(d.d_acc_edges); cudaFree(d.d_acc_nonedge); cudaFree(d.d_acc_bits); cudaFree(d.d_run); cudaFree(d.d_counts);
    cudaFree(d.d_whole); cudaFree(d.d_runs_all);
    cudaFree(d.d_kept[0]); cudaFree(d.d_kept[1]);
    if (d.h_runs_all) cudaFreeHost(d.h_runs_all);
    for (cudaEvent_t e : d.ev_step) cudaEventDestroy(e);
    if (d.h_cnt) cudaFreeHost(d.h_cnt);
    for (int k = 0; k < 6; k++) if (d.ev[k]) cudaEventDestroy(d.ev[k]);
    if (d.ws_event) cudaEventDestroy(d.ws_event);
    if (d.stream) cudaStreamDestroy(d.stream);
    if (d.s_copy) cudaStreamDestroy(d.s_copy);
    if (d.s_out) cudaStreamDestroy(d.s_out);
    d = DevCtx();
}


int ensure_tables(hc_store* s, DevCtx& d, double mismatch, cudaStream_t st) {
    {
        std::lock_guard<std::mutex> lk(s->mu);
        if (!s->tables_built || s->tables_mismatch != mismatch) {
            hc_build_tables(s->code_to_q, s->ncodes, mismatch, &s->tables);
            s->tables_built = true;
            s->tables_mismatch = mismatch;
            for (auto& dd : s->devs) dd.tables_valid = false;
        }
    }
    if (d.tables_valid && d.tables_mismatch == mismatch) return HC_OK;
    // tables change only when ps.mismatch changes (it never does in the drivers): wait on the host for every earlier call,
    // whatever its stream, then upload on this call's stream, ahead of its kernels (a pageable source is staged before
    // the copy returns, so the host tables may be rebuilt afterwards)
    CU(cudaEventSynchronize(d.ws_event));
    CU(cudaStreamSynchronize(st));
    const std::vector<uint32_t>& fx = s->packed ? s->tables.fx_packed : s->tables.fx;
    if (!d.fx_table) CU(cudaMalloc(&d.fx_table, fx.size() * sizeof(uint32_t)));
    if (!d.dbl_table) CU(cudaMalloc(&d.dbl_table, s->tables.dbl.size() * sizeof(double)));
    CU(cudaMemcpyAsync(d.fx_table, fx.data(), fx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d.dbl_table, s->tables.dbl.data(), s->tables.dbl.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    d.tables_valid = true;
    d.tables_mismatch = mismatch;
    d.has_void = s->tables.has_void;
    d.void_exact = s->tables.void_asymmetric;
    return HC_OK;
}

int ensure_workspace(DevCtx& d, uint64_t n) {
    if (n <= d.ws_cap && d.counters) return HC_OK;
    uint64_t cap = std::max<uint64_t>(n, 1024);
    CU(cudaEventSynchronize(d.ws_event));   // an earlier call on another stream may still be using the buffers
    cudaFree(d.tmp); cudaFree(d.cls); cudaFree(d.flagged); cudaFree(d.blockcounts);
    d.tmp = nullptr; d.cls = nullptr; d.flagged = nullptr; d.blockcounts = nullptr;
    d.ws_cap = 0;
    CU(cudaMalloc(&d.tmp, cap * sizeof(hc_tmp32)));
    CU(cudaMalloc(&d.cls, cap));
    CU(cudaMalloc(&d.flagged, cap * sizeof(uint32_t)));
    const uint64_t nb = hc_compact_blocks(cap) + 1;
    CU(cudaMalloc(&d.blockcounts, nb * 2 * sizeof(uint32_t) + 8 + nb * 2 * sizeof(uint64_t)));
    if (!d.counters) CU(cudaMalloc(&d.counters, HC_CNT_N * sizeof(unsigned long long)));
    d.ws_cap = cap;
    return HC_OK;
}

DevCtx* find_ctx(hc_store* s, int device) {
    for (auto& d : s->devs) if (d.device == device) return &d;
    return nullptr;
}

struct RunDev {                 // device-side run arrays of one batch of hc_candidate_entry records
    const uint32_t* anchor;     // [n_runs]
    const uint32_t* start;      // [n_runs + 1], relative to the batch
    uint32_t n_runs;
    uint32_t* tile_run;         // [ceil(n / 32)] scratch
};

// Enqueue the whole scoring pipeline for one shard on (d, st).
int enqueue_batch(hc_store* s, DevCtx& d, cudaStream_t st, const hc_params* p, const void* d_cand, int compact, uint64_t n,
                  hc_result* d_per_cand, hc_edge* d_edges, uint64_t edges_cap, uint64_t* d_nonedge, uint64_t nonedge_cap,
                  uint64_t* d_counts, uint64_t cand_offset, unsigned long long* d_run, cudaEvent_t k0, cudaEvent_t k1,
                  uint32_t* launches, const RunDev* runs = nullptr, int small_out = 0, uint32_t* d_bits = nullptr,
                  const hc_kept_dev* kept = nullptr) {
    if (n > 0xffffffffull) return fail(HC_ERR_ARG, "more than 2^32-1 candidates in one device batch");
    if (compact >= 3 && !runs) return fail(HC_ERR_ARG, "run-encoded candidates without run arrays");
    CU(cudaStreamWaitEvent(st, d.ws_event, 0));   // the previous call's use of the workspace, whatever its stream
    int rc = ensure_tables(s, d, p->mismatch, st);
    if (rc != HC_OK) return rc;
    rc = ensure_workspace(d, n);
    if (rc != HC_OK) return rc;
    int mono = 1;
    hc_kparams P;
    memset(&P, 0, sizeof(P));
    P.qual = d.qual; P.base2 = d.base2; P.nmask = d.nmask; P.rdesc = d.rdesc;
    P.pk = d.pk; P.packed = s->packed ? 1u : 0u;
    P.n_reads = (uint32_t)s->n_reads; P.n_single = (uint32_t)s->n_single;
    P.fx_table = d.fx_table; P.dbl_table = d.dbl_table; P.ncodes = (uint32_t)s->ncodes; P.has_void = d.has_void ? 1u : 0u;
    P.cand = d_cand; P.cand_compact = (uint32_t)compact; P.run = d_run; P.n = n; P.tmp = d.tmp; P.cls = d.cls; P.per_cand = d_per_cand; P.flagged = d.flagged;
    P.counters = d.counters;
    if (runs) { P.run_anchor = runs->anchor; P.run_start = runs->start; P.tile_run = runs->tile_run; }
    P.t_edge = hc_tables_exp_threshold(p->edge_threshold, &mono);
    if (!mono) return fail(HC_ERR_ARG, "host exp() is not monotone around edge_threshold");
    P.t_ov = hc_tables_exp_threshold(p->ov_threshold, &mono);
    if (!mono) return fail(HC_ERR_ARG, "host exp() is not monotone around ov_threshold");
    // fixed-point decision constants: mean = -S/(2^22*tl);  mean - margin >= t  <=>  S <= -(t+margin)*2^22 * tl
    P.ce_up = -(P.t_edge + HC_FX_MARGIN) * HC_FX_SCALE;
    P.ce_dn = -(P.t_edge - HC_FX_MARGIN) * HC_FX_SCALE;
    P.co_up = -(P.t_ov + HC_FX_MARGIN) * HC_FX_SCALE;
    P.co_dn = -(P.t_ov - HC_FX_MARGIN) * HC_FX_SCALE;
    P.never_edge = P.t_edge > 0.0;   // a mean log-likelihood is <= 0
    P.never_ov = P.t_ov > 0.0;
    P.merge_contigs = p->merge_contigs;
    P.merge_contigs_sign = p->merge_contigs > 0.0 ? 1 : (p->merge_contigs < 0.0 ? -1 : 0);
    P.min_read_len = p->min_read_len;
    P.zero_above_edge = 0.0 > p->edge_threshold;
    P.zero_above_ov = 0.0 > p->ov_threshold;
    P.exact_edges = (p->flags & HC_FLAG_EXACT_EDGE_SCORES) ? 1u : 0u;
    P.void_exact = d.void_exact ? 1u : 0u;
    CU(cudaMemsetAsync(d.counters, 0, HC_CNT_N * sizeof(unsigned long long), st));
    if (k0) CU(cudaEventRecord(k0, st));
    uint32_t nl = 0;
    if (n > 0) {
        hc_launch_cfg cfg = d.cfg;
        const uint64_t ntiles = (n + 31) / 32;
        const uint64_t warps_per_block = cfg.threads / 32;
        const uint64_t need_blocks = (ntiles + warps_per_block - 1) / warps_per_block;
        if ((uint64_t)cfg.blocks > need_blocks) cfg.blocks = (int)need_blocks;
        if (runs) { CU(hc_launch_tile_runs(runs->start, runs->n_runs, runs->tile_run, st)); nl += 1; }
        if (k0) CU(cudaEventRecord(d.ev[4], st));
        CU(hc_launch_score(P, cfg, st));
        if (k0) CU(cudaEventRecord(d.ev[5], st));
        CU(hc_launch_exact(P, st));
        nl += 2;
    }
    CU(hc_launch_compact(P, d_edges, edges_cap, d_nonedge, nonedge_cap, d.blockcounts, cand_offset, d_run, st, small_out, d_bits, kept));
    nl += (n > 0 ? 4 : 1) + (d_run ? 1 : 0) + ((n > 0 && small_out && d_bits) ? 1 : 0);   // count, scan, scatter, emit_edges (+ advance, + bit map)
    if (k1) CU(cudaEventRecord(k1, st));
    if (d_counts) {   // {n_edges, n_nonedges, n_exact} are contiguous in the counter block; [3] = invalid candidates
        CU(cudaMemcpyAsync(d_counts, d.counters + HC_CNT_EDGES, 3 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(d_counts + 3, d.counters + HC_CNT_ERRORS, sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    }
    CU(cudaEventRecord(d.ws_event, st));
    if (launches) *launches = nl;
    return HC_OK;
}

int add_stats(DevCtx& d, const unsigned long long* h, uint64_t n, hc_batch_stats* stats, cudaEvent_t k0, cudaEvent_t k1);

int read_stats(DevCtx& d, uint64_t n, hc_batch_stats* stats, cudaEvent_t k0, cudaEvent_t k1) {
    unsigned long long h[HC_CNT_N];
    CU(cudaMemcpy(h, d.counters, sizeof(h), cudaMemcpyDeviceToHost));
    return add_stats(d, h, n, stats, k0, k1);
}

int add_stats(DevCtx& d, const unsigned long long* h, uint64_t n, hc_batch_stats* stats, cudaEvent_t k0, cudaEvent_t k1) {
    if (stats) {
        stats->n_candidates += n;
        stats->n_edges += h[HC_CNT_EDGES];
        stats->n_nonedges += h[HC_CNT_NONEDGES];
        stats->n_exact += h[HC_CNT_EXACT];
        stats->n_windows += h[HC_CNT_WINDOWS];
        stats->n_positions += h[HC_CNT_POSITIONS];
        stats->algorithmic_bytes += h[HC_CNT_ALGBYTES];
        float ms = 0;
        if (k0 && k1 && cudaEventElapsedTime(&ms, k0, k1) == cudaSuccess) stats->kernel_ms = std::max(stats->kernel_ms, ms);
        if (k0 && n > 0 && cudaEventElapsedTime(&ms, d.ev[4], d.ev[5]) == cudaSuccess)
            stats->score_kernel_ms = std::max(stats->score_kernel_ms, ms);
    }
    if (h[HC_CNT_ERRORS]) {
        return fail(HC_ERR_ARG, std::to_string(h[HC_CNT_ERRORS]) +
                                    " candidate(s) with an invalid read index, a self overlap, or ORD not in {1,2} "
                                    "for a paired-paired overlap (the reference asserts, src/EdgeCalculator.cpp:184,369)");
    }
    return HC_OK;
}

}  // namespace

extern "C" {

const char* hc_last_error(void) { return g_err.c_str(); }
const char* hc_version(void) { return "haploconduct_b200 0.1 (sm_100a)"; }

int hc_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int hc_warm_up(int device) {
    if (hc_device_count() == 0) return fail(HC_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)");
    CU(cudaSetDevice(device));
    CU(cudaFree(nullptr));                 // creates the context
    void* p = nullptr;                      // first use of the pinned / device allocators
    CU(cudaMallocHost(&p, 1 << 20));
    CU(cudaFreeHost(p));
    return HC_OK;
}

double hc_phred_to_prob(int phred) { return hc_tables_phred_to_prob(phred); }

void hc_edge_extra_pos(uint32_t pos1, uint32_t pos2, char ord, uint32_t len1a, uint32_t len1b, uint32_t len2a, uint32_t len2b,
                       int32_t* pos3, int32_t* pos4) {
    const int p1 = len1b != 0, p2 = len2b != 0;     // src/EdgeCalculator.cpp:222, :262-263, :300-301, :361-372
    if (!p1 && !p2) { *pos3 = (int32_t)(len1a - pos1 - len2a); *pos4 = 0; }
    else if (!p1) { *pos3 = (int32_t)(len1a - pos2 - len2b); *pos4 = (int32_t)(len1a - pos1 - len2a); }
    else if (!p2) { *pos3 = (int32_t)(len1b + pos2 - len2a); *pos4 = (int32_t)(len2a + pos1 - len1a); }
    else {
        *pos3 = ord == '1' ? (int32_t)(len1b - pos2 - len2b) : (int32_t)(len1b + pos2 - len2b);
        *pos4 = (int32_t)(len1a - pos1 - len2a);
    }
}
double hc_exp_threshold(double threshold) { return hc_tables_exp_threshold(threshold, nullptr); }

uint64_t hc_store_n_reads(const hc_store* s) { return s ? s->n_reads : 0; }
uint64_t hc_store_n_single(const hc_store* s) { return s ? s->n_single : 0; }
int hc_store_n_devices(const hc_store* s) { return s ? (int)s->devs.size() : 0; }
int hc_store_quality_alphabet(const hc_store* s) { return s ? s->ncodes : 0; }
uint64_t hc_store_device_bytes(const hc_store* s) {
    if (!s) return 0;
    const uint64_t planes = s->packed ? s->total_positions : s->total_positions + s->total_positions / 4 + s->total_positions / 8;
    return planes + s->n_reads * sizeof(hc_rdesc);
}

void hc_store_destroy(hc_store* s) {
    if (!s) return;
    for (auto& d : s->devs) free_ctx(d);
    delete s;
}

namespace {

// Slot layout of reads with the given mate lengths: forward strand, then reverse complement, each in a
// zero-padded slot of hc_slot_size(len) positions.  0 ok, 2 empty first mate, 3 too large.
int layout_slots(const uint32_t* len2, uint64_t n_reads, std::vector<hc_rdesc>& rd, uint64_t* total) {
    rd.resize(n_reads);
    uint64_t pos = 0;   // in positions
    int bad = 0;
    for (uint64_t r = 0; r < n_reads; r++) {
        if (len2[2 * r] == 0) bad = 2;                      // empty sequence (src/FastqStorage.cpp:143-146)
        for (int m = 0; m < 2; m++) {
            const uint32_t len = len2[2 * r + m];
            if (len > HC_LEN_MAX) bad = 3;
            rd[r].slot16[m] = (uint32_t)(pos >> 4);
            rd[r].len[m] = len;
            if (len) pos += 2ull * hc_slot_size(len);
            if ((pos >> 4) > 0xffffffffull) bad = 3;
        }
    }
    *total = (pos + 63) & ~63ull;
    return bad;
}

cudaError_t init_ctx(hc_store* s, DevCtx& d, int device, bool* not_sm100) {
    d.device = device;
    cudaError_t e = cudaSetDevice(d.device);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, d.device);
    if (e == cudaSuccess && prop.major < 10) { *not_sm100 = true; return cudaErrorInvalidDevice; }
    if (e == cudaSuccess) {
        d.sm_count = prop.multiProcessorCount;
        d.smem_per_sm = prop.sharedMemPerMultiprocessor;
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.s_copy, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.s_out, cudaStreamNonBlocking);
    for (int j = 0; j < 2 && e == cudaSuccess; j++) {
        e = cudaEventCreateWithFlags(&d.ev_in[j], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.ev_done[j], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.ev_out[j], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaMalloc(&d.d_run, 2 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMallocHost(&d.h_cnt, 2 * HC_CNT_N * sizeof(unsigned long long));
    for (int j = 0; j < 6 && e == cudaSuccess; j++) e = cudaEventCreate(&d.ev[j]);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.ws_event, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&d.rdesc, s->n_reads * sizeof(hc_rdesc));
    if (e == cudaSuccess) e = cudaMalloc(&d.d_counts, 4 * sizeof(uint64_t));
    return e;
}

cudaError_t alloc_planes(hc_store* s, DevCtx& d, cudaStream_t st) {
    const uint64_t total = s->total_positions;
    uint8_t** bytes = s->packed ? &d.pk : &d.qual;   // one byte per position in either layout
    cudaError_t e = cudaMalloc(bytes, total + 64);
    if (e == cudaSuccess) e = cudaMemsetAsync(*bytes, 0, total + 64, st);
    if (e == cudaSuccess && !s->packed) e = cudaMalloc(&d.base2, (total / 16 + 16) * 4);
    if (e == cudaSuccess && !s->packed) e = cudaMalloc(&d.nmask, (total / 32 + 16) * 4);
    if (e == cudaSuccess && !s->packed) e = cudaMemsetAsync(d.base2, 0, (total / 16 + 16) * 4, st);
    if (e == cudaSuccess && !s->packed) e = cudaMemsetAsync(d.nmask, 0, (total / 32 + 16) * 4, st);
    return e;
}

// Validate, find the quality alphabet, pack both strands on the first device (text and source offsets are already
// there), then copy the planes to the other devices.  Returns HC_OK or an error code with the message set.
int build_store(hc_store* s, std::vector<hc_rdesc>& rd, const uint8_t* d_text, const hc_pack_src* d_src, uint64_t n_upper,
                int first_device, int n_devices) {
    const uint64_t n_reads = s->n_reads;
    s->devs.resize(n_devices);
    for (int k = 0; k < n_devices; k++) {
        bool not100 = false;
        const cudaError_t e = init_ctx(s, s->devs[k], first_device + k, &not100);
        if (not100) return fail(HC_ERR_CUDA, "device is not sm_100 class (this library ships sm_100a code only)");
        if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA, std::string("hc_store_create: ") + cudaGetErrorString(e));
    }
    DevCtx& d0 = s->devs[0];
    CU(cudaSetDevice(d0.device));
    unsigned long long* d_flags = nullptr;    // [0..127] occurrences of every quality character, [128] error bits
    uint8_t* d_lut = nullptr;
    unsigned long long h_flags[129];
    uint8_t lut[256];
    cudaError_t e = cudaMalloc(&d_flags, sizeof(h_flags));
    if (e == cudaSuccess) e = cudaMalloc(&d_lut, 256);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_flags, 0, sizeof(h_flags), d0.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d0.rdesc, rd.data(), n_reads * sizeof(hc_rdesc), cudaMemcpyHostToDevice, d0.stream);
    if (e == cudaSuccess)
        e = hc_pack_validate_launch(d_text, d_src, d0.rdesc, n_reads, n_upper, d_flags, reinterpret_cast<uint32_t*>(d_flags + 128), d0.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h_flags, d_flags, sizeof(h_flags), cudaMemcpyDeviceToHost, d0.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d0.stream);
    int rc = HC_OK;
    if (e == cudaSuccess && h_flags[128]) {
        rc = fail(HC_ERR_INPUT, (h_flags[128] & 1u)
                                    ? "invalid nucleotide (only upper-case A,C,G,T,N are accepted; the reference asserts in "
                                      "EdgeCalculator::score, src/EdgeCalculator.cpp:29-30)"
                                    : "quality character outside '!'..'~' (Phred 0..93; src/EdgeCalculator.cpp:61,93-98)");
    }
    if (e == cudaSuccess && rc == HC_OK) {
        memset(s->q_to_code, 0, sizeof(s->q_to_code));
        memset(lut, 0, sizeof(lut));
        s->ncodes = 0;
        s->code_to_q[0] = -1;
        // quality codes ranked by frequency, the most frequent value first (ties: the smaller Phred value); this order
        // decides which code each Phred value gets, and so the bytes of the stored planes
        std::vector<int> present;
        for (int c = 33; c <= 33 + 93; c++) if (h_flags[c]) present.push_back(c);
        std::stable_sort(present.begin(), present.end(), [&](int a, int b) { return h_flags[a] > h_flags[b]; });
        for (int c : present) {
            s->ncodes++;
            s->code_to_q[s->ncodes] = c - 33;
            s->q_to_code[c] = s->ncodes;
            lut[c] = (uint8_t)s->ncodes;
        }
        const char* layout = getenv("HC_STORE_LAYOUT");   // "planar" forces the three-plane layout (tests)
        s->packed = s->ncodes <= HC_PACKED_MAX_CODES && !(layout && strcmp(layout, "planar") == 0);
        e = cudaMemcpyAsync(d_lut, lut, 256, cudaMemcpyHostToDevice, d0.stream);
        if (e == cudaSuccess) e = alloc_planes(s, d0, d0.stream);
        if (e == cudaSuccess)
            e = hc_pack_write_launch(d_text, d_src, d0.rdesc, n_reads, n_upper, d_lut, s->packed, s->packed ? d0.pk : d0.qual, d0.base2,
                                     d0.nmask, d0.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(d0.stream);
    }
    cudaFree(d_flags);
    cudaFree(d_lut);
    if (rc != HC_OK) return rc;
    const uint64_t total = s->total_positions;
    for (int k = 0; k < n_devices && e == cudaSuccess; k++) {
        DevCtx& d = s->devs[k];
        e = cudaSetDevice(d.device);
        if (e == cudaSuccess) e = hc_score_occupancy((uint32_t)s->ncodes, d.sm_count, d.smem_per_sm, &d.cfg);
        if (k == 0 || e != cudaSuccess) continue;
        e = alloc_planes(s, d, d.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
        if (e == cudaSuccess) e = cudaMemcpyPeer(s->packed ? d.pk : d.qual, d.device, s->packed ? d0.pk : d0.qual, d0.device, total);
        if (e == cudaSuccess && !s->packed) e = cudaMemcpyPeer(d.base2, d.device, d0.base2, d0.device, total / 16 * 4);
        if (e == cudaSuccess && !s->packed) e = cudaMemcpyPeer(d.nmask, d.device, d0.nmask, d0.device, total / 32 * 4);
        if (e == cudaSuccess) e = cudaMemcpyPeer(d.rdesc, d.device, d0.rdesc, d0.device, n_reads * sizeof(hc_rdesc));
    }
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA, std::string("hc_store_create: ") + cudaGetErrorString(e));
    return HC_OK;
}

bool check_devices(int first_device, int n_devices) {
    if (n_devices < 1 || first_device < 0) { fail(HC_ERR_ARG, "hc_store_create: bad argument"); return false; }
    const int ndev = hc_device_count();
    if (ndev == 0) { fail(HC_ERR_CUDA, "no CUDA device available (this library has no CPU fallback)"); return false; }
    if (first_device + n_devices > ndev) { fail(HC_ERR_ARG, "hc_store_create: device range exceeds the devices present"); return false; }
    return true;
}

}  // namespace

hc_store* hc_store_create(const hc_read_desc* reads, uint64_t n_reads, uint64_t n_single, const char* bases,
                          const char* quals, int first_device, int n_devices) {
    if (!reads || !bases || !quals || n_reads == 0 || n_single > n_reads) {
        fail(HC_ERR_ARG, "hc_store_create: bad argument");
        return nullptr;
    }
    if (n_reads >= 0xffffffffull) { fail(HC_ERR_ARG, "hc_store_create: too many reads"); return nullptr; }
    if (!check_devices(first_device, n_devices)) return nullptr;

    hc_store* s = new hc_store();
    s->n_reads = n_reads;
    s->n_single = n_single;
    // ---- host: slot layout and where every mate's bytes lie in the two blobs
    std::vector<uint32_t> len2(2 * n_reads);
    std::vector<hc_pack_src> src(2 * n_reads);
    uint64_t blob = 0;
    int bad = 0;
    for (uint64_t r = 0; r < n_reads; r++) {
        const int paired = reads[r].seq_len[1] > 0;
        if ((r < n_single) == (paired != 0)) bad = 1;       // singles first, then pairs (src/FastqStorage.h:88-97)
        for (int m = 0; m < 2; m++) {
            len2[2 * r + m] = reads[r].seq_len[m];
            if (reads[r].seq_len[m]) blob = std::max<uint64_t>(blob, reads[r].seq_off[m] + reads[r].seq_len[m]);
        }
    }
    const uint64_t qbase = (blob + 15) & ~15ull;
    for (uint64_t r = 0; r < n_reads; r++)
        for (int m = 0; m < 2; m++) { src[2 * r + m].boff = reads[r].seq_off[m]; src[2 * r + m].qoff = qbase + reads[r].seq_off[m]; }
    std::vector<hc_rdesc> rd;
    if (!bad) bad = layout_slots(len2.data(), n_reads, rd, &s->total_positions);
    if (bad) {
        fail(bad == 1 ? HC_ERR_ARG : HC_ERR_INPUT,
             bad == 1 ? "hc_store_create: reads must be ordered singles first, then pairs"
                      : (bad == 2 ? "hc_store_create: read with an empty sequence" : "hc_store_create: store too large"));
        delete s;
        return nullptr;
    }
    // ---- device: raw bytes in, validate + pack there (no packed copy is ever built on the host)
    uint8_t* d_text = nullptr;
    hc_pack_src* d_src = nullptr;
    cudaError_t e = cudaSetDevice(first_device);
    if (e == cudaSuccess) e = cudaMalloc(&d_text, 2 * qbase + 16);
    if (e == cudaSuccess) e = cudaMalloc(&d_src, 2 * n_reads * sizeof(hc_pack_src));
    if (e == cudaSuccess) e = hc_copy_h2d(d_text, bases, blob);
    if (e == cudaSuccess) e = hc_copy_h2d(d_text + qbase, quals, blob);
    if (e == cudaSuccess) e = hc_copy_h2d(d_src, src.data(), 2 * n_reads * sizeof(hc_pack_src));
    int rc = HC_OK;
    if (e != cudaSuccess) rc = fail(e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA, std::string("hc_store_create: ") + cudaGetErrorString(e));
    else rc = build_store(s, rd, d_text, d_src, 0, first_device, n_devices);
    cudaSetDevice(first_device);
    cudaFree(d_text);
    cudaFree(d_src);
    if (rc != HC_OK) { const std::string keep = g_err; hc_store_destroy(s); g_err = keep; return nullptr; }
    return s;
}

// FastqStorage::FastqStorage (src/FastqStorage.h:58-98) from the text of the FASTQ files: the files go to the first
// device as they are; line index, record scan (ids, lengths), validation and packing all run there.
// file[k] != NULL: the text is in host memory; else fd[k] >= 0: it is streamed from the file (bytes[k] = its size)
static hc_store* store_from_fastq(const char* const file[3], const int fd[3], uint64_t bytes[3], uint64_t max_reads, int first_device,
                                  int n_devices) {
    if (!check_devices(first_device, n_devices)) return nullptr;
    uint64_t off[4] = {0, 0, 0, 0};
    for (int k = 0; k < 3; k++) off[k + 1] = off[k] + ((bytes[k] + 15) & ~15ull);
    hc_store* s = new hc_store();
    char* d_text = nullptr;
    unsigned long long* d_ls[3] = {nullptr, nullptr, nullptr};
    unsigned long long *d_ids = nullptr, *d_first = nullptr;
    uint32_t* d_len = nullptr;
    hc_pack_src* d_src = nullptr;
    void* d_tok = nullptr;
    uint64_t nl[3] = {0, 0, 0}, nrec[3] = {0, 0, 0};
    unsigned long long first_err = ~0ull;
    uint64_t n_single = 0, n_pairs = 0, n_reads = 0;
    std::vector<hc_rdesc> rd;
    int rc = HC_OK;
    cudaError_t e = cudaSetDevice(first_device);
    if (e == cudaSuccess) e = cudaMalloc(&d_text, off[3] + 16);
    for (int k = 0; k < 3 && e == cudaSuccess; k++) {
        if (!bytes[k]) continue;
        if (file[k]) e = hc_copy_h2d(d_text + off[k], file[k], bytes[k]);
        else { size_t got = 0; e = hc_copy_file_h2d(d_text + off[k], fd[k], bytes[k], &got); bytes[k] = got; }   // a file that shrank: what is there
    }
    for (int k = 0; k < 3 && e == cudaSuccess; k++) e = hc_fastq_index(d_text + off[k], bytes[k], max_reads, &d_ls[k], &nl[k], &nrec[k], 0);
    if (e == cudaSuccess) {
        n_single = nrec[0];
        n_pairs = std::min(nrec[1], nrec[2]);               // the loop runs while both files have lines, :176
        n_reads = n_single + n_pairs;
        if (n_reads == 0) rc = fail(HC_ERR_INPUT, "hc_store_create_fastq: no complete FASTQ record");
        else if (n_reads >= 0xffffffffull) rc = fail(HC_ERR_ARG, "hc_store_create_fastq: too many reads");
    }
    if (e == cudaSuccess && rc == HC_OK) {
        e = cudaMalloc(&d_ids, n_reads * sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMalloc(&d_len, 2 * n_reads * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc(&d_src, 2 * n_reads * sizeof(hc_pack_src));
        if (e == cudaSuccess) e = cudaMalloc(&d_tok, n_reads * 16);
        if (e == cudaSuccess) e = cudaMalloc(&d_first, sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMemset(d_len, 0, 2 * n_reads * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemset(d_src, 0, 2 * n_reads * sizeof(hc_pack_src));
        if (e == cudaSuccess) e = cudaMemset(d_first, 0xff, sizeof(unsigned long long));
        if (e == cudaSuccess) e = hc_fastq_records_launch(d_text, off[0], bytes[0], d_ls[0], nl[0], n_single, d_ids, d_len, d_src, d_tok, 0, 0, d_first, 0);
        if (e == cudaSuccess) e = hc_fastq_records_launch(d_text, off[1], bytes[1], d_ls[1], nl[1], n_pairs, d_ids, d_len, d_src, d_tok, 0, n_single, d_first, 0);
        if (e == cudaSuccess) e = hc_fastq_records_launch(d_text, off[2], bytes[2], d_ls[2], nl[2], n_pairs, d_ids, d_len, d_src, d_tok, 1, n_single, d_first, 0);
        if (e == cudaSuccess) e = cudaMemcpy(&first_err, d_first, sizeof(first_err), cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess && rc == HC_OK && first_err != ~0ull) {
        // the reference exits at this record (src/FastqStorage.cpp:107-110,143-146,181-192,217-220)
        const bool pair = first_err >= n_single;
        rc = fail(HC_ERR_INPUT, std::string("FASTQ record ") + std::to_string(pair ? first_err - n_single : first_err) + " of the " +
                                    (pair ? "paired" : "single-end") + " input is not acceptable: header without '@', mate headers "
                                    "that differ, an empty sequence, or sequence and quality lines of different lengths");
    }
    if (e == cudaSuccess && rc == HC_OK) {
        s->n_reads = n_reads;
        s->n_single = n_single;
        s->ids.resize(n_reads);
        s->lens.resize(2 * n_reads);
        e = cudaMemcpy(s->ids.data(), d_ids, n_reads * sizeof(uint64_t), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(s->lens.data(), d_len, 2 * n_reads * sizeof(uint32_t), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) {
            const int bad = layout_slots(s->lens.data(), n_reads, rd, &s->total_positions);
            if (bad) rc = fail(HC_ERR_INPUT, bad == 2 ? "hc_store_create_fastq: read with an empty sequence" : "hc_store_create_fastq: store too large");
        }
    }
    if (e != cudaSuccess && rc == HC_OK) rc = fail(e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA, std::string("hc_store_create_fastq: ") + cudaGetErrorString(e));
    if (rc == HC_OK) rc = build_store(s, rd, (const uint8_t*)d_text, d_src, n_single, first_device, n_devices);   // singles are upper-cased, :123
    cudaSetDevice(first_device);
    cudaFree(d_text); cudaFree(d_ids); cudaFree(d_len); cudaFree(d_src); cudaFree(d_tok); cudaFree(d_first);
    for (int k = 0; k < 3; k++) cudaFree(d_ls[k]);
    if (rc != HC_OK) { const std::string keep = g_err; hc_store_destroy(s); g_err = keep; return nullptr; }
    return s;
}

hc_store* hc_store_create_fastq(const char* singles, uint64_t singles_bytes, const char* paired1, uint64_t paired1_bytes,
                                const char* paired2, uint64_t paired2_bytes, uint64_t max_reads, int first_device, int n_devices) {
    if ((singles_bytes && !singles) || (paired1_bytes && !paired1) || (paired2_bytes && !paired2)) {
        fail(HC_ERR_ARG, "hc_store_create_fastq: NULL argument");
        return nullptr;
    }
    const char* file[3] = {singles_bytes ? singles : nullptr, paired1_bytes ? paired1 : nullptr, paired2_bytes ? paired2 : nullptr};
    const int fd[3] = {-1, -1, -1};
    uint64_t bytes[3] = {singles_bytes, paired1_bytes, paired2_bytes};
    return store_from_fastq(file, fd, bytes, max_reads, first_device, n_devices);
}

// The same from the files themselves, streamed: pieces of a file are read into a ring of pinned buffers by several host
// threads and go to the device from there, so the host never holds a file (src/FastqStorage.cpp:42-57 reads every line
// into a vector of strings first: twice the file in host memory; SURVEY 8f rank 4).  A path that is NULL, "" or "None" is
// an absent file (src/FastqStorage.h:66-75); a file that cannot be opened is the reference's "Unable to open" exit.
hc_store* hc_store_create_fastq_files(const char* singles_path, const char* paired1_path, const char* paired2_path, uint64_t max_reads,
                                      int first_device, int n_devices) {
    const char* path[3] = {singles_path, paired1_path, paired2_path};
    const char* file[3] = {nullptr, nullptr, nullptr};
    int fd[3] = {-1, -1, -1};
    uint64_t bytes[3] = {0, 0, 0};
    hc_store* s = nullptr;
    bool ok = true;
    for (int k = 0; k < 3 && ok; k++) {
        if (!path[k] || !*path[k] || !strcmp(path[k], "None")) continue;
        fd[k] = open(path[k], O_RDONLY);
        struct stat st;
        if (fd[k] < 0 || fstat(fd[k], &st) != 0) { fail(HC_ERR_INPUT, std::string("Unable to open fastq file ") + path[k]); ok = false; break; }
        bytes[k] = st.st_size > 0 ? (uint64_t)st.st_size : 0;
    }
    if (ok) s = store_from_fastq(file, fd, bytes, max_reads, first_device, n_devices);
    for (int k = 0; k < 3; k++) if (fd[k] >= 0) close(fd[k]);
    return s;
}

int hc_store_read_ids(const hc_store* s, uint64_t* ids, uint32_t* mate_lengths) {
    if (!s) return fail(HC_ERR_ARG, "hc_store_read_ids: NULL store");
    if (s->ids.size() != s->n_reads) return fail(HC_ERR_ARG, "hc_store_read_ids: the store was not built from FASTQ text");
    if (ids) memcpy(ids, s->ids.data(), s->n_reads * sizeof(uint64_t));
    if (mate_lengths) memcpy(mate_lengths, s->lens.data(), 2 * s->n_reads * sizeof(uint32_t));
    return HC_OK;
}

namespace {
__global__ void cons_lens(const hc_rdesc* __restrict__ rd, const hc_cons_seq* __restrict__ seqs, uint64_t n, uint32_t* len) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) len[j] = rd[seqs[j].read].len[seqs[j].mate] & HC_LEN_MASK;
}
}  // namespace

int hc_consensus(hc_store* s, const hc_cons_problem* problems, uint64_t n_problems, const hc_cons_seq* seqs, uint64_t n_seqs,
                 uint32_t min_clique_size, double min_qual, char* cons_seq, char* cons_qual, uint64_t out_bytes,
                 hc_cons_result* results) {
    if (!s || (n_problems && (!problems || !results)) || (n_seqs && !seqs) || (out_bytes && (!cons_seq || !cons_qual)))
        return fail(HC_ERR_ARG, "hc_consensus: NULL argument");
    if (n_problems == 0) return HC_OK;
    // ---- validate, tile index
    std::vector<unsigned long long> tile_off(n_problems + 1, 0);
    for (uint64_t p = 0; p < n_problems; p++) {
        const hc_cons_problem& P = problems[p];
        if (P.seq_begin > P.seq_end || P.seq_end > n_seqs || P.total_len < 0 || P.out_offset + (uint64_t)P.total_len > out_bytes)
            return fail(HC_ERR_ARG, "hc_consensus: problem " + std::to_string(p) + " is out of range");
        for (uint64_t j = P.seq_begin; j < P.seq_end; j++) {
            if (seqs[j].read >= s->n_reads || seqs[j].mate > 1 || seqs[j].pos < 0 || (j > P.seq_begin && seqs[j].pos < seqs[j - 1].pos))
                return fail(HC_ERR_ARG, "hc_consensus: problem " + std::to_string(p) + ": bad sequence entry (read index, mate, or "
                                        "start columns not ascending)");
        }
        if (P.seq_end > P.seq_begin && seqs[P.seq_begin].pos != 0)
            return fail(HC_ERR_ARG, "hc_consensus: the first start column of a problem must be 0 (the reference asserts, :449)");
        tile_off[p + 1] = tile_off[p] + (unsigned long long)((P.total_len + 255) / 256);
    }
    const uint64_t n_tiles = tile_off[n_problems];
    DevCtx& d = s->devs[0];
    CU(cudaSetDevice(d.device));
    double addend[94 * 2];
    hc_cons_addends(addend);
    int8_t c2q[HC_MAX_CODES + 1];
    for (int k = 0; k <= HC_MAX_CODES; k++) c2q[k] = (int8_t)(k <= s->ncodes && s->code_to_q[k] >= 0 ? s->code_to_q[k] : 0);
    hc_cons_problem* d_prob = nullptr;
    hc_cons_seq* d_seqs = nullptr;
    unsigned long long *d_toff = nullptr, *d_marked = nullptr, *d_nmarked = nullptr;
    double *d_add = nullptr, *d_sums = nullptr, *d_msums = nullptr;
    int8_t* d_c2q = nullptr;
    uint16_t* d_cnt = nullptr;
    uint32_t* d_len = nullptr;
    char *d_base = nullptr, *d_qual = nullptr;
    const uint64_t cols = out_bytes ? out_bytes : 1;
    uint64_t marked_cap = cols / 64 + 4096;
    unsigned long long n_marked = 0;
    std::unique_ptr<uint16_t[]> cnt;      // not zero-filled: the copy out writes every element that is read
    std::vector<uint32_t> lens(n_seqs ? n_seqs : 1);
    std::vector<unsigned long long> marked;
    std::vector<double> msums;
    int rc = HC_OK;
    const bool mark_all = getenv("HC_CONS_HOST_ALL") != nullptr;      // tests: every column through the host libm
    if (mark_all) marked_cap = cols;
    cudaError_t e = hc_scratch_alloc_on((void**)&d_prob, n_problems * sizeof(hc_cons_problem), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_seqs, (n_seqs ? n_seqs : 1) * sizeof(hc_cons_seq), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_toff, (n_problems + 1) * sizeof(unsigned long long), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_add, sizeof(addend), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_c2q, sizeof(c2q), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_sums, cols * 4 * sizeof(double), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_cnt, cols * sizeof(uint16_t), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_base, cols, d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_qual, cols, d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_marked, marked_cap * sizeof(unsigned long long), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_nmarked, sizeof(unsigned long long), d.stream);
    if (e == cudaSuccess) e = hc_scratch_alloc_on((void**)&d_len, (n_seqs ? n_seqs : 1) * sizeof(uint32_t), d.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_nmarked, 0, sizeof(unsigned long long), d.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_base, 0, cols, d.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_qual, 0, cols, d.stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_cnt, 0, cols * sizeof(uint16_t), d.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_prob, problems, n_problems * sizeof(hc_cons_problem), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess && n_seqs) e = cudaMemcpyAsync(d_seqs, seqs, n_seqs * sizeof(hc_cons_seq), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_toff, tile_off.data(), (n_problems + 1) * sizeof(unsigned long long), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_add, addend, sizeof(addend), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_c2q, c2q, sizeof(c2q), cudaMemcpyHostToDevice, d.stream);
    if (e == cudaSuccess) {
        hc_cons_dev D;
        D.pk = d.pk; D.qual = d.qual; D.base2 = d.base2; D.nmask = d.nmask; D.rdesc = d.rdesc; D.packed = s->packed ? 1 : 0;
        // (with HC_CONS_HOST_ALL the kernel gets a list of capacity 0: it still counts its marks but stores none, and the
        // host decides every column from the sums, all_cols below)
        e = hc_launch_cons_sums(D, d_prob, n_problems, d_seqs, d_toff, n_tiles, d_add, d_c2q, min_qual, d_sums, d_cnt, d_base, d_qual,
                                d_marked, mark_all ? 0 : marked_cap, d_nmarked, d.stream);
        if (e == cudaSuccess && n_seqs) {
            cons_lens<<<(unsigned)((n_seqs + 255) / 256), 256, 0, d.stream>>>(d.rdesc, d_seqs, n_seqs, d_len);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&n_marked, d_nmarked, sizeof(n_marked), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    if (e == cudaSuccess) {
        cnt.reset(new (std::nothrow) uint16_t[(size_t)cols]);
        if (!cnt) rc = fail(HC_ERR_NOMEM, "hc_consensus: host allocation failed");
    }
    if (e == cudaSuccess && rc == HC_OK && out_bytes) {
        // the stream has just been synchronised: the staged copies (pinned ring, several host threads) may run beside it
        e = hc_copy_d2h(cnt.get(), d_cnt, (size_t)out_bytes * sizeof(uint16_t));
        if (e == cudaSuccess) e = hc_copy_d2h(cons_seq, d_base, (size_t)out_bytes);
        if (e == cudaSuccess) e = hc_copy_d2h(cons_qual, d_qual, (size_t)out_bytes);
    }
    if (e == cudaSuccess && rc == HC_OK && n_seqs) e = cudaMemcpyAsync(lens.data(), d_len, n_seqs * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream);
    // ---- columns whose outcome is within the error bound of a decision: their scores come back and the host libm decides
    bool all_cols = mark_all || n_marked > marked_cap;     // (more marked columns than the list holds: redo every column)
    if (e == cudaSuccess && rc == HC_OK && !all_cols && n_marked) {
        marked.resize(n_marked);
        msums.resize(4 * n_marked);
        e = hc_scratch_alloc_on((void**)&d_msums, 4 * n_marked * sizeof(double), d.stream);
        if (e == cudaSuccess) e = hc_launch_cons_gather(d_marked, n_marked, d_sums, d_msums, d.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(marked.data(), d_marked, n_marked * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(msums.data(), d_msums, 4 * n_marked * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    }
    if (e == cudaSuccess && rc == HC_OK && all_cols && out_bytes) {
        try { msums.resize((size_t)out_bytes * 4); } catch (...) { rc = fail(HC_ERR_NOMEM, "hc_consensus: host allocation failed"); }
        if (rc == HC_OK) e = cudaMemcpyAsync(msums.data(), d_sums, (size_t)out_bytes * 4 * sizeof(double), cudaMemcpyDeviceToHost, d.stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    hc_scratch_free_on(d_prob, d.stream); hc_scratch_free_on(d_seqs, d.stream); hc_scratch_free_on(d_toff, d.stream); hc_scratch_free_on(d_add, d.stream); hc_scratch_free_on(d_c2q, d.stream); hc_scratch_free_on(d_sums, d.stream); hc_scratch_free_on(d_cnt, d.stream); hc_scratch_free_on(d_len, d.stream);
    hc_scratch_free_on(d_base, d.stream); hc_scratch_free_on(d_qual, d.stream); hc_scratch_free_on(d_marked, d.stream); hc_scratch_free_on(d_nmarked, d.stream); hc_scratch_free_on(d_msums, d.stream);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA, std::string("hc_consensus: ") + cudaGetErrorString(e));
    if (rc != HC_OK) return rc;
    if (all_cols) {
#pragma omp parallel for schedule(static)
        for (int64_t g = 0; g < (int64_t)out_bytes; g++) {
            char b = 'N', q = '$';
            if (!hc_cons_final_pos(msums[4 * g], msums[4 * g + 1], msums[4 * g + 2], msums[4 * g + 3], cnt[g], min_qual, &b, &q)) q = 0;
            cons_seq[g] = b;
            cons_qual[g] = q;
        }
    } else {
        for (uint64_t k = 0; k < n_marked; k++) {
            const uint64_t g = marked[k];
            char b = 'N', q = '$';
            if (!hc_cons_final_pos(msums[4 * k], msums[4 * k + 1], msums[4 * k + 2], msums[4 * k + 3], cnt[g], min_qual, &b, &q)) q = 0;
            cons_seq[g] = b;
            cons_qual[g] = q;
        }
    }
    // ---- the column walk of :447-513, problems in parallel (their output regions are disjoint)
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t p = 0; p < (int64_t)n_problems; p++)
        hc_cons_walk(&problems[p], seqs, lens.data(), cnt.get(), min_clique_size, cons_seq, cons_qual, &results[p]);
    if (getenv("HC_CONS_VERBOSE")) fprintf(stderr, "hc_consensus: %llu of %llu columns re-evaluated on the host\n",
                                           all_cols ? (unsigned long long)out_bytes : n_marked, (unsigned long long)out_bytes);
    return HC_OK;
}

int hc_score_batch_device(hc_store* s, int device, void* stream, const hc_params* p, const hc_candidate* d_cand, uint64_t n,
                          hc_result* d_per_cand, hc_edge* d_edges, uint64_t edges_cap, uint64_t* d_nonedge_idx,
                          uint64_t nonedge_cap, uint64_t* d_counts, hc_batch_stats* stats) {
    if (!s || !p || !d_counts || (n && !d_cand)) return fail(HC_ERR_ARG, "hc_score_batch_device: NULL argument");
    // the kernels read a candidate as two 16-byte loads and store 8-byte aligned records: a misaligned pointer would fault
    if (((uintptr_t)d_cand & 15u) || (((uintptr_t)d_per_cand | (uintptr_t)d_edges | (uintptr_t)d_nonedge_idx | (uintptr_t)d_counts) & 7u))
        return fail(HC_ERR_ARG, "hc_score_batch_device: d_cand must be 16-byte aligned; d_per_cand, d_edges, d_nonedge_idx and "
                                "d_counts 8-byte aligned");
    DevCtx* d = find_ctx(s, device);
    if (!d) return fail(HC_ERR_ARG, "hc_score_batch_device: the store has no replica on this device");
    CU(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t nl = 0;
    int rc = enqueue_batch(s, *d, st, p, d_cand, 0, n, d_per_cand, d_edges, edges_cap, d_nonedge_idx, nonedge_cap, d_counts, 0,
                           nullptr, stats ? d->ev[0] : nullptr, stats ? d->ev[1] : nullptr, &nl);
    if (rc != HC_OK) return rc;
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        CU(cudaStreamSynchronize(st));
        rc = read_stats(*d, n, stats, d->ev[0], d->ev[1]);
        stats->total_ms = stats->kernel_ms;
        stats->kernel_launches = nl;
    }
    return rc;
}

// Host-buffer path.  The batch is cut into contiguous per-device shards (rank order = input order) and
// every shard is streamed through its device in chunks: H2D of chunk k+1 (s_copy), kernels of chunk k
// (stream) and D2H of what chunk k-1 produced (s_out) overlap.  Outputs are compacted on the device
// behind the outputs of the earlier chunks (running totals stay on the device), so the host sees
// one ordered list per device.
struct RunsHost {               // caller's run arrays (hc_score_batch_runs)
    const uint32_t* anchor;     // [n_runs]
    const uint64_t* start;      // [n_runs + 1]
    uint64_t n_runs;
};

static int score_host(hc_store* s, const hc_params* p, const void* cand, int compact, uint64_t n, hc_result* per_cand,
                      hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges, uint64_t* nonedge_idx, uint64_t nonedge_cap,
                      uint64_t* n_nonedges, hc_batch_stats* stats, const RunsHost* runs = nullptr, int small_out = 0) {
    if (!s || !p || !n_edges || !n_nonedges || (n && !cand)) return fail(HC_ERR_ARG, "hc_score_batch: NULL argument");
    if (stats) memset(stats, 0, sizeof(*stats));
    *n_edges = 0;
    *n_nonedges = 0;
    const size_t rec = compact == 4 ? sizeof(hc_candidate_entry6) : compact == 3 ? sizeof(hc_candidate_entry)
                                    : (compact == 2 ? sizeof(hc_candidate_short) : (compact ? sizeof(hc_candidate_compact) : sizeof(hc_candidate)));
    const int G = (int)s->devs.size();
    uint64_t chunk = 0;            // candidates per pipeline step; 0 = the tapered default schedule
    if (const char* e = getenv("HC_HOST_CHUNK")) { const uint64_t v = strtoull(e, nullptr, 10); if (v) chunk = v; }   // tests
    size_t whole_max = (size_t)2 << 30;   // shards up to this many bytes of records are copied in ahead of the kernels
    if (const char* e = getenv("HC_HOST_WHOLE_MAX")) whole_max = (size_t)strtoull(e, nullptr, 10);                   // tests
    std::vector<uint64_t> lo(G + 1);
    for (int g = 0; g <= G; g++) lo[g] = g == G ? n : (n * (uint64_t)g / (uint64_t)G) & ~63ull;   // contiguous index ranges, cut at multiples of 64
    // size of an edge record on its way out, and (small outputs) the caller's bit map as 32-bit words
    const size_t erec = !small_out ? sizeof(hc_edge) : ((p->flags & HC_FLAG_EXACT_EDGE_SCORES) ? sizeof(hc_edge_small_exact) : sizeof(hc_edge_small));
    char* const edges_b = reinterpret_cast<char*>(edges);
    uint32_t* const bits_out = reinterpret_cast<uint32_t*>(nonedge_idx);
    if (small_out) nonedge_cap = 0;
    // Pipeline steps of device g: [cs[g][k], cs[g][k+1]).  Whole-shard mode (the shard's records fit `whole_max`): all
    // copies in are issued up front into one device buffer and run ahead of the kernels, so the steps can start small
    // (the first kernel waits for 1 M candidates, not 8 M), grow to 16 M (fewer launches) and end small (little left to
    // copy out after the last kernel).  Otherwise: two slots, the copy in of step k+1 behind the kernels of step k-1,
    // uniform steps of 8 M (measured: beats 2, 4 and 16 M in that mode).
    std::vector<std::vector<uint64_t>> cs(G);
    std::vector<char> whole(G, 0);
    for (int g = 0; g < G; g++) {
        const uint64_t m = lo[g + 1] - lo[g];
        whole[g] = m > 0 && m * rec <= whole_max;
        std::vector<uint64_t>& c = cs[g];
        c.push_back(lo[g]);
        uint64_t big = 16ull << 20;
        const uint64_t small = 1ull << 20;
        if (const char* e = getenv("HC_HOST_BIG")) { const uint64_t v = strtoull(e, nullptr, 10); if (v >= 2 * small) big = v; }   // experiments
        if (chunk || !whole[g] || m <= 2 * small) {
            const uint64_t step = ((chunk ? chunk : (8ull << 20)) + 63) & ~63ull;     // steps start at multiples of 64 (bit-map words)
            for (uint64_t o = step; o < m; o += step) c.push_back(lo[g] + o);
        } else {
            uint64_t done = 0, sz = small;
            while (sz < big && m - done > 4 * sz) { done += sz; c.push_back(lo[g] + done); sz *= 2; }          // 1, 2, 4, 8 M
            while (m - done > 2 * big) { done += big; c.push_back(lo[g] + done); }                            // 16 M ...
            while (m - done > 2 * small) { done += ((m - done + 1) / 2 + 63) & ~63ull; c.push_back(lo[g] + done); }   // halves (multiples of 64)
        }
        if (m > 0) c.push_back(lo[g + 1]);
    }
    uint32_t launches = 0;
    std::vector<uint64_t> dev_e(G, 0), dev_n(G, 0);
    int result = HC_OK;
    // ---- allocate / reset
    for (int g = 0; g < G; g++) {
        DevCtx& d = s->devs[g];
        const uint64_t m = lo[g + 1] - lo[g];
        uint64_t cap = 1;
        for (size_t k = 0; k + 1 < cs[g].size(); k++) cap = std::max<uint64_t>(cap, cs[g][k + 1] - cs[g][k]);
        CU(cudaSetDevice(d.device));
        {   // the kernels' workspace for the largest step, once: growing it step by step would free and reallocate
            // (a device-wide synchronisation each) right in the warm-up steps of the pipeline
            const int rcw = ensure_workspace(d, cap);
            if (rcw != HC_OK) return rcw;
        }
        if (whole[g]) {
            if (m * rec > d.whole_cap) {
                cudaFree(d.d_whole); d.d_whole = nullptr; d.whole_cap = 0;
                CU(cudaMalloc(&d.d_whole, m * rec));
                d.whole_cap = m * rec;
            }
            while (d.ev_step.size() + 1 < cs[g].size()) {
                cudaEvent_t ev;
                CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                d.ev_step.push_back(ev);
            }
        } else if (cap > d.slot_cap) {
            for (int k = 0; k < 2; k++) { cudaFree(d.d_cand[k]); d.d_cand[k] = nullptr; }
            d.slot_cap = 0;
            for (int k = 0; k < 2; k++) CU(cudaMalloc(&d.d_cand[k], cap * sizeof(hc_candidate)));
            d.slot_cap = cap;
        }
        if (per_cand && cap > d.pc_cap) {
            for (int k = 0; k < 2; k++) { cudaFree(d.d_per_cand[k]); d.d_per_cand[k] = nullptr; }
            d.pc_cap = 0;
            for (int k = 0; k < 2; k++) CU(cudaMalloc(&d.d_per_cand[k], cap * sizeof(hc_result)));
            d.pc_cap = cap;
        }
        if (runs && cap > d.tile_cap * 32) {
            const uint64_t tiles = (cap + 31) / 32;
            for (int k = 0; k < 2; k++) { cudaFree(d.d_tile_run[k]); d.d_tile_run[k] = nullptr; }
            d.tile_cap = 0;
            for (int k = 0; k < 2; k++) CU(cudaMalloc(&d.d_tile_run[k], tiles * sizeof(uint32_t)));
            d.tile_cap = tiles;
        }
        const uint64_t need_e = std::max<uint64_t>(std::min<uint64_t>(m, edges_cap), 1), need_n = std::max<uint64_t>(std::min<uint64_t>(m, nonedge_cap), 1);
        if (need_e > d.acc_e_cap) { cudaFree(d.d_acc_edges); d.d_acc_edges = nullptr; d.acc_e_cap = 0; CU(cudaMalloc(&d.d_acc_edges, need_e * sizeof(hc_edge))); d.acc_e_cap = need_e; }
        if (small_out && (m + 31) / 32 + 4 > d.acc_b_cap) {
            cudaFree(d.d_acc_bits); d.d_acc_bits = nullptr; d.acc_b_cap = 0;
            CU(cudaMalloc(&d.d_acc_bits, ((m + 31) / 32 + 4) * sizeof(uint32_t)));
            d.acc_b_cap = (m + 31) / 32 + 4;
        }
        if (need_n > d.acc_n_cap) { cudaFree(d.d_acc_nonedge); d.d_acc_nonedge = nullptr; d.acc_n_cap = 0; CU(cudaMalloc(&d.d_acc_nonedge, need_n * sizeof(uint64_t))); d.acc_n_cap = need_n; }
        CU(cudaMemsetAsync(d.d_run, 0, 2 * sizeof(unsigned long long), d.stream));
        CU(cudaEventRecord(d.ev[2], d.stream));
    }
    // ---- is the caller's record buffer pageable?  (registered / pinned memory goes to the copy engine as it is)
    bool pageable = false;
    if (n && !getenv("HC_NO_HOST_STAGING")) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, cand) != cudaSuccess) { cudaGetLastError(); pageable = true; }
        else pageable = at.type == cudaMemoryTypeUnregistered;
    }
    // ---- whole-shard mode: the copy in of step k (and its run arrays) is queued a few steps ahead of its kernels
    std::vector<std::vector<uint64_t>> run_off(G);    // per issued step: offset of its [anchors][starts] in d_runs_all (words), n_runs
    std::vector<uint64_t> run_words(G, 0);
    std::vector<size_t> copied(G, 0);
    for (int g = 0; g < G; g++) {
        if (!whole[g] || !runs) continue;
        DevCtx& d = s->devs[g];
        CU(cudaSetDevice(d.device));
        const uint64_t* st = runs->start;
        const size_t nsteps = cs[g].size() - 1;
        const uint64_t ra = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, lo[g]) - st) - 1;
        const uint64_t rb = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, lo[g + 1] - 1) - st) - 1;
        const uint64_t words = 2 * (rb - ra + 1 + nsteps) + nsteps;      // every step boundary may cut one run in two
        if (words > d.runs_all_cap) {
            cudaFree(d.d_runs_all); d.d_runs_all = nullptr;
            if (d.h_runs_all) { cudaFreeHost(d.h_runs_all); d.h_runs_all = nullptr; }
            d.runs_all_cap = 0;
            const uint64_t want = words + words / 8 + 1024;
            CU(cudaMalloc(&d.d_runs_all, want * sizeof(uint32_t)));
            CU(cudaMallocHost(&d.h_runs_all, want * sizeof(uint32_t)));
            d.runs_all_cap = want;
        }
    }
    auto issue_copy = [&](int g, size_t k) -> int {   // the current device is d.device
        DevCtx& d = s->devs[g];
        const uint64_t c0 = cs[g][k], cm = cs[g][k + 1] - c0;
        if (runs) {   // the runs that overlap [c0, c0 + cm): anchors as they are, starts clipped and made relative
            const uint64_t* st = runs->start;
            const uint64_t r0 = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, c0) - st) - 1;
            const uint64_t nr = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, c0 + cm - 1) - st) - r0;
            const uint64_t o = run_words[g];
            uint32_t* h = d.h_runs_all + o;
            memcpy(h, runs->anchor + r0, nr * sizeof(uint32_t));
            for (uint64_t j = 0; j < nr; j++) h[nr + j] = (uint32_t)(std::max<uint64_t>(st[r0 + j], c0) - c0);
            h[2 * nr] = (uint32_t)cm;
            run_off[g].push_back(o);
            run_off[g].push_back(nr);
            run_words[g] += 2 * nr + 1;
            CU(cudaMemcpyAsync(d.d_runs_all + o, h, (2 * nr + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, d.s_copy));
        }
        const char* src = (const char*)cand + c0 * rec;
        // pageable records (a std::vector, a numpy array) go through the pinned ring of hc_stage.cu, copied by several host threads
        if (pageable) CU(hc_copy_h2d_on(d.d_whole + (c0 - lo[g]) * rec, src, cm * rec, d.s_copy));
        else CU(cudaMemcpyAsync(d.d_whole + (c0 - lo[g]) * rec, src, cm * rec, cudaMemcpyHostToDevice, d.s_copy));
        CU(cudaEventRecord(d.ev_step[k], d.s_copy));
        return HC_OK;
    };
    const size_t copy_ahead = 3;
    // ---- chunk loop, all devices interleaved
    uint64_t max_chunks = 0;
    for (int g = 0; g < G; g++) max_chunks = std::max<uint64_t>(max_chunks, cs[g].empty() ? 0 : cs[g].size() - 1);
    std::vector<uint64_t> out_e(G, 0), out_n(G, 0);   // already copied out (G == 1 streams results out while computing)
    auto finalize_chunk = [&](int g, uint64_t k) -> int {   // chunk k of device g has been enqueued; wait for it, account, copy out
        DevCtx& d = s->devs[g];
        const int slot = (int)(k & 1);
        const uint64_t c0 = cs[g][k], cm = cs[g][k + 1] - c0;
        CU(cudaSetDevice(d.device));
        CU(cudaEventSynchronize(d.ev_done[slot]));
        const unsigned long long* h = d.h_cnt + slot * HC_CNT_N;
        int rc = add_stats(d, h, cm, stats, nullptr, nullptr);
        dev_e[g] += h[HC_CNT_EDGES];
        dev_n[g] += h[HC_CNT_NONEDGES];
        if (per_cand) {
            CU(cudaStreamWaitEvent(d.s_out, d.ev_done[slot], 0));
            CU(hc_copy_d2h_on(per_cand + c0, d.d_per_cand[slot], cm * sizeof(hc_result), d.s_out, nullptr));
        }
        if (G == 1) {   // offsets in the caller's arrays are known: stream this chunk's results out now
            const uint64_t e1 = std::min<uint64_t>(dev_e[g], d.acc_e_cap), n1 = std::min<uint64_t>(dev_n[g], d.acc_n_cap);
            CU(cudaStreamWaitEvent(d.s_out, d.ev_done[slot], 0));
            if (e1 > out_e[g] && e1 <= edges_cap)
                CU(hc_copy_d2h_on(edges_b + out_e[g] * erec, reinterpret_cast<char*>(d.d_acc_edges) + out_e[g] * erec, (e1 - out_e[g]) * erec, d.s_out, nullptr));
            if (!small_out && n1 > out_n[g] && n1 <= nonedge_cap)
                CU(hc_copy_d2h_on(nonedge_idx + out_n[g], d.d_acc_nonedge + out_n[g], (n1 - out_n[g]) * sizeof(uint64_t), d.s_out, nullptr));
            if (small_out && cm)     // this chunk's words of the bit map (chunks start at multiples of 64)
                CU(hc_copy_d2h_on(bits_out + c0 / 32, d.d_acc_bits + (c0 - lo[g]) / 32, ((cm + 31) / 32) * sizeof(uint32_t), d.s_out, nullptr));
            out_e[g] = std::max(out_e[g], e1);
            out_n[g] = std::max(out_n[g], n1);
        }
        CU(cudaEventRecord(d.ev_out[slot], d.s_out));
        return rc;
    };
    for (uint64_t k = 0; k < max_chunks; k++) {
        for (int g = 0; g < G; g++) {
            DevCtx& d = s->devs[g];
            if (k + 1 >= cs[g].size()) continue;
            const uint64_t c0 = cs[g][k], cm = cs[g][k + 1] - c0;
            const int slot = (int)(k & 1);
            CU(cudaSetDevice(d.device));
            if (k >= 2) {   // the slot's previous user (chunk k-2) must have been computed and copied out
                if (!whole[g]) CU(cudaStreamWaitEvent(d.s_copy, d.ev_done[slot], 0));
                CU(cudaStreamWaitEvent(d.stream, d.ev_out[slot], 0));
            }
            RunDev rdv{nullptr, nullptr, 0, nullptr};
            const void* d_cand_k = d.d_cand[slot];
            if (whole[g]) {   // nothing to wait for before queueing copies: the whole shard has its own place on the device
                while (copied[g] < cs[g].size() - 1 && copied[g] <= k + copy_ahead) {
                    const int rc = issue_copy(g, copied[g]);
                    if (rc != HC_OK) return rc;
                    copied[g]++;
                }
                d_cand_k = d.d_whole + (c0 - lo[g]) * rec;
                if (runs) {
                    const uint64_t o = run_off[g][2 * k], nr = run_off[g][2 * k + 1];
                    rdv.anchor = d.d_runs_all + o; rdv.start = d.d_runs_all + o + nr; rdv.n_runs = (uint32_t)nr; rdv.tile_run = d.d_tile_run[slot];
                }
                CU(cudaStreamWaitEvent(d.stream, d.ev_step[k], 0));
            } else {
            if (pageable) CU(hc_copy_h2d_on(d.d_cand[slot], (const char*)cand + c0 * rec, cm * rec, d.s_copy));
            else CU(cudaMemcpyAsync(d.d_cand[slot], (const char*)cand + c0 * rec, cm * rec, cudaMemcpyHostToDevice, d.s_copy));
            if (runs) {   // the runs that overlap [c0, c0 + cm): anchors as they are, starts clipped and made relative
                const uint64_t* st = runs->start;
                const uint64_t r0 = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, c0) - st) - 1;
                const uint64_t r1 = (uint64_t)(std::upper_bound(st, st + runs->n_runs + 1, c0 + cm - 1) - st) - 1;
                const uint64_t nr = r1 - r0 + 1;
                if (nr > d.runs_cap) {   // both slots grow together; the other slot's copy-in has long completed (finalize_chunk)
                    CU(cudaStreamSynchronize(d.s_copy));
                    CU(cudaStreamSynchronize(d.stream));
                    const uint64_t want = nr + nr / 4 + 1024;
                    for (int q = 0; q < 2; q++) {
                        cudaFree(d.d_runs[q]); d.d_runs[q] = nullptr;
                        if (d.h_runs[q]) { cudaFreeHost(d.h_runs[q]); d.h_runs[q] = nullptr; }
                    }
                    d.runs_cap = 0;
                    for (int q = 0; q < 2; q++) {
                        CU(cudaMalloc(&d.d_runs[q], (2 * want + 1) * sizeof(uint32_t)));
                        CU(cudaMallocHost(&d.h_runs[q], (2 * want + 1) * sizeof(uint32_t)));
                    }
                    d.runs_cap = want;
                }
                uint32_t* h = d.h_runs[slot];
                memcpy(h, runs->anchor + r0, nr * sizeof(uint32_t));
                for (uint64_t j = 0; j < nr; j++) h[nr + j] = (uint32_t)(std::max<uint64_t>(st[r0 + j], c0) - c0);
                h[2 * nr] = (uint32_t)cm;
                CU(cudaMemcpyAsync(d.d_runs[slot], h, (2 * nr + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, d.s_copy));
                rdv.anchor = d.d_runs[slot]; rdv.start = d.d_runs[slot] + nr; rdv.n_runs = (uint32_t)nr; rdv.tile_run = d.d_tile_run[slot];
            }
            CU(cudaEventRecord(d.ev_in[slot], d.s_copy));
            CU(cudaStreamWaitEvent(d.stream, d.ev_in[slot], 0));
            }
            uint32_t nl = 0;
            int rc = enqueue_batch(s, d, d.stream, p, d_cand_k, compact, cm, per_cand ? d.d_per_cand[slot] : nullptr,
                                   d.d_acc_edges, d.acc_e_cap * sizeof(hc_edge) / erec, small_out ? nullptr : d.d_acc_nonedge,
                                   small_out ? 0 : d.acc_n_cap, nullptr, c0, d.d_run,
                                   (stats && k == 0) ? d.ev[0] : nullptr, (stats && k == 0) ? d.ev[1] : nullptr, &nl,
                                   runs ? &rdv : nullptr, small_out, small_out ? d.d_acc_bits + (c0 - lo[g]) / 32 : nullptr);
            if (rc != HC_OK) return rc;
            launches += nl;
            CU(cudaMemcpyAsync(d.h_cnt + slot * HC_CNT_N, d.counters, HC_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream));
            CU(cudaEventRecord(d.ev_done[slot], d.stream));
        }
        if (k >= 1)
            for (int g = 0; g < G; g++)
                if (k < cs[g].size()) { int rc = finalize_chunk(g, k - 1); if (rc != HC_OK) result = rc; }
    }
    if (max_chunks >= 1)
        for (int g = 0; g < G; g++)
            if (max_chunks < cs[g].size()) { int rc = finalize_chunk(g, max_chunks - 1); if (rc != HC_OK) result = rc; }
    // ---- gather: rank order = input order
    uint64_t te = 0, tn = 0;
    for (int g = 0; g < G; g++) {
        DevCtx& d = s->devs[g];
        CU(cudaSetDevice(d.device));
        if (G > 1) {
            const uint64_t e1 = std::min<uint64_t>(dev_e[g], d.acc_e_cap), n1 = std::min<uint64_t>(dev_n[g], d.acc_n_cap);
            if (e1 && te + e1 <= edges_cap) CU(cudaMemcpyAsync(edges_b + te * erec, d.d_acc_edges, e1 * erec, cudaMemcpyDeviceToHost, d.s_out));
            if (!small_out && n1 && tn + n1 <= nonedge_cap) CU(cudaMemcpyAsync(nonedge_idx + tn, d.d_acc_nonedge, n1 * sizeof(uint64_t), cudaMemcpyDeviceToHost, d.s_out));
            if (small_out && lo[g + 1] > lo[g])
                CU(cudaMemcpyAsync(bits_out + lo[g] / 32, d.d_acc_bits, ((lo[g + 1] - lo[g] + 31) / 32) * sizeof(uint32_t), cudaMemcpyDeviceToHost, d.s_out));
        }
        te += dev_e[g];
        tn += dev_n[g];
    }
    float total_ms = 0;
    for (int g = 0; g < G; g++) {
        DevCtx& d = s->devs[g];
        CU(cudaSetDevice(d.device));
        CU(cudaStreamSynchronize(d.s_out));
        CU(cudaStreamSynchronize(d.stream));
        CU(cudaEventRecord(d.ev[3], d.stream));
        CU(cudaEventSynchronize(d.ev[3]));
        float ms = 0;
        if (cudaEventElapsedTime(&ms, d.ev[2], d.ev[3]) == cudaSuccess) total_ms = std::max(total_ms, ms);
        if (stats && lo[g + 1] > lo[g]) {
            if (cudaEventElapsedTime(&ms, d.ev[0], d.ev[1]) == cudaSuccess) stats->kernel_ms = std::max(stats->kernel_ms, ms);
            if (cudaEventElapsedTime(&ms, d.ev[4], d.ev[5]) == cudaSuccess) stats->score_kernel_ms = std::max(stats->score_kernel_ms, ms);
        }
    }
    *n_edges = te;
    *n_nonedges = tn;
    if (stats) { stats->total_ms = total_ms; stats->kernel_launches = launches; }
    if (result != HC_OK) return result;
    if (small_out && (n & 63)) {   // the last word of the bit map is written whole by the host: bits beyond n are 0
        const uint64_t last = n >> 6;
        nonedge_idx[last] &= (1ull << (n & 63)) - 1ull;
    }
    if (te > edges_cap || (!small_out && tn > nonedge_cap))
        return fail(HC_ERR_CAPACITY, "hc_score_batch: output buffer too small (required sizes returned in n_edges/n_nonedges)");
    return HC_OK;
}

int hc_score_batch(hc_store* s, const hc_params* p, const hc_candidate* cand, uint64_t n, hc_result* per_cand,
                   hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges, uint64_t* nonedge_idx, uint64_t nonedge_cap,
                   uint64_t* n_nonedges, hc_batch_stats* stats) {
    return score_host(s, p, cand, 0, n, per_cand, edges, edges_cap, n_edges, nonedge_idx, nonedge_cap, n_nonedges, stats);
}

int hc_score_batch_compact(hc_store* s, const hc_params* p, const hc_candidate_compact* cand, uint64_t n, hc_result* per_cand,
                           hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges, uint64_t* nonedge_idx, uint64_t nonedge_cap,
                           uint64_t* n_nonedges, hc_batch_stats* stats) {
    return score_host(s, p, cand, 1, n, per_cand, edges, edges_cap, n_edges, nonedge_idx, nonedge_cap, n_nonedges, stats);
}

int hc_score_batch_short(hc_store* s, const hc_params* p, const hc_candidate_short* cand, uint64_t n, hc_result* per_cand,
                         hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges, uint64_t* nonedge_idx, uint64_t nonedge_cap,
                         uint64_t* n_nonedges, hc_batch_stats* stats) {
    return score_host(s, p, cand, 2, n, per_cand, edges, edges_cap, n_edges, nonedge_idx, nonedge_cap, n_nonedges, stats);
}

int hc_score_batch_runs(hc_store* s, const hc_params* p, const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                        const hc_candidate_entry* entries, uint64_t n, hc_result* per_cand, hc_edge* edges, uint64_t edges_cap,
                        uint64_t* n_edges, uint64_t* nonedge_idx, uint64_t nonedge_cap, uint64_t* n_nonedges, hc_batch_stats* stats) {
    if (n && (!run_anchor || !run_start || n_runs == 0)) return fail(HC_ERR_ARG, "hc_score_batch_runs: NULL run arrays");
    if (s && s->n_reads > 0x7fffffffull) return fail(HC_ERR_ARG, "hc_score_batch_runs: more than 2^31-1 reads in the store");
    if (n) {
        if (run_start[0] != 0 || run_start[n_runs] != n) return fail(HC_ERR_ARG, "hc_score_batch_runs: run_start must begin at 0 and end at n");
        int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
        for (long long r = 0; r < (long long)n_runs; r++) bad |= (run_start[r] >= run_start[r + 1]);
        if (bad) return fail(HC_ERR_ARG, "hc_score_batch_runs: run_start must be strictly increasing (no empty runs)");
    }
    const RunsHost rh{run_anchor, run_start, n_runs};
    return score_host(s, p, entries, 3, n, per_cand, edges, edges_cap, n_edges, nonedge_idx, nonedge_cap, n_nonedges, stats,
                      n ? &rh : nullptr);
}

int hc_score_batch_runs_small(hc_store* s, const hc_params* p, const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                              const hc_candidate_entry* entries, uint64_t n, void* edges, uint64_t edges_cap, uint64_t* n_edges,
                              uint64_t* nonedge_bits, uint64_t* n_nonedges, hc_batch_stats* stats) {
    if (n && (!run_anchor || !run_start || n_runs == 0)) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: NULL run arrays");
    if (n && !nonedge_bits) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: NULL bit map");
    if (s && s->n_reads > 0x7fffffffull) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: more than 2^31-1 reads in the store");
    if (n > 0xffffffffull) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: a call takes fewer than 2^32 candidates");
    if (n) {
        if (run_start[0] != 0 || run_start[n_runs] != n) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: run_start must begin at 0 and end at n");
        int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
        for (long long r = 0; r < (long long)n_runs; r++) bad |= (run_start[r] >= run_start[r + 1]);
        if (bad) return fail(HC_ERR_ARG, "hc_score_batch_runs_small: run_start must be strictly increasing (no empty runs)");
    }
    const RunsHost rh{run_anchor, run_start, n_runs};
    return score_host(s, p, entries, 3, n, nullptr, reinterpret_cast<hc_edge*>(edges), edges_cap, n_edges, nonedge_bits, 0, n_nonedges, stats,
                      n ? &rh : nullptr, 1);
}

int hc_score_batch_runs6_small(hc_store* s, const hc_params* p, const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                               const hc_candidate_entry6* entries, uint64_t n, void* edges, uint64_t edges_cap, uint64_t* n_edges,
                               uint64_t* nonedge_bits, uint64_t* n_nonedges, hc_batch_stats* stats) {
    if (n && (!run_anchor || !run_start || n_runs == 0)) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: NULL run arrays");
    if (n && !nonedge_bits) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: NULL bit map");
    if (s && s->n_reads > (1ull << 25)) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: more than 2^25 reads in the store");
    if (n > 0xffffffffull) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: a call takes fewer than 2^32 candidates");
    if (n) {
        if (run_start[0] != 0 || run_start[n_runs] != n) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: run_start must begin at 0 and end at n");
        int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
        for (long long r = 0; r < (long long)n_runs; r++) bad |= (run_start[r] >= run_start[r + 1]);
        if (bad) return fail(HC_ERR_ARG, "hc_score_batch_runs6_small: run_start must be strictly increasing (no empty runs)");
    }
    const RunsHost rh{run_anchor, run_start, n_runs};
    return score_host(s, p, entries, 4, n, nullptr, reinterpret_cast<hc_edge*>(edges), edges_cap, n_edges, nonedge_bits, 0, n_nonedges, stats,
                      n ? &rh : nullptr, 1);
}

int hc_score_batch_short_small(hc_store* s, const hc_params* p, const hc_candidate_short* cand, uint64_t n, void* edges,
                               uint64_t edges_cap, uint64_t* n_edges, uint64_t* nonedge_bits, uint64_t* n_nonedges, hc_batch_stats* stats) {
    if (n && !nonedge_bits) return fail(HC_ERR_ARG, "hc_score_batch_short_small: NULL bit map");
    if (n > 0xffffffffull) return fail(HC_ERR_ARG, "hc_score_batch_short_small: a call takes fewer than 2^32 candidates");
    return score_host(s, p, cand, 2, n, nullptr, reinterpret_cast<hc_edge*>(edges), edges_cap, n_edges, nonedge_bits, 0, n_nonedges, stats, nullptr, 1);
}

// Text in, kept candidates and edges out.  The buffer is cut into pieces as hc_ingest_overlaps cuts it; on the id map's
// main stream every piece is parsed (hc_ingest_device) and scored (enqueue_batch in kept mode, running totals in d.d_run),
// and only what the host needs leaves the device.  The copy in of piece i + 1 runs on the copy stream and the copy out
// of piece i - 1 on the output stream while piece i is processed (two buffer sets).
int hc_ingest_score_overlaps(hc_store* s, const hc_idmap* cm, const char* text, uint64_t n_bytes, const hc_ingest_params* ip,
                             const hc_params* p, hc_candidate* kept, uint64_t* kept_line, uint8_t* kept_class, uint64_t kept_cap,
                             void* edges, uint64_t edges_cap, hc_overlap_rec* filtered, uint64_t* filtered_line, uint64_t filtered_cap,
                             hc_ingest_score_stats* stats) {
    if (!s || !cm || !ip || !p || !stats || (n_bytes && !text) || (kept_cap && (!kept || !kept_class)) || (edges_cap && !edges) ||
        (filtered_cap && !filtered))
        return fail(HC_ERR_ARG, "hc_ingest_score_overlaps: NULL argument");
    hc_idmap* m = const_cast<hc_idmap*>(cm);
    memset(stats, 0, sizeof(*stats));
    stats->ingest.first_error_line = ~0ull;
    DevCtx* dp = find_ctx(s, m->device);
    if (!dp) return fail(HC_ERR_ARG, "hc_ingest_score_overlaps: the store has no replica on the id map's device");
    if (n_bytes == 0) return HC_OK;
    DevCtx& d = *dp;
    CU(cudaSetDevice(d.device));
    const std::vector<uint64_t> cut = hc_ingest_cuts(text, n_bytes, hc_ingest_piece_bytes());
    const size_t n_pieces = cut.size() - 1;
    uint64_t max_piece = 0;
    for (size_t i = 0; i < n_pieces; i++) max_piece = std::max(max_piece, cut[i + 1] - cut[i]);
    const uint64_t cap = hc_ingest_rec_cap(max_piece);           // records of any kind one piece can produce
    const uint64_t tbytes = (max_piece + 16 + 255) & ~255ull;
    const size_t erec = (p->flags & HC_FLAG_EXACT_EDGE_SCORES) ? sizeof(hc_edge_small_exact) : sizeof(hc_edge_small);
    // a kept slot: [cand 32][line 8][edge record <= 32][edge_kept 4][class 1] bytes per record
    const uint64_t o_line = cap * sizeof(hc_candidate), o_edge = o_line + cap * sizeof(uint64_t);
    const uint64_t o_src = o_edge + cap * sizeof(hc_edge_small_exact), o_cls = o_src + cap * sizeof(uint32_t);
    if (cap > d.kept_cap) {
        for (int k = 0; k < 2; k++) { cudaFree(d.d_kept[k]); d.d_kept[k] = nullptr; }
        d.kept_cap = 0;
        for (int k = 0; k < 2; k++) CU(cudaMalloc(&d.d_kept[k], o_cls + cap));
        d.kept_cap = cap;
    }
    {
        const int rcw = ensure_workspace(d, cap);
        if (rcw != HC_OK) return rcw;
    }
    char* d_text = nullptr;
    hc_candidate* d_cand = nullptr;
    hc_overlap_rec* d_filt = nullptr;
    uint64_t *d_cl = nullptr, *d_fl = nullptr;
    CU(hc_idmap_ws(m, 11, 2 * tbytes, (void**)&d_text));
    CU(hc_idmap_ws(m, 12, 2 * cap * sizeof(hc_candidate), (void**)&d_cand));
    CU(hc_idmap_ws(m, 13, 2 * cap * sizeof(hc_overlap_rec), (void**)&d_filt));
    if (kept_line) CU(hc_idmap_ws(m, 14, 2 * cap * sizeof(uint64_t), (void**)&d_cl));
    if (filtered_line) CU(hc_idmap_ws(m, 15, 2 * cap * sizeof(uint64_t), (void**)&d_fl));
    hc_ingest_stats& is = stats->ingest;
    hc_batch_stats& bs = stats->score;
    bool overflow = false;
    uint64_t lines = 0, nk = 0, ne = 0, nf = 0;
    struct Out { int b; bool copy; uint64_t nk, pk, ne, pe, nf, pf; };   // a piece whose outputs wait to be copied out
    Out pend{};
    bool have_pend = false;
    auto copy_out = [&](const Out& o) -> int {
        const unsigned char* kb = d.d_kept[o.b];
        if (o.copy && o.pk) {
            CU(hc_copy_d2h_on(kept + o.nk, kb, o.pk * sizeof(hc_candidate), m->s_out, nullptr));
            if (kept_line) CU(hc_copy_d2h_on(kept_line + o.nk, kb + o_line, o.pk * sizeof(uint64_t), m->s_out, nullptr));
            CU(hc_copy_d2h_on(kept_class + o.nk, kb + o_cls, o.pk, m->s_out, nullptr));
        }
        if (o.copy && o.pe) CU(hc_copy_d2h_on(static_cast<char*>(edges) + o.ne * erec, kb + o_edge, o.pe * erec, m->s_out, nullptr));
        if (o.copy && o.pf) {
            CU(hc_copy_d2h_on(filtered + o.nf, d_filt + (size_t)o.b * cap, o.pf * sizeof(hc_overlap_rec), m->s_out, nullptr));
            if (filtered_line) CU(hc_copy_d2h_on(filtered_line + o.nf, d_fl + (size_t)o.b * cap, o.pf * sizeof(uint64_t), m->s_out, nullptr));
        }
        CU(cudaEventRecord(m->ev_out[o.b], m->s_out));
        return HC_OK;
    };
    auto run = [&]() -> int {
        hc_ingest_params pp = *ip;
        CU(cudaMemsetAsync(d.d_run, 0, 2 * sizeof(unsigned long long), m->s_main));
        CU(cudaEventRecord(d.ev[2], m->s_main));
        CU(hc_copy_h2d_on(d_text, text, cut[1] - cut[0], m->s_copy));
        CU(cudaEventRecord(m->ev_in[0], m->s_copy));
        for (size_t i = 0; i < n_pieces && lines < ip->max_overlaps; i++) {
            const int b = (int)(i & 1);
            if (i + 1 < n_pieces) {   // text buffer b ^ 1 was read by piece i - 1, which has completed
                CU(hc_copy_h2d_on(d_text + (size_t)(b ^ 1) * tbytes, text + cut[i + 1], cut[i + 2] - cut[i + 1], m->s_copy));
                CU(cudaEventRecord(m->ev_in[b ^ 1], m->s_copy));
            }
            CU(cudaStreamWaitEvent(m->s_main, m->ev_in[b], 0));
            if (i >= 2) CU(cudaEventSynchronize(m->ev_out[b]));          // buffer set b has been copied out
            hc_candidate* dc = d_cand + (size_t)b * cap;
            uint64_t* dcl = d_cl ? d_cl + (size_t)b * cap : nullptr;
            hc_ingest_stats st;
            pp.max_overlaps = ip->max_overlaps - lines;
            int rc = hc_ingest_device(m, d_text + (size_t)b * tbytes, cut[i + 1] - cut[i], &pp, dc, dcl, cap, d_filt + (size_t)b * cap,
                                      d_fl ? d_fl + (size_t)b * cap : nullptr, cap, &st, m->s_main, lines);
            if (rc != HC_OK) return rc;
            if (st.first_error_line != ~0ull && is.first_error_line == ~0ull) {
                is.first_error_line = lines + st.first_error_line;
                is.first_error_offset = cut[i] + st.first_error_offset;
                is.first_error_length = st.first_error_length;
                is.first_error_status = st.first_error_status;
            }
            unsigned char* kb = d.d_kept[b];
            const hc_kept_dev K{reinterpret_cast<hc_candidate*>(kb), kept_line ? reinterpret_cast<uint64_t*>(kb + o_line) : nullptr, kb + o_cls,
                                dcl, reinterpret_cast<uint32_t*>(kb + o_src)};
            uint32_t nl = 0;
            rc = enqueue_batch(s, d, m->s_main, p, dc, 0, st.n_scored, nullptr, reinterpret_cast<hc_edge*>(kb + o_edge), cap, nullptr, 0,
                               nullptr, 0, d.d_run, d.ev[0], d.ev[1], &nl, nullptr, 1, nullptr, &K);
            if (rc != HC_OK) return rc;
            CU(cudaMemcpyAsync(d.h_cnt, d.counters, HC_CNT_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, m->s_main));
            if (have_pend) { rc = copy_out(pend); have_pend = false; if (rc != HC_OK) return rc; }   // overlaps this piece's kernels
            CU(cudaStreamSynchronize(m->s_main));
            const unsigned long long* h = d.h_cnt;
            rc = add_stats(d, h, st.n_scored, &bs, nullptr, nullptr);     // the message of hc_score_batch* for rejected candidates
            if (rc != HC_OK) return rc;
            float ms = 0;
            if (cudaEventElapsedTime(&ms, d.ev[0], d.ev[1]) == cudaSuccess) bs.kernel_ms += ms;
            if (st.n_scored && cudaEventElapsedTime(&ms, d.ev[4], d.ev[5]) == cudaSuccess) bs.score_kernel_ms += ms;
            bs.kernel_launches += nl;
            const uint64_t pe = h[HC_CNT_EDGES], pk = pe + h[HC_CNT_NONEDGES];
            if (nk + pk > 0xffffffffull)
                return fail(HC_ERR_ARG, "hc_ingest_score_overlaps: 2^32 or more kept candidates (hc_edge_small.cand is 32 bits)");
            overflow = overflow || nk + pk > kept_cap || ne + pe > edges_cap || nf + st.n_filtered > filtered_cap;
            pend = Out{b, !overflow, nk, pk, ne, pe, nf, st.n_filtered};
            have_pend = true;
            lines += st.n_lines; nk += pk; ne += pe; nf += st.n_filtered;
            is.n_scored += st.n_scored; is.n_skipped += st.n_skipped; is.n_dropped += st.n_dropped; is.device_ms += st.device_ms;
        }
        if (have_pend) { have_pend = false; return copy_out(pend); }
        return HC_OK;
    };
    int rc = run();
    const cudaError_t e1 = cudaStreamSynchronize(m->s_out), e2 = cudaStreamSynchronize(m->s_copy);
    if (rc != HC_OK) return rc;
    CU(e1);
    CU(e2);
    CU(cudaEventRecord(d.ev[3], m->s_main));
    CU(cudaEventSynchronize(d.ev[3]));
    float ms = 0;
    if (cudaEventElapsedTime(&ms, d.ev[2], d.ev[3]) == cudaSuccess) bs.total_ms = ms;
    is.n_lines = lines; is.n_filtered = nf;
    stats->n_kept = nk;
    if (overflow) return fail(HC_ERR_CAPACITY, "hc_ingest_score_overlaps: output buffer too small (required sizes returned in stats)");
    return HC_OK;
}

int hc_overlap_score_multi(const char* seq1, uint32_t len1, const char* seq2, uint32_t len2, const char* qual1,
                           const char* qual2, const uint32_t* pos, uint32_t n_pos, const hc_params* p, double* scores,
                           double* mismatch_rates, uint8_t* above) {
    if (!seq1 || !seq2 || !qual1 || !qual2 || !p || len1 == 0 || len2 == 0 || (n_pos && !pos))
        return fail(HC_ERR_ARG, "hc_overlap_score_multi: bad argument");
    if (n_pos == 0) return HC_OK;
    std::string b(seq1, len1), q(qual1, len1);
    b.append(seq2, len2);
    q.append(qual2, len2);
    hc_read_desc rd[2];
    memset(rd, 0, sizeof(rd));
    rd[0].seq_off[0] = 0; rd[0].seq_len[0] = len1;
    rd[1].seq_off[0] = len1; rd[1].seq_len[0] = len2;
    int dev = 0;
    cudaGetDevice(&dev);
    hc_store* s = hc_store_create(rd, 2, 2, b.data(), q.data(), dev, 1);
    if (!s) return HC_ERR_CUDA;
    std::vector<hc_candidate> c(n_pos);
    memset(c.data(), 0, n_pos * sizeof(hc_candidate));
    for (uint32_t i = 0; i < n_pos; i++) {
        c[i].idx1 = 0; c[i].idx2 = 1; c[i].pos1 = pos[i]; c[i].ord = '-'; c[i].ori1 = 1; c[i].ori2 = 1; c[i].type1 = 's'; c[i].type2 = 's';
    }
    hc_params pp = *p;
    pp.merge_contigs = -1.0;   // class EDGE <=> score > edge_threshold, nothing else
    std::vector<hc_result> r(n_pos);
    std::vector<hc_edge> e(n_pos);
    std::vector<uint64_t> ni(n_pos);
    uint64_t ne = 0, nn = 0;
    int rc = hc_score_batch(s, &pp, c.data(), n_pos, r.data(), e.data(), n_pos, &ne, ni.data(), n_pos, &nn, nullptr);
    hc_store_destroy(s);
    if (rc != HC_OK) return rc;
    for (uint32_t i = 0; i < n_pos; i++) {
        if (scores) scores[i] = r[i].score;
        if (mismatch_rates) mismatch_rates[i] = r[i].mismatch_rate;
        if (above) above[i] = r[i].cls == HC_CLASS_EDGE;
    }
    return HC_OK;
}

double hc_overlap_score(const char* seq1, uint32_t len1, const char* seq2, uint32_t len2, const char* qual1,
                        const char* qual2, uint32_t pos, const hc_params* p, double* mismatch_rate) {
    double s = -1, mm = 1;
    if (hc_overlap_score_multi(seq1, len1, seq2, len2, qual1, qual2, &pos, 1, p, &s, &mm, nullptr) != HC_OK) return -1;
    if (mismatch_rate) *mismatch_rate = mm;
    return s;
}

}  // extern "C"
