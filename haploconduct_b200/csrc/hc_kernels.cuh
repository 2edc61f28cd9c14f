// hc_kernels.cuh -- kernel-side declarations shared by hc_kernels.cu and hc_api.cu
#ifndef HC_KERNELS_CUH_
#define HC_KERNELS_CUH_

#include <stdint.h>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_layout.h"

#ifndef HC_WARPS_MAX
#define HC_WARPS_MAX 12          // warps per CTA of the lane-chunk kernel
#endif
#ifndef HC_MIN_CTAS
#define HC_MIN_CTAS 2             // ... and resident CTAs per SM the register allocation aims at
#endif
#define HC_LANE_CHUNK 32u        // positions one lane handles per step (two 16-position halves)
#ifndef HC_PARTMAX
#define HC_PARTMAX 512u
#endif
//                            // lane-chunk partials per warp round (x 8 B = 4 KB of shared memory)
#define HC_BIG_CHUNKS 64u        // candidates with >= this many lane-chunks are scored warp-cooperatively
#define HC_WINSLOTS 64u          // 2 windows x 32 candidates
#define HC_VM_WORDS 64u          // tail-mask table of the packed layout (33 used), kept behind the score table
// per-warp scratch: partials + window descriptors (16 B + 8 B per slot) + head bitmap
#define HC_WARP_SCRATCH (HC_PARTMAX * 8u + HC_WINSLOTS * 16u + HC_WINSLOTS * 8u + (HC_PARTMAX / 32u) * 4u)

// class byte written per candidate: HC_CLASS_* in bits 0-1
#define HC_CLS_MASK 3u
#define HC_CLS_BOTH 4u           // every window is above edge_threshold (selects 0.5*(ov1+ov2) vs min, :256-261)
#define HC_CLS_EXACT 8u          // decided by the reference-order pass; hc_tmp32.S holds the exact mean logs

// Scratch record, written for accepted edges only: what the ordered compaction needs to emit hc_edge.
struct hc_tmp32 {
    unsigned long long S[2];     // fixed-point sum of -log p per window, or bits of the exact mean log (HC_CLS_EXACT)
    uint32_t tl[2];              // compared (non-N) positions per window; 0 = window not scored (score 0, mismatch rate 1.0)
    uint32_t mm[2];              // mismatches per window (the rate, an IEEE division, is taken when the edge is emitted)
};

struct hc_kparams {
    // read store planes (one replica)
    const uint8_t* qual;
    const uint32_t* base2;
    const uint32_t* nmask;
    const uint8_t* pk;          // packed layout: code | base << 6 per position (qual/base2/nmask are NULL then)
    const hc_rdesc* rdesc;
    uint32_t packed;
    uint32_t n_reads;
    uint32_t n_single;
    // tables
    const uint32_t* fx_table;   // (ncodes+1)*256 entries
    const double* dbl_table;    // (ncodes+1)^2*2 entries
    uint32_t ncodes;
    uint32_t has_void;
    // batch
    const void* cand;           // hc_candidate[n] (cand_compact == 0), hc_candidate_compact[n] (1), hc_candidate_short[n] (2)
    uint32_t cand_compact;      // or hc_candidate_entry[n] (3) with the three run arrays below
    const uint32_t* run_anchor; // [n_runs] read shared by the candidates of a run
    const uint32_t* run_start;  // [n_runs + 1] first candidate of each run within this batch, run_start[n_runs] = n
    const uint32_t* tile_run;   // [ceil(n / 32)] run that holds candidate 32 * t (hc_tile_runs)
    const unsigned long long* run;   // nullable: running {edges, non-edges} totals of earlier chunks = output base offsets
    uint64_t n;
    hc_tmp32* tmp;
    uint8_t* cls;
    hc_result* per_cand;        // nullable
    uint32_t* flagged;          // candidate indices that need the reference-order pass
    unsigned long long* counters;  // see HC_CNT_*
    // decisions (src/EdgeCalculator.cpp:404-413, thresholds moved into log space on the host)
    double t_edge;              // smallest mean with exp(mean) > edge_threshold
    double t_ov;                // smallest mean with exp(mean) > ov_threshold
    // fixed-point form: S <= c_up * total_len  <=>  surely above;  S > c_dn * total_len  <=>  surely below
    double ce_up, ce_dn, co_up, co_dn;
    double merge_contigs;
    int32_t merge_contigs_sign; // -1 / 0 / +1: with 0 (every driver's default) "mismatch rate <= merge_contigs" is "no mismatch at all"
    uint32_t min_read_len;
    uint32_t zero_above_edge;   // 0 > edge_threshold ?
    uint32_t zero_above_ov;     // 0 > ov_threshold ?
    uint32_t never_edge;        // t_edge > 0: a mean (<= 0) can never reach it
    uint32_t never_ov;
    uint32_t exact_edges;       // HC_FLAG_EXACT_EDGE_SCORES
    uint32_t void_exact;        // hc_tables::void_asymmetric: void hits are decided by the reference-order pass
};

enum {
    HC_CNT_FLAGGED = 0,   // number of entries in flagged[]
    HC_CNT_WINDOWS,
    HC_CNT_POSITIONS,
    HC_CNT_ALGBYTES,
    HC_CNT_ERRORS,        // candidates with invalid indices / ord
    HC_CNT_EDGES,         // written by the compaction
    HC_CNT_NONEDGES,
    HC_CNT_EXACT,
    HC_CNT_N
};

struct hc_launch_cfg {
    int blocks;
    int threads;
    size_t smem;
};

// Kept mode of the compaction (hc_ingest_score_overlaps): the candidates classified edge or non-edge are written out
// themselves, in batch order, and every edge names its kept index (plus the running totals P.run) as `cand`.
struct hc_kept_dev {
    hc_candidate* cand;          // [n] kept candidates of the batch
    uint64_t* line;              // nullable: their line numbers, taken from line_in
    uint8_t* cls;                // [n] their classes (HC_CLASS_EDGE / HC_CLASS_NONEDGE)
    const uint64_t* line_in;     // nullable: line number of every candidate of the batch
    uint32_t* edge_kept;         // [n] scratch: kept index of the batch's k-th edge
};

// host-callable launchers (hc_kernels.cu)
cudaError_t hc_launch_score(const hc_kparams& P, const hc_launch_cfg& cfg, cudaStream_t st);
cudaError_t hc_launch_exact(const hc_kparams& P, cudaStream_t st);
cudaError_t hc_launch_tile_runs(const uint32_t* run_start, uint32_t n_runs, uint32_t* tile_run, cudaStream_t st);
// small_out: d_edges receives hc_edge_small (hc_edge_small_exact with P.exact_edges) records and d_bits one bit per candidate
// of the batch (1 = non-edge overlap) instead of the index list.  kept != NULL (small_out, P.cand holds hc_candidate): kept
// mode, d_edges receives the batch's edges from index 0 and no non-edge list or bit map is written
cudaError_t hc_launch_compact(const hc_kparams& P, hc_edge* d_edges, uint64_t edges_cap, uint64_t* d_nonedge,
                              uint64_t nonedge_cap, uint32_t* d_blockcounts, uint64_t cand_offset, unsigned long long* d_run,
                              cudaStream_t st, int small_out = 0, uint32_t* d_bits = nullptr, const hc_kept_dev* kept = nullptr);
cudaError_t hc_score_occupancy(uint32_t ncodes, int sm_count, size_t smem_per_sm, hc_launch_cfg* cfg);
uint32_t hc_compact_blocks(uint64_t n);

#endif
