// hc_ingest.h -- internals of hc_ingest.cu that hc_api.cu shares: the id map, its workspace and the device-side
// ingestion of one buffer, so that hc_ingest_score_overlaps can hand the parsed candidates to the scoring pipeline
// without a trip through the host.
#ifndef HC_INGEST_H_
#define HC_INGEST_H_
#include <stdint.h>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"

struct hc_idmap {
    int device;
    uint64_t n;        // reads
    uint64_t mask;     // hash table size - 1 (open addressing, one 16-byte slot {id, index} per entry)
    ulonglong2* slots;
    uint64_t direct_n; // > 0: ids are dense, direct[id] = index for id < direct_n (fits L2 for 1e7 reads)
    uint32_t* direct;
    // grow-only workspace of hc_ingest_overlaps* (one call at a time per handle)
    void* ws[16];
    size_t ws_cap[16];
    cudaEvent_t e0, e1;
    // piece pipeline of the host-buffer entry point: copies in / kernels / copies out on three streams
    cudaStream_t s_main, s_copy, s_out;
    cudaEvent_t ev_in[2], ev_out[2];
};

// workspace slot k of the id map, grown to at least `bytes`
cudaError_t hc_idmap_ws(hc_idmap* m, int k, size_t bytes, void** out);

// Ingestion of text already on the device (slots 0-10 of the workspace).  Outputs are device buffers; returns synchronised
// with `stream`.  Output line numbers start at line_base.
// all_lines: the field rules of the Overlap constructor and the id lookup only -- no self-overlap test, no length /
// percentage pre-filter (p->min_overlap_len, min_overlap_perc and relax_PE_edges are not read).  Every line becomes a
// candidate, in file order; a line without 13 fields (HC_LINE_SKIPPED) is an error line like HC_LINE_ERROR and
// HC_LINE_UNKNOWN_ID, reported in st->first_error_*.  Nothing goes to d_filt.
int hc_ingest_device(const hc_idmap* m, const char* d_text, uint64_t n_bytes, const hc_ingest_params* p, hc_candidate* d_cand,
                     uint64_t* d_cand_line, uint64_t cand_cap, hc_overlap_rec* d_filt, uint64_t* d_filt_line, uint64_t filt_cap,
                     hc_ingest_stats* st, cudaStream_t stream, uint64_t line_base = 0, bool all_lines = false);

// A line that survives the Overlap constructor has 13 fields, five of them one character long (ORD, ORI1, ORI2, TYPE1,
// TYPE2): at least 17 bytes and its newline.  The candidates all_lines can produce from n_bytes of text:
static inline uint64_t hc_ingest_all_cap(uint64_t n_bytes) { return (n_bytes + 1) / 18 + 1; }

// Bytes per piece of a host buffer (32 MB; HC_INGEST_PIECE overrides it), and the cuts of `text` into pieces that end at
// a line end: piece k is [cut[k], cut[k + 1]).  A buffer of at most 1.5 pieces is one piece.
uint64_t hc_ingest_piece_bytes();
std::vector<uint64_t> hc_ingest_cuts(const char* text, uint64_t n_bytes, uint64_t piece);

// A line that reaches an output has 13 fields, i.e. at least 26 bytes with its newline: the records a piece can produce
static inline uint64_t hc_ingest_rec_cap(uint64_t piece_bytes) { return piece_bytes / 26 + 2; }

#endif
