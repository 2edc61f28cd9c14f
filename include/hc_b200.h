/* hc_b200.h -- C ABI of the B200-native overlap-edge scoring path.
 *
 * This is the drop-in boundary underneath the reference's two C++ interfaces
 *   EdgeCalculator::construct_edges()/process_overlaps()   src/EdgeCalculator.h:44-63, src/EdgeCalculator.cpp:389-423
 *   FastqStorage                                           src/FastqStorage.h:58-98
 * (FindNextOverlaps entry points are declared further down when that row is built).
 * Plain pointers and sizes only; no C++ or torch types cross it.  The library owns all device
 * memory; the caller owns every host buffer; no pointer handed out by the library outlives the
 * object it belongs to.  There is NO CPU fallback: every compute entry point fails with
 * HC_ERR_CUDA when no sm_100 device is usable.
 *
 * Error convention: every int-returning function returns HC_OK (0) or a negative HC_ERR_*;
 * hc_last_error() returns a thread-local, human readable description of the last failure.
 * The reference prints to stderr and exit(1)s (src/Overlap.h:109-163, src/EdgeCalculator.cpp:662-665);
 * the host shim above this ABI maps a negative return to exactly that behaviour.
 */
#ifndef HC_B200_H_
#define HC_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HC_OK              0
#define HC_ERR_ARG        -1   /* bad argument (NULL pointer, index out of range, bad ord/ori) */
#define HC_ERR_CUDA       -2   /* CUDA runtime/driver failure or no usable device */
#define HC_ERR_NOMEM      -3   /* host or device allocation failed */
#define HC_ERR_INPUT      -4   /* input the reference would exit(1)/assert on (invalid base, empty read, bad quality) */
#define HC_ERR_CAPACITY   -5   /* caller-provided output buffer too small */

/* ------------------------------------------------------------------------------------------
 * Read store  (replaces FastqStorage, src/FastqStorage.h:58-98 + src/Read.h:30-31)
 *
 * Reads are addressed by their dense index in the reference's m_read_vec order: all single-end
 * reads first, then all pairs (src/FastqStorage.h:88-97).  A single read has one sequence
 * (mate slot 0); a paired read has two (mate slots 0 and 1 = /1 and /2, stored exactly as read,
 * i.e. NOT reverse-complemented -- src/FastqStorage.cpp:196-205).
 * ------------------------------------------------------------------------------------------ */
typedef struct hc_store hc_store;

typedef struct {
    uint64_t seq_off[2];   /* byte offset of mate 0 / mate 1 in the bases[] and quals[] blobs        */
    uint32_t seq_len[2];   /* length of mate 0 / mate 1; seq_len[1] == 0  <=>  single-end read       */
} hc_read_desc;

/* Pack n_reads reads (n_single singles first, then pairs) into the device-resident SoA store
 * and replicate it on `n_devices` devices starting at `first_device` (pass n_devices = 1 and the
 * rank's local device in a one-process-per-GPU launch).
 *   bases: ASCII, upper-case A/C/G/T/N only (anything else -> HC_ERR_INPUT; the reference asserts
 *          on it in EdgeCalculator::score, src/EdgeCalculator.cpp:29-30).
 *   quals: raw FASTQ quality characters; Q = c - 33 must lie in [0, 93]
 *          (src/EdgeCalculator.cpp:93-96; outside it the reference's asserts :61,:97 fire).
 * Returns NULL on failure (see hc_last_error()). */
hc_store* hc_store_create(const hc_read_desc* reads, uint64_t n_reads, uint64_t n_single,
                          const char* bases, const char* quals,
                          int first_device, int n_devices);
/* The same store from the text of the FASTQ files, FastqStorage::FastqStorage (src/FastqStorage.h:58-98,
 * src/FastqStorage.cpp:42-235) on the device: at most 4 * max_reads lines per file (:46), records of four lines,
 * header = '@' + id token (first white-space delimited token, strtoul(.., 0), src/Types.h:99-102), single-end
 * sequences upper-cased (:123), mates taken verbatim (:196-197) with equal header tokens (:189-192); singles
 * first, then pairs.  Records the reference exits on give NULL + HC_ERR_INPUT; so does -- a deliberate deviation -- a
 * record whose sequence and quality lines differ in length, which the reference loads and only trips over when the
 * read is scored (src/EdgeCalculator.cpp:93-98).  Only the first file's header is tested for '@' (:181).  Pass NULL / 0 for an absent
 * file.  The id_correspondence table of the reference (--IDs) is not applied: use hc_store_create for that. */
hc_store* hc_store_create_fastq(const char* singles, uint64_t singles_bytes, const char* paired1, uint64_t paired1_bytes,
                                const char* paired2, uint64_t paired2_bytes, uint64_t max_reads,
                                int first_device, int n_devices);
/* The same from the files themselves, streamed through a ring of pinned buffers (the host never holds a file; the
 * reference reads every line into a vector of strings first, src/FastqStorage.cpp:42-57).  NULL, "" or "None" = absent
 * file; a file that cannot be opened gives NULL + HC_ERR_INPUT ("Unable to open fastq file", :54-56). */
hc_store* hc_store_create_fastq_files(const char* singles_path, const char* paired1_path, const char* paired2_path,
                                      uint64_t max_reads, int first_device, int n_devices);
/* ids (n_reads) and mate lengths (2 * n_reads) of a store built by hc_store_create_fastq*; either may be NULL */
int       hc_store_read_ids(const hc_store* s, uint64_t* ids, uint32_t* mate_lengths);
void      hc_store_destroy(hc_store* s);

uint64_t  hc_store_n_reads(const hc_store* s);
uint64_t  hc_store_n_single(const hc_store* s);
int       hc_store_n_devices(const hc_store* s);
/* bytes of device memory one replica occupies: both strands of every sequence, either packed
 * (<= 63 distinct quality values: one byte per base = 6-bit quality code | 2-bit base) or as three
 * planes (quality code bytes, 2-bit bases, 1-bit N mask) */
uint64_t  hc_store_device_bytes(const hc_store* s);
/* number of distinct quality values present (decides the packed vs three-plane layout) */
int       hc_store_quality_alphabet(const hc_store* s);

/* ------------------------------------------------------------------------------------------
 * Candidates  (replaces Overlap, src/Overlap.h:20-59; one record = one line of the 13-column
 * overlaps file after the host has mapped read IDs to dense indices)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint32_t idx1, idx2;     /* dense read indices of ID1 / ID2                                   */
    uint32_t pos1, pos2;     /* POS1 / POS2 ("-" -> 0, src/Overlap.h:55-59)                        */
    uint32_t len1, len2;     /* LEN1 / LEN2                                                        */
    uint8_t  perc1, perc2;   /* PERC1 / PERC2                                                      */
    uint8_t  ord;            /* '1', '2' or '-'                                                    */
    uint8_t  ori1, ori2;     /* 1 = '+', 0 = '-'                                                   */
    uint8_t  type1, type2;   /* 's' / 'p' as written in the file (host pre-filter only)           */
    uint8_t  reserved;       /* must be 0                                                          */
} hc_candidate;              /* 32 bytes */

/* Compact 16-byte form of the same record: only what the device reads (read types come from the
 * store).  Halves the host->device traffic of hc_score_batch_compact; LEN/PERC/TYPE stay with the
 * caller, who finds them again through hc_edge.cand. */
typedef struct {
    uint32_t idx1, idx2;
    uint32_t pos1_flags;     /* POS1 in bits 0-27; bit 28: ORI1 is '+'; bit 29: ORI2 is '+'; bits 30-31: ORD 0 '-', 1 '1', 2 '2' */
    uint32_t pos2;
} hc_candidate_compact;      /* 16 bytes */

/* 12-byte form for stores whose reads are shorter than 16384 bases (every short-read stage): three quarters of
 * the compact record again.  Positions that do not fit must use hc_candidate_compact. */
typedef struct {
    uint32_t idx1, idx2;
    uint32_t pos;            /* POS1 in bits 0-13, POS2 in bits 14-27; bit 28: ORI1 is '+'; bit 29: ORI2 is '+'; bits 30-31: ORD 0 '-', 1 '1', 2 '2' */
} hc_candidate_short;        /* 12 bytes */

/* Scoring parameters = the ProgramSettings fields the path reads (src/Types.h:19-67). */
typedef struct {
    double   edge_threshold;   /* src/EdgeCalculator.cpp:404 and per half :256,:294,:355 */
    double   ov_threshold;     /* :410 */
    double   merge_contigs;    /* :407 */
    double   mismatch;         /* :49  */
    uint32_t min_read_len;     /* :82  */
    uint32_t flags;            /* HC_FLAG_* */
} hc_params;

#define HC_FLAG_EXACT_EDGE_SCORES 1u  /* re-sum every accepted edge in the reference's order (slower) */

/* class of a candidate, src/EdgeCalculator.cpp:404-413 */
#define HC_CLASS_DISCARD 0
#define HC_CLASS_EDGE    1
#define HC_CLASS_NONEDGE 2

/* per-window status */
#define HC_WIN_UNUSED     0   /* S-S candidates have one window only                      */
#define HC_WIN_SCORED     1
#define HC_WIN_POS_OOR    2   /* pos >= len(A)            -> score 0, src/EdgeCalculator.cpp:76-79  */
#define HC_WIN_SHORT      3   /* a read < min_read_len    -> score 0, :82-84                          */
#define HC_WIN_VOID       4   /* some p < ps.mismatch     -> score 0, :49-51,:125-127                 */
#define HC_WIN_EMPTY      5   /* no non-N compared base   -> score 0, :129-131                        */

/* Optional per-candidate record (debug / parity); every field is what the reference's Edge holds
 * after compute_overlap (src/EdgeCalculator.cpp:143-385) plus the integer counts behind it. */
typedef struct {
    double   score;            /* Edge::score                                                       */
    double   mismatch_rate;    /* Edge::mismatch_rate                                               */
    int32_t  pos3, pos4;       /* Edge::pos3 / pos4 (src/EdgeCalculator.cpp:222,262-263,300-301,361-372) */
    uint32_t mismatches[2];    /* mismatch_count of window 1 / 2 (src/EdgeCalculator.cpp:105)       */
    uint32_t compared[2];      /* total_len of window 1 / 2 (non-N compared positions, :104)        */
    uint8_t  cls;              /* HC_CLASS_*                                                        */
    uint8_t  status[2];        /* HC_WIN_* per window                                               */
    uint8_t  exact;            /* 1 if the reference-order re-summation decided this candidate      */
    uint32_t indel_count;      /* always 0: the reference compares the windows gaplessly, position by position
                                  (src/EdgeCalculator.cpp:106-117); indels exist only upstream, in the candidate
                                  producers (OLA != OLB of rust-overlaps, CIGAR I/D of sam2overlaps.py)            */
} hc_result;                   /* 48 bytes */

/* One accepted edge, emitted in INPUT ORDER (= the reference's 1-thread order). */
typedef struct {
    uint64_t cand;             /* index into the candidate array of the call                        */
    double   score;            /* Edge::score, device exp()                                         */
    double   mismatch_rate;
    int32_t  pos3, pos4;
    double   mean_log[2];      /* (1.0/total_len)*total_score per window (src/EdgeCalculator.cpp:137); NaN for a
                                  window that was not scored.  With HC_FLAG_EXACT_EDGE_SCORES these are the
                                  reference's doubles bit for bit, so a host that needs Edge::score
                                  bit-identical to the reference evaluates exp() with its own libm (:138).  */
} hc_edge;                     /* 48 bytes */

/* Small outputs, for a host that keeps its candidate list (every real caller does: the non-edge overlaps are written
 * to nonedge_overlaps.txt from the host's own records, src/EdgeCalculator.cpp:546-555, and an Edge is built from the
 * overlap it came from, :415-422).  What travels back is one BIT per candidate for the non-edge overlaps and a 24-byte
 * record per accepted edge (32 bytes with HC_FLAG_EXACT_EDGE_SCORES) -- a third of the device->host bytes of hc_edge +
 * index lists.  Everything else of hc_edge follows from the candidate:
 *   mismatch_rate = max over the scored windows of (double)(float)mismatches[w] / compared[w]   (0 mismatches: 0.0;
 *                   a window with compared == 0 counts as 1.0; one window only unless HC_EDGE_TWO)          (:132,:254)
 *   score (exact) = HC_EDGE_TWO ? (HC_EDGE_BOTH ? 0.5*(exp(m0)+exp(m1)) : min(exp(m0), exp(m1))) : exp(m0), a window
 *                   with compared == 0 scoring 0                                                             (:138,:256-261)
 *   pos3 / pos4   = hc_edge_extra_pos() below                                                      (:222,:262-263,:300-301,:361-372) */
#define HC_EDGE_BOTH     1u   /* every window is above edge_threshold                                          */
#define HC_EDGE_TWO      2u   /* the candidate has two windows (a paired read is involved)                     */
#define HC_EDGE_EXACT    4u   /* decided / summed in the reference's order                                     */
#define HC_EDGE_OVERFLOW 8u   /* a count does not fit 16 bits (windows of 65536+ positions): use hc_score_batch* */
typedef struct {
    uint32_t cand;             /* index into the candidate array of the call (a call takes fewer than 2^32)    */
    uint16_t mismatches[2];    /* mismatch_count per window (src/EdgeCalculator.cpp:105)                       */
    uint16_t compared[2];      /* total_len per window (:104); 0 = window not scored                           */
    uint32_t flags;            /* HC_EDGE_*                                                                    */
    double   score;            /* Edge::score, device exp()                                                    */
} hc_edge_small;               /* 24 bytes */
typedef struct {
    uint32_t cand;
    uint16_t mismatches[2];
    uint16_t compared[2];
    uint32_t flags;
    double   mean_log[2];      /* (1.0/total_len)*total_score per window, the reference's doubles bit for bit (:137) */
} hc_edge_small_exact;         /* 32 bytes */

/* Edge::pos3 / pos4 of a candidate (size_t arithmetic truncated to int, as the reference's assignments do); host
 * arithmetic.  len1a/len1b: sequence lengths of read 1 (/1, /2; len1b == 0 for a single-end read), likewise read 2. */
void hc_edge_extra_pos(uint32_t pos1, uint32_t pos2, char ord, uint32_t len1a, uint32_t len1b, uint32_t len2a, uint32_t len2b,
                       int32_t* pos3, int32_t* pos4);

typedef struct {
    uint64_t n_candidates;
    uint64_t n_edges;
    uint64_t n_nonedges;
    uint64_t n_exact;          /* candidates re-summed in reference order (threshold-boundary cases) */
    uint64_t n_windows;        /* windows actually compared                                         */
    uint64_t n_positions;      /* sum of window lengths L = min(len(A)-pos, len(B))                 */
    uint64_t algorithmic_bytes;/* sum over candidates of 32 + sum_w(2*ceil(L/4)+2*ceil(L/8)+2L) + 16 */
    float    kernel_ms;        /* device time of the scoring kernels of this call (CUDA events)     */
    float    total_ms;         /* device time of the whole call incl. copies (CUDA events)          */
    uint32_t kernel_launches;  /* kernels launched by this call                                     */
    float    score_kernel_ms;  /* device time of the dominant kernel (hc_score_kernel) alone        */
} hc_batch_stats;

/* Score a batch of HOST candidates: the body of the omp-parallel region of
 * EdgeCalculator::process_overlaps (src/EdgeCalculator.cpp:395-423).
 * The batch is sharded by contiguous index range over the store's devices; outputs are gathered
 * in input order.
 *   per_cand      nullable; if given must hold n records.
 *   edges         must hold *edges_cap records; on return *n_edges are valid.
 *   nonedge_idx   candidate indices classified "non-edge overlap" (:410-413), input order.
 * Returns HC_ERR_CAPACITY (and the required sizes in *n_edges / *n_nonedges) if a buffer is too small. */
/* Host batches are streamed through the device in chunks: the copy of chunk k+1, the kernels of
 * chunk k and the copy-out of chunk k-1 overlap (chunk size: 16 M candidates). */
int hc_score_batch(hc_store* s, const hc_params* p,
                   const hc_candidate* cand, uint64_t n,
                   hc_result* per_cand,
                   hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges,
                   uint64_t* nonedge_idx, uint64_t nonedge_cap, uint64_t* n_nonedges,
                   hc_batch_stats* stats /* nullable */);

/* hc_score_batch on compact candidate records. */
int hc_score_batch_compact(hc_store* s, const hc_params* p,
                           const hc_candidate_compact* cand, uint64_t n,
                           hc_result* per_cand,
                           hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges,
                           uint64_t* nonedge_idx, uint64_t nonedge_cap, uint64_t* n_nonedges,
                           hc_batch_stats* stats /* nullable */);

/* hc_score_batch on 12-byte records (reads shorter than 16384 bases). */
int hc_score_batch_short(hc_store* s, const hc_params* p,
                         const hc_candidate_short* cand, uint64_t n,
                         hc_result* per_cand,
                         hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges,
                         uint64_t* nonedge_idx, uint64_t nonedge_cap, uint64_t* n_nonedges,
                         hc_batch_stats* stats /* nullable */);

/* hc_score_batch on run-encoded 8-byte records.  An overlaps file lists the overlaps of one read one after the other
 * (scripts/sfo2overlaps.py:52 sorts its lines by read; rust-overlaps emits them per read), so consecutive candidates
 * share a read: a RUN is a stretch of consecutive candidates that all contain the read run_anchor[r], as ID1 or as ID2,
 * and each candidate then only names the other read.  Any list can be cut into runs (a run may have length 1; the
 * order of the candidates is not changed).  run_start has n_runs + 1 entries, run_start[0] = 0, run_start[n_runs] = n,
 * strictly increasing.  Needs a store of fewer than 2^31 reads whose reads are shorter than 16384 bases; two thirds of
 * the host->device traffic of hc_score_batch_short.  Results are those of hc_score_batch on the decoded records. */
typedef struct {
    uint32_t other;          /* bits 0-30: dense index of the read that is not the run's anchor; bit 31: the anchor is ID2 */
    uint32_t pos;            /* as hc_candidate_short.pos */
} hc_candidate_entry;        /* 8 bytes */
int hc_score_batch_runs(hc_store* s, const hc_params* p,
                        const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                        const hc_candidate_entry* entries, uint64_t n,
                        hc_result* per_cand,
                        hc_edge* edges, uint64_t edges_cap, uint64_t* n_edges,
                        uint64_t* nonedge_idx, uint64_t nonedge_cap, uint64_t* n_nonedges,
                        hc_batch_stats* stats /* nullable */);

/* hc_score_batch_runs with small outputs: `edges` receives hc_edge_small records (hc_edge_small_exact when
 * p->flags has HC_FLAG_EXACT_EDGE_SCORES), in input order; nonedge_bits must hold ceil(n / 64) words and receives
 * bit (i % 64) of word i / 64 = 1 iff candidate i is a non-edge overlap (:410-413); *n_nonedges = their number. */
int hc_score_batch_runs_small(hc_store* s, const hc_params* p,
                              const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                              const hc_candidate_entry* entries, uint64_t n,
                              void* edges, uint64_t edges_cap, uint64_t* n_edges,
                              uint64_t* nonedge_bits, uint64_t* n_nonedges,
                              hc_batch_stats* stats /* nullable */);
/* The same on 6-byte run-encoded records, for stores of at most 2^25 reads whose reads are shorter than 512 bases (every
 * Illumina read set): the host->device copy of the records is what bounds a call on host buffers, so their size is
 * its speed.  A record is a 48-bit little-endian number: bits 0-24 the other read, 25 "the anchor is ID2", 26 ORI1 is
 * '+', 27 ORI2 is '+', 28-29 ORD (0 '-', 1 '1', 2 '2'), 30-38 POS1, 39-47 POS2. */
typedef struct { uint8_t b[6]; } hc_candidate_entry6;
int hc_score_batch_runs6_small(hc_store* s, const hc_params* p,
                               const uint32_t* run_anchor, const uint64_t* run_start, uint64_t n_runs,
                               const hc_candidate_entry6* entries, uint64_t n,
                               void* edges, uint64_t edges_cap, uint64_t* n_edges,
                               uint64_t* nonedge_bits, uint64_t* n_nonedges,
                               hc_batch_stats* stats /* nullable */);
/* The same on 12-byte records (lists that were not cut into runs). */
int hc_score_batch_short_small(hc_store* s, const hc_params* p,
                               const hc_candidate_short* cand, uint64_t n,
                               void* edges, uint64_t edges_cap, uint64_t* n_edges,
                               uint64_t* nonedge_bits, uint64_t* n_nonedges,
                               hc_batch_stats* stats /* nullable */);

/* Same, but every buffer is DEVICE memory on device `device` (one of the store's devices) and the
 * work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = default stream).
 * d_counts receives {n_edges, n_nonedges, n_exact, n_invalid} as uint64_t[4], where n_invalid counts the
 * candidates with an invalid read index, a self overlap, or a P-P candidate whose ORD is not '1' or '2'
 * (they are classified HC_CLASS_DISCARD).  With stats == NULL such a batch still returns HC_OK, so
 * d_counts[3] is the caller's only sign of them; with stats != NULL the call returns HC_ERR_ARG.
 * Asynchronous unless stats != NULL.
 * Capacities: when edges_cap or nonedge_cap is smaller than the list, the first edges_cap / nonedge_cap
 * records are written and the rest dropped; d_counts still holds the full counts and the call returns
 * HC_OK (unlike the host-buffer calls, which return HC_ERR_CAPACITY).  An output pointer may be NULL when
 * its capacity is 0.
 * Alignment: d_cand must be 16-byte aligned; d_per_cand, d_edges, d_nonedge_idx and d_counts 8-byte
 * aligned (cudaMalloc'ed buffers and whole records inside them are).  Anything else returns HC_ERR_ARG.
 * Ordering: calls on one store (this one, hc_score_batch* and hc_ingest_score_overlaps) share a device
 * workspace; each call's device work waits for the previous call's, whatever streams they use, so a
 * caller needs no synchronisation between them.  This holds for calls made from one host thread;
 * concurrent calls on one store from several host threads are not supported.
 * This is what the throughput benchmark times with inputs resident in HBM, and what a
 * device-side consumer (NCCL gather, GPU FindNextOverlaps) calls. */
int hc_score_batch_device(hc_store* s, int device, void* stream, const hc_params* p,
                          const hc_candidate* d_cand, uint64_t n,
                          hc_result* d_per_cand /* nullable */,
                          hc_edge* d_edges, uint64_t edges_cap,
                          uint64_t* d_nonedge_idx, uint64_t nonedge_cap,
                          uint64_t* d_counts,
                          hc_batch_stats* stats /* nullable; non-NULL makes the call synchronous */);

/* The scoring primitive on its own: EdgeCalculator::overlap_score (src/EdgeCalculator.cpp:67-139),
 * second caller SRBuilder::merge_self_overlap (src/SRBuilder.cpp:872-888).  Sequences are ASCII
 * host strings; runs one window on device 0 of a transient store.  Returns the score, writes the
 * mismatch rate; on error returns -1 and sets hc_last_error(). */
double hc_overlap_score(const char* seq1, uint32_t len1, const char* seq2, uint32_t len2,
                        const char* qual1, const char* qual2, uint32_t pos,
                        const hc_params* p, double* mismatch_rate);

/* The same primitive for many start positions of one sequence pair in ONE device batch -- the
 * access pattern of SRBuilder::merge_self_overlap (src/SRBuilder.cpp:880-888), which slides seq2 over
 * seq1 from pos = len1-15 downwards until score > 0.99.  above[i] (nullable) receives the exact
 * decision "overlap_score(pos[i]) > p->edge_threshold" (decided in the reference's own summation
 * order when the score is within 1e-7 of the threshold), so the caller's loop can test above[i]
 * instead of comparing a device exp() against the threshold. */
int hc_overlap_score_multi(const char* seq1, uint32_t len1, const char* seq2, uint32_t len2,
                           const char* qual1, const char* qual2, const uint32_t* pos, uint32_t n_pos,
                           const hc_params* p, double* scores, double* mismatch_rates, uint8_t* above);

/* Creates the CUDA context of `device` (a few tenths of a second per process).  Optional: every call does it on demand;
 * a host calls this from a second thread while it reads its input files, so that the two overlap. */
int hc_warm_up(int device);

/* Pinned host memory for the host-buffer entry points.  They accept any host memory (pageable buffers are staged through the
 * library's own pinned ring); buffers from here go to the copy engines as they are.  write_combined != 0: write-combined
 * memory, for buffers the host only WRITES front to back (candidate records on their way in) -- reading it back is slow.
 * NULL if the allocation fails. */
void* hc_host_alloc(uint64_t bytes, int write_combined);
void  hc_host_free(void* p);

/* EdgeCalculator::phred_to_prob (src/EdgeCalculator.cpp:59-63), host arithmetic: pow(10, -Q/10.0). */
double hc_phred_to_prob(int phred);

/* Smallest double x with exp(x) > threshold under the host libm (the decision
 * "exp(mean) > threshold" of src/EdgeCalculator.cpp:138,404 is evaluated as "mean >= x" on the device). */
double hc_exp_threshold(double threshold);

/* ------------------------------------------------------------------------------------------
 * FindNextOverlaps (FNO1): SRBuilder::findNextOverlaps, src/FindNextOverlaps.cpp:890-958 with
 * updateOverlap :25-327, findCliqueIndex :331-347, computeOverlapData :351-565.
 *
 * After an iteration has merged reads into super-reads, every edge / removed edge / non-edge overlap
 * (u, v) of the old graph is re-expressed between the NEW reads: the unmerged read itself, or every
 * super-read containing u resp. v, by index arithmetic on the sub-read positions.  Per unordered
 * pair of new reads the FIRST derivation in processing order wins, even if it then fails
 * (:84-97 precede :115-118).  The host keeps the graph walk that produces the edge stream
 * (:605-631, :635-697, :816-887); hc_fno1_text / hc_fno3_text below also build the text of
 * overlaps.txt on the device.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint32_t u, v;            /* old vertices                                                      */
    int32_t  pos1, pos2;      /* Edge::pos1 / pos2                                                 */
    int32_t  perc, len1, len2;/* Edge::overlap_perc / overlap_len1 / overlap_len2                  */
    uint8_t  ord;             /* '1', '2' or '-'                                                   */
    uint8_t  ori1, ori2;      /* Edge::ori1 / ori2 (1 = NORMAL)                                    */
    uint8_t  nonedge;         /* Edge::score == 0: non-edge overlap, ORI taken against the vertex labels (:34-37) */
} hc_fno_edge;                /* 32 bytes */

typedef struct {
    uint64_t id;              /* new read id: super-read id, or nodes_to_new_IDs[v] of an unmerged vertex */
    uint32_t len1, len2;      /* sequence length(s); len2 == 0 <=> single-end                      */
} hc_fno_read;                /* 16 bytes */

typedef struct { int32_t index1, index2, startpos1, startpos2; } hc_fno_subread;   /* SubreadInfo, src/Types.h:77-82 */

typedef struct {
    uint64_t n_vertices;
    const uint8_t*        visited;       /* [V] SRBuilder::visited                                   */
    const uint8_t*        label;         /* [V] OverlapGraph::getOrientation(v)                      */
    const hc_fno_read*    vertex_read;   /* [V] original read of the vertex: new id (if !visited) + lengths */
    const uint64_t*       sr_off;        /* [V+1] CSR of nodes_to_SR (:898-913)                       */
    const uint32_t*       sr_idx;        /* [sr_off[V]] super-read index per entry, list order        */
    const hc_fno_subread* sr_sub;        /* [sr_off[V]] get_subread_info(v) of that super-read        */
    uint64_t n_superreads;
    const hc_fno_read*    superread;     /* [n_superreads]                                            */
    uint8_t resolve_orientations;        /* ProgramSettings::resolve_orientations                     */
    uint8_t no_inclusions;               /* ProgramSettings::no_inclusions (drop perc == 100)          */
} hc_fno_input;

typedef struct {
    uint64_t id1, id2;        /* ID1 / ID2 of the emitted overlap line                             */
    int32_t  pos1, pos2, perc, len1, len2;
    uint8_t  ord, ori1, ori2, type1, type2;   /* characters: '1'/'2'/'-', '+'/'-', 's'/'p'          */
    uint8_t  reserved[3];
    int32_t  perc2;           /* PERC2: always 0 from hc_fno1 (the reference prints a literal 0, :136), set by hc_fno3 */
} hc_fno_overlap;             /* 48 bytes; line = id1 id2 pos1 pos2 ord ori1 ori2 perc perc2 len1 len2 type1 type2 */

/* Derives the next-iteration overlaps on `device`.  `out` receives the successful derivations in
 * processing order (edge order, then super-read list order); the caller formats, sorts and
 * de-duplicates the lines like the reference's std::set<std::string> (:918,:946-948).
 * Returns HC_ERR_CAPACITY (required size in *n_out) if out_cap is too small. */
int hc_fno1(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges,
            hc_fno_overlap* out, uint64_t out_cap, uint64_t* n_out, int device);

/* The same derivation with 24-byte result records (half the device->host bytes of hc_fno_overlap; the caller formats the
 * line from them): ids below 2^32, positions and lengths below 2^24, percentages below 256.  Returns HC_ERR_ARG (and
 * hc_last_error() says so) when a value of the result does not fit -- hc_fno1 / hc_fno3 take any input.
 *   pos1_perc  = pos1 | perc  << 24      pos2_perc2 = pos2 | perc2 << 24
 *   len1_flags = len1 | flags << 24      flags: bits 0-1 ord (0 '-', 1 '1', 2 '2'), bit 2 ori1 == '+', bit 3 ori2 == '+',
 *   len2                                        bit 4 type1 == 'p', bit 5 type2 == 'p'                                  */
typedef struct { uint32_t id1, id2, pos1_perc, pos2_perc2, len1_flags, len2; } hc_fno_overlap_small;   /* 24 bytes */
#define HC_FNO_SMALL_ORD(f)   (((f) & 3u) == 1u ? '1' : (((f) & 3u) == 2u ? '2' : '-'))
#define HC_FNO_SMALL_ORI1(f)  (((f) & 4u) ? '+' : '-')
#define HC_FNO_SMALL_ORI2(f)  (((f) & 8u) ? '+' : '-')
#define HC_FNO_SMALL_TYPE1(f) (((f) & 16u) ? 'p' : 's')
#define HC_FNO_SMALL_TYPE2(f) (((f) & 32u) ? 'p' : 's')

int hc_fno1_small(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges,
                  hc_fno_overlap_small* out, uint64_t out_cap, uint64_t* n_out, int device);

/* FindNextOverlaps3: SRBuilder::findNextOverlaps3 / nodeDictApproach / deduceOverlap,
 * src/FindNextOverlaps3.cpp:20-406.  Two new reads that share an ORIGINAL read overlap; the overlap
 * is deduced from the position of that original read inside both (OriginalIndex::index1/2,
 * src/Types.h:84-91).  Originals are visited in the iteration order of the reference's
 * std::unordered_map (:101) -- the host passes them in that order -- and per pair of new reads the
 * first original wins (:116-121).  Output = discovery order, not sorted (:139-166); entries the
 * reference drops (len1 <= 0, or perc == 100 under no_inclusions, :157-165) are not emitted. */
typedef struct { int32_t index1, index2; } hc_fno3_pos;

int hc_fno3(uint64_t n_originals, const uint64_t* off /* [n_originals+1] */, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos,
            uint64_t n_reads, const hc_fno_read* reads /* super-reads and trivial reads */, int no_inclusions,
            hc_fno_overlap* out, uint64_t out_cap, uint64_t* n_out, int device);
int hc_fno3_small(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos,
                  uint64_t n_reads, const hc_fno_read* reads, int no_inclusions,
                  hc_fno_overlap_small* out, uint64_t out_cap, uint64_t* n_out, int device);

/* The reference's overlaps.txt itself: the lines of the records hc_fno1 derives, formatted as
 * "%lu\t%lu\t%d\t%d\t%c\t%c\t%c\t%d\t%d\t%d\t%d\t%c\t%c" (src/FindNextOverlaps.cpp:122-148), unique and in
 * std::string (byte) order like the reference's std::set<std::string> (:918,:946-948); every line ends in '\n'.
 * *n_bytes / *n_lines receive the size of the file and its line count, *n_records (nullable) the records before
 * de-duplication.  HC_ERR_CAPACITY (sizes still written) if text_cap < *n_bytes; text may be NULL when text_cap is 0.
 * The arguments are checked as by hc_fno1; HC_ERR_ARG also for 2^32 or more records.  Sorting, de-duplication and
 * formatting run on the device; the text is the only thing copied back. */
int hc_fno1_text(const hc_fno_input* in, const hc_fno_edge* edges, uint64_t n_edges,
                 char* text, uint64_t text_cap, uint64_t* n_bytes, uint64_t* n_lines, uint64_t* n_records, int device);

/* hc_fno1_text for the stream head ++ N ++ tail, where N -- the non-edge overlaps the reference re-reads from
 * nonedge_overlaps.txt (reconsiderNonedgeOverlaps, src/FindNextOverlaps.cpp:635-697, --optimize=false) -- is parsed
 * from nonedge_text on m's device and never leaves it.  Same text, *n_bytes, *n_lines, *n_records and HC_ERR_CAPACITY
 * protocol as hc_fno1_text on that stream (text may be NULL with text_cap 0).
 *   head          head[0 .. n_adjacency) = the adj_out lists in vertex order (u non-decreasing), then branching_edges
 *   nonedge_text  host memory (pageable or pinned, any alignment): lines trimmed of outer tabs / spaces, split on tabs,
 *                 put through the Overlap constructor (src/Overlap.h:39-73) -- no self-overlap test, no pre-filter.
 *                 Line k becomes {u, v} = the store indices of ID1 / ID2 in m (vertex i is read i), POS1, POS2, ORD,
 *                 ORI1/2 == '+', perc = Overlap::get_perc(), LEN1, LEN2, nonedge = 1; an unterminated last line counts.
 *                 The line is dropped when checkEdge(v1, v2, true) > 0 (:694-696): the first adjacency entry (v1, v2),
 *                 or only if there is none the first (v2, v1), has nonedge == 0.  This reads a non-edge flag as
 *                 "score == 0" and any other entry as "score > 0": no adjacency edge may have a negative score.
 *                 Branching and tail edges are not in the graph and are not consulted.
 *   tail          the edges derived through removed inclusion vertices (:816-887)
 * A line the reference's loop would die on or leave undefined -- not 13 fields (an empty line too), a field the
 * constructor rejects, a trailing '\r', an id not in m -- gives HC_ERR_INPUT with the first such line in
 * stats->first_error_* and nothing written; the caller runs its own loop for the reference's message.
 * A call after HC_ERR_CAPACITY does all the work again, the parse of nonedge_text included: size text generously.
 * HC_ERR_ARG (checked before any device work): m on another device or m's read count != in->n_vertices,
 * n_adjacency > n_head, adjacency u decreasing, and every check of hc_fno1_text on head and tail. */
typedef struct {
    uint64_t n_lines;             /* lines of nonedge_text                                                  */
    uint64_t n_nonedges;          /* of them, lines whose pair is not an edge: the stream's middle segment   */
    uint64_t n_stream;            /* n_head + n_nonedges + n_tail                                           */
    uint64_t first_error_line;    /* 0-based, ~0 if none; and its byte offset / length in nonedge_text      */
    uint64_t first_error_offset, first_error_length;
    uint32_t first_error_status;  /* HC_LINE_SKIPPED (not 13 fields, empty), HC_LINE_ERROR, HC_LINE_UNKNOWN_ID */
    float    device_ms;           /* the stream built in HBM: head copy, pieces copied / parsed / probed / compacted, tail */
} hc_fno_nonedge_stats;           /* 56 bytes */

struct hc_idmap;                  /* hc_idmap_create, below */
int hc_fno1_text_nonedges(const hc_fno_input* in, const struct hc_idmap* m,
                          const hc_fno_edge* head, uint64_t n_head, uint64_t n_adjacency,
                          const char* nonedge_text, uint64_t nonedge_bytes,
                          const hc_fno_edge* tail, uint64_t n_tail,
                          char* text, uint64_t text_cap, uint64_t* n_bytes, uint64_t* n_lines, uint64_t* n_records,
                          hc_fno_nonedge_stats* stats, int device);

/* The same for hc_fno3: the lines in discovery order, not sorted, not de-duplicated (src/FindNextOverlaps3.cpp:139-166). */
int hc_fno3_text(uint64_t n_originals, const uint64_t* off, const uint32_t* sr_idx, const hc_fno3_pos* sr_pos,
                 uint64_t n_reads, const hc_fno_read* reads, int no_inclusions,
                 char* text, uint64_t text_cap, uint64_t* n_bytes, uint64_t* n_lines, int device);

/* ------------------------------------------------------------------------------------------
 * Duplicate-edge resolution of the graph insert (first "next" row, SURVEY 8f):
 * EdgeCalculator::process_overlaps, serial section, src/EdgeCalculator.cpp:429-545.
 *
 * The reference inserts accepted edges one by one; an edge whose (unordered vertex pair, "both
 * orientations equal" flag) already has an edge replaces it iff  score >= existing score, ties
 * broken by longer overlap, lower mismatch rate, smaller vertex1, ori1 true, ori2 true, smaller
 * pos1, smaller pos2, and -- everything equal -- the later one (:470-521).  That fold keeps, per
 * key, the LAST maximum of a lexicographic order, so it is a per-key arg-max: here one atomicCAS
 * loop per edge on a hash table.  The final adjacency lists are the survivors in input order
 * (a replaced edge is erased and the new one appended, :522-531), so the host only appends
 * `winner` edges, in order, to adj_out[vertex1].
 * Records carry the fields AFTER the reference's normalisation (:443-448: if pos1 == 0 and
 * v1 > v2, the reads are swapped and pos3/pos4 negated).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint32_t vertex1, vertex2;
    double   score, mismatch_rate;
    int32_t  pos1, pos2, pos3;
    int32_t  overlap_len;      /* Edge::get_len(0) = len1 + len2                                   */
    int32_t  perc;
    uint8_t  ori1, ori2;
    uint8_t  reserved[2];
} hc_dedup_edge;               /* 48 bytes */

/* winner[i] = 1 iff edge i is in the graph after all n edges have been inserted in order.
 * inclusions (nullable, n_vertices bytes, caller-zeroed) receives OverlapGraph::inclusions as the
 * reference sets it under ignore_inclusions (:459-468, decided by the FIRST edge of each key).
 * counts[0] = dup_count increment (:472,:537,:544), counts[1] = inclusion_count increment (:449-451). */
int hc_dedup_edges(const hc_dedup_edge* edges, uint64_t n, int ignore_inclusions, uint8_t* winner,
                   uint8_t* inclusions, uint64_t n_vertices, uint64_t counts[2], int device);

/* ------------------------------------------------------------------------------------------
 * Adjacency lists of the overlap graph (second half of the first "next" row, SURVEY 8f):
 * OverlapGraph::addEdge in insertion order (src/OverlapGraph.cpp:94-101) and OverlapGraph::sortEdges
 * (:722-764): every adjacency list ordered by Edge::get_nonoverlap_len() (src/Edge.h:58-63:
 * len(read1) + len(read2) - 2 * overlap_len, unsigned), then vertex2; adj_in rebuilt by walking the
 * sorted lists vertex by vertex.
 *
 * edges[i] with keep[i] != 0 (all if keep is NULL) are grouped by vertex1:
 *   out_off[v] .. out_off[v+1]   range of vertex v's list in out_perm            (out_off: n_vertices + 1)
 *   out_perm[p]                  index into edges[] of the p-th edge; inside a list: input order (sort == 0)
 *                                or (nonoverlap_len, vertex2, input order) (sort != 0)
 *   in_off / in_src              (optional) adj_in: in_src[in_off[w] ..] = the vertex1 of every edge into w, in the
 *                                order the walk over the lists meets them (:752-763)
 *   ties[v]                      (optional, n_vertices) 1 if a list of more than 16 edges holds two edges with equal
 *                                (nonoverlap_len, vertex2): std::sort does not say in which order it leaves them --
 *                                the host mirror sorts such a list with std::sort itself
 * ------------------------------------------------------------------------------------------ */
typedef struct { uint32_t vertex1, vertex2, nonoverlap_len, reserved; } hc_adj_edge;   /* 16 bytes */

int hc_build_adjacency(const hc_adj_edge* edges, uint64_t n, const uint8_t* keep, uint64_t n_vertices, int sort,
                       uint64_t* out_off, uint32_t* out_perm, uint64_t* in_off, uint32_t* in_src, uint8_t* ties,
                       uint64_t* n_kept, int device);

/* SRBuilder::calcSubreadInfo (src/SRBuilder.cpp:536-595) for many super-reads at once (third "next" row, SURVEY 8f:
 * the sub-read index records that hc_fno1 reads as sr_sub).  pos[] / vertex[] hold the pos_list / sorted_vertices lists of all
 * super-reads; a problem names its list 1 [begin1, end1), its list 2 [begin2, end2) (empty for a single-end super-read) and
 * what consensus() returned for the two sequences (trim_pos2 = -1: single-end).  For every entry k of a list 1:
 * first[k] = 1 if it is the first entry of its vertex in that list, and then info[k] = the SubreadInfo the reference's map
 * holds for that vertex ({index1, index2, startpos1, startpos2}, index2 = startpos2 = -1 when nothing sets them); entries of
 * a list 2 and repeated vertices get first[k] = 0.  List-1 ranges of different problems must not overlap. */
typedef struct {
    uint64_t begin1, end1, begin2, end2;
    int32_t  trim_pos1, trim_pos2;
} hc_subread_problem;            /* 40 bytes */
int hc_subread_info(const hc_subread_problem* problems, uint64_t n_problems, const int32_t* pos, const uint32_t* vertex,
                    uint64_t n_entries, hc_fno_subread* info, uint8_t* first, int device);

/* ------------------------------------------------------------------------------------------
 * Candidate ingestion (second "next" row, SURVEY 8f): the text loop of
 * EdgeCalculator::construct_edges, src/EdgeCalculator.cpp:581-645, on the device.
 *
 * Input is a buffer of complete lines of the 13-column overlaps file.  Every line is trimmed of
 * outer tabs/spaces (:584), split on tabs (or, with allow_spaces, on runs of tabs/spaces, :585-587),
 * must have 13 fields (:598-603), goes through the Overlap constructor (src/Overlap.h:39-73: ids by
 * strtoul(s, NULL, 0), numbers by atoi, "-" in POS2 zeroes POS2/PERC2/LEN2, ORD/ORI/TYPE stripped of
 * spaces when longer than one character), the self-overlap test (:605-607) and the length /
 * percentage pre-filter (:612-635).  Ids are mapped to store indices through hc_idmap =
 * FastqStorage::m_ID_to_index (src/FastqStorage.h:90-93, first insertion wins).
 * Outputs, both in file order: the candidates that reach process_overlaps (ready for
 * hc_score_batch*) and the overlaps the pre-filter sends to nonedge_overlaps.txt (:633-635).
 * A line the reference would exit(1)/assert/throw on is reported in stats (first such line);
 * nothing is guessed.
 * ------------------------------------------------------------------------------------------ */
#define HC_LINE_SCORE      1   /* passes the pre-filter -> process_overlaps                           */
#define HC_LINE_NONEDGE    2   /* fails the length tests -> nonedge_overlaps.txt (:633-635)           */
#define HC_LINE_DROPPED    3   /* self overlap (:605-607) or inside the band with perc < min_overlap_perc */
#define HC_LINE_SKIPPED    4   /* != 13 fields: "incorrect overlap; skipping" (:598-603)              */
#define HC_LINE_ERROR      5   /* a check of src/Overlap.h:107-165 fails: the reference exits/aborts  */
#define HC_LINE_UNKNOWN_ID 6   /* would be scored but an id is not in the store (map::at throws, :170-171) */

typedef struct hc_idmap hc_idmap;
/* ids[i] = read_id of store read i (m_read_vec order). */
hc_idmap* hc_idmap_create(const uint64_t* ids, uint64_t n_reads, int device);
void      hc_idmap_destroy(hc_idmap* m);

typedef struct {
    uint64_t max_overlaps;       /* ProgramSettings::max_overlaps: lines read at most (:581)           */
    uint32_t min_overlap_len;    /* :612,:618,:626                                                     */
    uint32_t min_overlap_perc;   /* :614,:621,:629                                                     */
    uint8_t  relax_PE_edges;     /* :626                                                               */
    uint8_t  allow_spaces;       /* :585                                                               */
    uint8_t  reserved[6];
} hc_ingest_params;              /* 24 bytes */

typedef struct {                 /* an Overlap as Overlap::get_overlap_line prints it (src/Overlap.h:234-237) */
    uint64_t id1, id2;
    uint32_t pos1, pos2, perc1, perc2, len1, len2;
    uint8_t  ord, ori1, ori2, type1, type2;   /* the characters of the file */
    uint8_t  reserved[3];
} hc_overlap_rec;                /* 48 bytes */

typedef struct {
    uint64_t n_lines;            /* lines read (clamped to max_overlaps)                               */
    uint64_t n_scored, n_filtered, n_skipped, n_dropped;
    uint64_t first_error_line;   /* 0-based line of the first HC_LINE_ERROR / HC_LINE_UNKNOWN_ID, ~0 if none */
    uint64_t first_error_offset; /* its byte offset and length in the buffer                           */
    uint64_t first_error_length;
    uint32_t first_error_status;
    float    device_ms;          /* newline index + parse + compaction kernels                         */
} hc_ingest_stats;               /* 72 bytes */

/* Host buffers.  cand_line / filtered_line (nullable) receive the 0-based line number of every
 * output record.  Returns HC_ERR_CAPACITY with the required sizes in stats->n_scored /
 * stats->n_filtered when a buffer is too small.  Lines after the first error line are still
 * classified; the caller decides (the host mirror dies with the reference's message). */
int hc_ingest_overlaps(const hc_idmap* m, const char* text, uint64_t n_bytes, const hc_ingest_params* p,
                       hc_candidate* cand, uint64_t* cand_line, uint64_t cand_cap,
                       hc_overlap_rec* filtered, uint64_t* filtered_line, uint64_t filtered_cap,
                       hc_ingest_stats* stats);
/* The same on DEVICE buffers of the id map's device; d_text may have any alignment (16-byte aligned
 * is fastest).  The candidates can be handed to hc_score_batch_device without leaving HBM. */
int hc_ingest_overlaps_device(const hc_idmap* m, void* stream, const char* d_text, uint64_t n_bytes,
                              const hc_ingest_params* p, hc_candidate* d_cand, uint64_t* d_cand_line, uint64_t cand_cap,
                              hc_overlap_rec* d_filtered, uint64_t* d_filtered_line, uint64_t filtered_cap,
                              hc_ingest_stats* stats);

/* Ingestion and scoring in one call: the text goes to the device, is parsed there and its candidates are scored there;
 * only the candidates scored as edges or non-edges, their edge records and the pre-filtered overlaps come back.  This is
 * EdgeCalculator::construct_edges (src/EdgeCalculator.cpp:561-666) up to the graph insert, for a host that keeps no
 * candidate list of its own.
 * Inputs
 *   text          host memory (pageable or pinned) holding complete lines, as for hc_ingest_overlaps.  Parsing, the
 *                 pre-filter, max_overlaps and the id lookup are those of hc_ingest_overlaps with `ip`; scoring is that of
 *                 hc_score_batch* with `p`, applied to the candidates the parser passes on.  Full hc_candidate records are
 *                 scored: no limit on read lengths or on the number of reads beyond the store's own.
 *   The work runs on the id map's device, where the store must have a replica (else HC_ERR_ARG).
 * Outputs, all in file order
 *   kept[k], kept_line[k], kept_class[k]   the scored candidates classified HC_CLASS_EDGE or HC_CLASS_NONEDGE, their 0-based
 *                 line in the text and their class.  Candidates classified HC_CLASS_DISCARD never leave the device.
 *   edges         hc_edge_small records (hc_edge_small_exact under HC_FLAG_EXACT_EDGE_SCORES); `cand` is the index of the
 *                 edge's candidate in kept[].  Every other field equals what hc_score_batch_short_small returns for the same
 *                 candidate, HC_EDGE_OVERFLOW included, so an Edge follows from kept[cand] as described above hc_edge_small.
 *   filtered, filtered_line   as from hc_ingest_overlaps.
 *   kept_line and filtered_line may be NULL; an output pointer may be NULL when its capacity is 0.
 * Errors
 *   Lines after the first error line are still classified and scored; stats->ingest.first_error_* reports that line and the
 *   caller decides (as for hc_ingest_overlaps).  A candidate the scorer rejects (e.g. a P-P candidate with ORD '-', an index
 *   outside the store) gives HC_ERR_ARG with the message of hc_score_batch*.  2^32 or more kept candidates give HC_ERR_ARG
 *   (cand is 32 bits).  A capacity that is too small gives HC_ERR_CAPACITY with the required sizes in stats->n_kept,
 *   stats->score.n_edges and stats->ingest.n_filtered. */
typedef struct {
    hc_ingest_stats ingest;    /* what hc_ingest_overlaps reports for the same text and parameters                      */
    hc_batch_stats  score;     /* what hc_score_batch* reports for the candidates the ingestion passed on (times: summed
                                  over the pieces the text is cut into; total_ms: the whole call)                          */
    uint64_t        n_kept;    /* scored candidates classified edge or non-edge (score.n_edges + score.n_nonedges)         */
} hc_ingest_score_stats;       /* 152 bytes */

int hc_ingest_score_overlaps(hc_store* s, const hc_idmap* m, const char* text, uint64_t n_bytes,
                             const hc_ingest_params* ip, const hc_params* p,
                             hc_candidate* kept, uint64_t* kept_line /* nullable */, uint8_t* kept_class, uint64_t kept_cap,
                             void* edges, uint64_t edges_cap,
                             hc_overlap_rec* filtered, uint64_t* filtered_line /* nullable */, uint64_t filtered_cap,
                             hc_ingest_score_stats* stats);

/* ------------------------------------------------------------------------------------------
 * Super-read consensus (third "next" row, SURVEY 8f): SRBuilder::consensus + consensus_pos,
 * src/SRBuilder.cpp:297-522, for many pile-ups at once.
 *
 * A problem is what SRBuilder::sort_vertices hands over (:688-700): sequences of the store (a read's
 * mate, forward or reverse-complemented) with their start columns, ascending from 0, the length of
 * the consensus, and the two flags.  For every column the device adds the reference's log10 terms
 * of the covering bases in list order (:318-341, addends from a host-libm table, so the four
 * scores are bit-identical) and evaluates :349-401 (pow / log10 / round) with its own libm while
 * bounding the error; columns within that bound of a decision come back with their scores and are
 * decided by the host libm, the same the reference links.  The host part of the call then walks
 * the columns like :447-513 (support trimming under error_correction, give-up cases).  Results
 * are the reference's strings.  Output regions of different problems must not overlap; the call owns the whole of
 * cons_seq / cons_qual [0, out_bytes): bytes between the regions of two problems are overwritten too (with zeros).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint32_t read;            /* store index of the read                                            */
    uint8_t  mate;            /* 0 / 1                                                              */
    uint8_t  rc;              /* 1: reverse complement, qualities reversed (src/Read.h:172-201)     */
    uint16_t reserved;
    int32_t  pos;             /* start column (pos_list), ascending within a problem                */
} hc_cons_seq;                /* 12 bytes */

typedef struct {
    uint64_t seq_begin, seq_end;   /* this problem's entries in the hc_cons_seq array               */
    uint64_t out_offset;           /* where its characters start in cons_seq / cons_qual; total_len bytes are reserved */
    int32_t  total_len;            /* consensus length handed to consensus() (:406)                 */
    uint8_t  subreads_needed, error_correction;
    uint8_t  reserved[2];
} hc_cons_problem;            /* 32 bytes */

typedef struct {
    int32_t ret;              /* consensus()'s return value: trim_pos, 0 (gave up) or -1 (not enough support) */
    int32_t length;           /* characters written at out_offset (0 where the reference clears the strings)  */
} hc_cons_result;

/* min_clique_size / min_qual = ProgramSettings::min_clique_size / min_qual (SRBuilder::minQual, src/SRBuilder.h:89).
 * out_bytes = size of cons_seq and of cons_qual. */
int hc_consensus(hc_store* s, const hc_cons_problem* problems, uint64_t n_problems, const hc_cons_seq* seqs, uint64_t n_seqs,
                 uint32_t min_clique_size, double min_qual, char* cons_seq, char* cons_qual, uint64_t out_bytes,
                 hc_cons_result* results);

int         hc_device_count(void);
const char* hc_last_error(void);
const char* hc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HC_B200_H_ */
