// hc_ingest.cu -- candidate ingestion on the device: the text loop of EdgeCalculator::construct_edges
// (src/EdgeCalculator.cpp:581-645) with the Overlap constructor (src/Overlap.h:39-73) and the
// id -> index map of FastqStorage (src/FastqStorage.h:90-93, used at src/EdgeCalculator.cpp:164-171).
// See hc_b200.h for the contract.  Byte work, HBM/L2-bound: newline index (count -> scan -> mark),
// one thread per line for the field parse, ordered compaction (count -> scan -> scatter).
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_ingest.h"

void hc_set_last_error(const char* msg);   // hc_api.cu

cudaError_t hc_idmap_ws(hc_idmap* m, int k, size_t bytes, void** out) {
    if (bytes > m->ws_cap[k]) {
        cudaFree(m->ws[k]);
        m->ws[k] = nullptr;
        m->ws_cap[k] = 0;
        const size_t want = bytes + bytes / 4 + 256;
        const cudaError_t e = cudaMalloc(&m->ws[k], want);
        if (e != cudaSuccess) return e;
        m->ws_cap[k] = want;
    }
    *out = m->ws[k];
    return cudaSuccess;
}

#include "hc_text.cuh"
#include "hc_stage.h"
#include "hc_scan.cuh"

namespace {

constexpr int LINES_PER_BLOCK = 1024; // lines per block in the compaction passes
constexpr u64 EMPTY = ~0ull;

struct IngTmp {            // one parsed line
    hc_overlap_rec r;
    uint32_t idx1, idx2;
};

__device__ __forceinline__ hc_candidate to_candidate(const IngTmp& t) {
    hc_candidate c;
    c.idx1 = t.idx1; c.idx2 = t.idx2; c.pos1 = t.r.pos1; c.pos2 = t.r.pos2; c.len1 = t.r.len1; c.len2 = t.r.len2;
    c.perc1 = (uint8_t)t.r.perc1; c.perc2 = (uint8_t)t.r.perc2; c.ord = t.r.ord;
    c.ori1 = t.r.ori1 == '+'; c.ori2 = t.r.ori2 == '+'; c.type1 = t.r.type1; c.type2 = t.r.type2; c.reserved = 0;
    return c;
}

__device__ __forceinline__ u64 hash64(u64 k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

// ---- id map ------------------------------------------------------------------------------------
struct IdMapDev {
    const ulonglong2* slots;
    u64 mask;
    const uint32_t* direct;
    u64 direct_n;
};

__global__ void idmap_insert(const u64* ids, u64 n, ulonglong2* slots, u64 mask) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64 key = ids[i];
        u64 h = hash64(key) & mask;
        while (true) {
            const u64 prev = atomicCAS(&slots[h].x, EMPTY, key);
            if (prev == EMPTY || prev == key) { atomicMin(&slots[h].y, i); break; }   // std::map::insert keeps the first
            h = (h + 1) & mask;
        }
    }
}

__global__ void idmap_insert_direct(const u64* ids, u64 n, uint32_t* direct) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) atomicMin(&direct[ids[i]], (uint32_t)i);
}

__device__ __forceinline__ uint32_t idmap_find(const IdMapDev& M, u64 key) {
    if (M.direct_n) return key < M.direct_n ? __ldg(M.direct + key) : 0xffffffffu;
    if (key == EMPTY) return 0xffffffffu;
    u64 h = hash64(key) & M.mask;
    while (true) {
        const ulonglong2 e = M.slots[h];
        if (e.x == key) return (uint32_t)e.y;
        if (e.x == EMPTY) return 0xffffffffu;
        h = (h + 1) & M.mask;
    }
}

// (unsigned int)atoi(s) = (unsigned int)(int)strtol(s, NULL, 10) on the field [p, q)
__device__ uint32_t dev_atoi(const char* t, u64 p, u64 q) {
    while (p < q && c_isspace(t[p])) p++;
    bool neg = false;
    if (p < q && (t[p] == '+' || t[p] == '-')) { neg = t[p] == '-'; p++; }
    u64 v = 0;
    bool ovf = false;
    const u64 cutoff = 0x7fffffffffffffffull / 10ull;            // LONG_MAX / 10 = |LONG_MIN| / 10
    const u64 cutlim = neg ? 8ull : 7ull;                        // |LONG_MIN| % 10, LONG_MAX % 10
    for (; p < q; p++) {
        const char c = t[p];
        if (c < '0' || c > '9') break;
        const u64 d = (u64)(c - '0');
        if (v > cutoff || (v == cutoff && d > cutlim)) ovf = true;
        else if (!ovf) v = v * 10ull + d;
    }
    long long r;
    if (ovf) r = neg ? (long long)0x8000000000000000ull : 0x7fffffffffffffffll;
    else r = neg ? -(long long)v : (long long)v;
    return (uint32_t)(int)r;
}

// one-character fields: ORI / ORD strip ' ' when the length is not 1 (src/Overlap.h:115-118,127-130), TYPE strips
// '\n', '\t', ' ' (:152-156); the result must be one character (assert) -- returns 0 when it is not
__device__ char dev_char_field(const char* t, u64 p, u64 q, bool is_type) {
    if (q - p == 1) return t[p];
    char out = 0;
    int cnt = 0;
    for (; p < q; p++) {
        const char c = t[p];
        const bool strip = c == ' ' || (is_type && (c == '\n' || c == '\t'));
        if (!strip) { out = c; cnt++; }
    }
    return cnt == 1 ? out : (char)0;
}

struct IngDev {
    const char* text;
    u64 n_bytes;
    const u64* line_start;
    u64 n_lines;           // lines considered (already clamped to max_overlaps)
    u64 n_newlines;
    IdMapDev ids;
    uint32_t min_overlap_len, min_overlap_perc;
    int relax, allow_spaces;
};

// src/EdgeCalculator.cpp:583-635 for line i; fills tmp and returns the status.  ALL: every line that survives the
// Overlap constructor is looked up and returned as HC_LINE_SCORE -- no self-overlap test, no pre-filter (the loop of
// src/FindNextOverlaps.cpp:635-697 over nonedge_overlaps.txt applies neither)
template <bool ALL>
__device__ uint8_t parse_line(const IngDev& D, u64 i, IngTmp& o) {
    const char* t = D.text;
    u64 s = D.line_start[i];
    u64 e = i < D.n_newlines ? D.line_start[i + 1] - 1 : D.n_bytes;    // without the '\n'
    while (s < e && (t[s] == '\t' || t[s] == ' ')) s++;                // trim_if(is_any_of("\t ")), :584
    while (e > s && (t[e - 1] == '\t' || t[e - 1] == ' ')) e--;
    if (s == e) return HC_LINE_SKIPPED;                                // no token at all
    u64 id1 = 0, id2 = 0;
    uint32_t num[6] = {0, 0, 0, 0, 0, 0};       // pos1 pos2 perc1 perc2 len1 len2
    char ch[5] = {0, 0, 0, 0, 0};               // ord ori1 ori2 type1 type2
    bool dash3 = false;
    uint32_t nf = 0;
    u64 p = s;
    while (true) {
        u64 q = p;
        if (D.allow_spaces) while (q < e && t[q] != '\t' && t[q] != ' ') q++;
        else while (q < e && t[q] != '\t') q++;
        switch (nf) {
            case 0: id1 = dev_strtoul0(t, p, q); break;
            case 1: id2 = dev_strtoul0(t, p, q); break;
            case 2: num[0] = dev_atoi(t, p, q); break;
            case 3: num[1] = dev_atoi(t, p, q); dash3 = (q - p == 1) && t[p] == '-'; break;
            case 4: ch[0] = dev_char_field(t, p, q, false); break;
            case 5: ch[1] = dev_char_field(t, p, q, false); break;
            case 6: ch[2] = dev_char_field(t, p, q, false); break;
            case 7: num[2] = dev_atoi(t, p, q); break;
            case 8: num[3] = dev_atoi(t, p, q); break;
            case 9: num[4] = dev_atoi(t, p, q); break;
            case 10: num[5] = dev_atoi(t, p, q); break;
            case 11: ch[3] = dev_char_field(t, p, q, true); break;
            case 12: ch[4] = dev_char_field(t, p, q, true); break;
            default: break;
        }
        nf++;
        if (q >= e) break;
        p = q + 1;
        if (D.allow_spaces) while (p < e && (t[p] == '\t' || t[p] == ' ')) p++;   // token_compress_on
    }
    if (nf != 13) return HC_LINE_SKIPPED;                              // :598-603
    if (dash3) { num[1] = 0; num[3] = 0; num[5] = 0; }                 // src/Overlap.h:55-59
    // the constructor's checks (:60-72); any failure ends the reference run
    bool bad = (int)num[0] < 0 || (int)num[1] < 0;                                         // check_pos
    bad |= (ch[1] != '+' && ch[1] != '-') || (ch[2] != '+' && ch[2] != '-');               // check_ori
    bad |= (int)num[2] < 0 || (int)num[2] > 100 || (int)num[3] < 0 || (int)num[3] > 100;   // check_perc
    bad |= (int)num[4] < 0 || (int)num[5] < 0;                                             // check_len
    bad |= (ch[3] != 's' && ch[3] != 'p') || (ch[4] != 's' && ch[4] != 'p');               // check_type
    if (!bad) {                                                                            // check_ord
        if (ch[3] == 's' || ch[4] == 's') bad = ch[0] != '-';
        else bad = ch[0] != '1' && ch[0] != '2';
    }
    if (bad) return HC_LINE_ERROR;
    o.r.id1 = id1; o.r.id2 = id2;
    o.r.pos1 = num[0]; o.r.pos2 = num[1]; o.r.perc1 = num[2]; o.r.perc2 = num[3]; o.r.len1 = num[4]; o.r.len2 = num[5];
    o.r.ord = (uint8_t)ch[0]; o.r.ori1 = (uint8_t)ch[1]; o.r.ori2 = (uint8_t)ch[2]; o.r.type1 = (uint8_t)ch[3]; o.r.type2 = (uint8_t)ch[4];
    o.r.reserved[0] = o.r.reserved[1] = o.r.reserved[2] = 0;
    o.idx1 = o.idx2 = 0xffffffffu;
    if (!ALL) {
        if (id1 == id2) return HC_LINE_DROPPED;                            // :605-607
        const uint32_t perc = num[3] > 0 ? (uint32_t)(0.5 * (double)(num[2] + num[3])) : num[2];   // Overlap::get_perc, :203-210
        const bool any_p = ch[3] == 'p' || ch[4] == 'p';
        const double half = 0.5 * (double)D.min_overlap_len;
        bool in_band;
        if (num[4] >= D.min_overlap_len && !any_p) in_band = true;                                      // :612-617
        else if ((double)num[4] >= half && (double)num[5] >= half && any_p) in_band = true;             // :618-624
        else in_band = D.relax && (uint32_t)(num[4] + num[5]) >= D.min_overlap_len && any_p;            // :626-632
        if (!in_band) return HC_LINE_NONEDGE;                                                           // :633-635
        if (perc < D.min_overlap_perc) return HC_LINE_DROPPED;
    }
    o.idx1 = idmap_find(D.ids, id1);
    o.idx2 = idmap_find(D.ids, id2);
    if (o.idx1 == 0xffffffffu || o.idx2 == 0xffffffffu) return HC_LINE_UNKNOWN_ID;                  // map::at throws, :170-171
    return HC_LINE_SCORE;
}

__global__ void __launch_bounds__(256) ing_parse(IngDev D, hc_candidate* tmp_c, hc_overlap_rec* tmp_f, uint8_t* status, u64* first_error) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D.n_lines) return;
    IngTmp o;
    const uint8_t st = parse_line<false>(D, i, o);
    status[i] = st;
    if (st == HC_LINE_SCORE) tmp_c[i] = to_candidate(o);      // only the record a line needs is written
    else if (st == HC_LINE_NONEDGE) tmp_f[i] = o.r;
    if (st == HC_LINE_ERROR || st == HC_LINE_UNKNOWN_ID) atomicMin(first_error, i);
}

// every line a candidate; anything else (also a line without 13 fields) is an error line
__global__ void __launch_bounds__(256) ing_parse_all(IngDev D, hc_candidate* tmp_c, uint8_t* status, u64* first_error) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D.n_lines) return;
    IngTmp o;
    const uint8_t st = parse_line<true>(D, i, o);
    status[i] = st;
    if (st == HC_LINE_SCORE) tmp_c[i] = to_candidate(o);
    else atomicMin(first_error, i);
}

// per block of LINES_PER_BLOCK lines: number of scored and of filtered lines
__global__ void __launch_bounds__(LINES_PER_BLOCK) ing_count(const uint8_t* status, u64 n, uint32_t* cnt_s, uint32_t* cnt_f,
                                                             u64* by_status) {
    const u64 i = (u64)blockIdx.x * LINES_PER_BLOCK + threadIdx.x;
    const uint8_t st = i < n ? status[i] : 0;
    const int a = __syncthreads_count(st == HC_LINE_SCORE);
    const int b = __syncthreads_count(st == HC_LINE_NONEDGE);
    const int c = __syncthreads_count(st == HC_LINE_SKIPPED);
    const int d = __syncthreads_count(st == HC_LINE_DROPPED);
    if (threadIdx.x == 0) {
        cnt_s[blockIdx.x] = (uint32_t)a;
        cnt_f[blockIdx.x] = (uint32_t)b;
        if (c) atomicAdd(&by_status[0], (u64)c);
        if (d) atomicAdd(&by_status[1], (u64)d);
    }
}

__global__ void __launch_bounds__(LINES_PER_BLOCK) ing_scatter(const uint8_t* status, const hc_candidate* tmp_c, const hc_overlap_rec* tmp_f, u64 n, const u64* off_s,
                                                               const u64* off_f, hc_candidate* cand, u64* cand_line,
                                                               hc_overlap_rec* filt, u64* filt_line, u64 line_base) {
    __shared__ uint32_t ws[32], wf[32];
    const u64 i = (u64)blockIdx.x * LINES_PER_BLOCK + threadIdx.x;
    const uint8_t st = i < n ? status[i] : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t bs = __ballot_sync(0xffffffffu, st == HC_LINE_SCORE), bf = __ballot_sync(0xffffffffu, st == HC_LINE_NONEDGE);
    if (lane == 0) { ws[warp] = __popc(bs); wf[warp] = __popc(bf); }
    __syncthreads();
    uint32_t ps = 0, pf = 0;
    for (int w = 0; w < warp; w++) { ps += ws[w]; pf += wf[w]; }
    const uint32_t lt = (1u << lane) - 1u;
    if (st == HC_LINE_SCORE) {
        const u64 k = off_s[blockIdx.x] + ps + __popc(bs & lt);
        cand[k] = tmp_c[i];
        if (cand_line) cand_line[k] = line_base + i;
    } else if (st == HC_LINE_NONEDGE) {
        const u64 k = off_f[blockIdx.x] + pf + __popc(bf & lt);
        filt[k] = tmp_f[i];
        if (filt_line) filt_line[k] = line_base + i;
    }
}

}  // namespace

#define ICU(call)                                                                            \
    do {                                                                                     \
        cudaError_t _e = (call);                                                             \
        if (_e != cudaSuccess) {                                                             \
            hc_set_last_error((std::string(#call) + ": " + cudaGetErrorString(_e)).c_str()); \
            rc = HC_ERR_CUDA;                                                                \
            goto done;                                                                       \
        }                                                                                    \
    } while (0)

extern "C" void hc_idmap_destroy(hc_idmap* m);

extern "C" hc_idmap* hc_idmap_create(const uint64_t* ids, uint64_t n_reads, int device) {
    if (n_reads && !ids) { hc_set_last_error("hc_idmap_create: NULL ids"); return nullptr; }
    if (n_reads >= 0xffffffffull) { hc_set_last_error("hc_idmap_create: too many reads"); return nullptr; }
    hc_idmap* m = new hc_idmap();
    m->device = device; m->n = n_reads; m->slots = nullptr; m->direct = nullptr; m->direct_n = 0; m->mask = 0;
    memset(m->ws, 0, sizeof(m->ws)); memset(m->ws_cap, 0, sizeof(m->ws_cap));
    m->e0 = m->e1 = nullptr;
    m->s_main = m->s_copy = m->s_out = nullptr;
    m->ev_in[0] = m->ev_in[1] = m->ev_out[0] = m->ev_out[1] = nullptr;
    u64 max_id = 0;
    for (u64 i = 0; i < n_reads; i++) max_id = std::max<u64>(max_id, ids[i]);
    if (n_reads && max_id == ~0ull) {   // the hash slots use this value as "empty" (strtoul yields it for "-1" or an overflowing header)
        hc_set_last_error("hc_idmap_create: read id 18446744073709551615 (ULONG_MAX) is not supported");
        delete m;
        return nullptr;
    }
    const bool dense = n_reads > 0 && max_id < 4 * n_reads + 1024;     // rename_fas.py numbers the reads 0..n-1
    int rc = HC_OK;
    u64* d_ids = nullptr;
    const int blocks = (int)std::min<u64>((n_reads + 255) / 256 + 1, 148 * 16);
    ICU(cudaSetDevice(device));
    if (n_reads) {
        ICU(cudaMalloc(&d_ids, n_reads * sizeof(u64)));
        ICU(cudaMemcpy(d_ids, ids, n_reads * sizeof(u64), cudaMemcpyHostToDevice));
    }
    if (dense) {
        m->direct_n = max_id + 1;
        ICU(cudaMalloc(&m->direct, m->direct_n * sizeof(uint32_t)));
        ICU(cudaMemset(m->direct, 0xff, m->direct_n * sizeof(uint32_t)));
        idmap_insert_direct<<<blocks, 256>>>(d_ids, n_reads, m->direct);
    } else {
        u64 cap = 64;
        while (cap < 2 * n_reads + 2) cap <<= 1;
        m->mask = cap - 1;
        ICU(cudaMalloc(&m->slots, cap * sizeof(ulonglong2)));
        ICU(cudaMemset(m->slots, 0xff, cap * sizeof(ulonglong2)));
        if (n_reads) idmap_insert<<<blocks, 256>>>(d_ids, n_reads, m->slots, m->mask);
    }
    ICU(cudaGetLastError());
    ICU(cudaDeviceSynchronize());
    ICU(cudaEventCreate(&m->e0));
    ICU(cudaEventCreate(&m->e1));
    ICU(cudaStreamCreateWithFlags(&m->s_main, cudaStreamNonBlocking));
    ICU(cudaStreamCreateWithFlags(&m->s_copy, cudaStreamNonBlocking));
    ICU(cudaStreamCreateWithFlags(&m->s_out, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) {
        ICU(cudaEventCreateWithFlags(&m->ev_in[k], cudaEventDisableTiming));
        ICU(cudaEventCreateWithFlags(&m->ev_out[k], cudaEventDisableTiming));
    }
done:
    cudaFree(d_ids);
    if (rc != HC_OK) { hc_idmap_destroy(m); return nullptr; }
    return m;
}

extern "C" void hc_idmap_destroy(hc_idmap* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaFree(m->slots);
    cudaFree(m->direct);
    for (int k = 0; k < 16; k++) cudaFree(m->ws[k]);
    if (m->e0) cudaEventDestroy(m->e0);
    if (m->e1) cudaEventDestroy(m->e1);
    for (int k = 0; k < 2; k++) { if (m->ev_in[k]) cudaEventDestroy(m->ev_in[k]); if (m->ev_out[k]) cudaEventDestroy(m->ev_out[k]); }
    if (m->s_main) cudaStreamDestroy(m->s_main);
    if (m->s_copy) cudaStreamDestroy(m->s_copy);
    if (m->s_out) cudaStreamDestroy(m->s_out);
    delete m;
}

// Device-side core: text already on the device.  Outputs are device buffers; counts[0..1] land in host memory.
int hc_ingest_device(const hc_idmap* cm, const char* d_text, uint64_t n_bytes, const hc_ingest_params* p, hc_candidate* d_cand,
                     uint64_t* d_cand_line, uint64_t cand_cap, hc_overlap_rec* d_filt, uint64_t* d_filt_line, uint64_t filt_cap,
                     hc_ingest_stats* st, cudaStream_t stream, uint64_t line_base, bool all_lines) {
    hc_idmap* m = const_cast<hc_idmap*>(cm);     // the workspace is the only thing a call changes
    int rc = HC_OK;
    const u64 n_tiles = (n_bytes + TILE - 1) / TILE;
    uint32_t *d_tcnt = nullptr, *d_cs = nullptr, *d_cf = nullptr;
    u64 *d_toff = nullptr, *d_tot = nullptr, *d_ls = nullptr, *d_os = nullptr, *d_of = nullptr, *d_misc = nullptr;
    hc_candidate* d_tmp_c = nullptr;
    hc_overlap_rec* d_tmp_f = nullptr;
    uint8_t* d_status = nullptr;
    u64 n_nl = 0, n_lines = 0, n_blocks = 0, misc[3] = {0, 0, EMPTY}, tot_s = 0, tot_f = 0;
    char last = '\n';
    IngDev D;
    memset(st, 0, sizeof(*st));
    st->first_error_line = EMPTY;
    if (n_bytes == 0) return HC_OK;
    ICU(hc_idmap_ws(m, 0, n_tiles * sizeof(uint32_t), (void**)&d_tcnt));
    ICU(hc_idmap_ws(m, 1, n_tiles * sizeof(u64), (void**)&d_toff));
    ICU(hc_idmap_ws(m, 2, (8 + hc_scan::blocks_for(n_tiles)) * sizeof(u64), (void**)&d_tot));
    d_misc = d_tot + 2;
    ICU(cudaEventRecord(m->e0, stream));
    nl_count<<<(unsigned)n_tiles, 256, 0, stream>>>(d_text, n_bytes, d_tcnt);
    hc_scan::exclusive_u32(d_tcnt, n_tiles, d_toff, d_tot, d_tot + 8, stream);
    ICU(cudaMemcpyAsync(&n_nl, d_tot, sizeof(u64), cudaMemcpyDeviceToHost, stream));
    ICU(cudaMemcpyAsync(&last, d_text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, stream));
    ICU(cudaStreamSynchronize(stream));
    n_lines = n_nl + (last != '\n' ? 1 : 0);          // getline also returns an unterminated last line
    ICU(hc_idmap_ws(m, 3, (n_nl + 2) * sizeof(u64), (void**)&d_ls));
    ICU(cudaMemsetAsync(d_ls, 0, sizeof(u64), stream));
    nl_mark<<<(unsigned)n_tiles, 256, 0, stream>>>(d_text, n_bytes, d_toff, d_ls);
    if (n_lines > p->max_overlaps) n_lines = p->max_overlaps;   // while (getline(...) && i < max_overlaps), :581
    st->n_lines = n_lines;
    if (n_lines == 0) { ICU(cudaStreamSynchronize(stream)); goto done; }
    n_blocks = (n_lines + LINES_PER_BLOCK - 1) / LINES_PER_BLOCK;
    ICU(hc_idmap_ws(m, 4, n_lines * sizeof(hc_candidate), (void**)&d_tmp_c));
    if (!all_lines) ICU(hc_idmap_ws(m, 5, n_lines * sizeof(hc_overlap_rec), (void**)&d_tmp_f));   // all_lines files no line as a non-edge
    ICU(hc_idmap_ws(m, 6, n_lines, (void**)&d_status));
    ICU(hc_idmap_ws(m, 7, n_blocks * sizeof(uint32_t), (void**)&d_cs));
    ICU(hc_idmap_ws(m, 8, n_blocks * sizeof(uint32_t), (void**)&d_cf));
    ICU(hc_idmap_ws(m, 9, n_blocks * sizeof(u64), (void**)&d_os));
    ICU(hc_idmap_ws(m, 10, n_blocks * sizeof(u64), (void**)&d_of));
    ICU(cudaMemcpyAsync(d_misc, misc, sizeof(misc), cudaMemcpyHostToDevice, stream));
    D.text = d_text; D.n_bytes = n_bytes; D.line_start = d_ls; D.n_lines = n_lines; D.n_newlines = n_nl;
    D.ids.slots = m->slots; D.ids.mask = m->mask; D.ids.direct = m->direct; D.ids.direct_n = m->direct_n;
    D.min_overlap_len = p->min_overlap_len; D.min_overlap_perc = p->min_overlap_perc; D.relax = p->relax_PE_edges != 0;
    D.allow_spaces = p->allow_spaces != 0;
    if (all_lines) ing_parse_all<<<(unsigned)((n_lines + 255) / 256), 256, 0, stream>>>(D, d_tmp_c, d_status, d_misc + 2);
    else ing_parse<<<(unsigned)((n_lines + 255) / 256), 256, 0, stream>>>(D, d_tmp_c, d_tmp_f, d_status, d_misc + 2);
    ing_count<<<(unsigned)n_blocks, LINES_PER_BLOCK, 0, stream>>>(d_status, n_lines, d_cs, d_cf, d_misc);
    scan_counts<<<1, 1024, 0, stream>>>(d_cs, n_blocks, d_os, d_tot);
    scan_counts<<<1, 1024, 0, stream>>>(d_cf, n_blocks, d_of, d_tot + 1);
    ICU(cudaMemcpyAsync(misc, d_misc, sizeof(misc), cudaMemcpyDeviceToHost, stream));
    ICU(cudaMemcpyAsync(&tot_s, d_tot, sizeof(u64), cudaMemcpyDeviceToHost, stream));
    ICU(cudaMemcpyAsync(&tot_f, d_tot + 1, sizeof(u64), cudaMemcpyDeviceToHost, stream));
    ICU(cudaStreamSynchronize(stream));
    st->n_scored = tot_s; st->n_filtered = tot_f; st->n_skipped = misc[0]; st->n_dropped = misc[1];
    st->first_error_line = misc[2];
    if (misc[2] != EMPTY) {
        uint8_t es = 0;
        u64 off[2] = {0, 0};
        ICU(cudaMemcpy(&es, d_status + misc[2], 1, cudaMemcpyDeviceToHost));
        ICU(cudaMemcpy(off, d_ls + misc[2], (misc[2] < n_nl ? 2 : 1) * sizeof(u64), cudaMemcpyDeviceToHost));
        st->first_error_status = es;
        st->first_error_offset = off[0];
        st->first_error_length = (misc[2] < n_nl ? off[1] - 1 : n_bytes) - off[0];
    }
    if (tot_s > cand_cap || tot_f > filt_cap) {
        hc_set_last_error("hc_ingest_overlaps: output buffer too small (required sizes returned in stats)");
        rc = HC_ERR_CAPACITY;
        goto done;
    }
    ing_scatter<<<(unsigned)n_blocks, LINES_PER_BLOCK, 0, stream>>>(d_status, d_tmp_c, d_tmp_f, n_lines, d_os, d_of, d_cand,
                                                                    reinterpret_cast<u64*>(d_cand_line), d_filt,
                                                                    reinterpret_cast<u64*>(d_filt_line), line_base);
    ICU(cudaEventRecord(m->e1, stream));
    ICU(cudaStreamSynchronize(stream));
    ICU(cudaGetLastError());
    ICU(cudaEventElapsedTime(&st->device_ms, m->e0, m->e1));
done:
    return rc;
}

extern "C" int hc_ingest_overlaps_device(const hc_idmap* m, void* stream, const char* d_text, uint64_t n_bytes,
                                         const hc_ingest_params* p, hc_candidate* d_cand, uint64_t* d_cand_line, uint64_t cand_cap,
                                         hc_overlap_rec* d_filtered, uint64_t* d_filtered_line, uint64_t filtered_cap,
                                         hc_ingest_stats* stats) {
    if (!m || !p || !stats || (n_bytes && !d_text)) { hc_set_last_error("hc_ingest_overlaps_device: NULL argument"); return HC_ERR_ARG; }
    if (cudaSetDevice(m->device) != cudaSuccess) { hc_set_last_error("hc_ingest_overlaps_device: cudaSetDevice failed"); return HC_ERR_CUDA; }
    return hc_ingest_device(m, d_text, n_bytes, p, d_cand, d_cand_line, cand_cap, d_filtered, d_filtered_line, filtered_cap, stats,
                         (cudaStream_t)stream);
}

uint64_t hc_ingest_piece_bytes() {
    u64 piece = 32ull << 20;
    if (const char* e = getenv("HC_INGEST_PIECE")) { const u64 v = strtoull(e, nullptr, 10); if (v) piece = v; }   // tests
    return piece;
}

std::vector<uint64_t> hc_ingest_cuts(const char* text, uint64_t n_bytes, uint64_t piece) {
    std::vector<uint64_t> cut(1, 0);
    if (n_bytes <= piece + piece / 2) { if (n_bytes) cut.push_back(n_bytes); return cut; }
    while (cut.back() < n_bytes) {
        u64 end = cut.back() + piece;
        if (end >= n_bytes) end = n_bytes;
        else {
            const void* nl = memrchr(text + cut.back(), '\n', end - cut.back());
            if (nl) end = (u64)((const char*)nl - text) + 1;
            else {   // a line longer than a piece: extend to its end
                const void* fw = memchr(text + end, '\n', n_bytes - end);
                end = fw ? (u64)((const char*)fw - text) + 1 : n_bytes;
            }
        }
        cut.push_back(end);
    }
    return cut;
}

// Large buffers are cut into pieces that end at a line end; the copy in of piece i + 1 and the copy out of piece i - 1
// overlap the kernels of piece i (three streams, two buffer sets).  hc_ingest_rec_cap bounds the records a piece can
// produce without counting its lines first.
static int ingest_pipelined(hc_idmap* m, const char* text, u64 n_bytes, const hc_ingest_params* p, hc_candidate* cand,
                            uint64_t* cand_line, u64 cand_cap, hc_overlap_rec* filtered, uint64_t* filtered_line, u64 filtered_cap,
                            hc_ingest_stats* stats, u64 piece) {
    int rc = HC_OK;
    const std::vector<uint64_t> cut = hc_ingest_cuts(text, n_bytes, piece);
    const size_t n_pieces = cut.size() - 1;
    u64 max_piece = 0;
    for (size_t i = 0; i < n_pieces; i++) max_piece = std::max<u64>(max_piece, cut[i + 1] - cut[i]);
    const u64 rec_cap = hc_ingest_rec_cap(max_piece);
    const u64 tbytes = (max_piece + 16 + 255) & ~255ull;
    char* d_text = nullptr;
    hc_candidate* d_cand = nullptr;
    hc_overlap_rec* d_filt = nullptr;
    uint64_t *d_cl = nullptr, *d_fl = nullptr;
    u64 lines = 0, ns = 0, nf = 0;
    bool overflow = false;
    hc_ingest_params pp = *p;
    ICU(hc_idmap_ws(m, 11, 2 * tbytes, (void**)&d_text));
    ICU(hc_idmap_ws(m, 12, 2 * rec_cap * sizeof(hc_candidate), (void**)&d_cand));
    ICU(hc_idmap_ws(m, 13, 2 * rec_cap * sizeof(hc_overlap_rec), (void**)&d_filt));
    if (cand_line) ICU(hc_idmap_ws(m, 14, 2 * rec_cap * sizeof(u64), (void**)&d_cl));
    if (filtered_line) ICU(hc_idmap_ws(m, 15, 2 * rec_cap * sizeof(u64), (void**)&d_fl));
    // pageable text / result buffers (a file read into memory, a std::vector) go through the pinned ring of hc_stage.cu,
    // copied by several host threads; pinned ones are handed to the copy engine as they are
    ICU(hc_copy_h2d_on(d_text, text, cut[1] - cut[0], m->s_copy));
    ICU(cudaEventRecord(m->ev_in[0], m->s_copy));
    for (size_t i = 0; i < n_pieces && lines < p->max_overlaps; i++) {
        const int b = (int)(i & 1);
        if (i + 1 < n_pieces) {   // buffer (i+1)&1 was read by piece i-1, whose kernels have completed (ingest_device returns synchronised)
            ICU(hc_copy_h2d_on(d_text + (size_t)(b ^ 1) * tbytes, text + cut[i + 1], cut[i + 2] - cut[i + 1], m->s_copy));
            ICU(cudaEventRecord(m->ev_in[b ^ 1], m->s_copy));
        }
        ICU(cudaStreamWaitEvent(m->s_main, m->ev_in[b], 0));
        if (i >= 2) ICU(cudaEventSynchronize(m->ev_out[b]));          // output set b has been copied out
        hc_ingest_stats st;
        pp.max_overlaps = p->max_overlaps - lines;
        const u64 room_s = overflow ? 0 : std::min<u64>(rec_cap, cand_cap - ns), room_f = overflow ? 0 : std::min<u64>(rec_cap, filtered_cap - nf);
        int prc = hc_ingest_device(m, d_text + (size_t)b * tbytes, cut[i + 1] - cut[i], &pp, d_cand + (size_t)b * rec_cap,
                                d_cl ? d_cl + (size_t)b * rec_cap : nullptr, room_s, d_filt + (size_t)b * rec_cap,
                                d_fl ? d_fl + (size_t)b * rec_cap : nullptr, room_f, &st, m->s_main, lines);
        if (prc == HC_ERR_CAPACITY) { overflow = true; prc = HC_OK; }   // keep counting: the caller gets the required sizes
        if (prc != HC_OK) { rc = prc; goto done; }
        if (st.first_error_line != EMPTY && stats->first_error_line == EMPTY) {
            stats->first_error_line = lines + st.first_error_line;
            stats->first_error_offset = cut[i] + st.first_error_offset;
            stats->first_error_length = st.first_error_length;
            stats->first_error_status = st.first_error_status;
        }
        if (!overflow) {
            if (st.n_scored) {
                ICU(hc_copy_d2h_on(cand + ns, d_cand + (size_t)b * rec_cap, st.n_scored * sizeof(hc_candidate), m->s_out, nullptr));
                if (cand_line) ICU(hc_copy_d2h_on(cand_line + ns, d_cl + (size_t)b * rec_cap, st.n_scored * sizeof(u64), m->s_out, nullptr));
            }
            if (st.n_filtered) {
                ICU(hc_copy_d2h_on(filtered + nf, d_filt + (size_t)b * rec_cap, st.n_filtered * sizeof(hc_overlap_rec), m->s_out, nullptr));
                if (filtered_line) ICU(hc_copy_d2h_on(filtered_line + nf, d_fl + (size_t)b * rec_cap, st.n_filtered * sizeof(u64), m->s_out, nullptr));
            }
        }
        ICU(cudaEventRecord(m->ev_out[b], m->s_out));
        lines += st.n_lines; ns += st.n_scored; nf += st.n_filtered;
        stats->n_skipped += st.n_skipped; stats->n_dropped += st.n_dropped; stats->device_ms += st.device_ms;
    }
    ICU(cudaStreamSynchronize(m->s_out));
    ICU(cudaStreamSynchronize(m->s_copy));
    stats->n_lines = lines; stats->n_scored = ns; stats->n_filtered = nf;
    if (overflow) {
        hc_set_last_error("hc_ingest_overlaps: output buffer too small (required sizes returned in stats)");
        rc = HC_ERR_CAPACITY;
    }
done:
    if (rc != HC_OK && rc != HC_ERR_CAPACITY) { cudaStreamSynchronize(m->s_copy); cudaStreamSynchronize(m->s_out); }
    return rc;
}

extern "C" int hc_ingest_overlaps(const hc_idmap* cm, const char* text, uint64_t n_bytes, const hc_ingest_params* p,
                                  hc_candidate* cand, uint64_t* cand_line, uint64_t cand_cap, hc_overlap_rec* filtered,
                                  uint64_t* filtered_line, uint64_t filtered_cap, hc_ingest_stats* stats) {
    if (!cm || !p || !stats || (n_bytes && !text)) { hc_set_last_error("hc_ingest_overlaps: NULL argument"); return HC_ERR_ARG; }
    hc_idmap* m = const_cast<hc_idmap*>(cm);
    int rc = HC_OK;
    char* d_text = nullptr;
    hc_candidate* d_cand = nullptr;
    hc_overlap_rec* d_filt = nullptr;
    uint64_t *d_cl = nullptr, *d_fl = nullptr;
    memset(stats, 0, sizeof(*stats));
    stats->first_error_line = EMPTY;
    if (n_bytes == 0) return HC_OK;
    ICU(cudaSetDevice(m->device));
    {
        const u64 piece = hc_ingest_piece_bytes();
        if (n_bytes > piece + piece / 2)
            return ingest_pipelined(m, text, n_bytes, p, cand, cand_line, cand_cap, filtered, filtered_line, filtered_cap, stats, piece);
    }
    ICU(hc_idmap_ws(m, 11, n_bytes + 16, (void**)&d_text));
    ICU(hc_copy_h2d(d_text, text, n_bytes));
    if (cand_cap) { ICU(hc_idmap_ws(m, 12, cand_cap * sizeof(hc_candidate), (void**)&d_cand)); if (cand_line) ICU(hc_idmap_ws(m, 14, cand_cap * sizeof(u64), (void**)&d_cl)); }
    if (filtered_cap) { ICU(hc_idmap_ws(m, 13, filtered_cap * sizeof(hc_overlap_rec), (void**)&d_filt)); if (filtered_line) ICU(hc_idmap_ws(m, 15, filtered_cap * sizeof(u64), (void**)&d_fl)); }
    rc = hc_ingest_device(m, d_text, n_bytes, p, d_cand, d_cl, cand_cap, d_filt, d_fl, filtered_cap, stats, m->s_main);
    if (rc != HC_OK) goto done;
    if (stats->n_scored) {
        ICU(hc_copy_d2h(cand, d_cand, stats->n_scored * sizeof(hc_candidate)));
        if (cand_line) ICU(hc_copy_d2h(cand_line, d_cl, stats->n_scored * sizeof(u64)));
    }
    if (stats->n_filtered) {
        ICU(hc_copy_d2h(filtered, d_filt, stats->n_filtered * sizeof(hc_overlap_rec)));
        if (filtered_line) ICU(hc_copy_d2h(filtered_line, d_fl, stats->n_filtered * sizeof(u64)));
    }
done:
    return rc;
}
