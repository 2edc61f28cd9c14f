// hc_fno_text.cu -- the bytes of FindNextOverlaps' overlaps.txt, built in HBM from the records fno_finish has compacted
// there.  A line is "%lu\t%lu\t%d\t%d\t%c\t%c\t%c\t%d\t%d\t%d\t%d\t%c\t%c\n" of id1 id2 pos1 pos2 ord ori1 ori2 perc perc2
// len1 len2 type1 type2 (src/FindNextOverlaps.cpp:122-148).
//
// FNO1 writes the reference's std::set<std::string>: the lines unique and in byte order (:918,:946-948).  A variable-length
// field holds only '0'-'9' and '-', all above the '\t' that ends it, so two lines compare as their 13 fields do, each
// field as a string in which "end of field" sorts below every byte.  Integer keys keep that order:
//   * a non-negative decimal v of d <= 10 digits: K(v) = v * 10^(10-d) * 10 + (d-1) (zero padding, ties by length:
//     "1" < "10" < "100" < "2"); ids are below 2^32, magnitudes of %d fields at most 2^31, so K < 2^37;
//   * a %d field x: negatives first ('-' < '0'), among them by K(|x|) ("-1" < "-10" < "-2"): x < 0 ? K(|x|) : 2^37 + K(x);
//   * a one-byte field (ord, ori1, ori2, type1, type2) compares as an unsigned byte at a fixed position.
// The records are sorted by (K(id1), K(id2)) with the LSD radix sort of hc_radix.cuh (stable, so a run of equal ids keeps
// record order), each run of equal ids is then ordered by the remaining fields by one thread (insertion sort up to 32
// entries, heap sort beyond, as adj_sort_groups), and a line is kept when its fields differ from its predecessor's.
// FNO3 keeps every record in record order (discovery order, src/FindNextOverlaps3.cpp:139-166).
//
// Byte offsets are the exclusive scan of the kept lines' lengths; the format kernel writes a block's lines into shared
// memory and stores its contiguous byte range with 16-byte stores (single bytes only in the two 16-byte words it shares
// with its neighbours); one hc_copy_d2h moves the text to the caller.
#include "hc_fno_text.h"
#include "hc_radix.cuh"
#include "hc_scan.cuh"
#include "hc_stage.h"

namespace {

typedef unsigned long long u64;

constexpr int MAX_LINE = 2 * 10 + 6 * 11 + 5 + 12 + 1;     // two ids < 2^32, six %d fields, five bytes, 12 tabs, '\n'
constexpr int FMT_THREADS = 256;                            // lines per block of the format kernel
constexpr int INSERTION_MAX = 32;

__device__ __forceinline__ hc_fno_overlap fields_of(const hc_fno_overlap& r) { return r; }
__device__ __forceinline__ hc_fno_overlap fields_of(const hc_fno_overlap_small& r) {
    hc_fno_overlap o;
    const uint32_t fl = r.len1_flags >> 24;
    o.id1 = r.id1; o.id2 = r.id2;
    o.pos1 = (int32_t)(r.pos1_perc & 0xffffffu); o.perc = (int32_t)(r.pos1_perc >> 24);
    o.pos2 = (int32_t)(r.pos2_perc2 & 0xffffffu); o.perc2 = (int32_t)(r.pos2_perc2 >> 24);
    o.len1 = (int32_t)(r.len1_flags & 0xffffffu); o.len2 = (int32_t)(r.len2 & 0xffffffu);
    o.ord = (uint8_t)HC_FNO_SMALL_ORD(fl); o.ori1 = (uint8_t)HC_FNO_SMALL_ORI1(fl); o.ori2 = (uint8_t)HC_FNO_SMALL_ORI2(fl);
    o.type1 = (uint8_t)HC_FNO_SMALL_TYPE1(fl); o.type2 = (uint8_t)HC_FNO_SMALL_TYPE2(fl);
    return o;
}

// every printed number fits 32 bits: ids are checked on entry, a %d magnitude is at most 2^31
__device__ __forceinline__ int ndigits(uint32_t v) {
    int d = 1;
    for (uint32_t p = 10; d < 10 && v >= p; p *= 10) d++;
    return d;
}
__device__ __forceinline__ uint32_t magnitude(int32_t x) { return x < 0 ? 0u - (uint32_t)x : (uint32_t)x; }
__device__ __forceinline__ int int_len(int32_t x) { return (x < 0) + ndigits(magnitude(x)); }

__device__ __forceinline__ u64 dec_key(uint32_t v) {
    const int d = ndigits(v);
    u64 k = v;
    for (int j = d; j < 10; j++) k *= 10;
    return k * 10 + (u64)(d - 1);
}
__device__ __forceinline__ u64 int_key(int32_t x) { return x < 0 ? dec_key(magnitude(x)) : (1ull << 37) + dec_key((uint32_t)x); }

__device__ __forceinline__ uint32_t line_len(const hc_fno_overlap& o) {
    return (uint32_t)(ndigits((uint32_t)o.id1) + ndigits((uint32_t)o.id2) + int_len(o.pos1) + int_len(o.pos2) + int_len(o.perc) +
                      int_len(o.perc2) + int_len(o.len1) + int_len(o.len2) + 5 + 12 + 1);
}

// byte order of the fields after id1 / id2 (pos1 pos2 ord ori1 ori2 perc perc2 len1 len2 type1 type2): <0, 0, >0
__device__ int cmp_rest(const hc_fno_overlap& a, const hc_fno_overlap& b) {
#define HC_CMP(x, y) do { const u64 _x = (x), _y = (y); if (_x != _y) return _x < _y ? -1 : 1; } while (0)
    HC_CMP(int_key(a.pos1), int_key(b.pos1));
    HC_CMP(int_key(a.pos2), int_key(b.pos2));
    HC_CMP(a.ord, b.ord);
    HC_CMP(a.ori1, b.ori1);
    HC_CMP(a.ori2, b.ori2);
    HC_CMP(int_key(a.perc), int_key(b.perc));
    HC_CMP(int_key(a.perc2), int_key(b.perc2));
    HC_CMP(int_key(a.len1), int_key(b.len1));
    HC_CMP(int_key(a.len2), int_key(b.len2));
    HC_CMP(a.type1, b.type1);
    HC_CMP(a.type2, b.type2);
#undef HC_CMP
    return 0;
}

__device__ __forceinline__ bool same_line(const hc_fno_overlap& a, const hc_fno_overlap& b) {
    return a.id1 == b.id1 && a.id2 == b.id2 && a.pos1 == b.pos1 && a.pos2 == b.pos2 && a.ord == b.ord && a.ori1 == b.ori1 &&
           a.ori2 == b.ori2 && a.perc == b.perc && a.perc2 == b.perc2 && a.len1 == b.len1 && a.len2 == b.len2 &&
           a.type1 == b.type1 && a.type2 == b.type2;
}

// per record: the line length; with SORT also the key (K(id1), K(id2)) and the record index
template <class R, bool SORT>
__global__ void text_keys(const R* __restrict__ rec, u64 n, uint32_t* __restrict__ len, ulonglong2* __restrict__ key,
                          uint32_t* __restrict__ idx) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const hc_fno_overlap o = fields_of(rec[i]);
        len[i] = line_len(o);
        if (SORT) {
            key[i] = make_ulonglong2(dec_key((uint32_t)o.id2), dec_key((uint32_t)o.id1));
            idx[i] = (uint32_t)i;
        }
    }
}

template <class R>
__device__ __forceinline__ bool rec_less(const R* rec, uint32_t a, uint32_t b) { return cmp_rest(fields_of(rec[a]), fields_of(rec[b])) < 0; }

template <class R>
__device__ void sift_down(const R* rec, uint32_t* v, uint32_t root, uint32_t m) {
    while (true) {
        uint32_t c = 2 * root + 1;
        if (c >= m) return;
        if (c + 1 < m && rec_less(rec, v[c], v[c + 1])) c++;
        if (!rec_less(rec, v[root], v[c])) return;
        const uint32_t t = v[root]; v[root] = v[c]; v[c] = t;
        root = c;
    }
}

// one thread per run of equal (id1, id2): order the run's record indices by the remaining fields
template <class R>
__global__ void text_runs(const ulonglong2* __restrict__ key, uint32_t* __restrict__ idx, u64 n, const R* __restrict__ rec) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const ulonglong2 k = key[i];
        if (i > 0) { const ulonglong2 p = key[i - 1]; if (p.x == k.x && p.y == k.y) continue; }
        u64 j = i + 1;
        while (j < n) { const ulonglong2 q = key[j]; if (q.x != k.x || q.y != k.y) break; j++; }
        const uint32_t m = (uint32_t)(j - i);
        if (m < 2) continue;
        uint32_t* v = idx + i;
        if (m <= INSERTION_MAX) {
            for (uint32_t a = 1; a < m; a++) {
                const uint32_t x = v[a];
                const hc_fno_overlap ox = fields_of(rec[x]);
                uint32_t b = a;
                while (b > 0 && cmp_rest(fields_of(rec[v[b - 1]]), ox) > 0) { v[b] = v[b - 1]; b--; }
                v[b] = x;
            }
        } else {
            for (uint32_t r = m / 2; r-- > 0;) sift_down(rec, v, r, m);
            for (uint32_t e = m - 1; e > 0; e--) {
                const uint32_t t = v[0]; v[0] = v[e]; v[e] = t;
                sift_down(rec, v, 0, e);
            }
        }
    }
}

// klen[i] = length of sorted line i if it differs from line i-1, else 0; *n_lines += kept lines
template <class R>
__global__ void text_marks(const uint32_t* __restrict__ idx, u64 n, const R* __restrict__ rec, const uint32_t* __restrict__ len,
                           uint32_t* __restrict__ klen, u64* __restrict__ n_lines) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 b = (u64)blockIdx.x * blockDim.x; b < n; b += stride) {      // whole warps per step: the ballot below
        const u64 i = b + threadIdx.x;
        bool keep = false;
        if (i < n) {
            const uint32_t r = idx[i];
            keep = i == 0 || !same_line(fields_of(rec[r]), fields_of(rec[idx[i - 1]]));
            klen[i] = keep ? len[r] : 0u;
        }
        const uint32_t kept = __ballot_sync(0xffffffffu, keep);
        if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_lines, (u64)__popc(kept));
    }
}

__device__ __forceinline__ char* put_dec(char* p, uint32_t v) {
    const int d = ndigits(v);
    for (int k = d - 1; k >= 0; k--) { p[k] = (char)('0' + v % 10u); v /= 10u; }
    return p + d;
}
__device__ __forceinline__ char* put_int(char* p, int32_t x) {
    if (x < 0) *p++ = '-';
    return put_dec(p, magnitude(x));
}

// Block b writes lines [b*256, b*256+256) (idx: sorted position -> record, nullptr = identity; klen[i] == 0: not kept).
// The lines go to shared memory at (byte offset - a0), a0 = the block's first byte rounded down to 16, so that the
// 16-byte words of the output and of the shared buffer line up; whole words go out as uint4 stores.
template <class R>
__global__ void __launch_bounds__(FMT_THREADS) text_format(const R* __restrict__ rec, const uint32_t* __restrict__ idx,
                                                           const uint32_t* __restrict__ klen, const u64* __restrict__ off,
                                                           const u64* __restrict__ total, u64 n, char* __restrict__ out) {
    __shared__ uint4 sbuf[(FMT_THREADS * MAX_LINE + 16 + 15) / 16];
    char* s = reinterpret_cast<char*>(sbuf);
    const u64 i0 = (u64)blockIdx.x * FMT_THREADS, i1 = i0 + FMT_THREADS < n ? i0 + FMT_THREADS : n;
    const u64 g0 = off[i0], g1 = i1 < n ? off[i1] : *total;
    if (g0 == g1) return;
    const u64 a0 = g0 & ~15ull;
    const u64 i = i0 + threadIdx.x;
    if (i < i1 && klen[i]) {
        const hc_fno_overlap o = fields_of(rec[idx ? idx[i] : (uint32_t)i]);
        char* p = s + (off[i] - a0);
        p = put_dec(p, (uint32_t)o.id1); *p++ = '\t';
        p = put_dec(p, (uint32_t)o.id2); *p++ = '\t';
        p = put_int(p, o.pos1); *p++ = '\t';
        p = put_int(p, o.pos2); *p++ = '\t';
        *p++ = (char)o.ord; *p++ = '\t';
        *p++ = (char)o.ori1; *p++ = '\t';
        *p++ = (char)o.ori2; *p++ = '\t';
        p = put_int(p, o.perc); *p++ = '\t';
        p = put_int(p, o.perc2); *p++ = '\t';
        p = put_int(p, o.len1); *p++ = '\t';
        p = put_int(p, o.len2); *p++ = '\t';
        *p++ = (char)o.type1; *p++ = '\t';
        *p++ = (char)o.type2; *p = '\n';
    }
    __syncthreads();
    const u64 w0 = g0 >> 4, w1 = (g1 + 15) >> 4;
    for (u64 w = w0 + threadIdx.x; w < w1; w += FMT_THREADS) {
        const u64 lo = w << 4, hi = lo + 16;
        if (lo >= g0 && hi <= g1) {
            reinterpret_cast<uint4*>(out)[w] = sbuf[w - w0];
        } else {                                             // a word shared with the neighbouring block: only our bytes
            for (u64 b = lo > g0 ? lo : g0; b < (hi < g1 ? hi : g1); b++) out[b] = s[b - a0];
        }
    }
}

inline int grid_for(u64 n, int threads) { const u64 b = (n + threads - 1) / threads; return (int)(b < 148 * 16 ? (b ? b : 1) : 148 * 16); }

}  // namespace

template <class R>
int fno_text(const R* d_rec, uint64_t n, const FnoText& t, FnoPhase& ph, const char* who) {
    int rc = HC_OK;
    *t.n_bytes = 0;
    *t.n_lines = 0;
    if (n == 0) return HC_OK;
    if (n >> 32) {
        hc_set_last_error((std::string(who) + ": 2^32 or more overlap records (the text stage indexes them with 32 bits)").c_str());
        return HC_ERR_ARG;
    }
    const int threads = 256, blocks = grid_for(n, threads);
    uint32_t *d_len = nullptr, *d_klen = nullptr, *d_idx = nullptr, *d_idx2 = nullptr, *d_order = nullptr;
    ulonglong2 *d_key = nullptr, *d_key2 = nullptr, *d_sorted = nullptr;
    u64 *d_off = nullptr, *d_total = nullptr, *d_bsum = nullptr, *d_lines = nullptr;
    char* d_text = nullptr;
    u64 bytes = 0, lines = n;
    FCU(hc_scratch_alloc((void**)&d_len, n * sizeof(uint32_t)));
    FCU(hc_scratch_alloc((void**)&d_off, n * sizeof(u64)));
    FCU(hc_scratch_alloc((void**)&d_total, sizeof(u64)));
    FCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(n) * sizeof(u64)));
    if (t.sort_unique) {
        FCU(hc_scratch_alloc((void**)&d_key, n * sizeof(ulonglong2))); FCU(hc_scratch_alloc((void**)&d_key2, n * sizeof(ulonglong2)));
        FCU(hc_scratch_alloc((void**)&d_idx, n * sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_idx2, n * sizeof(uint32_t)));
        FCU(hc_scratch_alloc((void**)&d_klen, n * sizeof(uint32_t))); FCU(hc_scratch_alloc((void**)&d_lines, sizeof(u64)));
        text_keys<R, true><<<blocks, threads>>>(d_rec, n, d_len, d_key, d_idx);
        FCU(cudaGetLastError());
        ph.mark("text: keys + lengths");
        FCU(hc_radix::sort_pairs(d_key, d_idx, d_key2, d_idx2, n, &d_sorted, &d_order));
        ph.mark("text: radix sort of the ids");
        text_runs<R><<<blocks, threads>>>(d_sorted, d_order, n, d_rec);
        FCU(cudaMemsetAsync(d_lines, 0, sizeof(u64)));
        text_marks<R><<<blocks, threads>>>(d_order, n, d_rec, d_len, d_klen, d_lines);
        FCU(cudaGetLastError());
        FCU(cudaMemcpy(&lines, d_lines, sizeof(u64), cudaMemcpyDeviceToHost));
        ph.mark("text: runs sorted, repeats marked");
    } else {
        text_keys<R, false><<<blocks, threads>>>(d_rec, n, d_len, nullptr, nullptr);
        FCU(cudaGetLastError());
        ph.mark("text: lengths");
    }
    hc_scan::exclusive_u32(t.sort_unique ? d_klen : d_len, n, d_off, d_total, d_bsum, 0);
    FCU(cudaMemcpy(&bytes, d_total, sizeof(u64), cudaMemcpyDeviceToHost));
    ph.mark("text: scan of line lengths");
    *t.n_bytes = bytes;
    *t.n_lines = lines;
    if (bytes > t.cap) {
        hc_set_last_error((std::string(who) + ": text buffer too small (required size returned in n_bytes)").c_str());
        rc = HC_ERR_CAPACITY;
        goto done;
    }
    FCU(hc_scratch_alloc((void**)&d_text, bytes));
    text_format<R><<<(unsigned)((n + FMT_THREADS - 1) / FMT_THREADS), FMT_THREADS>>>(d_rec, t.sort_unique ? d_order : nullptr,
                                                                                    t.sort_unique ? d_klen : d_len, d_off, d_total, n, d_text);
    FCU(cudaGetLastError());
    ph.mark("text: format");
    FCU(hc_copy_d2h(t.text, d_text, bytes));
    ph.mark("text: copy out");
done:
    hc_scratch_free(d_len); hc_scratch_free(d_klen); hc_scratch_free(d_idx); hc_scratch_free(d_idx2); hc_scratch_free(d_key);
    hc_scratch_free(d_key2); hc_scratch_free(d_off); hc_scratch_free(d_total); hc_scratch_free(d_bsum); hc_scratch_free(d_lines);
    hc_scratch_free(d_text);
    return rc;
}

template int fno_text<hc_fno_overlap_small>(const hc_fno_overlap_small*, uint64_t, const FnoText&, FnoPhase&, const char*);
template int fno_text<hc_fno_overlap>(const hc_fno_overlap*, uint64_t, const FnoText&, FnoPhase&, const char*);
