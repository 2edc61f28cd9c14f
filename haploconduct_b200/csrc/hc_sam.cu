// hc_sam.cu -- hc_sam2overlaps: single-end and interleaved paired-end SAM text -> the 13-column overlaps file of the
// reference-guided mode, built in HBM.  The host converter (host/hcb_sam2overlaps.cpp, scripts/sam2overlaps.py of the
// reference in C++) is the specification; the points below name its lines.
//
//   1. Lines and header (read_lines :225, :288).  Lines split on '\n' only; an unterminated last line counts and a '\r'
//      stays in the last field.  The header is the leading run of lines that are not empty and start with '@'; every
//      later line is an alignment (an empty one dies in parse_aln).
//   2. Parsing (parse_aln :69-93).  At most 11 tab-separated fields, the 11th takes the rest; fewer dies.  FLAG first
//      (to_long :41: optional sign, digits only); flag & 4 ends the line as unmapped, whatever its other fields.  Then
//      POS, MAPQ, PNEXT, TLEN must parse; the CIGAR's runs (cigar_runs :56: maximal runs of digits or of non-digits, so
//      an operation is a string and "MM" is neither "S" nor "I") must number 2 or more; the clip corrections of POS and
//      of len = |SEQ| follow :87-90.  The runs are kept as (length, class in {I, D, other}) plus two defects: D1, an odd
//      run count or a CIGAR that starts with a non-digit (every even run is then a non-digit and the first to_long of
//      overlap_pos dies, :100,:102,:107); D2, a zero-length run (the assertion of the back walk, :122).
//   3. Singles (:302-313).  Every mapped line of the single-end file is a record; its REF must be in the names table
//      (ref_of :297), the first line in file order that is not dies.
//   4. Pairing (:315-345).  The loop keeps at most one pending alignment: the paired_read vector never holds more than
//      two (the assertion :324 cannot fail) and the branch `pr.size() != 2` (:337) is unreachable.  Over the mapped lines
//      of the paired-end file in file order, in each maximal run of equal ids (bytes) offsets 0-1, 2-3, ... pair; an
//      odd run followed by another mapped line is one discard (:327), the leftover at the end of the file is not.  A pair
//      passes the orientation test of :330-336 (both reverse with POS0 >= POS1, a = the second; both forward with
//      POS0 < POS1, a = the first) or is one more discard.  reverse_p counts the accepted reverse pairs; only a's REF is
//      looked up.
//   5. Order (:350-364).  Stable order by (reference, position, singles before pairs), singles in file order and pairs
//      in formation order: one stable radix sort of (reference, position + 2^41, paired).
//   6. Records processed and window (:366-385).  Record k of a reference is processed iff the position of record
//      max(k - 1, 0) is below the reference length; max_len is the maximum of a.len over the processed records.  The
//      partners of record i > 0 are the records j < i with j == i - 1 or len_j - (pos_{i-1} - pos_j) >= min_ov (:383);
//      the bound of :379-380 only prunes (len_j <= max_len), and here it is a binary search.  One thread per record, j
//      increasing: the file is in (reference, i, j) order.
//   7. Overlap arithmetic (overlap_pos :98-133, overlap_line :142-151, merge :154-166, pair_overlap :177-223).  The
//      first overlap_pos(record.a behind, read.a in front) dies on D1 of either; D2 of the one behind only where the back
//      walk is reached (front_ref > pos1 - pos2).  overlap_line dies where m = min(len) == 0 or perc leaves [0, 100]
//      (possible with a negative min_ov); the second-end overlap_line runs whenever it is reached, before the output
//      test.  The second ends X (read's b, or its a when single) and Y (record's) are walked with the one further right
//      behind: Y for single-paired, X for paired-single (X left of Y is a "problem", :202), for paired-paired Y unless
//      Y.pos < X.pos.  merge's assertion (:158) cannot fail: the ids of a pair are equal, so ord is '2' iff X is behind
//      and the two pairs' ids differ.  perc = (long)round(ovlen / (double)m * 100.0), an IEEE division and
//      multiplication (__ddiv_rn, __dmul_rn: nothing contracted) and round-half-away, bit for bit the host's.
//   8. Warnings (:181, :186).  overlap_pos returns len = min(len2 - pos, len1) with pos >= 0, or len 0; lengths are
//      |SEQ| plus clips, never negative; so len > min(len1, len2) cannot hold and the warning lines never print.
//   9. Output.  No sort or uniq of output lines: per record its lines are counted (bytes, lines, ori types,
//      problems), scanned and then written, two passes as in hc_sfo.cu; the per-reference statistics are reductions of
//      the same counts over each reference's records.
//
// A line that dies is reported in three stages, as the host meets them: parsing (both files), the REF lookups, the
// sweep; inside a stage the smallest (file, line).  A sweep error names the alignment the host dies on.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>
#include <time.h>
#include <cuda_runtime.h>
#include "../../include/hc_b200.h"
#include "hc_radix.cuh"
#include "hc_scan.cuh"
#include "hc_stage.h"
#include "hc_text.cuh"

void hc_set_last_error(const char* msg);   // hc_api.cu

namespace {

typedef long long i64;

constexpr i64 BIG = 1ll << 40;             // |POS|, clips and CIGAR run lengths below this: no sum of them overflows
constexpr i64 POS_BIAS = 1ll << 41;        // corrected positions lie in (-2^41, 2^41)
constexpr i64 MIN_OV_CLAMP = 1ll << 50;    // min_ov beyond this compares like +-infinity with every length here
constexpr unsigned long long NO_ERR = ~0ull;
constexpr uint32_t CLS_OTHER = 0, CLS_I = 1, CLS_D = 2;

struct Aln {                               // a mapped alignment (host Aln :31)
    u64 id_off, cig_off, ops_off;          // text offsets of QNAME and CIGAR; first run in the ops array
    i64 pos, len;                          // clip-corrected POS, |SEQ| + hard clips
    uint32_t id_len, cig_len, n_ops;       // n_ops = (length, class) pairs, 0 when d1
    uint32_t line;                         // 0-based line in its file
    int32_t ref;                           // names-table index of REF, -1 if absent
    uint8_t file, rev, d1, d2;
};

struct Rec {                               // a single-end read or a pair (host Rec :35), in sorted order for the sweep
    i64 pos, len;                          // a.pos, a.len
    uint32_t a, b;                         // Aln indices (b == a for a single)
    int32_t ref;
    uint8_t paired, rc;
};

struct RefInfo { u64 rb, re, nproc; i64 max_len; };

struct Names { const char* t; const u64* off; const uint32_t* perm; const uint32_t* idx; uint32_t n; };

__device__ __forceinline__ unsigned long long err_key(uint32_t file, uint32_t line, uint32_t status) {
    return (unsigned long long)file << 34 | (unsigned long long)line << 2 | status;
}

// to_long (:41) of [b, e): 0 not a number, 1 ok, 2 more than 18 digits (the host's long may overflow)
__device__ int to_long(const char* t, u64 b, u64 e, i64* v) {
    if (b == e) return 0;
    bool neg = false;
    if (t[b] == '+' || t[b] == '-') { neg = t[b] == '-'; b++; }
    if (b == e) return 0;
    i64 x = 0;
    for (u64 p = b; p < e; p++) {
        const char c = t[p];
        if (c < '0' || c > '9') return 0;
        if (p - b < 18) x = x * 10 + (c - '0');
    }
    *v = neg ? -x : x;
    return e - b > 18 ? 2 : 1;
}

__device__ __forceinline__ bool is_digit(char c) { return c >= '0' && c <= '9'; }

// bytewise compare of two texts (std::string operator<=>)
__device__ int bcmp(const char* a, u64 la, const char* b, u64 lb) {
    const u64 m = la < lb ? la : lb;
    for (u64 i = 0; i < m; i++)
        if (a[i] != b[i]) return (unsigned char)a[i] < (unsigned char)b[i] ? -1 : 1;
    return la < lb ? -1 : (la > lb ? 1 : 0);
}

__device__ int32_t lookup(const Names& N, const char* s, u64 l) {
    uint32_t lo = 0, hi = N.n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) / 2, e = N.perm[mid];
        const int c = bcmp(N.t + N.off[e], N.off[e + 1] - N.off[e], s, l);
        if (c == 0) return (int32_t)N.idx[e];
        if (c < 0) lo = mid + 1; else hi = mid;
    }
    return -1;
}

__device__ __forceinline__ void line_span(const char* t, u64 n, const u64* ls, u64 n_nl, u64 k, u64* b, u64* le) {
    *b = ls[k];
    u64 e = k < n_nl ? ls[k + 1] : n;
    if (e > *b && t[e - 1] == '\n') e--;
    *le = e;
}

struct FileIn { const char* t; u64 base, n; const u64* ls; u64 n_nl, nl; uint32_t file; };

// the header's end: the first line that is empty or does not start with '@'
__global__ void sam_header(FileIn F, unsigned long long* first) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < F.nl; k += (u64)gridDim.x * blockDim.x) {
        u64 b, le;
        line_span(F.t, F.n, F.ls, F.n_nl, k, &b, &le);
        if (le == b || F.t[b] != '@') atomicMin(first, (unsigned long long)k);
    }
}

// one thread per line at or after the header: the Aln of a mapped line (ref looked up), mapped[g], nops[g], rev[g];
// a line the host dies on or the device declines -> err[0]; a mapped single whose REF is absent -> err[1]
__global__ void sam_parse(FileIn F, u64 first, u64 g0, Names N, Aln* __restrict__ aln, uint32_t* __restrict__ mapped,
                          uint32_t* __restrict__ nops, uint32_t* __restrict__ rev, unsigned long long* err) {
    for (u64 k = first + (u64)blockIdx.x * blockDim.x + threadIdx.x; k < F.nl; k += (u64)gridDim.x * blockDim.x) {
        const u64 g = g0 + (k - first);
        mapped[g] = 0; nops[g] = 0; rev[g] = 0;
        u64 b, le;
        line_span(F.t, F.n, F.ls, F.n_nl, k, &b, &le);
        const char* t = F.t;
        u64 fb[11], fe[11];
        int nf = 0;
        u64 p = b;
        while (nf < 11) {
            u64 q = p;
            while (q < le && t[q] != '\t') q++;
            fb[nf] = p;
            if (q == le || nf == 10) { fe[nf] = le; nf++; break; }
            fe[nf] = q; nf++;
            p = q + 1;
        }
        uint32_t die = 0, decline = 0;
        i64 flag = 0, POS = 0, dummy;
        int r;
        if (nf < 11) die = 1;
        if (!die) { r = to_long(t, fb[1], fe[1], &flag); die |= r == 0; decline |= r == 2; }
        if (!die && !decline && (flag & 4)) continue;                  // unmapped: nothing else is read
        if (!die && !decline) {
            r = to_long(t, fb[3], fe[3], &POS); die |= r == 0; decline |= r == 2 || POS >= BIG || POS <= -BIG;
            const int more[3] = {4, 7, 8};                             // MAPQ, PNEXT, TLEN: only their validity matters
            for (int f : more) { r = to_long(t, fb[f], fe[f], &dummy); die |= r == 0; decline |= r == 2; }
        }
        Aln a;
        uint32_t runs = 0, z = 0;
        i64 c0 = 0, prev_digit = 0, last_num = 0;
        bool c1S = false, c1H = false, lastH = false, first_digit = false;
        if (!die) {
            const u64 cb = fb[5], ce = fe[5];
            first_digit = cb < ce && is_digit(t[cb]);
            for (u64 q = cb; q < ce;) {
                const bool d = is_digit(t[q]);
                u64 e = q;
                while (e < ce && is_digit(t[e]) == d) e++;
                if (d) {
                    i64 v = 0;
                    for (u64 x = q; x < e && v < BIG; x++) v = v * 10 + (t[x] - '0');
                    if (v >= BIG) decline = 1;
                    if (v == 0) z = 1;
                    prev_digit = v;
                    if (runs == 0) c0 = v;
                } else {
                    const bool isS = e - q == 1 && t[q] == 'S', isH = e - q == 1 && t[q] == 'H';
                    if (runs == 1) { c1S = isS; c1H = isH; }
                    lastH = isH;
                    last_num = prev_digit;
                }
                runs++;
                q = e;
            }
            if (runs < 2) die = 1;
            if (runs > 0 && is_digit(t[ce - 1])) lastH = false;        // the last run is a number
        }
        if (die || decline) {
            atomicMin(&err[0], err_key(F.file, (uint32_t)k, die ? HC_SAM_DIES : HC_SAM_DECLINED));
            continue;
        }
        i64 len = (i64)(fe[9] - fb[9]);
        if (c1S) a.pos = POS - c0;                                      // c[1] is "S" or "H": c[0] is a number
        else if (c1H) { a.pos = POS - c0; len += c0; }
        else a.pos = POS;
        if (lastH) len += last_num;                                    // c[size - 2] is the number before the last "H"
        a.len = len;
        a.id_off = F.base + fb[0]; a.id_len = (uint32_t)(fe[0] - fb[0]);
        a.cig_off = F.base + fb[5]; a.cig_len = (uint32_t)(fe[5] - fb[5]);
        a.ops_off = 0;
        a.d1 = (runs & 1) || !first_digit;
        a.d2 = (uint8_t)z;
        a.n_ops = a.d1 ? 0 : runs / 2;
        a.line = (uint32_t)k;
        a.file = (uint8_t)F.file;
        a.rev = (flag & 16) != 0;
        a.ref = lookup(N, t + fb[2], fe[2] - fb[2]);
        if (F.file == 0 && a.ref < 0) atomicMin(&err[1], err_key(0, (uint32_t)k, HC_SAM_DIES));
        aln[g] = a;
        mapped[g] = 1; nops[g] = a.n_ops; rev[g] = a.rev;
    }
}

// the (length << 2 | class) runs of every mapped alignment without D1
__global__ void sam_ops(const char* __restrict__ t, const uint32_t* __restrict__ mapped, const u64* __restrict__ ooff, u64 ng,
                        Aln* __restrict__ aln, u64* __restrict__ ops) {
    for (u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (u64)gridDim.x * blockDim.x) {
        if (!mapped[g]) continue;
        const Aln a = aln[g];
        aln[g].ops_off = ooff[g];
        if (!a.n_ops) continue;
        u64* o = ops + ooff[g];
        const u64 cb = a.cig_off, ce = a.cig_off + a.cig_len;
        u64 v = 0;
        uint32_t r = 0;
        for (u64 q = cb; q < ce;) {
            const bool d = is_digit(t[q]);
            u64 e = q;
            while (e < ce && is_digit(t[e]) == d) e++;
            if (d) {
                v = 0;
                for (u64 x = q; x < e; x++) v = v * 10 + (t[x] - '0');
            } else {
                const uint32_t cls = e - q == 1 && t[q] == 'I' ? CLS_I : (e - q == 1 && t[q] == 'D' ? CLS_D : CLS_OTHER);
                o[r++] = v << 2 | cls;
            }
            q = e;
        }
    }
}

__global__ void sam_gather_mapped(const uint32_t* __restrict__ mapped, const u64* __restrict__ mpos, u64 g0, u64 n,
                                  uint32_t* __restrict__ midx) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (mapped[g0 + i]) midx[mpos[i]] = (uint32_t)(g0 + i);
}

__device__ __forceinline__ bool same_id(const char* t, const Aln& x, const Aln& y) {
    return x.id_len == y.id_len && bcmp(t + x.id_off, x.id_len, t + y.id_off, y.id_len) == 0;
}

// mapped paired-end alignment q starts a run of equal ids
__global__ void sam_run_starts(const char* __restrict__ t, const Aln* __restrict__ aln, const uint32_t* __restrict__ midx, u64 nm,
                               uint32_t* __restrict__ st) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < nm; q += (u64)gridDim.x * blockDim.x)
        st[q] = q == 0 || !same_id(t, aln[midx[q - 1]], aln[midx[q]]);
}

__global__ void sam_run_first(const uint32_t* __restrict__ st, const u64* __restrict__ rx, u64 nm, uint32_t* __restrict__ rfirst) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < nm; q += (u64)gridDim.x * blockDim.x)
        if (st[q]) rfirst[rx[q]] = (uint32_t)q;
}

__device__ __forceinline__ u64 run_offset(const uint32_t* st, const u64* rx, const uint32_t* rfirst, u64 q) {
    return q - rfirst[rx[q] + st[q] - 1];
}

// acc[q] = a pair ends at q and passes the orientation test; cnt[0] discards, cnt[1] reverse pairs; a's REF absent -> err[1]
__global__ void sam_pairs(const Aln* __restrict__ aln, const uint32_t* __restrict__ midx, const uint32_t* __restrict__ st,
                          const u64* __restrict__ rx, const uint32_t* __restrict__ rfirst, u64 nm, uint32_t* __restrict__ acc,
                          unsigned long long* cnt, unsigned long long* err) {
    unsigned disc = 0, revp = 0;
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < nm; q += (u64)gridDim.x * blockDim.x) {
        uint32_t ok = 0;
        if (q > 0 && st[q] && run_offset(st, rx, rfirst, q - 1) % 2 == 0) disc++;      // the pending end is dropped (:327)
        if (run_offset(st, rx, rfirst, q) % 2 == 1) {
            const Aln& x = aln[midx[q - 1]];
            const Aln& y = aln[midx[q]];
            const Aln* a = nullptr;
            if (x.pos >= y.pos) { if (x.rev && y.rev) { a = &y; revp++; } }
            else if (!x.rev && !y.rev) a = &x;
            if (a) {
                ok = 1;
                if (a->ref < 0) atomicMin(&err[1], err_key(1, a->line, HC_SAM_DIES));
            } else {
                disc++;
            }
        }
        acc[q] = ok;
    }
    disc = __reduce_add_sync(0xffffffffu, disc);
    revp = __reduce_add_sync(0xffffffffu, revp);
    if ((threadIdx.x & 31) == 0) {
        if (disc) atomicAdd(&cnt[0], (unsigned long long)disc);
        if (revp) atomicAdd(&cnt[1], (unsigned long long)revp);
    }
}

// records: the mapped singles in file order, then the accepted pairs in formation order; sort key and value
__global__ void sam_records(const Aln* __restrict__ aln, const uint32_t* __restrict__ smidx, u64 nsm, const uint32_t* __restrict__ pmidx,
                            const uint32_t* __restrict__ acc, const u64* __restrict__ apos, u64 nm, Rec* __restrict__ rec,
                            ulonglong2* __restrict__ key, uint32_t* __restrict__ val) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < nsm + nm; q += (u64)gridDim.x * blockDim.x) {
        Rec r;
        u64 at;
        if (q < nsm) {
            r.a = r.b = smidx[q];
            r.paired = 0; r.rc = 0;
            at = q;
        } else {
            const u64 m = q - nsm;
            if (!acc[m]) continue;
            const uint32_t i0 = pmidx[m - 1], i1 = pmidx[m];
            r.rc = aln[i0].pos >= aln[i1].pos;
            r.a = r.rc ? i1 : i0; r.b = r.rc ? i0 : i1;
            r.paired = 1;
            at = nsm + apos[m];
        }
        const Aln& a = aln[r.a];
        r.pos = a.pos; r.len = a.len; r.ref = a.ref;
        rec[at] = r;
        key[at] = make_ulonglong2((u64)(r.pos + POS_BIAS) << 1 | r.paired, (u64)(uint32_t)r.ref);
        val[at] = (uint32_t)at;
    }
}

__global__ void sam_gather(const uint32_t* __restrict__ ord, u64 n, const Rec* __restrict__ rec, Rec* __restrict__ srec) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) srec[k] = rec[ord[k]];
}

// one block per reference: its records [rb, re), those processed (:367-368) and max_len (:369-370)
__global__ void sam_ref_info(const Rec* __restrict__ srec, u64 n, const i64* __restrict__ ref_len, RefInfo* __restrict__ info) {
    __shared__ u64 s_rb, s_re, s_np;
    __shared__ unsigned long long s_max;
    const int32_t r = (int32_t)blockIdx.x;
    if (threadIdx.x == 0) {
        u64 lo = 0, hi = n;
        while (lo < hi) { const u64 m = (lo + hi) / 2; if (srec[m].ref < r) lo = m + 1; else hi = m; }
        const u64 rb = lo;
        hi = n;
        while (lo < hi) { const u64 m = (lo + hi) / 2; if (srec[m].ref <= r) lo = m + 1; else hi = m; }
        const u64 re = lo;
        lo = rb; hi = re;
        while (lo < hi) { const u64 m = (lo + hi) / 2; if (srec[m].pos < ref_len[r]) lo = m + 1; else hi = m; }
        const u64 c = lo - rb;                         // records inside the reference
        s_rb = rb; s_re = re;
        s_np = c == 0 ? 0 : (c + 1 < re - rb ? c + 1 : re - rb);
        s_max = 0;
    }
    __syncthreads();
    i64 m = 0;
    for (u64 k = s_rb + threadIdx.x; k < s_rb + s_np; k += blockDim.x) m = srec[k].len > m ? srec[k].len : m;
    if (m) atomicMax(&s_max, (unsigned long long)m);
    __syncthreads();
    if (threadIdx.x == 0) info[r] = RefInfo{s_rb, s_re, s_np, (i64)s_max};
}

struct Sink {                                         // counts bytes; writes them too when p != nullptr
    char* p;
    u64 n;
    __device__ void c(char x) { if (p) p[n] = x; n++; }
    __device__ void num(i64 v) {
        unsigned long long u = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
        int d = 1;
        for (unsigned long long x = u; x >= 10; x /= 10) d++;
        d += v < 0;
        if (p) {
            char* q = p + n;
            if (v < 0) *q = '-';
            for (int k = d - 1; k >= (v < 0); k--) { q[k] = (char)('0' + u % 10); u /= 10; }
        }
        n += d;
    }
    __device__ void str(const char* t, u64 b, u64 l) {
        if (p) for (u64 i = 0; i < l; i++) p[n + i] = t[b + i];
        n += l;
    }
};

struct Ctx { const char* t; const Aln* aln; const u64* ops; i64 min_ov; };

struct Ov { i64 pos, len; };

// overlap_pos (:98-133) with x behind (pos1) and y in front (pos2); *bad = the alignment the host dies on
__device__ Ov overlap_pos(const Ctx& X, uint32_t ix, uint32_t iy, uint32_t* bad) {
    const Aln& x = X.aln[ix];
    const Aln& y = X.aln[iy];
    Ov o = {-1, 0};
    if (x.d1) { *bad = ix; return o; }
    if (y.d1) { *bad = iy; return o; }
    const u64* c1 = X.ops + x.ops_off;
    const u64* c2 = X.ops + y.ops_off;
    const i64 d = x.pos - y.pos;
    i64 total_back = 0;
    for (uint32_t r = 0; r < x.n_ops; r++) if ((c1[r] & 3) != CLS_I) total_back += (i64)(c1[r] >> 2);
    const i64 max_len = d + total_back;
    i64 fs = 0, fr = 0, p = 0;
    for (uint32_t r = 0; r < y.n_ops && p < max_len; r++) {      // p never decreases: past max_len nothing changes
        const i64 n = (i64)(c2[r] >> 2), m = n < max_len - p ? n : max_len - p;
        const uint32_t cls = (uint32_t)(c2[r] & 3);
        if (cls != CLS_D) fs += m;
        if (cls != CLS_I) { fr += m; p += n; }
    }
    if (fr <= d) return o;
    if (x.d2) { *bad = ix; return o; }
    const i64 back_ref = fr - d;
    i64 bs = 0;
    p = 0;
    for (uint32_t r = 0; r < x.n_ops && p < back_ref; r++) {
        const i64 n = (i64)(c1[r] >> 2);
        const uint32_t cls = (uint32_t)(c1[r] & 3);
        if (cls != CLS_D) bs += n < back_ref - p ? n : back_ref - p;
        if (cls != CLS_I) p += n;
    }
    const i64 pos = d - ((fr - fs) - (back_ref - bs));
    if (pos >= 0) { o.pos = pos; o.len = y.len - pos < x.len ? y.len - pos : x.len; }
    return o;
}

// overlap_line's percentage (:145-149); false where the host dies
__device__ bool perc_of(i64 ovlen, i64 l1, i64 l2, i64* perc) {
    const i64 m = l1 < l2 ? l1 : l2;
    if (m == 0) return false;
    *perc = (i64)round(__dmul_rn(__ddiv_rn((double)ovlen, (double)m), 100.0));
    return *perc >= 0 && *perc <= 100;
}

struct PairOut { uint32_t bad; uint8_t line, problem, type; };

// pair_overlap (:177-223) of the read (earlier record R) and the record C; its line, if any, goes to s
__device__ PairOut pair_overlap(const Ctx& X, const Rec& R, const Rec& C, Sink& s) {
    PairOut out = {~0u, 0, 0, 0};
    const Aln& Ra = X.aln[R.a];
    const Aln& Ca = X.aln[C.a];
    const Ov o = overlap_pos(X, C.a, R.a, &out.bad);
    if (out.bad != ~0u) return out;
    if (o.len <= X.min_ov || o.pos < 0) return out;
    i64 perc1, perc2 = 0;
    if (!perc_of(o.len, Ra.len, Ca.len, &perc1)) { out.bad = Ra.len == 0 ? R.a : C.a; return out; }
    Ov v = {0, 0};
    char ord = '-', t1 = 's', t2 = 's';
    if (R.paired || C.paired) {
        const uint32_t ix = R.b, iy = C.b;                     // the second ends (b == a for a single)
        const Aln& x = X.aln[ix];
        const Aln& y = X.aln[iy];
        bool x_behind;
        if (R.paired && !C.paired) {
            if (x.pos < y.pos) { out.problem = 1; return out; }
            x_behind = true;
        } else {
            x_behind = y.pos < x.pos;
        }
        v = x_behind ? overlap_pos(X, ix, iy, &out.bad) : overlap_pos(X, iy, ix, &out.bad);
        if (out.bad != ~0u) return out;
        if (!perc_of(v.len, x.len, y.len, &perc2)) { out.bad = x.len == 0 ? ix : (y.len == 0 ? iy : (x_behind ? ix : iy)); return out; }
        if (!(v.len > X.min_ov && v.pos >= 0)) return out;
        t2 = 'p';
        if (R.paired && C.paired) { t1 = 'p'; ord = x_behind && !same_id(X.t, Ra, Ca) ? '2' : '1'; }
    }
    const char o1 = R.paired ? (R.rc ? '-' : '+') : (Ra.rev ? '-' : '+');
    const char o2 = C.paired ? (C.rc ? '-' : '+') : (Ca.rev ? '-' : '+');
    s.str(X.t, Ra.id_off, Ra.id_len); s.c('\t'); s.str(X.t, Ca.id_off, Ca.id_len); s.c('\t'); s.num(o.pos); s.c('\t');
    s.num(v.pos); s.c('\t'); s.c(ord); s.c('\t'); s.c(o1); s.c('\t'); s.c(o2); s.c('\t'); s.num(perc1); s.c('\t');
    s.num(perc2); s.c('\t'); s.num(o.len); s.c('\t'); s.num(v.len); s.c('\t'); s.c(t1); s.c('\t'); s.c(t2); s.c('\n');
    out.line = 1;
    out.type = (uint8_t)((o1 == '-') * 2 + (o2 == '-'));
    return out;
}

struct Sweep { Ctx X; const Rec* srec; const RefInfo* info; u64 n; };

struct RecCnt { uint32_t t[4], problems; };

// record k's partners (:379-385), each through pair_overlap into s; returns false if k is not a processed record > 0
template <typename F>
__device__ bool partners(const Sweep& S, u64 k, F&& each) {
    const Rec C = S.srec[k];
    const RefInfo I = S.info[C.ref];
    if (k == I.rb || k >= I.rb + I.nproc) return false;
    const i64 prev = S.srec[k - 1].pos;
    const i64 bound = prev - (I.max_len - S.X.min_ov);
    u64 lo = I.rb, hi = k - 1;                             // first j with pos >= bound, at most k - 1
    while (lo < hi) { const u64 m = (lo + hi) / 2; if (S.srec[m].pos < bound) lo = m + 1; else hi = m; }
    for (u64 j = lo; j < k; j++) {
        const Rec R = S.srec[j];
        if (j != k - 1 && !(R.len - (prev - R.pos) >= S.X.min_ov)) continue;
        each(R, C);
    }
    return true;
}

// per sorted record: bytes and per-type line counts of its lines, problems; a pair the host dies on -> err[2]
__global__ void sam_count(Sweep S, uint32_t* __restrict__ nb, RecCnt* __restrict__ rc, uint32_t* ovf, unsigned long long* err) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < S.n; k += (u64)gridDim.x * blockDim.x) {
        Sink s = {nullptr, 0};
        RecCnt c = {{0, 0, 0, 0}, 0};
        unsigned long long e = NO_ERR;
        partners(S, k, [&](const Rec& R, const Rec& C) {
            const PairOut o = pair_overlap(S.X, R, C, s);
            if (o.bad != ~0u) {
                const Aln& a = S.X.aln[o.bad];
                const unsigned long long key = err_key(a.file, a.line, HC_SAM_DIES);
                e = key < e ? key : e;
            }
            c.t[o.type] += o.line;
            c.problems += o.problem;
        });
        if (e != NO_ERR) atomicMin(&err[2], e);
        if (s.n >> 32) atomicOr(ovf, 1u);
        nb[k] = (uint32_t)s.n;
        rc[k] = c;
    }
}

__global__ void sam_format(Sweep S, const u64* __restrict__ off, char* __restrict__ out) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < S.n; k += (u64)gridDim.x * blockDim.x) {
        Sink s = {out + off[k], 0};
        partners(S, k, [&](const Rec& R, const Rec& C) { pair_overlap(S.X, R, C, s); });
    }
}

// one block per reference: hc_sam_ref_stats from the records' counts
__global__ void sam_ref_stats(const Rec* __restrict__ srec, const RecCnt* __restrict__ rc, const RefInfo* __restrict__ info,
                              hc_sam_ref_stats* __restrict__ rs) {
    __shared__ unsigned long long acc[7];                 // paired, problems, types[4], lines
    if (threadIdx.x < 7) acc[threadIdx.x] = 0;
    __syncthreads();
    const RefInfo I = info[blockIdx.x];
    unsigned long long v[7] = {0, 0, 0, 0, 0, 0, 0};
    for (u64 k = I.rb + threadIdx.x; k < I.re; k += blockDim.x) {
        v[0] += srec[k].paired;
        if (k < I.rb + I.nproc) {
            const RecCnt c = rc[k];
            v[1] += c.problems;
            for (int t = 0; t < 4; t++) { v[2 + t] += c.t[t]; v[6] += c.t[t]; }
        }
    }
    for (int i = 0; i < 7; i++) if (v[i]) atomicAdd(&acc[i], v[i]);
    __syncthreads();
    if (threadIdx.x == 0) {
        hc_sam_ref_stats r;
        r.n_alignments = I.re - I.rb;
        r.n_paired = acc[0];
        r.n_singles = r.n_alignments - acc[0];
        r.problems = acc[1];
        r.n_overlaps = acc[6];
        for (int t = 0; t < 4; t++) r.types[t] = acc[2 + t];
        rs[blockIdx.x] = r;
    }
}

inline int grid_for(u64 n, int threads) { const u64 b = (n + threads - 1) / threads; return (int)(b < 148 * 16 ? (b ? b : 1) : 148 * 16); }
inline double now_ms() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }

}  // namespace

// an allocation that fails is HC_ERR_NOMEM (the caller runs the host converter), anything else HC_ERR_CUDA
#define SCU(call)                                                                                              \
    do {                                                                                                       \
        cudaError_t _e = (call);                                                                               \
        if (_e != cudaSuccess) {                                                                               \
            hc_set_last_error((std::string("hc_sam2overlaps: ") + #call + ": " + cudaGetErrorString(_e)).c_str()); \
            rc = _e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA;                                 \
            if (rc == HC_ERR_NOMEM) cudaGetLastError();                                                        \
            goto done;                                                                                         \
        }                                                                                                      \
    } while (0)

extern "C" int hc_sam2overlaps(const char* sam_s, uint64_t n_s, const char* sam_p, uint64_t n_p, const char* ref_names,
                               const uint64_t* ref_name_off, const uint32_t* ref_name_idx, uint32_t n_names, const int64_t* ref_len,
                               uint32_t n_refs, int64_t min_overlap_len, char* text, uint64_t text_cap, uint64_t* n_text_bytes,
                               hc_sam_ref_stats* ref_stats, hc_sam_stats* stats, int device) {
    if (!n_text_bytes || !stats || (text_cap && !text) || (n_s && !sam_s) || (n_p && !sam_p) || (n_names && (!ref_name_off || !ref_name_idx)) ||
        (n_refs && !ref_len) || (n_names && ref_name_off[n_names] && !ref_names)) {
        hc_set_last_error("hc_sam2overlaps: NULL argument");
        return HC_ERR_ARG;
    }
    std::vector<uint32_t> perm(n_names);
    std::iota(perm.begin(), perm.end(), 0u);
    for (uint32_t e = 0; e < n_names; e++)
        if (ref_name_off[e + 1] < ref_name_off[e] || ref_name_idx[e] >= n_refs) {
            hc_set_last_error("hc_sam2overlaps: names table: offsets must not decrease and indices must be below n_refs");
            return HC_ERR_ARG;
        }
    auto name_cmp = [&](uint32_t a, uint32_t b) {
        const u64 la = ref_name_off[a + 1] - ref_name_off[a], lb = ref_name_off[b + 1] - ref_name_off[b];
        const int c = std::memcmp(ref_names + ref_name_off[a], ref_names + ref_name_off[b], la < lb ? la : lb);
        return c != 0 ? c : (la < lb ? -1 : (la > lb ? 1 : 0));
    };
    std::sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b) { return name_cmp(a, b) < 0; });
    for (uint32_t e = 1; e < n_names; e++)
        if (name_cmp(perm[e - 1], perm[e]) == 0) {
            hc_set_last_error("hc_sam2overlaps: names table: a name occurs twice");
            return HC_ERR_ARG;
        }
    *n_text_bytes = 0;
    memset(stats, 0, sizeof(*stats));
    stats->first_error_line = ~0ull;
    if (ref_stats) memset(ref_stats, 0, n_refs * sizeof(hc_sam_ref_stats));
    int rc = HC_OK;
    const int T = 256;
    const u64 n_all = n_s + n_p, names_bytes = n_names ? ref_name_off[n_names] : 0;
    char *d_text = nullptr, *d_names = nullptr, *d_out = nullptr;
    u64 *d_ls[2] = {nullptr, nullptr}, *d_noff = nullptr, *d_tot = nullptr, *d_bsum = nullptr, *d_ooff = nullptr, *d_ops = nullptr,
        *d_mpos = nullptr, *d_rx = nullptr, *d_apos = nullptr, *d_boff = nullptr;
    uint32_t *d_perm = nullptr, *d_nidx = nullptr, *d_mapped = nullptr, *d_nops = nullptr, *d_rev = nullptr, *d_smidx = nullptr,
             *d_pmidx = nullptr, *d_st = nullptr, *d_rfirst = nullptr, *d_acc = nullptr, *d_val = nullptr, *d_val2 = nullptr,
             *d_ord = nullptr, *d_nb = nullptr, *d_ovf = nullptr;
    unsigned long long* d_cnt = nullptr;      // [0..2] first error per stage, [3] header end, [4] discards, [5] reverse pairs
    i64* d_rlen = nullptr;
    Aln* d_aln = nullptr;
    Rec *d_rec = nullptr, *d_srec = nullptr;
    RefInfo* d_info = nullptr;
    RecCnt* d_rc = nullptr;
    hc_sam_ref_stats* d_rs = nullptr;
    ulonglong2 *d_key = nullptr, *d_key2 = nullptr, *d_skey = nullptr;
    u64 n_nl[2] = {0, 0}, nl[2] = {0, 0}, first[2] = {0, 0}, ng = 0, n_ops = 0, nsm = 0, nm = 0, nruns = 0, npairs = 0, nrec = 0,
        out_bytes = 0;
    unsigned long long cnt[6];
    uint32_t ovf = 0;
    double t0 = 0, t1 = 0;
    Names N;
    Sweep S;
    std::vector<hc_sam_ref_stats> rs(n_refs);
    const u64 nbytes[2] = {n_s, n_p};
    const i64 min_ov = min_overlap_len > MIN_OV_CLAMP ? MIN_OV_CLAMP : (min_overlap_len < -MIN_OV_CLAMP ? -MIN_OV_CLAMP : min_overlap_len);
    SCU(cudaSetDevice(device));
    t0 = now_ms();
    SCU(hc_scratch_alloc((void**)&d_text, n_all + 16));
    if (n_s) SCU(hc_copy_h2d(d_text, sam_s, n_s));
    if (n_p) SCU(hc_copy_h2d(d_text + n_s, sam_p, n_p));
    t1 = now_ms();
    stats->h2d_ms = (float)(t1 - t0);
    t0 = t1;
    // the names table (sorted here for the binary search) and the reference lengths
    SCU(hc_scratch_alloc((void**)&d_names, names_bytes + 1));
    SCU(hc_scratch_alloc((void**)&d_noff, (n_names + 1) * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_perm, (n_names + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_nidx, (n_names + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rlen, (n_refs + 1) * sizeof(i64)));
    if (names_bytes) SCU(cudaMemcpy(d_names, ref_names, names_bytes, cudaMemcpyHostToDevice));
    if (n_names) {
        SCU(cudaMemcpy(d_noff, ref_name_off, (n_names + 1) * sizeof(u64), cudaMemcpyHostToDevice));
        SCU(cudaMemcpy(d_perm, perm.data(), n_names * sizeof(uint32_t), cudaMemcpyHostToDevice));
        SCU(cudaMemcpy(d_nidx, ref_name_idx, n_names * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    if (n_refs) SCU(cudaMemcpy(d_rlen, ref_len, n_refs * sizeof(i64), cudaMemcpyHostToDevice));
    N = Names{d_names, d_noff, d_perm, d_nidx, n_names};
    // lines, header, parse
    for (int f = 0; f < 2; f++) SCU(hc_line_index(d_text + (f ? n_s : 0), nbytes[f], &d_ls[f], &n_nl[f], &nl[f], 0));
    if ((nl[0] + nl[1]) >> 32) {
        stats->first_error_file = nl[0] >> 32 ? 0 : 1;
        stats->first_error_line = 1ull << 32;
        stats->first_error_status = HC_SAM_DECLINED;
        hc_set_last_error("hc_sam2overlaps: 2^32 lines or more (the device path indexes lines with 32 bits)");
        rc = HC_ERR_INPUT;
        goto done;
    }
    for (int i = 0; i < 6; i++) cnt[i] = i < 3 ? NO_ERR : 0;
    SCU(hc_scratch_alloc((void**)&d_cnt, sizeof(cnt)));
    SCU(hc_scratch_alloc((void**)&d_ovf, sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_tot, sizeof(u64)));
    SCU(cudaMemset(d_ovf, 0, sizeof(uint32_t)));
    for (int f = 0; f < 2; f++) {
        cnt[3] = nl[f];
        SCU(cudaMemcpy(d_cnt + 3, &cnt[3], sizeof(u64), cudaMemcpyHostToDevice));
        if (nl[f]) {
            FileIn F = {d_text + (f ? n_s : 0), f ? n_s : 0, nbytes[f], d_ls[f], n_nl[f], nl[f], (uint32_t)f};
            sam_header<<<grid_for(nl[f], T), T>>>(F, d_cnt + 3);
            SCU(cudaGetLastError());
        }
        SCU(cudaMemcpy(&first[f], d_cnt + 3, sizeof(u64), cudaMemcpyDeviceToHost));
    }
    cnt[3] = 0;
    SCU(cudaMemcpy(d_cnt, cnt, sizeof(cnt), cudaMemcpyHostToDevice));
    ng = (nl[0] - first[0]) + (nl[1] - first[1]);
    SCU(hc_scratch_alloc((void**)&d_aln, (ng + 1) * sizeof(Aln)));
    SCU(hc_scratch_alloc((void**)&d_mapped, (ng + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_nops, (ng + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rev, (ng + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(ng + 1) * sizeof(u64)));
    for (int f = 0; f < 2; f++) {
        if (nl[f] == first[f]) continue;
        FileIn F = {d_text + (f ? n_s : 0), f ? n_s : 0, nbytes[f], d_ls[f], n_nl[f], nl[f], (uint32_t)f};
        sam_parse<<<grid_for(nl[f] - first[f], T), T>>>(F, first[f], f ? nl[0] - first[0] : 0, N, d_aln, d_mapped, d_nops, d_rev, d_cnt);
        SCU(cudaGetLastError());
    }
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (cnt[0] != NO_ERR || cnt[1] != NO_ERR) goto input_error;
    // the CIGAR runs
    SCU(hc_scratch_alloc((void**)&d_ooff, (ng + 1) * sizeof(u64)));
    hc_scan::exclusive_u32(d_nops, ng, d_ooff, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&n_ops, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_ops, (n_ops + 1) * sizeof(u64)));
    sam_ops<<<grid_for(ng, T), T>>>(d_text, d_mapped, d_ooff, ng, d_aln, d_ops);
    SCU(cudaGetLastError());
    hc_scratch_free(d_ooff); d_ooff = nullptr;
    // singles: the mapped lines of the single-end file in file order; counts
    SCU(hc_scratch_alloc((void**)&d_mpos, (ng + 1) * sizeof(u64)));
    {
        const u64 n0 = nl[0] - first[0], n1 = nl[1] - first[1];
        hc_scan::exclusive_u32(d_mapped, n0, d_mpos, d_tot, d_bsum, 0);
        SCU(cudaMemcpy(&nsm, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
        SCU(hc_scratch_alloc((void**)&d_smidx, (nsm + 1) * sizeof(uint32_t)));
        sam_gather_mapped<<<grid_for(n0, T), T>>>(d_mapped, d_mpos, 0, n0, d_smidx);
        hc_scan::exclusive_u32(d_rev, n0, d_mpos, d_tot, d_bsum, 0);
        SCU(cudaMemcpy(&stats->reverse_s, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
        stats->unmapped_s = n0 - nsm;
        hc_scan::exclusive_u32(d_mapped + n0, n1, d_mpos, d_tot, d_bsum, 0);
        SCU(cudaMemcpy(&nm, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
        stats->unmapped_p = n1 - nm;
        SCU(hc_scratch_alloc((void**)&d_pmidx, (nm + 1) * sizeof(uint32_t)));
        sam_gather_mapped<<<grid_for(n1, T), T>>>(d_mapped, d_mpos, n0, n1, d_pmidx);
        SCU(cudaGetLastError());
    }
    // pairing
    SCU(hc_scratch_alloc((void**)&d_st, (nm + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rx, (nm + 1) * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_acc, (nm + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_apos, (nm + 1) * sizeof(u64)));
    sam_run_starts<<<grid_for(nm, T), T>>>(d_text, d_aln, d_pmidx, nm, d_st);
    hc_scan::exclusive_u32(d_st, nm, d_rx, d_tot, d_bsum, 0);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(&nruns, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_rfirst, (nruns + 1) * sizeof(uint32_t)));
    sam_run_first<<<grid_for(nm, T), T>>>(d_st, d_rx, nm, d_rfirst);
    sam_pairs<<<grid_for(nm, T), T>>>(d_aln, d_pmidx, d_st, d_rx, d_rfirst, nm, d_acc, d_cnt + 4, d_cnt);
    hc_scan::exclusive_u32(d_acc, nm, d_apos, d_tot, d_bsum, 0);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(&npairs, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (cnt[1] != NO_ERR) goto input_error;
    stats->discarded = cnt[4];
    stats->reverse_p = cnt[5];
    // records in (reference, position, singles first) order
    nrec = nsm + npairs;
    stats->total_alns = nrec;
    SCU(hc_scratch_alloc((void**)&d_rec, (nrec + 1) * sizeof(Rec)));
    SCU(hc_scratch_alloc((void**)&d_key, (nrec + 1) * sizeof(ulonglong2)));
    SCU(hc_scratch_alloc((void**)&d_key2, (nrec + 1) * sizeof(ulonglong2)));
    SCU(hc_scratch_alloc((void**)&d_val, (nrec + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_val2, (nrec + 1) * sizeof(uint32_t)));
    sam_records<<<grid_for(nsm + nm, T), T>>>(d_aln, d_smidx, nsm, d_pmidx, d_acc, d_apos, nm, d_rec, d_key, d_val);
    SCU(cudaGetLastError());
    SCU(hc_radix::sort_pairs(d_key, d_val, d_key2, d_val2, nrec, &d_skey, &d_ord));
    SCU(hc_scratch_alloc((void**)&d_srec, (nrec + 1) * sizeof(Rec)));
    sam_gather<<<grid_for(nrec, T), T>>>(d_ord, nrec, d_rec, d_srec);
    SCU(cudaGetLastError());
    hc_scratch_free(d_rec); d_rec = nullptr;
    hc_scratch_free(d_key); d_key = nullptr;
    hc_scratch_free(d_key2); d_key2 = nullptr;
    SCU(hc_scratch_alloc((void**)&d_info, (n_refs + 1) * sizeof(RefInfo)));
    if (n_refs) sam_ref_info<<<n_refs, T>>>(d_srec, nrec, d_rlen, d_info);
    SCU(cudaGetLastError());
    // the sweep: count, scan, write
    S.X = Ctx{d_text, d_aln, d_ops, min_ov};
    S.srec = d_srec; S.info = d_info; S.n = nrec;
    SCU(hc_scratch_alloc((void**)&d_nb, (nrec + 1) * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rc, (nrec + 1) * sizeof(RecCnt)));
    SCU(hc_scratch_alloc((void**)&d_boff, (nrec + 1) * sizeof(u64)));
    hc_scratch_free(d_bsum); d_bsum = nullptr;
    SCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(nrec + 1) * sizeof(u64)));
    sam_count<<<grid_for(nrec, T), T>>>(S, d_nb, d_rc, d_ovf, d_cnt);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(&ovf, d_ovf, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (cnt[2] != NO_ERR) goto input_error;
    if (ovf) goto too_big;
    hc_scan::exclusive_u32(d_nb, nrec, d_boff, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&out_bytes, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_rs, (n_refs + 1) * sizeof(hc_sam_ref_stats)));
    if (n_refs) sam_ref_stats<<<n_refs, T>>>(d_srec, d_rc, d_info, d_rs);
    SCU(cudaGetLastError());
    if (n_refs) SCU(cudaMemcpy(rs.data(), d_rs, n_refs * sizeof(hc_sam_ref_stats), cudaMemcpyDeviceToHost));
    for (uint32_t r = 0; r < n_refs; r++) stats->n_out_lines += rs[r].n_overlaps;
    *n_text_bytes = out_bytes;
    if (out_bytes > text_cap) goto capacity;
    SCU(hc_scratch_alloc((void**)&d_out, out_bytes + 1));
    sam_format<<<grid_for(nrec, T), T>>>(S, d_boff, d_out);
    SCU(cudaGetLastError());
    SCU(cudaDeviceSynchronize());
    t1 = now_ms();
    stats->device_ms = (float)(t1 - t0);
    if (out_bytes) SCU(hc_copy_d2h(text, d_out, out_bytes));
    stats->d2h_ms = (float)(now_ms() - t1);
    if (ref_stats && n_refs) memcpy(ref_stats, rs.data(), n_refs * sizeof(hc_sam_ref_stats));
    goto done;
input_error:
    {
        const unsigned long long e = cnt[0] != NO_ERR ? cnt[0] : (cnt[1] != NO_ERR ? cnt[1] : cnt[2]);
        const uint32_t f = (uint32_t)(e >> 34);
        stats->first_error_file = f;
        stats->first_error_line = (e >> 2) & 0xffffffffull;
        stats->first_error_status = (uint32_t)(e & 3);
        u64 se[2] = {0, nbytes[f]};
        SCU(cudaMemcpy(se, d_ls[f] + stats->first_error_line, (stats->first_error_line < n_nl[f] ? 2 : 1) * sizeof(u64), cudaMemcpyDeviceToHost));
        stats->first_error_offset = se[0];
        stats->first_error_length = se[1] - se[0];
    }
    *n_text_bytes = 0;
    stats->n_out_lines = 0;
    hc_set_last_error((std::string("hc_sam2overlaps: line ") + std::to_string(stats->first_error_line) + " of the " +
                       (stats->first_error_file ? "paired-end" : "single-end") + " SAM text" +
                       (stats->first_error_status == HC_SAM_DIES ? " is one the host converter exits on" : " is outside what the device path covers")).c_str());
    rc = HC_ERR_INPUT;
    goto done;
too_big:
    hc_set_last_error("hc_sam2overlaps: one alignment's lines take 2^32 bytes or more (the device path counts them with 32 bits)");
    rc = HC_ERR_NOMEM;
    goto done;
capacity:
    hc_set_last_error("hc_sam2overlaps: text buffer too small (required size returned in n_text_bytes)");
    rc = HC_ERR_CAPACITY;
done:
    cudaFree(d_ls[0]); cudaFree(d_ls[1]);
    hc_scratch_free(d_text); hc_scratch_free(d_names); hc_scratch_free(d_out); hc_scratch_free(d_noff); hc_scratch_free(d_tot);
    hc_scratch_free(d_bsum); hc_scratch_free(d_ooff); hc_scratch_free(d_ops); hc_scratch_free(d_mpos); hc_scratch_free(d_rx);
    hc_scratch_free(d_apos); hc_scratch_free(d_boff); hc_scratch_free(d_perm); hc_scratch_free(d_nidx); hc_scratch_free(d_mapped);
    hc_scratch_free(d_nops); hc_scratch_free(d_rev); hc_scratch_free(d_smidx); hc_scratch_free(d_pmidx); hc_scratch_free(d_st);
    hc_scratch_free(d_rfirst); hc_scratch_free(d_acc); hc_scratch_free(d_val); hc_scratch_free(d_val2); hc_scratch_free(d_nb);
    hc_scratch_free(d_ovf); hc_scratch_free(d_cnt); hc_scratch_free(d_rlen); hc_scratch_free(d_aln);
    hc_scratch_free(d_rec); hc_scratch_free(d_srec); hc_scratch_free(d_info); hc_scratch_free(d_rc); hc_scratch_free(d_rs);
    hc_scratch_free(d_key); hc_scratch_free(d_key2);
    return rc;
}
