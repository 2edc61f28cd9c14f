// hc_sfo.cu -- hc_sfo2overlaps: the overlapper's SFO lines -> the 13-column overlaps file, built in HBM.  The host
// converter (host/hcb_sfo2overlaps.cpp, scripts/sfo2overlaps.py of the reference in C++) is the specification; the
// points below name its lines.
//
//   1. Temporary line (:311-348).  Each line is split on whitespace (split_ws :75), must have 8 fields (:318) and six
//      numeric fields parse_long accepts (:321,:325); the sfo ids map to original ids (original_id :89, asserting the
//      range when NP > 0).  Not flipped: put_long(na) \t put_long(nb) \t and then the original line byte for byte (:340:
//      spaces, repeated whitespace, a trailing '\r' stay; only '\n' is stripped, :315).  Flipped (na > nb, :323): ids
//      and sfo ids swap; for ori "I" OHA / OHB swap as strings, for any other ori they are negated and printed with
//      put_long (:331-336); OLA / OLB swap as strings and K follows as it was (:337).
//   2. Sort and uniq (:353-360).  Order by the numeric keys (idA, idB, sfoA, sfoB) (rec_less :186), ties by the bytes of
//      the temporary line, unsigned, the shorter first on a common prefix (text_cmp :52); adjacent lines with equal text
//      are dropped.  Equal text means equal keys, so the stable LSD radix sort of the 128-bit key (ids below 2^32) plus
//      a text order inside every run of equal keys is enough.
//   3. Kinds (:364-371).  idA == idB is skipped; neither id paired (is_paired :95) makes a single-single line
//      (s_s_overlap :106, put_ss_line :142); otherwise the line belongs to the group of its (idA, idB) (:375-388).
//   4. Groups (:398-412).  The lines of a group are matched pairwise, i < j, in sorted order (paired_overlap :148) with
//      the paired flags of the NEXT group's ids (:402-404); the last group is never matched and a one-line group writes
//      nothing (:401).
//   5. Output order and uniq (:415-432).  A group's lines come out immediately before the first line of the next group;
//      the final uniq drops every output line equal to the one before it in that order, across item boundaries (:423).
//   6. Floating point.  perc = min(round((double)(100 ovlen) / (double)minlen), 100) (:123-127): an IEEE division and
//      round-half-away, bit for bit the host's.  min(lenA, lenB) <= 0 is where the host dies (:121,:129).
//
// Device steps: newline index (hc_text.cuh) -> parse (record, key, temporary length) -> scan -> temporary text -> radix
// sort of (key, line) -> one thread per run of equal keys orders it by text -> repeats marked and compacted -> group
// starts (scan) -> per sorted line the bytes and lines of its item: a single-single line, or a row i of a matched group
// (the tests (i, j > i), so no thread is left with a group's m^2 / 2 tests) -> scans -> format -> the final uniq by
// comparing each output line with its predecessor -> compaction -> one hc_copy_d2h.
#include <cmath>
#include <cstring>
#include <string>
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

constexpr int INSERTION_MAX = 32;
constexpr i64 BIG = 1ll << 40;             // |OHA|, |OHB|, |OLA|, |OLB| below this: no sum or product of them overflows

struct SfoRec {                            // a temporary line's numbers (host Rec :44)
    uint32_t idA, idB, sfoA, sfoB;
    i64 oha, ohb, ola, olb;
    uint32_t tlen;                         // bytes of the temporary line
    uint8_t ori;                           // the ori field if it is one byte, else '?'
    uint8_t flip, isI;
};

struct Params { i64 ns, np, lim; };        // lim = NS + 2 NP (clamped): the sfo id range when NP > 0

__device__ __forceinline__ bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f' || c == '\n'; }

// split_ws (:75) of [b, e): the first 8 fields; returns the field count (9 means "more than 8")
__device__ int split8(const char* t, u64 b, u64 e, u64* fb, u64* fe) {
    int n = 0;
    u64 p = b;
    while (p < e) {
        while (p < e && is_ws(t[p])) p++;
        if (p >= e) break;
        const u64 s = p;
        while (p < e && !is_ws(t[p])) p++;
        if (n == 8) return 9;
        fb[n] = s; fe[n] = p;
        n++;
    }
    return n;
}

// parse_long (:59); *nd = digits after the sign (more than 18: the host's long may overflow, the value is not used)
__device__ bool parse_num(const char* t, u64 b, u64 e, i64* v, int* nd) {
    if (b == e) return false;
    bool neg = false;
    if (t[b] == '+' || t[b] == '-') { neg = t[b] == '-'; b++; }
    if (b == e) return false;
    *nd = (int)(e - b < 100 ? e - b : 100);
    i64 x = 0;
    for (u64 p = b; p < e; p++) {
        const char c = t[p];
        if (c < '0' || c > '9') return false;
        if (*nd <= 18) x = x * 10 + (c - '0');
    }
    *v = neg ? -x : x;
    return true;
}

__device__ __forceinline__ int dec_len(i64 v) {       // bytes put_long (:133) writes
    unsigned long long u = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
    int d = 1;
    while (u >= 10) { u /= 10; d++; }
    return d + (v < 0);
}

struct Sink {                                         // counts bytes; writes them too when p != nullptr
    char* p;
    u64 n;
    __device__ void c(char x) { if (p) p[n] = x; n++; }
    __device__ void num(i64 v) {
        const int d = dec_len(v);
        if (p) {
            unsigned long long u = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
            char* q = p + n;
            if (v < 0) *q = '-';
            for (int k = d - 1; k >= (v < 0); k--) { q[k] = (char)('0' + u % 10); u /= 10; }
        }
        n += d;
    }
    __device__ void str(const char* t, u64 b, u64 e) {
        if (p) for (u64 i = b; i < e; i++) p[n + (i - b)] = t[i];
        n += e - b;
    }
};

__device__ __forceinline__ void line_span(const char* t, u64 n, const u64* ls, u64 n_nl, u64 k, u64* b, u64* le) {
    *b = ls[k];
    u64 e = k < n_nl ? ls[k + 1] : n;
    while (e > *b && t[e - 1] == '\n') e--;
    *le = e;
}

// the temporary line (:328-342) into s; fb / fe: the 8 fields
__device__ void temp_line(Sink& s, const char* t, u64 b, u64 le, const u64* fb, const u64* fe, const SfoRec& r) {
    s.num(r.idA); s.c('\t'); s.num(r.idB); s.c('\t');
    if (!r.flip) { s.str(t, b, le); return; }
    s.str(t, fb[1], fe[1]); s.c('\t'); s.str(t, fb[0], fe[0]); s.c('\t'); s.str(t, fb[2], fe[2]); s.c('\t');
    if (r.isI) { s.str(t, fb[4], fe[4]); s.c('\t'); s.str(t, fb[3], fe[3]); }
    else { s.num(r.oha); s.c('\t'); s.num(r.ohb); }
    s.c('\t'); s.str(t, fb[6], fe[6]); s.c('\t'); s.str(t, fb[5], fe[5]); s.c('\t'); s.str(t, fb[7], fe[7]);
}

// one thread per line: record, key (idA, idB | sfoA, sfoB), temporary length; the first bad line -> *err = line << 2 | status
__global__ void sfo_parse(const char* __restrict__ t, u64 n, const u64* __restrict__ ls, u64 n_nl, u64 nl, Params P,
                          SfoRec* __restrict__ rec, ulonglong2* __restrict__ key, uint32_t* __restrict__ idx,
                          uint32_t* __restrict__ tlen, unsigned long long* err) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < nl; k += (u64)gridDim.x * blockDim.x) {
        u64 b, le, fb[8], fe[8];
        line_span(t, n, ls, n_nl, k, &b, &le);
        const int nf = split8(t, b, le, fb, fe);
        i64 v[7] = {0, 0, 0, 0, 0, 0, 0};
        int nd[7] = {0, 0, 0, 0, 0, 0, 0};
        uint32_t status = 0;
        if (nf != 8) status = HC_SFO_DIES;
        for (int f = 0; f < 7 && !status; f++)
            if (f != 2 && !parse_num(t, fb[f], fe[f], &v[f], &nd[f])) status = HC_SFO_DIES;
        for (int f = 0; f < 7 && !status; f++)
            if (f != 2 && nd[f] > 18) status = HC_SFO_DECLINED;
        const i64 sa = v[0], sb = v[1];
        if (!status && P.np > 0 && !(sa >= 0 && sa < P.lim && sb >= 0 && sb < P.lim)) status = HC_SFO_DIES;
        const i64 na = P.np == 0 ? sa : (sa < P.ns + P.np ? sa : sa - P.np);
        const i64 nb = P.np == 0 ? sb : (sb < P.ns + P.np ? sb : sb - P.np);
        if (!status && (sa < 0 || sa >= (1ll << 32) || sb < 0 || sb >= (1ll << 32) || na < 0 || nb < 0)) status = HC_SFO_DECLINED;
        for (int f = 3; f < 7 && !status; f++)
            if (v[f] >= BIG || v[f] <= -BIG) status = HC_SFO_DECLINED;
        if (status) {
            atomicMin(err, (unsigned long long)(k << 2 | status));
            tlen[k] = 0;
            continue;
        }
        SfoRec r;
        r.flip = na > nb;
        r.isI = fe[2] - fb[2] == 1 && t[fb[2]] == 'I';
        r.ori = fe[2] - fb[2] == 1 ? (uint8_t)t[fb[2]] : (uint8_t)'?';
        if (r.flip) {
            r.idA = (uint32_t)nb; r.idB = (uint32_t)na; r.sfoA = (uint32_t)sb; r.sfoB = (uint32_t)sa;
            if (r.isI) { r.oha = v[4]; r.ohb = v[3]; } else { r.oha = -v[3]; r.ohb = -v[4]; }
            r.ola = v[6]; r.olb = v[5];
        } else {
            r.idA = (uint32_t)na; r.idB = (uint32_t)nb; r.sfoA = (uint32_t)sa; r.sfoB = (uint32_t)sb;
            r.oha = v[3]; r.ohb = v[4]; r.ola = v[5]; r.olb = v[6];
        }
        Sink s = {nullptr, 0};
        temp_line(s, t, b, le, fb, fe, r);
        r.tlen = (uint32_t)s.n;
        rec[k] = r;
        key[k] = make_ulonglong2((u64)r.sfoA << 32 | r.sfoB, (u64)r.idA << 32 | r.idB);
        idx[k] = (uint32_t)k;
        tlen[k] = r.tlen;
    }
}

__global__ void sfo_temp(const char* __restrict__ t, u64 n, const u64* __restrict__ ls, u64 n_nl, u64 nl,
                         const SfoRec* __restrict__ rec, const u64* __restrict__ toff, char* __restrict__ tmp) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < nl; k += (u64)gridDim.x * blockDim.x) {
        u64 b, le, fb[8], fe[8];
        line_span(t, n, ls, n_nl, k, &b, &le);
        split8(t, b, le, fb, fe);
        Sink s = {tmp + toff[k], 0};
        temp_line(s, t, b, le, fb, fe, rec[k]);
    }
}

// text_cmp (:52) of the temporary lines of lines a and b
__device__ int tcmp(const char* tmp, const u64* toff, const SfoRec* rec, uint32_t a, uint32_t b) {
    const unsigned char* x = reinterpret_cast<const unsigned char*>(tmp + toff[a]);
    const unsigned char* y = reinterpret_cast<const unsigned char*>(tmp + toff[b]);
    const uint32_t la = rec[a].tlen, lb = rec[b].tlen, m = la < lb ? la : lb;
    for (uint32_t i = 0; i < m; i++) if (x[i] != y[i]) return x[i] < y[i] ? -1 : 1;
    return la < lb ? -1 : (la > lb ? 1 : 0);
}

struct TextLess {
    const char* tmp; const u64* toff; const SfoRec* rec;
    __device__ bool operator()(uint32_t a, uint32_t b) const { return tcmp(tmp, toff, rec, a, b) < 0; }
};

__device__ void sift_down(const TextLess& lt, uint32_t* v, uint32_t root, uint32_t m) {
    while (true) {
        uint32_t c = 2 * root + 1;
        if (c >= m) return;
        if (c + 1 < m && lt(v[c], v[c + 1])) c++;
        if (!lt(v[root], v[c])) return;
        const uint32_t x = v[root]; v[root] = v[c]; v[c] = x;
        root = c;
    }
}

__device__ __forceinline__ bool same_key(const ulonglong2& a, const ulonglong2& b) { return a.x == b.x && a.y == b.y; }

// one thread per run of equal keys: the run's lines in text order (insertion sort up to 32, heap sort beyond; on a run of
// identical lines the heap sort is linear)
__global__ void sfo_runs(const ulonglong2* __restrict__ key, uint32_t* __restrict__ ord, u64 n, TextLess lt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const ulonglong2 k = key[i];
        if (i > 0 && same_key(key[i - 1], k)) continue;
        u64 j = i + 1;
        while (j < n && same_key(key[j], k)) j++;
        const uint32_t m = (uint32_t)(j - i);
        if (m < 2) continue;
        uint32_t* v = ord + i;
        if (m <= INSERTION_MAX) {
            for (uint32_t a = 1; a < m; a++) {
                const uint32_t x = v[a];
                uint32_t c = a;
                while (c > 0 && lt(x, v[c - 1])) { v[c] = v[c - 1]; c--; }
                v[c] = x;
            }
        } else {
            for (uint32_t r = m / 2; r-- > 0;) sift_down(lt, v, r, m);
            for (uint32_t e = m - 1; e > 0; e--) {
                const uint32_t x = v[0]; v[0] = v[e]; v[e] = x;
                sift_down(lt, v, 0, e);
            }
        }
    }
}

// keep[i] = sorted line i differs from line i - 1 (uniq :355-360)
__global__ void sfo_marks(const ulonglong2* __restrict__ key, const uint32_t* __restrict__ ord, u64 n, TextLess lt,
                          uint32_t* __restrict__ keep) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        keep[i] = i == 0 || !same_key(key[i - 1], key[i]) || tcmp(lt.tmp, lt.toff, lt.rec, ord[i - 1], ord[i]) != 0;
}

__global__ void sfo_compact(const uint32_t* __restrict__ ord, const uint32_t* __restrict__ keep, const u64* __restrict__ pos, u64 n,
                            uint32_t* __restrict__ uq) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (keep[i]) uq[pos[i]] = ord[i];
}

__global__ void sfo_gather(const uint32_t* __restrict__ uq, u64 nu, const SfoRec* __restrict__ rec, SfoRec* __restrict__ srec) {
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < nu; u += (u64)gridDim.x * blockDim.x) srec[u] = rec[uq[u]];
}

__device__ __forceinline__ bool paired(const Params& P, uint32_t id) { return P.np > 0 && (i64)id >= P.ns; }   // is_paired :95
__device__ __forceinline__ int kind_of(const Params& P, const SfoRec& r) {                                    // :368-370
    if (r.idA == r.idB) return 0;
    return (!paired(P, r.idA) && !paired(P, r.idB)) ? 1 : 2;
}

// gf[u] = 1 iff unique line u is the first line of a group (srec: the unique lines in sorted order)
__global__ void sfo_group_firsts(const SfoRec* __restrict__ srec, u64 nu, Params P, uint32_t* __restrict__ gf) {
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < nu; u += (u64)gridDim.x * blockDim.x) {
        const SfoRec r = srec[u];
        bool f = kind_of(P, r) == 2;
        if (f && u > 0) { const SfoRec q = srec[u - 1]; f = q.idA != r.idA || q.idB != r.idB; }
        gf[u] = f;
    }
}

__global__ void sfo_group_starts(const uint32_t* __restrict__ gf, const u64* __restrict__ gx, u64 nu, uint32_t* __restrict__ gstart) {
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < nu; u += (u64)gridDim.x * blockDim.x)
        if (gf[u]) gstart[gx[u]] = (uint32_t)u;
}

struct SS { i64 id1, id2, pos1, perc, len1; char ori1, ori2; bool bad; };

__device__ SS s_s_overlap(const SfoRec& r) {           // :106-131
    SS o;
    const char ori = r.ori == 'N' ? '+' : '-';
    const i64 ovlen = r.ola < r.olb ? r.ola : r.olb;
    i64 lenA, lenB;
    if (r.oha >= 0) {
        if (r.ohb >= 0) { lenA = r.ola + r.oha; lenB = r.olb + r.ohb; }
        else { lenA = r.ola + r.oha - r.ohb; lenB = r.olb; }
        o.id1 = r.idA; o.id2 = r.idB; o.pos1 = r.oha; o.ori1 = '+'; o.ori2 = ori;
    } else {
        if (r.ohb >= 0) { lenA = r.ola; lenB = -r.oha + r.olb + r.ohb; }
        else { lenA = r.ola - r.ohb; lenB = -r.oha + r.olb; }
        o.id1 = r.idB; o.id2 = r.idA; o.pos1 = -r.oha; o.ori1 = ori; o.ori2 = '+';
    }
    const i64 minlen = lenA < lenB ? lenA : lenB;
    o.bad = minlen <= 0;
    o.perc = 0;
    if (!o.bad) {
        const double x = round((double)(100 * ovlen) / (double)minlen);
        o.perc = (i64)(x < 100.0 ? x : 100.0);
    }
    o.len1 = ovlen;
    return o;
}

__device__ void put_ss_line(Sink& s, const SS& o) {     // :142-145
    s.num(o.id1); s.c('\t'); s.num(o.id2); s.c('\t'); s.num(o.pos1); s.c('\t'); s.c('-'); s.c('\t'); s.c('-'); s.c('\t');
    s.c(o.ori1); s.c('\t'); s.c(o.ori2); s.c('\t'); s.num(o.perc); s.c('\t'); s.c('-'); s.c('\t'); s.num(o.len1);
    s.c('\t'); s.c('-'); s.c('\t'); s.c('s'); s.c('\t'); s.c('s'); s.c('\n');
}

// paired_overlap :148-184: 0 no match, else the line goes to s; *bad_line = the line whose s_s_overlap dies (or ~0)
__device__ bool paired_overlap(Sink& s, const SfoRec& c1, const SfoRec& c2, uint32_t l1, uint32_t l2, bool typeA, bool typeB,
                               unsigned long long* bad_line) {
    *bad_line = ~0ull;
    if (c1.ori != c2.ori) return false;
    int first = 0;
    const bool N = c1.ori == 'N', I = c1.ori == 'I';
    if (typeA && typeB) {
        if (N) { if (c1.sfoA < c2.sfoA && c1.sfoB < c2.sfoB) first = 1; else if (c1.sfoA > c2.sfoA && c1.sfoB > c2.sfoB) first = 2; }
        else if (I) { if (c1.sfoA < c2.sfoA && c1.sfoB > c2.sfoB) first = 1; else if (c1.sfoA > c2.sfoA && c1.sfoB < c2.sfoB) first = 2; }
    } else if (typeA && !typeB) {
        if (N) { if (c1.sfoA < c2.sfoA && c1.oha < c2.oha) first = 1; else if (c1.sfoA > c2.sfoA && c1.oha > c2.oha) first = 2; }
        else if (I) { if (c1.sfoA < c2.sfoA && c1.oha > c2.oha) first = 2; else if (c1.sfoA > c2.sfoA && c1.oha < c2.oha) first = 1; }
    } else {
        if (N) { if (c1.sfoB < c2.sfoB && c1.oha < c2.oha) first = 1; else if (c1.sfoB > c2.sfoB && c1.oha > c2.oha) first = 2; }
        else if (I) { if (c1.sfoB < c2.sfoB && c1.oha > c2.oha) first = 2; else if (c1.sfoB > c2.sfoB && c1.oha < c2.oha) first = 1; }
    }
    if (!first) return false;
    const SS o1 = s_s_overlap(first == 1 ? c1 : c2), o2 = s_s_overlap(first == 1 ? c2 : c1);
    if (o1.bad || o2.bad) {
        *bad_line = o1.bad ? (first == 1 ? l1 : l2) : (first == 1 ? l2 : l1);
        return true;
    }
    char t1, t2;
    if (o1.id1 == c1.idA) { t1 = typeA ? 'p' : 's'; t2 = typeB ? 'p' : 's'; }
    else { t1 = typeB ? 'p' : 's'; t2 = typeA ? 'p' : 's'; }
    char ord = '-';
    if (t1 == 'p' && t2 == 'p') ord = o1.id1 != o2.id1 ? '2' : '1';
    s.num(o1.id1); s.c('\t'); s.num(o1.id2); s.c('\t'); s.num(o1.pos1); s.c('\t'); s.num(o2.pos1); s.c('\t');
    s.c(ord); s.c('\t'); s.c(o1.ori1); s.c('\t'); s.c(o1.ori2); s.c('\t'); s.num(o1.perc); s.c('\t'); s.num(o2.perc); s.c('\t');
    s.num(o1.len1); s.c('\t'); s.num(o2.len1); s.c('\t'); s.c(t1); s.c('\t'); s.c(t2); s.c('\n');
    return true;
}

struct Groups {
    const uint32_t* uq; u64 nu; const SfoRec* rec; Params P;       // rec[u]: unique line u (sorted order), file line uq[u]
    const uint32_t* gf; const u64* gx; const uint32_t* gstart; u64 ng;
};

// The row of unique line u: its matched pairs (u, j > u) in j order, into s.  Returns false if u is not the row of a
// matched group (not a group line, or a line of the last group).
__device__ bool row(const Groups& G, u64 u, const SfoRec& r, Sink& s, uint32_t* cnt, unsigned long long* bad) {
    *cnt = 0;
    *bad = ~0ull;
    const u64 gid = G.gx[u] + G.gf[u] - 1;
    if (gid + 1 >= G.ng) return false;
    const SfoRec f = G.rec[G.gstart[gid + 1]];
    const bool ta = paired(G.P, f.idA), tb = paired(G.P, f.idB);
    for (u64 j = u + 1; j < G.nu; j++) {
        const SfoRec q = G.rec[j];
        if (q.idA != r.idA || q.idB != r.idB) break;
        unsigned long long b;
        if (paired_overlap(s, r, q, G.uq[u], G.uq[j], ta, tb, &b)) {
            if (b != ~0ull) { if (b < *bad) *bad = b; continue; }
            (*cnt)++;
        }
    }
    return true;
}

// per unique line: ss bytes (single-single), row bytes / lines (group line); dying lines -> *err; *ss_count, *ovf
__global__ void sfo_count(Groups G, uint32_t* __restrict__ sb, uint32_t* __restrict__ rb, uint32_t* __restrict__ rc,
                          unsigned long long* err, unsigned long long* ss_count, uint32_t* ovf) {
    unsigned long long n_ss = 0;
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < G.nu; u += (u64)gridDim.x * blockDim.x) {
        const uint32_t l = G.uq[u];
        const SfoRec r = G.rec[u];
        const int kind = kind_of(G.P, r);
        uint32_t s_bytes = 0, r_bytes = 0, r_cnt = 0;
        if (kind == 1) {
            const SS o = s_s_overlap(r);
            if (o.bad) atomicMin(err, (unsigned long long)l << 2 | HC_SFO_DIES);
            Sink s = {nullptr, 0};
            put_ss_line(s, o);
            s_bytes = (uint32_t)s.n;
            n_ss++;
        } else if (kind == 2) {
            Sink s = {nullptr, 0};
            unsigned long long bad;
            row(G, u, r, s, &r_cnt, &bad);
            if (bad != ~0ull) atomicMin(err, bad << 2 | HC_SFO_DIES);
            if (s.n >> 32) atomicOr(ovf, 1u);
            r_bytes = (uint32_t)s.n;
        }
        sb[u] = s_bytes; rb[u] = r_bytes; rc[u] = r_cnt;
    }
    n_ss = __reduce_add_sync(0xffffffffu, (unsigned)n_ss);     // blocks of whole warps; fewer than 2^32 lines
    if ((threadIdx.x & 31) == 0 && n_ss) atomicAdd(ss_count, n_ss);
}

// the item at unique line u: the previous group's rows (if u starts a group after the first) and then u's ss line
__global__ void sfo_slots(Groups G, const uint32_t* __restrict__ sb, const u64* __restrict__ rbx, const u64* __restrict__ rcx,
                          uint32_t* __restrict__ sl, uint32_t* __restrict__ sc, uint32_t* ovf) {
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < G.nu; u += (u64)gridDim.x * blockDim.x) {
        u64 gb = 0, gc = 0;
        if (G.gf[u] && G.gx[u] > 0) {
            const uint32_t p = G.gstart[G.gx[u] - 1];
            gb = rbx[u] - rbx[p];
            gc = rcx[u] - rcx[p];
        }
        const u64 bytes = gb + sb[u];
        if ((bytes >> 32) || (gc >> 32)) atomicOr(ovf, 1u);
        sl[u] = (uint32_t)bytes;
        sc[u] = (uint32_t)gc + (sb[u] != 0);
    }
}

// writes every item's lines at their places before the final uniq; ls_out[line] = its first byte
__global__ void sfo_format(Groups G, const uint32_t* __restrict__ sb, const uint32_t* __restrict__ rb, const u64* __restrict__ rbx,
                           const u64* __restrict__ rcx, const uint32_t* __restrict__ sl, const uint32_t* __restrict__ sc,
                           const u64* __restrict__ soff, const u64* __restrict__ loff, char* __restrict__ out, u64* __restrict__ ls_out) {
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < G.nu; u += (u64)gridDim.x * blockDim.x) {
        const SfoRec r = G.rec[u];
        if (sb[u]) {
            const u64 at = soff[u] + sl[u] - sb[u];
            ls_out[loff[u] + sc[u] - 1] = at;
            Sink s = {out + at, 0};
            put_ss_line(s, s_s_overlap(r));
        } else if (rb[u]) {
            const u64 gid = G.gx[u] + G.gf[u] - 1;
            const uint32_t f = G.gstart[gid + 1], g0 = G.gstart[gid];
            const u64 at = soff[f] + (rbx[u] - rbx[g0]);
            u64 li = loff[f] + (rcx[u] - rcx[g0]);
            const SfoRec nf = G.rec[f];
            const bool ta = paired(G.P, nf.idA), tb = paired(G.P, nf.idB);
            Sink s = {out + at, 0};
            for (u64 j = u + 1; j < G.nu; j++) {
                const SfoRec q = G.rec[j];
                if (q.idA != r.idA || q.idB != r.idB) break;
                const u64 before = s.n;
                unsigned long long b;
                if (paired_overlap(s, r, q, 0, 0, ta, tb, &b) && b == ~0ull) ls_out[li++] = at + before;
            }
        }
    }
}

// final uniq (:423): klen[L] = length of output line L if it differs from line L - 1, else 0
__global__ void sfo_out_marks(const char* __restrict__ out, const u64* __restrict__ ls_out, u64 nlines, uint32_t* __restrict__ klen,
                              unsigned long long* n_kept) {
    unsigned kept = 0;
    for (u64 L = (u64)blockIdx.x * blockDim.x + threadIdx.x; L < nlines; L += (u64)gridDim.x * blockDim.x) {
        const u64 s = ls_out[L], e = ls_out[L + 1];
        bool keep = true;
        if (L > 0) {
            const u64 ps = ls_out[L - 1];
            if (s - ps == e - s) {
                keep = false;
                for (u64 i = 0; i < e - s; i++) if (out[ps + i] != out[s + i]) { keep = true; break; }
            }
        }
        klen[L] = keep ? (uint32_t)(e - s) : 0u;
        kept += keep;
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_kept, (unsigned long long)kept);
}

__global__ void sfo_out_compact(const char* __restrict__ out, const u64* __restrict__ ls_out, const uint32_t* __restrict__ klen,
                                const u64* __restrict__ koff, u64 nlines, char* __restrict__ dst) {
    for (u64 L = (u64)blockIdx.x * blockDim.x + threadIdx.x; L < nlines; L += (u64)gridDim.x * blockDim.x) {
        const uint32_t m = klen[L];
        const char* s = out + ls_out[L];
        char* d = dst + koff[L];
        for (uint32_t i = 0; i < m; i++) d[i] = s[i];
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
            hc_set_last_error((std::string("hc_sfo2overlaps: ") + #call + ": " + cudaGetErrorString(_e)).c_str()); \
            rc = _e == cudaErrorMemoryAllocation ? HC_ERR_NOMEM : HC_ERR_CUDA;                                 \
            if (rc == HC_ERR_NOMEM) cudaGetLastError();                                                        \
            goto done;                                                                                         \
        }                                                                                                      \
    } while (0)

extern "C" int hc_sfo2overlaps(const char* sfo, uint64_t n_bytes, int64_t num_singles, int64_t num_pairs, char* text,
                               uint64_t text_cap, uint64_t* n_text_bytes, hc_sfo_stats* stats, int device) {
    if (!n_text_bytes || !stats || (text_cap && !text) || (n_bytes && !sfo)) {
        hc_set_last_error("hc_sfo2overlaps: NULL argument");
        return HC_ERR_ARG;
    }
    if (num_singles < 0 || num_pairs < 0) {
        hc_set_last_error("hc_sfo2overlaps: num_singles and num_pairs must not be negative");
        return HC_ERR_ARG;
    }
    *n_text_bytes = 0;
    memset(stats, 0, sizeof(*stats));
    stats->first_error_line = ~0ull;
    int rc = HC_OK;
    const int T = 256;
    Params P;
    P.ns = num_singles; P.np = num_pairs;
    P.lim = (num_singles >= (1ll << 61) || num_pairs >= (1ll << 60)) ? (1ll << 62) : num_singles + 2 * num_pairs;
    char *d_text = nullptr, *d_tmp = nullptr, *d_out = nullptr, *d_dst = nullptr;
    u64 *d_ls = nullptr, *d_toff = nullptr, *d_tot = nullptr, *d_bsum = nullptr, *d_pos = nullptr, *d_gx = nullptr, *d_rbx = nullptr,
        *d_rcx = nullptr, *d_soff = nullptr, *d_loff = nullptr, *d_lsout = nullptr, *d_koff = nullptr;
    unsigned long long* d_cnt = nullptr;        // [0] first error, [1] ss count, [2] kept output lines
    uint32_t *d_ovf = nullptr, *d_idx = nullptr, *d_idx2 = nullptr, *d_tlen = nullptr, *d_keep = nullptr, *d_uq = nullptr, *d_gf = nullptr,
             *d_gstart = nullptr, *d_sb = nullptr, *d_rb = nullptr, *d_rc = nullptr, *d_sl = nullptr, *d_sc = nullptr, *d_klen = nullptr;
    uint32_t *d_order = nullptr, ovf = 0;
    ulonglong2 *d_key = nullptr, *d_key2 = nullptr, *d_sorted = nullptr;
    SfoRec *d_rec = nullptr, *d_srec = nullptr;
    u64 n_nl = 0, nl = 0, tbytes = 0, nu = 0, ng = 0, pre_bytes = 0, pre_lines = 0, out_bytes = 0;
    unsigned long long cnt[3] = {~0ull, 0, 0};
    double t0 = 0, t1 = 0;
    TextLess lt;
    Groups G;
    SCU(cudaSetDevice(device));
    t0 = now_ms();
    if (n_bytes) {
        SCU(hc_scratch_alloc((void**)&d_text, n_bytes + 16));
        SCU(hc_copy_h2d(d_text, sfo, n_bytes));
    }
    t1 = now_ms();
    stats->h2d_ms = (float)(t1 - t0);
    t0 = t1;
    if (n_bytes == 0) goto finish;
    SCU(hc_line_index(d_text, n_bytes, &d_ls, &n_nl, &nl, 0));
    stats->n_lines = nl;
    if (nl >> 32) {
        stats->first_error_line = 1ull << 32;
        stats->first_error_status = HC_SFO_DECLINED;
        hc_set_last_error("hc_sfo2overlaps: 2^32 lines or more (the device path indexes lines with 32 bits)");
        rc = HC_ERR_INPUT;
        goto done;
    }
    SCU(hc_scratch_alloc((void**)&d_cnt, sizeof(cnt)));
    SCU(hc_scratch_alloc((void**)&d_ovf, sizeof(uint32_t)));
    SCU(cudaMemcpy(d_cnt, cnt, sizeof(cnt), cudaMemcpyHostToDevice));
    SCU(cudaMemset(d_ovf, 0, sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rec, nl * sizeof(SfoRec)));
    SCU(hc_scratch_alloc((void**)&d_key, nl * sizeof(ulonglong2)));
    SCU(hc_scratch_alloc((void**)&d_key2, nl * sizeof(ulonglong2)));
    SCU(hc_scratch_alloc((void**)&d_idx, nl * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_idx2, nl * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_tlen, nl * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_toff, nl * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_tot, sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(nl) * sizeof(u64)));
    sfo_parse<<<grid_for(nl, T), T>>>(d_text, n_bytes, d_ls, n_nl, nl, P, d_rec, d_key, d_idx, d_tlen, d_cnt);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    if (cnt[0] != ~0ull) goto input_error;
    hc_scan::exclusive_u32(d_tlen, nl, d_toff, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&tbytes, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_tmp, tbytes + 16));
    sfo_temp<<<grid_for(nl, T), T>>>(d_text, n_bytes, d_ls, n_nl, nl, d_rec, d_toff, d_tmp);
    SCU(cudaGetLastError());
    hc_scratch_free(d_text); d_text = nullptr;
    // sort | uniq
    SCU(hc_radix::sort_pairs(d_key, d_idx, d_key2, d_idx2, nl, &d_sorted, &d_order));
    lt.tmp = d_tmp; lt.toff = d_toff; lt.rec = d_rec;
    sfo_runs<<<grid_for(nl, T), T>>>(d_sorted, d_order, nl, lt);
    d_keep = d_tlen;                                   // the lengths are in d_toff now
    sfo_marks<<<grid_for(nl, T), T>>>(d_sorted, d_order, nl, lt, d_keep);
    SCU(cudaGetLastError());
    SCU(hc_scratch_alloc((void**)&d_pos, nl * sizeof(u64)));
    hc_scan::exclusive_u32(d_keep, nl, d_pos, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&nu, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    stats->n_unique = nu;
    d_uq = (d_order == d_idx) ? d_idx2 : d_idx;        // the buffer the sort did not leave its result in
    sfo_compact<<<grid_for(nl, T), T>>>(d_order, d_keep, d_pos, nl, d_uq);
    SCU(cudaGetLastError());
    hc_scratch_free(d_pos); d_pos = nullptr;
    hc_scratch_free(d_key); d_key = nullptr;
    hc_scratch_free(d_key2); d_key2 = nullptr;
    hc_scratch_free(d_tmp); d_tmp = nullptr;
    SCU(hc_scratch_alloc((void**)&d_srec, nu * sizeof(SfoRec)));
    sfo_gather<<<grid_for(nu, T), T>>>(d_uq, nu, d_rec, d_srec);
    SCU(cudaGetLastError());
    hc_scratch_free(d_rec); d_rec = nullptr;
    // groups
    SCU(hc_scratch_alloc((void**)&d_gf, nu * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_gx, nu * sizeof(u64)));
    sfo_group_firsts<<<grid_for(nu, T), T>>>(d_srec, nu, P, d_gf);
    hc_scan::exclusive_u32(d_gf, nu, d_gx, d_tot, d_bsum, 0);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(&ng, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_gstart, (ng + 1) * sizeof(uint32_t)));
    sfo_group_starts<<<grid_for(nu, T), T>>>(d_gf, d_gx, nu, d_gstart);
    // items: sizes, places, text
    G.uq = d_uq; G.nu = nu; G.rec = d_srec; G.P = P; G.gf = d_gf; G.gx = d_gx; G.gstart = d_gstart; G.ng = ng;
    SCU(hc_scratch_alloc((void**)&d_sb, nu * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rb, nu * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_rc, nu * sizeof(uint32_t)));
    sfo_count<<<grid_for(nu, T), T>>>(G, d_sb, d_rb, d_rc, d_cnt, d_cnt + 1, d_ovf);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(&ovf, d_ovf, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (cnt[0] != ~0ull) goto input_error;
    stats->s_s_count = cnt[1];
    if (ovf) goto too_big;
    SCU(hc_scratch_alloc((void**)&d_rbx, (nu + 1) * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_rcx, (nu + 1) * sizeof(u64)));
    hc_scan::exclusive_u32(d_rb, nu, d_rbx, d_tot, d_bsum, 0);
    hc_scan::exclusive_u32(d_rc, nu, d_rcx, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&stats->p_count, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(hc_scratch_alloc((void**)&d_sl, nu * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_sc, nu * sizeof(uint32_t)));
    sfo_slots<<<grid_for(nu, T), T>>>(G, d_sb, d_rbx, d_rcx, d_sl, d_sc, d_ovf);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(&ovf, d_ovf, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (ovf) goto too_big;
    SCU(hc_scratch_alloc((void**)&d_soff, nu * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_loff, nu * sizeof(u64)));
    hc_scan::exclusive_u32(d_sl, nu, d_soff, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&pre_bytes, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    hc_scan::exclusive_u32(d_sc, nu, d_loff, d_tot, d_bsum, 0);
    SCU(cudaMemcpy(&pre_lines, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    if (pre_lines == 0) goto finish;
    SCU(hc_scratch_alloc((void**)&d_out, pre_bytes));
    SCU(hc_scratch_alloc((void**)&d_lsout, (pre_lines + 1) * sizeof(u64)));
    SCU(cudaMemcpy(d_lsout + pre_lines, &pre_bytes, sizeof(u64), cudaMemcpyHostToDevice));
    sfo_format<<<grid_for(nu, T), T>>>(G, d_sb, d_rb, d_rbx, d_rcx, d_sl, d_sc, d_soff, d_loff, d_out, d_lsout);
    SCU(cudaGetLastError());
    // final uniq
    hc_scratch_free(d_bsum); d_bsum = nullptr;
    SCU(hc_scratch_alloc((void**)&d_bsum, hc_scan::blocks_for(pre_lines) * sizeof(u64)));
    SCU(hc_scratch_alloc((void**)&d_klen, pre_lines * sizeof(uint32_t)));
    SCU(hc_scratch_alloc((void**)&d_koff, pre_lines * sizeof(u64)));
    sfo_out_marks<<<grid_for(pre_lines, T), T>>>(d_out, d_lsout, pre_lines, d_klen, d_cnt + 2);
    hc_scan::exclusive_u32(d_klen, pre_lines, d_koff, d_tot, d_bsum, 0);
    SCU(cudaGetLastError());
    SCU(cudaMemcpy(&out_bytes, d_tot, sizeof(u64), cudaMemcpyDeviceToHost));
    SCU(cudaMemcpy(cnt, d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost));
    stats->n_out_lines = cnt[2];
    *n_text_bytes = out_bytes;
    if (out_bytes > text_cap) goto capacity;
    SCU(hc_scratch_alloc((void**)&d_dst, out_bytes));
    sfo_out_compact<<<grid_for(pre_lines, T), T>>>(d_out, d_lsout, d_klen, d_koff, pre_lines, d_dst);
    SCU(cudaGetLastError());
    SCU(cudaDeviceSynchronize());
    t1 = now_ms();
    stats->device_ms = (float)(t1 - t0);
    SCU(hc_copy_d2h(text, d_dst, out_bytes));
    stats->d2h_ms = (float)(now_ms() - t1);
    goto done;
finish:                                                 // no output line
    SCU(cudaDeviceSynchronize());
    stats->device_ms = (float)(now_ms() - t0);
    goto done;
input_error:
    stats->first_error_line = cnt[0] >> 2;
    stats->first_error_status = (uint32_t)(cnt[0] & 3);
    {
        u64 se[2] = {0, n_bytes};
        SCU(cudaMemcpy(se, d_ls + stats->first_error_line, (stats->first_error_line < n_nl ? 2 : 1) * sizeof(u64), cudaMemcpyDeviceToHost));
        stats->first_error_offset = se[0];
        stats->first_error_length = se[1] - se[0];
    }
    hc_set_last_error((std::string("hc_sfo2overlaps: line ") + std::to_string(stats->first_error_line) +
                       (stats->first_error_status == HC_SFO_DIES ? " is one the host converter exits on" : " is outside what the device path covers")).c_str());
    rc = HC_ERR_INPUT;
    goto done;
too_big:
    hc_set_last_error("hc_sfo2overlaps: a group writes 2^32 bytes or more (the device path counts them with 32 bits)");
    rc = HC_ERR_NOMEM;
    goto done;
capacity:
    hc_set_last_error("hc_sfo2overlaps: text buffer too small (required size returned in n_text_bytes)");
    rc = HC_ERR_CAPACITY;
done:
    cudaFree(d_ls);
    hc_scratch_free(d_text); hc_scratch_free(d_tmp); hc_scratch_free(d_out); hc_scratch_free(d_dst);
    hc_scratch_free(d_toff); hc_scratch_free(d_tot); hc_scratch_free(d_bsum); hc_scratch_free(d_pos); hc_scratch_free(d_gx);
    hc_scratch_free(d_rbx); hc_scratch_free(d_rcx); hc_scratch_free(d_soff); hc_scratch_free(d_loff); hc_scratch_free(d_lsout);
    hc_scratch_free(d_koff); hc_scratch_free(d_cnt); hc_scratch_free(d_ovf); hc_scratch_free(d_idx); hc_scratch_free(d_idx2);
    hc_scratch_free(d_tlen); hc_scratch_free(d_gf); hc_scratch_free(d_gstart); hc_scratch_free(d_sb); hc_scratch_free(d_rb);
    hc_scratch_free(d_rc); hc_scratch_free(d_sl); hc_scratch_free(d_sc); hc_scratch_free(d_klen); hc_scratch_free(d_key);
    hc_scratch_free(d_key2); hc_scratch_free(d_rec); hc_scratch_free(d_srec);
    return rc;
}
