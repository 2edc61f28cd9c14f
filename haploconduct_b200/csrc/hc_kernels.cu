// hc_kernels.cu -- sm_100a kernels of the overlap-edge scoring path.
//
// What the reference does per candidate (src/EdgeCalculator.cpp:143-385 -> :67-139 -> :26-56):
// pick one or two windows from read types / orientations / ord, walk each window base by base,
// add log p(q_A, q_B, match?) in double, count mismatches, skip N, then exp(mean) and three
// threshold tests (:404-413).
//
// How it is done here:
//   * hc_score_kernel     one warp owns a tile of 32 candidates.  Lane = candidate for window
//                         selection and for the final decision; in between, the tile's windows are
//                         cut into 32-position lane-chunks that are dealt round robin to the 32
//                         lanes, so short and long windows fill the warp equally well.  A lane-chunk
//                         is 2 aligned 128-bit loads of quality codes on the B side, up to 3 on the A
//                         side (re-aligned in registers: word mux + funnel shifts), 2-bit bases
//                         XOR/popc for the mismatch mask, and 32 shared-memory lookups of a
//                         fixed-point -log p table indexed by (code_A, code_B, mismatch) through one
//                         PRMT each.  Sums are integers, hence exact and order independent.
//                         Candidates whose mean lands within HC_FX_MARGIN of a threshold are queued for
//   * hc_exact_kernel     which re-adds the reference's own double addends in the reference's
//                         order (one thread per queued candidate), so every decision is bit-exact.
//   * hc_compact_*        order-preserving compaction of accepted edges / non-edge overlaps
//                         (count -> scan -> scatter): output order = input order = the reference's
//                         1-thread order.  The scatter places non-edge indices and, per edge, its source index;
//   * hc_emit_edges       one thread per accepted edge then evaluates exp() and the Edge fields (dense, so
//                         the 3.5 % of candidates that are edges do not stall the other lanes of the scatter).
// No tensor cores: nothing here is a contraction.
#include "hc_kernels.cuh"

namespace {

typedef unsigned long long u64;

struct Win {
    u64 xpos;         // position of A[pos] in the store's position space
    uint32_t ypos16;  // position of B[0] / 16
    uint32_t L;       // window length (src/EdgeCalculator.cpp:88); 0 when not scored
    uint32_t status;  // HC_WIN_*
    uint32_t hasN;    // a read of the window contains N
};

struct CandSetup {
    Win w[2];
    uint32_t two;   // two windows (any paired read involved)
    uint32_t err;
};

__device__ __forceinline__ hc_candidate load_candidate(const hc_kparams& P, u64 i) {
    hc_candidate c;
    if (P.cand_compact == 4u) {   // hc_candidate_entry6: 6 bytes (three 16-bit loads), run-encoded like hc_candidate_entry
        const uint16_t* hp = reinterpret_cast<const uint16_t*>(P.cand) + 3 * i;
        const uint32_t h0 = __ldg(hp), h1 = __ldg(hp + 1), h2 = __ldg(hp + 2);
        const uint32_t lo = h0 | (h1 << 16);               // bits 0-31 of the 48-bit record
        uint32_t r = __ldg(P.tile_run + (i >> 5));
        while ((uint32_t)i >= __ldg(P.run_start + r + 1)) r++;
        const uint32_t anchor = __ldg(P.run_anchor + r), other = lo & 0x01ffffffu;
        const bool anchor_is_2 = ((lo >> 25) & 1u) != 0u;
        c.idx1 = anchor_is_2 ? other : anchor;
        c.idx2 = anchor_is_2 ? anchor : other;
        c.pos1 = (lo >> 30) | ((h2 & 0x7fu) << 2);         // bits 30-38
        c.pos2 = h2 >> 7;                                  // bits 39-47
        c.len1 = c.len2 = 0; c.perc1 = c.perc2 = 0; c.type1 = c.type2 = 0; c.reserved = 0;
        c.ori1 = (lo >> 26) & 1u; c.ori2 = (lo >> 27) & 1u;
        const uint32_t o = (lo >> 28) & 3u;
        c.ord = o == 1 ? '1' : (o == 2 ? '2' : '-');
        return c;
    }
    if (P.cand_compact == 3u) {   // hc_candidate_entry: 8 bytes, the other read comes from the run the candidate lies in
        const uint2 e = __ldg(reinterpret_cast<const uint2*>(P.cand) + i);
        uint32_t r = __ldg(P.tile_run + (i >> 5));
        while ((uint32_t)i >= __ldg(P.run_start + r + 1)) r++;     // runs are rarely shorter than a tile
        const uint32_t anchor = __ldg(P.run_anchor + r), other = e.x & 0x7fffffffu;
        const bool anchor_is_2 = (e.x >> 31) != 0u;
        c.idx1 = anchor_is_2 ? other : anchor;
        c.idx2 = anchor_is_2 ? anchor : other;
        const uint32_t w = e.y;
        c.pos1 = w & 0x3fffu; c.pos2 = (w >> 14) & 0x3fffu;
        c.len1 = c.len2 = 0; c.perc1 = c.perc2 = 0; c.type1 = c.type2 = 0; c.reserved = 0;
        c.ori1 = (w >> 28) & 1u; c.ori2 = (w >> 29) & 1u;
        const uint32_t o = w >> 30;
        c.ord = o == 1 ? '1' : (o == 2 ? '2' : '-');
        return c;
    }
    if (P.cand_compact == 2u) {   // hc_candidate_short: 12 bytes, positions below 2^14
        const uint32_t* sp = reinterpret_cast<const uint32_t*>(P.cand) + 3 * i;
        const uint32_t w = __ldg(sp + 2);
        c.idx1 = __ldg(sp); c.idx2 = __ldg(sp + 1); c.pos1 = w & 0x3fffu; c.pos2 = (w >> 14) & 0x3fffu;
        c.len1 = c.len2 = 0; c.perc1 = c.perc2 = 0; c.type1 = c.type2 = 0; c.reserved = 0;
        c.ori1 = (w >> 28) & 1u; c.ori2 = (w >> 29) & 1u;
        const uint32_t o = w >> 30;
        c.ord = o == 1 ? '1' : (o == 2 ? '2' : '-');
        return c;
    }
    if (P.cand_compact) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(P.cand) + i);
        c.idx1 = a.x; c.idx2 = a.y; c.pos1 = a.z & 0x0fffffffu; c.pos2 = a.w;
        c.len1 = c.len2 = 0; c.perc1 = c.perc2 = 0; c.type1 = c.type2 = 0; c.reserved = 0;
        c.ori1 = (a.z >> 28) & 1u; c.ori2 = (a.z >> 29) & 1u;
        const uint32_t o = a.z >> 30;
        c.ord = o == 1 ? '1' : (o == 2 ? '2' : '-');
        return c;
    }
    const uint4* cp = reinterpret_cast<const uint4*>(P.cand) + 2 * i;
    const uint4 a = __ldg(cp), b = __ldg(cp + 1);
    c.idx1 = a.x; c.idx2 = a.y; c.pos1 = a.z; c.pos2 = a.w;
    c.len1 = b.x; c.len2 = b.y;
    c.perc1 = b.z & 0xff; c.perc2 = (b.z >> 8) & 0xff; c.ord = (b.z >> 16) & 0xff; c.ori1 = (b.z >> 24) & 0xff;
    c.ori2 = b.w & 0xff; c.type1 = (b.w >> 8) & 0xff; c.type2 = (b.w >> 16) & 0xff; c.reserved = 0;
    return c;
}

// overlap_score's guards and window length, src/EdgeCalculator.cpp:74-88.
// (rawA, slotA) / (rawB, slotB): length|HASN and forward slot start/16 of the two sequences.
__device__ __forceinline__ void make_window(const hc_kparams& P, uint32_t rawA, uint32_t slotA, int rcA, uint32_t rawB,
                                            uint32_t slotB, int rcB, uint32_t pos, Win& w) {
    const uint32_t lenA = rawA & HC_LEN_MASK, lenB = rawB & HC_LEN_MASK;
    w.L = 0;
    w.xpos = 0;
    w.ypos16 = 0;
    w.hasN = 0;
    if (pos >= lenA) { w.status = HC_WIN_POS_OOR; return; }
    if (lenA < P.min_read_len || lenB < P.min_read_len) { w.status = HC_WIN_SHORT; return; }
    const u64 sa = 16ull * slotA + (rcA ? hc_slot_size(lenA) : 0u);
    const u64 sb = 16ull * slotB + (rcB ? hc_slot_size(lenB) : 0u);
    w.xpos = sa + pos;
    w.ypos16 = (uint32_t)(sb >> 4);
    w.L = min(lenA - pos, lenB);
    w.status = HC_WIN_SCORED;
    w.hasN = ((rawA | rawB) & HC_HASN_BIT) ? 1u : 0u;
}

// Window selection of EdgeCalculator::compute_overlap, src/EdgeCalculator.cpp:199-351, written
// without the 13-way case split:
//   "first"/"second" mate of a paired read in orientation ori: (/1,/2) if '+', (/2,/1) if '-'  (:316-351)
//   window 1: A = read1.first (or its only sequence), B = read2.first                           pos1
//   window 2: a = read1.second (or its only sequence), b = read2.second (or its only sequence)  pos2
//             laid as (a, b), or as (b, a) for P-S (:278,:282,:286,:290) and for P-P with ord == 2
//             (:322,:331,:340,:349).
__device__ __forceinline__ void setup_windows(const hc_kparams& P, const hc_candidate& c, const uint4& r1, const uint4& r2,
                                              CandSetup& s) {
    // r.x/.y = slot16 of mate 0/1, r.z/.w = len|HASN of mate 0/1
    const int p1 = (r1.w & HC_LEN_MASK) != 0, p2 = (r2.w & HC_LEN_MASK) != 0;   // Read::is_paired()
    const int rc1 = c.ori1 ? 0 : 1, rc2 = c.ori2 ? 0 : 1;
    const int f1 = p1 ? rc1 : 0, s1 = p1 ? 1 - rc1 : 0;   // mate slot of first / second sequence of read 1
    const int f2 = p2 ? rc2 : 0, s2 = p2 ? 1 - rc2 : 0;
    s.two = (p1 | p2) ? 1u : 0u;
    s.err = 0;
    s.w[1].L = 0; s.w[1].xpos = 0; s.w[1].ypos16 = 0; s.w[1].hasN = 0; s.w[1].status = HC_WIN_UNUSED;
    if (p1 && p2) { if (c.ord != '1' && c.ord != '2') s.err = 1; }            // assert :369
    else if (P.n_single == 0) s.err = 1;                                        // :197, "Read types not recognized" :381
    make_window(P, f1 ? r1.w : r1.z, f1 ? r1.y : r1.x, rc1, f2 ? r2.w : r2.z, f2 ? r2.y : r2.x, rc2, c.pos1, s.w[0]);
    if (s.two) {
        const uint32_t ra = s1 ? r1.w : r1.z, sa = s1 ? r1.y : r1.x;
        const uint32_t rb = s2 ? r2.w : r2.z, sb = s2 ? r2.y : r2.x;
        const bool swapped = p1 && (!p2 || c.ord == '2');
        if (swapped) make_window(P, rb, sb, rc2, ra, sa, rc1, c.pos2, s.w[1]);
        else make_window(P, ra, sa, rc1, rb, sb, rc2, c.pos2, s.w[1]);
    }
    if (s.err) { s.w[0].L = s.w[1].L = 0; s.w[0].status = s.w[1].status = HC_WIN_UNUSED; }
}

// Edge::pos3 / pos4, src/EdgeCalculator.cpp:222, :262-263, :300-301, :361-372 (size_t arithmetic
// truncated to int == 32-bit wrap-around).
__device__ __forceinline__ void extra_pos(const hc_candidate& c, const uint4& r1, const uint4& r2, int32_t& pos3, int32_t& pos4) {
    const uint32_t l10 = r1.z & HC_LEN_MASK, l11 = r1.w & HC_LEN_MASK, l20 = r2.z & HC_LEN_MASK, l21 = r2.w & HC_LEN_MASK;
    const int p1 = l11 != 0, p2 = l21 != 0;
    if (!p1 && !p2) { pos3 = (int32_t)(l10 - c.pos1 - l20); pos4 = 0; }
    else if (!p1) { pos3 = (int32_t)(l10 - c.pos2 - l21); pos4 = (int32_t)(l10 - c.pos1 - l20); }
    else if (!p2) { pos3 = (int32_t)(l11 + c.pos2 - l20); pos4 = (int32_t)(l20 + c.pos1 - l10); }
    else {
        pos3 = c.ord == '1' ? (int32_t)(l11 - c.pos2 - l21) : (int32_t)(l11 + c.pos2 - l21);
        pos4 = (int32_t)(l10 - c.pos1 - l20);
    }
}

__device__ __forceinline__ bool load_and_setup(const hc_kparams& P, const hc_candidate& c, CandSetup& s, uint4& r1, uint4& r2) {
    if (c.idx1 >= P.n_reads || c.idx2 >= P.n_reads || c.idx1 == c.idx2) {
        s.err = 1; s.two = 0;
        s.w[0].L = s.w[1].L = 0; s.w[0].xpos = s.w[1].xpos = 0; s.w[0].ypos16 = s.w[1].ypos16 = 0;
        s.w[0].hasN = s.w[1].hasN = 0; s.w[0].status = s.w[1].status = HC_WIN_UNUSED;
        r1 = r2 = make_uint4(0, 0, 0, 0);
        return false;
    }
    r1 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + c.idx1));
    r2 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + c.idx2));
    setup_windows(P, c, r1, r2, s);
    return !s.err;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Pull the (randomly located) window data towards L2 while the tile is still being set up.
__device__ __forceinline__ void prefetch_window(const hc_kparams& P, const Win& w) {
    if (w.L == 0) return;
    const uint32_t n = min(w.L, 512u);
    if (P.packed) {
        const uint8_t* xa = P.pk + (w.xpos & ~127ull);
        const uint32_t xe = (uint32_t)(w.xpos & 127ull) + n;
        for (uint32_t o = 0; o < xe; o += 128) prefetch_l2(xa + o);
        const uint8_t* ya = P.pk + 16ull * w.ypos16;
        for (uint32_t o = 0; o < n; o += 128) prefetch_l2(ya + o);
        return;
    }
    const uint8_t* xa = P.qual + (w.xpos & ~127ull);
    const uint32_t xe = (uint32_t)(w.xpos & 127ull) + n;
    for (uint32_t o = 0; o < xe; o += 128) prefetch_l2(xa + o);
    const uint8_t* ya = P.qual + 16ull * w.ypos16;
    for (uint32_t o = 0; o < n; o += 128) prefetch_l2(ya + o);
    prefetch_l2(P.base2 + (w.xpos >> 4));
    prefetch_l2(P.base2 + ((w.xpos + n) >> 4));
    prefetch_l2(P.base2 + w.ypos16);
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// 32-byte load (LDG.256, sm_100): the L1 data pipe moves one 128-byte line per wavefront whatever the access width
// (tools/micro/l1_wavefronts.cu) and the lanes of a warp sit in about a dozen different lines, so what a lane-chunk
// costs there is its NUMBER of load instructions, not its bytes.
__device__ __forceinline__ void ldg256(const void* p, uint32_t* d) {
    asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7])
        : "l"(p));
}

// 16 positions: (A codes ^ swizzle(B codes)) | mismatch<<7 -> column byte, B code -> row byte,
// one PRMT per position builds the table index (upper bytes zero through PRMT's sign-replicate
// mode on the row byte, whose msb is always 0), 16 shared-memory lookups.
template <bool HAS_VOID>
__device__ __forceinline__ void lookup16(const uint32_t* __restrict__ T, const uint32_t* wa, const uint32_t* wy, uint32_t m,
                                         uint32_t& acc, uint32_t& orv) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        // mismatch bits of positions 4j..4j+3 (bits 0,2,4,6 of byte j of m) -> bit 7 of bytes 0..3
        const uint32_t mj = (m >> (8 * j)) & 0x55u;
        const uint32_t dep = (mj * 0x02082080u) & 0x80808080u;
        const uint32_t col = (wa[j] ^ hc_swz4(wy[j])) | dep;
        const uint32_t t0 = T[prmt(col, wy[j], 0xCC40u)];
        const uint32_t t1 = T[prmt(col, wy[j], 0xDD51u)];
        const uint32_t t2 = T[prmt(col, wy[j], 0xEE62u)];
        const uint32_t t3 = T[prmt(col, wy[j], 0xFF73u)];
        acc += (t0 + t1) + (t2 + t3);
        if (HAS_VOID) orv |= (t0 | t1) | (t2 | t3);
    }
}

// One 32-position lane-chunk of one window.  Returns the fixed-point sum of -log p over the chunk,
// the mismatch count, the number of N positions and whether a void (p < ps.mismatch) pair was hit.
template <bool HAS_VOID>
__device__ __forceinline__ void process32(const hc_kparams& P, const uint32_t* __restrict__ T, u64 xpos, uint32_t ypos16,
                                          uint32_t L, uint32_t hasN, uint32_t k, uint32_t& sum, uint32_t& mm, uint32_t& ncnt,
                                          uint32_t& vd) {
    const u64 xp = xpos + 32ull * k;
    const uint32_t n = min(L - 32u * k, 32u);   // 1..32 valid positions
    const uint32_t yq = ypos16 + 2u * k;        // even: slots start at multiples of 64 positions
    const uint32_t off = (uint32_t)xp & 15u;
    const bool two = n > 16u, x1 = off + n > 16u, x2 = off + n > 32u;
    const uint4 z4 = make_uint4(0, 0, 0, 0);
    // ---- loads, all issued before first use; blocks beyond the window are not touched
#ifndef HC_NO_LD256
    const uint32_t off32 = (uint32_t)xp & 31u;
    uint32_t QA[16], wy[8];
    const uint8_t* xb = P.qual + (xp & ~31ull);
    ldg256(xb, QA);
    if (off32 + n > 32u) ldg256(xb + 32, QA + 8);   // never beyond the slot: it holds window positions
    else {
#pragma unroll
        for (int i = 8; i < 16; i++) QA[i] = 0u;
    }
    ldg256(P.qual + 16ull * yq, wy);               // slots are padded by >= 32 zero bytes
    (void)two; (void)z4;
#else
    const uint4* xq = reinterpret_cast<const uint4*>(P.qual + (xp & ~15ull));
    const uint4 q0 = __ldg(xq);
    const uint4 q1 = x1 ? __ldg(xq + 1) : z4;
    const uint4 q2 = x2 ? __ldg(xq + 2) : z4;
    const uint4* yqp = reinterpret_cast<const uint4*>(P.qual) + yq;
    const uint4 y0 = __ldg(yqp);
    const uint4 y1 = two ? __ldg(yqp + 1) : z4;
#endif
    const uint32_t* bxp = P.base2 + (xp >> 4);
    const uint32_t b0 = __ldg(bxp);
    const uint32_t b1 = x1 ? __ldg(bxp + 1) : 0u;
    const uint32_t b2 = x2 ? __ldg(bxp + 2) : 0u;
    const uint2 by = __ldg(reinterpret_cast<const uint2*>(P.base2 + yq));
    // ---- mismatch masks in the 2-bit domain: XOR, fold pairs, popc
    const uint32_t bsh = off * 2u;
    const uint32_t xa0 = __funnelshift_r(b0, b1, bsh) ^ by.x;
    const uint32_t xa1 = __funnelshift_r(b1, b2, bsh) ^ by.y;
    uint32_t m0 = (xa0 | (xa0 >> 1)) & 0x55555555u;
    uint32_t m1 = (xa1 | (xa1 >> 1)) & 0x55555555u;
    if (n < 32u) {
        const uint32_t n0 = min(n, 16u), n1 = n - n0;
        m0 &= n0 >= 16u ? 0xffffffffu : ((1u << (2u * n0)) - 1u);
        m1 &= (1u << (2u * n1)) - 1u;   // n1 <= 15
    }
    ncnt = 0;
    if (hasN) {   // rare: either read contains an N (skipped positions, src/EdgeCalculator.cpp:35-39,122-124)
        const uint32_t* nap = P.nmask + (xp >> 5);
        const uint32_t na0 = __ldg(nap), na1 = __ldg(nap + 1);
        uint32_t nn = __funnelshift_r(na0, na1, (uint32_t)xp & 31u) | __ldg(P.nmask + (yq >> 1));
        if (n < 32u) nn &= (1u << n) - 1u;
        ncnt = __popc(nn);
        uint32_t s0 = nn & 0xffffu, s1 = nn >> 16;   // spread 16 bits to the even bit positions
        s0 = (s0 | (s0 << 8)) & 0x00ff00ffu; s1 = (s1 | (s1 << 8)) & 0x00ff00ffu;
        s0 = (s0 | (s0 << 4)) & 0x0f0f0f0fu; s1 = (s1 | (s1 << 4)) & 0x0f0f0f0fu;
        s0 = (s0 | (s0 << 2)) & 0x33333333u; s1 = (s1 | (s1 << 2)) & 0x33333333u;
        s0 = (s0 | (s0 << 1)) & 0x55555555u; s1 = (s1 | (s1 << 1)) & 0x55555555u;
        m0 &= ~s0;
        m1 &= ~s1;
    }
    mm = __popc(m0) + __popc(m1);
    // ---- A-side quality codes: select 9 of the 12 loaded words (word offset 0..3), then funnel by bytes
    const bool s2 = (off & 8u) != 0, s1 = (off & 4u) != 0;
    uint32_t V1[10], V[9];
#ifndef HC_NO_LD256
    const bool s4 = (off32 & 16u) != 0;
    uint32_t V2[12];
#pragma unroll
    for (int i = 0; i < 12; i++) V2[i] = s4 ? QA[i + 4] : QA[i];
#pragma unroll
    for (int i = 0; i < 10; i++) V1[i] = s2 ? V2[i + 2] : V2[i];
#else
    const uint32_t W[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
    for (int i = 0; i < 10; i++) V1[i] = s2 ? W[i + 2] : W[i];
    const uint32_t wy[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
#endif
#pragma unroll
    for (int i = 0; i < 9; i++) V[i] = s1 ? V1[i + 1] : V1[i];
    const uint32_t sh = (off & 3u) * 8u;
    uint32_t wa[8];
#pragma unroll
    for (int i = 0; i < 8; i++) wa[i] = __funnelshift_r(V[i], V[i + 1], sh);
    uint32_t acc = 0, orv = 0;
    lookup16<HAS_VOID>(T, wa, wy, m0, acc, orv);
    lookup16<HAS_VOID>(T, wa + 4, wy + 4, m1, acc, orv);
    sum = acc;
    vd = HAS_VOID ? ((orv & HC_VOID_BIT) ? 1u : 0u) : 0u;
}

// ---- packed layout (<= 63 quality codes): one byte per position = code | base << 6 ----------------------
// Re-align the A side exactly as in the planar kernel; the XOR of A and (swizzled) B bytes is at
// once the table column and, in bits 6-7, the base difference.  Mismatch flags of the 8 words are
// gathered into one 32-bit word (OR_j flags_j >> j) so that a single popc counts them.
#ifdef HC_NO_LD256
struct PkRow {          // the raw loads of one packed lane-chunk and what is needed to interpret them
    uint4 q0, q1, q2, y0, y1;
    uint32_t n, off, hasN;
};
#else
// 32-byte loads (ldg256) fetch the B side with one instruction and the A side with two instead of 2 + 3.
struct PkRow {
    uint32_t a[16];     // A side: the 64 bytes from the 32-byte boundary below the chunk (upper half zero when not needed)
    uint32_t y[8];      // B side: the chunk's 32 bytes (32-byte aligned by construction)
    uint32_t n, off, hasN;   // off = 0..31
};

#endif

__device__ __forceinline__ PkRow load32_packed(const hc_kparams& P, u64 xpos, uint32_t ypos16, uint32_t L, uint32_t hasN, uint32_t k) {
    PkRow r;
    const u64 xp = xpos + 32ull * k;
    r.n = min(L - 32u * k, 32u);   // 1..32 valid positions
    const uint32_t yq = ypos16 + 2u * k;
    r.hasN = hasN;
#ifndef HC_NO_LD256
    r.off = (uint32_t)xp & 31u;
    const uint8_t* xb = P.pk + (xp & ~31ull);
    ldg256(xb, r.a);
    if (r.off + r.n > 32u) ldg256(xb + 32, r.a + 8);   // never beyond the slot: it holds window positions
    else {
#pragma unroll
        for (int i = 8; i < 16; i++) r.a[i] = 0u;
    }
    ldg256(P.pk + 16ull * yq, r.y);                    // slots are padded by >= 32 zero bytes
    return r;
#else
    r.off = (uint32_t)xp & 15u;
    const bool two = r.n > 16u, x1 = r.off + r.n > 16u, x2 = r.off + r.n > 32u;
    const uint4 z4 = make_uint4(0, 0, 0, 0);
    const uint4* xq = reinterpret_cast<const uint4*>(P.pk + (xp & ~15ull));
    r.q0 = __ldg(xq);
    r.q1 = x1 ? __ldg(xq + 1) : z4;
    r.q2 = x2 ? __ldg(xq + 2) : z4;
    const uint4* yqp = reinterpret_cast<const uint4*>(P.pk) + yq;
    r.y0 = __ldg(yqp);
    r.y1 = two ? __ldg(yqp + 1) : z4;
    return r;
#endif
}

template <bool HAS_VOID>
__device__ __forceinline__ void compute32_packed(const uint32_t* __restrict__ T, const uint32_t* __restrict__ VM, const PkRow& r,
                                                 uint32_t& sum, uint32_t& mm, uint32_t& ncnt, uint32_t& vd) {
    const uint32_t n = r.n, off = r.off, hasN = r.hasN;
    const uint32_t vm = VM[n];
#ifndef HC_NO_LD256
    const bool s4 = (off & 16u) != 0, s2 = (off & 8u) != 0, s1 = (off & 4u) != 0;
    uint32_t V2[12], V1[10], V[9];
#pragma unroll
    for (int i = 0; i < 12; i++) V2[i] = s4 ? r.a[i + 4] : r.a[i];
#pragma unroll
    for (int i = 0; i < 10; i++) V1[i] = s2 ? V2[i + 2] : V2[i];
#pragma unroll
    for (int i = 0; i < 9; i++) V[i] = s1 ? V1[i + 1] : V1[i];
    const uint32_t sh = (off & 3u) * 8u;
    const uint32_t* wy = r.y;
#else
    const uint4 q0 = r.q0, q1 = r.q1, q2 = r.q2, y0 = r.y0, y1 = r.y1;
    const uint32_t W[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
    const bool s2 = (off & 8u) != 0, s1 = (off & 4u) != 0;
    uint32_t V1[10], V[9];
#pragma unroll
    for (int i = 0; i < 10; i++) V1[i] = s2 ? W[i + 2] : W[i];
#pragma unroll
    for (int i = 0; i < 9; i++) V[i] = s1 ? V1[i + 1] : V1[i];
    const uint32_t sh = (off & 3u) * 8u;
    const uint32_t wy[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
#endif
    uint32_t acc = 0, orv = 0, flags = 0, vw = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const uint32_t wa = __funnelshift_r(V[j], V[j + 1], sh);
        const uint32_t wb = wy[j];
        const uint32_t col = wa ^ hc_swz4_packed(wb);
        const uint32_t row = wb & 0x3f3f3f3fu;
        flags |= ((col | (col << 1)) & 0x80808080u) >> j;
        if (hasN) {   // a zero byte inside the window is an N (valid bases carry a code >= 1)
            const uint32_t nzA = (((wa & 0x7f7f7f7fu) + 0x7f7f7f7fu) | wa), nzB = (((wb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | wb);
            vw |= ((nzA & nzB) & 0x80808080u) >> j;
        }
        const uint32_t t0 = T[prmt(col, row, 0xCC40u)];
        const uint32_t t1 = T[prmt(col, row, 0xDD51u)];
        const uint32_t t2 = T[prmt(col, row, 0xEE62u)];
        const uint32_t t3 = T[prmt(col, row, 0xFF73u)];
        acc += (t0 + t1) + (t2 + t3);
        if (HAS_VOID) orv |= (t0 | t1) | (t2 | t3);
    }
    ncnt = 0;
    if (hasN) {
        const uint32_t valid = vw & vm;
        ncnt = n - __popc(valid);
        flags &= valid;
    } else {
        flags &= vm;
    }
    mm = __popc(flags);
    sum = acc;
    vd = HAS_VOID ? ((orv & HC_VOID_BIT) ? 1u : 0u) : 0u;
}

template <bool HAS_VOID>
__device__ __forceinline__ void process32_packed(const hc_kparams& P, const uint32_t* __restrict__ T,
                                                 const uint32_t* __restrict__ VM, u64 xpos, uint32_t ypos16, uint32_t L,
                                                 uint32_t hasN, uint32_t k, uint32_t& sum, uint32_t& mm, uint32_t& ncnt,
                                                 uint32_t& vd) {
    const PkRow r = load32_packed(P, xpos, ypos16, L, hasN, k);
    compute32_packed<HAS_VOID>(T, VM, r, sum, mm, ncnt, vd);
}

template <bool HAS_VOID, bool PACKED>
__device__ __forceinline__ void process_chunk(const hc_kparams& P, const uint32_t* __restrict__ T, const uint32_t* __restrict__ VM,
                                              u64 xpos, uint32_t ypos16, uint32_t L, uint32_t hasN, uint32_t k, uint32_t& sum,
                                              uint32_t& mm, uint32_t& ncnt, uint32_t& vd) {
    if (PACKED) process32_packed<HAS_VOID>(P, T, VM, xpos, ypos16, L, hasN, k, sum, mm, ncnt, vd);
    else process32<HAS_VOID>(P, T, xpos, ypos16, L, hasN, k, sum, mm, ncnt, vd);
}

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

struct WinAcc {
    u64 S;          // fixed-point sum of -log p
    uint32_t mm;    // mismatches
    uint32_t nn;    // N positions
    uint32_t vd;    // void
};

// Mismatch rate of one window, src/EdgeCalculator.cpp:132: float(mismatch_count)/total_len as a double; 1.0 for a window
// that was not scored (:71), exact on every device and host (an IEEE division of two small integers).
__device__ __forceinline__ double window_mm_rate(uint32_t mm, uint32_t tl) {
    if (tl == 0u) return 1.0;
    return mm ? (double)(float)(int)mm / (double)tl : 0.0;
}

// src/EdgeCalculator.cpp:254-261 (two windows) and :404-413, on per-window "above threshold" flags.  The rate itself is
// only divided out when merge_contigs is positive: "rate <= 0" is "no mismatch in any window", "rate <= negative" is never.
__device__ __forceinline__ uint32_t classify(const hc_kparams& P, uint32_t two, const uint32_t mmc[2], const uint32_t cmp[2],
                                             const int ae[2], const int ao[2]) {
    int both, ov_ok;
    if (two) {
        both = ae[0] && ae[1];
        ov_ok = ao[0] && ao[1];
    } else {
        both = ae[0];
        ov_ok = ao[0];
    }
    uint32_t cls;
    if (both) cls = HC_CLASS_EDGE;
    else {
        bool low;
        if (P.merge_contigs_sign == 0) low = cmp[0] != 0u && mmc[0] == 0u && (!two || (cmp[1] != 0u && mmc[1] == 0u));
        else if (P.merge_contigs_sign < 0) low = false;
        else {
            const double r0 = window_mm_rate(mmc[0], cmp[0]), r1 = window_mm_rate(mmc[1], cmp[1]);
            low = (two ? fmax(r0, r1) : r0) <= P.merge_contigs;
        }
        if (low) cls = HC_CLASS_EDGE;
        else if (ov_ok) cls = HC_CLASS_NONEDGE;
        else cls = HC_CLASS_DISCARD;
    }
    return cls | (both ? HC_CLS_BOTH : 0u);
}

// score of :138 / :256-261 from per-window scores
__device__ __forceinline__ double combine_score(uint32_t two, uint32_t both, double ov0, double ov1) {
    if (!two) return ov0;
    return both ? 0.5 * (ov0 + ov1) : fmin(ov0, ov1);
}

__device__ __forceinline__ double fx_mean(u64 S, uint32_t tl) { return -((double)S * (1.0 / HC_FX_SCALE)) / (double)tl; }

// (the candidate and its read descriptors are loaded again here rather than kept in registers across the chunk loops)
__device__ __noinline__ void write_per_cand(const hc_kparams& P, u64 i, double score, double mmrate, uint32_t cls,
                                            const uint32_t mmc[2], const uint32_t cmp[2], const uint32_t st[2], uint32_t exact) {
    hc_result r;
    r.score = score;
    r.mismatch_rate = mmrate;
    const hc_candidate c = load_candidate(P, i);
    uint4 r1 = make_uint4(0, 0, 0, 0), r2 = r1;
    if (c.idx1 < P.n_reads && c.idx2 < P.n_reads) {
        r1 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + c.idx1));
        r2 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + c.idx2));
    }
    extra_pos(c, r1, r2, r.pos3, r.pos4);
    r.mismatches[0] = mmc[0];
    r.mismatches[1] = mmc[1];
    r.compared[0] = cmp[0];
    r.compared[1] = cmp[1];
    r.cls = (uint8_t)(cls & HC_CLS_MASK);
    r.status[0] = (uint8_t)st[0];
    r.status[1] = (uint8_t)st[1];
    r.exact = (uint8_t)exact;
    r.indel_count = 0;
    P.per_cand[i] = r;
}

template <bool HAS_VOID, bool PACKED>
__global__ void __launch_bounds__(HC_WARPS_MAX * 32, HC_MIN_CTAS) hc_score_kernel(const hc_kparams P) {
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t* T = reinterpret_cast<uint32_t*>(smem);
    const uint32_t ntab = (P.ncodes + 1u) * 256u;                     // score table, then the tail masks, then per-warp scratch
    uint32_t* VM = T + ntab;
    for (uint32_t i = threadIdx.x; i < ntab; i += blockDim.x) T[i] = P.fx_table[i];
    if (threadIdx.x < HC_VM_WORDS) VM[threadIdx.x] = hc_packed_vmask(threadIdx.x);
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    unsigned char* scratch = smem + (size_t)(ntab + HC_VM_WORDS) * 4u + (size_t)warp * HC_WARP_SCRATCH;
    uint2* part = reinterpret_cast<uint2*>(scratch);                                     // [HC_PARTMAX]
    uint4* wdA = reinterpret_cast<uint4*>(scratch + HC_PARTMAX * 8u);                    // [64] xpos lo/hi, ypos16, L
    uint2* wdB = reinterpret_cast<uint2*>(scratch + HC_PARTMAX * 8u + HC_WINSLOTS * 16u); // [64] start chunk, hasN
    uint32_t* head = reinterpret_cast<uint32_t*>(scratch + HC_PARTMAX * 8u + HC_WINSLOTS * 24u);  // [HC_PARTMAX/32]

    const u64 ntiles = (P.n + 31ull) >> 5;
    const u64 gwarp = (u64)blockIdx.x * nwarps + warp;
    const u64 twarps = (u64)gridDim.x * nwarps;
    const uint32_t lane_le = 0xffffffffu >> (31 - lane);

    uint32_t st_windows = 0, st_positions = 0, st_bytes = 0, st_errors = 0;   // per lane: far below 2^32 for any batch a device holds

    for (u64 tile = gwarp; tile < ntiles; tile += twarps) {
        const u64 i = (tile << 5) + lane;
        const bool valid = i < P.n;
        CandSetup s;
        s.err = 0; s.two = 0;
        s.w[0].L = s.w[1].L = 0; s.w[0].status = s.w[1].status = HC_WIN_UNUSED;
        s.w[0].xpos = s.w[1].xpos = 0; s.w[0].ypos16 = s.w[1].ypos16 = 0; s.w[0].hasN = s.w[1].hasN = 0;
        if (valid) {
            const hc_candidate c = load_candidate(P, i);
            uint4 r1, r2;
            load_and_setup(P, c, s, r1, r2);
#ifndef HC_NO_PREFETCH
            prefetch_window(P, s.w[0]);
            prefetch_window(P, s.w[1]);
#endif
        }
        WinAcc acc[2];
        acc[0].S = acc[1].S = 0; acc[0].mm = acc[1].mm = 0; acc[0].nn = acc[1].nn = 0; acc[0].vd = acc[1].vd = 0;
        const uint32_t c0 = (s.w[0].L + 31u) >> 5, c1 = (s.w[1].L + 31u) >> 5;     // lane-chunks per window
        const uint32_t ct = c0 + c1;

        // ---- big candidates (>= 64 lane-chunks): the whole warp walks one window at a time
        uint32_t bigmask = __ballot_sync(0xffffffffu, ct >= HC_BIG_CHUNKS);
        while (bigmask) {
            const int src = __ffs(bigmask) - 1;
            bigmask &= bigmask - 1;
#pragma unroll
            for (int w = 0; w < 2; w++) {
                const uint32_t xl = __shfl_sync(0xffffffffu, (uint32_t)s.w[w].xpos, src);
                const uint32_t xh = __shfl_sync(0xffffffffu, (uint32_t)(s.w[w].xpos >> 32), src);
                const uint32_t yp = __shfl_sync(0xffffffffu, s.w[w].ypos16, src);
                const uint32_t Lw = __shfl_sync(0xffffffffu, s.w[w].L, src);
                const uint32_t hn = __shfl_sync(0xffffffffu, s.w[w].hasN, src);
                const uint32_t cw = (Lw + 31u) >> 5;
                if (cw == 0) continue;
                const u64 xpos = ((u64)xh << 32) | xl;
                u64 S = 0;
                uint32_t mm = 0, nn = 0, vd = 0;
                for (uint32_t k = lane; k < cw; k += 32) {
                    uint32_t sum, m1, n1, v1;
                    process_chunk<HAS_VOID, PACKED>(P, T, VM, xpos, yp, Lw, hn, k, sum, m1, n1, v1);
                    S += sum; mm += m1; nn += n1; vd |= v1;
                }
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    S += __shfl_xor_sync(0xffffffffu, S, d);
                    mm += __shfl_xor_sync(0xffffffffu, mm, d);
                    nn += __shfl_xor_sync(0xffffffffu, nn, d);
                    vd |= __shfl_xor_sync(0xffffffffu, vd, d);
                }
                if (lane == src) { acc[w].S = S; acc[w].mm = mm; acc[w].nn = nn; acc[w].vd = vd; }
            }
        }

        // ---- small candidates: rounds of at most HC_PARTMAX lane-chunks dealt round robin to the lanes
        uint32_t pending = __ballot_sync(0xffffffffu, ct > 0 && ct < HC_BIG_CHUNKS);
        while (pending) {
            const bool mine = (pending >> lane) & 1u;
            const uint32_t nwin = (c0 > 0) + (c1 > 0);
            const uint32_t v = mine ? (ct | (nwin << 16)) : 0u;
            const uint32_t incl = warp_incl_scan(v, lane);
            const bool fit = mine && ((incl & 0xffffu) <= HC_PARTMAX);
            const uint32_t take = __ballot_sync(0xffffffffu, fit);   // a prefix of the pending lanes, never empty
            const int last = 31 - __clz(take);
            const uint32_t C = __shfl_sync(0xffffffffu, incl, last) & 0xffffu;
            if (lane < (int)(HC_PARTMAX / 32u)) head[lane] = 0;
            __syncwarp();
            uint32_t start0 = 0, start1 = 0;
            if (fit) {
                start0 = (incl & 0xffffu) - ct;
                start1 = start0 + c0;
                uint32_t slot = (incl >> 16) - nwin;
                if (c0) {
                    wdA[slot] = make_uint4((uint32_t)s.w[0].xpos, (uint32_t)(s.w[0].xpos >> 32), s.w[0].ypos16, s.w[0].L);
                    wdB[slot] = make_uint2(start0, s.w[0].hasN);
                    atomicOr(&head[start0 >> 5], 1u << (start0 & 31u));
                    slot++;
                }
                if (c1) {
                    wdA[slot] = make_uint4((uint32_t)s.w[1].xpos, (uint32_t)(s.w[1].xpos >> 32), s.w[1].ypos16, s.w[1].L);
                    wdB[slot] = make_uint2(start1, s.w[1].hasN);
                    atomicOr(&head[start1 >> 5], 1u << (start1 & 31u));
                }
            }
            __syncwarp();
            uint32_t running = 0;
            for (uint32_t f0 = 0; f0 < C; f0 += 32) {
                const uint32_t hw = head[f0 >> 5];
                const uint32_t f = f0 + lane;
                if (f < C) {
                    const uint32_t slot = running + __popc(hw & lane_le) - 1u;
                    const uint4 a = wdA[slot];
                    const uint2 b = wdB[slot];
                    uint32_t sum, m1, n1, v1;
                    process_chunk<HAS_VOID, PACKED>(P, T, VM, ((u64)a.y << 32) | a.x, a.z, a.w, b.y, f - b.x, sum, m1, n1, v1);
                    part[f] = make_uint2(sum, m1 | (n1 << 12) | (v1 << 24));
                }
                running += __popc(hw);
            }
            __syncwarp();
            if (fit) {
                u64 S = 0;
                uint32_t pk = 0;
                for (uint32_t k = 0; k < c0; k++) { const uint2 e = part[start0 + k]; S += e.x; pk += e.y; }
                if (c0) { acc[0].S = S; acc[0].mm = pk & 0xfffu; acc[0].nn = (pk >> 12) & 0xfffu; acc[0].vd = pk >> 24; }
                S = 0; pk = 0;
                for (uint32_t k = 0; k < c1; k++) { const uint2 e = part[start1 + k]; S += e.x; pk += e.y; }
                if (c1) { acc[1].S = S; acc[1].mm = pk & 0xfffu; acc[1].nn = (pk >> 12) & 0xfffu; acc[1].vd = pk >> 24; }
            }
            __syncwarp();
            pending &= ~take;
        }

        // ---- decision (lane = candidate)
        bool flag = false;
        if (valid) {
            if (s.err) {
                st_errors++;
                P.cls[i] = HC_CLASS_DISCARD;
                if (P.per_cand) {
                    const uint32_t z[2] = {0, 0};
                    const uint32_t stt[2] = {HC_WIN_UNUSED, HC_WIN_UNUSED};
                    write_per_cand(P, i, 0.0, 1.0, HC_CLASS_DISCARD, z, z, stt, 0);
                }
            } else {
                int ae[2], ao[2];
                uint32_t mmc[2] = {0, 0}, cmp[2] = {0, 0}, stt[2];
#pragma unroll
                for (int w = 0; w < 2; w++) {
                    uint32_t status = s.w[w].status;
                    ae[w] = P.zero_above_edge;
                    ao[w] = P.zero_above_ov;
                    if (status == HC_WIN_SCORED) {
                        const uint32_t tl = s.w[w].L - acc[w].nn;
                        if (acc[w].vd) {
                            status = HC_WIN_VOID;               // :125-127, mismatch_rate stays 1.0
                            if (P.void_exact) flag = true;      // void in one order of the quality pair only: the reference's order decides
                        } else if (tl == 0) {
                            status = HC_WIN_EMPTY;              // :129-131
                        } else {
                            cmp[w] = tl;
                            mmc[w] = acc[w].mm;
                            const double dl = (double)tl, dS = (double)acc[w].S;
                            // mean = -S / (2^22 * tl) compared in the multiplied-out form (no division)
                            const bool up_e = !P.never_edge && (dS <= P.ce_up * dl);
                            const bool dn_e = P.never_edge || (dS > P.ce_dn * dl);
                            const bool up_o = !P.never_ov && (dS <= P.co_up * dl);
                            const bool dn_o = P.never_ov || (dS > P.co_dn * dl);
                            ae[w] = up_e;
                            ao[w] = up_o;
                            if (!(up_e || dn_e) || !(up_o || dn_o)) flag = true;
                        }
                        st_windows++;
                        st_positions += s.w[w].L;
                        st_bytes += 2u * ((s.w[w].L + 3u) >> 2) + 2u * ((s.w[w].L + 7u) >> 3) + 2u * s.w[w].L;
                    }
                    stt[w] = status;
                }
                st_bytes += 48;
                const uint32_t cls = classify(P, s.two, mmc, cmp, ae, ao);
                if (P.exact_edges && (cls & HC_CLS_MASK) == HC_CLASS_EDGE) flag = true;
                P.cls[i] = (uint8_t)cls;
                if ((cls & HC_CLS_MASK) == HC_CLASS_EDGE) {
                    hc_tmp32 t;
                    t.S[0] = acc[0].S; t.S[1] = acc[1].S;
                    t.tl[0] = cmp[0]; t.tl[1] = cmp[1];
                    t.mm[0] = mmc[0]; t.mm[1] = mmc[1];
                    P.tmp[i] = t;
                }
                if (P.per_cand) {
                    const double ov0 = cmp[0] ? exp(fx_mean(acc[0].S, cmp[0])) : 0.0;
                    const double ov1 = cmp[1] ? exp(fx_mean(acc[1].S, cmp[1])) : 0.0;
                    const double r0 = window_mm_rate(mmc[0], cmp[0]), r1 = window_mm_rate(mmc[1], cmp[1]);
                    write_per_cand(P, i, combine_score(s.two, cls & HC_CLS_BOTH, ov0, ov1), s.two ? fmax(r0, r1) : r0, cls, mmc, cmp, stt, 0);
                }
            }
        }
        // queue boundary cases for the reference-order pass (warp-aggregated append)
        const uint32_t fm = __ballot_sync(0xffffffffu, flag);
        if (fm) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&P.counters[HC_CNT_FLAGGED], (unsigned long long)__popc(fm));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (flag) P.flagged[base + __popc(fm & (lane_le >> 1))] = (uint32_t)i;
        }
    }
    // per-warp statistics, one atomic each at the very end
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        st_errors += __shfl_xor_sync(0xffffffffu, st_errors, d);
    }
    u64 w_windows = st_windows, w_positions = st_positions, w_bytes = st_bytes;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        w_windows += __shfl_xor_sync(0xffffffffu, w_windows, d);
        w_positions += __shfl_xor_sync(0xffffffffu, w_positions, d);
        w_bytes += __shfl_xor_sync(0xffffffffu, w_bytes, d);
    }
    if (lane == 0) {
        atomicAdd(&P.counters[HC_CNT_WINDOWS], w_windows);
        atomicAdd(&P.counters[HC_CNT_POSITIONS], w_positions);
        atomicAdd(&P.counters[HC_CNT_ALGBYTES], w_bytes);
        if (st_errors) atomicAdd(&P.counters[HC_CNT_ERRORS], (unsigned long long)st_errors);
    }
}

// ---- reference-order pass ---------------------------------------------------------------------------
// One thread re-adds one window exactly like src/EdgeCalculator.cpp:103-138: same double addends
// (host-built with the reference's expressions and libm), same order, IEEE add/mul/div with
// explicit _rn intrinsics so nothing is contracted into an FMA.
__device__ void exact_window(const hc_kparams& P, const double* __restrict__ sdbl, const Win& w, double& mean, double& mmrate, uint32_t& mmc,
                             uint32_t& cmp, uint32_t& status) {
    mean = 0.0;
    mmrate = 1.0;
    mmc = 0;
    cmp = 0;
    status = w.status;
    if (w.status != HC_WIN_SCORED) return;
    const uint32_t n1 = P.ncodes + 1u;
    double total = 0.0;
    uint32_t tl = 0, mm = 0;
    const u64 yp = 16ull * w.ypos16;
    if (P.packed) {
        // 32 positions per step, fetched like a lane-chunk of the score kernel (three 256-bit loads: a thread's window is its
        // own, so every load instruction of a warp costs 32 wavefronts -- few, wide ones); the addends come from the copy of
        // the double table in shared memory when there is one (sdbl); the additions stay strictly sequential in position
        // order (:106-121).
        const uint32_t nblk = (w.L + 31u) >> 5;
        for (uint32_t k = 0; k < nblk; k++) {
            const PkRow r = load32_packed(P, w.xpos, w.ypos16, w.L, 0u, k);
            const bool s4 = (r.off & 16u) != 0, s2 = (r.off & 8u) != 0, s1 = (r.off & 4u) != 0;
            uint32_t V2[12], V1[10], V[9];
#pragma unroll
            for (int i = 0; i < 12; i++) V2[i] = s4 ? r.a[i + 4] : r.a[i];
#pragma unroll
            for (int i = 0; i < 10; i++) V1[i] = s2 ? V2[i + 2] : V2[i];
#pragma unroll
            for (int i = 0; i < 9; i++) V[i] = s1 ? V1[i + 1] : V1[i];
            const uint32_t sh = (r.off & 3u) * 8u;
#pragma unroll
            for (uint32_t j = 0; j < 32; j++) {
                if (j < r.n) {
                    const uint32_t wa = __funnelshift_r(V[j >> 2], V[(j >> 2) + 1], sh);
                    const uint32_t a = (wa >> (8 * (j & 3))) & 0xffu, b = (r.y[j >> 2] >> (8 * (j & 3))) & 0xffu;
                    if (a != 0 && b != 0) {                                           // N, :35-39,:122-124
                        const uint32_t mis = (a >> 6) != (b >> 6);
                        mm += mis;
                        const uint32_t ti = hc_dbl_index(a & 63u, b & 63u, mis, n1);
                        const double lp = sdbl ? sdbl[ti] : __ldg(P.dbl_table + ti);
                        if (lp > 0.0) { status = HC_WIN_VOID; return; }              // :125-127
                        total = __dadd_rn(total, lp);                                 // :119
                        tl++;
                    }
                }
            }
        }
    } else {
        for (uint32_t i = 0; i < w.L; i++) {
            const u64 xa = w.xpos + i, xb = yp + i;
            const uint32_t nA = (P.nmask[xa >> 5] >> (xa & 31)) & 1u, nB = (P.nmask[xb >> 5] >> (xb & 31)) & 1u;
            if (nA | nB) continue;                                                    // :35-39,:122-124
            const uint32_t a = (P.base2[xa >> 4] >> (2 * (xa & 15))) & 3u, b = (P.base2[xb >> 4] >> (2 * (xb & 15))) & 3u;
            const uint32_t mis = a != b;
            mm += mis;
            const double lp = P.dbl_table[hc_dbl_index(P.qual[xa], P.qual[xb], mis, n1)];
            if (lp > 0.0) { status = HC_WIN_VOID; return; }                          // :125-127
            total = __dadd_rn(total, lp);                                             // :119
            tl++;
        }
    }
    if (tl == 0) { status = HC_WIN_EMPTY; return; }                      // :129-131
    mmc = mm;
    cmp = tl;
    const double dl = (double)tl;
    mmrate = __ddiv_rn((double)(float)(int)mm, dl);                      // :132
    mean = __dmul_rn(__ddiv_rn(1.0, dl), total);                         // :137
}

// The same sum with the addends in a WIDE shared-memory table, row = B code, column = A code | mismatch << 7 (256 doubles per
// row, like the fixed-point table of the score kernel): one PRMT builds an index, nothing is decided per position -- a
// position outside the window or with an N has a zero byte on one side (slots are zero padded) and its table entry is
// +0.0, which leaves a sum of non-positive addends bit for bit as it is; void entries (positive) are noticed per 32
// positions; compared and mismatching positions are counted on flag words.  Packed layout, one thread per window.
// (The first version decided j < n, N and void per position: 42 instructions per position, 5.3 ms for the 7.1 M edges of
// the benchmark step.)
__device__ void exact_window_wide(const hc_kparams& P, const double* __restrict__ T2, const Win& w, double& mean, double& mmrate,
                                  uint32_t& mmc, uint32_t& cmp, uint32_t& status) {
    mean = 0.0;
    mmrate = 1.0;
    mmc = 0;
    cmp = 0;
    status = w.status;
    if (w.status != HC_WIN_SCORED) return;
    double total = 0.0;
    uint32_t tl = 0, mm = 0;
    const uint32_t nblk = (w.L + 31u) >> 5;
    for (uint32_t k = 0; k < nblk; k++) {
        const PkRow r = load32_packed(P, w.xpos, w.ypos16, w.L, 0u, k);
        const bool s4 = (r.off & 16u) != 0, s2 = (r.off & 8u) != 0, s1 = (r.off & 4u) != 0;
        uint32_t V2[12], V1[10], V[9];
#pragma unroll
        for (int i = 0; i < 12; i++) V2[i] = s4 ? r.a[i + 4] : r.a[i];
#pragma unroll
        for (int i = 0; i < 10; i++) V1[i] = s2 ? V2[i + 2] : V2[i];
#pragma unroll
        for (int i = 0; i < 9; i++) V[i] = s1 ? V1[i + 1] : V1[i];
        const uint32_t sh = (r.off & 3u) * 8u;
        uint32_t flags = 0, vw = 0;
        bool vd = false;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint32_t wa = __funnelshift_r(V[j], V[j + 1], sh), wb = r.y[j];
            const uint32_t x = wa ^ wb;                                         // bits 6-7 of a byte: base difference
            const uint32_t mf = (x | (x << 1)) & 0x80808080u;
            const uint32_t col = (wa & 0x3f3f3f3fu) | mf, row = wb & 0x3f3f3f3fu;
            const uint32_t nzA = (((wa & 0x7f7f7f7fu) + 0x7f7f7f7fu) | wa), nzB = (((wb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | wb);
            flags |= mf >> j;
            vw |= ((nzA & nzB) & 0x80808080u) >> j;
            const double l0 = T2[prmt(col, row, 0xCC40u)], l1 = T2[prmt(col, row, 0xDD51u)];
            const double l2 = T2[prmt(col, row, 0xEE62u)], l3 = T2[prmt(col, row, 0xFF73u)];
            vd = vd || l0 > 0.0 || l1 > 0.0 || l2 > 0.0 || l3 > 0.0;
            total = __dadd_rn(total, l0);                                       // :119, position order
            total = __dadd_rn(total, l1);
            total = __dadd_rn(total, l2);
            total = __dadd_rn(total, l3);
        }
        if (vd) { status = HC_WIN_VOID; return; }                               // :125-127
        tl += __popc(vw);
        mm += __popc(flags & vw);
    }
    if (tl == 0) { status = HC_WIN_EMPTY; return; }                      // :129-131
    mmc = mm;
    cmp = tl;
    const double dl = (double)tl;
    mmrate = __ddiv_rn((double)(float)(int)mm, dl);                      // :132
    mean = __dmul_rn(__ddiv_rn(1.0, dl), total);                         // :137
}

// The same window by a whole warp: the lanes fetch 32 positions' addends at once, the additions still run in position
// order (every lane repeats the chain on shuffled values).  Used when only a few candidates are queued -- the usual
// case, a few dozen per batch -- where one thread per candidate means a chain of ~265 dependent loads.
__device__ void exact_window_warp(const hc_kparams& P, const Win& w, int lane, double& mean, double& mmrate, uint32_t& mmc,
                                  uint32_t& cmp, uint32_t& status) {
    mean = 0.0;
    mmrate = 1.0;
    mmc = 0;
    cmp = 0;
    status = w.status;
    if (w.status != HC_WIN_SCORED) return;
    const uint32_t n1 = P.ncodes + 1u;
    double total = 0.0;
    uint32_t tl = 0, mm = 0;
    const u64 yp = 16ull * w.ypos16;
    for (uint32_t i0 = 0; i0 < w.L; i0 += 32) {
        const uint32_t i = i0 + lane;
        bool valid = false;
        uint32_t mis = 0;
        double lp = 0.0;
        if (i < w.L) {
            const u64 xa = w.xpos + i, xb = yp + i;
            if (P.packed) {
                const uint32_t a = P.pk[xa], b = P.pk[xb];
                if (a != 0 && b != 0) {                                               // N, :35-39,:122-124
                    valid = true;
                    mis = (a >> 6) != (b >> 6);
                    lp = __ldg(P.dbl_table + hc_dbl_index(a & 63u, b & 63u, mis, n1));
                }
            } else {
                const uint32_t nA = (P.nmask[xa >> 5] >> (xa & 31)) & 1u, nB = (P.nmask[xb >> 5] >> (xb & 31)) & 1u;
                if (!(nA | nB)) {
                    valid = true;
                    const uint32_t a = (P.base2[xa >> 4] >> (2 * (xa & 15))) & 3u, b = (P.base2[xb >> 4] >> (2 * (xb & 15))) & 3u;
                    mis = a != b;
                    lp = P.dbl_table[hc_dbl_index(P.qual[xa], P.qual[xb], mis, n1)];
                }
            }
        }
        const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
        const uint32_t mmask = __ballot_sync(0xffffffffu, valid && mis);
        if (__any_sync(0xffffffffu, valid && lp > 0.0)) { status = HC_WIN_VOID; return; }   // :125-127
        mm += __popc(mmask);
        tl += __popc(vmask);
        for (uint32_t rem = vmask; rem; rem &= rem - 1)
            total = __dadd_rn(total, __shfl_sync(0xffffffffu, lp, __ffs(rem) - 1));           // :119, position order
    }
    if (tl == 0) { status = HC_WIN_EMPTY; return; }                      // :129-131
    mmc = mm;
    cmp = tl;
    const double dl = (double)tl;
    mmrate = __ddiv_rn((double)(float)(int)mm, dl);                      // :132
    mean = __dmul_rn(__ddiv_rn(1.0, dl), total);                         // :137
}

__global__ void hc_exact_kernel(const hc_kparams P, uint32_t table_in_smem) {
    extern __shared__ __align__(16) unsigned char smem[];
    const u64 nf = P.counters[HC_CNT_FLAGGED];
    const u64 nthreads = (u64)gridDim.x * blockDim.x;
    const bool warp_mode = nf * 32ull <= nthreads;     // every queued candidate can have a warp of its own
    // many queued candidates (HC_FLAG_EXACT_EDGE_SCORES: every accepted edge): one thread each, and the table of addends in
    // shared memory -- the lookups of a warp are 32 different addresses, which the global-memory path pays with up to 32
    // wavefronts each and shared memory with a few
    const double* sdbl = nullptr;
    const double* swide = nullptr;
    if (table_in_smem == 1u && !warp_mode && nf > 0) {
        double* t = reinterpret_cast<double*>(smem);
        const uint32_t nent = (P.ncodes + 1u) * (P.ncodes + 1u) * 2u;
        for (uint32_t k = threadIdx.x; k < nent; k += blockDim.x) t[k] = P.dbl_table[k];
        __syncthreads();
        sdbl = t;
    }
    if (table_in_smem == 2u && !warp_mode && nf > 0) {   // wide table: [B code][A code | mismatch << 7]; N / padding (code 0) adds +0.0
        double* t = reinterpret_cast<double*>(smem);
        const uint32_t n1 = P.ncodes + 1u, nent = n1 * 256u;
        for (uint32_t k = threadIdx.x; k < nent; k += blockDim.x) {
            const uint32_t b = k >> 8, a = k & 63u, m = (k >> 7) & 1u;
            t[k] = (a == 0u || b == 0u || a >= n1 || (k & 64u)) ? 0.0 : P.dbl_table[hc_dbl_index(a, b, m, n1)];
        }
        __syncthreads();
        swide = t;
    }
    const int lane = threadIdx.x & 31;
    const u64 tid = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool writer = !warp_mode || lane == 0;
    for (u64 t = warp_mode ? tid >> 5 : tid; t < nf; t += warp_mode ? nthreads >> 5 : nthreads) {
        const u64 i = P.flagged[t];
        const hc_candidate c = load_candidate(P, i);
        CandSetup s;
        uint4 r1, r2;
        if (!load_and_setup(P, c, s, r1, r2)) continue;
        double mean[2], mmr[2] = {1.0, 1.0};
        int ae[2], ao[2];
        uint32_t mmc[2], cmp[2], stt[2];
#pragma unroll
        for (int w = 0; w < 2; w++) {
            if (warp_mode) exact_window_warp(P, s.w[w], lane, mean[w], mmr[w], mmc[w], cmp[w], stt[w]);
            else if (swide) exact_window_wide(P, swide, s.w[w], mean[w], mmr[w], mmc[w], cmp[w], stt[w]);
            else exact_window(P, sdbl, s.w[w], mean[w], mmr[w], mmc[w], cmp[w], stt[w]);
            if (stt[w] == HC_WIN_SCORED) {
                ae[w] = mean[w] >= P.t_edge;   // <=> host-libm exp(mean) > edge_threshold
                ao[w] = mean[w] >= P.t_ov;
            } else {
                ae[w] = P.zero_above_edge;
                ao[w] = P.zero_above_ov;
            }
        }
        const uint32_t cls = classify(P, s.two, mmc, cmp, ae, ao) | HC_CLS_EXACT;
        const double mmrate = s.two ? fmax(mmr[0], mmr[1]) : mmr[0];
        if (!writer) continue;
        P.cls[i] = (uint8_t)cls;
        if ((cls & HC_CLS_MASK) == HC_CLASS_EDGE) {
            hc_tmp32 tm;
            tm.S[0] = (u64)__double_as_longlong(mean[0]);
            tm.S[1] = (u64)__double_as_longlong(mean[1]);
            tm.tl[0] = cmp[0]; tm.tl[1] = cmp[1];
            tm.mm[0] = mmc[0]; tm.mm[1] = mmc[1];
            P.tmp[i] = tm;
        }
        if (P.per_cand) {
            const double ov0 = cmp[0] ? exp(mean[0]) : 0.0, ov1 = cmp[1] ? exp(mean[1]) : 0.0;
            write_per_cand(P, i, combine_score(s.two, cls & HC_CLS_BOTH, ov0, ov1), mmrate, cls, mmc, cmp, stt, 1);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) P.counters[HC_CNT_EXACT] = nf;
}

// ---- order-preserving compaction ----------------------------------------------------------------------
#define HC_CB_THREADS 256
#define HC_CB_ITEMS 4096   // candidates per block

// class bytes: low two bits = class; per 32-bit word the number of bytes equal to 1 (edge) / 2 (non-edge)
__device__ __forceinline__ void count_classes4(uint32_t w, uint32_t& e, uint32_t& o) {
    const uint32_t lo = w & 0x01010101u, hi = (w >> 1) & 0x01010101u;
    e += __popc(lo & ~hi);
    o += __popc(hi & ~lo);
}

__global__ void __launch_bounds__(HC_CB_THREADS) hc_compact_count(const uint8_t* __restrict__ cls, u64 n, uint32_t* blockcounts) {
    const u64 base = (u64)blockIdx.x * HC_CB_ITEMS;
    uint32_t e = 0, o = 0;
    if (base + HC_CB_ITEMS <= n) {            // full block: one 16-byte load per thread (4096 = 256 x 16)
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(cls + base) + threadIdx.x);
        count_classes4(v.x, e, o); count_classes4(v.y, e, o); count_classes4(v.z, e, o); count_classes4(v.w, e, o);
    } else {
        for (uint32_t k = threadIdx.x; k < HC_CB_ITEMS; k += HC_CB_THREADS) {
            const u64 i = base + k;
            if (i < n) {
                const uint32_t c = cls[i] & HC_CLS_MASK;
                e += c == HC_CLASS_EDGE;
                o += c == HC_CLASS_NONEDGE;
            }
        }
    }
    __shared__ uint32_t se[HC_CB_THREADS / 32], so[HC_CB_THREADS / 32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, d);
        o += __shfl_xor_sync(0xffffffffu, o, d);
    }
    if ((threadIdx.x & 31) == 0) { se[threadIdx.x >> 5] = e; so[threadIdx.x >> 5] = o; }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t te = 0, to = 0;
        for (int w = 0; w < HC_CB_THREADS / 32; w++) { te += se[w]; to += so[w]; }
        blockcounts[2 * blockIdx.x] = te;
        blockcounts[2 * blockIdx.x + 1] = to;
    }
}

// single block: exclusive scan of the per-block counts (64-bit running totals kept in blockoffs)
__global__ void __launch_bounds__(1024) hc_compact_scan(const uint32_t* blockcounts, uint32_t nblocks, u64* blockoffs,
                                                        unsigned long long* counters) {
    __shared__ u64 wsum_e[32], wsum_o[32];
    __shared__ u64 carry_e, carry_o;
    if (threadIdx.x == 0) { carry_e = 0; carry_o = 0; }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t b0 = 0; b0 < nblocks; b0 += 1024) {
        const uint32_t b = b0 + threadIdx.x;
        u64 e = b < nblocks ? blockcounts[2 * b] : 0, o = b < nblocks ? blockcounts[2 * b + 1] : 0;
        u64 ie = e, io = o;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            u64 te = __shfl_up_sync(0xffffffffu, ie, d), to = __shfl_up_sync(0xffffffffu, io, d);
            if (lane >= d) { ie += te; io += to; }
        }
        if (lane == 31) { wsum_e[warp] = ie; wsum_o[warp] = io; }
        __syncthreads();
        if (warp == 0) {
            u64 ve = wsum_e[lane], vo = wsum_o[lane];
            u64 se = ve, so = vo;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                u64 te = __shfl_up_sync(0xffffffffu, se, d), to = __shfl_up_sync(0xffffffffu, so, d);
                if (lane >= d) { se += te; so += to; }
            }
            wsum_e[lane] = se - ve;
            wsum_o[lane] = so - vo;
        }
        __syncthreads();
        const u64 ce = carry_e, co = carry_o;
        if (b < nblocks) {
            blockoffs[2 * b] = ce + wsum_e[warp] + ie - e;
            blockoffs[2 * b + 1] = co + wsum_o[warp] + io - o;
        }
        __syncthreads();
        if (threadIdx.x == 1023) { carry_e = ce + wsum_e[31] + ie; carry_o = co + wsum_o[31] + io; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { counters[HC_CNT_EDGES] = carry_e; counters[HC_CNT_NONEDGES] = carry_o; }
}

// Edge::score (:138, :256-261) and the extra positions for one accepted edge
__device__ __forceinline__ void emit_edge(const hc_kparams& P, u64 i, uint32_t cfull, u64 cand_offset, hc_edge* dst) {
    const hc_candidate cd = load_candidate(P, i);
    const uint4 r1 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + cd.idx1));
    const uint4 r2 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + cd.idx2));
    const hc_tmp32 t = P.tmp[i];
    double ov[2], ml[2];
#pragma unroll
    for (int w = 0; w < 2; w++) {
        if (t.tl[w] == 0) ml[w] = __longlong_as_double(0x7ff8000000000000LL);   // NaN: window not scored
        else if (cfull & HC_CLS_EXACT) ml[w] = __longlong_as_double((long long)t.S[w]);
        else ml[w] = fx_mean(t.S[w], t.tl[w]);
        ov[w] = t.tl[w] ? exp(ml[w]) : 0.0;
    }
    const uint32_t two = ((r1.w | r2.w) & HC_LEN_MASK) != 0;
    hc_edge e;
    e.cand = i + cand_offset;
    e.score = combine_score(two, cfull & HC_CLS_BOTH, ov[0], ov[1]);
    const double mr0 = window_mm_rate(t.mm[0], t.tl[0]), mr1 = window_mm_rate(t.mm[1], t.tl[1]);
    e.mismatch_rate = two ? fmax(mr0, mr1) : mr0;                              // :132, :254
    extra_pos(cd, r1, r2, e.pos3, e.pos4);
    e.mean_log[0] = ml[0];
    e.mean_log[1] = ml[1];
    *dst = e;
}

// The same edge as a small record (hc_edge_small / hc_edge_small_exact): what a host that keeps the candidate list cannot
// derive itself -- counts, flags and the score resp. the exact mean logs.
template <bool EXACT>
__device__ __forceinline__ void emit_edge_small(const hc_kparams& P, u64 i, uint32_t cfull, u64 cand_offset, void* dst_base, u64 k) {
    const hc_candidate cd = load_candidate(P, i);
    const uint4 r1 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + cd.idx1));
    const uint4 r2 = __ldg(reinterpret_cast<const uint4*>(P.rdesc + cd.idx2));
    const hc_tmp32 t = P.tmp[i];
    double ml[2];
#pragma unroll
    for (int w = 0; w < 2; w++) {
        if (t.tl[w] == 0) ml[w] = __longlong_as_double(0x7ff8000000000000LL);   // NaN: window not scored
        else if (cfull & HC_CLS_EXACT) ml[w] = __longlong_as_double((long long)t.S[w]);
        else ml[w] = fx_mean(t.S[w], t.tl[w]);
    }
    const uint32_t two = ((r1.w | r2.w) & HC_LEN_MASK) != 0;
    const uint32_t flags = ((cfull & HC_CLS_BOTH) ? HC_EDGE_BOTH : 0u) | (two ? HC_EDGE_TWO : 0u) | ((cfull & HC_CLS_EXACT) ? HC_EDGE_EXACT : 0u);
    const uint32_t m0 = min(t.mm[0], 0xffffu), m1 = min(t.mm[1], 0xffffu), l0 = min(t.tl[0], 0xffffu), l1 = min(t.tl[1], 0xffffu);
    if (EXACT) {
        hc_edge_small_exact e;
        e.cand = (uint32_t)(i + cand_offset);
        e.mismatches[0] = (uint16_t)m0; e.mismatches[1] = (uint16_t)m1;
        e.compared[0] = (uint16_t)l0; e.compared[1] = (uint16_t)l1;
        e.flags = flags | ((t.tl[0] > 0xffffu || t.tl[1] > 0xffffu) ? HC_EDGE_OVERFLOW : 0u);
        e.mean_log[0] = ml[0];
        e.mean_log[1] = ml[1];
        reinterpret_cast<hc_edge_small_exact*>(dst_base)[k] = e;
    } else {
        hc_edge_small e;
        e.cand = (uint32_t)(i + cand_offset);
        e.mismatches[0] = (uint16_t)m0; e.mismatches[1] = (uint16_t)m1;
        e.compared[0] = (uint16_t)l0; e.compared[1] = (uint16_t)l1;
        e.flags = flags | ((t.tl[0] > 0xffffu || t.tl[1] > 0xffffu) ? HC_EDGE_OVERFLOW : 0u);
        e.score = combine_score(two, cfull & HC_CLS_BOTH, t.tl[0] ? exp(ml[0]) : 0.0, t.tl[1] ? exp(ml[1]) : 0.0);
        reinterpret_cast<hc_edge_small*>(dst_base)[k] = e;
    }
}

// Each thread owns four consecutive candidates (one 32-bit load of class bytes); ranks come from a warp scan of the
// packed (edges | non-edges << 16) counts and the per-warp totals, so the lists keep the input order.
__global__ void __launch_bounds__(HC_CB_THREADS) hc_compact_scatter(const hc_kparams P, const u64* __restrict__ blockoffs,
                                                                   uint32_t* edge_src, uint64_t* nonedge, u64 nonedge_cap,
                                                                   u64 cand_offset) {
    __shared__ uint32_t wtot[HC_CB_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 base = (u64)blockIdx.x * HC_CB_ITEMS;
    const u64 run_e = P.run ? P.run[0] : 0ull;
    u64 eoff = blockoffs[2 * blockIdx.x] + run_e, ooff = blockoffs[2 * blockIdx.x + 1] + (P.run ? P.run[1] : 0ull);
    for (uint32_t k0 = 0; k0 < HC_CB_ITEMS; k0 += 4 * HC_CB_THREADS) {
        const u64 i0 = base + k0 + 4ull * threadIdx.x;
        uint32_t w4 = 0;                                           // class bytes of candidates i0 .. i0+3 (0 = discard beyond n)
        if (i0 + 4 <= P.n) w4 = __ldg(reinterpret_cast<const uint32_t*>(P.cls + i0));
        else for (int j = 0; j < 4; j++) if (i0 + j < P.n) w4 |= (uint32_t)P.cls[i0 + j] << (8 * j);
        uint32_t ce = 0, co = 0;
        count_classes4(w4, ce, co);
        const uint32_t mine = ce | (co << 16);
        uint32_t inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < HC_CB_THREADS / 32; w++) {
            if (w < warp) before += wtot[w];
            total += wtot[w];
        }
        const uint32_t ex = before + inc - mine;
        u64 de = eoff + (ex & 0xffffu), dn = ooff + (ex >> 16);
        if (mine) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t cfull = (w4 >> (8 * j)) & 0xffu;
                const uint32_t c = cfull & HC_CLS_MASK;
                if (c == HC_CLASS_EDGE) {
                    edge_src[de - run_e] = (uint32_t)(i0 + j);        // rank within this batch -> candidate; emitted by hc_emit_edges
                    de++;
                } else if (c == HC_CLASS_NONEDGE) {
                    if (dn < nonedge_cap) nonedge[dn] = i0 + j + cand_offset;
                    dn++;
                }
            }
        }
        eoff += total & 0xffffu;
        ooff += total >> 16;
        __syncthreads();
    }
}

// Kept mode of hc_compact_scatter (the same ranks; that kernel stays as it is): a kept candidate's index is its rank
// among the edges plus its rank among the non-edges.  The candidate, its line and its class are written at that index
// relative to the batch (the running totals P.run taken off), and an edge's absolute kept index goes to K.edge_kept for
// hc_emit_edges_kept.
__global__ void __launch_bounds__(HC_CB_THREADS) hc_compact_scatter_kept(const hc_kparams P, const u64* __restrict__ blockoffs,
                                                                        uint32_t* edge_src, const hc_kept_dev K) {
    __shared__ uint32_t wtot[HC_CB_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 base = (u64)blockIdx.x * HC_CB_ITEMS;
    const u64 run_e = P.run ? P.run[0] : 0ull, run_n = P.run ? P.run[1] : 0ull;
    u64 eoff = blockoffs[2 * blockIdx.x] + run_e, ooff = blockoffs[2 * blockIdx.x + 1] + run_n;
    const hc_candidate* cand = reinterpret_cast<const hc_candidate*>(P.cand);
    for (uint32_t k0 = 0; k0 < HC_CB_ITEMS; k0 += 4 * HC_CB_THREADS) {
        const u64 i0 = base + k0 + 4ull * threadIdx.x;
        uint32_t w4 = 0;
        if (i0 + 4 <= P.n) w4 = __ldg(reinterpret_cast<const uint32_t*>(P.cls + i0));
        else for (int j = 0; j < 4; j++) if (i0 + j < P.n) w4 |= (uint32_t)P.cls[i0 + j] << (8 * j);
        uint32_t ce = 0, co = 0;
        count_classes4(w4, ce, co);
        const uint32_t mine = ce | (co << 16);
        uint32_t inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wtot[warp] = inc;
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < HC_CB_THREADS / 32; w++) {
            if (w < warp) before += wtot[w];
            total += wtot[w];
        }
        const uint32_t ex = before + inc - mine;
        u64 de = eoff + (ex & 0xffffu), dn = ooff + (ex >> 16);
        if (mine) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t c = (w4 >> (8 * j)) & HC_CLS_MASK;
                if (c != HC_CLASS_EDGE && c != HC_CLASS_NONEDGE) continue;
                const u64 r = (de - run_e) + (dn - run_n);
                K.cand[r] = cand[i0 + j];
                if (K.line) K.line[r] = K.line_in[i0 + j];
                K.cls[r] = (uint8_t)c;
                if (c == HC_CLASS_EDGE) {
                    edge_src[de - run_e] = (uint32_t)(i0 + j);
                    K.edge_kept[de - run_e] = (uint32_t)(de + dn);
                    de++;
                } else {
                    dn++;
                }
            }
        }
        eoff += total & 0xffffu;
        ooff += total >> 16;
        __syncthreads();
    }
}

// One thread per accepted edge of the batch (dense: no idle lanes next to the exp() and the random loads)
__global__ void __launch_bounds__(256) hc_emit_edges(const hc_kparams P, const uint32_t* __restrict__ edge_src, hc_edge* edges,
                                                     u64 edges_cap, u64 cand_offset) {
    const u64 n_edges = P.counters[HC_CNT_EDGES];
    const u64 run_e = P.run ? P.run[0] : 0ull;
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n_edges; k += (u64)gridDim.x * blockDim.x) {
        if (run_e + k >= edges_cap) break;
        const u64 i = edge_src[k];
        emit_edge(P, i, P.cls[i], cand_offset, edges + run_e + k);
    }
}

template <bool EXACT>
__global__ void __launch_bounds__(256) hc_emit_edges_small(const hc_kparams P, const uint32_t* __restrict__ edge_src, void* edges,
                                                           u64 edges_cap, u64 cand_offset) {
    const u64 n_edges = P.counters[HC_CNT_EDGES];
    const u64 run_e = P.run ? P.run[0] : 0ull;
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n_edges; k += (u64)gridDim.x * blockDim.x) {
        if (run_e + k >= edges_cap) break;
        const u64 i = edge_src[k];
        emit_edge_small<EXACT>(P, i, P.cls[i], cand_offset, edges, run_e + k);
    }
}

// Kept mode: the batch's k-th edge goes to edges[k] and names its kept index as `cand` (emit_edge_small writes
// i + cand_offset, so the offset is the kept index minus i, modulo 2^64)
template <bool EXACT>
__global__ void __launch_bounds__(256) hc_emit_edges_kept(const hc_kparams P, const uint32_t* __restrict__ edge_src,
                                                          const uint32_t* __restrict__ edge_kept, void* edges) {
    const u64 n_edges = P.counters[HC_CNT_EDGES];
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n_edges; k += (u64)gridDim.x * blockDim.x) {
        const u64 i = edge_src[k];
        emit_edge_small<EXACT>(P, i, P.cls[i], (u64)edge_kept[k] - i, edges, k);
    }
}

// One bit per candidate: 1 = non-edge overlap (:410-413).  One thread per 32 candidates; bits[w] covers candidates 32w..32w+31.
__global__ void __launch_bounds__(256) hc_nonedge_bits(const uint8_t* __restrict__ cls, u64 n, uint32_t* __restrict__ bits) {
    const u64 words = (n + 31) >> 5;
    for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (u64)gridDim.x * blockDim.x) {
        const u64 i0 = w << 5;
        uint32_t out = 0;
        if (i0 + 32 <= n) {
            const uint4 a = __ldg(reinterpret_cast<const uint4*>(cls + i0)), b = __ldg(reinterpret_cast<const uint4*>(cls + i0) + 1);
            const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const uint32_t ne = (v[q] >> 1) & ~v[q] & 0x01010101u;          // class bits 10 = non-edge
                out |= (((ne * 0x01020408u) >> 24) & 0xfu) << (4 * q);          // bits 0, 8, 16, 24 -> bits 0..3 of a nibble
            }
        } else {
            for (u64 j = i0; j < n; j++) out |= (uint32_t)((cls[j] & HC_CLS_MASK) == HC_CLASS_NONEDGE) << (j - i0);
        }
        bits[w] = out;
    }
}

// tile_run[t] = the run that holds candidate 32 * t; one thread per run writes the tiles that start inside it
__global__ void hc_tile_runs(const uint32_t* __restrict__ run_start, uint32_t n_runs, uint32_t* __restrict__ tile_run) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_runs; r += gridDim.x * blockDim.x) {
        const uint32_t s = run_start[r], e = run_start[r + 1];
        for (uint32_t t = (s + 31u) >> 5; ((u64)t << 5) < e; t++) tile_run[t] = r;
    }
}

__global__ void hc_compact_advance(unsigned long long* run, const unsigned long long* counters) {
    run[0] += counters[HC_CNT_EDGES];
    run[1] += counters[HC_CNT_NONEDGES];
}

}  // namespace

// ---- launchers ----------------------------------------------------------------------------------------
// grid cap of the streaming helper kernels (grid-stride loops): eight blocks per SM of the current device
static unsigned hc_grid_cap() {
    static int sms[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148u * 8u;
    if (!sms[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        sms[dev] = n;
    }
    return (unsigned)sms[dev] * 8u;
}

cudaError_t hc_score_occupancy(uint32_t ncodes, int sm_count, size_t smem_per_sm, hc_launch_cfg* cfg) {
    const size_t table = (size_t)(ncodes + 1u) * 1024u + HC_VM_WORDS * 4u;    // score table + tail masks, per CTA
    const int max_ctas = HC_MIN_CTAS;                                            // what the register allocation allows
    int best_warps = 0, best_nw = 0, best_ctas = 0;
    for (int nw = HC_WARPS_MAX; nw >= 4; nw -= 4) {                              // the table is per CTA: prefer large CTAs
        const size_t per_cta = table + (size_t)nw * HC_WARP_SCRATCH + 1024u;   // +1 KB the driver reserves per CTA
        if (per_cta > 227u * 1024u) continue;
        int ctas = (int)(smem_per_sm / per_cta);
        if (ctas > max_ctas) ctas = max_ctas;
        if (ctas * nw * 32 > 2048) ctas = 2048 / (nw * 32);
        if (ctas < 1) continue;
        if (ctas * nw > best_warps) { best_warps = ctas * nw; best_nw = nw; best_ctas = ctas; }
    }
    if (best_nw == 0) return cudaErrorInvalidConfiguration;
    cfg->threads = best_nw * 32;
    cfg->smem = table + (size_t)best_nw * HC_WARP_SCRATCH;
    cfg->blocks = sm_count * best_ctas;
    return cudaSuccess;
}

cudaError_t hc_launch_score(const hc_kparams& P, const hc_launch_cfg& cfg, cudaStream_t st) {
    void (*fn)(const hc_kparams);
    if (P.packed) fn = P.has_void ? hc_score_kernel<true, true> : hc_score_kernel<false, true>;
    else fn = P.has_void ? hc_score_kernel<true, false> : hc_score_kernel<false, false>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.smem);
    if (e != cudaSuccess) return e;
    fn<<<cfg.blocks, cfg.threads, cfg.smem, st>>>(P);
    return cudaGetLastError();
}

cudaError_t hc_launch_tile_runs(const uint32_t* run_start, uint32_t n_runs, uint32_t* tile_run, cudaStream_t st) {
    if (n_runs == 0) return cudaSuccess;
    const unsigned blocks = (n_runs + 255u) / 256u;
    hc_tile_runs<<<blocks < hc_grid_cap() ? blocks : hc_grid_cap(), 256, 0, st>>>(run_start, n_runs, tile_run);
    return cudaGetLastError();
}

cudaError_t hc_launch_exact(const hc_kparams& P, cudaStream_t st) {
    // Every accepted edge is queued (HC_FLAG_EXACT_EDGE_SCORES), packed layout: the wide double table, (K+1) * 2 KB -- 68 KB
    // for 33 quality values --, blocks of 256 threads, as many per SM as the table leaves room for.
    const size_t wide = (size_t)(P.ncodes + 1u) * 256u * sizeof(double);
    if (P.packed && P.exact_edges && wide <= 200u * 1024u) {
        int dev = 0, sms = 148;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaError_t e = cudaFuncSetAttribute(hc_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wide);
        if (e != cudaSuccess) return e;
        const size_t per_sm = 224u * 1024u / (wide + 1024u);
        const unsigned bps = (unsigned)(per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm));
        hc_exact_kernel<<<(unsigned)sms * bps, 256, wide, st>>>(P, 2u);
        return cudaGetLastError();
    }
    // a few boundary candidates (one warp each) or, rarely, many: the compact table ((K+1)^2 * 2 addends, 18 KB for 33
    // quality values) next to 128 threads
    const size_t tbl = (size_t)(P.ncodes + 1u) * (P.ncodes + 1u) * 2u * sizeof(double);
    const bool in_smem = P.packed && tbl <= 96u * 1024u;
    if (in_smem) {
        cudaError_t e = cudaFuncSetAttribute(hc_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tbl);
        if (e != cudaSuccess) return e;
    }
    hc_exact_kernel<<<hc_grid_cap(), 128, in_smem ? tbl : 0, st>>>(P, in_smem ? 1u : 0u);
    return cudaGetLastError();
}

uint32_t hc_compact_blocks(uint64_t n) { return (uint32_t)((n + HC_CB_ITEMS - 1) / HC_CB_ITEMS); }

// d_blockcounts: uint32[2*nblocks] followed (8-byte aligned) by uint64[2*nblocks] block offsets
cudaError_t hc_launch_compact(const hc_kparams& P, hc_edge* d_edges, uint64_t edges_cap, uint64_t* d_nonedge,
                              uint64_t nonedge_cap, uint32_t* d_blockcounts, uint64_t cand_offset, unsigned long long* d_run,
                              cudaStream_t st, int small_out, uint32_t* d_bits, const hc_kept_dev* kept) {
    const uint32_t nb = hc_compact_blocks(P.n);
    u64* offs = reinterpret_cast<u64*>(d_blockcounts + 2ull * nb + (2ull * nb & 1ull));
    if (nb > 0) {
        hc_compact_count<<<nb, HC_CB_THREADS, 0, st>>>(P.cls, P.n, d_blockcounts);
    }
    hc_compact_scan<<<1, 1024, 0, st>>>(d_blockcounts, nb, offs, P.counters);
    if (nb > 0 && kept) {
        hc_compact_scatter_kept<<<nb, HC_CB_THREADS, 0, st>>>(P, offs, P.flagged, *kept);
        const u64 want = (P.n + 255) / 256;
        const unsigned eb = (unsigned)(want < (unsigned long long)hc_grid_cap() ? want : (unsigned long long)hc_grid_cap());
        if (P.exact_edges) hc_emit_edges_kept<true><<<eb, 256, 0, st>>>(P, P.flagged, kept->edge_kept, d_edges);
        else hc_emit_edges_kept<false><<<eb, 256, 0, st>>>(P, P.flagged, kept->edge_kept, d_edges);
    } else if (nb > 0) {
        // P.flagged has been consumed by the reference-order pass; it now carries the source index of every edge
        hc_compact_scatter<<<nb, HC_CB_THREADS, 0, st>>>(P, offs, P.flagged, d_nonedge, nonedge_cap, cand_offset);
        const u64 want = (P.n + 255) / 256;
        const unsigned eb = (unsigned)(want < (unsigned long long)hc_grid_cap() ? want : (unsigned long long)hc_grid_cap());
        if (!small_out) hc_emit_edges<<<eb, 256, 0, st>>>(P, P.flagged, d_edges, edges_cap, cand_offset);
        else if (P.exact_edges) hc_emit_edges_small<true><<<eb, 256, 0, st>>>(P, P.flagged, d_edges, edges_cap, cand_offset);
        else hc_emit_edges_small<false><<<eb, 256, 0, st>>>(P, P.flagged, d_edges, edges_cap, cand_offset);
        if (small_out && d_bits) {
            const u64 wantb = (((P.n + 31) >> 5) + 255) / 256;
            hc_nonedge_bits<<<(unsigned)(wantb < (unsigned long long)hc_grid_cap() ? wantb : (unsigned long long)hc_grid_cap()), 256, 0, st>>>(P.cls, P.n, d_bits);
        }
    }
    if (d_run) hc_compact_advance<<<1, 1, 0, st>>>(d_run, P.counters);
    return cudaGetLastError();
}
