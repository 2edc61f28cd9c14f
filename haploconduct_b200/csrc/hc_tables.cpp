// hc_tables.cpp -- host-side score tables (compiled with g++ -O2 -ffp-contract=off, no FMA, like
// the reference build, makefile:6).
//
// Every addend of the reference's per-base log-likelihood is a pure function of (Q_A, Q_B, match?):
//   P(Q)      = pow(10, -Q/10.0)                                       src/EdgeCalculator.cpp:59-63
//   match     p = (1-p1)*(1-p2) + (p1*p2)/3.0                          :41
//   mismatch  p = p1*(1-p2)/3.0 + p2*(1-p1)/3.0 + (2/9.0)*p1*p2        :44
//   void      p < ps.mismatch                                          :49-51
//   addend    log(p)                                                   :52
// with (p1, p2) = (quality of the A side, quality of the B side) -- the mismatch expression is not
// bit-symmetric, so the table is indexed by the ORDERED pair.  Built with the host libm so the
// double table is bit-identical to what the reference adds up; the device never calls pow/log.
#include <cmath>
#include <cstring>
#include <vector>
#include "hc_tables.h"

double hc_tables_phred_to_prob(int phred) { return pow(10, -phred / 10.0); }

// fixed-point addend of one ordered pair of codes; *is_void when p < ps.mismatch (:49-51)
static double pair_log(int qa, int qb, int mm, double mismatch_param, bool* is_void) {
    double p1 = hc_tables_phred_to_prob(qa);
    double p2 = hc_tables_phred_to_prob(qb);
    double p;
    if (!mm) p = (1 - p1) * (1 - p2) + (p1 * p2) / 3.0;
    else p = p1 * (1 - p2) / 3.0 + p2 * (1 - p1) / 3.0 + (2 / 9.0) * p1 * p2;
    *is_void = p < mismatch_param;
    return *is_void ? 2.0 : log(p);   // sentinel > 0: "unacceptable mismatch", the whole overlap is void
}

void hc_build_tables(const int* code_to_q, int ncodes, double mismatch_param, hc_tables* out) {
    const int n1 = ncodes + 1;
    out->ncodes = ncodes;
    out->dbl.assign((size_t)n1 * n1 * 2, 0.0);
    out->fx.assign((size_t)n1 * 256, 0u);
    const bool packed = ncodes <= HC_PACKED_MAX_CODES;
    out->fx_packed.assign(packed ? (size_t)n1 * 256 : 0, 0u);
    out->has_void = false;
    out->void_asymmetric = false;
    for (int ca = 1; ca <= ncodes; ca++) {
        for (int cb = 1; cb <= ncodes; cb++) {
            for (int mm = 0; mm < 2; mm++) {
                bool v_ab, v_ba;
                const double lp = pair_log(code_to_q[ca], code_to_q[cb], mm, mismatch_param, &v_ab);
                // The fixed-point table is SYMMETRIC: both orders take the value of (min code, max code).  The reference's
                // expression :44 is not bit-symmetric, but the two orders differ by a few ulp of a double, far below the
                // 2^-23 rounding of the table (HC_FX_MARGIN keeps 1e-9 of slack for it).  A void decision that differs
                // between the two orders (ps.mismatch within an ulp of some p) sends void hits to the reference-order pass.
                const int lo = ca < cb ? ca : cb, hi = ca < cb ? cb : ca;
                const double lps = pair_log(code_to_q[lo], code_to_q[hi], mm, mismatch_param, &v_ba);
                bool v_other;
                pair_log(code_to_q[cb], code_to_q[ca], mm, mismatch_param, &v_other);
                if (v_ab != v_other) out->void_asymmetric = true;
                const bool v_any = v_ab || v_other;
                uint32_t fx;
                if (v_any) {
                    fx = HC_VOID_BIT;
                    out->has_void = true;
                } else {
                    double v = -lps * HC_FX_SCALE;
                    fx = (uint32_t)llround(v);
                    if (fx >= HC_VOID_BIT) fx = HC_VOID_BIT - 1;  // cannot happen for Q in [0,93]
                }
                (void)v_ba;
                out->dbl[hc_dbl_index(ca, cb, mm, n1)] = lp;
                out->fx[hc_fx_index(ca, cb, mm)] = fx;
                if (packed) {
                    if (!mm) out->fx_packed[hc_fx_index_packed(ca, cb, 0)] = fx;
                    else for (uint32_t bx = 1; bx < 4; bx++) out->fx_packed[hc_fx_index_packed(ca, cb, bx)] = fx;
                }
            }
        }
    }
}

// Smallest double x with exp(x) > thr under the host libm.  The reference decides
// "exp(mean) > thr" (src/EdgeCalculator.cpp:138,404); the device decides "mean >= x".
// exp is monotone non-decreasing in glibc; the bisection runs on the ordered bit patterns and the
// result is verified on a +-64 ulp neighbourhood.
static inline int64_t d2o(double d) {
    int64_t i;
    memcpy(&i, &d, 8);
    return i < 0 ? (int64_t)0x8000000000000000LL - i : i;
}
static inline double o2d(int64_t o) {
    int64_t i = o < 0 ? (int64_t)0x8000000000000000LL - o : o;
    double d;
    memcpy(&d, &i, 8);
    return d;
}

double hc_tables_exp_threshold(double thr, int* monotone_ok) {
    if (monotone_ok) *monotone_ok = 1;
    if (!(thr == thr)) return INFINITY;
    if (thr < 0) return -INFINITY;   // exp(x) > negative for every x
    int64_t lo = d2o(-800.0), hi = d2o(800.0);
    if (exp(o2d(hi)) <= thr) return INFINITY;
    if (exp(o2d(lo)) > thr) return -INFINITY;
    // invariant: exp(lo) <= thr < exp(hi)
    while ((__int128)hi - (__int128)lo > 1) {
        int64_t mid = (int64_t)(((__int128)lo + (__int128)hi) >> 1);   // hi - lo overflows int64
        if (exp(o2d(mid)) > thr) hi = mid; else lo = mid;
    }
    if (monotone_ok) {
        for (int k = 1; k <= 64; k++) {
            if (!(exp(o2d(hi + k)) > thr) || (exp(o2d(lo - k)) > thr)) *monotone_ok = 0;
        }
    }
    return o2d(hi);
}
