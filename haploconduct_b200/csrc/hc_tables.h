// hc_tables.h -- host-built score tables (see hc_tables.cpp)
#ifndef HC_TABLES_H_
#define HC_TABLES_H_
#include <stdint.h>
#include <vector>
#include "hc_layout.h"

struct hc_tables {
    int ncodes;                  // K: quality codes 1..K
    bool has_void;               // some (qa,qb,mm) has p < ps.mismatch
    std::vector<double> dbl;     // [(K+1)*(K+1)*2] log(p), exact reference addends (2.0 = void sentinel)
    std::vector<uint32_t> fx;    // [(K+1)*256] round(-log(p)*2^22), swizzled layout of hc_fx_index()
    std::vector<uint32_t> fx_packed;  // same values in the hc_fx_index_packed() layout (K <= 63 only, else empty)
    bool void_asymmetric;        // some (qa,qb) is void in one order only: void hits are decided by the reference-order pass
};

double hc_tables_phred_to_prob(int phred);
void hc_build_tables(const int* code_to_q, int ncodes, double mismatch_param, hc_tables* out);
double hc_tables_exp_threshold(double thr, int* monotone_ok);
#endif
