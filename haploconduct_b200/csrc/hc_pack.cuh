// hc_pack.cuh -- device-side construction of the read store (hc_pack.cu), called from hc_api.cu.
#ifndef HC_PACK_CUH_
#define HC_PACK_CUH_
#include <cstdint>
#include <cuda_runtime.h>
#include "hc_layout.h"

struct hc_pack_src {      // per (read, mate): where its bases and its quality characters start in the device text buffer
    unsigned long long boff, qoff;
};

// quality alphabet (d_hist[128]: occurrences of every quality character) and validity (d_err: bit 0 invalid nucleotide,
// bit 1 quality out of range) of all reads; the first n_upper reads are upper-cased first (singles, src/FastqStorage.cpp:123)
cudaError_t hc_pack_validate_launch(const uint8_t* d_text, const hc_pack_src* d_src, const hc_rdesc* d_rd, uint64_t n_reads,
                                    uint64_t n_upper, unsigned long long* d_hist, uint32_t* d_err, cudaStream_t stream);
// both strands of every read into the (zeroed) planes; sets HC_HASN_BIT in d_rd
cudaError_t hc_pack_write_launch(const uint8_t* d_text, const hc_pack_src* d_src, hc_rdesc* d_rd, uint64_t n_reads, uint64_t n_upper,
                                 const uint8_t* d_q2code, int packed, uint8_t* qplane, uint32_t* base2, uint32_t* nmask,
                                 cudaStream_t stream);
// newline index of one FASTQ file on the device; n_records = complete 4-line records within 4 * max_reads lines
cudaError_t hc_fastq_index(const char* d_file, uint64_t n_bytes, uint64_t max_reads, unsigned long long** d_line_start,
                           uint64_t* n_newlines, uint64_t* n_records, cudaStream_t stream);
// records of one file -> ids (mate 0), lengths, source offsets; mate 1 compares its header token with mate 0's
cudaError_t hc_fastq_records_launch(const char* d_text, uint64_t file_off, uint64_t n_bytes, const unsigned long long* d_line_start,
                                    uint64_t n_newlines, uint64_t n_rec, unsigned long long* d_ids, uint32_t* d_len, hc_pack_src* d_src,
                                    void* d_tok, int mate, uint64_t out0, unsigned long long* d_first_err, cudaStream_t stream);
#endif
