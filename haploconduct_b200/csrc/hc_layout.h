// hc_layout.h -- data layout shared by the host packer / table builder and the sm_100a kernels.
//
// Device read store (replaces FastqStorage's vector<Read>, src/FastqStorage.h:83-97, src/Read.h:30-31):
//
//   Every stored sequence (a single read, or one mate of a pair) owns TWO slots in one global
//   "position space": its forward strand and its reverse complement (Read::get_rev_comp /
//   get_rev_phred, src/Read.h:172-201, materialised once at pack time instead of per call).
//   A slot starts at a multiple of HC_SLOT_ALIGN positions, holds `len` positions and is padded
//   with zeros up to slot_size(len) = round_up(len + HC_SLOT_PAD, HC_SLOT_ALIGN); the rc slot
//   follows the forward slot immediately.  Three structure-of-arrays planes are indexed by position:
//
//     qual  : uint8  per position   quality CODE (0 = padding or N, 1..K = rank of the Phred value
//                                   among the distinct values present in the store)
//     base2 : 2 bits per position   A=0 C=1 G=2 T=3 (N and padding = 0), 16 positions per uint32
//     nmask : 1 bit  per position   1 = N, 32 positions per uint32
//
//   Because a window always lays B[0..L) over A[pos..pos+L) (src/EdgeCalculator.cpp:86-88,106-117),
//   the B side of every 16-position chunk is 16-byte / word aligned and only the A side needs
//   funnel shifts.  Zero padding makes every over-read contribute exactly 0 to the score sum.
//
// Per-read descriptor (16 bytes, one LDG.128): slot start / 16 and length for both mates.
#ifndef HC_LAYOUT_H_
#define HC_LAYOUT_H_

#include <stdint.h>

#define HC_SLOT_ALIGN 64u
#define HC_SLOT_PAD 32u
#define HC_CHUNK 16u            // positions per lane-chunk
#define HC_MAX_CODES 127        // quality codes 1..127 (7 bits), 0 = null
#define HC_FX_SHIFT 22          // fixed point: entry = round(-log(p) * 2^22)
#define HC_FX_SCALE 4194304.0   // 2^22
// |mean_fx - mean_ref| <= 2^-23 (table rounding, 0.5 ulp per term) + double-rounding slack
#define HC_FX_MARGIN (1.1920928955078125e-07 + 1.0e-9)
#define HC_VOID_BIT 0x08000000u // 2^27 > any real entry (max -log p = 22.6 -> 9.5e7 < 2^27)
#define HC_LEN_MASK 0x3fffffffu  // sequence lengths are below 2^30
#define HC_LEN_MAX 0x3fffffffu
#define HC_HASN_BIT 0x80000000u  // the sequence contains an N

#if defined(__CUDACC__)
#define HC_HD __host__ __device__ __forceinline__
#else
#define HC_HD static inline
#endif

struct hc_rdesc {          // device read descriptor
    uint32_t slot16[2];    // forward-slot start / 16 for mate 0 / 1
    uint32_t len[2];       // length | HC_HASN_BIT ; len[1] == 0 <=> single-end read
};

HC_HD uint32_t hc_slot_size(uint32_t len) {
    return (len + HC_SLOT_PAD + HC_SLOT_ALIGN - 1u) & ~(HC_SLOT_ALIGN - 1u);
}

// Bank swizzle of the score table: the table row is the B-side code, the column is
// (A-side code XOR g(B-side code)) | mismatch << 7.  g spreads the (q,q) diagonal and equal-A-quality
// runs over the 32 shared-memory banks.  Works on 4 packed bytes at once (codes are < 128).
HC_HD uint32_t hc_swz4(uint32_t wb) { return ((wb << 1) & 0x7e7e7e7eu) | (wb & 0x01010101u); }
HC_HD uint32_t hc_swz1(uint32_t cb) { return ((cb << 1) & 0x7eu) | (cb & 1u); }

// index into the fixed-point table: 256 columns per row
HC_HD uint32_t hc_fx_index(uint32_t ca, uint32_t cb, uint32_t mm) {
    return (cb << 8) | ((ca ^ hc_swz1(cb)) & 0x7fu) | (mm << 7);
}
// Packed ("narrow") layout, used when the store has at most 63 distinct quality values:
//   one byte per position = quality code (bits 0-5, 0 = N or padding) | 2-bit base << 6.
// XOR of an A byte with a B byte then carries the base difference in bits 6-7 for free; the table
// column is ((code_A ^ g6(code_B)) & 63) | (base_A ^ base_B) << 6  (columns 64..255 = mismatch).
#define HC_PACKED_MAX_CODES 63
#ifdef HC_NO_SWZ   // experiment: no bank swizzle (column = A code)
HC_HD uint32_t hc_swz4_packed(uint32_t wb) { return wb & 0xc0c0c0c0u; }
HC_HD uint32_t hc_swz1_packed(uint32_t cb) { (void)cb; return 0u; }
#else
HC_HD uint32_t hc_swz4_packed(uint32_t wb) { return ((wb << 1) & 0x3e3e3e3eu) | (wb & 0xc1c1c1c1u); }
HC_HD uint32_t hc_swz1_packed(uint32_t cb) { return ((cb << 1) & 0x3eu) | (cb & 1u); }
#endif
HC_HD uint32_t hc_fx_index_packed(uint32_t ca, uint32_t cb, uint32_t bx) {
    return (cb << 8) | ((ca ^ hc_swz1_packed(cb)) & 0x3fu) | (bx << 6);
}
// Mismatch flags of a 32-position lane-chunk are gathered as OR_j (flags(word j) >> j): position
// p = 4j + t lands on bit 8t + 7 - j.  Mask of the first n positions in that bit order:
HC_HD uint32_t hc_packed_vmask(uint32_t n) {
    uint32_t m = 0;
    for (uint32_t p = 0; p < n && p < 32u; p++) m |= 1u << (8u * (p & 3u) + 7u - (p >> 2));
    return m;
}

// index into the double table used by the reference-order pass
HC_HD uint32_t hc_dbl_index(uint32_t ca, uint32_t cb, uint32_t mm, uint32_t ncodes1) {
    return ((ca * ncodes1) + cb) * 2u + mm;
}

#endif
