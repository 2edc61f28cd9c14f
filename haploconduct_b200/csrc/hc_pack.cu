// hc_pack.cu -- building the read store on the device.
//   * validation + quality alphabet + packing of both strands (what FastqStorage / Read keep as strings,
//     src/Read.h:144-201: get_seq / get_phred / get_rev_comp / get_rev_phred) from raw bases / qualities,
//   * the FASTQ record scan of FastqStorage::read_singles / read_pairs (src/FastqStorage.cpp:92-235).
// Byte work, one warp per (read, mate); the only host work left is the slot layout (a prefix sum over reads).
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>
#include "hc_layout.h"
#include "hc_pack.cuh"
#include "hc_text.cuh"

namespace {

__device__ __forceinline__ int dev_base_code(unsigned char c) {
    switch (c) {
        case 'A': return 0;
        case 'C': return 1;
        case 'G': return 2;
        case 'T': return 3;
        case 'N': return 4;
        default: return -1;
    }
}

__device__ __forceinline__ unsigned char dev_upper(unsigned char c) { return (c >= 'a' && c <= 'z') ? (unsigned char)(c - 32) : c; }

// hist[128]: how often every quality character occurs (quality codes are ranked by frequency, see build_store in hc_api.cu);
// err: 1 invalid nucleotide, 2 quality out of range
__global__ void __launch_bounds__(256) pack_validate(const uint8_t* __restrict__ text, const hc_pack_src* __restrict__ src,
                                                     const hc_rdesc* __restrict__ rd, u64 n_reads, u64 n_upper,
                                                     unsigned long long* hist, uint32_t* err) {
    __shared__ uint32_t shist[128];
    if (threadIdx.x < 128) shist[threadIdx.x] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const u64 gw = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((u64)gridDim.x * blockDim.x) >> 5;
    uint32_t lerr = 0;
    for (u64 t = gw; t < 2 * n_reads; t += nw) {
        const u64 r = t >> 1;
        const int m = (int)(t & 1);
        const uint32_t len = rd[r].len[m] & HC_LEN_MASK;
        if (!len) continue;
        const uint8_t* b = text + src[t].boff;
        const uint8_t* q = text + src[t].qoff;
        const bool up = r < n_upper;
        for (uint32_t i = lane; i < len; i += 32) {
            const unsigned char bc = up ? dev_upper(b[i]) : b[i];
            const unsigned char qc = q[i];
            if (dev_base_code(bc) < 0) lerr |= 1u;
            if (qc < 33 || qc > 33 + 93) lerr |= 2u;
            else atomicAdd(&shist[qc], 1u);          // a block sees far fewer than 2^32 characters between two flushes
        }
    }
    __syncthreads();
    if (threadIdx.x < 128 && shist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)shist[threadIdx.x]);
    if (lerr) atomicOr(err, lerr);
}

// forward strand at the slot start, reverse complement (reversed qualities) one slot size further; planes are zeroed
template <bool PACKED>
__global__ void __launch_bounds__(256) pack_write(const uint8_t* __restrict__ text, const hc_pack_src* __restrict__ src, hc_rdesc* rd,
                                                  u64 n_reads, u64 n_upper, const uint8_t* __restrict__ q2code, uint8_t* qplane,
                                                  uint32_t* base2, uint32_t* nmask) {
    __shared__ uint8_t lut[256];
    lut[threadIdx.x] = q2code[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const u64 gw = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 t = gw; t < 2 * n_reads; t += nw) {
        const u64 r = t >> 1;
        const int m = (int)(t & 1);
        const uint32_t len = rd[r].len[m] & HC_LEN_MASK;
        if (!len) continue;
        const uint8_t* b = text + src[t].boff;
        const uint8_t* q = text + src[t].qoff;
        const bool up = r < n_upper;
        const u64 fwd = 16ull * rd[r].slot16[m], rev = fwd + hc_slot_size(len);
        bool hasN = false;
        for (uint32_t i0 = 0; i0 < len; i0 += 32) {
            const uint32_t i = i0 + lane;
            if (i >= len) continue;
            const int bc = dev_base_code(up ? dev_upper(b[i]) : b[i]);
            const u64 pf = fwd + i, pr = rev + (len - 1 - i);
            if (bc == 4) {
                hasN = true;          // N: quality code 0 (contributes nothing), base bits 0, mask bit set
                if (!PACKED) {
                    atomicOr(&nmask[pf >> 5], 1u << (pf & 31));
                    atomicOr(&nmask[pr >> 5], 1u << (pr & 31));
                }
            } else {
                const uint8_t code = lut[q[i]];
                if (PACKED) {
                    qplane[pf] = (uint8_t)(code | (bc << 6));
                    qplane[pr] = (uint8_t)(code | ((3 - bc) << 6));          // reversed qualities + complement
                } else {
                    qplane[pf] = code;
                    qplane[pr] = code;                                       // src/Read.h:187-201
                    atomicOr(&base2[pf >> 4], (uint32_t)bc << (2 * (pf & 15)));
                    atomicOr(&base2[pr >> 4], (uint32_t)(3 - bc) << (2 * (pr & 15)));   // src/Types.h:109-129
                }
            }
        }
        if (__any_sync(0xffffffffu, hasN) && lane == 0) rd[r].len[m] |= HC_HASN_BIT;
    }
}

// One FASTQ record (4 lines) per thread: header check, id, sequence / quality line extents.  A record the
// reference exits on (header without '@' :107-110,:181-184; mate headers that differ :189-192; empty sequence
// :143-146,:217-220) or whose sequence and quality lengths differ lowers *first_err to its index; the host then
// looks at that record itself and reports why.
__global__ void __launch_bounds__(256) fq_records(const char* __restrict__ text, u64 file_off, u64 n_bytes,
                                                  const u64* __restrict__ line_start, u64 n_newlines, u64 n_rec, u64* ids,
                                                  uint32_t* len, hc_pack_src* src, ulonglong2* tok, int mate, u64 out0, u64* first_err) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_rec) return;
    const char* f = text + file_off;
    u64 ls[4], le[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const u64 li = 4 * k + j;
        ls[j] = line_start[li];
        le[j] = li < n_newlines ? line_start[li + 1] - 1 : n_bytes;
    }
    // the reference tests the '@' of the first file's header only (src/FastqStorage.cpp:107-110,:181-184); mate 2's is just skipped
    bool bad = le[0] == ls[0] || (mate == 0 && f[ls[0]] != '@');
    // stringstream(line.substr(1)) >> token: skip white space, read up to the next white space (:111-113)
    u64 p = ls[0] + 1;
    while (p < le[0] && c_isspace(f[p])) p++;
    u64 q = p;
    while (q < le[0] && !c_isspace(f[q])) q++;
    if (bad) p = q = ls[0];
    const u64 o = out0 + k;
    if (mate == 0) {
        ids[o] = dev_strtoul0(f, p, q);                     // str_to_read_id, src/Types.h:99-102
        tok[o] = make_ulonglong2(file_off + p, q - p);
    } else {
        const ulonglong2 t0 = tok[o];
        if (t0.y != q - p) bad = true;
        else for (u64 j = 0; j < t0.y && !bad; j++) bad = text[t0.x + j] != f[p + j];
    }
    const u64 slen = le[1] - ls[1], qlen = le[3] - ls[3];
    if (slen != qlen || slen == 0 || slen > HC_LEN_MAX) bad = true;
    len[2 * o + mate] = bad ? 0u : (uint32_t)slen;
    src[2 * o + mate].boff = file_off + ls[1];
    src[2 * o + mate].qoff = file_off + ls[3];
    if (bad) atomicMin(first_err, o);
}

}  // namespace

cudaError_t hc_pack_validate_launch(const uint8_t* d_text, const hc_pack_src* d_src, const hc_rdesc* d_rd, uint64_t n_reads,
                                    uint64_t n_upper, unsigned long long* d_hist, uint32_t* d_err, cudaStream_t stream) {
    const u64 warps = 2 * n_reads;
    const unsigned blocks = (unsigned)std::min<u64>((warps + 7) / 8, 148ull * 32);
    pack_validate<<<blocks ? blocks : 1, 256, 0, stream>>>(d_text, d_src, d_rd, n_reads, n_upper, d_hist, d_err);
    return cudaGetLastError();
}

cudaError_t hc_pack_write_launch(const uint8_t* d_text, const hc_pack_src* d_src, hc_rdesc* d_rd, uint64_t n_reads, uint64_t n_upper,
                                 const uint8_t* d_q2code, int packed, uint8_t* qplane, uint32_t* base2, uint32_t* nmask,
                                 cudaStream_t stream) {
    const u64 warps = 2 * n_reads;
    const unsigned blocks = (unsigned)std::min<u64>((warps + 7) / 8, 148ull * 32);
    if (packed) pack_write<true><<<blocks ? blocks : 1, 256, 0, stream>>>(d_text, d_src, d_rd, n_reads, n_upper, d_q2code, qplane, base2, nmask);
    else pack_write<false><<<blocks ? blocks : 1, 256, 0, stream>>>(d_text, d_src, d_rd, n_reads, n_upper, d_q2code, qplane, base2, nmask);
    return cudaGetLastError();
}

cudaError_t hc_fastq_index(const char* d_text, uint64_t n_bytes, uint64_t max_reads, unsigned long long** d_line_start,
                           uint64_t* n_newlines, uint64_t* n_records, cudaStream_t stream) {
    u64 nl = 0, lines = 0;
    cudaError_t e = hc_line_index(d_text, n_bytes, d_line_start, &nl, &lines, stream);
    if (e != cudaSuccess) return e;
    if (max_reads < (~0ull >> 2) && lines > 4 * max_reads) lines = 4 * max_reads;   // count < 4*MAX, src/FastqStorage.cpp:46
    *n_newlines = nl;
    *n_records = lines / 4;                                                         // a record is stored at its 4th line
    return cudaSuccess;
}

cudaError_t hc_fastq_records_launch(const char* d_text, uint64_t file_off, uint64_t n_bytes, const unsigned long long* d_line_start,
                                    uint64_t n_newlines, uint64_t n_rec, unsigned long long* d_ids, uint32_t* d_len, hc_pack_src* d_src,
                                    void* d_tok, int mate, uint64_t out0, unsigned long long* d_first_err, cudaStream_t stream) {
    if (n_rec == 0) return cudaSuccess;
    fq_records<<<(unsigned)((n_rec + 255) / 256), 256, 0, stream>>>(d_text, file_off, n_bytes, d_line_start, n_newlines, n_rec, d_ids, d_len,
                                                                    d_src, reinterpret_cast<ulonglong2*>(d_tok), mate, out0, d_first_err);
    return cudaGetLastError();
}
