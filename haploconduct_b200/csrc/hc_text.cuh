// hc_text.cuh -- text primitives shared by the ingestion kernels (hc_ingest.cu: overlaps file, hc_pack.cu: FASTQ) and the
// converters (hc_sfo.cu, hc_sam.cu): newline index of a device buffer (count -> scan -> mark), the lines it delimits, the
// glibc number parsers the reference calls, the converters' number parser and their count-then-write output sink.
#ifndef HC_TEXT_CUH_
#define HC_TEXT_CUH_
#include <cstdint>
#include <cuda_runtime.h>

namespace {

typedef unsigned long long u64;
constexpr int TILE = 4096;            // text bytes per block in the newline passes (256 threads x 16 B)

// ---- newline index -----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t nl_mask16(const char* text, u64 n, u64 p) {   // bit b = text[p + b] == '\n'
    uint32_t m = 0;
    if (p + 16 <= n && ((reinterpret_cast<uintptr_t>(text) & 15u) == 0)) {
        const uint4 v = *reinterpret_cast<const uint4*>(text + p);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t x = w[j] ^ 0x0a0a0a0au;                      // zero byte <=> newline
            uint32_t z = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;   // exact zero-byte detector
            z = (z >> 7) * 0x00204081u;                                 // gather bits 0,8,16,24 into bits 24..27
            m |= ((z >> 21) & 0xfu) << (4 * j);
        }
    } else {
        for (int b = 0; b < 16 && p + b < n; b++) m |= (uint32_t)(text[p + b] == '\n') << b;
    }
    return m;
}

__global__ void __launch_bounds__(256) nl_count(const char* text, u64 n, uint32_t* tile_cnt) {
    const u64 p = (u64)blockIdx.x * TILE + 16ull * threadIdx.x;
    const int c = p < n ? __popc(nl_mask16(text, n, p)) : 0;
    __shared__ int wsum[8];
    int v = c;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
        for (int w = 0; w < 8; w++) s += wsum[w];
        tile_cnt[blockIdx.x] = (uint32_t)s;
    }
}

// single-block exclusive scan of uint32 counts -> u64 offsets (the inputs are per-tile / per-block counts)
__global__ void __launch_bounds__(1024) scan_counts(const uint32_t* in, u64 n, u64* out, u64* total) {
    __shared__ u64 wsum[32];
    __shared__ u64 carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (u64 b0 = 0; b0 < n; b0 += 1024) {
        const u64 i = b0 + threadIdx.x;
        const u64 v = i < n ? in[i] : 0;
        u64 inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u64 t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const u64 w = wsum[lane];
            u64 s = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u64 t = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += t;
            }
            wsum[lane] = s - w;
        }
        __syncthreads();
        const u64 c = carry;
        if (i < n) out[i] = c + wsum[warp] + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c + wsum[31] + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// line_start[k + 1] = offset behind the k-th newline (line_start[0] = 0 is set by the host)
__global__ void __launch_bounds__(256) nl_mark(const char* text, u64 n, const u64* tile_off, u64* line_start) {
    const u64 p = (u64)blockIdx.x * TILE + 16ull * threadIdx.x;
    const uint32_t m = p < n ? nl_mask16(text, n, p) : 0u;
    const int c = __popc(m);
    __shared__ int wsum[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; w++) base += wsum[w];
    u64 k = tile_off[blockIdx.x] + (u64)(base + inc - c);
    uint32_t mm = m;
    while (mm) {
        const int b = __ffs(mm) - 1;
        mm &= mm - 1;
        line_start[++k] = p + b + 1;
    }
}

// ---- field parsers (glibc semantics of what src/Types.h:99-102 and src/Overlap.h:42-50 call) -----
__device__ __forceinline__ bool c_isspace(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// strtoul(s, NULL, 0) on the field [p, q)
__device__ u64 dev_strtoul0(const char* t, u64 p, u64 q) {
    while (p < q && c_isspace(t[p])) p++;
    bool neg = false;
    if (p < q && (t[p] == '+' || t[p] == '-')) { neg = t[p] == '-'; p++; }
    int base = 10;
    if (p < q && t[p] == '0') {
        if (p + 2 < q + 0 && (t[p + 1] == 'x' || t[p + 1] == 'X')) {
            const char h = t[p + 2];
            if ((h >= '0' && h <= '9') || (h >= 'a' && h <= 'f') || (h >= 'A' && h <= 'F')) { base = 16; p += 2; }
            else base = 8;      // "0x" without a hex digit: the "0" is the number
        } else base = 8;
    }
    u64 v = 0;
    bool ovf = false;
    // glibc's cutoff / cutlim test instead of a division per digit
    const u64 cutoff = base == 10 ? ~0ull / 10ull : (base == 16 ? ~0ull >> 4 : ~0ull >> 3);
    const int cutlim = base == 10 ? (int)(~0ull % 10ull) : base - 1;
    for (; p < q; p++) {
        const char c = t[p];
        int d;
        if (c >= '0' && c <= '9') d = c - '0';
        else if (c >= 'a' && c <= 'z') d = c - 'a' + 10;
        else if (c >= 'A' && c <= 'Z') d = c - 'A' + 10;
        else break;
        if (d >= base) break;
        if (v > cutoff || (v == cutoff && d > cutlim)) ovf = true;
        else v = v * (u64)base + (u64)d;
    }
    if (ovf) return ~0ull;                     // ULONG_MAX, whatever the sign
    return neg ? 0ull - v : v;
}

// parse_long of both host converters on [b, e): an optional sign, then decimal digits only.  0: not a number; 1: ok, *v set;
// 2: more than 18 digits (the host's long may overflow; *v holds the first 18 and the caller declines the field).
__device__ int parse_long(const char* t, u64 b, u64 e, long long* v) {
    if (b == e) return 0;
    bool neg = false;
    if (t[b] == '+' || t[b] == '-') { neg = t[b] == '-'; b++; }
    if (b == e) return 0;
    long long x = 0;
    for (u64 p = b; p < e; p++) {
        const char c = t[p];
        if (c < '0' || c > '9') return 0;
        if (p - b < 18) x = x * 10 + (c - '0');
    }
    *v = neg ? -x : x;
    return e - b > 18 ? 2 : 1;
}

// ---- lines and output ----------------------------------------------------------------------------
// Line k of a text with the newline index ls (n_nl newlines, hc_line_index): [*b, *le) without its '\n'.  The span up to
// the next line start ends in its only newline, so one strip is all there is.
__device__ __forceinline__ void line_span(const char* t, u64 n, const u64* ls, u64 n_nl, u64 k, u64* b, u64* le) {
    *b = ls[k];
    u64 e = k < n_nl ? ls[k + 1] : n;
    if (e > *b && t[e - 1] == '\n') e--;
    *le = e;
}

// A thread's output text: counts the bytes, and writes them too when p != nullptr (the converters size every line with
// one pass, scan the sizes and write with a second)
struct Sink {
    char* p;
    u64 n;
    __device__ void c(char x) { if (p) p[n] = x; n++; }
    __device__ void num(long long v) {                   // printf("%ld")
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
    __device__ void str(const char* t, u64 b, u64 e) {   // the bytes t[b, e)
        if (p) for (u64 i = b; i < e; i++) p[n + (i - b)] = t[i];
        n += e - b;
    }
};

// Newline index of d_text[0, n): *d_line_start (cudaMalloc'ed here, n_newlines + 2 entries) holds the offset of every
// line start, entry 0 = 0.  n_lines counts an unterminated last line too (std::getline returns it).
inline cudaError_t hc_line_index(const char* d_text, u64 n, u64** d_line_start, u64* n_newlines, u64* n_lines, cudaStream_t stream) {
    *d_line_start = nullptr; *n_newlines = 0; *n_lines = 0;
    if (n == 0) return cudaSuccess;
    const u64 n_tiles = (n + TILE - 1) / TILE;
    uint32_t* d_tcnt = nullptr;
    u64 *d_toff = nullptr, *d_tot = nullptr;
    char last = '\n';
    cudaError_t e = cudaMalloc(&d_tcnt, n_tiles * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&d_toff, n_tiles * sizeof(u64));
    if (e == cudaSuccess) e = cudaMalloc(&d_tot, sizeof(u64));
    if (e == cudaSuccess) {
        nl_count<<<(unsigned)n_tiles, 256, 0, stream>>>(d_text, n, d_tcnt);
        scan_counts<<<1, 1024, 0, stream>>>(d_tcnt, n_tiles, d_toff, d_tot);
        e = cudaMemcpyAsync(n_newlines, d_tot, sizeof(u64), cudaMemcpyDeviceToHost, stream);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&last, d_text + n - 1, 1, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e == cudaSuccess) {
        *n_lines = *n_newlines + (last != '\n' ? 1 : 0);
        e = cudaMalloc(d_line_start, (*n_newlines + 2) * sizeof(u64));
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(*d_line_start, 0, sizeof(u64), stream);
    if (e == cudaSuccess) {
        nl_mark<<<(unsigned)n_tiles, 256, 0, stream>>>(d_text, n, d_toff, *d_line_start);
        e = cudaStreamSynchronize(stream);      // d_toff is freed below
    }
    cudaFree(d_tcnt); cudaFree(d_toff); cudaFree(d_tot);
    if (e != cudaSuccess) { cudaFree(*d_line_start); *d_line_start = nullptr; }
    return e;
}

}  // namespace
#endif
