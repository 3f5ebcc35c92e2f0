// ingest.cu — K0-GL: the per-genotype likelihood columns of a tgls file parsed on the GPU (readTGLSData's
// `ss >> gl` loop, garlic-data.cpp:1538-1554; SURVEY §8f.1).  The host hands over, per line, the raw text that follows
// the 4th field; token k of a line (blank-separated) is individual k's value.  One CTA per line: every thread scans 16
// characters, a block scan ranks the token starts, and the thread that owns a start converts its token to fp64 and
// stores it into the individual-major matrix garlic_gpu_put_gl fills (this rank keeps its own individuals' tokens, or
// with SEL the columns listed in local[n_input], common.cuh:select_local).
// Consecutive lines are handled by neighbouring CTAs, so the 8-byte stores of one individual's row merge into whole
// sectors in L2 before they reach HBM.
//
// Decimal → binary is exact where one IEEE operation suffices (Clinger's fast path: at most 15 significant digits and a
// power of ten up to 10^22 — every phred-scaled or short fixed-point value); anything else (long mantissas, huge
// exponents, inf / nan / hex, malformed tokens) is listed and converted by the caller's strtod, so the matrix equals the
// host reader's bit for bit.
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"
#include "kernels.h"

namespace garlic {

namespace {

constexpr int kTglsChars = 16;

__constant__ double c_pow10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11,
                                   1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

__device__ __forceinline__ bool is_blank(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n'; }

// token = p[0 .. n) up to the first blank; *hard = the host must convert it
__device__ double parse_decimal(const char* p, long long n, bool* hard)
{
    long long i = 0;
    bool neg = false;
    if (i < n && (p[i] == '-' || p[i] == '+')) { neg = p[i] == '-'; ++i; }
    unsigned long long m = 0;
    int nd = 0, e10 = 0;
    bool any = false, dot = false, bad = false;
    for (; i < n; ++i) {
        const char c = p[i];
        if (c >= '0' && c <= '9') {
            any = true;
            if (m == 0ull && c == '0') { if (dot) --e10; }               // leading zeros carry no digits
            else if (nd < 19) { m = m * 10ull + (unsigned long long)(c - '0'); ++nd; if (dot) --e10; }
            else { bad = true; if (!dot) ++e10; }                          // more digits than 64 bits hold exactly
        } else if (c == '.' && !dot) dot = true;
        else break;
    }
    if (i < n && (p[i] == 'e' || p[i] == 'E')) {
        ++i;
        bool eneg = false;
        if (i < n && (p[i] == '-' || p[i] == '+')) { eneg = p[i] == '-'; ++i; }
        int ex = 0, nex = 0;
        for (; i < n && p[i] >= '0' && p[i] <= '9'; ++i, ++nex) ex = ex < 100000 ? ex * 10 + (p[i] - '0') : ex;
        if (!nex) bad = true;
        e10 += eneg ? -ex : ex;
    }
    if (i < n && !is_blank(p[i])) bad = true;                             // trailing characters: inf, nan, hex, junk
    if (!any) bad = true;
    double v = 0.0;
    if (!bad && m != 0ull) {
        if (nd <= 15 && e10 >= -22 && e10 <= 22) {
            v = (double)m;                                                 // exact: m < 10^15 < 2^53
            v = e10 < 0 ? v / c_pow10[-e10] : v * c_pow10[e10];            // one correctly rounded operation
        } else bad = true;
    }
    *hard = bad;
    return neg ? -v : v;
}

template <bool SEL>
__global__ void __launch_bounds__(256)
tokenize_tgls_kernel(const char* __restrict__ text, const long long* __restrict__ off, int n_snp, int n_ind, int ind_lo,
                     const int* __restrict__ local, int n_input, double* __restrict__ out, int64_t out_stride, long long snp0,
                     int* __restrict__ n_tokens, int2* __restrict__ hard_list, unsigned* __restrict__ hard_count, unsigned hard_cap)
{
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int l = blockIdx.x; l < n_snp; l += gridDim.x) {
        const char* line = text + off[l];
        const long long len = off[l + 1] - off[l];
        if (threadIdx.x == 0) s_base = 0;
        __syncthreads();
        for (long long t0 = 0; t0 < len; t0 += 256 * kTglsChars) {
            const long long i0 = t0 + (long long)threadIdx.x * kTglsChars;
            // a token starts at a non-blank character whose predecessor is blank (or the start of the text)
            bool prev_blank = (i0 == 0 || i0 > len) ? true : is_blank(line[i0 - 1]);
            unsigned starts = 0u;
            int n = 0;
#pragma unroll
            for (int k = 0; k < kTglsChars; ++k) {
                const bool b = (i0 + k < len) ? is_blank(line[i0 + k]) : true;
                if (!b && prev_blank) { starts |= 1u << k; ++n; }
                prev_blank = b;
            }
            int incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            int wbase = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) wbase += s_warp[w];
            int k = s_base + wbase + incl - n;                           // rank of this thread's first token
            for (; starts; starts &= starts - 1u, ++k) {
                int j;
                if (SEL) { j = select_local(local, n_input, k); if (j < 0) continue; }
                else { if (k < ind_lo || k >= ind_lo + n_ind) continue; j = k - ind_lo; }
                const long long at = i0 + (__ffs((int)starts) - 1);
                bool hard = false;
                const double v = parse_decimal(line + at, len - at, &hard);
                out[(int64_t)j * out_stride + snp0 + l] = v;
                if (hard) {
                    const unsigned slot = atomicAdd(hard_count, 1u);
                    if (slot < hard_cap) hard_list[slot] = make_int2(l, k);
                }
            }
            __syncthreads();
            if (threadIdx.x == 255) s_base += wbase + incl;
            __syncthreads();
        }
        if (threadIdx.x == 0) n_tokens[l] = s_base;
        __syncthreads();
    }
}

}  // namespace

cudaError_t launch_tokenize_tgls(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, const int* local,
                                 int n_input, double* out, int64_t out_stride, long long snp0, int* n_tokens, int2* hard_list,
                                 unsigned* hard_count, unsigned hard_cap, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    const unsigned blocks = n_snp < 148 * 8 ? n_snp : 148 * 8;
    if (local)
        tokenize_tgls_kernel<true><<<blocks, 256, 0, st>>>(text, off, n_snp, n_ind, ind_lo, local, n_input, out, out_stride, snp0,
                                                           n_tokens, hard_list, hard_count, hard_cap);
    else
        tokenize_tgls_kernel<false><<<blocks, 256, 0, st>>>(text, off, n_snp, n_ind, ind_lo, nullptr, 0, out, out_stride, snp0,
                                                            n_tokens, hard_list, hard_count, hard_cap);
    return cudaGetLastError();
}

}  // namespace garlic
