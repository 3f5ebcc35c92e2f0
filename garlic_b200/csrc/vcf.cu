// vcf.cu — VCF tokeniser (sm_100a): the sample columns of VCF records → allele index bytes in the [n_snp][n_ind][2] block
// that K1 (kernels.cu: first_allele_kernel, code_alleles_kernel) codes with missing = 255.
//
// One CTA per record, as K0 (tokenize_tped_kernel): each thread looks at 16 characters of a tile, a block scan ranks the
// column starts (position 0 of a non-empty record and every position after a '\t'), and the thread that owns a column
// start parses that column's GT (vcf_gt.cuh:parse_gt) from global memory.  Every rank parses every column so that the
// per-record diagnostics are the same on all ranks; it stores only the columns of its own individuals
// [ind_lo, ind_lo + n_ind).
#include <climits>
#include <cstdint>

#include "kernels.h"
#include "vcf_gt.cuh"

namespace garlic {

namespace {

constexpr int kVcfChars = 16;   // characters per thread per tile

__global__ void __launch_bounds__(256)
tokenize_vcf_kernel(const char* __restrict__ text, const long long* __restrict__ off, int n_snp, int n_ind, int ind_lo,
                    uint8_t* __restrict__ alleles, int* __restrict__ n_cols, int* __restrict__ max_allele,
                    int* __restrict__ bad_col)
{
    __shared__ int s_warp[8];
    __shared__ int s_base, s_max, s_bad;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long c_lo = ind_lo, c_hi = (long long)ind_lo + n_ind;
    for (int l = blockIdx.x; l < n_snp; l += gridDim.x) {
        const char* line = text + off[l];
        const long long len = off[l + 1] - off[l];
        uint8_t* dst = alleles + (size_t)l * n_ind * 2;
        if (threadIdx.x == 0) { s_base = 0; s_max = -1; s_bad = INT_MAX; }
        __syncthreads();
        int my_max = -1, my_bad = INT_MAX;
        // position len is scanned too: a record that ends in a tab has an empty last column (an empty record has none)
        for (long long t0 = 0; t0 <= len; t0 += 256 * kVcfChars) {
            const long long i0 = t0 + (long long)threadIdx.x * kVcfChars;
            unsigned starts = 0;                       // bit k: a column starts at i0 + k
            char prev = i0 == 0 ? (len ? '\t' : ' ') : (i0 - 1 < len ? line[i0 - 1] : ' ');
#pragma unroll
            for (int k = 0; k < kVcfChars; ++k) {
                const char c = i0 + k < len ? line[i0 + k] : ' ';
                if (i0 + k <= len && prev == '\t') starts |= 1u << k;
                prev = c;
            }
            const int n = __popc(starts);
            int incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            int wbase = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) wbase += s_warp[w];
            long long col = (long long)s_base + wbase + incl - n;   // rank of this thread's first column start
            while (starts) {
                const int k = __ffs(starts) - 1;
                starts &= starts - 1;
                const long long i = i0 + k;
                int a, b;
                if (parse_gt(line + i, len - i, &a, &b)) {
                    if (col >= c_lo && col < c_hi) {
                        dst[2 * (col - c_lo)] = (uint8_t)a;
                        dst[2 * (col - c_lo) + 1] = (uint8_t)b;
                    }
                    if (a != kVcfMissing && a > my_max) my_max = a;
                    if (b != kVcfMissing && b > my_max) my_max = b;
                } else if (col < my_bad) {
                    my_bad = (int)col;
                }
                ++col;
            }
            __syncthreads();
            if (threadIdx.x == 255) s_base += wbase + incl;
            __syncthreads();
        }
        for (int o = 16; o; o >>= 1) {
            my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, o));
            my_bad = min(my_bad, __shfl_xor_sync(0xffffffffu, my_bad, o));
        }
        if (lane == 0) { atomicMax(&s_max, my_max); atomicMin(&s_bad, my_bad); }
        __syncthreads();
        if (threadIdx.x == 0) {
            n_cols[l] = s_base;
            max_allele[l] = s_max;
            bad_col[l] = s_bad == INT_MAX ? -1 : s_bad;
        }
        __syncthreads();
    }
}

}  // namespace

cudaError_t launch_tokenize_vcf(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, uint8_t* alleles,
                                int* n_cols, int* max_allele, int* bad_col, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    tokenize_vcf_kernel<<<n_snp < 148 * 8 ? n_snp : 148 * 8, 256, 0, st>>>(text, off, n_snp, n_ind, ind_lo, alleles, n_cols,
                                                                          max_allele, bad_col);
    return cudaGetLastError();
}

}  // namespace garlic
