// bed.cu — PLINK 1 binary genotypes (.bed, SNP-major mode) coded on the GPU: the same two phases as K1 (kernels.cu), so
// that the "1" allele can be MIN-reduced across GPUs between them.
//
// A .bed row holds one SNP, individual i at bits 2(i%4) of byte i/4, PLINK's values 0 = hom A1, 1 = missing, 2 = het,
// 3 = hom A2.  The equivalent tped writes hom A1 as "A1 A1", het as "A1 A2", hom A2 as "A2 A2", missing as "0 0", so the
// "1" allele (the first non-missing character, garlic-data.cpp:112-113) is A2 iff the first present call is hom A2.
// The caller stages, per SNP, the byte columns that hold its own individuals: field sh + i of a staged row is this
// rank's individual i (sh = ind_offset % 4), the fields around them belong to other ranks and are ignored.
//   phase a (bed_count_kernel, per uploaded block): first-allele key ((2·global_ind) << 8 | id, id 1 = A1, 2 = A2 —
//            the key format of first_allele_kernel) and the four counters, nalleles counting copies of A2;
//   phase b (bed_code): nalleles of the SNPs whose "1" allele is A1 become total - nalleles, then the 2-bit transpose
//            into the individual-major packed matrix with the per-SNP recode as whole-word bit operations.
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"
#include "kernels.h"

namespace garlic {

namespace {

constexpr uint32_t kEven32 = 0x55555555u;
constexpr uint64_t kEven64 = 0x5555555555555555ull;

// even-bit mask of the fields [lo, hi) of a 16-field word (0 <= lo, hi <= 16)
__device__ __forceinline__ uint32_t field_mask(int lo, int hi)
{
    if (hi <= lo) return 0u;
    const uint64_t m = ((1ull << (2 * hi)) - 1ull) & ~((1ull << (2 * lo)) - 1ull);
    return (uint32_t)m & kEven32;
}

// one warp per SNP; lanes stride over the staged row's 32-bit words (16 fields each)
__global__ void __launch_bounds__(256)
bed_count_kernel(const uint8_t* __restrict__ stage, int64_t stride, int n_snp, int sh, int n_ind, int ind_offset,
                 int* __restrict__ counts, long long L0, unsigned long long* __restrict__ key)
{
    const int lane = threadIdx.x & 31;
    const int n_words = (sh + n_ind + 15) >> 4;
    for (long long s = blockIdx.x * 8ll + (threadIdx.x >> 5); s < n_snp; s += gridDim.x * 8ll) {
        const uint32_t* row = reinterpret_cast<const uint32_t*>(stage + s * stride);
        int n_a2 = 0, n_miss = 0, n_valid = 0, n_hom = 0;
        unsigned long long best = ~0ull;
        for (int j = lane; j < n_words; j += 32) {
            const uint32_t v = field_mask(max(sh - 16 * j, 0), min(sh + n_ind - 16 * j, 16));
            const uint32_t x = row[j];
            const uint32_t hi = (x >> 1) & v, lo = x & v;
            const uint32_t miss = lo & ~hi;
            n_a2 += __popc(hi) + __popc(hi & lo);
            n_miss += __popc(miss);
            n_valid += __popc(v);
            n_hom += __popc(~(hi ^ lo) & v);
            const uint32_t present = v & ~miss;
            if (best == ~0ull && present) {
                const int b = __ffs((int)present) - 1;
                const long long ind = ind_offset + 16ll * j + (b >> 1) - sh;
                best = ((unsigned long long)(2 * ind) << 8) | (((hi & lo) >> b) & 1u ? 2u : 1u);
            }
        }
        for (int o = 16; o; o >>= 1) {
            n_a2 += __shfl_xor_sync(0xffffffffu, n_a2, o);
            n_miss += __shfl_xor_sync(0xffffffffu, n_miss, o);
            n_valid += __shfl_xor_sync(0xffffffffu, n_valid, o);
            n_hom += __shfl_xor_sync(0xffffffffu, n_hom, o);
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other < best ? other : best;
        }
        if (lane == 0) {
            const int nonmiss = n_valid - n_miss;
            counts[s] = n_a2;
            counts[L0 + s] = 2 * nonmiss;
            counts[2 * L0 + s] = n_hom;
            counts[3 * L0 + s] = nonmiss;
            key[s] = best;
        }
    }
}

// thread per SNP: the "1" allele is A1 → nalleles = total - (copies of A2); bit s%32 of a1_words[s/32] records it
__global__ void bed_fix_kernel(const unsigned long long* __restrict__ key, long long L0, int* __restrict__ counts,
                               uint32_t* __restrict__ a1_words)
{
    const long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool a1 = s < L0 && key[s] != ~0ull && (key[s] & 0xff) == 1;
    if (a1) counts[s] = counts[L0 + s] - counts[s];
    const unsigned b = __ballot_sync(0xffffffffu, a1);
    if ((threadIdx.x & 31) == 0 && s < L0) a1_words[s >> 5] = b;
}

// one stage of a 16x16 transpose of 2-bit elements held in 16 words (element k of word r at bits 2k): swap the
// J x J blocks off the diagonal
template <int J, uint32_t M>
__device__ __forceinline__ void swap_blocks(uint32_t* x)
{
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        if (r & J) continue;
        const uint32_t t = ((x[r] >> (2 * J)) ^ x[r + J]) & M;
        x[r] ^= t << (2 * J);
        x[r + J] ^= t;
    }
}
__device__ __forceinline__ void transpose16x2(uint32_t* x)
{
    swap_blocks<8, 0x0000ffffu>(x);
    swap_blocks<4, 0x00ff00ffu>(x);
    swap_blocks<2, 0x0f0f0f0fu>(x);
    swap_blocks<1, 0x33333333u>(x);
}

// bit b of w → bit 2b of the result
__device__ __forceinline__ uint64_t spread_bits(uint32_t w)
{
    uint64_t x = w;
    x = (x | (x << 16)) & 0x0000ffff0000ffffull;
    x = (x | (x << 8)) & 0x00ff00ff00ff00ffull;
    x = (x | (x << 4)) & 0x0f0f0f0f0f0f0f0full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    x = (x | (x << 1)) & kEven64;
    return x;
}

// Tile = 1024 SNPs (blockIdx.x) x 128 fields, i.e. 32 bytes of each staged row (blockIdx.y).  The CTA loads the tile
// with 16-byte loads (whole 32-byte sectors) into shared memory laid out [column of 16 fields][SNP] with one pad word per 32 SNPs, so that warp w
// (= column) lane l (= 32-SNP word) reads its 32 words conflict-free; the lane transposes them in registers into the
// 16 packed words of its column's individuals, recodes them and stores word l of 16 rows — a warp's store is 256
// contiguous bytes of one row.
constexpr int kBedSnps = 1024, kBedCols = 8, kBedColStride = kBedSnps + kBedSnps / 32;

__global__ void __launch_bounds__(256)
bed_transpose_kernel(const uint8_t* __restrict__ stage, int64_t stride, long long L0, int sh, int n_ind,
                     const uint32_t* __restrict__ a1_words, uint64_t* __restrict__ geno, int64_t row_words)
{
    __shared__ uint32_t tile[kBedCols * kBedColStride];
    const long long s0 = (long long)blockIdx.x * kBedSnps;
    const int64_t byte0 = (int64_t)blockIdx.y * (kBedCols * 4);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int idx = it * 256 + threadIdx.x;
        const int r = idx >> 1, half = idx & 1;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (s0 + r < L0) v = *reinterpret_cast<const uint4*>(stage + (s0 + r) * stride + byte0 + 16 * half);
        uint32_t* d = tile + (4 * half) * kBedColStride + r + (r >> 5);
        d[0] = v.x; d[kBedColStride] = v.y; d[2 * kBedColStride] = v.z; d[3 * kBedColStride] = v.w;
    }
    __syncthreads();
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long word = (s0 >> 5) + lane;
    if (word >= (L0 + 31) >> 5) return;
    uint32_t x[32];
    const uint32_t* src = tile + w * kBedColStride + 33 * lane;
#pragma unroll
    for (int r = 0; r < 32; ++r) x[r] = src[r];
    transpose16x2(x);
    transpose16x2(x + 16);
    const uint64_t m = spread_bits(a1_words[word]);        // SNPs whose "1" allele is A1
    const int ind0 = ((int)blockIdx.y * kBedCols + w) * 16 - sh;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const int i = ind0 + k;
        if (i < 0 || i >= n_ind) continue;
        const uint64_t v = (uint64_t)x[k] | ((uint64_t)x[16 + k] << 32);
        const uint64_t hi = (v >> 1) & kEven64, lo = v & kEven64;
        // copies of A2: odd bit = lo, even bit = hi ^ lo; copies of A1: odd bit = ~hi, even bit = hi ^ lo (missing → 3)
        const uint64_t odd = ((lo & ~m) | (~hi & m)) & kEven64;
        geno[(int64_t)i * row_words + word] = (odd << 1) | (hi ^ lo);
    }
}

}  // namespace

cudaError_t launch_bed_count(const uint8_t* stage, int64_t stride, int n_snp, int sh, int n_ind, int ind_offset,
                             int* counts, long long L0, unsigned long long* key, cudaStream_t st)
{
    if (n_snp <= 0) return cudaSuccess;
    const int blocks = (n_snp + 7) / 8 < 148 * 16 ? (n_snp + 7) / 8 : 148 * 16;
    bed_count_kernel<<<blocks, 256, 0, st>>>(stage, stride, n_snp, sh, n_ind, ind_offset, counts, L0, key);
    return cudaGetLastError();
}

// stride must be a multiple of 32 bytes covering fields [0, sh + n_ind); a1_words: ceil(L0/32) words of scratch
cudaError_t launch_bed_code(const uint8_t* stage, int64_t stride, long long L0, int sh, int n_ind,
                            const unsigned long long* key, int* counts, uint32_t* a1_words, uint64_t* geno,
                            int64_t row_words, cudaStream_t st)
{
    if (L0 <= 0) return cudaSuccess;
    bed_fix_kernel<<<(unsigned)((L0 + 255) / 256), 256, 0, st>>>(key, L0, counts, a1_words);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const dim3 grid((unsigned)((L0 + kBedSnps - 1) / kBedSnps), (unsigned)(stride / (kBedCols * 4)));
    bed_transpose_kernel<<<grid, 256, 0, st>>>(stage, stride, L0, sh, n_ind, a1_words, geno, row_words);
    return cudaGetLastError();
}

}  // namespace garlic
