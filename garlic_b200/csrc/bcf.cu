// bcf.cu — BCF GT decoder (sm_100a): the GT vectors of BCF records → allele index bytes in the [n_snp][n_ind][2] block
// that K1 (kernels.cu: first_allele_kernel, code_alleles_kernel) codes with missing = 255.
//
// A BCF states every field's width, so there is nothing to tokenise: record l's n_samples × count values of `width`
// bytes start at gt + off[l] (a multiple of 4).  One CTA per record, grid-stride over records.  The common case, int8
// with count 2, is read as 32-bit words of two samples each, four words per thread in flight, coalesced across the
// warp; a word whose four bytes are all non-negative is a valid pair of calls and is decoded with byte-SIMD
// ((v >> 1) - 1 per byte, which is also 255 for a missing 0 or 1).  Any other word, and the int16 / int32 / count-1
// layouts, go through bcf_gt.cuh:decode_gt one sample per thread.  Every rank decodes every sample so that the
// per-record diagnostics are the same on all ranks; it stores only its own individuals [ind_lo, ind_lo + n_ind), or with
// SEL the samples listed in local[n_input] (common.cuh:select_local; the loads stay as they are, only the stores move).  The
// diagnostics are reduced per warp and folded in with global atomics on arrays pre-set to -1 (atomicMax for the
// largest allele index, an unsigned atomicMin for the first malformed sample), so a CTA never waits on a barrier.
//
// With FILTER (--vcf-min-gq / --vcf-min-dp) the record's GQ and DP vectors (count 1, one value per sample, staged in
// their own buffer, kernels.h:CallFilter) are read alongside GT, coalesced the same way: in the int8 count-2 path an
// int8 GQ / DP is one 16-bit load per word of two samples.  bcf_gt.cuh:bcf_value decides each value; a call that fails
// a threshold is stored as two missing alleles.  The GT rule and the largest allele index apply to the calls as
// written.  The first sample with a malformed value goes to bad_val (unsigned atomicMin on an array pre-set to -1), and
// the stored calls with a present allele set missing are counted per thread and added once per warp at the end.
#include <cstdint>

#include "bcf_gt.cuh"
#include "kernels.h"

namespace garlic {

namespace {

constexpr int kBcfThreads = 256;
constexpr int kBcfWords = 4;      // 32-bit words per thread in flight (int8, count 2)

__device__ __forceinline__ int32_t load_value(const uint8_t* p, long long k, int width)
{
    if (width == 1) return (int8_t)__ldg(p + k);
    if (width == 2) return __ldg((const int16_t*)p + k);
    return __ldg((const int32_t*)p + k);
}

// returns whether sample i is one of this handle's individuals (and was stored)
template <bool SEL>
__device__ __forceinline__ bool store_call(uint8_t* dst, long long i, long long lo, long long hi, const int* local, int n_input,
                                           uint32_t ab)
{
    if (SEL) {
        const int j = select_local(local, n_input, i);
        if (j >= 0) *(uint16_t*)(dst + 2 * j) = (uint16_t)ab;
        return j >= 0;
    }
    if (i >= lo && i < hi) { *(uint16_t*)(dst + 2 * (i - lo)) = (uint16_t)ab; return true; }
    return false;
}

// The GQ or DP values of samples i and, if two, i + 1 of a count-1 vector of `type` at p (raw bits, sign-extended):
// an int8 pair is one 16-bit load (i is even and p a multiple of 4 in the int8 count-2 path)
__device__ __forceinline__ void load_values(const uint8_t* p, int type, long long i, bool two, int32_t* v)
{
    if (type == 1 && two) {
        const uint16_t w = __ldg((const uint16_t*)(p + i));
        v[0] = (int8_t)w;
        v[1] = (int8_t)(w >> 8);
    } else {
        const int width = type == 1 ? 1 : type == 2 ? 2 : 4;
        v[0] = load_value(p, i, width);
        if (two) v[1] = load_value(p, i + 1, width);
    }
}

// the filtered values of one record (kernels.h:CallFilter); a null pointer: absent or that filter off
struct RecFilter {
    const uint8_t *gq = nullptr, *dp = nullptr;
    int gq_t = 0, dp_t = 0;
};

// the call filter on samples i (and i + 1 if two): bit j of the result set = call j fails a threshold; a malformed
// value lowers *bad to its sample
__device__ __forceinline__ unsigned filter_calls(const RecFilter& f, const CallFilter& cf, long long i, bool two, unsigned* bad)
{
    int32_t g[2] = {0, 0}, d[2] = {0, 0};
    if (f.gq) load_values(f.gq, f.gq_t, i, two, g);
    if (f.dp) load_values(f.dp, f.dp_t, i, two, d);
    unsigned fail = 0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        if (j && !two) break;
        const int rg = f.gq ? bcf_value(g[j], f.gq_t, cf.min_gq) : 1;
        const int rd = f.dp ? bcf_value(d[j], f.dp_t, cf.min_dp) : 1;
        if (rg < 0 || rd < 0) { if ((unsigned)(i + j) < *bad) *bad = (unsigned)(i + j); }
        else if (!rg || !rd) fail |= 1u << j;
    }
    return fail;
}

template <bool SEL, bool FILTER>
__global__ void __launch_bounds__(kBcfThreads)
decode_bcf_gt_kernel(const uint8_t* __restrict__ gt, const long long* __restrict__ off, const uint8_t* __restrict__ type,
                     int n_snp, int n_samples, int n_ind, int ind_lo, const int* __restrict__ local, int n_input,
                     uint8_t* __restrict__ alleles,
                     int* __restrict__ max_allele, unsigned* __restrict__ bad_sample, CallFilter cf)
{
    const long long lo = ind_lo, hi = (long long)ind_lo + n_ind;
    unsigned long long my_set = 0;                 // FILTER: stored calls set missing, over every record of this thread
    for (int l = blockIdx.x; l < n_snp; l += gridDim.x) {
        const uint8_t* p = gt + off[l];
        uint8_t* dst = alleles + (size_t)l * n_ind * 2;
        const int count = type[l] >> 4, t = type[l] & 15, width = t == 1 ? 1 : t == 2 ? 2 : 4;
        int my_max = -1;
        unsigned my_bad = 0xffffffffu, my_badv = 0xffffffffu;
        RecFilter f;
        if (FILTER) {
            const int2 ps = cf.fv_pos[l];
            const uint8_t* base = cf.fv + cf.fv_off[l];
            if (cf.min_gq && ps.x >= 0) { f.gq = base + ps.x; f.gq_t = cf.fv_type[2 * l] & 15; }
            if (cf.min_dp && ps.y >= 0) { f.dp = base + ps.y; f.dp_t = cf.fv_type[2 * l + 1] & 15; }
        }
        const bool filt = FILTER && (f.gq || f.dp);
        if (width == 1 && count == 2) {
            const uint32_t* w = (const uint32_t*)p;
            const int n_words = (n_samples + 1) / 2;
            uint32_t hmax = 0;                                   // per byte: the largest (v >> 1) of a fast word
            for (int k0 = 0; k0 < n_words; k0 += kBcfWords * kBcfThreads) {
                uint32_t x[kBcfWords];
#pragma unroll
                for (int u = 0; u < kBcfWords; ++u) {
                    const int k = k0 + u * kBcfThreads + threadIdx.x;
                    x[u] = k < n_words ? __ldg(w + k) : 0u;
                }
#pragma unroll
                for (int u = 0; u < kBcfWords; ++u) {
                    const int k = k0 + u * kBcfThreads + threadIdx.x;
                    if (k >= n_words) continue;
                    const long long i = 2LL * k;                 // the word's first sample
                    uint32_t v = x[u];
                    if (i + 1 >= n_samples) v &= 0xffffu;         // an odd sample count: the pad is not a sample
                    uint32_t out;
                    if (!(v & 0x80808080u)) {                    // four non-negative values: two valid calls
                        const uint32_t h = (v >> 1) & 0x7f7f7f7fu;
                        hmax = __vmaxu4(hmax, h);
                        out = __vsub4(h, 0x01010101u);
                    } else {
                        out = 0xffffffffu;
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            if (i + j >= n_samples) break;
                            int a, b;
                            if (decode_gt((int8_t)(v >> (16 * j)), (int8_t)(v >> (16 * j + 8)), 2, 1, &a, &b)) {
                                out = (out & ~(0xffffu << (16 * j))) | (uint32_t)(a | b << 8) << (16 * j);
                                if (a != kBcfMissing) my_max = max(my_max, a);
                                if (b != kBcfMissing) my_max = max(my_max, b);
                            } else if ((unsigned)(i + j) < my_bad) {
                                my_bad = (unsigned)(i + j);
                            }
                        }
                    }
                    unsigned drop = 0;
                    if (filt) {
                        drop = filter_calls(f, cf, i, i + 1 < n_samples, &my_badv);
                        if ((out & 0xffffu) == 0xffffu) drop &= ~1u;      // already two missing alleles: not counted
                        if ((out >> 16) == 0xffffu) drop &= ~2u;
                        out |= (drop & 1 ? 0xffffu : 0u) | (drop & 2 ? 0xffff0000u : 0u);
                    }
                    const bool s0 = store_call<SEL>(dst, i, lo, hi, local, n_input, out);
                    const bool s1 = store_call<SEL>(dst, i + 1, lo, hi, local, n_input, out >> 16);
                    if (FILTER) my_set += (s0 && (drop & 1)) + (s1 && (drop & 2));
                }
            }
            const uint32_t m = max(max(hmax & 0xff, (hmax >> 8) & 0xff), max((hmax >> 16) & 0xff, hmax >> 24));
            my_max = max(my_max, (int)m - 1);
        } else {
            for (int i = threadIdx.x; i < n_samples; i += kBcfThreads) {
                int a = kBcfMissing, b = kBcfMissing, ok = 0;
                if (count >= 1 && count <= 2) {
                    const long long k = (long long)i * count;
                    ok = decode_gt(load_value(p, k, width), count == 2 ? load_value(p, k + 1, width) : 0, count, width, &a, &b);
                }
                if (ok) {
                    if (a != kBcfMissing) my_max = max(my_max, a);
                    if (b != kBcfMissing) my_max = max(my_max, b);
                } else if ((unsigned)i < my_bad) {
                    my_bad = (unsigned)i;
                }
                bool drop = false;
                if (filt) drop = filter_calls(f, cf, i, false, &my_badv) && ok && (a != kBcfMissing || b != kBcfMissing);
                const bool s = store_call<SEL>(dst, i, lo, hi, local, n_input, ok && !drop ? (uint32_t)(a | b << 8) : 0xffffu);
                if (FILTER) my_set += s && drop;
            }
        }
        for (int o = 16; o; o >>= 1) {
            my_max = max(my_max, __shfl_xor_sync(0xffffffffu, my_max, o));
            my_bad = min(my_bad, __shfl_xor_sync(0xffffffffu, my_bad, o));
            if (FILTER) my_badv = min(my_badv, __shfl_xor_sync(0xffffffffu, my_badv, o));
        }
        if ((threadIdx.x & 31) == 0) {
            if (my_max >= 0) atomicMax(max_allele + l, my_max);
            if (my_bad != 0xffffffffu) atomicMin(bad_sample + l, my_bad);
            if (FILTER && my_badv != 0xffffffffu) atomicMin((unsigned*)cf.bad_val + l, my_badv);
        }
    }
    if (FILTER) {
        for (int o = 16; o; o >>= 1) my_set += __shfl_xor_sync(0xffffffffu, my_set, o);
        if ((threadIdx.x & 31) == 0 && my_set) atomicAdd(cf.n_set_missing, my_set);
    }
}

template <bool SEL>
void launch_bcf(unsigned blocks, const uint8_t* gt, const long long* off, const uint8_t* type, int n_snp, int n_samples,
                int n_ind, int ind_lo, const int* local, int n_input, uint8_t* alleles, int* max_allele, int* bad_sample,
                const CallFilter& cf, cudaStream_t st)
{
    if (cf.fv)
        decode_bcf_gt_kernel<SEL, true><<<blocks, kBcfThreads, 0, st>>>(gt, off, type, n_snp, n_samples, n_ind, ind_lo, local,
                                                                        n_input, alleles, max_allele, (unsigned*)bad_sample, cf);
    else
        decode_bcf_gt_kernel<SEL, false><<<blocks, kBcfThreads, 0, st>>>(gt, off, type, n_snp, n_samples, n_ind, ind_lo, local,
                                                                         n_input, alleles, max_allele, (unsigned*)bad_sample, cf);
}

}  // namespace

cudaError_t launch_decode_bcf_gt(const uint8_t* gt, const long long* off, const uint8_t* type, int n_snp, int n_samples,
                                 int n_ind, int ind_lo, const int* local, int n_input, uint8_t* alleles, int* max_allele,
                                 int* bad_sample, const CallFilter& cf, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    // -1 in each: "no allele" for atomicMax, and as unsigned the identity of atomicMin ("no malformed sample")
    cudaError_t e = cudaMemsetAsync(max_allele, 0xff, (size_t)n_snp * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(bad_sample, 0xff, (size_t)n_snp * sizeof(int), st);
    if (e == cudaSuccess && cf.fv) e = cudaMemsetAsync(cf.bad_val, 0xff, (size_t)n_snp * sizeof(int), st);
    if (e != cudaSuccess) return e;
    const unsigned blocks = n_snp < 148 * 8 ? n_snp : 148 * 8;
    if (local)
        launch_bcf<true>(blocks, gt, off, type, n_snp, n_samples, n_ind, ind_lo, local, n_input, alleles, max_allele, bad_sample, cf, st);
    else
        launch_bcf<false>(blocks, gt, off, type, n_snp, n_samples, n_ind, ind_lo, nullptr, 0, alleles, max_allele, bad_sample, cf, st);
    return cudaGetLastError();
}

}  // namespace garlic
