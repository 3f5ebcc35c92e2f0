// bcf_gt.cuh — the rule of one BCF genotype (GT) call.  __host__ __device__ so that tests/bcf_emu.cpp and the driver's
// messages run the same code on the CPU that bcf.cu:decode_bcf_gt_kernel runs on the GPU.
//
// A BCF 2.2 GT field is a typed integer vector of `count` values per sample, int8, int16 or int32.  Each value is
// (allele + 1) << 1 | phased, so 0 and 1 are a missing allele; end-of-vector (0x81, 0x8001, 0x80000001) pads a sample
// with fewer values than `count`.  Accepted, phase ignored: two values, each a missing allele or an allele index
// 0..254; a missing first allele followed by end-of-vector (a lone '.', two missing alleles); and a count-1 field whose
// one value is a missing allele (every sample a lone '.').  Everything else is rejected: haploid calls with an allele
// present, end-of-vector in the first slot, the missing-value markers (0x80, 0x8000, 0x80000000) and the other negative
// values, indices of 255 or more, and counts other than 1 and 2.
#pragma once
#include "common.cuh"

namespace garlic {

constexpr int kBcfMissing = 255;    // allele index byte of a missing allele (as kVcfMissing)
constexpr int kBcfMaxAllele = 254;  // largest allele index a GT may name

// end-of-vector of a value `width` bytes wide, sign-extended to int32
GHD int32_t bcf_eov(int width) { return width == 1 ? -127 : width == 2 ? -32767 : (int32_t)0x80000001u; }

// v0, v1: one sample's first two values, sign-extended from `width` bytes (v1 is ignored when count == 1).  Returns 1
// and the two allele index bytes (kBcfMissing for a missing allele) of a valid call, 0 otherwise.
GHD int decode_gt(int32_t v0, int32_t v1, int count, int width, int* a, int* b)
{
    if (count < 1 || count > 2 || v0 < 0 || (v0 >> 1) - 1 > kBcfMaxAllele) return 0;
    if (count == 1 || v1 == bcf_eov(width)) {        // a lone value: only a missing allele
        if (v0 > 1) return 0;
        *a = *b = kBcfMissing;
        return 1;
    }
    if (v1 < 0 || (v1 >> 1) - 1 > kBcfMaxAllele) return 0;
    *a = v0 > 1 ? (v0 >> 1) - 1 : kBcfMissing;
    *b = v1 > 1 ? (v1 >> 1) - 1 : kBcfMissing;
    return 1;
}

// One GQ or DP value of a count-1 field of `type` (1/2/3 = int8/int16/int32, 5 = float) against an integer threshold
// thr >= 1.  raw: the integer sign-extended from its width, or the float's bits.  Returns 1 if the call passes (value
// >= thr, or the missing or end-of-vector sentinel of its type), 0 if it is below thr, -1 if it is malformed (a float
// NaN other than the two sentinels 0x7F800001 / 0x7F800002, or an infinity).  Other integers compare as integers.
GHD int bcf_value(int32_t raw, int type, int thr)
{
    if (type == 5) {
        if (raw == 0x7F800001 || raw == 0x7F800002) return 1;
        if ((raw & 0x7F800000) == 0x7F800000) return -1;
        // a finite float passes iff its integer part (toward -inf) reaches thr; exact without a float compare
        const int e = ((raw >> 23) & 0xff) - 127;
        if (raw < 0 && (raw & 0x7fffffff)) return 0;   // negative (not -0)
        if (e < 0) return 0 >= thr;
        if (e >= 31) return 1;
        const uint32_t m = (uint32_t)(raw & 0x7fffff) | 0x800000u;
        const uint32_t ip = e >= 23 ? m << (e - 23) : m >> (23 - e);
        return ip >= (uint32_t)thr;
    }
    const int width = type == 1 ? 1 : type == 2 ? 2 : 4;
    const int32_t miss = width == 1 ? -128 : width == 2 ? -32768 : (int32_t)0x80000000u;
    if (raw == miss || raw == bcf_eov(width)) return 1;
    return raw >= thr;
}

}  // namespace garlic
