// vcf_gt.cuh — the grammar of one VCF genotype (GT) field.  __host__ __device__ so that tests/vcf_emu.cpp runs the same
// code on the CPU that vcf.cu:tokenize_vcf_kernel runs on the GPU.
//
// The GT is the start of a sample column, up to ':' (more FORMAT keys follow), '\t' (the next sample) or the end of the
// line.  Accepted: two alleles separated by '/' or '|', each '.' (missing) or a decimal allele index 0..254, or a lone
// '.' (both alleles missing).  Everything else is rejected: haploid and polyploid calls, empty fields, signs, letters,
// and indices of 255 or more (a VCF record's alleles are coded in one byte, 255 being the missing code).
#pragma once
#include "common.cuh"

namespace garlic {

constexpr int kVcfMissing = 255;    // allele index byte of a missing allele
constexpr int kVcfMaxAllele = 254;  // largest allele index a GT may name

GHD bool gt_end(const char* p, long long i, long long n) { return i >= n || p[i] == ':' || p[i] == '\t'; }

// p: the first character of a sample column, n: characters left on the line.  Returns 1 and the two allele index bytes
// (kVcfMissing for '.') of a valid GT, 0 otherwise.
GHD int parse_gt(const char* p, long long n, int* a, int* b)
{
    int v[2] = {0, 0};
    long long i = 0;
    for (int k = 0; k < 2; ++k) {
        if (i < n && p[i] == '.') {
            v[k] = kVcfMissing;
            ++i;
        } else {
            int x = 0, digits = 0;
            for (; i < n && p[i] >= '0' && p[i] <= '9'; ++i, ++digits) {
                x = 10 * x + (p[i] - '0');
                if (x > kVcfMaxAllele) return 0;
            }
            if (!digits) return 0;
            v[k] = x;
        }
        if (k == 0) {
            if (v[0] == kVcfMissing && gt_end(p, i, n)) { *a = *b = kVcfMissing; return 1; }   // lone '.'
            if (i >= n || (p[i] != '/' && p[i] != '|')) return 0;
            ++i;
        }
    }
    if (!gt_end(p, i, n)) return 0;
    *a = v[0];
    *b = v[1];
    return 1;
}

}  // namespace garlic
