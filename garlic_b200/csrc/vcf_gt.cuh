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

// One FORMAT value (GQ or DP) against an integer threshold thr >= 1: p is the value's first character, it ends at ':',
// '\t' or the end of the line.  Returns 1 if the call passes (value >= thr, or the value is missing: empty or '.'), 0
// if it is below thr, -1 if it is malformed.  Accepted: an optional '-', one or more digits, then optionally '.' and
// one or more digits; I.F passes iff I >= thr, so no floating-point parse is needed, and the digits saturate once they
// reach thr.  Everything else (letters, exponents, "nan", a lone '-') is malformed.
GHD int fmt_value(const char* p, long long n, int thr)
{
    if (gt_end(p, 0, n) || (p[0] == '.' && gt_end(p, 1, n))) return 1;
    const bool neg = p[0] == '-';
    long long i = neg, x = 0;
    for (; i < n && p[i] >= '0' && p[i] <= '9'; ++i)
        if (x < thr) x = 10 * x + (p[i] - '0');
    if (i == neg) return -1;
    if (i < n && p[i] == '.') {
        const long long f0 = ++i;
        while (i < n && p[i] >= '0' && p[i] <= '9') ++i;
        if (i == f0) return -1;
    }
    if (!gt_end(p, i, n)) return -1;
    return !neg && x >= thr;
}

// The call filter of one sample column: p its first character (the GT), n the characters left on the line; k_gq /
// k_dp the FORMAT indices of GQ and DP in this record (-1: absent, or that filter is off), min_gq / min_dp their
// thresholds.  Returns 0 if the call passes, 1 if a value is below its threshold (the call is set missing), -1 if a
// value is malformed, with *field = 0 (GQ) or 1 (DP).  A subfield the column omits (trailing fields dropped) passes.
GHD int call_filter(const char* p, long long n, int k_gq, int min_gq, int k_dp, int min_dp, int* field)
{
    const int k_last = k_gq > k_dp ? k_gq : k_dp;
    int fail = 0;
    long long i = 0;
    for (int k = 0; k <= k_last; ++k) {
        if (k == k_gq || k == k_dp) {
            const int r = fmt_value(p + i, n - i, k == k_gq ? min_gq : min_dp);
            if (r < 0) { *field = k == k_gq ? 0 : 1; return -1; }
            fail |= r == 0;
        }
        while (i < n && p[i] != ':' && p[i] != '\t') ++i;
        if (i >= n || p[i] == '\t') break;
        ++i;
    }
    return fail;
}

}  // namespace garlic
