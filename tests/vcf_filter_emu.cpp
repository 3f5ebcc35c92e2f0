// vcf_filter_emu.cpp — the call filter's rules (garlic_b200/csrc/vcf_gt.cuh:fmt_value / call_filter, bcf_gt.cuh:
// bcf_value) and the driver's loader with GQ / DP (garlic_b200/host/io.cpp:load_vcf with call_keys) behind a C
// interface, so that tests/test_vcf_call_filter.py can check them without a GPU.  TEST HARNESS ONLY: built with io.cpp
// and cli.cpp; on the GPU the same rules run inside vcf.cu:tokenize_vcf_kernel and bcf.cu:decode_bcf_gt_kernel.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../garlic_b200/csrc/common.cuh"
#include "../garlic_b200/csrc/bcf_gt.cuh"
#include "../garlic_b200/csrc/vcf_gt.cuh"
#include "../garlic_b200/host/garlic_host.h"

extern "C" {

int emu_fmt_value(const char* p, long long n, int thr) { return garlic::fmt_value(p, n, thr); }

// returns call_filter's result; *field = -1 unless a value is malformed
int emu_call_filter(const char* p, long long n, int k_gq, int min_gq, int k_dp, int min_dp, int* field)
{
    *field = -1;
    return garlic::call_filter(p, n, k_gq, min_gq, k_dp, min_dp, field);
}

void emu_bcf_value(const int32_t* raw, int n, int type, int thr, int32_t* out)
{
    for (int i = 0; i < n; ++i) out[i] = garlic::bcf_value(raw[i], type, thr);
}

// load_vcf(path, call_keys); errors go to <log_base>.error.  On success returns the number of records and fills, as
// '\n'-separated lines: Vcf::fmt_index, Vcf::fv as hex, Vcf::fv_off, Vcf::fv_pos, Vcf::fv_type (space-separated
// numbers), then Tped::text as hex.  Returns -1 on failure, -2 if out is too small (need holds the size).
long long emu_load_filter(const char* path, const char* log_base, unsigned call_keys, char* out, long long cap, long long* need)
{
    gh::LOG.open(log_base);
    gh::Tped t;
    gh::Vcf v;
    const bool ok = gh::load_vcf(path, t, v, call_keys);
    gh::LOG.close();
    if (!ok) return -1;
    std::string s;
    auto nums = [&](const auto& a) {
        for (size_t i = 0; i < a.size(); ++i) s += (i ? " " : "") + std::to_string((long long)a[i]);
        s += "\n";
    };
    auto hex = [&](const auto& a) {
        char hx[3];
        for (size_t i = 0; i < a.size(); ++i) { snprintf(hx, sizeof(hx), "%02x", (unsigned char)a[i]); s += hx; }
        s += "\n";
    };
    nums(v.fmt_index);
    hex(v.fv);
    nums(v.fv_off);
    nums(v.fv_pos);
    nums(v.fv_type);
    hex(t.text);
    *need = (long long)s.size();
    if ((long long)s.size() > cap) return -2;
    memcpy(out, s.data(), s.size());
    return t.n_loci;
}

}
