// bcf_emu.cpp — the BCF GT rule (garlic_b200/csrc/bcf_gt.cuh:decode_gt) and the driver's VCF / BCF loader
// (garlic_b200/host/io.cpp:load_vcf) behind a C interface, so that tests/test_bcf_ingest.py can check them without a
// GPU.  TEST HARNESS ONLY: built with io.cpp and cli.cpp; on the GPU the same decode_gt runs inside
// bcf.cu:decode_bcf_gt_kernel.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../garlic_b200/csrc/common.cuh"
#include "../garlic_b200/csrc/bcf_gt.cuh"
#include "../garlic_b200/host/garlic_host.h"

extern "C" {

// decode_gt of n calls (v0[i], v1[i]); out[3i..3i+2] = ok, a, b
void emu_decode_gt(const int32_t* v0, const int32_t* v1, int n, int count, int width, int32_t* out)
{
    for (int i = 0; i < n; ++i) {
        int a = -1, b = -1;
        out[3 * i] = garlic::decode_gt(v0[i], v1[i], count, width, &a, &b);
        out[3 * i + 1] = a;
        out[3 * i + 2] = b;
    }
}

// load_vcf(path); errors go to <log_base>.error.  On success returns the number of records and fills, as one
// '\n'-separated text: the samples (tab-separated), then per record CHROM, POS, ID, REF, the ALTs (',' joined, '.'
// for none), Vcf::line and the GT descriptor (-1 for VCF text) (tab-separated), then per record its Tped::text span as
// hex, then Tped::text_off (space-separated).  Returns -1 on failure, -2 if out is too small (need holds the size).
long long emu_load_vcf(const char* path, const char* log_base, char* out, long long cap, long long* need)
{
    gh::LOG.open(log_base);
    gh::Tped t;
    gh::Vcf v;
    const bool ok = gh::load_vcf(path, t, v);
    gh::LOG.close();
    if (!ok) return -1;
    std::string s;
    for (size_t i = 0; i < v.samples.size(); ++i) s += (i ? "\t" : "") + v.samples[i];
    s += "\n";
    for (int64_t l = 0; l < t.n_loci; ++l) {
        size_t c = 0;
        while (t.chr_off[c + 1] <= l) ++c;
        std::string alts;
        for (size_t k = 0; k < v.alts[l].size(); ++k) alts += (k ? "," : "") + v.alts[l][k];
        s += t.chr_names[c] + "\t" + std::to_string(t.pos[l]) + "\t" + t.snp_id[l] + "\t" + v.ref[l] + "\t" +
             (alts.empty() ? "." : alts) + "\t" + std::to_string(v.line[l]) + "\t" +
             std::to_string(v.gt_type.empty() ? -1 : (int)v.gt_type[l]) + "\n";
    }
    char hx[3];
    for (int64_t l = 0; l < t.n_loci; ++l) {
        for (int64_t k = t.text_off[l]; k < t.text_off[l + 1]; ++k) {
            snprintf(hx, sizeof(hx), "%02x", (unsigned char)t.text[k]);
            s += hx;
        }
        s += "\n";
    }
    for (size_t l = 0; l < t.text_off.size(); ++l) s += (l ? " " : "") + std::to_string(t.text_off[l]);
    s += "\n";
    *need = (long long)s.size();
    if ((long long)s.size() > cap) return -2;
    memcpy(out, s.data(), s.size());
    return t.n_loci;
}

}
