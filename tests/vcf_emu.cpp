// vcf_emu.cpp — the VCF GT grammar (garlic_b200/csrc/vcf_gt.cuh:parse_gt) and the driver's VCF loader
// (garlic_b200/host/io.cpp:load_vcf, with its BGZF reader) behind a C interface, so that tests/test_vcf_ingest.py can
// check them without a GPU.  TEST HARNESS ONLY: built with io.cpp and cli.cpp; on the GPU the same parse_gt runs inside
// vcf.cu:tokenize_vcf_kernel.
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../garlic_b200/csrc/common.cuh"
#include "../garlic_b200/csrc/vcf_gt.cuh"
#include "../garlic_b200/host/garlic_host.h"

extern "C" {

int emu_parse_gt(const char* p, long long n, int* a, int* b) { return garlic::parse_gt(p, n, a, b); }

// load_vcf(path); errors go to <log_base>.error.  On success returns the number of records and fills, as one
// '\n'-separated text: the samples (tab-separated), then per record CHROM, POS, ID, REF, the ALTs (',' joined,
// '.' for none) and its line number (tab-separated), then the records' sample text each followed by '\n'.
// Returns -1 on failure, -2 if out is too small (need holds the size).
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
             (alts.empty() ? "." : alts) + "\t" + std::to_string(v.line[l]) + "\n";
    }
    for (int64_t l = 0; l < t.n_loci; ++l) {
        s.append(t.text.data() + t.text_off[l], (size_t)(t.text_off[l + 1] - t.text_off[l]));
        s += "\n";
    }
    *need = (long long)s.size();
    if ((long long)s.size() > cap) return -2;
    memcpy(out, s.data(), s.size());
    return t.n_loci;
}

}
