// cli.cpp — flag parsing with the reference's surface and rules (src/garlic-cli.cpp:15-174 flag names and
// defaults, src/param_t.cpp:230-400 parsing rules: bool flags toggle, list flags run to the next flag,
// numbers may not use exponent notation, duplicates are errors), plus .log / .error handling
// (src/garlic-errlog.cpp).
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <set>
#include <sstream>

#include "garlic_host.h"

namespace gh {

const char* const kVersion = "1.1.6a";
Log LOG;

bool Log::open(const std::string& base)
{
    log = fopen((base + ".log").c_str(), "w");
    if (!log) { fprintf(stderr, "ERROR: Could not open %s.log for logging.\n", base.c_str()); return false; }
    err = fopen((base + ".error").c_str(), "w");
    if (!err) { fprintf(stderr, "ERROR: Could not open %s.error for logging.\n", base.c_str()); return false; }
    return true;
}
void Log::close()
{
    if (log) fclose(log);
    if (err) fclose(err);
    log = err = nullptr;
}
void Log::line(const std::string& s)
{
    if (hold) { held.push_back(s); return; }
    if (log) { fputs(s.c_str(), log); fputc('\n', log); fflush(log); }
}
void Log::error(const std::string& s)
{
    last = s;
    fprintf(stderr, "%s\n", s.c_str());
    if (err) { fputs(s.c_str(), err); fputc('\n', err); fflush(err); }
}

std::string fmt_g(double v)
{
    std::ostringstream ss;   // exactly what `ostream << double` prints in the reference
    ss << v;
    return ss.str();
}
std::string fmt_bool(bool b) { return b ? "TRUE" : "FALSE"; }

static bool good_double(const std::string& s)   // param_t::goodDouble: digits, one '.', leading '-'
{
    int dots = 0;
    for (size_t i = 0; i < s.size(); ++i) {
        const char c = s[i];
        if (!isdigit((unsigned char)c) && c != '.' && c != '-') return false;
        if (c == '.') dots++;
        if (c == '-' && i != 0) return false;
        if (dots > 1) return false;
    }
    return true;
}
static bool good_int(const std::string& s)
{
    for (size_t i = 0; i < s.size(); ++i) {
        const char c = s[i];
        if (!isdigit((unsigned char)c) && c != '-') return false;
        if (c == '-' && i != 0) return false;
    }
    return true;
}

static const char* kHelp =
    "\ngarlic_b200 -- B200-native implementation of the GARLIC v1.1.6a LOD/wLOD -> ROH path.\n"
    "Flags (same names, defaults and meaning as garlic): --tped --tfam --tgls --gl-type --map --weighted --cm\n"
    "  --winsize --winsize-multi --auto-winsize --auto-winsize-step --overlap-frac --auto-overlap-frac --error\n"
    "  --max-gap --lod-cutoff --size-bounds --kde-subsample --ld-subsample --no-kde-thinning --nclust --M --mu\n"
    "  --build --centromere --tped-missing --threads --resample --out --raw-lod\n"
    "Extensions: --bfile <prefix> (PLINK 1 binary fileset prefix.bed/.bim/.fam in place of --tped/--tfam; not with --phased),\n"
    "  --vcf <file> (VCF, plain, gzip or BGZF, or BCF 2.2, uncompressed or BGZF, in place of --tped; FORMAT must start\n"
    "  with GT and every GT must be diploid, so restrict the input to the autosomes; QUAL, FILTER and INFO are ignored and\n"
    "  no filter is applied except --vcf-min-gq / --vcf-min-dp; --tfam is optional:\n"
    "  its IDs must equal the VCF samples in order and it names the population, which is VCF without it; not with\n"
    "  --host-tokenize),\n"
    "  --vcf-min-gq <T>, --vcf-min-dp <D> (--vcf input only, integers >= 1: a call whose FORMAT GQ is below T, or whose DP\n"
    "  is below D, is set missing, as if written ./.; a missing or absent value passes; QUAL, FILTER and INFO are still\n"
    "  ignored),\n"
    "  --gpus <n> (shard individuals over n GPUs), --exact (whole-segment chains), --device <n>, --seed <n> (subsample RNG seed), --device-lut, --kde-direct, --kde-gpu (the KDE itself on the GPU: exact Gauss transform of the thinned windows still in HBM), --host-tokenize (tped allele columns extracted on the host instead of the GPU tokeniser)\n"
    "  --by-pop (a tfam or .fam with several population IDs, the first column: each population, in order of first\n"
    "  appearance, is analysed as a separate run with the same flags would analyse it, its outputs under <out>.<pop>;\n"
    "  <out>.log lists the populations; with --gpus n each population is sharded over min(n, its size) GPUs)\n";

int parse_cli(int argc, char** argv, Options& o, std::string& cmdline)
{
    cmdline.clear();
    for (int i = 0; i < argc; ++i) { cmdline += argv[i]; cmdline += " "; }
    std::map<std::string, bool*> fb = {{"--weighted", &o.weighted}, {"--cm", &o.cm}, {"--auto-winsize", &o.auto_winsize},
        {"--auto-overlap-frac", &o.auto_overlap}, {"--raw-lod", &o.raw_lod}, {"--freq-only", &o.freq_only},
        {"--phased", &o.phased}, {"--no-kde-thinning", &o.no_kde_thinning}, {"--exact", &o.exact}, {"--device-lut", &o.device_lut}, {"--kde-direct", &o.kde_direct}, {"--kde-gpu", &o.kde_gpu}, {"--host-tokenize", &o.host_tokenize},
        {"--by-pop", &o.by_pop}};
    std::map<std::string, int*> fi = {{"--winsize", &o.winsize}, {"--auto-winsize-step", &o.auto_winsize_step},
        {"--max-gap", &o.max_gap}, {"--resample", &o.resample}, {"--threads", &o.threads}, {"--M", &o.M},
        {"--nclust", &o.nclust}, {"--kde-subsample", &o.kde_subsample}, {"--ld-subsample", &o.ld_subsample},
        {"--device", &o.device}, {"--gpus", &o.gpus}, {"--vcf-min-gq", &o.vcf_min_gq}, {"--vcf-min-dp", &o.vcf_min_dp}};
    std::map<std::string, double*> fd = {{"--error", &o.error}, {"--overlap-frac", &o.overlap_frac},
        {"--lod-cutoff", &o.lod_cutoff}, {"--mu", &o.mu}};
    std::map<std::string, std::string*> fs = {{"--tped", &o.tped}, {"--tfam", &o.tfam}, {"--tgls", &o.tgls},
        {"--gl-type", &o.gl_type}, {"--map", &o.map}, {"--out", &o.out}, {"--build", &o.build},
        {"--centromere", &o.centromere}, {"--freq-file", &o.freq_file}, {"--bfile", &o.bfile}, {"--vcf", &o.vcf}};
    auto is_flag = [&](const std::string& s) {
        return fb.count(s) || fi.count(s) || fd.count(s) || fs.count(s) || s == "--winsize-multi" || s == "--size-bounds" ||
               s == "--tped-missing" || s == "--seed" || s == "--help";
    };
    std::set<std::string> seen;
    if (argc < 2) { fputs(kHelp, stderr); return 1; }
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        if (a == "--help") { fputs(kHelp, stderr); return 1; }
        if (seen.count(a)) { fprintf(stderr, "ERROR: Duplicate %s found.\n", a.c_str()); return -1; }
        if (fb.count(a)) { *fb[a] = !*fb[a]; seen.insert(a); continue; }
        if (!is_flag(a)) { fprintf(stderr, "ERROR: %s is not a valid flag.\n", a.c_str()); return -1; }
        if (i + 1 >= argc) { fprintf(stderr, "ERROR: No argument found for %s.\n", a.c_str()); return -1; }
        const std::string v = argv[i + 1];
        if (fi.count(a)) {
            if (!good_int(v)) { fprintf(stderr, "ERROR: %s is not a valid integer.\n", v.c_str()); return -1; }
            *fi[a] = atoi(v.c_str());
            if ((a == "--vcf-min-gq" || a == "--vcf-min-dp") && *fi[a] < 1) {
                fprintf(stderr, "ERROR: %s must be an integer >= 1.\n", a.c_str());
                return -1;
            }
            ++i;
        } else if (a == "--seed") {
            if (!good_int(v)) { fprintf(stderr, "ERROR: %s is not a valid integer.\n", v.c_str()); return -1; }
            o.seed = atol(v.c_str());
            ++i;
        } else if (fd.count(a)) {
            if (!good_double(v)) { fprintf(stderr, "ERROR: %s is not a valid double.\n", v.c_str()); return -1; }
            *fd[a] = atof(v.c_str());
            ++i;
        } else if (fs.count(a)) {
            *fs[a] = v;
            ++i;
        } else if (a == "--tped-missing") {
            if (v.size() > 1) { fprintf(stderr, "ERROR: %s is not a valid character.\n", v.c_str()); return -1; }
            o.tped_missing = v[0];
            ++i;
        } else if (a == "--winsize-multi") {
            o.winsize_multi.clear();
            while (i + 1 < argc) {
                const std::string w = argv[i + 1];
                if (good_int(w)) { o.winsize_multi.push_back(atoi(w.c_str())); ++i; }
                else if (!is_flag(w)) { fprintf(stderr, "ERROR: %s is not a valid integer.\n", w.c_str()); return -1; }
                else break;
            }
            if (o.winsize_multi.empty()) { fprintf(stderr, "ERROR: No arguments found for %s.\n", a.c_str()); return -1; }
        } else if (a == "--size-bounds") {
            o.size_bounds.clear();
            while (i + 1 < argc) {
                const std::string w = argv[i + 1];
                if (good_double(w)) { o.size_bounds.push_back(atof(w.c_str())); ++i; }
                else if (!is_flag(w)) { fprintf(stderr, "ERROR: %s is not a valid double.\n", w.c_str()); return -1; }
                else break;
            }
            if (o.size_bounds.empty()) { fprintf(stderr, "ERROR: No arguments found for %s.\n", a.c_str()); return -1; }
        }
        seen.insert(a);
    }
    return 0;
}

}  // namespace gh
