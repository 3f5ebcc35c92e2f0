// garlic_host.h — host side of the B200 GARLIC driver (command line, text loaders, KDE/GMM, writers).
//
// The process boundary of the reference (SURVEY.md §8b.1): same flags, same input files, same output
// files as `garlic` v1.1.6a (src/garlic-cli.cpp:15-174, src/garlic-main.cpp:25-421).  Everything per
// genotype runs on the GPU through include/garlic_b200.h; what is here is the per-run / per-SNP host
// work the reference also does once: parsing, map interpolation, KDE (FIGTree) + cutoff heuristic,
// GMM size classes, writers.
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <vector>

namespace gh {

extern const char* const kVersion;   // "1.1.6a": printed in the BED track lines (garlic-roh.cpp:603-605)

// ---- logging (.log / .error; errors also to stderr — garlic-errlog.cpp:24-65) -------------------
struct Log {
    FILE* log = nullptr;
    FILE* err = nullptr;
    bool open(const std::string& base);
    void close();
    void line(const std::string& s);        // to .log
    void error(const std::string& s);       // to stderr and .error
};
extern Log LOG;
std::string fmt_g(double v);                 // C++ ostream default formatting (precision 6)
std::string fmt_bool(bool b);                // TRUE / FALSE

// ---- options (garlic-cli.cpp) ---------------------------------------------------------------------
struct Options {
    std::string tped = "none", tfam = "none", tgls = "none", gl_type = "none", map = "none", out = "outfile";
    std::string build = "none", centromere = "none", freq_file = "none";
    std::string bfile = "none";  // PLINK 1 binary fileset PREFIX.bed / .bim / .fam in place of --tped / --tfam
    std::string vcf = "none";    // VCF in place of --tped (--tfam optional)
    bool weighted = false, cm = false, auto_winsize = false, auto_overlap = false, raw_lod = false;
    bool freq_only = false, phased = false, no_kde_thinning = false;
    int winsize = 0, auto_winsize_step = 10, max_gap = 200000, resample = 0, threads = 1, M = 7, nclust = 3;
    int kde_subsample = 20, ld_subsample = 0;
    std::vector<int> winsize_multi{-1};
    std::vector<double> size_bounds{-1};
    double error = -1, overlap_frac = 0.25, lod_cutoff = -999999, mu = 1e-9;
    char tped_missing = '0';
    bool exact = false;          // extension: whole-segment chains everywhere (--exact)
    int device = 0;              // extension: first CUDA device (--device)
    int gpus = 1;                // extension: shard the individuals over this many GPUs (--gpus)
    bool device_lut = false;     // extension: build the per-SNP LOD table on the GPU (--device-lut)
    bool host_tokenize = false;  // extension: extract the tped allele characters on the host instead of K0 (--host-tokenize)
    bool kde_direct = false;     // extension: exact (reproducible) Gauss transform for the KDE (--kde-direct)
    bool kde_gpu = false;        // extension: computeKDE on the GPU, from the thinned windows still in HBM (--kde-gpu)
    long seed = -1;              // extension: RNG seed for the KDE / LD subsamples (--seed; default time)
};
// returns 0 = run, 1 = help printed (exit 0), -1 = error
int parse_cli(int argc, char** argv, Options& o, std::string& cmdline);

// ---- inputs -------------------------------------------------------------------------------------------
struct Tped {
    int n_ind = 0;
    int64_t n_loci = 0;
    std::vector<std::string> chr_names;          // as written in the file
    std::vector<int64_t> chr_off;                // [C+1]
    std::vector<int32_t> pos;
    std::vector<std::string> snp_id;
    std::vector<uint8_t> alleles;                // [L0][N][2]  (only with --host-tokenize)
    std::vector<char> text;                      // raw genotype columns of every line (what follows the 4th field) …
    std::vector<int64_t> text_off;               // … line l = text[text_off[l], text_off[l+1]): tokenised on the GPU (K0)
};
// host_tokenize: extract the allele characters here (the pre-K0 path, kept for A/B timing) instead of keeping raw text
bool load_tped(const std::string& path, char missing, Tped& t, bool host_tokenize = false);
struct Tfam { std::string pop; std::vector<std::string> ids; };
bool load_tfam(const std::string& path, Tfam& f);
// PLINK .bim: chr / id / cM / bp fill the tped's first four columns (same chromosome log lines as load_tped); a1 / a2 =
// the allele names of columns 5 and 6
bool load_bim(const std::string& path, Tped& t, std::vector<std::string>& a1, std::vector<std::string>& a2);
// PLINK .bed header and size: magic 6c 1b, SNP-major mode 01, 3 + n_loci * ceil(n_ind/4) bytes; leaves f after the header
bool open_bed(const std::string& path, int n_ind, int64_t n_loci, FILE*& f);
// VCF (plain, gzip or BGZF — the last inflated block-parallel): the #CHROM line's samples take the place of the tfam's
// individuals; per record CHROM / ID / POS fill the tped's columns 1 / 2 / 4 (same chromosome log lines as load_tped),
// and the sample columns (the text after FORMAT's tab) go to Tped::text / text_off for the GPU (garlic_gpu_put_vcf_text).
// FORMAT must be GT or start with GT:.  QUAL, FILTER and INFO are ignored.
struct Vcf {
    std::vector<std::string> samples;
    std::vector<std::string> ref;                 // per record
    std::vector<std::vector<std::string>> alts;   // per record, ALT split on ',' ('.' = none)
    std::vector<int64_t> line;                    // per record, its line number in the file (for messages)
};
bool load_vcf(const std::string& path, Tped& t, Vcf& v);
struct Scaffold { std::string chr; std::vector<int32_t> pos; std::vector<double> gen; };
bool load_map(const std::string& path, std::vector<Scaffold>& s);
// values individual-major [N][L0]
bool load_tgls(const std::string& path, const Tped& t, std::vector<double>& values);
// K0-GL: the tgls file streamed in blocks of lines; per block the raw value columns (what follows the 4th field of every
// line) and their offsets, converted on the GPU (garlic_gpu_put_tgls_text).  A missing line yields an empty tail, which
// fails the column check exactly as the reference's getline on a short file does (garlic-data.cpp:1529-1536).
struct TglsBlocks {
    void* impl = nullptr;
    bool open(const std::string& path);
    // up to max_lines lines: text / off[n+1]; returns the number of lines delivered (short files: padded with empty lines)
    int next(int max_lines, std::vector<char>& text, std::vector<int64_t>& off);
    ~TglsBlocks();
};
// readFreqData (garlic-data.cpp:1345-1440): CHR SNP POS ALLELE FREQ rows in tped order; 1 - freq where ALLELE is not the
// "1" allele.  one_allele: its name per SNP; by_name = false compares the first character of ALLELE as the reference's
// `ss >> char` does (tped input), true the whole token (.bim allele names may be longer than one character)
bool load_freq_file(const std::string& path, const Tped& t, const std::vector<std::string>& one_allele, bool by_name,
                    std::vector<double>& freq);
std::string chr_label(const std::string& name);   // checkChrName, garlic-data.cpp:1886-1891
// centromere table: build = hg18/hg19/hg38 or custom file "<chr> <start> <end>"
bool load_centromeres(const std::string& build, const std::string& file, std::map<std::string, std::pair<int, int>>& cen);
// interpolateGeneticmap / getMapInfo / interpolate (garlic-data.cpp:702-757)
bool interpolate_map(const int32_t* pos, int64_t n, const Scaffold& s, double* gpos, int& n_interp);

// ---- KDE + cutoff (garlic-kde.cpp) ----------------------------------------------------------------
struct Kde { std::vector<double> x, y; };
void compute_kde(std::vector<double>& data, Kde& k, bool direct = false);   // sorts data in place (nrd0)
double min_between_modes(const Kde& k, int wsize);             // get_min_btw_modes
double wiggle(Kde& k, int fit = 20);                           // calculateWiggle (scales y by 100 in place)
bool write_kde(const Kde& k, const std::string& path);

// ---- GMM size classes (gmm.cpp, BoundFinder.cpp, garlic-roh.cpp:935-1003) ---------------------------
bool size_classes(const std::vector<double>& lengths, int nclust, std::vector<double>& bounds);

// ---- writers ------------------------------------------------------------------------------------------
bool write_freq_gz(const std::string& path, const Tped& t, const std::vector<std::string>& one_allele,
                   const std::vector<double>& freq);
struct Roh { int ind, chr; double start, stop, length; };
bool write_bed(const std::string& path, const std::vector<Roh>& roh, const std::vector<std::string>& ind_ids,
               const std::vector<std::string>& chr_labels, const std::vector<double>& bounds, const std::string& pop,
               bool cm);

}  // namespace gh
