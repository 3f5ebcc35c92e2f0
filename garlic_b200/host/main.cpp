// main.cpp — `garlic_b200`: command-line driver with the reference's process boundary (flags, inputs, outputs,
// order of operations and log lines of src/garlic-main.cpp:25-421), calling the hand-written kernels through
// the C ABI of include/garlic_b200.h.  There is no CPU path for the per-genotype work: without a CUDA device
// the program stops at garlic_gpu_create.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <random>
#include <thread>

#include <zlib.h>

#include "../../include/garlic_b200.h"
#include "garlic_host.h"
#include "../csrc/bcf_gt.cuh"
#include "../csrc/vcf_gt.cuh"

using namespace gh;

namespace {

// --gpus G: individuals are sharded over G GPUs (rank r = individuals [lo_r, hi_r)); rank 0 is the main thread,
// ranks 1..G-1 are follower threads that mirror every GPU call (the library's NCCL collectives inside
// code_alleles / filter / windows_gather need all ranks in the call at the same time).
struct Rank {
    int rank = 0, lo = 0, hi = 0;
    garlic_gpu_t* g = nullptr;
    std::vector<garlic_roh_t> rec;
    int64_t n_roh = 0;
    std::string err;
};

struct Team {
    std::vector<Rank> ranks;                 // ranks[0] is the main thread's
    std::vector<std::thread> threads;
    std::mutex mu;
    std::condition_variable cv;
    std::function<bool(Rank&)> job;
    long generation = 0;
    int pending = 0;
    bool quit = false, failed = false;

    void follower(int r, long seen)
    {
        for (;;) {
            std::function<bool(Rank&)> j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return quit || generation != seen; });
                if (quit) return;
                seen = generation;
                j = job;
            }
            const bool ok = j(ranks[r]);
            std::lock_guard<std::mutex> lk(mu);
            if (!ok) failed = true;
            --pending;
            cv.notify_all();
        }
    }
    // run `j` on every rank at the same time (rank 0 on the calling thread); false if any rank failed
    bool all(const std::function<bool(Rank&)>& j)
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            job = j;
            pending = (int)ranks.size() - 1;
            ++generation;
        }
        cv.notify_all();
        const bool ok0 = j(ranks[0]);
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return pending == 0; });
        if (!ok0) failed = true;
        return !failed;
    }
    void start(int G)
    {
        ranks.assign(G, Rank());
        quit = failed = false;
        for (int r = 1; r < G; ++r) threads.emplace_back(&Team::follower, this, r, generation);
    }
    void stop()
    {
        { std::lock_guard<std::mutex> lk(mu); quit = true; }
        cv.notify_all();
        for (auto& t : threads) t.join();
        threads.clear();
    }
    ~Team() { if (!threads.empty()) stop(); }
    std::string first_error() const
    {
        for (const Rank& r : ranks) if (!r.err.empty()) return "rank " + std::to_string(r.rank) + ": " + r.err;
        return "unknown error";
    }
};

// BCF: the first sample of record s whose GT names an allele index above n_alt (bcf_gt.cuh:decode_gt, the rule the GPU
// applies), -1 if none
int bcf_sample_above(const Tped& t, const Vcf& v, int64_t s, int n_alt)
{
    const int count = v.gt_type[s] >> 4, type = v.gt_type[s] & 15, w = type == 3 ? 4 : type;
    const unsigned char* p = (const unsigned char*)t.text.data() + t.text_off[s];
    auto value = [&](int64_t k) -> int32_t {
        const unsigned char* q = p + k * w;
        return w == 1 ? (int8_t)q[0] : w == 2 ? (int16_t)(q[0] | q[1] << 8) : (int32_t)(q[0] | q[1] << 8 | q[2] << 16 | (uint32_t)q[3] << 24);
    };
    for (int i = 0; i < t.n_ind && count <= 2; ++i) {
        int a, b;
        if (garlic::decode_gt(value((int64_t)i * count), count == 2 ? value((int64_t)i * count + 1) : 0, count, w, &a, &b) &&
            ((a != garlic::kBcfMissing && a > n_alt) || (b != garlic::kBcfMissing && b > n_alt)))
            return i;
    }
    return -1;
}

bool rank_ok(Rank& r, int rc, const char* what)
{
    if (rc == 0) return true;
    r.err = std::string(what) + ": " + garlic_gpu_last_error(r.g);
    return false;
}

struct Ctx {
    Options o;
    Team team;
    garlic_gpu_t* g = nullptr;               // = team.ranks[0].g
    Tped tped;
    Tfam tfam;
    std::vector<Scaffold> scaffold;
    std::map<std::string, std::pair<int, int>> cen;
    std::vector<std::string> labels;            // chr labels ("chr1", …) in data order
    std::vector<int32_t> cen_arr;               // [C][2]
    int64_t L = 0;
    std::vector<int32_t> pos;                   // kept positions
    std::vector<int64_t> chr_off;               // kept offsets [C+1]
    std::vector<double> gpos;                   // kept genetic positions (weighted / cm)
    std::mt19937 rng;
};

bool gpu_ok(Ctx& c, int rc, const char* what)
{
    if (rc == 0) return true;
    LOG.error(std::string("ERROR: ") + what + ": " + garlic_gpu_last_error(c.g));
    return false;
}

// gsl_ran_choose (selection sampling, keeps source order) with gsl_rng_uniform = mt19937()/2^32
std::vector<int32_t> choose(Ctx& c, int k, int n)
{
    std::vector<int32_t> out;
    for (int i = 0; i < n && (int)out.size() < k; ++i)
        if ((n - i) * (c.rng() / 4294967296.0) < k - (int)out.size()) out.push_back(i);
    return out;
}

// calcLDData (garlic-data.cpp:330-375) on every rank at once: `ld` lists individuals of the whole sample (empty =
// all); each GPU contributes the bit-planes of the LD individuals it holds and the library all-reduces them.
bool ld_band_all(Ctx& c, int W, const std::vector<int32_t>& ld)
{
    if (!c.team.all([&](Rank& R) {
            garlic_gpu_set_wlod(R.g, c.o.mu, c.o.M);
            garlic_gpu_set_phased(R.g, c.o.phased ? 1 : 0);     // calcR2LD instead of calcHR2LD (garlic-data.cpp:371)
            return rank_ok(R, garlic_gpu_ld_band(R.g, W, ld.empty() ? nullptr : ld.data(), (int)ld.size(), nullptr), "ld_band");
        })) { LOG.error("ERROR: " + c.team.first_error()); return false; }
    return true;
}

// convert[Subset]WinData2DoubleData (garlic-data.cpp:2026-2150): chr → individual → locus, MISSING/NaN dropped.
// inds: global individual indices (ascending) or nullptr for all; every rank computes the windows of its own
// individuals and the library all-gathers them (rank order = individual order).
bool thinned_windows(Ctx& c, int W, int step, const std::vector<int32_t>* inds, std::vector<double>& out)
{
    const int G = (int)c.team.ranks.size();
    std::vector<std::vector<int32_t>> local(G);
    int rows = 0;
    for (int r = 0; r < G; ++r) {
        const Rank& R = c.team.ranks[r];
        if (inds) { for (int i : *inds) if (i >= R.lo && i < R.hi) local[r].push_back(i - R.lo); }
        else { for (int i = R.lo; i < R.hi; ++i) local[r].push_back(i - R.lo); }
        rows = std::max(rows, (int)local[r].size());
    }
    const int64_t slots = garlic_gpu_window_slots(c.g, step);
    std::vector<double> m((size_t)G * rows * slots);
    const bool weighted = c.o.weighted;
    if (!c.team.all([&](Rank& R) {
            std::vector<double> scratch;
            double* dst = R.rank == 0 ? m.data() : (scratch.resize(m.size()), scratch.data());
            return rank_ok(R, garlic_gpu_windows_gather(R.g, W, step, weighted, local[R.rank].data(), (int)local[R.rank].size(), rows,
                                                        1 /* whole-segment chains */, dst), "windows");
        })) { LOG.error("ERROR: " + c.team.first_error()); return false; }
    out.clear();
    int64_t base = 0;
    for (size_t ch = 0; ch + 1 < c.chr_off.size(); ++ch) {
        const int64_t ns = (c.chr_off[ch + 1] - c.chr_off[ch] + step - 1) / step;
        for (int r = 0; r < G; ++r)
            for (size_t i = 0; i < local[r].size(); ++i)
                for (int64_t sl = 0; sl < ns; ++sl) {
                    const double v = m[((size_t)r * rows + i) * slots + base + sl];
                    if (v != GARLIC_MISSING && !std::isnan(v)) out.push_back(v);
                }
        base += ns;
    }
    return true;
}

// --kde-gpu: computeKDE (garlic-kde.cpp:14-101) on the GPU, from the thinned windows the gather left in rank 0's HBM
// (every rank holds the whole gathered matrix); the 512 sums come back, the normalisation (:86-95) is done here.
bool compute_kde_gpu(Ctx& c, size_t n_expected, Kde& k)
{
    const int M = 512;
    LOG.line("KDE with " + std::to_string(n_expected) + " points.");
    k.x.assign(M, 0.0);
    k.y.assign(M, 0.0);
    int64_t n = 0;
    double h = 0;
    if (!gpu_ok(c, garlic_gpu_kde(c.g, nullptr, 0, M, k.x.data(), k.y.data(), &n, &h), "kde")) return false;
    if ((size_t)n != n_expected) { LOG.error("ERROR: device KDE saw " + std::to_string(n) + " values, expected " + std::to_string(n_expected)); return false; }
    const double spacing = k.x[1] - k.x[0];
    double sum = 0;
    for (int i = 0; i < M; ++i) sum += k.y[i];
    for (int i = 0; i < M; ++i) k.y[i] /= (sum * spacing);
    return true;
}

double lod_host(int g, double freq, double error)   // garlic-roh.cpp:355-386
{
    double a, na;
    if (freq == 0 || freq == 1 || g == 3) { a = 1; na = 1; }
    else if (g == 0) { na = (1 - freq) * (1 - freq); a = (1 - error) * (1 - freq) + error * na; }
    else if (g == 1) { na = 2 * (freq) * (1 - freq); a = error * na; }
    else { na = (freq) * (freq); a = (1 - error) * (freq) + error * na; }
    return std::log10(a / na);
}

double calc_density(const Ctx& c)   // calcDensity, garlic-data.cpp:318-328
{
    double length = 0;
    for (size_t ch = 0; ch + 1 < c.chr_off.size(); ++ch) {
        const int64_t lo = c.chr_off[ch], hi = c.chr_off[ch + 1];
        length += c.pos[hi - 1] - c.pos[lo] + 1 - (c.cen_arr[2 * ch + 1] - c.cen_arr[2 * ch]);
    }
    return double(c.L) / length;
}

// one gz file per chromosome, one line per individual, "NA" for MISSING, 6 significant digits; individuals are
// streamed in blocks so that the window matrix never exists as a whole
bool write_raw_lod(Ctx& c, int W)
{
    const int C = (int)c.labels.size(), N = (int)c.tfam.ids.size();
    std::vector<gzFile> f(C);
    for (int ch = 0; ch < C; ++ch) {
        const std::string fn = c.o.out + "." + c.tfam.pop + "." + c.labels[ch] + ".raw.lod.windows.gz";
        f[ch] = gzopen(fn.c_str(), "wb");
        if (!f[ch]) { LOG.error("ERROR: Failed to open " + fn); return false; }
    }
    const int64_t slots = garlic_gpu_window_slots(c.g, 1);
    const int blk = (int)std::max<int64_t>(1, std::min<int64_t>(N, (int64_t)(256 << 20) / (slots * 8)));
    std::vector<double> m((size_t)blk * slots);
    std::vector<int32_t> idx(blk);
    std::string line;
    // individuals in file order = rank order; each rank dumps the windows of its own shard (no exchange involved)
    for (Rank& R : c.team.ranks)
    for (int i0 = 0; i0 < R.hi - R.lo; i0 += blk) {
        const int n = std::min(blk, R.hi - R.lo - i0);
        for (int i = 0; i < n; ++i) idx[i] = i0 + i;
        if (garlic_gpu_windows(R.g, W, 1, c.o.weighted, idx.data(), n, 1, m.data())) {
            LOG.error(std::string("ERROR: windows: ") + garlic_gpu_last_error(R.g));
            return false;
        }
        for (int ch = 0; ch < C; ++ch) {
            const int64_t lo = c.chr_off[ch], hi = c.chr_off[ch + 1];
            for (int i = 0; i < n; ++i) {
                line.clear();
                for (int64_t s = lo; s < hi; ++s) {
                    const double v = m[(size_t)i * slots + s];
                    if (v == GARLIC_MISSING) line += "NA"; else line += fmt_g(v);
                    if (s < hi - 1) line += ' ';
                }
                line += '\n';
                gzwrite(f[ch], line.data(), (unsigned)line.size());
            }
        }
    }
    for (int ch = 0; ch < C; ++ch) {
        gzclose(f[ch]);
        fprintf(stderr, "Wrote %s.%s.%s.raw.lod.windows.gz\n", c.o.out.c_str(), c.tfam.pop.c_str(), c.labels[ch].c_str());
    }
    return true;
}

std::string join(const std::vector<double>& v) { std::string s; for (double x : v) s += " " + fmt_g(x); return s; }
std::string join(const std::vector<int>& v) { std::string s; for (int x : v) s += " " + std::to_string(x); return s; }

}  // namespace

int main(int argc, char** argv)
{
    Ctx c;
    Options& o = c.o;
    std::string cmdline;
    const int pr = parse_cli(argc, argv, o, cmdline);
    if (pr > 0) return 0;
    if (pr < 0) return -1;
    if (!LOG.open(o.out)) return -1;
    LOG.line(cmdline);
    LOG.hold = o.by_pop;                       // --by-pop: <out>.log lists the populations; these lines go to theirs
    LOG.line("Output file basename: " + o.out);

    // ---- validation and parameter log, in the reference's order (garlic-main.cpp:39-183) ----
    const bool bed = o.bfile != "none", vcf = o.vcf != "none";
    const bool call_filter = o.vcf_min_gq > 0 || o.vcf_min_dp > 0;
    if (vcf) {
        if (o.tped != "none" || bed) { LOG.error("ERROR: Provide exactly one input: --tped/--tfam, --bfile or --vcf."); return -1; }
        if (o.host_tokenize) { LOG.error("ERROR: --host-tokenize applies to tped input only, not to --vcf."); return -1; }
        LOG.line("VCF file: " + o.vcf);
        if (o.tfam != "none") LOG.line("TFAM file: " + o.tfam);
        if (o.vcf_min_gq > 0) LOG.line("Minimum genotype quality (GQ) of a call: " + std::to_string(o.vcf_min_gq));
        if (o.vcf_min_dp > 0) LOG.line("Minimum read depth (DP) of a call: " + std::to_string(o.vcf_min_dp));
    } else if (call_filter) {
        LOG.error("ERROR: --vcf-min-gq and --vcf-min-dp apply to --vcf input (VCF or BCF) only, not to --tped or --bfile.");
        return -1;
    } else if (bed) {
        if (o.tped != "none" || o.tfam != "none") { LOG.error("ERROR: Provide either --bfile or --tped and --tfam, not both."); return -1; }
        if (o.phased) { LOG.error("ERROR: --phased cannot be used with --bfile: a PLINK .bed stores unphased genotypes."); return -1; }
        LOG.line("PLINK binary fileset: " + o.bfile);
    } else {
        if (o.tped == "none" || o.tfam == "none") { LOG.error("ERROR: Must provide both a tped and tfam file."); return -1; }
        LOG.line("TPED file: " + o.tped);
        LOG.line(std::string("TPED missing data code: ") + o.tped_missing);
        LOG.line("TFAM file: " + o.tfam);
    }
    LOG.line("TGLS file: " + o.tgls);
    const bool use_gl = o.tgls != "none";
    if (use_gl && o.gl_type != "GQ" && o.gl_type != "GL" && o.gl_type != "PL") {
        LOG.error("ERROR: Must choose GQ/GL/PL for genotype likelihood format or provide a single error rate with --error.");
        return -1;
    }
    LOG.line("Genotype likelihood format: " + o.gl_type);
    if (o.cm && o.map == "none") { LOG.error("ERROR: Must provide mapfile if you wish to construct ROH in genetic map units."); return -1; }
    LOG.line("Measure ROH in genetic distance units: " + fmt_bool(o.cm));
    if (o.map == "none" && (o.weighted || o.cm)) { LOG.error("ERROR: Weighted LOD score method requires a map file."); return -1; }
    LOG.line("Weighted LOD: " + fmt_bool(o.weighted));
    if (o.weighted) LOG.line("Map file: " + o.map);
    if (o.build != "hg18" && o.build != "hg19" && o.build != "hg38" && o.build != "none") {
        LOG.error("ERROR: Must choose hg18/hg19/hg38 for build version or provide a custom centromere file.");
        return -1;
    }
    LOG.line("Genome build: " + o.build);
    if (o.build == "none" && o.centromere == "none") {
        LOG.error("ERROR: Must choose hg18/hg19/hg38 for build version or provide a custom centromere file.");
        return -1;
    }
    LOG.line("User defined centromere file: " + o.centromere);

    const bool auto_freq = (o.freq_file == "none");
    if (!auto_freq && o.freq_only) { LOG.error("ERROR: Specifying a frequency file and --freq-only is redundant."); return -1; }
    LOG.line("Calculate allele frequencies only: " + fmt_bool(o.freq_only));
    LOG.line("Calculate allele frequencies from data: " + fmt_bool(auto_freq));
    if (!auto_freq) LOG.line("Allele frequencies file: " + o.freq_file);
    else if (o.resample <= 0) LOG.line("Allele frequencies resampled: FALSE");
    else LOG.line("Allele frequencies resampled: " + std::to_string(o.resample));
    bool explore = false;
    if (o.winsize_multi[0] != -1) {
        for (int w : o.winsize_multi)
            if (w <= 0) { LOG.error("ERROR: SNP window sizes must be > 1."); return -1; }
        explore = true;
    }
    LOG.line("Explore window sizes: " + fmt_bool(explore));
    if (explore) LOG.line("User defined window sizes:" + join(o.winsize_multi));
    LOG.line("Automatic window size: " + fmt_bool(o.auto_winsize));
    if (o.auto_winsize_step <= 0) { LOG.error("ERROR: Automatic window step size must be > 0."); return -1; }
    LOG.line("Automatic window step size: " + std::to_string(o.auto_winsize_step));
    int winsize = o.winsize;
    if (winsize <= 1 && !explore && !(o.auto_winsize && o.weighted)) {
        LOG.error("ERROR: SNP window size must be > 1. If using --auto-winsize, this is the starting value.");
        return -1;
    }
    if (!explore && !o.auto_winsize) LOG.line("User defined window size: " + std::to_string(winsize));
    double cutoff = o.lod_cutoff;
    const bool auto_cutoff = (o.lod_cutoff == -999999);
    LOG.line("Choose LOD score cutoff automatically: " + fmt_bool(auto_cutoff));
    if (!auto_cutoff) LOG.line("User defined LOD score cutoff: " + fmt_g(cutoff));
    std::vector<double> bounds = o.size_bounds;
    bool auto_bounds = true;
    if (!(bounds.size() == 1 && bounds[0] == -1)) {
        for (size_t i = 0; i < bounds.size(); ++i)
            if (bounds[i] <= 0 || (i && bounds[i] <= bounds[i - 1])) {
                LOG.error("ERROR: ROH size boundaries must be positive and in increasing order.");
                return -1;
            }
        auto_bounds = false;
    }
    LOG.line("Choose ROH class thresholds automatically: " + fmt_bool(auto_bounds));
    if (!auto_bounds) LOG.line("User defined ROH class thresholds:" + join(bounds));
    if (o.threads <= 0) { LOG.error("ERROR: Number of threads must be > 0."); return -1; }
    LOG.line("Threads: " + std::to_string(o.threads));
    if ((o.error <= 0 || o.error >= 1) && !use_gl) {
        LOG.error("ERROR: Genotype error rate must be > 0 and < 1, or a TGLS file must be provided.");
        return -1;
    }
    LOG.line("Genotyping error: " + fmt_g(o.error));
    if (o.max_gap < 0) { LOG.error("ERROR: Max gap must be > 0."); return -1; }
    LOG.line("Max gap: " + std::to_string(o.max_gap));
    if (o.overlap_frac < 0 || o.overlap_frac > 1) { LOG.error("ERROR: Overlap fraction must be >= 0 and <= 1."); return -1; }
    if (o.auto_overlap) LOG.line("Overlap fraction: automatic");
    else if (o.overlap_frac != 0) LOG.line("Overlap fraction: " + fmt_g(o.overlap_frac));
    else LOG.line("Overlap fraction: 1/winsize");
    if (o.mu <= 0) { LOG.error("ERROR: Mutation rate must be > 0."); return -1; }
    LOG.line("mu: " + fmt_g(o.mu));
    if (o.M <= 0) { LOG.error("ERROR: Number of meioses must be > 0."); return -1; }
    LOG.line("M: " + std::to_string(o.M));
    if (o.nclust <= 0) { LOG.error("ERROR: Must choose positive number for number of GMM clusters."); return -1; }
    LOG.line("# GMM clusters: " + std::to_string(o.nclust));
    LOG.line(o.kde_subsample <= 0 ? std::string("# of rand individuals for KDE: ALL") : "# of rand individuals for KDE: " + std::to_string(o.kde_subsample));
    LOG.line(o.ld_subsample <= 0 ? std::string("# of rand individuals for LD: ALL") : "# of rand individuals for LD: " + std::to_string(o.ld_subsample));
    LOG.line("Output raw LOD scores: " + fmt_bool(o.raw_lod));
    LOG.line("Use r2 for weighting phased data: " + fmt_bool(o.phased));
    const bool thin = !o.no_kde_thinning;
    LOG.line("Use thinning for KDE estimation: " + fmt_bool(thin));
    c.rng.seed(o.seed >= 0 ? (o.seed == 0 ? 4357u : (unsigned)o.seed) : (unsigned)time(nullptr));

    // ---- inputs ----
    if (!load_centromeres(o.build, o.centromere, c.cen)) return -1;
    std::vector<std::string> a1, a2;                   // .bim allele names (--bfile)
    Vcf vc;                                            // VCF samples and allele names (--vcf)
    const unsigned call_keys = (o.vcf_min_gq > 0 ? 1u : 0u) | (o.vcf_min_dp > 0 ? 2u : 0u);
    if (vcf ? !load_vcf(o.vcf, c.tped, vc, call_keys)
            : bed ? !load_bim(o.bfile + ".bim", c.tped, a1, a2) : !load_tped(o.tped, o.tped_missing, c.tped, o.host_tokenize)) return 1;
    Tped& t = c.tped;
    LOG.line("Total loci: " + std::to_string(t.n_loci));
    if (vcf) {
        // the samples are the individuals; a --tfam must list the same IDs in the same order and names the population
        if (o.tfam == "none") { c.tfam.pop = "VCF"; c.tfam.ids = vc.samples; c.tfam.pops.assign(vc.samples.size(), "VCF"); }
        else {
            if (!load_tfam(o.tfam, c.tfam, o.by_pop)) return 1;
            for (size_t i = 0; i < std::max(c.tfam.ids.size(), vc.samples.size()); ++i)
                if (i >= c.tfam.ids.size() || i >= vc.samples.size() || c.tfam.ids[i] != vc.samples[i]) {
                    LOG.error("ERROR: " + o.tfam + " and " + o.vcf + " differ at individual " + std::to_string(i + 1) + ": " +
                              (i < c.tfam.ids.size() ? c.tfam.ids[i] : std::string("(none)")) + " in the tfam, " +
                              (i < vc.samples.size() ? vc.samples[i] : std::string("(none)")) + " in the VCF header.");
                    return 1;
                }
        }
    } else if (!load_tfam(bed ? o.bfile + ".fam" : o.tfam, c.tfam, o.by_pop)) return 1;
    if (bed) t.n_ind = (int)c.tfam.ids.size();
    else if ((int)c.tfam.ids.size() != t.n_ind) { LOG.error("ERROR: tfam and tped disagree on the number of individuals."); return 1; }
    FILE* bed_in = nullptr;
    if (bed) {                                          // the size check, once for the whole file
        if (!open_bed(o.bfile + ".bed", t.n_ind, t.n_loci, bed_in)) return 1;
        fclose(bed_in);
    }
    std::vector<double> gl;
    const bool oob = o.weighted || o.cm;

    // ---- populations: in order of first appearance, each the individuals (input columns) carrying its ID ----
    std::vector<std::string> pop_ids;
    std::vector<std::vector<int32_t>> pop_cols;
    if (!o.by_pop) { pop_ids.push_back(c.tfam.pop); pop_cols.emplace_back(); }
    else
        for (int i = 0; i < t.n_ind; ++i) {
            const std::string& p = c.tfam.pops[i];
            const size_t k = std::find(pop_ids.begin(), pop_ids.end(), p) - pop_ids.begin();
            if (k == pop_ids.size()) {
                if (p == "." || p == ".." || p.find('/') != std::string::npos) {
                    LOG.error("ERROR: Population ID " + p + " cannot be part of a file name (--by-pop writes <out>." + p + ".*).");
                    return 1;
                }
                pop_ids.push_back(p);
                pop_cols.emplace_back();
            }
            pop_cols[k].push_back(i);
        }
    const Tfam all = c.tfam;
    const std::string out_base = o.out;
    const int winsize0 = winsize;
    const double cutoff0 = cutoff;
    const std::vector<double> bounds0 = bounds;

    // one population (without --by-pop: the whole input, cols empty): what a separate run does from here on
    auto run_population = [&](const std::string& pop, const std::vector<int32_t>& cols, bool last_pop) -> int {
    const bool sel = !cols.empty();
    const int N = sel ? (int)cols.size() : t.n_ind;
    int winsize = winsize0;
    double cutoff = cutoff0;
    std::vector<double> bounds = bounds0;
    c.rng.seed(o.seed >= 0 ? (o.seed == 0 ? 4357u : (unsigned)o.seed) : (unsigned)time(nullptr));
    c.tfam.pop = pop;
    if (sel) { c.tfam.ids.clear(); for (int i : cols) c.tfam.ids.push_back(all.ids[i]); }
    c.labels.clear(); c.cen_arr.clear(); c.scaffold.clear();
    if (bed && !open_bed(o.bfile + ".bed", t.n_ind, t.n_loci, bed_in)) return 1;
    LOG.line("Population: " + c.tfam.pop);
    LOG.line("Total diploid individuals: " + std::to_string(N));
    // (K0-GL streams the file to the GPUs below; --host-tokenize reads it once, for every population)
    if (use_gl && o.host_tokenize && gl.empty() && !load_tgls(o.tgls, t, gl)) return 1;
    if (oob) {
        if (!load_map(o.map, c.scaffold)) return 1;
        if (c.scaffold.size() != t.chr_names.size()) {
            LOG.error("ERROR: Scaffold genetic map does not have the same number of chromosomes as data.");
            return -1;
        }
    }
    const int C = (int)t.chr_names.size();
    bool warned = false;
    for (int ch = 0; ch < C; ++ch) {
        c.labels.push_back(chr_label(t.chr_names[ch]));
        auto it = c.cen.find(c.labels.back());
        if (it == c.cen.end()) {   // centromere::centromereStart/End: 0/0 + warning (garlic-centromeres.cpp:33-59)
            LOG.error("WARNING: No centromere start information for chr: " + c.labels.back());
            if (!warned) LOG.error("WARNING: If you provided custom centromeres check that chromosome names match between data files.");
            warned = true;
            c.cen_arr.push_back(0); c.cen_arr.push_back(0);
        } else { c.cen_arr.push_back(it->second.first); c.cen_arr.push_back(it->second.second); }
    }

    // ---- GPU: coding, counts, freq, filter (K1-K3), individuals sharded over --gpus ranks ----
    const int G = o.by_pop ? std::min(o.gpus, N) : o.gpus;
    if (G < 1 || G > N) { LOG.error("ERROR: --gpus must be between 1 and the number of individuals."); return -1; }
    Team& team = c.team;
    team.start(G);
    uint8_t comm_id[128];
    if (G > 1 && garlic_gpu_comm_id(comm_id)) { LOG.error("ERROR: ncclGetUniqueId failed."); return 1; }
    const int per = (N + G - 1) / G;
    for (int r = 0; r < G; ++r) { team.ranks[r].rank = r; team.ranks[r].lo = std::min(N, r * per); team.ranks[r].hi = std::min(N, (r + 1) * per); }
    auto fail = [&](int code) { LOG.error("ERROR: " + team.first_error()); team.stop(); return code; };
    const int64_t blk = 1 << 12;                       // tped lines per upload (multiple of 32)
    const bool bcf = !vc.gt_type.empty();
    auto vcf_record = [&](int64_t s) {                 // names a VCF / BCF record: file, line or record, CHROM:POS
        const int ch = (int)(std::upper_bound(t.chr_off.begin(), t.chr_off.end(), s) - t.chr_off.begin()) - 1;
        return o.vcf + (bcf ? " record " : " line ") + std::to_string(vc.line[s]) + " (" + t.chr_names[ch] + ":" + std::to_string(t.pos[s]) + "): ";
    };
    // the checks of a record's GT diagnostics (first malformed sample, largest allele index) against its ALT count
    auto vcf_record_error = [&](int64_t s, int bad, int max_allele) -> std::string {
        if (bad >= 0)
            return vcf_record(s) + "the GT of sample " + vc.samples[bad] +
                   (bcf ? " is not two allele indices 0..254 (or missing), nor a lone missing value."
                        : " is not two allele indices 0..254 (or '.') separated by / or |, nor a lone '.'.") +
                   " Haploid calls (chrX in males, chrY, chrM) are not supported: restrict the input to the autosomes.";
        const int n_alt = (int)vc.alts[s].size();
        if (max_allele > n_alt) {
            std::string e = vcf_record(s) + "allele index " + std::to_string(max_allele) + " but only " + std::to_string(n_alt) + " ALT allele(s).";
            const int i = bcf ? bcf_sample_above(t, vc, s, n_alt) : -1;
            if (i >= 0) e += " First in sample " + vc.samples[i] + ".";
            return e;
        }
        return "";
    };
    // the message of record s's first malformed GQ / DP value, in sample bad (the rule the GPU applied, run here again)
    auto value_error = [&](int64_t s, int bad) -> std::string {
        const int32_t k_gq = vc.fmt_index[2 * s], k_dp = vc.fmt_index[2 * s + 1];
        int field = 0;
        std::string value;
        if (bcf) {
            const unsigned char* p = (const unsigned char*)vc.fv.data() + vc.fv_off[s];
            for (int f = 1; f >= 0; --f) {                  // GQ is named when both are malformed
                const int32_t at = vc.fv_pos[2 * s + f], type = vc.fv_type[2 * s + f] & 15, w = type == 1 ? 1 : type == 2 ? 2 : 4;
                if (at < 0) continue;
                const unsigned char* q = p + at + (int64_t)bad * w;
                const int32_t raw = w == 1 ? (int8_t)q[0] : w == 2 ? (int16_t)(q[0] | q[1] << 8) : (int32_t)(q[0] | q[1] << 8 | q[2] << 16 | (uint32_t)q[3] << 24);
                if (garlic::bcf_value(raw, type, f ? o.vcf_min_dp : o.vcf_min_gq) < 0) {
                    field = f;
                    char hex[16];
                    snprintf(hex, sizeof(hex), "0x%08x", (unsigned)raw);
                    value = hex;
                }
            }
            return vcf_record(s) + "the " + (field ? "DP" : "GQ") + " of sample " + vc.samples[bad] + " is float " + value +
                   ", an infinity or NaN that is not the missing value.";
        }
        const char* p = t.text.data() + t.text_off[s];
        const char* e = t.text.data() + t.text_off[s + 1];
        for (int i = 0; i < bad && p < e; ++i) { const char* tab = (const char*)memchr(p, '\t', e - p); p = tab ? tab + 1 : e; }
        garlic::call_filter(p, e - p, k_gq, o.vcf_min_gq, k_dp, o.vcf_min_dp, &field);
        const int k = field ? k_dp : k_gq;
        for (int i = 0; i < k && p < e; ++i) {
            while (p < e && *p != ':' && *p != '\t') ++p;
            if (p < e && *p == ':') ++p;
        }
        const char* ve = p;
        while (ve < e && *ve != ':' && *ve != '\t') ++ve;
        return vcf_record(s) + "the " + (field ? "DP" : "GQ") + " of sample " + vc.samples[bad] + " (" + std::string(p, ve) +
               ") is not a number: digits with an optional '-' and decimal part, or '.'.";
    };
    if (!team.all([&](Rank& R) {
            if (garlic_gpu_create(o.device + R.rank, &R.g)) { R.err = "no usable CUDA device " + std::to_string(o.device + R.rank) + "; garlic_b200 has no CPU path"; return false; }
            if (G > 1 && !rank_ok(R, garlic_gpu_comm_init(R.g, comm_id, R.rank, G), "comm_init")) return false;
            const int n = R.hi - R.lo;
            if (!rank_ok(R, garlic_gpu_set_shape(R.g, n, R.lo, t.n_loci, C, t.chr_off.data(), t.pos.data()), "set_shape")) return false;
            // --by-pop: every rank parses every input column and keeps its own individuals of the population
            if (sel && !rank_ok(R, garlic_gpu_select_columns(R.g, cols.data() + R.lo, t.n_ind), "select_columns")) return false;
            if (call_filter && !rank_ok(R, garlic_gpu_set_call_filter(R.g, o.vcf_min_gq, o.vcf_min_dp), "set_call_filter")) return false;
            std::vector<uint8_t> slice;
            std::vector<int32_t> nb;
            std::vector<int32_t> nc, mx, bc, bv;
            for (int64_t s0 = 0; s0 < t.n_loci && vcf; s0 += blk) {
                // the VCF sample columns (or the BCF GT vectors) go to every rank, which keeps its own individuals'
                // allele indices; every rank parses every sample, so each finds the same malformed records
                const int ns = (int)std::min(blk, t.n_loci - s0);
                nc.resize(ns); mx.resize(ns); bc.resize(ns); bv.assign(ns, -1);
                const int rc = call_filter
                    ? (bcf ? garlic_gpu_put_bcf_gt_filtered(R.g, (const uint8_t*)t.text.data(), t.text_off.data() + s0, vc.gt_type.data() + s0,
                                                            t.n_ind, s0, ns, vc.fv.data(), vc.fv_off.data() + s0, vc.fv_pos.data() + 2 * s0,
                                                            vc.fv_type.data() + 2 * s0, mx.data(), bc.data(), bv.data())
                           : garlic_gpu_put_vcf_text_filtered(R.g, t.text.data(), t.text_off.data() + s0, s0, ns, vc.fmt_index.data() + 2 * s0,
                                                              nc.data(), mx.data(), bc.data(), bv.data()))
                    : (bcf ? garlic_gpu_put_bcf_gt(R.g, (const uint8_t*)t.text.data(), t.text_off.data() + s0, vc.gt_type.data() + s0,
                                                   t.n_ind, s0, ns, mx.data(), bc.data())
                           : garlic_gpu_put_vcf_text(R.g, t.text.data(), t.text_off.data() + s0, s0, ns, nc.data(), mx.data(), bc.data()));
                if (!rank_ok(R, rc, bcf ? "put_bcf_gt" : "put_vcf_text")) return false;
                for (int k = 0; k < ns; ++k) {
                    if (!bcf && nc[k] != t.n_ind) {
                        R.err = vcf_record(s0 + k) + std::to_string(nc[k]) + " sample columns, but the #CHROM header names " + std::to_string(t.n_ind) + " samples.";
                        return false;
                    }
                    R.err = vcf_record_error(s0 + k, bc[k], mx[k]);
                    if (R.err.empty() && bv[k] >= 0) R.err = value_error(s0 + k, bv[k]);
                    if (!R.err.empty()) return false;
                }
            }
            for (int64_t s0 = 0; s0 < t.n_loci && !bed && !vcf && !o.host_tokenize; s0 += blk) {
                // K0: the raw genotype columns go to every rank, which keeps its own individuals' characters
                const int ns = (int)std::min(blk, t.n_loci - s0);
                nb.resize(ns);
                if (!rank_ok(R, garlic_gpu_put_tped_text(R.g, t.text.data(), t.text_off.data() + s0, s0, ns, o.tped_missing, nb.data()), "put_tped_text")) return false;
                for (int k = 0; k < ns; ++k)
                    if (nb[k] != 2 * t.n_ind) {      // loadTPEDData's column check (garlic-data.cpp:73-80), per line
                        R.err = "line " + std::to_string(s0 + k + 1) + " of " + o.tped + (nb[k] < 2 * t.n_ind ? " is truncated." : " has a different number of columns.");
                        return false;
                    }
            }
            for (int64_t s0 = 0; s0 < t.n_loci && !bed && o.host_tokenize; s0 += blk) {
                const int ns = (int)std::min(blk, t.n_loci - s0);
                const uint8_t* src_ = t.alleles.data() + (size_t)s0 * t.n_ind * 2;
                if (sel) {                                     // this rank's columns of the population
                    slice.resize((size_t)ns * n * 2);
                    for (int k = 0; k < ns; ++k)
                        for (int i = 0; i < n; ++i)
                            memcpy(slice.data() + ((size_t)k * n + i) * 2, src_ + ((size_t)k * t.n_ind + cols[R.lo + i]) * 2, 2);
                    src_ = slice.data();
                } else if (G > 1) {                            // this rank's columns of the block
                    slice.resize((size_t)ns * n * 2);
                    for (int k = 0; k < ns; ++k) memcpy(slice.data() + (size_t)k * n * 2, src_ + ((size_t)k * t.n_ind + R.lo) * 2, (size_t)n * 2);
                    src_ = slice.data();
                }
                if (!rank_ok(R, garlic_gpu_put_alleles(R.g, src_, s0, ns, o.tped_missing), "put_alleles")) return false;
            }
            if (!bed && !rank_ok(R, garlic_gpu_code_alleles(R.g), "code_alleles")) return false;     // MIN all-reduce of the first-allele keys
            if (use_gl && o.host_tokenize) {
                const int type = o.gl_type == "GQ" ? GARLIC_GL_GQ : o.gl_type == "GL" ? GARLIC_GL_GL : GARLIC_GL_PL;
                std::vector<double> rows;
                if (sel)
                    for (int i = R.lo; i < R.hi; ++i) rows.insert(rows.end(), gl.begin() + (size_t)cols[i] * t.n_loci, gl.begin() + (size_t)(cols[i] + 1) * t.n_loci);
                if (!rank_ok(R, garlic_gpu_put_gl(R.g, sel ? rows.data() : gl.data() + (size_t)R.lo * t.n_loci, type), "put_gl")) return false;
            }
            return true;
        })) return fail(1);
    if (bed) {
        // the .bed streams through two page-locked buffers of blk whole SNP rows: the next block is read while every rank
        // copies its own byte columns of the current one (garlic_gpu_put_bed); the whole file is never held
        const int64_t stride = (t.n_ind + 3) / 4;
        uint8_t* buf[2] = {(uint8_t*)garlic_gpu_host_alloc((size_t)(blk * stride)), (uint8_t*)garlic_gpu_host_alloc((size_t)(blk * stride))};
        auto rd = [&](int k, int64_t s0) {
            const int64_t ns = std::min(blk, t.n_loci - s0);
            return fread(buf[k], (size_t)stride, (size_t)ns, bed_in) == (size_t)ns;
        };
        bool have = buf[0] && buf[1] && rd(0, 0), put = true;
        for (int64_t s0 = 0; have && put && s0 < t.n_loci; s0 += blk) {
            const int k = (int)((s0 / blk) & 1), ns = (int)std::min(blk, t.n_loci - s0);
            bool next = true;
            std::thread reader;
            if (s0 + blk < t.n_loci) reader = std::thread([&, k, s0] { next = rd(k ^ 1, s0 + blk); });
            put = team.all([&](Rank& R) { return rank_ok(R, garlic_gpu_put_bed(R.g, buf[k], stride, s0, ns), "put_bed"); });
            if (reader.joinable()) reader.join();
            have = next;
        }
        fclose(bed_in);
        garlic_gpu_host_free(buf[0]);
        garlic_gpu_host_free(buf[1]);
        if (!put) return fail(1);
        if (!have) { LOG.error("ERROR: Failed to read " + o.bfile + ".bed"); team.stop(); return 1; }
        if (!team.all([&](Rank& R) { return rank_ok(R, garlic_gpu_code_alleles(R.g), "code_alleles"); })) return fail(1);
    }
    if (use_gl && !o.host_tokenize) {
        // K0-GL: the likelihood file goes to the GPUs as raw text, a block of lines at a time; every rank converts its
        // own individuals' columns (readTGLSData's parsing, garlic-data.cpp:1516-1554)
        const int type = o.gl_type == "GQ" ? GARLIC_GL_GQ : o.gl_type == "GL" ? GARLIC_GL_GL : GARLIC_GL_PL;
        TglsBlocks in;
        if (!in.open(o.tgls)) { team.stop(); return 1; }
        std::vector<char> text;
        std::vector<int64_t> off;
        std::vector<std::vector<int32_t>> ntok(G);
        for (int64_t s0 = 0; s0 < t.n_loci; s0 += blk) {
            const int ns = (int)std::min(blk, t.n_loci - s0);
            in.next(ns, text, off);
            if (text.empty()) text.push_back(' ');
            if (!team.all([&](Rank& R) {
                    ntok[R.rank].resize(ns);
                    return rank_ok(R, garlic_gpu_put_tgls_text(R.g, text.data(), off.data(), s0, ns, type, ntok[R.rank].data()), "put_tgls_text");
                })) return fail(1);
            for (int k = 0; k < ns; ++k)
                if (ntok[0][k] != t.n_ind) {                   // the reference counts the 4 leading fields as well (:1531)
                    LOG.error("ERROR: Incorrect number of columns in tgls file:  " + std::to_string(ntok[0][k] ? ntok[0][k] + 4 : 0) + ". Expected:  " + std::to_string(t.n_ind));
                    team.stop();
                    return 1;
                }
        }
    }
    c.g = team.ranks[0].g;
    if (call_filter) {
        uint64_t n_set = 0;
        for (Rank& R : team.ranks) n_set += garlic_gpu_calls_set_missing(R.g);
        int64_t lacking = 0;
        for (int64_t s = 0; s < t.n_loci; ++s)
            lacking += (o.vcf_min_gq > 0 && vc.fmt_index[2 * s] < 0) || (o.vcf_min_dp > 0 && vc.fmt_index[2 * s + 1] < 0);
        LOG.line("Calls set missing by the GQ/DP filter: " + std::to_string(n_set) + "; records whose FORMAT lacks " +
                 (o.vcf_min_gq > 0 && o.vcf_min_dp > 0 ? "GQ or DP" : o.vcf_min_gq > 0 ? "GQ" : "DP") + ": " + std::to_string(lacking));
    }
    if (last_pop) {                                    // the parsed input stays on the host until the last population
        std::vector<uint8_t>().swap(t.alleles);
        std::vector<char>().swap(t.text);
        std::vector<double>().swap(gl);
    }
    std::vector<int32_t> chr_param;
    if (oob)
        for (int ch = 0; ch < C; ++ch) {
            chr_param.push_back(c.scaffold[ch].pos.front()); chr_param.push_back(c.scaffold[ch].pos.back());
            chr_param.push_back(c.cen_arr[2 * ch]); chr_param.push_back(c.cen_arr[2 * ch + 1]);
        }
    std::vector<double> freq0(t.n_loci);
    std::vector<uint8_t> one(t.n_loci);
    const uint8_t no_one = vcf ? 255 : (uint8_t)o.tped_missing;     // get_one_allele's value for "no allele present"
    if (!gpu_ok(c, garlic_gpu_get_one_allele(c.g, one.data(), (char)no_one), "get_one_allele")) return 1;
    std::vector<std::string> one_name(t.n_loci);       // what .freq.gz prints and --freq-file is compared with
    for (int64_t s = 0; s < t.n_loci; ++s)
        one_name[s] = vcf ? (one[s] == 255 ? std::string("0") : one[s] == 0 ? vc.ref[s] : vc.alts[s][one[s] - 1])
                    : !bed ? std::string(1, (char)one[s]) : one[s] == 1 ? a1[s] : one[s] == 2 ? a2[s] : std::string("0");
    std::vector<double> panel;
    if (!auto_freq) {   // readFreqData (garlic-data.cpp:1345-1440): panel frequencies, flipped where the row names the other allele
        printf("Loading user provided allele frequencies from %s\n", o.freq_file.c_str());
        if (!load_freq_file(o.freq_file, t, one_name, bed || vcf, panel)) { team.stop(); return -1; }
    }
    if (!team.all([&](Rank& R) {                               // SUM all-reduce of the per-SNP counters inside
            int64_t L = 0;
            const bool ok = rank_ok(R, garlic_gpu_filter(R.g, oob, oob ? chr_param.data() : nullptr, auto_freq ? nullptr : panel.data(),
                                                         R.rank == 0 ? freq0.data() : nullptr, nullptr, &L), "filter");
            if (R.rank == 0) c.L = L;
            return ok;
        })) return fail(1);
    if (auto_freq && o.resample > 0) {
        // --resample n (garlic-data.cpp:140-148, 296-303): each frequency is replaced by a binomial draw count/n made of
        // n uniform deviates (gsl_rng_uniform = mt19937()/2^32, seeded from the clock in the reference; --seed here);
        // the filter, tables and everything downstream then use the resampled frequencies
        for (int64_t s = 0; s < t.n_loci; ++s) {
            // total != 0 (garlic-data.cpp:142) <=> some non-missing allele <=> the line has a "1" allele
            if (one[s] == no_one) continue;
            int count = 0;
            for (int i = 0; i < o.resample; ++i) count += (c.rng() / 4294967296.0) <= freq0[s];
            freq0[s] = double(count) / double(o.resample);
        }
        panel = freq0;
        if (!team.all([&](Rank& R) {
                int64_t L = 0;
                const bool ok = rank_ok(R, garlic_gpu_filter(R.g, oob, oob ? chr_param.data() : nullptr, panel.data(), nullptr, nullptr, &L), "filter");
                if (R.rank == 0) c.L = L;
                return ok;
            })) return fail(1);
    }
    if (auto_freq && !write_freq_gz(o.out + ".freq.gz", t, one_name, freq0)) { team.stop(); return 1; }
    auto shutdown = [&]() { team.all([](Rank& R) { garlic_gpu_destroy(R.g); R.g = nullptr; return true; }); team.stop(); };
    if (o.freq_only) { shutdown(); return 0; }   // freqOnly (garlic-data.cpp:238-315): the .freq.gz is the output
    std::vector<int32_t> src(c.L);
    if (!gpu_ok(c, garlic_gpu_get_kept_index(c.g, src.data()), "get_kept_index")) return fail(1);
    c.pos.resize(c.L);
    c.chr_off.assign(C + 1, 0);
    {
        int ch = 0;
        for (int64_t d = 0; d < c.L; ++d) {
            while (src[d] >= t.chr_off[ch + 1]) { ++ch; c.chr_off[ch] = d; }
            c.pos[d] = t.pos[src[d]];
        }
        for (++ch; ch <= C; ++ch) c.chr_off[ch] = c.L;
    }
    if (oob) {
        LOG.line("Monomorphic or out of bounds loci filtered: " + std::to_string(t.n_loci - c.L));
        c.gpos.resize(c.L);
        int n_interp = 0;
        for (int ch = 0; ch < C; ++ch)
            if (!interpolate_map(c.pos.data() + c.chr_off[ch], c.chr_off[ch + 1] - c.chr_off[ch], c.scaffold[ch], c.gpos.data() + c.chr_off[ch], n_interp)) {
                LOG.error("ERROR: Sites outside of map scaffold should have been filtered out.");
                return 1;
            }
        LOG.line("Number of genetic map locations interpolated: " + std::to_string(n_interp));
    } else LOG.line("Monomorphic loci filtered: " + std::to_string(t.n_loci - c.L));
    LOG.line("Total loci used for analysis: " + std::to_string(c.L));
    std::vector<double> lut;
    if (!use_gl && !o.device_lut) {
        // per-SNP LOD table with the HOST libm (lod(), garlic-roh.cpp:355-386, same operation order): the
        // reference's windows then come out bit-identical for whole-segment chains, which keeps the FIGTree
        // input of the cutoff selection the reference's own.  --device-lut builds it with K4 instead (≤ 1 ulp).
        lut.resize((size_t)c.L * 4);
        for (int64_t d = 0; d < c.L; ++d)
            for (int g = 0; g < 4; ++g) lut[(size_t)d * 4 + g] = lod_host(g, freq0[src[d]], o.error);
    }
    if (!team.all([&](Rank& R) {
            if (!rank_ok(R, garlic_gpu_set_tables(R.g, o.error, o.max_gap, c.cen_arr.data(), oob ? c.gpos.data() : nullptr), "set_tables")) return false;
            return lut.empty() || rank_ok(R, garlic_gpu_set_lut(R.g, lut.data()), "set_lut");
        })) return fail(1);
    double density = -1;
    if ((o.auto_winsize && o.weighted) || o.auto_overlap) density = calc_density(c);

    // ---- window size (garlic-main.cpp:295-336; garlic-roh.cpp:699-933) ----
    Kde selected;
    bool have_kde = false;
    if (explore || (o.auto_winsize && !o.weighted)) {
        std::vector<int32_t> sub;
        const std::vector<int32_t>* subp = nullptr;
        if (o.kde_subsample > 0 && o.kde_subsample < N) {   // subsetData, garlic-data.cpp:2171-2244
            sub = choose(c, o.kde_subsample, N);
            std::string s = "Individuals used for KDE: ";
            for (int i : sub) s += c.tfam.ids[i] + " ";
            LOG.line(s);
            subp = &sub;
        }
        auto kde_for = [&](int W, Kde& k) -> bool {
            if (o.weighted) {
                std::vector<int32_t> ld;
                if (o.ld_subsample > 0 && o.ld_subsample < N) ld = choose(c, o.ld_subsample, N);
                if (!ld_band_all(c, W, ld)) return false;
            }
            std::vector<double> data;
            if (!thinned_windows(c, W, thin ? W : 1, subp, data)) return false;
            if (data.size() < 2) { LOG.error("ERROR: no valid windows for window size " + std::to_string(W)); return false; }
            if (o.kde_gpu) return compute_kde_gpu(c, data.size(), k);
            compute_kde(data, k, o.kde_direct);
            return true;
        };
        if (explore && !(o.auto_winsize && !o.weighted)) {          // exploreWinsizes: KDE files only
            for (int W : o.winsize_multi) {
                Kde k;
                if (!kde_for(W, k)) return 1;
                if (!write_kde(k, o.out + "." + std::to_string(W) + "SNPs.kde")) return 1;
            }
            shutdown();
            return 0;
        }
        LOG.line("Searching for acceptable window size, smoothness threshold: 0.5");
        LOG.line("winsize\tsmoothness");
        if (explore) {                                               // selectWinsizeFromList
            for (size_t i = 0; i < o.winsize_multi.size(); ++i) {
                Kde k;
                const int W = o.winsize_multi[i];
                if (!kde_for(W, k)) return 1;
                const double mse = wiggle(k);
                LOG.line(" " + std::to_string(W) + "\t " + fmt_g(mse));   // LOG.log("",W,false) + LOG.log("\t",mse)
                if (mse <= 0.5 || i + 1 == o.winsize_multi.size()) { selected = k; winsize = W; have_kde = true; break; }
            }
        } else {                                                     // selectWinsize
            for (int W = winsize;; W += o.auto_winsize_step) {
                Kde k;
                if (!kde_for(W, k)) return 1;
                const double mse = wiggle(k);
                LOG.line(" " + std::to_string(W) + "\t " + fmt_g(mse));
                if (mse <= 0.5) { selected = k; winsize = W; have_kde = true; break; }
            }
        }
        if (!write_kde(selected, o.out + "." + std::to_string(winsize) + "SNPs.kde")) return 1;
        if (!explore) LOG.line("Selected window size: " + std::to_string(winsize));
    } else if (o.auto_winsize) {                                     // selectWinsizeWeighted, garlic-roh.cpp:3-9
        const int size = int(8.3235 * std::log(density) + 138.0521 + 0.5);
        winsize = size >= 10 ? size : 10;
        LOG.line("Selected window size: " + std::to_string(winsize));
    }
    printf("Window size: %d\n", winsize);
    double overlap = o.overlap_frac;
    if (o.auto_overlap) {                                            // selectOverlapFrac, garlic-data.cpp:3-8
        overlap = (6.375 * std::log(density) + 63.888) / 100.0;
        if (overlap > 1) overlap = 1.0;
        if (overlap <= 0) overlap = 1.0 / double(winsize);
        LOG.line("Selected overlap fraction: " + fmt_g(overlap));
    }

    // ---- LD band for wLOD (K6) ----
    if (o.weighted) {
        fprintf(stderr, "Calculating LD matrix.\n");
        std::vector<int32_t> ld;
        if (o.ld_subsample > 0 && o.ld_subsample < N) ld = choose(c, o.ld_subsample, N);
        if (!ld_band_all(c, winsize, ld)) return 1;
    }

    // ---- --raw-lod: every window of every individual (writeWinData, garlic-data.cpp:1704-1747) ----
    if (o.raw_lod && !write_raw_lod(c, winsize)) return -1;

    // ---- pass 1: thinned windows → KDE → cutoff (host, FIGTree) ----
    if (auto_cutoff) {
        if (!have_kde) {
            std::vector<int32_t> sub;
            const std::vector<int32_t>* subp = nullptr;
            if (o.kde_subsample > 0) {
                if (o.kde_subsample < N) sub = choose(c, o.kde_subsample, N);
                else { sub.resize(N); for (int i = 0; i < N; ++i) sub[i] = i; }
                std::string s = "Individuals used for KDE: ";
                for (int i : sub) s += c.tfam.ids[i] + " ";
                LOG.line(s);
                subp = &sub;
            }
            std::vector<double> data;
            if (!thinned_windows(c, winsize, thin ? winsize : 1, subp, data)) return 1;
            if (data.size() < 2) { LOG.error("ERROR: no valid windows to estimate the LOD score density."); return 1; }
            fprintf(stderr, "Estimating distribution of raw LOD score windows:\n");
            if (o.kde_gpu) { if (!compute_kde_gpu(c, data.size(), selected)) return 1; }
            else compute_kde(data, selected, o.kde_direct);
            if (!write_kde(selected, o.out + "." + std::to_string(winsize) + "SNPs.kde")) return -1;
        }
        cutoff = min_between_modes(selected, winsize);
        LOG.line("Selected LOD score cutoff: " + fmt_g(cutoff));
        printf("Selected LOD score cutoff (17 digits): %.17g\n", cutoff);
    } else printf("User defined LOD score cutoff: %s\n", fmt_g(cutoff).c_str());

    // ---- pass 2: windows → cutoff → coverage → ROH (fused K5) ----
    printf("Assembling ROH windows\n");
    if (!team.all([&](Rank& R) {
            R.rec.resize(1 << 16);
            for (;;) {
                if (!rank_ok(R, garlic_gpu_call_roh(R.g, winsize, cutoff, overlap, o.weighted, o.exact, R.rec.data(), (int64_t)R.rec.size(), &R.n_roh), "call_roh")) return false;
                if (R.n_roh <= (int64_t)R.rec.size()) return true;
                R.rec.resize(R.n_roh + 1024);
            }
        })) return fail(1);
    std::vector<Roh> roh;
    std::vector<double> lengths;
    for (const Rank& R : team.ranks)                                  // rank order = individual order
        for (int64_t r = 0; r < R.n_roh; ++r) {
            const int a = R.rec[r].start_idx, b = R.rec[r].stop_idx;
            Roh x;
            x.ind = R.lo + R.rec[r].ind; x.chr = R.rec[r].chr;
            x.start = c.pos[a]; x.stop = c.pos[b];
            x.length = o.cm ? c.gpos[b] - c.gpos[a] : double(c.pos[b] - c.pos[a] + 1);   // garlic-roh.cpp:478-484
            roh.push_back(x);
            lengths.push_back(x.length);
        }
    shutdown();

    // ---- size classes (host GMM) and output ----
    if (auto_bounds) {
        printf("Fitting %d-component GMM for size classification\n", o.nclust);
        if (!size_classes(lengths, o.nclust, bounds)) return 1;
        LOG.line("Selected ROH size boundaries = (" + join(bounds) + " )");
    } else LOG.line("User provided ROH size boundaries = (" + join(bounds) + " )");
    printf("Writing ROH tracts.\n");
    if (!write_bed(o.out + ".roh.bed", roh, c.tfam.ids, c.labels, bounds, c.tfam.pop, o.cm)) return 1;
    printf("Finished.\n");
    LOG.close();
    return 0;
    };

    if (!o.by_pop) return run_population(c.tfam.pop, {}, true);
    // --by-pop: the parameter and input lines a separate run writes before "Population:" go to each population's log
    LOG.hold = false;
    const std::vector<std::string> held = LOG.held;
    Log top = LOG;
    for (size_t k = 0; k < pop_ids.size(); ++k) {
        const std::string prefix = out_base + "." + pop_ids[k];
        top.line("Population " + pop_ids[k] + ": " + std::to_string(pop_cols[k].size()) + " individuals, output prefix " + prefix);
        LOG = Log();
        if (!LOG.open(prefix)) { top.close(); return -1; }
        LOG.line(cmdline);
        LOG.line("Output file basename: " + prefix);
        for (size_t i = 1; i < held.size(); ++i) LOG.line(held[i]);
        o.out = prefix;
        const int rc = run_population(pop_ids[k], pop_cols[k], k + 1 == pop_ids.size());
        const std::string msg = LOG.last;
        LOG.close();
        if (rc) {
            top.error("ERROR: population " + pop_ids[k] + ": " + (msg.empty() ? std::string("failed") : msg));
            top.close();
            return rc;
        }
    }
    top.close();
    return 0;
}
