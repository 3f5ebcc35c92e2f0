// capi.cu — extern "C" layer of libgarlic_b200.so (see include/garlic_b200.h).
// Host-side glue only: device memory, the segment table (closed form of the reference's window
// validity, SURVEY §3.4), kernel launches, stitching of chunk-boundary runs.  All arithmetic of the
// hot path happens in the kernels of kernels.cu / wlod.cu.
#include <cuda_runtime.h>
#include <nccl.h>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <unistd.h>
#include <string>
#include <vector>

#include "../../include/garlic_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "wlod.h"
#include "segments.h"
#include "bound.cuh"

using namespace garlic;

namespace {
constexpr int kPad = 4096 + 64;   // over-read slack (SNP entries) behind every per-SNP array / row
constexpr int kMaxW = 4096;
constexpr unsigned kBreakCap = 1u << 20, kBreakFirst = 4096;   // bad-pair list of set_tables: capacity, entries copied eagerly

}

struct garlic_gpu {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    int n_ind = 0, ind_offset = 0, n_chr = 0;
    int64_t L0 = 0, L = 0;
    std::vector<int64_t> chr_off0, chr_off;
    std::vector<int32_t> pos0, pos, src, cen;
    std::vector<double> gpos;
    std::vector<Stretch> stretches;   // gap/centromere-free SNP stretches (set_tables finds the breaks, the first consumer sorts them)
    bool stretches_pending = false;   // the break list is on its way to brk_pin; ev_tables marks its arrival
    uint8_t* brk_pin = nullptr;       // page-locked: count + the first breaks
    cudaEvent_t ev_tables = nullptr;
    bool have_geno0 = false, filtered = false, tables = false, have_gl = false, have_ld = false;
    int gl_type = GARLIC_GL_ERROR;
    double error = -1, mu = 1e-9;
    int max_gap = 200000, M = 7, ld_W = 0;
    double amax = 0;   // bound on |LOD table entry| of the table in use (ambiguity tolerance, see lod_bound())
    double fmin = 0.5; // smallest min(f, 1-f) a caller-supplied frequency vector held (freq_override)
    int* d_corr = nullptr;   // count_packed's correction vectors (2 x L0)
    int missing_char = '0';
    // device
    uint8_t* d_alleles = nullptr;
    unsigned long long* d_key = nullptr;
    uint8_t* d_bed = nullptr;         // put_bed staging: [L0][bed_stride] bytes, SNP-major, this rank's byte columns
    uint8_t* d_bed_rows = nullptr;    // put_bed: whole rows of one block as the caller passed them (handle spans every column)
    uint32_t* d_a1 = nullptr;         // per 32-SNP word: SNPs whose "1" allele is the .bim's A1
    int64_t bed_stride = 0;
    bool bed_input = false;           // the genotypes came from a .bed (no allele characters, no phase)
    bool vcf_input = false;           // d_alleles holds VCF allele index bytes (put_vcf_text), not tped characters
    uint64_t *d_geno0 = nullptr, *d_geno = nullptr;
    int64_t row_words0 = 0, row_words = 0;
    int* d_counts = nullptr;
    double *d_gl0 = nullptr, *d_gl = nullptr;
    int64_t gl_stride = 0;
    double *d_freq0 = nullptr, *d_freq = nullptr, *d_lut = nullptr, *d_gpos = nullptr;
    double *d_nomut = nullptr, *d_norec = nullptr, *d_wlut = nullptr, *d_invld = nullptr, *d_homf = nullptr;
    char* d_text = nullptr;           // K0 staging: raw tped line tails, their offsets, non-blank counts
    long long* d_textoff = nullptr;
    int* d_nonblank = nullptr;
    int2* d_hard = nullptr;           // K0-GL: tokens the device conversion leaves to strtod
    StitchScratch stitch_scratch;     // host buffers of call_roh kept between calls
    std::vector<RohRec> recs_buf, ambs_buf, merged_buf, tmp_buf;
    uint64_t* d_ldplanes = nullptr;   // LD scratch: bit-planes and the ordered pair matrix (kept between calls)
    double* d_ldpairs = nullptr;
    uint8_t* d_keep = nullptr;
    int *d_src = nullptr, *d_pos0 = nullptr, *d_chr_of0 = nullptr, *d_pos = nullptr, *d_chr_of = nullptr,
        *d_chr_start = nullptr, *d_chr_param = nullptr;
    RohRec *d_out = nullptr, *d_amb = nullptr, *d_sorted = nullptr;
    unsigned* d_hist = nullptr;       // run records per individual → bucket offsets
    unsigned* d_kept = nullptr;       // final runs per individual → offsets of the dense output
    size_t last_final = 0;            // final runs of the previous call_roh (size of the speculative first copy)
    // pass-2 items of the pruned pass, built (and uploaded) while the GPU is busy with pass 1 (windows_common)
    std::vector<Segment> p2_segs;
    std::vector<Item> p2_items;
    Item* d_items_p2 = nullptr;
    int p2_W = 0, p2_tile = 0, p2_chunk = 0, p2_slice = 0;
    uint64_t tables_gen = 0, p2_gen = 0;
    size_t sorted_cap = 0;
    unsigned out_cap = 0, amb_cap = 0;
    unsigned* d_cnt = nullptr;
    Item* d_items = nullptr;
    double* d_dump = nullptr;
    size_t items_cap = 0;
    int* d_indlist = nullptr;
    size_t indlist_cap = 0;
    double stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int64_t stats_items = 0;
    int* d_scan = nullptr;         // block counts of the keep scan, total, kept chromosome offsets
    int* d_breaks = nullptr;       // bad-pair list
    uint32_t* d_badbits = nullptr; // bit i: no window may hold SNPs i-1 and i (gap / centromere pair, chromosome start)
    int* d_thin = nullptr;         // segment + chromosome tables of the thinned pass 1
    // K3 is deferred to the first consumer of the compacted rows so that it can run fused with the pruning bound
    // (squeeze.cu): filter() only builds the plan.  The pruned pass 2 of window sizes from 32 on never needs them: its
    // bound reads the uncompacted rows and its walker compacts its candidates' slices (kernels.cu:walk_units_kernel)
    bool geno_pending = false;
    uint4 *d_plan_head = nullptr, *d_plan_seg = nullptr;
    int2* d_plan_rng = nullptr;
    uint4* d_bhw = nullptr;        // bound tables (bound.cuh) per half-word, valid for bound_tables_W
    uint16_t* d_plan_fast = nullptr;
    int* d_bflag = nullptr;        // != 0: the table in use breaks the bound's assumptions (every pair is a candidate)
    int bound_tables_W = 0;
    uint32_t* d_pmax = nullptr;    // [n_pieces][pmax_stride] piece maxima of every individual, valid for bound_W
    int64_t pmax_stride = 0;
    int n_pieces = 0, bound_W = 0;
    int* d_cand_list = nullptr;
    unsigned* d_cand_cnt = nullptr;
    int2* d_units = nullptr;       // work queue of the pruned pass 2: (item, first candidate)
    unsigned* d_nunits = nullptr;  // [0] units appended, [1] candidate pairs (inside the block of d_cnt: ensure_zero_block)
    size_t zero_cap = 0, zero_n = 0;
    cudaEvent_t ev_sq0 = nullptr, ev_sq1 = nullptr;   // around the last compaction and / or bound launch
    bool sq_timed = false;
    int item_pieces = 1;           // pieces per item of the pruned pass (GARLIC_ITEM_PIECES)
    bool prune = true;             // GARLIC_NO_PRUNE=1 disables the pruning pass
    bool precounted = false;       // d_counts already holds K2's counts of the rows put_packed copied
    bool phased = false;           // --phased: LD band from r2 between haplotypes instead of hr2
    bool wlod_mma = true;          // GARLIC_NO_MMA=1: weighted pass 2 with the exact kernel only
    ncclComm_t comm = nullptr;     // one rank per GPU, individuals sharded across ranks (DESIGN.md §7)
    int comm_rank = 0, comm_world = 1;
    // d_counts = [nalleles, total, hom, nonmiss] x L0.  Across ranks the first two rows (what freq and the filter need)
    // are summed as soon as the local counts exist; the other two (homFreq: only --weighted) when the LD band asks
    bool counts_reduced = false, counts_hi_reduced = false;
    bool counts_nccl_mem = false;      // d_counts came from ncclMemAlloc (symmetric-window capable)
    // NVLink exchange (xchg.cu): [flags | counters | freq0 | keep] of this rank in one IPC-exported block, peers' blocks mapped
    uint8_t* xslab = nullptr;
    void* xpeer[kXchgMaxRanks] = {nullptr};
    size_t x_off_counts = 0, x_off_freq = 0, x_off_keep = 0;
    bool xchg_tried = false, xchg_ok = false;
    unsigned xchg_seq = 0;
    ncclWindow_t counts_win = nullptr; // d_counts registered with the communicator as a symmetric window
    bool counts_win_tried = false;
    double* d_gather = nullptr;    // all-gathered thinned windows
    const double* kde_src = nullptr;   // the window matrix the last pass-1 call left on the device (garlic_gpu_kde)
    int64_t kde_src_n = 0;
    double *d_kde = nullptr, *d_kde_in = nullptr;   // scratch of the device KDE; uploaded host values
    cudaEvent_t ev2 = nullptr;
    cudaStream_t copy_stream = nullptr;   // device-to-host copies that overlap the kernels behind them (filter)
    cudaStream_t aux_stream = nullptr;    // thinned pass 1 beside the compaction (windows_common)
    cudaEvent_t ev_aux_in = nullptr, ev_aux_out = nullptr;
    cudaEvent_t ev_copy = nullptr;
    // GARLIC_TIMELINE=1: host clock and stream position (CUDA events) at marked points of the entry points, printed at destroy
    bool tl_on = false;
    std::vector<cudaEvent_t> tl_ev;
    std::vector<const char*> tl_name;
    std::vector<double> tl_host;
    bool out_pending = false;      // filter's freq / keep copies into page-locked caller buffers are still in flight
    uint8_t* pin = nullptr;        // pinned host staging buffer
    size_t pin_cap = 0;
    std::map<void*, size_t> cap;   // bytes behind each device pointer slot (keyed by the slot's address)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

// GARLIC_TIMING=1: wall-clock laps of the host-side phases of an entry point, to stderr
struct Laps {
    bool on;
    int rank = 0;
    const char* name;
    std::chrono::steady_clock::time_point t0;
    std::string out;
    explicit Laps(const char* n) : on(getenv("GARLIC_TIMING") != nullptr), name(n), t0(std::chrono::steady_clock::now()) {}
    void lap(const char* what)
    {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        char b[96];
        snprintf(b, sizeof b, " %s=%.3f", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        out += b;
        t0 = t1;
    }
    ~Laps() { if (on) fprintf(stderr, "[garlic_b200 r%d] %s:%s ms\n", rank, name, out.c_str()); }
};

static void tl_mark(garlic_gpu* h, const char* name)
{
    if (!h->tl_on) return;
    if (h->tl_ev.size() >= 4096) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, h->stream);
    h->tl_ev.push_back(e);
    h->tl_name.push_back(name);
    h->tl_host.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count());
}
static void tl_dump(garlic_gpu* h)
{
    if (!h->tl_on || h->tl_ev.empty()) return;
    cudaStreamSynchronize(h->stream);
    const size_t n = h->tl_ev.size(), first = n > 120 ? n - 120 : 0;
    for (size_t i = first; i < n; ++i) {
        float g = 0;
        cudaEventElapsedTime(&g, h->tl_ev[first], h->tl_ev[i]);
        fprintf(stderr, "[timeline r%d] %-28s host %9.3f  stream %9.3f ms\n", h->comm_rank, h->tl_name[i], h->tl_host[i] - h->tl_host[first], g);
    }
    for (cudaEvent_t e : h->tl_ev) cudaEventDestroy(e);
    h->tl_ev.clear();
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)
#define LAUNCH(call) do { CK(call); h->launches++; } while (0)
#define FAIL(msg) do { h->err = (msg); return 1; } while (0)

// (re)allocate a device array; an existing allocation that is large enough is kept (repeated runs
// of the path on the same shape — window-size scans, benchmark steps — then allocate nothing)
template <typename T>
static int dev_alloc(garlic_gpu* h, T** p, size_t n)
{
    if (n == 0) n = 1;
    const size_t bytes = n * sizeof(T);
    auto it = h->cap.find((void*)p);
    if (*p && it != h->cap.end() && it->second >= bytes) return 0;
    if (*p) { cudaFree(*p); *p = nullptr; }
    CK(cudaMalloc((void**)p, bytes));
    h->cap[(void*)p] = bytes;
    return 0;
}
template <typename T>
static void dev_free(T*& p) { if (p) cudaFree(p); p = nullptr; }

static int pin_alloc(garlic_gpu* h, size_t bytes)
{
    if (h->pin && h->pin_cap >= bytes) return 0;
    if (h->pin) { cudaFreeHost(h->pin); h->pin = nullptr; h->pin_cap = 0; }
    CK(cudaMallocHost((void**)&h->pin, bytes));
    h->pin_cap = bytes;
    return 0;
}

// Bound on |lod()| for the table in use (garlic-roh.cpp:355-386).  With e in [1e-16, 1] (readTGLSData's clamp, or the
// global --error) and f in (0,1):  lod(het) = log10(e) >= log10(e_min);  lod(hom) = log10((1-e)/(1-f) + e) lies in
// [0, -log10(min(f,1-f))].  Frequencies made from counts are multiples of 1/(2 N_total); caller-supplied ones
// (--freq-file) are scanned in garlic_gpu_filter.  One decade of slack on top.
static double lod_bound(const garlic_gpu* h)
{
    const double n_total = 2.0 * ((double)h->n_ind + 1.0) * (double)std::max(1, h->comm_world);
    double fmin = 1.0 / n_total;
    if (h->fmin > 0 && h->fmin < fmin) fmin = h->fmin;
    const double emin = h->have_gl ? 1e-16 : ((h->error > 0 && h->error < 1) ? h->error : 1e-16);
    return std::max(-std::log10(emin), -std::log10(fmin)) + 1.0;
}

#define NCK(call)                                                                             \
    do {                                                                                      \
        ncclResult_t r_ = (call);                                                             \
        if (r_ != ncclSuccess) {                                                              \
            h->err = std::string(#call) + ": " + ncclGetErrorString(r_);                      \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

// the path's one data collective (SURVEY §8e), stream-ordered on the library's stream: every rank calls it at the same
// points of the call sequence (count_packed / filter; ld_band / get_hom_freq for the second half)
static int reduce_counts(garlic_gpu* h, bool hi)
{
    if (!h->comm) return 0;
    // GARLIC_NCCL_WINDOW=1: the counters live in memory from ncclMemAlloc and are registered with the communicator as a
    // symmetric window (same buffer, same offset on every rank) so that NCCL may run its symmetric kernels for this
    // all-reduce.  Measured on 8 B200 (profiles/r02i): no gain at 4.8 MB (1.28 ms per step against 1.24 without), hence
    // opt-in.  Registration is a collective, done once per shape; if it is refused the all-reduce runs unregistered.
    if (!h->counts_win_tried && h->counts_nccl_mem) {
        h->counts_win_tried = true;
        if (getenv("GARLIC_NCCL_WINDOW") != nullptr) {
            if (ncclCommWindowRegister(h->comm, h->d_counts, (size_t)4 * h->L0 * sizeof(int), &h->counts_win, NCCL_WIN_COLL_SYMMETRIC) != ncclSuccess)
                h->counts_win = nullptr;
        }
    }
    if (!h->counts_reduced) {
        NCK(ncclAllReduce(h->d_counts, h->d_counts, (size_t)2 * h->L0, ncclInt32, ncclSum, h->comm, h->stream));
        h->counts_reduced = true;
    }
    if (hi && !h->counts_hi_reduced) {
        NCK(ncclAllReduce(h->d_counts + 2 * h->L0, h->d_counts + 2 * h->L0, (size_t)2 * h->L0, ncclInt32, ncclSum, h->comm, h->stream));
        h->counts_hi_reduced = true;
    }
    return 0;
}

static void free_counts(garlic_gpu* h)
{
    if (!h->d_counts) return;
    if (h->xchg_ok) return;                            // inside the exchange block: xchg_teardown owns it
    if (h->counts_win && h->comm) ncclCommWindowDeregister(h->comm, h->counts_win);
    h->counts_win = nullptr; h->counts_win_tried = false;
    if (h->counts_nccl_mem) ncclMemFree(h->d_counts); else cudaFree(h->d_counts);
    h->d_counts = nullptr; h->counts_nccl_mem = false;
    h->cap.erase((void*)&h->d_counts);
}

// the per-SNP counters [4][L0]: from NCCL's allocator so that they can become a symmetric window (reduce_counts)
static int alloc_counts(garlic_gpu* h, size_t n)
{
    const size_t bytes = n * sizeof(int);
    auto it = h->cap.find((void*)&h->d_counts);
    if (h->d_counts && it != h->cap.end() && it->second == bytes) return 0;   // (a window is registered with its exact size)
    free_counts(h);
    void* p = nullptr;
    if (getenv("GARLIC_NCCL_WINDOW") != nullptr && ncclMemAlloc(&p, bytes) == ncclSuccess && p) {
        h->d_counts = static_cast<int*>(p);
        h->counts_nccl_mem = true;
    } else {
        cudaGetLastError();
        CK(cudaMalloc((void**)&h->d_counts, bytes));
    }
    h->cap[(void*)&h->d_counts] = bytes;
    return 0;
}

// ---- NVLink exchange of the counters (xchg.cu) ----------------------------------------------------------------
static void xchg_teardown(garlic_gpu* h)
{
    if (!h->xslab) { h->xchg_tried = false; h->xchg_ok = false; return; }
    cudaStreamSynchronize(h->stream);
    for (int p = 0; p < kXchgMaxRanks; ++p) {
        if (h->xpeer[p] && h->xpeer[p] != (void*)h->xslab) cudaIpcCloseMemHandle(h->xpeer[p]);
        h->xpeer[p] = nullptr;
    }
    if (h->xchg_ok) {                                  // the three tables lived inside the block
        h->d_counts = nullptr; h->d_freq0 = nullptr; h->d_keep = nullptr;
        h->cap.erase((void*)&h->d_counts); h->cap.erase((void*)&h->d_freq0); h->cap.erase((void*)&h->d_keep);
    }
    cudaFree(h->xslab);
    h->xslab = nullptr;
    h->xchg_tried = false; h->xchg_ok = false; h->xchg_seq = 0;
}

// One-time, collective (every rank of the communicator calls it at the same point): allocate this rank's block, exchange
// the IPC handles over the communicator, map the peers' blocks, agree that every rank succeeded, and move the counters /
// freq / keep tables into the block.  Any failure (one process driving several GPUs, IPC not permitted, more than 16
// ranks) leaves the NCCL all-reduce in place on every rank.
static int ensure_xchg(garlic_gpu* h)
{
    if (h->xchg_tried) return 0;
    h->xchg_tried = true;
    h->xchg_ok = false;
    if (!h->comm || h->comm_world < 2 || h->comm_world > kXchgMaxRanks || h->counts_nccl_mem) return 0;
    if (getenv("GARLIC_NO_XCHG") != nullptr) return 0;
    const int N = h->comm_world;
    const size_t L0 = (size_t)h->L0;
    h->x_off_counts = 256;
    h->x_off_freq = (h->x_off_counts + 16 * L0 + 255) & ~(size_t)255;
    h->x_off_keep = h->x_off_freq + 8 * L0;
    const size_t total = ((h->x_off_keep + L0 + 255) & ~(size_t)255);
    struct Rec { cudaIpcMemHandle_t hdl; int pid; int ok; long long L0; char pad[128 - sizeof(cudaIpcMemHandle_t) - 16]; };
    static_assert(sizeof(Rec) == 128, "exchange record is 128 bytes");
    Rec mine;
    memset(&mine, 0, sizeof(mine));
    mine.pid = (int)getpid(); mine.L0 = h->L0; mine.ok = 1;
    if (cudaMalloc((void**)&h->xslab, total) != cudaSuccess) { cudaGetLastError(); h->xslab = nullptr; mine.ok = 0; }
    if (mine.ok) {
        cudaMemsetAsync(h->xslab, 0, 256, h->stream);
        cudaStreamSynchronize(h->stream);
        if (cudaIpcGetMemHandle(&mine.hdl, h->xslab) != cudaSuccess) { cudaGetLastError(); mine.ok = 0; }
    }
    // the records travel over the communicator (the only channel the library has)
    Rec* d_rec = nullptr;
    std::vector<Rec> all(N);
    CK(cudaMalloc((void**)&d_rec, (size_t)(N + 1) * sizeof(Rec)));
    CK(cudaMemcpyAsync(d_rec + N, &mine, sizeof(Rec), cudaMemcpyHostToDevice, h->stream));
    NCK(ncclAllGather(d_rec + N, d_rec, sizeof(Rec), ncclUint8, h->comm, h->stream));
    CK(cudaMemcpyAsync(all.data(), d_rec, (size_t)N * sizeof(Rec), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int ok = 1;
    for (int p = 0; p < N; ++p) {
        if (!all[p].ok || all[p].L0 != h->L0) ok = 0;
        if (p != h->comm_rank && all[p].pid == mine.pid) ok = 0;   // several GPUs driven by one process: no IPC mapping of one's own memory
    }
    for (int p = 0; p < N && ok; ++p) {
        if (p == h->comm_rank) { h->xpeer[p] = h->xslab; continue; }
        void* ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, all[p].hdl, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
        h->xpeer[p] = ptr;
    }
    // agreement: every rank mapped every peer, or nobody uses the path
    int* d_ok = reinterpret_cast<int*>(d_rec);
    CK(cudaMemcpyAsync(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice, h->stream));
    NCK(ncclAllReduce(d_ok, d_ok, 1, ncclInt32, ncclMin, h->comm, h->stream));
    CK(cudaMemcpyAsync(&ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(d_rec);
    if (!ok) {
        for (int p = 0; p < N; ++p) {
            if (h->xpeer[p] && h->xpeer[p] != (void*)h->xslab) cudaIpcCloseMemHandle(h->xpeer[p]);
            h->xpeer[p] = nullptr;
        }
        if (h->xslab) cudaFree(h->xslab);
        h->xslab = nullptr;
        return 0;
    }
    // the tables move into the block (the counters with what the count kernel has already put there)
    int* nc = reinterpret_cast<int*>(h->xslab + h->x_off_counts);
    if (h->d_counts) CK(cudaMemcpyAsync(nc, h->d_counts, 16 * L0, cudaMemcpyDeviceToDevice, h->stream));
    else CK(cudaMemsetAsync(nc, 0, 16 * L0, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    free_counts(h);
    if (h->d_freq0) { cudaFree(h->d_freq0); h->d_freq0 = nullptr; }
    if (h->d_keep) { cudaFree(h->d_keep); h->d_keep = nullptr; }
    h->d_counts = nc;
    h->d_freq0 = reinterpret_cast<double*>(h->xslab + h->x_off_freq);
    h->d_keep = h->xslab + h->x_off_keep;
    h->cap[(void*)&h->d_counts] = 16 * L0;
    h->cap[(void*)&h->d_freq0] = 8 * L0;
    h->cap[(void*)&h->d_keep] = L0;
    h->xchg_ok = true;
    h->xchg_seq = 0;
    return 0;
}

// filter() does not wait for its copies into page-locked caller buffers; every later call that hands data to the host
// (windows, call_roh, kde, the get_* accessors) and garlic_gpu_sync complete them first
static int finish_outputs(garlic_gpu* h)
{
    if (!h->out_pending) return 0;
    CK(cudaStreamSynchronize(h->copy_stream));
    h->out_pending = false;
    return 0;
}

static bool is_pinned(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// host copy of the gather list (kept SNP → pre-filter index), fetched from the device on first use
static int fetch_src(garlic_gpu* h)
{
    if ((int64_t)h->src.size() == h->L) return 0;
    h->src.resize(h->L);
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(h->src.data(), h->d_src, h->L * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

static int ensure_geno(garlic_gpu* h, int W_hint);   // runs the deferred compaction (K3), fused with the bound when it can be

extern "C" {

int garlic_gpu_create(int device, garlic_gpu_t** out)
{
    if (!out) return 1;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= device || device < 0) {
        fprintf(stderr, "garlic_b200: no usable CUDA device %d (found %d) — there is no CPU fallback\n", device, n);
        return 2;
    }
    garlic_gpu* h = new garlic_gpu;
    h->device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete h;
        return 3;
    }
    cudaEventCreate(&h->ev0);
    cudaEventCreate(&h->ev1);
    cudaEventCreate(&h->ev2);
    cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_tables, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&h->ev_aux_in, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_aux_out, cudaEventDisableTiming);
    h->prune = getenv("GARLIC_NO_PRUNE") == nullptr;
    h->tl_on = getenv("GARLIC_TIMELINE") != nullptr;
    cudaEventCreate(&h->ev_sq0);
    cudaEventCreate(&h->ev_sq1);
    if (const char* e = getenv("GARLIC_ITEM_PIECES")) { const int m = atoi(e); if (m >= 1 && m <= 16) h->item_pieces = m; }
    h->wlod_mma = getenv("GARLIC_NO_MMA") == nullptr;
    cudaMalloc((void**)&h->d_cnt, 8 * sizeof(unsigned));
    h->zero_cap = 8;
    *out = h;
    return 0;
}

void garlic_gpu_destroy(garlic_gpu_t* h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    tl_dump(h);
    xchg_teardown(h);
    dev_free(h->d_alleles); dev_free(h->d_key); dev_free(h->d_bed); dev_free(h->d_bed_rows); dev_free(h->d_a1); dev_free(h->d_geno0); dev_free(h->d_geno);
    free_counts(h);
    dev_free(h->d_gl0); dev_free(h->d_gl); dev_free(h->d_freq0); dev_free(h->d_freq); dev_free(h->d_lut);
    dev_free(h->d_ldplanes); dev_free(h->d_ldpairs); dev_free(h->d_text); dev_free(h->d_textoff); dev_free(h->d_nonblank);
    dev_free(h->d_gpos); dev_free(h->d_nomut); dev_free(h->d_norec); dev_free(h->d_wlut); dev_free(h->d_invld);
    dev_free(h->d_homf); dev_free(h->d_keep); dev_free(h->d_src); dev_free(h->d_pos0); dev_free(h->d_chr_of0);
    dev_free(h->d_pos); dev_free(h->d_chr_of); dev_free(h->d_chr_start); dev_free(h->d_chr_param);
    dev_free(h->d_out); dev_free(h->d_amb); dev_free(h->d_sorted); dev_free(h->d_items_p2); dev_free(h->d_cnt); dev_free(h->d_items); dev_free(h->d_indlist); dev_free(h->d_dump);
    dev_free(h->d_scan); dev_free(h->d_breaks); dev_free(h->d_thin); dev_free(h->d_badbits);
    if (h->pin) cudaFreeHost(h->pin);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->ev_copy) cudaEventDestroy(h->ev_copy);
    if (h->ev_tables) cudaEventDestroy(h->ev_tables);
    if (h->brk_pin) cudaFreeHost(h->brk_pin);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->aux_stream) { cudaStreamSynchronize(h->aux_stream); cudaStreamDestroy(h->aux_stream); }
    if (h->ev_aux_in) cudaEventDestroy(h->ev_aux_in);
    if (h->ev_aux_out) cudaEventDestroy(h->ev_aux_out);
    dev_free(h->d_plan_head); dev_free(h->d_plan_seg); dev_free(h->d_plan_rng); dev_free(h->d_bhw); dev_free(h->d_plan_fast); dev_free(h->d_bflag);
    dev_free(h->d_pmax); dev_free(h->d_cand_list); dev_free(h->d_cand_cnt); dev_free(h->d_units);
    if (h->ev_sq0) cudaEventDestroy(h->ev_sq0);
    if (h->ev_sq1) cudaEventDestroy(h->ev_sq1);
    if (h->comm) ncclCommDestroy(h->comm);
    dev_free(h->d_gather); dev_free(h->d_corr); dev_free(h->d_kde); dev_free(h->d_kde_in); dev_free(h->d_hard);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

const char* garlic_gpu_last_error(const garlic_gpu_t* h) { return h ? h->err.c_str() : "null handle"; }
uint64_t garlic_gpu_launch_count(const garlic_gpu_t* h) { return h ? h->launches : 0; }
void* garlic_gpu_stream(const garlic_gpu_t* h) { return h ? (void*)h->stream : nullptr; }
void* garlic_gpu_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void garlic_gpu_host_free(void* p) { if (p) cudaFreeHost(p); }

int garlic_gpu_comm_id(uint8_t* id128)
{
    ncclUniqueId id;
    if (ncclGetUniqueId(&id) != ncclSuccess) return 1;
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return 0;
}

int garlic_gpu_comm_init(garlic_gpu_t* h, const uint8_t* id128, int rank, int world)
{
    CK(cudaSetDevice(h->device));
    if (world < 1 || rank < 0 || rank >= world) FAIL("comm_init: bad rank / world size");
    xchg_teardown(h);
    if (h->comm) {
        if (h->counts_win) ncclCommWindowDeregister(h->comm, h->counts_win);
        ncclCommDestroy(h->comm); h->comm = nullptr;
    }
    h->counts_win = nullptr; h->counts_win_tried = false;
    h->comm_rank = rank; h->comm_world = world;
    if (world == 1) return 0;
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    NCK(ncclCommInitRank(&h->comm, world, id, rank));
    return 0;
}

int garlic_gpu_sync(garlic_gpu_t* h)
{
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return finish_outputs(h);
}

int garlic_gpu_set_shape(garlic_gpu_t* h, int n_ind, int ind_offset, int64_t n_loci, int n_chr,
                         const int64_t* chr_offsets, const int32_t* pos)
{
    if (!h) return 1;
    CK(cudaSetDevice(h->device));
    if (n_ind < 1 || n_loci < 1 || n_chr < 1) FAIL("set_shape: number of individuals, loci and chromosomes must be positive");
    if (n_loci > 0x7ffffff0ll - kPad) FAIL("set_shape: too many loci");
    if (chr_offsets[0] != 0 || chr_offsets[n_chr] != n_loci) FAIL("set_shape: chr_offsets must span [0, n_loci]");
    h->n_ind = n_ind; h->ind_offset = ind_offset; h->L0 = n_loci; h->n_chr = n_chr;
    h->chr_off0.assign(chr_offsets, chr_offsets + n_chr + 1);
    h->pos0.assign(pos, pos + n_loci);
    h->row_words0 = (((n_loci + kPad + 31) >> 5) + 3) & ~(int64_t)1;
    if (dev_alloc(h, &h->d_geno0, (size_t)n_ind * h->row_words0)) return 1;
    CK(cudaMemsetAsync(h->d_geno0, 0xff, (size_t)n_ind * h->row_words0 * 8, h->stream));
    if (h->xslab && (h->cap.find((void*)&h->d_counts) == h->cap.end() || h->cap[(void*)&h->d_counts] != (size_t)16 * n_loci)) xchg_teardown(h);
    if (alloc_counts(h, (size_t)4 * n_loci)) return 1;
    CK(cudaMemsetAsync(h->d_counts, 0, (size_t)4 * n_loci * sizeof(int), h->stream));
    if (dev_alloc(h, &h->d_pos0, (size_t)n_loci)) return 1;
    CK(cudaMemcpyAsync(h->d_pos0, pos, n_loci * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    std::vector<int> chr_of(n_loci);
    for (int c = 0; c < n_chr; ++c)
        for (int64_t s = chr_offsets[c]; s < chr_offsets[c + 1]; ++s) chr_of[s] = c;
    if (dev_alloc(h, &h->d_chr_of0, (size_t)n_loci)) return 1;
    CK(cudaMemcpyAsync(h->d_chr_of0, chr_of.data(), n_loci * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->have_geno0 = false; h->filtered = false; h->tables = false; h->have_gl = false; h->have_ld = false;
    dev_free(h->d_alleles); dev_free(h->d_key); dev_free(h->d_bed);
    h->bed_input = false; h->vcf_input = false;
    return 0;
}

int garlic_gpu_put_alleles(garlic_gpu_t* h, const uint8_t* alleles, int64_t snp0, int n_snp, char missing)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_alleles: call set_shape first");
    if (snp0 % 32 != 0 || snp0 < 0 || snp0 + n_snp > h->L0) FAIL("put_alleles: bad SNP range (snp0 must be a multiple of 32)");
    if (h->bed_input) FAIL("put_alleles: this handle holds .bed input");
    if (h->vcf_input) FAIL("put_alleles: this handle holds VCF input");
    if (!h->d_alleles) {
        if (dev_alloc(h, &h->d_alleles, (size_t)h->L0 * h->n_ind * 2)) return 1;
        if (dev_alloc(h, &h->d_key, (size_t)h->L0)) return 1;
    }
    uint8_t* dst = h->d_alleles + (size_t)snp0 * h->n_ind * 2;
    CK(cudaMemcpyAsync(dst, alleles, (size_t)n_snp * h->n_ind * 2, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ev_copy, h->stream));
    LAUNCH(launch_first_allele(dst, n_snp, h->n_ind, h->ind_offset, (unsigned char)missing, h->d_key + snp0, h->stream));
    h->missing_char = (unsigned char)missing;
    CK(cudaEventSynchronize(h->ev_copy));   // the copy has left the caller's buffer (it may be page-locked and reused)
    return 0;
}

int garlic_gpu_put_tped_text(garlic_gpu_t* h, const char* text, const int64_t* line_off, int64_t snp0, int n_snp,
                             char missing, int32_t* nonblank)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_tped_text: call set_shape first");
    if (snp0 % 32 != 0 || snp0 < 0 || snp0 + n_snp > h->L0) FAIL("put_tped_text: bad SNP range (snp0 must be a multiple of 32)");
    if (n_snp <= 0) return 0;
    if (h->bed_input) FAIL("put_tped_text: this handle holds .bed input");
    if (h->vcf_input) FAIL("put_tped_text: this handle holds VCF input");
    if (!h->d_alleles) {
        if (dev_alloc(h, &h->d_alleles, (size_t)h->L0 * h->n_ind * 2)) return 1;
        if (dev_alloc(h, &h->d_key, (size_t)h->L0)) return 1;
    }
    const int64_t bytes = line_off[n_snp] - line_off[0];
    if (bytes < 0) FAIL("put_tped_text: line offsets must ascend");
    if (dev_alloc(h, &h->d_text, (size_t)bytes + 16)) return 1;
    if (dev_alloc(h, &h->d_textoff, (size_t)n_snp + 1)) return 1;
    if (dev_alloc(h, &h->d_nonblank, (size_t)n_snp)) return 1;
    std::vector<long long> rel(n_snp + 1);
    for (int i = 0; i <= n_snp; ++i) rel[i] = (long long)(line_off[i] - line_off[0]);
    CK(cudaMemcpyAsync(h->d_text, text + line_off[0], (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_textoff, rel.data(), rel.size() * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    uint8_t* dst = h->d_alleles + (size_t)snp0 * h->n_ind * 2;
    // a short line leaves its tail untouched: pre-fill with the missing character so that nothing undefined is coded
    CK(cudaMemsetAsync(dst, (unsigned char)missing, (size_t)n_snp * h->n_ind * 2, h->stream));
    LAUNCH(launch_tokenize_tped(h->d_text, h->d_textoff, n_snp, h->n_ind, h->ind_offset, dst, h->d_nonblank, h->stream));
    LAUNCH(launch_first_allele(dst, n_snp, h->n_ind, h->ind_offset, (unsigned char)missing, h->d_key + snp0, h->stream));
    h->missing_char = (unsigned char)missing;
    if (nonblank) CK(cudaMemcpyAsync(nonblank, h->d_nonblank, (size_t)n_snp * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // the caller may reuse its text buffer
    return 0;
}

int garlic_gpu_put_vcf_text(garlic_gpu_t* h, const char* text, const int64_t* line_off, int64_t snp0, int n_snp,
                            int32_t* n_cols, int32_t* max_allele, int32_t* bad_col)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_vcf_text: call set_shape first");
    if (snp0 % 32 != 0 || snp0 < 0 || snp0 + n_snp > h->L0) FAIL("put_vcf_text: bad SNP range (snp0 must be a multiple of 32)");
    if (n_snp <= 0) return 0;
    if (h->bed_input) FAIL("put_vcf_text: this handle holds .bed input");
    if (h->d_alleles && !h->vcf_input) FAIL("put_vcf_text: this handle holds tped input");
    if (!h->d_alleles) {
        if (dev_alloc(h, &h->d_alleles, (size_t)h->L0 * h->n_ind * 2)) return 1;
        if (dev_alloc(h, &h->d_key, (size_t)h->L0)) return 1;
        h->vcf_input = true;
    }
    const int64_t bytes = line_off[n_snp] - line_off[0];
    if (bytes < 0) FAIL("put_vcf_text: line offsets must ascend");
    if (dev_alloc(h, &h->d_text, (size_t)bytes + 16)) return 1;
    if (dev_alloc(h, &h->d_textoff, (size_t)n_snp + 1)) return 1;
    if (dev_alloc(h, &h->d_nonblank, (size_t)3 * n_snp)) return 1;     // column count, largest index, first bad column
    std::vector<long long> rel(n_snp + 1);
    for (int i = 0; i <= n_snp; ++i) rel[i] = (long long)(line_off[i] - line_off[0]);
    CK(cudaMemcpyAsync(h->d_text, text + line_off[0], (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_textoff, rel.data(), rel.size() * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    uint8_t* dst = h->d_alleles + (size_t)snp0 * h->n_ind * 2;
    // a short record leaves its tail untouched: pre-fill with the missing code so that nothing undefined is coded
    CK(cudaMemsetAsync(dst, 255, (size_t)n_snp * h->n_ind * 2, h->stream));
    int* diag = h->d_nonblank;
    LAUNCH(launch_tokenize_vcf(h->d_text, h->d_textoff, n_snp, h->n_ind, h->ind_offset, dst, diag, diag + n_snp,
                               diag + 2 * n_snp, h->stream));
    LAUNCH(launch_first_allele(dst, n_snp, h->n_ind, h->ind_offset, 255, h->d_key + snp0, h->stream));
    h->missing_char = 255;
    int32_t* out[3] = {n_cols, max_allele, bad_col};
    for (int k = 0; k < 3; ++k)
        if (out[k]) CK(cudaMemcpyAsync(out[k], diag + (size_t)k * n_snp, (size_t)n_snp * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // the caller may reuse its text buffer
    return 0;
}

void* garlic_gpu_first_allele_keys_dev(garlic_gpu_t* h) { return h ? (void*)h->d_key : nullptr; }

// .bed rows of the whole file → this handle's byte columns of SNPs [snp0, snp0 + n_snp), then phase a (bed.cu)
static int put_bed_common(garlic_gpu* h, const void* rows, int64_t stride, int64_t snp0, int n_snp, cudaMemcpyKind kind)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_bed: call set_shape first");
    if (snp0 % 32 != 0 || snp0 < 0 || n_snp < 0 || snp0 + n_snp > h->L0) FAIL("put_bed: bad SNP range (snp0 must be a multiple of 32)");
    if (h->d_alleles) FAIL("put_bed: this handle holds allele input");
    const int64_t byte0 = h->ind_offset / 4, sh = h->ind_offset % 4;
    const int64_t width = (sh + h->n_ind + 3) / 4;
    if (stride < byte0 + width) FAIL("put_bed: SNP row stride smaller than the bytes of this handle's individuals");
    if (!h->d_bed) {
        h->bed_stride = (width + 31) / 32 * 32;               // whole 32-byte sectors per row (bed_transpose_kernel)
        if (dev_alloc(h, &h->d_bed, (size_t)h->L0 * h->bed_stride)) return 1;
        if (dev_alloc(h, &h->d_key, (size_t)h->L0)) return 1;
        h->bed_input = true;
    }
    if (n_snp == 0) return 0;
    uint8_t* dst = h->d_bed + (size_t)snp0 * h->bed_stride;
    if (kind == cudaMemcpyHostToDevice && width == stride) {
        // a pitched host-to-device copy costs about 0.13 us per row (76 ms for the 600 k rows of a 2,000-individual file
        // on a B200 box): a handle that keeps every column takes the rows in one piece and re-pitches them on the device
        if (dev_alloc(h, &h->d_bed_rows, (size_t)n_snp * stride)) return 1;
        CK(cudaMemcpyAsync(h->d_bed_rows, rows, (size_t)n_snp * stride, kind, h->stream));
        rows = h->d_bed_rows;
        kind = cudaMemcpyDeviceToDevice;
    }
    CK(cudaMemcpy2DAsync(dst, (size_t)h->bed_stride, (const uint8_t*)rows + byte0, (size_t)stride, (size_t)width, (size_t)n_snp,
                         kind, h->stream));
    CK(cudaEventRecord(h->ev_copy, h->stream));
    LAUNCH(launch_bed_count(dst, h->bed_stride, n_snp, (int)sh, h->n_ind, h->ind_offset, h->d_counts + snp0, h->L0,
                            h->d_key + snp0, h->stream));
    h->counts_reduced = false; h->counts_hi_reduced = false;
    CK(cudaEventSynchronize(h->ev_copy));   // the copy has left the caller's buffer (it may be page-locked and reused)
    return 0;
}

int garlic_gpu_put_bed(garlic_gpu_t* h, const uint8_t* rows, int64_t snp_stride_bytes, int64_t snp0, int n_snp)
{
    return put_bed_common(h, rows, snp_stride_bytes, snp0, n_snp, cudaMemcpyHostToDevice);
}
int garlic_gpu_put_bed_dev(garlic_gpu_t* h, const void* rows_dev, int64_t snp_stride_bytes, int64_t snp0, int n_snp)
{
    return put_bed_common(h, rows_dev, snp_stride_bytes, snp0, n_snp, cudaMemcpyDeviceToDevice);
}

int garlic_gpu_code_alleles(garlic_gpu_t* h)
{
    CK(cudaSetDevice(h->device));
    if (!h->d_alleles && !h->d_bed) FAIL("code_alleles: no alleles uploaded");
    const int missing = h->missing_char;
    h->counts_reduced = false; h->counts_hi_reduced = false;
    // the "1" allele is the first non-missing character over ALL individuals: MIN over the shards' keys
    if (h->comm) NCK(ncclAllReduce(h->d_key, h->d_key, (size_t)h->L0, ncclUint64, ncclMin, h->comm, h->stream));
    if (h->d_bed) {
        // put_bed's phase a left the counters of every SNP; nothing reads the staged rows after the transpose
        if (dev_alloc(h, &h->d_a1, (size_t)(h->L0 + 31) / 32)) return 1;
        LAUNCH(launch_bed_code(h->d_bed, h->bed_stride, h->L0, h->ind_offset % 4, h->n_ind, h->d_key, h->d_counts, h->d_a1,
                               h->d_geno0, h->row_words0, h->stream));
        h->launches++;                     // (two kernels)
        CK(cudaStreamSynchronize(h->stream));
        dev_free(h->d_bed); dev_free(h->d_bed_rows);
        h->have_geno0 = true;
        return 0;
    }
    CK(cudaMemsetAsync(h->d_counts, 0, (size_t)4 * h->L0 * sizeof(int), h->stream));
    // chunks of SNPs so the grid stays within limits; all chunks start on a 32-SNP boundary
    const int64_t chunk = 1 << 20;
    for (int64_t s0 = 0; s0 < h->L0; s0 += chunk) {
        const int n = (int)std::min<int64_t>(chunk, h->L0 - s0);
        LAUNCH(launch_code_alleles(h->d_alleles + (size_t)s0 * h->n_ind * 2, n, h->n_ind, missing, h->d_key + s0, s0,
                                   h->d_geno0, h->row_words0, h->d_counts, h->L0, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    h->have_geno0 = true;
    return 0;
}

static int put_packed_common(garlic_gpu* h, const void* rows, int64_t stride, cudaMemcpyKind kind)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_packed: call set_shape first");
    const int64_t need = (h->L0 + 3) / 4;
    if (stride < need) FAIL("put_packed: row stride smaller than ceil(n_loci/4)");
    h->precounted = false;
    if (kind == cudaMemcpyHostToDevice && h->n_ind >= 256 && h->d_counts) {
        // host rows: the copy goes in slices of individuals on the copy stream and K2 counts each slice as soon as it has
        // landed, so the column reduction hides behind the PCIe transfer (garlic_gpu_count_packed then has nothing to do)
        const int n_slices = 8;
        const int per = ((h->n_ind + n_slices - 1) / n_slices + 15) / 16 * 16;
        CK(cudaMemsetAsync(h->d_counts, 0, (size_t)4 * h->L0 * sizeof(int), h->stream));
        CK(cudaEventRecord(h->ev_copy, h->stream));
        CK(cudaStreamWaitEvent(h->copy_stream, h->ev_copy, 0));            // earlier work on the rows is done
        for (int r0 = 0; r0 < h->n_ind; r0 += per) {
            const int n = std::min(per, h->n_ind - r0);
            uint64_t* dst = h->d_geno0 + (size_t)r0 * h->row_words0;
            CK(cudaMemcpy2DAsync(dst, (size_t)h->row_words0 * 8, (const char*)rows + (size_t)r0 * stride, (size_t)stride, (size_t)need,
                                 (size_t)n, kind, h->copy_stream));
            CK(cudaEventRecord(h->ev_copy, h->copy_stream));
            CK(cudaStreamWaitEvent(h->stream, h->ev_copy, 0));
            LAUNCH(launch_count_packed(dst, h->row_words0, n, h->L0, h->d_counts, h->stream));
        }
        CK(cudaStreamSynchronize(h->copy_stream));                          // the caller may reuse its buffer
        h->precounted = true;
        h->counts_reduced = false; h->counts_hi_reduced = false;
        h->have_geno0 = true;
        return 0;
    }
    CK(cudaMemcpy2DAsync(h->d_geno0, (size_t)h->row_words0 * 8, rows, (size_t)stride, (size_t)need, (size_t)h->n_ind, kind, h->stream));
    // bits of the last partial word beyond n_loci may hold anything; they are never read as SNPs < L0
    CK(cudaStreamSynchronize(h->stream));
    h->have_geno0 = true;
    return 0;
}

int garlic_gpu_put_packed(garlic_gpu_t* h, const uint8_t* rows, int64_t row_stride_bytes)
{
    return put_packed_common(h, rows, row_stride_bytes, cudaMemcpyHostToDevice);
}
int garlic_gpu_put_packed_dev(garlic_gpu_t* h, const void* rows_dev, int64_t row_stride_bytes)
{
    return put_packed_common(h, rows_dev, row_stride_bytes, cudaMemcpyDeviceToDevice);
}

// adds host correction vectors to device counts
__global__ void add_corr_kernel(int* counts, long long L0, const int* na, const int* tot)
{
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < L0; s += (long long)gridDim.x * blockDim.x) {
        if (na) counts[s] += na[s];
        if (tot) counts[L0 + s] += tot[s];
    }
}

int garlic_gpu_count_packed(garlic_gpu_t* h, const int32_t* nalleles_corr, const int32_t* total_corr)
{
    CK(cudaSetDevice(h->device));
    if (!h->have_geno0) FAIL("count_packed: no genotypes loaded");
    tl_mark(h, "count_packed:in");
    h->counts_reduced = false; h->counts_hi_reduced = false;
    if (h->precounted) {
        h->precounted = false;             // garlic_gpu_put_packed counted the rows while they arrived
    } else {
        CK(cudaMemsetAsync(h->d_counts, 0, (size_t)4 * h->L0 * sizeof(int), h->stream));
        LAUNCH(launch_count_packed(h->d_geno0, h->row_words0, h->n_ind, h->L0, h->d_counts, h->stream));
    }
    if (nalleles_corr || total_corr) {
        if (dev_alloc(h, &h->d_corr, (size_t)2 * h->L0)) return 1;     // scratch kept on the handle
        int *d_a = nalleles_corr ? h->d_corr : nullptr, *d_t = total_corr ? h->d_corr + h->L0 : nullptr;
        if (d_a) CK(cudaMemcpyAsync(d_a, nalleles_corr, h->L0 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        if (d_t) CK(cudaMemcpyAsync(d_t, total_corr, h->L0 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        add_corr_kernel<<<(unsigned)std::min<int64_t>((h->L0 + 255) / 256, 148 * 16), 256, 0, h->stream>>>(h->d_counts, h->L0, d_a, d_t);
        CK(cudaGetLastError());
        h->launches++;
        CK(cudaStreamSynchronize(h->stream));                          // the caller may reuse its vectors
    }
    if (h->xchg_ok) return 0;              // the sums are formed by the NVLink exchange fused with freq + keep (filter)
    return reduce_counts(h, false);        // starts right behind the count kernel; filter() finds the sums ready
}

void* garlic_gpu_counts_dev(garlic_gpu_t* h) { return h ? (void*)h->d_counts : nullptr; }

int garlic_gpu_get_counts(garlic_gpu_t* h, int32_t* na, int32_t* tot, int32_t* hom, int32_t* nm)
{
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    int32_t* dst[4] = {na, tot, hom, nm};
    for (int c = 0; c < 4; ++c)
        if (dst[c]) CK(cudaMemcpy(dst[c], h->d_counts + (size_t)c * h->L0, h->L0 * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

int garlic_gpu_get_one_allele(garlic_gpu_t* h, uint8_t* allele, char missing)
{
    CK(cudaSetDevice(h->device));
    if (!h->d_key) FAIL("get_one_allele: alleles were not ingested on this handle");
    std::vector<unsigned long long> k(h->L0);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(k.data(), h->d_key, h->L0 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    for (int64_t s = 0; s < h->L0; ++s) allele[s] = (k[s] == ~0ull) ? (uint8_t)missing : (uint8_t)(k[s] & 0xff);
    return 0;
}

static int put_gl_common(garlic_gpu* h, const void* v, int gl_type, cudaMemcpyKind kind)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_gl: call set_shape first");
    if (gl_type < -1 || gl_type > 2) FAIL("put_gl: bad gl_type");
    if (dev_alloc(h, &h->d_gl0, (size_t)h->n_ind * h->L0)) return 1;
    CK(cudaMemcpyAsync(h->d_gl0, v, (size_t)h->n_ind * h->L0 * sizeof(double), kind, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->gl_type = gl_type;
    h->have_gl = true;
    return 0;
}
int garlic_gpu_put_tgls_text(garlic_gpu_t* h, const char* text, const int64_t* line_off, int64_t snp0, int n_snp,
                             int gl_type, int32_t* n_tokens)
{
    CK(cudaSetDevice(h->device));
    if (!h->L0) FAIL("put_tgls_text: call set_shape first");
    if (gl_type < -1 || gl_type > 2) FAIL("put_tgls_text: bad gl_type");
    if (snp0 < 0 || n_snp < 0 || snp0 + n_snp > h->L0) FAIL("put_tgls_text: bad SNP range");
    if (n_snp == 0) return 0;
    const int64_t bytes = line_off[n_snp] - line_off[0];
    if (bytes < 0) FAIL("put_tgls_text: line offsets must ascend");
    if (dev_alloc(h, &h->d_gl0, (size_t)h->n_ind * h->L0)) return 1;
    if (dev_alloc(h, &h->d_text, (size_t)bytes + 16)) return 1;
    if (dev_alloc(h, &h->d_textoff, (size_t)n_snp + 1)) return 1;
    if (dev_alloc(h, &h->d_nonblank, (size_t)n_snp)) return 1;
    const unsigned hard_cap = 1u << 16;
    if (dev_alloc(h, &h->d_hard, (size_t)hard_cap + 1)) return 1;
    unsigned* d_hard_n = reinterpret_cast<unsigned*>(h->d_hard + hard_cap);
    std::vector<long long> rel(n_snp + 1);
    for (int i = 0; i <= n_snp; ++i) rel[i] = (long long)(line_off[i] - line_off[0]);
    const char* base = text + line_off[0];
    CK(cudaMemcpyAsync(h->d_text, base, (size_t)bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_textoff, rel.data(), rel.size() * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(d_hard_n, 0, sizeof(unsigned), h->stream));
    LAUNCH(launch_tokenize_tgls(h->d_text, h->d_textoff, n_snp, h->n_ind, h->ind_offset, h->d_gl0, h->L0, snp0, h->d_nonblank,
                                h->d_hard, d_hard_n, hard_cap, h->stream));
    std::vector<int32_t> ntok_local;
    if (!n_tokens) { ntok_local.resize(n_snp); n_tokens = ntok_local.data(); }
    unsigned n_hard = 0;
    CK(cudaMemcpyAsync(n_tokens, h->d_nonblank, (size_t)n_snp * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&n_hard, d_hard_n, sizeof(unsigned), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));   // the caller may reuse its text buffer
    if (n_hard) {
        // tokens outside the exact fast path: converted here with strtod, exactly what the host reader does.  More of them
        // than the list holds: every token of this rank's columns is converted on the host (correct, only slow).
        auto token_at = [&](int l, int k) -> const char* {
            const char* p = base + rel[l];
            const char* e = base + rel[l + 1];
            for (int t = 0;; ++t) {
                while (p < e && (*p == ' ' || *p == '\t' || *p == '\r' || *p == '\n')) ++p;
                if (p >= e) return nullptr;
                if (t == k) return p;
                while (p < e && !(*p == ' ' || *p == '\t' || *p == '\r' || *p == '\n')) ++p;
            }
        };
        auto convert = [&](const char* p, int l) -> double {
            const char* e = base + rel[l + 1];
            const char* q = p;
            while (q < e && !(*q == ' ' || *q == '\t' || *q == '\r' || *q == '\n')) ++q;
            const std::string tok(p, q);                                   // strtod needs a terminated string
            return strtod(tok.c_str(), nullptr);
        };
        std::vector<int2> list;
        if (n_hard <= hard_cap) {
            list.resize(n_hard);
            CK(cudaMemcpy(list.data(), h->d_hard, n_hard * sizeof(int2), cudaMemcpyDeviceToHost));
        } else {
            for (int l = 0; l < n_snp; ++l)
                for (int k = h->ind_offset; k < h->ind_offset + h->n_ind; ++k) list.push_back(make_int2(l, k));
        }
        std::sort(list.begin(), list.end(), [](const int2& a, const int2& b) { return a.x != b.x ? a.x < b.x : a.y < b.y; });
        for (const int2& t : list) {
            const char* p = token_at(t.x, t.y);
            if (!p) continue;
            const double v = convert(p, t.x);
            CK(cudaMemcpyAsync(h->d_gl0 + (size_t)(t.y - h->ind_offset) * h->L0 + snp0 + t.x, &v, sizeof(double), cudaMemcpyHostToDevice, h->stream));
            CK(cudaStreamSynchronize(h->stream));                          // v lives on this stack frame
        }
    }
    h->gl_type = gl_type;
    h->have_gl = true;
    return 0;
}

int garlic_gpu_get_gl(garlic_gpu_t* h, double* values)
{
    CK(cudaSetDevice(h->device));
    if (!h->have_gl || !h->d_gl0) FAIL("get_gl: no likelihoods loaded");
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(values, h->d_gl0, (size_t)h->n_ind * h->L0 * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

int garlic_gpu_put_gl(garlic_gpu_t* h, const double* values, int gl_type) { return put_gl_common(h, values, gl_type, cudaMemcpyHostToDevice); }
int garlic_gpu_put_gl_dev(garlic_gpu_t* h, const void* values_dev, int gl_type) { return put_gl_common(h, values_dev, gl_type, cudaMemcpyDeviceToDevice); }

int garlic_gpu_filter(garlic_gpu_t* h, int oob, const int32_t* chr_param, const double* freq_override,
                      double* freq_out, uint8_t* keep_out, int64_t* n_kept)
{
    CK(cudaSetDevice(h->device));
    if (!h->have_geno0) FAIL("filter: no genotypes loaded");
    if (oob && !chr_param) FAIL("filter: oob filtering needs chr_param");
    const int64_t L0 = h->L0;
    Laps laps("filter");
    laps.rank = h->comm_rank;
    if (finish_outputs(h)) return 1;
    tl_mark(h, "filter:in");
    if (!freq_override) h->fmin = 0.5;
    bool freq_direct = false, keep_direct = false, copies_in_flight = false;
    if (dev_alloc(h, &h->d_freq0, (size_t)L0)) return 1;
    if (dev_alloc(h, &h->d_keep, (size_t)L0)) return 1;
    if (oob) {
        if (dev_alloc(h, &h->d_chr_param, (size_t)4 * h->n_chr)) return 1;
        CK(cudaMemcpyAsync(h->d_chr_param, chr_param, 4 * h->n_chr * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    }
    // pinned staging: freq0[L0] doubles | keep[L0] bytes | total, chr_off_kept[C+1] ints
    const int n_blocks = (int)((L0 + 1023) / 1024);
    const size_t off_keep = (size_t)L0 * 8, off_meta = (off_keep + (size_t)L0 + 63) & ~(size_t)63;
    if (pin_alloc(h, off_meta + (size_t)(h->n_chr + 2) * 4 + 64)) return 1;
    double* freq0 = reinterpret_cast<double*>(h->pin);
    uint8_t* keep = h->pin + off_keep;
    int32_t* meta = reinterpret_cast<int32_t*>(h->pin + off_meta);
    if (freq_override) {
        // --freq-file: frequencies come from the caller; the predicate is evaluated on the host copy
        h->fmin = 0.5;
        for (int64_t s = 0; s < L0; ++s) {
            const double f = freq_override[s];
            bool k = (f > 0 && f < 1);
            if (k) h->fmin = std::min(h->fmin, std::min(f, 1.0 - f));
            if (oob) {
                int c = (int)(std::upper_bound(h->chr_off0.begin(), h->chr_off0.end(), s) - h->chr_off0.begin()) - 1;
                const int32_t* cp = chr_param + 4 * c;
                const int p = h->pos0[s];
                k = k && !(p < cp[0]) && !(p > cp[1]) && !(p > cp[2] && p < cp[3]);
            }
            freq0[s] = f; keep[s] = k;
        }
        CK(cudaMemcpyAsync(h->d_freq0, freq0, L0 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_keep, keep, L0, cudaMemcpyHostToDevice, h->stream));
    } else {
        // the one data-path collective (SURVEY §8e): per-SNP counters of all shards, summed in place on this stream
        if (h->comm && !h->xchg_tried && ensure_xchg(h)) return 1;
        if (h->xchg_ok && !h->counts_reduced) {
            // one kernel over NVLink peer memory: counters of all ranks summed, freq and keep evaluated, all three stored
            // into every rank's tables (xchg.cu) — instead of ncclAllReduce + freq_keep_kernel
            XchgParams X;
            memset(&X, 0, sizeof(X));
            for (int p = 0; p < h->comm_world; ++p) {
                uint8_t* base = static_cast<uint8_t*>(h->xpeer[p]);
                X.flags[p] = reinterpret_cast<unsigned*>(base);
                X.counts[p] = reinterpret_cast<int*>(base + h->x_off_counts);
                X.freq[p] = reinterpret_cast<double*>(base + h->x_off_freq);
                X.keep[p] = base + h->x_off_keep;
            }
            X.n = h->comm_world; X.rank = h->comm_rank; X.seq = ++h->xchg_seq; X.L0 = L0;
            X.pos = h->d_pos0; X.chr_of = h->d_chr_of0; X.chr_param = h->d_chr_param; X.oob = oob;
            X.done_counter = reinterpret_cast<unsigned*>(h->xslab) + 48;
            LAUNCH(launch_xchg_freq_keep(X, h->stream));
            h->counts_reduced = true;
        } else {
            if (reduce_counts(h, false)) return 1;
            LAUNCH(launch_freq_keep(h->d_counts, L0, h->d_pos0, h->d_chr_of0, h->d_chr_param, oob, h->d_freq0, h->d_keep, h->stream));
        }
        // page-locked caller buffers (garlic_gpu_host_alloc) are written by the copy engine directly
        freq_direct = freq_out && is_pinned(freq_out);
        keep_direct = keep_out && is_pinned(keep_out);
        // freq[] / keep[] travel to the host on a second stream, behind the kernel that made them, while the keep-mask
        // scan and the compaction run on: the host only waits for them at the end of this call
        copies_in_flight = freq_out || keep_out;     // (enqueued below, behind the few bytes this call itself waits for)
    }
    // exclusive scan of the keep mask on the device: gather list, keep bits per input word, per output word
    // the input word it starts in, kept offset of every chromosome
    if (dev_alloc(h, &h->d_src, (size_t)L0)) return 1;
    if (dev_alloc(h, &h->d_scan, (size_t)n_blocks + h->n_chr + 8)) return 1;
    int* d_total = h->d_scan + n_blocks;
    int* d_chr_off_kept = d_total + 1;
    CK(launch_keep_scan(h->d_keep, L0, h->d_chr_of0, h->n_chr, h->d_scan, d_total, h->d_src, d_chr_off_kept, h->stream));
    h->launches += 3;
    CK(cudaMemcpyAsync(meta, d_total, (size_t)(h->n_chr + 2) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (copies_in_flight) {
        // freq[] / keep[] travel to the host on a second stream while the path runs on.  They start behind the copy of
        // the kept-SNP count above: device-to-host copies share one engine, and 5 MB in front of those few bytes would
        // hold this call's synchronisation for 0.1 ms.
        CK(cudaEventRecord(h->ev_copy, h->stream));
        CK(cudaStreamWaitEvent(h->copy_stream, h->ev_copy, 0));
        if (freq_out) CK(cudaMemcpyAsync(freq_direct ? freq_out : freq0, h->d_freq0, L0 * sizeof(double), cudaMemcpyDeviceToHost, h->copy_stream));
        if (keep_out) CK(cudaMemcpyAsync(keep_direct ? keep_out : keep, h->d_keep, L0, cudaMemcpyDeviceToHost, h->copy_stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    laps.lap("freq_keep+scan");
    tl_mark(h, "filter:after-sync");
    if (freq_override) {
        if (freq_out) memcpy(freq_out, freq0, L0 * sizeof(double));
        if (keep_out) memcpy(keep_out, keep, L0);
    }
    const int64_t L = meta[0];
    h->chr_off.assign(h->n_chr + 1, 0);
    for (int c = 0; c <= h->n_chr; ++c) h->chr_off[c] = meta[1 + c];
    h->src.clear();          // host copies of the gather list / kept positions are fetched on demand
    h->pos.clear();
    h->L = L;
    if (n_kept) *n_kept = L;
    if (L < 1) FAIL("filter: no polymorphic loci left");
    h->row_words = (((L + kPad + 31) >> 5) + 3) & ~(int64_t)1;   // even: rows are whole 16-byte quads
    // the compaction itself, and the compacted matrix, wait for their first consumer (ensure_geno): here only its plan,
    // from the gather list
    h->n_pieces = (int)((L + kPiece - 1) / kPiece);
    {
        const long long n_q = 16ll * (h->n_pieces + 4);
        if (dev_alloc(h, &h->d_plan_head, (size_t)n_q)) return 1;
        if (dev_alloc(h, &h->d_plan_seg, (size_t)n_q * kPlanSegMax)) return 1;
        if (dev_alloc(h, &h->d_plan_rng, (size_t)h->n_pieces + 4)) return 1;
        if (dev_alloc(h, &h->d_plan_fast, (size_t)n_q)) return 1;
        LAUNCH(launch_plan(h->d_src, d_total, n_q, h->d_plan_head, h->d_plan_seg, h->d_plan_fast, h->d_plan_rng, h->stream));
    }
    h->geno_pending = true; h->bound_W = 0; h->bound_tables_W = 0;
    if (dev_alloc(h, &h->d_freq, (size_t)L + kPad)) return 1;
    CK(cudaMemsetAsync(h->d_freq, 0, (size_t)(L + kPad) * sizeof(double), h->stream));
    LAUNCH(launch_gather_f64(h->d_freq0, h->d_src, L, h->d_freq, h->stream));
    if (h->have_gl) {
        h->gl_stride = L + kPad;
        // lane-interleaved [groups of 32 individuals][gl_stride][32] (common.cuh:gl_lane); the kernel writes every element
        if (dev_alloc(h, &h->d_gl, (size_t)((h->n_ind + 31) / 32) * 32 * h->gl_stride)) return 1;
        LAUNCH(launch_compact_gl(h->d_gl0, L0, h->d_src, L, h->d_geno0, h->row_words0, h->d_freq0, h->d_gl, h->gl_stride, h->n_ind,
                                 h->gl_type, h->stream));
    }
    // per-SNP position / chromosome arrays of the kept SNPs (device-side gathers)
    std::vector<int> chr_start(h->n_chr);
    for (int c = 0; c < h->n_chr; ++c) chr_start[c] = (int)h->chr_off[c];
    if (dev_alloc(h, &h->d_pos, (size_t)L)) return 1;
    if (dev_alloc(h, &h->d_chr_of, (size_t)L)) return 1;
    if (dev_alloc(h, &h->d_chr_start, (size_t)h->n_chr)) return 1;
    LAUNCH(launch_gather_i32(h->d_pos0, h->d_src, L, h->d_pos, h->stream));
    LAUNCH(launch_gather_i32(h->d_chr_of0, h->d_src, L, h->d_chr_of, h->stream));
    CK(cudaMemcpyAsync(h->d_chr_start, chr_start.data(), h->n_chr * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    laps.lap("enqueue");   // compaction and gathers run stream-ordered behind this call
    if (copies_in_flight) {
        const bool all_direct = (!freq_out || freq_direct) && (!keep_out || keep_direct);
        if (all_direct) {
            // page-locked caller buffers: the copy engine fills them behind this call (include/garlic_b200.h)
            h->out_pending = true;
        } else {
            CK(cudaStreamSynchronize(h->copy_stream));
            if (freq_out && !freq_direct) memcpy(freq_out, freq0, L0 * sizeof(double));
            if (keep_out && !keep_direct) memcpy(keep_out, keep, L0);
        }
        laps.lap("freq/keep d2h");
    }
    h->filtered = true; h->tables = false; h->have_ld = false;
    tl_mark(h, "filter:out");
    return 0;
}

int64_t garlic_gpu_n_kept(const garlic_gpu_t* h) { return h ? h->L : 0; }

int garlic_gpu_get_genotypes(garlic_gpu_t* h, int filtered, uint8_t* rows, int64_t row_stride_bytes)
{
    CK(cudaSetDevice(h->device));
    if (filtered ? !h->filtered : !h->have_geno0) FAIL("get_genotypes: nothing loaded");
    const int64_t n = filtered ? h->L : h->L0;
    const int64_t need = (n + 3) / 4;
    if (row_stride_bytes < need) FAIL("get_genotypes: row stride too small");
    if (filtered && ensure_geno(h, 0)) return 1;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy2D(rows, (size_t)row_stride_bytes, filtered ? h->d_geno : h->d_geno0,
                    (size_t)(filtered ? h->row_words : h->row_words0) * 8, (size_t)need, (size_t)h->n_ind, cudaMemcpyDeviceToHost));
    return 0;
}

int garlic_gpu_get_kept_index(garlic_gpu_t* h, int32_t* src_index)
{
    if (!h->filtered) FAIL("get_kept_index: call filter first");
    if (fetch_src(h)) return 1;
    memcpy(src_index, h->src.data(), h->L * sizeof(int32_t));
    return 0;
}

int garlic_gpu_set_tables(garlic_gpu_t* h, double error, int max_gap, const int32_t* centromeres, const double* gpos)
{
    CK(cudaSetDevice(h->device));
    if (!h->filtered) FAIL("set_tables: call filter first");
    h->error = error; h->max_gap = max_gap;
    Laps laps("set_tables");
    laps.rank = h->comm_rank;
    tl_mark(h, "set_tables:in");
    h->cen.assign(2 * h->n_chr, 0);
    if (centromeres) h->cen.assign(centromeres, centromeres + 2 * h->n_chr);
    const int64_t L = h->L;
    if (dev_alloc(h, &h->d_lut, (size_t)(L + kPad) * 4)) return 1;
    CK(cudaMemsetAsync(h->d_lut, 0, (size_t)(L + kPad) * 4 * sizeof(double), h->stream));
    LAUNCH(launch_build_lut(h->d_freq, L, error, h->d_lut, h->stream));
    h->gpos.clear();
    if (gpos) {
        h->gpos.assign(gpos, gpos + L);
        if (dev_alloc(h, &h->d_gpos, (size_t)L)) return 1;
        CK(cudaMemcpyAsync(h->d_gpos, gpos, L * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    }
    h->amax = lod_bound(h);   // enters the ambiguity tolerance of the chunked / tensor-core passes
    // gap/centromere-free stretches: bad adjacent pairs found on the device (a short list); the count and the first
    // entries travel to a page-locked block behind the kernels above.  Nobody waits here: the first consumer of the
    // stretches (ensure_stretches) does, after it has put its own first kernels — the compaction — on the stream.
    {
        if (dev_alloc(h, &h->d_breaks, (size_t)kBreakCap + 2 * h->n_chr + 4)) return 1;
        int* d_cen = h->d_breaks + kBreakCap;
        unsigned* d_n = reinterpret_cast<unsigned*>(d_cen + 2 * h->n_chr);
        CK(cudaMemcpyAsync(d_cen, h->cen.data(), 2 * h->n_chr * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemsetAsync(d_n, 0, sizeof(unsigned), h->stream));
        if (dev_alloc(h, &h->d_badbits, (size_t)((L + 31) >> 5) + 4)) return 1;
        LAUNCH(launch_bad_pairs(h->d_pos, h->d_chr_of, d_cen, max_gap, L, h->d_breaks, d_n, kBreakCap, h->d_badbits, h->stream));
        if (!h->brk_pin) CK(cudaMallocHost((void**)&h->brk_pin, 64 + kBreakFirst * sizeof(int)));
        CK(cudaMemcpyAsync(h->brk_pin, d_n, sizeof(unsigned), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(h->brk_pin + 64, h->d_breaks, kBreakFirst * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev_tables, h->stream));
        h->stretches_pending = true;
        h->stretches.clear();
    }
    laps.lap("enqueue");
    tl_mark(h, "set_tables:out");
    h->tables = true; h->have_ld = false; h->bound_W = 0; h->bound_tables_W = 0; h->tables_gen++;
    return 0;
}

int garlic_gpu_set_lut(garlic_gpu_t* h, const double* lut)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("set_lut: call set_tables first");
    CK(cudaMemcpy(h->d_lut, lut, (size_t)h->L * 4 * sizeof(double), cudaMemcpyHostToDevice));
    double m = 0;                                           // the caller's table: its own largest magnitude
    for (int64_t i = 0; i < h->L * 4; ++i) { const double a = std::fabs(lut[i]); if (a > m && std::isfinite(a)) m = a; }
    h->amax = std::max(lod_bound(h), m + 1.0);
    dev_free(h->d_wlut);   // the weighted score table is rebuilt on demand
    h->bound_W = 0; h->bound_tables_W = 0;   // and so are the pruning tables and the piece maxima
    return 0;
}

int garlic_gpu_get_lut(garlic_gpu_t* h, double* lut)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("get_lut: call set_tables first");
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(lut, h->d_lut, (size_t)h->L * 4 * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

int garlic_gpu_get_hom_freq(garlic_gpu_t* h, double* hom_freq)
{
    CK(cudaSetDevice(h->device));
    if (!h->filtered) FAIL("get_hom_freq: call filter first");
    std::vector<int> hom(h->L0), nm(h->L0);
    if (reduce_counts(h, true)) return 1;      // (with a communicator attached: a collective, every rank calls it)
    if (garlic_gpu_get_counts(h, nullptr, nullptr, hom.data(), nm.data())) return 1;
    if (fetch_src(h)) return 1;
    for (int64_t d = 0; d < h->L; ++d) {
        double total = nm[h->src[d]], fh = hom[h->src[d]];
        fh /= total;   // 0/0 → NaN exactly as the reference (garlic-data.cpp:672)
        hom_freq[d] = fh;
    }
    return 0;
}

int garlic_gpu_set_prune(garlic_gpu_t* h, int on)
{
    h->prune = on != 0;
    return 0;
}

int garlic_gpu_set_phased(garlic_gpu_t* h, int phased)
{
    h->phased = phased != 0;
    h->have_ld = false;
    return 0;
}

int garlic_gpu_set_wlod(garlic_gpu_t* h, double mu, int M)
{
    h->mu = mu; h->M = M;
    dev_free(h->d_wlut);
    return 0;
}

}  // extern "C"

// the break list of set_tables has arrived: sort it into the per-chromosome stretches
static int ensure_stretches(garlic_gpu* h)
{
    if (!h->stretches_pending) return 0;
    CK(cudaEventSynchronize(h->ev_tables));
    const unsigned nb = *reinterpret_cast<const unsigned*>(h->brk_pin);
    const int* first_host = reinterpret_cast<const int*>(h->brk_pin + 64);
    if (nb > kBreakCap) FAIL("set_tables: more than 2^20 gaps; raise --max-gap");
    std::vector<int> breaks(first_host, first_host + std::min(nb, kBreakFirst));
    if (nb > kBreakFirst) {
        breaks.resize(nb);
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpy(breaks.data() + kBreakFirst, h->d_breaks + kBreakFirst, (nb - kBreakFirst) * sizeof(int), cudaMemcpyDeviceToHost));
    }
    std::sort(breaks.begin(), breaks.end());
    h->stretches.clear();
    size_t bi = 0;
    for (int c = 0; c < h->n_chr; ++c) {
        int a = (int)h->chr_off[c];
        const int hi = (int)h->chr_off[c + 1];
        while (bi < breaks.size() && breaks[bi] < hi) {
            if (breaks[bi] > a) h->stretches.push_back({c, a, breaks[bi]});
            a = breaks[bi++];
        }
        if (hi > a) h->stretches.push_back({c, a, hi});
    }
    h->stretches_pending = false;
    return 0;
}

// counters every pass 2 starts from zero, in one block (one memset): [cnt 4 | work units 4 | hist n_ind+1 | kept n_ind+1]
static int ensure_zero_block(garlic_gpu* h)
{
    const size_t n = 8 + 2 * ((size_t)h->n_ind + 1);
    if (h->zero_cap < n) {
        if (h->d_cnt) cudaFree(h->d_cnt);
        h->d_cnt = nullptr;
        CK(cudaMalloc((void**)&h->d_cnt, n * sizeof(unsigned)));
        CK(cudaMemsetAsync(h->d_cnt, 0, n * sizeof(unsigned), h->stream));
        h->zero_cap = n;
    }
    h->d_nunits = h->d_cnt + 4;
    h->d_hist = h->d_cnt + 8;
    h->d_kept = h->d_hist + h->n_ind + 1;
    h->zero_n = n;
    return 0;
}

static int upload_items(garlic_gpu* h, const std::vector<Item>& items)
{
    if (items.size() > h->items_cap) {
        if (dev_alloc(h, &h->d_items, items.size() + 1024)) return 1;
        h->items_cap = items.size() + 1024;
    }
    if (!items.empty()) CK(cudaMemcpyAsync(h->d_items, items.data(), items.size() * sizeof(Item), cudaMemcpyHostToDevice, h->stream));
    return 0;
}

static int upload_indlist(garlic_gpu* h, const int32_t* list, int n, cudaStream_t st = nullptr)
{
    if (!st) st = h->stream;
    if ((size_t)n > h->indlist_cap) {
        if (dev_alloc(h, &h->d_indlist, (size_t)n + 1024)) return 1;
        h->indlist_cap = (size_t)n + 1024;
    }
    CK(cudaMemcpyAsync(h->d_indlist, list, n * sizeof(int), cudaMemcpyHostToDevice, st));
    return 0;
}

static WalkParams base_params(const garlic_gpu* h, int W)
{
    WalkParams P;
    memset(&P, 0, sizeof(P));
    P.geno = h->d_geno; P.row_words = h->row_words;
    P.lut = h->d_lut; P.gl = h->have_gl ? h->d_gl : nullptr; P.freq = h->d_freq; P.gl_stride = h->gl_stride;
    P.ind_list = nullptr; P.n_lanes = h->n_ind; P.W = W; P.thr = 1; P.cutoff = 0; P.tol = 0;
    P.out = h->d_out; P.out_count = h->d_cnt; P.out_cap = h->out_cap; P.amb = h->d_amb; P.amb_cap = h->amb_cap;
    P.hist = nullptr;
    P.dump = nullptr; P.dump_stride = 0; P.dump_step = 1;
    return P;
}

static int ensure_weighted(garlic_gpu* h, int W);   // wlod tables + LD band present for this W
static int launch_any_walk(garlic_gpu* h, const WalkParams& P, const Item* items, int n_items, int weighted, bool roh, bool dump,
                           int tile_snps, const CandList& cl = CandList())
{
    if (weighted) {
        WlodParams Q;
        Q.base = P; Q.wlut = h->d_wlut; Q.invld = h->d_invld; Q.nomut = h->d_nomut; Q.norec = h->d_norec;
        // tolerance-checked fast pass on the FP64 tensor cores; exact mul-then-add sums otherwise (dumps, exact mode,
        // re-evaluation of ambiguous pairs)
        if (P.tol > 0 && roh && !dump && h->wlod_mma && P.W >= kWlodMmaMinW) LAUNCH(launch_wlod_mma(Q, items, n_items, h->have_gl, h->stream));
        else LAUNCH(launch_wlod_walk(Q, items, n_items, h->have_gl, roh, dump, h->stream));
    } else {
        LAUNCH(launch_walk(P, items, n_items, h->have_gl, roh, dump, tile_snps <= kTileSnpsMax ? tile_snps : 0, cl, h->stream));
    }
    return 0;
}

// ---- deferred compaction (K3) and the pruning bound (squeeze.cu, bound.cuh) ----
static bool can_bound(const garlic_gpu* h, int W)
{
    return h->prune && h->tables && !h->have_gl && W >= kBoundMinW && W <= 1280;   // (a piece plus its lead-in must fit the walker's table tile)
}

// Will the pruned pass 2 of window size W run as work units (walk_units_kernel)?  That walker builds its candidates'
// compacted slices itself, so the pass in front of it is the bound alone.  Conservative in the item table's tile (the
// largest an item of kPiece * item_pieces owned SNPs and its W - 1 lead-in windows can need): a false "no" only costs
// the compaction the pass did before.
static bool units_walk(const garlic_gpu* h, int W)
{
    const int span = kPiece * h->item_pieces + W - 2;          // slide steps of the longest item
    return can_bound(h, W) && !bound_partial(W) && 32 * ((span + 31) / 32) + W <= kTileSnpsMax;
}

static int ensure_bound_tables(garlic_gpu* h, int W)
{
    if (h->bound_tables_W == W) return 0;
    const long long n_hw = 16ll * (h->n_pieces + 4);           // 256 (n_pieces + 4) + W + 16 < L + kPad table entries
    if (dev_alloc(h, &h->d_bhw, (size_t)n_hw)) return 1;
    if (dev_alloc(h, &h->d_bflag, (size_t)4)) return 1;
    CK(cudaMemsetAsync(h->d_bflag, 0, 4 * sizeof(int), h->stream));
    LAUNCH(launch_bound_tables(h->d_lut, h->L + kPad, n_hw, h->L, W, h->d_bhw, h->d_bflag, h->stream));
    h->bound_tables_W = W;
    return 0;
}

static SqueezeParams squeeze_params(garlic_gpu* h, bool squeeze, int W)
{
    SqueezeParams Q;
    memset(&Q, 0, sizeof(Q));
    Q.gin = squeeze ? h->d_geno0 : h->d_geno;
    Q.in_words = squeeze ? h->row_words0 : h->row_words;
    Q.gout = h->d_geno; Q.out_words = h->row_words;
    Q.plan_head = h->d_plan_head; Q.plan_seg = h->d_plan_seg; Q.piece_rng = h->d_plan_rng;
    Q.plan_fast = reinterpret_cast<const uint32_t*>(h->d_plan_fast); Q.src = h->d_src; Q.n_kept = h->d_scan + (int)((h->L0 + 1023) / 1024);
    Q.n_ind = h->n_ind;
    Q.hw = h->d_bhw;
    Q.lag = bound_lag(W);
    Q.partial = (W > 0 && bound_partial(W)) ? 1 : 0;
    Q.low_mask = W > 0 ? bound_low_mask(W) : 0u;
    Q.pmax = h->d_pmax; Q.pmax_stride = h->pmax_stride;
    Q.n_pieces = h->n_pieces;
    return Q;
}

static int alloc_pmax(garlic_gpu* h)
{
    h->pmax_stride = ((int64_t)h->n_ind + 31) & ~(int64_t)31;
    return dev_alloc(h, &h->d_pmax, (size_t)h->n_pieces * h->pmax_stride);
}

// The compacted rows are needed now.  W_hint > 0: the caller is about to work with unweighted table-mode windows of
// that size, so the pruning bound for it rides along in the same pass over the matrix.
static int ensure_geno(garlic_gpu* h, int W_hint)
{
    if (!h->geno_pending) return 0;
    // the slack words behind each row are only ever over-read (their lookups are masked), so they need
    // no defined content; a fresh allocation is filled once so that dumps stay reproducible
    const bool fresh = h->cap.find((void*)&h->d_geno) == h->cap.end() || !h->d_geno ||
                       h->cap[(void*)&h->d_geno] < (size_t)h->n_ind * h->row_words * 8;
    if (dev_alloc(h, &h->d_geno, (size_t)h->n_ind * h->row_words)) return 1;
    if (fresh) CK(cudaMemsetAsync(h->d_geno, 0xff, (size_t)h->n_ind * h->row_words * 8, h->stream));
    int c2 = 0;
    if (W_hint > 0 && can_bound(h, W_hint) && h->bound_W != W_hint) {
        if (ensure_bound_tables(h, W_hint)) return 1;
        if (alloc_pmax(h)) return 1;
        c2 = bound_c2(W_hint);
    }
    const SqueezeParams Q = squeeze_params(h, true, W_hint);
    CK(cudaEventRecord(h->ev_sq0, h->stream));
    LAUNCH(launch_squeeze_bound(Q, true, true, c2, h->stream));
    CK(cudaEventRecord(h->ev_sq1, h->stream));
    h->sq_timed = true;
    h->geno_pending = false;
    if (c2) h->bound_W = W_hint;
    return 0;
}

// Items of the pruned pass 2 for window size W: piece-aligned chunks of the segments, uploaded to their own buffer.
// Built once per (tables, W) — windows_common calls this while the GPU is busy with pass 1, call_roh finds them ready.
static int prepare_p2_items(garlic_gpu* h, int W)
{
    if (h->p2_gen == h->tables_gen && h->p2_W == W) return 0;
    if (ensure_stretches(h)) return 1;
    segments_from_stretches(h->stretches, W, h->p2_segs);
    build_items_aligned(h->chr_off, W, h->p2_segs, kPiece * h->item_pieces, h->p2_items);
    h->p2_chunk = 0;
    for (const Item& it : h->p2_items) h->p2_chunk = std::max(h->p2_chunk, it.own_hi - it.own_lo);
    h->p2_tile = items_tile_snps(h->p2_items, W);
    h->p2_slice = items_slice_words(h->p2_items, W);
    if (dev_alloc(h, &h->d_items_p2, h->p2_items.size() + 1)) return 1;
    if (!h->p2_items.empty())
        CK(cudaMemcpyAsync(h->d_items_p2, h->p2_items.data(), h->p2_items.size() * sizeof(Item), cudaMemcpyHostToDevice, h->stream));
    h->p2_gen = h->tables_gen; h->p2_W = W;
    return 0;
}

// Piece maxima for window size W present, without compacting rows where it can: over the compacted rows if they
// exist, else over the uncompacted ones, compacted in registers only.  Window sizes below 32 whose rows are not
// compacted yet take the fused pass instead: their pruned walker (launch_walk) reads compacted rows.
static int ensure_bound(garlic_gpu* h, int W)
{
    if (h->bound_W == W) return 0;
    if (h->geno_pending && bound_partial(W)) return ensure_geno(h, W);
    if (ensure_bound_tables(h, W)) return 1;
    if (alloc_pmax(h)) return 1;
    const bool raw = h->geno_pending;
    const SqueezeParams Q = squeeze_params(h, raw, W);
    CK(cudaEventRecord(h->ev_sq0, h->stream));
    LAUNCH(launch_squeeze_bound(Q, raw, false, bound_c2(W), h->stream));
    CK(cudaEventRecord(h->ev_sq1, h->stream));
    h->sq_timed = true;
    h->bound_W = W;
    return 0;
}

// Thinned pass 1 in table mode (what the KDE needs) does not depend on the compaction: it reads the uncompacted matrix
// through the gather list, on a second stream, while the fused compaction + bound pass runs on the main one — the host
// gets its windows 0.3 ms earlier and has pass 2 enqueued before the compaction is over.
static bool side_pass1(const garlic_gpu* h, int weighted, int exact, int step)
{
    static const bool off = getenv("GARLIC_NO_SIDE_PASS1") != nullptr;
    return !off && !weighted && !exact && step >= 8 && !h->have_gl && h->have_geno0 && h->aux_stream != nullptr;
}
// the side stream starts behind what the main stream holds now (tables, gather list), not behind what follows
static int begin_side(garlic_gpu* h)
{
    CK(cudaEventRecord(h->ev_aux_in, h->stream));
    CK(cudaStreamWaitEvent(h->aux_stream, h->ev_aux_in, 0));
    return 0;
}
// … and the main stream's later work (the KDE on the device, another pass 1) sees the side stream's results
static int end_side(garlic_gpu* h)
{
    CK(cudaEventRecord(h->ev_aux_out, h->aux_stream));
    CK(cudaStreamWaitEvent(h->stream, h->ev_aux_out, 0));
    return 0;
}

extern "C" {

int64_t garlic_gpu_window_slots(garlic_gpu_t* h, int step)
{
    if (!h || !h->filtered || step < 1) return -1;
    int64_t n = 0;
    for (int c = 0; c < h->n_chr; ++c) n += (h->chr_off[c + 1] - h->chr_off[c] + step - 1) / step;
    return n;
}

static int windows_common(garlic_gpu_t* h, int winsize, int step, int weighted, const int32_t* individuals, int n,
                          int exact, double* out, void** out_dev);

int garlic_gpu_windows(garlic_gpu_t* h, int winsize, int step, int weighted, const int32_t* individuals, int n,
                       int exact, double* out)
{
    return windows_common(h, winsize, step, weighted, individuals, n, exact, out, nullptr);
}

int garlic_gpu_windows_dev(garlic_gpu_t* h, int winsize, int step, int weighted, const int32_t* individuals, int n,
                           int exact, void** out_dev)
{
    if (!out_dev) return 1;
    return windows_common(h, winsize, step, weighted, individuals, n, exact, nullptr, out_dev);
}

// Thinned windows of the KDE individuals of ALL shards: this rank computes the windows of its own individuals
// (n <= rows_per_rank local indices), one ncclAllGather on the library's stream collects every rank's
// MISSING-padded [rows_per_rank][n_slots] block, and out receives [world*rows_per_rank][n_slots] (rank order).
int garlic_gpu_windows_gather(garlic_gpu_t* h, int winsize, int step, int weighted, const int32_t* individuals, int n,
                              int rows_per_rank, int exact, double* out)
{
    if (n > rows_per_rank) FAIL("windows_gather: more individuals than rows_per_rank");
    const int64_t slots = garlic_gpu_window_slots(h, step);
    if (slots < 0) FAIL("windows_gather: call filter first");
    void* dptr = nullptr;
    if (n > 0 && windows_common(h, winsize, step, weighted, individuals, n, exact, nullptr, &dptr)) return 1;
    CK(cudaSetDevice(h->device));
    // the exchange follows the windows on their stream (the side stream in table mode: not behind the compaction)
    const bool side = h->filtered && h->tables && side_pass1(h, weighted, exact, step);
    cudaStream_t ws = side ? h->aux_stream : h->stream;
    if (side && n == 0 && begin_side(h)) return 1;
    const size_t blk = (size_t)rows_per_rank * slots;
    if (dev_alloc(h, &h->d_gather, blk * (h->comm_world + 1))) return 1;
    double* send = h->d_gather + blk * h->comm_world;
    LAUNCH(launch_fill_f64(send, blk, kMissing, ws));
    if (n > 0) CK(cudaMemcpyAsync(send, dptr, (size_t)n * slots * sizeof(double), cudaMemcpyDeviceToDevice, ws));
    if (h->comm) NCK(ncclAllGather(send, h->d_gather, blk, ncclDouble, h->comm, ws));
    else CK(cudaMemcpyAsync(h->d_gather, send, blk * sizeof(double), cudaMemcpyDeviceToDevice, ws));
    h->kde_src = h->d_gather; h->kde_src_n = (int64_t)(blk * h->comm_world);
    if (!out) return side ? end_side(h) : 0;   // a rank that only contributes: nothing travels to its host, nobody waits
    const size_t bytes = blk * h->comm_world * sizeof(double);
    const bool direct = is_pinned(out);
    const bool staged = !direct && bytes <= ((size_t)64 << 20) && !pin_alloc(h, bytes);
    CK(cudaMemcpyAsync(direct ? (void*)out : (staged ? (void*)h->pin : (void*)out), h->d_gather, bytes, cudaMemcpyDeviceToHost, ws));
    CK(cudaStreamSynchronize(ws));
    if (side && end_side(h)) return 1;
    if (finish_outputs(h)) return 1;
    if (staged) memcpy(out, h->pin, bytes);
    return 0;
}

static int windows_common(garlic_gpu_t* h, int winsize, int step, int weighted, const int32_t* individuals, int n,
                          int exact, double* out, void** out_dev)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("windows: call set_tables first");
    if (winsize < 2 || winsize > kMaxW) FAIL("windows: winsize out of range [2,4096]");
    if (step < 1) FAIL("windows: step must be >= 1");
    tl_mark(h, "windows:in");
    if (weighted && ensure_weighted(h, winsize)) return 1;
    const int W = winsize;
    const int n_lanes = individuals ? n : h->n_ind;
    if (individuals)
        for (int i = 0; i < n; ++i) if (individuals[i] < 0 || individuals[i] >= h->n_ind) FAIL("windows: individual index out of range");
    const int64_t slots = garlic_gpu_window_slots(h, step);
    // thinned pass 1 (unweighted, tolerance 1e-9): sum only the windows the KDE will look at
    const bool direct = !weighted && !exact && step >= 8;
    const bool side = direct && side_pass1(h, weighted, exact, step);
    cudaStream_t ws = h->stream;                                   // the stream this call's copies to the host run on
    int rc = 0;
    double* d_dump = nullptr;
    if (direct) {
        // Everything this pass reads is on the device already — the table, the gather list, the bad-pair bit map of
        // set_tables — so in table mode (`side`) it goes FIRST, over the uncompacted matrix: its windows travel to the host
        // on the side stream while the main stream runs the fused compaction + bound pass, and the host has pass 2
        // enqueued before that is over.  (GL mode: the likelihood matrix was compacted by filter(); same kernel.)
        if (!side && ensure_geno(h, winsize)) return 1;
        if (individuals && upload_indlist(h, individuals, n)) return 1;
        if (dev_alloc(h, &h->d_dump, (size_t)n_lanes * slots)) return 1;
        d_dump = h->d_dump;
        LAUNCH(launch_fill_f64(d_dump, (size_t)n_lanes * slots, kMissing, h->stream));
        std::vector<int2> meta(h->n_chr);
        int base = 0;
        for (int c = 0; c < h->n_chr; ++c) {
            meta[c].x = (int)h->chr_off[c]; meta[c].y = base;
            base += (int)((h->chr_off[c + 1] - h->chr_off[c] + step - 1) / step);
        }
        if (dev_alloc(h, &h->d_thin, (size_t)2 * h->n_chr + 8)) return 1;
        int2* d_meta = reinterpret_cast<int2*>(h->d_thin);
        CK(cudaMemcpyAsync(d_meta, meta.data(), meta.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
        LAUNCH(launch_thin_windows(side ? h->d_geno0 : h->d_geno, side ? h->row_words0 : h->row_words, h->d_lut,
                                   individuals ? h->d_indlist : nullptr, n_lanes, h->d_badbits, h->L, d_meta, h->n_chr, slots, step, W,
                                   d_dump, slots, h->have_gl ? h->d_gl : nullptr, h->gl_stride, side ? h->d_src : nullptr, h->stream));
        if (side) {
            if (begin_side(h)) return 1;                           // the side stream takes over behind the windows …
            ws = h->aux_stream;
            // … and the main stream goes on with the bound for pass 2, fused with the compaction unless pass 2 will
            // not need compacted rows
            if (units_walk(h, W) ? ensure_bound(h, W) : ensure_geno(h, winsize)) return 1;
        }
        tl_mark(h, "windows:squeeze-enqueued");
        // the GPU is busy: the host gets pass 2's items ready meanwhile
        if (h->bound_W == W && prepare_p2_items(h, W)) return 1;
    } else {
        if (ensure_geno(h, weighted ? 0 : winsize)) return 1;
        if (individuals && upload_indlist(h, individuals, n)) return 1;
        std::vector<Segment> segs;
        std::vector<Item> items;
        if (ensure_stretches(h)) return 1;                 // (the compaction above is already on the stream)
        segments_from_stretches(h->stretches, W, segs);
        if (dev_alloc(h, &h->d_dump, (size_t)n_lanes * slots)) return 1;
        d_dump = h->d_dump;
        LAUNCH(launch_fill_f64(d_dump, (size_t)n_lanes * slots, kMissing, h->stream));
        int chunk = 0;
        if (weighted) chunk = std::max(64, pick_chunk(h->L, W, n_lanes, 0) / 8);   // every wLOD window is a fresh sum
        else if (!exact) chunk = pick_chunk(h->L, W, n_lanes, h->have_gl ? 0 : kTileSnpsMax);   // GL mode has no table tile
        build_items(h->chr_off, W, segs, chunk, step, items);
        if (upload_items(h, items)) return 1;
        WalkParams P = base_params(h, W);
        P.ind_list = individuals ? h->d_indlist : nullptr;
        P.n_lanes = n_lanes;
        P.cutoff = 0; P.thr = 1; P.tol = 0;
        P.dump = d_dump; P.dump_stride = slots; P.dump_step = step;
        CK(cudaMemsetAsync(h->d_cnt, 0, 4 * sizeof(unsigned), h->stream));
        rc = launch_any_walk(h, P, h->d_items, (int)items.size(), weighted, false, true, items_tile_snps(items, W));
    }
    if (!rc) { h->kde_src = d_dump; h->kde_src_n = (int64_t)n_lanes * slots; }
    tl_mark(h, "windows:enqueued");
    if (!rc && finish_outputs(h)) rc = 1;
    if (!rc && out_dev) {
        *out_dev = d_dump;
        cudaError_t e = cudaStreamSynchronize(ws);
        if (e != cudaSuccess) { h->err = std::string("windows: ") + cudaGetErrorString(e); rc = 1; }
    } else if (!rc) {
        const size_t bytes = (size_t)n_lanes * slots * sizeof(double);
        const bool staged = !is_pinned(out) && bytes <= ((size_t)64 << 20) && !pin_alloc(h, bytes);
        cudaError_t e = cudaMemcpyAsync(staged ? (void*)h->pin : (void*)out, d_dump, bytes, cudaMemcpyDeviceToHost, ws);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ws);
        if (e != cudaSuccess) { h->err = std::string("windows: ") + cudaGetErrorString(e); rc = 1; }
        else if (staged) memcpy(out, h->pin, bytes);
    }
    tl_mark(h, "windows:out");
    return rc;
}

int garlic_gpu_kde(garlic_gpu_t* h, const double* values, int64_t n_values, int m_targets, double* x, double* y,
                   int64_t* n_used, double* bandwidth)
{
    CK(cudaSetDevice(h->device));
    if (m_targets < 2 || m_targets > 1024) FAIL("kde: number of targets out of range [2,1024]");
    if (!x || !y) FAIL("kde: null output");
    const double* src = h->kde_src;
    int64_t n = h->kde_src_n;
    if (values) {
        if (n_values < 1) FAIL("kde: no values");
        if (dev_alloc(h, &h->d_kde_in, (size_t)n_values)) return 1;
        CK(cudaMemcpyAsync(h->d_kde_in, values, (size_t)n_values * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        src = h->d_kde_in; n = n_values;
    }
    if (!src || n < 1) FAIL("kde: no window matrix on the device (call garlic_gpu_windows first, or pass values)");
    if (dev_alloc(h, &h->d_kde, kde_scratch_doubles(m_targets))) return 1;
    double* d_res = nullptr;
    int launches = 0;
    CK(launch_kde(src, (long long)n, m_targets, h->d_kde, &d_res, &launches, h->stream));
    h->launches += launches;
    const size_t bytes = (size_t)(8 + 2 * m_targets) * sizeof(double);
    if (pin_alloc(h, bytes)) return 1;
    CK(cudaMemcpyAsync(h->pin, d_res, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (finish_outputs(h)) return 1;
    const double* r = reinterpret_cast<const double*>(h->pin);
    if (n_used) *n_used = (int64_t)r[0];
    if (bandwidth) *bandwidth = r[5];
    if (r[0] < 2) FAIL("kde: fewer than two valid window values");
    memcpy(x, r + 8, (size_t)m_targets * sizeof(double));
    memcpy(y, r + 8 + m_targets, (size_t)m_targets * sizeof(double));
    return 0;
}

int garlic_gpu_call_roh(garlic_gpu_t* h, int winsize, double cutoff, double overlap_frac, int weighted, int exact,
                        garlic_roh_t* out, int64_t cap, int64_t* count)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("call_roh: call set_tables first");
    if (winsize < 2 || winsize > kMaxW) FAIL("call_roh: winsize out of range [2,4096]");
    // MISSING windows must fail the cutoff test (garlic-roh.cpp:450); at or below the sentinel the
    // reference overruns inWin[] (:452), so there is no behaviour to reproduce
    if (!(cutoff > kMissing)) FAIL("call_roh: LOD cutoff must be greater than the MISSING sentinel (-9999)");
    if (weighted && ensure_weighted(h, winsize)) return 1;
    const int W = winsize;
    Laps laps("call_roh");
    laps.rank = h->comm_rank;
    tl_mark(h, "call_roh:in");
    // pruned pass (bound.cuh): unweighted table mode, window sizes the bound covers, cutoffs inside its fixed-point range
    int cut_ok = 0;
    bound_cut_store(cutoff, 1.0, &cut_ok);
    bool prune = !exact && !weighted && can_bound(h, W) && cut_ok;
    // the bound, and the compacted rows unless the pruned walker will build its own slices (checked again below)
    if (prune && units_walk(h, W) ? ensure_bound(h, W) : ensure_geno(h, prune ? W : 0)) return 1;
    // garlic-roh.cpp:422-424, compared against integers at :466 and :477
    double thr_d = overlap_frac * W;
    thr_d = (thr_d >= 1) ? thr_d : 1;
    thr_d = (thr_d <= W) ? thr_d : W;
    const int thr = (int)std::ceil(thr_d);

    std::vector<Segment> segs;
    std::vector<Item> items;
    if (ensure_stretches(h)) return 1;
    segments_from_stretches(h->stretches, W, segs);
    int chunk = 0;
    // weighted windows are fresh sums: a chunk only pays its W-1 lead-in windows, so chunks are kept long for the
    // tensor-core pass and short (more parallel items) for the exact kernel
    if (weighted) chunk = (!exact && h->wlod_mma && W >= kWlodMmaMinW) ? std::max(256, pick_chunk(h->L, W, h->n_ind, 0) / 2)
                                                                      : std::max(64, pick_chunk(h->L, W, h->n_ind, 0) / 8);
    else if (!exact) chunk = pick_chunk(h->L, W, h->n_ind, h->have_gl ? 0 : kTileSnpsMax);
    if (prune) {
        if (prepare_p2_items(h, W)) return 1;
        prune = h->p2_tile <= kTileSnpsMax && (int64_t)h->p2_items.size() * h->n_ind < (1ll << 31);
        if (prune) chunk = h->p2_chunk;
    }
    if (!(prune && !bound_partial(W)) && ensure_geno(h, 0)) return 1;   // every walker but the work units reads compacted rows
    const Item* d_its = h->d_items;                    // the items in use: the cached piece-aligned ones, or `items`
    const std::vector<Item>* its = &items;
    if (prune) {
        d_its = h->d_items_p2; its = &h->p2_items;
    } else {
        build_items(h->chr_off, W, segs, chunk, 0, items);
        if (upload_items(h, items)) return 1;
        d_its = h->d_items;                            // (the upload may have moved the buffer)
    }
    int64_t n_win = 0;
    for (const Segment& s : segs) n_win += s.we - s.ws;
    // note: the reference also "evaluates" invalid window starts (they come out MISSING); the unit
    // of work N·Σ_c(L_c-W+1) counts those too (SURVEY §8)
    int64_t units = 0;
    for (int c = 0; c < h->n_chr; ++c) units += std::max<int64_t>(0, h->chr_off[c + 1] - h->chr_off[c] - W + 1);
    units *= h->n_ind;

    if (!h->d_out) {
        h->out_cap = 1u << 22;
        if (dev_alloc(h, &h->d_out, h->out_cap)) return 1;
        h->amb_cap = 1u << 16;
        if (dev_alloc(h, &h->d_amb, h->amb_cap)) return 1;
    }
    laps.lap("items");
    std::vector<RohRec>&recs = h->recs_buf, &ambs = h->ambs_buf;
    recs.clear(); ambs.clear();
    size_t n_stage = 0;            // records waiting in the pinned staging buffer
    bool done = false;
    float ms = 0, ms_select = 0;
    bool pruned = false;
    double n_cand = -1.0;
    for (int attempt = 0; attempt < 3; ++attempt) {
        WalkParams P = base_params(h, W);
        P.cutoff = cutoff; P.thr = thr;
        if (!exact && !weighted) {
            // |fast − reference chain| ≤ |reference chain − exact sum| + |chunked chain − exact sum|
            //   ≤ (longest + W)·2ε·(W+1)·amax + (chunk + 2W)·2ε·(W+1)·amax,  2ε = 2^-52 — see DESIGN.md §5
            int64_t longest = 0;
            for (const Segment& s : segs) longest = std::max<int64_t>(longest, s.we - s.ws);
            P.tol = (double)(longest + chunk + 3 * W) * 2.220446049250313e-16 * (W + 1) * h->amax;
        }
        if (!exact && weighted && h->wlod_mma && W >= kWlodMmaMinW) {
            // |DMMA sum − reference mul-then-add sum| ≤ (W+8)·2ε·W·amax: scores are bounded by amax (nomut, norec ≤ 1)
            // and 1/LD ≤ 1 because every LD sum contains the diagonal term 1 (garlic-data.cpp:521-527)
            P.tol = (double)(W + 8) * 2.0 * 2.220446049250313e-16 * W * h->amax;
        }
        if (ensure_zero_block(h)) return 1;
        CK(cudaMemsetAsync(h->d_cnt, 0, h->zero_n * sizeof(unsigned), h->stream));
        P.out_count = h->d_cnt;
        // pruned pass: the piece maxima (computed with the compaction, or now) are thresholded into dense per-item
        // candidate lists and a queue of work units; the walker below only visits those
        const int tile_snps = prune ? h->p2_tile : items_tile_snps(*its, W);
        const bool prune_now = prune && !exact;
        const int n_its = (int)its->size();
        CandList cl;
        unsigned unit_cap = 0;
        CK(cudaEventRecord(h->ev0, h->stream));
        if (prune_now) {
            if (ensure_bound(h, W)) return 1;
            int ok = 0;
            const int cut_store = bound_cut_store(cutoff, P.tol, &ok);
            const int per_item = (h->n_ind + kUnitThreads - 1) / kUnitThreads;
            unit_cap = (unsigned)std::min<int64_t>((int64_t)n_its * per_item, 1ll << 28);
            if (dev_alloc(h, &h->d_cand_list, (size_t)n_its * h->n_ind)) return 1;
            if (dev_alloc(h, &h->d_cand_cnt, (size_t)n_its + 1)) return 1;
            if (dev_alloc(h, &h->d_units, (size_t)unit_cap)) return 1;
            LAUNCH(launch_select(d_its, n_its, h->d_pmax, h->pmax_stride, h->n_ind, cut_store, h->d_bflag,
                                 h->d_cand_list, h->n_ind, h->d_cand_cnt, h->d_units, h->d_nunits, unit_cap, kUnitThreads, bound_c2(W), h->stream));
            cl.list = h->d_cand_list; cl.cnt = h->d_cand_cnt; cl.stride = h->n_ind;
        }
        CK(cudaEventRecord(h->ev2, h->stream));
        // run records are bucketed by individual, ordered, stitched and packed on the device
        // (kernels.cu:launch_bucket_by_individual): the final runs end up dense in d_out, their number in d_cnt[2]
        if (dev_alloc(h, &h->d_sorted, (size_t)h->out_cap)) return 1;
        P.hist = h->d_hist;
        // window sizes below 32 leave a quarter of the pairs (a short window is homozygous by chance often enough): eight-warp
        // CTAs over the candidate lists share one table tile among 256 candidates, where a work unit would stage it for 64
        if (prune_now && !bound_partial(W)) {
            RawRows R;                                 // (the compacted rows, if another consumer has made them)
            R.rows = h->geno_pending ? h->d_geno0 : nullptr; R.row_words = h->row_words0;
            R.head = h->d_plan_head; R.segs = h->d_plan_seg; R.L = h->L;
            LAUNCH(launch_walk_units(P, R, d_its, h->d_units, h->d_nunits, unit_cap, tile_snps, h->p2_slice, cl, h->stream));
        }
        else if (prune_now) LAUNCH(launch_walk(P, d_its, n_its, false, true, false, tile_snps, cl, h->stream));
        else if (launch_any_walk(h, P, d_its, n_its, weighted, true, false, tile_snps)) return 1;
        CK(cudaEventRecord(h->ev1, h->stream));
        LAUNCH(launch_bucket_by_individual(h->d_out, h->d_cnt, h->out_cap, h->d_hist, h->n_ind, h->d_sorted, thr, h->d_kept,
                                           h->d_cnt + 2, h->stream));
        // one synchronisation: the counters and — speculatively, sized by the previous call — the final runs and the
        // ambiguous pairs travel together; only a larger result costs a second copy
        const size_t guess = std::min<size_t>(h->out_cap, std::max<size_t>(4096, h->last_final + h->last_final / 4));
        const size_t amb_guess = 256;
        if (pin_alloc(h, 64 + (guess + std::max<size_t>(amb_guess, h->amb_cap)) * sizeof(RohRec))) return 1;
        unsigned* cnt = reinterpret_cast<unsigned*>(h->pin);
        RohRec* stage = reinterpret_cast<RohRec*>(h->pin + 64);
        CK(cudaMemcpyAsync(cnt, h->d_cnt, 4 * sizeof(unsigned), cudaMemcpyDeviceToHost, h->stream));
        cnt[4] = 0; cnt[5] = 0;                                // work units / candidate pairs of the pruned pass ride along
        if (prune_now) CK(cudaMemcpyAsync(cnt + 4, h->d_nunits, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(stage, h->d_out, guess * sizeof(RohRec), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(stage + guess, h->d_amb, amb_guess * sizeof(RohRec), cudaMemcpyDeviceToHost, h->stream));
        tl_mark(h, "call_roh:enqueued");
        CK(cudaStreamSynchronize(h->stream));
        if (finish_outputs(h)) return 1;
        tl_mark(h, "call_roh:synced");
        CK(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        CK(cudaEventElapsedTime(&ms_select, h->ev0, h->ev2));
        pruned = prune_now;
        n_cand = prune_now ? (double)cnt[5] : -1.0;
        const unsigned n_raw = cnt[0], n_amb = cnt[1], n_fin = cnt[2];
        if (n_raw > h->out_cap) {
            h->out_cap = n_raw + n_raw / 4 + 1024;
            if (dev_alloc(h, &h->d_out, h->out_cap)) return 1;
            continue;
        }
        if (n_amb > h->amb_cap) {   // pathological: (nearly) everything ambiguous → exact everywhere
            exact = 1; prune = false;
            if (ensure_geno(h, 0)) return 1;
            build_items(h->chr_off, W, segs, 0, 0, items);
            if (upload_items(h, items)) return 1;
            d_its = h->d_items; its = &items;
            continue;
        }
        recs.resize(n_fin);
        ambs.resize(n_amb);
        if (n_fin) memcpy(recs.data(), stage, std::min<size_t>(n_fin, guess) * sizeof(RohRec));
        if (n_fin > guess) CK(cudaMemcpy(recs.data() + guess, h->d_out + guess, (n_fin - guess) * sizeof(RohRec), cudaMemcpyDeviceToHost));
        if (n_amb) memcpy(ambs.data(), stage + guess, std::min<size_t>(n_amb, amb_guess) * sizeof(RohRec));
        if (n_amb > amb_guess) CK(cudaMemcpy(ambs.data() + amb_guess, h->d_amb + amb_guess, (n_amb - amb_guess) * sizeof(RohRec), cudaMemcpyDeviceToHost));
        n_stage = n_raw;
        h->last_final = n_fin;
        done = true;
        break;
    }
    if (!done) FAIL("call_roh: record buffers still overflowing after three attempts");
    laps.lap("kernel+d2h");
    // exact re-evaluation of (individual, segment) pairs that had a window within rounding
    // distance of the cutoff: one whole-segment launch per distinct segment
    int64_t n_amb_pairs = 0;
    if (!ambs.empty()) {
        if (ensure_geno(h, 0)) return 1;                  // whole-segment chains read compacted rows
        std::map<int, std::vector<int>> by_seg;
        for (const RohRec& a : ambs) by_seg[a.tag].push_back(a.ind);
        std::vector<RohRec> fixed;
        for (auto& kv : by_seg) {
            std::vector<int>& inds = kv.second;
            std::sort(inds.begin(), inds.end());
            inds.erase(std::unique(inds.begin(), inds.end()), inds.end());
            n_amb_pairs += (int64_t)inds.size();
            std::vector<Segment> one(1, segs[kv.first]);
            std::vector<Item> its;
            build_items(h->chr_off, W, one, 0, 0, its);
            its[0].seg = kv.first;
            if (upload_items(h, its)) return 1;
            if (upload_indlist(h, inds.data(), (int)inds.size())) return 1;
            WalkParams P = base_params(h, W);
            P.cutoff = cutoff; P.thr = thr; P.tol = 0;
            P.ind_list = h->d_indlist; P.n_lanes = (int)inds.size();
            CK(cudaMemsetAsync(h->d_cnt, 0, 4 * sizeof(unsigned), h->stream));
            if (launch_any_walk(h, P, h->d_items, 1, weighted, true, false, items_tile_snps(its, W))) return 1;
            unsigned cnt[4];
            CK(cudaMemcpyAsync(cnt, h->d_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            if (cnt[0] > h->out_cap) FAIL("call_roh: ROH buffer overflow during exact re-evaluation");
            const size_t base = fixed.size();
            fixed.resize(base + cnt[0]);
            if (cnt[0]) CK(cudaMemcpy(fixed.data() + base, h->d_out, cnt[0] * sizeof(RohRec), cudaMemcpyDeviceToHost));
            // drop the fast pass's records of these pairs
            recs.erase(std::remove_if(recs.begin(), recs.end(), [&](const RohRec& r) {
                return (r.tag >> 2) == kv.first && std::binary_search(inds.begin(), inds.end(), r.ind);
            }), recs.end());
        }
        recs.insert(recs.end(), fixed.begin(), fixed.end());
    }
    // sort by (individual, start) and stitch runs that were cut at chunk boundaries
    laps.lap("ambiguous");
    // the device's runs are final (ordered, stitched, minimum length applied); with re-evaluated pairs spliced in the
    // host sorts and stitches once more
    std::vector<RohRec>& merged = ambs.empty() ? recs : h->merged_buf;
    if (!ambs.empty()) stitch_runs(recs, thr, merged, &h->stitch_scratch);
    laps.lap("stitch");
    if (laps.on) fprintf(stderr, "[garlic_b200] call_roh: %zu raw records, %zu ambiguous pairs, %zu runs after stitching\n", n_stage, ambs.size(), merged.size());
    const int64_t n_out = (int64_t)merged.size();
    for (int64_t r = 0; r < n_out && r < cap && out; ++r) {
        out[r].ind = merged[r].ind;
        out[r].chr = segs[merged[r].tag >> 2].chr;
        out[r].start_idx = merged[r].a;
        out[r].stop_idx = merged[r].b;
    }
    if (count) *count = n_out;
    h->stats[0] = (double)its->size();
    h->stats[1] = (double)units;
    h->stats[2] = (double)n_amb_pairs;
    h->stats[3] = ms;
    h->stats[4] = ms_select;
    h->stats[5] = pruned ? n_cand : -1;
    h->stats[6] = (double)its->size() * h->n_ind;
    h->stats_items = 0;
    laps.lap("out");
    tl_mark(h, "call_roh:out");
    return 0;
}

int garlic_gpu_last_stats(garlic_gpu_t* h, double* s)
{
    if (h->stats_items > 0) {   // candidate (individual, item) pairs that went to the walker
        unsigned nu[2] = {0, 0};
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpy(nu, h->d_nunits, sizeof(nu), cudaMemcpyDeviceToHost));
        h->stats[5] = (double)nu[1];
        h->stats_items = 0;
    }
    if (h->sq_timed) {          // the last compaction (+ bound) launch
        float ms = 0;
        CK(cudaSetDevice(h->device));
        CK(cudaEventSynchronize(h->ev_sq1));
        CK(cudaEventElapsedTime(&ms, h->ev_sq0, h->ev_sq1));
        h->stats[7] = ms;
    }
    for (int i = 0; i < 8; ++i) s[i] = h->stats[i];
    return 0;
}

int garlic_gpu_get_piece_bounds(garlic_gpu_t* h, int winsize, uint32_t* out, int64_t cap_entries, int64_t* n_pieces)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("get_piece_bounds: call set_tables first");
    if (!can_bound(h, winsize)) FAIL("get_piece_bounds: no bound for this mode / window size (unweighted table mode, winsize >= 16)");
    if (ensure_bound(h, winsize)) return 1;
    if (n_pieces) *n_pieces = h->n_pieces;
    if ((int64_t)h->n_pieces * h->n_ind > cap_entries) FAIL("get_piece_bounds: output buffer too small");
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy2D(out, (size_t)h->n_ind * 4, h->d_pmax, (size_t)h->pmax_stride * 4, (size_t)h->n_ind * 4, (size_t)h->n_pieces,
                    cudaMemcpyDeviceToHost));
    return 0;
}

int garlic_gpu_ld_band(garlic_gpu_t* h, int winsize, const int32_t* ld_individuals, int n_ld, double* out_ld)
{
    CK(cudaSetDevice(h->device));
    if (!h->tables) FAIL("ld_band: call set_tables first");
    if (winsize < 2 || winsize > kMaxW) FAIL("ld_band: winsize out of range [2,4096]");
    if (ensure_geno(h, 0)) return 1;
    const int64_t L = h->L;
    const int W = winsize;
    // sharded run: indices address the whole sample (this rank holds [ind_offset, ind_offset + n_ind))
    int n_total = h->n_ind;
    if (h->comm) {
        int* d_n = reinterpret_cast<int*>(h->d_cnt);
        CK(cudaMemcpyAsync(d_n, &h->n_ind, sizeof(int), cudaMemcpyHostToDevice, h->stream));
        NCK(ncclAllReduce(d_n, d_n, 1, ncclInt32, ncclSum, h->comm, h->stream));
        CK(cudaMemcpyAsync(&n_total, d_n, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    std::vector<int> all;
    if (!ld_individuals) {
        all.resize(n_total);
        for (int i = 0; i < n_total; ++i) all[i] = i;
        ld_individuals = all.data(); n_ld = n_total;
    }
    for (int i = 0; i < n_ld; ++i)
        if (ld_individuals[i] < 0 || ld_individuals[i] >= n_total) {
            h->err = "ld_band: individual index " + std::to_string(ld_individuals[i]) + " out of range [0, " + std::to_string(n_total) + ")";
            return 1;
        }
    if (upload_indlist(h, ld_individuals, n_ld)) return 1;
    Laps laps("ld_band");
    // homFreq over ALL individuals from the reduced counts (garlic-data.cpp:656-676)
    if (reduce_counts(h, true)) return 1;
    if (dev_alloc(h, &h->d_homf, (size_t)L)) return 1;
    LAUNCH(launch_hom_freq(h->d_counts, h->L0, h->d_src, L, h->d_homf, h->stream));
    // zero-padded weight rows (wlod.h); rows of windows that do not exist stay all-zero
    if (dev_alloc(h, &h->d_invld, (size_t)(L + kPad) * inv_stride(W))) return 1;
    CK(cudaMemsetAsync(h->d_invld, 0, (size_t)(L + kPad) * inv_stride(W) * sizeof(double), h->stream));
    LdPhase ph;
    if (h->phased) {
        if (h->bed_input) FAIL("ld_band: --phased needs phased haplotypes, and a PLINK .bed stores unphased genotypes");
        if (!h->d_alleles || !h->d_key) FAIL("ld_band: --phased needs the allele characters (put_alleles / put_tped_text), not pre-packed genotypes");
        ph.alleles = h->d_alleles; ph.key = h->d_key; ph.src = h->d_src; ph.missing = h->missing_char; ph.freq = h->d_freq;
    }
    if (dev_alloc(h, &h->d_ldplanes, ld_planes_words(L, n_ld, h->phased))) return 1;
    if (dev_alloc(h, &h->d_ldpairs, ld_pairs_doubles(L, W))) return 1;
    double* d_ld = nullptr;
    if (out_ld) CK(cudaMalloc(&d_ld, (size_t)L * W * sizeof(double)));
    laps.lap("alloc");
    int launches = 0;
    cudaError_t e = launch_ld_band(h->d_geno, h->row_words, h->d_indlist, n_ld, h->d_homf, h->d_chr_of, h->d_chr_start,
                                   h->n_chr, L, W, h->d_invld, d_ld, h->stream, &launches, h->comm,
                                   h->comm ? h->ind_offset : 0, h->n_ind, h->d_ldplanes, h->d_ldpairs, ph);
    h->launches += launches + 1;
    if (e != cudaSuccess) { if (d_ld) cudaFree(d_ld); h->err = std::string("ld_band: ") + cudaGetErrorString(e); return 1; }
    if (out_ld) {
        e = cudaMemcpyAsync(out_ld, d_ld, (size_t)L * W * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        cudaFree(d_ld);
        if (e != cudaSuccess) { h->err = std::string("ld_band: ") + cudaGetErrorString(e); return 1; }
    }
    CK(cudaStreamSynchronize(h->stream));
    laps.lap("kernels");
    h->have_ld = true; h->ld_W = W;
    return 0;
}

}  // extern "C"

static int ensure_weighted(garlic_gpu* h, int W)
{
    if (h->gpos.empty()) FAIL("weighted: genetic positions were not given to set_tables");
    if (!h->have_ld || h->ld_W != W) FAIL("weighted: call ld_band with this window size first");
    if (!h->d_wlut) {
        const int64_t L = h->L;
        if (dev_alloc(h, &h->d_nomut, (size_t)L + kPad)) return 1;
        if (dev_alloc(h, &h->d_norec, (size_t)L + kPad)) return 1;
        CK(cudaMemsetAsync(h->d_nomut, 0, (size_t)(L + kPad) * sizeof(double), h->stream));
        CK(cudaMemsetAsync(h->d_norec, 0, (size_t)(L + kPad) * sizeof(double), h->stream));
        LAUNCH(launch_wlod_weights(h->d_pos, h->d_gpos, h->d_chr_of, h->d_chr_start, L, h->mu, h->M, h->d_nomut, h->d_norec, h->stream));
        if (dev_alloc(h, &h->d_wlut, (size_t)(L + kPad) * 4)) return 1;
        CK(cudaMemsetAsync(h->d_wlut, 0, (size_t)(L + kPad) * 4 * sizeof(double), h->stream));
        LAUNCH(launch_build_wlut(h->d_lut, h->d_nomut, h->d_norec, L, h->d_wlut, h->stream));
    }
    return 0;
}
