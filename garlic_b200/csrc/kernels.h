// kernels.h — launch wrappers of the hand-written kernels (internal C++ interface; the public
// boundary is the C ABI in include/garlic_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace garlic {

constexpr int kWalkThreads = 256;     // 8 individual groups (warps) of one item per CTA
constexpr int kTileSnpsMax = 1536;    // table tile staged per CTA: 1536 SNPs × 32 B = 48 KB
constexpr int kUnitThreads = 64;      // pruned pass 2: two warps = up to 64 candidate individuals per work unit

// dense per-item individual lists produced by the pruning pass (list == nullptr: every individual)
struct CandList {
    const int* list = nullptr;       // [n_items][stride]
    const unsigned* cnt = nullptr;   // [n_items]
    int stride = 0;
};

// tile_snps > 0: every item touches at most tile_snps SNPs → stage its table slice in shared memory
cudaError_t launch_walk(const WalkParams& P, const Item* items, int n_items, bool gl_mode, bool roh,
                        bool dump, int tile_snps, const CandList& cl, cudaStream_t st);
// The uncompacted rows and the compaction plan (bound.cuh:plan_half), from which the pruned walker builds the
// compacted slices of its candidates (bound.cuh:plan_slice)
struct RawRows {
    const uint64_t* rows;      // [n_ind][row_words] uncompacted
    int64_t row_words;
    const uint4* head;         // plan head per output half-word
    const uint4* segs;         // [n_q][kPlanSegMax] plan segments
    long long L;               // kept SNPs
};
// the walker over the queue of (item, 64 candidates) work units left by the bound (squeeze.cu); every lane reads its
// candidate's compacted words [w0 >> 5, that + slice_words) from a slice it builds out of R first (R.rows == nullptr:
// from the compacted rows P.geno instead)
cudaError_t launch_walk_units(const WalkParams& P, const RawRows& R, const Item* items, const int2* units, const unsigned* n_units,
                              unsigned unit_cap, int tile_snps, int slice_words, const CandList& cl, cudaStream_t st);

// K3 + pruning bound, fused (squeeze.cu, bound.cuh)
struct SqueezeParams {
    const uint64_t* gin;       // rows to read: the uncompacted matrix (squeeze) or the compacted one (bound only)
    int64_t in_words;
    uint64_t* gout;            // compacted rows (squeeze)
    int64_t out_words;
    const uint4* plan_head;    // compaction plan per output half-word (bound.cuh:plan_half): the slow path's
    const uint4* plan_seg;
    const uint32_t* plan_fast; // two-byte codes of the branch-free path (bound.cuh:plan_fast_code), two per word
    const int2* piece_rng;     // per piece: first input half-word it reads; span << 16 | bit mask of slow-path half-words
    const int* src;            // gather list (kept SNP -> source SNP)
    const int* n_kept;         // device-resident number of kept SNPs
    int n_ind;
    const uint4* hw;           // bound tables per half-word (bound.cuh:bound_hw_entry; w = Bmax of block q - C2)
    int lag;                   // C2 - c1: 1 or 2
    int partial;               // window sizes below 32: partial-half-word core (bound.cuh)
    uint32_t low_mask;         // bound_low_mask(W)
    uint32_t* pmax;            // [n_pieces][pmax_stride]: piece maxima per individual (bound.cuh:bound_pack)
    int64_t pmax_stride;
    int n_pieces, pieces_per_task, n_col_tasks;
};
// n_tab: entries the table holds (L + padding); entries beyond read as zero
cudaError_t launch_bound_tables(const double* lut, long long n_tab, long long n_hw, long long L, int W, uint4* hw, int* invalid, cudaStream_t st);
cudaError_t launch_plan(const int* src, const int* n_kept, long long n_q, uint4* head, uint4* segs, uint16_t* fast,
                        int2* piece_rng, cudaStream_t st);
// c2 > 0: with the bound for that window size class; squeeze = false: bound only, over compacted rows;
// squeeze and not store: bound only, over the uncompacted rows (compacted in registers, nothing written)
cudaError_t launch_squeeze_bound(SqueezeParams P, bool squeeze, bool store, int c2, cudaStream_t st);
cudaError_t launch_select(const Item* items, int n_items, const uint32_t* pmax, int64_t stride, int n_ind, int cut_store,
                          const int* invalid, int* cand_list, int cand_stride, unsigned* cand_cnt, int2* units, unsigned* n_units,
                          unsigned unit_cap, int lanes_per_unit, int c2, cudaStream_t st);
cudaError_t launch_thin_windows(const uint64_t* geno, int64_t row_words, const double* lut, const int* ind_list, int n_lanes,
                                const uint32_t* bad_bits, long long L, const int2* meta, int n_chr, long long n_slots, int step, int W,
                                double* dump, int64_t dump_stride, const double* gl, int64_t gl_stride, const int* src, cudaStream_t st);
cudaError_t launch_fill_f64(double* p, size_t n, double v, cudaStream_t st);
cudaError_t launch_bucket_by_individual(RohRec* in, const unsigned* count, unsigned cap, unsigned* hist, int n_ind,
                                        RohRec* out, int thr, unsigned* kept, unsigned* total, cudaStream_t st);
cudaError_t launch_tokenize_tped(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, uint8_t* alleles,
                                 int* nonblank, cudaStream_t st);
// vcf.cu: VCF sample columns → allele index bytes (255 = missing) and per record the column count, the largest allele
// index (-1 if none) and the first column whose GT is malformed (-1 if none)
cudaError_t launch_tokenize_vcf(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, uint8_t* alleles,
                                int* n_cols, int* max_allele, int* bad_col, cudaStream_t st);
cudaError_t launch_first_allele(const uint8_t* alleles, int n_snp, int n_ind, int ind_offset, int missing,
                                unsigned long long* key, cudaStream_t st);
cudaError_t launch_code_alleles(const uint8_t* alleles, int n_snp, int n_ind, int missing,
                                const unsigned long long* key, long long snp0, uint64_t* geno,
                                int64_t row_words, int* counts, long long L0, cudaStream_t st);
cudaError_t launch_count_packed(const uint64_t* geno, int64_t row_words, int n_ind, long long L0,
                                int* counts, cudaStream_t st);
// bed.cu: PLINK .bed rows staged SNP-major ([n_snp][stride] bytes, this rank's individual i at field sh + i)
cudaError_t launch_bed_count(const uint8_t* stage, int64_t stride, int n_snp, int sh, int n_ind, int ind_offset,
                             int* counts, long long L0, unsigned long long* key, cudaStream_t st);
cudaError_t launch_bed_code(const uint8_t* stage, int64_t stride, long long L0, int sh, int n_ind,
                            const unsigned long long* key, int* counts, uint32_t* a1_words, uint64_t* geno,
                            int64_t row_words, cudaStream_t st);
cudaError_t launch_freq_keep(const int* counts, long long L0, const int* pos, const int* chr_of,
                             const int* chr_param, int oob, double* freq, uint8_t* keep, cudaStream_t st);
cudaError_t launch_keep_scan(const uint8_t* keep, long long L0, const int* chr_of0, int n_chr, int* block_counts,
                             int* total, int* src, int* chr_off_kept, cudaStream_t st);
cudaError_t launch_bad_pairs(const int* pos, const int* chr_of, const int* cen, int max_gap, long long L, int* list,
                             unsigned* count, unsigned cap, uint32_t* bad_bits, cudaStream_t st);
cudaError_t launch_gather_i32(const int* in, const int* src, long long L, int* out, cudaStream_t st);
cudaError_t launch_compact_gl(const double* in, int64_t in_stride, const int* src, long long L, const uint64_t* geno0,
                              int64_t row_words0, const double* freq0, double* out, int64_t out_stride, int n_ind, int type,
                              cudaStream_t st);
cudaError_t launch_gather_f64(const double* in, const int* src, long long L, double* out, cudaStream_t st);
cudaError_t launch_build_lut(const double* freq, long long L, double error, double* lut, cudaStream_t st);
cudaError_t launch_wlod_weights(const int* pos, const double* gpos, const int* chr_of, const int* chr_start,
                                long long L, double mu, int M, double* nomut, double* norec, cudaStream_t st);
cudaError_t launch_build_wlut(const double* lut, const double* nomut, const double* norec, long long L,
                              double* wlut, cudaStream_t st);
// K0-GL (ingest.cu): tgls value columns from raw text into the individual-major matrix out[(k - ind_lo) * out_stride + snp0 + l]
cudaError_t launch_tokenize_tgls(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, double* out,
                                 int64_t out_stride, long long snp0, int* n_tokens, int2* hard_list, unsigned* hard_count,
                                 unsigned hard_cap, cudaStream_t st);
// the counter exchange over NVLink peer memory, fused with freq + keep (xchg.cu)
constexpr int kXchgMaxRanks = 16, kXchgReady = 0, kXchgDone = 16;   // flag words per rank: ready[16] | done[16]
struct XchgParams {
    int* counts[kXchgMaxRanks];        // every rank's counters [4][L0] (rows 0, 1 are exchanged)
    double* freq[kXchgMaxRanks];       // every rank's freq0[L0]
    uint8_t* keep[kXchgMaxRanks];      // every rank's keep[L0]
    unsigned* flags[kXchgMaxRanks];    // every rank's flag words
    int n, rank;
    unsigned seq;                      // call number, the same on every rank
    long long L0;
    const int* pos; const int* chr_of; const int* chr_param; int oob;
    unsigned* done_counter;            // local: CTAs of this launch that have finished their slice
};
cudaError_t launch_xchg_freq_keep(const XchgParams& P, cudaStream_t st);
// computeKDE on the device (kde.cu): scratch size in doubles; out → state[8] | x[m] | y[m] inside the scratch
size_t kde_scratch_doubles(int m);
cudaError_t launch_kde(const double* v, long long n, int m, double* scratch, double** out, int* launches, cudaStream_t st);

}  // namespace garlic
