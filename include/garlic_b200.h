/*
 * garlic_b200.h — C ABI of the B200-native GARLIC hot path (libgarlic_b200.so).
 *
 * GARLIC (szpiech/garlic v1.1.6a) has no FFI of its own: the hot path sits between the loaders
 * and the writers inside main() (reference src/garlic-main.cpp:216-406).  Each entry point below
 * replaces one of those calls; the reference-side binding a maintainer would add is shown in
 * INTEGRATION.md.  Conventions: opaque handle, plain pointers and sizes, int status return
 * (0 = ok, non-zero = error, text via garlic_gpu_last_error), no exceptions cross the boundary,
 * caller-owned HOST buffers unless a name ends in _dev.  One handle drives one GPU; multi-GPU
 * runs use one process (and one handle) per GPU and shard by individual (DESIGN.md §7).
 *
 * There is no CPU fallback: every compute entry point launches hand-written sm_100a kernels and
 * fails if no CUDA device is usable.
 */
#ifndef GARLIC_B200_H
#define GARLIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct garlic_gpu garlic_gpu_t;

#define GARLIC_MISSING (-9999.0)   /* reference MISSING sentinel for windows (garlic-data.h) */

/* genotype-likelihood encodings, reference readTGLSData (src/garlic-data.cpp:1557-1570) */
#define GARLIC_GL_GQ 0
#define GARLIC_GL_GL 1
#define GARLIC_GL_PL 2
#define GARLIC_GL_ERROR (-1)   /* values are already per-genotype error rates */

/* One ROH as the reference stores it in ROHData (src/garlic-roh.h:43-50), plus SNP indices. */
typedef struct {
    int32_t ind;        /* individual index (local to this handle) */
    int32_t chr;        /* chromosome index */
    int32_t start_idx;  /* index of first SNP in the filtered, concatenated SNP axis */
    int32_t stop_idx;   /* index of last SNP (inclusive) */
} garlic_roh_t;

/* ---- lifecycle -------------------------------------------------------------------------- */
int garlic_gpu_create(int device, garlic_gpu_t **out);
void garlic_gpu_destroy(garlic_gpu_t *h);
const char *garlic_gpu_last_error(const garlic_gpu_t *h);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
uint64_t garlic_gpu_launch_count(const garlic_gpu_t *h);
/* CUDA stream (cudaStream_t) all kernels of this handle are launched on */
void *garlic_gpu_stream(const garlic_gpu_t *h);
int garlic_gpu_sync(garlic_gpu_t *h);
/* page-locked host memory: buffers from here are read / written by the copy engine without staging
 * (put_packed, filter's freq_out / keep_out); ordinary memory works everywhere, only slower */
void *garlic_gpu_host_alloc(size_t bytes);
void garlic_gpu_host_free(void *p);

/* ---- multi-GPU: one handle (rank) per GPU, individuals sharded across ranks (DESIGN.md §7) ---------------
 * Rank 0 obtains 128 bytes with garlic_gpu_comm_id and hands them to the other ranks by any channel; every
 * rank then calls garlic_gpu_comm_init.  With a communicator the library performs the path's exchanges itself,
 * on its own stream, over NCCL: SUM all-reduce of the per-SNP counters inside garlic_gpu_filter, MIN all-reduce
 * of the first-allele keys inside garlic_gpu_code_alleles, all-gather in garlic_gpu_windows_gather.  Without
 * one (world = 1) those calls are local and the *_dev accessors below let the caller run the collectives. */
int garlic_gpu_comm_id(uint8_t *id128);
int garlic_gpu_comm_init(garlic_gpu_t *h, const uint8_t *id128, int rank, int world);

/* ---- K1: loadTPEDData's coding + allele counting (src/garlic-data.cpp:103-150) -------------
 * n_ind individuals on this GPU starting at global individual ind_offset; n_loci SNPs before
 * filtering; chr_offsets[n_chr+1] into the SNP axis; pos[n_loci] physical positions. */
int garlic_gpu_set_shape(garlic_gpu_t *h, int n_ind, int ind_offset, int64_t n_loci, int n_chr,
                         const int64_t *chr_offsets, const int32_t *pos);
/* Column selection: columns[n_ind] lists the input columns (individuals of the input, counted from 0) that this handle
 * holds, strictly ascending, each below n_input, the number of individuals the input holds.  put_tped_text,
 * put_vcf_text, put_bcf_gt, put_tgls_text and put_bed / put_bed_dev then store the listed columns (individual i of
 * the handle = input column columns[i]) instead of [ind_offset, ind_offset+n_ind); every column is still parsed, so
 * the per-line diagnostics are those of the whole input.  ind_offset keeps its meaning: the handle's first individual
 * within the analysed sample (the first-allele keys and the LD individual lists address that sample), so a sample of
 * several handles lists disjoint columns.  put_alleles, put_gl, put_packed and their _dev forms receive only this
 * handle's individuals and ignore the selection.  Call after set_shape (which resets the selection) and before the
 * first put_*.  Fails on an unsorted or out-of-range list and after a put_*. */
int garlic_gpu_select_columns(garlic_gpu_t *h, const int32_t *columns, int n_input);
/* alleles: [n_snp][n_ind][2] characters for SNPs [snp0, snp0+n_snp), snp0 % 32 == 0.
 * Uploads them and records, per SNP, the first non-missing allele in file order (phase a). */
int garlic_gpu_put_alleles(garlic_gpu_t *h, const uint8_t *alleles, int64_t snp0, int n_snp, char missing);
/* device pointer to the uint64 first-allele keys [n_loci]; with several GPUs, MIN-all-reduce it
 * between put_alleles and code_alleles */
void *garlic_gpu_first_allele_keys_dev(garlic_gpu_t *h);
/* phase b: code every call to 2 bits (individual-major packed matrix), count alleles */
/* K0: the same from raw text.  text + line_off[i] .. line_off[i+1] is what follows the 4th field of tped line snp0 + i
 * (blanks, tabs, CR allowed anywhere): its k-th non-blank character is allele k, as `stringstream >> char` reads it
 * (src/garlic-data.cpp:105-133).  Every rank gets the whole line and keeps its own individuals' characters.
 * nonblank (may be NULL): [n_snp] number of non-blank characters found per line, for the caller's column-count check. */
int garlic_gpu_put_tped_text(garlic_gpu_t *h, const char *text, const int64_t *line_off, int64_t snp0, int n_snp,
                             char missing, int32_t *nonblank);
/* PLINK 1 binary genotypes: rows = whole SNP-major .bed rows of SNPs [snp0, snp0+n_snp), snp0 % 32 == 0, of the WHOLE
 * fileset (snp_stride_bytes = ceil(N_total/4): individual i at bits 2(i%4) of byte i/4, PLINK values 0 hom A1,
 * 1 missing, 2 het, 3 hom A2), without the 3 magic bytes.  One cudaMemcpy2DAsync copies only the byte columns that hold
 * this handle's individuals [ind_offset, ind_offset+n_ind); a kernel then records per SNP the first-allele key and the
 * counters (phase a).  The calls are coded as the tped that writes hom A1 "A1 A1", het "A1 A2", hom A2 "A2 A2" and
 * missing "0 0" would be: the "1" allele is A2 iff the first present call over all individuals is hom A2.
 * garlic_gpu_code_alleles then runs the transpose (phase b) and frees the staging rows.  --phased is refused on such
 * a handle (a .bed stores no phase).  _dev: rows on this GPU, complete before the call.  With a column selection the
 * stride must cover ceil(n_input/4) bytes; the rows are copied whole and a kernel gathers the listed columns. */
int garlic_gpu_put_bed(garlic_gpu_t *h, const uint8_t *rows, int64_t snp_stride_bytes, int64_t snp0, int n_snp);
int garlic_gpu_put_bed_dev(garlic_gpu_t *h, const void *rows_dev, int64_t snp_stride_bytes, int64_t snp0, int n_snp);
/* VCF genotypes: text = per record the characters after the FORMAT column's tab (the sample columns, separated by
 * '\t'), record l of the block = text[line_off[l], line_off[l+1]), SNPs [snp0, snp0+n_snp), snp0 % 32 == 0.  Each GT
 * (the start of a sample column, up to ':', '\t' or the end) must be two alleles separated by '/' or '|', each '.' or
 * an allele index 0..254, or a lone '.'; this handle's individuals [ind_offset, ind_offset+n_ind) are stored as allele
 * index bytes, 255 = missing.  A record means exactly the tped line that writes each sample's two alleles in GT order
 * by name (REF for index 0, the k-th ALT for index k, the missing code for '.'), so the "1" allele is the first
 * present allele in file order, half-missing calls count their present allele, and a multi-allelic record is coded
 * "1" allele against the rest.  Phase ('|' or '/') is not checked; --phased reads the alleles in GT order.  The block
 * is pre-filled with 255 and every call synchronises (the caller may reuse text).  Every handle parses every column,
 * so the diagnostics are the same on all ranks; per record (each may be NULL): n_cols = sample columns,
 * max_allele = largest allele index (-1 if none), bad_col = first column whose GT is malformed (-1 if none).  The
 * caller checks them against the header's sample count and the record's ALT count.  Fails on a handle that holds
 * tped or .bed input.  garlic_gpu_code_alleles then codes the block with missing = 255. */
int garlic_gpu_put_vcf_text(garlic_gpu_t *h, const char *text, const int64_t *line_off, int64_t snp0, int n_snp,
                            int32_t *n_cols, int32_t *max_allele, int32_t *bad_col);
/* BCF 2.2 genotypes: per record the GT field's values (n_samples x count values of the width its typed descriptor
 * names), record l of the block at gt + rec_off[l] (rec_off: n_snp + 1 entries, rec_off[l] % 4 == 0, the payloads in
 * ascending order), gt_type[l] = the GT's descriptor byte (count << 4 | type, type 1/2/3 = int8/int16/int32; count 15
 * = 15 or more), SNPs [snp0, snp0+n_snp), snp0 % 32 == 0.  Each value is (allele + 1) << 1 | phased; a call must be two
 * values, each a missing allele (0 or 1) or an allele index 0..254, or a missing allele then end-of-vector (a lone '.'),
 * or a count-1 field whose value is a missing allele.  Phase bits are ignored.  n_samples is the file's sample count:
 * this handle's individuals [ind_offset, ind_offset+n_ind) are stored as allele index bytes, 255 = missing, and a
 * record means exactly the VCF text record with the same GTs (garlic_gpu_put_vcf_text), so the coding, the "1" allele
 * and --phased are the same.  Every handle decodes every sample, so the diagnostics are the same on all ranks; per
 * record (each may be NULL): max_allele = largest allele index (-1 if none), bad_sample = first sample whose GT is
 * malformed (-1 if none).  The caller checks max_allele against the record's ALT count.  Fails on a descriptor of
 * another type or of count 0, a payload shorter than its descriptor needs, an offset that is not a multiple of 4, and
 * a handle that holds tped or .bed input; BCF and VCF text blocks may be mixed on one handle.  Every call
 * synchronises (the caller may reuse its buffers).  garlic_gpu_code_alleles then codes the block with missing = 255. */
int garlic_gpu_put_bcf_gt(garlic_gpu_t *h, const uint8_t *gt, const int64_t *rec_off, const uint8_t *gt_type,
                          int n_samples, int64_t snp0, int n_snp, int32_t *max_allele, int32_t *bad_sample);
/* Call filter of VCF / BCF input (--vcf-min-gq / --vcf-min-dp): a call whose FORMAT GQ is below min_gq, or whose DP is
 * below min_dp, is stored as two missing alleles, so a filtered put means exactly the unfiltered put of the file in
 * which every such call is written ./. (0 = that filter off; both 0 = no filter).  A missing value passes: '.', an
 * empty or omitted trailing subfield, a record without the key, the BCF missing and end-of-vector values.  Call it
 * after set_shape (which turns the filter off) and before the first put_*; it resets the count of calls set missing.
 * Only the _filtered puts below apply it; put_vcf_text and put_bcf_gt never filter. */
int garlic_gpu_set_call_filter(garlic_gpu_t *h, int min_gq, int min_dp);
/* put_vcf_text with the call filter.  fmt_index[2*l] / [2*l+1] = the FORMAT index (GT = 0) of GQ / DP in record l,
 * -1 if its FORMAT lacks the key.  A value is an optional '-', digits, then optionally '.' and digits (I.F passes iff
 * I >= the threshold), or missing; anything else is malformed while its filter is on.  bad_value[l] (may be NULL) =
 * the first sample of record l with a malformed GQ or DP, -1 if none; the GT checks (bad_col, max_allele) apply to
 * every call as written, filtered or not. */
int garlic_gpu_put_vcf_text_filtered(garlic_gpu_t *h, const char *text, const int64_t *line_off, int64_t snp0, int n_snp,
                                     const int32_t *fmt_index, int32_t *n_cols, int32_t *max_allele, int32_t *bad_col,
                                     int32_t *bad_value);
/* put_bcf_gt with the call filter.  Record l's GQ and DP vectors lie in fv[fv_off[l], fv_off[l+1]) (fv_off: n_snp + 1
 * ascending entries, multiples of 4): GQ at fv + fv_off[l] + fv_pos[2*l], DP at + fv_pos[2*l+1] (multiples of 4, -1 if
 * the record lacks the key), with descriptors fv_type[2*l] / [2*l+1].  A filtered field must have count 1 and type
 * int8, int16, int32 or float (5), else the call fails naming the record.  Integers other than the missing / end-of-
 * vector values compare as integers; a float must be finite or one of its two sentinels (0x7F800001, 0x7F800002), an
 * other NaN or an infinity is malformed.  fv may be NULL when fv_off[n_snp] == fv_off[0] (no record of the block holds
 * a GQ or DP vector: every call passes).  bad_value[l] (may be NULL) as for put_vcf_text_filtered. */
int garlic_gpu_put_bcf_gt_filtered(garlic_gpu_t *h, const uint8_t *gt, const int64_t *rec_off, const uint8_t *gt_type,
                                   int n_samples, int64_t snp0, int n_snp, const uint8_t *fv, const int64_t *fv_off,
                                   const int32_t *fv_pos, const uint8_t *fv_type, int32_t *max_allele, int32_t *bad_sample,
                                   int32_t *bad_value);
/* calls of this handle's individuals with at least one present allele that the call filter set missing, since
 * set_call_filter (a call already ./. is not counted) */
uint64_t garlic_gpu_calls_set_missing(const garlic_gpu_t *h);
int garlic_gpu_code_alleles(garlic_gpu_t *h);

/* ---- pre-coded input: packed 2-bit rows (codes 0/1/2, 3 = missing) -------------------------
 * rows: [n_ind][row_stride_bytes] on the host (or, for _dev, on this GPU); SNP s of a row is
 * bits 2*(s%4) of byte s/4.  The library works on its own stream (garlic_gpu_stream): device buffers
 * handed to a _dev entry point must be complete (producer stream synchronised) before the call. */
int garlic_gpu_put_packed(garlic_gpu_t *h, const uint8_t *rows, int64_t row_stride_bytes);
int garlic_gpu_put_packed_dev(garlic_gpu_t *h, const void *rows_dev, int64_t row_stride_bytes);
/* K2: per-SNP allele / missingness / homozygote counts by column reduction of the packed matrix
 * (replaces the counting inside loadTPEDData and calculateGenoFreq, src/garlic-data.cpp:656-676).
 * Optional corrections (may be NULL) add half-missing calls to nalleles / total. */
int garlic_gpu_count_packed(garlic_gpu_t *h, const int32_t *nalleles_corr, const int32_t *total_corr);

/* counts [4][n_loci] int32 on the device: nalleles, total, hom, nonmiss — SUM-all-reduce across
 * GPUs before garlic_gpu_filter. */
void *garlic_gpu_counts_dev(garlic_gpu_t *h);
int garlic_gpu_get_counts(garlic_gpu_t *h, int32_t *nalleles, int32_t *total, int32_t *hom, int32_t *nonmiss);
/* the "1" allele per SNP after code_alleles (missing char if all calls missing).  After put_bed: 1 = the .bim's A1
 * (5th column), 2 = its A2 (6th column), missing if no call is present.  After put_vcf_text: the allele index
 * (0 = REF, k = the k-th ALT), or 255 if no allele is present (pass missing = (char)0xFF); the same after put_bcf_gt */
int garlic_gpu_get_one_allele(garlic_gpu_t *h, uint8_t *allele, char missing);

/* ---- optional per-genotype likelihoods (readTGLSData, src/garlic-data.cpp:1516-1586) -------
 * values: [n_ind][n_loci] (individual-major) raw GQ/GL/PL values; transformed to per-genotype
 * error on the device during garlic_gpu_filter. */
int garlic_gpu_put_gl(garlic_gpu_t *h, const double *values, int gl_type);
int garlic_gpu_put_gl_dev(garlic_gpu_t *h, const void *values_dev, int gl_type);
/* K0-GL: the same matrix from raw text.  text + line_off[i] .. line_off[i+1] is what follows the 4th field of tgls line
 * snp0 + i; its k-th blank-separated token is individual k's value (`ss >> gl`, src/garlic-data.cpp:1538-1554).  Every
 * rank gets the whole line and keeps its own individuals' tokens.  Tokens are converted on the device where one IEEE
 * operation is exact (<= 15 significant digits, |power of ten| <= 22); the few others by the host's strtod, so the
 * values equal the host reader's bit for bit.  n_tokens (may be NULL): [n_snp] tokens found per line, for the caller's
 * column check (:1531-1536).  Call for every SNP range before garlic_gpu_filter. */
int garlic_gpu_put_tgls_text(garlic_gpu_t *h, const char *text, const int64_t *line_off, int64_t snp0, int n_snp,
                             int gl_type, int32_t *n_tokens);

/* the raw likelihood matrix back to the host, [n_ind][n_loci] individual-major, as put_gl / put_tgls_text stored it (parity checks) */
int garlic_gpu_get_gl(garlic_gpu_t *h, double *values);

/* ---- freq + filterMonomorphic[AndOOB]Sites + K3 compaction (src/garlic-data.cpp:141,871-1195)
 * freq = nalleles/total from the (all-reduced) counts; keep iff 0<freq<1 [and, if oob, inside
 * the map scaffold and not strictly inside the centromere]. chr_param: [n_chr][4] =
 * scaffold first bp, scaffold last bp, centromere start, centromere end (NULL if !oob).
 * freq_override (may be NULL): use these frequencies instead (--freq-file).
 * Outputs: freq_out[n_loci] (may be NULL), keep_out[n_loci] (may be NULL); returns L via n_kept.
 * Ordinary host buffers are complete on return.  Page-locked ones (garlic_gpu_host_alloc) are filled by the copy engine
 * behind the call — the path goes on without waiting for 5 MB to cross PCIe — and are complete when the next call that
 * hands data to the host returns (garlic_gpu_windows*, garlic_gpu_call_roh, garlic_gpu_kde) or after garlic_gpu_sync. */
int garlic_gpu_filter(garlic_gpu_t *h, int oob, const int32_t *chr_param, const double *freq_override,
                      double *freq_out, uint8_t *keep_out, int64_t *n_kept);

/* ---- per-SNP tables (K4; lod(), src/garlic-roh.cpp:355-386; inGap/centromeres :11-16) -------
 * centromeres: [n_chr][2] start,end (0,0 if unknown); max_gap as --max-gap. Builds the LOD table
 * on the device from freq and error (ignored when GL data are loaded). gpos (may be NULL):
 * genetic positions [L] of the kept SNPs (needed for --weighted). */
int garlic_gpu_set_tables(garlic_gpu_t *h, double error, int max_gap, const int32_t *centromeres,
                          const double *gpos);
/* host-supplied LOD table [L][4] (g = 0,1,2,missing) replacing the device-built one: the C++ driver uses
 * it to evaluate lod() with the host libm, so whole-segment chains are bit-identical to the reference's */
int garlic_gpu_set_lut(garlic_gpu_t *h, const double *lut);
int garlic_gpu_get_lut(garlic_gpu_t *h, double *lut);
/* homFreq per kept SNP (calculateGenoFreq) from the reduced counts.  With a communicator attached this sums the
 * hom / non-missing counters across ranks first (a collective: every rank calls it, as with garlic_gpu_ld_band) */
int garlic_gpu_get_hom_freq(garlic_gpu_t *h, double *hom_freq);

/* ---- K6: calcLDData / calcHR2LD (src/garlic-data.cpp:330-424,474-527,558-583) ---------------
 * LD individuals (ascending as gsl_ran_choose returns them) or NULL for all.  With a communicator attached
 * (garlic_gpu_comm_init) the indices address the WHOLE sample, every rank passes the same list, and the LD bit-planes
 * of the ranks' shards are combined by one ncclAllReduce inside the call; otherwise they are this handle's rows.
 * out_ld (may be NULL): the LD sums [L][W] as the reference's LDData (rows ≥ L_c-W+1 are 0). */
int garlic_gpu_ld_band(garlic_gpu_t *h, int winsize, const int32_t *ld_individuals, int n_ld, double *out_ld);
/* --phased: the LD band is built from r2 between haplotypes (calcR2LD / r2, src/garlic-data.cpp:426-471,585-617) with
 * the first-copy bit of every call = (first allele character == the "1" allele) (:129); needs allele input. */
int garlic_gpu_set_phased(garlic_gpu_t *h, int phased);
/* wLOD parameters (--mu, --M), call before weighted windows */
int garlic_gpu_set_wlod(garlic_gpu_t *h, double mu, int M);

/* ---- K5 pass 1: windows for the KDE (convert[Subset]WinData2DoubleData, src/garlic-data.cpp:
 * 2026-2150) and --raw-lod --------------------------------------------------------------------
 * Computes windows of the listed individuals (NULL = all) at locus index 0,step,2·step… of each
 * chromosome. out: [n][n_slots] with n_slots = Σ_c ceil(L_c/step), slot order chromosome-major;
 * GARLIC_MISSING where the reference has MISSING. exact != 0: whole-segment chains (bit-identical
 * to the reference's running sums). */
int64_t garlic_gpu_window_slots(garlic_gpu_t *h, int step);
int garlic_gpu_windows(garlic_gpu_t *h, int winsize, int step, int weighted, const int32_t *individuals,
                       int n, int exact, double *out);
/* same, but the [n][n_slots] matrix stays on the GPU (valid until the next windows call): *out_dev receives
 * the device pointer — multi-GPU runs all-gather it before the one copy to the host */
int garlic_gpu_windows_dev(garlic_gpu_t *h, int winsize, int step, int weighted, const int32_t *individuals,
                           int n, int exact, void **out_dev);
/* the KDE individuals of ALL ranks: this rank computes its n <= rows_per_rank local individuals, one all-gather
 * collects every rank's MISSING-padded block; out: [world*rows_per_rank][n_slots] in rank order, or NULL on ranks that
 * only contribute (the gathered matrix stays on their GPU, the call does not wait) */
int garlic_gpu_windows_gather(garlic_gpu_t *h, int winsize, int step, int weighted, const int32_t *individuals,
                              int n, int rows_per_rank, int exact, double *out);

/* ---- computeKDE on the device (src/garlic-kde.cpp:14-101, nrd0 :130-140; SURVEY §8f.4) --------------------------
 * Density of the window values pass 1 left on this GPU — values == NULL: the matrix of the last garlic_gpu_windows /
 * _windows_dev / _windows_gather call, MISSING and NaN slots skipped in place — or of n_values host values.
 * Bandwidth = nrd0 (gsl_stats_sd, gsl quantiles), m_targets (the reference: 512; 2..1024) equally spaced targets
 * from min - 3h to max + 3h, and the Gauss transform  y[j] = sum_i (1/n) exp(-(x[j] - v_i)^2 / h^2)  evaluated
 * exactly (the sum FIGTree approximates to eps = 1e-2 for the reference).  x[m], y[m] (not yet divided by
 * sum(y) * spacing: garlic-kde.cpp:86-95 stays with the caller), *n_used values, *bandwidth = h.  Reproducible:
 * every reduction runs in a fixed order. */
int garlic_gpu_kde(garlic_gpu_t *h, const double *values, int64_t n_values, int m_targets, double *x, double *y,
                   int64_t *n_used, double *bandwidth);

/* ---- K5 pass 2: calc[w]LODWindows + assembleROHWindows fused (src/garlic-roh.cpp:279-347,409-546)
 * overlap_frac as --overlap-frac. out: capacity cap records, sorted by (ind, chr, start);
 * *count receives the number of ROH (may exceed cap: call again with a larger buffer).
 * exact: 0 = chunked fast pass + exact re-evaluation of windows within rounding distance of the
 * cutoff (same ROH as exact), 1 = whole-segment chains everywhere. */
int garlic_gpu_call_roh(garlic_gpu_t *h, int winsize, double cutoff, double overlap_frac, int weighted,
                        int exact, garlic_roh_t *out, int64_t cap, int64_t *count);
/* pruning bound of pass 2 on (default) / off: off walks every (individual, item) pair — same ROH, for measurements */
int garlic_gpu_set_prune(garlic_gpu_t *h, int on);
/* statistics of the last call_roh, 8 doubles: [0] items, [1] individual-windows decided (N·Σ_c(L_c-W+1)),
 * [2] ambiguous (individual, segment) pairs re-evaluated exactly, [3] kernel milliseconds of pass 2 (candidate
 * selection + walker), [4] of which selection, [5] (individual, item) pairs that went to the walker (-1: no
 * pruning), [6] all (individual, item) pairs, [7] milliseconds of the last compaction (K3) or pruning-bound launch —
 * the bound alone, over the uncompacted rows, when the pruned pass 2 needs no compacted matrix */
int garlic_gpu_last_stats(garlic_gpu_t *h, double *stats8);
/* the pruning bound of pass 2 (a sufficient test that an individual has NO window >= cutoff in a 256-SNP piece,
 * evaluated from the packed genotypes alone): out [n_pieces][n_ind], per entry two int16 — low = maximum over the
 * piece's 16-SNP blocks of window starts, high = over its last (winsize+14)/16 blocks — in units of 1/64 LOD,
 * rounded up; *n_pieces = ceil(L/256).  Unweighted table mode, 32 <= winsize <= 209.  Introspection / parity tests. */
int garlic_gpu_get_piece_bounds(garlic_gpu_t *h, int winsize, uint32_t *out, int64_t cap_entries, int64_t *n_pieces);

/* packed 2-bit genotype rows back to the host (parity checks; --phased / debugging): filtered = 0 →
 * the matrix as ingested [n_ind][ceil(n_loci/4)], 1 → after compaction [n_ind][ceil(L/4)];
 * row_stride_bytes >= that width. */
int garlic_gpu_get_genotypes(garlic_gpu_t *h, int filtered, uint8_t *rows, int64_t row_stride_bytes);

/* sizes after filtering */
int64_t garlic_gpu_n_kept(const garlic_gpu_t *h);
int garlic_gpu_get_kept_index(garlic_gpu_t *h, int32_t *src_index); /* [L] pre-filter index of kept SNP */

#ifdef __cplusplus
}
#endif
#endif
