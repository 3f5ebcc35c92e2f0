// common.cuh — shared types for the garlic_b200 CUDA path (sm_100a).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GHD __host__ __device__ __forceinline__
#else
#define GHD inline
struct uint2 { unsigned x, y; };   // host-side stand-ins for the CUDA vector types used by shared code
struct int2 { int x, y; };
struct uint4 { unsigned x, y, z, w; };
struct int4 { int x, y, z, w; };
#endif

namespace garlic {

constexpr double kMissing = -9999.0;   // reference MISSING sentinel (garlic-data.h)

// One unit of the segment table (DESIGN.md §4).  A *segment* is a maximal run of valid window
// starts [ws, we) on one chromosome (closed form of garlic-roh.cpp:55-123, SURVEY §3.4); its SNP
// stretch is [ws, we+W-1).  An item is a chunk of a segment; items partition the stretch into
// owned SNP ranges [own_lo, own_hi).  Indices are global over the filtered, concatenated SNP axis.
struct Item {
    int w0;         // first window this item computes (fresh sum) = max(ws, own_lo-W+1)
    int we;         // end (exclusive) of the segment's valid windows
    int own_lo;     // first owned SNP
    int own_hi;     // end (exclusive) of owned SNPs
    int seg;        // segment id
    int flags;      // bit0: a previous item of the same segment exists; bit1: a next item exists
    int chr_start;  // global index of the chromosome's first SNP (thinning origin, garlic-data.cpp:2037)
    int thin_base;  // first thinned slot of this chromosome in the dump matrix
};

// One emitted run of covered SNPs (global SNP indices, inclusive).
struct RohRec {
    int ind;   // individual (index into the kernel's individual list)
    int a, b;  // first / last SNP index of the run
    int tag;   // seg<<2 | open_right<<1 | open_left
};

struct WalkParams {
    const uint64_t* geno;   // packed rows, 32 genotypes per 64-bit word, SNP s at bits 2*(s&31) of word s>>5
    int64_t row_words;      // row stride in 64-bit words (>= ceil(L/32)+2, padded)
    const double* lut;      // [L+pad][4] per-SNP LOD of g=0,1,2,missing (unweighted, global --error)
    const double* gl;       // per-genotype LOD (GL mode: lod() of every genotype, built at compaction), or nullptr;
                            // lane-interleaved: [ceil(N/32)][gl_stride SNPs][32 individuals] — see gl_lane()
    const double* freq;     // [L] (GL mode)
    int64_t gl_stride;
    const int* ind_list;    // optional indirection: lane k works on individual ind_list[k]
    int n_lanes;            // number of individuals to process (length of ind_list, or N)
    int W;                  // window size in SNPs
    int thr;                // integer coverage threshold = ceil(clamp(overlap_frac*W,1,W))
    double cutoff;          // LOD cutoff (garlic-roh.cpp:450)
    double tol;             // ambiguity half-width (0 = exact mode, no check)
    // outputs
    RohRec* out;            // ROH records
    unsigned* out_count;    // [0]=records appended, [1]=ambiguous (lane,item) pairs
    unsigned out_cap;
    unsigned* hist;         // optional [n_ind]: records appended per individual (for the device-side bucketing)
    RohRec* amb;            // ambiguous pairs (ind, seg) recorded as RohRec{ind,0,0,seg}
    unsigned amb_cap;
    double* dump;           // window dump matrix [n_lanes][dump_stride] or nullptr
    int64_t dump_stride;
    int dump_step;          // keep windows with (t-chr_start) % dump_step == 0
};

// GL-mode value of individual `ind` at SNP s: gl_lane(P, ind)[s * kGlLanes].  The 32 individuals of a group sit
// next to each other for every SNP, so a warp walking 32 consecutive individuals reads 256 contiguous bytes per SNP
// and a group's SNP range is one contiguous slab (what gl_walk_kernel copies with cp.async.bulk).
constexpr int kGlLanes = 32;
// Column selection of the ingest kernels (garlic_gpu_select_columns): local[col] is the handle's individual that input
// column col holds, or -1.  Columns at or beyond n_input (the extra columns of a malformed line) are never stored.
GHD int select_local(const int* local, int n_input, long long col)
{
    return col < n_input ? local[col] : -1;
}

GHD const double* gl_lane(const WalkParams& P, int ind)
{
    return P.gl + ((int64_t)(ind >> 5) * P.gl_stride) * kGlLanes + (ind & 31);
}

}  // namespace garlic
