// kernels.cu — hand-written sm_100a kernels for the GARLIC LOD/wLOD → ROH hot path.
// Kernel inventory (DESIGN.md §5): here K0 tokenize_tped, K1 code_alleles, K2 count_packed, compact_gl, K4 build_lut,
// K5 walk / walk_units (fused windows→ROH / window dump), thin_windows, the run-record bucketing; K3 + the pruning bound
// live in squeeze.cu, K6 and K5-W in wlod.cu, the counter exchange in xchg.cu, K0-GL in ingest.cu, the KDE in kde.cu.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <stdint.h>
#include <algorithm>
#include "common.cuh"
#include "walk.cuh"
#include "bound.cuh"
#include "kernels.h"

namespace garlic {

// ------------------------------------------------------------------------------------------
// K5: fused windows → ROH.  One warp = 32 individuals walking one item (a chunk of SNPs) in
// lock-step; the warps of a CTA take neighbouring individual groups of the SAME item, so the item's
// slice of the per-SNP LOD table is staged ONCE per CTA into shared memory by a TMA bulk copy
// (cp.async.bulk + mbarrier) and every table lookup of the walk is a conflict-free LDS (all lanes of a
// step read the same 32-byte entry).  Genotype words stream from HBM (each lane its own row; 8-byte
// reads that hit the same 32-byte sector four blocks in a row).
// TILE = false: table read from global memory (whole-segment exact chains, very large windows).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <int SRC, bool ROH, bool DUMP, bool TILE>
__global__ void __launch_bounds__(kWalkThreads, TILE ? 4 : 2)
walk_kernel(const WalkParams P, const Item* __restrict__ items, int n_items, int n_groups, int tile_bytes,
            const int* __restrict__ cand_list, const unsigned* __restrict__ cand_cnt, int cand_stride)
{
    extern __shared__ __align__(128) unsigned char walk_smem[];
    // layout: [tile (tile_bytes, TILE only)] [ring: NW * blockDim words] [mbarrier]
    unsigned char* tile_s = walk_smem;
    uint32_t* ring_smem = reinterpret_cast<uint32_t*>(walk_smem + (TILE ? tile_bytes : 0));
    const int NW = ((P.W + 31) >> 5) + 1;
    uint64_t* bar = reinterpret_cast<uint64_t*>(ring_smem + NW * blockDim.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gpb = blockDim.x >> 5;
    const int gblocks = (n_groups + gpb - 1) / gpb;
    const long long total = (long long)n_items * gblocks;
    if (TILE) {
        if (threadIdx.x == 0) mbar_init(bar, 1);
        __syncthreads();
    }
    uint32_t phase = 0;
    for (long long u = blockIdx.x; u < total; u += gridDim.x) {
        const int item = (int)(u / gblocks);
        const int group = (int)(u % gblocks) * gpb + warp;
        // pruned pass: this item's individuals are the dense candidate list written by select_kernel (squeeze.cu)
        int n_lanes = P.n_lanes;
        const int* list = nullptr;
        if (cand_list) {
            n_lanes = (int)cand_cnt[item];
            list = cand_list + (int64_t)item * cand_stride;
            if ((int)(u % gblocks) * gpb * 32 >= n_lanes) continue;      // whole CTA: nothing left in this item
        }
        const Item it = items[item];
        const char* tile = reinterpret_cast<const char*>(P.lut);
        int tile_lo = 0;
        if (TILE) {
            // SNPs the walk touches: [w0, w0 + 32*nblk + W) (fresh sum, slide-in / slide-out streams)
            const int nblk = (it.own_hi - 1 - it.w0 + 31) >> 5;
            const uint32_t bytes = (uint32_t)(32 * nblk + P.W) * 32u;
            if (threadIdx.x == 0) {
                mbar_expect_tx(bar, bytes);
                tma_load_1d(tile_s, P.lut + (int64_t)it.w0 * 4, bytes, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1u;
            tile = reinterpret_cast<const char*>(tile_s);
            tile_lo = it.w0;
        }
        if (group * 32 < n_lanes) {
            const int k = group * 32 + lane;
            const bool active = k < n_lanes;
            const int kk = active ? k : n_lanes - 1;
            walk_item<SRC, ROH, DUMP>(P, it, kk, active, ring_smem + threadIdx.x, blockDim.x, tile, tile_lo,
                                      list ? list[kk] : -1);
        }
        if (TILE) __syncthreads();   // every warp is done with the tile before the next copy lands
    }
}

// ------------------------------------------------------------------------------------------
// K5 pass 2 on the candidates the bound left (squeeze.cu:select_kernel): one CTA of two warps per work unit = up to 64
// candidate individuals of one piece-sized item, taken from a device-resident queue (the host never learns its length).
// The item's slice of the per-SNP table (about 14 KB at W = 50) is staged by one bulk copy per unit; two-warp CTAs keep
// the barrier around it cheap and let some ten units share an SM.  The compacted matrix is never written on this path:
// while the copy lands, every lane builds its candidate's compacted words of the item (about 14 at W = 50) from the
// uncompacted row by the compaction plan (bound.cuh:plan_slice) into its own stretch of shared memory — a few percent of
// the rows are read, where the compaction would have written all of them.  Where a compacted matrix exists already
// (R.rows == nullptr: another consumer needed it) the lanes read their rows from there, as the other walkers do.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kUnitThreads, 16)
walk_units_kernel(const WalkParams P, const RawRows R, const Item* __restrict__ items, const int2* __restrict__ units,
                  const unsigned* __restrict__ n_units, unsigned unit_cap, int tile_bytes, int slice_stride,
                  const int* __restrict__ cand_list, const unsigned* __restrict__ cand_cnt, int cand_stride)
{
    extern __shared__ __align__(128) unsigned char walk_smem[];
    // layout: [tile (tile_bytes)] [slices: slice_stride words per thread] [ring: NW words per thread] [mbarrier]
    unsigned char* tile_s = walk_smem;
    uint64_t* slice_s = reinterpret_cast<uint64_t*>(walk_smem + tile_bytes) + (size_t)threadIdx.x * slice_stride;
    uint32_t* ring_smem = reinterpret_cast<uint32_t*>(walk_smem + tile_bytes + (size_t)slice_stride * kUnitThreads * 8);
    const int NW = ((P.W + 31) >> 5) + 1;
    uint64_t* bar = reinterpret_cast<uint64_t*>(ring_smem + NW * kUnitThreads);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    unsigned nu = *n_units;
    nu = nu < unit_cap ? nu : unit_cap;
    uint32_t phase = 0;
    for (unsigned u = blockIdx.x; u < nu; u += gridDim.x) {
        const int2 un = units[u];
        const Item it = items[un.x];
        int n_lanes = (int)cand_cnt[un.x] - un.y;
        n_lanes = n_lanes < kUnitThreads ? n_lanes : kUnitThreads;
        const int* list = cand_list + (int64_t)un.x * cand_stride + un.y;
        const int nblk = (it.own_hi - 1 - it.w0 + 31) >> 5;
        const uint32_t bytes = (uint32_t)(32 * nblk + P.W) * 32u;
        if (threadIdx.x == 0) {
            mbar_expect_tx(bar, bytes);
            tma_load_1d(tile_s, P.lut + (int64_t)it.w0 * 4, bytes, bar);
        }
        const bool busy = warp * 32 < n_lanes;
        const int k = warp * 32 + lane;
        const bool active = k < n_lanes;
        const int kk = active ? k : n_lanes - 1;
        const int ind = busy ? list[kk] : 0;
        const int wlo = it.w0 >> 5;
        if (busy && R.rows) {
            const int n_w = ((it.w0 + P.W) >> 5) + nblk + 2 - wlo;   // (items_slice_words)
            plan_slice(R.head, R.segs, R.L, reinterpret_cast<const uint32_t*>(R.rows + (int64_t)ind * R.row_words), wlo, n_w, slice_s);
        }
        mbar_wait(bar, phase);
        phase ^= 1u;
        if (busy)
            walk_item<0, true, false>(P, it, kk, active, ring_smem + threadIdx.x, kUnitThreads,
                                      reinterpret_cast<const char*>(tile_s), it.w0, ind, R.rows ? slice_s : nullptr, wlo);
        __syncthreads();   // both warps are done with the tile before the next copy lands
    }
}

cudaError_t launch_walk_units(const WalkParams& P, const RawRows& R, const Item* items, const int2* units, const unsigned* n_units,
                              unsigned unit_cap, int tile_snps, int slice_words, const CandList& cl, cudaStream_t st)
{
    const int NW = ((P.W + 31) >> 5) + 1;
    const int tile_bytes = tile_snps * 32;
    const int slice_stride = R.rows ? slice_words | 1 : 0;   // odd: the lanes' 8-byte reads of the same word k fall in distinct banks
    const size_t smem = (size_t)tile_bytes + (size_t)slice_stride * kUnitThreads * 8 + (size_t)NW * kUnitThreads * sizeof(uint32_t) + 16;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(walk_units_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    per_sm = per_sm > 16 ? 16 : (per_sm < 1 ? 1 : per_sm);
    walk_units_kernel<<<148 * per_sm, kUnitThreads, smem, st>>>(P, R, items, units, n_units, unit_cap, tile_bytes, slice_stride,
                                                               cl.list, cl.cnt, cl.stride);
    return cudaGetLastError();
}

template <int SRC, bool ROH, bool DUMP>
static cudaError_t launch_walk_t(const WalkParams& P, const Item* items, int n_items, int tile_snps, const CandList& cl,
                                 cudaStream_t st)
{
    if (n_items == 0 || P.n_lanes == 0) return cudaSuccess;
    const int threads = kWalkThreads;
    const int n_groups = (P.n_lanes + 31) / 32;
    const int gpb = threads / 32;
    const long long total = (long long)n_items * ((n_groups + gpb - 1) / gpb);
    const int NW = ((P.W + 31) >> 5) + 1;
    const bool tile = (SRC == 0) && tile_snps > 0;
    const int tile_bytes = tile ? tile_snps * 32 : 0;
    const size_t smem = (size_t)tile_bytes + (size_t)NW * threads * sizeof(uint32_t) + 16;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long grid = total;
    const long long cap = (long long)sms * 4 * 16;   // persistent-ish: ≤ 16 waves of 4 CTAs/SM
    if (grid > cap) grid = cap;
    if (tile) {
        auto kern = walk_kernel<SRC, ROH, DUMP, true>;
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<(unsigned)grid, threads, smem, st>>>(P, items, n_items, n_groups, tile_bytes, cl.list, cl.cnt, cl.stride);
    } else {
        auto kern = walk_kernel<SRC, ROH, DUMP, false>;
        if (smem > 48 * 1024) {                                // flag history of very large windows
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<(unsigned)grid, threads, smem, st>>>(P, items, n_items, n_groups, 0, cl.list, cl.cnt, cl.stride);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// K5-GL pass 2: the fused window → cutoff → coverage → ROH walker for per-genotype likelihoods (--tgls).
// Here every genotype has its own LOD (8 bytes per individual-window of compulsory HBM traffic, SURVEY §8d: the
// HBM-bound config), so the kernel is organised around the copy:
//   * one CTA = one warp = the 32 individuals of a group walking one item, lane = individual;
//   * the group's values for the item's SNPs are ONE contiguous slab of the lane-interleaved matrix
//     (common.cuh:gl_lane).  It streams through a per-warp shared-memory ring in pieces of kGlPiece SNPs (4 KB) moved
//     by cp.async.bulk, each completing on its own mbarrier.  The ring holds the last W SNPs (= the slide-out values
//     of garlic-roh.cpp:98-100, so nothing is read twice from HBM or L2) plus the pieces in flight ahead;
//   * per step: two conflict-free LDS.64 (slide-in, slide-out), the window update in the reference's order (exact) or
//     win + (in − out) with the cutoff ± tol test (tolerance-checked pass, DESIGN.md §5), then cover_block as in the
//     table-mode walker.
// ------------------------------------------------------------------------------------------
constexpr int kGlPiece = 16;                              // SNPs per bulk copy
constexpr int kGlPieceBytes = kGlPiece * kGlLanes * 8;    // 4 KB

__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

template <bool CHK>
__global__ void __launch_bounds__(32)
gl_walk_kernel(const WalkParams P, const Item* __restrict__ items, int n_items, int n_groups, int NS)
{
    extern __shared__ __align__(128) unsigned char gl_smem[];
    const int lane = threadIdx.x;
    const int W = P.W;
    const int NW = ((W + 31) >> 5) + 1;
    const double* ring = reinterpret_cast<const double*>(gl_smem);
    uint32_t* fring = reinterpret_cast<uint32_t*>(gl_smem + (size_t)NS * kGlPieceBytes) + lane;   // flag-word history
    uint64_t* bars = reinterpret_cast<uint64_t*>(gl_smem + (size_t)NS * kGlPieceBytes + (size_t)NW * 128);
    if (lane == 0) for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
    __syncwarp();
    const int R = NS * kGlPiece;                           // ring length in SNPs (NS is even: R is a multiple of 32)
    uint64_t par = 0;                                      // bit s: parity the next completion of slot s will have
    const double cut_hi = CHK ? P.cutoff + P.tol : P.cutoff, cut_lo = P.cutoff - P.tol;
    const int r = (32 - (W & 31)) & 31;
    const long long total = (long long)n_items * n_groups;
    for (long long u = blockIdx.x; u < total; u += gridDim.x) {
        const int item = (int)(u / n_groups), group = (int)(u % n_groups);
        const Item it = items[item];
        const int ind = group * 32 + lane;
        const bool active = ind < P.n_lanes;
        const unsigned char* slab = reinterpret_cast<const unsigned char*>(P.gl + ((int64_t)group * P.gl_stride + it.w0) * kGlLanes);
        const int M = it.own_hi - 1 - it.w0;               // slide steps
        const int nblk = (M + 31) >> 5;
        const int NQ = (W + 32 * nblk + kGlPiece - 1) / kGlPiece;   // pieces this walk consumes
        int issued = 0, waited = 0;
        int islot = 0, wslot = 0;                          // ring slots of piece `issued` / `waited` (no runtime modulo)
        // lanes are done reading a slot before lane 0 hands it back to the copy engine
        auto issue_upto = [&](int qmax) {
            const int hi = qmax + 1 < NQ ? qmax + 1 : NQ;
            if (hi <= issued) return;
            __syncwarp();
            if (lane == 0) fence_proxy_async();
            for (; issued < hi; ++issued) {
                if (lane == 0) {
                    mbar_expect_tx(&bars[islot], kGlPieceBytes);
                    tma_load_1d(gl_smem + (size_t)islot * kGlPieceBytes, slab + (size_t)issued * kGlPieceBytes, kGlPieceBytes,
                                &bars[islot]);
                }
                if (++islot == NS) islot = 0;
            }
        };
        auto wait_upto = [&](int q) {
            for (; waited <= q; ++waited) {
                mbar_wait(&bars[wslot], (uint32_t)(par >> wslot) & 1u);
                par ^= 1ull << wslot;
                if (++wslot == NS) wslot = 0;
            }
        };
        issue_upto(NS - 1);
        // fresh sum for window w0, ascending (garlic-roh.cpp:57-71); these pieces sit in slots 0, 1, …
        double win = 0.0;
        for (int q = 0; q * kGlPiece < W; ++q) {
            wait_upto(q);
            const int n = W - q * kGlPiece < kGlPiece ? W - q * kGlPiece : kGlPiece;
            const double* p = ring + (size_t)q * kGlPiece * kGlLanes + lane;
            for (int i = 0; i < n; ++i) win += p[i * kGlLanes];
        }
        LaneState S;
        S.win = win; S.run_start = -1; S.fw = 0; S.ambig = false;
        const bool f0 = win >= cut_hi;
        if (CHK) S.ambig = (f0 != (win >= cut_lo));
        S.cov = (int)f0;
        S.hist = (uint32_t)f0 << 31;
        if (it.w0 >= it.own_lo && S.cov >= P.thr) S.run_start = it.w0;
        if (W > 32) {
            for (int w = 0; w < NW; ++w) fring[w * 32] = 0;
            fring[0] = (uint32_t)f0 << 31;
        }
        int wr = 1 % NW;
        int tblk = it.w0 + 1;
        int pin = W % R, pout = 0;                         // ring positions of the block's first slide-in / slide-out SNP
        for (int j = 0; j < nblk; ++j, tblk += 32) {
            wait_upto((W + 32 * j + 31) / kGlPiece);
            const int kwrap = R - pin;                     // slide-in steps k >= kwrap sit at the start of the ring
            const double* p_in = ring + (size_t)pin * kGlLanes + lane;
            const double* p_in2 = p_in - (size_t)R * kGlLanes;
            const double* p_out = ring + (size_t)pout * kGlLanes + lane;
            uint32_t vm = 0xffffffffu;
            const int nv = it.we - tblk;
            if (nv < 32) vm = nv <= 0 ? 0u : ((1u << nv) - 1u);
            // all 64 shared-memory reads of the block are issued before the dependent chain starts (one warp per
            // scheduler: nothing else hides the LDS latency); d[] then holds the block's window values.  Only one block
            // in NS/2 has its slide-in range wrap around the ring: the others read at compile-time offsets.
            uint32_t fhi = 0, flo = 0;
            double d[32], o[CHK ? 1 : 32];
            if (kwrap >= 32) {
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    if (CHK) d[k] = p_in[k * kGlLanes] - p_out[k * kGlLanes];
                    else { d[k] = p_in[k * kGlLanes]; o[k] = p_out[k * kGlLanes]; }
                }
            } else {
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    const double a_in = (k < kwrap ? p_in : p_in2)[k * kGlLanes];
                    if (CHK) d[k] = a_in - p_out[k * kGlLanes];
                    else { d[k] = a_in; o[k] = p_out[k * kGlLanes]; }
                }
            }
            if (CHK) {
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    win = win + d[k];
                    d[k] = win;
                    if (win >= cut_lo) flo |= 1u << k;
                }
                // a window at or above cutoff + tol is also above cutoff − tol: the second test only runs where needed
                if (__any_sync(0xffffffffu, flo != 0u)) {
#pragma unroll
                    for (int k = 0; k < 32; ++k) if (d[k] >= cut_hi) fhi |= 1u << k;   // garlic-roh.cpp:450
                }
            } else {
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    win = (win - o[k]) + d[k];             // garlic-roh.cpp:98-100
                    if (win >= cut_hi) fhi |= 1u << k;     // garlic-roh.cpp:450
                }
            }
            S.win = win;
            fhi &= vm;
            if (CHK) { flo &= vm; S.ambig |= (fhi != flo); }
            uint32_t ow = 0;
            if (W > 32) {
                int r0 = wr + 1; if (r0 >= NW) r0 -= NW;
                int r1 = r0 + 1; if (r1 >= NW) r1 -= NW;
                const uint32_t w0_ = fring[r0 * 32], w1_ = fring[r1 * 32];
                ow = r ? ((w0_ >> r) | (w1_ << (32 - r))) : w0_;
            }
            const bool full = (tblk + 31 < it.we) && (tblk >= it.own_lo) && (tblk + 31 < it.own_hi);
            if (full) cover_block<true>(P, it, S, ind, active, fhi, ow, tblk);
            else cover_block<false>(P, it, S, ind, active, fhi, ow, tblk);
            if (W > 32) {
                fring[wr * 32] = S.fw;
                if (++wr >= NW) wr = 0;
            }
            pin += 32; if (pin >= R) pin -= R;
            pout += 32; if (pout >= R) pout -= R;
            // slide-out pieces 2j, 2j+1 are dead now: their slots take pieces 2j+NS, 2j+1+NS
            issue_upto(2 * j + 1 + NS);
        }
        if (S.run_start >= 0) emit_run(P, it, ind, active, S.run_start, it.own_hi - 1);
        if (CHK && S.ambig && active) {
            const unsigned p = atomicAdd(P.out_count + 1, 1u);
            if (p < P.amb_cap) {
                RohRec rr;
                rr.ind = ind; rr.a = 0; rr.b = 0; rr.tag = it.seg;
                P.amb[p] = rr;
            }
        }
        wait_upto(NQ - 1);                                 // nothing of this walk is still landing (only when nblk == 0)
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// K5-GL pass 2, relay form (tolerance-checked pass only).  One warp per scheduler cannot hide its own instruction
// latencies, and shared memory (the W-SNP history) caps the CTAs per SM at about three.  Here K warps (2..4) share ONE
// ring and take the item's 32-window blocks in turn (block j → warp j mod K).  A warp loads its block's 64 values,
// forms d = in − out and their running sum P inside the block without waiting for anybody; only then does it take the
// window value at the end of block j−1 (`base`, 32 doubles handed through shared memory), publishes base + P[31] for
// the next warp at once, and tests base + P[k] against cutoff ± tol.  The coverage / run state (cover_block) travels
// the same way one step behind.  Sums are re-associated (base + prefix instead of one chain): same error bound as the
// chunked chain (DESIGN.md §5), windows within tol of the cutoff are re-walked exactly.
// Safety of slot reuse with K warps (a warp may lag K−1 blocks): floor(W/16) >= 2K, checked by the launcher.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void seq_wait(const volatile int* p, int v)
{
    while (*p < v) { }
    __threadfence_block();
}
__device__ __forceinline__ void seq_post(volatile int* p, int v, int lane)
{
    __threadfence_block();
    __syncwarp();
    if (lane == 0) *p = v;
}

__global__ void __launch_bounds__(128)
gl_relay_kernel(const WalkParams P, const Item* __restrict__ items, int n_items, int n_groups, int NS)
{
    extern __shared__ __align__(128) unsigned char gl_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, K = blockDim.x >> 5;
    const int W = P.W;
    const int NW = ((W + 31) >> 5) + 1;
    const double* ring = reinterpret_cast<const double*>(gl_smem);
    unsigned char* aux = gl_smem + (size_t)NS * kGlPieceBytes;
    uint32_t* fring = reinterpret_cast<uint32_t*>(aux) + lane;                       // [NW][32] flag-word history
    uint64_t* bars = reinterpret_cast<uint64_t*>(aux + (size_t)NW * 128);           // [64]
    double* sbase = reinterpret_cast<double*>(aux + (size_t)NW * 128 + 512) + lane;   // [32] window value handed on
    int* scov = reinterpret_cast<int*>(aux + (size_t)NW * 128 + 512 + 256) + lane;    // [3][32] cov, run_start, hist
    volatile int* seq = reinterpret_cast<volatile int*>(aux + (size_t)NW * 128 + 512 + 256 + 384);   // [0] base, [1] cover
    if (threadIdx.x == 0) for (int s = 0; s < NS; ++s) mbar_init(&bars[s], 1);
    __syncthreads();
    const int R = NS * kGlPiece;
    uint64_t par = 0;                                      // every warp follows every piece: same parity history
    const double cut_hi = P.cutoff + P.tol, cut_lo = P.cutoff - P.tol;
    const int r = (32 - (W & 31)) & 31;
    const long long total = (long long)n_items * n_groups;
    for (long long u = blockIdx.x; u < total; u += gridDim.x) {
        const int item = (int)(u / n_groups), group = (int)(u % n_groups);
        const Item it = items[item];
        const int ind = group * 32 + lane;
        const bool active = ind < P.n_lanes;
        const unsigned char* slab = reinterpret_cast<const unsigned char*>(P.gl + ((int64_t)group * P.gl_stride + it.w0) * kGlLanes);
        const int M = it.own_hi - 1 - it.w0;
        const int nblk = (M + 31) >> 5;
        const int NQ = (W + 32 * nblk + kGlPiece - 1) / kGlPiece;
        __syncthreads();                                   // every warp is done with the previous walk's shared state
        if (threadIdx.x == 0) { seq[0] = -1; seq[1] = -1; }
        __syncthreads();
        int waited = 0, wslot = 0;
        auto wait_upto = [&](int q) {
            for (; waited <= q; ++waited) {
                mbar_wait(&bars[wslot], (uint32_t)(par >> wslot) & 1u);
                par ^= 1ull << wslot;
                if (++wslot == NS) wslot = 0;
            }
        };
        auto issue = [&](int q0, int q1) {                 // pieces [q0, q1) ∩ [0, NQ), by this warp's lane 0
            if (q1 > NQ) q1 = NQ;
            if (q0 >= q1) return;
            __syncwarp();
            if (lane == 0) {
                fence_proxy_async();
                int sl = q0 % NS;
                for (int q = q0; q < q1; ++q) {
                    mbar_expect_tx(&bars[sl], kGlPieceBytes);
                    tma_load_1d(gl_smem + (size_t)sl * kGlPieceBytes, slab + (size_t)q * kGlPieceBytes, kGlPieceBytes, &bars[sl]);
                    if (++sl == NS) sl = 0;
                }
            }
        };
        if (warp == 0) issue(0, NS);
        // every warp sees the first pieces land before any slot can be reused (keeps the parity history in step)
        wait_upto((W + 31) / kGlPiece < NQ ? (W + 31) / kGlPiece : NQ - 1);
        bool ambig = false;
        if (warp == 0) {
            // fresh sum for window w0, ascending (garlic-roh.cpp:57-71); these pieces sit in slots 0, 1, …
            double win = 0.0;
            for (int q = 0; q * kGlPiece < W; ++q) {
                const int n = W - q * kGlPiece < kGlPiece ? W - q * kGlPiece : kGlPiece;
                const double* p = ring + (size_t)q * kGlPiece * kGlLanes + lane;
                for (int i = 0; i < n; ++i) win += p[i * kGlLanes];
            }
            const bool f0 = win >= cut_hi;
            ambig = (f0 != (win >= cut_lo));
            const int cov0 = (int)f0;
            sbase[0] = win;
            scov[0] = cov0;
            scov[32] = (it.w0 >= it.own_lo && cov0 >= P.thr) ? it.w0 : -1;
            scov[64] = (int)((uint32_t)f0 << 31);
            if (W > 32) {
                for (int w = 0; w < NW; ++w) fring[w * 32] = 0;
                fring[0] = (uint32_t)f0 << 31;
            }
            seq_post(&seq[0], 0, lane);
            seq_post(&seq[1], 0, lane);
        }
        __syncthreads();                                   // no slot is handed back while the fresh sum still reads the ring
        int wr = (1 + warp) % NW;
        int pin = (W + 32 * warp) % R, pout = (32 * warp) % R;
        for (int j = warp; j < nblk; j += K) {
            const int tblk = it.w0 + 1 + 32 * j;
            wait_upto((W + 32 * j + 31) / kGlPiece);
            const int kwrap = R - pin;
            const double* p_in = ring + (size_t)pin * kGlLanes + lane;
            const double* p_in2 = p_in - (size_t)R * kGlLanes;
            const double* p_out = ring + (size_t)pout * kGlLanes + lane;
            double d[32];
            if (kwrap >= 32) {
#pragma unroll
                for (int k = 0; k < 32; ++k) d[k] = p_in[k * kGlLanes] - p_out[k * kGlLanes];
            } else {
#pragma unroll
                for (int k = 0; k < 32; ++k) d[k] = (k < kwrap ? p_in : p_in2)[k * kGlLanes] - p_out[k * kGlLanes];
            }
#pragma unroll
            for (int k = 1; k < 32; ++k) d[k] = d[k - 1] + d[k];
            // this block's slide-out pieces 2j, 2j+1 are dead: their slots take pieces 2j+NS, 2j+1+NS
            issue(2 * j + NS, 2 * j + 2 + NS);
            seq_wait(&seq[0], j);
            const double base = sbase[0];
            sbase[0] = base + d[31];
            seq_post(&seq[0], j + 1, lane);
            uint32_t vm = 0xffffffffu;
            const int nv = it.we - tblk;
            if (nv < 32) vm = nv <= 0 ? 0u : ((1u << nv) - 1u);
            uint32_t fhi = 0, flo = 0;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                d[k] = base + d[k];
                if (d[k] >= cut_lo) flo |= 1u << k;
            }
            if (__any_sync(0xffffffffu, flo != 0u)) {
#pragma unroll
                for (int k = 0; k < 32; ++k) if (d[k] >= cut_hi) fhi |= 1u << k;   // garlic-roh.cpp:450
            }
            fhi &= vm; flo &= vm;
            ambig |= (fhi != flo);
            // coverage / run state of block j−1 → this block
            seq_wait(&seq[1], j);
            LaneState S;
            S.win = 0; S.fw = 0; S.ambig = false;
            S.cov = scov[0]; S.run_start = scov[32]; S.hist = (uint32_t)scov[64];
            uint32_t ow = 0;
            if (W > 32) {
                int r0 = wr + 1; if (r0 >= NW) r0 -= NW;
                int r1 = r0 + 1; if (r1 >= NW) r1 -= NW;
                const uint32_t w0_ = fring[r0 * 32], w1_ = fring[r1 * 32];
                ow = r ? ((w0_ >> r) | (w1_ << (32 - r))) : w0_;
            }
            const bool full = (tblk + 31 < it.we) && (tblk >= it.own_lo) && (tblk + 31 < it.own_hi);
            if (full) cover_block<true>(P, it, S, ind, active, fhi, ow, tblk);
            else cover_block<false>(P, it, S, ind, active, fhi, ow, tblk);
            if (W > 32) fring[wr * 32] = S.fw;
            if (j == nblk - 1) {
                if (S.run_start >= 0) emit_run(P, it, ind, active, S.run_start, it.own_hi - 1);
            } else {
                scov[0] = S.cov; scov[32] = S.run_start; scov[64] = (int)S.hist;
                seq_post(&seq[1], j + 1, lane);
            }
            wr += K; while (wr >= NW) wr -= NW;
            pin += 32 * K; while (pin >= R) pin -= R;
            pout += 32 * K; while (pout >= R) pout -= R;
        }
        if (nblk == 0 && warp == 0) {
            const int rs = scov[32];
            if (rs >= 0) emit_run(P, it, ind, active, rs, it.own_hi - 1);
        }
        if (ambig && active) {
            const unsigned p = atomicAdd(P.out_count + 1, 1u);
            if (p < P.amb_cap) {
                RohRec rr;
                rr.ind = ind; rr.a = 0; rr.b = 0; rr.tag = it.seg;
                P.amb[p] = rr;
            }
        }
        wait_upto(NQ - 1);                                 // every warp has followed every piece of this walk
    }
}

// ring slots for window size W (even; 0 = the ring does not fit, use the generic walker)
static int gl_ring_slots(int W, size_t* smem_bytes)
{
    const int span = (W + 31) / kGlPiece + 1;              // pieces a block's slide-out .. slide-in range touches
    const int NW = ((W + 31) >> 5) + 1;
    const size_t fixed = (size_t)NW * 128 + 64 * 8 + 256 + 384 + 128;     // flag ring, mbarriers, relay hand-over area
    const size_t budget = 227 * 1024;
    int ns_min = span + 3; ns_min += ns_min & 1;
    if (ns_min > 56 || (size_t)ns_min * kGlPieceBytes + fixed > budget) return 0;
    // as many CTAs per SM as the minimum ring allows, then spend the rest of that share on pieces in flight
    int ctas = (int)((budget - 1024) / ((size_t)ns_min * kGlPieceBytes + fixed + 1024));
    if (const char* e = getenv("GARLIC_GL_CTAS")) { const int c = atoi(e); if (c >= 1 && c < ctas) ctas = c; }
    int ns = (int)(((budget - 1024) / (ctas > 0 ? ctas : 1) - fixed - 1024) / kGlPieceBytes);
    if (ns > span + 24) ns = span + 24;
    if (ns > 56) ns = 56;
    ns -= ns & 1;
    if (ns < ns_min) ns = ns_min;
    *smem_bytes = (size_t)ns * kGlPieceBytes + fixed;
    return ns;
}

static cudaError_t launch_gl_walk(const WalkParams& P, const Item* items, int n_items, int NS, size_t smem, cudaStream_t st)
{
    const int n_groups = (P.n_lanes + 31) / 32;
    const long long total = (long long)n_items * n_groups;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int per_sm = (int)((227 * 1024) / (smem + 1024));
    long long grid = (long long)sms * (per_sm > 0 ? per_sm : 1);   // persistent: every CTA slot of the chip, once
    if (grid > total) grid = total;
    cudaError_t e;
    if (P.tol > 0) {
        // relay warps per ring: floor(W/16) >= 2K keeps slot reuse safe with a warp lagging K-1 blocks
        int K = 1;
        // and (W+31)/16 >= 4K-1 keeps every warp's mbarrier parity history in step (a slot completes at most once unseen)
        while (K < 4 && (P.W / kGlPiece) >= 2 * (K + 1) && (P.W + 31) / kGlPiece >= 4 * (K + 1) - 1) ++K;
        if (const char* ev = getenv("GARLIC_GL_WARPS")) { const int k = atoi(ev); if (k >= 1 && k < K) K = k; }
        if (K >= 2) {
            e = cudaFuncSetAttribute(gl_relay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            gl_relay_kernel<<<(unsigned)grid, 32 * K, smem, st>>>(P, items, n_items, n_groups, NS);
            return cudaGetLastError();
        }
        e = cudaFuncSetAttribute(gl_walk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        gl_walk_kernel<true><<<(unsigned)grid, 32, smem, st>>>(P, items, n_items, n_groups, NS);
    } else {
        e = cudaFuncSetAttribute(gl_walk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        gl_walk_kernel<false><<<(unsigned)grid, 32, smem, st>>>(P, items, n_items, n_groups, NS);
    }
    return cudaGetLastError();
}

cudaError_t launch_walk(const WalkParams& P, const Item* items, int n_items, bool gl_mode, bool roh,
                        bool dump, int tile_snps, const CandList& cl, cudaStream_t st)
{
    if (gl_mode) {
        if (roh && !dump && !P.ind_list && n_items && P.n_lanes) {
            size_t smem = 0;
            const int NS = gl_ring_slots(P.W, &smem);
            if (NS && !getenv("GARLIC_NO_GL_RING")) return launch_gl_walk(P, items, n_items, NS, smem, st);
        }
        if (roh && !dump) return launch_walk_t<1, true, false>(P, items, n_items, 0, cl, st);
        if (!roh && dump) return launch_walk_t<1, false, true>(P, items, n_items, 0, cl, st);
        return launch_walk_t<1, true, true>(P, items, n_items, 0, cl, st);
    }
    if (roh && !dump) return launch_walk_t<0, true, false>(P, items, n_items, tile_snps, cl, st);
    if (!roh && dump) return launch_walk_t<0, false, true>(P, items, n_items, tile_snps, cl, st);
    return launch_walk_t<0, true, true>(P, items, n_items, tile_snps, cl, st);
}

// ------------------------------------------------------------------------------------------
// K5 pass 1, thinned: the KDE only looks at windows at locus 0, step, 2·step, … of each chromosome
// (convert[Subset]WinData2DoubleData, garlic-data.cpp:2026-2150) for a handful of individuals, so each of those
// windows is summed directly (ascending, like a fresh sum of calcLOD, garlic-roh.cpp:57-71) by its own thread
// instead of walking every window in between.  meta: per chromosome (first kept SNP, first slot).
// Valid windows are those inside a segment [ws, we); the others keep the MISSING the buffer was filled with.
// ------------------------------------------------------------------------------------------
__global__ void thin_windows_kernel(const uint64_t* __restrict__ geno, int64_t row_words, const double* __restrict__ lut,
                                    const int* __restrict__ ind_list, const uint32_t* __restrict__ bad_bits, long long L,
                                    const int2* __restrict__ meta, int n_chr, long long n_slots, int step, int W,
                                    double* __restrict__ dump, int64_t dump_stride, const double* __restrict__ gl,
                                    int64_t gl_stride, const int* __restrict__ src)
{
    // src != nullptr: geno is the UNCOMPACTED matrix and kept SNP s sits at column src[s] (pass 1 then does not have to wait
    // for the compaction)
    const int k = blockIdx.y;
    const int ind = ind_list ? ind_list[k] : k;
    const uint64_t* row = geno + (int64_t)ind * row_words;
    // GL mode: per-genotype LOD values, lane-interleaved (common.cuh:gl_lane)
    const double* glrow = gl ? gl + ((int64_t)(ind >> 5) * gl_stride) * kGlLanes + (ind & 31) : nullptr;
    for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n_slots; j += (long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = n_chr - 1;                       // chromosome of slot j: last c with meta[c].y <= j
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (meta[mid].y <= j) lo = mid; else hi = mid - 1; }
        const int t = meta[lo].x + (int)(j - meta[lo].y) * step;
        // a valid window: inside the data and no bad pair / chromosome start among SNPs t+1 … t+W-1 (the closed form of the
        // reference's MISSING logic, DESIGN.md §4, tested on the bit map bad_pairs_kernel leaves)
        if ((long long)t + W > L) continue;
        bool ok = true;
        const int b0 = t + 1, b1 = t + W - 1;
        for (int w = b0 >> 5; w <= (b1 >> 5); ++w) {
            uint32_t m = bad_bits[w];
            if (w == (b0 >> 5)) m &= ~((1u << (b0 & 31)) - 1u);
            if (w == (b1 >> 5) && (b1 & 31) != 31) m &= (1u << ((b1 & 31) + 1)) - 1u;
            ok = ok && m == 0u;
        }
        if (!ok) continue;
        double win = 0.0;
        if (glrow) {
            for (int i = 0; i < W; ++i) win += glrow[(int64_t)(t + i) * kGlLanes];
        } else {
            // eight table lookups in flight at a time; the sum itself stays ascending (a fresh sum of calcLOD)
            int i = 0;
            for (; i + 8 <= W; i += 8) {
                double v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int s = t + i + k;
                    const int c = src ? src[s] : s;
                    const int g = (int)(row[c >> 5] >> (2 * (c & 31))) & 3;
                    v[k] = lut[(int64_t)s * 4 + g];
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) win += v[k];
            }
            for (; i < W; ++i) {
                const int s = t + i;
                const int c = src ? src[s] : s;
                const int g = (int)(row[c >> 5] >> (2 * (c & 31))) & 3;
                win += lut[(int64_t)s * 4 + g];
            }
        }
        dump[(int64_t)k * dump_stride + j] = win;
    }
}

cudaError_t launch_thin_windows(const uint64_t* geno, int64_t row_words, const double* lut, const int* ind_list, int n_lanes,
                                const uint32_t* bad_bits, long long L, const int2* meta, int n_chr, long long n_slots, int step, int W,
                                double* dump, int64_t dump_stride, const double* gl, int64_t gl_stride, const int* src, cudaStream_t st)
{
    if (!n_lanes || !n_slots) return cudaSuccess;
    long long bx = (n_slots + 127) / 128;
    if (bx > 4096) bx = 4096;
    dim3 grid((unsigned)bx, (unsigned)n_lanes);
    thin_windows_kernel<<<grid, 128, 0, st>>>(geno, row_words, lut, ind_list, bad_bits, L, meta, n_chr, n_slots, step, W, dump,
                                               dump_stride, gl, gl_stride, src);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Run records leave the walkers in arbitrary order (one atomic append each).  The reference's output order is
// (individual, chromosome, start): the counting sort on the individual is done here — emit_run kept a histogram —
// and each individual's handful of runs is then ordered and stitched by one thread.  hist: [n_ind] counts → offsets.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) bucket_scan_kernel(unsigned* __restrict__ hist, int n)
{
    __shared__ unsigned s_part[1024];
    const int per = (n + 1023) / 1024;
    const int lo = threadIdx.x * per, hi = min(n, lo + per);
    unsigned sum = 0;
    for (int i = lo; i < hi; ++i) sum += hist[i];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const unsigned v = threadIdx.x >= o ? s_part[threadIdx.x - o] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned run = s_part[threadIdx.x] - sum;
    for (int i = lo; i < hi; ++i) { const unsigned c = hist[i]; hist[i] = run; run += c; }
}

__global__ void bucket_scatter_kernel(const RohRec* __restrict__ in, const unsigned* __restrict__ count, unsigned cap,
                                      unsigned* __restrict__ offs, RohRec* __restrict__ out)
{
    const unsigned n = min(*count, cap);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const RohRec r = in[i];
        out[atomicAdd(offs + r.ind, 1u)] = r;
    }
}

// One warp per individual: order its runs by start, merge the pieces of runs that were cut at item borders and
// apply the minimum-length rule (garlic-roh.cpp:477) — segments.h:stitch_runs, in place; dropped slots get ind = -1.
// Up to kStitchSmem runs (the piece-sized items of the pruned pass cut a long ROH into several): the bucket is ranked
// by all lanes against a copy in shared memory, dropped into a second shared array in order, and lane 0 merges from
// there.  Larger buckets (cutoffs that flag nearly everything) are ranked in global memory through `scratch`.
// ends: the bucket offsets after the scatter (= end of every individual's bucket).
constexpr int kStitchSmem = 256;
__global__ void __launch_bounds__(128)
bucket_stitch_kernel(RohRec* __restrict__ recs, RohRec* __restrict__ scratch, const unsigned* __restrict__ ends, int n_ind, int thr,
                     unsigned* __restrict__ kept)
{
    __shared__ RohRec s_in[4][kStitchSmem];
    __shared__ RohRec s_rec[4][kStitchSmem];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = blockIdx.x * 4 + warp; i < n_ind; i += gridDim.x * 4) {
        const unsigned lo = i ? ends[i - 1] : 0u, hi = ends[i];
        const unsigned n = hi - lo;
        if (n == 0u) { if (lane == 0) kept[i] = 0u; continue; }
        const RohRec* src;
        if (n <= (unsigned)kStitchSmem) {
            for (unsigned j = lane; j < n; j += 32) s_in[warp][j] = recs[lo + j];
            __syncwarp();
            for (unsigned j = lane; j < n; j += 32) {
                const RohRec mine = s_in[warp][j];
                unsigned rank = 0;
                // starts of one individual's runs are distinct; ties are broken by position anyway
                for (unsigned k = 0; k < n; ++k) { const int ak = s_in[warp][k].a; rank += (ak < mine.a) || (ak == mine.a && k < j); }
                s_rec[warp][rank] = mine;
            }
            __syncwarp();
            src = s_rec[warp];
        } else {
            for (unsigned j = lane; j < n; j += 32) {
                const RohRec mine = recs[lo + j];
                unsigned rank = 0;
                for (unsigned k = 0; k < n; ++k) { const int ak = recs[lo + k].a; rank += (ak < mine.a) || (ak == mine.a && k < j); }
                scratch[lo + rank] = mine;
            }
            __threadfence_block();
            __syncwarp();
            src = scratch + lo;
        }
        if (lane == 0) {
            unsigned w = lo, k = 0;
            while (k < n) {
                RohRec cur = src[k++];
                while ((cur.tag & 2) && k < n) {
                    const RohRec nx = src[k];
                    if (!((nx.tag & 1) && nx.a == cur.b + 1 && (nx.tag >> 2) == (cur.tag >> 2))) break;
                    cur.b = nx.b;
                    cur.tag = (cur.tag & ~2) | (nx.tag & 2);
                    ++k;
                }
                if (cur.b - cur.a + 1 >= thr) recs[w++] = cur;   // src is a copy: no record still to be read is overwritten
            }
            kept[i] = w - lo;                                    // the individual's final runs sit at recs[lo, lo + kept)
            for (; w < hi; ++w) recs[w].ind = -1;
        }
        __syncwarp();
    }
}

// final runs of all individuals, dense and in (individual, start) order: kept_off = exclusive scan of kept[]
__global__ void __launch_bounds__(128)
bucket_compact_kernel(const RohRec* __restrict__ recs, const unsigned* __restrict__ ends, const unsigned* __restrict__ kept_off,
                      int n_ind, RohRec* __restrict__ out, unsigned* __restrict__ total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = blockIdx.x * 4 + warp; i < n_ind; i += gridDim.x * 4) {
        const unsigned lo = i ? ends[i - 1] : 0u;
        const unsigned o0 = kept_off[i], o1 = kept_off[i + 1];
        for (unsigned j = lane; j < o1 - o0; j += 32) out[o0 + j] = recs[lo + j];
        if (i == n_ind - 1 && lane == 0) *total = o1;
    }
}

// in: the walkers' records (arbitrary order) → out: bucketed by individual, ordered, stitched → in: the final runs, dense;
// *total = their number.  hist: [n_ind + 1] records per individual (by emit_run); kept: [n_ind + 1] scratch.
cudaError_t launch_bucket_by_individual(RohRec* in, const unsigned* count, unsigned cap, unsigned* hist, int n_ind,
                                        RohRec* out, int thr, unsigned* kept, unsigned* total, cudaStream_t st)
{
    if (!n_ind) return cudaSuccess;
    const int grid = (n_ind + 3) / 4 < 148 * 8 ? (n_ind + 3) / 4 : 148 * 8;
    bucket_scan_kernel<<<1, 1024, 0, st>>>(hist, n_ind);
    bucket_scatter_kernel<<<148, 256, 0, st>>>(in, count, cap, hist, out);
    // `in` is free once scattered: the stitch kernel's scratch for buckets too large for shared memory, then the output
    bucket_stitch_kernel<<<grid, 128, 0, st>>>(out, in, hist, n_ind, thr, kept);
    bucket_scan_kernel<<<1, 1024, 0, st>>>(kept, n_ind + 1);      // kept[n_ind] = 0 → the total lands there
    bucket_compact_kernel<<<grid, 128, 0, st>>>(out, hist, kept, n_ind, in, total);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// fill
// ------------------------------------------------------------------------------------------
__global__ void fill_f64_kernel(double* p, size_t n, double v)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
cudaError_t launch_fill_f64(double* p, size_t n, double v, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    fill_f64_kernel<<<(unsigned)blocks, 256, 0, st>>>(p, n, v);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// K1: genotype coding from allele characters (garlic-data.cpp:105-133), two phases so that the
// "1" allele (first non-missing character in file order over ALL individuals) can be min-reduced
// across GPUs between them.
//   phase a: per SNP key = min over local calls of ((global_call_index << 8) | char)
//   phase b: code each call, count nalleles / total (half-missing calls count their present
//            allele, :115-127), and transpose into the individual-major 2-bit matrix.
// alleles: [n_snp][n_ind][2] bytes (one tped line per SNP).
// ------------------------------------------------------------------------------------------
__global__ void first_allele_kernel(const uint8_t* __restrict__ alleles, int n_snp, int n_ind,
                                    int ind_offset, int missing, unsigned long long* __restrict__ key)
{
    // one warp per SNP; lanes stride over the 2*n_ind allele characters
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (long long s = blockIdx.x * (long long)warps_per_block + (threadIdx.x >> 5); s < n_snp;
         s += (long long)gridDim.x * warps_per_block) {
        const uint8_t* a = alleles + (size_t)s * n_ind * 2;
        unsigned long long best = ~0ull;
        for (int c = lane; c < 2 * n_ind; c += 32) {
            const uint8_t ch = a[c];
            if (ch != missing) {
                best = (((unsigned long long)(2ll * ind_offset + c)) << 8) | ch;
                break;   // lanes visit their calls in ascending order
            }
        }
        for (int o = 16; o; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other < best ? other : best;
        }
        if (lane == 0) key[s] = best;
    }
}

// ------------------------------------------------------------------------------------------
// K0: tped tokeniser.  The reference reads a line's genotype columns with `stringstream >> char`, i.e. the k-th
// non-blank character after the 4th field is allele k (garlic-data.cpp:105-133).  The host keeps those line tails as
// raw text; here one CTA per line ranks the non-blank characters (per-thread count, block scan) and scatters the ones
// belonging to this GPU's individuals [ind_lo, ind_lo + n_ind) into the [n_snp][n_ind][2] allele block K1 works on.
// nonblank[l] = number of non-blank characters of line l (the host checks it against 2 x individuals).
// ------------------------------------------------------------------------------------------
constexpr int kTokChars = 16;   // characters per thread per tile
__global__ void __launch_bounds__(256)
tokenize_tped_kernel(const char* __restrict__ text, const long long* __restrict__ off, int n_snp, int n_ind, int ind_lo,
                     uint8_t* __restrict__ alleles, int* __restrict__ nonblank)
{
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long k_lo = 2ll * ind_lo, k_hi = 2ll * (ind_lo + n_ind);
    for (int l = blockIdx.x; l < n_snp; l += gridDim.x) {
        const char* line = text + off[l];
        const long long len = off[l + 1] - off[l];
        uint8_t* dst = alleles + (size_t)l * n_ind * 2;
        if (threadIdx.x == 0) s_base = 0;
        __syncthreads();
        for (long long t0 = 0; t0 < len; t0 += 256 * kTokChars) {
            const long long i0 = t0 + (long long)threadIdx.x * kTokChars;
            char c[kTokChars];
            int n = 0;
#pragma unroll
            for (int k = 0; k < kTokChars; ++k) {
                c[k] = (i0 + k < len) ? line[i0 + k] : ' ';
                n += (c[k] != ' ' && c[k] != '\t' && c[k] != '\r' && c[k] != '\n');
            }
            // exclusive scan of n over the block
            int incl = n;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            int wbase = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) if (w < warp) wbase += s_warp[w];
            long long k = (long long)s_base + wbase + incl - n;      // rank of this thread's first non-blank character
#pragma unroll
            for (int q = 0; q < kTokChars; ++q)
                if (c[q] != ' ' && c[q] != '\t' && c[q] != '\r' && c[q] != '\n') {
                    if (k >= k_lo && k < k_hi) dst[k - k_lo] = (uint8_t)c[q];
                    ++k;
                }
            __syncthreads();
            if (threadIdx.x == 255) s_base += wbase + incl;
            __syncthreads();
        }
        if (threadIdx.x == 0) nonblank[l] = s_base;
        __syncthreads();
    }
}

cudaError_t launch_tokenize_tped(const char* text, const long long* off, int n_snp, int n_ind, int ind_lo, uint8_t* alleles,
                                 int* nonblank, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    tokenize_tped_kernel<<<n_snp < 148 * 8 ? n_snp : 148 * 8, 256, 0, st>>>(text, off, n_snp, n_ind, ind_lo, alleles, nonblank);
    return cudaGetLastError();
}

cudaError_t launch_first_allele(const uint8_t* alleles, int n_snp, int n_ind, int ind_offset, int missing,
                                unsigned long long* key, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    int blocks = (n_snp + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    first_allele_kernel<<<blocks, 256, 0, st>>>(alleles, n_snp, n_ind, ind_offset, missing, key);
    return cudaGetLastError();
}

// phase b.  Tile = 32 SNPs (one 64-bit packed word per individual) × 32 individuals per warp pass.
// Block = 256 threads = 8 warps; block handles SNPs [32*blockIdx.x, +32) and loops individuals.
// counts: [4][L0] int32 = nalleles, total, hom(g∈{0,2}), nonmiss.
__global__ void __launch_bounds__(256)
code_alleles_kernel(const uint8_t* __restrict__ alleles, int n_snp, int n_ind, int missing,
                    const unsigned long long* __restrict__ key, long long snp0,
                    uint64_t* __restrict__ geno, int64_t row_words, int* __restrict__ counts, long long L0)
{
    __shared__ uint8_t tile[32][257];          // [snp][ind-in-chunk] genotype codes, padded
    __shared__ int s_cnt[4][32];
    const int s_base = blockIdx.x * 32;
    if (threadIdx.x < 128) s_cnt[threadIdx.x >> 5][threadIdx.x & 31] = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n_ind; i0 += 256) {
        // code: each thread handles one individual for the 32 SNPs?  no — coalesce on the character
        // axis: for SNP r, threads read consecutive individuals (2 bytes each)
        for (int r = 0; r < 32; ++r) {
            const int s = s_base + r;
            const int i = i0 + threadIdx.x;
            uint8_t code = 3;
            int na = 0, tot = 0;
            if (s < n_snp && i < n_ind) {
                const uint16_t two = reinterpret_cast<const uint16_t*>(alleles + (size_t)s * n_ind * 2)[i];
                const int a1 = two & 0xff, a2 = two >> 8;
                const unsigned long long k = key[s];
                const int one = (k == ~0ull) ? missing : (int)(k & 0xff);
                int d = 0;
                if (a1 == missing) d = -9; else { tot++; if (a1 == one) { d += 1; na++; } }
                if (a2 == missing) d += -9; else { tot++; if (a2 == one) { d += 1; na++; } }
                code = d < 0 ? 3 : (uint8_t)d;
            }
            // warp-shuffle reduction of the per-SNP counts (all lanes participate), then one
            // shared atomic per warp
            int v_na = na, v_tot = tot, v_hom = (code == 0 || code == 2), v_nm = (code != 3);
            for (int o = 16; o; o >>= 1) {
                v_na += __shfl_xor_sync(0xffffffffu, v_na, o);
                v_tot += __shfl_xor_sync(0xffffffffu, v_tot, o);
                v_hom += __shfl_xor_sync(0xffffffffu, v_hom, o);
                v_nm += __shfl_xor_sync(0xffffffffu, v_nm, o);
            }
            if ((threadIdx.x & 31) == 0 && v_tot + v_nm + v_hom) {
                atomicAdd(&s_cnt[0][r], v_na); atomicAdd(&s_cnt[1][r], v_tot);
                atomicAdd(&s_cnt[2][r], v_hom); atomicAdd(&s_cnt[3][r], v_nm);
            }
            tile[r][threadIdx.x] = code;
        }
        __syncthreads();
        // pack: thread = individual; 32 SNP codes → one 64-bit word of its row
        const int i = i0 + threadIdx.x;
        if (i < n_ind) {
            uint64_t w = 0;
#pragma unroll
            for (int r = 0; r < 32; ++r) w |= (uint64_t)tile[r][threadIdx.x] << (2 * r);
            geno[(int64_t)i * row_words + ((snp0 + s_base) >> 5)] = w;
        }
        __syncthreads();
    }
    if (threadIdx.x < 128) {
        const int c = threadIdx.x >> 5, r = threadIdx.x & 31;
        if (s_base + r < n_snp) atomicAdd(&counts[(long long)c * L0 + snp0 + s_base + r], s_cnt[c][r]);
    }
}

cudaError_t launch_code_alleles(const uint8_t* alleles, int n_snp, int n_ind, int missing,
                                const unsigned long long* key, long long snp0, uint64_t* geno,
                                int64_t row_words, int* counts, long long L0, cudaStream_t st)
{
    if (!n_snp) return cudaSuccess;
    // snp0 must be a multiple of 32 so that tiles map to whole packed words
    code_alleles_kernel<<<(n_snp + 31) / 32, 256, 0, st>>>(alleles, n_snp, n_ind, missing, key, snp0, geno,
                                                          row_words, counts, L0);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// K2: per-SNP counts from the packed matrix (pre-coded input path): column reduction over the GPU's
// individuals (replaces the counting inside loadTPEDData, garlic-data.cpp:115-127, and calculateGenoFreq,
// :656-676).  A thread owns one 64-bit word column (32 SNPs) for every 8th row of its block's row range; lanes of a
// warp read 256 contiguous bytes of one row.  Counting is bit-sliced: per row two words (the packed word itself — even
// bits = g in {1, missing}, odd bits = g in {2, missing} — and a missing indicator) are fed 8 rows at a time through a carry-save adder tree (LOP3: sum 0x96, carry 0xE8)
// into vertical counters ones/twos/fours/eights…; every 248 rows the 8 bit-planes are turned into per-SNP byte
// counts (nibble → 4 bytes by multiplication) and added to shared, then global, integer counters.
// counts: [4][L0] = nalleles (Σ g over g<3), total (2·nonmiss), hom, nonmiss.
// ------------------------------------------------------------------------------------------
struct VCounter {
    uint64_t p[8];   // bit-planes: ones, twos, fours, eights, …, 128s
};

__device__ __forceinline__ void csa(uint64_t& sum, uint64_t& carry, uint64_t a, uint64_t b, uint64_t c)
{
    const uint64_t u = a ^ b;
    carry = (a & b) | (u & c);
    sum = u ^ c;
}

__device__ __forceinline__ void vc_add8(VCounter& v, const uint64_t x[8])
{
    uint64_t t2a, t2b, t2c, t2d, t4a, t4b, e8;
    csa(v.p[0], t2a, v.p[0], x[0], x[1]);
    csa(v.p[0], t2b, v.p[0], x[2], x[3]);
    csa(v.p[1], t4a, v.p[1], t2a, t2b);
    csa(v.p[0], t2c, v.p[0], x[4], x[5]);
    csa(v.p[0], t2d, v.p[0], x[6], x[7]);
    csa(v.p[1], t4b, v.p[1], t2c, t2d);
    csa(v.p[2], e8, v.p[2], t4a, t4b);
#pragma unroll
    for (int l = 3; l < 8; ++l) {   // ripple the eights into the higher planes
        const uint64_t c = v.p[l] & e8;
        v.p[l] ^= e8;
        e8 = c;
    }
}

// Turn the 8 planes (64 bit positions = 32 SNPs x {even, odd}) into counts and add them to this thread's slots of
// the CTA's shared counters, laid out [kind][SNP within word (32)][column (256, stride kCntCol = 257)] so that a warp's
// accesses are consecutive and every slot has exactly one owner (plain adds, no atomics); the odd stride makes the final
// read-out (consecutive SNPs = consecutive rows of this layout) conflict-free as well.
// 4 bit positions at a time: nibble n of plane l → bytes (bit j → byte j) by (n * 0x00204081) & 0x01010101.
constexpr int kCntCol = 257;
__device__ __noinline__ void vc_flush(VCounter& v, int* __restrict__ even_cnt, int* __restrict__ odd_cnt)
{
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        uint32_t acc = 0;
#pragma unroll
        for (int l = 0; l < 8; ++l) {
            const uint32_t nib = (uint32_t)(v.p[l] >> (4 * g)) & 0xfu;
            acc += ((nib * 0x00204081u) & 0x01010101u) << l;
        }
        even_cnt[(2 * g) * kCntCol] += acc & 0xff;
        even_cnt[(2 * g + 1) * kCntCol] += (acc >> 16) & 0xff;
        if (odd_cnt) {
            odd_cnt[(2 * g) * kCntCol] += (acc >> 8) & 0xff;
            odd_cnt[(2 * g + 1) * kCntCol] += acc >> 24;
        }
    }
#pragma unroll
    for (int l = 0; l < 8; ++l) v.p[l] = 0;
}

// block = 256 consecutive word columns (2 KB of every row, contiguous), thread = one column, rows of the block's
// row range in groups of 8.
__global__ void __launch_bounds__(256, 2)
count_packed_kernel(const uint64_t* __restrict__ geno, int64_t row_words, int n_ind, long long L0,
                    int rows_per_block, int* __restrict__ counts)
{
    extern __shared__ int s_cnt[];             // [3][32][kCntCol]: n1, n2, missing
    for (int i = threadIdx.x; i < 3 * 32 * kCntCol; i += 256) s_cnt[i] = 0;
    __syncthreads();
    const long long word = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long n_words = (L0 + 31) >> 5;
    const int r0 = blockIdx.y * rows_per_block;
    const int r1 = min(n_ind, r0 + rows_per_block);
    if (word < n_words && r0 < r1) {
        const uint64_t M = 0x5555555555555555ull;
        VCounter va, vm;
#pragma unroll
        for (int l = 0; l < 8; ++l) { va.p[l] = 0; vm.p[l] = 0; }
        int groups = 0;
        const uint64_t* col = geno + word;
        int* mine = s_cnt + threadIdx.x;
        for (int rb = r0; rb < r1; rb += 16) {
            // 16 rows in flight per thread (128 B each from 16 different DRAM pages), consumed as two groups of 8
            uint64_t w[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int r = rb + i;
                w[i] = r < r1 ? col[(int64_t)r * row_words] : 0ull;                 // 0 = g==0: adds to no counter
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                uint64_t xa[8], xm[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    // the packed word itself is counted: its even bits are set for g in {1, missing}, its odd bits for
                    // g in {2, missing}; the missing calls are counted separately and taken off at the end
                    xa[i] = w[8 * h + i];
                    xm[i] = w[8 * h + i] & (w[8 * h + i] >> 1) & M;   // missing at the even bit
                }
                vc_add8(va, xa);
                vc_add8(vm, xm);
            }
            groups += 2;
            if (groups >= 30) {                               // 240 rows: the planes hold at most 255
                vc_flush(va, mine, mine + 32 * kCntCol);
                vc_flush(vm, mine + 2 * 32 * kCntCol, nullptr);
                groups = 0;
            }
        }
        if (groups) {
            vc_flush(va, mine, mine + 32 * kCntCol);
            vc_flush(vm, mine + 2 * 32 * kCntCol, nullptr);
        }
    }
    __syncthreads();
    const int rows = max(0, r1 - r0);
    for (int i = threadIdx.x; i < 32 * 256; i += 256) {       // i = SNP within the CTA's 8192: consecutive → coalesced
        const long long s = (long long)blockIdx.x * 8192 + i;
        if (s >= L0) continue;
        const int slot = (i & 31) * kCntCol + (i >> 5);
        const int nm = s_cnt[2 * 32 * kCntCol + slot];
        const int n1 = s_cnt[slot] - nm, n2 = s_cnt[32 * kCntCol + slot] - nm;
        const int nonmiss = rows - nm;
        atomicAdd(&counts[0 * L0 + s], n1 + 2 * n2);
        atomicAdd(&counts[1 * L0 + s], 2 * nonmiss);
        atomicAdd(&counts[2 * L0 + s], nonmiss - n1);
        atomicAdd(&counts[3 * L0 + s], nonmiss);
    }
}

cudaError_t launch_count_packed(const uint64_t* geno, int64_t row_words, int n_ind, long long L0,
                                int* counts, cudaStream_t st)
{
    if (!n_ind || !L0) return cudaSuccess;
    const long long n_words = (L0 + 31) >> 5;
    const unsigned gx = (unsigned)((n_words + 255) / 256);
    int gy = (int)((148ll * 2 + gx - 1) / gx);            // about one wave of 2 CTAs per SM
    gy = std::max(1, std::min(gy, (n_ind + 63) / 64));
    int rpb = (n_ind + gy - 1) / gy;
    rpb = ((rpb + 15) / 16) * 16;
    gy = (n_ind + rpb - 1) / rpb;
    dim3 grid(gx, gy);
    const size_t smem = 3 * 32 * kCntCol * sizeof(int);       // 96 KB
    cudaError_t e = cudaFuncSetAttribute(count_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    count_packed_kernel<<<grid, 256, smem, st>>>(geno, row_words, n_ind, L0, rpb, counts);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// freq + keep mask (garlic-data.cpp:141, :968, :1070-1073) from reduced counts.
// ------------------------------------------------------------------------------------------
__global__ void freq_keep_kernel(const int* __restrict__ counts, long long L0, const int* __restrict__ pos,
                                 const int* __restrict__ chr_of, const int* __restrict__ chr_param /*[C][4]*/,
                                 int oob, double* __restrict__ freq, uint8_t* __restrict__ keep)
{
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < L0; s += (long long)gridDim.x * blockDim.x) {
        const int na = counts[s], tot = counts[L0 + s];
        const double f = (tot == 0) ? 0.0 : ((double)na / (double)tot);
        freq[s] = f;
        bool k = (f > 0 && f < 1);
        if (oob) {
            const int* cp = chr_param + 4 * chr_of[s];   // scaffold first, last, centromere start, end
            const int p = pos[s];
            k = k && !(p < cp[0]) && !(p > cp[1]) && !(p > cp[2] && p < cp[3]);
        }
        keep[s] = k;
    }
}

cudaError_t launch_freq_keep(const int* counts, long long L0, const int* pos, const int* chr_of,
                             const int* chr_param, int oob, double* freq, uint8_t* keep, cudaStream_t st)
{
    if (!L0) return cudaSuccess;
    long long blocks = (L0 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    freq_keep_kernel<<<(unsigned)blocks, 256, 0, st>>>(counts, L0, pos, chr_of, chr_param, oob, freq, keep);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// Keep-mask bookkeeping on the device (the exclusive scan behind filterMonomorphic*Sites' compaction):
// one thread per SNP, a warp = one 32-SNP input word, so the keep bits of a word are a ballot.
//   keep_count_kernel   : kept SNPs per 1024-SNP block
//   keep_scan_kernel    : exclusive scan of the block counts (single CTA), total → *total
//   keep_scatter_kernel : gather list src[] (kept SNP -> source SNP; the compaction plan of squeeze.cu is made from it),
//                         kept offset of each chromosome
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
keep_count_kernel(const uint8_t* __restrict__ keep, long long L0, int* __restrict__ block_counts)
{
    __shared__ int s_w[32];
    const long long s = (long long)blockIdx.x * 1024 + threadIdx.x;
    const bool k = s < L0 && keep[s];
    const unsigned m = __ballot_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = __popc(m);
    __syncthreads();
    if (threadIdx.x < 32) {
        int v = s_w[threadIdx.x];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) block_counts[blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(1024)
keep_scan_kernel(int* __restrict__ block_counts, int n_blocks, int* __restrict__ total)
{
    __shared__ int s_w[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < n_blocks; base += 1024) {
        const int i = base + threadIdx.x;
        const int v = i < n_blocks ? block_counts[i] : 0;
        int incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) s_w[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            const int w = s_w[threadIdx.x];
            int wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (threadIdx.x >= o) wi += t;
            }
            s_w[threadIdx.x] = wi - w;   // exclusive warp offsets
        }
        __syncthreads();
        const int carry = s_carry;
        if (i < n_blocks) block_counts[i] = carry + s_w[threadIdx.x >> 5] + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_w[31] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

__global__ void __launch_bounds__(1024)
keep_scatter_kernel(const uint8_t* __restrict__ keep, long long L0, const int* __restrict__ block_offsets,
                    const int* __restrict__ chr_of0, int n_chr, const int* __restrict__ total, int* __restrict__ src,
                    int* __restrict__ chr_off_kept)
{
    __shared__ int s_w[32];
    const long long s = (long long)blockIdx.x * 1024 + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool k = s < L0 && keep[s];
    const unsigned m = __ballot_sync(0xffffffffu, k);
    const int before = __popc(m & ((1u << lane) - 1u));
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x < 32) {
        const int w = s_w[threadIdx.x];
        int wi = w;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (threadIdx.x >= o) wi += t;
        }
        s_w[threadIdx.x] = wi - w;
    }
    __syncthreads();
    if (s >= L0) return;
    const int d = block_offsets[blockIdx.x] + s_w[warp] + before;   // kept SNPs before s
    if (k) src[d] = (int)s;
    if (s == 0 || chr_of0[s] != chr_of0[s - 1]) chr_off_kept[chr_of0[s]] = d;
    if (s == 0) chr_off_kept[n_chr] = *total;
}

cudaError_t launch_keep_scan(const uint8_t* keep, long long L0, const int* chr_of0, int n_chr, int* block_counts,
                             int* total, int* src, int* chr_off_kept, cudaStream_t st)
{
    if (!L0) return cudaSuccess;
    const int n_blocks = (int)((L0 + 1023) / 1024);
    keep_count_kernel<<<n_blocks, 1024, 0, st>>>(keep, L0, block_counts);
    keep_scan_kernel<<<1, 1024, 0, st>>>(block_counts, n_blocks, total);
    keep_scatter_kernel<<<n_blocks, 1024, 0, st>>>(keep, L0, block_counts, chr_of0, n_chr, total, src, chr_off_kept);
    return cudaGetLastError();
}

// Bad adjacent pairs (gap > MAX_GAP or overlapping the centromere, inGap garlic-roh.cpp:11-16,60-61) of the kept
// SNPs: appends i for every bad pair (i-1,i) inside a chromosome; the host sorts the short list into stretches.
__global__ void bad_pairs_kernel(const int* __restrict__ pos, const int* __restrict__ chr_of, const int* __restrict__ cen,
                                 int max_gap, long long L, int* __restrict__ list, unsigned* __restrict__ count, unsigned cap,
                                 uint32_t* __restrict__ bad_bits)
{
    // bad_bits: bit i set <=> no window may hold both SNP i-1 and SNP i (a gap / centromere pair, or a chromosome start):
    // what the thinned pass 1 tests on the device, so that it needs nothing from the host (thin_windows_kernel)
    const long long n_round = (L + 31) & ~31ll;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_round; i += (long long)gridDim.x * blockDim.x) {
        bool bad = false;
        if (i >= 1 && i < L) {
            const int c = chr_of[i];
            if (c != chr_of[i - 1]) bad = true;
            else {
                const int qs = pos[i - 1], qe = pos[i], ts = cen[2 * c], te = cen[2 * c + 1];
                const bool gap = (ts <= qs && te >= qs) || (ts <= qe && te >= qe) || (ts >= qs && te <= qe);
                if ((qe - qs > max_gap) || gap) {
                    bad = true;
                    const unsigned p = atomicAdd(count, 1u);
                    if (p < cap) list[p] = (int)i;
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, bad);
        if ((threadIdx.x & 31) == 0) bad_bits[i >> 5] = m;
    }
}
cudaError_t launch_bad_pairs(const int* pos, const int* chr_of, const int* cen, int max_gap, long long L, int* list,
                             unsigned* count, unsigned cap, uint32_t* bad_bits, cudaStream_t st)
{
    if (L < 1) return cudaSuccess;
    long long blocks = (L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    bad_pairs_kernel<<<(unsigned)blocks, 256, 0, st>>>(pos, chr_of, cen, max_gap, L, list, count, cap, bad_bits);
    return cudaGetLastError();
}

// gather a per-SNP int array through src[]
__global__ void gather_i32_kernel(const int* in, const int* src, long long L, int* out)
{
    for (long long d = blockIdx.x * (long long)blockDim.x + threadIdx.x; d < L; d += (long long)gridDim.x * blockDim.x) out[d] = in[src[d]];
}
cudaError_t launch_gather_i32(const int* in, const int* src, long long L, int* out, cudaStream_t st)
{
    if (!L) return cudaSuccess;
    long long blocks = (L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    gather_i32_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, src, L, out);
    return cudaGetLastError();
}

// GL rows: gather kept columns, apply the GQ/GL/PL → per-genotype error transform (garlic-data.cpp:1555-1577) and
// evaluate lod() of every genotype in the same pass, so that the walker only streams per-genotype LOD values.
// type: 0 GQ, 1 GL, 2 PL, -1 = already an error.
__device__ __forceinline__ double gl_to_error(double gl, int type)
{
    if (type == 0) {
        gl /= (-10.0);
        gl = (gl > -10) ? gl : -10;
        gl = pow(10.0, gl);
    } else if (type == 1) {
        gl = (gl > -10) ? gl : -10;
        gl = 1 - pow(10.0, gl);
    } else if (type == 2) {
        gl /= (-10.0);
        gl = (gl > -10) ? gl : -10;
        gl = 1 - pow(10.0, gl);
    } else return gl;
    if (gl <= 0) gl = 0.0000000000000001;
    if (gl > 1) gl = 1;
    return gl;
}

// K3-GL: compaction of the per-genotype likelihood matrix fused with readTGLSData's error transform and lod()
// (evaluated once per genotype here instead of twice per window step in the walker), written lane-interleaved
// (common.cuh:gl_lane): out[group][d][lane].  A CTA transposes a tile of 32 individuals x 64 kept SNPs through shared
// memory: reads run along the SNP axis of the caller's individual-major matrix, writes are whole 16 KB slabs.
// Covers d in [0, out_stride) and all 32 lanes of the last group: pad SNPs and absent individuals are written as 0.
//
// The error transform is a pow() per genotype, and likelihood files hold few distinct values (phred-scaled integers):
// every warp keeps a direct-mapped memo of (raw value -> error) in shared memory, filled with the results of the same
// gl_to_error() call, so a hit returns bit for bit what the call would.  One lane per slot writes (match_any), the
// warp synchronises between the write and the next probe: no torn entries.  All-distinct data only pay the probe.
constexpr int kGlTile = 64;
constexpr int kGlMemo = 128;                // entries per warp (16 B each): 8 warps x 2 KB
struct GlMemoEntry { unsigned long long key; double val; };

__device__ __forceinline__ double gl_error_memo(double raw, int type, bool on, GlMemoEntry* memo)
{
    // every lane of the warp calls this (inactive ones with on = false)
    const unsigned long long key = (unsigned long long)__double_as_longlong(raw);
    const unsigned slot = (unsigned)((key * 0x9E3779B97F4A7C15ull) >> 57);       // 7 bits
    const GlMemoEntry e = memo[slot];
    const bool hit = on && e.key == key;
    double v = e.val;
    const bool miss = on && !hit;
    if (__any_sync(0xffffffffu, miss)) {
        if (miss) v = gl_to_error(raw, type);
        // one writer per slot: the lowest missing lane among those that map to it
        const unsigned peers = __match_any_sync(0xffffffffu, miss ? slot : 0xffffffffu);
        if (miss && (int)(__ffs((int)peers) - 1) == (int)(threadIdx.x & 31)) { memo[slot].key = key; memo[slot].val = v; }
        __syncwarp();
    }
    return v;
}

__global__ void __launch_bounds__(256)
compact_gl_kernel(const double* __restrict__ in, int64_t in_stride, const int* __restrict__ src,
                  long long L, const uint64_t* __restrict__ geno0, int64_t row_words0,
                  const double* __restrict__ freq0, double* __restrict__ out, int64_t out_stride,
                  int n_ind, int type)
{
    __shared__ double tile[kGlTile][33];
    __shared__ GlMemoEntry memo_s[8][kGlMemo];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    GlMemoEntry* memo = memo_s[warp];
    // an impossible key: the bit pattern of a NaN payload no text or caller value produces by accident matters little —
    // a raw value with exactly these bits would read val = 0 once; use the one pattern gl_to_error maps to itself
    for (int i = lane; i < kGlMemo; i += 32) { memo[i].key = 0xfff8dead0000beefull; memo[i].val = gl_to_error(__longlong_as_double((long long)0xfff8dead0000beefull), type); }
    __syncwarp();
    const bool use_memo = type >= 0;
    const long long tiles_per_group = (out_stride + kGlTile - 1) / kGlTile;
    const long long total = tiles_per_group * ((n_ind + 31) / 32);
    for (long long u = blockIdx.x; u < total; u += gridDim.x) {
        const int group = (int)(u / tiles_per_group);
        const long long d0 = (u % tiles_per_group) * kGlTile;
#pragma unroll
        for (int h = 0; h < kGlTile / 32; ++h) {
            const long long d = d0 + lane + 32 * h;
            const int s = d < L ? src[d] : -1;
            const double f = s >= 0 ? freq0[s] : 0.0;
            // the four rows' raw values and genotype words first: independent loads in flight before any arithmetic
            double raw[4];
            uint64_t gw[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int i = group * 32 + warp + 8 * r;
                const bool on = s >= 0 && i < n_ind;
                raw[r] = on ? in[(int64_t)i * in_stride + s] : 0.0;
                gw[r] = on ? geno0[(int64_t)i * row_words0 + (s >> 5)] : 0ull;
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int il = warp + 8 * r, i = group * 32 + il;
                const bool on = s >= 0 && i < n_ind;
                double v = 0.0;
                // per-genotype error (readTGLSData) → per-genotype LOD (lod(), garlic-roh.cpp:355-386)
                const double e = use_memo ? gl_error_memo(raw[r], type, on, memo) : raw[r];
                if (on) v = lod_eval((int)(gw[r] >> (2 * (s & 31))) & 3, f, e);
                tile[lane + 32 * h][il] = v;
            }
        }
        __syncthreads();
        double* o = out + ((int64_t)group * out_stride + d0) * kGlLanes;
        const int rows = (int)((out_stride - d0) < kGlTile ? (out_stride - d0) : kGlTile);
        for (int e = threadIdx.x; e < rows * 32; e += 256) o[e] = tile[e >> 5][e & 31];
        __syncthreads();
    }
}

cudaError_t launch_compact_gl(const double* in, int64_t in_stride, const int* src, long long L, const uint64_t* geno0,
                              int64_t row_words0, const double* freq0, double* out, int64_t out_stride, int n_ind, int type,
                              cudaStream_t st)
{
    if (!n_ind) return cudaSuccess;
    long long blocks = ((out_stride + kGlTile - 1) / kGlTile) * ((n_ind + 31) / 32);
    if (blocks > 148 * 32) blocks = 148 * 32;
    compact_gl_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, in_stride, src, L, geno0, row_words0, freq0, out, out_stride, n_ind, type);
    return cudaGetLastError();
}

// gather a per-SNP double / int array through src[]
__global__ void gather_f64_kernel(const double* in, const int* src, long long L, double* out)
{
    for (long long d = blockIdx.x * (long long)blockDim.x + threadIdx.x; d < L; d += (long long)gridDim.x * blockDim.x) out[d] = in[src[d]];
}
cudaError_t launch_gather_f64(const double* in, const int* src, long long L, double* out, cudaStream_t st)
{
    if (!L) return cudaSuccess;
    long long blocks = (L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    gather_f64_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, src, L, out);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// K4: per-SNP LOD table lut[s][g], g = 0,1,2,missing, for a global --error (garlic-roh.cpp:355-386)
// and, for wLOD, the per-SNP score table lod*nomut*norec evaluated left to right (:246-249).
// ------------------------------------------------------------------------------------------
__global__ void build_lut_kernel(const double* __restrict__ freq, long long L, double error, double* __restrict__ lut)
{
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < L; s += (long long)gridDim.x * blockDim.x) {
        const double f = freq[s];
        double4 v;
        v.x = lod_eval(0, f, error); v.y = lod_eval(1, f, error); v.z = lod_eval(2, f, error); v.w = 0.0;
        reinterpret_cast<double4*>(lut)[s] = v;
    }
}
cudaError_t launch_build_lut(const double* freq, long long L, double error, double* lut, cudaStream_t st)
{
    if (!L) return cudaSuccess;
    long long blocks = (L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    build_lut_kernel<<<(unsigned)blocks, 256, 0, st>>>(freq, L, error, lut);
    return cudaGetLastError();
}

// wLOD per-SNP weights: nomut = exp(-2*M*mu*Δbp), norec = exp(-2*M*1*Δcm); Δ of a chromosome's
// first SNP is its absolute position (garlic-roh.cpp:134-140, :246-247).
__global__ void wlod_weights_kernel(const int* __restrict__ pos, const double* __restrict__ gpos,
                                    const int* __restrict__ chr_of, const int* __restrict__ chr_start, long long L,
                                    double mu, int M, double* __restrict__ nomut, double* __restrict__ norec)
{
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < L; s += (long long)gridDim.x * blockDim.x) {
        const bool first = (s == chr_start[chr_of[s]]);
        const double pi = first ? (double)pos[s] : (double)(pos[s] - pos[s - 1]);
        const double gi = first ? gpos[s] : (gpos[s] - gpos[s - 1]);
        nomut[s] = exp(-2.0 * M * mu * pi);
        norec[s] = exp(-2.0 * M * 1 * gi);
    }
}
cudaError_t launch_wlod_weights(const int* pos, const double* gpos, const int* chr_of, const int* chr_start,
                                long long L, double mu, int M, double* nomut, double* norec, cudaStream_t st)
{
    if (!L) return cudaSuccess;
    long long blocks = (L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    wlod_weights_kernel<<<(unsigned)blocks, 256, 0, st>>>(pos, gpos, chr_of, chr_start, L, mu, M, nomut, norec);
    return cudaGetLastError();
}

// score table for wLOD with a global error: slut[s][g] = lod(g)*nomut[s]*norec[s]
__global__ void build_wlut_kernel(const double* __restrict__ lut, const double* __restrict__ nomut,
                                  const double* __restrict__ norec, long long L, double* __restrict__ wlut)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < 4 * L; t += (long long)gridDim.x * blockDim.x) {
        const long long s = t >> 2;
        wlut[t] = lut[t] * nomut[s] * norec[s];
    }
}
cudaError_t launch_build_wlut(const double* lut, const double* nomut, const double* norec, long long L,
                              double* wlut, cudaStream_t st)
{
    if (!L) return cudaSuccess;
    long long blocks = (4 * L + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    build_wlut_kernel<<<(unsigned)blocks, 256, 0, st>>>(lut, nomut, norec, L, wlut);
    return cudaGetLastError();
}

}  // namespace garlic
