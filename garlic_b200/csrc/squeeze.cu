// squeeze.cu — K3 (column compaction of the packed genotype matrix, filterMonomorphic[AndOOB]Sites,
// garlic-data.cpp:871-1195, as a bit-level gather) fused with the pruning bound of K5 pass 2 (bound.cuh), and the
// candidate selection that follows once the cutoff is known.
//
// squeeze_bound_kernel: one lane = one individual, one warp = 32 individuals marching along the SNP axis over a range of
// 256-SNP pieces.  The rows' input half-words stream through a per-warp shared-memory ring filled by cp.async (each
// copy instruction moves 128 contiguous bytes of two rows, so global reads are whole lines instead of one sector per
// lane); the compaction plan (which input half-words make up an output half-word) is the same for every individual and
// is read with warp-uniform loads; the compacted half-word goes (a) through a shared staging tile to coalesced
// 128-byte row stores and (b), still in its register, into the bound (three POPC and a dozen integer operations).
// SQUEEZE = false: bound only, over rows that are already compacted (another window size on the same data).
// BOUND = false: compaction only (GL / weighted modes, window sizes outside the bound's range).
// STORE = false (with SQUEEZE): the bound over the uncompacted rows, compacted in registers only and never written —
// when the only consumer is the pruned walker (walk_units_kernel), which compacts its few candidates' slices itself.
// Without the output tile a CTA needs 36 KB instead of 54 KB of shared memory: five CTAs per SM instead of four.
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include "common.cuh"
#include "bound.cuh"
#include "kernels.h"

namespace garlic {

namespace {
constexpr int kSqWarps = 4;                               // 54 KB (36 KB without the output tile) of shared memory per CTA
constexpr int kSqStages = 4;                              // ring = 4 stages of 16 input half-words (64 B) per row
constexpr int kSqStageHw = 16, kSqStageShift = 4;
constexpr int kSqRingHw = kSqStages * kSqStageHw;         // input half-word a of a row sits at ring position a & 63
constexpr int kSqRowBytes = kSqRingHw * 4 + 8;            // + 8 B pad: rows start 2 banks apart
constexpr int kSqRingBytes = 32 * kSqRowBytes;            // 32 rows
constexpr int kSqOutRowBytes = 144;                       // output staging: 16 words (128 B) per row + 16 B pad
constexpr int kSqOutBytes = 32 * kSqOutRowBytes;
constexpr int kSqStashBytes = 32 + 256 + 256;             // the current piece's plan codes, bound tables, full plan heads
constexpr int kSqWarpBytes = kSqRingBytes + kSqOutBytes + kSqStashBytes;
constexpr int kSqWarpBytesNoTile = kSqRingBytes + kSqStashBytes;
// CTAs per SM: the tiled layout is held to four by shared memory (and runs at up to 128 registers); without the tile six
// would fit, but the bound's register state (two 16-entry prefix rings, the 20-register input window, 16 half-words)
// spills below 96 registers, which allow five
constexpr int kSqCtasPerSm = 4, kSqCtasPerSmNoTile = 5;

__device__ __forceinline__ uint32_t sq_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async8(uint32_t dst_smem, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_dyn(int pending)     // at most `pending` (0..7) newest groups still in flight
{
    switch (pending) {
        case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
        case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
        case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
        case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
        case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
        default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
    }
}
}  // namespace

// ------------------------------------------------------------------------------------------
// tables of the bound for window size W (bound.cuh): one thread per half-word / block
// ------------------------------------------------------------------------------------------
// A CTA makes the entries of kBtHw consecutive half-words.  The table rows they look at — 16 SNPs each for the level
// planes, and the W + 15 SNPs behind block q - C2 for its Bmax — overlap almost completely between neighbours, so the
// CTA's whole range of the per-SNP table is staged once by one bulk copy (cp.async.bulk) and the (unchanged, strictly
// ordered) arithmetic of bound.cuh then runs out of shared memory: one thread per half-word reading 512 contiguous
// bytes of global memory per step had made this little kernel cost as much as the thinned pass 1.
constexpr int kBtHw = 128;
namespace {
__device__ __forceinline__ void bt_mbar_init(uint64_t* bar)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sq_smem_u32(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bt_bulk_load(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sq_smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(sq_smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(sq_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bt_mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BT_WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra BT_WAIT_DONE;\n"
        "bra BT_WAIT_LOOP;\n"
        "BT_WAIT_DONE:\n"
        "}\n" ::"r"(sq_smem_u32(bar)), "r"(parity) : "memory");
}
}  // namespace

__global__ void __launch_bounds__(kBtHw)
bound_tables_kernel(const double* __restrict__ lut, long long n_hw, long long L, int W, uint4* __restrict__ hw, int* __restrict__ invalid,
                    int stage_snps, long long n_tab)
{
    extern __shared__ __align__(128) double bt_smem[];       // [stage_snps][4] | mbarrier
    uint64_t* bar = reinterpret_cast<uint64_t*>(bt_smem + (size_t)stage_snps * 4);
    const int c2 = bound_c2(W);
    if (threadIdx.x == 0) bt_mbar_init(bar);
    __syncthreads();
    uint32_t phase = 0;
    for (long long k0 = (long long)blockIdx.x * kBtHw; k0 < n_hw; k0 += (long long)gridDim.x * kBtHw) {
        // SNPs [s_lo, s_lo + stage_snps): from block k0 - c2 (never below 0) to the end of half-word k0 + kBtHw - 1
        const long long kb = k0 >= c2 ? k0 - c2 : 0;
        const long long s_lo = kb * 16;
        __syncthreads();                                   // the previous range has been read
        const long long have = n_tab - s_lo < stage_snps ? n_tab - s_lo : stage_snps;   // table entries that exist
        if (threadIdx.x == 0) bt_bulk_load(bt_smem, lut + s_lo * 4, (uint32_t)(have * 32), bar);   // one bulk copy per range
        for (long long i = have * 4 + threadIdx.x; i < (long long)stage_snps * 4; i += kBtHw) bt_smem[i] = 0.0;   // beyond the table: zero
        bt_mbar_wait(bar, phase);
        phase ^= 1u;
        __syncthreads();
        const long long k = k0 + threadIdx.x;
        if (k < n_hw) {
            const double* tab = bt_smem - s_lo * 4;           // tab + s * 4 is SNP s of the staged range
            int bad = 0;
            uint4 e = bound_hw_entry(tab, k, L, &bad);
            e.w = k >= c2 ? (uint32_t)bound_block_max(tab, k - c2, W) : 0u;   // what the step at half-word k evaluates
            hw[k] = e;
            if (bad) atomicOr(invalid, 1);
        }
    }
}

cudaError_t launch_bound_tables(const double* lut, long long n_tab, long long n_hw, long long L, int W, uint4* hw, int* invalid, cudaStream_t st)
{
    if (!n_hw) return cudaSuccess;
    // staged SNPs: the kBtHw half-words themselves plus C2 blocks in front, and behind block k - C2 its last window
    // (start + 15 + W); whichever reaches further
    const int c2 = bound_c2(W);
    const int stage_snps = std::max(16 * (kBtHw + c2), 16 * (kBtHw - 1) + 16 + W + 16);
    const size_t smem = (size_t)stage_snps * 32 + 16;
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(bound_tables_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long blocks = (n_hw + kBtHw - 1) / kBtHw;
    if (blocks > 148 * 8) blocks = 148 * 8;
    bound_tables_kernel<<<(unsigned)blocks, kBtHw, smem, st>>>(lut, n_hw, L, W, hw, invalid, stage_snps, n_tab);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// compaction plan: one thread per output half-word (bound.cuh:plan_half) from the gather list src[]
// ------------------------------------------------------------------------------------------
__global__ void plan_kernel(const int* __restrict__ src, const int* __restrict__ n_kept, long long n_q,
                            uint4* __restrict__ head, uint4* __restrict__ segs, uint16_t* __restrict__ fast,
                            int2* __restrict__ piece_rng)
{
    const long long L = *n_kept;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n_q; q += (long long)gridDim.x * blockDim.x) {
        uint4 hd;
        plan_half(src, L, q, &hd, segs + q * kPlanSegMax);
        head[q] = hd;
        const long long d0 = (q & ~15ll) * 16;             // first kept SNP of the piece
        const int a0 = d0 < L ? src[d0] >> 4 : -1;         // first input half-word the piece reads
        const uint32_t code = a0 >= 0 ? plan_fast_code(hd, a0 & ~1, (int)(q & 15)) : 0xffffu;
        fast[q] = (uint16_t)code;
        // per piece: x = first input half-word (-1: nothing to read), y = (last - first, saturated) << 16 | mask of the
        // half-words that need the slow path — eight bytes, both used: a wider load with a dead component would make
        // its register wait for the load at once
        const unsigned slow = __ballot_sync(__activemask(), code == 0xffffu);
        if ((q & 15) == 0) {
            int2 r = make_int2(-1, 0);
            if (a0 >= 0) {
                const long long d1 = d0 + kPiece - 1 < L ? d0 + kPiece - 1 : L - 1;
                const int a1 = src[d1] >> 4;
                r.x = a0;
                r.y = (int)((unsigned)(a1 - a0 < 0xffff ? a1 - a0 : 0xffff) << 16);
            }
            r.y |= (int)((slow >> (threadIdx.x & 16)) & 0xffffu);
            piece_rng[q >> 4] = r;
        }
    }
}

cudaError_t launch_plan(const int* src, const int* n_kept, long long n_q, uint4* head, uint4* segs, uint16_t* fast,
                        int2* piece_rng, cudaStream_t st)
{
    if (!n_q) return cudaSuccess;
    long long blocks = (n_q + 127) / 128;
    if (blocks > 148 * 16) blocks = 148 * 16;
    plan_kernel<<<(unsigned)blocks, 128, 0, st>>>(src, n_kept, n_q, head, segs, fast, piece_rng);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// the fused pass
// ------------------------------------------------------------------------------------------
template <bool SQUEEZE, bool STORE, bool BOUND, int C2, int LAG, bool PARTIAL>
__global__ void __launch_bounds__(kSqWarps * 32, SQUEEZE && STORE ? 0 : kSqCtasPerSmNoTile)
squeeze_bound_kernel(const SqueezeParams P)
{
    constexpr bool TILE = SQUEEZE && STORE;               // the output staging tile exists
    extern __shared__ __align__(16) unsigned char sq_smem[];
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform for the compiler
    const int lane = threadIdx.x & 31;
    unsigned char* ring_s = sq_smem + (size_t)warp * (TILE ? kSqWarpBytes : kSqWarpBytesNoTile);
    unsigned char* out_s = ring_s + kSqRingBytes;
    const uint32_t* my_ring = reinterpret_cast<const uint32_t*>(ring_s + lane * kSqRowBytes);
    const uint2* my_ring64 = reinterpret_cast<const uint2*>(ring_s + lane * kSqRowBytes);
    uint32_t* my_out = reinterpret_cast<uint32_t*>(out_s + lane * kSqOutRowBytes);   // this lane's 32 output half-words
    uint32_t* sh_fast = reinterpret_cast<uint32_t*>(out_s + (TILE ? kSqOutBytes : 0));   // the piece's 16 two-byte plan codes
    uint4* sh_tab = reinterpret_cast<uint4*>(sh_fast + 8);                 // its 16 bound table entries (lanes 0..15)
    uint4* sh_head = sh_tab + 16;                                          // its 16 full plan heads (lanes 16..31): slow path
    const int c4 = lane & 7, rsel4 = lane >> 3;           // copies and flushes: a quarter-warp covers one row
    const uint32_t ring_u32 = sq_smem_u32(ring_s);
    const int n_rg = (P.n_ind + 31) >> 5;
    const long long n_kept = TILE ? (long long)*P.n_kept : 0;
    const long long n_out_words = TILE ? (n_kept + 31) >> 5 : 0;
    const long long n_tasks = (long long)n_rg * P.n_col_tasks;
    for (long long task = (long long)blockIdx.x * kSqWarps + warp; task < n_tasks; task += (long long)gridDim.x * kSqWarps) {
        const int rg = (int)(task % n_rg), ct = (int)(task / n_rg);
        const int pc_lo = ct * P.pieces_per_task;
        const int pc_hi = min(P.n_pieces, pc_lo + P.pieces_per_task);
        const int row = rg * 32 + lane;
        const bool active = row < P.n_ind;
        const uint32_t* grow32 = reinterpret_cast<const uint32_t*>(P.gin + (int64_t)(active ? row : P.n_ind - 1) * P.in_words);
        // ---- input ring: stage t = input half-words [16 t, 16 t + 16) of the 32 rows, in ring positions (16 t) & 63 …
        int issued = 0;                                    // stages below this one have been issued (or skipped)
        // the eight rows this lane copies for every stage (row 4 i + lane / 8, eight bytes at column lane % 8)
        const uint64_t* cp_src[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int gr = rg * 32 + 4 * i + rsel4;
            gr = gr < P.n_ind ? gr : P.n_ind - 1;
            cp_src[i] = P.gin + (int64_t)gr * P.in_words + c4;
        }
        const uint32_t cp_dst = ring_u32 + (uint32_t)(rsel4 * kSqRowBytes + c4 * 8);
        auto issue = [&](int t) {
            const long long w0 = (long long)t * (kSqStageHw / 2);   // first 64-bit word of the stage
            if (w0 + kSqStageHw / 2 <= P.in_words) {
                const uint32_t dst = cp_dst + (uint32_t)((t & (kSqStages - 1)) * (kSqStageHw * 4));
#pragma unroll
                for (int i = 0; i < 8; ++i) cp_async8(dst + i * 4 * kSqRowBytes, cp_src[i] + w0);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        // Input half-words [a_lo, a_hi] must be readable: at most three stages (the usual case: a piece reads about 17
        // consecutive input half-words), the fourth ring stage stays in flight ahead.  Returns false when the range is
        // wider (a long run of dropped SNPs inside the piece): that piece reads global memory directly.
        auto stage_in = [&](int a_lo, int a_hi) -> bool {
            if (a_hi < a_lo) return true;                  // nothing to read
            const int lo_st = a_lo >> kSqStageShift, hi_st = a_hi >> kSqStageShift;
            if (hi_st - lo_st > 2) return false;           // (the register window of phase A spans at most three stages)
            if (issued < lo_st) {                          // stages nobody reads are never copied; what is still in
                asm volatile("cp.async.wait_group 0;" ::: "memory");   // flight lands before its slot gets a new owner
                issued = lo_st;
            }
            __syncwarp();                                  // every lane is done with the stages about to be overwritten
#pragma unroll 1
            while (issued <= lo_st + kSqStages - 1) issue(issued++);
            cp_async_wait_dyn(issued - 1 - hi_st);
            __syncwarp();
            return true;
        };

        BoundState S;
        bound_reset(S);
        // The plan codes and bound tables of a piece are the same for every individual: a few lanes fetch them with one
        // coalesced load each, one piece ahead (the L2 latency hides behind a whole piece of work), and park them in
        // shared memory, from where every half-word step takes them with broadcast reads.
        uint32_t r_fast = 0u;
        uint4 r_tab = make_uint4(0u, 0u, 0u, 0u);         // lanes 0..15: bound table entry; lanes 16..31: full plan head
        int2 r_rng = make_int2(-1, 0);
        const uint4* tab_src = lane < 16 ? P.hw + lane : P.plan_head + (lane - 16);
        const bool tab_on = lane < 16 ? BOUND : SQUEEZE;
        auto fetch = [&](int piece) {
            if (SQUEEZE && lane < 8) r_fast = P.plan_fast[(long long)piece * 8 + lane];
            if (tab_on) r_tab = tab_src[(long long)piece * 16];
            r_rng = SQUEEZE ? P.piece_rng[piece] : make_int2(piece * 16, 15 << 16);
        };
        fetch(pc_lo);
        const int pi_end = BOUND ? pc_hi + 1 : pc_hi;     // one more piece drains the bound's C2 half-words of lag
#pragma unroll 1
        for (int pi = pc_lo; pi < pi_end; ++pi) {
            const long long qb = (long long)pi * 16;
            __syncwarp();                                  // the previous piece's stash has been read
            const int2 rng = r_rng;
            const bool ring_ok = stage_in(rng.x, rng.x < 0 ? -2 : rng.x + (int)((unsigned)rng.y >> 16));
            if (SQUEEZE && lane < 8) sh_fast[lane] = r_fast;
            if (tab_on) sh_tab[lane] = r_tab;              // lanes 16..31 land in sh_head
            __syncwarp();
            fetch(pi + 1);                                 // the tables have four pieces of slack
            uint32_t hreg[16];                             // the piece's 16 half-words (registers: every index is static)
            uint32_t* dst = my_out + ((pi & 1) << 4);
            if (SQUEEZE) {
                // ---- phase A: the piece's 16 output half-words.  Its input window — 20 half-words from the (even) first
                // source half-word on — is read into registers with ten conflict-free 8-byte loads; the usual output
                // half-word (16 consecutive sources, at most one dropped SNP in between) is then a funnel shift of the
                // 64-bit window at register I + k, k <= 2, with the fields above the dropped SNP moved down by one: no
                // branches, no further shared-memory traffic.  The others (`slow` bits of the piece) are redone below.
                uint32_t w[20];
                const uint32_t u0 = (uint32_t)rng.x >> 1;
#pragma unroll
                for (int j = 0; j < 10; ++j) {
                    const uint2 v = my_ring64[(u0 + j) & (kSqRingHw / 2 - 1)];
                    w[2 * j] = v.x; w[2 * j + 1] = v.y;
                }
#pragma unroll
                for (int I = 0; I < 16; ++I) {
                    const uint32_t cw = sh_fast[I >> 1];
                    const uint32_t b0 = __byte_perm(cw, 0u, (I & 1) ? 0x4442u : 0x4440u);   // k | sh << 2
                    const uint32_t p2 = __byte_perm(cw, 0u, (I & 1) ? 0x4443u : 0x4441u);   // 2 p
                    const uint32_t k = b0 & 3u, sh = b0 >> 2;
                    const uint32_t x0 = k == 0u ? w[I] : (k == 1u ? w[I + 1] : w[I + 2]);
                    const uint32_t x1 = k == 0u ? w[I + 1] : (k == 1u ? w[I + 2] : w[I + 3]);
                    const uint32_t x2 = k == 0u ? w[I + 2] : (k == 1u ? w[I + 3] : w[I + 4]);
                    const uint32_t lo = __funnelshift_r(x0, x1, sh), hi = __funnelshift_r(x1, x2, sh);
                    const uint32_t m = __funnelshift_lc(0xffffffffu, 0u, p2);             // the fields below the dropped one
                    hreg[I] = (lo & m) | (__funnelshift_r(lo, hi, 2u) & ~m);
                }
                if (TILE) {
#pragma unroll
                    for (int I = 0; I < 16; I += 4) *reinterpret_cast<uint4*>(dst + I) = make_uint4(hreg[I], hreg[I + 1], hreg[I + 2], hreg[I + 3]);
                }
                unsigned slow = ring_ok ? ((unsigned)rng.y & 0xffffu) : 0xffffu;
                if (slow) {                                // several dropped SNPs, long dropped runs, the end of the data
#pragma unroll 1
                    for (; slow; slow &= slow - 1u) {
                        const int I = __ffs((int)slow) - 1;
                        const uint4 hd = sh_head[I];
                        uint32_t h;
                        if (hd.x & 0x100u) {
                            const uint32_t a = hd.y;
                            if (ring_ok) h = plan_window(hd, my_ring[a & (kSqRingHw - 1)], my_ring[(a + 1) & (kSqRingHw - 1)], my_ring[(a + 2) & (kSqRingHw - 1)]);
                            else h = plan_window(hd, grow32[a], plan_need1(hd) ? grow32[a + 1] : 0u, plan_need2(hd) ? grow32[a + 2] : 0u);
                        } else {
                            h = hd.w;
                            const uint4* sg = P.plan_seg + (qb + I) * kPlanSegMax;
                            const int ns = (int)hd.x;
#pragma unroll 1
                            for (int k = 0; k < ns; ++k) {
                                const uint4 g = sg[k];
                                const uint32_t x = ring_ok ? my_ring[g.x & (kSqRingHw - 1)] : grow32[g.x];
                                h |= ((x >> g.y) & g.z) << g.w;
                            }
                        }
                        if (TILE) {
                            dst[I] = h;
                        } else {                           // (warp-uniform I: a select per register, no divergence)
#pragma unroll
                            for (int J = 0; J < 16; ++J) hreg[J] = J == I ? h : hreg[J];
                        }
                    }
                    if (TILE) {
                        __syncwarp();
#pragma unroll
                        for (int I = 0; I < 16; ++I) hreg[I] = dst[I];
                    }
                }
            } else {
                const uint4* hsrc = reinterpret_cast<const uint4*>(my_ring + (qb & (kSqRingHw - 1)));   // a piece = one stage
#pragma unroll
                for (int I = 0; I < 16; I += 4) { const uint2 v0 = reinterpret_cast<const uint2*>(hsrc)[I >> 1], v1 = reinterpret_cast<const uint2*>(hsrc)[(I >> 1) + 1]; hreg[I] = v0.x; hreg[I + 1] = v0.y; hreg[I + 2] = v1.x; hreg[I + 3] = v1.y; }
            }
            if (BOUND) {
                // ---- phase B: the bound over the 16 half-words, ring indices compile-time
#pragma unroll
                for (int I = 0; I < 16; ++I) {
                    const long long q = qb + I;
                    bound_step<C2, LAG, PARTIAL>(S, hreg[I], sh_tab[I], I, P.low_mask);
                    if (((I - C2) & 15) == 15) {           // block k = q - C2 closes its piece
                        const int piece = (int)((q - C2) >> 4);
                        if (piece >= pc_lo && piece < pc_hi && active)
                            P.pmax[(int64_t)piece * P.pmax_stride + row] = bound_pack(S.pm_all, S.pm_tail);
                        S.pm_all = -0x40000000; S.pm_tail = -0x40000000;
                    }
                }
            }
            // ---- two pieces = 16 output words per row: flush through shared memory, 128 B per row and quarter-warp
            if (TILE && pi < pc_hi && ((pi & 1) || pi == pc_hi - 1)) {
                __syncwarp();
                const long long wd = 16ll * (pi >> 1) + 2 * c4;
                if (2 * c4 < ((pi & 1) ? 16 : 8) && wd < n_out_words) {
                    const unsigned char* sp = out_s + rsel4 * kSqOutRowBytes + c4 * 16;
                    uint64_t* gp = P.gout + (int64_t)(rg * 32 + rsel4) * P.out_words + wd;
                    const int rows = min(32, P.n_ind - rg * 32);           // rows of this group that exist
#pragma unroll 4
                    for (int r = rsel4; r < rows; r += 4, sp += 4 * kSqOutRowBytes, gp += 4 * P.out_words)
                        *reinterpret_cast<uint4*>(gp) = *reinterpret_cast<const uint4*>(sp);
                }
                __syncwarp();
            }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");   // nothing of this task is still landing
        __syncwarp();
    }
}

template <bool SQUEEZE, bool STORE, bool BOUND, int C2, int LAG, bool PARTIAL>
static cudaError_t launch_sq_t(const SqueezeParams& P, unsigned grid, size_t smem, cudaStream_t st)
{
    auto kern = squeeze_bound_kernel<SQUEEZE, STORE, BOUND, C2, LAG, PARTIAL>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, kSqWarps * 32, smem, st>>>(P);
    return cudaGetLastError();
}

template <bool SQUEEZE, bool STORE, int LAG>
static cudaError_t launch_sq_c2(const SqueezeParams& P, int c2, unsigned grid, size_t smem, cudaStream_t st)
{
    switch (c2) {
        case 2: return launch_sq_t<SQUEEZE, STORE, true, 2, LAG, false>(P, grid, smem, st);
        case 3: return launch_sq_t<SQUEEZE, STORE, true, 3, LAG, false>(P, grid, smem, st);
        case 4: return launch_sq_t<SQUEEZE, STORE, true, 4, LAG, false>(P, grid, smem, st);
        case 5: return launch_sq_t<SQUEEZE, STORE, true, 5, LAG, false>(P, grid, smem, st);
        case 6: return launch_sq_t<SQUEEZE, STORE, true, 6, LAG, false>(P, grid, smem, st);
        case 7: return launch_sq_t<SQUEEZE, STORE, true, 7, LAG, false>(P, grid, smem, st);
        case 8: return launch_sq_t<SQUEEZE, STORE, true, 8, LAG, false>(P, grid, smem, st);
        case 9: return launch_sq_t<SQUEEZE, STORE, true, 9, LAG, false>(P, grid, smem, st);
        case 10: return launch_sq_t<SQUEEZE, STORE, true, 10, LAG, false>(P, grid, smem, st);
        case 11: return launch_sq_t<SQUEEZE, STORE, true, 11, LAG, false>(P, grid, smem, st);
        case 12: return launch_sq_t<SQUEEZE, STORE, true, 12, LAG, false>(P, grid, smem, st);
        case 13: return launch_sq_t<SQUEEZE, STORE, true, 13, LAG, false>(P, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

// window sizes below 32: the core is a partial half-word (bound.cuh: bound_step<…, true>), C2 = LAG = 1 or 2
template <bool SQUEEZE, bool STORE>
static cudaError_t launch_sq_partial(const SqueezeParams& P, int c2, unsigned grid, size_t smem, cudaStream_t st)
{
    if (c2 == 1) return launch_sq_t<SQUEEZE, STORE, true, 1, 1, true>(P, grid, smem, st);
    if (c2 == 2) return launch_sq_t<SQUEEZE, STORE, true, 2, 2, true>(P, grid, smem, st);
    return cudaErrorInvalidValue;
}

// pieces per warp task: enough tasks for three waves of the warps an SM holds, an even number of pieces (the output
// staging tile holds two), and long enough that the extra piece the bound drains costs a few percent
int squeeze_pieces_per_task(int n_ind, int n_pieces, int warps_per_sm)
{
    const int n_rg = (n_ind + 31) / 32;
    const int want_tasks = 148 * warps_per_sm * 3;
    int n_col = std::max(1, (want_tasks + n_rg - 1) / n_rg);
    int ppt = (n_pieces + n_col - 1) / n_col;
    ppt = std::max(ppt, 16);
    ppt += ppt & 1;
    return ppt;
}

cudaError_t launch_squeeze_bound(SqueezeParams P, bool squeeze, bool store, int c2, cudaStream_t st)
{
    if (!P.n_ind || !P.n_pieces) return cudaSuccess;
    if (!squeeze) store = false;                           // bound over compacted rows: nothing to write
    if (c2 <= 0 && !(squeeze && store)) return cudaErrorInvalidValue;
    if (squeeze && !store && P.partial) return cudaErrorInvalidValue;   // (window sizes below 32 walk compacted rows)
    const int ctas_per_sm = store ? kSqCtasPerSm : kSqCtasPerSmNoTile;
    P.pieces_per_task = squeeze_pieces_per_task(P.n_ind, P.n_pieces, ctas_per_sm * kSqWarps);
    P.n_col_tasks = (P.n_pieces + P.pieces_per_task - 1) / P.pieces_per_task;
    const int n_rg = (P.n_ind + 31) / 32;
    const long long n_tasks = (long long)n_rg * P.n_col_tasks;
    long long grid = (n_tasks + kSqWarps - 1) / kSqWarps;
    if (grid > 148ll * ctas_per_sm * 8) grid = 148ll * ctas_per_sm * 8;
    const unsigned g = (unsigned)grid;
    const size_t smem = (size_t)kSqWarps * (store ? kSqWarpBytes : kSqWarpBytesNoTile);
    if (c2 <= 0) return launch_sq_t<true, true, false, 2, 1, false>(P, g, smem, st);
    if (P.partial) return squeeze ? launch_sq_partial<true, true>(P, c2, g, smem, st) : launch_sq_partial<false, false>(P, c2, g, smem, st);
    if (P.lag != 1 && P.lag != 2) return cudaErrorInvalidValue;
    if (!squeeze) return P.lag == 1 ? launch_sq_c2<false, false, 1>(P, c2, g, smem, st) : launch_sq_c2<false, false, 2>(P, c2, g, smem, st);
    if (!store) return P.lag == 1 ? launch_sq_c2<true, false, 1>(P, c2, g, smem, st) : launch_sq_c2<true, false, 2>(P, c2, g, smem, st);
    return P.lag == 1 ? launch_sq_c2<true, true, 1>(P, c2, g, smem, st) : launch_sq_c2<true, true, 2>(P, c2, g, smem, st);
}

// ------------------------------------------------------------------------------------------
// candidate selection: one CTA per item thresholds the piece maxima of every individual (bound.cuh:
// bound_item_candidate), writes the item's dense candidate list (in no particular order) and appends one work unit per
// `lanes_per_unit` candidates to the walker's queue.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
select_kernel(const Item* __restrict__ items, int n_items, const uint32_t* __restrict__ pmax, int64_t stride, int n_ind,
              int cut_store, const int* __restrict__ invalid, int* __restrict__ cand_list, int cand_stride,
              unsigned* __restrict__ cand_cnt, int2* __restrict__ units, unsigned* __restrict__ n_units, unsigned unit_cap,
              int lanes_per_unit, int c2)
{
    __shared__ int s_n;
    const int lane = threadIdx.x & 31;
    if (*invalid) cut_store = -32768;                      // the table breaks the bound's assumptions: keep everybody
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const Item it = items[item];
        __syncthreads();                                   // s_n of the previous item has been read
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
        // one pass: a thread takes individuals t, t + 256, … (independent loads), a warp appends its candidates with one
        // shared atomic per round; the list comes out in no particular order — the runs are sorted afterwards
        int* list = cand_list + (int64_t)item * cand_stride;
        const int rounds = (n_ind + 255) >> 8;
        for (int r = 0; r < rounds; ++r) {
            const int ind = r * 256 + threadIdx.x;
            const bool c = ind < n_ind && bound_item_candidate(pmax, stride, ind, it, cut_store, c2);
            const unsigned m = __ballot_sync(0xffffffffu, c);
            if (m) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&s_n, __popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (c) list[base + __popc(m & ((1u << lane) - 1u))] = ind;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int total = s_n;
            cand_cnt[item] = (unsigned)total;
            const int nu = (total + lanes_per_unit - 1) / lanes_per_unit;
            if (nu) {
                const unsigned b = atomicAdd(n_units, (unsigned)nu);
                for (int u = 0; u < nu; ++u)
                    if (b + u < unit_cap) units[b + u] = make_int2(item, u * lanes_per_unit);
                atomicAdd(n_units + 1, (unsigned)total);  // total candidate pairs (statistics)
            }
        }
    }
}

cudaError_t launch_select(const Item* items, int n_items, const uint32_t* pmax, int64_t stride, int n_ind, int cut_store,
                          const int* invalid, int* cand_list, int cand_stride, unsigned* cand_cnt, int2* units, unsigned* n_units,
                          unsigned unit_cap, int lanes_per_unit, int c2, cudaStream_t st)
{
    if (!n_items || !n_ind) return cudaSuccess;
    const int grid = n_items < 148 * 8 ? n_items : 148 * 8;
    select_kernel<<<grid, 256, 0, st>>>(items, n_items, pmax, stride, n_ind, cut_store, invalid, cand_list, cand_stride, cand_cnt, units,
                                        n_units, unit_cap, lanes_per_unit, c2);
    return cudaGetLastError();
}

}  // namespace garlic
