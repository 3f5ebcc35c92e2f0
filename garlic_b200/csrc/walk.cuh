// walk.cuh — the per-lane fused LOD-window → cutoff → coverage → run-length walker (K5).
//
// One lane = one individual walking one Item (a chunk of a segment of valid windows) along the
// SNP axis.  Replaces, fused and without ever materialising the window matrix:
//   * calcLOD's running update win[l] = win[l-1] - lod(out) + lod(in), fresh sum at each restart
//     (reference src/garlic-roh.cpp:50-123) — same operation order, so with items = whole
//     segments the window values are bit-identical to the reference chain;
//   * the cutoff test and per-SNP coverage count inWin[] (garlic-roh.cpp:446-454) as a sliding
//     count of the last W window flags;
//   * the run-length state machine (garlic-roh.cpp:462-532) as bit-parallel edge detection on
//     32-step words of "covered" bits;
//   * optional window dump for the KDE thinning (garlic-data.cpp:2026-2069) / --raw-lod.
//
// Written __host__ __device__ so tests can run the identical logic on the CPU
// (tests/host_emu.cpp) where no GPU is available; the product path only ever runs it on the GPU.
#pragma once
#include <math.h>
#include "common.cuh"

namespace garlic {

// lod(): log10(P(g|autozygous)/P(g|non-autozygous)), exact operation order of
// garlic-roh.cpp:355-386.  Compiled with FMA contraction disabled (-fmad=false).
GHD double lod_eval(int g, double f, double e)
{
    if (f == 0 || f == 1 || g == 3) return 0.0;   // log10(1/1)
    double a, na;
    if (g == 0) {
        na = (1 - f) * (1 - f);
        a = (1 - e) * (1 - f) + e * na;
    } else if (g == 1) {
        na = 2 * (f) * (1 - f);
        a = e * na;
    } else {
        na = (f) * (f);
        a = (1 - e) * (f) + e * na;
    }
    return log10(a / na);
}

// Where a lane reads its per-SNP LOD from.  SRC 0: the per-SNP table (4 doubles per SNP: g=0,1,2,missing)
// seen through `tile`, which holds the entries of SNPs tile_lo, tile_lo+1, … — either the whole table
// in global memory (tile_lo = 0) or the item's slice staged into shared memory by TMA (kernels.cu).
// SRC 1: per-genotype LOD values (GL mode; lod() of each genotype's own error rate, evaluated at compaction).
template <int SRC>
struct LaneCtx {
    const uint64_t* row;    // word k of the row sits at row[k - row_base]
    int row_base;
    const char* tile;
    int tile_lo;
    const double* freq;
    const double* glrow;
    GHD double aval(int s, int g) const
    {
        if (SRC == 0) return *reinterpret_cast<const double*>(tile + ((uint32_t)(s - tile_lo) * 32u + (uint32_t)g * 8u));
        return glrow[(int64_t)s * kGlLanes];   // GL mode: per-genotype LOD, evaluated once by compact_gl_kernel
    }
};

struct LaneState {
    double win;
    int cov;
    int run_start;
    uint32_t fw;
    uint32_t hist;
    bool ambig;
};

GHD void emit_run(const WalkParams& P, const Item& it, int ind, bool active, int a, int b)
{
    const int ol = (a == it.own_lo) && (it.flags & 1);
    const int orr = (b == it.own_hi - 1) && (it.flags & 2);
    if (!active) return;
    if (!(ol | orr) && (b - a + 1 < P.thr)) return;   // garlic-roh.cpp:477 (min #SNPs)
#ifdef __CUDA_ARCH__
    unsigned p = atomicAdd(P.out_count, 1u);
#else
    unsigned p = P.out_count[0]++;
#endif
    if (p < P.out_cap) {
        RohRec r;
        r.ind = ind; r.a = a; r.b = b; r.tag = (it.seg << 2) | (orr << 1) | ol;
        P.out[p] = r;
#ifdef __CUDA_ARCH__
        if (P.hist) atomicAdd(P.hist + ind, 1u);
#endif
    }
}

template <bool DUMP>
GHD void dump_window(const WalkParams& P, const Item& it, int k, bool active, int t, double win)
{
    if (!DUMP) return;
    const int d = t - it.chr_start;
    // a window is dumped by the item that owns its first SNP (lead-in windows belong to the previous chunk)
    if (active && t >= it.own_lo && (d % P.dump_step) == 0)
        P.dump[(int64_t)k * P.dump_stride + it.thin_base + d / P.dump_step] = win;
}

GHD int popc32(uint32_t x)
{
#ifdef __CUDA_ARCH__
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// position of the n-th (1-based) set bit of x; the caller guarantees 1 <= n <= popc(x)
GHD int nth_set_bit(uint32_t x, int n)
{
    int pos = 0, c;
    c = popc32(x & 0xffffu); if (n > c) { n -= c; pos += 16; x >>= 16; }
    c = popc32(x & 0xffu);   if (n > c) { n -= c; pos += 8;  x >>= 8; }
    c = popc32(x & 0xfu);    if (n > c) { n -= c; pos += 4;  x >>= 4; }
    c = popc32(x & 0x3u);    if (n > c) { n -= c; pos += 2;  x >>= 2; }
    c = (int)(x & 1u);       if (n > c) { pos += 1; }
    return pos;
}

// byte offset (g*8) of genotype k's table entry, straight from the packed word: no multiply
GHD uint32_t lut_off(uint32_t w, int kk)
{
    return kk >= 2 ? ((w >> (2 * kk - 3)) & 24u) : ((w << (3 - 2 * kk)) & 24u);
}

// Phase 2 of a 32-window block: from the block's window-flag word fw (bit k = window tblk+k reached the cutoff)
// and ow (the flag stream delayed by W, only used when W > 32) to per-SNP coverage, covered bits and run records.
template <bool FULL>
GHD void cover_block(const WalkParams& P, const Item& it, LaneState& S, int ind, bool active, uint32_t fw, uint32_t ow,
                     int tblk)
{
    const int W = P.W;
    S.fw = fw;   // the block's window-flag word, stored to the history ring by the caller

    bool busy = (fw | (uint32_t)S.cov) != 0u;   // an open run implies cov >= thr >= 1
#ifdef __CUDA_ARCH__
    busy = __any_sync(0xffffffffu, busy);
#endif
    if (!busy) {
        if (W <= 32) S.hist = 0;   // = fw
        return;
    }
    // flags leaving the W-window during this block: the flag stream delayed by W steps
    uint32_t owv = ow;
    if (W <= 32) owv = (W == 32) ? S.hist : ((fw << W) | (S.hist >> (32 - W)));
    // cov(k) = cov + #d1 bits ≤ k − #d2 bits ≤ k  (sliding form of garlic-roh.cpp:446-454); covered = cov ≥ thr (:466)
    const uint32_t d1 = fw & ~owv, d2 = owv & ~fw;
    int cov = S.cov;
    uint32_t cw;
    bool mixed = (d1 != 0u) && (d2 != 0u);
#ifdef __CUDA_ARCH__
    mixed = __any_sync(0xffffffffu, mixed);
#endif
    if (mixed) {                 // a run starts and another ends within W steps of each other: per-step count
        cw = 0;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            cov += (int)((d1 >> k) & 1u) - (int)((d2 >> k) & 1u);
            cw |= (uint32_t)(cov >= P.thr) << k;
        }
    } else if (d1) {             // only increments: covered from the step of the (thr-cov)-th one on
        const int n = P.thr - cov, c = popc32(d1);
        cw = n <= 0 ? 0xffffffffu : (n > c ? 0u : (0xffffffffu << nth_set_bit(d1, n)));
        cov += c;
    } else if (d2) {             // only decrements: covered until the (cov-thr+1)-th one
        const int m = cov - P.thr, c = popc32(d2);
        cw = m < 0 ? 0u : (m >= c ? 0xffffffffu : ((1u << nth_set_bit(d2, m + 1)) - 1u));
        cov -= c;
    } else {
        cw = cov >= P.thr ? 0xffffffffu : 0u;
    }
    S.cov = cov;
    if (W <= 32) S.hist = fw;
    // run-length on the 32 covered bits (bit-parallel edge detection)
    uint32_t em = 0xffffffffu;
    if (!FULL) {
        const int lo = it.own_lo - tblk, hi = it.own_hi - tblk;          // owned steps are [lo, hi)
        const uint32_t mlo = lo <= 0 ? 0xffffffffu : (lo >= 32 ? 0u : ~((1u << lo) - 1u));
        const uint32_t mhi = hi >= 32 ? 0xffffffffu : (hi <= 0 ? 0u : ((1u << hi) - 1u));
        em = mlo & mhi;
    }
    const uint32_t x = cw & em;
    const uint32_t inr = S.run_start >= 0 ? 1u : 0u;
    uint32_t trans = x ^ ((x << 1) | inr);
    while (trans) {
#ifdef __CUDA_ARCH__
        const int k = __ffs((int)trans) - 1;
#else
        const int k = __builtin_ctz(trans);
#endif
        trans &= trans - 1;
        const int t = tblk + k;
        if ((x >> k) & 1u) S.run_start = t;
        else { emit_run(P, it, ind, active, S.run_start, t - 1); S.run_start = -1; }
    }
}

// One block of 32 slide steps, in two phases.
//   phase 1: the window chain win = (win - lod(out)) + lod(in) (garlic-roh.cpp:98-100) and the cutoff
//            test (:450) for all 32 steps → flag word(s).  With CHK the test is made against
//            cutoff±tol: where both agree they equal the test against the cutoff itself, where they
//            differ the (individual, segment) pair is marked for exact re-evaluation.
//   phase 2: coverage count (sliding form of :446-454) and run-length on the 32 flag bits — skipped by
//            the whole warp when no lane has a flag in this block or a flag still inside its last W
//            windows (the common case outside ROH).
// FULL: every step is a valid window and inside the owned range.
template <int SRC, bool ROH, bool DUMP, bool FULL, bool CHK>
GHD void walk_block(const WalkParams& P, const Item& it, const LaneCtx<SRC>& C, LaneState& S, int ind,
                    int k_slot, bool active, uint64_t gin, uint64_t gout, int tblk, uint32_t ow)
{
    const int W = P.W;
    const double cut_hi = CHK ? P.cutoff + P.tol : P.cutoff, cut_lo = P.cutoff - P.tol;
    const int s_in0 = tblk + W - 1, s_out0 = tblk - 1;
    uint32_t vm = 0xffffffffu;             // valid-window mask of the block
    if (!FULL) {
        const int n = it.we - tblk;
        vm = n >= 32 ? 0xffffffffu : (n <= 0 ? 0u : ((1u << n) - 1u));
    }
    uint32_t fhi = 0, flo = 0;
    double win = S.win;
    if (SRC == 0) {
        const uint32_t bi = (uint32_t)(s_in0 - C.tile_lo) * 32u, bo = (uint32_t)(s_out0 - C.tile_lo) * 32u;
        const uint32_t gi0 = (uint32_t)gin, gi1 = (uint32_t)(gin >> 32);
        const uint32_t go0 = (uint32_t)gout, go1 = (uint32_t)(gout >> 32);
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            const uint32_t oi = lut_off(k < 16 ? gi0 : gi1, k & 15), oo = lut_off(k < 16 ? go0 : go1, k & 15);
            const double a_in = *reinterpret_cast<const double*>(C.tile + ((bi | oi) + k * 32));
            const double a_out = *reinterpret_cast<const double*>(C.tile + ((bo | oo) + k * 32));
            // exact chains keep the reference's order (garlic-roh.cpp:98-100); the tolerance-checked
            // pass takes the difference off the dependent chain (same error bound, DESIGN.md §6)
            if (CHK) win = win + (a_in - a_out);
            else win = (win - a_out) + a_in;
            if (ROH) {
                if (win >= cut_hi) fhi |= 1u << k;                           // garlic-roh.cpp:450
                if (CHK) { if (win >= cut_lo) flo |= 1u << k; }
            }
            if (DUMP) { if ((vm >> k) & 1u) dump_window<DUMP>(P, it, k_slot, active, tblk + k, win); }
        }
    } else {
#pragma unroll 4
        for (int k = 0; k < 32; ++k) {
            const int go = (int)(gout >> (2 * k)) & 3, gi = (int)(gin >> (2 * k)) & 3;
            win = (win - C.aval(s_out0 + k, go)) + C.aval(s_in0 + k, gi);
            if (ROH) {
                if (win >= cut_hi) fhi |= 1u << k;
                if (CHK) { if (win >= cut_lo) flo |= 1u << k; }
            }
            if (DUMP) { if ((vm >> k) & 1u) dump_window<DUMP>(P, it, k_slot, active, tblk + k, win); }
        }
    }
    S.win = win;
    if (!ROH) return;
    fhi &= vm;
    if (CHK) { flo &= vm; S.ambig |= (fhi != flo); }
    cover_block<FULL>(P, it, S, ind, active, fhi, ow, tblk);
}

// Walk one item for one individual.  ring: this lane's flag-history ring (NW words, stride rstride).
// row: the words [row_base, …) of the individual's compacted row, if the caller holds them (else P.geno's row).
template <int SRC, bool ROH, bool DUMP>
GHD void walk_item(const WalkParams& P, const Item& it, int k_slot, bool active, uint32_t* ring, int rstride,
                   const char* tile, int tile_lo, int ind_in = -1, const uint64_t* row = nullptr, int row_base = 0)
{
    const int W = P.W;
    const int ind = ind_in >= 0 ? ind_in : (P.ind_list ? P.ind_list[k_slot] : k_slot);
    LaneCtx<SRC> C;
    C.row = row ? row : P.geno + (int64_t)ind * P.row_words;
    C.row_base = row ? row_base : 0;
    C.tile = tile;
    C.tile_lo = tile_lo;
    C.freq = P.freq;
    C.glrow = (SRC == 1) ? gl_lane(P, ind) : nullptr;
    const int NW = ((W + 31) >> 5) + 1;
    const bool chk = P.tol > 0;

    // fresh sum for window w0, ascending (garlic-roh.cpp:57-71)
    double win = 0.0;
    for (int i = 0; i < W; ++i) {
        const int s = it.w0 + i;
        const int g = (int)(C.row[(s >> 5) - C.row_base] >> (2 * (s & 31))) & 3;
        win += C.aval(s, g);
    }
    LaneState S;
    S.win = win; S.run_start = -1; S.fw = 0; S.ambig = false;
    const bool f0 = win >= (chk ? P.cutoff + P.tol : P.cutoff);
    if (chk) S.ambig = (f0 != (win >= P.cutoff - P.tol));
    dump_window<DUMP>(P, it, k_slot, active, it.w0, win);
    S.cov = (int)f0;
    S.hist = (uint32_t)f0 << 31;   // flag stream of the previous 32 steps: window w0 sits at position 31
    if (ROH && it.w0 >= it.own_lo && S.cov >= P.thr) S.run_start = it.w0;
    if (W > 32) {
        for (int w = 0; w < NW; ++w) ring[w * rstride] = 0;
        ring[0] = (uint32_t)f0 << 31;   // window w0 sits at bit-stream position 31
    }

    const int M = it.own_hi - 1 - it.w0;   // number of slide steps
    const int sa = 2 * ((it.w0 + W) & 31), sb = 2 * (it.w0 & 31);
    const uint64_t* pa = C.row + (((it.w0 + W) >> 5) - C.row_base);   // slide-in stream
    const uint64_t* pb = C.row + ((it.w0 >> 5) - C.row_base);         // slide-out stream
    uint64_t a_lo = pa[0], b_lo = pb[0];
    uint64_t a_hi = pa[1], b_hi = pb[1];
    pa += 2; pb += 2;
    const int r = (32 - (W & 31)) & 31;
    // ring of flag words (W > 32): block j writes slot (j+1) mod NW and reads the two slots after it,
    // which hold stream words j+1-nwords and j+2-nwords (NW = nwords+1); indices advance by compare-and-wrap
    int wr = 1 % NW;
    int tblk = it.w0 + 1;
    for (int m0 = 0; m0 < M; m0 += 32, tblk += 32) {
        // next block's words are requested before this block's arithmetic (rows are padded)
        const uint64_t a_nx = *pa++, b_nx = *pb++;
        const uint64_t gin = sa ? ((a_lo >> sa) | (a_hi << (64 - sa))) : a_lo;
        const uint64_t gout = sb ? ((b_lo >> sb) | (b_hi << (64 - sb))) : b_lo;
        a_lo = a_hi; b_lo = b_hi; a_hi = a_nx; b_hi = b_nx;
        uint32_t ow = 0;
        if (ROH && W > 32) {
            int r0 = wr + 1; if (r0 >= NW) r0 -= NW;
            int r1 = r0 + 1; if (r1 >= NW) r1 -= NW;
            const uint32_t w0_ = ring[r0 * rstride], w1_ = ring[r1 * rstride];
            ow = r ? ((w0_ >> r) | (w1_ << (32 - r))) : w0_;
        }
        const bool full = (tblk + 31 < it.we) && (tblk >= it.own_lo) && (tblk + 31 < it.own_hi);
        if (chk) {
            if (full) walk_block<SRC, ROH, DUMP, true, true>(P, it, C, S, ind, k_slot, active, gin, gout, tblk, ow);
            else walk_block<SRC, ROH, DUMP, false, true>(P, it, C, S, ind, k_slot, active, gin, gout, tblk, ow);
        } else {
            if (full) walk_block<SRC, ROH, DUMP, true, false>(P, it, C, S, ind, k_slot, active, gin, gout, tblk, ow);
            else walk_block<SRC, ROH, DUMP, false, false>(P, it, C, S, ind, k_slot, active, gin, gout, tblk, ow);
        }
        if (ROH && W > 32) {
            ring[wr * rstride] = S.fw;
            if (++wr >= NW) wr = 0;
        }
    }
    if (ROH && S.run_start >= 0) emit_run(P, it, ind, active, S.run_start, it.own_hi - 1);
    if (chk && S.ambig && active) {
#ifdef __CUDA_ARCH__
        unsigned p = atomicAdd(P.out_count + 1, 1u);
#else
        unsigned p = P.out_count[1]++;
#endif
        if (p < P.amb_cap) {
            RohRec rr;
            rr.ind = ind; rr.a = 0; rr.b = 0; rr.tag = it.seg;
            P.amb[p] = rr;
        }
    }
}

}  // namespace garlic
