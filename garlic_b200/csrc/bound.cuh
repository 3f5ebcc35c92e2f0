// bound.cuh — the pruning bound in front of the fused window → ROH walker (K5 pass 2, unweighted, table mode) and the
// bit-level column compaction (K3) it is fused with (squeeze.cu).  __host__ __device__ so that tests/host_emu.cpp runs
// the identical logic on the CPU.
//
// Most windows are nowhere near the cutoff: outside runs of homozygosity a window holds many heterozygous calls, each
// worth about log10(error) < 0.  This pass proves that cheaply for every individual and every 16-SNP block of window
// starts from bit operations on the packed genotypes alone — no per-genotype table lookup, no floating point:
//
//   lod(s,g) = base[s] + { 0            for the homozygote with the smaller table value,
//                          D[s] >= 0    for the other homozygote ("rare" below),
//                          lut[s][1] - base[s] <= chet   for a heterozygote,
//                          lut[s][3] - base[s] <= 0      for a missing call }
//   base[s] = min(lut[s][0], lut[s][2]),  D[s] = |lut[s][0] - lut[s][2]|   (the table is lod(), garlic-roh.cpp:355-386)
//
//   => every window starting in block k (t in [16k, 16k+16)) satisfies
//        win(t) <= Bmax[k] + sum_{q in core(k)} chet[q] * nhet(q) + sum_{q in span(k)} step[q] * nlev(q)
//      core(k) = half-words every such window contains  (k+1 .. k+c1,  c1 = (W-16)>>4)
//      span(k) = half-words any such window touches     (k   .. k+C2,  C2 = (W+14)>>4)
//      Bmax[k] = max_t sum_{s in [t,t+W)} base[s]
//      chet[q] = max_{s in q} (lut[s][1] - base[s])                      (one coefficient per half-word)
//      nlev(q) = sum over rare homozygotes of level(s), level(s) in {0,1,2,3} the smallest with level*step[q] >= D[s],
//                step[q] = max_{s in q} D[s] / 3: two bit-planes p0, p1 per half-word, nlev = popc(r&p0) + 2 popc(r&p1)
//
// evaluated in integers (fixed point 2^-8, every table entry rounded towards a larger bound).  Per individual and
// 256-SNP piece the kernel keeps the maximum over the piece's 16 blocks (and, separately, over its last C2 blocks: the
// only ones whose windows reach into the next piece); an (individual, item) pair none of whose blocks reaches
// cutoff - tol holds no flagged window (garlic-roh.cpp:450), hence no coverage and no ROH, and is never walked.
// The maxima do not depend on the cutoff, so the pass runs once per window size — fused with the compaction, while the
// compacted half-word is still in a register — before the cutoff is known (KDE, pass 1).
#pragma once
#include "common.cuh"
#include "walk.cuh"

namespace garlic {

constexpr int kBoundShift = 8;          // fixed-point scale of the bound: 1/256
constexpr int kBoundStoreShift = 2;     // the stored maxima are >> 2 (rounded up): int16 covers +-512 LOD
constexpr int kPiece = 256;             // SNPs per piece = 16 half-words = 8 packed words
constexpr int kBoundMinW = 16;          // below: the windows of a 16-start block share no SNP but one
constexpr int kBoundPartialW = 32;      // below: no whole half-word lies inside every window of a block — the core is the
                                        // block's last SNP plus the first W - 16 SNPs of the next half-word (bound_step<…, true>)
constexpr int kBoundMaxC2 = 13;         // ring of 16 prefix sums per lane: geometry of window sizes up to 209
constexpr int kBoundGeomMaxW = 209;     // larger windows: this geometry for their first 209 SNPs, the remaining W - 209 SNPs
                                        // enter Bmax with the larger homozygote's value (bound_block_max), whatever the genotype
constexpr int kPlanSegMax = 16;

GHD int bound_geom_w(int W) { return W > kBoundGeomMaxW ? kBoundGeomMaxW : W; }
GHD int bound_c2(int W) { return (bound_geom_w(W) + 14) >> 4; }
GHD int bound_c1(int W) { const int c = (bound_geom_w(W) - 16) >> 4; return c > 0 ? c : 0; }
GHD int bound_lag(int W) { return bound_c2(W) - bound_c1(W); }   // 1 or 2 for W >= kBoundMinW
GHD bool bound_partial(int W) { return W < kBoundPartialW; }
// even-bit mask of the SNPs of half-word k + c1 + 1 that every window of block k contains: its first (W - 16) & 15
GHD uint32_t bound_low_mask(int W) { const int r = (bound_geom_w(W) - 16) & 15; return r ? ((1u << (2 * r)) - 1u) & 0x55555555u : 0u; }

// Per half-word table entry, one 16-byte load per step:
//   x = orientation (even bits: bit 2i set <=> genotype 2 is the "rare" homozygote at SNP 16q+i) | plane p0 << 1 (odd bits)
//   y = plane p1 (even bits)
//   z = step (low 16 bits) | -chet (high 16 bits), fixed point, rounded towards a larger bound
//   w = filled in by the caller: Bmax of block q - C2 (what the step at half-word q evaluates)
GHD uint4 bound_hw_entry(const double* lut, long long q, long long L, int* invalid)
{
    const double scale = (double)(1 << kBoundShift);
    double D[16], dmax = 0.0, chet = -1e300;
    uint32_t mo = 0u;
    for (int i = 0; i < 16; ++i) {
        const long long s = q * 16 + i;
        const double* e = lut + s * 4;
        const double base = e[0] < e[2] ? e[0] : e[2];
        D[i] = fabs(e[0] - e[2]);
        if (!(D[i] >= 0.0) || D[i] > 1e6) { D[i] = 0.0; if (s < L) *invalid = 1; }      // NaN / inf tables: no bound
        if (e[2] > e[0]) mo |= 1u << (2 * i);
        if (D[i] > dmax) dmax = D[i];
        if (s < L) {
            const double dh = e[1] - base;
            if (dh > chet) chet = dh;
            if (e[3] - base > 0.0) *invalid = 1;      // a missing call worth more than a homozygote
            if (!(dh <= 0.0)) *invalid = 1;           // a heterozygote worth more than a homozygote (or NaN)
        }
    }
    uint32_t step = dmax > 0.0 ? (uint32_t)ceil(dmax / 3.0 * scale) + 1u : 0u;
    if (step > 0xffffu) { step = 0xffffu; *invalid = 1; }
    uint32_t p0 = 0u, p1 = 0u;
    for (int i = 0; i < 16; ++i) {
        int lev = 0;
        if (D[i] > 0.0) {
            lev = (int)ceil(D[i] * scale / (double)step);
            if (lev < 1) lev = 1;
            if (lev > 3) lev = 3;                     // 3*step >= dmax*scale by construction
        }
        if (lev & 1) p0 |= 1u << (2 * i);
        if (lev & 2) p1 |= 1u << (2 * i);
    }
    uint32_t ch = 0u;                                 // magnitude, rounded towards zero (a less negative coefficient)
    if (chet > -1e299 && chet < 0.0) { const double m = floor(-chet * scale); ch = m > 65535.0 ? 0xffffu : (uint32_t)m; }
    uint4 o;
    o.x = mo | (p0 << 1); o.y = p1; o.z = step | (ch << 16); o.w = 0u;
    return o;
}

// Bmax[k] in fixed point, rounded up (+2 of slack for the fp64 sums): the largest, over the 16 window starts t of
// block k, of  sum_{s in [t, t+Wg)} base[s]  +  sum_{s in [t+Wg, t+W)} top[s],  Wg = bound_geom_w(W) — the second sum
// (window sizes beyond the ring's geometry) takes every SNP at its best genotype, top[s] = max(lut[s][0], lut[s][2]).
GHD int bound_block_max(const double* lut, long long k, int W)
{
    const int Wg = bound_geom_w(W);
    const long long s0 = k * 16;
    double b = 0.0;
    for (int i = 0; i < Wg; ++i) { const double* e = lut + (s0 + i) * 4; b += e[0] < e[2] ? e[0] : e[2]; }
    for (int i = Wg; i < W; ++i) { const double* e = lut + (s0 + i) * 4; b += e[0] < e[2] ? e[2] : e[0]; }
    double bmax = b;
    for (int j = 1; j < 16; ++j) {
        const double* eo = lut + (s0 + j - 1) * 4;            // leaves the base part
        const double* ei = lut + (s0 + j - 1 + W) * 4;        // enters the last part
        b -= (eo[0] < eo[2] ? eo[0] : eo[2]);
        if (W > Wg) {
            const double* em = lut + (s0 + j - 1 + Wg) * 4;   // moves from the optimistic part to the base part
            b -= (em[0] < em[2] ? em[2] : em[0]);
            b += (em[0] < em[2] ? em[0] : em[2]);
            b += (ei[0] < ei[2] ? ei[2] : ei[0]);
        } else {
            b += (ei[0] < ei[2] ? ei[0] : ei[2]);
        }
        if (b > bmax) bmax = b;
    }
    const double v = ceil(bmax * (double)(1 << kBoundShift)) + 2.0;
    return v > 1.0e9 ? 1000000000 : (v < -1.0e9 ? -1000000000 : (int)v);
}

// Running state of one individual's scan: prefix sums of the het and rare terms, the last 16 of each in a ring
// (indices are compile-time after unrolling, so the ring lives in registers), the piece maxima.
struct BoundState {
    uint32_t PH[16], PR[16];   // modular arithmetic: only differences over at most 16 half-words are used
    uint32_t ph, pr;
    uint32_t top1, top2, low1; // PARTIAL: het term of the last SNP of the previous two half-words, low-mask term of the previous one
    int pm_all, pm_tail;
};

GHD void bound_reset(BoundState& S)
{
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int i = 0; i < 16; ++i) { S.PH[i] = 0u; S.PR[i] = 0u; }
    S.ph = 0u; S.pr = 0u;
    S.top1 = 0u; S.top2 = 0u; S.low1 = 0u;
    S.pm_all = -0x40000000; S.pm_tail = -0x40000000;
}

// One half-word h (16 genotypes) at ring position I = q & 15 (a constant after unrolling: the ring stays in registers);
// evaluates block k = q - C2, whose Bmax is t.w.  LAG = C2 - c1: 1 or 2.  PH accumulates the magnitude of the (negative)
// het term.
// PARTIAL = false (W >= 32): the het term counts the whole half-words k+1 … k+c1 every window of the block contains.
// PARTIAL = true (16 <= W < 32, where c1 = 0): it counts exactly the SNPs those windows share, [16k + 15, 16k + W) — the
// last SNP of half-word k and the first W - 16 of half-word k + 1 (low_mask).  The ring then holds the prefix up to
// SNP 14 of each half-word, the two scalars the last-SNP terms of the two half-words before this one.
template <int C2, int LAG, bool PARTIAL = false>
GHD void bound_step(BoundState& S, uint32_t h, const uint4& t, const int I, const uint32_t low_mask = 0u)
{
    const uint32_t M = 0x55555555u;
    const uint32_t s = h >> 1;
    const uint32_t het = h & ~s & M;                   // g == 1
    const uint32_t x = ~h & ~(s ^ t.x);                // even bits: homozygous with the "rare" orientation
    const int n0 = popc32(x & (t.x >> 1) & M), n1 = popc32(x & t.y), nh = popc32(het);
    S.pr += (uint32_t)(n0 + 2 * n1) * (t.z & 0xffffu);
    S.PR[I] = S.pr;
    int ub;
    if (!PARTIAL) {
        S.ph += (uint32_t)nh * (t.z >> 16);
        S.PH[I] = S.ph;
        ub = (int)t.w + (int)(S.pr - S.PR[(I - C2 - 1) & 15]) + (int)(S.PH[(I - C2) & 15] - S.PH[(I - LAG) & 15]);
    } else {
        const uint32_t ch = t.z >> 16;
        const uint32_t top = ((het >> 30) & 1u) * ch, low = (uint32_t)popc32(het & low_mask) * ch;
        S.PH[I] = S.ph + (uint32_t)nh * ch - top;      // prefix up to SNP 14 of this half-word
        S.ph += (uint32_t)nh * ch;
        // het magnitude over [16k + 15, end of half-word q - LAG] + the low part of half-word q - LAG + 1
        const uint32_t top_lag = LAG == 1 ? S.top1 : S.top2;
        const uint32_t low_next = LAG == 1 ? low : S.low1;
        const uint32_t core = (S.PH[(I - LAG) & 15] + top_lag) - S.PH[(I - C2) & 15] + low_next;
        ub = (int)t.w + (int)(S.pr - S.PR[(I - C2 - 1) & 15]) - (int)core;
        S.top2 = S.top1; S.top1 = top; S.low1 = low;
    }
    S.pm_all = ub > S.pm_all ? ub : S.pm_all;
    if (((I - C2) & 15) >= 16 - C2) S.pm_tail = ub > S.pm_tail ? ub : S.pm_tail;   // compile-time condition
}

// the two maxima as stored: int16 each (all | tail << 16), >> kBoundStoreShift rounded up, clamped
GHD uint32_t bound_pack(int pm_all, int pm_tail)
{
    int a = (pm_all + (1 << kBoundStoreShift) - 1) >> kBoundStoreShift, b = (pm_tail + (1 << kBoundStoreShift) - 1) >> kBoundStoreShift;
    a = a > 32767 ? 32767 : (a < -32768 ? -32768 : a);
    b = b > 32767 ? 32767 : (b < -32768 ? -32768 : b);
    return ((uint32_t)a & 0xffffu) | ((uint32_t)b << 16);
}

// cutoff - tol as compared against the stored maxima (rounded down, with slack); out of the int16 range: *ok = 0
GHD int bound_cut_store(double cutoff, double tol, int* ok)
{
    const double c = floor((cutoff - tol) * (double)(1 << kBoundShift)) - 2.0;
    *ok = (c > -8.0e6 && c < 8.0e6);
    if (!*ok) return 0;
    const int s = (int)c >> kBoundStoreShift;          // arithmetic shift: floor
    if (s > 32000 || s < -32000) *ok = 0;
    return s;
}

// Is (individual, item) a candidate?  Windows the item's walk evaluates start in [w0, own_hi): the pieces of own_lo …
// own_hi - 1 in full; of the lead-in (w0 < own_lo) the pieces before them in full too, except that the piece of w0 only
// contributes its last C2 blocks when the lead-in starts inside those (always, for window sizes up to 209).
GHD bool bound_item_candidate(const uint32_t* pmax, int64_t stride, int ind, const Item& it, int cut_store, int c2)
{
    const int p_own = it.own_lo >> 8, p_hi = (it.own_hi - 1) >> 8, p_w0 = it.w0 >> 8;
    bool c = false;
    for (int p = (p_w0 < p_own ? p_w0 + 1 : p_own); p <= p_hi; ++p) c |= (int)(int16_t)(pmax[(int64_t)p * stride + ind] & 0xffffu) >= cut_store;
    if (p_w0 < p_own) {
        const uint32_t v = pmax[(int64_t)p_w0 * stride + ind];
        const bool tail_covers = it.w0 >= 256 * (p_w0 + 1) - 16 * c2;
        c |= (int)(int16_t)(tail_covers ? (v >> 16) : (v & 0xffffu)) >= cut_store;
    }
    return c;
}

// ---------------------------------------------------------------------------------------------------------------
// K3 as a plan: how output half-word q (kept SNPs 16q .. 16q+15) is put together from input half-words.
//   x & 0x100: the 16 sources are consecutive but for d = (x >> 4) & 15 <= 3 dropped SNPs in between: take the window of
//              input half-words y, y+1, y+2 shifted right by (z & 255) bits and delete the fields at positions
//              (z >> 8) & 255, (z >> 16) & 255, z >> 24 (window coordinates after the earlier deletions, all < 16);
//   otherwise: x = number of segments (0..16), y = the last segment's input half-word (-1 if none), and
//              seg = {input half-word, right shift, mask, left shift} per run of kept SNPs inside one input half-word.
//   w = tail (bits of SNPs >= L read as missing); in the window form (always 16 SNPs) instead the mask of the fields
//       below the first deleted one (all ones without deletion): the kernel's branch-free path handles d <= 1 with it.
// ---------------------------------------------------------------------------------------------------------------
GHD void plan_half(const int* src, long long L, long long q, uint4* head, uint4* segs)
{
    const long long d0 = q * 16;
    int n = 0;
    if (d0 < L) { const long long r = L - d0; n = r < 16 ? (int)r : 16; }
    uint4 hd;
    hd.w = n < 16 ? (0xffffffffu << (2 * n)) : 0u;
    hd.z = 0u;
    if (n == 16) {
        const int d = src[d0 + 15] - src[d0] - 15;
        if (d >= 0 && d <= 3) {
            uint32_t z = (uint32_t)(2 * (src[d0] & 15));
            int k = 0;
            for (int i = 0; i < 15; ++i)
                for (int g = src[d0 + i + 1] - src[d0 + i] - 1; g > 0; --g) z |= (uint32_t)(i + 1) << (8 * ++k);
            hd.x = 0x100u | ((uint32_t)d << 4); hd.y = (uint32_t)(src[d0] >> 4); hd.z = z;
            hd.w = d ? ((1u << (2u * ((z >> 8) & 255u))) - 1u) : 0xffffffffu;
            *head = hd;
            return;
        }
    }
    int ns = 0, i = 0, last = -1;
    while (i < n) {
        const int s0 = src[d0 + i];
        int len = 1;
        while (i + len < n && src[d0 + i + len] == s0 + len && ((s0 + len) >> 4) == (s0 >> 4)) ++len;
        uint4 sg;
        sg.x = (uint32_t)(s0 >> 4); sg.y = (uint32_t)(2 * (s0 & 15));
        sg.z = len >= 16 ? 0xffffffffu : ((1u << (2 * len)) - 1u);
        sg.w = (uint32_t)(2 * i);
        segs[ns++] = sg;
        last = s0 >> 4;
        i += len;
    }
    hd.x = (uint32_t)ns; hd.y = (uint32_t)last;
    *head = hd;
}

// the window form: x0, x1, x2 = input half-words y, y+1, y+2 (x1 / x2 only read when plan_need1 / plan_need2)
// The kernel's branch-free path: the piece's input window sits in 20 registers (half-words a_base … a_base + 19,
// a_base even = the piece's first source half-word rounded down); output half-word I of the piece takes the 64-bit window at
// register I + k shifted right by sh bits, and the fields from p on move down by one (p = 16: no deletion).
// Two bytes per half-word: k | sh << 2, then 2 p.  0xffff: not expressible (several deletions, general form, a window
// further than two half-words ahead after many dropped SNPs) — the half-word takes the slow path.
GHD uint32_t plan_fast_code(const uint4& hd, int a_base, int I)
{
    if (!(hd.x & 0x100u) || ((hd.x >> 4) & 15u) > 1u) return 0xffffu;
    const int rel = 32 * ((int)hd.y - a_base - I) + (int)(hd.z & 255u);
    if (rel < 0 || rel >= 96) return 0xffffu;
    const uint32_t p = ((hd.x >> 4) & 15u) ? ((hd.z >> 8) & 255u) : 16u;
    return (uint32_t)(rel >> 5) | ((uint32_t)(rel & 31) << 2) | ((2u * p) << 8);
}
// r[0..4] = window registers I .. I + 4
GHD uint32_t plan_fast_apply(uint32_t code, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, uint32_t r4)
{
    const uint32_t k = code & 3u, sh = (code >> 2) & 31u, p2 = (code >> 8) & 255u;
    const uint32_t x0 = k == 0u ? r0 : (k == 1u ? r1 : r2), x1 = k == 0u ? r1 : (k == 1u ? r2 : r3), x2 = k == 0u ? r2 : (k == 1u ? r3 : r4);
    const uint32_t lo = sh ? ((x0 >> sh) | (x1 << (32u - sh))) : x0, hi = sh ? ((x1 >> sh) | (x2 << (32u - sh))) : x1;
    const uint32_t m = p2 >= 32u ? 0xffffffffu : ((1u << p2) - 1u);
    return (lo & m) | (((lo >> 2) | (hi << 30)) & ~m);
}
GHD bool plan_need1(const uint4& hd) { return ((hd.z & 255u) != 0u) || ((hd.x >> 4) & 15u); }
GHD bool plan_need2(const uint4& hd) { return ((hd.z & 255u) >> 1) + 15u + ((hd.x >> 4) & 15u) >= 32u; }
GHD uint32_t plan_window(const uint4& hd, uint32_t x0, uint32_t x1, uint32_t x2)
{
    const uint32_t sh = hd.z & 255u;
    uint32_t lo = sh ? ((x0 >> sh) | (x1 << (32u - sh))) : x0;
    uint32_t d = (hd.x >> 4) & 15u;
    if (d) {
        uint32_t hi = sh ? ((x1 >> sh) | (x2 << (32u - sh))) : x1;
        uint32_t z = hd.z >> 8;
        for (; d; --d, z >>= 8) {
            const uint32_t m = (1u << (2u * (z & 255u))) - 1u;     // fields below the deleted one stay
            const uint32_t slo = (lo >> 2) | (hi << 30);
            hi >>= 2;
            lo = (lo & m) | (slo & ~m);
        }
    }
    return lo;
}

// Output half-word q of one row, gathered from the row's uncompacted half-words hin by its plan head hd and segments sg
GHD uint32_t plan_gather(const uint4& hd, const uint4* sg, const uint32_t* hin)
{
    if (hd.x & 0x100u) return plan_window(hd, hin[hd.y], plan_need1(hd) ? hin[hd.y + 1] : 0u, plan_need2(hd) ? hin[hd.y + 2] : 0u);
    uint32_t h = hd.w;
    for (uint32_t k = 0; k < hd.x; ++k) { const uint4 g = sg[k]; h |= ((hin[g.x] >> g.y) & g.z) << g.w; }
    return h;
}

// Compacted words [wlo, wlo + n) of one row into out[0 .. n): what K3 writes there, built from the uncompacted row hin
// (32-bit view) by the plan (head / segs of every output half-word, bound.cuh:plan_half).  Half-words from SNP L on read
// as missing calls.  The plan is the same for every row: on the GPU a warp's lanes read it with uniform loads and
// only the row loads differ between lanes (the pruned walker, kernels.cu:walk_units_kernel).
GHD void plan_slice(const uint4* head, const uint4* segs, long long L, const uint32_t* hin, long long wlo, int n, uint64_t* out)
{
    for (int j = 0; j < n; ++j) {
        const long long q = 2 * (wlo + j);
        const uint32_t lo = 16 * q < L ? plan_gather(head[q], segs + q * kPlanSegMax, hin) : 0xffffffffu;
        const uint32_t hi = 16 * (q + 1) < L ? plan_gather(head[q + 1], segs + (q + 1) * kPlanSegMax, hin) : 0xffffffffu;
        out[j] = (uint64_t)hi << 32 | lo;
    }
}

}  // namespace garlic
