// segments.h — host-side segment table and run stitching (pure C++, shared by capi.cu and the CPU
// emulation test).  Closed form of the reference's window validity: a window is MISSING iff it
// contains an adjacent SNP pair with a gap > MAX_GAP or overlapping the centromere
// (src/garlic-roh.cpp:55-123, inGap :11-16; equivalence verified in SURVEY §3.4 and by
// tests/test_host_emu.py against the literal oracle).
#pragma once
#include <algorithm>
#include <cstdint>
#include <vector>
#include "common.cuh"

namespace garlic {

struct Segment { int chr, ws, we; };   // valid window starts [ws,we); SNP stretch [ws, we+W-1)

inline bool in_gap(int qs, int qe, int ts, int te)
{
    return (ts <= qs && te >= qs) || (ts <= qe && te >= qe) || (ts >= qs && te <= qe);
}

// Maximal stretches [a,b) of SNPs of one chromosome without a bad adjacent pair (independent of W).
struct Stretch { int chr, a, b; };

inline void build_stretches(const std::vector<int64_t>& chr_off, const std::vector<int32_t>& pos,
                            const std::vector<int32_t>& cen, int max_gap, std::vector<Stretch>& out)
{
    out.clear();
    const int n_chr = (int)chr_off.size() - 1;
    for (int c = 0; c < n_chr; ++c) {
        const int lo = (int)chr_off[c], hi = (int)chr_off[c + 1];
        const int cs = cen[2 * c], ce = cen[2 * c + 1];
        int a = lo;
        for (int i = lo + 1; i <= hi; ++i) {
            bool brk = (i == hi);
            if (!brk) {
                const int p0 = pos[i - 1], p1 = pos[i];
                brk = (p1 - p0 > max_gap) || in_gap(p0, p1, cs, ce);   // garlic-roh.cpp:60-61
            }
            if (brk) {
                if (i > a) out.push_back({c, a, i});
                a = i;
            }
        }
    }
}

inline void segments_from_stretches(const std::vector<Stretch>& st, int W, std::vector<Segment>& segs)
{
    segs.clear();
    for (const Stretch& s : st)
        if (s.b - s.a >= W) segs.push_back({s.chr, s.a, s.b - W + 1});
}

inline void build_segments(const std::vector<int64_t>& chr_off, const std::vector<int32_t>& pos,
                           const std::vector<int32_t>& cen, int max_gap, int W, std::vector<Segment>& segs)
{
    std::vector<Stretch> st;
    build_stretches(chr_off, pos, cen, max_gap, st);
    segments_from_stretches(st, W, segs);
}

// Chunk length (owned SNPs per item) of the chunked fast pass.  Preferred: the largest chunk whose
// table slice (owned SNPs + W-1 lead-in windows + W slide-in SNPs + block rounding) fits the shared-
// memory tile of tile_max SNPs; windows too large for that fall back to a chunk sized to fill the GPU.
inline int pick_chunk(int64_t L, int W, int n_lanes, int tile_max)
{
    const int c_tile = (tile_max - 2 * W - 32) / 32 * 32;
    if (c_tile >= 256) return c_tile;
    const int n_groups = (n_lanes + 31) / 32;
    const int64_t target_items = std::max<int64_t>(1, (148 * 16 * 4 + n_groups - 1) / n_groups);
    int64_t ch = L / target_items;
    const int64_t lo = std::max(256, 8 * W);
    ch = std::max<int64_t>(lo, std::min<int64_t>(ch, 8192));
    return (int)((ch + 31) / 32 * 32);
}

// SNPs an item's walk touches: [w0, w0 + 32*ceil((own_hi-1-w0)/32) + W)  (see walk_kernel)
inline int items_tile_snps(const std::vector<Item>& items, int W)
{
    int m = 0;
    for (const Item& it : items) m = std::max(m, 32 * ((it.own_hi - 1 - it.w0 + 31) >> 5) + W);
    return m;
}

// packed words of a row the walker reads for an item (walk.cuh:walk_item): from word w0 >> 5 through the slide-in
// stream's two-word lookahead behind its last block; the largest over the items
inline int items_slice_words(const std::vector<Item>& items, int W)
{
    int m = 0;
    for (const Item& it : items)
        m = std::max(m, ((it.w0 + W) >> 5) + ((it.own_hi - 1 - it.w0 + 31) >> 5) + 2 - (it.w0 >> 5));
    return m;
}

// chunk = 0: one item per segment (exact chains).  step > 0: thinning slots for window dumps.
inline void build_items(const std::vector<int64_t>& chr_off, int W, const std::vector<Segment>& segs, int chunk,
                        int step, std::vector<Item>& items)
{
    items.clear();
    const int n_chr = (int)chr_off.size() - 1;
    std::vector<int> thin_base(n_chr + 1, 0);
    for (int c = 0; c < n_chr; ++c) {
        const int Lc = (int)(chr_off[c + 1] - chr_off[c]);
        thin_base[c + 1] = thin_base[c] + (step > 0 ? (Lc + step - 1) / step : 0);
    }
    for (size_t si = 0; si < segs.size(); ++si) {
        const Segment& s = segs[si];
        const int a = s.ws, b = s.we + W - 1;
        int n = 1, size = b - a;
        if (chunk > 0 && b - a > chunk) {
            n = (b - a + chunk - 1) / chunk;
            size = std::min(chunk, ((b - a + n - 1) / n + 31) / 32 * 32);
            n = (b - a + size - 1) / size;
        }
        for (int i = 0; i < n; ++i) {
            Item it;
            it.own_lo = a + i * size;
            it.own_hi = std::min(b, it.own_lo + size);
            it.w0 = std::max(a, it.own_lo - W + 1);
            it.we = s.we;
            it.seg = (int)si;
            it.flags = (i > 0 ? 1 : 0) | (i + 1 < n ? 2 : 0);
            it.chr_start = (int)chr_off[s.chr];
            it.thin_base = thin_base[s.chr];
            items.push_back(it);
        }
    }
}

// Items aligned to the pruning pieces (bound.cuh): a segment's SNP stretch is cut at the multiples of `piece` that lie
// inside it, except those closer than piece/4 to either end (no sliver items).
inline void build_items_aligned(const std::vector<int64_t>& chr_off, int W, const std::vector<Segment>& segs, int piece,
                                std::vector<Item>& items)
{
    items.clear();
    std::vector<int> cuts;
    for (size_t si = 0; si < segs.size(); ++si) {
        const Segment& s = segs[si];
        const int a = s.ws, b = s.we + W - 1;
        cuts.clear();
        cuts.push_back(a);
        for (int c = (a / piece + 1) * piece; c < b; c += piece)
            if (c - a >= piece / 4 && b - c >= piece / 4) cuts.push_back(c);
        cuts.push_back(b);
        const int n = (int)cuts.size() - 1;
        for (int i = 0; i < n; ++i) {
            Item it;
            it.own_lo = cuts[i];
            it.own_hi = cuts[i + 1];
            it.w0 = std::max(a, it.own_lo - W + 1);
            it.we = s.we;
            it.seg = (int)si;
            it.flags = (i > 0 ? 1 : 0) | (i + 1 < n ? 2 : 0);
            it.chr_start = (int)chr_off[s.chr];
            it.thin_base = 0;
            items.push_back(it);
        }
    }
}

// buffers of stitch_runs kept between calls (a fresh 400 KB vector per call costs more than the sort)
struct StitchScratch {
    std::vector<uint32_t> first, cur;
    std::vector<std::pair<uint64_t, uint32_t>> key;
};

// Sort by (individual, start), merge runs cut at chunk boundaries, apply the minimum-length rule
// (garlic-roh.cpp:477).  Returns the merged runs; tag keeps seg<<2.

inline void stitch_runs(std::vector<RohRec>& recs, int thr, std::vector<RohRec>& out, StitchScratch* scratch = nullptr)
{
    StitchScratch local;
    StitchScratch& S = scratch ? *scratch : local;
    // sort by (individual, start): counting sort on the individual, then each individual's few runs by start
    int n_ind = 0;
    for (const RohRec& r : recs) n_ind = std::max(n_ind, r.ind + 1);
    std::vector<uint32_t>& first = S.first;
    first.assign(n_ind + 1, 0);
    for (const RohRec& r : recs) first[r.ind + 1]++;
    for (int i = 0; i < n_ind; ++i) first[i + 1] += first[i];
    std::vector<std::pair<uint64_t, uint32_t>>& key = S.key;
    key.resize(recs.size());
    {
        std::vector<uint32_t>& cur = S.cur;
        cur.assign(first.begin(), first.end() - 1);
        for (size_t i = 0; i < recs.size(); ++i)
            key[cur[recs[i].ind]++] = {((uint64_t)(uint32_t)recs[i].ind << 32) | (uint32_t)recs[i].a, (uint32_t)i};
    }
    for (int i = 0; i < n_ind; ++i) {
        const uint32_t lo = first[i], hi = first[i + 1];
        if (hi - lo > 24) std::sort(key.begin() + lo, key.begin() + hi);
        else
            for (uint32_t a = lo + 1; a < hi; ++a) {          // insertion sort: a handful of runs per individual
                const auto v = key[a];
                uint32_t b = a;
                while (b > lo && key[b - 1] > v) { key[b] = key[b - 1]; --b; }
                key[b] = v;
            }
    }
    out.clear();
    out.reserve(recs.size());
    size_t i = 0;
    while (i < key.size()) {
        RohRec cur = recs[key[i++].second];
        while ((cur.tag & 2) && i < key.size()) {
            const RohRec& nx = recs[key[i].second];
            if (!(nx.ind == cur.ind && (nx.tag & 1) && nx.a == cur.b + 1 && (nx.tag >> 2) == (cur.tag >> 2))) break;
            cur.b = nx.b;
            cur.tag = (cur.tag & ~2) | (nx.tag & 2);
            ++i;
        }
        if (cur.b - cur.a + 1 < thr) continue;
        out.push_back(cur);
    }
}

// Records stitched on the device (kernels.cu:bucket_stitch_kernel) arrive ordered by (individual, start) with the
// dropped slots marked ind = -1: keep the rest.
inline void take_stitched(const RohRec* recs, size_t n, std::vector<RohRec>& out)
{
    out.resize(n);
    RohRec* o = out.data();
    size_t m = 0;
    for (size_t i = 0; i < n; ++i) {
        o[m] = recs[i];
        m += recs[i].ind >= 0;
    }
    out.resize(m);
}

}  // namespace garlic
