"""Python mirror of the reference's hot-path call sequence (garlic-main.cpp:216-406) on top of the
C ABI — used by tests, bench.py and smoke().  The C++ command-line driver (garlic_b200/host/) follows
the same order.  Host-only steps here are the ones the reference also does once per run on scalars /
per-SNP vectors (map interpolation, density heuristics); everything per genotype runs on the GPU.
"""
from __future__ import annotations

import math

import numpy as np

from .api import GarlicGPU, overlap_threshold  # noqa: F401


def chr_label(name: str) -> str:
    """checkChrName, garlic-data.cpp:1886-1891."""
    return name if name[0] == "c" else "chr" + name


def interpolate_map(pos, spos, sgen):
    """interpolateGeneticmap / getMapInfo / interpolate (garlic-data.cpp:702-757): exact scaffold hits
    take the scaffold value (last duplicate wins, as the reference's std::map assignment does);
    other positions are interpolated with the reference's slope/intercept expression."""
    pos = np.asarray(pos, np.int64)
    spos = np.asarray(spos, np.int64)
    sgen = np.asarray(sgen, np.float64)
    if len(pos) and (pos.min() < spos[0] or pos.max() > spos[-1]):
        raise ValueError("Sites outside of map scaffold should have been filtered out")
    hi = np.searchsorted(spos, pos, side="right") - 1          # last index with spos <= pos
    exact = spos[hi] == pos
    lo = np.clip(hi, 0, len(spos) - 2)
    x0 = spos[lo].astype(np.float64)
    x1 = spos[lo + 1].astype(np.float64)
    y0, y1 = sgen[lo], sgen[lo + 1]
    q = pos.astype(np.float64)
    with np.errstate(all="ignore"):
        slope = (y1 - y0) / (x1 - x0)
        val = slope * q + (y0 - slope * x0)
    out = np.where(exact, sgen[hi], val)
    return out, int((~exact).sum())


def calc_density(n_loci, chr_pos, chr_cen):
    """calcDensity, garlic-data.cpp:318-328."""
    length = 0.0
    for p, c in zip(chr_pos, chr_cen):
        length += int(p[-1]) - int(p[0]) + 1 - (c[1] - c[0])
    return float(n_loci) / length


def select_overlap_frac(density, winsize):
    """selectOverlapFrac, garlic-data.cpp:3-8."""
    frac = (6.375 * math.log(density) + 63.888) / 100.0
    if frac > 1:
        frac = 1.0
    if frac <= 0:
        frac = 1.0 / float(winsize)
    return frac


def select_winsize_weighted(density):
    """selectWinsizeWeighted, garlic-roh.cpp:3-9."""
    size = int(8.3235 * math.log(density) + 138.0521 + 0.5)
    return size if size >= 10 else 10


class HotPath:
    """Runs load → count → filter → tables → [LD] → windows / ROH on one GPU for a synth.Dataset-like
    object (fields: chr_names, chr_offsets, pos, alleles | codes, centromeres, map_pos/map_cm, gl)."""

    def __init__(self, device=0):
        self.g = GarlicGPU(device)

    def close(self):
        self.g.close()

    def load(self, ds, weighted=False, cm=False, error=None, max_gap=200000, packed_rows=None,
             nalleles_corr=None, total_corr=None, mu=1e-9, M=7, bed=None, vcf=None, bcf=None, columns=None, n_input=None):
        """bed: uint8[L0, ceil(N/4)] SNP-major .bed rows (plink.Fileset.rows) in place of ds.alleles.
        vcf: (text, offsets) of the VCF sample columns (vcf.sample_text) in place of ds.alleles.
        bcf: (payload, offsets, descriptors) of the BCF GT vectors (bcf.gt_payload) in place of ds.alleles.
        columns: the individuals of a bed / vcf / bcf input of n_input individuals that form the analysed sample
        (ascending; GarlicGPU.select_columns); ds.gl, if any, holds the sample's individuals only."""
        g = self.g
        N = ds.n_ind if packed_rows is None else packed_rows.shape[0]
        if columns is not None:
            N = len(columns)
        g.set_shape(N, len(ds.pos), ds.chr_offsets, ds.pos)
        if columns is not None:
            g.select_columns(columns, n_input)
        n_samples = N if n_input is None else n_input
        if bed is not None:
            for s0 in range(0, len(ds.pos), 4096):
                g.put_bed(bed[s0:s0 + 4096], s0)
            g.code_alleles()
        elif vcf is not None:
            text, off = vcf
            for s0 in range(0, len(ds.pos), 4096):
                o = off[s0:s0 + 4097]
                nc, mx, bad = g.put_vcf_text(text, o, s0)
                if (nc != n_samples).any() or (bad >= 0).any():
                    raise ValueError("malformed VCF records in block %d" % s0)
            g.code_alleles()
        elif bcf is not None:
            gt, off, types = bcf
            for s0 in range(0, len(ds.pos), 4096):
                _, bad = g.put_bcf_gt(gt, off[s0:s0 + 4097], types[s0:s0 + 4096], n_samples, s0)
                if (bad >= 0).any():
                    raise ValueError("malformed BCF records in block %d" % s0)
            g.code_alleles()
        elif packed_rows is None:
            step = 1 << 16
            for s0 in range(0, len(ds.pos), step):
                g.put_alleles(ds.alleles[s0:s0 + step], s0, ds.tped_missing)
            g.code_alleles()
        else:
            g.put_packed(packed_rows)
            g.count_packed(nalleles_corr, total_corr)
        if getattr(ds, "gl", None) is not None:
            g.put_gl(np.ascontiguousarray(ds.gl.T), ds.gl_type)
        labels = [chr_label(n) for n in ds.chr_names]
        cens = [ds.centromeres.get(l, (0, 0)) for l in labels]
        oob = weighted or cm
        chr_param = None
        if oob:
            chr_param = np.array([[ds.map_pos[c][0], ds.map_pos[c][-1], cens[c][0], cens[c][1]]
                                  for c in range(len(labels))], np.int32)
        self.freq0, self.keep, self.L = g.filter(oob, chr_param)
        self.labels, self.cens = labels, cens
        kept = g.get_kept_index()
        self.pos = np.asarray(ds.pos)[kept]
        co0 = np.asarray(ds.chr_offsets)
        self.chr_off = np.searchsorted(kept, co0)          # kept offsets per chromosome
        self.gpos = None
        self.n_interp = 0
        if oob:
            gp = np.empty(self.L)
            for c in range(len(labels)):
                lo, hi = self.chr_off[c], self.chr_off[c + 1]
                gp[lo:hi], k = interpolate_map(self.pos[lo:hi], ds.map_pos[c], ds.map_cm[c])
                self.n_interp += k
            self.gpos = gp
        g.set_tables(error, max_gap, np.array(cens, np.int32), self.gpos)
        if weighted:
            g.set_wlod(mu, M)
        return self

    def density(self):
        return calc_density(self.L, [self.pos[self.chr_off[c]:self.chr_off[c + 1]] for c in range(len(self.labels))],
                            self.cens)

    def roh(self, W, cutoff, overlap_frac, weighted=False, exact=False, cm=False):
        """→ list of (ind, chr_index, start_bp, stop_bp, length, start_idx, stop_idx) in reference order."""
        arr = self.g.call_roh(W, cutoff, overlap_frac, weighted, exact)
        out = []
        for ind, c, a, b in arr:
            if cm:
                ln = float(self.gpos[b] - self.gpos[a])          # garlic-roh.cpp:478
            else:
                ln = float(int(self.pos[b]) - int(self.pos[a]) + 1)
            out.append((int(ind), int(c), int(self.pos[a]), int(self.pos[b]), ln, int(a), int(b)))
        return out

    def thinned(self, W, step, individuals=None, weighted=False, exact=True):
        """KDE input: windows at locus 0,step,… per chromosome, MISSING/NaN dropped, in the reference's
        chr → individual → locus order (garlic-data.cpp:2026-2069)."""
        m = self.g.windows(W, step, weighted, individuals, exact)
        vals = []
        base = 0
        for c in range(len(self.labels)):
            n = (int(self.chr_off[c + 1] - self.chr_off[c]) + step - 1) // step
            blk = m[:, base:base + n].reshape(-1)
            vals.append(blk[(blk != -9999.0) & ~np.isnan(blk)])
            base += n
        return np.concatenate(vals) if vals else np.empty(0)


def bad_pair_bits(pos, chr_off, cens, max_gap):
    """bool[L]: bit i set <=> no window may hold both SNP i-1 and SNP i — a gap / centromere pair (inGap, garlic-roh.cpp:11-16)
    or a chromosome start.  What csrc/kernels.cu:bad_pairs_kernel leaves on the device for the thinned pass 1."""
    pos = np.asarray(pos, np.int64)
    bad = np.zeros(len(pos), bool)
    for c in range(len(chr_off) - 1):
        lo, hi = int(chr_off[c]), int(chr_off[c + 1])
        if hi <= lo:
            continue
        if lo > 0:
            bad[lo] = True
        qs, qe = pos[lo:hi - 1], pos[lo + 1:hi]
        ts, te = cens[c]
        gap = ((ts <= qs) & (te >= qs)) | ((ts <= qe) & (te >= qe)) | ((ts >= qs) & (te <= qe))
        bad[lo + 1:hi] = (qe - qs > max_gap) | gap
    return bad


def window_valid(bad, W):
    """bool[L]: window starting at t is not MISSING <=> t + W <= L and no bad pair among SNPs t+1 … t+W-1
    (thin_windows_kernel's test on the bit map; DESIGN.md §4)."""
    L = len(bad)
    cs = np.concatenate([[0], np.cumsum(bad.astype(np.int64))])
    ok = np.zeros(L, bool)
    t = np.arange(0, max(0, L - W + 1))
    ok[:len(t)] = (cs[t + W] - cs[t + 1]) == 0
    return ok


_POW10 = [10.0 ** k for k in range(23)]


def parse_decimal_fast(tok):
    """The decimal -> fp64 conversion of csrc/ingest.cu:parse_decimal, statement for statement: (value, hard).  hard = the
    device leaves the token to the host's strtod (more than 15 significant digits, a power of ten beyond 10^22, inf / nan /
    hex, malformed); otherwise value is exact — one correctly rounded IEEE operation on exact operands."""
    n, i = len(tok), 0
    neg = False
    if i < n and tok[i] in "+-":
        neg = tok[i] == "-"
        i += 1
    m, nd, e10 = 0, 0, 0
    any_digit = dot = bad = False
    while i < n:
        c = tok[i]
        if "0" <= c <= "9":
            any_digit = True
            if m == 0 and c == "0":
                if dot:
                    e10 -= 1
            elif nd < 19:
                m = m * 10 + (ord(c) - 48)
                nd += 1
                if dot:
                    e10 -= 1
            else:
                bad = True
                if not dot:
                    e10 += 1
        elif c == "." and not dot:
            dot = True
        else:
            break
        i += 1
    if i < n and tok[i] in "eE":
        i += 1
        eneg = False
        if i < n and tok[i] in "+-":
            eneg = tok[i] == "-"
            i += 1
        ex = nex = 0
        while i < n and "0" <= tok[i] <= "9":
            ex = ex * 10 + (ord(tok[i]) - 48) if ex < 100000 else ex
            nex += 1
            i += 1
        if not nex:
            bad = True
        e10 += -ex if eneg else ex
    if i < n:
        bad = True
    if not any_digit:
        bad = True
    v = 0.0
    if not bad and m != 0:
        if nd <= 15 and -22 <= e10 <= 22:
            v = float(m)
            v = v / _POW10[-e10] if e10 < 0 else v * _POW10[e10]
        else:
            bad = True
    return (-v if neg else v), bad
