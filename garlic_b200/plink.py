"""PLINK 1 binary filesets (.bed / .bim / .fam) in numpy: reader, writer, and the convention that makes a fileset the
same input as a tped.

A .bed is SNP-major: after the magic bytes 6c 1b 01, one row of ceil(N/4) bytes per SNP, individual i at bits 2(i%4) of
byte i/4, with PLINK's values 0 = hom A1, 1 = missing, 2 = het, 3 = hom A2.  The fileset means exactly the tped that
writes hom A1 as "A1 A1", het as "A1 A2", hom A2 as "A2 A2" and missing as "0 0" with the .bim's allele names, the .fam
in the role of the .tfam and the .bim's chr / id / cM / bp as the tped's first four columns.  So the "1" allele
(the first non-missing character, reference loadTPEDData) is A2 iff the first present call is hom A2, A1 if it is
hom A1 or het, and there is none if no call is present (csrc/bed.cu computes the same on the GPU).
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np

MAGIC = bytes([0x6C, 0x1B])
HOM_A1, MISSING, HET, HOM_A2 = 0, 1, 2, 3


class PlinkError(ValueError):
    pass


@dataclass
class Bim:
    chr: list        # chromosome names as written
    ids: list        # SNP ids
    cm: list         # genetic positions as written (strings)
    bp: np.ndarray   # int32 physical positions
    a1: list         # allele names (strings, '0' = unknown)
    a2: list


@dataclass
class Fileset:
    rows: np.ndarray   # uint8[L0, ceil(N/4)] .bed rows without the magic bytes
    bim: Bim
    fam: list          # [(family / population, individual id)] per individual

    @property
    def n_ind(self):
        return len(self.fam)

    @property
    def n_loci(self):
        return self.rows.shape[0]

    def codes(self):
        """uint8[L0, N] PLINK values (padding bits of the last byte dropped)."""
        return codes_from_rows(self.rows, self.n_ind)


def codes_from_rows(rows, n_ind):
    rows = np.asarray(rows, np.uint8)
    out = np.empty((rows.shape[0], rows.shape[1], 4), np.uint8)
    for k in range(4):
        out[:, :, k] = (rows >> (2 * k)) & 3
    return out.reshape(rows.shape[0], -1)[:, :n_ind]


def rows_from_codes(codes, pad=0):
    """uint8[L0, N] PLINK values → .bed rows; the padding fields of the last byte get the value `pad`."""
    codes = np.asarray(codes, np.uint8)
    L0, N = codes.shape
    nb = (N + 3) // 4
    q = np.full((L0, nb * 4), pad & 3, np.uint8)
    q[:, :N] = codes
    q = q.reshape(L0, nb, 4)
    return (q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)).astype(np.uint8)


def _table(path, ncol):
    with open(path) as f:
        rows = [l.split() for l in f if l.strip()]
    for k, r in enumerate(rows):
        if len(r) < ncol:
            raise PlinkError("%s line %d: expected %d columns, found %d" % (path, k + 1, ncol, len(r)))
    return rows


def read_bim(path):
    t = _table(path, 6)
    return Bim(chr=[r[0] for r in t], ids=[r[1] for r in t], cm=[r[2] for r in t],
               bp=np.array([int(r[3]) for r in t], np.int32), a1=[r[4] for r in t], a2=[r[5] for r in t])


def read_fam(path):
    return [(r[0], r[1]) for r in _table(path, 6)]


def check_header(head, size, n_ind, n_snp):
    """The checks every reader of a .bed makes: magic bytes, SNP-major mode, size 3 + L0·ceil(N/4)."""
    if len(head) < 3 or bytes(head[:2]) != MAGIC:
        raise PlinkError("not a PLINK .bed file (the first bytes are not 6c 1b)")
    if head[2] == 0:
        raise PlinkError("individual-major .bed (mode byte 00) is not supported; rewrite it SNP-major with plink --make-bed")
    if head[2] != 1:
        raise PlinkError("unknown .bed mode byte %02x" % head[2])
    want = 3 + n_snp * ((n_ind + 3) // 4)
    if size != want:
        raise PlinkError(".bed has %d bytes, but %d SNPs (.bim) x %d individuals (.fam) need %d" % (size, n_snp, n_ind, want))


def read_fileset(prefix):
    bim, fam = read_bim(prefix + ".bim"), read_fam(prefix + ".fam")
    data = np.fromfile(prefix + ".bed", np.uint8)
    check_header(data[:3].tobytes(), len(data), len(fam), len(bim.bp))
    return Fileset(rows=data[3:].reshape(len(bim.bp), (len(fam) + 3) // 4), bim=bim, fam=fam)


def write_fileset(prefix, codes, bim, fam, pad=0):
    """codes uint8[L0, N] PLINK values; fam [(population, id)]; pad = value of the padding fields."""
    d = os.path.dirname(prefix)
    if d:
        os.makedirs(d, exist_ok=True)
    with open(prefix + ".bed", "wb") as f:
        f.write(MAGIC + b"\x01")
        f.write(rows_from_codes(codes, pad).tobytes())
    with open(prefix + ".bim", "w") as f:
        for c, i, g, p, a, b in zip(bim.chr, bim.ids, bim.cm, bim.bp, bim.a1, bim.a2):
            f.write("%s\t%s\t%s\t%d\t%s\t%s\n" % (c, i, g, int(p), a, b))
    with open(prefix + ".fam", "w") as f:
        for pop, i in fam:
            f.write("%s %s 0 0 0 -9\n" % (pop, i))
    return prefix


def one_allele(codes):
    """int8[L0]: 1 if the "1" allele is A1, 2 if A2, 0 if no call is present (the first present call decides)."""
    codes = np.asarray(codes, np.uint8)
    present = codes != MISSING
    first = np.argmax(present, axis=1)
    fc = codes[np.arange(len(codes)), first]
    return np.where(~present.any(1), 0, np.where(fc == HOM_A2, 2, 1)).astype(np.int8)


def tped_tokens(codes, a1, a2):
    """The equivalent tped's genotype columns: list per SNP of 2N allele names."""
    codes = np.asarray(codes, np.uint8)
    out = []
    for s in range(codes.shape[0]):
        pick = {HOM_A1: (a1[s], a1[s]), HET: (a1[s], a2[s]), HOM_A2: (a2[s], a2[s]), MISSING: ("0", "0")}
        out.append([t for c in codes[s] for t in pick[int(c)]])
    return out


def tped_alleles(codes, a1, a2):
    """uint8[L0, N, 2] allele characters of the equivalent tped (allele names of one character)."""
    codes = np.asarray(codes, np.uint8)
    c1 = np.frombuffer("".join(a1).encode(), np.uint8)[:, None]
    c2 = np.frombuffer("".join(a2).encode(), np.uint8)[:, None]
    if len(c1) != codes.shape[0] or len(c2) != codes.shape[0]:
        raise ValueError("tped_alleles needs allele names of one character")
    zero = np.uint8(ord("0"))
    first = np.where(codes == HOM_A2, c2, np.where(codes == MISSING, zero, c1))
    second = np.where(codes == HOM_A1, c1, np.where(codes == MISSING, zero, c2))
    return np.stack([first, second], axis=2).astype(np.uint8)


def write_tped(prefix, fs: Fileset):
    """The equivalent tped / tfam of a fileset."""
    toks = tped_tokens(fs.codes(), fs.bim.a1, fs.bim.a2)
    b = fs.bim
    with open(prefix + ".tped", "w") as f:
        for s in range(fs.n_loci):
            f.write("%s %s %s %d %s\n" % (b.chr[s], b.ids[s], b.cm[s], int(b.bp[s]), " ".join(toks[s])))
    with open(prefix + ".tfam", "w") as f:
        for pop, i in fs.fam:
            f.write("%s %s 0 0 0 0\n" % (pop, i))
    return prefix + ".tped", prefix + ".tfam"


def from_alleles(alleles, seed=0, missing=ord("0")):
    """A tped allele matrix uint8[L0, N, 2] → (codes uint8[L0, N], a1, a2): half-missing calls become missing, and each
    SNP's two letters are named A1 / A2 in a seeded random order, so that heterozygotes are written A1 first and some
    SNPs' "1" allele is A2.  A SNP with fewer than two letters gets a stand-in letter for the absent one."""
    alleles = np.asarray(alleles, np.uint8)
    L0 = alleles.shape[0]
    rng = np.random.default_rng(seed)
    swap = rng.random(L0) < 0.5
    codes = np.full(alleles.shape[:2], MISSING, np.uint8)
    a1, a2 = [], []
    for s in range(L0):
        x = alleles[s]
        ok = (x[:, 0] != missing) & (x[:, 1] != missing)
        letters = list(dict.fromkeys(x[ok].reshape(-1).tolist()))
        if len(letters) > 2:
            raise ValueError("SNP %d has more than two alleles" % s)
        for c in b"ACGT":
            if len(letters) >= 2:
                break
            if c not in letters:
                letters.append(c)
        p, q = (letters[1], letters[0]) if swap[s] else (letters[0], letters[1])
        n2 = (x[:, 0] == q).astype(np.int32) + (x[:, 1] == q)
        codes[s] = np.where(~ok, MISSING, np.where(n2 == 0, HOM_A1, np.where(n2 == 1, HET, HOM_A2)))
        a1.append(chr(p))
        a2.append(chr(q))
    return codes, a1, a2


def bed_dataset(ds, seed=0):
    """A bed-representable copy of a synth.Dataset → (dataset, codes, a1, a2): its alleles are those of the equivalent
    tped of from_alleles' fileset."""
    import copy
    codes, a1, a2 = from_alleles(ds.alleles, seed, ord(ds.tped_missing))
    out = copy.copy(ds)
    out.alleles = tped_alleles(codes, a1, a2)
    return out, codes, a1, a2


def bim_of(ds, a1, a2):
    """The .bim of a synth.Dataset (cM 0, as its tped writer writes)."""
    chrs = []
    for c in range(len(ds.chr_names)):
        chrs += [ds.chr_names[c]] * int(ds.chr_offsets[c + 1] - ds.chr_offsets[c])
    return Bim(chr=chrs, ids=list(ds.snp_ids), cm=["0"] * len(ds.pos), bp=np.asarray(ds.pos, np.int32), a1=list(a1),
               a2=list(a2))
