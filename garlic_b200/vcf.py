"""VCF genotypes in numpy: the CPU reference of the VCF input path, and a writer for test data (plain, gzip or BGZF).

A VCF means exactly the tped that writes each sample's two GT alleles in GT order by name — REF for index 0, the k-th
ALT for index k, the missing code for '.' (a lone '.' GT is two missing alleles) — with CHROM / ID / POS as the tped's
columns 1 / 2 / 4 and the #CHROM line's samples in place of the tfam's individuals.  So the "1" allele is the first
present allele in file order, half-missing calls count their present allele, and a multi-allelic record is coded "1"
allele against the rest.  csrc/vcf.cu parses the same GT grammar on the GPU (csrc/vcf_gt.cuh:parse_gt).

Alleles are held as index bytes, 255 = missing.
"""
from __future__ import annotations

import gzip
import struct
import zlib
from dataclasses import dataclass

import numpy as np

MISSING = 255
MAX_ALLELE = 254
FORMATS = ("GT", "GT:AD:DP:GQ:PL")


class VcfError(ValueError):
    pass


@dataclass
class Vcf:
    samples: list
    chrom: list        # per record
    pos: np.ndarray    # int64 per record
    ids: list
    ref: list
    alts: list         # per record: list of ALT names ([] for '.')
    idx: np.ndarray    # uint8[L0, N, 2] allele indices, 255 = missing


def parse_gt(col):
    """The GT of one sample column (text up to ':' / end) → (a, b) allele index bytes, or None if malformed."""
    gt = col.split(":", 1)[0]
    if gt == ".":
        return MISSING, MISSING
    parts = gt.replace("|", "/").split("/")
    if len(parts) != 2:
        return None
    out = []
    for p in parts:
        if p == ".":
            out.append(MISSING)
        elif p and all("0" <= c <= "9" for c in p) and int(p) <= MAX_ALLELE:
            out.append(int(p))
        else:
            return None
    return tuple(out)


# ------------------------------------------------------------------------------------------------ BGZF
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_block(data: bytes, level=6) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    cdata = c.compress(data) + c.flush()
    bsize = 12 + 6 + len(cdata) + 8
    if bsize > 65536:
        raise ValueError("BGZF block larger than 64 KiB")
    head = bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1)
    return head + cdata + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data))


def bgzf_compress(data: bytes, block_size=65280) -> bytes:
    """BGZF of data: blocks of block_size input bytes (at most 65,280, as htslib writes) and the empty EOF block."""
    out = [bgzf_block(data[i:i + block_size]) for i in range(0, len(data), block_size)]
    return b"".join(out) + BGZF_EOF


def _open_text(path):
    with open(path, "rb") as f:
        magic = f.read(2)
    return gzip.open(path, "rt") if magic == b"\x1f\x8b" else open(path)


# ------------------------------------------------------------------------------------------------ reader
def read_vcf(path) -> Vcf:
    """Pure-Python reader (plain, gzip or BGZF) with the checks of the driver's loader and of the GPU tokeniser."""
    samples, chrom, pos, ids, ref, alts, idx = None, [], [], [], [], [], []
    with _open_text(path) as f:
        for no, line in enumerate(f, 1):
            line = line.rstrip("\r\n")
            if samples is None:
                if line.startswith("##"):
                    continue
                if not line.startswith("#CHROM"):
                    raise VcfError("line %d: no #CHROM header line before the first record" % no)
                cols = line.split("\t")
                if len(cols) < 9 or cols[8] != "FORMAT":
                    raise VcfError("the #CHROM header has no FORMAT column")
                if len(cols) == 9:
                    raise VcfError("the #CHROM header names no samples")
                samples = cols[9:]
                if len(set(samples)) != len(samples):
                    raise VcfError("duplicate sample ID")
                continue
            if not line:
                continue
            cols = line.split("\t")
            where = "line %d (%s:%s)" % (no, cols[0], cols[1] if len(cols) > 1 else "")
            if len(cols) < 9:
                raise VcfError(where + ": fewer than 9 fixed columns")
            if not cols[1].isdigit():
                raise VcfError(where + ": POS is not an integer")
            if cols[8] != "GT" and not cols[8].startswith("GT:"):
                raise VcfError(where + ": FORMAT does not start with GT")
            if len(cols) - 9 != len(samples):
                raise VcfError(where + ": %d sample columns, the header names %d" % (len(cols) - 9, len(samples)))
            a = cols[4].split(",") if cols[4] != "." else []
            row = []
            for c in cols[9:]:
                g = parse_gt(c)
                if g is None:
                    raise VcfError(where + ": malformed GT %r" % c)
                if max((x for x in g if x != MISSING), default=-1) > len(a):
                    raise VcfError(where + ": allele index above the ALT count")
                row.append(g)
            chrom.append(cols[0])
            pos.append(int(cols[1]))
            ids.append(cols[2])
            ref.append(cols[3])
            alts.append(a)
            idx.append(row)
    if samples is None:
        raise VcfError("no #CHROM header line")
    arr = np.array(idx, np.uint8).reshape(len(idx), len(samples), 2)
    return Vcf(samples=samples, chrom=chrom, pos=np.array(pos, np.int64), ids=ids, ref=ref, alts=alts, idx=arr)


def sample_text(path):
    """(bytes, int64 offsets[L0+1]): per record the text after the FORMAT column's tab, as the driver uploads it."""
    parts, off = [], [0]
    with _open_text(path) as f:
        for line in f:
            line = line.rstrip("\r\n")
            if not line or line.startswith("#"):
                continue
            cols = line.split("\t", 9)
            t = cols[9].encode() if len(cols) > 9 else b""
            parts.append(t)
            off.append(off[-1] + len(t))
    return b"".join(parts), np.array(off, np.int64)


# ------------------------------------------------------------------------------------------------ writer
def _gt_table(max_idx, sep, lone_missing):
    """table[a, b] → GT text for allele index bytes a, b (255 = '.')."""
    names = [str(i) for i in range(max_idx + 1)]
    tab = {}
    for a in list(range(max_idx + 1)) + [MISSING]:
        for b in list(range(max_idx + 1)) + [MISSING]:
            na = "." if a == MISSING else names[a]
            nb = "." if b == MISSING else names[b]
            tab[(a, b)] = "." if (lone_missing and a == MISSING and b == MISSING) else na + sep + nb
    return tab


def vcf_text(v: Vcf, fmt="GT", sep="/", lone_missing=False) -> bytes:
    """The VCF file's text.  fmt "GT:AD:DP:GQ:PL" adds filler values after each GT; sep "/" or "|"; lone_missing
    writes a call with both alleles missing as a lone '.'."""
    if fmt not in FORMATS or sep not in "/|":
        raise ValueError("fmt must be one of %s and sep '/' or '|'" % (FORMATS,))
    idx = np.asarray(v.idx, np.uint8)
    present = idx[idx != MISSING]
    top = int(present.max()) if present.size else 0
    tab = _gt_table(top, sep, lone_missing)
    codes = idx[:, :, 0].astype(np.int64) * 256 + idx[:, :, 1]
    keys = sorted(tab)
    lut = np.empty(256 * 256, object)
    for a, b in keys:
        lut[a * 256 + b] = tab[(a, b)]
    out = ["##fileformat=VCFv4.2\n", '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n',
           "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(v.samples) + "\n"]
    for s in range(len(v.chrom)):
        gts = lut[codes[s]]
        if fmt != "GT":
            n = 1 + len(v.alts[s])
            extra = ":" + ",".join(["3"] * n) + ":%d:30:" % (3 * n) + ",".join(["0"] + ["20"] * (n * (n + 1) // 2 - 1))
            gts = [g + extra for g in gts]
        alt = ",".join(v.alts[s]) if v.alts[s] else "."
        out.append("%s\t%d\t%s\t%s\t%s\t.\tPASS\t.\t%s\t%s\n" % (v.chrom[s], int(v.pos[s]), v.ids[s], v.ref[s], alt, fmt,
                                                                "\t".join(gts)))
    return "".join(out).encode()


def write_vcf(path, v: Vcf, fmt="GT", sep="/", lone_missing=False, compress=None, block_size=65280):
    """compress: None (plain), "gz" (one gzip member) or "bgzf" (blocks of block_size input bytes)."""
    data = vcf_text(v, fmt, sep, lone_missing)
    if compress == "gz":
        data = gzip.compress(data, compresslevel=1)
    elif compress == "bgzf":
        data = bgzf_compress(data, block_size)
    elif compress is not None:
        raise ValueError("compress must be None, 'gz' or 'bgzf'")
    with open(path, "wb") as f:
        f.write(data)
    return path


# ------------------------------------------------------------------------------------------------ convention
def from_dataset(ds, seed=0) -> Vcf:
    """The VCF of a synth.Dataset whose tped alleles are exactly ds.alleles: per SNP the letters present, in a seeded
    random order, become REF and the ALTs (so the "1" allele is sometimes REF, sometimes an ALT); a SNP with no
    letter gets REF "A" and no ALT."""
    alleles = np.asarray(ds.alleles, np.uint8)
    miss = ord(ds.tped_missing)
    rng = np.random.default_rng(seed)
    L0, N, _ = alleles.shape
    idx = np.full((L0, N, 2), MISSING, np.uint8)
    ref, alts, chrom = [], [], []
    for c in range(len(ds.chr_names)):
        chrom += [ds.chr_names[c]] * int(ds.chr_offsets[c + 1] - ds.chr_offsets[c])
    for s in range(L0):
        x = alleles[s]
        letters = [l for l in dict.fromkeys(x.reshape(-1).tolist()) if l != miss]
        letters = [letters[i] for i in rng.permutation(len(letters))] or [ord("A")]
        for k, l in enumerate(letters):
            idx[s][x == l] = k
        ref.append(chr(letters[0]))
        alts.append([chr(l) for l in letters[1:]])
    return Vcf(samples=list(ds.ind_ids), chrom=chrom, pos=np.asarray(ds.pos, np.int64), ids=list(ds.snp_ids), ref=ref,
               alts=alts, idx=idx)


def tped_alleles(idx, ref, alts, missing="0"):
    """uint8[L0, N, 2] allele characters of the equivalent tped (allele names of one character)."""
    idx = np.asarray(idx, np.uint8)
    out = np.full(idx.shape, ord(missing), np.uint8)
    for s in range(idx.shape[0]):
        names = [ref[s]] + list(alts[s])
        if any(len(n) != 1 for n in names):
            raise ValueError("tped_alleles needs allele names of one character")
        lut = np.full(256, ord(missing), np.uint8)
        lut[:len(names)] = np.frombuffer("".join(names).encode(), np.uint8)
        out[s] = lut[idx[s]]
    return out


def one_allele(idx):
    """uint8[L0]: the "1" allele's index (the first present allele in file order), 255 if no allele is present."""
    flat = np.asarray(idx, np.uint8).reshape(len(idx), -1)
    present = flat != MISSING
    first = np.argmax(present, axis=1)
    return np.where(present.any(1), flat[np.arange(len(flat)), first], MISSING).astype(np.uint8)
