"""BCF input: a spec-written BCF, the Python reader / writer, the GT rule (csrc/bcf_gt.cuh:decode_gt through
tests/bcf_emu.cpp) and the driver's loader (host/io.cpp) on the CPU; on the GPU, put_bcf_gt + code_alleles against
put_vcf_text + code_alleles of the same records, the per-record diagnostics, sharded handles, ROH against the oracle,
and driver runs with --vcf x.bcf against --vcf x.vcf.gz."""
import ctypes as C
import gzip
import os
import shutil
import struct
import subprocess
import tempfile

import numpy as np
import pytest

from garlic_b200 import bcf, vcf
from tests.common import GOLDEN, arg, load_case, oracle_roh_idx

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
M = vcf.MISSING
_EMU = None


def emu():
    """tests/bcf_emu.cpp + host/io.cpp + host/cli.cpp, built into a temporary directory."""
    global _EMU
    if _EMU is None:
        so = os.path.join(tempfile.mkdtemp(prefix="garlic_bcf_emu_"), "bcf_emu.so")
        host = os.path.join(ROOT, "garlic_b200", "host")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "bcf_emu.cpp"),
                               os.path.join(host, "io.cpp"), os.path.join(host, "cli.cpp"), "-lz", "-pthread"])
        _EMU = C.CDLL(so)
        _EMU.emu_load_vcf.restype = C.c_longlong
    return _EMU


def emu_decode_gt(v0, v1, count, width):
    """→ int32[n, 3]: ok, a, b per call, from the host build of decode_gt."""
    v0, v1 = np.ascontiguousarray(v0, np.int32), np.ascontiguousarray(v1, np.int32)
    out = np.empty((len(v0), 3), np.int32)
    emu().emu_decode_gt(v0.ctypes.data_as(C.c_void_p), v1.ctypes.data_as(C.c_void_p), C.c_int(len(v0)), C.c_int(count),
                        C.c_int(width), out.ctypes.data_as(C.c_void_p))
    return out


def emu_load(path, log_base):
    """→ (samples, [(chrom, pos, id, ref, alts, line, gt_type)], [payload bytes per record], offsets) or the .error text."""
    cap = 1 << 20
    while True:
        buf = C.create_string_buffer(cap)
        need = C.c_longlong(0)
        n = emu().emu_load_vcf(path.encode(), log_base.encode(), buf, C.c_longlong(cap), C.byref(need))
        if n == -2:
            cap = need.value + 1
            continue
        if n < 0:
            return open(log_base + ".error").read()
        lines = buf.raw[:need.value].decode().split("\n")
        recs = [tuple(l.split("\t")) for l in lines[1:1 + n]]
        payloads = [bytes.fromhex(h) for h in lines[1 + n:1 + 2 * n]]
        off = np.array(lines[1 + 2 * n].split(), np.int64)
        return lines[0].split("\t"), recs, payloads, off


LETTERS = "ACGT"


def random_vcf(seed, N, L0, miss=0.08):
    """Records with 0..3 ALTs (one-letter names), half-missing calls, all-missing records and leading missing calls."""
    rng = np.random.default_rng(seed)
    n_alt = rng.integers(0, 4, L0)
    idx = (rng.random((L0, N, 2)) * (n_alt[:, None, None] + 1)).astype(np.uint8)
    idx[rng.random((L0, N, 2)) < miss] = vcf.MISSING
    idx[rng.random((L0, N)) < miss] = vcf.MISSING
    idx[0] = vcf.MISSING
    if L0 > 3:
        idx[1, :N // 2] = vcf.MISSING
        idx[2, 0, 0] = vcf.MISSING
    ref, alts = [], []
    for s in range(L0):
        perm = rng.permutation(4)
        ref.append(LETTERS[perm[0]])
        alts.append([LETTERS[p] for p in perm[1:1 + n_alt[s]]])
    half = L0 // 2
    return vcf.Vcf(samples=["s%d" % i for i in range(N)], chrom=["1"] * half + ["2"] * (L0 - half),
                   pos=np.arange(1, L0 + 1, dtype=np.int64) * 1000, ids=["rs%d" % i for i in range(L0)], ref=ref,
                   alts=alts, idx=idx)


def same_vcf(a, b):
    assert a.samples == b.samples and a.chrom == b.chrom and a.ids == b.ids and a.ref == b.ref and a.alts == b.alts
    assert np.array_equal(a.pos, b.pos) and np.array_equal(a.idx, b.idx)


def wide_vcf(seed, N, L0):
    """random_vcf with one record of 5 alleles (PL count 15) and one naming allele index 70 (int16 GT values)."""
    v = random_vcf(seed, N, L0)
    v.alts[4] = ["C", "G", "T", "<DEL>"]
    v.idx[4, :, 0] = np.arange(N) % 5
    v.alts[6] = ["A%d" % k for k in range(1, 71)]
    v.idx[6, 0] = (70, 0)
    return v


# ------------------------------------------------------------------------------------------------ spec pin
def _typed_str(s):
    b = s.encode()
    return (bytes([len(b) << 4 | 7]) if len(b) < 15 else bytes([0xF7, 0x11, len(b)])) + b


def _rec(shared_hex, alleles, indiv_hex):
    """A record: shared part = the fixed fields and ID (hex), then the allele strings, then FILTER (PASS)."""
    sh = bytes.fromhex(shared_hex) + b"".join(_typed_str(a) for a in alleles) + bytes.fromhex("11 00")
    ind = bytes.fromhex(indiv_hex)
    return struct.pack("<II", len(sh), len(ind)) + sh + ind


SPEC_HEADER = ("##fileformat=VCFv4.3\n"
               '##FILTER=<ID=PASS,Description="All filters passed",IDX=0>\n'
               '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype, with a quoted comma",IDX=3>\n'
               "##contig=<ID=1,length=1000000,IDX=0>\n"
               "##contig=<ID=2,length=1000000,IDX=2>\n"
               "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ta\tb\n").encode() + b"\0"
SPEC_ALTS70 = ["A%d" % k for k in range(1, 71)]
SPEC_RECORDS = [
    # CHROM 0, POS 99 (VCF 100), rlen 1, QUAL missing, n_allele 2, n_fmt 1 | n_sample 2, ID "rs1"; GT (key 3) int8
    # x 2: 0/1 = 02 04, 0|1 = 02 05
    _rec("00000000 63000000 01000000 0100807f 02000000 02000001 37 727331", ["A", "G"], "11 03 21 02 04 02 05"),
    # CHROM 0, POS 149, no ALT, ID missing (07); every sample a lone '.': count 1, value 00
    _rec("00000000 95000000 01000000 0100807f 01000000 02000001 07", ["A"], "11 03 11 00 00"),
    # CHROM 2 ("2"), POS 4999, ID of 20 characters (count 15: typed int 0x14 follows); ./. = 00 00, lone . = 00 81
    _rec("02000000 87130000 01000000 0100807f 02000000 02000001 f7 11 14" + "rs_long_identifier_x".encode().hex(),
         ["C", "T"], "11 03 21 00 00 00 81"),
    # CHROM 2, POS 5999, ID "rs4", REF G and 70 ALTs; GT int16 x 2: 70/0 = 008e 0002, 0|70 = 0002 008f
    _rec("02000000 6f170000 01000000 0100807f 47000000 02000001 37 727334", ["G"] + SPEC_ALTS70,
         "11 03 22 8e00 0200 0200 8f00"),
]
SPEC_BCF = b"BCF\x02\x02" + struct.pack("<I", len(SPEC_HEADER)) + SPEC_HEADER + b"".join(SPEC_RECORDS)
SPEC_WANT = vcf.Vcf(samples=["a", "b"], chrom=["1", "1", "2", "2"], pos=np.array([100, 150, 5000, 6000], np.int64),
                    ids=["rs1", ".", "rs_long_identifier_x", "rs4"], ref=["A", "A", "C", "G"],
                    alts=[["G"], [], ["T"], SPEC_ALTS70],
                    idx=np.array([[[0, 1], [0, 1]], [[M, M], [M, M]], [[M, M], [M, M]], [[70, 0], [0, 70]]], np.uint8))


@pytest.mark.parametrize("compress", [None, "bgzf"])
def test_spec_bcf_reads_as_written(tmp_path, compress):
    path = str(tmp_path / "spec.bcf")
    open(path, "wb").write(SPEC_BCF if compress is None else vcf.bgzf_compress(SPEC_BCF, 50))
    same_vcf(bcf.read_bcf(path), SPEC_WANT)
    res = emu_load(path, str(tmp_path / "log"))
    assert not isinstance(res, str), res
    samples, recs, payloads, off = res
    assert samples == ["a", "b"]
    assert [r[:6] for r in recs] == [("1", "100", "rs1", "A", "G", "1"), ("1", "150", ".", "A", ".", "2"),
                                     ("2", "5000", "rs_long_identifier_x", "C", "T", "3"),
                                     ("2", "6000", "rs4", "G", ",".join(SPEC_ALTS70), "4")]
    assert [int(r[6]) for r in recs] == [0x21, 0x11, 0x21, 0x22]
    assert payloads == [bytes.fromhex(h) for h in ("02040205", "00000000", "00000081", "8e00020002008f00")]
    assert list(off) == [0, 4, 8, 12, 20]
    assert "Chromosome chr1: 2 sites." in open(str(tmp_path / "log") + ".log").read()
    g, o, t = bcf.gt_payload(path)
    assert g == b"".join(payloads) and np.array_equal(o, off) and list(t) == [0x21, 0x11, 0x21, 0x22]


# ------------------------------------------------------------------------------------------------ round trips
ROUND_TRIPS = [(w, fmt, lone, compress, idx) for w in (None, 2, 4) for fmt in vcf.FORMATS for lone in (False, True)
               for compress, idx in ((None, True), ("bgzf", False), ("gz", True))]


@pytest.mark.parametrize("width,fmt,lone,compress,idx", ROUND_TRIPS)
def test_round_trip(tmp_path, width, fmt, lone, compress, idx):
    v = wide_vcf(1, 13, 57)
    path = bcf.write_bcf(str(tmp_path / "x.bcf"), v, fmt, lone, width, compress, idx, block_size=97)
    same_vcf(bcf.read_bcf(path), v)
    _, recs = bcf._parse(path)
    w = {None: 2, 2: 2, 4: 4}[width]                               # record 6 names allele 70: int16 at least
    assert {r["gt_type"] & 15 for r in recs} == {bcf.TYPE_OF_WIDTH[w]}
    assert (recs[0]["gt_type"] >> 4) == (1 if lone else 2)         # record 0: every sample missing
    if fmt != "GT":
        assert recs[4]["format"]["PL"].shape == (13, 15)            # 5 alleles: PL count 15 (overflow descriptor)
    v1 = random_vcf(2, 5, 20)
    same_vcf(bcf.read_bcf(bcf.write_bcf(str(tmp_path / "y.bcf"), v1, fmt, lone, width, compress, idx)), v1)
    if width is None:
        assert {r["gt_type"] & 15 for r in bcf._parse(str(tmp_path / "y.bcf"))[1]} == {bcf.INT8}


# ------------------------------------------------------------------------------------------------ loader = VCF loader
@pytest.mark.parametrize("compress,width,fmt,lone", [(None, None, "GT", False), ("bgzf", 2, "GT:AD:DP:GQ:PL", True),
                                                     ("gz", 4, "GT", True), ("bgzf", None, "GT:AD:DP:GQ:PL", False)])
def test_loader_equals_vcf_loader(tmp_path, compress, width, fmt, lone):
    v = random_vcf(7, 21, 300)
    pv = vcf.write_vcf(str(tmp_path / "x.vcf.gz"), v, fmt, "|", lone, "bgzf")
    pb = bcf.write_bcf(str(tmp_path / "x.bcf"), v, fmt, lone, width, compress, block_size=1000)
    rv, rb = emu_load(pv, str(tmp_path / "lv")), emu_load(pb, str(tmp_path / "lb"))
    assert not isinstance(rv, str) and not isinstance(rb, str), (rv, rb)
    assert rb[0] == rv[0]
    assert [r[:5] for r in rb[1]] == [r[:5] for r in rv[1]]
    assert [int(r[5]) for r in rb[1]] == list(range(1, 301))         # record numbers
    assert open(str(tmp_path / "lb.log")).read() == open(str(tmp_path / "lv.log")).read()
    g, off, types = bcf.gt_payload(pb)
    assert b"".join(rb[2]) == g and np.array_equal(rb[3], off) and [int(r[6]) for r in rb[1]] == list(types)
    assert all(o % 4 == 0 for o in off)
    text, toff = vcf.sample_text(pv)
    for s in range(300):
        count, w = types[s] >> 4, bcf.WIDTH[types[s] & 15]
        vals = np.frombuffer(rb[2][s][:21 * count * w], {1: "<i1", 2: "<i2", 4: "<i4"}[w]).reshape(21, count)
        got = emu_decode_gt(vals[:, 0], vals[:, 1] if count > 1 else np.zeros(21), count, w)
        cols = text[toff[s]:toff[s + 1]].decode().split("\t")
        assert got[:, 0].all()
        assert [tuple(x) for x in got[:, 1:]] == [vcf.parse_gt(c) for c in cols]


# ------------------------------------------------------------------------------------------------ decode_gt
def _check_decode(v0, v1, count, width):
    got = emu_decode_gt(v0, v1, count, width)
    for k in range(len(v0)):
        want = bcf.decode_gt(int(v0[k]), int(v1[k]), count, width)
        assert (tuple(got[k, 1:]) if got[k, 0] else None) == want, (v0[k], v1[k], count, width)


def test_decode_gt_every_int8_pair():
    pairs = np.arange(65536)
    v0, v1 = (pairs >> 8).astype(np.int8).astype(np.int32), (pairs & 255).astype(np.int8).astype(np.int32)
    for count in (1, 2, 3):
        _check_decode(v0, v1, count, 1)
    ok = [bcf.decode_gt(int(a), int(b), 2, 1) is not None for a, b in zip(v0, v1)]
    assert sum(ok) == 128 * 128 + 2                                   # every non-negative pair, and 00 81 / 01 81
    assert bcf.decode_gt(2, -127, 2, 1) is None and bcf.decode_gt(-127, 0, 2, 1) is None   # haploid; EOV first
    assert bcf.decode_gt(0, 0, 1, 1) == (M, M) and bcf.decode_gt(2, 0, 1, 1) is None
    assert bcf.decode_gt(2, 5, 2, 1) == (0, 1) and bcf.decode_gt(0, -127, 2, 1) == (M, M)


@pytest.mark.parametrize("width", [2, 4])
def test_decode_gt_wide_boundaries(width):
    eov, miss = bcf.EOV[width], bcf.EOV[width] - 1
    edge = [0, 1, 2, 3, 510, 511, 512, 513, 140, 141, -1, -2, eov, miss, eov + 1, eov + 6, -200,
            (1 << (8 * width - 1)) - 1]
    v0, v1 = np.array([a for a in edge for _ in edge]), np.array([b for _ in edge for b in edge])
    for count in (1, 2, 3):
        _check_decode(v0, v1, count, width)
    assert bcf.decode_gt(510, 511, 2, width) == (254, 254)             # index 254
    assert bcf.decode_gt(512, 2, 2, width) is None and bcf.decode_gt(2, 513, 2, width) is None    # index 255
    assert bcf.decode_gt(1, eov, 2, width) == (M, M) and bcf.decode_gt(eov, 1, 2, width) is None
    assert bcf.decode_gt(miss, 2, 2, width) is None and bcf.decode_gt(2, miss, 2, width) is None


# ------------------------------------------------------------------------------------------------ rejections
def _layout(data):
    """→ (header end, [(record start, l_shared, l_indiv)]) of an uncompressed BCF."""
    i = 9 + struct.unpack_from("<I", data, 5)[0]
    recs = []
    while i < len(data):
        ls, li = struct.unpack_from("<II", data, i)
        recs.append((i, ls, li))
        i += 8 + ls + li
    return recs


def _patch(data, at, new):
    return data[:at] + new + data[at + len(new):]


def _header(data, fn):
    n = struct.unpack_from("<I", data, 5)[0]
    text = fn(data[9:9 + n].decode()).encode()
    return data[:5] + struct.pack("<I", len(text)) + text + data[9 + n:]


def _base():
    v = random_vcf(3, 4, 12)
    return bcf.bcf_bytes(v, "GT:AD:DP:GQ:PL"), v


def _rec_field(k, off, new):
    def f(d):
        r = _layout(d)[k][0]
        return _patch(d, r + 8 + off, new)
    return f


def _indiv(k, off, new):
    def f(d):
        r, ls, _ = _layout(d)[k]
        return _patch(d, r + 8 + ls + off, new)
    return f


def _lengths(k, fn):
    def f(d):
        r, ls, li = _layout(d)[k]
        return _patch(d, r, struct.pack("<II", *fn(ls, li)))
    return f


def _gt_only(d):
    return bcf.bcf_bytes(random_vcf(3, 4, 12), "GT")


REJECT = [
    ("version", lambda d: b"BCF\x02\x01" + d[5:], "BCF version 2.1", None),
    ("trunc_header", lambda d: d[:40], "truncated header", None),
    ("trunc_record", lambda d: d[:_layout(d)[5][0] + 30], "record 6: truncated record", None),
    ("trunc_lengths", _lengths(11, lambda ls, li: (ls, li + 1000)), "run past the end of the file", 12),
    ("trunc_8", lambda d: d[:_layout(d)[3][0] + 5], "record 4: truncated record", None),
    ("l_shared", _lengths(2, lambda ls, li: (20, li + ls - 20)), "l_shared (20) is too small", 3),
    ("l_shared_alleles", _lengths(2, lambda ls, li: (27, li + ls - 27)), "l_shared (27) is too small", 3),
    ("no_chrom", lambda d: _header(d, lambda t: t.replace("#CHROM", "#XHROM")), "no #CHROM header line", None),
    ("no_samples", lambda d: _header(d, lambda t: t.replace("\ts0\ts1\ts2\ts3", "")), "names no samples", None),
    ("dup_samples", lambda d: _header(d, lambda t: t.replace("\ts2", "\ts1")), "duplicate sample ID", None),
    ("mixed_idx", lambda d: _header(d, lambda t: t.replace(",IDX=1>", ">", 1)), "mix lines with and without IDX=",
     None),
    ("n_sample", _rec_field(4, 20, struct.pack("<I", 1 << 24 | 5)), "5 samples, but the #CHROM header names 4", 5),
    ("chrom", _rec_field(3, 0, struct.pack("<i", 7)), "CHROM index 7 is not in the header's contig dictionary", 4),
    ("key", _indiv(2, 0, bytes([0x11, 9])), "FORMAT key 9 is not in the header's dictionary of strings", 3),
    ("not_gt", _indiv(2, 0, bytes([0x11, 3])), "FORMAT does not start with GT (DP)", 3),
    ("gt_float", _indiv(2, 2, bytes([0x25])), "the GT field is of type 5, not int8, int16 or int32", 3),
    ("gt_count0", _indiv(2, 2, bytes([0x01])), "the GT field has a count of 0", 3),
    ("gt_long", lambda d: _indiv(2, 2, bytes([0x51]))(_gt_only(d)), "is longer than l_indiv", 3),
]


@pytest.mark.parametrize("name,damage,msg,rec", REJECT, ids=[r[0] for r in REJECT])
def test_loader_rejects(tmp_path, name, damage, msg, rec):
    data, v = _base()
    path = str(tmp_path / "x.bcf")
    open(path, "wb").write(damage(data))
    res = emu_load(path, str(tmp_path / "log"))
    assert isinstance(res, str) and msg in res, res
    assert path in res
    if rec is not None:
        assert "record %d (%s:%d)" % (rec, v.chrom[rec - 1], v.pos[rec - 1]) in res or \
            ("record %d:" % rec in res and name in ("chrom", "trunc_lengths")), res
    with pytest.raises(vcf.VcfError):
        bcf.read_bcf(path)


def _first_block_end(z):
    return int.from_bytes(z[16:18], "little") + 1


@pytest.mark.parametrize("damage,msg", [
    (lambda z: z[:_first_block_end(z) - 8] + bytes([z[_first_block_end(z) - 8] ^ 1]) + z[_first_block_end(z) - 7:],
     "CRC32 mismatch"),
    (lambda z: z[:-40], "truncated BGZF block"),
    (lambda z: z[:_first_block_end(z) + 7], "truncated BGZF block header"),
])
def test_bgzf_damage_is_an_error(tmp_path, damage, msg):
    path = str(tmp_path / "x.bcf")
    bcf.write_bcf(path, random_vcf(2, 9, 40), "GT:AD:DP:GQ:PL", block_size=300)
    z = open(path, "rb").read()
    open(path, "wb").write(damage(z))
    res = emu_load(path, str(tmp_path / "log"))
    assert isinstance(res, str) and msg in res and path in res, res


# ------------------------------------------------------------------------------------------------ GPU
def _shape(g, N, L0, ind_offset=0):
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 1000
    g.set_shape(N, L0, np.array([0, L0 // 2, L0], np.int64), pos, ind_offset=ind_offset)


def _put_bcf(g, payload, N, block=1024):
    gt, off, types = payload
    diag = [g.put_bcf_gt(gt, off[s0:s0 + block + 1], types[s0:s0 + block], N, s0) for s0 in range(0, len(types), block)]
    return [np.concatenate(d) for d in zip(*diag)]


def _put_vcf(g, text, off, block=1024):
    diag = [g.put_vcf_text(text, off[s0:s0 + block + 1], s0) for s0 in range(0, len(off) - 1, block)]
    return [np.concatenate(d) for d in zip(*diag)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,L0,width", [(1, 3001, 1), (3, 2333, 2), (29, 5017, 4), (77, 4100, 1), (513, 3075, 1),
                                        (513, 3075, 2)])
def test_bcf_coding_equals_vcf_coding(tmp_path, N, L0, width):
    from garlic_b200 import synth
    from garlic_b200.api import GarlicGPU
    v = random_vcf(N + 5, N, L0)
    v.idx[5] = M                                                   # a second all-missing record (count 1)
    lone = N % 2 == 1
    pv = vcf.write_vcf(str(tmp_path / "x.vcf"), v, "GT", "/", lone)
    pb = bcf.write_bcf(str(tmp_path / "x.bcf"), v, "GT:AD:DP:GQ:PL", lone, width)
    payload = bcf.gt_payload(pb)
    assert (payload[2] & 15 == bcf.TYPE_OF_WIDTH[width]).all() and ((payload[2] >> 4) == 1).any() == lone
    out = []
    for kind in ("vcf", "bcf"):
        g = GarlicGPU(0)
        _shape(g, N, L0)
        if kind == "vcf":
            nc, mx, bad = _put_vcf(g, *vcf.sample_text(pv))
        else:
            mx, bad = _put_bcf(g, payload, N, block=4096)             # ragged last block
        assert (bad == -1).all()
        g.code_alleles()
        f, keep, L = g.filter()
        out.append(dict(mx=mx, one=g.get_one_allele(255), counts=np.array(g.get_counts()), f=f.copy(), keep=keep.copy(),
                        all=synth.unpack_codes(g.get_genotypes(False), L0),
                        kept=synth.unpack_codes(g.get_genotypes(True), L)))
        g.close()
    a, b = out
    assert np.array_equal(b["one"], vcf.one_allele(v.idx))
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _diag_payload(rows, width=1):
    """rows: per record (count, values[N * count]) → payload, offsets, descriptors."""
    parts, off, types = [], [0], []
    dt = {1: "<i1", 2: "<i2", 4: "<i4"}[width]
    for count, vals in rows:
        raw = np.array(vals, np.int64).astype(dt).tobytes()
        raw += b"\0" * (-len(raw) % 4)
        parts.append(raw)
        off.append(off[-1] + len(raw))
        types.append(count << 4 | bcf.TYPE_OF_WIDTH[width])
    return b"".join(parts), np.array(off, np.int64), np.array(types, np.uint8)


def _diag_rows(N, width):
    e = bcf.EOV[width]
    ok = [2, 4] * N
    rows, want = [], []

    def put(vals, mx, bad, count=2):
        rows.append((count, vals))
        want.append((mx, bad))
    put(ok, 1, -1)
    put([4, 2] + ok[2:], 1, -1)
    for where in (0, N // 2, N - 1):                                   # first, middle, last sample
        too_big = [-126, 2] if width == 1 else [512, 2]             # int8: a reserved value; else allele index 255
        for bad_call in ([2, e], [e, 2], [e - 1, 2], [2, -3], too_big):
            vals = list(ok)
            vals[2 * where:2 * where + 2] = bad_call
            put(vals, 1, where)
    put([0, e] * N, -1, -1)
    put([0] * N, -1, -1, count=1)
    put([2] + [0] * (N - 1), -1, 0, count=1)                           # a haploid call with an allele present
    put([2, 2, 2] * N, -1, 0, count=3)
    put([2, 4] + [2, 8] * (N - 1), 3, -1)                              # index 3: above a small ALT count, reported
    if width > 1:
        put([2, 510] * N, 254, -1)
    return rows, want


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1, 2, 4])
@pytest.mark.parametrize("lo,n", [(0, 7), (1, 2), (6, 1), (3, 4)])
def test_bcf_diagnostics(width, lo, n):
    from garlic_b200.api import GarlicGPU
    N = 7
    rows, want = _diag_rows(N, width)
    rows, want = rows * 3, want * 3                                   # spans several CTAs' grid-stride loop
    gt, off, types = _diag_payload(rows, width)
    g = GarlicGPU(0)
    _shape(g, n, len(rows), ind_offset=lo)
    mx, bad = g.put_bcf_gt(gt, off, types, N, 0)
    assert list(mx) == [w[0] for w in want] and list(bad) == [w[1] for w in want]
    g.close()
    long_vals = [2, 4] * 3000                                          # more than one pass of the CTA's loop
    long_vals[2 * 2999:] = [2, 6]
    long_vals[2 * 2500:2 * 2500 + 2] = [4, 0]
    gt, off, types = _diag_payload([(2, long_vals)], width)
    g = GarlicGPU(0)
    _shape(g, n, 1, ind_offset=lo)
    mx, bad = g.put_bcf_gt(gt, off, types, 3000, 0)
    assert list(mx) == [2] and list(bad) == [-1]
    long_vals[2 * 2999 + 1] = e = bcf.EOV[width]
    gt, off, types = _diag_payload([(2, long_vals)], width)
    mx, bad = g.put_bcf_gt(gt, off, types, 3000, 0)
    assert list(mx) == [1] and list(bad) == [2999]
    g.close()


class _DevArray:
    """A device buffer of the library as a torch tensor (no copy)."""
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


@pytest.mark.gpu
@pytest.mark.parametrize("N,cuts,width", [(77, [1, 30], 1), (29, [3, 4], 2), (513, [130, 259], 1)])
def test_sharded_handles_equal_one_handle(tmp_path, N, cuts, width):
    import torch
    from garlic_b200 import synth
    from garlic_b200.api import GarlicGPU
    L0 = 4100
    v = random_vcf(N, N, L0)
    payload = bcf.gt_payload(bcf.write_bcf(str(tmp_path / "x.bcf"), v, "GT", True, width))
    whole = GarlicGPU(0)
    _shape(whole, N, L0)
    want_diag = _put_bcf(whole, payload, N)
    whole.code_alleles()
    want_rows = synth.unpack_codes(whole.get_genotypes(False), L0)
    want_counts = whole.get_counts()
    bounds = [0] + cuts + [N]
    hs = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        g = GarlicGPU(0)
        _shape(g, hi - lo, L0, ind_offset=lo)
        diag = _put_bcf(g, payload, N)                               # every handle decodes every sample
        assert all(np.array_equal(a, b) for a, b in zip(diag, want_diag))
        g.sync()
        hs.append(g)
    keys = [torch.as_tensor(_DevArray(g.first_allele_keys_dev(), L0, "<i8"), device="cuda") for g in hs]
    mn = np.minimum.reduce([k.cpu().numpy().view(np.uint64) for k in keys])
    for k in keys:
        k.copy_(torch.from_numpy(mn.view(np.int64)))
    torch.cuda.synchronize()
    got_rows, got_counts = [], np.zeros((4, L0), np.int64)
    for g in hs:
        g.code_alleles()
        got_rows.append(synth.unpack_codes(g.get_genotypes(False), L0))
        got_counts += np.array(g.get_counts())
    assert np.array_equal(np.concatenate(got_rows), want_rows)
    assert np.array_equal(got_counts, np.array(want_counts))
    assert all(np.array_equal(g.get_one_allele(255), whole.get_one_allele(255)) for g in hs)
    for g in hs + [whole]:
        g.close()


@pytest.mark.gpu
def test_put_bcf_gt_refusals(tmp_path):
    from garlic_b200.api import GarlicError, GarlicGPU
    v = random_vcf(5, 8, 64)
    gt, off, types = bcf.gt_payload(bcf.write_bcf(str(tmp_path / "x.bcf"), v))
    g = GarlicGPU(0)
    _shape(g, 8, 64)
    g.put_alleles(vcf.tped_alleles(v.idx, v.ref, v.alts))
    with pytest.raises(GarlicError, match="tped input"):
        g.put_bcf_gt(gt, off, types, 8, 0)
    _shape(g, 8, 64)
    g.put_bed(np.zeros((64, 2), np.uint8))
    with pytest.raises(GarlicError, match=".bed input"):
        g.put_bcf_gt(gt, off, types, 8, 0)
    _shape(g, 8, 64)
    for bad_types, msg in ((np.where(np.arange(64) == 9, 0x25, types), "descriptor"),
                           (np.where(np.arange(64) == 9, 0x01, types), "descriptor"),
                           (np.where(np.arange(64) == 9, 0x41, types), "shorter")):
        with pytest.raises(GarlicError, match=msg):
            g.put_bcf_gt(gt, off, bad_types.astype(np.uint8), 8, 0)
    with pytest.raises(GarlicError, match="multiple of 4"):
        g.put_bcf_gt(gt, off + np.where(np.arange(65) == 3, 2, 0), types, 8, 0)
    with pytest.raises(GarlicError, match="n_samples"):
        g.put_bcf_gt(gt, off, types, 7, 0)
    g.put_bcf_gt(gt, off, types, 8, 0)                                # BCF is VCF input: put_alleles refuses it
    with pytest.raises(GarlicError, match="VCF input"):
        g.put_alleles(vcf.tped_alleles(v.idx, v.ref, v.alts))
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lod_0", "lod_small", "wlod_cm"])
def test_roh_from_bcf_equal_oracle(tmp_path, name):
    from garlic_b200.pipeline import HotPath
    from oracle import oracle as orc
    ds, args = load_case(name)
    W = arg(args, "--winsize", cast=int)
    err = arg(args, "--error", None, float)
    cutoff = arg(args, "--lod-cutoff", None, float)
    ov = arg(args, "--overlap-frac", 0.25, float)
    weighted, cm = "--weighted" in args, "--cm" in args
    res = orc.run_pipeline(ds, W, err, cutoff, ov, weighted=weighted, cm=cm)
    path = bcf.write_bcf(str(tmp_path / "x.bcf"), vcf.from_dataset(ds, seed=5), "GT:AD:DP:GQ:PL", True)
    hp = HotPath().load(ds, weighted=weighted, cm=cm, error=err, bcf=bcf.gt_payload(path))
    assert hp.L == res["n_used"]
    if weighted:
        hp.g.ld_band(W)
    got = hp.roh(W, cutoff, res["overlap_frac"], weighted=weighted, cm=cm)
    assert got and [(r[0], r[1], r[5], r[6]) for r in got] == oracle_roh_idx(res)
    hp.close()


# ------------------------------------------------------------------------------------------------ CLI (GPU)
BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")


def _cli_inputs(name, tmp, fmt="GT", lone=False, n_ind=None, rename=None):
    """Writes a golden case as tped/tfam (syn.*), as a BGZF VCF and as BCF (BGZF and uncompressed); returns (base argv
    without input or output, tfam, {kind: path}, the Vcf).  rename = (snp, name): that SNP's "1" allele gets a longer
    name."""
    ds, args = load_case(name)
    if n_ind is not None:
        ds.alleles, ds.ind_ids = ds.alleles[:, :n_ind], ds.ind_ids[:n_ind]
    ds.write(tmp)
    if os.path.exists(os.path.join(GOLDEN, name, "in.freq")):
        shutil.copy(os.path.join(GOLDEN, name, "in.freq"), os.path.join(tmp, "syn.freq"))
    v = vcf.from_dataset(ds, seed=11)
    if rename is not None:
        s, new = rename
        k = vcf.one_allele(v.idx)[s]
        if k == 0:
            v.ref[s] = new
        else:
            v.alts[s][k - 1] = new
    paths = {"vcf": vcf.write_vcf(os.path.join(tmp, "in.vcf.gz"), v, fmt, "|", lone, "bgzf", block_size=4000),
             "bcf": bcf.write_bcf(os.path.join(tmp, "in.bcf"), v, fmt, lone, block_size=4000),
             "ubcf": bcf.write_bcf(os.path.join(tmp, "in.u.bcf"), v, fmt, lone, compress=None)}
    with open(os.path.join(GOLDEN, name, "cmd.txt")) as f:
        cmd = [a.replace("<tmp>", tmp) for a in f.readline().split()[1:] if a != "--raw-lod"]
    i = cmd.index("--out")
    del cmd[i:i + 2]
    i = cmd.index("--tped")
    tfam = cmd[i + 3]
    return cmd[:i] + cmd[i + 4:], tfam, paths, v


def _run(argv, out):
    os.makedirs(os.path.dirname(out), exist_ok=True)
    return subprocess.run([BIN] + argv + ["--out", out], capture_output=True, text=True, timeout=300)


def _same_outputs(a, b, subs):
    """Outputs of prefix a and b byte for byte; in b's .log every (old, new) of subs is replaced first."""
    for ext in (".roh.bed", ".freq.gz"):
        assert os.path.exists(a + ext) == os.path.exists(b + ext), ext
        if os.path.exists(a + ext):
            assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), ext
    da, db = os.path.dirname(a), os.path.dirname(b)
    ka = sorted(f for f in os.listdir(da) if f.endswith(".kde"))
    assert ka == sorted(f for f in os.listdir(db) if f.endswith(".kde"))
    for f in ka:
        assert open(os.path.join(da, f)).read() == open(os.path.join(db, f)).read()
    log = open(b + ".log").read()
    for old, new in subs:
        log = log.replace(old, new)
    assert open(a + ".log").read() == log


@pytest.mark.gpu
@pytest.mark.parametrize("name,extra,fmt,lone,kinds", [
    ("lod_0", [], "GT", False, ("bcf", "ubcf")),
    ("lod_small", ["TFAM"], "GT:AD:DP:GQ:PL", True, ("bcf", "ubcf")),
    ("wlod_phased", [], "GT:AD:DP:GQ:PL", False, ("bcf",)),           # --phased (in the case's command)
    ("lod_1", ["--freq-only"], "GT", True, ("bcf", "ubcf")),
    ("auto_cutoff", ["--kde-direct", "--seed", "5"], "GT", True, ("bcf",)),
    ("freq_file", [], "GT:AD:DP:GQ:PL", True, ("ubcf",)),
])
def test_cli_bcf_equals_vcf(tmp_path, name, extra, fmt, lone, kinds):
    tmp = str(tmp_path)
    base, tfam, paths, _ = _cli_inputs(name, tmp, fmt, lone)
    if "TFAM" in extra:
        extra = ["--tfam", tfam]
    r = _run(base + ["--vcf", paths["vcf"]] + extra, os.path.join(tmp, "v", "o"))
    assert r.returncode == 0, r.stderr[-2000:]
    for kind in kinds:
        out = os.path.join(tmp, kind, "o")
        r = _run(base + ["--vcf", paths[kind]] + extra, out)
        assert r.returncode == 0, r.stderr[-2000:]
        _same_outputs(os.path.join(tmp, "v", "o"), out, [(paths[kind], paths["vcf"]), (out, os.path.join(tmp, "v", "o"))])
        assert "VCF file: " + paths[kind] in open(out + ".log").read()


@pytest.mark.gpu
def test_cli_bcf_long_allele_name_and_freq_file(tmp_path):
    """A "1" allele named by more than one character: .freq.gz prints it and --freq-file compares whole tokens."""
    tmp = str(tmp_path)
    s = 40
    base, _, paths, v = _cli_inputs("freq_file", tmp, "GT", False, rename=(s, "<DEL:ME>"))
    ds = load_case("freq_file")[0]
    rows = open(os.path.join(tmp, "syn.freq")).read().splitlines(True)
    t = rows[s + 1].split()
    k = vcf.one_allele(v.idx)[s]
    old = chr(ds.alleles[s][v.idx[s] == k][0])
    t[3] = "<DEL:ME>" if t[3] == old else t[3]
    rows[s + 1] = "\t".join(t) + "\n"
    open(os.path.join(tmp, "vcf.freq"), "w").write("".join(rows))
    base[base.index("--freq-file") + 1] = os.path.join(tmp, "vcf.freq")
    r = _run(base + ["--vcf", paths["vcf"]], os.path.join(tmp, "v", "o"))
    assert r.returncode == 0, r.stderr[-2000:]
    out = os.path.join(tmp, "b", "o")
    r = _run(base + ["--vcf", paths["bcf"]], out)
    assert r.returncode == 0, r.stderr[-2000:]
    _same_outputs(os.path.join(tmp, "v", "o"), out, [(paths["bcf"], paths["vcf"]), (out, os.path.join(tmp, "v", "o"))])
    i = base.index("--freq-file")                                    # .freq.gz prints the whole name
    base = base[:i] + base[i + 2:] + ["--freq-only"]
    for kind in ("vcf", "bcf"):
        r = _run(base + ["--vcf", paths[kind]], os.path.join(tmp, kind + "f", "o"))
        assert r.returncode == 0, r.stderr[-2000:]
    freq = gzip.open(os.path.join(tmp, "bcff", "o.freq.gz"), "rt").read()
    assert "<DEL:ME>" in freq.splitlines()[s + 1]
    assert freq == gzip.open(os.path.join(tmp, "vcff", "o.freq.gz"), "rt").read()


@pytest.mark.gpu
def test_cli_bcf_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tmp = str(tmp_path)
    base, _, paths, _ = _cli_inputs("lod_small", tmp, n_ind=29)
    r1 = _run(base + ["--vcf", paths["vcf"]], os.path.join(tmp, "a", "o"))
    r2 = _run(base + ["--vcf", paths["bcf"], "--gpus", "2"], os.path.join(tmp, "b", "o"))
    assert r1.returncode == 0 and r2.returncode == 0, r1.stderr[-1000:] + r2.stderr[-1000:]
    log_b = open(os.path.join(tmp, "b", "o.log")).read()
    assert "--gpus 2" in log_b
    open(os.path.join(tmp, "b", "o.log"), "w").write(log_b.replace(" --gpus 2", ""))
    _same_outputs(os.path.join(tmp, "a", "o"), os.path.join(tmp, "b", "o"),
                  [(paths["bcf"], paths["vcf"]), (os.path.join(tmp, "b", "o"), os.path.join(tmp, "a", "o"))])


def _edit_gt(path, s, vals):
    """Rewrites record s's GT values (an uncompressed BCF with int8 count-2 GTs) with vals (sample, v0, v1)."""
    data = bytearray(open(path, "rb").read())
    r, ls, _ = _layout(bytes(data))[s]
    p = r + 8 + ls + 3
    for i, a, b in vals:
        data[p + 2 * i:p + 2 * i + 2] = bytes([a & 255, b & 255])
    open(path, "wb").write(bytes(data))


@pytest.mark.gpu
@pytest.mark.parametrize("vals,msg", [
    ([(3, 4, 0x81)], "the GT of sample %s is not two allele indices"),          # a haploid call with an allele present
    ([(3, 2 + 2 * 40, 2)], "allele index 40 but only"),
])
def test_cli_bcf_errors(tmp_path, vals, msg):
    tmp = str(tmp_path)
    base, _, paths, v = _cli_inputs("lod_0", tmp)
    _edit_gt(paths["ubcf"], 100, vals)
    r = _run(base + ["--vcf", paths["ubcf"]], os.path.join(tmp, "b", "o"))
    assert r.returncode != 0
    err = open(os.path.join(tmp, "b", "o.error")).read()
    where = "%s record 101 (%s:%d): " % (paths["ubcf"], v.chrom[100], v.pos[100])
    assert where in err, err
    assert (msg % v.samples[3] if "%s" in msg else msg) in err, err
    assert v.samples[3] in err and ("autosomes" in err) == ("%s" in msg)
