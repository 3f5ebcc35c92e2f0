"""VCF input: the Python reader / writer, the GT grammar (csrc/vcf_gt.cuh through tests/vcf_emu.cpp) and the driver's
loader with its BGZF reader (host/io.cpp) on the CPU; on the GPU, put_vcf_text + code_alleles against the tped coding
path (orc.code_tped of the equivalent alleles), the per-record diagnostics, sharded handles, ROH against the oracle, and
driver runs with --vcf against the same data as --tped."""
import ctypes as C
import gzip
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from garlic_b200 import synth, vcf
from tests.common import GOLDEN, arg, load_case, oracle_roh_idx

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_EMU = None


def emu():
    """tests/vcf_emu.cpp + host/io.cpp + host/cli.cpp, built into a temporary directory."""
    global _EMU
    if _EMU is None:
        so = os.path.join(tempfile.mkdtemp(prefix="garlic_vcf_emu_"), "vcf_emu.so")
        host = os.path.join(ROOT, "garlic_b200", "host")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "vcf_emu.cpp"),
                               os.path.join(host, "io.cpp"), os.path.join(host, "cli.cpp"), "-lz", "-pthread"])
        _EMU = C.CDLL(so)
        _EMU.emu_load_vcf.restype = C.c_longlong
    return _EMU


def emu_parse_gt(s):
    a, b = C.c_int(-1), C.c_int(-1)
    raw = s.encode()
    ok = emu().emu_parse_gt(C.c_char_p(raw), C.c_longlong(len(raw)), C.byref(a), C.byref(b))
    return (a.value, b.value) if ok else None


def emu_load_vcf(path, log_base):
    """→ (samples, [(chrom, pos, id, ref, alts, line)], [sample text per record]) or the .error text on failure."""
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
        return lines[0].split("\t"), recs, lines[1 + n:1 + 2 * n]


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


# ------------------------------------------------------------------------------------------------ CPU
WRITE_CASES = [(None, "GT", "/", False), ("gz", "GT:AD:DP:GQ:PL", "|", True), ("bgzf", "GT", "|", True),
               ("bgzf", "GT:AD:DP:GQ:PL", "/", False)]


@pytest.mark.parametrize("compress,fmt,sep,lone", WRITE_CASES)
def test_round_trip(tmp_path, compress, fmt, sep, lone):
    v = random_vcf(1, 13, 57)
    v.alts[5] = v.alts[5] + ["<DEL>"]                       # long names survive the round trip
    path = vcf.write_vcf(str(tmp_path / "x.vcf"), v, fmt, sep, lone, compress, block_size=97)
    got = vcf.read_vcf(path)
    same_vcf(got, v)
    text, off = vcf.sample_text(path)
    assert len(off) == 58
    # the driver's loader (and its BGZF reader, blocks of 97 bytes: lines cross blocks) sees the same records
    res = emu_load_vcf(path, str(tmp_path / "log"))
    assert not isinstance(res, str), res
    samples, recs, texts = res
    assert samples == v.samples
    assert [r[:5] for r in recs] == [(v.chrom[s], str(v.pos[s]), v.ids[s], v.ref[s], ",".join(v.alts[s]) or ".")
                                     for s in range(57)]
    assert [int(r[5]) for r in recs] == list(range(4, 61))          # two meta lines and the header come first
    assert [t.encode() for t in texts] == [text[off[s]:off[s + 1]] for s in range(57)]
    if lone:
        both = (v.idx == vcf.MISSING).all(2)
        assert both.any() and any(c.split(":")[0] == "." for t in texts for c in t.split("\t"))


def test_bgzf_blocks_are_standard(tmp_path):
    data = b"".join(b"line %d\n" % i for i in range(3000))
    z = vcf.bgzf_compress(data, 1000)
    assert gzip.decompress(z) == data                            # multi-member gzip
    assert z.endswith(vcf.BGZF_EOF) and z[12:16] == b"BC\x02\x00"


@pytest.mark.parametrize("name", ["lod_0", "lod_small", "wlod_cm", "wlod_phased", "gl_pl", "freq_file"])
def test_dataset_vcf_is_the_tped(name):
    ds, _ = load_case(name)
    v = vcf.from_dataset(ds, seed=3)
    assert np.array_equal(vcf.tped_alleles(v.idx, v.ref, v.alts), ds.alleles)
    one = vcf.one_allele(v.idx)
    assert (one == 0).any() and ((one > 0) & (one < 255)).any()
    half = (v.idx == vcf.MISSING).sum(2) == 1
    assert half.any()


def test_multi_allelic_convention():
    M = vcf.MISSING
    idx = np.array([[[M, M], [M, M]],          # nothing present: no "1" allele
                    [[M, 2], [0, 1]],          # half-missing first call: its present allele (index 2) is the "1" allele
                    [[1, 0], [2, 2]]], np.uint8)
    ref, alts = ["A", "C", "G"], [["T"], ["G", "T"], ["A", "C"]]
    assert list(vcf.one_allele(idx)) == [M, 2, 1]
    al = vcf.tped_alleles(idx, ref, alts)
    assert bytes(al[1].reshape(-1)) == b"0TCG" and bytes(al[2].reshape(-1)) == b"AGCC"


GT_TABLE = [("0/1", (0, 1)), ("1|0", (1, 0)), ("./.", (255, 255)), (".", (255, 255)), ("0/.", (0, 255)),
            ("./1", (255, 1)), ("12/3", (12, 3)), ("254/0", (254, 0)), ("0/1:3,4:7", (0, 1)), (".:5", (255, 255)),
            ("1|1:0,9:9:27:255,27,0", (1, 1)), ("007/1", (7, 1)),
            ("255/0", None), ("0", None), ("0/1/2", None), ("", None), ("a/b", None), ("-1/0", None), ("0//1", None),
            ("0/", None), ("/1", None), ("1000/0", None), (":", None), ("0 /1", None), ("0\\1", None)]


@pytest.mark.parametrize("gt,want", GT_TABLE)
def test_parse_gt_device_grammar_equals_reader(gt, want):
    assert vcf.parse_gt(gt) == want
    assert emu_parse_gt(gt) == want
    assert emu_parse_gt(gt + "\t0/0") == want                    # a tab ends the column


def _write_lines(path, lines):
    with open(path, "w") as f:
        f.write("".join(l + "\n" for l in lines))
    return path


HEAD = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT"


@pytest.mark.parametrize("lines,msg", [
    (["##fileformat=VCFv4.2", "1\t10\tr1\tA\tG\t.\t.\t.\tGT\t0/1"], "no #CHROM header"),
    ([HEAD[:-7]], "no FORMAT column"),
    ([HEAD], "names no samples"),
    ([HEAD + "\ta\tb\ta"], "duplicate sample ID"),
    ([HEAD + "\ta", "1\t10\tr1\tA\tG\t.\t.\t.", "1\t11\tr2\tA\tG\t.\t.\t.\tGT\t0/1"], "line 2 (1:10): fewer than 9"),
    ([HEAD + "\ta", "1\t10\tr1\tA\tG\t.\t.\t.\tGT\t0/1", "2\t1e5\tr2\tA\tG\t.\t.\t.\tGT\t0/1"], "line 3 (2:1e5): POS is not"),
    ([HEAD + "\ta", "1\t10\tr1\tA\tG\t.\t.\t.\tDP:GT\t5:0/1"], "(1:10): FORMAT does not start with GT"),
    ([HEAD + "\ta", "1\t10\tr1\tA\tG\t.\t.\t.\tGTX\t0/1"], "FORMAT does not start with GT"),
    ([HEAD + "\ta"], "has no records"),
])
def test_load_vcf_rejects(tmp_path, lines, msg):
    path = _write_lines(str(tmp_path / "x.vcf"), lines)
    res = emu_load_vcf(path, str(tmp_path / "log"))
    assert isinstance(res, str) and msg in res, res
    assert str(path) in res
    if msg != "has no records":
        with pytest.raises(vcf.VcfError):
            vcf.read_vcf(path)


def _first_block_end(z):
    return int.from_bytes(z[16:18], "little") + 1


@pytest.mark.parametrize("damage,msg", [
    (lambda z: z[:_first_block_end(z) - 8] + bytes([z[_first_block_end(z) - 8] ^ 1]) + z[_first_block_end(z) - 7:],
     "CRC32 mismatch"),
    (lambda z: z[:-40], "truncated BGZF block"),
    (lambda z: z[:_first_block_end(z) + 7], "truncated BGZF block header"),
    (lambda z: z[:_first_block_end(z) - 4] + (5000).to_bytes(4, "little") + z[_first_block_end(z):], "ISIZE"),
])
def test_bgzf_damage_is_an_error(tmp_path, damage, msg):
    v = random_vcf(2, 9, 40)
    path = str(tmp_path / "x.vcf.gz")
    vcf.write_vcf(path, v, compress="bgzf", block_size=300)
    z = open(path, "rb").read()
    open(path, "wb").write(damage(z))
    res = emu_load_vcf(path, str(tmp_path / "log"))
    assert isinstance(res, str) and msg in res, res


def test_plain_gzip_and_bgzf_load_alike(tmp_path):
    v = random_vcf(4, 21, 300)
    outs = []
    for compress in (None, "gz", "bgzf"):
        p = vcf.write_vcf(str(tmp_path / ("x%s.vcf" % compress)), v, "GT:AD:DP:GQ:PL", "|", True, compress, 1 << 12)
        outs.append(emu_load_vcf(p, str(tmp_path / "log")))
    assert outs[0] == outs[1] == outs[2]


# ------------------------------------------------------------------------------------------------ GPU
def _shape(g, N, L0, ind_offset=0):
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 1000
    g.set_shape(N, L0, np.array([0, L0 // 2, L0], np.int64), pos, ind_offset=ind_offset)


def _put(g, text, off, block=1024):
    diag = []
    for s0 in range(0, len(off) - 1, block):
        diag.append(g.put_vcf_text(text, off[s0:s0 + block + 1], s0))
    return [np.concatenate(d) for d in zip(*diag)]


@pytest.mark.gpu
@pytest.mark.parametrize("N,L0", [(1, 3001), (3, 2333), (29, 5000 + 17), (77, 4100), (513, 3075)])
def test_vcf_coding_equals_tped_coding(tmp_path, N, L0):
    from garlic_b200.api import GarlicGPU
    from oracle import oracle as orc
    v = random_vcf(N + 11, N, L0)
    geno, na, tot, one, freq = orc.code_tped(vcf.tped_alleles(v.idx, v.ref, v.alts))
    names = [[r] + a for r, a in zip(v.ref, v.alts)]
    w = vcf.Vcf(**{**v.__dict__, "alts": [list(a) for a in v.alts]})
    for s in range(0, L0, 7):                                      # long ALT names do not change the coding
        w.alts[s] = [x + "<INS:ME>" if k % 2 else x for k, x in enumerate(w.alts[s])]
    compress, fmt, sep, lone = WRITE_CASES[N % len(WRITE_CASES)]
    path = vcf.write_vcf(str(tmp_path / "x.vcf"), w, fmt, sep, lone, compress, block_size=5000)
    text, off = vcf.sample_text(path)
    g = GarlicGPU(0)
    _shape(g, N, L0)
    nc, mx, bad = _put(g, text, off)                               # ragged last block
    assert (nc == N).all() and (bad == -1).all()
    present = np.where(v.idx == vcf.MISSING, -1, v.idx.astype(np.int64)).reshape(L0, -1).max(1)
    assert np.array_equal(mx, present)
    g.code_alleles()
    c_na, c_tot, c_hom, c_nm = g.get_counts()
    assert np.array_equal(c_na, na) and np.array_equal(c_tot, tot)
    k = g.get_one_allele(255)
    assert np.array_equal(k, vcf.one_allele(v.idx))
    assert np.array_equal(np.array([ord(names[s][k[s]]) if k[s] != 255 else ord("0") for s in range(L0)], np.uint8), one)
    want = geno.astype(np.uint8)
    assert np.array_equal(c_nm, (want != 3).sum(1))
    assert np.array_equal(c_hom, ((want == 0) | (want == 2)).sum(1))
    assert np.array_equal(synth.unpack_codes(g.get_genotypes(False), L0), want.T)
    f, keep, L = g.filter()
    assert np.array_equal(f, freq)
    assert np.array_equal(keep, (freq > 0) & (freq < 1))
    assert np.array_equal(synth.unpack_codes(g.get_genotypes(True), L), want[keep].T)
    g.close()


DIAG_RECORDS = [("0/1\t1/0\t0|0\t./.", 4, 1, -1),
                ("0/1\t1/0\t0|0", 3, 1, -1),                       # one column short
                ("0/1\t1/0\t0|0\t./.\t2/2", 5, 2, -1),              # one extra
                ("0\t0/1\t0/1\t0/1", 4, 1, 0),                      # haploid
                ("0/1\t0/1/1\t0/1\t0/1", 4, 1, 1),                  # triploid
                ("0/1\t0/1\tx/y\t0/1:3", 4, 1, 2),                  # junk
                ("0/1\t0/1\t0/1\t255/0", 4, 1, 3),                  # index 255
                ("0/1\t0/1:3,4\t12/3:5:6\t.", 4, 12, -1),           # index above a small ALT count: reported, not refused
                ("./.\t.\t.:1\t.|.", 4, -1, -1),
                ("", 0, -1, -1),
                ("\t0/1\t0/1\t0/1", 4, 1, 0),                       # empty first column
                ("1/1\t0/1\t1/0\t", 4, 1, 3)]                       # empty last column


@pytest.mark.gpu
@pytest.mark.parametrize("lo,n", [(0, 4), (1, 2), (3, 1)])
def test_vcf_diagnostics(lo, n):
    from garlic_b200.api import GarlicGPU
    recs = [r[0].encode() for r in DIAG_RECORDS] * 3                # spans several CTAs' grid-stride loop
    long_rec = "\t".join(["1/0"] * 4) + "\t" + "\t".join(["0/0"] * 3000)     # more than one 4,096-character tile
    recs.append(long_rec.encode())
    off = np.concatenate([[0], np.cumsum([len(r) for r in recs])]).astype(np.int64)
    g = GarlicGPU(0)
    _shape(g, n, len(recs), ind_offset=lo)
    nc, mx, bad = g.put_vcf_text(b"".join(recs), off, 0)
    want = DIAG_RECORDS * 3
    assert list(nc[:-1]) == [r[1] for r in want] and nc[-1] == 3004
    assert list(mx[:-1]) == [r[2] for r in want] and mx[-1] == 1
    assert list(bad[:-1]) == [r[3] for r in want] and bad[-1] == -1
    g.close()


class _DevArray:
    """A device buffer of the library as a torch tensor (no copy)."""
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


@pytest.mark.gpu
@pytest.mark.parametrize("N,cuts", [(77, [1, 30]), (29, [3, 4]), (513, [130, 259])])
def test_sharded_handles_equal_one_handle(tmp_path, N, cuts):
    import torch
    from garlic_b200.api import GarlicGPU
    L0 = 4100
    v = random_vcf(N, N, L0)
    text, off = vcf.sample_text(vcf.write_vcf(str(tmp_path / "x.vcf"), v, "GT", "|", True))
    whole = GarlicGPU(0)
    _shape(whole, N, L0)
    want_diag = _put(whole, text, off)
    whole.code_alleles()
    want_rows = synth.unpack_codes(whole.get_genotypes(False), L0)
    want_counts = whole.get_counts()
    bounds = [0] + cuts + [N]
    hs = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        g = GarlicGPU(0)
        _shape(g, hi - lo, L0, ind_offset=lo)
        diag = _put(g, text, off)                                   # every handle parses every column
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
def test_handle_input_kinds_do_not_mix(tmp_path):
    from garlic_b200.api import GarlicError, GarlicGPU
    v = random_vcf(5, 8, 64)
    text, off = vcf.sample_text(vcf.write_vcf(str(tmp_path / "x.vcf"), v))
    g = GarlicGPU(0)
    _shape(g, 8, 64)
    g.put_alleles(vcf.tped_alleles(v.idx, v.ref, v.alts))
    with pytest.raises(GarlicError, match="tped input"):
        g.put_vcf_text(text, off, 0)
    _shape(g, 8, 64)
    g.put_vcf_text(text, off, 0)
    with pytest.raises(GarlicError, match="VCF input"):
        g.put_alleles(vcf.tped_alleles(v.idx, v.ref, v.alts))
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lod_0", "lod_small", "wlod_cm"])
def test_roh_from_vcf_equal_oracle(tmp_path, name):
    from garlic_b200.pipeline import HotPath
    from oracle import oracle as orc
    ds, args = load_case(name)
    W = arg(args, "--winsize", cast=int)
    err = arg(args, "--error", None, float)
    cutoff = arg(args, "--lod-cutoff", None, float)
    ov = arg(args, "--overlap-frac", 0.25, float)
    weighted, cm = "--weighted" in args, "--cm" in args
    res = orc.run_pipeline(ds, W, err, cutoff, ov, weighted=weighted, cm=cm)
    path = vcf.write_vcf(str(tmp_path / "x.vcf.gz"), vcf.from_dataset(ds, seed=5), "GT:AD:DP:GQ:PL", "/", True, "bgzf")
    hp = HotPath().load(ds, weighted=weighted, cm=cm, error=err, vcf=vcf.sample_text(path))
    assert hp.L == res["n_used"]
    if weighted:
        hp.g.ld_band(W)
    got = hp.roh(W, cutoff, res["overlap_frac"], weighted=weighted, cm=cm)
    assert got and [(r[0], r[1], r[5], r[6]) for r in got] == oracle_roh_idx(res)
    hp.close()


# ------------------------------------------------------------------------------------------------ CLI (GPU)
BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")


def _cli_inputs(name, tmp, compress=None, fmt="GT", sep="/", lone=False, n_ind=None, rename=None):
    """Writes a golden case twice — as tped/tfam (syn.*) and as a VCF — and returns (tped argv, vcf argv with --tfam,
    vcf argv without, the VCF) without the output prefix.  rename = (snp, name): that SNP's "1" allele gets a longer
    name in the VCF (the tped keeps the one-character name)."""
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
    path = os.path.join(tmp, "in.vcf" + (".gz" if compress else ""))
    vcf.write_vcf(path, v, fmt, sep, lone, compress, block_size=4000)
    with open(os.path.join(GOLDEN, name, "cmd.txt")) as f:
        cmd = [a.replace("<tmp>", tmp) for a in f.readline().split()[1:] if a != "--raw-lod"]
    i = cmd.index("--out")
    del cmd[i:i + 2]
    i = cmd.index("--tped")
    assert cmd[i + 2] == "--tfam"
    base = cmd[:i] + cmd[i + 4:]
    return cmd, base + ["--vcf", path, "--tfam", cmd[i + 3]], base + ["--vcf", path], v


def _run(argv, out):
    return subprocess.run([BIN] + argv + ["--out", out], capture_output=True, text=True, timeout=300)


def _same_outputs(tmp, a, b, freq_sub=None):
    assert os.path.exists(a + ".roh.bed") == os.path.exists(b + ".roh.bed")       # (--freq-only writes none)
    if os.path.exists(a + ".roh.bed"):
        assert open(a + ".roh.bed").read() == open(b + ".roh.bed").read()
    if os.path.exists(a + ".freq.gz"):
        fa = gzip.open(a + ".freq.gz", "rt").read()
        if freq_sub:
            rows = fa.splitlines(True)
            s, new = freq_sub
            t = rows[s + 1].split("\t")
            rows[s + 1] = "\t".join(t[:3] + [new] + t[4:])
            fa = "".join(rows)
        assert fa == gzip.open(b + ".freq.gz", "rt").read()
    else:
        assert not os.path.exists(b + ".freq.gz")
    ka = sorted(f for f in os.listdir(tmp) if f.startswith(os.path.basename(a) + ".") and f.endswith(".kde"))
    kb = sorted(f for f in os.listdir(tmp) if f.startswith(os.path.basename(b) + ".") and f.endswith(".kde"))
    assert [f.split(".", 1)[1] for f in ka] == [f.split(".", 1)[1] for f in kb]
    for x, y in zip(ka, kb):
        assert open(os.path.join(tmp, x)).read() == open(os.path.join(tmp, y)).read()

    def log(p):
        return [l for l in open(p + ".log").read().splitlines()[1:] if tmp not in l and not l.startswith("TPED missing")]
    assert log(a) == log(b)


@pytest.mark.gpu
@pytest.mark.parametrize("name,extra,compress,fmt,sep,lone", [
    ("lod_0", [], None, "GT", "/", False),
    ("lod_small", [], "gz", "GT:AD:DP:GQ:PL", "/", True),
    ("wlod_cm", [], "bgzf", "GT", "/", True),
    ("wlod_phased", [], "bgzf", "GT:AD:DP:GQ:PL", "|", False),       # --phased (in the case's command) with '|' GTs
    ("gl_pl", [], None, "GT:AD:DP:GQ:PL", "/", True),                # --tgls rows follow the VCF records
    ("lod_1", ["--freq-only"], "gz", "GT", "|", False),
    ("lod_3", ["--resample", "50", "--seed", "7"], "bgzf", "GT", "/", False),
    ("auto_cutoff", ["--kde-direct", "--seed", "5"], None, "GT", "|", True),
    ("freq_file", [], "bgzf", "GT:AD:DP:GQ:PL", "/", True),
])
def test_cli_vcf_equals_tped(tmp_path, name, extra, compress, fmt, sep, lone):
    tmp = str(tmp_path)
    tped, with_tfam, _, _ = _cli_inputs(name, tmp, compress, fmt, sep, lone)
    r1 = _run(tped + extra, os.path.join(tmp, "t"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(with_tfam + extra, os.path.join(tmp, "v"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _same_outputs(tmp, os.path.join(tmp, "t"), os.path.join(tmp, "v"))
    log = open(os.path.join(tmp, "v.log")).read()
    assert "VCF file: " + with_tfam[with_tfam.index("--vcf") + 1] in log and "TPED file" not in log


@pytest.mark.gpu
@pytest.mark.parametrize("name,extra", [("freq_file", []), ("lod_2", ["--freq-only"])])
def test_cli_vcf_long_allele_names(tmp_path, name, extra):
    """A REF / ALT name longer than one character: .freq.gz prints it and --freq-file compares whole tokens."""
    tmp = str(tmp_path)
    s = 40
    tped, with_tfam, _, v = _cli_inputs(name, tmp, "bgzf", rename=(s, "<DEL:ME>"))
    k = vcf.one_allele(v.idx)[s]
    assert k != 255
    if "--freq-file" in with_tfam:
        rows = open(os.path.join(tmp, "syn.freq")).read().splitlines(True)
        t = rows[s + 1].split()
        old = chr(load_case(name)[0].alleles[s][v.idx[s] == k][0])
        t[3] = "<DEL:ME>" if t[3] == old else t[3]
        rows[s + 1] = "\t".join(t) + "\n"
        open(os.path.join(tmp, "vcf.freq"), "w").write("".join(rows))
        with_tfam[with_tfam.index("--freq-file") + 1] = os.path.join(tmp, "vcf.freq")
    r1 = _run(tped + extra, os.path.join(tmp, "t"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(with_tfam + extra, os.path.join(tmp, "v"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _same_outputs(tmp, os.path.join(tmp, "t"), os.path.join(tmp, "v"), freq_sub=(s, "<DEL:ME>"))


@pytest.mark.gpu
def test_cli_vcf_population(tmp_path):
    tmp = str(tmp_path)
    tped, with_tfam, without, _ = _cli_inputs("lod_small", tmp, "gz")
    r = _run(without, os.path.join(tmp, "v"))
    assert r.returncode == 0, r.stderr[-2000:]
    bed = open(os.path.join(tmp, "v.roh.bed")).read()
    assert "Pop:VCF ROH" in bed and "Population: VCF" in open(os.path.join(tmp, "v.log")).read()
    r1 = _run(tped, os.path.join(tmp, "t"))
    assert r1.returncode == 0
    pop = load_case("lod_small")[0].pop
    assert open(os.path.join(tmp, "t.roh.bed")).read().replace("Pop:%s " % pop, "Pop:VCF ") == bed
    tfam = with_tfam[with_tfam.index("--tfam") + 1]
    rows = open(tfam).read().splitlines(True)
    t = rows[3].split()
    rows[3] = " ".join([t[0], "other"] + t[2:]) + "\n"
    open(os.path.join(tmp, "bad.tfam"), "w").write("".join(rows))
    with_tfam[with_tfam.index("--tfam") + 1] = os.path.join(tmp, "bad.tfam")
    r = _run(with_tfam, os.path.join(tmp, "b"))
    assert r.returncode != 0
    assert "differ at individual 4" in open(os.path.join(tmp, "b.error")).read()


def _edit_record(path, s, fn):
    lines = open(path).read().splitlines(True)
    first = next(i for i, l in enumerate(lines) if not l.startswith("#"))
    cols = lines[first + s].rstrip("\n").split("\t")
    lines[first + s] = "\t".join(fn(cols)) + "\n"
    open(path, "w").write("".join(lines))


@pytest.mark.gpu
@pytest.mark.parametrize("edit,extra,msg", [
    (lambda c: c[:-1], [], "sample columns, but the #CHROM header names"),
    (lambda c: c[:9] + ["1"] + c[10:], [], "Haploid calls"),
    (lambda c: c[:4] + ["."] + c[5:9] + ["1/0"] + c[10:], [], "allele index 1 but only 0 ALT"),
    (lambda c: c[:8] + ["DP:GT"] + c[9:], [], "FORMAT does not start with GT"),
    (None, ["--host-tokenize"], "--host-tokenize"),
    (None, ["--tped", "x.tped"], "exactly one input"),
    (None, ["--bfile", "x"], "exactly one input"),
])
def test_cli_vcf_errors(tmp_path, edit, extra, msg):
    tmp = str(tmp_path)
    _, with_tfam, _, _ = _cli_inputs("lod_0", tmp)
    path = with_tfam[with_tfam.index("--vcf") + 1]
    if edit is not None:
        _edit_record(path, 100, edit)
    r = _run(with_tfam + extra, os.path.join(tmp, "v"))
    assert r.returncode != 0
    err = open(os.path.join(tmp, "v.error")).read()
    assert msg in err, err
    if edit is not None:
        assert "line 104 (" in err                                  # two meta lines and the header before record 0


@pytest.mark.gpu
def test_cli_vcf_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tmp = str(tmp_path)
    _, with_tfam, _, _ = _cli_inputs("lod_small", tmp, "bgzf", n_ind=29)
    r1 = _run(with_tfam, os.path.join(tmp, "a"))
    r2 = _run(with_tfam + ["--gpus", "2"], os.path.join(tmp, "b"))
    assert r1.returncode == 0 and r2.returncode == 0, r1.stderr[-1000:] + r2.stderr[-1000:]
    _same_outputs(tmp, os.path.join(tmp, "a"), os.path.join(tmp, "b"))
