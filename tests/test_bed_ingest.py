"""PLINK .bed/.bim/.fam input: the numpy reader / writer and the fileset → tped convention on the CPU; on the GPU, put_bed +
code_alleles against the tped coding path (orc.code_tped of the equivalent alleles), sharded handles, and ROH against
the oracle."""
import os

import numpy as np
import pytest

from garlic_b200 import plink, synth
from tests.common import arg, load_case, oracle_roh_idx


def random_fileset_codes(seed, N, L0, miss=0.08):
    """PLINK values uint8[L0, N] with the first-call cases pinned at the start: SNP 0 all missing, SNPs 1-3 first call
    hom A1 / het / hom A2 after leading missing calls, SNPs 4-6 the same without them."""
    rng = np.random.default_rng(seed)
    p = rng.uniform(0.05, 0.95, L0)
    g = (rng.random((L0, N)) < p[:, None]).astype(np.int64) + (rng.random((L0, N)) < p[:, None])
    codes = np.choose(g, [plink.HOM_A1, plink.HET, plink.HOM_A2]).astype(np.uint8)
    codes[rng.random((L0, N)) < miss] = plink.MISSING
    mono = rng.random(L0) < 0.03
    codes[mono] = np.where(codes[mono] == plink.MISSING, plink.MISSING, plink.HOM_A2)
    codes[0] = plink.MISSING
    lead = N // 2
    for k, first in enumerate([plink.HOM_A1, plink.HET, plink.HOM_A2]):
        codes[1 + k, :lead] = plink.MISSING
        codes[1 + k, lead] = first
        codes[4 + k, 0] = first
    return codes


def random_names(seed, L0):
    rng = np.random.default_rng(seed + 1)
    i1 = rng.integers(0, 4, L0)
    i2 = (i1 + rng.integers(1, 4, L0)) % 4
    return [chr(b"ACGT"[i]) for i in i1], [chr(b"ACGT"[i]) for i in i2]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("N", [1, 3, 4, 6, 29])
def test_fileset_round_trip_ignores_padding(tmp_path, N):
    L0 = 37
    codes = random_fileset_codes(N, N, L0)
    a1, a2 = random_names(N, L0)
    bim = plink.Bim(chr=["1"] * 20 + ["2"] * 17, ids=["s%d" % i for i in range(L0)], cm=["0"] * L0,
                    bp=np.arange(1, L0 + 1, dtype=np.int32) * 100, a1=a1, a2=a2)
    fam = [("POP", "i%d" % i) for i in range(N)]
    for pad in (0, 1, 3):                                           # padding fields of the last byte hold anything
        plink.write_fileset(str(tmp_path / "x"), codes, bim, fam, pad=pad)
        fs = plink.read_fileset(str(tmp_path / "x"))
        assert np.array_equal(fs.codes(), codes)
        assert fs.fam == fam and fs.bim.a1 == a1 and fs.bim.a2 == a2 and fs.bim.chr == bim.chr
        assert np.array_equal(fs.bim.bp, bim.bp)
        assert os.path.getsize(str(tmp_path / "x.bed")) == 3 + L0 * ((N + 3) // 4)
    if N % 4:
        assert (plink.rows_from_codes(codes, 3)[:, -1] >> (2 * (N % 4))).min() > 0


def _write_small(tmp_path, N=5, L0=8):
    codes = random_fileset_codes(0, N, L0)
    bim = plink.Bim(chr=["1"] * L0, ids=["s%d" % i for i in range(L0)], cm=["0"] * L0,
                    bp=np.arange(1, L0 + 1, dtype=np.int32), a1=["A"] * L0, a2=["G"] * L0)
    return plink.write_fileset(str(tmp_path / "x"), codes, bim, [("P", "i%d" % i) for i in range(N)])


@pytest.mark.parametrize("damage,msg", [
    (lambda b: b"\x6c\x1c" + b[2:], "6c 1b"),
    (lambda b: b[:2] + b"\x00" + b[3:], "individual-major"),
    (lambda b: b[:2] + b"\x02" + b[3:], "mode byte"),
    (lambda b: b + b"\x00", "bytes"),
    (lambda b: b[:-1], "bytes"),
])
def test_malformed_bed_raises(tmp_path, damage, msg):
    prefix = _write_small(tmp_path)
    with open(prefix + ".bed", "rb") as f:
        b = f.read()
    with open(prefix + ".bed", "wb") as f:
        f.write(damage(b))
    with pytest.raises(plink.PlinkError, match=msg):
        plink.read_fileset(prefix)


@pytest.mark.parametrize("which", ["bim", "fam"])
def test_row_count_mismatch_raises(tmp_path, which):
    prefix = _write_small(tmp_path)
    with open(prefix + "." + which) as f:
        lines = f.readlines()
    with open(prefix + "." + which, "w") as f:
        f.writelines(lines[:-1])
    with pytest.raises(plink.PlinkError, match="bytes"):
        plink.read_fileset(prefix)


def test_bed_to_tped_convention(tmp_path):
    M, A1, HET, A2 = plink.MISSING, plink.HOM_A1, plink.HET, plink.HOM_A2
    codes = np.array([[M, M, M],          # no call: no "1" allele
                      [A1, A2, HET],      # first call hom A1 → A1
                      [HET, A2, A2],      # het → A1
                      [A2, A1, HET],      # hom A2 → A2
                      [M, A1, A2],        # missing, then hom A1 → A1
                      [M, HET, A1],       # missing, then het → A1
                      [M, M, A2]],        # missing, then hom A2 → A2
                     np.uint8)
    a1, a2 = ["A", "C", "GT", "T", "A", "C", "G"], ["G", "T", "G", "C", "C", "A", "T"]
    assert list(plink.one_allele(codes)) == [0, 1, 1, 2, 1, 1, 2]
    toks = plink.tped_tokens(codes, a1, a2)
    assert toks[0] == ["0"] * 6
    assert toks[1] == ["C", "C", "T", "T", "C", "T"]
    assert toks[2] == ["GT", "G", "G", "G", "G", "G"]                  # het: A1 first, names longer than one character
    bim = plink.Bim(chr=["1"] * 7, ids=["s%d" % i for i in range(7)], cm=["0"] * 7, bp=np.arange(1, 8, dtype=np.int32),
                    a1=a1, a2=a2)
    plink.write_fileset(str(tmp_path / "x"), codes, bim, [("P", "a"), ("P", "b"), ("P", "c")], pad=2)
    tped, tfam = plink.write_tped(str(tmp_path / "t"), plink.read_fileset(str(tmp_path / "x")))
    with open(tped) as f:
        lines = f.read().splitlines()
    assert lines[3] == "1 s3 0 4 C C T T T C"
    with open(tfam) as f:
        assert f.read().splitlines()[1] == "P b 0 0 0 0"
    # the tped reader's first non-missing character is the "1" allele named above
    single = [0, 1, 3, 4, 5, 6]
    al = plink.tped_alleles(codes[single], [a1[i] for i in single], [a2[i] for i in single])
    flat = al.reshape(len(single), -1)
    first = [next((chr(c) for c in row if c != ord("0")), None) for row in flat]
    names = {1: a1, 2: a2}
    assert first == [None if plink.one_allele(codes)[i] == 0 else names[plink.one_allele(codes)[i]][i] for i in single]


def test_bed_dataset_is_representable_and_names_a2_sometimes():
    ds, _ = load_case("lod_0")
    dsb, codes, a1, a2 = plink.bed_dataset(ds, seed=3)
    assert np.array_equal(dsb.alleles, plink.tped_alleles(codes, a1, a2))
    half = (ds.alleles == ord("0")).sum(2) == 1
    assert half.any() and (codes[half] == plink.MISSING).all()
    one = plink.one_allele(codes)
    assert (one == 1).any() and (one == 2).any() and (one == 0).any()
    # calls both datasets have in full keep their letters (heterozygotes up to order)
    full = (ds.alleles != ord("0")).all(2)
    assert np.array_equal(np.sort(ds.alleles[full], 1), np.sort(dsb.alleles[full], 1))


# ------------------------------------------------------------------------------------------------ GPU
def _shape(g, N, L0, ind_offset=0):
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 1000
    g.set_shape(N, L0, np.array([0, L0 // 2, L0], np.int64), pos, ind_offset=ind_offset)


def _put(g, rows, block=1024):
    for s0 in range(0, rows.shape[0], block):
        g.put_bed(rows[s0:s0 + block], s0)


@pytest.mark.gpu
@pytest.mark.parametrize("N,L0", [(1, 3001), (3, 2333), (29, 5000 + 17), (77, 4100), (513, 3075)])
def test_bed_coding_equals_tped_coding(N, L0):
    from garlic_b200.api import GarlicGPU
    from oracle import oracle as orc
    codes = random_fileset_codes(N + 11, N, L0)
    a1, a2 = random_names(N, L0)
    geno, na, tot, one, freq = orc.code_tped(plink.tped_alleles(codes, a1, a2))
    g = GarlicGPU(0)
    _shape(g, N, L0)
    _put(g, plink.rows_from_codes(codes, pad=1))                   # ragged last block, non-zero padding
    g.code_alleles()
    c_na, c_tot, c_hom, c_nm = g.get_counts()
    assert np.array_equal(c_na, na) and np.array_equal(c_tot, tot)
    k = g.get_one_allele()
    c1, c2 = np.frombuffer("".join(a1).encode(), np.uint8), np.frombuffer("".join(a2).encode(), np.uint8)
    assert set(np.unique(k)) <= {1, 2, ord("0")}
    assert np.array_equal(np.where(k == 1, c1, np.where(k == 2, c2, k)), one)
    want = geno.astype(np.uint8)
    assert np.array_equal(c_nm, (want != 3).sum(1))
    assert np.array_equal(c_hom, ((want == 0) | (want == 2)).sum(1))
    assert np.array_equal(synth.unpack_codes(g.get_genotypes(False), L0), want.T)
    f, keep, L = g.filter()
    assert np.array_equal(f, freq)
    assert np.array_equal(keep, (freq > 0) & (freq < 1))
    assert np.array_equal(synth.unpack_codes(g.get_genotypes(True), L), want[keep].T)
    g.close()


class _DevArray:
    """A device buffer of the library as a torch tensor (no copy)."""
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


@pytest.mark.gpu
@pytest.mark.parametrize("N,cuts", [(77, [1, 30]), (29, [3, 4]), (513, [130, 259])])
def test_sharded_handles_equal_one_handle(N, cuts):
    import torch
    from garlic_b200.api import GarlicGPU
    L0 = 4100
    codes = random_fileset_codes(N, N, L0)
    rows = plink.rows_from_codes(codes, pad=2)
    whole = GarlicGPU(0)
    _shape(whole, N, L0)
    _put(whole, rows)
    whole.code_alleles()
    want_rows = synth.unpack_codes(whole.get_genotypes(False), L0)
    want_counts = whole.get_counts()
    bounds = [0] + cuts + [N]
    hs = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        g = GarlicGPU(0)
        _shape(g, hi - lo, L0, ind_offset=lo)
        _put(g, rows)                                               # every handle gets whole rows, keeps its columns
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
    assert all(np.array_equal(g.get_one_allele(), whole.get_one_allele()) for g in hs)
    for g in hs + [whole]:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lod_0", "lod_small", "wlod_cm"])
def test_roh_from_bed_equal_oracle(name):
    from garlic_b200.pipeline import HotPath
    from oracle import oracle as orc
    ds, args = load_case(name)
    dsb, codes, a1, a2 = plink.bed_dataset(ds, seed=5)
    W = arg(args, "--winsize", cast=int)
    err = arg(args, "--error", None, float)
    cutoff = arg(args, "--lod-cutoff", None, float)
    ov = arg(args, "--overlap-frac", 0.25, float)
    weighted, cm = "--weighted" in args, "--cm" in args
    res = orc.run_pipeline(dsb, W, err, cutoff, ov, weighted=weighted, cm=cm)
    hp = HotPath().load(dsb, weighted=weighted, cm=cm, error=err, bed=plink.rows_from_codes(codes, pad=3))
    assert hp.L == res["n_used"]
    if weighted:
        hp.g.ld_band(W)
    got = hp.roh(W, cutoff, res["overlap_frac"], weighted=weighted, cm=cm)
    assert got and [(r[0], r[1], r[5], r[6]) for r in got] == oracle_roh_idx(res)
    if weighted:
        hp.g.set_phased(True)
        with pytest.raises(Exception, match="unphased"):
            hp.g.ld_band(W)
    hp.close()


# ------------------------------------------------------------------------------------------------ CLI (GPU)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")


def _cli_inputs(name, tmp, n_ind=None, rename=None):
    """Writes the bed-representable dataset of a golden case twice — as tped/tfam (syn.*) and as a fileset (bed.*) — and
    returns (tped argv, bfile argv) without the output prefix.  rename = (snp, name): that SNP's "1" allele gets a longer
    name in the fileset (the tped keeps the one-character name)."""
    from tests.common import GOLDEN
    ds, args = load_case(name)
    dsb, codes, a1, a2 = plink.bed_dataset(ds, seed=11)
    if n_ind is not None:
        dsb.alleles, dsb.ind_ids, codes = dsb.alleles[:, :n_ind], dsb.ind_ids[:n_ind], codes[:, :n_ind]
    dsb.write(tmp)
    one = plink.one_allele(codes)
    b1, b2 = list(a1), list(a2)
    if rename is not None:
        s, new = rename
        (b1 if one[s] == 1 else b2)[s] = new
    plink.write_fileset(os.path.join(tmp, "bed"), codes, plink.bim_of(dsb, b1, b2), [(dsb.pop, i) for i in dsb.ind_ids],
                        pad=3)
    with open(os.path.join(GOLDEN, name, "cmd.txt")) as f:
        cmd = [a.replace("<tmp>", tmp) for a in f.readline().split()[1:] if a != "--raw-lod"]
    i = cmd.index("--out")
    del cmd[i:i + 2]
    i = cmd.index("--tped")
    base = cmd[:i] + cmd[i + 4:]
    assert cmd[i + 2] == "--tfam"
    return cmd, base + ["--bfile", os.path.join(tmp, "bed")], one, a1, a2


def _run(argv, out):
    import subprocess
    return subprocess.run([BIN] + argv + ["--out", out], capture_output=True, text=True, timeout=300)


def _same_outputs(tmp, a, b, freq_sub=None):
    import gzip
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
@pytest.mark.parametrize("name,extra", [("lod_0", []), ("lod_small", []), ("wlod_cm", []), ("gl_pl", []),
                                        ("lod_1", ["--freq-only"]), ("lod_3", ["--resample", "50", "--seed", "7"]),
                                        ("auto_cutoff", ["--kde-direct", "--seed", "5"])])
def test_cli_bfile_equals_tped(tmp_path, name, extra):
    tmp = str(tmp_path)
    tped, bfile, *_ = _cli_inputs(name, tmp)
    r1 = _run(tped + extra, os.path.join(tmp, "t"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(bfile + extra, os.path.join(tmp, "b"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _same_outputs(tmp, os.path.join(tmp, "t"), os.path.join(tmp, "b"))
    log = open(os.path.join(tmp, "b.log")).read()
    assert "PLINK binary fileset: " + os.path.join(tmp, "bed") in log and "TPED file" not in log


@pytest.mark.gpu
@pytest.mark.parametrize("name,extra", [("freq_file", []), ("lod_2", ["--freq-only"])])
def test_cli_bfile_long_allele_names(tmp_path, name, extra):
    """A .bim allele name longer than one character: .freq.gz prints it and --freq-file compares whole tokens."""
    tmp = str(tmp_path)
    from tests.common import GOLDEN
    s = 40
    tped, bfile, one, a1, a2 = _cli_inputs(name, tmp, rename=(s, "ACGT"))
    assert one[s] in (1, 2)
    if os.path.exists(os.path.join(GOLDEN, name, "in.freq")):
        rows = open(os.path.join(GOLDEN, name, "in.freq")).read().splitlines(True)
        open(os.path.join(tmp, "syn.freq"), "w").write("".join(rows))
        t = rows[s + 1].split()
        old = (a1 if one[s] == 1 else a2)[s]
        t[3] = "ACGT" if t[3] == old else t[3]
        rows[s + 1] = "\t".join(t) + "\n"
        open(os.path.join(tmp, "bed.freq"), "w").write("".join(rows))
        i = bfile.index("--freq-file")
        bfile[i + 1] = os.path.join(tmp, "bed.freq")
    r1 = _run(tped + extra, os.path.join(tmp, "t"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(bfile + extra, os.path.join(tmp, "b"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _same_outputs(tmp, os.path.join(tmp, "t"), os.path.join(tmp, "b"), freq_sub=(s, "ACGT"))


@pytest.mark.gpu
def test_cli_bfile_two_gpus_equal_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tmp = str(tmp_path)
    _, bfile, *_ = _cli_inputs("lod_small", tmp, n_ind=29)
    r1 = _run(bfile, os.path.join(tmp, "a"))
    r2 = _run(bfile + ["--gpus", "2"], os.path.join(tmp, "b"))
    assert r1.returncode == 0 and r2.returncode == 0, r1.stderr[-1000:] + r2.stderr[-1000:]
    _same_outputs(tmp, os.path.join(tmp, "a"), os.path.join(tmp, "b"))


def _damage_magic(p):
    b = open(p + ".bed", "rb").read()
    open(p + ".bed", "wb").write(b"\x6c\x1c" + b[2:])


def _damage_mode(p):
    b = open(p + ".bed", "rb").read()
    open(p + ".bed", "wb").write(b[:2] + b"\x00" + b[3:])


def _damage_size(p):
    b = open(p + ".bed", "rb").read()
    open(p + ".bed", "wb").write(b[:-1])


def _damage_fam(p):
    rows = open(p + ".fam").read().splitlines(True)
    open(p + ".fam", "w").write("".join(rows[:-2]))


@pytest.mark.gpu
@pytest.mark.parametrize("damage,msg", [(None, "--phased"), (_damage_magic, "6c 1b"), (_damage_mode, "individual-major"),
                                        (_damage_size, "bytes"), (_damage_fam, "bytes")])
def test_cli_bfile_errors(tmp_path, damage, msg):
    tmp = str(tmp_path)
    _, bfile, *_ = _cli_inputs("lod_0", tmp)
    if damage is None:
        bfile = bfile + ["--phased"]
    else:
        damage(os.path.join(tmp, "bed"))
    r = _run(bfile, os.path.join(tmp, "b"))
    assert r.returncode != 0
    assert msg in open(os.path.join(tmp, "b.error")).read()
