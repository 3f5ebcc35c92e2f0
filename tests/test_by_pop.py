"""Column selection (garlic_gpu_select_columns): a handle that holds a listed subset of the input's individuals, such as
one population of a multi-population file.  On the CPU: the .bed gather rule (bed_select.cuh, through
tests/bed_select_emu.cpp) against a numpy gather, and the rejected column lists.  On the GPU: for every text, binary and
likelihood input, a handle with select_columns(cols) equals a handle given the input restricted to cols; a sample split
over two selecting handles equals one handle; pruned ROH of a selected handle equal the oracle on that sample."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from garlic_b200 import bcf, plink, synth, vcf
from tests.common import arg, load_case, oracle_roh_idx
from tests.test_bed_ingest import random_fileset_codes
from tests.test_vcf_ingest import random_vcf

HERE = os.path.dirname(os.path.abspath(__file__))
_EMU = None


def emu():
    """tests/bed_select_emu.cpp (bed_select.cuh:bed_gather_byte for the CPU), built into a temporary directory."""
    global _EMU
    if _EMU is None:
        so = os.path.join(tempfile.mkdtemp(prefix="garlic_bed_select_emu_"), "bed_select_emu.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, os.path.join(HERE, "bed_select_emu.cpp")])
        _EMU = C.CDLL(so)
    return _EMU


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def emu_bed_select(rows, cols):
    rows = np.ascontiguousarray(rows, np.uint8)
    cols = np.ascontiguousarray(cols, np.int32)
    out = np.zeros((rows.shape[0], (len(cols) + 3) // 4), np.uint8)
    emu().emu_bed_select(_p(rows), C.c_int64(rows.shape[1]), C.c_int(rows.shape[0]), _p(cols), C.c_int(len(cols)), _p(out))
    return out


def random_columns(rng, n_input):
    """A non-empty ascending subset of range(n_input)."""
    k = int(rng.integers(1, n_input + 1))
    return np.sort(rng.choice(n_input, k, replace=False)).astype(np.int32)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("N", [1, 3, 4, 5, 29, 77, 513])
def test_bed_gather_rule_equals_numpy(N):
    rng = np.random.default_rng(N)
    codes = rng.integers(0, 4, (37, N)).astype(np.uint8)
    rows = plink.rows_from_codes(codes, pad=3)                         # non-zero padding of a ragged last byte
    lists = [random_columns(rng, N) for _ in range(6)]
    lists += [np.arange(N), np.array([0]), np.array([N - 1]), np.array(sorted({0, N - 1}))]
    lists += [np.arange(s, N, 3) for s in range(min(4, N))]            # every bit offset of the first column
    for cols in lists:
        got = emu_bed_select(rows, cols)
        assert np.array_equal(got, plink.rows_from_codes(codes[:, cols], pad=0)), cols


def _unbound_handle(n_ind):
    """A GarlicGPU without a device: select_columns' own checks run before the library is called."""
    from garlic_b200 import api
    g = api.GarlicGPU.__new__(api.GarlicGPU)
    g.lib, g.h, g.n_ind = api.load_library(), C.c_void_p(), n_ind
    return g


@pytest.mark.parametrize("cols,n_input,msg", [
    ([0, 2, 1], 4, "ascending"),
    ([0, 2, 2], 4, "ascending"),
    ([0, 1, 4], 4, "outside"),
    ([-1, 1, 2], 4, "outside"),
    ([0, 1], 4, "2 columns for a handle of 3"),
    ([0, 1, 2, 3], 4, "4 columns for a handle of 3"),
])
def test_select_columns_rejects(cols, n_input, msg):
    from garlic_b200 import api
    if not os.path.exists(api.LIB_PATH):
        pytest.skip("libgarlic_b200.so is not built")
    with pytest.raises(api.GarlicError, match=msg):
        _unbound_handle(3).select_columns(cols, n_input)


# ------------------------------------------------------------------------------------------------ GPU
L0S = {1: 3001, 3: 2333, 29: 5017, 77: 4100, 513: 3075}
KINDS = ["tped", "vcf_gt", "vcf_full", "bcf_int8", "bcf_int16", "bcf_lone", "bed", "bed_dev", "tgls"]


def _tped_text(alleles):
    """Line tails of a tped (alleles uint8[L0, N, 2]) and their offsets."""
    lines = [b" ".join(bytes([c]) for c in row.reshape(-1)) for row in alleles]
    off = np.zeros(len(lines) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in lines])
    return b"".join(lines), off


def _tgls_tokens(rng, L0, N):
    tok = np.array([[str(x) for x in row] for row in rng.integers(0, 99, (L0, N))], dtype=object)
    hard = rng.random((L0, N)) < 0.01                                   # long mantissas: the host strtod path
    tok[hard] = "0.12345678901234567"
    tok[rng.random((L0, N)) < 0.01] = "1e-30"
    return tok


def _tgls_text(tok):
    lines = [" ".join(row).encode() for row in tok]
    off = np.zeros(len(lines) + 1, np.int64)
    off[1:] = np.cumsum([len(x) for x in lines])
    return b"".join(lines), off


class Input:
    """One input of N individuals of a kind, and how to load it (or its restriction to some columns) into a handle."""

    def __init__(self, kind, N, L0, tmp, seed):
        self.kind, self.N, self.L0, self.tmp = kind, N, L0, tmp
        rng = np.random.default_rng(seed)
        if kind == "tped":
            self.alleles = rng.choice(np.frombuffer(b"0ACGT", np.uint8), (L0, N, 2), p=[0.08, 0.46, 0.46, 0, 0])
            self.alleles[0] = ord("0")
        elif kind.startswith("vcf") or kind.startswith("bcf"):
            self.v = random_vcf(seed, N, L0)
            if kind == "bcf_int16":
                self.v.alts[6] = ["A%d" % k for k in range(1, 71)]
                self.v.idx[6, 0] = (70, 0)
        elif kind.startswith("bed"):
            self.codes = random_fileset_codes(seed, N, L0)
        else:
            self.tok = _tgls_tokens(rng, L0, N)

    def _sub(self, cols):
        """(payload of the input restricted to cols — all columns for None —, n_input)."""
        idx = np.arange(self.N) if cols is None else np.asarray(cols)
        name = "full" if cols is None else "sub"
        k = self.kind
        if k == "tped":
            return _tped_text(self.alleles[:, idx]), len(idx)
        if k.startswith("vcf") or k.startswith("bcf"):
            v = vcf.Vcf(**{**self.v.__dict__, "samples": [self.v.samples[i] for i in idx], "idx": self.v.idx[:, idx]})
            if k.startswith("vcf"):
                fmt, compress = ("GT", None) if k == "vcf_gt" else ("GT:AD:DP:GQ:PL", "bgzf")
                path = vcf.write_vcf(str(self.tmp / (name + ".vcf")), v, fmt, "/", k == "vcf_full", compress)
                return vcf.sample_text(path), len(idx)
            path = str(self.tmp / (name + ".bcf"))
            bcf.write_bcf(path, v, "GT", lone_missing=k == "bcf_lone", width=2 if k == "bcf_int16" else None)
            return bcf.gt_payload(path), len(idx)
        if k.startswith("bed"):
            return plink.rows_from_codes(self.codes[:, idx], pad=2), len(idx)
        return _tgls_text(self.tok[:, idx]), len(idx)

    def load(self, g, cols=None, select=True, ind_offset=0):
        """set_shape for len(cols) individuals, select_columns(cols) if select, then upload the whole input (select) or
        the input restricted to cols (not select)."""
        import torch
        n = self.N if cols is None else len(cols)
        pos = np.arange(1, self.L0 + 1, dtype=np.int32) * 1000
        g.set_shape(n, self.L0, np.array([0, self.L0 // 2, self.L0], np.int64), pos, ind_offset=ind_offset)
        if select and cols is not None:
            g.select_columns(cols, self.N)
        data, n_input = self._sub(None if select else cols)
        k, B = self.kind, 1024
        for s0 in range(0, self.L0, B):
            s1 = min(self.L0, s0 + B)
            if k == "tped":
                nb = g.put_tped_text(data[0], data[1][s0:s1 + 1], s0)
                assert (nb == 2 * n_input).all()
            elif k.startswith("vcf"):
                nc, _, bad = g.put_vcf_text(data[0], data[1][s0:s1 + 1], s0)
                assert (nc == n_input).all() and (bad == -1).all()
            elif k.startswith("bcf"):
                _, bad = g.put_bcf_gt(data[0], data[1][s0:s1 + 1], data[2][s0:s1], n_input, s0)
                assert (bad == -1).all()
            elif k == "bed":
                g.put_bed(data[s0:s1], s0)
            elif k == "bed_dev":
                if s0 == 0:
                    self._dev = torch.from_numpy(np.ascontiguousarray(data)).cuda()
                    torch.cuda.synchronize()
                g.put_bed_dev(self._dev.data_ptr() + s0 * data.shape[1], data.shape[1], s1 - s0, s0)
            else:
                ntok = g.put_tgls_text(data[0], data[1][s0:s1 + 1], "PL", snp0=s0)
                assert (ntok == n_input).all()
        g.sync()

    def missing(self):
        return ord("0") if self.kind == "tped" or self.kind.startswith("bed") else 255


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


def _keys(g, L0):
    import torch
    return torch.as_tensor(_DevArray(g.first_allele_keys_dev(), L0, "<i8"), device="cuda").cpu().numpy().view(np.uint64).copy()


def _state(inp, g):
    """What a handle holds after ingest: GL matrix (tgls), or keys, then after code_alleles the packed matrix, the
    counters and the "1" allele."""
    if inp.kind == "tgls":
        return [g.get_gl()]
    keys = _keys(g, inp.L0)
    g.code_alleles()
    return [keys, synth.unpack_codes(g.get_genotypes(False), inp.L0), np.array(g.get_counts()), g.get_one_allele(inp.missing())]


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N", sorted(L0S))
def test_selected_handle_equals_restricted_input(tmp_path, kind, N):
    from garlic_b200.api import GarlicGPU
    inp = Input(kind, N, L0S[N], tmp_path, seed=N + 7)
    rng = np.random.default_rng(N)
    lists = [random_columns(rng, N), np.arange(N)]
    if kind.startswith("bed"):
        lists += [np.arange(s, N, 3) for s in range(1, min(4, N))]      # first column at every bit offset
    for cols in lists:
        a, b = GarlicGPU(0), GarlicGPU(0)
        inp.load(a, cols, select=True)
        inp.load(b, cols, select=False)
        _same(_state(inp, a), _state(inp, b))
        a.close()
        b.close()
    # selecting every column is no selection
    a, b = GarlicGPU(0), GarlicGPU(0)
    inp.load(a, np.arange(N), select=True)
    inp.load(b, None)
    _same(_state(inp, a), _state(inp, b))
    a.close()
    b.close()


@pytest.mark.gpu
def test_select_columns_on_the_handle():
    from garlic_b200.api import GarlicError, GarlicGPU
    inp = Input("bed", 9, 100, None, seed=1)
    g = GarlicGPU(0)
    pos = np.arange(1, 101, dtype=np.int32)
    g.set_shape(3, 100, np.array([0, 100], np.int64), pos)
    for cols, n_input, msg in [([0, 2, 1], 9, "ascending"), ([0, 1, 9], 9, "outside"), ([-1, 1, 2], 9, "outside")]:
        with pytest.raises(GarlicError, match=msg):
            g.select_columns(cols, n_input)
    g.select_columns([1, 4, 8], 9)
    with pytest.raises(GarlicError, match="ceil"):
        g.put_bed(plink.rows_from_codes(inp.codes[:32, :8]), 0)           # stride of 8 individuals, not 9
    g.put_bed(plink.rows_from_codes(inp.codes[:32]), 0)
    with pytest.raises(GarlicError, match="before the first put"):
        g.select_columns([1, 4, 8], 9)
    g.set_shape(3, 100, np.array([0, 100], np.int64), pos)                # resets the selection: rows of 3 individuals
    g.put_bed(plink.rows_from_codes(inp.codes[:32, :3]), 0)
    v = random_vcf(3, 9, 64)
    path = tempfile.mkdtemp(prefix="garlic_sel_") + "/x.bcf"
    bcf.write_bcf(path, v)
    gt, off, types = bcf.gt_payload(path)
    g.set_shape(3, 64, np.array([0, 64], np.int64), pos[:64])
    g.select_columns([1, 4, 8], 9)
    with pytest.raises(GarlicError, match="n_samples"):
        g.put_bcf_gt(gt, off, types, 8, 0)
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["tped", "vcf_gt", "bcf_int8", "bed"])
def test_split_sample_equals_one_handle(tmp_path, kind):
    """A sample (columns cols of the input) split over two handles, with ind_offset and the MIN of the first-allele keys
    as the driver's ranks do them, equals one handle of the whole sample."""
    import torch
    from garlic_b200.api import GarlicGPU
    N, L0 = 77, 4100
    inp = Input(kind, N, L0, tmp_path, seed=5)
    cols = np.sort(np.random.default_rng(2).choice(N, 40, replace=False)).astype(np.int32)
    whole = GarlicGPU(0)
    inp.load(whole, cols)
    want = _state(inp, whole)
    hs = []
    for lo, hi in [(0, 13), (13, 40)]:
        g = GarlicGPU(0)
        inp.load(g, cols[lo:hi], ind_offset=lo)
        hs.append(g)
    keys = [torch.as_tensor(_DevArray(g.first_allele_keys_dev(), L0, "<i8"), device="cuda") for g in hs]
    mn = np.minimum.reduce([k.cpu().numpy().view(np.uint64) for k in keys])
    for k in keys:
        k.copy_(torch.from_numpy(mn.view(np.int64)))
    torch.cuda.synchronize()
    assert np.array_equal(mn, want[0])
    rows, counts = [], np.zeros((4, L0), np.int64)
    for g in hs:
        g.code_alleles()
        rows.append(synth.unpack_codes(g.get_genotypes(False), L0))
        counts += np.array(g.get_counts())
    assert np.array_equal(np.concatenate(rows), want[1])
    assert np.array_equal(counts, want[2])
    assert all(np.array_equal(g.get_one_allele(inp.missing()), want[3]) for g in hs)
    for g in hs + [whole]:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lod_0", "wlod_cm"])
def test_roh_of_selected_sample_equal_oracle(tmp_path, name):
    """The golden case's individuals interleaved with others in one VCF; the handle that selects them calls the ROH the
    oracle calls on the case alone."""
    from garlic_b200.pipeline import HotPath
    from oracle import oracle as orc
    ds, args = load_case(name)
    W = arg(args, "--winsize", cast=int)
    err = arg(args, "--error", None, float)
    cutoff = arg(args, "--lod-cutoff", None, float)
    ov = arg(args, "--overlap-frac", 0.25, float)
    weighted, cm = "--weighted" in args, "--cm" in args
    res = orc.run_pipeline(ds, W, err, cutoff, ov, weighted=weighted, cm=cm)
    v = vcf.from_dataset(ds, seed=5)
    N = len(v.samples)
    rng = np.random.default_rng(1)
    n_input = 2 * N + 3
    cols = np.sort(rng.choice(n_input, N, replace=False)).astype(np.int32)
    others = np.setdiff1d(np.arange(n_input), cols)
    idx = np.empty((v.idx.shape[0], n_input, 2), np.uint8)
    idx[:, cols] = v.idx
    idx[:, others] = v.idx[:, rng.integers(0, N, len(others))]
    samples = ["x%d" % i for i in range(n_input)]
    full = vcf.Vcf(**{**v.__dict__, "samples": samples, "idx": idx})
    path = vcf.write_vcf(str(tmp_path / "all.vcf.gz"), full, "GT", "/", False, "bgzf")
    hp = HotPath().load(ds, weighted=weighted, cm=cm, error=err, vcf=vcf.sample_text(path), columns=cols, n_input=n_input)
    assert hp.L == res["n_used"]
    if weighted:
        hp.g.ld_band(W)
    got = hp.roh(W, cutoff, res["overlap_frac"], weighted=weighted, cm=cm)
    assert got and [(r[0], r[1], r[5], r[6]) for r in got] == oracle_roh_idx(res)
    hp.close()


# ------------------------------------------------------------------------------------------------ driver --by-pop (GPU)
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")
GOLDEN = os.path.join(HERE, "golden")
POPS = ("AFR", "EUR", "EAS")


def _pop_of(N):
    """Three populations interleaved so that none is contiguous or byte-aligned in a .bed row."""
    return [POPS[(i + i // 4) % 3] for i in range(N)]


def _write_input(ds, tmp, kind):
    """ds as the input files of one run in directory tmp; → the argv that names them."""
    os.makedirs(tmp, exist_ok=True)
    paths = ds.write(tmp)
    if kind == "bfile":
        dsb, codes, a1, a2 = ds._bed
        plink.write_fileset(os.path.join(tmp, "syn"), codes, plink.bim_of(dsb, a1, a2),
                            [(p, i) for p, i in zip(ds._pops, ds.ind_ids)])
        return ["--bfile", os.path.join(tmp, "syn")]
    if kind in ("vcf", "bcf"):
        v = ds._vcf
        p = os.path.join(tmp, "in.vcf.gz" if kind == "vcf" else "in.bcf")
        vcf.write_vcf(p, v, compress="bgzf") if kind == "vcf" else bcf.write_bcf(p, v)
        return ["--vcf", p, "--tfam", paths["tfam"]]
    return ["--tped", paths["tped"], "--tfam", paths["tfam"]] + (["--host-tokenize"] if kind == "host" else [])


def _restrict(ds, cols, pops):
    import copy
    d = copy.copy(ds)
    d.alleles = ds.alleles[:, cols]
    d.ind_ids = [ds.ind_ids[i] for i in cols]
    d._pops = [pops[i] for i in cols]
    if getattr(ds, "gl", None) is not None:
        d.gl = ds.gl[:, cols]
    if hasattr(ds, "_vcf"):
        d._vcf = vcf.Vcf(**{**ds._vcf.__dict__, "samples": [ds._vcf.samples[i] for i in cols], "idx": ds._vcf.idx[:, cols]})
    if hasattr(ds, "_bed"):
        dsb, codes, a1, a2 = ds._bed
        d._bed = (dsb, codes[:, cols], a1, a2)
    return d


def _write_tfam(path, ids, pops):
    with open(path, "w") as f:
        for p, i in zip(pops, ids):
            f.write("%s %s 0 0 0 0\n" % (p, i))


def _case_argv(name, tmp, extra):
    with open(os.path.join(GOLDEN, name, "cmd.txt")) as f:
        cmd = [a.replace("<tmp>", tmp) for a in f.readline().split()[1:] if a != "--raw-lod"]
    i = cmd.index("--out")
    del cmd[i:i + 2]
    i = cmd.index("--tped")
    cmd = cmd[:i] + cmd[i + 4:]
    for k, flag in enumerate(extra):                                    # a flag of extra replaces the case's own
        if flag.startswith("--") and flag in cmd:
            j = cmd.index(flag) + 1
            while j < len(cmd) and not cmd[j].startswith("--"):
                j += 1
            del cmd[cmd.index(flag):j]
    return cmd + extra


def _prepare(name, tmp, kind):
    """The golden case with three interleaved populations: the whole input in tmp/all, each population's restriction
    in tmp/<P>.  → (populations, dataset)."""
    import shutil
    ds, _ = load_case(name)
    if kind == "bfile":
        ds = plink.bed_dataset(ds, seed=3)[0]
        ds._bed = plink.bed_dataset(load_case(name)[0], seed=3)
    pops = _pop_of(ds.n_ind)
    ds._pops = pops
    if kind in ("vcf", "bcf"):
        ds._vcf = vcf.from_dataset(ds, seed=11)
    dirs = {"all": (ds, pops)}
    for p in POPS:
        cols = [i for i in range(ds.n_ind) if pops[i] == p]
        d = _restrict(ds, cols, pops)
        d.pop = p
        dirs[p] = (d, [p] * len(cols))
    argv = {}
    for key, (d, pp) in dirs.items():
        t = os.path.join(tmp, key)
        argv[key] = _write_input(d, t, kind)
        _write_tfam(os.path.join(t, "syn.tfam"), d.ind_ids, pp)
        if os.path.exists(os.path.join(GOLDEN, name, "in.freq")):
            shutil.copy(os.path.join(GOLDEN, name, "in.freq"), os.path.join(t, "syn.freq"))
    return argv


def _run_cli(argv, out):
    return subprocess.run([BIN] + argv + ["--out", out], capture_output=True, text=True, timeout=600)


def _outputs(prefix):
    """name suffix → content of every output file of a run (logs without the command line and the lines naming a
    path)."""
    import glob
    import gzip
    out = {}
    for f in glob.glob(prefix + ".*"):
        suf = f[len(prefix):]
        if suf.endswith(".gz"):
            out[suf] = gzip.open(f, "rb").read()
        elif suf == ".log":
            out[suf] = [l for l in open(f).read().splitlines()[1:] if os.sep not in l]
        else:
            out[suf] = open(f, "rb").read()
    return out


BY_POP_CASES = [
    ("lod_0", "tped", []), ("lod_0", "host", []), ("lod_0", "bfile", []), ("lod_0", "vcf", []), ("lod_0", "bcf", []),
    ("gl_pl", "tped", []), ("wlod_cm", "tped", ["--ld-subsample", "5", "--seed", "3"]), ("wlod_phased", "vcf", []),
    ("lod_1", "tped", ["--freq-only"]), ("lod_3", "tped", ["--resample", "50", "--seed", "7"]),
    ("auto_cutoff", "tped", ["--kde-direct", "--seed", "5"]), ("freq_file", "tped", []),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind,extra", BY_POP_CASES)
def test_cli_by_pop_equals_separate_runs(tmp_path, name, kind, extra):
    tmp = str(tmp_path)
    argv = _prepare(name, tmp, kind)
    base = _case_argv(name, os.path.join(tmp, "all"), extra)
    r = _run_cli(base + argv["all"] + ["--by-pop"], os.path.join(tmp, "all", "out"))
    assert r.returncode == 0, r.stderr[-2000:]
    top = open(os.path.join(tmp, "all", "out.log")).read().splitlines()
    pops = _pop_of(load_case(name)[0].n_ind)
    assert top[1:] == ["Population %s: %d individuals, output prefix %s" % (p, pops.count(p), os.path.join(tmp, "all", "out." + p))
                       for p in POPS]
    for p in POPS:
        d = os.path.join(tmp, p)
        rs = _run_cli(_case_argv(name, d, extra) + argv[p], os.path.join(d, "out"))
        assert rs.returncode == 0, rs.stderr[-2000:]
        want, got = _outputs(os.path.join(d, "out")), _outputs(os.path.join(tmp, "all", "out." + p))
        assert sorted(want) == sorted(got)
        for k in want:
            assert want[k] == got[k], (p, k)


@pytest.mark.gpu
def test_cli_by_pop_two_gpus(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tmp = str(tmp_path)
    argv = _prepare("lod_0", tmp, "tped")
    base = _case_argv("lod_0", os.path.join(tmp, "all"), [])
    for g, sub in [("1", "a"), ("2", "b")]:
        r = _run_cli(base + argv["all"] + ["--by-pop", "--gpus", g], os.path.join(tmp, "all", sub))
        assert r.returncode == 0, r.stderr[-2000:]
    for p in POPS:
        assert _outputs(os.path.join(tmp, "all", "a." + p)) == _outputs(os.path.join(tmp, "all", "b." + p))


@pytest.mark.gpu
def test_cli_by_pop_refusals(tmp_path):
    tmp = str(tmp_path)
    argv = _prepare("lod_0", tmp, "tped")
    base = _case_argv("lod_0", os.path.join(tmp, "all"), [])
    out = os.path.join(tmp, "all", "x")
    r = _run_cli(base + argv["all"], out)                              # several population IDs without --by-pop
    assert r.returncode != 0 and "Found multiple population IDs" in open(out + ".error").read()
    ds, _ = load_case("lod_0")
    tfam = argv["all"][argv["all"].index("--tfam") + 1]
    pops = _pop_of(ds.n_ind)
    _write_tfam(tfam, ds.ind_ids, ["a/b" if p == "EUR" else p for p in pops])
    r = _run_cli(base + argv["all"] + ["--by-pop"], out)
    assert r.returncode != 0 and "a/b cannot be part of a file name" in open(out + ".error").read()
    assert not os.path.exists(out + ".AFR.log")                        # refused before any population runs


@pytest.mark.gpu
def test_cli_by_pop_failure_names_the_population(tmp_path):
    """A window size the library refuses: the first population's separate run fails, and the --by-pop run stops with
    that run's message prefixed by the population's ID."""
    tmp = str(tmp_path)
    argv = _prepare("auto_cutoff", tmp, "tped")
    extra = ["--winsize", "1000000"]
    out = os.path.join(tmp, "all", "y")
    r = _run_cli(_case_argv("auto_cutoff", os.path.join(tmp, "all"), extra) + argv["all"] + ["--by-pop"], out)
    assert r.returncode != 0
    d = os.path.join(tmp, "AFR")
    rs = _run_cli(_case_argv("auto_cutoff", d, extra) + argv["AFR"], os.path.join(d, "y"))
    assert rs.returncode == r.returncode
    msg = open(os.path.join(d, "y.error")).read().strip().splitlines()[-1]
    assert "winsize out of range" in msg
    assert open(out + ".error").read().splitlines()[-1] == "ERROR: population AFR: " + msg
    assert open(out + ".AFR.error").read() == open(os.path.join(d, "y.error")).read()
    assert not os.path.exists(out + ".EUR.log")
