"""The call filter of VCF / BCF input (--vcf-min-gq / --vcf-min-dp): a run with the flags equals the run on the file in
which every failing call is written ./. .  On the CPU: the text grammar (csrc/vcf_gt.cuh through
tests/vcf_filter_emu.cpp) against vcf.py's restatement, the BCF value rule against bcf.py's, the loader's GQ / DP
indices and vectors against the Python readers, and apply_call_filter against rewrite-then-read.  On the GPU: the
filtered puts against the plain puts of the rewritten input, the diagnostics and the set-missing count, sharded and
selecting handles, and driver runs with the flags against runs on the rewritten VCF."""
import ctypes as C
import itertools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from garlic_b200 import bcf, synth, vcf
from tests.common import load_case

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
M = vcf.MISSING
_EMU = None


def emu():
    """tests/vcf_filter_emu.cpp + host/io.cpp + host/cli.cpp, built into a temporary directory."""
    global _EMU
    if _EMU is None:
        so = os.path.join(tempfile.mkdtemp(prefix="garlic_filter_emu_"), "vcf_filter_emu.so")
        host = os.path.join(ROOT, "garlic_b200", "host")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                               os.path.join(HERE, "vcf_filter_emu.cpp"), os.path.join(host, "io.cpp"),
                               os.path.join(host, "cli.cpp"), "-lz", "-pthread"])
        _EMU = C.CDLL(so)
        _EMU.emu_load_filter.restype = C.c_longlong
    return _EMU


def emu_call_filter(text, k_gq, min_gq, k_dp, min_dp):
    b = text.encode()
    field = C.c_int(0)
    r = emu().emu_call_filter(b, C.c_longlong(len(b)), k_gq, min_gq, k_dp, min_dp, C.byref(field))
    return r, (field.value if r < 0 else None)


def emu_load(path, log_base, keys):
    cap = 1 << 20
    while True:
        buf = C.create_string_buffer(cap)
        need = C.c_longlong(0)
        n = emu().emu_load_filter(path.encode(), log_base.encode(), C.c_uint(keys), buf, C.c_longlong(cap), C.byref(need))
        if n == -2:
            cap = need.value + 1
            continue
        if n < 0:
            return open(log_base + ".error").read()
        lines = buf.raw[:need.value].decode().split("\n")
        nums = [np.array(l.split(), np.int64) if k != 1 else None for k, l in enumerate(lines[:5])]
        return dict(fmt_index=nums[0], fv=bytes.fromhex(lines[1]), fv_off=nums[2], fv_pos=nums[3], fv_type=nums[4],
                    text=bytes.fromhex(lines[5]))


def random_calls(seed, N, L0, miss=0.08, decimals=True):
    """A Vcf with 0..2 ALTs, missing calls, and GQ / DP values in [0, 60) with NaN (missing) and decimals."""
    rng = np.random.default_rng(seed)
    n_alt = rng.integers(0, 3, L0)
    idx = (rng.random((L0, N, 2)) * (n_alt[:, None, None] + 1)).astype(np.uint8)
    idx[rng.random((L0, N, 2)) < miss] = M
    idx[rng.random((L0, N)) < miss] = M
    gq = rng.integers(0, 60, (L0, N)).astype(float)
    dp = rng.integers(0, 40, (L0, N)).astype(float)
    if decimals:
        gq[rng.random((L0, N)) < 0.1] += 0.5
    gq[rng.random((L0, N)) < 0.05] = np.nan
    dp[rng.random((L0, N)) < 0.05] = np.nan
    chrom = ["1"] * (L0 // 2) + ["2"] * (L0 - L0 // 2)
    return vcf.Vcf(samples=["s%d" % i for i in range(N)], chrom=chrom, pos=np.arange(1, L0 + 1) * 100,
                   ids=["r%d" % s for s in range(L0)], ref=["A"] * L0,
                   alts=[["C", "G"][:int(k)] for k in n_alt], idx=idx, gq=gq, dp=dp)


def rewritten_text(text, off, fk, min_gq, min_dp):
    """The sample text with every call that fails a threshold (vcf.call_filter) written ./. ."""
    parts, new_off = [], [0]
    for s in range(len(off) - 1):
        cols = text[off[s]:off[s + 1]].decode().split("\t")
        out = []
        for c in cols:
            r, _ = vcf.call_filter(c, int(fk[s, 0]) if min_gq else -1, min_gq, int(fk[s, 1]) if min_dp else -1, min_dp)
            out.append("./." + c[len(c.split(":")[0]):] if r == 1 else c)
        parts.append("\t".join(out).encode())
        new_off.append(new_off[-1] + len(parts[-1]))
    return b"".join(parts), np.array(new_off, np.int64)


# ------------------------------------------------------------------------------------------------ CPU
ALPHABET = "0159.-:\ta"


def test_text_grammar_exhaustive():
    for n in range(0, 5):
        for t in itertools.product(ALPHABET, repeat=n):
            s = "".join(t)
            for thr in (1, 5, 19):
                b = s.encode()
                assert emu().emu_fmt_value(b, C.c_longlong(len(b)), thr) == vcf.fmt_value(s.split("\t")[0].split(":")[0], thr), (s, thr)
            col = "0/1:" + s
            for k_gq, k_dp in ((1, -1), (-1, 1), (1, 2), (2, 1), (3, 1)):
                assert emu_call_filter(col, k_gq, 5, k_dp, 10) == vcf.call_filter(col, k_gq, 5, k_dp, 10), (col, k_gq, k_dp)


@pytest.mark.parametrize("text,thr,want", [("20", 20, 1), ("19", 20, 0), ("19.99", 20, 0), ("20.0", 20, 1), (".", 20, 1),
                                           ("", 20, 1), ("-5", 1, 0), ("-0", 1, 0), ("0", 1, 0), ("99999999999999", 7, 1),
                                           ("1e3", 1, -1), ("nan", 1, -1), ("-", 1, -1), ("1.", 1, -1), (".5", 1, -1),
                                           ("..", 1, -1), ("+3", 1, -1), ("3a", 1, -1)])
def test_value_grammar_cases(text, thr, want):
    assert vcf.fmt_value(text, thr) == want
    b = text.encode()
    assert emu().emu_fmt_value(b, C.c_longlong(len(b)), thr) == want


@pytest.mark.parametrize("fmt", ["GT:AD:DP:GQ:PL", "GT:GQ:DP", "GT:DP:GQ:AD", "GT:GQ", "GT:DP", "GT:AD"])
def test_random_columns_with_dropped_fields(fmt):
    v = random_calls(3, 40, 60)
    drop = np.random.default_rng(4).integers(0, len(fmt.split(":")), (60, 40))
    text = vcf.vcf_text(v, fmt, drop=drop).decode().splitlines()
    k_gq, k_dp = vcf.format_index(fmt)
    for s, line in enumerate(l for l in text if not l.startswith("#")):
        for i, col in enumerate(line.split("\t")[9:]):
            for mg, md in ((25, 0), (0, 12), (25, 12)):
                kg, kd = (k_gq if mg else -1), (k_dp if md else -1)
                got = emu_call_filter(col, kg, mg, kd, md)
                assert got == vcf.call_filter(col, kg, mg, kd, md)
                kept = len(fmt.split(":")) - drop[s, i]
                gq = v.gq[s, i] if 0 <= kg < kept else np.nan
                dp = v.dp[s, i] if 0 <= kd < kept else np.nan
                assert got[0] == int((mg and gq < mg) or (md and dp < md))


def test_bcf_value_rule():
    cases = [(bcf.INT8, np.arange(-128, 128)),
             (bcf.INT16, np.array([-32768, -32767, -32766, -1, 0, 1, 19, 20, 127, 128, 32767])),
             (bcf.INT32, np.array([-2**31, -2**31 + 1, -2**31 + 2, -1, 0, 1, 20, 2**31 - 1]))]
    floats = np.array([0.0, -0.0, 0.5, 0.99, 1.0, 19.999, 20.0, 20.5, 1e9, 3e38, -1.0, -20.0, 1e-40], np.float32)
    fbits = np.concatenate([floats.view(np.uint32),
                            np.array([0x7F800001, 0x7F800002, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x7F800003,
                                      0x7FFFFFFF], np.uint32)])
    cases.append((bcf.FLOAT, fbits.view(np.int32)))
    for typ, raw in cases:
        raw = np.ascontiguousarray(raw, np.int32)
        for thr in (1, 20, 2**31 - 1):
            out = np.empty(len(raw), np.int32)
            emu().emu_bcf_value(raw.ctypes.data_as(C.c_void_p), C.c_int(len(raw)), C.c_int(typ), C.c_int(thr),
                                out.ctypes.data_as(C.c_void_p))
            want = [bcf.value_rule(int(r), typ, thr) for r in raw]
            assert list(out) == want, (typ, thr)
    assert bcf.value_rule(0x7F800001, bcf.FLOAT, 5) == 1 and bcf.value_rule(0x7F800000, bcf.FLOAT, 5) == -1
    assert bcf.value_rule(-128, bcf.INT8, 5) == 1 and bcf.value_rule(-127, bcf.INT8, 5) == 1
    assert bcf.value_rule(-126, bcf.INT8, 5) == 0


@pytest.mark.parametrize("fmt", ["GT:AD:DP:GQ:PL", "GT:GQ:DP", "GT:DP:GQ", "GT:AD", "GT"])
@pytest.mark.parametrize("keys", [1, 2, 3])
def test_loader_vcf_indices(tmp_path, fmt, keys):
    v = random_calls(5, 7, 90)
    path = vcf.write_vcf(str(tmp_path / "x.vcf.gz"), v, fmt, compress="bgzf", block_size=3000)
    got = emu_load(path, str(tmp_path / "log"), keys)
    fk = vcf.format_indices(path)
    fk[:, 0] = fk[:, 0] if keys & 1 else -1
    fk[:, 1] = fk[:, 1] if keys & 2 else -1
    assert np.array_equal(got["fmt_index"].reshape(-1, 2), fk)
    assert got["text"] == vcf.sample_text(path)[0]
    assert got["fv"] == b"" and len(got["fv_off"]) == 0


@pytest.mark.parametrize("fmt,call_type", [("GT:AD:DP:GQ:PL", None), ("GT:GQ:DP", bcf.INT16), ("GT:DP:GQ", bcf.INT32),
                                           ("GT:GQ:DP", bcf.FLOAT), ("GT:AD", None)])
@pytest.mark.parametrize("keys", [1, 2, 3])
def test_loader_bcf_vectors(tmp_path, fmt, call_type, keys):
    v = random_calls(6, 9, 70, decimals=call_type == bcf.FLOAT)
    path = bcf.write_bcf(str(tmp_path / "x.bcf"), v, fmt, call_type=call_type, block_size=3000)
    got = emu_load(path, str(tmp_path / "log"), keys)
    want_keys = tuple(k for j, k in enumerate(("GQ", "DP")) if keys >> j & 1)
    fv, fv_off, fv_pos, fv_type, fidx = bcf.call_values(path, want_keys)
    assert got["fv"] == fv and np.array_equal(got["fv_off"], fv_off)
    assert np.array_equal(got["fv_pos"].reshape(-1, 2), fv_pos)
    assert np.array_equal(got["fv_type"].reshape(-1, 2), fv_type)
    assert np.array_equal(got["fmt_index"].reshape(-1, 2), fidx)
    payload, off, _ = bcf.gt_payload(path)
    assert got["text"] == payload
    r = bcf.read_bcf(path)
    for key, arr in (("GQ", r.gq), ("DP", r.dp)):
        if key in fmt.split(":"):
            src = v.gq if key == "GQ" else v.dp
            assert np.array_equal(np.isnan(arr), np.isnan(src))
            ok = ~np.isnan(src)
            assert np.array_equal(arr[ok], src[ok] if call_type == bcf.FLOAT else src[ok].astype(int))


def test_loader_bcf_rejects_gq_shape(tmp_path):
    v = random_calls(7, 4, 5)
    raw = bytearray(bcf.bcf_bytes(v, "GT:GQ", call_type=bcf.INT8))
    path = str(tmp_path / "x.bcf")
    # the first record's GQ descriptor (count 1, int8) becomes count 1, char: refused only while GQ is filtered
    i = raw.index(bytes([0x11, 0x02, 0x11]), 9) + 2           # typed key 2 (GQ), then its descriptor
    raw[i] = 0x17
    open(path, "wb").write(bytes(raw))
    err = emu_load(path, str(tmp_path / "log"), 1)
    assert isinstance(err, str) and "record 1" in err and "the GQ field has count 1 and type 7" in err
    assert isinstance(emu_load(path, str(tmp_path / "log2"), 2), dict)


def test_readers_accept_malformed_values(tmp_path):
    """A malformed GQ / DP is read (as NaN, flagged) and refused only by a filter on that key, as the driver does."""
    v = random_calls(9, 5, 6)
    path = vcf.write_vcf(str(tmp_path / "x.vcf"), v, "GT:AD:DP:GQ:PL")
    lines = open(path).read().split("\n")
    body = [i for i, l in enumerate(lines) if l and not l.startswith("#")]
    cols = lines[body[2]].split("\t")
    sub = cols[9 + 1].split(":")
    sub[3] = "2e1"
    cols[9 + 1] = ":".join(sub)
    lines[body[2]] = "\t".join(cols)
    open(path, "w").write("\n".join(lines))
    r = vcf.read_vcf(path)
    assert np.isnan(r.gq[2, 1]) and r.bad[2, 1, 0] and r.bad.sum() == 1
    vcf.apply_call_filter(r, 0, 12)
    with pytest.raises(vcf.VcfError, match="record 3 .*malformed GQ of sample s1"):
        vcf.apply_call_filter(r, 25, 0)
    w = random_calls(9, 5, 6, decimals=True)
    p2 = str(tmp_path / "x.bcf")
    raw = bytearray(bcf.bcf_bytes(w, "GT:GQ:DP", call_type=bcf.FLOAT))
    inf = np.array([np.inf], np.float32).tobytes()
    first = np.array([w.gq[0, 0]], np.float32).tobytes()
    at = raw.index(bytes([0x11, 0x02, 0x15]) + first) + 3              # the first record's GQ vector, sample 0
    raw[at:at + 4] = inf
    open(p2, "wb").write(bytes(raw))
    r = bcf.read_bcf(p2)
    assert np.isnan(r.gq[0, 0]) and r.bad[0, 0, 0] and r.bad.sum() == 1
    vcf.apply_call_filter(r, 0, 12)
    with pytest.raises(vcf.VcfError, match="malformed GQ"):
        vcf.apply_call_filter(r, 25, 0)


@pytest.mark.parametrize("min_gq,min_dp", [(25, 0), (0, 12), (25, 12)])
def test_apply_call_filter_equals_rewrite_then_read(tmp_path, min_gq, min_dp):
    v = random_calls(8, 11, 80)
    path = vcf.write_vcf(str(tmp_path / "x.vcf"), v, "GT:AD:DP:GQ:PL")
    r = vcf.read_vcf(path)
    got = vcf.apply_call_filter(r, min_gq, min_dp)
    text, off = vcf.sample_text(path)
    new, new_off = rewritten_text(text, off, vcf.format_indices(path), min_gq, min_dp)
    lines = open(path).read().splitlines()
    head = [l for l in lines if l.startswith("#")]
    body = [l for l in lines if not l.startswith("#")]
    out = head + ["\t".join(b.split("\t")[:9]) + "\t" + new[new_off[s]:new_off[s + 1]].decode() for s, b in enumerate(body)]
    p2 = str(tmp_path / "y.vcf")
    open(p2, "w").write("\n".join(out) + "\n")
    assert np.array_equal(vcf.read_vcf(p2).idx, got.idx)
    assert vcf.calls_set_missing(r, min_gq, min_dp) == int(((r.idx != M).any(2) & (got.idx == M).all(2)).sum())


# ------------------------------------------------------------------------------------------------ GPU: kernels
def _shape(g, N, L0, ind_offset=0):
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 1000
    g.set_shape(N, L0, np.array([0, L0 // 2, L0], np.int64), pos, ind_offset=ind_offset)


def _state(g, L0):
    g.code_alleles()
    return (synth.unpack_codes(g.get_genotypes(False), L0), [np.array(c) for c in g.get_counts()], g.get_one_allele(255))


def _same_state(a, b):
    assert np.array_equal(a[0], b[0])
    assert all(np.array_equal(x, y) for x, y in zip(a[1], b[1]))
    assert np.array_equal(a[2], b[2])


FILTERS = [(25, 0), (0, 12), (25, 12)]


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 3, 29, 77, 513])
@pytest.mark.parametrize("min_gq,min_dp", FILTERS)
def test_vcf_filtered_put_equals_rewritten(tmp_path, N, min_gq, min_dp):
    from garlic_b200.api import GarlicGPU
    L0 = 1500
    v = random_calls(N, N, L0)
    fmt = ["GT:AD:DP:GQ:PL", "GT:GQ:DP", "GT:DP"][N % 3]
    drop = np.random.default_rng(N).integers(0, 2, (L0, N)) * np.random.default_rng(N + 1).integers(0, 3, (L0, N))
    path = vcf.write_vcf(str(tmp_path / "x.vcf"), v, fmt, drop=drop)
    text, off = vcf.sample_text(path)
    fk = vcf.format_indices(path)
    new, new_off = rewritten_text(text, off, fk, min_gq, min_dp)
    want = vcf.apply_call_filter(vcf.read_vcf(path), min_gq, min_dp)
    a = GarlicGPU(0)
    _shape(a, N, L0)
    a.set_call_filter(min_gq, min_dp)
    diag = [a.put_vcf_text_filtered(text, off[s0:s0 + 1025], fk[s0:s0 + 1024], s0) for s0 in range(0, L0, 1024)]
    nc, mx, bad, badv = (np.concatenate(d) for d in zip(*diag))
    assert (nc == N).all() and (bad == -1).all() and (badv == -1).all()
    present = np.where(v.idx == M, -1, v.idx.astype(np.int64)).reshape(L0, -1).max(1)
    assert np.array_equal(mx, present)                             # the allele check sees the calls as written
    r = vcf.read_vcf(path)
    assert a.calls_set_missing() == vcf.calls_set_missing(r, min_gq, min_dp)
    b = GarlicGPU(0)
    _shape(b, N, L0)
    for s0 in range(0, L0, 1024):
        b.put_vcf_text(new, new_off[s0:s0 + 1025], s0)
    sa, sb = _state(a, L0), _state(b, L0)
    _same_state(sa, sb)
    assert np.array_equal(sa[2], vcf.one_allele(want.idx))
    a.close()
    b.close()


def _gt_vectors(idx, width):
    """(payload, rec_off, gt_type) of GT vectors of idx (count 2) at `width` bytes per value."""
    typ = bcf.TYPE_OF_WIDTH[width]
    parts, off = [], [0]
    for s in range(len(idx)):
        _, vals = bcf._gt_field(idx[s], False, width)
        raw = vals.astype(bcf._DT[typ]).tobytes()
        raw += b"\0" * (-len(raw) % 4)
        parts.append(raw)
        off.append(off[-1] + len(raw))
    return b"".join(parts), np.array(off, np.int64), np.full(len(idx), 2 << 4 | typ, np.uint8)


def _value_vectors(v, typ, fmt_keys, rng, eov_rate=0.03):
    """(fv, fv_off, fv_pos, fv_type, gq, dp) with the raw GQ / DP vectors of v as typ, in the order of fmt_keys (a
    random share of the values replaced by the end-of-vector sentinel; missing values are the missing sentinel)."""
    parts, off = [], [0]
    L0, N = v.idx.shape[:2]
    pos = np.full((L0, 2), -1, np.int32)
    types = np.zeros((L0, 2), np.uint8)
    out = {"GQ": np.full((L0, N), np.nan), "DP": np.full((L0, N), np.nan)}
    for s in range(L0):
        span = b""
        for key in fmt_keys:
            j = ("GQ", "DP").index(key)
            vals = bcf.value_array((v.gq if key == "GQ" else v.dp)[s], typ)
            eov = rng.random(N) < eov_rate if eov_rate else np.zeros(N, bool)
            if typ == bcf.FLOAT:
                vals.view(np.uint32)[eov] = bcf.FLOAT_EOV
            else:
                vals[eov] = bcf.EOV[bcf.WIDTH[typ]]
            out[key][s] = bcf.values_float(vals, typ)
            pos[s, j], types[s, j] = len(span), 1 << 4 | typ
            raw = vals.tobytes()
            span += raw + b"\0" * (-len(raw) % 4)
        parts.append(span)
        off.append(off[-1] + len(span))
    return b"".join(parts), np.array(off, np.int64), pos, types, out["GQ"], out["DP"]


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 3, 29, 77, 513])
@pytest.mark.parametrize("typ", [bcf.INT8, bcf.INT16, bcf.INT32, bcf.FLOAT])
@pytest.mark.parametrize("min_gq,min_dp", FILTERS)
@pytest.mark.parametrize("width", [1, 2, 4])                       # GT int8 (count-2 word path), int16, int32 (per sample)
def test_bcf_filtered_put_equals_rewritten(N, typ, min_gq, min_dp, width):
    from garlic_b200.api import GarlicGPU
    L0 = 1100
    rng = np.random.default_rng(N * 7 + typ)
    v = random_calls(N + typ, N, L0, decimals=typ == bcf.FLOAT)
    keys = [("GQ", "DP"), ("DP", "GQ"), ("GQ",), ("DP",)][(N + typ) % 4]
    fv, fv_off, fv_pos, fv_type, gq, dp = _value_vectors(v, typ, keys, rng)
    w = vcf.Vcf(**{**v.__dict__, "gq": gq, "dp": dp})
    want = vcf.apply_call_filter(w, min_gq, min_dp)
    gt, rec_off, gt_type = _gt_vectors(v.idx, width)
    a = GarlicGPU(0)
    _shape(a, N, L0)
    a.set_call_filter(min_gq, min_dp)
    mx, bad, badv = a.put_bcf_gt_filtered(gt, rec_off, gt_type, N, fv, fv_off, fv_pos, fv_type)
    assert (bad == -1).all() and (badv == -1).all()
    present = np.where(v.idx == M, -1, v.idx.astype(np.int64)).reshape(L0, -1).max(1)
    assert np.array_equal(mx, present)
    assert a.calls_set_missing() == vcf.calls_set_missing(w, min_gq, min_dp)
    gt2, off2, type2 = _gt_vectors(want.idx, width)
    b = GarlicGPU(0)
    _shape(b, N, L0)
    b.put_bcf_gt(gt2, off2, type2, N)
    _same_state(_state(a, L0), _state(b, L0))
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["vcf", "bcf", "bcf16"])         # bcf16: int16 GT, the per-sample path
def test_selected_and_sharded_handles(tmp_path, kind):
    """A selecting handle equals a handle given the restricted input; two sharded handles equal one handle."""
    from garlic_b200.api import GarlicGPU
    N, L0, mg, md = 77, 1300, 25, 12
    v = random_calls(11, N, L0, decimals=False)
    if kind != "vcf":                                              # the values as the vectors hold them (EOV: NaN)
        _, _, _, _, gq, dp = _value_vectors(v, bcf.INT8, ("GQ", "DP"), np.random.default_rng(1))
        v = vcf.Vcf(**{**v.__dict__, "gq": gq, "dp": dp})

    def putter(w, name):
        """put(g) of the input w (all its samples) → the per-record malformed-value diagnostic."""
        if kind == "vcf":
            path = vcf.write_vcf(str(tmp_path / name), w, "GT:AD:DP:GQ:PL")
            text, off = vcf.sample_text(path)
            fk = vcf.format_indices(path)
            return lambda g: g.put_vcf_text_filtered(text, off, fk)[3]
        fv, fv_off, fv_pos, fv_type, _, _ = _value_vectors(w, bcf.INT8, ("GQ", "DP"), None, eov_rate=0)
        gt, rec_off, gt_type = _gt_vectors(w.idx, 2 if kind == "bcf16" else 1)
        n = len(w.samples)
        return lambda g: g.put_bcf_gt_filtered(gt, rec_off, gt_type, n, fv, fv_off, fv_pos, fv_type)[2]

    put = putter(v, "x.vcf")
    whole = GarlicGPU(0)
    _shape(whole, N, L0)
    whole.set_call_filter(mg, md)
    assert (put(whole) == -1).all()
    want = _state(whole, L0)
    whole_set = whole.calls_set_missing()
    cols = np.array([i for i in range(N) if (i + i // 4) % 3 == 1], np.int32)
    sel = GarlicGPU(0)
    _shape(sel, len(cols), L0)
    sel.select_columns(cols, N)
    sel.set_call_filter(mg, md)
    assert (put(sel) == -1).all()
    assert sel.calls_set_missing() == vcf.calls_set_missing(v, mg, md, cols)
    sub = vcf.Vcf(**{**v.__dict__, "samples": [v.samples[i] for i in cols], "idx": v.idx[:, cols], "gq": v.gq[:, cols],
                     "dp": v.dp[:, cols]})
    res = GarlicGPU(0)
    _shape(res, len(cols), L0)
    res.set_call_filter(mg, md)
    assert (putter(sub, "sub.vcf")(res) == -1).all()
    assert res.calls_set_missing() == sel.calls_set_missing()
    _same_state(_state(sel, L0), _state(res, L0))
    sel.close()
    res.close()
    # two shards: the first-allele keys are MIN-reduced across the handles before coding, as the driver's ranks do
    import torch
    hs = []
    for lo, hi in ((0, 40), (40, N)):
        g = GarlicGPU(0)
        _shape(g, hi - lo, L0, ind_offset=lo)
        g.set_call_filter(mg, md)
        assert (put(g) == -1).all()
        g.sync()
        hs.append(g)
    assert sum(g.calls_set_missing() for g in hs) == whole_set == vcf.calls_set_missing(v, mg, md)
    keys = [torch.as_tensor(_DevArray(g.first_allele_keys_dev(), L0, "<i8"), device="cuda") for g in hs]
    mn = np.minimum.reduce([k.cpu().numpy().view(np.uint64) for k in keys])
    for k in keys:
        k.copy_(torch.from_numpy(mn.view(np.int64)))
    torch.cuda.synchronize()
    rows = np.concatenate([_state(g, L0)[0] for g in hs])
    assert np.array_equal(rows, want[0])
    for g in hs + [whole]:
        g.close()


class _DevArray:
    """A device buffer of the library as a torch tensor (no copy)."""
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = dict(shape=(n,), typestr=typestr, data=(ptr, False), version=2)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1, 2])
def test_filter_without_values_stores_every_call(tmp_path, width):
    """Filters on, but no record holds GQ or DP: the filtered puts store what the plain puts store and set nothing
    missing (the BCF value buffer is empty and goes to the library as NULL)."""
    from garlic_b200.api import GarlicGPU
    N, L0 = 29, 700
    v = random_calls(31, N, L0)
    v.gq = v.dp = None
    gt, rec_off, gt_type = _gt_vectors(v.idx, width)
    text, off = vcf.sample_text(vcf.write_vcf(str(tmp_path / "x.vcf"), v))
    states = []
    for filtered in (False, True):
        for kind in ("vcf", "bcf"):
            g = GarlicGPU(0)
            _shape(g, N, L0)
            if filtered:
                g.set_call_filter(20, 10)
                if kind == "vcf":
                    assert (g.put_vcf_text_filtered(text, off, np.full((L0, 2), -1, np.int32))[3] == -1).all()
                else:
                    assert (g.put_bcf_gt_filtered(gt, rec_off, gt_type, N, b"", np.zeros(L0 + 1, np.int64),
                                                  np.full((L0, 2), -1, np.int32), np.zeros((L0, 2), np.uint8))[2] == -1).all()
                assert g.calls_set_missing() == 0
            elif kind == "vcf":
                g.put_vcf_text(text, off)
            else:
                g.put_bcf_gt(gt, rec_off, gt_type, N)
            states.append(_state(g, L0))
            g.close()
    for st in states[1:]:
        _same_state(states[0], st)


@pytest.mark.gpu
def test_malformed_value_diagnostics():
    from garlic_b200.api import GarlicGPU
    recs = ["0/1:30:10\t1/1:3x:10\t0/0:abc:1", "0/1:30:10\t0/1:30:-\t0/0:30:1e2", "0/1:.:\t0/1::\t./.:1:1",
            "0/1:nan:5\t0/1:5:5\t0/1:5:5"]
    fk = np.array([[1, 2]] * 4, np.int32)
    text = "".join(recs).encode()
    off = np.concatenate([[0], np.cumsum([len(r) for r in recs])]).astype(np.int64)
    for mg, md, want in ((20, 0, [1, -1, -1, 0]), (0, 5, [-1, 1, -1, -1]), (20, 5, [1, 1, -1, 0])):
        g = GarlicGPU(0)
        _shape(g, 3, 4)
        g.set_call_filter(mg, md)
        nc, mx, bad, badv = g.put_vcf_text_filtered(text, off, fk)
        assert list(badv) == want and (bad == -1).all()
        g.close()
    # BCF: a NaN that is not a sentinel, or an infinity, is malformed
    idx = np.zeros((2, 5, 2), np.uint8)
    gt, rec_off, gt_type = _gt_vectors(idx, 1)
    vals = np.array([[30, 30, 0x7F800000, 30, 0x7FC00000], [0x7F800001, 0x7F800002, 1, 30, 0xFF800000]], np.uint32)
    vals = np.where(vals < 100, np.array(vals, np.float32).view(np.uint32), vals).astype(np.uint32)
    fv = b"".join(r.tobytes() for r in vals)
    g = GarlicGPU(0)
    _shape(g, 5, 2)
    g.set_call_filter(20, 0)
    mx, bad, badv = g.put_bcf_gt_filtered(gt, rec_off, gt_type, 5, fv, np.array([0, 20, 40]),
                                          np.array([[0, -1], [0, -1]], np.int32), np.full((2, 2), 0x15, np.uint8))
    assert list(badv) == [2, 4]
    g.close()
    g = GarlicGPU(0)
    _shape(g, 5, 2)
    g.set_call_filter(20, 0)
    with pytest.raises(Exception, match="GQ descriptor"):
        g.put_bcf_gt_filtered(gt, rec_off, gt_type, 5, fv, np.array([0, 20, 40]), np.array([[0, -1], [0, -1]], np.int32),
                              np.full((2, 2), 0x25, np.uint8))
    g.close()


# ------------------------------------------------------------------------------------------------ GPU: driver
BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")


def _case(name, tmp, seed):
    """A golden case's command (without input or output) and its Vcf with GQ / DP values."""
    ds, _ = load_case(name)
    ds.write(tmp)
    v = vcf.from_dataset(ds, seed=11)
    L0, N = v.idx.shape[:2]
    r = random_calls(seed, N, L0, decimals=False)
    v.gq, v.dp = r.gq, r.dp
    with open(os.path.join(HERE, "golden", name, "cmd.txt")) as f:
        cmd = [a.replace("<tmp>", tmp) for a in f.readline().split()[1:] if a != "--raw-lod"]
    i = cmd.index("--out")
    del cmd[i:i + 2]
    i = cmd.index("--tped")
    return cmd[:i] + cmd[i + 4:], cmd[i + 3], v


def _write(kind, path, v, call_type=None):
    if kind == "bcf":
        return bcf.write_bcf(path + ".bcf", v, "GT:AD:DP:GQ:PL", call_type=call_type, block_size=4000)
    comp = {"plain": None, "gz": "gz", "bgzf": "bgzf"}[kind]
    return vcf.write_vcf(path + (".vcf" if comp is None else ".vcf.gz"), v, "GT:AD:DP:GQ:PL", compress=comp, block_size=4000)


def _run(argv, out):
    return subprocess.run([BIN] + argv + ["--out", out], capture_output=True, text=True, timeout=300)


NEW_LINES = ("Minimum genotype quality", "Minimum read depth", "Calls set missing by the GQ/DP filter")


def _compare(tmp, a, b, count=None):
    for ext in (".roh.bed", ".freq.gz"):
        assert os.path.exists(a + ext) == os.path.exists(b + ext), ext
        if os.path.exists(a + ext):
            assert open(a + ext, "rb").read() == open(b + ext, "rb").read(), ext
    ka = sorted(f[len(os.path.basename(a)):] for f in os.listdir(tmp) if f.startswith(os.path.basename(a) + ".") and f.endswith(".kde"))
    kb = sorted(f[len(os.path.basename(b)):] for f in os.listdir(tmp) if f.startswith(os.path.basename(b) + ".") and f.endswith(".kde"))
    assert ka == kb
    for k in ka:
        assert open(a + k).read() == open(b + k).read()
    la = open(a + ".log").read().splitlines()[1:]
    lines = [l for l in la if l.startswith("Calls set missing")]
    if count is not None:
        assert len(lines) == 1 and lines[0].startswith("Calls set missing by the GQ/DP filter: %d;" % count), lines
    keep = [l for l in la if tmp not in l and not l.startswith(NEW_LINES)]
    assert keep == [l for l in open(b + ".log").read().splitlines()[1:] if tmp not in l]


@pytest.mark.gpu
@pytest.mark.parametrize("name,kind,min_gq,min_dp,call_type", [
    ("lod_0", "plain", 25, 0, None),
    ("lod_small", "gz", 0, 12, None),
    ("wlod_cm", "bgzf", 25, 12, None),
    ("gl_pl", "bgzf", 20, 5, None),
    ("lod_small", "bcf", 25, 12, None),
    ("wlod_cm", "bcf", 30, 0, bcf.INT16),
    ("lod_0", "bcf", 0, 10, bcf.FLOAT),
])
def test_cli_filter_equals_rewritten(tmp_path, name, kind, min_gq, min_dp, call_type):
    tmp = str(tmp_path)
    base, _, v = _case(name, tmp, 17)
    src = _write(kind, os.path.join(tmp, "in"), v, call_type)
    rew = _write(kind, os.path.join(tmp, "rw"), vcf.apply_call_filter(v, min_gq, min_dp), call_type)
    flags = (["--vcf-min-gq", str(min_gq)] if min_gq else []) + (["--vcf-min-dp", str(min_dp)] if min_dp else [])
    r1 = _run(base + ["--vcf", src] + flags, os.path.join(tmp, "f"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(base + ["--vcf", rew], os.path.join(tmp, "r"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _compare(tmp, os.path.join(tmp, "f"), os.path.join(tmp, "r"), vcf.calls_set_missing(v, min_gq, min_dp))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,fmt,flags", [
    ("plain", "GT", ["--vcf-min-gq", "20"]),
    ("bgzf", "GT", ["--vcf-min-dp", "10"]),
    ("bcf", "GT", ["--vcf-min-gq", "20", "--vcf-min-dp", "10"]),
    ("bcf", "GT", ["--vcf-min-dp", "10"]),
    ("bcf", "GT:GQ", ["--vcf-min-dp", "10"]),                     # GQ present, DP absent everywhere
    ("gz", "GT:GQ", ["--vcf-min-dp", "10"]),
])
def test_cli_filter_on_absent_keys(tmp_path, kind, fmt, flags):
    """A filtered key that no record holds: every call passes, the outputs equal the unfiltered run, and the log counts
    every record as lacking the key."""
    tmp = str(tmp_path)
    base, _, v = _case("lod_small", tmp, 37)
    if "GQ" not in fmt:
        v.gq = None
    v.dp = None
    if kind == "bcf":
        src = bcf.write_bcf(os.path.join(tmp, "in.bcf"), v, fmt, block_size=4000)
    else:
        comp = None if kind == "plain" else kind
        src = vcf.write_vcf(os.path.join(tmp, "in.vcf" + (".gz" if comp else "")), v, fmt, compress=comp, block_size=4000)
    r1 = _run(base + ["--vcf", src] + flags, os.path.join(tmp, "f"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(base + ["--vcf", src], os.path.join(tmp, "r"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    _compare(tmp, os.path.join(tmp, "f"), os.path.join(tmp, "r"), 0)
    line = [l for l in open(os.path.join(tmp, "f.log")).read().splitlines() if l.startswith("Calls set missing")][0]
    assert line.endswith(": %d" % len(v.chrom)), line


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", ["1", "2"])
def test_cli_filter_by_pop_and_gpus(tmp_path, gpus):
    import torch
    if gpus == "2" and torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tmp = str(tmp_path)
    base, _, v = _case("lod_small", tmp, 23)
    N = v.idx.shape[1]
    pops = ["P%d" % ((i + i // 4) % 3) for i in range(N)]
    tfam = os.path.join(tmp, "pops.tfam")
    with open(tfam, "w") as f:
        for p, s in zip(pops, v.samples):
            f.write("%s %s 0 0 0 0\n" % (p, s))
    src = _write("bgzf", os.path.join(tmp, "in"), v)
    rew = _write("bgzf", os.path.join(tmp, "rw"), vcf.apply_call_filter(v, 25, 12))
    extra = ["--tfam", tfam, "--by-pop", "--gpus", gpus]
    r1 = _run(base + ["--vcf", src, "--vcf-min-gq", "25", "--vcf-min-dp", "12"] + extra, os.path.join(tmp, "f"))
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = _run(base + ["--vcf", rew] + extra, os.path.join(tmp, "r"))
    assert r2.returncode == 0, r2.stderr[-2000:]
    for p in ("P0", "P1", "P2"):
        cols = [i for i in range(N) if pops[i] == p]
        _compare(tmp, os.path.join(tmp, "f." + p), os.path.join(tmp, "r." + p), vcf.calls_set_missing(v, 25, 12, cols))


@pytest.mark.gpu
def test_cli_filter_refusals_and_errors(tmp_path):
    tmp = str(tmp_path)
    base, tfam, v = _case("lod_small", tmp, 29)
    tped = ["--tped", os.path.join(tmp, "syn.tped"), "--tfam", tfam]
    for flag in ("--vcf-min-gq", "--vcf-min-dp"):
        r = _run(base + tped + [flag, "10"], os.path.join(tmp, "t"))
        assert r.returncode != 0 and "apply to --vcf input" in r.stderr
        r = _run(base + ["--bfile", os.path.join(tmp, "nothing"), flag, "10"], os.path.join(tmp, "b"))
        assert r.returncode != 0 and "apply to --vcf input" in r.stderr
        for bad in ("0", "-3"):
            src = _write("plain", os.path.join(tmp, "in"), v)
            r = _run(base + ["--vcf", src, flag, bad], os.path.join(tmp, "z"))
            assert r.returncode != 0 and flag + " must be an integer >= 1" in r.stderr
    v.gq = np.array(v.gq)
    v.gq[5, 3] = np.nan
    src = _write("plain", os.path.join(tmp, "in"), v)
    lines = open(src).read().split("\n")
    body = [i for i, l in enumerate(lines) if l and not l.startswith("#")]
    cols = lines[body[5]].split("\t")
    sub = cols[9 + 3].split(":")
    sub[3] = "2e1"
    cols[9 + 3] = ":".join(sub)
    lines[body[5]] = "\t".join(cols)
    open(src, "w").write("\n".join(lines))
    r = _run(base + ["--vcf", src, "--vcf-min-gq", "10"], os.path.join(tmp, "m"))
    assert r.returncode != 0
    want = "%s line %d (%s:%d): the GQ of sample %s (2e1) is not a number" % (src, body[5] + 1, v.chrom[5], v.pos[5], v.samples[3])
    assert want in r.stderr, r.stderr[-1000:]
    r = _run(base + ["--vcf", src, "--vcf-min-dp", "10"], os.path.join(tmp, "ok"))   # GQ not filtered: not checked
    assert r.returncode == 0, r.stderr[-1000:]
