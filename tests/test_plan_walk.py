"""The pruned pass 2 without a compacted matrix: the bound over the uncompacted rows (squeeze.cu, no output tile), the
walker's own compacted slices (bound.cuh:plan_slice, kernels.cu:walk_units_kernel) and the lazy compaction behind
every consumer that still reads compacted rows (capi.cu:ensure_geno)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from garlic_b200 import synth
from tests.test_host_emu import _p, synth_pack

PAD = 4160
HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def plan_emu():
    """tests/plan_emu.cpp (bound.cuh:plan_slice for the CPU), built into a temporary directory."""
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="garlic_plan_emu_"), "plan_emu.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-o", so,
                               os.path.join(HERE, "plan_emu.cpp")])
        _LIB = C.CDLL(so)
    return _LIB


def _slices(codes, keep, wlo, n):
    src = np.flatnonzero(keep).astype(np.int32)
    L = len(src)
    N, L0 = codes.shape
    in_words = (((L0 + PAD + 31) >> 5) + 3) & ~1
    rows_in = synth_pack(codes, in_words)
    out = np.zeros((N, n), np.uint64)
    plan_emu().emu_plan_slice(_p(rows_in), C.c_int64(in_words), _p(src), C.c_longlong(L), C.c_int(N), C.c_longlong(wlo), C.c_int(n),
                         _p(out))
    out_words = (((L + PAD + 31) >> 5) + 3) & ~1
    full = synth_pack(codes[:, keep], out_words)
    # beyond the kept SNPs the slice reads as missing calls (code 3): what the compacted matrix's tail holds
    tail = np.full((N, max(0, wlo + n - out_words)), 0xFFFFFFFFFFFFFFFF, np.uint64)
    want = np.concatenate([full, tail], 1)[:, wlo:wlo + n].copy()
    last = L - 32 * wlo                                    # kept SNPs inside the slice
    for w in range(n):                                     # SNPs from L on: missing, whatever the packing left there
        lo = last - 32 * w
        if lo < 32:
            m = np.uint64(0) if lo <= 0 else np.uint64((1 << (2 * lo)) - 1)
            want[:, w] = (want[:, w] & m) | (np.uint64(0xFFFFFFFFFFFFFFFF) & ~m)
    return out, want, L


def test_plan_slice_equals_column_gather():
    """Random item ranges of the walker's slices, bit for bit against dropping the columns: single and several dropped
    SNPs per half-word, dropped runs longer than 16 SNPs (the plan's segment form), the last piece, ragged L."""
    rng = np.random.default_rng(11)
    N = 33
    for L0, drop in ((9000, 0.02), (7777, 0.1), (6001, 0.4), (5000, 0.0)):
        codes = rng.integers(0, 4, (N, L0)).astype(np.uint8)
        keep = rng.random(L0) >= drop
        keep[2000:2040] = False                            # a dropped run of 40 SNPs
        keep[3000:3017] = False                            # … and one of 17
        L = int(keep.sum())
        n_w = (L + 31) // 32
        ranges = [(0, 14), (n_w - 14, 14), (n_w - 3, 8), (max(0, n_w - 52), 52)]     # the last piece, past the end
        ranges += [(int(rng.integers(0, n_w - 20)), int(rng.integers(1, 53))) for _ in range(12)]
        for wlo, n in ranges:
            got, want, _ = _slices(codes, keep, wlo, n)
            assert np.array_equal(got, want), (L0, drop, wlo, n)


# --------------------------------------------------------------------------------------------------- GPU
def _handle(n_ind, L0, seed, prune=True):
    from garlic_b200.pipeline import HotPath
    names, offs, pos, cens = synth.make_positions_genomewide(seed, L0)
    codes = synth.make_codes(seed, n_ind, L0)
    if not prune:
        os.environ["GARLIC_NO_PRUNE"] = "1"
    try:
        hp = HotPath()
    finally:
        os.environ.pop("GARLIC_NO_PRUNE", None)
    g = hp.g
    g.set_shape(n_ind, L0, offs, pos)
    g.put_packed(synth.pack_codes(codes))
    g.count_packed()
    freq, keep, L = g.filter()
    g.set_tables(0.001, 200000, np.array([cens["chr" + n] for n in names], np.int32))
    return hp, g, codes, keep.copy(), L


@pytest.mark.gpu
@pytest.mark.parametrize("n_ind,L0,W,W2", [(300, 80000, 50, 100), (77, 30011, 32, 209), (513, 20000, 64, 250)])
def test_bound_over_uncompacted_rows_equals_host_emulation(n_ind, L0, W, W2):
    """The no-store bound pass (thinned windows first, as the benchmarked step runs them) and a second window size on
    the same, still uncompacted, data: piece maxima equal bound.cuh on the CPU bit for bit."""
    from tests.test_gpu_parity import _emu_bounds
    hp, g, codes, keep, L = _handle(n_ind, L0, 13)
    g.windows(W, W, individuals=np.arange(0, n_ind, 37, dtype=np.int32), exact=False)
    assert g.last_stats()["squeeze_ms"] > 0
    n0 = g.launch_count()
    got = g.piece_bounds(W2)                               # no compacted rows yet: the no-store pass again
    assert g.launch_count() - n0 == 2                      # (its tables, the pass)
    lut = g.get_lut()
    assert np.array_equal(got, _emu_bounds(codes[:, keep], lut, L, W2))
    assert np.array_equal(g.piece_bounds(W), _emu_bounds(codes[:, keep], lut, L, W))
    hp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,cutoff", [(50, 2.0), (32, 0.5), (100, 5.0), (209, 20.0), (60, -3.0), (10, 1.0), (16, 1.0), (30, 1.5), (31, 2.0),
                                      (250, 25.0), (400, 40.0), (600, 50.0)])
def test_pruned_pass_without_compacted_rows_equals_exact_and_unpruned(W, cutoff):
    """The step as the benchmark runs it (thinned windows, then call_roh; from W 32 on no compacted matrix) == the
    unpruned pass == whole-segment exact chains, over the window-size classes and cutoffs of the pruned-pass test."""
    outs = {}
    for mode in ("pruned", "unpruned"):
        hp, g, codes, keep, L = _handle(330, 70000, 4, prune=mode == "pruned")
        g.windows(W, W, individuals=np.arange(0, 330, 17, dtype=np.int32), exact=False)
        outs[mode] = g.call_roh(W, cutoff, 0.25).copy()
        if mode == "pruned":
            outs["exact"] = g.call_roh(W, cutoff, 0.25, exact=True).copy()
        hp.close()
    assert len(outs["exact"]) > (50 if W <= 400 else -1)
    assert np.array_equal(outs["pruned"], outs["exact"])
    assert np.array_equal(outs["unpruned"], outs["exact"])


@pytest.mark.gpu
def test_c2_shaped_step_launches_no_compaction_and_rows_compact_lazily():
    """windows -> call_roh at W 50 launches no compaction: the first consumer of compacted rows afterwards
    (get_genotypes) launches exactly one kernel, the compaction, and gets the column gather; a second call launches none."""
    hp, g, codes, keep, L = _handle(300, 80000, 21)
    g.windows(50, 50, individuals=np.arange(0, 300, 15, dtype=np.int32), exact=False)
    roh = g.call_roh(50, 2.0, 0.25).copy()
    st = g.last_stats()
    assert 0 <= st["candidate_pairs"] < st["all_pairs"] and len(roh) > 100
    n0 = g.launch_count()
    packed = g.get_genotypes(True)
    assert g.launch_count() - n0 == 1
    assert np.array_equal(synth.unpack_codes(packed, L), codes[:, keep])
    n1 = g.launch_count()
    g.get_genotypes(True)
    assert g.launch_count() == n1
    assert np.array_equal(g.call_roh(50, 2.0, 0.25), roh)                                # now over compacted rows too
    hp.close()


@pytest.mark.gpu
def test_ambiguous_pairs_rewalk_after_the_pass_without_compacted_rows():
    """A cutoff on a window value: the pruned pass over uncompacted rows marks the pair ambiguous, the whole-segment
    re-walk compacts the rows on demand and the result equals the oracle."""
    from oracle import oracle as orc
    from garlic_b200.pipeline import HotPath
    from tests.common import flatten, load_case, oracle_roh_idx
    ds, args = load_case("lod_small")
    W = 50
    res0 = orc.run_pipeline(ds, W, 0.001, None)
    F = flatten(res0, 0.001)
    win = res0["chroms"][0]["win"]
    vals = np.sort(win[win != orc.MISSING])
    cutoff = float(vals[len(vals) // 2])
    res = orc.run_pipeline(ds, W, 0.001, cutoff)
    hp = HotPath().load(ds, error=0.001)
    hp.g.set_lut(F["lut"][:hp.L])
    n0 = hp.g.launch_count()
    got = hp.roh(W, cutoff, 0.25, exact=False)
    assert hp.g.last_stats()["ambiguous_pairs"] >= 1
    assert hp.g.last_stats()["candidate_pairs"] >= 0
    assert hp.g.launch_count() > n0
    assert [(r[0], r[1], r[5], r[6]) for r in got] == oracle_roh_idx(res)
    hp.close()
