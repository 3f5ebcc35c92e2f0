"""bench.py --dump-outputs: the files it writes stay within the size limit and are the same from run to run, and on
the GPU they hold what the timed steps computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _outputs():
    rng = np.random.default_rng(3)
    return dict(freq=rng.random(200_000), keep=rng.random(200_000) < 0.9, kde_windows=rng.random((20, 5000)),
                roh=rng.integers(0, 600_000, (9000, 4)).astype(np.int32), absent=None)


def _load(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_below_the_limit_is_whole(tmp_path):
    arrays = _outputs()
    bench.dump_outputs(str(tmp_path), arrays)
    got = _load(str(tmp_path))
    assert sorted(got) == ["freq.npy", "kde_windows.npy", "keep.npy", "roh.npy"]
    assert got["keep.npy"].dtype == np.float32 and got["freq.npy"].dtype == np.float64
    for k in ("freq", "keep", "kde_windows", "roh"):
        assert np.array_equal(got[k + ".npy"], arrays[k])


def test_dump_above_the_limit_is_a_fixed_sample(tmp_path):
    arrays, limit = _outputs(), 1 << 20
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), arrays, limit=limit)
    bench.dump_outputs(str(b), arrays, limit=limit)
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= limit
    got, again = _load(str(a)), _load(str(b))
    assert sorted(got) == sorted(again)
    assert all(np.array_equal(got[f], again[f]) for f in got)
    for k in ("freq", "keep", "kde_windows", "roh"):
        rows = got[k + "_rows.npy"].astype(np.int64)
        assert len(rows) > 0 and np.all(np.diff(rows) > 0)
        assert np.array_equal(got[k + ".npy"], arrays[k][rows])


@pytest.mark.gpu
def test_bench_dump_holds_the_timed_steps_outputs(tmp_path):
    """Two bench runs with different --steps dump the same arrays, and these equal the frequencies, keep mask and ROH
    calls recomputed on the host from the same seeded genotypes."""
    import torch
    n, L = 256, 60_000
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--n-ind", str(n), "--n-loci", str(L), "--warmup", "1", "--no-cpu"]
    dumps = []
    for steps in (3, 1):
        d = tmp_path / ("steps%d" % steps)
        r = subprocess.run(cmd + ["--steps", str(steps), "--dump-outputs", str(d)], cwd=ROOT, capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        dumps.append(_load(str(d)))
    got, again = dumps
    assert sorted(got) == ["freq.npy", "kde_windows.npy", "keep.npy", "roh.npy"]
    assert all(np.array_equal(got[f], again[f]) for f in got)
    assert len(got["roh.npy"]) == line["roh_found"] > 0

    from garlic_b200 import synth
    cfg = bench.CFG
    names, chr_off, pos, cens = synth.make_positions_genomewide(cfg["seed"], L)
    row_bytes = ((L + 3) // 4 + 15) // 16 * 16
    rows = bench.make_rows_torch(torch, torch.device("cuda", 0), n, L, cfg["seed"], 1000, row_bytes).cpu().numpy()
    codes = bench.unpack_rows(rows, L)
    called = codes != 3
    tot = 2 * called.sum(0)
    freq = np.where(tot > 0, np.where(called, codes, 0).sum(0) / np.maximum(tot, 1), 0.0)
    keep = (freq > 0) & (freq < 1)
    assert np.array_equal(got["freq.npy"], freq)
    assert np.array_equal(got["keep.npy"], keep.astype(np.float32))

    chroms = bench.cpu_chroms(codes, keep, freq, pos, chr_off, names, cens)
    _, want = bench.CpuSample(chroms, n, cfg["winsize"], cfg["error"], cfg["cutoff"], cfg["overlap_frac"],
                              cfg["max_gap"], 4).run()
    pos_k = pos[keep]
    roh = got["roh.npy"].astype(np.int64)
    assert sorted((int(i), int(c), int(pos_k[a]), int(pos_k[b])) for i, c, a, b in roh) == sorted(want)
