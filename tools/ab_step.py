#!/usr/bin/env python3
"""A/B of the benchmarked step between two checkouts of this repository, in one job on one GPU.

    python tools/ab_step.py --a OLD_TREE --b NEW_TREE [--runs 3] [--steps 30] [--warmup 5] [--out DIR]

Each tree must hold a built library (garlic_b200/libgarlic_b200.so).  The two trees' `bench.py --no-configs --no-cpu`
runs alternate (A B A B …), so drifting clocks and neighbours on the host hit both alike.  Per run it records
ms_per_step, roofline.kernel_ms (the bound pass, or the fused compaction + bound pass), roofline.pass2.ms and
select_ms; the card's name, power limit and clocks are read once before and once after.  With --out, the last run of
each tree also writes its outputs (bench.py --dump-outputs) and the script reports whether freq, keep, kde_windows and
roh are identical.

The bound pass is reported against the bytes it has to read — the uncompacted rows, the piece maxima it writes and the
per-SNP tables — not bench.py's algorithmic_bytes_per_launch, which also counts the write of a compacted matrix.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys


def card():
    q = "name,power.limit,clocks.sm,clocks.mem,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def run(tree, steps, warmup, dump):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-configs", "--no-cpu"]
    if dump:
        cmd += ["--dump-outputs", dump]
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stderr[-2000:])
        raise SystemExit("bench.py failed in %s" % tree)
    line = json.loads([x for x in r.stdout.splitlines() if x.startswith("{")][-1])
    rf = line["roofline"]
    snps, n_ind, lk = line["config"]["snps"], line["config"]["individuals_per_gpu"], line["loci_used"]
    read_bytes = n_ind * snps / 4.0 + ((lk + 255) // 256) * n_ind * 4.0 + (lk / 16.0) * (16 + 4 + 16) + snps * 4.0
    return dict(ms_per_step=line["ms_per_step"], kernel_ms=rf["kernel_ms"], pass2_ms=rf["pass2"]["ms"],
                select_ms=rf["pass2"]["select_ms"], candidate_pair_fraction=rf["pass2"]["candidate_pair_fraction"],
                bound_read_gbs=read_bytes / (rf["kernel_ms"] / 1e3) / 1e9, read_bytes=read_bytes, roh=line["roh_found"])


def same_outputs(da, db):
    import numpy as np
    res = {}
    for name in ("freq", "keep", "kde_windows", "roh"):
        pa, pb = os.path.join(da, name + ".npy"), os.path.join(db, name + ".npy")
        if not (os.path.exists(pa) and os.path.exists(pb)):
            res[name] = "missing"
            continue
        a, b = np.load(pa), np.load(pb)
        res[name] = "identical" if a.shape == b.shape and np.array_equal(a, b, equal_nan=True) else "DIFFERENT"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="tree of the old build")
    ap.add_argument("--b", required=True, help="tree of the new build")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", help="directory for the outputs of the last run of each tree (a/, b/)")
    a = ap.parse_args()
    if a.runs < 3:
        ap.error("--runs must be at least 3")
    trees = {"a": os.path.abspath(a.a), "b": os.path.abspath(a.b)}
    rec = dict(card_before=card(), runs={"a": [], "b": []}, trees=trees)
    for i in range(a.runs):
        for k in ("a", "b"):
            dump = os.path.join(os.path.abspath(a.out), k) if (a.out and i == a.runs - 1) else None
            r = run(trees[k], a.steps, a.warmup, dump)
            rec["runs"][k].append(r)
            print(json.dumps(dict(tree=k, run=i, **r)), flush=True)
    rec["card_after"] = card()
    summ = {}
    for k in ("a", "b"):
        rs = rec["runs"][k]
        summ[k] = {f: dict(median=statistics.median(r[f] for r in rs), min=min(r[f] for r in rs), max=max(r[f] for r in rs))
                   for f in ("ms_per_step", "kernel_ms", "pass2_ms", "select_ms", "bound_read_gbs")}
    rec["summary"] = summ
    rec["ms_per_step_gain"] = summ["a"]["ms_per_step"]["median"] - summ["b"]["ms_per_step"]["median"]
    rec["ms_per_step_spread"] = max(summ[k]["ms_per_step"]["max"] - summ[k]["ms_per_step"]["min"] for k in ("a", "b"))
    if a.out:
        rec["outputs"] = same_outputs(os.path.join(a.out, "a"), os.path.join(a.out, "b"))
    print(json.dumps(dict(summary=rec["summary"], gain=rec["ms_per_step_gain"], spread=rec["ms_per_step_spread"],
                          outputs=rec.get("outputs"), card_before=rec["card_before"], card_after=rec["card_after"])), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "ab_step.json"), "w") as f:
            json.dump(rec, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
