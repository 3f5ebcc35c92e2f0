#!/usr/bin/env python3
"""Cost of the call filter (--vcf-min-gq / --vcf-min-dp) on the GPU:

1. the kernels alone (torch.profiler, CUDA activities) at 2,000 individuals x 600,000 records, in 4,096-record blocks
   (one block, generated once, is uploaded for every block): tokenize_vcf_kernel on GT:AD:DP:GQ:PL text, and
   decode_bcf_gt_kernel on int8 GT vectors with int8 GQ and DP vectors, each with the filter off (put_vcf_text /
   put_bcf_gt) and with both thresholds on (the _filtered puts, GQ >= 20 and DP >= 10);
2. the C++ driver's --freq-only wall time (best of 3) at 2,000 x 20,000 on the same data as a BGZF VCF and a BGZF
   BCF, without and with --vcf-min-gq 20 --vcf-min-dp 10.

    python tools/call_filter_bench.py [n_ind] [n_snps] [cli_n_ind] [cli_n_snps] > out.json
"""
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from garlic_b200 import bcf, synth, vcf  # noqa: E402
from garlic_b200.api import GarlicGPU  # noqa: E402

BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")
N = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
L0 = int(sys.argv[2]) if len(sys.argv) > 2 else 600000
CLI_N = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
CLI_L = int(sys.argv[4]) if len(sys.argv) > 4 else 20000
BLK = 4096
MIN_GQ, MIN_DP = 20, 10


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def block(seed):
    """BLK records x N samples: allele indices (2 % missing), GQ in [0, 99], DP in [0, 49]."""
    rng = np.random.default_rng(seed)
    idx = (rng.random((BLK, N, 2)) < rng.uniform(0.05, 0.95, (BLK, 1, 1))).astype(np.uint8)
    idx[rng.random((BLK, N, 2)) < 0.02] = vcf.MISSING
    return idx, rng.integers(0, 100, (BLK, N)), rng.integers(0, 50, (BLK, N))


def vcf_block(idx, gq, dp):
    """GT:AD:DP:GQ:PL sample text, every column "a/b:3,3:DD:GG:0,20,20"."""
    ch = np.where(idx == vcf.MISSING, ord("."), idx + ord("0")).astype(np.uint8)
    c = np.empty((BLK, N, 22), np.uint8)
    c[:] = np.frombuffer(b"0/0:3,3:00:00:0,20,20\t", np.uint8)
    c[:, :, 0], c[:, :, 2] = ch[:, :, 0], ch[:, :, 1]
    c[:, :, 8], c[:, :, 9] = dp // 10 + ord("0"), dp % 10 + ord("0")
    c[:, :, 11], c[:, :, 12] = gq // 10 + ord("0"), gq % 10 + ord("0")
    rows = c.reshape(BLK, N * 22)[:, :-1]
    return rows.tobytes(), np.arange(BLK + 1, dtype=np.int64) * rows.shape[1], np.tile([[3, 2]], (BLK, 1)).astype(np.int32)


def bcf_block(idx, gq, dp):
    gt = np.where(idx == vcf.MISSING, 0, (idx.astype(np.int64) + 1) << 1).astype(np.int8).reshape(BLK, -1)
    pad = (-gt.shape[1]) % 4
    gt = np.pad(gt, ((0, 0), (0, pad)))
    vpad = (-N) % 4
    fv = np.concatenate([np.pad(gq.astype(np.int8), ((0, 0), (0, vpad))), np.pad(dp.astype(np.int8), ((0, 0), (0, vpad)))], 1)
    span = fv.shape[1]
    return (gt.tobytes(), np.arange(BLK + 1, dtype=np.int64) * gt.shape[1], np.full(BLK, 0x21, np.uint8),
            fv.tobytes(), np.arange(BLK + 1, dtype=np.int64) * span,
            np.tile([[0, span // 2]], (BLK, 1)).astype(np.int32), np.full((BLK, 2), 0x11, np.uint8))


def kernels():
    from torch.profiler import ProfilerActivity, profile
    idx, gq, dp = block(1)
    text, off, fk = vcf_block(idx, gq, dp)
    gt, rec_off, gt_type, fv, fv_off, fv_pos, fv_type = bcf_block(idx, gq, dp)
    g = GarlicGPU(0)
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 500
    co = np.array([0, L0], np.int64)

    def run(kind, on):
        g.set_shape(N, L0, co, pos)
        if on:
            g.set_call_filter(MIN_GQ, MIN_DP)
        for s0 in range(0, L0, BLK):
            n = min(BLK, L0 - s0)
            if kind == "vcf" and on:
                assert (g.put_vcf_text_filtered(text, off[:n + 1], fk[:n], s0)[3] < 0).all()
            elif kind == "vcf":
                g.put_vcf_text(text, off[:n + 1], s0)
            elif on:
                assert (g.put_bcf_gt_filtered(gt, rec_off[:n + 1], gt_type[:n], N, fv, fv_off[:n + 1], fv_pos[:n], fv_type[:n], s0)[2] < 0).all()
            else:
                g.put_bcf_gt(gt, rec_off[:n + 1], gt_type[:n], N, s0)

    res = {}
    kname = {"vcf": "tokenize_vcf_kernel", "bcf": "decode_bcf_gt_kernel"}
    for rep in range(2):                    # two alternating rounds: the spread between them is the run-to-run noise
        for kind in ("vcf", "bcf"):
            for on in (False, True):
                run(kind, on)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    run(kind, on)
                t = sum(e.device_time_total for e in prof.key_averages() if kname[kind] in e.key) / 1e3
                res.setdefault("%s_%s_ms" % (kname[kind], "on" if on else "off"), []).append(round(t, 3))
                if on:
                    res["%s_calls_set_missing" % kind] = g.calls_set_missing()
    g.close()
    return res


def driver():
    ds = synth.make_dataset(seed=3, n_ind=CLI_N, chr_sizes=(CLI_L // 2, CLI_L - CLI_L // 2))
    v = vcf.from_dataset(ds, seed=4)
    rng = np.random.default_rng(5)
    v.gq = rng.integers(0, 100, v.idx.shape[:2]).astype(float)
    v.dp = rng.integers(0, 50, v.idx.shape[:2]).astype(float)
    res = dict(cli_n_ind=CLI_N, cli_n_snps=CLI_L)
    with tempfile.TemporaryDirectory() as tmp:
        paths = ds.write(tmp)
        files = {"vcf_bgzf": vcf.write_vcf(os.path.join(tmp, "x.vcf.gz"), v, "GT:AD:DP:GQ:PL", compress="bgzf"),
                 "bcf_bgzf": bcf.write_bcf(os.path.join(tmp, "x.bcf"), v, "GT:AD:DP:GQ:PL")}
        common = ["--freq-only", "--centromere", paths["centromere"], "--winsize", "50", "--error", "0.001"]
        flags = {"off": [], "on": ["--vcf-min-gq", str(MIN_GQ), "--vcf-min-dp", str(MIN_DP)]}
        for rep in range(3):
            for name, p in files.items():
                for k, f in flags.items():
                    t0 = time.perf_counter()
                    r = subprocess.run([BIN, "--vcf", p] + common + f + ["--out", os.path.join(tmp, name + k)],
                                       capture_output=True, text=True)
                    dt = time.perf_counter() - t0
                    assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
                    key = "%s_freq_only_%s_s" % (name, k)
                    res[key] = round(min(res.get(key, 1e9), dt), 3)
    return res


if __name__ == "__main__":
    out = dict(card=card(), n_ind=N, n_snps=L0, min_gq=MIN_GQ, min_dp=MIN_DP)
    out.update(kernels())
    out.update(driver())
    print(json.dumps(out))
