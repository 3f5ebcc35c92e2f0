#!/usr/bin/env python3
"""BCF ingest on the GPU:

1. the C++ driver, --freq-only wall time (best of 3) at 2,000 individuals x 20,000 SNPs (the shape of
   r05_vcf_ingest.json's driver runs) from the same genotypes as VCF (GT plain, GT BGZF) and as BCF (GT BGZF,
   GT:AD:DP:GQ:PL BGZF, GT uncompressed); every run's .freq.gz must be identical;
2. the decoder kernel alone (torch.profiler, CUDA activities) at 2,000 x 600,000: put_bcf_gt in 4,096-record blocks of
   int8 GT payloads built in numpy (one block, generated once, is uploaded for every block), as bytes moved (2 B read +
   2 B written per genotype) per second against the device-to-device copy peak measured in the same run (read + write
   bytes of a 4 GB copy / CUDA event time); also put_bcf_gt + code_alleles wall time for the whole matrix.

    python tools/bcf_ingest_bench.py [n_ind] [n_snps] [cli_n_ind] [cli_n_snps] > out.json
"""
import gzip
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


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def copy_peak():
    import torch
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 10 * 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3)


def block_payload(seed):
    """int8 GT payloads of BLK records x N samples (count 2): indices 0 / 1, 2 % missing alleles, unphased."""
    rng = np.random.default_rng(seed)
    idx = (rng.random((BLK, N, 2)) < rng.uniform(0.05, 0.95, (BLK, 1, 1))).astype(np.int8)
    vals = (idx + 1) << 1
    vals[rng.random((BLK, N, 2)) < 0.02] = 0
    rows = vals.reshape(BLK, 2 * N)
    pad = -rows.shape[1] % 4
    rows = np.concatenate([rows, np.zeros((BLK, pad), np.int8)], 1)
    off = np.arange(BLK + 1, dtype=np.int64) * rows.shape[1]
    return rows.tobytes(), off, np.full(BLK, 0x21, np.uint8)


def device_path():
    from torch.profiler import ProfilerActivity, profile
    gt, off, types = block_payload(1)
    g = GarlicGPU(0)
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 500
    co = np.array([0, L0], np.int64)

    def run():
        g.set_shape(N, L0, co, pos)
        for s0 in range(0, L0, BLK):
            n = min(BLK, L0 - s0)
            _, bad = g.put_bcf_gt(gt, off[:n + 1], types[:n], N, s0)
            assert (bad < 0).all()
        g.code_alleles()

    run()
    walls = []
    for _ in range(3):
        t0 = time.perf_counter()
        run()
        walls.append(time.perf_counter() - t0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
    res = dict(put_bcf_gt_code_alleles_s=round(min(walls), 3))
    for e in prof.key_averages():
        if "decode_bcf_gt_kernel" in e.key:
            total = e.device_time_total / 1e6                    # s over all blocks
            nbytes = 2 * L0 * N + 2 * L0 * N                     # GT values read + allele index bytes written
            res.update(decode_bcf_gt_kernel_total_ms=round(total * 1e3, 3), decode_bcf_gt_launches=e.count,
                       bytes_moved=nbytes, decode_GBps=round(nbytes / total / 1e9, 1))
    g.close()
    return res


def driver():
    ds = synth.make_dataset(seed=3, n_ind=CLI_N, chr_sizes=(CLI_L // 2, CLI_L - CLI_L // 2))
    v = vcf.from_dataset(ds, seed=4)
    res = dict(cli_n_ind=CLI_N, cli_n_snps=CLI_L)
    with tempfile.TemporaryDirectory() as tmp:
        paths = ds.write(tmp)
        files = {"vcf_gt_plain": vcf.write_vcf(os.path.join(tmp, "gt.vcf"), v),
                 "vcf_gt_bgzf": vcf.write_vcf(os.path.join(tmp, "gt.vcf.gz"), v, compress="bgzf"),
                 "bcf_gt_bgzf": bcf.write_bcf(os.path.join(tmp, "gt.bcf"), v),
                 "bcf_gt_ad_dp_gq_pl_bgzf": bcf.write_bcf(os.path.join(tmp, "full.bcf"), v, "GT:AD:DP:GQ:PL"),
                 "bcf_gt_uncompressed": bcf.write_bcf(os.path.join(tmp, "gt.u.bcf"), v, compress=None)}
        common = ["--freq-only", "--centromere", paths["centromere"], "--winsize", "50", "--error", "0.001"]
        outs = {}
        for name, p in files.items():
            res[name + "_mb"] = round(os.path.getsize(p) / 1e6, 2)
            best = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                r = subprocess.run([BIN, "--vcf", p, "--tfam", paths["tfam"]] + common + ["--out", os.path.join(tmp, name)],
                                   capture_output=True, text=True)
                best = min(best, time.perf_counter() - t0)
                assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
            res["%s_freq_only_s" % name] = round(best, 3)
            outs[name] = gzip.open(os.path.join(tmp, name + ".freq.gz"), "rt").read()
        res["freq_gz_identical"] = len(set(outs.values())) == 1
    return res


if __name__ == "__main__":
    out = dict(card=card(), n_ind=N, n_snps=L0)
    out["d2d_copy_peak_TBps"] = round(copy_peak() / 1e12, 2)
    out.update(device_path())
    if "decode_GBps" in out:
        out["decode_fraction_of_copy_peak"] = round(out["decode_GBps"] * 1e9 / (out["d2d_copy_peak_TBps"] * 1e12), 3)
    out.update(driver())
    print(json.dumps(out))
