#!/usr/bin/env python3
"""VCF ingest on the GPU:

1. the C++ driver, --freq-only wall time (best of 3) at 2,000 individuals x 20,000 SNPs (the shape of
   r04_bed_ingest.json's driver runs) from the same genotypes as tped (plain, gz) and as VCF (GT plain, GT BGZF,
   GT:AD:DP:GQ:PL BGZF); every run's .freq.gz must be identical;
2. the tokeniser kernel alone (torch.profiler, CUDA activities) at 2,000 x 600,000: put_vcf_text in 4,096-record blocks
   of GT-only text (one block's text, generated once, is uploaded for every block), as text bytes per second against
   the device-to-device copy peak measured in the same run (read + write bytes of a 4 GB copy / CUDA event time);
   also put_vcf_text + code_alleles wall time for the whole matrix.

    python tools/vcf_ingest_bench.py [n_ind] [n_snps] [cli_n_ind] [cli_n_snps] > out.json
"""
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from garlic_b200 import synth, vcf  # noqa: E402
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


def block_text(seed):
    """GT-only sample text of BLK records x N samples, single-digit indices, 2 % missing alleles."""
    rng = np.random.default_rng(seed)
    idx = (rng.random((BLK, N, 2)) < rng.uniform(0.05, 0.95, (BLK, 1, 1))).astype(np.uint8)
    ch = (idx + ord("0")).astype(np.uint8)
    ch[rng.random((BLK, N, 2)) < 0.02] = ord(".")
    b = np.empty((BLK, N, 4), np.uint8)
    b[:, :, 0], b[:, :, 1], b[:, :, 2], b[:, :, 3] = ch[:, :, 0], ord("/"), ch[:, :, 1], ord("\t")
    rows = b.reshape(BLK, N * 4)[:, :-1]
    off = np.arange(BLK + 1, dtype=np.int64) * rows.shape[1]
    return rows.tobytes(), off


def device_path():
    from torch.profiler import ProfilerActivity, profile
    text, off = block_text(1)
    g = GarlicGPU(0)
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 500
    co = np.array([0, L0], np.int64)

    def run():
        g.set_shape(N, L0, co, pos)
        for s0 in range(0, L0, BLK):
            n = min(BLK, L0 - s0)
            nc, _, bad = g.put_vcf_text(text, off[:n + 1], s0)
            assert (nc == N).all() and (bad < 0).all()
        g.code_alleles()

    run()
    walls = []
    for _ in range(3):
        t0 = time.perf_counter()
        run()
        walls.append(time.perf_counter() - t0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
    res = dict(put_vcf_text_code_alleles_s=round(min(walls), 3))
    for e in prof.key_averages():
        if "tokenize_vcf_kernel" in e.key:
            total = e.device_time_total / 1e6                    # s over all blocks
            nbytes = sum(int(off[min(BLK, L0 - s0)]) for s0 in range(0, L0, BLK))
            res.update(tokenize_vcf_kernel_total_ms=round(total * 1e3, 3), tokenize_vcf_launches=e.count,
                       text_bytes=nbytes, tokenize_text_GBps=round(nbytes / total / 1e9, 1))
    g.close()
    return res


def driver():
    ds = synth.make_dataset(seed=3, n_ind=CLI_N, chr_sizes=(CLI_L // 2, CLI_L - CLI_L // 2))
    v = vcf.from_dataset(ds, seed=4)
    res = dict(cli_n_ind=CLI_N, cli_n_snps=CLI_L)
    with tempfile.TemporaryDirectory() as tmp:
        paths = ds.write(tmp)
        with open(paths["tped"], "rb") as fi, gzip.open(paths["tped"] + ".gz", "wb", compresslevel=1) as fo:
            shutil.copyfileobj(fi, fo)
        files = {"vcf_gt_plain": vcf.write_vcf(os.path.join(tmp, "gt.vcf"), v),
                 "vcf_gt_bgzf": vcf.write_vcf(os.path.join(tmp, "gt.vcf.gz"), v, compress="bgzf"),
                 "vcf_gt_ad_dp_gq_pl_bgzf": vcf.write_vcf(os.path.join(tmp, "full.vcf.gz"), v, "GT:AD:DP:GQ:PL",
                                                           compress="bgzf")}
        runs = {"tped_plain": ["--tped", paths["tped"], "--tfam", paths["tfam"]],
                "tped_gz": ["--tped", paths["tped"] + ".gz", "--tfam", paths["tfam"]]}
        for k, p in files.items():
            runs[k] = ["--vcf", p, "--tfam", paths["tfam"]]
            res[k + "_mb"] = round(os.path.getsize(p) / 1e6, 2)
        res["tped_plain_mb"] = round(os.path.getsize(paths["tped"]) / 1e6, 2)
        res["tped_gz_mb"] = round(os.path.getsize(paths["tped"] + ".gz") / 1e6, 2)
        common = ["--freq-only", "--centromere", paths["centromere"], "--winsize", "50", "--error", "0.001"]
        outs = {}
        for name, argv in runs.items():
            best = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                r = subprocess.run([BIN] + argv + common + ["--out", os.path.join(tmp, name)], capture_output=True, text=True)
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
    if "tokenize_text_GBps" in out:
        out["tokenize_fraction_of_copy_peak"] = round(out["tokenize_text_GBps"] * 1e9 / (out["d2d_copy_peak_TBps"] * 1e12), 3)
    out.update(driver())
    print(json.dumps(out))
