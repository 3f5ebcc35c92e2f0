#!/usr/bin/env python3
"""PLINK .bed ingest on the GPU, at the C2 shape by default (2,000 individuals x 600,000 SNPs, one rank):

1. device path: put_bed (4,096-SNP blocks) + code_alleles against put_packed + count_packed of the same genotypes, host
   clock around calls that end synchronised, and the bytes each copies host-to-device;
2. the kernels alone (torch.profiler, CUDA activities): bed_transpose_kernel and bed_count_kernel, their achieved
   bandwidth (bytes the algorithm must move / kernel time) against the 6.56 TB/s copy peak measured on this B200
   (profiles/README.md);
3. the C++ driver: --bfile --freq-only against --tped --freq-only on the same data, plain and gz tped (like
   tools/ingest_bench.py), at a smaller shape (text generation dominates otherwise).

    python tools/bed_ingest_bench.py [n_ind] [n_snps] [cli_n_ind] [cli_n_snps] > out.json
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
from garlic_b200 import plink  # noqa: E402
from garlic_b200.api import GarlicGPU  # noqa: E402

BIN = os.path.join(ROOT, "garlic_b200", "host", "garlic_b200")
COPY_PEAK = 6.56e12
N = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
L0 = int(sys.argv[2]) if len(sys.argv) > 2 else 600000
CLI_N = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
CLI_L = int(sys.argv[4]) if len(sys.argv) > 4 else 20000
REPS = 5


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def codes_rows(seed, n, L):
    rng = np.random.default_rng(seed)
    p = rng.uniform(0.05, 0.95, L).astype(np.float32)
    out = np.empty((L, (n + 3) // 4), np.uint8)
    for s0 in range(0, L, 20000):
        pp = p[s0:s0 + 20000, None]
        g = (rng.random((len(pp), n), np.float32) < pp).astype(np.uint8) + (rng.random((len(pp), n), np.float32) < pp)
        c = np.choose(g, [plink.HOM_A1, plink.HET, plink.HOM_A2]).astype(np.uint8)
        c[rng.random(c.shape, np.float32) < 0.01] = plink.MISSING
        out[s0:s0 + 20000] = plink.rows_from_codes(c)
    return out


def device_path(rows):
    import torch
    g = GarlicGPU(0)
    pos = np.arange(1, L0 + 1, dtype=np.int32) * 500
    co = np.array([0, L0], np.int64)
    packed = None
    res = {}
    host_rows = g.host_array(rows.size, np.uint8).reshape(rows.shape)
    host_rows[:] = rows
    t_bed, t_packed = [], []
    for rep in range(REPS + 1):
        g.set_shape(N, L0, co, pos)
        g.sync()
        t0 = time.perf_counter()
        for s0 in range(0, L0, 4096):
            g.put_bed(host_rows[s0:s0 + 4096], s0)
        g.code_alleles()
        t_bed.append(time.perf_counter() - t0)
        if packed is None:
            packed = g.host_array(N * ((L0 + 3) // 4), np.uint8).reshape(N, -1)
            packed[:] = g.get_genotypes(False)
        g.set_shape(N, L0, co, pos)
        g.sync()
        t0 = time.perf_counter()
        g.put_packed(packed)
        g.count_packed()
        g.sync()
        t_packed.append(time.perf_counter() - t0)
    res["put_bed_code_alleles_ms"] = round(1e3 * float(np.median(t_bed[1:])), 3)
    res["put_packed_count_packed_ms"] = round(1e3 * float(np.median(t_packed[1:])), 3)
    width = (N + 3) // 4
    res["h2d_bytes_put_bed"] = L0 * width
    res["h2d_bytes_put_packed"] = N * ((L0 + 3) // 4)
    # kernels alone: the rows already on the device (put_bed_dev), torch.profiler around code_alleles
    d_rows = torch.from_numpy(rows).cuda()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for rep in range(REPS):
            g.set_shape(N, L0, co, pos)
            g.put_bed_dev(d_rows.data_ptr(), width, L0, 0)
            g.code_alleles()
    times = {}
    for e in prof.key_averages():
        for k in ("bed_transpose_kernel", "bed_count_kernel", "bed_fix_kernel"):
            if k in e.key:
                times[k] = e.device_time_total / max(1, e.count) / 1e3       # ms per launch
    staged = L0 * ((width + 31) // 32 * 32)
    out_bytes = N * ((L0 + 31) // 32) * 8
    res["kernel_ms"] = {k: round(v, 4) for k, v in times.items()}
    if "bed_transpose_kernel" in times:
        bw = (staged + out_bytes) / (times["bed_transpose_kernel"] * 1e-3)
        res["transpose_bytes"] = staged + out_bytes
        res["transpose_TBps"] = round(bw / 1e12, 3)
        res["transpose_fraction_of_copy_peak"] = round(bw / COPY_PEAK, 3)
    if "bed_count_kernel" in times:
        bw = staged / (times["bed_count_kernel"] * 1e-3)
        res["count_TBps"] = round(bw / 1e12, 3)
        res["count_fraction_of_copy_peak"] = round(bw / COPY_PEAK, 3)
    g.close()
    return res


def driver():
    rows = codes_rows(2, CLI_N, CLI_L)
    codes = plink.codes_from_rows(rows, CLI_N)
    a1, a2 = ["A"] * CLI_L, ["G"] * CLI_L
    bim = plink.Bim(chr=["1"] * CLI_L, ids=["rs%d" % i for i in range(CLI_L)], cm=["0"] * CLI_L,
                    bp=np.arange(CLI_L, dtype=np.int32) * 500 + 1000, a1=a1, a2=a2)
    res = dict(cli_n_ind=CLI_N, cli_n_snps=CLI_L)
    with tempfile.TemporaryDirectory() as tmp:
        prefix = plink.write_fileset(os.path.join(tmp, "s"), codes, bim, [("POP", "ind%d" % i) for i in range(CLI_N)])
        tped, _ = plink.write_tped(prefix, plink.read_fileset(prefix))
        with open(tped, "rb") as fi, gzip.open(tped + ".gz", "wb", compresslevel=1) as fo:
            fo.write(fi.read())
        res["bed_mb"] = round(os.path.getsize(prefix + ".bed") / 1e6, 2)
        res["tped_mb"] = round(os.path.getsize(tped) / 1e6, 2)
        common = ["--freq-only", "--build", "hg19", "--winsize", "50", "--error", "0.001"]
        runs = {"bfile": ["--bfile", prefix], "tped_plain": ["--tped", tped, "--tfam", prefix + ".tfam"],
                "tped_gz": ["--tped", tped + ".gz", "--tfam", prefix + ".tfam"]}
        outs = {}
        for name, argv in runs.items():
            best = 1e9
            for _ in range(2):
                t0 = time.perf_counter()
                r = subprocess.run([BIN] + argv + common + ["--out", os.path.join(tmp, name)], capture_output=True, text=True)
                best = min(best, time.perf_counter() - t0)
                assert r.returncode == 0, r.stdout[-500:] + r.stderr[-500:]
            res["%s_freq_only_s" % name] = round(best, 3)
            outs[name] = gzip.open(os.path.join(tmp, name + ".freq.gz"), "rt").read()
        res["freq_gz_identical"] = outs["bfile"] == outs["tped_plain"] == outs["tped_gz"]
    return res


if __name__ == "__main__":
    out = dict(card=card(), n_ind=N, n_snps=L0, bed_mb=round(L0 * ((N + 3) // 4) / 1e6, 1))
    out.update(device_path(codes_rows(1, N, L0)))
    out.update(driver())
    print(json.dumps(out))
