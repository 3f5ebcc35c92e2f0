#!/usr/bin/env python3
"""Column selection (garlic_gpu_select_columns) on the GPU, kernels alone (torch.profiler, CUDA activities):
1. decode_bcf_gt_kernel at N_input x L0 int8 GT payloads (one numpy block of 4,096 records uploaded for every block):
   a handle of the first N_input/2 samples (range form) against a handle of every other sample (selected form); both
   read every sample and write N_input/2;
2. bed_select_kernel at the same shape: whole .bed rows on the device (put_bed_dev, one 4,096-row block reused), every
   other column selected; bytes moved = ceil(N_input/4) read + ceil(N_input/8) written per SNP, against the
   device-to-device copy peak measured in the same run (read + write bytes of a 4 GB copy / CUDA event time).
    python tools/select_bench.py [n_input] [n_snps] > out.json
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from garlic_b200.api import GarlicGPU  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
L0 = int(sys.argv[2]) if len(sys.argv) > 2 else 600000
BLK = 4096


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
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


def kernel_ms(prof, name):
    tot, n = 0.0, 0
    for e in prof.key_averages():
        if name in e.key:
            tot += e.device_time_total / 1e3
            n += e.count
    return round(tot, 3), n


def shape(g, n):
    g.set_shape(n, L0, np.array([0, L0], np.int64), np.arange(1, L0 + 1, dtype=np.int32) * 500)


def bcf_forms():
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(1)
    idx = (rng.random((BLK, N, 2)) < rng.uniform(0.05, 0.95, (BLK, 1, 1))).astype(np.int8)
    rows = ((idx + 1) << 1).reshape(BLK, 2 * N)
    rows = np.concatenate([rows, np.zeros((BLK, -rows.shape[1] % 4), np.int8)], 1)
    gt, off, types = rows.tobytes(), np.arange(BLK + 1, dtype=np.int64) * rows.shape[1], np.full(BLK, 0x21, np.uint8)
    half = N // 2
    res = {}
    for form, cols in [("range", None), ("selected", np.arange(0, N, 2)[:half])]:
        g = GarlicGPU(0)

        def run():
            shape(g, half)
            if cols is not None:
                g.select_columns(cols, N)
            for s0 in range(0, L0, BLK):
                n = min(BLK, L0 - s0)
                g.put_bcf_gt(gt, off[:n + 1], types[:n], N, s0)
            g.sync()
        run()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run()
        ms, launches = kernel_ms(prof, "decode_bcf_gt_kernel")
        res["decode_bcf_gt_%s_ms" % form] = ms
        res["decode_bcf_gt_%s_launches" % form] = launches
        g.close()
    return res


def bed_select():
    import torch
    from torch.profiler import ProfilerActivity, profile
    stride = (N + 3) // 4
    rows = torch.from_numpy(np.random.default_rng(2).integers(0, 256, (BLK, stride), dtype=np.uint8)).cuda()
    torch.cuda.synchronize()
    cols = np.arange(0, N, 2)
    g = GarlicGPU(0)

    def run():
        shape(g, len(cols))
        g.select_columns(cols, N)
        for s0 in range(0, L0, BLK):
            g.put_bed_dev(rows.data_ptr(), stride, min(BLK, L0 - s0), s0)
        g.sync()
    run()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
    ms, launches = kernel_ms(prof, "bed_select_kernel")
    nbytes = L0 * (stride + (len(cols) + 3) // 4)
    g.close()
    return dict(bed_select_ms=ms, bed_select_launches=launches, bed_select_bytes=nbytes,
                bed_select_GBps=round(nbytes / (ms * 1e-3) / 1e9, 1))


if __name__ == "__main__":
    out = dict(card=card(), n_input=N, n_snps=L0)
    out["d2d_copy_peak_TBps"] = round(copy_peak() / 1e12, 2)
    out.update(bcf_forms())
    out.update(bed_select())
    out["bed_select_fraction_of_copy_peak"] = round(out["bed_select_GBps"] * 1e9 / (out["d2d_copy_peak_TBps"] * 1e12), 3)
    print(json.dumps(out))
