#!/usr/bin/env python3
"""bench.py — GARLIC LOD → ROH hot path on B200: individual-windows/s (BASELINE.json metric).

Own arm (default):  python bench.py --gpus N --steps K --warmup W
    Workload = BASELINE.json configs[1]: synthetic array, 2,000 individuals x 600k SNPs (22 autosomes,
    hg19 centromeres, 0.1 % gaps > 200 kb), --winsize 50, --error 0.001, unweighted LOD, --overlap-frac 0.25,
    fixed --lod-cutoff (host KDE excluded, SURVEY §8d).  One step = one pass of the hot path over the batch:
    [H2D of the packed genotypes, e2e only] -> K2 allele/missingness counts -> freq + monomorphic filter (N>1: the
    counters of all ranks are summed, and freq / keep evaluated, by one kernel over NVLink peer memory inside the library)
    -> keep-mask scan, K3's plan -> K4 LOD table, gap bit map -> K5 pass 1 (thinned windows of the 20 KDE individuals ->
    host of rank 0; N>1: all-gather) beside K3 fused with the pruning bound of pass 2 -> K5 pass 2 (candidate selection,
    windows -> cutoff -> coverage -> ROH, fused) -> ROH records to the host.  Sharded by individual: every rank holds
    2,000 individuals (weak scaling).
    `value` has the packed matrix resident in HBM; `e2e` goes through the C ABI with pinned HOST buffers.
    --dump-outputs DIR writes what the last resident step returned (freq, keep mask, thinned KDE windows, ROH records)
    as DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output.  Under N ranks every rank
    writes its ROH records as roh_rank<r>.npy, with individuals counted within the rank.

Reference arm:      python bench.py --impl reference --gpus N --steps K --warmup W
    The reference's own calcLODWindows + assembleROHWindows (oracle/_ref/ref_driver, compiled from
    /root/reference/src) on the host cores, one process per core, each on a bounded sample of the same
    workload (same SNPs, frequencies and genotypes).  Falls back to the C port (oracle/liboracle.so).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "individual_windows_per_sec"
UNIT = "individual-windows/s"
CFG = dict(n_ind=2000, n_loci=600_000, winsize=50, error=0.001, cutoff=2.0, overlap_frac=0.25, max_gap=200000,
           kde_subsample=20, seed=2)
WORKLOAD = "configs[1]: synthetic array 2000 ind x 600k SNPs, 22 autosomes, --winsize 50 --error 0.001 unweighted"


# ------------------------------------------------------------------------------------------------
# synthetic workload (device-side generation with torch: plumbing only)
# ------------------------------------------------------------------------------------------------
def make_rows_torch(torch, dev, n_ind, L, seed, ind_seed, row_bytes, chunk=250):
    """Packed 2-bit rows uint8[n_ind, row_bytes] on `dev`: Binomial(2,p_l) genotypes, 2 % monomorphic columns,
    5 planted homozygous tracts (200-2000 SNPs) per individual, 0.5 % missing (SURVEY §8d)."""
    gp = torch.Generator(device=dev)
    gp.manual_seed(seed)                       # per-SNP frequencies: identical on every rank
    p = torch.rand(L, generator=gp, device=dev) * 0.9 + 0.05
    mono = torch.rand(L, generator=gp, device=dev) < 0.02
    p = torch.where(mono, torch.zeros_like(p), p)
    gi = torch.Generator(device=dev)
    gi.manual_seed(ind_seed)                   # genotypes: differ per rank
    rows = torch.full((n_ind, row_bytes), 0xFF, dtype=torch.uint8, device=dev)
    ar = torch.arange(L, device=dev)
    L4 = (L + 3) // 4
    for i0 in range(0, n_ind, chunk):
        n = min(chunk, n_ind - i0)
        h0 = torch.rand((n, L), generator=gi, device=dev) < p
        h1 = torch.rand((n, L), generator=gi, device=dev) < p
        for _ in range(5):
            ln = torch.randint(200, 2000, (n, 1), generator=gi, device=dev)
            st = (torch.rand((n, 1), generator=gi, device=dev) * (L - 2000)).long()
            m = (ar >= st) & (ar < st + ln)
            h1 = torch.where(m, h0, h1)
        g = h0.to(torch.uint8) + h1.to(torch.uint8)
        miss = torch.rand((n, L), generator=gi, device=dev) < 0.005
        g = torch.where(miss, torch.full_like(g, 3), g)
        if L % 4:
            g = torch.nn.functional.pad(g, (0, 4 - L % 4), value=3)
        q = g.view(n, L4, 4)
        rows[i0:i0 + n, :L4] = q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)
    return rows


def unpack_rows(rows_u8, L):
    b = rows_u8[:, :(L + 3) // 4]
    out = np.empty((b.shape[0], b.shape[1], 4), np.uint8)
    for k in range(4):
        out[:, :, k] = (b >> (2 * k)) & 3
    return out.reshape(b.shape[0], -1)[:, :L]


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
_SAMPLER_SRC = r"""
import json, sys, time
import pynvml as nv
nv.nvmlInit()
hs = [nv.nvmlDeviceGetHandleByIndex(int(i)) for i in sys.argv[1:]]
mx = float(nv.nvmlDeviceGetMaxClockInfo(hs[0], nv.NVML_CLOCK_SM))
sys.stdout.write("ready\n"); sys.stdout.flush()
sys.stdin.readline()                      # "go"
import select
sm, mask = [], 0
while True:
    for h in hs:
        try:
            sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            pass
    if select.select([sys.stdin], [], [], 0.001)[0]:
        break
print(json.dumps(dict(sm=sm, mask=mask, mx=mx)))
"""


class ClockSampler:
    """Polls NVML (SM clock, clocks-event reasons) about every millisecond while the timed region runs: the region lasts
    tens of milliseconds, too short for `nvidia-smi -lms`.  The polling runs in a helper PROCESS — a thread inside rank 0
    would take the interpreter lock from the thread that drives the GPU some sixteen times per millisecond when it watches
    eight GPUs, and every rank waits for rank 0 at the next exchange.  Falls back to one nvidia-smi query."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20))

    def __init__(self, index, n_devices=1):
        """index: first local GPU; n_devices: how many consecutive local GPUs the helper watches — under torchrun rank 0
        starts one helper for every GPU of the job."""
        self.index, self.p = index, None
        try:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            ids = [int(x) for x in vis.split(",")] if vis and all(x.strip().isdigit() for x in vis.split(",")) else None
            phys = [str(ids[index + k] if ids else index + k) for k in range(n_devices)]
            self.p = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC] + phys, stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            if self.p.stdout.readline().strip() != "ready":
                raise RuntimeError("sampler did not start")
        except Exception:
            if self.p is not None:
                self.p.kill()
            self.p = None

    def start(self):
        if self.p is None:
            return
        self.p.stdin.write("go\n")
        self.p.stdin.flush()

    def stop(self):
        if self.p is not None:
            try:
                self.p.stdin.write("stop\n")
                self.p.stdin.flush()
                r = json.loads(self.p.stdout.readline())
                self.p.wait(timeout=5)
                reasons = sorted(nm for nm, bit in self.REASONS if r["mask"] & bit)
                return dict(sm_mhz=float(np.median(r["sm"])) if r["sm"] else None, sm_max_mhz=r["mx"], reasons=reasons,
                            samples=len(r["sm"]), how="NVML polled about every ms by a helper process during the timed region")
            except Exception:
                self.p.kill()
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
            a, b = [float(x) for x in out.strip().split(",")]
            return dict(sm_mhz=a, sm_max_mhz=b, reasons=[], samples=1, how="one nvidia-smi query after the region")
        except Exception:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml and nvidia-smi unavailable"], samples=0)


def bind_near_gpu(index):
    """Run this rank on the host cores next to its GPU (NVML's ideal CPU set) before any page-locked buffer is
    allocated: with 8 ranks on a two-socket host, pinned buffers on the wrong socket make every H2D copy cross it."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        ids = [int(x) for x in vis.split(",")] if vis and all(x.strip().isdigit() for x in vis.split(",")) else None
        h = pynvml.nvmlDeviceGetHandleByIndex(ids[index] if ids else index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1 and 64 * w + b < n_cpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


# ------------------------------------------------------------------------------------------------
# CPU arm helpers (the checker / baseline; never on the product path)
# ------------------------------------------------------------------------------------------------
def cpu_chroms(codes_ind_major, keep, freq0, pos0, chr_off0, names, cens):
    """Filtered per-chromosome SNP-major arrays for oracle/refdrv from the bench's own tables."""
    chroms = []
    for c, nm in enumerate(names):
        lo, hi = int(chr_off0[c]), int(chr_off0[c + 1])
        k = keep[lo:hi]
        chroms.append(dict(name="chr" + nm, cen=cens["chr" + nm], pos=np.ascontiguousarray(pos0[lo:hi][k]),
                           freq=np.ascontiguousarray(freq0[lo:hi][k]), gpos=None, gl=None,
                           geno=np.ascontiguousarray(codes_ind_major[:, lo:hi][:, k].T.astype(np.int8))))
    return chroms


class CpuSample:
    """The reference functions (oracle/_ref/ref_driver) or, if that binary is absent, the C port
    (oracle/liboracle.so) on `n` individuals split over `procs` processes / threads."""

    def __init__(self, chroms, n, W, error, cutoff, ov, max_gap, procs):
        from oracle import refdrv
        self.refdrv, self.chroms, self.n, self.W = refdrv, chroms, n, W
        self.args = (error, cutoff, ov, max_gap)
        self.units = n * sum(max(0, len(ch["pos"]) - W + 1) for ch in chroms)
        self.bounds = np.linspace(0, n, procs + 1).astype(int)
        self.procs = procs
        self.kind = "reference" if refdrv.available() else "port"
        self.tmp = None
        if self.kind == "reference":
            self.tmp = tempfile.TemporaryDirectory()
            self.jobs = []
            for p in range(procs):
                a, b = int(self.bounds[p]), int(self.bounds[p + 1])
                if b <= a:
                    continue
                sub = [dict(ch, geno=np.ascontiguousarray(ch["geno"][:, a:b])) for ch in chroms]
                pin, pout = os.path.join(self.tmp.name, "in%d.bin" % p), os.path.join(self.tmp.name, "out%d.bin" % p)
                refdrv.write_input(pin, sub, b - a, W, error, cutoff=cutoff, overlap_frac=ov, max_gap=max_gap,
                                   dump_windows=False)
                self.jobs.append((a, b, [dict(pos=ch["pos"]) for ch in sub], pin, pout))

    def run(self):
        """→ (seconds, roh).  seconds = compute time of calcLODWindows + assembleROHWindows in the slowest
        process (input parsing and process start-up excluded)."""
        error, cutoff, ov, max_gap = self.args
        W = self.W
        if self.kind == "reference":
            ps = [subprocess.Popen([self.refdrv.BIN, j[3], j[4]], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                  for j in self.jobs]
            if any(p.wait() for p in ps):
                raise RuntimeError("ref_driver failed")
            outs = [self.refdrv.read_output(j[4], j[2], j[1] - j[0], W, dump_windows=False) for j in self.jobs]
            secs = max(o["t_windows"] + o["t_roh"] for o in outs)
            roh = []
            for j, o in zip(self.jobs, outs):
                roh += [(r[0] + j[0], r[1], r[2], r[3]) for r in o["roh"]]
            return secs, roh
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle as orc

        def work(p):
            a, b = int(self.bounds[p]), int(self.bounds[p + 1])
            roh = []
            for ci, ch in enumerate(self.chroms):
                if b <= a:
                    continue
                win = orc.calc_lod(np.ascontiguousarray(ch["geno"][:, a:b]), ch["freq"], ch["pos"], W, error, max_gap,
                                   ch["cen"])
                for i in range(b - a):
                    s_, e_, _ = orc.assemble(win[i], ch["pos"], None, cutoff, W, max_gap, ov, False, ch["cen"])
                    roh += [(a + i, ci, int(ch["pos"][x]), int(ch["pos"][y])) for x, y in zip(s_, e_)]
            return roh
        t0 = time.perf_counter()
        with ThreadPoolExecutor(self.procs) as ex:
            parts = list(ex.map(work, range(self.procs)))
        return time.perf_counter() - t0, sorted(sum(parts, []))


def dump_outputs(out_dir, arrays, limit=64 << 20, seed=0):
    """Writes each array as out_dir/<name>.npy, in float64 (bool as float32).  If together they would exceed `limit`
    bytes, every array keeps the same fixed, seeded fraction of its rows, and the row indices kept go to <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float32 if v.dtype == np.bool_ else np.float64) for k, v in arrays.items() if v is not None}
    total = sum(v.nbytes for v in arrays.values())
    frac = 1.0 if total <= limit else (limit - (1 << 16)) / (total + sum(8 * len(v) for v in arrays.values()))
    rng = np.random.default_rng(seed)
    for k, v in arrays.items():
        if frac < 1.0:
            rows = np.sort(rng.choice(len(v), min(len(v), max(1, int(len(v) * frac))), replace=False))
            np.save(os.path.join(out_dir, k + "_rows.npy"), rows.astype(np.float64))
            v = v[rows]
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n-ind", type=int, default=CFG["n_ind"])
    ap.add_argument("--n-loci", type=int, default=CFG["n_loci"])
    ap.add_argument("--cpu-sample", type=int, default=400, help="individuals in the cpu_baseline sample")
    ap.add_argument("--cpu-sample-multi", type=int, default=48, help="individuals per rank in the N>1 parity sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--exact", action="store_true", help="whole-segment chains in pass 2")
    ap.add_argument("--no-configs", action="store_true", help="skip the full-size C4 / C3 runs that follow the headline at N=1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    a.warmup = max(a.warmup, 0)
    # exactly one JSON line on stdout: libraries (NCCL prints its version) get stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    from garlic_b200 import synth

    W, err, cutoff, ov, max_gap = CFG["winsize"], CFG["error"], CFG["cutoff"], CFG["overlap_frac"], CFG["max_gap"]
    n_ind, L0 = a.n_ind, a.n_loci
    names, chr_off0, pos0, cens = synth.make_positions_genomewide(CFG["seed"], L0)
    cen_arr = np.array([cens["chr" + nm] for nm in names], np.int32)
    row_bytes = ((L0 + 3) // 4 + 15) // 16 * 16
    config = dict(workload=WORKLOAD if (n_ind, L0) == (CFG["n_ind"], CFG["n_loci"]) else
                  "REDUCED %d ind x %d SNPs (not the BASELINE config)" % (n_ind, L0),
                  individuals_per_gpu=n_ind, snps=L0, winsize=W, error=err, lod_cutoff=cutoff, overlap_frac=ov,
                  kde_subsample=CFG["kde_subsample"], sharding="by individual, %d GPU(s)" % world,
                  l2="inputs (packed matrix %.0f MB per GPU) larger than the 126 MB L2" % (n_ind * row_bytes / 1e6))

    # -------------------------------------------------------------------------------- reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        if not torch.cuda.is_available():
            dev = "cpu"
        else:
            dev = "cuda:0"
        procs = os.cpu_count() or 1
        per = max(1, min(16, n_ind // procs))      # individuals per process per step (bounded sample)
        n_s = procs * per
        rows = make_rows_torch(torch, dev, max(n_s, 256), L0, CFG["seed"], 1000, row_bytes).cpu().numpy()
        codes_all = unpack_rows(rows, L0)
        # frequencies of the sample's population: the same tables the GPU arm derives, from these rows
        nm_ = (codes_all != 3)
        tot = 2 * nm_.sum(0)
        na = np.where(nm_, codes_all, 0).sum(0)
        freq0 = np.where(tot > 0, na / np.maximum(tot, 1), 0.0)
        keep = (freq0 > 0) & (freq0 < 1)
        chroms = cpu_chroms(codes_all[:n_s], keep, freq0, pos0, chr_off0, names, cens)
        cs = CpuSample(chroms, n_s, W, err, cutoff, ov, max_gap, procs)
        kind, times = cs.kind, []
        for it in range(a.warmup + a.steps):
            secs, _ = cs.run()
            if it >= a.warmup:
                times.append(secs)
        units = cs.units
        ms = 1e3 * float(np.mean(times))
        val = units / (ms / 1e3)
        sample = "%d individuals x %d SNPs (of the %d-individual workload) per step, %d processes x %d individuals" % (
            n_s, int(keep.sum()), n_ind, procs, per)
        emit((dict(metric=METRIC, value=val, unit=UNIT, impl="reference", n_gpus=a.gpus, steps=a.steps,
                              warmup=a.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak",
                              vs_baseline=None, dtype="f64", data="synthetic", config=config,
                              cpu_baseline=dict(value=val, unit=UNIT, cores=procs, kind=kind, sample=sample),
                              e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return 0

    # -------------------------------------------------------------------------------------- own arm
    if not torch.cuda.is_available():
        sys.stderr.write("bench.py: no CUDA device; garlic_b200 has no CPU fallback\n")
        return 1
    from garlic_b200.api import GarlicGPU
    from garlic_b200 import shard
    near = bind_near_gpu(local) if world > 1 else 0
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    rows_dev = make_rows_torch(torch, dev, n_ind, L0, CFG["seed"], 1000 + rank, row_bytes)
    rows_host = torch.empty((n_ind, row_bytes), dtype=torch.uint8, pin_memory=True)
    rows_host.copy_(rows_dev)
    torch.cuda.synchronize()
    rows_host_np = rows_host.numpy()

    g = GarlicGPU(local)
    g.set_shape(n_ind, L0, chr_off0, pos0, ind_offset=rank * n_ind)
    stream = torch.cuda.ExternalStream(g.stream(), device=dev)
    if dist is not None:
        # the library runs the path's collectives itself (NCCL on its own stream); torch.distributed only carries
        # the 128-byte communicator id, the timing barrier and the max-over-ranks of the measured time
        ids = [GarlicGPU.comm_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        g.comm_init(ids[0], rank, world)
    # the KDE subsample: 20 individuals of the whole job, spread evenly; this rank computes its own
    n_total = n_ind * world
    kde_global = np.unique(np.linspace(0, n_total - 1, CFG["kde_subsample"]).astype(np.int64))
    kde_parts = [(kde_global[(kde_global // n_ind) == r] - r * n_ind).astype(np.int32) for r in range(world)]
    kde_local = kde_parts[rank]
    kde_max = max(len(x) for x in kde_parts)
    state = {}

    phases = {}

    def lap(name, t0):
        if phases is not None and "on" in phases:
            g.sync()
            phases[name] = phases.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
        return time.perf_counter()

    def step(resident, all_outputs=False):
        """One pass of the hot path.  As in the reference's main() — and in garlic_b200's own driver (host/main.cpp) — the
        per-SNP outputs that are identical on every rank (freq[] for the .freq file, the keep mask, the thinned windows of
        the KDE individuals) travel to the host of rank 0 only; every rank fetches its own ROH records.  all_outputs:
        every rank fetches everything (the untimed step that feeds the parity checks)."""
        lead = rank == 0 or all_outputs
        t0 = time.perf_counter()
        if not resident:
            g.put_packed(rows_host_np)                       # H2D from pinned host memory
            t0 = lap("put_packed_h2d", t0)
        g.count_packed()                                     # K2; N>1: + the all-reduce of the allele counters, in stream order
        t0 = lap("count_packed_allreduce" if dist is not None else "count_packed", t0)
        freq, keep, L = g.filter(want_freq=lead, want_keep=lead, wait=False)   # freq, keep mask -> page-locked host buffers
        # (rank 0), filled behind the call and complete when pass 1 returns; K3's plan
        t0 = lap("filter_compact", t0)
        g.set_tables(err, max_gap, cen_arr)                  # K4
        t0 = lap("set_tables", t0)
        if dist is None:
            thin = g.windows(W, W, individuals=kde_local, exact=False, reuse=True)
        else:                                                # rank 0 gets all KDE individuals' thinned LODs
            thin = g.windows_gather(W, W, kde_local, kde_max, world, want=lead)
        t0 = lap("pass1_thinned_windows", t0)
        roh = g.call_roh(W, cutoff, ov, exact=a.exact, copy=False)   # K5 pass 2 (fused) -> ROH records on the host
        t0 = lap("pass2_call_roh", t0)
        st = g.last_stats()
        nb = lambda x: 0 if x is None else x.nbytes
        state.update(freq=freq, keep=keep, L=L, thin=thin, roh=roh, stats=st,
                     h2d=(0 if resident else rows_host_np.nbytes) + pos0.nbytes + chr_off0.nbytes,
                     d2h=nb(freq) + nb(keep) + nb(thin) + roh.nbytes + 16)
        return st

    def timed(resident, steps, warmup, sample_clocks):
        for _ in range(warmup):
            step(resident)
        kms, sqms, launches0 = [], [], g.launch_count()
        # one sampling thread for the whole job: rank 0 watches every GPU
        cs = ClockSampler(0, world) if (sample_clocks and rank == 0) else None
        barrier()
        if cs:
            cs.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            st = step(resident)
            kms.append(st["kernel_ms"])
            sqms.append(st["squeeze_ms"])
        e1.record(stream)
        barrier()
        clocks = cs.stop() if cs else None
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), (float(np.mean(kms)), float(np.mean(sqms))), g.launch_count() - launches0, clocks

    g.put_packed_dev(rows_dev.data_ptr(), row_bytes)
    ms_res, (kms, sqms), launches, clocks = timed(True, a.steps, a.warmup, True)
    # copied now: the steps that follow overwrite the page-locked buffers these arrays live in
    last_outputs = {name: None if state[k] is None else np.array(state[k])
                    for name, k in (("freq", "freq"), ("keep", "keep"), ("kde_windows", "thin"), ("roh", "roh"))}
    units_local = state["stats"]["units"]
    units_total = units_local * world
    value = units_total * a.steps / (ms_res / 1e3)
    n_roh, n_amb, n_items, Lk = len(state["roh"]), state["stats"]["ambiguous_pairs"], state["stats"]["items"], state["L"]
    roh_dev = state["roh"].copy()
    ms_e2e, _, _, _ = timed(False, a.steps, min(a.warmup, 2) if a.warmup else 0, False)
    e2e_val = units_total * a.steps / (ms_e2e / 1e3)
    e2e = dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=int(state["h2d"]), d2h_bytes_per_step=int(state["d2h"]),
               ms_per_step=ms_e2e / a.steps,
               note="bytes of rank 0 (freq[], keep mask and the thinned windows go to rank 0's host only; every rank "
                    "uploads its own packed rows and fetches its own ROH records)" if world > 1 else "")
    assert np.array_equal(roh_dev, state["roh"]), "resident and host-buffer runs disagree"
    phases["on"] = 1                                         # one extra, untimed step with a sync after each call
    step(False)
    phases.pop("on")
    saved_phases = dict(phases)
    phases.clear()
    step(True, all_outputs=True)                             # untimed: every rank fetches freq / keep for its parity check below
    g.sync()
    phases.update(saved_phases)
    # how much the headline depends on the cutoff: pass-2 kernel time and candidate fraction at three cutoffs and
    # with the pruning bound switched off (every pair walked) — same data, same tables, pass 2 only
    sens = {}
    if rank == 0:
        def p2(c):
            for _ in range(2):
                r = g.call_roh(W, c, ov)
            st = g.last_stats()
            return dict(kernel_ms=round(st["kernel_ms"], 4), roh=len(r),
                        candidate_pair_fraction=(st["candidate_pairs"] / st["all_pairs"]) if st["candidate_pairs"] >= 0 else None)
        for c in (0.0, 1.0, 2.0):
            sens["cutoff_%g" % c] = p2(c)
        g.set_prune(False)
        sens["pruning_off_cutoff_%g" % cutoff] = p2(cutoff)
        g.set_prune(True)
        sens["note"] = "pass-2 kernels only (selection + walker); the compaction + bound pass (roofline.kernel_ms) does not depend on the cutoff"

    # roofline of the dominant kernel: the fused compaction + pruning-bound pass (squeeze_bound_kernel, K3 + the bound of
    # K5 pass 2), timed live with CUDA events on the library's stream around its launch in every step.  Algorithmic
    # bytes per launch (DESIGN.md §5): the uncompacted matrix read once, the compacted matrix written once, the piece
    # maxima written once, the per-SNP tables read once.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    n_pieces = (Lk + 255) // 256
    alg_bytes = n_ind * L0 / 4.0 + n_ind * Lk / 4.0 + n_pieces * n_ind * 4.0 + (Lk / 16.0) * (16 + 4 + 16) + L0 * 4.0
    achieved = alg_bytes / (sqms / 1e3) / 1e9
    cand = (state["stats"]["candidate_pairs"] / state["stats"]["all_pairs"]) if state["stats"]["candidate_pairs"] >= 0 else None
    walk_bytes = (cand or 1.0) * n_ind * Lk / 4.0 + n_pieces * n_ind * 4.0 + n_items * 32.0 + n_roh * 16.0
    roofline = dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=None,
                    kernel="squeeze_bound_kernel<1,1,C2> (K3 column compaction fused with the pruning bound of K5 pass 2)",
                    kernel_ms=sqms, algorithmic_bytes_per_launch=alg_bytes,
                    bytes_per_individual_window=alg_bytes / units_local,
                    peak_source="MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
                    kernel_units_per_s=units_local / (sqms / 1e3),
                    frac_of_nominal_8000_gbs=achieved / 8000.0,     # BASELINE.json quotes "roughly 8 TB/s" (SURVEY §8d: report both)
                    pass2=dict(kernels="select_kernel + walk_units_kernel (windows -> cutoff -> coverage -> ROH on the "
                                       "candidates the bound leaves)", ms=kms, select_ms=state["stats"]["select_ms"],
                               candidate_pair_fraction=cand, algorithmic_bytes=walk_bytes,
                               achieved_gbs=walk_bytes / (kms / 1e3) / 1e9),
                    pair_ms=sqms + kms,
                    pair_achieved_gbs=(alg_bytes + walk_bytes) / ((sqms + kms) / 1e3) / 1e9,
                    pair_frac=(alg_bytes + walk_bytes) / ((sqms + kms) / 1e3) / 1e9 / peak,
                    note="traffic: dram__bytes of one ncu --set full capture of this kernel (profiles/), per launch")
    tr = os.path.join(ROOT, "profiles", "r02_squeeze_traffic.json")
    if os.path.exists(tr):
        try:
            roofline["traffic"] = json.load(open(tr)).get("dram_bytes_per_launch")
        except Exception:
            pass

    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
                ms_per_step=ms_res / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic", config=config, e2e=e2e, gpu_launches=int(launches), roofline=roofline,
                clocks=clocks, host_cores_bound_per_rank=int(near), roh_found=int(n_roh), loci_used=int(Lk), ambiguous_pairs_reevaluated=int(n_amb),
                individual_windows_per_step=int(units_total), pruning_sensitivity=sens,
                phases_ms_one_synchronised_step={k: round(v, 3) for k, v in phases.items()})

    # cpu_baseline: rank 0, N=1 only, bounded sample of the same workload; the same run doubles as the parity check.
    # At N > 1 every rank checks a (smaller) sample of ITS OWN individuals against the reference's functions, and rank 0
    # checks the all-reduced frequencies against counts made on the host from all ranks' rows.
    if not a.no_cpu:
        n_s = min(a.cpu_sample if world == 1 else a.cpu_sample_multi, n_ind)
        codes = unpack_rows(rows_host_np[:n_s], L0)
        chroms = cpu_chroms(codes, state["keep"], state["freq"], pos0, chr_off0, names, cens)
        cs = CpuSample(chroms, n_s, W, err, cutoff, ov, max_gap, 1)
        secs, roh_cpu = cs.run()
        rate, kind = cs.units / secs, cs.kind
        if rank == 0 and world == 1:
            line["cpu_baseline"] = dict(value=rate, unit=UNIT, cores=1, kind=kind, seconds=secs,
                                        sample="first %d of the %d individuals x %d SNPs, same tables; the reference's "
                                               "unweighted calcLOD/assembleROHWindows are single-threaded" % (n_s, n_ind, Lk))
        pos_k = pos0[state["keep"]]
        got = sorted((int(r[0]), int(r[1]), int(pos_k[r[2]]), int(pos_k[r[3]])) for r in roh_dev if r[0] < n_s)
        mine = "identical ROH (%d)" % len(got) if got == sorted(roh_cpu) else \
            "MISMATCH: gpu %d vs cpu %d" % (len(got), len(roh_cpu))
        # frequencies: host-side counts of this rank's packed rows, summed over ranks, against the library's freq[]
        na = np.zeros(L0, np.int64)
        tot = np.zeros(L0, np.int64)
        L4 = (L0 + 3) // 4
        for i0 in range(0, n_ind, 250):
            b = rows_host_np[i0:i0 + 250, :L4]
            for k in range(4):
                gk = (b >> (2 * k)) & 3
                cols = np.arange(k, L0, 4)
                na[cols] += np.where(gk != 3, gk, 0).sum(0, dtype=np.int64)[:len(cols)]
                tot[cols] += 2 * (gk != 3).sum(0, dtype=np.int64)[:len(cols)]
        if dist is not None:
            t = torch.from_numpy(np.stack([na, tot])).to(dev)
            dist.all_reduce(t)
            na, tot = t.cpu().numpy()
        freq_cpu = np.where(tot > 0, na / np.maximum(tot, 1), 0.0)
        freq_ok = bool(np.array_equal(freq_cpu, state["freq"]))
        if dist is not None:
            allp = [None] * world
            dist.all_gather_object(allp, mine)
        else:
            allp = [mine]
        kind_s = "reference functions" if kind == "reference" else "C port of the reference"
        if all(x.startswith("identical") for x in allp):
            line["parity_vs_cpu_sample"] = "identical ROH on %s (%s; first %d individuals of every rank vs the %s)" % (
                "all %d ranks" % world if world > 1 else "the sample", ", ".join(x.split("(")[1].rstrip(")") for x in allp), n_s, kind_s)
        else:
            line["parity_vs_cpu_sample"] = "; ".join("rank %d: %s" % (r, x) for r, x in enumerate(allp))
        line["parity_freq_vs_host_counts"] = ("identical freq[] (%d SNPs, counts of all %d ranks' rows)" % (L0, world)) if freq_ok \
            else "MISMATCH in freq[]"
    g.close()
    # The other single-GPU configs of BASELINE.json at FULL size, after the headline (N = 1 only): C4 (500 x 10 M,
    # per-genotype PL likelihoods, W 200: the HBM-bound pass) and C3 (5,000 x 1 M, --weighted wLOD with an LD band over 500
    # individuals, W 72: the fp64 tensor-core pass), each with its kernel time, roofline and a parity check against the
    # reference's own functions (tools/run_configs.py).  Data are generated on the device.
    if rank == 0 and world == 1 and not a.no_configs and not a.no_cpu and (n_ind, L0) == (CFG["n_ind"], CFG["n_loci"]):
        del rows_dev
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        cfgs = {}
        try:
            import run_configs
            for key, fn, args_ in (("c4", run_configs.c4, (500, 10_000_000)), ("c3", run_configs.c3, (5000, 1_000_000, 500, False))):
                t0 = time.perf_counter()
                try:
                    r = fn(*args_)
                    r["wall_s"] = round(time.perf_counter() - t0, 1)
                    cfgs[key] = r
                except Exception as e:          # the headline line must survive a failure here
                    cfgs[key] = dict(error=repr(e)[:300])
                torch.cuda.empty_cache()
        except Exception as e:
            cfgs["error"] = repr(e)[:300]
        line["configs"] = cfgs
    if a.dump_outputs:
        # ROH records are (individual, chromosome, first kept SNP, last kept SNP), the individual counted within this rank
        # (rank r holds the global individuals r * n_ind ...); freq / keep / kde_windows reach rank 0 only
        suffix = "_rank%d" % rank if world > 1 else ""
        dump_outputs(a.dump_outputs, {k + suffix: v for k, v in last_outputs.items()})
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
