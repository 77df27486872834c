#!/usr/bin/env python
"""UniFrac sample-pairs/sec on B200 (BASELINE.json metric), one JSON line.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on host cores

A step = one full pass of the hot path (branch embedding + every pair of the lower triangle) over one
synthetic batch.  Headline workload at N=1 is BASELINE.json configs[1]: unweighted UniFrac, synthetic
10k-leaf tree x 5k samples (SURVEY.md 8d generator, seeds 1002 / 2002).  For N>1 the sample count grows
with sqrt(N) so that pairs per GPU stay fixed ("weak").

  value      pairs/s with inputs resident in HBM (frc_restart + drain, distances stay in HBM); one process
             per GPU, tile bands dealt to the ranks, CUDA events, max over ranks
  e2e        pairs/s through the C ABI from HOST buffers to pinned HOST distances, every step
             frc_create -> frc_next_f32* -> frc_destroy.  N>1: ONE process (rank 0) drives all N GPUs
             through opts.n_devices and reads one ordered stream -- the path behind the reference's seam
             (frcfrc.go:58-62); the other ranks idle at a CPU barrier.  e2e.per_rank_processes is the same
             workload with one process per GPU each reading its own bands.
  roofline   dominant kernel timed alone (one band, one launch); roofline_embed: the embedding stage vs HBM
  accuracy   the headline stream against the oracle on sampled rows, measured inside this run
  weighted   (N=1) BASELINE config 3 -- weighted, 50k-leaf tree x 20k samples -- with the same keys
  sharded    (N>1) the same workload with the sample-sharded embedding (peer stores + NCCL) per rank
  strong     fixed-size run (cfg4s: 100k-leaf tree x 30k samples) for strong scaling over N

--dump-outputs DIR writes the distances the `value` leg computed in its last timed step (see OutputDump), so that
two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DUMP_BYTES = 60_000_000  # --dump-outputs: data bytes in all, under 64 MB with the .npy headers
DUMP_SEED = 0

CONFIGS = {
    # name: (mode, leaves, samples, density, tree_seed, table_seed)
    "cfg2": ("unweighted", 10_000, 5_000, 0.02, 1002, 2002),
    "cfg2w": ("weighted", 10_000, 5_000, 0.02, 1002, 2002),
    "cfg3": ("weighted", 50_000, 20_000, 0.02, 1003, 2003),
    "cfg3u": ("unweighted", 50_000, 20_000, 0.02, 1003, 2003),
    "cfg4": ("unweighted", 100_000, 100_000, 0.02, 1004, 2004),
    "cfg4s": ("unweighted", 100_000, 30_000, 0.02, 1004, 2004),
    "cfg4w": ("weighted", 100_000, 100_000, 0.02, 1004, 2004),
    # 150 GB of u8 operands: more than one GPU holds -> the pair kernel expands its tiles from the bit rows
    "cfg4x": ("unweighted", 100_000, 250_000, 0.02, 1004, 2004),
    # BASELINE config 5: 320 GB of fp32 panels -> capacity mode over 8 GPUs (panels stay sharded, tiles read peers' HBM);
    # cfg5h is the same tree with half the samples (160 GB of panels: still more than one GPU holds)
    "cfg5": ("weighted", 200_000, 200_000, 0.02, 1005, 2005),
    "cfg5h": ("weighted", 200_000, 100_000, 0.02, 1005, 2005),
    "tiny": ("unweighted", 1_000, 512, 0.02, 1009, 2009),
    "tinyw": ("weighted", 1_000, 512, 0.02, 1009, 2009),
}


def load_traffic(config: str, kernel: str, world: int):
    """dram bytes per launch of the dominant kernel from the committed ncu capture of this config (1 GPU)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if world != 1 or not os.path.exists(p):
        return None
    with open(p) as f:
        d = json.load(f)
    e = d.get(f"{config}:{kernel}")
    return e["bytes"] if e else None


def measure_int8_peak():
    """Dense int8 tensor peak measured the way MEASURED_PEAKS.json measures bf16: a cuBLASLt GEMM
    (torch._int_mm, 8192^3, best of 10, CUDA events).  None when this torch build cannot run it."""
    try:
        import torch

        n = 8192
        a = torch.randint(-4, 4, (n, n), dtype=torch.int8, device="cuda")
        b = torch.randint(-4, 4, (n, n), dtype=torch.int8, device="cuda")
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        return 2.0 * n ** 3 / (best / 1e3) / 1e12
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.windows = []  # (t0, t1) of timed regions, perf_counter

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [r for t, r in self.rows if any(a - 0.05 <= t <= b + 0.15 for a, b in self.windows)]
        window = "timed regions"
        if len(inside) < 3:  # regions shorter than the sampling period: use the whole loaded phase
            inside, window = [r for _, r in self.rows], "warm-up + timed regions"
        for r in inside:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def make_workload(name: str, world: int, fixed: bool = False):
    from frackyfrac_b200 import synth

    mode, leaves, samples, density, ts, bs = CONFIGS[name]
    if world > 1 and not fixed:  # weak scaling: pairs per GPU constant
        samples = int(round(samples * math.sqrt(world)))
    tree = synth.random_tree(leaves, ts)
    rp, col, val = synth.random_table(tree, samples, density, bs)
    return mode, tree, (rp, col, val), samples, leaves, density


def cpu_baseline(tree, csr, weighted, target_s=12.0, threads=None):
    """The oracle (a port of the reference algorithm) on the host cores, bounded sample."""
    from oracle import oracle as orc

    threads = threads or os.cpu_count() or 1
    rp, col, val = csr
    n = len(rp) - 1
    ot = orc.Tree.from_flat(tree.parent, tree.length)
    tab = orc.Table.from_csr(rp, col, val)
    # calibrate on the last few rows, then size the sample for ~target_s of pair work
    r0 = max(1, n - max(2, threads // 2))
    _, emb_s, pair_s = orc.unifrac_rows(tab, ot, weighted, 1, threads, r0, n)
    cal_pairs = n * (n - 1) // 2 - r0 * (r0 - 1) // 2
    rate = cal_pairs / max(pair_s, 1e-6)
    want_pairs = min(n * (n - 1) // 2, int(rate * target_s))
    rows = max(1, min(n - 1, int(round(want_pairs / max(n - 1, 1)))))
    rb = n - rows
    _, emb_s, pair_s = orc.unifrac_rows(tab, ot, weighted, 1, threads, rb, n)
    pairs = n * (n - 1) // 2 - rb * (rb - 1) // 2
    total_pairs = n * (n - 1) // 2
    # whole-job rate implied by the sample: embedding charged in proportion
    t = pair_s + emb_s * pairs / total_pairs
    return {"value": pairs / t, "unit": "sample-pairs/s", "cores": threads, "kind": "port",
            "sample": f"rows [{rb},{n}) of the triangle = {pairs} pairs in {pair_s:.2f}s pair stage + "
                      f"{emb_s:.2f}s embedding of all {n} samples (charged pro rata)",
            "embed_s": emb_s, "pair_s": pair_s, "pairs": pairs}


def accuracy_against_oracle(flat, tree, csr, weighted, n_rows=24):
    """Max relative error (1e-7 floor, NaN must match NaN) of three blocks of rows of the triangle."""
    from oracle import oracle as orc

    rp, col, val = csr
    n = len(rp) - 1
    ot, tab = orc.Tree.from_flat(tree.parent, tree.length), orc.Table.from_csr(rp, col, val)
    worst, checked = 0.0, 0
    for r0 in sorted({1, max(1, n // 2 - n_rows // 2), max(1, n - n_rows)}):
        r1 = min(n, r0 + n_rows)
        want, _, _ = orc.unifrac_rows(tab, ot, weighted, 1, os.cpu_count() or 1, r0, r1)
        got = np.asarray(flat[r0 * (r0 - 1) // 2: r1 * (r1 - 1) // 2], np.float64)
        nan_w = np.isnan(want)
        if not np.array_equal(nan_w, np.isnan(got)):
            return {"max_rel_err": float("inf"), "pairs_checked": checked, "note": "NaN pattern differs"}
        if (~nan_w).any():
            worst = max(worst, float(np.max(np.abs(got[~nan_w] - want[~nan_w]) / np.maximum(np.abs(want[~nan_w]), 1e-7))))
        checked += len(want)
    return {"max_rel_err": worst, "pairs_checked": checked, "tolerance": 1e-5, "ok": worst < 1e-5,
            "against": "oracle (C port of frcfrc/unifrac.go) on three blocks of rows, same inputs"}


def run_reference(args, world, rank):
    if rank != 0:
        return
    mode, tree, csr, samples, leaves, density = make_workload(args.config, world, args.fixed_size)
    weighted = mode == "weighted"
    vals, last = [], None
    t_all0 = time.perf_counter()
    # every step is a bounded sample of the workload, sized so that the W + K
    # steps the driver asked for end within ~2.5 minutes of CPU work
    per_step = min(args.ref_seconds, max(0.25, 150.0 / max(1, args.steps + args.warmup)))
    n_warm, n_steps = args.warmup, args.steps
    for it in range(n_warm + n_steps):
        last = cpu_baseline(tree, csr, weighted, target_s=per_step)
        if it >= n_warm:
            vals.append(last)
    ms = 1e3 * np.mean([v["pair_s"] + v["embed_s"] * v["pairs"] / (samples * (samples - 1) // 2) for v in vals])
    v = float(np.mean([x["value"] for x in vals]))
    out = {"impl": "reference", "metric": f"UniFrac sample-pairs/sec ({mode})", "value": v, "unit": "sample-pairs/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(args.config, mode, leaves, samples, density, world),
           "cpu_baseline": {"value": v, "unit": "sample-pairs/s", "cores": last["cores"], "kind": "port",
                            "sample": last["sample"]},
           "e2e": {"value": v, "unit": "sample-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "note": "Go toolchain absent: oracle/ (C port of frcfrc/unifrac.go, pthreads on all host cores) stands in "
                   "for `frcfrc -p $(nproc)`; each step is a bounded sample of the workload; "
                   f"{n_steps} timed steps of ~{per_step:.2f} s CPU work each after {n_warm} warm-up steps",
           "wall_s": time.perf_counter() - t_all0}
    print(json.dumps(out), flush=True)


def workload_config(name, mode, leaves, samples, density, world, shard=False):
    return {"workload": f"{name}: {mode} UniFrac, synthetic {leaves}-leaf random-join tree ({2 * leaves - 1} nodes) x "
                        f"{samples} samples, leaf density {density}, lognormal counts",
            "leaves": leaves, "nodes": 2 * leaves - 1, "samples": samples, "pairs": samples * (samples - 1) // 2,
            "parallelism": (f"value: one process per GPU, tile-band sharding x{world}, embedding " +
                            ("sample-sharded + exchanged (peer stores / NCCL)" if shard else "rebuilt per rank") +
                            f"; e2e: one process driving {world} GPUs, sample-sharded embedding exchanged over peer "
                            "memory, one ordered stream") if world > 1 else "single GPU",
            "l2": "operands (3 x samples x nodes, u8 or bf16 = 0.3 / 0.6 GB at cfg2) exceed the 126 MB L2 and "
                  "every step rewrites them: no L2 flush needed"}


class Harness:
    """Ranks, barriers and reductions of one bench process."""

    def __init__(self, world, rank, local_rank):
        import torch

        self.torch, self.world, self.rank, self.local_rank = torch, world, rank, local_rank
        torch.cuda.set_device(local_rank)
        self.dist, self.cpu_group = None, None
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist
            # barriers that keep the GPUs idle (an NCCL barrier parks a spinning kernel on every device):
            # used around the phase in which rank 0 alone drives all GPUs
            self.cpu_group = dist.new_group(backend="gloo")

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def cpu_barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier(group=self.cpu_group)

    def maxreduce(self, x: float) -> float:
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


class _DeviceArray:
    """A float32 device buffer of the engine, seen by torch through the CUDA array interface (no copy)."""

    def __init__(self, addr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (addr, False), "version": 2}


class OutputDump:
    """--dump-outputs: the flat lower triangle (IterPairs order, float32) that the `value` leg's last timed step
    left in HBM, as DIR/distances.npy.  When it exceeds DUMP_BYTES, a fixed seeded sample of pairs instead, with
    their flat indices (exact in float64) as DIR/distances_index.npy.  Each band is copied on the device when the
    engine hands it out (it is complete then, and its buffer is reused after the next call); with several ranks
    every rank fills its own bands and a sum over the ranks joins them."""

    def __init__(self, directory, n_pairs, device):
        import torch

        self.torch, self.dir = torch, directory
        self.index = None
        m = n_pairs
        if 4 * n_pairs > DUMP_BYTES:
            self.index = np.unique(np.random.default_rng(DUMP_SEED).integers(0, n_pairs, DUMP_BYTES // 12))
            self.index_dev = torch.from_numpy(self.index).to(device)
            m = len(self.index)
        self.out = torch.zeros(m, dtype=torch.float32, device=device)
        self.stream = torch.cuda.Stream(device)
        torch.cuda.synchronize(device)

    def drain(self, job):
        """job.drain() that also copies every band into the dump."""
        while True:
            addr, first, n = job.next_raw_f32()
            if n == 0:
                return
            band = self.torch.as_tensor(_DeviceArray(addr, n), device=self.out.device)
            with self.torch.cuda.stream(self.stream):
                if self.index is None:
                    self.out[first:first + n] = band
                else:
                    lo, hi = np.searchsorted(self.index, [first, first + n])
                    self.out[lo:hi] = band[self.index_dev[lo:hi] - first]
            self.stream.synchronize()

    def write(self, h):
        if h.dist is not None:
            h.dist.all_reduce(self.out)
        if h.rank == 0:
            os.makedirs(self.dir, exist_ok=True)
            np.save(os.path.join(self.dir, "distances.npy"), self.out.cpu().numpy())
            if self.index is not None:
                np.save(os.path.join(self.dir, "distances_index.npy"), self.index.astype(np.float64))


def device_leg(h, ctx, tree, csr, weighted, flags, steps, warmup, sampler=None, dump=None):
    """`value`: inputs resident in HBM, distances stay in HBM; CUDA events, max over ranks.  `dump`: an OutputDump
    that receives the last timed step's distances."""
    from frackyfrac_b200 import engine

    rp, col, val = csr
    job = engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                     rank=h.rank, world=h.world, flags=engine.FLAG_NO_D2H | flags)
    job.drain()
    for _ in range(warmup):
        job.restart(); job.drain()
    h.barrier()
    t0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    for s in range(steps):
        job.restart()
        if dump is not None and s == steps - 1:
            dump.drain(job)
        else:
            job.drain()
        info = job.info()
        dev_ms += info.run_ms
        launches += info.kernel_launches
    h.barrier()
    wall = time.perf_counter() - t0
    if sampler is not None:
        sampler.mark(t0, t0 + wall)
    dev_s = h.maxreduce(dev_ms / 1e3)
    wall_s = h.maxreduce(wall)
    info = job.info()
    job.close()
    return dev_s, wall_s, launches, info


def host_leg(tree, csr, weighted, flags, steps, warmup, ctx=None, devices=None, f32=True, rank=0, world=1, keep=False):
    """`e2e`: host buffers -> frc_create -> frc_next* -> frc_destroy, every step.  Returns (seconds, last info,
    the last step's distances when keep)."""
    from frackyfrac_b200 import engine

    rp, col, val = csr
    n = len(rp) - 1
    flat = np.zeros(n * (n - 1) // 2, np.float32) if keep else None

    def step(collect=False):
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                        rank=rank, world=world, flags=flags) as j:
            if collect:
                for first, a in j.chunks_f32(copy=False):
                    flat[first:first + len(a)] = a
            else:
                j.drain(f32=f32)
            return j.info()

    info = None
    for _ in range(warmup):
        info = step()
    t0 = time.perf_counter()
    for _ in range(steps):
        info = step()
    dt = time.perf_counter() - t0
    if keep:
        step(collect=True)
    return dt, info, flat


def d2h_floor(n_devices, bytes_total, chunk_bytes, reps=5):
    """The host-link bound of `e2e`: the same bytes, in band-sized chunks, copied device -> pinned host from all
    `n_devices` GPUs at once with plain cudaMemcpyAsync (torch), nothing else running.  On this pool's 8-GPU box the
    GPUs share the host links: the aggregate saturates near 95 GB/s, not 8 x 55."""
    import torch

    per = max(chunk_bytes, bytes_total // n_devices)
    n_chunks = max(1, per // max(chunk_bytes, 1))
    src, dst, streams = [], [], []
    for d in range(n_devices):
        with torch.cuda.device(d):
            src.append(torch.empty(chunk_bytes, dtype=torch.uint8, device=f"cuda:{d}"))
            dst.append(torch.empty(chunk_bytes * min(n_chunks, 8), dtype=torch.uint8).pin_memory())
            streams.append(torch.cuda.Stream(device=d))
    best = 1e9
    for _ in range(reps + 1):
        for d in range(n_devices):
            torch.cuda.synchronize(d)
        t0 = time.perf_counter()
        for c in range(n_chunks):
            for d in range(n_devices):
                with torch.cuda.stream(streams[d]):
                    k = c % min(n_chunks, 8)
                    dst[d][k * chunk_bytes:(k + 1) * chunk_bytes].copy_(src[d], non_blocking=True)
        for d in range(n_devices):
            streams[d].synchronize()
        best = min(best, time.perf_counter() - t0)
    moved = n_chunks * chunk_bytes * n_devices
    return {"ms": 1e3 * best * bytes_total / moved, "aggregate_gbs": moved / best / 1e9, "per_device_gbs": moved / best / 1e9 / n_devices,
            "how": f"{n_chunks} x {chunk_bytes} B per device, {n_devices} device(s) at once, cudaMemcpyAsync to pinned host, best of {reps}"}


def kernel_roofline(ctx, tree, csr, weighted, flags, config, total_pairs, samples, peaks, peaks_kind, reps):
    """The dominant kernel timed alone: one band over the whole triangle, nothing else on the device."""
    from frackyfrac_b200 import engine

    rp, col, val = csr
    rj = engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                    band_rows=1 << 20, flags=engine.FLAG_NO_D2H | flags)
    rj.drain()
    ms, emb = [], []
    for _ in range(max(3, reps)):
        rj.restart(); rj.drain()
        i = rj.info()
        ms.append(i.pairs_ms)
        emb.append(i.embed_ms)
    ri = rj.info()
    rj.close()
    k_ms = float(np.median(ms))
    B = tree.n_nodes
    if weighted:
        # SURVEY 8d: 2 FP32 lane-ops per (pair, node); peak = SMs * 128 lanes * clock
        peak = 148 * 128 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        ach = total_pairs * 2.0 * B / (k_ms / 1e3) / 1e12
        roof = {"bound": "fp32", "kernel": "k_weighted_tiles", "achieved": ach, "peak": peak,
                "unit": "T lane-op/s", "frac": ach / peak,
                "traffic": load_traffic(config, "k_weighted_tiles", 1), "kernel_ms": k_ms,
                "peak_source": "derived: 148 SM x 128 lanes x sm_max_mhz"}
    else:
        # algorithmic work = one multiply-add per (pair, node) = 2*B flops per pair (SURVEY 8d).
        # bf16 hi/lo kernel: executes 2 bf16 planes on the kind::f16 pipe -> peak = measured bf16 burst.
        # u8 kernel: executes 2 u8 planes on the kind::i8 pipe, whose rate is 2x the bf16 one
        # (no measured int8 figure in MEASURED_PEAKS.json: derived as 2 x bf16_tflops, stated).
        i8 = ri.operand_kind >= 2
        int8_measured = measure_int8_peak() if i8 else None
        # the larger of the two estimates of the int8 peak, so that frac is not flattered
        peak = max(int8_measured or 0.0, peaks["bf16_tflops"] * 2.0) if i8 else peaks["bf16_tflops"]
        ach = total_pairs * 2.0 * B / (k_ms / 1e3) / 1e12
        n_tiles = sum(t + 1 for t in range((samples + 127) // 128))
        executed = n_tiles * 128 * 128 * ri.n_nodes_padded * 2 * 2.0 / (k_ms / 1e3) / 1e12
        kname = "k_unweighted_tc2<u8>" if i8 else "k_unweighted_tc2<bf16>"
        roof = {"bound": "tensor", "kernel": kname,
                "achieved": ach, "peak": peak,
                "unit": "TOP/s" if i8 else "TFLOP/s", "frac": ach / peak,
                "traffic": load_traffic(config, kname, 1), "kernel_ms": k_ms,
                "executed_tflops": executed, "executed_frac": executed / peak,
                "achieved_vs_bf16_peak": ach / peaks["bf16_tflops"],
                "int8_peak_measured_cublaslt": int8_measured,
                "peak_source": (f"max(2 x {peaks_kind} bf16_tflops [kind::i8 issues at twice the kind::f16 rate], "
                                "int8 GEMM measured live with torch._int_mm 8192^3 best of 10)" if i8 else
                                f"{peaks_kind} bf16_tflops") + " (burst; kernel timed alone, one launch over all tiles)",
                "note": "algorithmic ops = 2*B per pair; the kernel executes 2 operand planes and full "
                        "diagonal tiles over the padded contraction length, reported as executed_* (the "
                        "CTA-pair kernel also runs one masked tile above each second diagonal tile, not counted)"}
    e_ms = float(np.median(emb))
    gbs = ri.embed_bytes / (e_ms / 1e3) / 1e9 if e_ms > 0 else 0.0
    roof_embed = {"bound": "hbm", "stage": "embedding (CSR -> presence bits -> row sums -> K-major operands)" if not weighted else
                  "embedding (CSR -> fp64 subtree sums per slab -> totals -> fp32 tile panels + denominators)",
                  "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                  "algorithmic_bytes": int(ri.embed_bytes), "stage_ms": e_ms,
                  "peak_source": f"{peaks_kind} hbm_gbs", "timed": "CUDA events around the stage, median over restarts"}
    return roof, roof_embed, ri


def dtype_of(weighted, info):
    if weighted:
        return "f32 numerator tiles + f32 output, f64 embedding / denominators"
    if info.operand_kind == 1:
        return "bf16 x bf16 -> f32 (tcgen05 kind::f16), f64 row sums, f32 ratio / output"
    return "u8 x u8 -> s32 (tcgen05 kind::i8, exact), s64 chunk / row sums, f32 ratio / output"


def sub_record(h, ctx, args, name, steps, warmup, peaks, peaks_kind, fixed, legs=("value", "e2e", "roofline", "cpu", "accuracy")):
    """One workload measured like the headline, with fewer steps (a sub-record of the JSON line)."""
    from frackyfrac_b200 import engine

    mode, tree, csr, samples, leaves, density = make_workload(name, h.world, fixed)
    weighted = mode == "weighted"
    total_pairs = samples * (samples - 1) // 2
    rec = {"config": workload_config(name, mode, leaves, samples, density, h.world), "steps": steps, "warmup": warmup,
           "scaling": "strong" if fixed else "weak"}
    flags = 0
    if "value" in legs:
        shard = h.world > 1 and samples * (2 * leaves - 1) >= 2_000_000_000
        if shard:
            flags |= engine.FLAG_SHARD_EMBED
        dev_s, wall_s, launches, info = device_leg(h, ctx, tree, csr, weighted, flags, steps, warmup)
        rec.update({"value": total_pairs * steps / dev_s, "unit": "sample-pairs/s", "ms_per_step": 1e3 * dev_s / steps,
                    "dtype": dtype_of(weighted, info), "gpu_launches": int(launches), "embedding_sharded": bool(shard),
                    "stages_ms": {"embed": info.embed_ms, "run": info.run_ms}})
    if "e2e" in legs:
        h.cpu_barrier()
        if h.rank == 0:
            mctx = engine.Context(devices=list(range(h.world))) if h.world > 1 else ctx
            dt, ei, flat = host_leg(tree, csr, weighted, 0, steps, warmup, ctx=mctx, keep="accuracy" in legs)
            rec["e2e"] = {"value": total_pairs * steps / dt, "unit": "sample-pairs/s", "ms_per_step": 1e3 * dt / steps,
                          "h2d_bytes_per_step": int(ei.h2d_bytes), "d2h_bytes_per_step": int(ei.d2h_bytes),
                          "n_devices": int(ei.n_devices), "create_ms": ei.create_ms}
            if "accuracy" in legs:
                rec["accuracy"] = accuracy_against_oracle(flat, tree, csr, weighted)
            if mctx is not ctx:
                mctx.close()
        h.cpu_barrier()
    if h.rank == 0 and h.world == 1 and "roofline" in legs:
        roof, roof_embed, _ = kernel_roofline(ctx, tree, csr, weighted, 0, name, total_pairs, samples, peaks, peaks_kind, 3)
        rec["roofline"], rec["roofline_embed"] = roof, roof_embed
    if h.rank == 0 and "cpu" in legs:
        cpu = cpu_baseline(tree, csr, weighted, target_s=min(8.0, args.ref_seconds))
        rec["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    return rec


def run_ours(args, world, rank, local_rank):
    from frackyfrac_b200 import engine

    h = Harness(world, rank, local_rank)
    t_bench0 = time.perf_counter()
    mode, tree, csr, samples, leaves, density = make_workload(args.config, world, args.fixed_size)
    weighted = mode == "weighted"
    rp, col, val = csr
    total_pairs = samples * (samples - 1) // 2
    ctx = engine.Context(local_rank)
    peaks, peaks_kind = load_peaks()
    uw_flags = engine.FLAG_UW_BF16 if args.uw_kernel == "bf16" else 0
    # one process per GPU (`value`): the sample-sharded embedding (FRC_FLAG_SHARD_EMBED: peer stores of the bit
    # columns + NCCL all-gather of the row sums) pays when the shardable part outweighs the meeting of the ranks
    # (~140 us at 8 ranks).  At the cfg2-derived sizes of the scaling run it is a wash, so the default is
    # size-based; --shard-embed / --no-shard-embed force either; the `sharded` sub-record always measures it.
    shard = world > 1 and not args.no_shard_embed and (args.shard_embed or samples * (2 * leaves - 1) >= 2_000_000_000)
    if world > 1:
        from frackyfrac_b200 import dist as fdist
        fdist.init_comm(ctx, rank, world)
    flags = uw_flags | (engine.FLAG_SHARD_EMBED if shard else 0)

    # ---------------------------------------------- value: inputs resident in HBM, one process per GPU
    dump = OutputDump(args.dump_outputs, total_pairs, local_rank) if args.dump_outputs else None
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_s, wall_s, launches, info = device_leg(h, ctx, tree, csr, weighted, flags, args.steps, args.warmup, sampler, dump)
    value = total_pairs * args.steps / dev_s
    if dump is not None:
        dump.write(h)

    # ---------------------------------------------- sharded sub-record (N > 1): the exchange path per rank
    sharded = None
    if world > 1 and not args.quick:
        sf = uw_flags | engine.FLAG_SHARD_EMBED
        s_dev, _, _, s_info = device_leg(h, ctx, tree, csr, weighted, sf, args.steps, args.warmup)
        # byte identity of the two streams on this rank's bands (host route, fp32 bands as delivered)
        def my_stream(f):
            with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                            rank=rank, world=world, flags=f) as j:
                return np.concatenate([a for _, a in j.chunks_f32()] or [np.zeros(0, np.float32)])
        same = bool(np.array_equal(my_stream(sf), my_stream(uw_flags), equal_nan=True))
        same = h.maxreduce(0.0 if same else 1.0) == 0.0
        sharded = {"value": total_pairs * args.steps / s_dev, "unit": "sample-pairs/s", "ms_per_step": 1e3 * s_dev / args.steps,
                   "embed_ms": s_info.embed_ms, "embed_ms_unsharded": info.embed_ms, "gather_bytes_per_rank": int(s_info.gather_bytes),
                   "identical_to_unsharded_stream": same,
                   "how": "FRC_FLAG_SHARD_EMBED: each rank builds the bit columns of its sample shard and stores them into "
                          "every rank's HBM over NVLink (CUDA IPC mappings) from inside the embedding kernel; one NCCL "
                          "all-gather of the row sums (8 B per sample) is where the ranks meet"}

    # ---------------------------------------------- e2e: host buffers through the C ABI
    e2e = None
    e2e_flat = None
    if not args.no_e2e:
        # (a) one process per GPU, each rank yields its own bands
        h.barrier()
        t0 = time.perf_counter()
        dt_r, ei_r, _ = host_leg(tree, csr, weighted, flags, args.steps, args.warmup, ctx=ctx, rank=rank, world=world)
        sampler.mark(t0, time.perf_counter())
        ranks_s = max(h.maxreduce(dt_r), 1e-9)
        per_rank = {"value": total_pairs * args.steps / ranks_s, "ms_per_step": 1e3 * ranks_s / args.steps,
                    "h2d_bytes_per_step_per_rank": int(ei_r.h2d_bytes), "d2h_bytes_per_step_per_rank": int(ei_r.d2h_bytes),
                    "h2d_ms": ei_r.h2d_ms}
        # (b) one process drives every GPU and reads ONE ordered stream (rank 0; the others idle, GPUs free)
        h.cpu_barrier()
        if rank == 0:
            mctx = engine.Context(devices=list(range(world))) if world > 1 else ctx
            t0 = time.perf_counter()
            dt, ei, e2e_flat = host_leg(tree, csr, weighted, uw_flags, args.steps, args.warmup, ctx=mctx, keep=not args.quick)
            sampler.mark(t0, t0 + dt)
            f64 = None
            if world == 1:
                dt64, ei64, _ = host_leg(tree, csr, weighted, uw_flags, args.steps, args.warmup, ctx=mctx, f32=False)
                f64 = {"value": total_pairs * args.steps / dt64, "ms_per_step": 1e3 * dt64 / args.steps,
                       "note": "the same stream through frc_next (float64 at the boundary: fp32 bands widened on the host)"}
            e2e = {"value": total_pairs * args.steps / dt, "unit": "sample-pairs/s",
                   "h2d_bytes_per_step": int(ei.h2d_bytes), "d2h_bytes_per_step": int(ei.d2h_bytes),
                   "ms_per_step": 1e3 * dt / args.steps, "n_devices": int(ei.n_devices), "processes": 1,
                   "stages_ms": {"create_host": ei.create_ms, "h2d": ei.h2d_ms, "embed": ei.embed_ms},
                   "float64": f64, "per_rank_processes": per_rank if world > 1 else None,
                   "timed": "host wall clock around frc_create..frc_next_f32*..frc_destroy (host validation, pinned staging, "
                            "H2D, kernels, D2H of every distance as fp32 into pinned host memory)" +
                            (f"; one process, {world} GPUs, one ordered stream (opts.n_devices)" if world > 1 else "")}
            if mctx is not ctx:
                mctx.close()
            if not args.quick:
                fl = d2h_floor(world, int(ei.d2h_bytes), max(1 << 20, int(ei.d2h_bytes) // max(1, int(ei.n_bands_total))))
                e2e["d2h_floor"] = fl
                e2e["frac_of_d2h_floor"] = fl["ms"] / e2e["ms_per_step"]
        h.cpu_barrier()
    clocks = sampler.stop()

    # ---------------------------------------------- roofline of the dominant kernel + embedding stage (rank 0, timed alone)
    roofline, roofline_embed, cpu, accuracy = None, None, None, None
    if rank == 0 and not args.no_roofline:
        roofline, roofline_embed, _ = kernel_roofline(ctx, tree, csr, weighted, uw_flags, args.config, total_pairs, samples,
                                                      peaks, peaks_kind, args.steps)
        if world > 1:
            roofline["note_n"] = "kernel timed alone on ONE GPU over the whole triangle of this N's workload"
    if rank == 0 and e2e_flat is not None:
        accuracy = accuracy_against_oracle(e2e_flat, tree, csr, weighted)
        e2e_flat = None
    if rank == 0 and not args.no_cpu:
        cpu = cpu_baseline(tree, csr, weighted, target_s=args.ref_seconds)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # ---------------------------------------------- sub-records: the other half of the metric, strong scaling
    weighted_rec, strong_rec = None, None
    if not args.quick and not weighted:
        if world == 1:
            weighted_rec = sub_record(h, ctx, args, "cfg3", 2, 1, peaks, peaks_kind, fixed=False)
        strong_rec = sub_record(h, ctx, args, "cfg4s", 5, 2, peaks, peaks_kind, fixed=True, legs=("value", "e2e"))

    if rank == 0:
        out = {"metric": f"UniFrac sample-pairs/sec ({mode})", "value": value, "unit": "sample-pairs/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dev_s / args.steps,
               "higher_is_better": True, "scaling": "strong" if args.fixed_size else "weak", "vs_baseline": None,
               "dtype": dtype_of(weighted, info), "data": "synthetic",
               "config": workload_config(args.config, mode, leaves, samples, density, world, shard),
               "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
               "roofline": roofline, "roofline_embed": roofline_embed, "accuracy": accuracy, "cpu_baseline": cpu,
               "stages_ms": {"embed": info.embed_ms, "run": info.run_ms,
                             "note": "value leg, this rank: CUDA events (embedding stage; embedding start -> last band done)"},
               "weighted": weighted_rec, "sharded": sharded, "strong": strong_rec,
               "timing": "value: CUDA events on the engine's streams (embedding start -> last band done), summed over "
                         "steps, max over ranks; wall clock of the same region = %.3f ms/step" % (1e3 * wall_s / args.steps),
               "flagged_pairs": int(info.flagged_pairs), "bands": int(info.n_bands_total),
               "tree_height": int(info.tree_height), "bench_wall_s": time.perf_counter() - t_bench0}
        print(json.dumps(out), flush=True)
    ctx.close()
    h.close()


def main():
    sys.dont_write_bytecode = True  # the tree may be read-only: leave no __pycache__ in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--ref-seconds", type=float, default=12.0, help="CPU work per reference sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (configs whose output exceeds host RAM)")
    ap.add_argument("--no-roofline", action="store_true", help="skip the kernel-alone timing leg")
    ap.add_argument("--quick", action="store_true", help="headline only: no weighted / sharded / strong sub-records, no accuracy")
    ap.add_argument("--min-warmup", type=int, default=3)
    ap.add_argument("--fixed-size", action="store_true",
                    help="N>1: keep the config's sample count (strong scaling) instead of growing it with sqrt(N)")
    ap.add_argument("--shard-embed", action="store_true", help="N>1: force the sharded embedding + exchange in the value leg")
    ap.add_argument("--no-shard-embed", action="store_true",
                    help="N>1: every rank rebuilds the whole embedding (no exchange) in the value leg")
    ap.add_argument("--uw-kernel", default="u8", choices=["u8", "bf16"],
                    help="operand encoding of the unweighted tensor-core kernel (FRC_FLAG_UW_BF16)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the distances of the value leg's last timed step to DIR (.npy, float32; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under it
        port = os.environ.get("MASTER_PORT", "29517")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", port, os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    args.warmup = max(args.warmup, args.min_warmup) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args, world, rank)
    else:
        run_ours(args, world, rank, local_rank)


if __name__ == "__main__":
    main()
