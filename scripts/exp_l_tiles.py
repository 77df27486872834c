"""Flag -l as the reference codes it (normalize = 0) at BASELINE config 3 size: the key-matched FP32 tiles
(FRC_FLAG_L_TILES) against the exact list walk and against the unkeyed tiles of normalize = 2 (the ceiling).

  python scripts/exp_l_tiles.py [--config cfg3] [--reps 5] [--exact-samples 4096] [--out profiles]

Writes one JSON line per leg to <out>/l_tiles_<config>.jsonl and prints them.  Legs:
  keyed      pair stage of the keyed tiles alone (one band over the whole triangle, FRC_FLAG_NO_D2H, median over
             frc_restart): pairs/s, lane-op rate against the FP32 issue peak (148 SMs x 128 lanes x max SM clock)
             -- algorithmic 2 ops per (pair, node) as bench.py counts the unkeyed kernel, and executed 4
             (ISETP + FSEL + FADD + FADD) -- and the max relative error against the oracle (normalize = 0) on sampled rows
  documented the same job with normalize = 2 on the unkeyed kernel
  exact      the exact list walk on the first --exact-samples samples (its rate does not depend on the sample
             count: one thread per pair walks two lists); 0 skips it
The card's name, power limit and max SM clock are read in the same run and go into every line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {"cfg3": (50_000, 20_000, 0.02, 1003, 2003), "cfg2": (10_000, 5_000, 0.02, 1002, 2002)}


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi query failed: " + q.stderr)
    name, plim, mhz = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit_w": float(plim), "sm_max_mhz": float(mhz)}


def pair_stage(ctx, tree, csr, normalize, flags, reps, n_samples=None):
    """Median device time of the pair stage (pairs_ms, fixup_ms) of one band over the whole triangle."""
    from frackyfrac_b200 import engine

    rp, col, val = csr
    if n_samples is not None:
        rp, col, val = rp[:n_samples + 1], col[:rp[n_samples]], val[:rp[n_samples]]
    path = engine.PATH_EXACT if normalize == 0 and not flags else engine.PATH_FAST
    job = engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, normalize=normalize, path=path, ctx=ctx,
                     band_rows=1 << 20, flags=engine.FLAG_NO_D2H | flags)
    job.drain()
    pm, fm, em = [], [], []
    for _ in range(reps):
        job.restart()
        job.drain()
        i = job.info()
        pm.append(i.pairs_ms); fm.append(i.fixup_ms); em.append(i.embed_ms)
    info = job.info()
    job.close()
    return float(np.median(pm)), float(np.median(fm)), float(np.median(em)), info


def max_rel_err(ctx, tree, csr, n_rows=24):
    """The keyed job's fp32 stream against the oracle (normalize = 0) on three blocks of rows."""
    from frackyfrac_b200 import engine
    from oracle import oracle as orc

    rp, col, val = csr
    n = len(rp) - 1
    flat = np.empty(n * (n - 1) // 2, np.float32)
    with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, normalize=0, path=engine.PATH_FAST, ctx=ctx,
                    flags=engine.FLAG_L_TILES) as job:
        for first, a in job.chunks_f32(copy=False):
            flat[first:first + len(a)] = a
            xi, xv = job.exceptions()
            flat[xi] = xv
        flagged = job.info().flagged_pairs
    ot, tab = orc.Tree.from_flat(tree.parent, tree.length), orc.Table.from_csr(rp, col, val)
    worst, checked = 0.0, 0
    for r0 in sorted({1, n // 2 - n_rows // 2, n - n_rows}):
        want, _, _ = orc.unifrac_rows(tab, ot, True, 0, os.cpu_count() or 1, r0, r0 + n_rows)
        got = flat[r0 * (r0 - 1) // 2:(r0 + n_rows) * (r0 + n_rows - 1) // 2].astype(np.float64)
        ok = ~np.isnan(want)
        assert np.array_equal(np.isnan(got), ~ok), "NaN pattern differs"
        worst = max(worst, float(np.max(np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-7))))
        checked += len(want)
    return worst, checked, flagged


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--exact-samples", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()

    from frackyfrac_b200 import engine, synth

    hw = card()
    leaves, samples, density, ts, bs = CONFIGS[args.config]
    t0 = time.time()
    tree = synth.random_tree(leaves, ts)
    csr = synth.random_table(tree, samples, density, bs)
    gen_s = time.time() - t0
    B = tree.n_nodes
    peak = 148 * 128 * hw["sm_max_mhz"] * 1e6 / 1e12
    ctx = engine.Context(0)
    base = {"config": args.config, "leaves": leaves, "samples": samples, "nodes": B, **hw,
            "fp32_issue_peak_t_lane_ops": peak, "timing": "CUDA events, one band, FRC_FLAG_NO_D2H, median of "
            f"{args.reps} frc_restart runs", "generator_s": gen_s}
    lines = []

    def rate(pairs, ms, per):
        return pairs * per * B / (ms / 1e3) / 1e12

    pairs = samples * (samples - 1) // 2
    k_ms, k_fix, k_emb, ki = pair_stage(ctx, tree, csr, 0, engine.FLAG_L_TILES, args.reps)
    err, checked, flagged = max_rel_err(ctx, tree, csr)
    lines.append({**base, "leg": "keyed", "normalize": 0, "kernel": "k_weighted_tiles<keyed>", "path_taken": ki.path_taken,
                  "pairs_ms": k_ms, "fixup_ms": k_fix, "embed_ms": k_emb, "pairs_per_s": pairs / (k_ms / 1e3),
                  "alg_t_lane_ops": rate(pairs, k_ms, 2), "alg_frac": rate(pairs, k_ms, 2) / peak,
                  "exec_t_lane_ops": rate(pairs, k_ms, 4), "exec_frac": rate(pairs, k_ms, 4) / peak,
                  "flagged_pairs": flagged, "max_rel_err": err, "pairs_checked": checked,
                  "against": "oracle normalize=0 on three blocks of 24 rows"})
    print(json.dumps(lines[-1]), flush=True)
    d_ms, d_fix, d_emb, _ = pair_stage(ctx, tree, csr, 2, 0, args.reps)
    lines.append({**base, "leg": "documented", "normalize": 2, "kernel": "k_weighted_tiles", "pairs_ms": d_ms,
                  "fixup_ms": d_fix, "embed_ms": d_emb, "pairs_per_s": pairs / (d_ms / 1e3),
                  "alg_t_lane_ops": rate(pairs, d_ms, 2), "alg_frac": rate(pairs, d_ms, 2) / peak,
                  "keyed_over_documented_time": k_ms / d_ms})
    print(json.dumps(lines[-1]), flush=True)
    if args.exact_samples > 0:
        n = min(samples, args.exact_samples)
        e_ms, _, e_emb, ei = pair_stage(ctx, tree, csr, 0, 0, max(1, args.reps // 2), n_samples=n)
        ep = n * (n - 1) // 2
        lines.append({**base, "leg": "exact", "normalize": 0, "kernel": "k_unsorted_pairs", "samples_run": n,
                      "path_taken": ei.path_taken, "pairs_ms": e_ms, "embed_ms": e_emb, "pairs_per_s": ep / (e_ms / 1e3),
                      "keyed_speedup_pairs_per_s": (pairs / (k_ms / 1e3)) / (ep / (e_ms / 1e3))})
        print(json.dumps(lines[-1]), flush=True)
    ctx.close()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, f"l_tiles_{args.config}.jsonl"), "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
