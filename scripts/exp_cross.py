"""Query x reference distances (frc_create_cross) against the triangle jobs a user would otherwise run.

  python scripts/exp_cross.py [--reps 5] [--out profiles]

Legs, one JSON line each, written to <out>/cross_unweighted_cfg2.jsonl and <out>/cross_weighted_cfg3.jsonl:
  pair_stage  the pair kernel alone: one band over the whole job, FRC_FLAG_NO_D2H, median pairs_ms over frc_restart
              runs -> pairs/s; for the cross job and for the triangle over the reference samples alone
  e2e         wall clock of frc_create + reading the whole stream with frc_next_f32 (host output), median of --reps
              jobs on one context: the cross job, and the user's alternative, the triangle over n_ref + n_q samples
Unweighted: BASELINE config 2 tree (10k leaves), n_ref = 5000, n_q in {1024, 5000}.  Weighted: config 3 tree (50k
leaves), n_ref = 20000, n_q = 2048.  The card's name and power limit are read in the same run and go into every line.
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

CTA_PAIRS = 74  # clusters of two CTAs resident at once on 148 SMs


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi query failed: " + q.stderr)
    name, plim, mhz = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit_w": float(plim), "sm_max_mhz": float(mhz)}


def rows(csr, s0, s1):
    rp, col, val = csr
    return rp[s0:s1 + 1] - rp[s0], col[rp[s0]:rp[s1]], val[rp[s0]:rp[s1]]


def pair_stage(ctx, tree, ref, query, weighted, reps):
    """Median pairs_ms / fixup_ms of one NO_D2H band; query None = the triangle over `ref`."""
    from frackyfrac_b200 import engine

    job = engine.Job(tree.parent, tree.length, *ref, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                     band_rows=1 << 30, flags=engine.FLAG_NO_D2H, query=query)
    job.drain()
    pm, fm = [], []
    for _ in range(reps):
        job.restart()
        job.drain()
        i = job.info()
        pm.append(i.pairs_ms)
        fm.append(i.fixup_ms)
    info = job.info()
    job.close()
    assert info.n_bands_total == 1
    return float(np.median(pm)), float(np.median(fm)), info


def e2e(ctx, tree, ref, query, weighted, reps):
    """Median wall clock of create + drain through frc_next_f32."""
    from frackyfrac_b200 import engine

    ts = []
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        with engine.Job(tree.parent, tree.length, *ref, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                        query=query) as job:
            n = job.drain(f32=True)
            info = job.info()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts[1:])), n, info


def run(hw, label, tree, table, n_ref, n_qs, weighted, reps, out):
    from frackyfrac_b200 import engine

    ctx = engine.Context(0)
    ref = rows(table, 0, n_ref)
    base = {"workload": label, "weighted": weighted, "nodes": tree.n_nodes, "n_ref": n_ref, **hw}
    lines = []

    def emit(d):
        lines.append({**base, **d})
        print(json.dumps(lines[-1]), flush=True)

    t_ms, t_fix, ti = pair_stage(ctx, tree, ref, None, weighted, reps)
    tri_pairs = n_ref * (n_ref - 1) // 2
    emit({"leg": "pair_stage", "job": "triangle(ref)", "pairs": tri_pairs, "pairs_ms": t_ms, "fixup_ms": t_fix,
          "pairs_per_s": tri_pairs / (t_ms / 1e3), "timing": f"CUDA events, one band, NO_D2H, median of {reps}"})
    for n_q in n_qs:
        query = rows(table, n_ref, n_ref + n_q)
        c_ms, c_fix, ci = pair_stage(ctx, tree, ref, query, weighted, reps)
        pairs = n_q * n_ref
        assert ci.n_pairs_total == pairs
        q_tiles, r_tiles = -(-n_q // 128), -(-n_ref // 128)
        d = {"leg": "pair_stage", "job": "cross", "n_q": n_q, "pairs": pairs, "pairs_ms": c_ms, "fixup_ms": c_fix,
             "pairs_per_s": pairs / (c_ms / 1e3), "rate_vs_triangle": (pairs / c_ms) / (tri_pairs / t_ms),
             "timing": f"CUDA events, one band, NO_D2H, median of {reps}"}
        if not weighted:   # CTA-pair tiles (128 query rows x 256 reference columns) over 74 resident clusters
            d.update(cta_pair_tiles=q_tiles * -(-r_tiles // 2), waves=q_tiles * -(-r_tiles // 2) / CTA_PAIRS)
        else:
            d.update(ctas=q_tiles * r_tiles)
        emit(d)
        x_ms, xn, _ = e2e(ctx, tree, ref, query, weighted, reps)
        both = rows(table, 0, n_ref + n_q)
        a_ms, an, _ = e2e(ctx, tree, both, None, weighted, reps)
        emit({"leg": "e2e", "n_q": n_q, "cross_ms": x_ms, "cross_pairs": xn, "triangle_all_ms": a_ms,
              "triangle_all_pairs": an, "speedup": a_ms / x_ms,
              "timing": f"host wall clock, frc_create + frc_next_f32 to the end, median of {reps} after one warm-up"})
    ctx.close()
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, f"cross_{label}.jsonl"), "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()

    from frackyfrac_b200 import synth

    hw = card()
    tree = synth.random_tree(10_000, 1002)
    table = synth.random_table(tree, 10_000, 0.02, 2002)
    run(hw, "unweighted_cfg2", tree, table, 5000, (1024, 5000), False, args.reps, args.out)
    tree = synth.random_tree(50_000, 1003)
    table = synth.random_table(tree, 22_048, 0.02, 2003)
    run(hw, "weighted_cfg3", tree, table, 20_000, (2048,), True, max(2, args.reps // 2), args.out)


if __name__ == "__main__":
    main()
