"""FRC_FLAG_PRUNE: a large reference tree with a table that observes a small part of it, and the flag's cost where
there is nothing to prune.

  python scripts/exp_prune.py [--leaves 2000000] [--samples 20000] [--observed 50000] [--per-sample 1000]
                              [--reps 5] [--out profiles]

Writes one JSON line per leg to <out>/prune_reference.jsonl and <out>/prune_overhead.jsonl and prints them.
  reference  random tree of --leaves leaves, --samples samples each holding --per-sample of the same --observed
             leaves; weighted (normalize 1) and unweighted, flag on and off.  Per leg: create_ms (host wall clock of
             frc_create), embed_ms and pairs_ms (one band over the whole triangle, FRC_FLAG_NO_D2H, median of
             frc_restart runs), n_nodes_padded, and with the flag the max relative error of all pairs of the first 64
             samples against the oracle on the whole tree.  A leg that fails records the engine's status and message
             (the weighted panels of the unpruned tree exceed one device).
  overhead   create_ms at BASELINE config 2 and 3 sizes (every leaf observed: nothing to prune), flag on and off
             alternated in the same process.
The card's name and power limit are read in the same run and go into every line.
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

OVERHEAD_CONFIGS = {"cfg2": (10_000, 5_000, 0.02, 1002, 2002), "cfg3": (50_000, 20_000, 0.02, 1003, 2003)}


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    if q.returncode:
        raise RuntimeError("nvidia-smi query failed: " + q.stderr)
    name, plim = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit_w": float(plim)}


def observed_table(tree, n_samples, n_observed, per_sample, seed):
    rng = np.random.default_rng(seed)
    pool = rng.choice(tree.leaf_ids, size=n_observed, replace=False)
    rp = np.arange(n_samples + 1, dtype=np.int64) * per_sample
    col = np.concatenate([rng.choice(pool, size=per_sample, replace=False) for _ in range(n_samples)]).astype(np.int32)
    val = np.ceil(rng.lognormal(3.0, 1.5, len(col)))
    return rp, col, val


def pair_stage(ctx, tree, csr, weighted, flags, reps):
    """create_ms, median embed_ms / pairs_ms / fixup_ms of one band over the whole triangle, and the job's info."""
    from frackyfrac_b200 import engine

    rp, col, val = csr
    job = engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST, ctx=ctx,
                     band_rows=1 << 20, flags=engine.FLAG_NO_D2H | flags)
    try:
        create_ms = job.info().create_ms
        job.drain()
        em, pm, fm = [], [], []
        for _ in range(reps):
            job.restart()
            job.drain()
            i = job.info()
            em.append(i.embed_ms); pm.append(i.pairs_ms); fm.append(i.fixup_ms)
        info = job.info()
    finally:
        job.close()
    return create_ms, float(np.median(em)), float(np.median(pm)), float(np.median(fm)), info


def max_rel_err(ctx, tree, csr, weighted, flags, n=64):
    from frackyfrac_b200 import engine
    from oracle import oracle as orc

    rp, col, val = csr
    rp, col, val = rp[:n + 1], col[:rp[n]], val[:rp[n]]
    got = engine.unifrac(tree.parent, tree.length, rp, col, val, weighted, path=engine.PATH_FAST, ctx=ctx, flags=flags)
    want = orc.unifrac(orc.Table.from_csr(rp, col, val), orc.Tree.from_flat(tree.parent, tree.length), weighted, 1,
                       os.cpu_count() or 1)
    ok = ~np.isnan(want)
    assert np.array_equal(np.isnan(got), ~ok), "NaN pattern differs"
    return float(np.max(np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-7))), len(want)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--leaves", type=int, default=2_000_000)
    ap.add_argument("--samples", type=int, default=20_000)
    ap.add_argument("--observed", type=int, default=50_000)
    ap.add_argument("--per-sample", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--overhead-reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()

    from frackyfrac_b200 import engine, synth

    hw = card()
    os.makedirs(args.out, exist_ok=True)
    ctx = engine.Context(0)

    # ---- the reference-tree case
    t0 = time.time()
    tree = synth.random_tree(args.leaves, 4001)
    csr = observed_table(tree, args.samples, args.observed, args.per_sample, 4002)
    base = {"case": "reference", "leaves": args.leaves, "nodes": tree.n_nodes, "samples": args.samples,
            "observed_leaves": args.observed, "per_sample": args.per_sample, **hw,
            "timing": f"create_ms: host wall clock of frc_create; embed/pairs/fixup: CUDA events, one band, "
                      f"FRC_FLAG_NO_D2H, median of {args.reps} frc_restart runs", "generator_s": time.time() - t0}
    lines = []
    for weighted in (True, False):
        for prune in (True, False):
            flags = engine.FLAG_PRUNE if prune else 0
            line = {**base, "weighted": weighted, "prune": prune}
            try:
                c_ms, e_ms, p_ms, f_ms, info = pair_stage(ctx, tree, csr, weighted, flags, args.reps if prune else 1)
                line.update(create_ms=c_ms, embed_ms=e_ms, pairs_ms=p_ms, fixup_ms=f_ms,
                            n_nodes_padded=info.n_nodes_padded, tree_height=info.tree_height,
                            operand_kind=info.operand_kind, flagged_pairs=info.flagged_pairs)
                if prune:
                    err, checked = max_rel_err(ctx, tree, csr, weighted, flags)
                    line.update(max_rel_err=err, pairs_checked=checked,
                                against="oracle on the whole tree, all pairs of the first 64 samples")
            except engine.FrcError as e:
                line.update(status=e.code, error=str(e))
            lines.append(line)
            print(json.dumps(line), flush=True)
    with open(os.path.join(args.out, "prune_reference.jsonl"), "w") as f:
        f.writelines(json.dumps(ln) + "\n" for ln in lines)
    del tree, csr

    # ---- nothing to prune: what the marking pass costs frc_create
    lines = []
    for cfg, (leaves, samples, density, ts, bs) in OVERHEAD_CONFIGS.items():
        tree = synth.random_tree(leaves, ts)
        rp, col, val = synth.random_table(tree, samples, density, bs)
        for weighted in (False, True):
            ms = {0: [], 1: []}
            for _ in range(args.overhead_reps):
                for prune in (0, 1):
                    with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=engine.PATH_FAST,
                                    ctx=ctx, band_rows=1 << 20,
                                    flags=engine.FLAG_NO_D2H | (engine.FLAG_PRUNE if prune else 0)) as job:
                        ms[prune].append(job.info().create_ms)
                        job.drain()
            line = {"case": "overhead", "config": cfg, "leaves": leaves, "nodes": tree.n_nodes, "samples": samples,
                    "weighted": weighted, **hw, "timing": "host wall clock of frc_create, flag off / on alternated, "
                    f"{args.overhead_reps} each", "create_ms_off": ms[0], "create_ms_on": ms[1],
                    "median_off": float(np.median(ms[0])), "median_on": float(np.median(ms[1]))}
            lines.append(line)
            print(json.dumps(line), flush=True)
    with open(os.path.join(args.out, "prune_overhead.jsonl"), "w") as f:
        f.writelines(json.dumps(ln) + "\n" for ln in lines)
    ctx.close()


if __name__ == "__main__":
    main()
