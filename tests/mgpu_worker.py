"""Worker of tests/test_multi_gpu.py, launched by torchrun with one rank per GPU.

Every rank runs its bands of the triangle with the embedding built sample-sharded and
all-gathered (FRC_FLAG_SHARD_EMBED); rank 0 also runs the whole job alone.  The cases cover every
array the weighted exchange carries (normalisers with normalize=1, key panels with -l as coded on
the tiles) and, with FRC_PEER_PUSH=0, the NCCL all-gather of the unweighted bit columns.  The merged
multi-rank stream must equal the single-rank one byte for byte (SURVEY §8e) and stay within
1e-5 of the oracle.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from frackyfrac_b200 import dist as fdist, engine, synth  # noqa: E402


def main():
    rank, world, local = fdist.env_rank_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = engine.Context(local)
    fdist.init_comm(ctx, rank, world)
    tree = synth.random_tree(1500, 301)
    rp, col, val = synth.random_table(tree, 1100, 0.03, 302)
    n = 1100
    ok = True
    cases = (  # weighted, normalize, flags, FRC_PEER_PUSH
        (False, 1, 0, None), (False, 1, engine.FLAG_UW_BF16, None), (False, 1, engine.FLAG_UW_BITS, None),
        (False, 1, 0, "0"), (True, 1, 0, None), (True, 2, 0, None), (True, 0, engine.FLAG_L_TILES, None))
    for weighted, norm, uw_flags, peer_push in cases:
        # (every rank sets it before the job is created: the peer-push decision is collective)
        if peer_push is not None:
            os.environ["FRC_PEER_PUSH"] = peer_push
        chunks = []
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, normalize=norm, path=engine.PATH_FAST,
                        ctx=ctx, rank=rank, world=world, band_rows=128, flags=uw_flags | engine.FLAG_SHARD_EMBED) as job:
            for first, a in job.chunks():
                chunks.append((first, a))
            info = job.info()
        assert info.gather_bytes > 0, "the embedding was not all-gathered"
        full = fdist.gather_distances(chunks, n)
        if rank == 0:
            alone = engine.unifrac(tree.parent, tree.length, rp, col, val, weighted, normalize=norm, path=engine.PATH_FAST,
                                   ctx=ctx, band_rows=128, flags=uw_flags)
            same = np.array_equal(full, alone, equal_nan=True)
            from oracle import oracle as orc
            want = orc.unifrac(orc.Table.from_csr(rp, col, val), orc.Tree.from_flat(tree.parent, tree.length), weighted, norm, 8)
            err = np.max(np.abs(full - want) / np.maximum(np.abs(want), 1e-12))
            print(f"weighted={weighted} normalize={norm} flags={uw_flags} peer_push={peer_push} world={world} "
                  f"identical={same} max_rel_err={err:.2e} gather_bytes={info.gather_bytes}", flush=True)
            ok = ok and same and err < 1e-5
        os.environ.pop("FRC_PEER_PUSH", None)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.broadcast(flag, src=0)
    ctx.close()
    dist.destroy_process_group()
    if rank == 0:
        print("MGPU_OK" if ok else "MGPU_FAIL", flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
