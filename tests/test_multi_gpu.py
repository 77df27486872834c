"""Multi-GPU path on real devices (skipped with fewer than 2 GPUs): sample-sharded embedding,
NCCL all-gather of the compact form inside libfrcfrc_cuda, band-sharded pair stage."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_embedding_all_gather_matches_single_gpu(built):
    import torch

    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2 if n < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "mgpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "MGPU_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def _stream(job):
    """All chunks of a job; asserts they are contiguous and strictly increasing."""
    import numpy as np

    out, expect = [], 0
    for first, a in job.chunks():
        assert first == expect, (first, expect)
        expect += len(a)
        out.append(a)
    return np.concatenate(out) if out else np.zeros(0)


def test_one_process_many_gpus_one_ordered_stream(built, monkeypatch):
    """opts.n_devices: ONE process validates and stages the inputs once, every GPU computes the bands it owns, and
    frc_next hands them out in flat-index order (the single ordered iter.Seq behind frcfrc.go:58-62).  The stream
    must be byte-identical for 1, 2, 4 and 8 devices (SURVEY 8e), with the sample shards of the embedding exchanged
    over peer memory or with every device rebuilding it (FRC_SHARD=0)."""
    import numpy as np
    import torch

    from frackyfrac_b200 import engine, synth
    from tests.helpers import oracle_flat, rel_err

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree = synth.random_tree(1500, 301)
    rp, col, val = synth.random_table(tree, 1100, 0.03, 302, integer_counts=False)
    m = rp[1]
    col[m:2 * m] = col[:m]; val[m:2 * m] = val[:m]                       # an identical pair
    col[5 * m:6 * m] = col[:m]; val[5 * m:6 * m] = val[:m] * (1 + 1e-4 * (np.arange(m) % 3 == 0))  # fix-up territory
    one = engine.Context(0)
    cases = [(False, 0, engine.PATH_FAST), (False, engine.FLAG_UW_BF16, engine.PATH_FAST), (False, engine.FLAG_UW_BITS, engine.PATH_FAST),
             (True, 0, engine.PATH_FAST), (True, 0, engine.PATH_EXACT)]
    ref = {}
    for weighted, flags, path in cases:
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=path, ctx=one, band_rows=128, flags=flags) as job:
            ref[(weighted, flags, path)] = _stream(job)
            assert job.info().n_devices == 1
    one.close()
    want = {w: oracle_flat(tree, (rp, col, val), w) for w in (False, True)}
    for nd in [k for k in (2, 4, 8) if k <= n_gpu]:
        ctx = engine.Context(devices=list(range(nd)))
        for shard in ("1", "0"):
            monkeypatch.setenv("FRC_SHARD", shard)
            for weighted, flags, path in cases:
                for band_rows in (128, 0):
                    with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, path=path, ctx=ctx,
                                    band_rows=band_rows, flags=flags) as job:
                        got = _stream(job)
                        info = job.info()
                    assert info.n_devices == nd and info.n_bands_mine == info.n_bands_total
                    if path == engine.PATH_FAST and shard == "1":
                        assert info.gather_bytes > 0, "the sample shards were not exchanged between the devices"
                    key = (weighted, flags, path)
                    assert np.array_equal(got, ref[key], equal_nan=True), (nd, shard, key, band_rows)
                    assert rel_err(got, want[weighted]).max() < 1e-5
        # restart on resident inputs gives the same stream again
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=False, path=engine.PATH_FAST, ctx=ctx) as job:
            a = _stream(job)
            job.restart()
            b = _stream(job)
        assert np.array_equal(a, b) and np.array_equal(a, ref[(False, 0, engine.PATH_FAST)])
        ctx.close()
    # a job may also bring its own devices (no context): opts.n_devices = -1 = every visible GPU
    with engine.Job(tree.parent, tree.length, rp, col, val, weighted=False, path=engine.PATH_FAST, devices=-1) as job:
        assert np.array_equal(_stream(job), ref[(False, 0, engine.PATH_FAST)]) and job.info().n_devices == min(n_gpu, 8)


def test_weighted_capacity_mode_reads_panels_from_peers(built, monkeypatch):
    """BASELINE config 5 in the small: when the fp32 panels of all samples do not fit one GPU they stay sharded over
    the devices (two shards each) and the column shards visit every device in turn through two visiting buffers filled
    over NVLink (start_pairs_capacity in csrc/job.cu, PanelMap in csrc/weighted.cu).  Forced here with FRC_CAPACITY=1:
    the stream must be the resident path's, byte for byte -- same tiles, same arithmetic, only the address of a panel
    changes."""
    import numpy as np
    import torch

    from frackyfrac_b200 import engine, synth
    from tests.helpers import oracle_flat, rel_err

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree = synth.random_tree(900, 401)
    rp, col, val = synth.random_table(tree, 1300, 0.04, 402, integer_counts=False)
    m = rp[1]
    col[9 * m:10 * m] = col[:m]; val[9 * m:10 * m] = val[:m] * (1 + 1e-4 * (np.arange(m) % 3 == 0))   # fix-up territory
    one = engine.Context(0)
    ref = {}
    for normalize in (1, 2):
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, normalize=normalize, path=engine.PATH_FAST, ctx=one) as job:
            ref[normalize] = _stream(job)
    one.close()
    want = oracle_flat(tree, (rp, col, val), True)
    assert rel_err(ref[1], want).max() < 1e-5
    for nd in [k for k in (2, 4, 8) if k <= n_gpu]:
        ctx = engine.Context(devices=list(range(nd)))
        monkeypatch.setenv("FRC_CAPACITY", "1")
        for normalize in (1, 2):
            for band_rows, slab in ((0, "0"), (128, "128")):
                monkeypatch.setenv("FRC_WS_SLAB", slab)
                with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, normalize=normalize, path=engine.PATH_FAST,
                                ctx=ctx, band_rows=band_rows) as job:
                    got = _stream(job)
                    info = job.info()
                # the other devices' shards visited this one: their panels crossed NVLink
                assert info.n_devices == nd and info.gather_bytes > 4 * tree.n_nodes * 128 * nd
                assert np.array_equal(got, ref[normalize], equal_nan=True), (nd, normalize, band_rows)
        monkeypatch.setenv("FRC_CAPACITY", "0")
        monkeypatch.delenv("FRC_WS_SLAB")
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, path=engine.PATH_FAST, ctx=ctx) as job:
            assert np.array_equal(_stream(job), ref[1], equal_nan=True)
        ctx.close()


def test_weighted_capacity_mode_counts_each_group_once(built, monkeypatch):
    """In capacity mode one fix-up output serves all the bands of a row-shard group: its flagged pairs and its
    distances below fp32's range must reach frc_job_info once per pass, and frc_chunk_exceptions must hand each of
    those distances out with the band it lies in -- exactly as the resident path does, and again after a restart."""
    import numpy as np
    import torch

    from frackyfrac_b200 import engine, synth

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree = synth.random_tree(900, 411)
    tree.length = tree.length.copy()
    # two sibling leaves a, b on branches of 1e-60: samples that differ only in which of them they hold lie ~1e-60
    # apart, below fp32's range
    kids = {}
    for v in range(1, tree.n_nodes):
        kids.setdefault(int(tree.parent[v]), []).append(v)
    leaves = set(tree.leaf_ids.tolist())
    a, b = next(c for c in kids.values() if len(c) == 2 and set(c) <= leaves)
    tree.length[[a, b]] = 1e-60
    n = 2100  # with band_rows = 128: at least two bands in every row-shard group on up to 8 devices
    rp, col, val = synth.random_table(tree, n, 0.04, 412, integer_counts=False)
    rows = []
    for s in range(n):
        c, v = col[rp[s]:rp[s + 1]], val[rp[s]:rp[s + 1]]
        keep = (c != a) & (c != b)
        rows.append((c[keep], v[keep]))
    c0, v0 = rows[0]
    rows[9] = (c0, v0 * (1 + 1e-4 * (np.arange(len(v0)) % 3 == 0)))  # a near duplicate of sample 0: fix-up territory
    variants = list(range(40, n, 100))  # sample 0 plus leaf a or leaf b, spread over many bands
    for k, s in enumerate(variants):
        rows[s] = (np.append(c0, a if k % 2 else b), np.append(v0, 1.0))
    rp = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int64)
    col = np.concatenate([c for c, _ in rows]).astype(np.int32)
    val = np.concatenate([v for _, v in rows])
    n_ab = (len(variants) // 2) * ((len(variants) + 1) // 2)

    def drain(job):
        got, ex, expect = [], [], 0
        for first, d in job.chunks_f32():
            assert first == expect, (first, expect)
            xi, xv = job.exceptions()
            assert ((xi >= first) & (xi < first + len(d))).all(), (first, len(d), xi)
            ex += zip(xi.tolist(), xv.tolist())
            got.append(d)
            expect += len(d)
        i = job.info()
        return np.concatenate(got), sorted(ex), (i.n_pairs_total, i.flagged_pairs, i.exceptions, i.d2h_bytes)

    for nd in [k for k in (2, 4, 8) if k <= n_gpu]:
        ctx = engine.Context(devices=list(range(nd)))
        passes = {}
        for cap in ("0", "1"):
            monkeypatch.setenv("FRC_CAPACITY", cap)
            with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, path=engine.PATH_FAST, ctx=ctx,
                            band_rows=128) as job:
                passes[cap] = [drain(job)]
                job.restart()
                passes[cap].append(drain(job))
        got, ex, counts = passes["0"][0]
        assert len(ex) == n_ab and all(0 < x < 1e-38 for _, x in ex)
        assert counts == (n * (n - 1) // 2, counts[1], n_ab, 4 * n * (n - 1) // 2) and counts[1] > n_ab
        for cap in ("0", "1"):
            for k, (g, e, c) in enumerate(passes[cap]):
                assert g.tobytes() == got.tobytes(), (nd, cap, k)
                assert e == ex, (nd, cap, k)
                assert c == counts, (nd, cap, k, c, counts)
        ctx.close()


def test_cli_on_all_gpus_reproduces_the_reference_fixtures(built, tmp_path):
    """The CLI stand-in with every visible GPU behind it: the six testdata/*.want files, byte for byte."""
    import torch

    from frackyfrac_b200 import hostlib
    from tests import kat

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    golden = os.path.join(ROOT, "tests", "golden")
    env = dict(os.environ, FRCFRC_DEVICES=str(min(8, torch.cuda.device_count())))
    for fixture, sparse, weighted in kat.CLI:
        out = tmp_path / "got"
        cmd = [hostlib.CLI_PATH, "-i", os.path.join(golden, fixture + (".sparse" if sparse else ".dense")),
               "-t", os.path.join(golden, fixture + ".tree"), "-o", str(out)] + (["-s"] if sparse else []) + (["-w"] if weighted else [])
        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
        assert r.returncode == 0, r.stderr
        assert out.read_text() == open(os.path.join(golden, fixture + ".want")).read()
    # and a fast-path sized input: same bytes from 1 GPU and from all of them
    from frackyfrac_b200 import synth

    tree = synth.random_tree(3000, 7)
    rp, col, val = synth.random_table(tree, 1500, 0.03, 8)
    (tmp_path / "t.tree").write_text(synth.to_newick(tree))
    (tmp_path / "t.sparse").write_text(synth.to_sparse_text(tree, rp, col, val))
    outs = []
    for nd in ("1", env["FRCFRC_DEVICES"]):
        for w in ([], ["-w"]):
            o = tmp_path / f"o{nd}{len(w)}"
            r = subprocess.run([hostlib.CLI_PATH, "-s", "-i", str(tmp_path / "t.sparse"), "-t", str(tmp_path / "t.tree"), "-o", str(o),
                                "-p", "4"] + w, capture_output=True, text=True, env=dict(os.environ, FRCFRC_DEVICES=nd, FRCFRC_PATH="fast"))
            assert r.returncode == 0, r.stderr
            outs.append(o.read_bytes())
    assert outs[0] == outs[2] and outs[1] == outs[3] and outs[0] != outs[1] and len(outs[0]) > 5_000_000
