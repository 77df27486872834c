"""bench.py --dump-outputs: the distances of the value leg's last timed step, as the stream delivers them."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _host_stream(ctx, tree, csr):
    from frackyfrac_b200 import engine

    with engine.Job(tree.parent, tree.length, *csr, weighted=False, path=engine.PATH_FAST, ctx=ctx) as job:
        return np.concatenate([a for _, a in job.chunks_f32()])


def test_dump_outputs_is_the_distance_stream(gpu_ctx, tmp_path):
    """The whole triangle of the `tiny` config, bit for bit what frc_next_f32 hands a host caller."""
    import bench

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "tiny", "--steps", "2", "--warmup", "1",
                        "--quick", "--no-cpu", "--no-e2e", "--no-roofline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["distances.npy"]
    got = np.load(tmp_path / "distances.npy")
    _, tree, csr, samples, _, _ = bench.make_workload("tiny", 1)
    assert got.dtype == np.float32 and len(got) == samples * (samples - 1) // 2
    assert np.array_equal(got, _host_stream(gpu_ctx, tree, csr), equal_nan=True)


def test_dump_outputs_samples_a_large_triangle(gpu_ctx, tmp_path, monkeypatch):
    """Past DUMP_BYTES the dump is a fixed sample of pairs, with their flat indices, gathered across bands."""
    import bench
    from frackyfrac_b200 import engine

    monkeypatch.setattr(bench, "DUMP_BYTES", 120_000)
    _, tree, csr, samples, _, _ = bench.make_workload("tiny", 1)
    dump = bench.OutputDump(str(tmp_path), samples * (samples - 1) // 2, 0)
    with engine.Job(tree.parent, tree.length, *csr, weighted=False, path=engine.PATH_FAST, ctx=gpu_ctx, band_rows=128,
                    flags=engine.FLAG_NO_D2H) as job:
        dump.drain(job)
        assert job.info().n_bands_mine > 1
    dump.write(types.SimpleNamespace(dist=None, rank=0))
    idx = np.load(tmp_path / "distances_index.npy")
    got = np.load(tmp_path / "distances.npy")
    assert idx.dtype == np.float64 and got.dtype == np.float32
    assert len(got) == len(idx) > 5000 and 4 * len(got) + 8 * len(idx) <= 120_000 and (np.diff(idx) > 0).all()
    assert np.array_equal(got, _host_stream(gpu_ctx, tree, csr)[idx.astype(np.int64)], equal_nan=True)
