"""Query x reference distances: frc_create_cross.

A cross job stages [reference rows; empty rows up to q0 = n_ref rounded up to 256; query rows] as one table and
computes only the block of pairs (n_ref + q, r) of the triangle over [ref; query], streamed query-major with flat
index q * n_ref + r.  The CPU tests check the band and tile plans (csrc/plan.cpp) and the argument checks; the GPU
tests check that every route gives the triangle's bytes for those pairs, and the oracle, edge cases, the CLI and
several GPUs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import kat

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MB = 1024 * 1024


@pytest.fixture(scope="module")
def L(built):
    from frackyfrac_b200 import engine

    lib = engine.lib()
    lib.frc_debug_cross_bands.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int64]
    lib.frc_debug_cross_bands.restype = C.c_int64
    lib.frc_debug_cross_tiles.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64]
    lib.frc_debug_cross_tiles.restype = C.c_int64
    return lib


def cross_bands(L, n_ref, n_q, world, d2h, band_rows=0):
    n = L.frc_debug_cross_bands(n_ref, n_q, band_rows, world, int(d2h), 0, 8, None, 0)
    out = np.zeros((max(n, 1), 5), np.int64)
    L.frc_debug_cross_bands(n_ref, n_q, band_rows, world, int(d2h), 0, 8, out.ctypes.data, n)
    return out[:n]


def cross_tiles(L, row0, row1, n_ref, pair_tiles):
    n = L.frc_debug_cross_tiles(row0, row1, n_ref, int(pair_tiles), None, 0)
    out = np.zeros((max(n, 1), 2), np.int32)
    L.frc_debug_cross_tiles(row0, row1, n_ref, int(pair_tiles), out.ctypes.data, n)
    return out[:n]


# ------------------------------------------------------------------ CPU: the plan
@pytest.mark.parametrize("n_ref", [1, 127, 128, 129, 255, 256, 257, 1000])
def test_bands_partition_the_block(L, n_ref):
    q0 = -(-n_ref // 256) * 256
    for n_q in (1, 128, 129, 1000):
        for world in range(1, 9):
            for d2h in (False, True):
                b = cross_bands(L, n_ref, n_q, world, d2h)
                row0, row1, first, count, owner = b.T
                assert row0[0] == q0 and row1[-1] == q0 + n_q, (n_q, world, d2h)
                assert (row0[1:] == row1[:-1]).all() and ((row0 - q0) % 128 == 0).all()
                assert (first == (row0 - q0) * n_ref).all() and (count == (row1 - row0) * n_ref).all()
                assert first[0] == 0 and first[-1] + count[-1] == n_q * n_ref and (count > 0).all()
                assert ((owner >= 0) & (owner < world)).all()
                # the byte caps of the triangle's plan, up to the rounding to whole query tiles
                cap = (96 if d2h else 1536) * MB
                assert (8 * count <= cap + 8 * 128 * n_ref).all()
    # explicit band_rows counts query rows (whole tiles); the empty block has no band
    b = cross_bands(L, 300, 1000, 1, True, band_rows=200)
    assert list(b[:, 1] - b[:, 0]) == [256, 256, 256, 232]
    assert len(cross_bands(L, 0, 100, 1, True)) == 0 and len(cross_bands(L, 100, 0, 1, True)) == 0


def test_bands_follow_the_byte_caps_and_owners(L):
    # 2000 x 50000 pairs of 8 bytes: 763 MB streamed -> bands of at most ~96 MB (+ one tile row of rounding)
    b = cross_bands(L, 50_000, 2000, 1, True)
    assert len(b) >= 8 and (8 * b[:, 3] <= 96 * MB + 8 * 128 * 50_000).all()
    # in HBM: one band on one device, two per device otherwise; owners balanced
    assert len(cross_bands(L, 5000, 1024, 1, False)) == 1
    b = cross_bands(L, 5000, 4096, 4, False)
    assert len(b) == 8 and sorted(np.bincount(b[:, 4], minlength=4)) == [2, 2, 2, 2]


@pytest.mark.parametrize("pair_tiles", [True, False])
def test_tiles_cover_each_band_rectangle_once(L, pair_tiles):
    for n_ref in (1, 127, 128, 129, 255, 256, 257, 1000):
        q0 = -(-n_ref // 256) * 256
        ref_tiles = -(-n_ref // 128)
        for n_q in (1, 128, 129, 1000):
            for row0, row1, _, _, _ in cross_bands(L, n_ref, n_q, 1, True, band_rows=256):
                t = cross_tiles(L, row0, row1, n_ref, pair_tiles)
                assert (t[:, 0] >= q0 // 128).all()
                want = {(ti, tj) for ti in range(row0 // 128, (row1 - 1) // 128 + 1) for tj in range(ref_tiles)}
                if pair_tiles:
                    assert (t[:, 1] % 2 == 0).all()
                    assert len({tuple(x) for x in t}) == len(t)
                    got = [(ti, tj + c) for ti, tj in t for c in (0, 1) if tj + c < ref_tiles]
                    assert (t[:, 1] + 1 < q0 // 128).all()   # the odd partner tile lies in the padding rows
                else:
                    got = [tuple(x) for x in t]
                assert len(got) == len(want) and set(got) == want, (n_ref, n_q, row0)


# ------------------------------------------------------------------ CPU: argument checks before the device
def _tables():
    parent, length = np.array([-1, 0, 0], np.int32), np.array([0, 1, 1.0])
    ref = (np.array([0, 1, 2], np.int64), np.array([1, 2], np.int32), np.array([1.0, 1.0]))
    query = (np.array([0, 1], np.int64), np.array([2], np.int32), np.array([1.0]))
    return parent, length, ref, query


def _create_error(**kw):
    from frackyfrac_b200 import engine

    parent, length, ref, query = _tables()
    a = dict(ref=ref, query=query, weighted=False)
    a.update(kw)
    with pytest.raises(engine.FrcError) as e:
        engine.Job(parent, length, *a.pop("ref"), **a)
    return e.value.code, str(e.value)


def test_argument_errors_come_before_the_device(built):
    import torch

    from frackyfrac_b200 import engine

    parent, length, ref, query = _tables()
    L = engine.lib()
    t = engine._Tree(3, parent.ctypes.data, length.ctypes.data)
    keep = []
    a = engine._csr(keep, *ref)
    o = engine._Opts(0, 1, -1, -1, 0, 1, 0, 0, 0, None)
    h = C.c_void_p()
    assert L.frc_create_cross(None, C.byref(t), C.byref(a), None, C.byref(o), C.byref(h)) == 1
    assert "query table is NULL" in L.frc_last_error(None).decode()

    code, msg = _create_error(ref=(np.array([0, 2, 1, 3], np.int64), np.array([1, 2, 1], np.int32), np.ones(3)))
    assert code == 1 and "reference table: row_ptr is not monotone at reference sample #2" in msg, msg
    code, msg = _create_error(query=(np.array([0, 1, 0, 1], np.int64), np.array([2], np.int32), np.array([1.0])))
    assert code == 1 and "query table: row_ptr is not monotone at query sample #2" in msg, msg
    code, msg = _create_error(query=(np.array([1, 1], np.int64), np.array([2], np.int32), np.array([1.0])))
    assert code == 1 and "query table: row_ptr[0] != 0" in msg, msg
    code, msg = _create_error(world=2, rank=0)
    assert code == 5 and "world" in msg, msg
    code, msg = _create_error(flags=engine.FLAG_SHARD_EMBED)
    assert code == 5 and "FRC_FLAG_SHARD_EMBED" in msg, msg
    code, msg = _create_error(weighted=False, normalize=0)
    assert code == 1 and "-l can only be used with weighted" in msg
    if not torch.cuda.is_available():
        code, _ = _create_error(ref=ref)   # a good call: only now the missing device shows
        assert code in (2, 5)


# ------------------------------------------------------------------ GPU
def _table(tree, n, seed, dup_of=None):
    """n samples over the tree; with dup_of = (rp, col, val), the first rows are exact and near copies of its rows
    (presence: one leaf dropped) so that both fix-ups run."""
    from frackyfrac_b200 import synth

    rp, col, val = synth.random_table(tree, n, 0.08, seed, integer_counts=False)
    rows = [(col[rp[s]:rp[s + 1]].copy(), val[rp[s]:rp[s + 1]].copy()) for s in range(n)]
    if dup_of is not None:
        drp, dcol, dval = dup_of
        rng = np.random.default_rng(seed)
        for k in range(min(6, n, len(drp) - 1)):
            c, v = dcol[drp[k]:drp[k + 1]].copy(), dval[drp[k]:drp[k + 1]].copy()
            if k % 3 == 1:
                v = v * (1.0 + 1e-4 * rng.random(len(v)))
            elif k % 3 == 2 and len(c) > 1:
                c, v = c[1:], v[1:]
            rows[k] = (c, v)
    if n > 7:
        rows[7] = (rows[7][0][:0], rows[7][1][:0])   # an empty sample
    rp = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int64)
    col = np.concatenate([c for c, _ in rows]).astype(np.int32) if n else np.zeros(0, np.int32)
    val = np.concatenate([v for _, v in rows]) if n else np.zeros(0)
    return rp, col, val


def _concat(a, b):
    return (np.concatenate([a[0], a[0][-1] + b[0][1:]]).astype(np.int64), np.concatenate([a[1], b[1]]),
            np.concatenate([a[2], b[2]]))


def _block(tri, n_ref, n_q):
    i = n_ref + np.arange(n_q, dtype=np.int64)
    return tri[(i * (i - 1) // 2)[:, None] + np.arange(n_ref, dtype=np.int64)[None, :]].ravel()


def _stream(job, mode):
    """The whole stream: 'f64' (frc_next), 'f32' (frc_next_f32 + exceptions, widened) or 'dev' (FRC_FLAG_NO_D2H)."""
    import torch

    n = job.info().n_pairs_total
    out = np.full(n, -7.0)
    f32 = job.info().value_bytes == 4
    if mode == "f64":
        for first, a in job.chunks():
            out[first:first + len(a)] = a
        return out
    if mode == "f32":
        for first, a in job.chunks_f32():
            d = a.astype(np.float64)
            xi, xv = job.exceptions()
            d[xi - first] = xv
            out[first:first + len(a)] = d
        return out
    nxt = job.next_raw_f32 if f32 else job.next_raw
    while True:
        addr, first, cnt = nxt()
        if cnt == 0:
            return out
        dev = type("D", (), {})()
        dev.__cuda_array_interface__ = {"shape": (cnt,), "typestr": "<f4" if f32 else "<f8", "data": (addr, False),
                                        "version": 2}
        out[first:first + cnt] = torch.as_tensor(dev, device="cuda").cpu().numpy().astype(np.float64)


_TREES = {}


def _tree(neg):
    from frackyfrac_b200 import synth

    if neg not in _TREES:
        tree = synth.random_tree(300, 71)
        if neg:
            tree.length = tree.length.copy()
            tree.length[np.random.default_rng(72).random(tree.n_nodes) < 0.1] *= -1.0
        _TREES[neg] = tree
    return _TREES[neg]


ROUTES = {   # name: (weighted, normalize, path, flags, environment, negative lengths, operand_kind)
    "exact-uw": (False, 1, 1, 0, {}, False, 0),
    "exact-w1": (True, 1, 1, 0, {}, False, 0),
    "exact-w0": (True, 0, 1, 0, {}, False, 0),
    "exact-w2": (True, 2, 1, 0, {}, False, 0),
    "u8-int": (False, 1, 0, 0, {}, False, 2),
    "u8-f64": (False, 1, 0, 0, {"FRC_U8_ACC": "f64"}, False, 2),
    "bf16": (False, 1, 0, 2, {}, False, 1),
    "bits": (False, 1, 0, 8, {}, False, 3),
    "w1": (True, 1, 0, 0, {}, False, 0),
    "w2": (True, 2, 0, 0, {}, False, 0),
    "w1-neg": (True, 1, 0, 0, {}, True, 0),
    "w2-neg": (True, 2, 0, 0, {}, True, 0),
    "l-tiles": (True, 0, 0, 16, {}, False, 0),
}
SIZES = [(1, 1), (129, 130), (300, 513), (1000, 130), (1, 513), (257, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("prune", [False, True])
@pytest.mark.parametrize("route", list(ROUTES))
def test_block_is_the_triangles_bytes(gpu_ctx, monkeypatch, route, prune):
    """Every route: the cross stream (f64, f32 and the NO_D2H device bands, many bands) equals the triangle's entries
    (n_ref + q, r) over [ref; query] byte for byte."""
    from frackyfrac_b200 import engine

    weighted, normalize, path, flags, env, neg, kind = ROUTES[route]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    flags |= engine.FLAG_PRUNE if prune else 0
    tree = _tree(neg)
    for n_ref, n_q in SIZES:
        ref = _table(tree, n_ref, 100 + n_ref)
        query = _table(tree, n_q, 200 + n_q, dup_of=ref)
        kw = dict(weighted=weighted, normalize=normalize, path=path, ctx=gpu_ctx)
        full = _concat(ref, query)
        modes = ("f64", "dev") if path == engine.PATH_EXACT else ("f64", "f32", "dev")
        with engine.Job(tree.parent, tree.length, *full, flags=flags, **kw) as job:   # (fast paths: fp32, widened)
            want = _block(_stream(job, "f64"), n_ref, n_q)
        for mode in modes:
            fl = flags | (engine.FLAG_NO_D2H if mode == "dev" else 0)
            with engine.Job(tree.parent, tree.length, *ref, query=query, flags=fl, band_rows=128, **kw) as job:
                info = job.info()
                assert info.n_pairs_total == n_q * n_ref and info.n_bands_total == -(-n_q // 128)
                assert info.operand_kind == kind and info.path_taken == path
                got = _stream(job, mode)
            assert got.tobytes() == want.tobytes(), (route, n_ref, n_q, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("weighted,normalize,flags", [(False, 1, 0), (True, 1, 0), (True, 2, 0), (True, 0, 16)])
def test_oracle(gpu_ctx, weighted, normalize, flags):
    from frackyfrac_b200 import engine, synth
    from oracle import oracle as orc
    from tests.helpers import rel_err

    tree = synth.random_tree(3000, 81)
    ref = _table(tree, 700, 82)
    query = _table(tree, 300, 83, dup_of=ref)
    got = engine.unifrac_cross(tree.parent, tree.length, ref, query, weighted, normalize, path=engine.PATH_FAST,
                               flags=flags, ctx=gpu_ctx)
    assert got.shape == (300, 700)
    rows, _, _ = orc.unifrac_rows(orc.Table.from_csr(*_concat(ref, query)), orc.Tree.from_flat(tree.parent, tree.length),
                                  weighted, normalize, 4, 700, 1000)
    i = 700 + np.arange(300)
    want = rows[(i * (i - 1) // 2 - 700 * 699 // 2)[:, None] + np.arange(700)[None, :]]
    assert rel_err(got.ravel(), want.ravel()).max() < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("weighted,path", [(False, 0), (True, 0), (False, 1), (True, 1)])
def test_edge_cases(gpu_ctx, weighted, path):
    from frackyfrac_b200 import engine

    tree = _tree(False)
    ref = _table(tree, 300, 91)
    query = _table(tree, 130, 92, dup_of=ref)
    kw = dict(weighted=weighted, path=path, ctx=gpu_ctx)
    none = (np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0))
    for a, b in ((none, query), (ref, none), (none, none)):
        with engine.Job(tree.parent, tree.length, *a, query=b, **kw) as job:
            assert job.info().n_pairs_total == 0 and job.drain() == 0
    # empty samples on both sides: the pair of two empty samples is NaN (0/0), as in the triangle
    got = engine.unifrac_cross(tree.parent, tree.length, ref, query, **kw)
    assert np.isnan(got[7, 7]) and not np.isnan(got[0, 0]) and got[0, 0] == 0.0   # query 0 is a copy of ref 0
    # frc_restart gives the same bytes
    with engine.Job(tree.parent, tree.length, *ref, query=query, band_rows=128, **kw) as job:
        a = _stream(job, "f64")
        job.restart()
        assert _stream(job, "f64").tobytes() == a.tobytes()
    # a bad entry is reported with its table and row
    col = query[1].copy()
    col[query[0][2]] = tree.n_nodes
    with pytest.raises(engine.FrcError) as e:
        engine.Job(tree.parent, tree.length, *ref, query=(query[0], col, query[2]), **kw)
    assert e.value.code == 1 and f"query sample #3: entry 1 (node {tree.n_nodes}): node id out of range" in str(e.value)
    col = ref[1].copy()
    col[ref[0][4]] = -1
    with pytest.raises(engine.FrcError) as e:
        engine.Job(tree.parent, tree.length, ref[0], col, ref[2], query=query, **kw)
    assert e.value.code == 1 and "reference sample #5: entry 1 (node -1): node id out of range" in str(e.value)


def _split_text(text, sparse, k):
    lines = text.splitlines(keepends=True)
    head, rows = ([], lines) if sparse else (lines[:1], lines[1:])
    return "".join(head + rows[:k]), "".join(head + rows[k:])


CLI_CASES = [(f, ".sparse" if s else ".dense", s, w, 1) for f, s, w in kat.CLI] + [
    ("synth_a", ".dense", False, False, 1), ("synth_a", ".sparse", True, True, 1), ("synth_a", ".dense", False, True, 1),
    ("synth_a", ".sparse", True, True, 0), ("wtd", ".sparse", True, True, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("fixture,suffix,sparse,weighted,normalize", CLI_CASES)
def test_cli(built, tmp_path, fixture, suffix, sparse, weighted, normalize):
    """FRCFRC_QUERY: -i is the reference, the output is the query x reference block in (q1,r1) ... (q1,rR), (q2,r1)
    order, byte for byte the oracle's lines for those pairs of the whole table."""
    from frackyfrac_b200 import hostlib
    from oracle import oracle as orc

    text = open(os.path.join(GOLDEN, fixture + suffix)).read()
    tree_text = open(os.path.join(GOLDEN, fixture + ".tree")).read()
    n = len(text.splitlines()) - (0 if sparse else 1)
    k = max(1, n // 3)
    ref_text, query_text = _split_text(text, sparse, k)
    (tmp_path / "ref").write_text(ref_text)
    (tmp_path / "query").write_text(query_text)
    out = tmp_path / "got"
    cmd = [hostlib.CLI_PATH, "-t", os.path.join(GOLDEN, fixture + ".tree"), "-i", str(tmp_path / "ref"), "-o", str(out)]
    cmd += (["-s"] if sparse else []) + (["-w"] if weighted else []) + (["-l"] if normalize != 1 else [])
    r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, FRCFRC_QUERY=str(tmp_path / "query")))
    assert r.returncode == 0, r.stderr
    tri = orc.unifrac(orc.Table.parse(text, sparse), orc.Tree.parse(tree_text), weighted, normalize, 1)
    assert out.read_bytes() == hostlib.format_lines(_block(tri, k, n - k))


@pytest.mark.gpu
def test_several_gpus(built):
    import torch

    from frackyfrac_b200 import engine

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree = _tree(False)
    ref = _table(tree, 1000, 111)
    query = _table(tree, 513, 112, dup_of=ref)
    for weighted, normalize, flags in ((False, 1, 0), (True, 1, 0), (True, 0, engine.FLAG_L_TILES)):
        kw = dict(weighted=weighted, normalize=normalize, path=engine.PATH_FAST, flags=flags, band_rows=128)
        one = engine.unifrac_cross(tree.parent, tree.length, ref, query, device=0, **kw)
        for devices in ([0, 1], -1):
            got = engine.unifrac_cross(tree.parent, tree.length, ref, query, devices=devices, **kw)
            assert got.tobytes() == one.tobytes(), (weighted, normalize, devices)
