"""Pruning the tree to the table's support: FRC_FLAG_PRUNE.

A node whose subtree holds no listed leaf is 0 in every sample and adds nothing; a surviving non-root node with one
surviving child holds the same value as that child in every sample, so the fast paths merge such chains into their
lowest node (lengths summed) and weigh that node by the chain's node count in the default normaliser.  DESIGN.md has
the rule and its proof.  The CPU tests check the pruning itself (csrc/plan.cpp) against a plain-Python restatement and
the rule against the oracle; the GPU tests run every path on the pruned tree."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests import kat
from tests.helpers import oracle_flat, rel_err

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def L(built):
    from frackyfrac_b200 import engine

    lib = engine.lib()
    lib.frc_debug_prune.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32] + [C.c_void_p] * 4
    lib.frc_debug_prune.restype = C.c_int32
    return lib


def debug_prune(L, parent, length, leaves, merge):
    """(parent, length, mult, new_of_old) of the pruned tree, as frc_create builds it."""
    B = len(parent)
    parent = np.ascontiguousarray(parent, np.int32)
    length = np.ascontiguousarray(length, np.float64)
    marks = np.zeros(B, np.uint8)
    marks[np.asarray(leaves, np.int64)] = 1
    op, ol, om, no = np.zeros(B, np.int32), np.zeros(B), np.zeros(B, np.int32), np.zeros(B, np.int32)
    n = L.frc_debug_prune(parent.ctypes.data, length.ctypes.data, B, marks.ctypes.data, int(merge), op.ctypes.data,
                          ol.ctypes.data, om.ctypes.data, no.ctypes.data)
    assert n >= 1
    return op[:n], ol[:n], om[:n], no


# ------------------------------------------------------------------ the rule, restated in plain Python
def py_prune(parent, length, leaves, merge):
    B = len(parent)
    in_s = [False] * B
    in_s[0] = True
    for leaf in leaves:
        v = int(leaf)
        while not in_s[v]:
            in_s[v] = True
            v = int(parent[v])
    kids = [0] * B
    for v in range(1, B):
        if in_s[v]:
            kids[parent[v]] += 1
    drop = [bool(merge) and v > 0 and in_s[v] and kids[v] == 1 for v in range(B)]
    new, par, ln, mu = [-1] * B, [], [], []
    for v in range(B):
        if not in_s[v] or drop[v]:
            continue
        chain, p = [], int(parent[v]) if v else -1
        while p >= 0 and drop[p]:
            chain.append(p)
            p = int(parent[p])
        s = float(length[v])
        if chain:                        # summed from the top of the chain down
            s = float(length[chain[-1]])
            for u in reversed(chain[:-1]):
                s += float(length[u])
            s += float(length[v])
        new[v] = len(par)
        par.append(new[p] if p >= 0 else -1)
        ln.append(s)
        mu.append(len(chain) + 1)
    return np.array(par, np.int32), np.array(ln), np.array(mu, np.int32), np.array(new, np.int32), np.array(in_s)


def _is_preorder(parent):
    path = [0]
    for v in range(1, len(parent)):
        if not (0 <= parent[v] < v) or parent[v] not in path:
            return False
        path = path[:path.index(parent[v]) + 1] + [v]
    return True


def restated(parent, length, mult, rp, col, val, weighted, normalize):
    """Distances on a (pruned) tree in IterPairs order; mult = None drops the multiplicities from the normaliser."""
    B, N = len(parent), len(rp) - 1
    E = np.zeros((N, B))
    K = np.full((N, B), -1, np.int64)
    for s in range(N):
        c = col[rp[s]:rp[s + 1]]
        E[s, c] = val[rp[s]:rp[s + 1]]
        K[s, c] = c
    for v in range(B - 1, 0, -1):
        E[:, parent[v]] += E[:, v]
        K[:, parent[v]] = np.maximum(K[:, parent[v]], K[:, v])
    if weighted and normalize == 1:
        T = E @ (np.ones(B) if mult is None else mult)
        E = np.divide(E, T[:, None], out=np.zeros_like(E), where=T[:, None] > 0)
    out = []
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(N):
            a, b = E[i], E[:i]
            if not weighted:
                pa, pb = a > 0, b > 0
                num, den = (pa ^ pb) @ length, (pa | pb) @ length
            else:
                diff = np.abs(a - b)
                if normalize == 0:
                    diff = np.where(K[i] == K[:i], diff, a + b)
                num, den = diff @ length, (a + b) @ length
            out.extend(num / den)
    return np.array(out)


def _observed_table(tree, n_samples, n_observed, per_sample, seed, integer_counts=False):
    """A table whose samples draw from a few observed leaves of a large tree."""
    rng = np.random.default_rng(seed)
    pool = rng.choice(tree.leaf_ids, size=n_observed, replace=False)
    rp = np.arange(n_samples + 1, dtype=np.int64) * per_sample
    col = np.concatenate([rng.choice(pool, size=per_sample, replace=False) for _ in range(n_samples)]).astype(np.int32)
    val = np.ceil(rng.lognormal(3.0, 1.5, len(col)))
    if not integer_counts:
        val = val * rng.random(len(val)) + 1e-3
    return rp, col, val


def _small_cases():
    from frackyfrac_b200 import synth

    out = []
    for shape, seed in (("random", 3), ("caterpillar", 4), ("balanced", 5)):
        tree = synth.random_tree(300, seed, shape=shape)
        length = tree.length.copy()
        length[np.random.default_rng(seed).random(len(length)) < 0.1] = 0.0
        tree = synth.Tree(tree.parent, length, tree.leaf_ids, tree.names)
        rp, col, val = _observed_table(tree, 12, 30, 8, seed + 10)
        rp = np.concatenate([rp[:4], rp[3:4], rp[3:]])              # samples 3 and 4 are empty
        out.append((tree, (rp, col, val)))
    return out


def test_prune_matches_the_restatement(L):
    """(a) frc_debug_prune against the plain-Python rule: random, caterpillar and balanced trees, leaf subsets from
    none to all, merge on and off."""
    from frackyfrac_b200 import synth

    rng = np.random.default_rng(7)
    for shape in ("random", "caterpillar", "balanced"):
        for n in (1, 2, 3, 57, 400):
            tree = synth.random_tree(n, 11 + n, shape=shape)
            subsets = [[], tree.leaf_ids[:1], tree.leaf_ids, rng.choice(tree.leaf_ids, size=max(1, n // 7), replace=False),
                       rng.choice(tree.leaf_ids, size=max(1, n // 2), replace=False)]
            for leaves in subsets:
                for merge in (0, 1):
                    par, ln, mu, new = debug_prune(L, tree.parent, tree.length, leaves, merge)
                    wpar, wln, wmu, wnew, in_s = py_prune(tree.parent, tree.length, leaves, merge)
                    assert np.array_equal(par, wpar) and np.array_equal(ln, wln) and np.array_equal(mu, wmu)
                    assert np.array_equal(new, wnew)
                    kept = new >= 0
                    assert kept[0] and new[0] == 0 and par[0] == -1               # root kept, still the root
                    assert not (kept & ~in_s).any()                                # only support nodes survive
                    if not merge:
                        assert np.array_equal(kept, in_s) and (mu == 1).all()
                        assert np.array_equal(ln, tree.length[kept])              # lengths verbatim
                    assert mu.sum() == in_s.sum()
                    assert _is_preorder(par)
                    assert (np.diff(new[kept]) == 1).all()                         # order preserved
                    lv = new[np.asarray(leaves, np.int64)]
                    assert (lv >= 0).all()
                    assert not np.isin(lv, par).any()                              # listed leaves stay leaves
                    if merge:
                        assert len(par) <= max(1, 2 * len(np.unique(leaves)))


def test_prune_refuses_a_tree_that_is_not_preorder(L):
    """(b) frc_create prunes nothing when parent[] fails the pre-order check (the unpruned walks then report it)."""
    marks = np.ones(4, np.uint8)
    out = [np.zeros(4, np.int32), np.zeros(4), np.zeros(4, np.int32), np.zeros(4, np.int32)]
    for parent, bad in (([-1, 0, 0, 1], 3), ([-1, 0, 3, 1], 2)):
        p = np.array(parent, np.int32)
        n = L.frc_debug_prune(p.ctypes.data, np.ones(4).ctypes.data, 4, marks.ctypes.data, 1, *[a.ctypes.data for a in out])
        assert n == -1 - bad


@pytest.mark.parametrize("weighted,normalize", [(False, 1), (True, 1), (True, 2), (True, 0)])
def test_rule_on_the_pruned_tree_matches_the_oracle(L, weighted, normalize):
    """(c) The distances restated on the merged tree, with multiplicities in the default normaliser, are the oracle's
    on the whole tree to 1e-12 (normalize = 0 through the key rule); without the multiplicities the default
    normaliser misses by far more than 1e-5."""
    worst_without = 0.0
    for tree, (rp, col, val) in _small_cases():
        want = oracle_flat(tree, (rp, col, val), weighted, normalize)
        leaves = np.unique(col)
        par, ln, mu, new = debug_prune(L, tree.parent, tree.length, leaves, 1)
        assert len(par) < tree.n_nodes // 4
        got = restated(par, ln, mu, rp, new[col], val, weighted, normalize)
        assert np.isnan(want).any()
        e = rel_err(got, want)
        assert e.max() < 1e-12, e.max()
        worst_without = max(worst_without, rel_err(restated(par, ln, None, rp, new[col], val, weighted, normalize),
                                                   want).max())
    if weighted and normalize == 1:
        assert worst_without > 1e-4, worst_without
    else:
        assert worst_without < 1e-12


# ------------------------------------------------------------------ GPU
_BIG = {}


def _big(shape):
    """A 20k-leaf tree and a table of 200 samples over 300 observed leaves."""
    from frackyfrac_b200 import synth

    if shape not in _BIG:
        seed = {"random": 21, "caterpillar": 22, "balanced": 23}[shape]
        tree = synth.random_tree(20_000, seed, shape=shape)
        _BIG[shape] = (tree, _observed_table(tree, 200, 300, 25, seed + 100))
    return _BIG[shape]


def _run(tree, csr, weighted, normalize=1, path=None, flags=0, ctx=None, f32=False, **kw):
    from frackyfrac_b200 import engine

    rp, col, val = csr
    with engine.Job(tree.parent, tree.length, rp, col, val, weighted=weighted, normalize=normalize,
                    path=engine.PATH_FAST if path is None else path, ctx=ctx, flags=flags, **kw) as job:
        if not f32:
            got = [a for _, a in job.chunks()]
        else:
            got = []
            for first, a in job.chunks_f32():
                d = a.astype(np.float64)
                xi, xv = job.exceptions()
                d[xi - first] = xv
                got.append(d)
        return (np.concatenate(got) if got else np.zeros(0)), job.info()   # (counters of the delivered bands)


def _with_lengths(tree, negative):
    from frackyfrac_b200 import synth

    length = tree.length.copy()
    if negative:
        neg = np.random.default_rng(5).random(len(length)) < 0.05
        length[neg] = -0.1 * length[neg]
    return synth.Tree(tree.parent, length, tree.leaf_ids, tree.names)


FAST_MODES = [  # (id, weighted, normalize, extra flags, operand_kind, negative lengths)
    ("u8", False, 1, 0, 2, False), ("bf16", False, 1, 2, 1, False), ("bits", False, 1, 8, 3, False),
    ("w1", True, 1, 0, 0, False), ("w2", True, 2, 0, 0, False), ("w0_tiles", True, 0, 16, 0, False),
    ("uw_neg", False, 1, 0, 1, True), ("w1_neg", True, 1, 0, 0, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "caterpillar", "balanced"])
@pytest.mark.parametrize("mode", FAST_MODES, ids=[m[0] for m in FAST_MODES])
def test_fast_paths_match_the_oracle_on_the_whole_tree(gpu_ctx, L, shape, mode):
    """(d) Every fast kernel on the pruned tree is within 1e-5 of the oracle on the unpruned tree; the weighted paths
    contract over round_up(B', 64) nodes."""
    from frackyfrac_b200 import engine

    _, weighted, normalize, flags, kind, negative = mode
    tree, csr = _big(shape)
    tree = _with_lengths(tree, negative)
    want = oracle_flat(tree, csr, weighted, normalize, threads=os.cpu_count() or 4)
    got, info = _run(tree, csr, weighted, normalize, flags=flags | engine.FLAG_PRUNE, ctx=gpu_ctx)
    assert info.path_taken == engine.PATH_FAST
    e = rel_err(got, want)
    assert e.max() < 1e-5, f"max rel err {e.max():.3e}"
    par, _, _, _ = debug_prune(L, tree.parent, tree.length, np.unique(csr[1]), 1)
    assert len(par) <= 600
    if weighted:
        assert info.n_nodes_padded == (len(par) + 63) // 64 * 64
    else:
        assert info.operand_kind == kind and info.n_nodes_padded < 1024


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "caterpillar"])
def test_exact_path_is_byte_identical(gpu_ctx, shape):
    """(e) The exact path prunes without merging: flag on and off give the same bytes in every mode, the -l list walk
    included."""
    from frackyfrac_b200 import engine

    tree, csr = _big(shape)
    for weighted, normalize in ((False, 1), (True, 1), (True, 2), (True, 0)):
        off, i0 = _run(tree, csr, weighted, normalize, path=engine.PATH_EXACT, ctx=gpu_ctx)
        on, i1 = _run(tree, csr, weighted, normalize, path=engine.PATH_EXACT, flags=engine.FLAG_PRUNE, ctx=gpu_ctx)
        assert i1.path_taken == engine.PATH_EXACT and i1.n_nodes_padded < i0.n_nodes_padded
        assert off.tobytes() == on.tobytes(), (weighted, normalize)


@pytest.mark.gpu
@pytest.mark.parametrize("fixture,sparse,weighted", kat.CLI)
def test_cli_golden_with_the_flag(built, tmp_path, fixture, sparse, weighted):
    """(f) The CLI stand-in with FRCFRC_PRUNE=1 prints the committed bytes (uwtd2 has a leaf no sample holds)."""
    from frackyfrac_b200 import hostlib

    out = tmp_path / "got"
    cmd = [hostlib.CLI_PATH, "-i", os.path.join(GOLDEN, fixture + (".sparse" if sparse else ".dense")),
           "-t", os.path.join(GOLDEN, fixture + ".tree"), "-o", str(out)]
    cmd[1:1] = (["-s"] if sparse else []) + (["-w"] if weighted else [])
    r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, FRCFRC_PRUNE="1"))
    assert r.returncode == 0, r.stderr
    assert out.read_text() == open(os.path.join(GOLDEN, fixture + ".want")).read()


@pytest.mark.gpu
@pytest.mark.parametrize("fixture,suffix,sparse,tag,weighted,normalize", kat.SYNTH)
def test_cli_synthetic_golden_with_the_flag(built, tmp_path, fixture, suffix, sparse, tag, weighted, normalize):
    from frackyfrac_b200 import hostlib

    out = tmp_path / "got"
    cmd = [hostlib.CLI_PATH, "-t", os.path.join(GOLDEN, fixture + ".tree"), "-i", os.path.join(GOLDEN, fixture + suffix),
           "-o", str(out)]
    cmd += (["-s"] if sparse else []) + (["-w"] if weighted else []) + (["-l"] if normalize != 1 else [])
    env = dict(os.environ, FRCFRC_PRUNE="1")
    if normalize == 2:
        env["FRCFRC_L"] = "documented"
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    assert out.read_text() == open(os.path.join(GOLDEN, f"{fixture}.{tag}.want")).read()


@pytest.mark.gpu
def test_nothing_to_prune_changes_no_byte(gpu_ctx, L):
    """(g) Every leaf observed and no unary node: the fast paths give the same bytes with and without the flag."""
    from frackyfrac_b200 import engine, synth

    tree = synth.random_tree(2000, 31)
    csr = synth.random_table(tree, 5000, 0.02, 32)
    par, _, _, _ = debug_prune(L, tree.parent, tree.length, np.unique(csr[1]), 1)
    assert len(par) == tree.n_nodes
    for weighted, normalize, flags in ((False, 1, 0), (False, 1, engine.FLAG_UW_BF16), (True, 1, 0), (True, 2, 0),
                                       (True, 0, engine.FLAG_L_TILES)):
        off, _ = _run(tree, csr, weighted, normalize, flags=flags, ctx=gpu_ctx, f32=True)
        on, _ = _run(tree, csr, weighted, normalize, flags=flags | engine.FLAG_PRUNE, ctx=gpu_ctx, f32=True)
        assert off.tobytes() == on.tobytes(), (weighted, normalize, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("weighted,normalize,flags", [(False, 1, 0), (True, 1, 0), (True, 2, 0), (True, 0, 16)])
def test_edge_cases_with_the_flag(gpu_ctx, weighted, normalize, flags):
    """(h) Identical samples give exactly 0, near-copies go through the fix-up, empty samples give NaN, a table without
    entries gives all NaN, fewer than two samples an empty stream, and the f32 and f64 streams agree."""
    from frackyfrac_b200 import engine

    flags |= engine.FLAG_PRUNE
    tree, (rp, col, val) = _big("random")
    rp, col, val = rp[:41].copy(), col[:rp[40]].copy(), val[:rp[40]].copy()
    m = int(rp[1])
    rng = np.random.default_rng(9)
    for k, eps in enumerate((1e-2, 1e-3, 1e-4, 1e-5, 1e-6), start=1):
        col[k * m:(k + 1) * m] = col[:m]
        val[k * m:(k + 1) * m] = val[:m] * (1.0 + eps * rng.random(m) * (rng.random(m) < 0.3))
    col[6 * m:7 * m] = col[:m]                                  # an exact copy of sample 0
    val[6 * m:7 * m] = val[:m]
    keep = np.ones(len(col), bool)
    keep[rp[8]:rp[10]] = False                                  # samples 8 and 9 empty
    lens = np.diff(rp)
    lens[8:10] = 0
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col, val = col[keep], val[keep]
    want = oracle_flat(tree, (rp, col, val), weighted, normalize)
    got, info = _run(tree, (rp, col, val), weighted, normalize, flags=flags, ctx=gpu_ctx)
    assert rel_err(got, want).max() < 1e-5
    assert got[6 * 5 // 2] == 0.0                               # pair (6, 0)
    assert np.isnan(got[9 * 8 // 2 + 8])                        # pair (9, 8)
    if weighted:                                                # (presence: the near-copies are exact copies)
        assert info.flagged_pairs >= 5
        near = [k * (k - 1) // 2 for k in range(1, 6)]          # pairs (k, 0)
        assert (np.abs(got[near] - want[near]) <= 1.2e-7 * want[near] + 1e-15).all()
    narrow, _ = _run(tree, (rp, col, val), weighted, normalize, flags=flags, ctx=gpu_ctx, f32=True)
    assert np.array_equal(narrow, got, equal_nan=True)
    empty = np.zeros(6, np.int64)
    got, _ = _run(tree, (empty, col[:0], val[:0]), weighted, normalize, flags=flags, ctx=gpu_ctx)
    assert len(got) == 10 and np.isnan(got).all()
    for n in (0, 1):
        got, info = _run(tree, (rp[:n + 1], col[:rp[n]], val[:rp[n]]), weighted, normalize, flags=flags, ctx=gpu_ctx)
        assert len(got) == 0 and info.n_pairs_total == 0


@pytest.mark.gpu
def test_bad_inputs_give_the_same_errors(gpu_ctx):
    """(i) Every invalid input is refused with the same status and message with and without the flag (original node
    ids in the messages)."""
    from frackyfrac_b200 import engine, synth

    tree = synth.random_tree(20, 61)
    rp, col, val = synth.random_table(tree, 3, 0.2, 62)
    internal = int(np.setdiff1d(np.arange(tree.n_nodes), tree.leaf_ids)[1])
    cases = []
    for k, bad in ((0, internal), (2, tree.n_nodes), (3, -1)):
        c = col.copy(); c[k] = bad
        cases += [dict(col=c, weighted=False), dict(col=c, weighted=True)]
    v = val.copy(); v[1] = 0.0
    cases.append(dict(val=v, weighted=True))
    v = val.copy(); v[2] = np.inf
    cases.append(dict(val=v, weighted=True))
    c = col.copy(); c[1] = c[0]
    cases.append(dict(col=c, weighted=True))
    p = tree.parent.copy(); p[3] = 7
    cases += [dict(parent=p, weighted=False), dict(parent=p, weighted=True, path=engine.PATH_EXACT)]
    ln = tree.length.copy(); ln[int(np.setdiff1d(np.arange(1, tree.n_nodes), col)[0])] = np.nan  # an unobserved node
    cases.append(dict(length=ln, weighted=True, path=engine.PATH_FAST))
    cases.append(dict(weighted=False, normalize=0))
    cases.append(dict(weighted=True, normalize=0, path=engine.PATH_FAST))
    cases.append(dict(parent=np.array([-1, 0, 0, 1], np.int32), length=np.ones(4), rp=np.array([0, 1, 2], np.int64),
                      col=np.array([2, 3], np.int32), val=np.ones(2), weighted=False))
    for case in cases:
        case = dict(case)
        args = [case.pop(k, d) for k, d in (("parent", tree.parent), ("length", tree.length), ("rp", rp), ("col", col),
                                           ("val", val))]
        errs = []
        for flags in (0, engine.FLAG_PRUNE):
            with pytest.raises(engine.FrcError) as e:
                engine.Job(*args, ctx=gpu_ctx, flags=flags, **case)
            errs.append((e.value.code, str(e.value)))
        assert errs[0] == errs[1], errs


@pytest.mark.gpu
def test_flag_over_several_gpus(built, monkeypatch):
    """(j) One process over 2 / 4 / 8 GPUs, sharded or not, gives the one-GPU stream byte for byte; the capacity mode
    (unkeyed weighted) gives the resident bytes."""
    import torch

    from frackyfrac_b200 import engine

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree, csr = _big("random")
    one = engine.Context(0)
    modes = ((False, 1, 0), (True, 1, 0), (True, 2, 0), (True, 0, engine.FLAG_L_TILES))
    ref = {m: _run(tree, csr, m[0], m[1], flags=m[2] | engine.FLAG_PRUNE, ctx=one)[0] for m in modes}
    one.close()
    for nd in (2, 4, 8):
        if nd > n_gpu:
            break
        for shard in ("1", "0"):
            monkeypatch.setenv("FRC_SHARD", shard)
            for m in modes:
                got, info = _run(tree, csr, m[0], m[1], flags=m[2] | engine.FLAG_PRUNE, devices=list(range(nd)))
                assert info.n_devices == nd
                assert np.array_equal(got, ref[m], equal_nan=True), (nd, shard, m)
    monkeypatch.setenv("FRC_SHARD", "1")
    monkeypatch.setenv("FRC_CAPACITY", "1")
    for m in modes[1:3]:
        got, _ = _run(tree, csr, m[0], m[1], flags=engine.FLAG_PRUNE, devices=[0, 1])
        assert np.array_equal(got, ref[m], equal_nan=True), m
