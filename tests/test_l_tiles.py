"""Flag -l as the reference codes it (normalize = 0) on the FP32 tile kernel: FRC_FLAG_L_TILES.

Without normalizeFlatNodes the reference's merge-join (frcfrc/unifrac.go:174-205) walks per-sample lists in
post-order.  Which nodes it pairs up has a closed form: with key_s(v) = the largest present leaf id under v,
node v takes the |a - b| branch iff both samples hold it and key_A(v) == key_B(v); every other present node is
added one-sided.  The CPU tests check that rule against the oracle and against a literal walk; the GPU tests run
the keyed tiles (csrc/weighted.cu) and their fix-up."""
import os
import subprocess

import numpy as np
import pytest

from tests.helpers import oracle_flat, rel_err

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

# a multifurcating tree with a name carried by two leaves ("a") and a name that is also an internal node's ("x")
NWK = "((a:0.1,b:0.25,c:0.7,a:0.3)x:0.5,(d:1.5,(e:0.125,f:0.3):0,x:0.9):0.05,g:2)r:0.75;"
NWK_TABLE = "a:0.3 d:7 x:5\nb:1.1 e:2 g:0.01\nc:3 f:1e-3 a:2\n\n\nd:1 e:1 f:1 g:1 x:2\nb:2 c:1 e:4\nb:1 c:3 e:2\n"


# ------------------------------------------------------------------ the rule, restated in plain Python
def _embed(parent, rp, col, val):
    """Raw subtree sums E[s][v] and keys K[s][v] (largest present leaf id under v, -1 when absent)."""
    B, N = len(parent), len(rp) - 1
    E = np.zeros((N, B))
    K = np.full((N, B), -1, np.int64)
    for s in range(N):
        c = col[rp[s]:rp[s + 1]]
        E[s, c] = val[rp[s]:rp[s + 1]]
        K[s, c] = c
    for v in range(B - 1, 0, -1):   # pre-order ids: every child after its parent
        p = parent[v]
        E[:, p] += E[:, v]
        K[:, p] = np.maximum(K[:, p], K[:, v])
    assert ((K >= 0) == (E > 0)).all()
    return E, K


def keyed_distances(parent, length, rp, col, val):
    """numer = sum_v len_v * (key_i(v) == key_j(v) ? |a - b| : a + b), denom = W_i + W_j, in IterPairs order."""
    E, K = _embed(parent, rp, col, val)
    out = []
    with np.errstate(invalid="ignore", divide="ignore"):
        for i in range(len(E)):
            for j in range(i):
                a, b = E[i], E[j]
                t = np.where(K[i] == K[j], np.abs(a - b), a + b)
                out.append(np.dot(length, t) / np.dot(length, a + b))
    return np.array(out)


def _post_order_lists(parent, E):
    B = len(parent)
    children = [[] for _ in range(B)]
    for v in range(1, B):
        children[parent[v]].append(v)
    order, stack = [], [(0, False)]
    while stack:
        v, done = stack.pop()
        if done:
            order.append(v)
            continue
        stack.append((v, True))
        stack.extend((c, False) for c in reversed(children[v]))
    return [[v for v in order if E[s, v] > 0] for s in range(len(E))]


def walk_matched(la, lb):
    """The nodes the reference's two-pointer walk over two post-order lists takes the |a - b| branch for."""
    i = j = 0
    matched = set()
    while i < len(la) and j < len(lb):
        if la[i] < lb[j]:
            i += 1
        elif la[i] > lb[j]:
            j += 1
        else:
            matched.add(la[i])
            i += 1
            j += 1
    return matched


def _cases():
    from frackyfrac_b200 import synth

    out = []
    for shape, seed in (("random", 3), ("caterpillar", 4), ("balanced", 5)):
        tree = synth.random_tree(70, seed, shape=shape)
        L = tree.length.copy()
        L[np.random.default_rng(seed).random(len(L)) < 0.1] = 0.0     # zero-length branches
        rp, col, val = synth.random_table(tree, 14, 0.15, seed + 10, integer_counts=False)
        rows = [(col[rp[s]:rp[s + 1]], val[rp[s]:rp[s + 1]]) for s in range(14)]
        rows[5] = (rows[0][0], rows[0][1][::-1].copy())               # sample 0's leaves with other values
        rows[3] = rows[9] = (rows[0][0][:0], rows[0][1][:0])          # two empty samples
        rp = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int64)
        col = np.concatenate([c for c, _ in rows]).astype(np.int32)
        val = np.concatenate([v for _, v in rows])
        out.append((tree.parent, L, rp, col, val))
    return out


def _newick_case():
    from frackyfrac_b200 import hostlib

    tree = hostlib.Tree(NWK)
    rp, col, val = hostlib.Table(NWK_TABLE, True).resolve(tree)
    return tree.parent, tree.length, rp, col, val


def _oracle(parent, length, rp, col, val, normalize):
    from oracle import oracle as orc

    return orc.unifrac(orc.Table.from_csr(rp, col, val), orc.Tree.from_flat(parent, length), True, normalize, 1)


def _close(got, want, tol):
    assert (np.isnan(got) == np.isnan(want)).all()
    ok = ~np.isnan(want)
    assert (np.abs(got[ok] - want[ok]) <= tol * np.abs(want[ok])).all(), np.max(np.abs(got[ok] - want[ok]))


def test_key_rule_reproduces_the_reference_walk(built):
    """(a) The key rule gives the oracle's normalize = 0 distances to 1e-12 and the literal walk's matched sets, on
    random, caterpillar and balanced trees with zero-length branches and an empty sample, and on a multifurcating
    Newick tree with a name on two leaves and a named internal node."""
    from oracle import oracle as orc

    cases = _cases() + [_newick_case()]
    for parent, length, rp, col, val in cases:
        got = keyed_distances(parent, length, rp, col, val)
        _close(got, _oracle(parent, length, rp, col, val, 0), 1e-12)
        assert np.isnan(got).any()                                   # the two empty samples: 0 / 0
        E, K = _embed(parent, rp, col, val)
        lists = _post_order_lists(parent, E)
        for i in range(len(E)):
            for j in range(i):
                rule = {v for v in range(len(parent)) if K[i, v] >= 0 and K[i, v] == K[j, v]}
                assert walk_matched(lists[i], lists[j]) == rule, (i, j)
    # the Newick case parsed by the oracle itself gives the same distances as the resolved arrays
    parent, length, rp, col, val = _newick_case()
    want = orc.unifrac(orc.Table.parse(NWK_TABLE, True), orc.Tree.parse(NWK), True, 0, 1)
    _close(keyed_distances(parent, length, rp, col, val), want, 1e-12)


def test_identical_leaf_sets_give_the_documented_value(built):
    """(b) When two samples hold the same leaves every key agrees, nothing is mis-paired, and normalize = 0 equals
    the documented -l (normalize = 2)."""
    for parent, length, rp, col, val in _cases() + [_newick_case()]:
        E, _ = _embed(parent, rp, col, val)
        as_coded = _oracle(parent, length, rp, col, val, 0)
        documented = _oracle(parent, length, rp, col, val, 2)
        same = [k for k, (i, j) in enumerate((i, j) for i in range(len(E)) for j in range(i))
                if ((E[i] > 0) == (E[j] > 0)).all() and (E[i] > 0).any()]
        assert same
        _close(as_coded[same], documented[same], 1e-12)
        _close(keyed_distances(parent, length, rp, col, val)[same], documented[same], 1e-12)


def test_flag_argument_handling_before_the_device(built):
    """(c) Without FRC_FLAG_L_TILES, path FAST with normalize = 0 is still refused ("as coded"); with it the options
    are valid and a box without a GPU reports the missing device instead."""
    import torch

    from frackyfrac_b200 import engine

    if torch.cuda.is_available():
        pytest.skip("runs on the CPU box (the GPU tests below run the same options on a device)")
    parent, length = np.array([-1, 0, 0], np.int32), np.array([0, 1, 1.0])
    rp, col, val = np.array([0, 1, 2], np.int64), np.array([1, 2], np.int32), np.array([1.0, 1.0])

    def code(**kw):
        with pytest.raises(engine.FrcError) as e:
            engine.Job(parent, length, rp, col, val, weighted=True, **kw)
        return e.value.code, str(e.value)

    c, msg = code(normalize=0, path=engine.PATH_FAST)
    assert c == 5 and "as coded" in msg
    for kw in (dict(normalize=0, path=engine.PATH_FAST), dict(normalize=0, path=engine.PATH_AUTO),
               dict(normalize=1, path=engine.PATH_FAST), dict(normalize=2, path=engine.PATH_FAST)):
        c, msg = code(flags=engine.FLAG_L_TILES, **kw)
        assert c in (2, 5) and "as coded" not in msg, (kw, c, msg)
    with pytest.raises(engine.FrcError) as e:   # -l still needs weighted (frcfrc.go:84-86), flag or not
        engine.Job(parent, length, rp, col, val, weighted=False, normalize=0, flags=engine.FLAG_L_TILES)
    assert e.value.code == 1


# ------------------------------------------------------------------ GPU
def _tiles(tree_parent, length, rp, col, val, ctx, path=None, **kw):
    from frackyfrac_b200 import engine

    with engine.Job(tree_parent, length, rp, col, val, weighted=True, normalize=0,
                    path=engine.PATH_FAST if path is None else path, ctx=ctx,
                    flags=engine.FLAG_L_TILES | kw.pop("flags", 0), **kw) as job:
        got = np.concatenate([a for _, a in job.chunks()]) if job.info().n_pairs_total else np.zeros(0)
        return got, job.info()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "caterpillar", "balanced"])
@pytest.mark.parametrize("lengths", ["prescaled", "negative"])
def test_tiles_match_the_oracle(gpu_ctx, shape, lengths):
    """(d) Key-matched tiles within 1e-5 of the reference's -l on three tree shapes, with non-negative lengths
    (pre-scaled operand) and with some negative ones (FFMA form)."""
    from frackyfrac_b200 import engine, synth

    tree = synth.random_tree(900, 41, shape=shape)
    L = tree.length.copy()
    if lengths == "negative":
        neg = np.random.default_rng(42).random(len(L)) < 0.05
        L[neg] = -0.1 * L[neg]
    tree = synth.Tree(tree.parent, L, tree.leaf_ids, tree.names)
    csr = synth.random_table(tree, 300, 0.03, 43, integer_counts=False)
    want = oracle_flat(tree, csr, True, 0)
    got, info = _tiles(tree.parent, tree.length, *csr, gpu_ctx)
    assert info.path_taken == engine.PATH_FAST and info.value_bytes == 4
    e = rel_err(got, want)
    assert e.max() < 1e-5, f"max rel err {e.max():.3e}"
    # the rule mis-pairs real nodes here: the documented -l differs
    assert rel_err(oracle_flat(tree, csr, True, 2), want).max() > 1e-3


@pytest.mark.gpu
def test_tiles_small_distances_go_through_the_fixup(gpu_ctx):
    """(e) Near-copies (relative perturbations 1e-2 .. 1e-7) are flagged and recomputed in fixed point with the keys
    of the panels: within 1.2e-7 after the fix-up (one fp32 rounding)."""
    from frackyfrac_b200 import synth

    tree = synth.random_tree(1200, 85)
    rp, col, val = synth.random_table(tree, 160, 0.04, 86, integer_counts=False)
    m = rp[1]
    rng = np.random.default_rng(87)
    for k, eps in enumerate((1e-2, 1e-3, 1e-4, 1e-5, 1e-6, 1e-7), start=1):
        col[k * m:(k + 1) * m] = col[:m]
        val[k * m:(k + 1) * m] = val[:m] * (1.0 + eps * rng.random(m) * (rng.random(m) < 0.2))
    col[7 * m:8 * m] = col[:m]               # an exact copy: 0 exactly
    val[7 * m:8 * m] = val[:m]
    want = oracle_flat(tree, (rp, col, val), True, 0)
    got, info = _tiles(tree.parent, tree.length, rp, col, val, gpu_ctx)
    assert (want[:21] < 1 / 32).all() and want[:21].min() < 1e-6
    assert info.flagged_pairs >= 21
    assert rel_err(got, want).max() < 1e-5
    assert (np.abs(got[:21] - want[:21]) <= 1.2e-7 * want[:21] + 1e-15).all()
    assert got[7 * 6 // 2] == 0.0            # pair (7, 0)


@pytest.mark.gpu
def test_tiles_empty_and_tiny_inputs(gpu_ctx):
    """(f) Two empty samples give NaN, an empty one against a non-empty one gives 1; fewer than two samples give an
    empty stream."""
    from frackyfrac_b200 import engine, synth

    tree = synth.random_tree(50, 3)
    rp, col, val = synth.random_table(tree, 4, 0.1, 4)
    m = rp[1]
    rp = np.array([0, m, m, 2 * m, 2 * m], np.int64)  # samples 1 and 3 empty
    got, _ = _tiles(tree.parent, tree.length, rp, col[:2 * m], val[:2 * m], gpu_ctx)
    want = oracle_flat(tree, (rp, col[:2 * m], val[:2 * m]), True, 0)
    assert np.isnan(want[4]) and np.isnan(got[4])     # pair (3, 1)
    assert got[0] == 1.0 and want[0] == 1.0           # pair (1, 0)
    assert rel_err(got, want).max() < 1e-5
    for n in (0, 1):
        for path in (engine.PATH_AUTO, engine.PATH_FAST):
            got, info = _tiles(tree.parent, tree.length, rp[:n + 1], col[:rp[n]], val[:rp[n]], gpu_ctx, path=path)
            assert len(got) == 0 and info.n_pairs_total == 0 and info.n_bands_total == 0


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["synth_a", "synth_b"])
def test_auto_with_the_flag(gpu_ctx, fixture):
    """(g) AUTO + flag keeps the AUTO rule of every mode: a small input takes the bit-exact walk (the committed
    bytes), a large one the tiles."""
    from frackyfrac_b200 import engine, hostlib, synth

    tree = hostlib.Tree(open(os.path.join(GOLDEN, fixture + ".tree")).read())
    rp, col, val = hostlib.Table(open(os.path.join(GOLDEN, fixture + ".sparse")).read(), True).resolve(tree)
    got, info = _tiles(tree.parent, tree.length, rp, col, val, gpu_ctx, path=engine.PATH_AUTO)
    assert info.path_taken == engine.PATH_EXACT
    assert "".join(hostlib.format_go(v) + "\n" for v in got) == open(os.path.join(GOLDEN, fixture + ".wl.want")).read()
    big = synth.random_tree(2000, 51)                 # 3999 nodes x 134940 pairs > 2^28
    csr = synth.random_table(big, 520, 0.01, 52)
    got, info = _tiles(big.parent, big.length, *csr, gpu_ctx, path=engine.PATH_AUTO)
    assert info.path_taken == engine.PATH_FAST
    rows = slice(0, 200 * 199 // 2)                   # the first 200 rows against the oracle
    from oracle import oracle as orc
    want, _, _ = orc.unifrac_rows(orc.Table.from_csr(*csr), orc.Tree.from_flat(big.parent, big.length), True, 0,
                                  os.cpu_count() or 1, 0, 200)
    assert rel_err(got[rows], want).max() < 1e-5


@pytest.mark.gpu
def test_tiles_f32_stream_and_band_layout(gpu_ctx):
    """(h) frc_next_f32 carries the same numbers as frc_next, and the band decomposition changes no byte."""
    from frackyfrac_b200 import engine, synth

    tree = synth.random_tree(1500, 301)
    rp, col, val = synth.random_table(tree, 1100, 0.03, 302)
    m = rp[1]
    col[m:2 * m] = col[:m]; val[m:2 * m] = val[:m]
    col[2 * m:3 * m] = col[:m]; val[2 * m:3 * m] = val[:m] * (1.0 + 1e-3 * (np.arange(m) % 5 == 0))

    def run(f32, band_rows=0):
        with engine.Job(tree.parent, tree.length, rp, col, val, weighted=True, normalize=0, path=engine.PATH_FAST,
                        ctx=gpu_ctx, band_rows=band_rows, flags=engine.FLAG_L_TILES) as job:
            if not f32:
                return np.concatenate([a for _, a in job.chunks()])
            out = []
            for first, a in job.chunks_f32():
                d = a.astype(np.float64)
                xi, xv = job.exceptions()
                d[xi - first] = xv
                out.append(d)
            return np.concatenate(out)

    narrow, wide, ragged, other = run(True), run(False), run(True, 128), run(True, 384)
    assert np.array_equal(narrow, wide, equal_nan=True)
    assert np.array_equal(narrow, ragged, equal_nan=True) and np.array_equal(narrow, other, equal_nan=True)
    assert narrow[0] == 0.0
    assert rel_err(narrow, oracle_flat(tree, (rp, col, val), True, 0)).max() < 1e-5


@pytest.mark.gpu
def test_tiles_over_several_gpus(built, monkeypatch):
    """(i) One process over 2 / 4 / 8 GPUs (key panels exchanged over peer memory, or rebuilt everywhere) gives the
    one-GPU stream byte for byte; the capacity mode, which would shard the panels, is refused."""
    import torch

    from frackyfrac_b200 import engine, synth

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    tree = synth.random_tree(1500, 311)
    rp, col, val = synth.random_table(tree, 1100, 0.03, 312, integer_counts=False)
    m = rp[1]
    col[5 * m:6 * m] = col[:m]; val[5 * m:6 * m] = val[:m] * (1 + 1e-4 * (np.arange(m) % 3 == 0))
    one = engine.Context(0)
    ref, _ = _tiles(tree.parent, tree.length, rp, col, val, one)
    one.close()
    for nd in (2, 4, 8):
        if nd > n_gpu:
            break
        for shard in ("1", "0"):
            monkeypatch.setenv("FRC_SHARD", shard)
            got, info = _tiles(tree.parent, tree.length, rp, col, val, None, devices=list(range(nd)))
            assert info.n_devices == nd
            assert np.array_equal(got, ref, equal_nan=True), (nd, shard)
    monkeypatch.setenv("FRC_SHARD", "1")
    monkeypatch.setenv("FRC_CAPACITY", "1")
    with pytest.raises(engine.FrcError) as e:
        _tiles(tree.parent, tree.length, rp, col, val, None, devices=[0, 1])
    assert e.value.code == 5 and "capacity" in str(e.value)


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["synth_a", "synth_b"])
def test_cli_fast_path_with_l(built, tmp_path, fixture):
    """(j) The CLI stand-in with -w -l and FRCFRC_PATH=fast runs the tiles: within 1e-5 of the committed values."""
    from frackyfrac_b200 import hostlib

    out = tmp_path / "got"
    cmd = [hostlib.CLI_PATH, "-w", "-l", "-s", "-t", os.path.join(GOLDEN, fixture + ".tree"),
           "-i", os.path.join(GOLDEN, fixture + ".sparse"), "-o", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, FRCFRC_PATH="fast"))
    assert r.returncode == 0, r.stderr
    want = np.array([float(x) for x in open(os.path.join(GOLDEN, fixture + ".wl.want")).read().split()])
    got = np.array([float(x) for x in out.read_text().split()])
    assert rel_err(got, want).max() < 1e-5
