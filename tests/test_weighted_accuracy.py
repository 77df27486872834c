"""Worst-case accuracy of the weighted FP32 pair tiles (k_weighted_tiles, csrc/weighted.cu) against the reference.

Random trees with random values make the fp32 rounding errors of the tile sums cancel, and their distances sit near
0.8 or below the 1/32 at which pairs are recomputed exactly.  The inputs here are the ones where the kernel's error
model is weakest:
  - regular terms at large B (equal lengths and counts): every rounding of the running sums goes the same way;
  - keyed -l tiles just above the fix-up threshold, where a numerator formed as W_i + W_j - 2 S would cancel.
tests/weighted_model.py restates the kernel's arithmetic in numpy: the CPU tests show on it why each input is here
and that the kernel as built stays within 5e-6 on all of them; the GPU tests check the kernel against the oracle
(and, for the unkeyed constant terms, against the model's bytes, which pins the summation order)."""
import functools

import numpy as np
import pytest

from tests import weighted_model as wm
from tests.helpers import oracle_flat, rel_err

OPERANDS = (0x3fa6f700, 0x3ffe2580, 0x3f800001, 0x3fcccccd)   # fp32 bits of the operand constants
KEYED_STARS = {   # (leaves, branch length, leaves of sample 0; sample 1 holds all leaves): d = 0.03896, not flagged
    "star4k-0.1": (4000, 0.1, 3700), "star4k-0.37": (4000, 0.37, 3700), "star4k-1.3": (4000, 1.3, 3700),
    "star20k-0.1": (20000, 0.1, 18500)}
BUDGET = 5e-6     # what the model of the kernel as built must stay within (the contract is 1e-5)


def f32(bits):
    return np.array([bits], np.uint32).view(np.float32)[0]


def keyed_star(n_leaves, length, n0):
    parent, L = wm.star(n_leaves, length)
    rp, col, val = wm.csr([(np.arange(1, n0 + 1), np.ones(n0)), (np.arange(1, n_leaves + 1), np.ones(n_leaves))])
    return parent, L, (rp, col, val)


@functools.lru_cache(maxsize=None)
def random_tree_case():
    """synth.random_tree(50 000, 9): sample 0 = 25 000 random leaves with counts 1..49, sample 1 = sample 0 plus the
    1 250 lowest-id leaves it lacks (they change few keys: d = 0.0351 under -l as coded)."""
    from frackyfrac_b200 import synth

    tree = synth.random_tree(50_000, 9)
    rng = np.random.default_rng(10)
    leaves = rng.permutation(tree.leaf_ids)
    base, extra = np.sort(leaves[:25_000]), np.sort(leaves[25_000:])
    cb, ce = rng.integers(1, 50, 25_000).astype(float), rng.integers(1, 50, 25_000).astype(float)
    return tree, base, cb, extra, ce


def model_error(parent, length, csr, keyed, normalize, scheme):
    """(oracle-free fp64 distance, relative error of the model) of pair (1, 0)."""
    E, K = wm.embed(parent, *csr)
    if normalize == 1:
        E = E / E.sum(axis=1)[:, None]
    A, W = wm.operands(E, length)
    want = wm.exact(E, K, length, [(1, 0)], keyed)[0]
    got = wm.distances(A, W, [(1, 0)], K if keyed else None, scheme=scheme)[0]
    return want, abs(float(got) - want) / want


# ------------------------------------------------------------------ CPU: the model
def test_model_reproduces_the_keyed_failures_before_the_fix():
    """The keyed star inputs at d = 0.03896 (above the 1/32 threshold, so not recomputed): with the fp32 total and the
    cancelling numerator W_i + W_j - 2 S the modelled error is 1.8e-5 .. 6.8e-5; the random tree's 1.1e-5."""
    want = {"star4k-0.1": 6.1e-5, "star4k-0.37": 4.4e-5, "star4k-1.3": 1.8e-5, "star20k-0.1": 6.8e-5}
    for name, (n, length, n0) in KEYED_STARS.items():
        d, err = model_error(*keyed_star(n, length, n0), True, 0, "f32tot")
        assert abs(d - 30 / 770) < 1e-12
        assert err == pytest.approx(want[name], rel=0.03), (name, err)
    tree, base, cb, extra, ce = random_tree_case()
    csr = wm.csr([(base, cb), (np.concatenate([base, extra[:1250]]), np.concatenate([cb, ce[:1250]]))])
    d, err = model_error(tree.parent, tree.length, csr, True, 0, "f32tot")
    assert 1 / 32 < d < 0.04 and err > 1e-5, (d, err)


def test_model_reproduces_the_unkeyed_failure_before_the_fix():
    """Star with 2^18 leaves on disjoint halves, every operand the fp32 0x3fa6f700: d = 1 exactly, and the fp32
    total of 1024 equal flushes is off by 1.45e-5; 0x3ffe2580 by 7.8e-6."""
    n = 1 << 18
    for bits, want in ((0x3fa6f700, 1.44e-5), (0x3ffe2580, 7.8e-6)):
        c = np.array([f32(bits)])
        err = abs(wm.constant_sum(c, n, lead=1, scheme="f32tot")[0] / (np.float64(c[0]) * n) - 1)
        assert err == pytest.approx(want, rel=0.03), (hex(bits), err)


def test_model_constant_sum_is_the_general_model():
    """The vectorised constant-term sum gives the general model's bytes on a small star (root first, then leaves)."""
    for scheme in ("f32tot", "f64tot"):
        for n in (1, 255, 256, 257, 3000):
            c = f32(0x3fa6f700)
            t = np.zeros((n + 1, 1), np.float32)
            t[1:] = c
            tot, acc = wm.accumulate(t, scheme=scheme)
            general = (tot + acc.astype(np.float64)) if scheme == "f64tot" else (tot + acc).astype(np.float64)
            assert general[0] ==wm.constant_sum(np.array([c]), n, lead=1, scheme=scheme)[0]


def test_model_of_the_kernel_stays_within_budget_on_the_designed_inputs():
    """The kernel as built (fp64 total, direct keyed numerator) models within 5e-6 on every input above."""
    assert wm.SCHEME == "f64tot"
    for name, (n, length, n0) in KEYED_STARS.items():
        _, err = model_error(*keyed_star(n, length, n0), True, 0, wm.SCHEME)
        assert err <= BUDGET, (name, err)
    tree, base, cb, extra, ce = random_tree_case()
    csr = wm.csr([(base, cb), (np.concatenate([base, extra[:1250]]), np.concatenate([cb, ce[:1250]]))])
    _, err = model_error(tree.parent, tree.length, csr, True, 0, wm.SCHEME)
    assert err <= BUDGET, err
    for bits in OPERANDS:
        c = np.array([f32(bits)])
        for n in (1 << 14, 1 << 17, 1 << 18):
            err = abs(wm.constant_sum(c, n, lead=1)[0] / (np.float64(c[0]) * n) - 1)
            assert err <= BUDGET, (hex(bits), n, err)


def test_model_of_the_kernel_stays_within_budget_on_a_sweep_of_constants():
    """2 * 10^5 random fp32 mantissas as constant terms at B = 2^18 + 1 (root, then 2^18 leaves): the kernel as built
    stays within 5e-6 on all of them (only the 256-term fp32 level rounds); the fp32 total did not."""
    rng = np.random.default_rng(2024)
    c = (rng.integers(0, 1 << 23, 200_000).astype(np.uint32) | np.uint32(0x3f800000)).view(np.float32)
    n = 1 << 18
    exact = c.astype(np.float64) * n
    new = np.abs(wm.constant_sum(c, n, lead=1) / exact - 1)
    old = np.abs(wm.constant_sum(c, n, lead=1, scheme="f32tot") / exact - 1)
    assert new.max() <= BUDGET, new.max()
    assert old.max() > 1e-5


# ------------------------------------------------------------------ GPU
def _job(parent, length, csr, normalize, ctx, **kw):
    from frackyfrac_b200 import engine

    flags = engine.FLAG_L_TILES if normalize == 0 else 0
    with engine.Job(parent, length, *csr, weighted=True, normalize=normalize, path=engine.PATH_FAST, ctx=ctx,
                    flags=flags, **kw) as job:
        got = np.concatenate([a for _, a in job.chunks()])
        info = job.info()
    assert info.path_taken == engine.PATH_FAST and info.value_bytes == 4
    return got, info


def _constant_star(n, bits, normalize, neg_leaf=False):
    """Star with n leaves (n a power of two) and two samples on the even and odd leaves, unit counts, lengths set so
    that every leaf's pre-scaled operand is the fp32 with these bits.  neg_leaf: one more leaf, unobserved, with a
    negative length (the FFMA form of the kernel)."""
    scale = 1.0 / n if normalize == 1 else 1.0        # normalize 1: a leaf's proportion is 1 / (n/2 + n/2 at the root)
    parent, L = wm.star(n + int(neg_leaf), wm.length_for_operand(bits, scale))
    if neg_leaf:
        L[-1] = -0.5
    csr = wm.csr([(np.arange(2, n + 1, 2), np.ones(n // 2)), (np.arange(1, n + 1, 2), np.ones(n // 2))])
    return parent, L, csr


def _constant_model(n, bits, normalize):
    """The model's fp32 distance of the constant star: root first (operand 0), then n leaves with operand c; every fp64
    stage is exact (n a power of two), so the model's bytes are the kernel's."""
    c = f32(bits)
    num = wm.constant_sum(np.array([c]), n, lead=1)
    w = np.float64(c) * (n // 2)
    return wm.epilogue(num, np.zeros(1, np.float32), w, w)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("normalize", [1, 2])
@pytest.mark.parametrize("n", [1 << 14, 1 << 17, 1 << 18])
def test_constant_terms_match_the_oracle_and_the_model_bytes(gpu_ctx, n, normalize):
    """Unkeyed, equal terms: within 1e-5 of the oracle (d = 1), and the kernel's bytes are the model's."""
    from frackyfrac_b200 import synth

    for bits in OPERANDS:
        parent, L, csr = _constant_star(n, bits, normalize)
        want = oracle_flat(synth.Tree(parent, L, None, None), csr, True, normalize)
        got, _ = _job(parent, L, csr, normalize, gpu_ctx)
        err = rel_err(got, want).max()
        print(f"constant n={n} normalize={normalize} operand={bits:#x}: d={got[0]!r} max rel err {err:.3e}")
        assert want[0] == 1.0
        assert np.float32(got[0]).view(np.uint32) == _constant_model(n, bits, normalize).view(np.uint32), hex(bits)
        assert err < 1e-5, (hex(bits), err)


def _sweep_case(tree_name, counts):
    """(parent, length, csr): sample 0 and 127 variants that add increasing sets of extra leaves to it, so that the
    distances (k, 0) sweep about [1/32, 0.3] under -l as coded."""
    rng = np.random.default_rng(77)
    if tree_name == "random":
        tree, base, cb, extra, ce = random_tree_case()
        parent, L = tree.parent, tree.length
        m = np.unique(np.geomspace(1170, 11000, 127).astype(int))
        if counts == "unit":
            cb, ce = np.ones_like(cb), np.ones_like(ce)
    else:
        n_leaves, length = {"star-0.1": (4000, 0.1), "star-0.37": (4000, 0.37), "star-1.3": (4000, 1.3),
                            "star20k-0.1": (20000, 0.1)}[tree_name]
        parent, L = wm.star(n_leaves, length)
        n0 = n_leaves // 2
        base, extra = np.arange(1, n0 + 1), np.arange(n0 + 1, n_leaves + 1)
        cb = np.ones(n0) if counts == "unit" else rng.integers(1, 50, n0).astype(float)
        ce = np.ones(n_leaves - n0) if counts == "unit" else rng.integers(1, 50, n_leaves - n0).astype(float)
        # d(k, 0) = extra mass / (2 base mass + extra mass) on a star (root length 0): pick the masses of the targets
        target = np.geomspace(1 / 32 * 1.001, 0.3, 127)
        mass = np.cumsum(ce)
        m = np.unique(np.searchsorted(mass, 2 * cb.sum() * target / (1 - target)) + 1)
    rows = [(base, cb)] + [(np.concatenate([base, extra[:k]]), np.concatenate([cb, ce[:k]])) for k in m]
    return parent, L, wm.csr(rows)


SWEEPS = ["star-0.1", "star-0.37", "star-1.3", "star20k-0.1", "random"]


@pytest.mark.gpu
@pytest.mark.parametrize("counts", ["unit", "1..49"])
@pytest.mark.parametrize("tree_name", SWEEPS)
@pytest.mark.parametrize("normalize", [0, 1, 2])
def test_sweep_above_the_fixup_threshold(gpu_ctx, normalize, tree_name, counts):
    """Every pair within 1e-5 of the oracle, and no pair at d >= 1/32 is flagged for the fix-up (so the tiles, not the
    recompute, carry these pairs).  normalize 0 (keyed -l tiles) is where a cancelling numerator fails; 1 and 2
    (unkeyed) check the operand-rounding bound 6e-8 / d."""
    from frackyfrac_b200 import synth

    parent, L, csr = _sweep_case(tree_name, counts)
    want = oracle_flat(synth.Tree(parent, L, None, None), csr, True, normalize)
    got, info = _job(parent, L, csr, normalize, gpu_ctx)
    n = len(csr[0]) - 1
    k0 = np.array([k * (k - 1) // 2 for k in range(1, n)])          # pairs (k, 0)
    above = want >= 1 / 32
    err = rel_err(got, want)
    print(f"sweep {tree_name} {counts} normalize={normalize}: {n - 1} variants, d(k,0) in "
          f"[{want[k0].min():.4f}, {want[k0].max():.4f}], {above.sum()} pairs >= 1/32, flagged {info.flagged_pairs}, "
          f"max rel err {err.max():.3e} (>= 1/32: {rel_err(got[above], want[above]).max():.3e})")
    if normalize == 0:
        assert want[k0].min() < 0.04 and want[k0].max() > 0.25 and (want[k0] >= 1 / 32).all()
    assert info.flagged_pairs <= (want < 1 / 32).sum()
    assert err.max() < 1e-5


@pytest.mark.gpu
def test_ffma_form_with_a_negative_unobserved_length(gpu_ctx):
    """Negative lengths switch the kernel to the FFMA form (operand a, len applied by fmaf): an unkeyed constant star
    and the keyed star sweep with one more leaf that no sample observes, of length -0.5, within 1e-5."""
    from frackyfrac_b200 import synth

    for normalize in (1, 2):
        parent, L, csr = _constant_star(1 << 18, 0x3fa6f700, normalize, neg_leaf=True)
        want = oracle_flat(synth.Tree(parent, L, None, None), csr, True, normalize)
        got, _ = _job(parent, L, csr, normalize, gpu_ctx)
        err = rel_err(got, want).max()
        print(f"ffma constant normalize={normalize}: max rel err {err:.3e}")
        assert err < 1e-5
    parent, L, csr = _sweep_case("star-0.1", "1..49")
    parent, L = np.append(parent, 0).astype(np.int32), np.append(L, -0.5)
    want = oracle_flat(synth.Tree(parent, L, None, None), csr, True, 0)
    got, info = _job(parent, L, csr, 0, gpu_ctx)
    err = rel_err(got, want).max()
    print(f"ffma keyed sweep: flagged {info.flagged_pairs}, max rel err {err:.3e}")
    assert info.flagged_pairs <= (want < 1 / 32).sum()
    assert err < 1e-5


@pytest.mark.gpu
def test_rect_tiles(gpu_ctx):
    """The rectangular instantiation (engine.unifrac_cross): the unkeyed constant star (reference = sample 0, query =
    sample 1) gives the model's bytes; the keyed star sweep (reference = sample 0, query = the variants) is within
    1e-5 of the oracle's triangle over [reference; query]."""
    from frackyfrac_b200 import engine, synth

    def split(csr, n_ref):
        rp, col, val = csr
        k = rp[n_ref]
        return (rp[:n_ref + 1], col[:k], val[:k]), (rp[n_ref:] - k, col[k:], val[k:])

    parent, L, csr = _constant_star(1 << 18, 0x3fa6f700, 1)
    ref, qry = split(csr, 1)
    got = engine.unifrac_cross(parent, L, ref, qry, True, 1, path=engine.PATH_FAST, ctx=gpu_ctx)
    print(f"rect constant: d={got[0, 0]!r}")
    assert np.float32(got[0, 0]).view(np.uint32) == _constant_model(1 << 18, 0x3fa6f700, 1).view(np.uint32)
    parent, L, csr = _sweep_case("star-0.1", "unit")
    ref, qry = split(csr, 1)
    got = engine.unifrac_cross(parent, L, ref, qry, True, 0, path=engine.PATH_FAST, ctx=gpu_ctx,
                               flags=engine.FLAG_L_TILES)
    tri = oracle_flat(synth.Tree(parent, L, None, None), csr, True, 0)
    n_q = len(qry[0]) - 1
    want = np.array([tri[(1 + q) * q // 2] for q in range(n_q)])    # pairs (1 + q, 0) of the triangle
    err = rel_err(got[:, 0], want).max()
    print(f"rect keyed sweep: max rel err {err:.3e}")
    assert err < 1e-5
