"""Table staging of frc_create (frackyfrac_b200/csrc/plan.cpp) on the CPU box: the caller's CSR entries checked and
copied into the staged table, the PRUNE leaf marks, and which rows a part reads.

The checks are frc_create's only guard on the entries a caller hands in, and their messages name the row, the entry
and the node.  frc_debug_stage runs the same functions frc_create runs (StagedTable, chunk_rows, stage_entries,
first_error, mark_table_leaves), so these tests pin the staged bytes and every message without a device."""
import ctypes as C

import numpy as np
import pytest

from frackyfrac_b200 import synth

TREE = synth.random_tree(300, 17)
B = TREE.n_nodes
LEAVES = np.sort(TREE.leaf_ids)
INNER = next(v for v in range(1, B - 1) if TREE.parent[v + 1] == v)  # a node that is not a leaf (not the root)


@pytest.fixture(scope="module")
def L(built):
    from frackyfrac_b200 import engine

    lib = engine.lib()
    P = C.c_void_p
    lib.frc_debug_stage.argtypes = [P, C.c_int32, C.c_int64, P, P, P, C.c_int64, P, P, P, P, C.c_int32, P, C.c_int64,
                                    P, P, P, P, C.c_char_p, C.c_int64]
    lib.frc_debug_stage.restype = C.c_int64
    lib.frc_debug_rows_read.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int32, P]
    lib.frc_debug_rows_read.restype = None
    lib.frc_debug_shards.argtypes = [C.c_int64, C.c_int32, C.c_int32, P, P, C.c_int64, P, C.c_int64]
    lib.frc_debug_shards.restype = C.c_int64
    lib.frc_debug_prune.argtypes = [P, P, C.c_int32, P, C.c_int32] + [P] * 4
    lib.frc_debug_prune.restype = C.c_int32
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data


def _table(n, seed, leaves=LEAVES[60:260], most=12):
    """n rows of 0..most distinct leaves (empty rows included) with positive finite values."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, most + 1, n)
    rp = np.zeros(n + 1, np.int64)
    rp[1:] = np.cumsum(counts)
    col = np.concatenate([rng.choice(leaves, c, replace=False) for c in counts] + [np.zeros(0)]).astype(np.int32)
    val = rng.lognormal(0.0, 2.0, len(col))
    return rp, col, val


def _q0(n_ref):
    return -(-n_ref // 256) * 256


def stage(L, ref, query=None, new_of_old=None, values=True, chunks=1, stamp=None, tag=0, marks=False):
    """What frc_create stages: (row_ptr, col, val or None, reported message, marks or None)."""
    n_ref = len(ref[0]) - 1
    n_q = len(query[0]) - 1 if query is not None else -1
    N = _q0(n_ref) + n_q if query is not None else n_ref
    nnz = len(ref[1]) + (len(query[1]) if query is not None else 0)
    q = query if query is not None else (None, None, None)
    rp = np.full(N + 1, -7, np.int64)
    col = np.full(nnz, -7, np.int32)
    val = np.full(nnz, -7.0) if values else None
    if values and stamp is None:
        stamp = np.full(B, -1, np.int64)
    mk = np.zeros(B, np.uint8) if marks else None
    no = None if new_of_old is None else np.ascontiguousarray(new_of_old, np.int32)
    msg = C.create_string_buffer(512)
    got = L.frc_debug_stage(TREE.parent.ctypes.data, B, n_ref, *map(_ptr, ref), n_q, *map(_ptr, q), _ptr(no), chunks,
                            _ptr(stamp), tag, rp.ctypes.data, col.ctypes.data, _ptr(val), _ptr(mk), msg, len(msg))
    assert got == N
    return rp, col, val, msg.value.decode(), mk


def model(ref, query=None, new_of_old=None):
    """The staged table in numpy: reference rows, empty rows up to q0 = n_ref rounded up to 256, query rows."""
    rp, col, val = ref
    if query is not None:
        n_ref, nnz_a = len(rp) - 1, rp[-1]
        rp = np.concatenate([rp, np.full(_q0(n_ref) - n_ref, nnz_a), nnz_a + query[0][1:]])
        col, val = np.concatenate([col, query[1]]), np.concatenate([val, query[2]])
    if new_of_old is not None:
        col = np.asarray(new_of_old)[col]
    return rp, col.astype(np.int32), val


def _new_of_old(L, leaves, merge):
    marks = np.zeros(B, np.uint8)
    marks[leaves] = 1
    op, ol, om, no = np.zeros(B, np.int32), np.zeros(B), np.zeros(B, np.int32), np.zeros(B, np.int32)
    n = L.frc_debug_prune(TREE.parent.ctypes.data, TREE.length.ctypes.data, B, marks.ctypes.data, int(merge),
                          op.ctypes.data, ol.ctypes.data, om.ctypes.data, no.ctypes.data)
    assert 1 <= n < B
    return no


def _check_bytes(L, ref, query, prune, values, chunks):
    leaves = np.unique(np.concatenate([ref[1]] + ([query[1]] if query is not None else [])))
    no = None if prune is None else _new_of_old(L, leaves, prune == "merge")
    rp, col, val, msg, _ = stage(L, ref, query, new_of_old=no, values=values, chunks=chunks)
    want_rp, want_col, want_val = model(ref, query, no)
    assert msg == ""
    assert rp.tobytes() == want_rp.tobytes()
    assert col.tobytes() == want_col.tobytes()
    if values:
        assert val.tobytes() == want_val.tobytes()
    if no is not None:
        assert (col >= 0).all() and not np.array_equal(col, model(ref, query)[1])


@pytest.mark.parametrize("chunks", [1, 7])
@pytest.mark.parametrize("values", [True, False])
@pytest.mark.parametrize("prune", [None, "prune", "merge"])
def test_triangle_table_bytes(L, prune, values, chunks):
    _check_bytes(L, _table(300, 1), None, prune, values, chunks)


@pytest.mark.parametrize("chunks", [1, 7])
@pytest.mark.parametrize("values", [True, False])
@pytest.mark.parametrize("prune", [None, "prune", "merge"])
@pytest.mark.parametrize("n_ref", [1, 255, 256, 257, 700])
def test_cross_table_bytes(L, n_ref, prune, values, chunks):
    ref = _table(n_ref, 2 + n_ref, leaves=LEAVES[40:160])
    query = _table(130, 3 + n_ref, leaves=LEAVES[120:270])
    _check_bytes(L, ref, query, prune, values, chunks)
    rp = stage(L, ref, query, values=values, chunks=chunks)[0]
    assert len(rp) == _q0(n_ref) + 130 + 1 and (rp[n_ref:_q0(n_ref) + 1] == len(ref[1])).all()


def _broken(table, row, entry, col=None, val=None):
    rp, c, v = table[0], table[1].copy(), table[2].copy()
    k = rp[row] + entry - 1
    assert rp[row] <= k < rp[row + 1]
    if col is not None:
        c[k] = col
    if val is not None:
        v[k] = val
    return rp, c, v


def _row_with(table, at_least, start=0):
    """First row from `start` on with at least that many entries."""
    return next(s for s in range(start, len(table[0]) - 1) if table[0][s + 1] - table[0][s] >= at_least)


@pytest.mark.parametrize("values", [True, False])
def test_entry_messages(L, values):
    t = _table(40, 5)
    s = _row_with(t, 3)
    name = f"sample #{s + 1}: entry 3"
    cases = [(dict(col=-1), f"{name} (node -1): node id out of range"),
             (dict(col=B), f"{name} (node {B}): node id out of range"),
             (dict(col=INNER), f"{name} (node {INNER}): node is not a leaf"),
             (dict(col=0), f"{name} (node 0): node is not a leaf")]
    leaf = int(t[1][t[0][s] + 2])
    for bad in (0.0, -1.5, np.inf, np.nan):
        cases.append((dict(val=bad), f"{name} (node {leaf}): bad value"))
    for change, want in cases:
        assert stage(L, _broken(t, s, 3, **change), values=values)[3] == want, change
    # a leaf listed twice in a row: an error only when values are used (presence is an OR)
    first = int(t[1][t[0][s]])
    dup = _broken(t, s, 3, col=first)
    rp, col, _, msg, _ = stage(L, dup, values=values)
    if values:
        assert msg == f"{name} (node {first}): leaf listed twice"
    else:
        assert msg == "" and col.tobytes() == dup[1].tobytes()


def test_check_order(L):
    """An entry with two faults reports the earlier check: range, leaf, value, duplicate."""
    t = _table(40, 6)
    s = _row_with(t, 3)
    first = int(t[1][t[0][s]])
    name = f"sample #{s + 1}: entry 3"
    cases = [(dict(col=-1, val=0.0), f"{name} (node -1): node id out of range"),
             (dict(col=B, val=np.nan), f"{name} (node {B}): node id out of range"),
             (dict(col=INNER, val=-1.0), f"{name} (node {INNER}): node is not a leaf"),
             (dict(col=first, val=np.inf), f"{name} (node {first}): bad value")]
    for change, want in cases:
        assert stage(L, _broken(t, s, 3, **change))[3] == want, change


def test_cross_messages_name_the_table(L):
    ref, query = _table(300, 7), _table(90, 8)
    r, q = _row_with(ref, 2), _row_with(query, 2, start=40)
    got = stage(L, _broken(ref, r, 2, col=-1), query)[3]
    assert got == f"reference sample #{r + 1}: entry 2 (node -1): node id out of range"
    got = stage(L, ref, _broken(query, q, 2, col=B))[3]
    assert got == f"query sample #{q + 1}: entry 2 (node {B}): node id out of range"
    got = stage(L, ref, _broken(query, q, 2, val=0.0))[3]
    assert got == f"query sample #{q + 1}: entry 2 (node {int(query[1][query[0][q] + 1])}): bad value"


@pytest.mark.parametrize("chunks", [1, 2, 3, 8, 64])
def test_first_bad_entry_in_row_order_whatever_the_chunking(L, chunks):
    t = _table(600, 9)
    rows = [s for s in range(600) if t[0][s + 1] - t[0][s] >= 6]
    a, b, c = rows[40], rows[len(rows) // 2], rows[-3]
    bad = _broken(t, a, 5, val=-2.0)
    bad = _broken(bad, a, 6, col=-1)       # a later entry of the same row
    bad = _broken(bad, b, 1, col=INNER)
    bad = _broken(bad, c, 2, col=B)
    want = f"sample #{a + 1}: entry 5 (node {int(t[1][t[0][a] + 4])}): bad value"
    assert stage(L, bad, chunks=chunks)[3] == want
    # without the first fault the next row's is reported
    bad = _broken(_broken(bad, a, 5, val=1.0), a, 6, col=int(t[1][t[0][a] + 5]))
    assert stage(L, bad, chunks=chunks)[3] == f"sample #{b + 1}: entry 1 (node {INNER}): node is not a leaf"
    # cross: a query fault never hides a reference fault
    q = _table(200, 10)
    qbad = _broken(q, _row_with(q, 1), 1, col=-1)
    r = _row_with(t, 1)
    got = stage(L, _broken(t, r, 1, col=B), qbad, chunks=chunks)[3]
    assert got == f"reference sample #{r + 1}: entry 1 (node {B}): node id out of range"


def test_stamps_carry_across_jobs(L):
    """The duplicate stamps persist between jobs; each job's tag lies past the previous job's marks."""
    t = _table(300, 11, most=30)
    N = len(t[0]) - 1
    stamp = np.full(B, -1, np.int64)
    epoch = 0
    for _ in range(3):
        assert stage(L, t, stamp=stamp, tag=epoch)[3] == ""
        # a listed leaf holds the tag + the last row that listed it
        last = np.full(B, -1, np.int64)
        for s in range(N):
            last[t[1][t[0][s]:t[0][s + 1]]] = epoch + s
        assert stamp.tobytes() == np.where(last >= 0, last, stamp).tobytes() and (stamp[last < 0] < epoch).all()
        epoch += N + 1   # frc_create: stamp_epoch += N + 1
    # a duplicate inside one row is still found under a fresh tag
    s = _row_with(t, 4)
    dup = _broken(t, s, 4, col=int(t[1][t[0][s] + 1]))
    got = stage(L, dup, stamp=stamp, tag=epoch)[3]
    assert got == f"sample #{s + 1}: entry 4 (node {int(t[1][t[0][s] + 1])}): leaf listed twice"


def test_prune_marks_are_the_union_of_both_tables_leaves(L):
    ref = _table(300, 12, leaves=LEAVES[:120])
    query = _table(150, 13, leaves=LEAVES[90:260])
    for q in (None, query):
        mk = stage(L, ref, q, marks=True)[4]
        want = np.zeros(B, np.uint8)
        want[ref[1]] = 1
        if q is not None:
            want[q[1]] = 1
        assert mk.tobytes() == want.tobytes()
    # ids out of range mark nothing (staging reports them)
    bad = _broken(_broken(query, _row_with(query, 2), 1, col=-1), _row_with(query, 2), 2, col=B)
    mk = stage(L, ref, bad, marks=True)[4]
    want = np.zeros(B, np.uint8)
    want[ref[1]] = 1
    want[bad[1][(bad[1] >= 0) & (bad[1] < B)]] = 1
    assert mk.tobytes() == want.tobytes()


def _shard_range(L, n, owners, owner):
    info, shards, ranges = np.zeros(3, np.int64), np.zeros((64, 2), np.int32), np.zeros((64, 4), np.int64)
    k = L.frc_debug_shards(n, owners, 1, info.ctypes.data, shards.ctypes.data, len(shards), ranges.ctypes.data,
                           len(ranges))
    assert k == owners
    (_, s0, s1, _), = [r for r in ranges[:k] if r[0] == owner]
    return min(n, s0), min(n, s1)


@pytest.mark.parametrize("n", [0, 1, 127, 128, 1000, 5000])
def test_rows_read(L, n):
    out = np.zeros(2, np.int64)
    for owners in range(1, 9):
        covered = []
        for owner in range(owners):
            L.frc_debug_rows_read(n, owners, owner, 1, out.ctypes.data)
            assert tuple(out) == _shard_range(L, n, owners, owner)
            covered.append(tuple(out))
            L.frc_debug_rows_read(n, owners, owner, 0, out.ctypes.data)
            assert tuple(out) == (0, n)
        # the owners' rows tile [0, n)
        assert covered[0][0] == 0 and covered[-1][1] == n
        assert all(covered[k][1] == covered[k + 1][0] for k in range(owners - 1))
