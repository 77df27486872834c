"""The host-only planning units of frc_create (frackyfrac_b200/csrc/plan.cpp) on the CPU box: band plan,
tile lists, operand column plan, tree walk.  They decide what every GPU computes, so they are tested without one."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def L(built):
    from frackyfrac_b200 import engine

    lib = engine.lib()
    lib.frc_debug_bands.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64]
    lib.frc_debug_bands.restype = C.c_int64
    lib.frc_debug_band_tiles.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64]
    lib.frc_debug_band_tiles.restype = C.c_int64
    lib.frc_debug_plan_columns.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.frc_debug_plan_columns.restype = C.c_int32
    lib.frc_debug_tree.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p] * 6
    lib.frc_debug_tree.restype = C.c_int32
    return lib


def _bands(L, n, band_rows=0, world=1, d2h=1, per_rank=0):
    out = np.zeros((4096, 5), np.int64)
    k = L.frc_debug_bands(n, band_rows, world, d2h, per_rank, 8, out.ctypes.data, len(out))
    assert 0 <= k <= len(out)
    return out[:k]


def _tiles(L, row0, row1, pair):
    out = np.zeros((1 << 16, 2), np.int32)
    k = L.frc_debug_band_tiles(row0, row1, pair, out.ctypes.data, len(out))
    assert k <= len(out)
    return out[:k]


def test_bands_partition_the_triangle_and_balance_the_owners(L):
    for n in (2, 129, 1000, 5000, 14142, 100_000):
        total = n * (n - 1) // 2
        for world in (1, 2, 4, 8):
            for d2h in (0, 1):
                b = _bands(L, n, world=world, d2h=d2h)
                assert b[0, 0] == 0 and b[-1, 1] == n and (b[1:, 0] == b[:-1, 1]).all()
                assert (b[:, 0] % 128 == 0).all()
                assert b[0, 2] == 0 and (b[1:, 2] == np.cumsum(b[:-1, 3])).all() and b[:, 3].sum() == total
                assert set(b[:, 4].tolist()) <= set(range(world))
                if n >= 14142:
                    load = np.bincount(b[:, 4], weights=b[:, 3], minlength=world)
                    assert load.max() / load.mean() < 1.10, (n, world, load)
    # the band plan the public helper reports is the same one
    from frackyfrac_b200 import engine

    b = _bands(L, 14142, world=8)
    for r in range(8):
        f, c = engine.plan_bands(14142, r, 8)
        mine = b[b[:, 4] == r]
        assert f.tolist() == mine[:, 2].tolist() and c.tolist() == mine[:, 3].tolist()
    assert len(_bands(L, 5000, per_rank=3)) == 3 + 1   # (one device, streamed: the first band is cut again)


@pytest.mark.parametrize("pair", [0, 1])
def test_band_tiles_cover_every_pair_once(L, pair):
    for row0, row1 in ((0, 5000), (0, 100), (1280, 2560), (4864, 5000), (128, 256), (0, 128)):
        t = _tiles(L, row0, row1, pair)
        t0, t1 = row0 // 128, (row1 - 1) // 128
        seen = set()
        for ti, tj in t.tolist():
            assert t0 <= ti <= t1
            cols = (tj, tj + 1) if pair else (tj,)
            assert tj % 2 == 0 or not pair
            assert tj <= ti
            for c in cols:
                assert (ti, c) not in seen
                seen.add((ti, c))
        need = {(ti, tj) for ti in range(t0, t1 + 1) for tj in range(ti + 1)}
        assert need <= seen
        # a pair tile may add the masked tile right of the diagonal, nothing else
        assert all(tj == ti + 1 and ti % 2 == 0 for ti, tj in seen - need)


def _plan(L, length, want_i8=1, gb=3, force_f64=0):
    n = len(length)
    cap = ((n + 127) // 128 + 24) * 128
    order, cexp, lcol = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap)
    cend, cscale, cshift, info = np.zeros(64, np.int32), np.zeros(64), np.zeros(64, np.int32), np.zeros(5, np.int32)
    length = np.ascontiguousarray(length, np.float64)
    kp = L.frc_debug_plan_columns(length.ctypes.data, n, want_i8, gb, force_f64, order.ctypes.data, cexp.ctypes.data,
                                  lcol.ctypes.data, cap, cend.ctypes.data, cscale.ctypes.data, cshift.ctypes.data,
                                  info.ctypes.data)
    assert kp > 0
    nc = int(info[4])
    return dict(kp=kp, order=order[:kp], cexp=cexp[:kp], lcol=lcol[:kp], cend=cend[:nc], cscale=cscale[:nc],
                cshift=cshift[:nc], i8=bool(info[0]), intacc=bool(info[1]), biased=bool(info[2]), e_min=int(info[3]))


def test_u8_column_plan_places_every_positive_length_once(L):
    rng = np.random.default_rng(3)
    for kind in ("exp", "heavy", "zeros", "const", "one_huge"):
        n = 5000
        length = rng.exponential(0.05, n)
        if kind == "heavy":
            length = np.exp(rng.normal(-3, 4, n))
        elif kind == "zeros":
            length[rng.random(n) < 0.3] = 0.0
        elif kind == "const":
            length[:] = 0.37
        elif kind == "one_huge":
            length[17] = 1e6
        p = _plan(L, length)
        assert p["i8"] and p["kp"] % 128 == 0
        cols = p["order"][p["order"] >= 0]
        assert sorted(cols.tolist()) == np.flatnonzero(length > 0).tolist()          # each once, zero lengths none
        assert np.array_equal(p["lcol"][p["order"] >= 0], length[cols]) and (p["lcol"][p["order"] < 0] == 0).all()
        # the chunk exponent leaves x = len / 2^e below 2^23 (so a * m with a <= 255, m <= 65535 reaches it) and every
        # aligned block of 128 columns has one exponent
        x = p["lcol"] / np.exp2(p["cexp"].astype(float))
        assert (x < 2.0 ** 23).all()
        assert (p["cexp"].reshape(-1, 128) == p["cexp"].reshape(-1, 128)[:, :1]).all()
        # chunks: ends ascending, last = kp / 128, runs of at most 128 blocks (plane sums < 2^31), scale = 2^exp
        assert (np.diff(p["cend"]) > 0).all() and p["cend"][-1] == p["kp"] // 128
        assert (np.diff(np.concatenate([[0], p["cend"]])) <= 128).all()
        for c, (b0, b1) in enumerate(zip(np.concatenate([[0], p["cend"][:-1]]), p["cend"])):
            assert (p["cexp"][b0 * 128:b1 * 128] == np.log2(p["cscale"][c])).all()
        span = np.log2(p["cscale"]).max() - np.log2(p["cscale"]).min()
        assert p["intacc"] == (span <= 16) and p["e_min"] == int(np.log2(p["cscale"]).min())
        assert (p["cshift"] == np.log2(p["cscale"]) - p["e_min"]).all()
    assert not _plan(L, rng.exponential(0.05, 3000), force_f64=1)["intacc"]
    # bf16 plan: identity order, uniform chunks of 64 K blocks
    p = _plan(L, rng.exponential(0.05, 3000), want_i8=0)
    assert not p["i8"] and p["kp"] == 3008 and p["order"][:3000].tolist() == list(range(3000)) and (p["order"][3000:] == -1).all()


def _py_tree(parent):
    n = len(parent)
    children = [[] for _ in range(n)]
    for v in range(1, n):
        children[parent[v]].append(v)
    height = [0] * n
    for v in range(n - 1, 0, -1):
        height[parent[v]] = max(height[parent[v]], height[v] + 1)
    post = []
    stack = [(0, 0)]
    while stack:
        v, k = stack.pop()
        if k < len(children[v]):
            stack.append((v, k + 1))
            stack.append((children[v][k], 0))
        else:
            post.append(v)
    return children, height, post


def test_tree_walk_levels_children_post_order(L):
    from frackyfrac_b200 import synth

    for shape, n in (("random", 700), ("caterpillar", 300), ("balanced", 256)):
        tree = synth.random_tree(n, 5, shape=shape)
        parent = np.ascontiguousarray(tree.parent, np.int32)
        B = len(parent)
        lvl, lpar, lptr = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B + 2, np.int32)
        cptr, cidx, post = np.zeros(B + 1, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
        H = L.frc_debug_tree(parent.ctypes.data, B, lvl.ctypes.data, lpar.ctypes.data, lptr.ctypes.data, cptr.ctypes.data,
                             cidx.ctypes.data, post.ctypes.data)
        children, height, want_post = _py_tree(parent.tolist())
        assert H == height[0]
        assert post.tolist() == want_post                        # abundanceToFlatNodes' visiting order (unifrac.go:32-53)
        for v in range(B):
            assert cidx[cptr[v]:cptr[v + 1]].tolist() == children[v]   # file order
        assert lptr[0] == 0 and lptr[H + 1] == B
        for h in range(H + 1):
            nodes = lvl[lptr[h]:lptr[h + 1]].tolist()
            assert nodes == [v for v in range(B) if height[v] == h]    # leaves first, ascending id inside a level
        assert all(lpar[k] == (parent[lvl[k]] if lvl[k] else 0) for k in range(B))
    # not a pre-order numbering / a parent that is not a smaller id
    bad = np.array([-1, 0, 0, 1], np.int32)
    z = [np.zeros(8, np.int32) for _ in range(6)]
    assert L.frc_debug_tree(bad.ctypes.data, 4, *[a.ctypes.data for a in z]) == -1 - 3
    bad = np.array([-1, 0, 5, 1, 1, 1], np.int32)
    assert L.frc_debug_tree(bad.ctypes.data, 6, *[a.ctypes.data for a in z]) == -1 - 2


def test_capacity_bands_respect_the_shards(L):
    """Capacity mode of the weighted path: 2G row shards, shard s on device s or 2G-1-s; no band straddles a shard,
    the triangle is covered once and the devices' pair counts are balanced."""
    L.frc_debug_bands_capacity.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_int64]
    L.frc_debug_bands_capacity.restype = C.c_int64
    for n, G in ((1100, 2), (5000, 4), (20000, 8), (200_000, 8), (300, 2)):
        np_ = -(-n // (256 * G)) * 256 * G
        R = np_ // (2 * G)
        for d2h in (0, 1):
            for band_rows in (0, 128):
                out = np.zeros((1 << 14, 5), np.int64)
                k = L.frc_debug_bands_capacity(n, np_, G, band_rows, d2h, out.ctypes.data, len(out))
                b = out[:k]
                assert b[0, 0] == 0 and b[-1, 1] == n and (b[1:, 0] == b[:-1, 1]).all()
                assert (b[1:, 2] == np.cumsum(b[:-1, 3])).all() and b[:, 3].sum() == n * (n - 1) // 2
                shard = b[:, 0] // R
                assert (shard == (b[:, 1] - 1) // R).all()
                assert (b[:, 4] == np.where(shard < G, shard, 2 * G - 1 - shard)).all()
                if n >= 5000:
                    load = np.bincount(b[:, 4], weights=b[:, 3], minlength=G)
                    assert load.max() / load.mean() < 1.06, (n, G, load)


def test_capacity_groups_cover_every_tile_once_in_visiting_order(L):
    """Capacity mode, per device: the rows of each of its two shards form a group whose tiles are listed by the column
    shard they read (the order the shards visit in).  Over all devices every tile of the triangle appears exactly
    once, every tile sits in the segment of its own column shard, and rows only ever belong to the device's shards."""
    L.frc_debug_capacity_groups.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p,
                                            C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.frc_debug_capacity_groups.restype = C.c_int64
    for n, G in ((1300, 2), (5000, 4), (9000, 8), (300, 2)):
        np_ = -(-n // (256 * G)) * 256 * G
        R, T, S = np_ // (2 * G), np_ // (2 * G) // 128, 2 * G
        seen = {}
        pairs = 0
        for dev in range(G):
            groups = np.zeros((4, 4), np.int64)
            coff = np.zeros((4, S + 1), np.int32)
            tiles = np.zeros((1 << 20, 2), np.int32)
            nt = C.c_int64()
            k = L.frc_debug_capacity_groups(n, np_, G, dev, 0, 1, groups.ctypes.data, coff.ctypes.data, 4, tiles.ctypes.data,
                                            len(tiles), C.byref(nt))
            assert 1 <= k <= 2
            for g in range(k):
                shard, first, count, off = groups[g].tolist()
                assert shard in (dev, S - 1 - dev)
                r0, r1 = shard * R, min(n, (shard + 1) * R)
                assert first == (r0 * (r0 - 1) // 2 if r0 >= 2 else 0) and count == r1 * (r1 - 1) // 2 - first
                pairs += count
                assert coff[g][0] == 0 and (np.diff(coff[g]) >= 0).all() and (coff[g][shard + 1:] == coff[g][shard + 1]).all()
                for c in range(S):
                    seg = tiles[off + coff[g][c]: off + coff[g][c + 1]]
                    for ti, tj in seg.tolist():
                        assert tj // T == c and ti // T == shard and tj <= ti and ti * 128 < n
                        assert (ti, tj) not in seen
                        seen[(ti, tj)] = dev
        nt_rows = (n + 127) // 128
        assert pairs == n * (n - 1) // 2
        assert set(seen) == {(ti, tj) for ti in range(nt_rows) for tj in range(ti + 1)}


def _bands_capacity(L, n, np_, G, band_rows=0, d2h=1):
    L.frc_debug_bands_capacity.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_int64]
    L.frc_debug_bands_capacity.restype = C.c_int64
    out = np.zeros((1 << 14, 5), np.int64)
    k = L.frc_debug_bands_capacity(n, np_, G, band_rows, d2h, out.ctypes.data, len(out))
    assert 0 <= k <= len(out)
    return out[:k]


def _shards(L, n, owners, mode):
    L.frc_debug_shards.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
    L.frc_debug_shards.restype = C.c_int64
    info, shards, ranges = np.zeros(3, np.int64), np.zeros((64, 2), np.int32), np.zeros((64, 4), np.int64)
    k = L.frc_debug_shards(n, owners, mode, info.ctypes.data, shards.ctypes.data, len(shards), ranges.ctypes.data,
                           len(ranges))
    assert k > 0
    np_, n_shards, shard_rows = info.tolist()
    return np_, n_shards, shard_rows, shards[:n_shards], ranges[:k]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_sample_shards_partition_the_padded_samples(L, mode):
    """The sample shards of the embedding (0: every owner builds everything, 1: one shard per owner, 2: capacity
    mode, two per device): padded to whole tiles of every shard, every sample built once (mode 0: by every owner)."""
    for n in (1, 127, 128, 1000, 14142, 100_000):
        for owners in range(1, 9):
            np_, n_shards, R, shards, ranges = _shards(L, n, owners, mode)
            assert n_shards == (1, owners, 2 * owners)[mode]
            assert np_ >= n and np_ % (128 * n_shards) == 0 and R * n_shards == np_
            assert sorted(set(ranges[:, 0].tolist())) == list(range(owners))
            assert (ranges[:, 1:3] % 128 == 0).all()
            if mode == 0:
                assert shards.tolist() == [[-1, 0]]
                assert ranges.tolist() == [[r, 0, np_, 0] for r in range(owners)]
                continue
            cover = np.zeros(np_, np.int32)
            for owner, s0, s1, slot in ranges.tolist():
                cover[s0:s1] += 1
                assert s1 == s0 + R and shards[s0 // R].tolist() == [owner, slot]
            assert (cover == 1).all()
            if mode == 1:
                # what the in-place all-gather relies on: owner r holds exactly shard r, at its global place
                assert ranges.tolist() == [[r, r * R, (r + 1) * R, r] for r in range(owners)]
            else:
                # device d holds shards d and 2G-1-d, in slots 0 and 1
                assert ranges.tolist() == [x for d in range(owners) for x in
                                           ([d, d * R, (d + 1) * R, 0], [d, (2 * owners - 1 - d) * R, (2 * owners - d) * R, 1])]
                for row0, row1, _, _, owner in _bands_capacity(L, n, np_, owners).tolist():
                    assert (row1 - 1) // R == row0 // R and owner == shards[row0 // R, 0]
