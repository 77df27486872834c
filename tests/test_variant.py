"""Which variant of the fast path frc_create runs (frackyfrac_b200/csrc/plan.cpp: plan_exchange, plan_variant) on the
CPU box: how the sample shards meet, the capacity mode of the weighted panels, the unweighted operand kind, the bits
feed, and the flags the stages read from that decision.

Two choices are automatic and depend on device 0's free HBM: the capacity mode (panels over 24 GiB and over 55 % of
it) and the bits feed (u8 operands over 32 GiB and over 80 % of it).  A wrong gate sends a large job out of memory or
runs a job that fits at about half the speed.  frc_debug_plan_variant takes the free HBM as a number and counts how
often it is asked, so every branch is tested here without a device.  The knobs are read from the environment, as
frc_create reads them.  Every expected outcome is written out by hand."""
import ctypes as C
import types

import numpy as np
import pytest

FIELDS = ("exchange", "fused_embed", "sharded_fast_uw", "capacity", "shard_mode", "want_i8", "bits_feed",
          "rowsum_in_expand", "rowsum_split", "peer_store", "peer_push", "need_blocks", "operand_kind", "intacc", "kp",
          "asked")
NONE, IN_PROCESS, NCCL = 0, 1, 2    # Variant::Exchange
WHOLE, SHARDED, CAPACITY = 0, 1, 2  # ShardPlan::Mode
OK, ERR_STATE, ERR_UNSUPPORTED = 0, 4, 5
SHARD_EMBED, UW_BF16, UW_BITS = 4, 2, 8  # FRC_FLAG_*
GiB = 1 << 30
KNOBS = ("FRC_SHARD", "FRC_EMBED_LEVELS", "FRC_CAPACITY", "FRC_UW_KERNEL", "FRC_UW_FEED", "FRC_U8_ACC", "FRC_PEER_PUSH",
         "FRC_U8_GROUP_BINADES")

MSG_COMM = ("FRC_FLAG_SHARD_EMBED needs a context whose communicator (frc_ctx_comm_init) matches opts->rank / "
            "opts->world")
MSG_LEVELS = "FRC_EMBED_LEVELS=1 cannot build a sample shard"
MSG_RECT = ("frc_create_cross keeps the weighted panels of all samples on every device; the capacity mode, which shards "
            "them over the devices when they exceed about half of one device's free HBM (or with FRC_CAPACITY=1), only "
            "runs triangle jobs")
MSG_KEYED = ("the key-matched tiles of -l as coded (FRC_FLAG_L_TILES) keep the value and key panels of all samples on "
             "every device; the capacity mode, which shards them over the devices when they exceed about half of one "
             "device's free HBM (or with FRC_CAPACITY=1), does not carry keys")

# Gate boundaries.  Weighted panels of 1024 nodes over two devices (np = N rounded up to 512): 4 * 1024 * np bytes.
CAP_AT_24 = 6291456         # panels exactly 24 GiB: not over the gate
CAP_OVER_24 = 6291457       # np 6291968: panels 25771900928 bytes
CAP_FREE_CHOSEN = 46858001687   # panels > 0.55 x this
CAP_FREE_NOT = 46858001688      # panels < 0.55 x this
KEYED_AT_24 = 3145728       # keyed: 8 bytes per entry, exactly 24 GiB
KEYED_OVER_24 = 3145729     # keyed 25773998080 bytes; 4 bytes per entry would be half that
# u8 operands of 1024 equal lengths (kp 1024) on one device (np = N rounded up to 128): 3 * np * kp bytes.
U8_UNDER_32 = 11184768      # 34359607296 bytes
U8_OVER_32 = 11184769       # np 11184896: 34360000512 bytes
U8_FREE_CHOSEN = 42950000639    # need > 0.80 x this
U8_FREE_NOT = 42950000641       # need < 0.80 x this


@pytest.fixture(scope="module")
def L(built):
    from frackyfrac_b200 import engine

    lib = engine.lib()
    i32, P = C.c_int32, C.c_void_p
    lib.frc_debug_plan_variant.argtypes = [i32, i32, i32, i32, C.c_uint32, i32, i32, C.c_int64, P, i32, i32, i32, i32,
                                           i32, i32, C.c_int64, P, C.c_char_p, C.c_int64]
    lib.frc_debug_plan_variant.restype = i32
    return lib


@pytest.fixture
def plan(L, monkeypatch):
    def run(weighted=False, exact=False, keyed=False, rect=False, flags=0, world=1, rank=0, N=1000, B=1024,
            n_parts=1, peer_ok=True, comm=None, neg_len=False, free=200 * GiB, **env):
        """The variant of one job: env holds the FRC_* knobs (every other knob unset); comm = (world, rank) of the
        context's communicator; free < 0: the free-HBM query fails."""
        for k in KNOBS:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, str(v))
        length = np.ones(B)
        cw, cr = comm if comm is not None else (-1, -1)
        out = np.full(len(FIELDS), -7, np.int64)
        msg = C.create_string_buffer(1024)
        rc = L.frc_debug_plan_variant(int(weighted), int(exact), int(keyed), int(rect), flags, world, rank, N,
                                      length.ctypes.data, B, n_parts, int(peer_ok), cw, cr, int(neg_len), free,
                                      out.ctypes.data, msg, len(msg))
        return types.SimpleNamespace(rc=rc, msg=msg.value.decode(), **dict(zip(FIELDS, out.tolist())))
    return run


def expect(r, **want):
    got = {k: getattr(r, k) for k in want}
    assert got == want


# ------------------------------------------------------------------ how the sample shards meet
@pytest.mark.parametrize("job, want", [
    (dict(exact=True, n_parts=2), dict(exchange=NONE, sharded_fast_uw=0, shard_mode=WHOLE)),
    (dict(n_parts=2), dict(exchange=IN_PROCESS, sharded_fast_uw=1, shard_mode=SHARDED)),
    (dict(n_parts=2, weighted=True), dict(exchange=IN_PROCESS, sharded_fast_uw=0, shard_mode=SHARDED)),
    (dict(n_parts=2, peer_ok=False), dict(exchange=NONE, sharded_fast_uw=0, shard_mode=WHOLE)),
    (dict(n_parts=2, FRC_SHARD=0), dict(exchange=NONE, sharded_fast_uw=0, shard_mode=WHOLE)),
    (dict(n_parts=2, FRC_EMBED_LEVELS=1), dict(exchange=NONE, fused_embed=0, shard_mode=WHOLE)),
    (dict(n_parts=2, weighted=True, FRC_EMBED_LEVELS=1), dict(exchange=IN_PROCESS, fused_embed=0, shard_mode=SHARDED)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1)), dict(exchange=NCCL, sharded_fast_uw=1, shard_mode=SHARDED)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1), weighted=True),
     dict(exchange=NCCL, sharded_fast_uw=0, shard_mode=SHARDED)),
    (dict(world=4, rank=1, comm=(4, 1)), dict(exchange=NONE, sharded_fast_uw=0, shard_mode=WHOLE)),
    (dict(flags=SHARD_EMBED), dict(exchange=NONE, shard_mode=WHOLE)),
])
def test_exchange(plan, job, want):
    r = plan(**job)
    assert (r.rc, r.msg) == (OK, "")
    expect(r, **want)


@pytest.mark.parametrize("job, rc, msg", [
    (dict(), ERR_STATE, MSG_COMM),                                 # no communicator
    (dict(comm=(2, 1)), ERR_STATE, MSG_COMM),                      # another world
    (dict(comm=(4, 0)), ERR_STATE, MSG_COMM),                      # another rank
    (dict(comm=(4, 1), FRC_EMBED_LEVELS=1), ERR_UNSUPPORTED, MSG_LEVELS),
    (dict(FRC_EMBED_LEVELS=1), ERR_STATE, MSG_COMM),               # both: the communicator first
    (dict(comm=(4, 1), FRC_EMBED_LEVELS=1, weighted=True), OK, ""),  # the weighted path builds its shard per slab
])
def test_nccl_refusals(plan, job, rc, msg):
    r = plan(world=4, rank=1, flags=SHARD_EMBED, **job)
    assert (r.rc, r.msg) == (rc, msg)


# ------------------------------------------------------------------ capacity mode of the weighted panels
@pytest.mark.parametrize("job, capacity, mode, asked", [
    (dict(FRC_CAPACITY=1), 1, CAPACITY, 0),
    (dict(FRC_CAPACITY=0, N=CAP_OVER_24, free=1), 0, SHARDED, 0),
    (dict(FRC_CAPACITY=1, N=1), 0, SHARDED, 0),
    (dict(FRC_CAPACITY=1, weighted=False), 0, SHARDED, 0),
    (dict(FRC_CAPACITY=1, peer_ok=False), 0, WHOLE, 0),
    (dict(FRC_CAPACITY=1, FRC_SHARD=0), 0, WHOLE, 0),
    (dict(N=CAP_OVER_24, free=1, peer_ok=False), 0, WHOLE, 0),
    (dict(N=CAP_AT_24, free=1), 0, SHARDED, 0),                   # at the gate: free HBM is not asked
    (dict(N=CAP_OVER_24, free=CAP_FREE_CHOSEN), 1, CAPACITY, 1),
    (dict(N=CAP_OVER_24, free=CAP_FREE_NOT), 0, SHARDED, 1),
    (dict(N=CAP_OVER_24, free=-1), 0, SHARDED, 1),                # the query failed: not chosen
    (dict(N=KEYED_AT_24, keyed=True, free=1 << 40), 0, SHARDED, 0),
    (dict(N=KEYED_OVER_24, keyed=True, free=1 << 40), 0, SHARDED, 1),  # 8 bytes per keyed entry
    (dict(N=KEYED_OVER_24, free=1), 0, SHARDED, 0),                    # 4 bytes unkeyed: under the gate
    (dict(N=CAP_OVER_24, rect=True, free=CAP_FREE_NOT), 0, SHARDED, 1),
])
def test_capacity_mode(plan, job, capacity, mode, asked):
    r = plan(**{"weighted": True, "n_parts": 2, **job})
    assert (r.rc, r.msg) == (OK, "")
    expect(r, capacity=capacity, shard_mode=mode, asked=asked)


@pytest.mark.parametrize("job, msg", [
    (dict(rect=True, FRC_CAPACITY=1), MSG_RECT),
    (dict(rect=True, N=CAP_OVER_24, free=CAP_FREE_CHOSEN), MSG_RECT),
    (dict(keyed=True, FRC_CAPACITY=1), MSG_KEYED),
    (dict(keyed=True, N=KEYED_OVER_24, free=1), MSG_KEYED),
    (dict(rect=True, keyed=True, FRC_CAPACITY=1), MSG_RECT),
])
def test_capacity_refusals(plan, job, msg):
    r = plan(weighted=True, n_parts=2, **job)
    assert (r.rc, r.msg) == (ERR_UNSUPPORTED, msg)


# ------------------------------------------------------------------ unweighted operands
@pytest.mark.parametrize("job, kind, want_i8, intacc, bits", [
    (dict(), 2, 1, 1, 0),
    (dict(flags=UW_BF16), 1, 0, 0, 0),
    (dict(FRC_UW_KERNEL="bf16"), 1, 0, 0, 0),
    (dict(neg_len=True), 1, 0, 0, 0),
    (dict(FRC_EMBED_LEVELS=1), 1, 0, 0, 0),
    (dict(FRC_U8_ACC="f64"), 2, 1, 0, 0),
    (dict(FRC_U8_ACC="f64", flags=UW_BITS), 2, 1, 0, 0),   # the bits feed needs the integer mode
    (dict(FRC_U8_ACC="f64", FRC_UW_FEED="bits"), 2, 1, 0, 0),
    (dict(flags=UW_BITS), 3, 1, 1, 1),
    (dict(FRC_UW_FEED="bits"), 3, 1, 1, 1),
    (dict(flags=UW_BF16 | UW_BITS), 1, 0, 0, 0),
    (dict(weighted=True), 0, 0, 0, 0),
    (dict(exact=True), 0, 0, 0, 0),
])
def test_operand_kind(plan, job, kind, want_i8, intacc, bits):
    r = plan(**job)
    assert (r.rc, r.msg) == (OK, "")
    expect(r, operand_kind=kind, want_i8=want_i8, intacc=intacc, bits_feed=bits, asked=0)


@pytest.mark.parametrize("job, bits, asked", [
    (dict(N=U8_UNDER_32, free=1), 0, 0),                 # under the gate: free HBM is not asked
    (dict(N=U8_UNDER_32, free=1, n_parts=2), 1, 1),      # np of two shards: 11184896
    (dict(N=U8_UNDER_32, free=1, world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1)), 1, 1),  # four shards: 11185152
    (dict(N=U8_OVER_32, free=U8_FREE_CHOSEN), 1, 1),
    (dict(N=U8_OVER_32, free=U8_FREE_NOT), 0, 1),
    (dict(N=U8_OVER_32, free=-1), 0, 1),                 # the query failed: not chosen
    (dict(N=U8_OVER_32, free=1, flags=UW_BITS), 1, 0),   # forced: nothing to ask
    (dict(N=U8_OVER_32, free=1, FRC_U8_ACC="f64"), 0, 0),
    (dict(N=U8_OVER_32, free=1, flags=UW_BF16), 0, 0),
    (dict(N=U8_OVER_32, free=1, weighted=True), 0, 0),
])
def test_bits_feed_gate(plan, job, bits, asked):
    r = plan(**job)
    assert (r.rc, r.msg) == (OK, "")
    if not job.get("weighted") and not job.get("flags", 0) & UW_BF16:
        assert r.kp == 1024
    expect(r, bits_feed=bits, asked=asked)


# ------------------------------------------------------------------ what the stages read
@pytest.mark.parametrize("job, want", [
    (dict(), dict(rowsum_in_expand=1, rowsum_split=0, peer_store=0, peer_push=0, need_blocks=0)),
    (dict(flags=UW_BF16), dict(rowsum_in_expand=0, rowsum_split=1, peer_store=0, need_blocks=0)),
    (dict(flags=UW_BITS), dict(rowsum_in_expand=0, rowsum_split=1, peer_store=0, need_blocks=0)),
    (dict(FRC_EMBED_LEVELS=1), dict(rowsum_in_expand=0, rowsum_split=0, need_blocks=0)),
    (dict(n_parts=2), dict(rowsum_in_expand=1, rowsum_split=0, peer_store=1, peer_push=0, need_blocks=1)),
    (dict(n_parts=2, flags=UW_BITS), dict(rowsum_in_expand=0, rowsum_split=0, peer_store=0, need_blocks=1)),
    (dict(n_parts=2, flags=UW_BF16), dict(rowsum_in_expand=0, rowsum_split=0, peer_store=1, need_blocks=1)),
    (dict(n_parts=2, peer_ok=False, flags=UW_BF16), dict(rowsum_split=1, peer_store=0, need_blocks=1)),
    (dict(n_parts=2, FRC_EMBED_LEVELS=1), dict(rowsum_split=0, peer_store=0, need_blocks=0)),
    (dict(world=4, rank=1), dict(peer_push=0, need_blocks=1, rowsum_split=0)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1)),
     dict(peer_push=1, peer_store=0, need_blocks=1, rowsum_split=0, rowsum_in_expand=1)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1), FRC_PEER_PUSH=1), dict(peer_push=1)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1), FRC_PEER_PUSH=0), dict(peer_push=0)),
    (dict(world=8, rank=7, flags=SHARD_EMBED, comm=(8, 7)), dict(peer_push=1)),
    (dict(world=9, rank=1, flags=SHARD_EMBED, comm=(9, 1)), dict(peer_push=0)),
    (dict(world=4, rank=1, flags=SHARD_EMBED | UW_BITS, comm=(4, 1)), dict(peer_push=0, rowsum_split=0)),
    (dict(world=4, rank=1, flags=SHARD_EMBED, comm=(4, 1), weighted=True), dict(peer_push=0, need_blocks=0)),
    (dict(n_parts=2, weighted=True), dict(peer_store=0, need_blocks=0, rowsum_split=0)),
])
def test_stage_flags(plan, job, want):
    r = plan(**job)
    assert (r.rc, r.msg) == (OK, "")
    expect(r, **want)
