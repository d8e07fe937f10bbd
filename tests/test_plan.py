"""The CUDA backend's call planner (csrc/include/accl/cuda/plan.hpp) as a pure function: protocol, algorithm
and channel-count decisions must be identical on every rank and follow the documented rules (docs/tuning.md).
Runs without a GPU (the planner is host/device-shared code); skipped on emulator-only builds."""
import pytest

import accl_b200 as A
from accl_b200 import DataType

pytestmark = pytest.mark.skipif(not A._C.with_cuda, reason="built without the CUDA backend")
Op = A._C.Operation
F32 = DataType.float32


# the configuration these tests were written against: 128 channels, 1 MiB staging / 256 KiB LL regions, 64 KiB eager
# limits; every other option at its CudaConfig default
PINNED = dict(max_ctas=128, stage_kb=1024, ll_kb=256, max_eager_bytes=64 << 10, eager_rx_buf_bytes=64 << 10)


def plan(op, nbytes, world=8, dtype=F32, esz=4, **kw):
    return A._C.cuda_plan(op, nbytes // esz, dtype, world, **{**PINNED, **kw})


ONE_WAY = ("eager", "ll", "staged")  # protocols without a meeting: slot ring, flag-in-data, payload + flag


def test_eager_vs_rendezvous_threshold():
    assert plan(Op.allreduce, 64 << 10)["algo"] in ONE_WAY           # bytes <= max_eager_size
    assert plan(Op.allreduce, (64 << 10) + 4)["algo"] not in ONE_WAY
    assert plan(Op.allreduce, 64 << 20, compressed=True)["algo"] == "eager"   # compressed calls always use slots
    assert plan(Op.send, 1 << 20)["algo"] == "p2p" and plan(Op.recv, 1 << 20)["algo"] == "p2p"
    assert plan(Op.send, 1024)["algo"] == "eager" and plan(Op.send, 1024)["n_ctas"] == 1  # eager point to point: one channel


def test_one_way_protocol_selection():
    # all-reduce: one hop (everybody sends everything) while tiny, reduce-scatter + all-gather above
    p = plan(Op.allreduce, 1024)
    assert p["algo"] == "ll" and p["oneshot"] and p["n_ctas"] == 1
    p = plan(Op.allreduce, 64 << 10)
    assert p["algo"] == "ll" and not p["oneshot"]                     # shards of 8 KiB through the flag-in-data protocol
    p = plan(Op.allreduce, 2 << 20, max_eager_bytes=4 << 20, ll_kb=2048)
    assert p["algo"] == "ll" and not p["oneshot"] and p["n_ctas"] == 32   # shards of 256 KiB: 32 K lines over all channels
    # what does not fit the LL region: the payload + flag protocol when that is enabled, else the slot ring while
    # that is a handful of segments, else the rendezvous algorithms
    assert plan(Op.allreduce, 2 << 20, max_eager_bytes=4 << 20)["algo"] == "nvls"
    assert plan(Op.allreduce, 2 << 20, max_eager_bytes=4 << 20, staged_max_bytes=1 << 20)["algo"] == "staged"
    assert plan(Op.allgather, 128 << 10, max_eager_bytes=4 << 20, ll_kb=128)["algo"] == "eager"   # 2 segments of 64 KiB
    assert plan(Op.allgather, 256 << 10, max_eager_bytes=4 << 20)["algo"] == "p2p"     # 4 segments: user buffer to user buffer
    # sizes that do not split into 16-byte shards go one-shot while small, to the other paths otherwise
    assert plan(Op.allreduce, 20000)["oneshot"]
    assert plan(Op.allreduce, (1 << 20) + 4, max_eager_bytes=4 << 20)["algo"] == "nvls"
    # per-peer message decides for the others
    assert plan(Op.allgather, 8 << 10)["algo"] == "ll"
    assert plan(Op.reduce_scatter, 16 << 10)["algo"] == "ll"
    assert plan(Op.bcast, 32 << 10)["algo"] == "ll"
    assert plan(Op.bcast, 32 << 10, ll_max_bytes=16384, staged_max_bytes=1 << 20)["algo"] == "staged"   # the crossover is a knob
    assert plan(Op.allgather, 256 << 10, max_eager_bytes=1 << 20, staged_max_bytes=1 << 20)["algo"] == "staged"   # 256 KiB > LL capacity of 128 KiB
    assert plan(Op.allgather, 256 << 10, max_eager_bytes=1 << 20, ll_kb=2048)["algo"] == "ll"
    # flag-in-data doubles the wire bytes: budgeted on message x (P - 1) peers (2 MiB), so the crossover moves with P
    big = dict(max_eager_bytes=4 << 20, ll_kb=2048)
    assert plan(Op.allgather, 256 << 10, world=8, **big)["algo"] == "ll"      # 7 x 256 KiB
    assert plan(Op.allgather, 512 << 10, world=8, **big)["algo"] == "p2p"     # 7 x 512 KiB: user buffer to user buffer
    assert plan(Op.allgather, 512 << 10, world=4, **big)["algo"] == "ll"      # 3 x 512 KiB
    assert plan(Op.allreduce, 4 << 20, world=8, **big)["algo"] == "nvls"      # shards of 512 KiB to 7 peers
    assert plan(Op.allreduce, 2 << 20, world=2, **big)["algo"] == "ll"        # one shard of 1 MiB to one peer
    assert plan(Op.bcast, 512 << 10, world=8, **big)["algo"] == "nvls"        # the root would push 7 x 512 KiB x 2
    # no staging configured: everything one-way is the slot ring
    assert plan(Op.allreduce, 1024, stage_kb=0, ll_kb=0)["algo"] == "eager"
    # channel counts: every channel owns 1/32 of a region
    assert plan(Op.allgather, 256 << 10, max_eager_bytes=1 << 20, staged_max_bytes=1 << 20)["n_ctas"] == 8   # 32 KiB per channel
    # inside the engine a message that fits one channel stays on one (executed inline by the control CTA)
    assert plan(Op.allreduce, 8 << 10, ll_kb=2048, engine_mode=True)["n_ctas"] == 1
    assert plan(Op.allreduce, 8 << 10, ll_kb=2048)["n_ctas"] == 2


def test_allreduce_algorithm_by_size_and_world():
    # one-shot while bytes * P <= 2 MiB, then two-shot: through the switch from 3 ranks, peer load/store below
    assert plan(Op.allreduce, 128 << 10, world=8)["algo"] == "p2p_oneshot"
    assert plan(Op.allreduce, 512 << 10, world=8)["algo"] == "nvls"
    assert plan(Op.allreduce, 512 << 10, world=2)["algo"] == "p2p_oneshot"
    assert plan(Op.allreduce, 128 << 10, world=8, max_eager_bytes=1 << 20)["algo"] in ONE_WAY
    assert plan(Op.allreduce, 4 << 20, world=2)["algo"] == "p2p"
    assert plan(Op.allreduce, 4 << 20, world=8, has_mc=False)["algo"] == "p2p"
    assert plan(Op.allreduce, 4 << 20, world=4, nvls_min_ranks=99)["algo"] == "p2p"


def test_nvls_only_for_ops_that_win_through_the_switch():
    for op in (Op.allreduce, Op.bcast, Op.reduce):
        assert plan(op, 16 << 20)["algo"] == "nvls"
    for op in (Op.allgather, Op.reduce_scatter, Op.scatter, Op.gather, Op.alltoall):
        assert plan(op, 1 << 20)["algo"] == "p2p"                     # less traffic per link with peer stores / loads


def test_channel_counts():
    assert plan(Op.allreduce, 256 << 20, max_ctas=128)["n_ctas"] == 32      # measured: few channels win through the switch
    assert plan(Op.allreduce, 64 << 20, world=2, max_ctas=128)["n_ctas"] == 128    # peer loads / stores want them all
    assert plan(Op.allreduce, 256 << 20, world=2, max_ctas=128)["n_ctas"] == 128
    assert plan(Op.reduce_scatter, 32 << 20, max_ctas=128)["n_ctas"] == 128  # 8 x 32 MiB moved: all channels
    assert plan(Op.allgather, 128 << 10, max_ctas=128)["n_ctas"] == 8        # 8 x 128 KiB moved at 128 KiB per channel
    assert plan(Op.allreduce, 1024, max_ctas=128)["n_ctas"] == 1
    assert plan(Op.allreduce, 64 << 10, max_ctas=128, stage_kb=0, ll_kb=0)["n_ctas"] == 4   # slot ring: 16 KiB per channel, <= 16 channels
    assert plan(Op.allreduce, 256 << 20, max_ctas=1000, nvls_min_ranks=99)["n_ctas"] <= 128   # never more channels than sync pads
    assert plan(Op.copy, 1 << 30)["algo"] == "local" and plan(Op.copy, 1 << 30)["n_ctas"] == 296
    assert plan(Op.barrier, 0)["n_ctas"] == 1 and plan(Op.nop, 0)["algo"] == "local"


# ---- invariants over random calls and configurations (the planner runs on every rank and on the device: whatever it
# returns must be executable by the protocol it names)
from hypothesis import HealthCheck, given, settings, strategies as st  # noqa: E402

COLLECTIVES = [Op.allreduce, Op.allgather, Op.reduce_scatter, Op.bcast, Op.scatter, Op.gather, Op.reduce, Op.alltoall]


@settings(max_examples=600, deadline=None, suppress_health_check=[HealthCheck.too_slow])
@given(op=st.sampled_from(COLLECTIVES + [Op.send, Op.recv]), count=st.integers(1, 1 << 28), world=st.integers(2, 8),
       max_eager=st.sampled_from([1024, 64 << 10, 1 << 20, 4 << 20]), max_ctas=st.sampled_from([1, 8, 32, 64, 128, 1000]),
       has_mc=st.booleans(), ll_kb=st.sampled_from([0, 64, 256, 2048]), stage_kb=st.sampled_from([0, 1024]),
       staged_max=st.sampled_from([0, 1 << 20]), engine_mode=st.booleans(), compressed=st.booleans())
def test_plans_are_executable(op, count, world, max_eager, max_ctas, has_mc, ll_kb, stage_kb, staged_max, engine_mode, compressed):
    p = A._C.cuda_plan(op, count, F32, world, max_eager_bytes=max_eager, eager_rx_buf_bytes=64 << 10, max_ctas=max_ctas,
                       has_mc=has_mc, ll_kb=ll_kb, stage_kb=stage_kb, staged_max_bytes=staged_max, engine_mode=engine_mode,
                       compressed=compressed)
    nbytes = count * 4
    assert p["algo"] in ("eager", "nvls", "p2p", "p2p_oneshot", "ll", "staged", "wire")
    assert 1 <= p["n_ctas"] <= min(max(max_ctas, 1), 128)                     # never more channels than sync pads / the cap
    if p["algo"] in ("ll", "staged"):
        assert nbytes <= max_eager and not compressed and op not in (Op.send, Op.recv)
        assert p["n_ctas"] <= 32                                              # staging regions are cut into 32 channel slices
        m = nbytes // world if (op == Op.allreduce and not p["oneshot"]) else nbytes
        region = (ll_kb if p["algo"] == "ll" else stage_kb) << 10
        assert 0 < m <= region // (2 if p["algo"] == "ll" else 1)             # the message fits its staging region
        if p["algo"] == "ll":
            assert m * (world - 1) <= 2 << 20                                 # the fan-out budget
    if p["oneshot"]:
        assert op == Op.allreduce and p["algo"] in ("ll", "staged")
    if p["algo"] == "nvls":
        assert has_mc and world >= 3 and op in (Op.allreduce, Op.bcast, Op.reduce)
    if p["algo"] == "p2p_oneshot":
        assert op == Op.allreduce and nbytes * world <= 2 << 20
    if op in (Op.send, Op.recv):
        assert p["algo"] in ("eager", "p2p") and (p["algo"] == "p2p" or p["n_ctas"] == 1)
    if nbytes > max_eager and not compressed:
        assert p["algo"] in ("nvls", "p2p", "p2p_oneshot")                    # rendezvous class


@settings(max_examples=200, deadline=None)
@given(op=st.sampled_from(COLLECTIVES), world=st.integers(2, 8), lo=st.integers(1, 1 << 20))
def test_channel_count_grows_with_the_message_within_one_protocol(op, world, lo):
    """Within one algorithm a larger message never gets fewer channels."""
    a = plan(op, lo * 4, world=world, max_eager_bytes=4 << 20, ll_kb=2048)
    b = plan(op, lo * 8, world=world, max_eager_bytes=4 << 20, ll_kb=2048)
    if a["algo"] == b["algo"] and a["oneshot"] == b["oneshot"]:
        assert b["n_ctas"] >= a["n_ctas"], (a, b)


def test_options_default_to_the_device_configuration():
    """No option given plans as a device built with every CudaConfig default; unknown names are refused."""
    nvls_ops = (1 << int(Op.allreduce)) | (1 << int(Op.bcast)) | (1 << int(Op.reduce))
    defaults = dict(heap_mb=1024, multicast=1, engine=0, engine_workers=0, engine_idle_us=1000, oneshot_kb=2048,
                    nvls_ops=nvls_ops, host_pipeline_chunk_kb=16 << 10, max_ctas=32, nvls_min_ranks=3, nvls_ctas=32,
                    hybrid_16ths=0, nvls_unroll=4, reduce_push=0, bcast_flags=0, split_phases=0, ll_max_bytes=2 << 20,
                    ll_oneshot_max=32 << 10, oneshot_max_bytes=2 << 20, wire_min_bytes=256 << 10, staged_max_bytes=0,
                    stream_loopback=1)
    geometry = dict(max_eager_bytes=4 << 20, eager_rx_buf_bytes=64 << 10, stage_kb=1024, ll_kb=256)
    for op in COLLECTIVES + [Op.send]:
        for nbytes in (1024, 64 << 10, 1 << 20, 16 << 20, 256 << 20):
            for world in (2, 4, 8):
                for engine_mode in (False, True):
                    call = (op, nbytes // 4, F32, world)
                    assert (A._C.cuda_plan(*call, engine_mode=engine_mode, **geometry) ==
                            A._C.cuda_plan(*call, engine_mode=engine_mode, **geometry, **defaults)), (call, engine_mode)
    with pytest.raises(ValueError, match="unknown CUDA backend option 'no_such_knob'"):
        A._C.cuda_plan(Op.allreduce, 1024, F32, 8, **geometry, no_such_knob=1)
