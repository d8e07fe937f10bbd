"""The emulator running the B200 backend's schedules (`Accl.set_one_hop_schedules`): one-hop all-gather /
reduce-scatter, everybody-sends-everything and reduce-scatter + all-gather all-reduce, flat rooted collectives —
in the eager and in the rendezvous configuration, in place, with ranks arriving late (parked calls), mixed with
other calls.  The data flow and the in-place hazards of the GPU schedules are exercised without a GPU
(SURVEY 7.4: one description of the schedules for both backends; the selection rules are plan.hpp's).
"""
import time

import pytest
import torch

import accl_b200 as A
from accl_b200 import MAX, SUM

EAGER = dict(n_egr_rx_bufs=16, egr_rx_buf_size=1024, max_egr_size=1 << 20, max_rndzv_size=1 << 24)
RNDZV = dict(n_egr_rx_bufs=16, egr_rx_buf_size=64, max_egr_size=64, max_rndzv_size=1 << 20)
PROTOCOLS = [pytest.param(EAGER, id="eager"), pytest.param(RNDZV, id="rndzv")]
WORLDS = [2, 3, 4, 5]


def data(count, rank, salt=0, dtype=torch.float32):
    g = torch.Generator().manual_seed(4321 + 31 * rank + salt)
    return torch.randint(-50, 50, (count,), generator=g).to(dtype)   # integer valued: sums are exact in any order


def run(world, fn, cfg):
    def body(a, r, w):
        a.set_one_hop_schedules(True)
        return fn(a, r, w)
    return A.run_ranks(world, body, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("func", [SUM, MAX])
def test_allreduce_one_shot_two_shot_and_odd_counts(world, cfg, func):
    # 24: one hop (small); 8192 * world elements: two hops, shards split evenly; 9001: does not split (flag-in-data class: one hop);
    # 200003: rendezvous class, bytes x P > 2 MiB and a remainder: two hops, the last rank's shard absorbs the remainder
    for count in (24, 8192 * world, 9001, 200003):
        def fn(a, r, w, count=count):
            s, d = a.create_buffer(count), a.create_buffer(count)
            s.host[:] = data(count, r)
            a.allreduce(s, d, count, func)
            ref = torch.stack([data(count, q) for q in range(w)])
            ref = ref.sum(0) if func == SUM else ref.max(0).values
            assert torch.equal(d.host, ref), (count, r)
            assert torch.equal(s.host, data(count, r))                # the source is left alone
        run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", [2, 3, 4])
def test_allreduce_in_place_repeated(world, cfg):
    """src == dst: the fold that writes the result must not run before this rank's own contributions have left."""
    for count in (100, 4096 * world):
        def fn(a, r, w, count=count):
            b = a.create_buffer(count)
            ref = None
            for it in range(3):
                b.host[:] = data(count, r, salt=it)
                a.allreduce(b, b, count, SUM)
                ref = torch.stack([data(count, q, salt=it) for q in range(w)]).sum(0)
                assert torch.equal(b.host, ref), (count, it, r)
        run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", WORLDS)
def test_allgather_and_reduce_scatter(world, cfg):
    count = 777

    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count * w)
        s.host[:] = data(count, r)
        a.allgather(s, d, count)
        assert torch.equal(d.host, torch.cat([data(count, q) for q in range(w)]))
        big, out = a.create_buffer(count * w), a.create_buffer(count)
        big.host[:] = data(count * w, r, salt=5)
        a.reduce_scatter(big, out, count, SUM)
        ref = torch.stack([data(count * w, q, salt=5) for q in range(w)]).sum(0)[r * count:(r + 1) * count]
        assert torch.equal(out.host, ref)
    run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", [3, 4, 5])
def test_rooted_collectives_take_their_flat_forms(world, cfg):
    count = 500

    def fn(a, r, w):
        for root in range(w):
            s, d = a.create_buffer(count), a.create_buffer(count)
            s.host[:] = data(count, r, salt=root)
            a.reduce(s, d, count, root, SUM)
            if r == root:
                assert torch.equal(d.host, torch.stack([data(count, q, salt=root) for q in range(w)]).sum(0))
            g = a.create_buffer(count * w)
            a.gather(s, g, count, root)
            if r == root:
                assert torch.equal(g.host, torch.cat([data(count, q, salt=root) for q in range(w)]))
            b = a.create_buffer(count)
            if r == root:
                b.host[:] = data(count, root, salt=99)
            a.bcast(b, count, root)
            assert torch.equal(b.host, data(count, root, salt=99))
    run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_late_ranks_park_the_call_instead_of_failing(cfg):
    """Rendezvous form: a rank whose peers have not arrived yet returns NOT_READY and is resumed at its saved step."""
    count, world = 6000, 4

    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        time.sleep(0.05 * r)                                   # ranks enter the call 50 ms apart
        a.allreduce(s, d, count, SUM)
        assert torch.equal(d.host, torch.stack([data(count, q) for q in range(w)]).sum(0))
        time.sleep(0.03 * (w - r))
        out = a.create_buffer(count // w)
        a.reduce_scatter(s, out, count // w, SUM)
        ref = torch.stack([data(count, q) for q in range(w)]).sum(0)
        assert torch.equal(out.host, ref[r * (count // w):(r + 1) * (count // w)])
    run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_mixed_sequence_with_point_to_point_and_subcommunicator(cfg):
    world, count = 4, 1200

    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        for it in range(3):
            a.allreduce(s, d, count, SUM)
            nxt, prv = (r + 1) % w, (r - 1) % w
            t = a.create_buffer(count)
            q = a.send(s, count, nxt, tag=it, run_async=True)
            a.recv(t, count, prv, tag=it)
            q.wait()
            assert torch.equal(t.host, data(count, prv))
            g = a.create_buffer(count * w)
            a.allgather(s, g, count)
            assert torch.equal(g.host[r * count:(r + 1) * count], s.host)
        assert torch.equal(d.host, torch.stack([data(count, q) for q in range(w)]).sum(0))
        # a sub-communicator of the even ranks runs the same schedules on its own sequence space
        ranks = A.Accl.generate_ranks(w)
        if r % 2 == 0:
            comm = a.create_communicator([ranks[0], ranks[2]], r // 2)
            a.allreduce(s, d, count, SUM, comm_id=comm)
            assert torch.equal(d.host, data(count, 0) + data(count, 2))
    run(world, fn, cfg)


def test_reference_schedules_are_the_default_and_agree():
    """Same call, both schedule families, same answer; the register defaults to the reference's rings / trees."""
    count, world = 3000, 4

    def fn(a, r, w):
        s, d1, d2 = a.create_buffer(count), a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        a.allreduce(s, d1, count, SUM)
        a.barrier()
        a.set_one_hop_schedules(True)
        a.barrier()
        a.allreduce(s, d2, count, SUM)
        assert torch.equal(d1.host, d2.host)
        a.barrier()
        a.set_one_hop_schedules(False)
        return True
    assert all(A.run_ranks(world, fn, EAGER))


def _dispatches(a):
    txt = A._C.emu_debug_state(a.impl)
    return int(txt.split("one_hop_dispatches=")[1].split()[0])


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_the_one_hop_handlers_really_run(cfg):
    """The statistic in the engine's state dump counts calls dispatched to the one-hop handlers: it moves with the
    register on, stands still with it off and for calls the handlers do not take (compressed wire)."""
    count, world = 2048, 3

    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        a.barrier()
        n0 = _dispatches(a)
        a.barrier()
        a.allreduce(s, d, count, SUM)                 # register off: ring / tree
        a.barrier()
        n1 = _dispatches(a)
        a.barrier()
        a.set_one_hop_schedules(True)
        a.allreduce(s, d, count, SUM)
        a.reduce_scatter(s, d, count // 4, SUM)
        a.barrier()
        n2 = _dispatches(a)
        a.barrier()
        a.allreduce(s, d, count, SUM, compress_dtype=torch.float16)   # compressed: not a one-hop call
        a.barrier()
        n3 = _dispatches(a)
        a.barrier()
        return n0, n1, n2, n3
    for n0, n1, n2, n3 in A.run_ranks(world, fn, cfg):
        assert n1 == n0 and n2 >= n1 + 2 * world and n3 == n2


def _stat(a, name):
    return int(A._C.emu_debug_state(a.impl).split(name + "=")[1].split()[0])


@pytest.mark.skipif(not A._C.with_cuda, reason="the planner hook lives in the CUDA build")
@pytest.mark.parametrize("cfg,max_eager", [(EAGER, 1 << 20), (RNDZV, 64)], ids=["eager", "rndzv"])
def test_one_shot_or_two_shot_is_the_planners_decision(cfg, max_eager):
    """For the same (count, world, eager threshold) the emulator takes the form `plan_call` picks for the GPU:
    flag-in-data class: one hop up to 32 KiB; rendezvous class: one hop while bytes x P <= 2 MiB."""
    world = 4
    Op = A._C.Operation
    for count in (256, 8192, 65536, 262144):
        p = A._C.cuda_plan(Op.allreduce, count, A.DataType.float32, world, max_eager_bytes=max_eager,
                           eager_rx_buf_bytes=64 << 10, max_ctas=128, stage_kb=1024, ll_kb=2048)
        want_one_shot = p["algo"] in ("p2p_oneshot", "eager") or (p["algo"] in ("ll", "staged") and p["oneshot"])

        def fn(a, r, w, count=count):
            s, d = a.create_buffer(count), a.create_buffer(count)
            s.host[:] = data(count, r)
            a.barrier()
            one0, two0 = _stat(a, "allreduce_one_shot"), _stat(a, "allreduce_two_shot")
            a.barrier()
            a.allreduce(s, d, count, SUM)
            a.barrier()
            one1, two1 = _stat(a, "allreduce_one_shot"), _stat(a, "allreduce_two_shot")
            a.barrier()
            assert torch.equal(d.host, torch.stack([data(count, q) for q in range(w)]).sum(0))
            return one1 - one0, two1 - two0
        for one, two in run(world, fn, dict(cfg, max_rndzv_size=1 << 22)):
            assert (one >= world and two == 0) if want_one_shot else (two >= world and one == 0), (count, p, one, two)
