"""GPU tests of the one-way staged protocols (ALGO_LL: flag carried in the data; ALGO_STAGED: payload + release
flag; csrc/src/cuda/staged.cuh).  Sizes are chosen so that every branch of the planner is taken: one-hop and
two-hop all-reduce, one and several channels, unaligned tails, in-place operands, long call sequences (staging
parity reuse and credits), mixed operations on one communicator, rooted patterns from every root, sub-communicators.
Reference matrix: test/host/xrt/src/test.cpp (bcast :508, scatter :558, gather :592, allgather :667, reduce :834,
reduce_scatter :1020, allreduce :1068, segmentation +-1 :345-393)."""
import pytest
import torch

import accl_b200 as A
from accl_b200 import MAX, SUM

pytestmark = pytest.mark.gpu
NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0
ONEWAY = dict(n_egr_rx_bufs=4, egr_rx_buf_size=16 << 10, max_egr_size=4 << 20, max_rndzv_size=1 << 30)


def devices(world):
    return [r % max(NGPU, 1) for r in range(world)]


def data(count, rank, dtype=torch.float32, salt=0):
    g = torch.Generator().manual_seed(977 + 131 * rank + salt)
    if dtype in (torch.int32, torch.int64):
        return torch.randint(-1000, 1000, (count,), generator=g, dtype=dtype)
    return (torch.rand(count, generator=g, dtype=torch.float32) * 8 - 4).to(dtype)


def ref_reduce(world, count, func, dtype=torch.float32, salt=0):
    xs = [data(count, r, dtype, salt).to(torch.float64 if dtype.is_floating_point else torch.int64) for r in range(world)]
    out = xs[0].clone()
    for x in xs[1:]:
        out = out + x if func == SUM else torch.maximum(out, x)
    return out


def close(a, b, rtol=1e-5, atol=1e-5):
    return torch.allclose(a.cpu().to(torch.float64), b.cpu().to(torch.float64), rtol=rtol, atol=atol)


def run(world, fn, **kw):
    # staged_max_bytes: also exercise the payload + release-flag protocol for what does not fit the LL regions
    cfg = dict(heap_mb=256, max_ctas=16, ll_kb=512, staged_max_bytes=2 << 20)
    cfg.update(kw)
    return A.run_cuda_ranks(devices(world), fn, ONEWAY, **cfg)


def algo(a, op, count, dtype=A.DataType.float32):
    """what the planner picks for this call on this device (same on every rank)"""
    return A._C.cuda_plan_call(a.impl, op, count, dtype)


# counts (fp32): 1 elem, odd tiny, 1 KiB, LL one-hop limit, two-hop LL, LL/staged crossover, staged, odd staged
SIZES = [1, 7, 256, 8192, 8192 + 1, 12288, 16384, 65536, 65536 - 1, 262144, 262144 + 3, 786432, 1 << 20]


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("func", [SUM, MAX])
def test_allreduce_sizes(world, func):
    seen = set()

    def fn(a, r, w):
        for n in SIZES:
            s, d = a.create_buffer(n), a.create_buffer(n)
            s.dev.copy_(data(n, r, salt=n).cuda(a.cuda_device))
            d.dev.zero_()
            a.allreduce(s, d, n, func, from_fpga=True, to_fpga=True)
            torch.cuda.current_stream().synchronize()
            assert close(d.dev, ref_reduce(w, n, func, salt=n), 1e-5, 1e-4), f"allreduce n={n} rank {r}"
            if r == 0:
                p = algo(a, A._C.Operation.allreduce, n)
                seen.add((p["algo"], p["oneshot"]))
    run(world, fn)
    assert ("ll", True) in seen and ("staged", False) in seen, seen
    if world >= 3:
        assert ("ll", False) in seen, seen  # 48 KiB: shards of <= 16 KiB go through the forwarding LL exchange


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64, torch.int32, torch.int64])
def test_allreduce_dtypes(dtype):
    def fn(a, r, w):
        for n in (5, 1000, 16384, 200000):
            s, d = a.create_buffer(n, dtype), a.create_buffer(n, dtype)
            s.host[:] = data(n, r, dtype)
            a.allreduce(s, d, n, SUM)
            tol = {torch.float16: 2e-2, torch.bfloat16: 1e-1}.get(dtype, 1e-9)
            assert close(d.host, ref_reduce(w, n, SUM, dtype), tol, tol), (dtype, n)
    run(3, fn)


def test_allreduce_in_place_and_repeated():
    # the same buffers over and over: staging parity reuse, credits, and no rank may run ahead into a buffer
    # that a peer has not consumed yet
    def fn(a, r, w):
        for n in (64, 8192, 65536, 1 << 19):
            b = a.create_buffer(n)
            for it in range(12):
                b.dev.copy_(data(n, r, salt=it).cuda(a.cuda_device))
                a.allreduce(b, b, n, SUM, from_fpga=True, to_fpga=True, run_async=True).free()
                torch.cuda.current_stream().synchronize()
                assert close(b.dev, ref_reduce(w, n, SUM, salt=it), 1e-5, 1e-4), (n, it)
    run(4, fn)


@pytest.mark.parametrize("world", [2, 4])
def test_allgather_reduce_scatter_alltoall(world):
    def fn(a, r, w):
        for n in (3, 512, 4096, 4096 + 1, 40000, 200000):
            s, d = a.create_buffer(n * w), a.create_buffer(n)
            s.host[:] = data(n * w, r, salt=n)
            a.reduce_scatter(s, d, n, SUM)
            assert close(d.host, ref_reduce(w, n * w, SUM, salt=n)[r * n:(r + 1) * n], 1e-5, 1e-4), ("rs", n)
            g = a.create_buffer(n * w)
            a.allgather(d, g, n)
            assert close(g.host, ref_reduce(w, n * w, SUM, salt=n), 1e-5, 1e-4), ("ag", n)
            t = a.create_buffer(n * w)
            a.alltoall(s, t, n)
            ref = torch.cat([data(n * w, q, salt=n)[r * n:(r + 1) * n] for q in range(w)])
            assert torch.equal(t.host, ref), ("a2a", n)
    run(world, fn)


@pytest.mark.parametrize("world", [2, 3])
def test_rooted_from_every_root(world):
    def fn(a, r, w):
        for n in (9, 2048, 30000):
            for root in range(w):
                b = a.create_buffer(n)
                if r == root:
                    b.host[:] = data(n, root, salt=root)
                a.bcast(b, n, root)
                assert torch.equal(b.host, data(n, root, salt=root)), ("bcast", n, root)
                send, recv = a.create_buffer(n * w), a.create_buffer(n)
                full = data(n * w, root, salt=7)
                if r == root:
                    send.host[:] = full
                a.scatter(send, recv, n, root)
                assert torch.equal(recv.host, full[r * n:(r + 1) * n]), ("scatter", n, root)
                out = a.create_buffer(n * w)
                a.gather(recv, out, n, root)
                if r == root:
                    assert torch.equal(out.host, full), ("gather", n, root)
                s, d = a.create_buffer(n), a.create_buffer(n)
                s.host[:] = data(n, r, salt=root)
                a.reduce(s, d, n, root, MAX)
                if r == root:
                    assert close(d.host, ref_reduce(w, n, MAX, salt=root), 0, 0), ("reduce", n, root)
    run(world, fn)


def test_mixed_sequence_on_one_communicator():
    # different operations, sizes and protocols back to back on the same message streams
    def fn(a, r, w):
        bufs = {n: (a.create_buffer(n * w), a.create_buffer(n * w)) for n in (100, 5000, 70000)}
        for it in range(6):
            for n, (s, d) in bufs.items():
                s.dev.copy_(data(n * w, r, salt=it).cuda(a.cuda_device))
                kw = dict(from_fpga=True, to_fpga=True)
                a.allreduce(s, d, n, SUM, **kw)
                torch.cuda.current_stream().synchronize()
                assert close(d.dev[:n], ref_reduce(w, n * w, SUM, salt=it)[:n], 1e-5, 1e-4)
                a.allgather(s, d, n, **kw)
                torch.cuda.current_stream().synchronize()
                assert torch.equal(d.dev.cpu(), torch.cat([data(n * w, q, salt=it)[:n] for q in range(w)]))
                a.bcast(s, n, it % w, **kw)
                torch.cuda.current_stream().synchronize()
                assert torch.equal(s.dev[:n].cpu(), data(n * w, it % w, salt=it)[:n])
            a.barrier()
    run(3, fn)


def test_subcommunicators_use_their_own_state():
    # two overlapping groups: the world and {0, 2}; calls interleave on the same ranks
    def fn(a, r, w):
        ranks = A.Accl.generate_ranks(w)
        group = [0, 2]
        comm = a.create_communicator([ranks[g] for g in group], group.index(r)) if r in group else None
        for n in (33, 9000, 100000):
            s, d = a.create_buffer(n), a.create_buffer(n)
            s.host[:] = data(n, r, salt=n)
            a.allreduce(s, d, n, SUM)
            assert close(d.host, ref_reduce(w, n, SUM, salt=n), 1e-5, 1e-4)
            if comm is not None:
                a.allreduce(s, d, n, SUM, comm_id=comm)
                ref = data(n, 0, salt=n).double() + data(n, 2, salt=n).double()
                assert close(d.host, ref, 1e-5, 1e-4)
        a.barrier()
    run(3, fn)


def test_two_streams_two_communicators_in_flight():
    # reference multicomm test (test.cpp:756-832): calls on two overlapping communicators, here issued on two
    # CUDA streams of the same rank without waiting in between — each communicator has its own bank of state
    def fn(a, r, w):
        ranks = A.Accl.generate_ranks(w)
        group = [0, 1]
        comm = a.create_communicator([ranks[g] for g in group], group.index(r)) if r in group else None
        n1, n2 = 300000, 50000
        s1, d1 = a.create_buffer(n1), a.create_buffer(n1)
        s2, d2 = a.create_buffer(n2), a.create_buffer(n2)
        s1.dev.copy_(data(n1, r).cuda(a.cuda_device))
        s2.dev.copy_(data(n2, r, salt=5).cuda(a.cuda_device))
        torch.cuda.current_stream().synchronize()
        st1, st2 = torch.cuda.Stream(a.cuda_device), torch.cuda.Stream(a.cuda_device)
        reqs = []
        for it in range(8):
            with torch.cuda.stream(st1):
                reqs.append(a.allreduce(s1, d1, n1, SUM, from_fpga=True, to_fpga=True, run_async=True))
            if comm is not None:
                with torch.cuda.stream(st2):
                    reqs.append(a.allreduce(s2, d2, n2, SUM, comm_id=comm, from_fpga=True, to_fpga=True, run_async=True))
        for q in reqs:
            q.wait()
            assert q.retcode() == 0
        st1.synchronize()
        st2.synchronize()
        assert close(d1.dev, ref_reduce(w, n1, SUM), 1e-5, 1e-4)
        if comm is not None:
            ref = data(n2, 0, salt=5).double() + data(n2, 1, salt=5).double()
            assert close(d2.dev, ref, 1e-5, 1e-4)
        a.barrier()
    # rendezvous sized on the world communicator, one-way sized on the pair
    A.run_cuda_ranks(devices(3), fn, dict(n_egr_rx_bufs=4, egr_rx_buf_size=16 << 10, max_egr_size=256 << 10, max_rndzv_size=1 << 30),
                     heap_mb=256, max_ctas=8)


def test_cuda_graph_replay_of_small_allreduces():
    # launch-bound inner loops belong in a CUDA graph: calls are capturable (no host-visible completion record)
    def fn(a, r, w):
        n = 2048
        s, d = a.create_buffer(n), a.create_buffer(n)
        s.dev.copy_(data(n, r).cuda(a.cuda_device))
        st = torch.cuda.Stream(a.cuda_device)
        with torch.cuda.stream(st):
            a.allreduce(s, d, n, SUM, from_fpga=True, to_fpga=True, run_async=True).free()  # warm-up outside the graph
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            # (ranks are threads of one process here: only this thread's calls belong to the capture)
            with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
                for _ in range(10):
                    a.allreduce(s, d, n, SUM, from_fpga=True, to_fpga=True, run_async=True).free()
            for _ in range(3):
                g.replay()
            st.synchronize()
        assert close(d.dev, ref_reduce(w, n, SUM), 1e-5, 1e-4)
        a.barrier()
    run(2, fn)


# ------------------------------------------------------------------------------------------------------------------
# wire-compressed collectives at bandwidth (ALGO_WIRE, csrc/src/cuda/compress.cuh): operands keep their dtype, the
# NVLink traffic is fp16 / bf16 / block-scaled fp8.  Tolerances as the reference's compressed tests
# (test/host/xrt/src/test.cpp:22-27: rtol 5e-3 / atol 5e-2 for fp16), wider for fp8.
WIRE = dict(n_egr_rx_bufs=4, egr_rx_buf_size=16 << 10, max_egr_size=64 << 10, max_rndzv_size=1 << 30)
WIRE_TOL = {torch.float16: dict(rtol=5e-3, atol=5e-2), torch.bfloat16: dict(rtol=2e-2, atol=1e-1),
            "float8_e4m3": dict(rtol=0.13, atol=0.8)}


@pytest.mark.parametrize("wire", [torch.float16, torch.bfloat16, "float8_e4m3"])
@pytest.mark.parametrize("world", [2, 3])
def test_wire_compressed_collectives(wire, world):
    def fn(a, r, w):
        tol = WIRE_TOL[wire]
        for n in (100000, 100003, 1 << 20):
            s, d = a.create_buffer(n), a.create_buffer(n)
            s.dev.copy_(data(n, r, salt=n).cuda(a.cuda_device))
            for func in (SUM, MAX):
                d.dev.zero_()
                a.allreduce(s, d, n, func, compress_dtype=wire, from_fpga=True, to_fpga=True)
                torch.cuda.current_stream().synchronize()
                assert close(d.dev, ref_reduce(w, n, func, salt=n), **tol), ("allreduce", wire, n, func)
            per = n // w
            rs = a.create_buffer(per)
            a.reduce_scatter(s, rs, per, SUM, compress_dtype=wire, from_fpga=True, to_fpga=True)
            torch.cuda.current_stream().synchronize()
            assert close(rs.dev, ref_reduce(w, n, SUM, salt=n)[r * per:(r + 1) * per], **tol), ("reduce_scatter", wire, n)
            g = a.create_buffer(per * w)
            a.allgather(rs, g, per, compress_dtype=wire, from_fpga=True, to_fpga=True)
            torch.cuda.current_stream().synchronize()
            assert close(g.dev, ref_reduce(w, n, SUM, salt=n)[:per * w], rtol=2 * tol["rtol"], atol=2 * tol["atol"]), ("allgather", wire, n)
            # in place, twice in a row (scratch halves are reused without a trailing meeting)
            for it in range(2):
                s.dev.copy_(data(n, r, salt=n + it).cuda(a.cuda_device))
                a.allreduce(s, s, n, SUM, compress_dtype=wire, from_fpga=True, to_fpga=True)
                torch.cuda.current_stream().synchronize()
                assert close(s.dev, ref_reduce(w, n, SUM, salt=n + it), **tol), ("in place", wire, n, it)
    A.run_cuda_ranks(devices(world), fn, WIRE, heap_mb=256, max_ctas=16)

