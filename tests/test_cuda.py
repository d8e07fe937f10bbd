"""GPU tests of the CUDA backend (run on a B200 box: `pytest -m gpu`).

Ranks are threads of this process.  With >= 2 GPUs each rank drives its own
GPU over NVLink (NVLS paths included); with a single GPU the ranks share it
(peer pointers alias the same device, no multicast) so protocol logic, flags
and every kernel body still execute.  Numerics are compared against plain
PyTorch fp32/fp64 references of the same op.  Matrix follows the reference's
suite (test/host/xrt/src/test.cpp) like tests/test_emulator.py.
"""
import pytest
import torch

import accl_b200 as A
from accl_b200 import MAX, SUM

pytestmark = pytest.mark.gpu

NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0
EAGER = dict(n_egr_rx_bufs=4, egr_rx_buf_size=16 << 10, max_egr_size=64 << 10, max_rndzv_size=1 << 30)
RNDZV = dict(n_egr_rx_bufs=4, egr_rx_buf_size=1024, max_egr_size=1024, max_rndzv_size=1 << 30)
PROTOCOLS = [pytest.param(EAGER, id="eager"), pytest.param(RNDZV, id="rndzv")]
COUNT = 5000  # 20 KB fp32: eager in EAGER (segmented: slot is 16 KB), rendezvous in RNDZV; not vector aligned per rank


def devices(world):
    return [r % max(NGPU, 1) for r in range(world)]


def worlds():
    return sorted({2, min(4, max(2, NGPU)), 3})


def data(count, rank, dtype=torch.float32, salt=0):
    g = torch.Generator().manual_seed(4321 + 31 * rank + salt)
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


def run(world, fn, cfg=EAGER, **kw):
    return A.run_cuda_ranks(devices(world), fn, cfg, heap_mb=64, max_ctas=4, **kw)


def run_shared_gpu(world, fn, cfg=EAGER, **kw):
    """All ranks on cuda:0 (a supported deployment: ranks sharing a GPU talk through the same heap windows)."""
    return A.run_cuda_ranks([0] * world, fn, cfg, heap_mb=64, max_ctas=4, **kw)


def test_probe_and_describe():
    def fn(a, r, w):
        return a.describe()
    out = run(2, fn)
    assert "CudaDevice rank 0/2" in out[0]
    print(out, A._C.cuda_probe(0))


def test_copy_combine_nop():
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
        s.host[:] = data(COUNT, 0)
        a.copy(s, d, COUNT)
        assert torch.equal(s.host, d.host)
        x, y, z = a.create_buffer(COUNT), a.create_buffer(COUNT), a.create_buffer(COUNT)
        x.host[:] = data(COUNT, 1)
        y.host[:] = data(COUNT, 2)
        a.combine(COUNT, SUM, x, y, z)
        assert close(z.host, x.host + y.host)
        a.combine(COUNT, MAX, x, y, z)
        assert torch.equal(z.host, torch.maximum(x.host, y.host))
        req = a.nop()
        assert req.retcode() == 0 and req.duration_ns() < 5_000_000
        h = a.create_buffer(COUNT, torch.float16)
        a.copy(s, h, COUNT)  # mixed dtype copy = cast lane
        assert close(h.host, s.host.half(), 0, 0)
    run(1, fn)


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_sendrecv(cfg):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
        s.host[:] = data(COUNT, r)
        nxt, prv = (r + 1) % w, (r - 1) % w
        if r % 2 == 0:
            a.send(s, COUNT, nxt, tag=5)
            a.recv(d, COUNT, prv, tag=5)
        else:
            a.recv(d, COUNT, prv, tag=5)
            a.send(s, COUNT, nxt, tag=5)
        assert torch.equal(d.host, data(COUNT, prv))
    run(2, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", worlds())
@pytest.mark.parametrize("func", [SUM, MAX])
def test_allreduce(cfg, world, func):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
        s.host[:] = data(COUNT, r)
        a.allreduce(s, d, COUNT, func)
        assert close(d.host, ref_reduce(w, COUNT, func), 1e-5, 1e-5)
    run(world, fn, cfg)


@pytest.mark.parametrize("count", [1, 7, 1 << 18, (1 << 20) + 3])
def test_allreduce_sizes_twoshot(count):
    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        a.allreduce(s, d, count, SUM)
        assert close(d.host, ref_reduce(w, count, SUM), 1e-5, 1e-4)
    run(2, fn, RNDZV, oneshot_kb=64)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64, torch.int32, torch.int64])
@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_allreduce_dtypes(dtype, cfg):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT, dtype), a.create_buffer(COUNT, dtype)
        s.host[:] = data(COUNT, r, dtype)
        a.allreduce(s, d, COUNT, SUM)
        tol = {torch.float16: 2e-2, torch.bfloat16: 1e-1}.get(dtype, 1e-9)
        assert close(d.host, ref_reduce(w, COUNT, SUM, dtype), tol, tol)
    run(2, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", worlds())
def test_reduce_scatter_allgather(cfg, world):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT * w), a.create_buffer(COUNT)
        s.host[:] = data(COUNT * w, r)
        a.reduce_scatter(s, d, COUNT, SUM)
        assert close(d.host, ref_reduce(w, COUNT * w, SUM)[r * COUNT:(r + 1) * COUNT], 1e-5, 1e-5)
        g = a.create_buffer(COUNT * w)
        a.allgather(d, g, COUNT)
        assert close(g.host, ref_reduce(w, COUNT * w, SUM), 1e-5, 1e-5)
    run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("world", worlds())
def test_rooted_collectives(cfg, world):
    def fn(a, r, w):
        for root in range(w):
            b = a.create_buffer(COUNT)
            if r == root:
                b.host[:] = data(COUNT, root, salt=root)
            a.bcast(b, COUNT, root)
            assert torch.equal(b.host, data(COUNT, root, salt=root))
            send, recv = a.create_buffer(COUNT * w), a.create_buffer(COUNT)
            full = data(COUNT * w, root, salt=7)
            if r == root:
                send.host[:] = full
            a.scatter(send, recv, COUNT, root)
            assert torch.equal(recv.host, full[r * COUNT:(r + 1) * COUNT])
            out = a.create_buffer(COUNT * w)
            a.gather(recv, out, COUNT, root)
            if r == root:
                assert torch.equal(out.host, full)
            s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
            s.host[:] = data(COUNT, r, salt=root)
            a.reduce(s, d, COUNT, root, SUM)
            if r == root:
                assert close(d.host, ref_reduce(w, COUNT, SUM, salt=root), 1e-5, 1e-5)
    run(world, fn, cfg)


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_alltoall_barrier(cfg):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT * w), a.create_buffer(COUNT * w)
        s.host[:] = data(COUNT * w, r)
        a.alltoall(s, d, COUNT)
        ref = torch.cat([data(COUNT * w, q)[r * COUNT:(r + 1) * COUNT] for q in range(w)])
        assert torch.equal(d.host, ref)
        a.barrier()
    run(3, fn, cfg)


@pytest.mark.parametrize("wire", [torch.float16, torch.bfloat16, "float8_e4m3"])
def test_allreduce_compressed_wire(wire):
    def fn(a, r, w):
        s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
        s.host[:] = data(COUNT, r)
        a.allreduce(s, d, COUNT, SUM, compress_dtype=wire)
        tol = dict(rtol=5e-3, atol=5e-2) if wire != "float8_e4m3" else dict(rtol=0.1, atol=0.6)
        assert close(d.host, ref_reduce(w, COUNT, SUM), **tol)
        b = a.create_buffer(COUNT)
        if r == 0:
            b.host[:] = data(COUNT, 0)
        a.bcast(b, COUNT, 0, compress_dtype=wire)
        assert close(b.host, data(COUNT, 0), **tol)
    run(2, fn, EAGER)


def test_device_resident_tensors_and_streams():
    # zero-copy: operands are torch tensors aliasing the symmetric heap, calls are stream ordered
    def fn(a, r, w):
        n = 1 << 16
        s, d = a.create_buffer(n), a.create_buffer(n)
        x = s.dev
        x.copy_(data(n, r).cuda(a.cuda_device))
        x.mul_(2.0)                       # producer kernel on the torch stream
        req = a.allreduce(s, d, n, SUM, from_fpga=True, to_fpga=True, run_async=True)
        y = d.dev * 0.5                   # consumer kernel, ordered after the collective
        req.wait()
        assert close(y, ref_reduce(w, n, SUM), 1e-5, 1e-4)
        assert req.duration_ns() > 0
    run(2, fn, RNDZV)


def test_subcommunicator():
    def fn(a, r, w):
        ranks = A.Accl.generate_ranks(w)
        group = [0, 2]
        if r in group:
            comm = a.create_communicator([ranks[g] for g in group], group.index(r))
            s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
            s.host[:] = data(COUNT, r)
            a.allreduce(s, d, COUNT, SUM, comm_id=comm)
            ref = data(COUNT, 0).double() + data(COUNT, 2).double()
            assert close(d.host, ref, 1e-5, 1e-5)
        a.barrier()
    run(3, fn, RNDZV)


def test_host_only_buffers_are_staged():
    def fn(a, r, w):
        s, d = a.create_buffer_host(COUNT), a.create_buffer_host(COUNT)
        s.host[:] = data(COUNT, r)
        a.allreduce(s, d, COUNT, SUM)
        assert close(d.host, ref_reduce(w, COUNT, SUM), 1e-5, 1e-5)
    run(2, fn, RNDZV)


@pytest.mark.multigpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_nvls_paths_when_available(dtype):
    # force the in-switch algorithms even at 2 ranks
    n = 1 << 20

    def fn(a, r, w):
        s, d = a.create_buffer(n, dtype), a.create_buffer(n, dtype)
        s.host[:] = data(n, r, dtype)
        a.allreduce(s, d, n, SUM)
        tol = 1e-4 if dtype == torch.float32 else 1e-1
        assert close(d.host, ref_reduce(w, n, SUM, dtype), tol, tol)
        g = a.create_buffer(n * w, dtype)
        a.allgather(s, g, n)
        assert torch.equal(g.host, torch.cat([data(n, q, dtype) for q in range(w)]))
        rs = a.create_buffer(n // w, dtype)
        a.reduce_scatter(s, rs, n // w, SUM)
        assert close(rs.host, ref_reduce(w, n, SUM, dtype)[r * (n // w):(r + 1) * (n // w)], tol, tol)
        return a.describe()
    out = A.run_cuda_ranks(list(range(min(NGPU, 4))), fn, RNDZV, heap_mb=128, max_ctas=8, nvls_min_ranks=2, oneshot_kb=0, nvls_ops=0xFFFF)
    print(out[0])


def test_host_resident_allreduce_is_pipelined_and_correct():
    n = 12 << 20  # 48 MiB fp32: above the 2 x 16 MiB pipelining threshold, not a multiple of the chunk

    def fn(a, r, w):
        s, d = a.create_buffer(n + 5), a.create_buffer(n + 5)
        s.host[:] = float(r + 1)
        s.host[-1] = 7.0
        a.allreduce(s, d, n + 5, SUM)   # host-resident operands, blocking: H2D / collective / D2H overlap per chunk
        assert float(d.host[0]) == sum(range(1, w + 1)) and float(d.host[n]) == sum(range(1, w + 1))
        assert float(d.host[-1]) == 7.0 * w
    A.run_cuda_ranks(devices(2), fn, RNDZV, heap_mb=256, max_ctas=8)


def test_stream_operands_and_stream_put():
    # the device-side stream port is a FIFO in the heap; results pushed with RES_STREAM are what
    # OP0_STREAM consumers pop (the reference's emulator runs the same tests with kernel loopback)
    from accl_b200 import DataType
    n = 3000

    def fn(a, r, w):
        s, d = a.create_buffer(n), a.create_buffer(n)
        s.host[:] = data(n, r)
        a.copy_to_stream(s, n)
        a.copy_from_stream(d, n)
        assert torch.equal(s.host, d.host)
        a.copy_to_stream(s, n)
        a.copy_from_to_stream(DataType.float32, n)
        a.copy_from_stream(d, n)
        assert torch.equal(s.host, d.host)
        nxt, prv = (r + 1) % w, (r - 1) % w
        # memory -> network -> stream -> memory
        req = a.send(s, n, nxt, tag=9, run_async=True)
        a.recv_to_stream(DataType.float32, n, prv, tag=9)
        req.wait()
        a.copy_from_stream(d, n)
        assert torch.equal(d.host, data(n, prv))
        # memory -> stream -> network -> memory
        a.copy_to_stream(s, n)
        req = a.send_from_stream(DataType.float32, n, nxt, tag=11, run_async=True)
        a.recv(d, n, prv, tag=11)
        req.wait()
        assert torch.equal(d.host, data(n, prv))
        # one-sided put into the peer's stream, no matching recv
        a.barrier()
        a.stream_put(s, n, nxt, 9)
        a.copy_from_stream(d, n)
        assert torch.equal(d.host, data(n, prv))
        # reduce: stream -> memory and memory -> stream
        a.copy_to_stream(s, n)
        a.reduce_stream2mem(DataType.float32, d, n, 0, SUM)
        if r == 0:
            assert close(d.host, ref_reduce(w, n, SUM), 1e-5, 1e-5)
        a.reduce_mem2stream(s, DataType.float32, n, 0, SUM)
        if r == 0:
            a.copy_from_stream(d, n)
            assert close(d.host, ref_reduce(w, n, SUM), 1e-5, 1e-5)
    run(2, fn, EAGER)


def test_large_reduce_is_distributed_over_workers():
    n = (1 << 19) + 3   # > 1 MiB: the non-root ranks each reduce a slice and store it into the root

    def fn(a, r, w):
        for root in (0, w - 1):
            s, d = a.create_buffer(n), a.create_buffer(n)
            s.host[:] = data(n, r, salt=root)
            a.reduce(s, d, n, root, SUM)
            if r == root:
                assert close(d.host, ref_reduce(w, n, SUM, salt=root), 1e-5, 1e-4)
    run(3, fn, RNDZV)


@pytest.mark.parametrize("func", [SUM, MAX])
def test_large_reduce_12mib_chunked(func):
    """12 MiB + tail: the size class of the chunked rooted-reduce schemes — the distributed pull (default) and the
    write-only push through the scratch area (tuning knob reduce_push)."""
    n = (3 << 20) + 5

    def fn(a, r, w):
        for push in (0, 1):
            a.set_tuning("reduce_push", push)
            s, d = a.create_buffer(n), a.create_buffer(n)
            s.host[:] = data(n, r, salt=3 + push)
            a.reduce(s, d, n, 1, func)
            if r == 1:
                assert close(d.host, ref_reduce(w, n, func, salt=3 + push), 1e-5, 1e-4), push
    A.run_cuda_ranks(devices(3), fn, RNDZV, heap_mb=256, max_ctas=8)


@pytest.mark.multigpu
@pytest.mark.skipif(NGPU < 3, reason="pipelined NVLS broadcast needs >= 3 GPUs")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_large_bcast_and_reduce_through_the_switch(dtype):
    n = (6 << 20) + 8   # 24 MiB fp32: pipelined scatter + multimem.st broadcast; distributed NVLS reduce
    w_ = min(NGPU, 8)

    def fn(a, r, w):
        for root in (0, w - 1):
            b = a.create_buffer(n, dtype)
            if r == root:
                b.host[:] = data(n, root, dtype, salt=root)
            a.bcast(b, n, root)
            assert torch.equal(b.host, data(n, root, dtype, salt=root))
            s, d = a.create_buffer(n, dtype), a.create_buffer(n, dtype)
            s.host[:] = data(n, r, dtype, salt=root)
            a.reduce(s, d, n, root, SUM)
            if r == root:
                tol = 1e-4 if dtype == torch.float32 else 2e-1
                assert close(d.host, ref_reduce(w, n, SUM, dtype, salt=root), tol, tol)
    A.run_cuda_ranks(list(range(w_)), fn, RNDZV, heap_mb=512, max_ctas=16)


@pytest.mark.parametrize("flags", [0, 1])
def test_large_bcast_is_pipelined_over_workers(flags):
    n = (33 << 20) + 4   # 132 MiB fp32 (>= 128 MiB): the root deals slices, the workers forward them
    # flags = 0: one meeting per chunk; flags = 1: one-way "chunk landed" counters (tuning knob bcast_flags)

    def fn(a, r, w):
        a.set_tuning("bcast_flags", flags)
        for root in (0, 1):
            b = a.create_buffer(n)
            if r == root:
                b.host[:] = data(n, root, salt=root)
            a.bcast(b, n, root)
            assert torch.equal(b.host, data(n, root, salt=root))
    A.run_cuda_ranks(devices(3), fn, RNDZV, heap_mb=768, max_ctas=8)


@pytest.mark.parametrize("cfg", PROTOCOLS)
def test_stress_sendrecv_ring(cfg):
    """2000 tagged exchanges around a ring without re-initialising (reference stress.cpp:24-33):
    slot credits, sequence numbers and sync pads must survive wrap-around of the small rings."""
    iters = 2000

    def fn(a, r, w):
        s, d = a.create_buffer(COUNT), a.create_buffer(COUNT)
        nxt, prv = (r + 1) % w, (r - 1) % w
        for i in range(iters):
            s.dev.fill_(float(r * 10000 + i))
            if r % 2 == 0:
                a.send(s, COUNT, nxt, tag=i & 0xFF, from_fpga=True)
                a.recv(d, COUNT, prv, tag=i & 0xFF, to_fpga=True)
            else:
                a.recv(d, COUNT, prv, tag=i & 0xFF, to_fpga=True)
                a.send(s, COUNT, nxt, tag=i & 0xFF, from_fpga=True)
            if i % 250 == 0 or i == iters - 1:
                torch.cuda.synchronize()
                assert float(d.dev[0]) == float(prv * 10000 + i) and float(d.dev[-1]) == float(prv * 10000 + i)
    run(2, fn, cfg)


@pytest.mark.parametrize("count", [(128 << 10) // 4, (256 << 10) // 4 + 3, (1 << 20) // 4])
def test_allreduce_in_place_rendezvous_oneshot_sizes(count):
    """In-place all-reduce in the size class of the rendezvous one-shot (everybody pulls everything): a peer must
    never read a source that its owner has already overwritten with the result — the kernel takes the two-shot
    body when any rank runs in place."""
    def fn(a, r, w):
        b = a.create_buffer(count)
        for it in range(4):
            b.dev.copy_(data(count, r, salt=it).cuda(a.cuda_device))
            a.allreduce(b, b, count, SUM, from_fpga=True, to_fpga=True)
            torch.cuda.current_stream().synchronize()
            assert close(b.dev, ref_reduce(w, count, SUM, salt=it), 1e-5, 1e-4), it
    A.run_cuda_ranks(devices(3), fn, RNDZV, heap_mb=64, max_ctas=8)


@pytest.mark.parametrize("cfg", PROTOCOLS)
@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_sendrecv_segmentation(cfg, k, delta):
    """count = k * segment + {-1, 0, 1} (reference ACCLSegmentationTest, test/host/xrt/src/test.cpp:345-393, 1154-1159):
    the eager path cuts messages at the RX-buffer size, rendezvous moves them whole."""
    seg = (16 << 10) // 4 if cfg is EAGER else 1024 // 4   # elements per eager segment of the configuration
    count = k * seg + delta

    def fn(a, r, w):
        s, d = a.create_buffer(count), a.create_buffer(count)
        s.host[:] = data(count, r)
        nxt, prv = (r + 1) % w, (r - 1) % w
        if r % 2 == 0:
            a.send(s, count, nxt, tag=3)
            a.recv(d, count, prv, tag=3)
        else:
            a.recv(d, count, prv, tag=3)
            a.send(s, count, nxt, tag=3)
        assert torch.equal(d.host, data(count, prv))
        # and through a collective of the same size
        out = a.create_buffer(count)
        a.allreduce(s, out, count, SUM)
        assert close(out.host, ref_reduce(w, count, SUM), 1e-5, 1e-5)
    run(2, fn, cfg)


def test_stream_ids_do_not_interleave():
    """With the loop-back off, stream id s is served by its own FIFO (reference: ids 9..246 travel as TDEST,
    dma_mover.cpp:312,644): two stream_puts with different ids can be drained in either order, and the vadd_put
    user kernel (data.push while computing, then the consumer's data.pull) lands in the id it names."""
    from accl_b200.ops import stream_pull, vadd_put
    n = 5000

    def fn(a, r, w):
        a.set_tuning("stream_loopback", 0)
        nxt, prv = (r + 1) % w, (r - 1) % w
        s1, s2, d1, d2 = (a.create_buffer(n) for _ in range(4))
        s1.host[:] = data(n, r, salt=1)
        s2.host[:] = data(n, r, salt=2)
        a.stream_put(s1, n, nxt, 9)
        a.stream_put(s2, n, nxt, 10)
        a.barrier()
        st2 = stream_pull(a, d2, n, stream_id=10)   # the later put first
        st1 = stream_pull(a, d1, n, stream_id=9)
        torch.cuda.current_stream().synchronize()
        assert int(st1.item()) == 0 and int(st2.item()) == 0
        assert torch.equal(d1.dev.cpu(), data(n, prv, salt=1)) and torch.equal(d2.dev.cpu(), data(n, prv, salt=2))
        # the reference's vadd_put example: x + 1 pushed into stream 11 of the next rank while computing
        s1.sync_to_device()
        st = vadd_put(a, s1, n, nxt, stream_id=11)
        sp = stream_pull(a, d1, n, stream_id=11)
        torch.cuda.current_stream().synchronize()
        assert int(st.item()) == 0 and int(sp.item()) == 0
        assert torch.equal(d1.dev.cpu(), data(n, prv, salt=1) + 1.0)
        a.barrier()
    run(2, fn, EAGER)


# run-time knob: (value set, value read back), in range and out of range
TUNING = {
    "hybrid_16ths": [(3, 3), (99, 15), (-1, 0)],
    "nvls_unroll": [(8, 8), (16, 16), (3, 4), (0, 4)],
    "reduce_push": [(2, 2), (3, 0), (-1, 0)],
    "bcast_flags": [(1, 1), (5, 0), (-2, 0)],
    "split_phases": [(1, 1), (7, 1), (0, 0)],
    "nvls_ctas": [(16, 16), (1 << 20, 1 << 20)],
    "nvls_min_ranks": [(2, 2), (99, 99)],
    "max_ctas": [(64, 64), (126, 126), (127, 126), (1000, 126), (0, 1), (-5, 1)],
    "ll_max_bytes": [(1 << 20, 1 << 20), (1 << 40, 1 << 40), (-1, -1)],
    "ll_oneshot_max": [(8 << 10, 8 << 10), (1 << 40, 1 << 40)],
    "oneshot_max_bytes": [(1 << 20, 1 << 20), (1 << 40, 1 << 40)],
    "wire_min_bytes": [(0, 0), (1 << 40, 1 << 40)],
    "staged_max_bytes": [(1 << 20, 1 << 20), (1 << 40, 1 << 40)],
    "stream_loopback": [(0, 0), (5, 1), (1, 1)],
}


def test_set_tuning_clamps_and_get_tuning_reads_back():
    """Every run-time knob takes an in-range value as it is and clamps (or stores) an out-of-range one; the options
    fixed at construction are refused by set_tuning and unknown to get_tuning; max_ctas=128 at construction stays 128."""
    def fn(a, r, w):
        assert a.get_tuning("max_ctas") == 128
        for name, pairs in TUNING.items():
            for value, want in pairs:
                a.set_tuning(name, value)
                assert a.get_tuning(name) == want, (name, value)
        for name in ("heap_mb", "multicast", "engine", "engine_workers", "engine_idle_us", "oneshot_kb", "nvls_ops",
                     "stage_kb", "ll_kb", "host_pipeline_chunk_kb", "stage_bytes", "ll_bytes", "no_such_knob"):
            with pytest.raises(ValueError):
                a.set_tuning(name, 1)
        for name in ("engine_workers", "stage_kb", "oneshot_kb", "no_such_knob"):
            assert a.get_tuning(name) == -1, name
        assert a.get_tuning("stage_bytes") > 0 and a.get_tuning("ll_bytes") > 0
    A.run_cuda_ranks([0], fn, EAGER, heap_mb=64, max_ctas=128)
