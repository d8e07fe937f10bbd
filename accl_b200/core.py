"""Python face of the library: `Accl` (one per rank) and `Buffer`.

Thin by design — every call lands in the C++ facade `accl::ACCL`
(csrc/include/accl/accl.hpp), which mirrors the reference API
(driver/xrt/include/accl.hpp).  What Python adds: torch/numpy views of buffer
memory, dtype mapping, stream plumbing (the current torch CUDA stream is
forwarded to the backend) and world construction helpers.
"""
import os
import threading

import numpy as np
import torch

from . import _C
from .utils.dtypes import to_accl, to_torch

DataType = _C.DataType
ReduceFunction = _C.ReduceFunction
BufferKind = _C.BufferKind
TAG_ANY = _C.TAG_ANY
GLOBAL_COMM = _C.GLOBAL_COMM
SUM = _C.ReduceFunction.SUM
MAX = _C.ReduceFunction.MAX


try:
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:  # pragma: no cover - older torch
    def _raw_stream(device):
        return torch.cuda.current_stream(device).cuda_stream


class _CudaView:
    """Minimal __cuda_array_interface__ carrier so torch can alias heap memory."""

    def __init__(self, ptr, nbytes, owner):
        self.__cuda_array_interface__ = {
            "shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None,
        }
        self._owner = owner


class Buffer:
    """A library buffer: `.host` is a torch tensor aliasing the host side,
    `.dev` (CUDA backend) a torch tensor aliasing the device side inside the
    symmetric NVLink heap (zero-copy operand for every collective)."""

    def __init__(self, impl, accl):
        self._b = impl
        self._accl = accl
        self._host = None
        self._dev = None

    @property
    def impl(self):
        return self._b

    @property
    def dtype(self):
        return self._b.dtype

    @property
    def length(self):
        return self._b.length

    @property
    def nbytes(self):
        return self._b.size

    @property
    def address(self):
        return self._b.address

    @property
    def host(self):
        if self._host is None:
            self._host = torch.frombuffer(self._b.host_view(), dtype=torch.uint8).view(to_torch(self._b.dtype))
        return self._host

    @property
    def numpy(self):
        return self.host.numpy() if self.host.dtype in (torch.float16, torch.float32, torch.float64, torch.int32,
                                                         torch.int64, torch.int8) else self.host.view(torch.uint8).numpy()

    @property
    def dev(self):
        if self._dev is None:
            ptr = self._b.device_ptr
            if not ptr:
                raise RuntimeError("buffer has no CUDA device pointer (emulator backend?)")
            idx = self._accl.cuda_device
            view = _CudaView(ptr, self._b.size, self)
            t = torch.as_tensor(view, device=torch.device("cuda", idx))
            self._dev = t.view(to_torch(self._b.dtype))
        return self._dev

    def sync_to_device(self):
        self._b.sync_to_device()

    def sync_from_device(self):
        self._b.sync_from_device()

    def slice(self, start, end):
        return Buffer(self._b.slice(start, end), self._accl)

    def __len__(self):
        return self._b.length


def _impl(buf):
    return buf._b if isinstance(buf, Buffer) else buf


class Accl:
    """One rank's handle.  Method names and argument order follow accl::ACCL."""

    def __init__(self, impl, rank, world, cuda_device=None):
        self._a = impl
        self.rank = rank
        self.world = world
        self.cuda_device = cuda_device
        self.initialized = False
        self._cuda = impl.device_type() == _C.DeviceType.cuda

    # ---- setup -----------------------------------------------------------
    @staticmethod
    def generate_ranks(world=None, base_port=5500, max_segment_size=1024, ips=None, config_file=None):
        """Rank table (reference: accl_network_utils::generate_ranks): from a list of IPs, from the reference's
        JSON rank file {"ips": [...]} (`config_file`), or `world` local ranks on 127.0.0.1."""
        if config_file is not None:
            return _C.generate_ranks_from_file(str(config_file), base_port, max_segment_size)
        if ips is None:
            ips = ["127.0.0.1"] * world
        return _C.generate_ranks(list(ips), base_port, max_segment_size)

    def initialize(self, ranks=None, local_rank=None, n_egr_rx_bufs=16, egr_rx_buf_size=1024, max_egr_size=1024,
                   max_rndzv_size=32 * 1024):
        if ranks is None:
            ranks = self.generate_ranks(self.world, max_segment_size=egr_rx_buf_size)
        self._a.initialize(ranks, self.rank if local_rank is None else local_rank, n_egr_rx_bufs, egr_rx_buf_size,
                           max_egr_size, max_rndzv_size)
        self.initialized = True
        return self

    def deinit(self):
        self._a.deinit()
        self.initialized = False

    @property
    def impl(self):
        return self._a

    @property
    def is_cuda(self):
        return self._a.device_type() == _C.DeviceType.cuda

    def describe(self):
        return self._a.describe()

    # ---- buffers ---------------------------------------------------------
    def create_buffer(self, length, dtype=DataType.float32, kind=BufferKind.device):
        return Buffer(self._a.create_buffer(int(length), to_accl(dtype), kind), self)

    def create_buffer_host(self, length, dtype=DataType.float32):
        return self.create_buffer(length, dtype, BufferKind.host_only)

    def create_buffer_p2p(self, length, dtype=DataType.float32):
        return self.create_buffer(length, dtype, BufferKind.p2p)

    # -- zero-copy operands for torch tensors (CUDA backend) -----------------
    def heap_contains(self, t) -> bool:
        """True when the CUDA tensor `t` lives inside this rank's symmetric heap (a `Buffer.dev` view, or a tensor
        allocated from `heap_mem_pool()`)."""
        if not (self.is_cuda and isinstance(t, torch.Tensor) and t.is_cuda and t.numel()):
            return False
        rng = getattr(self, "_heap_range", None)
        if rng is None:
            rng = self._heap_range = _C.cuda_heap_range(self._a)   # fixed for the life of the backend
        base, size = rng
        p = t.data_ptr()
        return base <= p and p + t.numel() * t.element_size() <= base + size

    def wrap_device(self, t: "torch.Tensor") -> "Buffer":
        """A Buffer over a contiguous CUDA tensor that already lives in the heap: zero-copy operand, nothing is
        allocated.  The tensor must stay alive while calls on the buffer are in flight."""
        assert t.is_contiguous(), "wrap_device needs a contiguous tensor"
        b = Buffer(_C.cuda_wrap_device(self._a, t.data_ptr(), t.numel(), to_accl(t.dtype)), self)
        b._dev = t.view(-1)
        return b

    def heap_mem_pool(self):
        """A `torch.cuda.MemPool` whose allocations come from the symmetric heap:

            pool = accl.heap_mem_pool()
            with torch.cuda.use_mem_pool(pool):
                ddp = DistributedDataParallel(model, ...)      # gradient buckets land in the heap
                x = torch.empty(n, device="cuda")               # so does this

        Tensors allocated this way are zero-copy operands of every collective (`TensorGroup` / the "accl"
        torch.distributed backend recognise them).  Every rank must allocate in the same order."""
        if getattr(self, "_mem_pool", None) is None:
            _C.cuda_heap_pool_attach(self._a)
            alloc = torch.cuda.memory.CUDAPluggableAllocator(_C.__file__, "accl_heap_pool_alloc", "accl_heap_pool_free")
            self._pool_allocator = alloc
            self._mem_pool = torch.cuda.MemPool(alloc.allocator())
        return self._mem_pool

    def wrap(self, array):
        """Wrap caller-owned host memory (numpy array or CPU torch tensor)."""
        if isinstance(array, torch.Tensor):
            assert array.device.type == "cpu" and array.is_contiguous()
            b = self._a.wrap_buffer(array.data_ptr(), array.numel(), to_accl(array.dtype))
        else:
            array = np.ascontiguousarray(array)
            b = self._a.wrap_buffer(array.ctypes.data, array.size, to_accl(array.dtype))
        buf = Buffer(b, self)
        buf._keep = array
        return buf

    # ---- call helpers ----------------------------------------------------
    def _stream(self):
        if self._cuda and self.cuda_device is not None:
            # raw handle of torch's current stream (no Stream object: this runs on every call)
            h = _raw_stream(self.cuda_device)
            # 0 is torch's legacy default stream: name it explicitly (cudaStreamLegacy)
            # so calls stay ordered with tensor ops issued on it
            self._a.set_stream(h if h else 1)

    def _cd(self, compress_dtype):
        return DataType.none if compress_dtype is None else to_accl(compress_dtype)

    # ---- primitives ------------------------------------------------------
    def nop(self, run_async=False):
        self._stream()
        return self._a.nop(run_async)

    def send(self, srcbuf, count, dst, tag=TAG_ANY, comm_id=GLOBAL_COMM, from_fpga=False, compress_dtype=None,
             run_async=False):
        self._stream()
        return self._a.send(_impl(srcbuf), count, dst, tag, comm_id, from_fpga, self._cd(compress_dtype), run_async)

    def send_from_stream(self, dtype, count, dst, tag=TAG_ANY, comm_id=GLOBAL_COMM, compress_dtype=None,
                         run_async=False):
        return self._a.send_from_stream(to_accl(dtype), count, dst, tag, comm_id, self._cd(compress_dtype), run_async)

    def stream_put(self, srcbuf, count, dst, stream_id, comm_id=GLOBAL_COMM, from_fpga=False, compress_dtype=None,
                   run_async=False):
        self._stream()
        return self._a.stream_put(_impl(srcbuf), count, dst, stream_id, comm_id, from_fpga, self._cd(compress_dtype),
                                  run_async)

    def recv(self, dstbuf, count, src, tag=TAG_ANY, comm_id=GLOBAL_COMM, to_fpga=False, compress_dtype=None,
             run_async=False):
        self._stream()
        return self._a.recv(_impl(dstbuf), count, src, tag, comm_id, to_fpga, self._cd(compress_dtype), run_async)

    def recv_to_stream(self, dtype, count, src, tag=TAG_ANY, comm_id=GLOBAL_COMM, compress_dtype=None,
                       run_async=False):
        return self._a.recv_to_stream(to_accl(dtype), count, src, tag, comm_id, self._cd(compress_dtype), run_async)

    def copy(self, srcbuf, dstbuf, count, from_fpga=False, to_fpga=False, run_async=False):
        self._stream()
        return self._a.copy(_impl(srcbuf), _impl(dstbuf), count, from_fpga, to_fpga, run_async)

    def copy_from_stream(self, dstbuf, count, to_fpga=False, run_async=False):
        return self._a.copy_from_stream(_impl(dstbuf), count, to_fpga, run_async)

    def copy_to_stream(self, srcbuf, count, from_fpga=False, run_async=False):
        return self._a.copy_to_stream(_impl(srcbuf), count, from_fpga, run_async)

    def copy_from_to_stream(self, dtype, count, run_async=False):
        return self._a.copy_from_to_stream(to_accl(dtype), count, run_async)

    def combine(self, count, function, val1, val2, result, val1_from_fpga=False, val2_from_fpga=False, to_fpga=False,
                run_async=False):
        self._stream()
        return self._a.combine(count, function, _impl(val1), _impl(val2), _impl(result), val1_from_fpga,
                               val2_from_fpga, to_fpga, run_async)

    # ---- collectives -----------------------------------------------------
    def bcast(self, buf, count, root, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False, compress_dtype=None,
              run_async=False):
        self._stream()
        return self._a.bcast(_impl(buf), count, root, comm_id, from_fpga, to_fpga, self._cd(compress_dtype), run_async)

    def scatter(self, sendbuf, recvbuf, count, root, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
                compress_dtype=None, run_async=False):
        self._stream()
        return self._a.scatter(_impl(sendbuf), _impl(recvbuf), count, root, comm_id, from_fpga, to_fpga,
                               self._cd(compress_dtype), run_async)

    def gather(self, sendbuf, recvbuf, count, root, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
               compress_dtype=None, run_async=False):
        self._stream()
        return self._a.gather(_impl(sendbuf), _impl(recvbuf), count, root, comm_id, from_fpga, to_fpga,
                              self._cd(compress_dtype), run_async)

    def allgather(self, sendbuf, recvbuf, count, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
                  compress_dtype=None, run_async=False):
        self._stream()
        return self._a.allgather(_impl(sendbuf), _impl(recvbuf), count, comm_id, from_fpga, to_fpga,
                                 self._cd(compress_dtype), run_async)

    def reduce(self, sendbuf, recvbuf, count, root, func=SUM, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
               compress_dtype=None, run_async=False):
        self._stream()
        return self._a.reduce(_impl(sendbuf), _impl(recvbuf), count, root, func, comm_id, from_fpga, to_fpga,
                              self._cd(compress_dtype), run_async)

    def reduce_stream2mem(self, src_dtype, recvbuf, count, root, func=SUM, comm_id=GLOBAL_COMM, to_fpga=False,
                          compress_dtype=None, run_async=False):
        return self._a.reduce_stream2mem(to_accl(src_dtype), _impl(recvbuf), count, root, func, comm_id, to_fpga,
                                         self._cd(compress_dtype), run_async)

    def reduce_mem2stream(self, sendbuf, dst_dtype, count, root, func=SUM, comm_id=GLOBAL_COMM, from_fpga=False,
                          compress_dtype=None, run_async=False):
        return self._a.reduce_mem2stream(_impl(sendbuf), to_accl(dst_dtype), count, root, func, comm_id, from_fpga,
                                         self._cd(compress_dtype), run_async)

    def reduce_stream2stream(self, src_dtype, dst_dtype, count, root, func=SUM, comm_id=GLOBAL_COMM,
                             compress_dtype=None, run_async=False):
        return self._a.reduce_stream2stream(to_accl(src_dtype), to_accl(dst_dtype), count, root, func, comm_id,
                                            self._cd(compress_dtype), run_async)

    def allreduce(self, sendbuf, recvbuf, count, func=SUM, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
                  compress_dtype=None, run_async=False):
        self._stream()
        return self._a.allreduce(_impl(sendbuf), _impl(recvbuf), count, func, comm_id, from_fpga, to_fpga,
                                 self._cd(compress_dtype), run_async)

    def reduce_scatter(self, sendbuf, recvbuf, count, func=SUM, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
                       compress_dtype=None, run_async=False):
        self._stream()
        return self._a.reduce_scatter(_impl(sendbuf), _impl(recvbuf), count, func, comm_id, from_fpga, to_fpga,
                                      self._cd(compress_dtype), run_async)

    def alltoall(self, sendbuf, recvbuf, count, comm_id=GLOBAL_COMM, from_fpga=False, to_fpga=False,
                 compress_dtype=None, run_async=False):
        self._stream()
        return self._a.alltoall(_impl(sendbuf), _impl(recvbuf), count, comm_id, from_fpga, to_fpga,
                                self._cd(compress_dtype), run_async)

    def barrier(self, comm_id=GLOBAL_COMM):
        self._stream()
        return self._a.barrier(comm_id)

    # ---- communicators / config / introspection --------------------------
    def create_communicator(self, ranks, local_rank):
        return self._a.create_communicator(ranks, local_rank)

    def get_comm_group(self, comm_id=GLOBAL_COMM):
        return self._a.get_comm_group(comm_id)

    def get_comm_rank(self, comm_id=GLOBAL_COMM):
        return self._a.get_comm_rank(comm_id)

    def set_timeout(self, value):
        self._a.set_timeout(value)

    def set_max_eager_msg_size(self, value):
        self._a.set_max_eager_msg_size(value)

    def set_max_rendezvous_msg_size(self, value):
        self._a.set_max_rendezvous_msg_size(value)

    def set_one_hop_schedules(self, on=True):
        """Emulator: execute the schedules of the B200 backend (one-hop all-gather / reduce-scatter / one-shot and
        two-shot all-reduce, flat rooted collectives) instead of the reference's rings and trees.  Same value on every rank."""
        self._a.set_one_hop_schedules(bool(on))

    def dump_communicator(self):
        return self._a.dump_communicator()

    def dump_exchange_memory(self):
        return self._a.dump_exchange_memory()

    def set_tuning(self, name, value):
        """CUDA backend: runtime knob (hybrid_16ths, nvls_unroll, nvls_ctas, reduce_push, bcast_flags, ll_max_bytes,
        ll_oneshot_max, max_ctas, stream_loopback ...); must be set identically on every rank."""
        _C.cuda_set_tuning(self._a, name, int(value))

    def get_tuning(self, name):
        return _C.cuda_get_tuning(self._a, name)

    def drain(self):
        """CUDA backend: wait until every call started so far has completed."""
        _C.cuda_drain(self._a)

    def cuda_debug_state(self):
        """CUDA backend: sync-pad / eager counters of this rank's control block.
        Safe to call from another thread while a call hangs."""
        return _C.cuda_debug_state(self._a)

    def dump_eager_rx_buffers(self, dump_data=False):
        return self._a.dump_eager_rx_buffers(dump_data)

    def __getattr__(self, name):  # anything not wrapped above goes straight to C++
        return getattr(self._a, name)


def _raise_rank_errors(errors, hung, timeout):
    """Report the most informative failure of a multi-rank run: a rank that timed out waiting for a peer is
    usually a consequence, the peer's own error (assertion, bad argument...) the cause — show that one first and list
    the others."""
    failed = [(r, e) for r, e in enumerate(errors) if e is not None]
    if failed:
        def secondary(item):
            return "TIMEOUT" in str(item[1][0]) or "NOT_READY" in str(item[1][0])
        primary = next((f for f in failed if not secondary(f)), failed[0])
        others = "".join(f"\n  also rank {r}: {type(e[0]).__name__}: {str(e[0]).splitlines()[0] if str(e[0]) else ''}"
                         for r, e in failed if r != primary[0])
        if hung:
            others += f"\n  ranks {hung} still running after {timeout}s"
        raise RuntimeError(f"rank {primary[0]} failed:\n{primary[1][1]}{others}") from primary[1][0]
    if hung:
        raise TimeoutError(f"ranks {hung} did not finish within {timeout}s")


def emulator_world(world_size, mem_mb=256):
    """N un-initialised ranks of an in-process CPU emulator (drive each from its own thread)."""
    return [Accl(a, r, world_size) for r, a in enumerate(_C.make_emu_world(world_size, mem_mb))]


def run_ranks(world_size, fn, init_kwargs=None, mem_mb=64, timeout=120.0):
    """Run fn(accl, rank, world) on every rank of a fresh emulator world, one
    thread per rank; re-raises the most informative failure (a peer's own error before the time-outs it caused).  The harness used by the CPU
    test-suite (the reference uses mpirun + one emulator process per rank)."""
    accls = emulator_world(world_size, mem_mb)
    errors = [None] * world_size
    results = [None] * world_size

    def body(r):
        try:
            accls[r].initialize(**(init_kwargs or {}))
            results[r] = fn(accls[r], r, world_size)
        except BaseException as e:  # noqa: BLE001 - reported to the caller
            import traceback
            errors[r] = (e, traceback.format_exc())

    threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(world_size)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    hung = [r for r, t in enumerate(threads) if t.is_alive()]
    _raise_rank_errors(errors, hung, timeout)
    for a in accls:
        a.deinit()
    return results


def socket_rank(rank=None, world_size=None, addr="127.0.0.1", base_port=None, mem_mb=256):
    """One emulator rank per process (torchrun / mpirun style), loopback TCP between ranks."""
    rank = int(os.environ.get("RANK", 0)) if rank is None else rank
    world_size = int(os.environ.get("WORLD_SIZE", 1)) if world_size is None else world_size
    if base_port is None:
        base_port = int(os.environ.get("ACCL_EMU_PORT", int(os.environ.get("MASTER_PORT", 29500)) + 100))
    return Accl(_C.make_emu_socket(rank, world_size, addr, base_port, mem_mb), rank, world_size)


def remote_rank(rank=None, world_size=None, addr="127.0.0.1", ctrl_port=None, connect_timeout_s=60):
    """Driver for a stand-alone engine process (`build/bin/cclo_emu`, see
    accl_b200.models.emulator.spawn_engines): the reference's SimDevice <-> cclo_emu split."""
    rank = int(os.environ.get("RANK", 0)) if rank is None else rank
    world_size = int(os.environ.get("WORLD_SIZE", 1)) if world_size is None else world_size
    if ctrl_port is None:
        ctrl_port = int(os.environ.get("ACCL_EMU_PORT", 5500)) + 1000 + rank
    return Accl(_C.make_emu_remote(rank, world_size, addr, ctrl_port, connect_timeout_s), rank, world_size)


# --------------------------------------------------------------------- CUDA
def _prepare_cuda_env():
    # ranks sharing one process/GPU need independent hardware queues, or one
    # rank's spinning kernel can block the launch of the peer it waits for
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    # Note: with CUDA's lazy module loading the FIRST launch of any kernel may synchronise the
    # context.  The library preloads its own kernels; if an application keeps the persistent
    # engine pinned while launching brand-new kernels, export CUDA_MODULE_LOADING=EAGER.


def cuda_world(devices, heap_mb=256, multicast=True, max_ctas=8, engine=False, nvls_min_ranks=3, oneshot_kb=2048,
               nvls_ops=-1, **extra):
    """In-process world on real GPUs: rank i drives devices[i] (a device may
    appear several times: ranks then share that GPU, without NVLS).  `extra`: engine_workers, engine_idle_us,
    stage_kb, ll_kb and every `set_tuning` knob."""
    _prepare_cuda_env()
    options = dict(extra, heap_mb=heap_mb, multicast=multicast, max_ctas=max_ctas, engine=engine,
                   nvls_min_ranks=nvls_min_ranks, oneshot_kb=oneshot_kb, nvls_ops=nvls_ops)
    impls = _C.make_cuda_world(list(devices), {k: int(v) for k, v in options.items()})
    return [Accl(a, r, len(devices), cuda_device=devices[r]) for r, a in enumerate(impls)]


def bind_to_gpu_numa_node(device):
    """Pin this process to the CPUs nearest to `device` (NVML affinity) so that pinned staging
    buffers and the launch path stay on the GPU's NUMA node.  Best effort; returns the CPU set."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:  # noqa: BLE001
        return set()


def cuda_rank(rank=None, world_size=None, device=None, addr=None, port=None, heap_mb=1024, multicast=True,
              max_ctas=128, engine=False, nvls_min_ranks=3, oneshot_kb=2048, nvls_ops=-1, **extra):
    """One rank per process (torchrun): RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT."""
    _prepare_cuda_env()
    rank = int(os.environ.get("RANK", 0)) if rank is None else rank
    world_size = int(os.environ.get("WORLD_SIZE", 1)) if world_size is None else world_size
    device = int(os.environ.get("LOCAL_RANK", rank)) if device is None else device
    addr = os.environ.get("MASTER_ADDR", "127.0.0.1") if addr is None else addr
    if addr == "localhost":
        addr = "127.0.0.1"
    if port is None:
        port = int(os.environ.get("ACCL_PORT", int(os.environ.get("MASTER_PORT", 29500)) + 137))
    if os.environ.get("ACCL_BIND_NUMA", "1") != "0":
        bind_to_gpu_numa_node(device)
    options = dict(extra, heap_mb=heap_mb, multicast=multicast, max_ctas=max_ctas, engine=engine,
                   nvls_min_ranks=nvls_min_ranks, oneshot_kb=oneshot_kb, nvls_ops=nvls_ops)
    impl = _C.make_cuda_rank(rank, world_size, device, addr, port, {k: int(v) for k, v in options.items()})
    return Accl(impl, rank, world_size, cuda_device=device)


def run_cuda_ranks(devices, fn, init_kwargs=None, timeout=180.0, **cfg):
    """Threads-as-ranks harness on GPUs (the CUDA twin of run_ranks)."""
    accls = cuda_world(devices, **cfg)
    world = len(devices)
    errors = [None] * world
    results = [None] * world

    def body(r):
        try:
            torch.cuda.set_device(devices[r])
            # one torch stream per rank: ranks sharing a GPU must never queue on the same stream
            with torch.cuda.stream(torch.cuda.Stream(devices[r])):
                accls[r].initialize(**(init_kwargs or {}))
                results[r] = fn(accls[r], r, world)
                torch.cuda.current_stream().synchronize()
        except BaseException as e:  # noqa: BLE001
            import traceback
            errors[r] = (e, traceback.format_exc())

    threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    hung = [r for r, t in enumerate(threads) if t.is_alive()]
    _raise_rank_errors(errors, hung, timeout)
    for a in accls:
        a.deinit()
    del accls
    return results
