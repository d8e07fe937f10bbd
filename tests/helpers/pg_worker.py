"""Worker of tests/test_emulator_multiprocess.py::test_torch_distributed_backend (one process per rank)."""
import faulthandler, os, sys
faulthandler.dump_traceback_later(int(os.environ.get("PG_WATCHDOG_S", 90)), exit=True)  # a hang prints where, then exits
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch, torch.distributed as dist
import accl_b200.parallel.process_group  # noqa
import accl_b200 as A  # noqa: E402
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
use_cuda = torch.cuda.is_available() and A._C.with_cuda and A._C.cuda_driver_available()
if use_cuda:  # same choice init_from_env makes inside the backend; then every tensor lives on this rank's GPU
    os.environ["LOCAL_RANK"] = str(int(os.environ.get("LOCAL_RANK", rank)) % torch.cuda.device_count())  # ranks may share a GPU
    torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
    torch.set_default_device(torch.device("cuda", int(os.environ["LOCAL_RANK"])))
port = os.environ.get("PG_PORT") or str(int(os.environ.get("MASTER_PORT", 29500)) + 7)
if "TORCHELASTIC_RUN_ID" in os.environ:   # under torchrun the agent already hosts the store at MASTER_ADDR:MASTER_PORT
    dist.init_process_group("accl", init_method="env://", rank=rank, world_size=world)
else:
    dist.init_process_group("accl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
if not use_cuda:
    # emulator ranks are separate processes that can reach a collective more than the engine's default receive
    # timeout (1 s) apart on a busy host: give them the budget the CUDA backend has by default (32 s)
    accl_b200.parallel.process_group._primary["accl"].set_timeout(32_000_000)
t = torch.full((1000,), float(rank + 1))
dist.all_reduce(t)
assert torch.all(t == world * (world + 1) / 2), t[:4]
dist.all_reduce(t, op=dist.ReduceOp.MAX)
b = torch.full((33,), float(rank)); dist.broadcast(b, src=1); assert torch.all(b == 1)
out = torch.empty(4 * world); dist.all_gather_into_tensor(out, torch.full((4,), float(rank)))
assert torch.equal(out[::4], torch.arange(world, dtype=torch.float32))
lst = [torch.empty(3) for _ in range(world)]; dist.all_gather(lst, torch.full((3,), float(rank)))
assert all(torch.all(lst[q] == q) for q in range(world))
rs = torch.empty(5); dist.reduce_scatter_tensor(rs, torch.ones(5 * world)); assert torch.all(rs == world)
a2a = torch.empty(2 * world); dist.all_to_all_single(a2a, torch.arange(2 * world, dtype=torch.float32) + 100 * rank)
assert torch.equal(a2a[::2], torch.tensor([100.0 * q + 2 * rank for q in range(world)]))
r = torch.full((7,), float(rank)); dist.reduce(r, dst=0, op=dist.ReduceOp.SUM)
if rank == 0: assert torch.all(r == sum(range(world)))
if rank == 0: dist.send(torch.arange(10, dtype=torch.float32), dst=1)
if rank == 1:
    x = torch.empty(10); dist.recv(x, src=0); assert torch.equal(x, torch.arange(10, dtype=torch.float32))
dist.barrier()
# sub-groups are communicators on the same engine (each with its own protocol-state bank)
members = [0, world - 1] if world > 2 else [0, 1]
sub = dist.new_group(members)
if rank in members:
    sgt = torch.full((257,), float(rank + 1)); dist.all_reduce(sgt, group=sub)
    assert torch.all(sgt == sum(m + 1 for m in members)), sgt[:4]
    nc = torch.arange(12, dtype=torch.float32).view(3, 4).t()   # non-contiguous destination
    dist.broadcast(nc, src=members[0], group=sub)
dist.barrier()
# DistributedDataParallel on top
torch.manual_seed(0)
model = torch.nn.Linear(8, 4)
ddp = torch.nn.parallel.DistributedDataParallel(model)
xs = torch.randn(16, 8, generator=torch.Generator(device="cpu").manual_seed(rank), device="cpu").to(model.weight.device)
ddp(xs).sum().backward()
g = model.weight.grad.clone()
chk = g.clone(); dist.all_reduce(chk, op=dist.ReduceOp.MAX)
assert torch.allclose(chk, g), "DDP gradients differ across ranks"
dist.barrier()
print(f"pg rank {rank}: ok", flush=True)
dist.destroy_process_group()
