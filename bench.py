#!/usr/bin/env python
"""Headline benchmark: all-reduce bus bandwidth (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # N=1: plain python
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N \
      --master-addr 127.0.0.1 --master-port P bench.py --gpus N --steps K --warmup W

One rank per GPU.  The timed region is K all-reduces of `--bytes` (default
256 MiB fp32 per GPU, larger than the 126 MB L2) on device-resident buffers of
the library's symmetric heap, bracketed by barrier + torch.cuda.synchronize()
and timed with CUDA events; the reported time is the max over ranks.  `value`
is NCCL-tests bus bandwidth (algbw * 2(P-1)/P; algbw itself for P=1).  The
`e2e` block repeats the measurement through the public API with host-resident
data (pinned H2D of the input and D2H of the result inside every step — the
library's default calling convention, reference accl.cpp:780-826).

`--impl reference` reports why the reference cannot run here; `--impl nccl`
measures torch.distributed/NCCL on the same buffers sizes for comparison.
The reference's own sweep benchmark is test/host/xrt/src/bench.cpp:25-61.

`--dump-outputs DIR` writes, after the timed steps, the all-reduce result of
the last step as DIR/allreduce_out.npy (rank 0; float32, float64 for float64
runs).  Results larger than DUMP_MAX_ELEMS are sampled at positions drawn from
a fixed seed.  The operands are seeded too, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def busbw_factor(p):
    return 2.0 * (p - 1) / p if p > 1 else 1.0


DUMP_MAX_ELEMS = 4 << 20  # 16 MiB as float32, 32 MiB as float64


def dump_output(out_dir, name, t):
    """Write the 1-D result `t` (or a seeded sample of it) as out_dir/<name>.npy in float32 / float64."""
    import numpy as np
    import torch
    if t.numel() > DUMP_MAX_ELEMS:
        g = torch.Generator().manual_seed(0)
        idx = torch.randint(0, t.numel(), (DUMP_MAX_ELEMS,), generator=g).sort().values
        t = t[idx.to(t.device)]
    t = t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t.start()

    def stop(self):
        self._stop.set()
        self._t.join(timeout=6)
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for n, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="accl", choices=["accl", "reference", "nccl"])
    ap.add_argument("--bytes", type=int, default=256 << 20)
    ap.add_argument("--dtype", default="float32")
    ap.add_argument("--max-ctas", type=int, default=int(os.environ.get("ACCL_MAX_CTAS", 128)))
    ap.add_argument("--engine", action="store_true", help="route calls through the persistent engine kernel")
    ap.add_argument("--tune", default="", help="name=value,... runtime knobs (Accl.set_tuning), identical on every rank")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-nccl", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the result of the last timed step to DIR/allreduce_out.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        print(json.dumps({"impl": "reference", "unavailable":
                          "Xilinx/ACCL is an FPGA design (HLS kernels + MicroBlaze firmware + XRT/Coyote host driver); "
                          "no setup.py/pyproject, needs XRT, Vitis, ZMQ, jsoncpp and an Alveo card or its RTL simulator: "
                          "`pip install --target baseline/_ref /root/reference` fails with 'not installable'"}))
        return 0

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    torch.cuda.set_device(local)
    use_dist = world > 1
    if use_dist:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    dt = getattr(torch, args.dtype)
    esz = torch.empty((), dtype=dt).element_size()
    n = args.bytes // esz
    nbytes = n * esz
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if not use_dist:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warm):
        for _ in range(warm):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        barrier()
        return max_over_ranks(ms)

    sampler = ClockSampler(local) if rank == 0 else None
    result = {}
    if args.impl == "nccl":
        x = torch.ones(n, dtype=dt, device="cuda")
        fn = (lambda: dist.all_reduce(x)) if use_dist else (lambda: x.add_(0))
        if sampler:
            sampler.start()
        ms = timed(fn, K, W)
        if args.dump_outputs and rank == 0:
            dump_output(args.dump_outputs, "allreduce_out", x)
        launches = K
        impl_name = "nccl"
        e2e = None
    else:
        import accl_b200 as A
        heap_mb = max(512, (4 * nbytes >> 20) + 256)
        acc = A.cuda_rank(rank, world, local, heap_mb=heap_mb, max_ctas=args.max_ctas, engine=args.engine)
        acc.initialize(n_egr_rx_bufs=4, egr_rx_buf_size=64 << 10, max_egr_size=64 << 10, max_rndzv_size=1 << 30)
        for kv in filter(None, args.tune.split(",")):
            k, v = kv.split("=")
            acc.set_tuning(k, int(v))
        src = acc.create_buffer(n, dt)
        dst = acc.create_buffer(n, dt)
        # rank-dependent pseudo-random operands; the guard below compares the WHOLE result with a float64 reference
        g = torch.Generator(device="cuda").manual_seed(1234 + rank)
        src.dev.copy_((torch.rand(n, device="cuda", generator=g) * 2 - 1).to(dt))
        dst.dev.zero_()

        def fn():
            acc.allreduce(src, dst, n, A.SUM, from_fpga=True, to_fpga=True, run_async=True).free()

        # correctness guard: a wrong (mis-sharded, permuted, partially reduced) answer must not produce a number
        fn()
        torch.cuda.synchronize()
        chunk = 32 << 20
        worst = 0.0
        for o in range(0, n, chunk):
            ref = src.dev[o:o + chunk].double()
            if use_dist:
                dist.all_reduce(ref)
            worst = max(worst, float((dst.dev[o:o + chunk].double() - ref).abs().max()))
            del ref
        tol = {torch.float32: 1e-5, torch.float16: 2e-2, torch.bfloat16: 1e-1}.get(dt, 1e-5) * max(world, 1)
        assert worst <= tol, f"allreduce wrong: max abs error {worst} > {tol}"
        result["max_abs_err_vs_fp64_ref"] = worst
        if sampler:
            sampler.start()
        ms = timed(fn, K, W)
        if args.dump_outputs and rank == 0:
            # before the e2e pass below, which writes dst
            dump_output(args.dump_outputs, "allreduce_out", dst.dev)
        # kernels of this library launched inside the timed region: one k_call per all-reduce (direct launch), or one
        # k_submit proxy per all-reduce handing the command to the resident k_engine kernel (engine mode)
        launches = K
        impl_name = "accl_b200"
        e2e = None
        nccl = None
        if use_dist and not args.no_nccl:
            x = src.dev.clone() if nbytes <= (1 << 30) else torch.ones(n, dtype=dt, device="cuda")
            ms_n = timed(lambda: dist.all_reduce(x), max(3, K // 2), 3)
            nccl = {"ms_per_step": ms_n, "busbw_GBps": nbytes / ms_n * 1e-6 * busbw_factor(world)}
            del x
        if not args.no_e2e:
            # public API, host-resident operands: pinned H2D of the input and D2H of the result every step
            src.host.copy_(torch.rand(n, generator=torch.Generator().manual_seed(99 + rank)).to(dt))

            def fn_e2e():
                acc.allreduce(src, dst, n, A.SUM)  # from_fpga=False, to_fpga=False, blocking

            e_steps = max(3, min(K, 10))
            ms_e = timed(fn_e2e, e_steps, 3)
            # the value that came back must be the sum of what went in (first / last elements against a float64 reference)
            probe = torch.cat([src.host[:1024], src.host[-1024:]]).double().cuda()
            if use_dist:
                dist.all_reduce(probe)
            got = torch.cat([dst.host[:1024], dst.host[-1024:]]).double().cuda()
            assert float((got - probe).abs().max()) <= tol, "e2e allreduce wrong"
            e2e = {"value": nbytes / ms_e * 1e-6 * busbw_factor(world), "unit": "GB/s", "ms_per_step": ms_e,
                   "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes, "steps": e_steps,
                   "note": "accl allreduce(sendbuf, recvbuf) with host-resident data: sync_to_device + collective + sync_from_device"}
            if use_dist and not args.no_nccl:
                # the same end-to-end step on NCCL: pinned H2D, dist.all_reduce, D2H, blocking
                hx = torch.empty(n, dtype=dt).pin_memory()
                hy = torch.empty(n, dtype=dt).pin_memory()
                hx.copy_(src.host)
                dx = torch.empty(n, dtype=dt, device="cuda")

                def nccl_e2e():
                    dx.copy_(hx, non_blocking=True)
                    dist.all_reduce(dx)
                    hy.copy_(dx, non_blocking=True)
                    torch.cuda.current_stream().synchronize()

                ms_ne = timed(nccl_e2e, e_steps, 3)
                e2e["nccl_e2e"] = {"value": nbytes / ms_ne * 1e-6 * busbw_factor(world), "ms_per_step": ms_ne}
                del hx, hy, dx
        result["nccl_same_run"] = nccl
        result["backend"] = acc.describe()
        result["mode"] = "engine" if args.engine else "direct"
    clocks = sampler.stop() if sampler else None
    algbw = nbytes / ms * 1e-6
    value = algbw * busbw_factor(world)
    if rank == 0:
        out = {
            "metric": "allreduce_bus_bandwidth", "value": value, "unit": "GB/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic", "impl": impl_name,
            "config": {"model": "allreduce SUM, device-resident symmetric-heap buffers", "global_batch": nbytes * world,
                       "seq_len": n, "bytes_per_gpu": nbytes, "parallelism": f"dp{world}",
                       "l2": "operands (2 x %d MiB per GPU) exceed the 126 MB L2; no flush needed" % (nbytes >> 20),
                       "busbw": "algbw*2(P-1)/P (NCCL-tests convention); P=1 reports algbw of the local copy",
                       "roofline_GBps_per_dir": 900, "timer": "CUDA events, max over ranks"},
            "algbw_GBps": algbw, "gpu_launches": launches, "clocks": clocks,
        }
        if world > 1:
            # bytes per direction per GPU: in-switch two-shot moves M (1 + 1/P), peer two-shot 2 M (P-1)/P
            # (the NVLink byte counters confirm both: profiles/nvlink_traffic_*.jsonl)
            in_switch = "nvls=yes" in str(result.get("backend", "")) and world >= 3
            per_dir = nbytes * (1 + 1.0 / world) if in_switch else 2.0 * nbytes * (world - 1) / world
            out["link_GBps_per_dir"] = per_dir / ms * 1e-6
            out["link_accounting"] = "in-switch two-shot: M (1 + 1/P)" if in_switch else "peer two-shot: 2 M (P-1)/P"
            out["frac_of_900_GBps_link"] = out["link_GBps_per_dir"] / 900.0
        if e2e is not None:
            out["e2e"] = e2e
        out.update(result)
        print(json.dumps(out), flush=True)
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
