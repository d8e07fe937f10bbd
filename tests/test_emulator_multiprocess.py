"""One emulator rank per process over loopback TCP (SocketFabric): the
multi-process deployment of the CPU backend, as CI runs the reference's
emulator under mpirun (.github/workflows/build-and-test.yml:52-101)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [2, 3])
def test_selftest_over_sockets(world):
    r = subprocess.run([sys.executable, "-m", "accl_b200.models.emulator", "-n", str(world), "--selftest"], cwd=ROOT,
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count(": ok") == world


def test_standalone_engine_processes_with_remote_drivers():
    """Engines as separate processes (build/bin/cclo_emu), drivers attach over the control socket:
    the reference's cclo_emu + SimDevice deployment (test/model/emulator/run.py, simdevice.cpp)."""
    import threading

    import torch

    import accl_b200 as A
    from accl_b200.models.emulator import spawn_engines

    world = 3
    procs, base = spawn_engines(world, mem_mb=32, stderr=subprocess.DEVNULL)
    errors = []

    def driver(r):
        try:
            a = A.remote_rank(r, world, ctrl_port=base + 1000 + r)
            assert "RemoteDevice" in a.describe()
            a.initialize(n_egr_rx_bufs=16, egr_rx_buf_size=1024, max_egr_size=1024, max_rndzv_size=32768)
            for n in (16, 300, 20000):  # eager, segmented eager, rendezvous
                s, d = a.create_buffer(n), a.create_buffer(n)
                s.host[:] = torch.arange(n, dtype=torch.float32) + r
                nxt, prv = (r + 1) % world, (r - 1) % world
                req = a.send(s, n, nxt, tag=3, run_async=True)
                a.recv(d, n, prv, tag=3)
                req.wait()
                assert torch.equal(d.host, torch.arange(n, dtype=torch.float32) + prv)
                req = a.allreduce(s, d, n, A.SUM, run_async=True)
                req.wait()
                d.sync_from_device()  # async call with a host-resident result: the read-back is ours
                assert req.duration_ns() > 0
                ref = sum(torch.arange(n, dtype=torch.float32) + q for q in range(world))
                assert torch.allclose(d.host, ref)
            # the one-hop schedules of the B200 backend inside a stand-alone engine: the register travels over the control socket
            a.barrier()
            a.set_one_hop_schedules(True)
            for n in (300, 6000):   # rendezvous class, one hop: the whole vector lands in a scratch buffer (<= max_rndzv_size)
                s, d = a.create_buffer(n), a.create_buffer(n)
                s.host[:] = torch.arange(n, dtype=torch.float32) + r
                a.allreduce(s, d, n, A.SUM)
                assert torch.equal(d.host, sum(torch.arange(n, dtype=torch.float32) + q for q in range(world)))
            assert "one_hop_dispatches=" in A._C.emu_remote_debug_state(a.impl)
            assert int(A._C.emu_remote_debug_state(a.impl).split("one_hop_dispatches=")[1].split()[0]) >= 2
            a.barrier()
            a.set_one_hop_schedules(False)
            # stream port through the control connection (kernel loopback is on by default)
            s, d = a.create_buffer(64), a.create_buffer(64)
            s.host[:] = torch.arange(64, dtype=torch.float32) * (r + 1)
            a.copy_to_stream(s, 64)
            a.copy_from_stream(d, 64)
            assert torch.equal(s.host, d.host)
            a.barrier()
            a.deinit()
            A._C.emu_remote_shutdown(a.impl)
        except BaseException as e:  # noqa: BLE001
            errors.append((r, repr(e)))

    ts = [threading.Thread(target=driver, args=(r,)) for r in range(world)]
    try:
        for t in ts:
            t.start()
        for t in ts:
            t.join(timeout=120)
        assert not errors, errors
        assert all(not t.is_alive() for t in ts), "driver hung"
        for p in procs:
            assert p.wait(timeout=30) == 0
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()


def test_cpp_suite_binary():
    """The C++ API test list (csrc/tools/emu_suite.cpp, counterpart of the reference's gtest binary)."""
    from accl_b200.utils import build as b
    exe = os.path.join(ROOT, "build", "bin", "emu_suite")
    if not os.path.exists(exe):
        b.build_tool("emu_suite")
    r = subprocess.run([exe, "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " 0 failed" in r.stdout


@pytest.mark.parametrize("zero", [0, 1])
def test_data_parallel_mlp_trains(zero):
    """End-to-end consumer: DDP / ZeRO-1 training of a small MLP, one emulator process per rank."""
    import json
    r = subprocess.run([sys.executable, "-m", "accl_b200.models.emulator", "-n", "2", "--", sys.executable, "-m",
                        "accl_b200.models.dp_mlp", "--backend", "emulator", "--zero", str(zero), "--steps", "20"], cwd=ROOT,
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][0]
    out = json.loads(line)
    assert out["ok"] and out["replicas_identical"] and out["loss_last"] < out["loss_first"]


def test_cpp_example_links_against_the_static_library(tmp_path):
    """examples/cpp/allreduce_emulator.cpp against build/lib/libaccl.a: the path a C++ user of the reference's
    driver takes (no Python anywhere)."""
    from accl_b200.utils import build as b
    lib = os.path.join(ROOT, "build", "lib", "libaccl.a")
    if not os.path.exists(lib):
        pytest.skip("static library not built (python -m accl_b200.utils.build)")
    exe = str(tmp_path / "allreduce_emulator")
    cmd = [b.CXX, "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "csrc", "include"),
           os.path.join(ROOT, "examples", "cpp", "allreduce_emulator.cpp"), lib]
    cudart = "/usr/local/cuda/lib64/libcudart_static.a"
    import accl_b200 as A
    if A._C.with_cuda and os.path.exists(cudart):
        cmd.append(cudart)
    cmd += ["-lpthread", "-ldl", "-lrt", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "all ranks ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("one_hop", ["0", "1"], ids=["rings", "one_hop"])
@pytest.mark.parametrize("world", [2, 3])
def test_torch_distributed_backend(world, one_hop):
    """`dist.init_process_group("accl")`: all_reduce / broadcast / all_gather / reduce_scatter / all_to_all /
    reduce / send / recv / barrier and DistributedDataParallel through the standard torch.distributed API."""
    import random
    # no GPU visible: the backend picks the CUDA path whenever it can (test_cuda_engine.py covers that one)
    env = dict(os.environ, PG_PORT=str(random.randint(20000, 40000)), ACCL_EMU_ONE_HOP=one_hop, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "accl_b200.models.emulator", "-n", str(world), "--", sys.executable,
                        os.path.join(ROOT, "tests", "helpers", "pg_worker.py")], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count(": ok") == world


def test_engine_process_survives_garbage_on_the_control_port():
    """A stray client sending a malformed frame must not crash or wedge the engine process: unknown request
    types are answered with an error reply, an absurd length closes the connection and the process exits cleanly."""
    import socket
    import struct
    from accl_b200.models.emulator import spawn_engines
    procs, base = spawn_engines(1, mem_mb=16, stderr=subprocess.DEVNULL)
    try:
        s = None
        for _ in range(200):
            try:
                s = socket.create_connection(("127.0.0.1", base + 1000), timeout=5)
                break
            except OSError:
                import time
                time.sleep(0.05)
        assert s is not None
        # frame: type, seq, a, b, len, aux  (32 bytes, little endian)
        s.sendall(struct.pack("<IIQQII", 999, 1, 0, 0, 0, 0))
        hdr = s.recv(32, socket.MSG_WAITALL)
        typ, seq, _, _, ln, aux = struct.unpack("<IIQQII", hdr)
        assert typ == 0x8000 and seq == 1 and aux == 1       # REPLY with the error flag
        msg = s.recv(ln, socket.MSG_WAITALL)
        assert b"unknown request" in msg
        s.sendall(struct.pack("<IIQQII", 5, 2, 0, 0, 0xFFFFFFF0, 0))   # 4 GiB "payload"
        assert s.recv(32) == b""                              # connection dropped
        s.close()
        assert procs[0].wait(timeout=20) == 0
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()


def test_cpp_fuzz_binary():
    """csrc/tools/emu_fuzz.cpp: random call programs through the C++ API (the binary the TSan / ASan campaigns use)."""
    from accl_b200.utils import build as b
    exe = os.path.join(ROOT, "build", "bin", "emu_fuzz")
    if not os.path.exists(exe):
        b.build_tool("emu_fuzz")
    r = subprocess.run([exe, "400", "5"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and " 0 failed" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
