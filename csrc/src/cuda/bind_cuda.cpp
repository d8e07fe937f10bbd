// pybind11 glue for the CUDA backend (kept out of pyaccl.cpp so that the
// emulator-only build has no CUDA dependency).
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <map>

#include "accl/accl.hpp"
#include "accl/cuda/cudadevice.hpp"
#include "accl/cuda/driver_api.hpp"
#include "accl/cuda/plan.hpp"
#include "accl/cuda/plugins.hpp"

namespace py = pybind11;

namespace accl {
namespace cuda {

using OptionMap = std::map<std::string, long>;

static CudaConfig config_from(const OptionMap &options) {
  CudaConfig c;
  for (auto &kv : options)
    if (!set_option(c, kv.first, kv.second, false)) throw std::invalid_argument("unknown CUDA backend option '" + kv.first + "'");
  return c;
}

static CudaDevice *cuda_device(ACCL &a) {
  auto *d = dynamic_cast<CudaDevice *>(a.device());
  if (!d) throw std::runtime_error("not a CUDA backend");
  return d;
}

static py::dict plan_dict(const WorkItem &w) {
  static const char *names[] = {"auto", "local", "eager", "nvls", "p2p", "p2p_oneshot", "ll", "staged", "wire"};
  py::dict d;
  d["algo"] = w.algo < 9 ? names[w.algo] : "?";
  d["n_ctas"] = w.n_ctas;
  d["use_mc"] = (w.flags & WF_USE_MC) != 0;
  d["oneshot"] = (w.flags & WF_ONESHOT) != 0;
  return d;
}

void bind_cuda(py::module_ &m) {
  m.def("cuda_driver_available", [] { return DriverApi::available(); });
  // The call planner (plan.hpp) as a pure function, for unit tests on machines without a GPU: which protocol /
  // algorithm / channel count a call of `count` elements of `dtype` gets on `world` ranks, given the eager limits (default
  // 64 KiB), the staging regions (1 MiB, LL 256 KiB), and any backend options (CudaConfig defaults otherwise).
  m.def("cuda_plan", [](operation op, uint32_t count, dataType dtype, uint32_t world, uint32_t max_eager_bytes,
                        uint32_t eager_rx_buf_bytes, bool has_mc, uint32_t stage_kb, uint32_t ll_kb, bool engine_mode,
                        bool compressed, const py::kwargs &options) {
    const CudaConfig cfg = config_from(options.cast<OptionMap>());
    std::vector<uint32_t> exch(exchmem::SIZE_WORDS, 0);
    exch[exchmem::MAX_EAGER_SIZE / 4] = max_eager_bytes;
    exch[exchmem::EAGER_RX_BUF_SIZE / 4] = eager_rx_buf_bytes;
    // the worker CTAs an engine would start (engine.cu), without its cap by the SM count
    const uint32_t workers = static_cast<uint32_t>(std::max(1, cfg.engine_workers > 0 ? cfg.engine_workers : cfg.max_ctas));
    WorkItem w{};
    w.desc.scenario = static_cast<uint32_t>(op);
    w.desc.count = count;
    w.desc.compression_flags = compressed ? 1u : 0u;
    w.comm_size = world;
    w.udtype = static_cast<uint32_t>(dtype);
    plan_call(exch.data(),
              make_plan_cfg(cfg, has_mc, world, size_t{stage_kb} << 10, size_t{ll_kb} << 10, engine_mode ? workers : 0u), w);
    return plan_dict(w);
  }, py::arg("op"), py::arg("count"), py::arg("dtype"), py::arg("world"), py::kw_only(), py::arg("max_eager_bytes") = 64u << 10,
        py::arg("eager_rx_buf_bytes") = 64u << 10, py::arg("has_mc") = true, py::arg("stage_kb") = 1024, py::arg("ll_kb") = 256,
        py::arg("engine_mode") = false, py::arg("compressed") = false);
  // how a live device plans a call: its exchange memory and plan_cfg(), without running the call
  m.def("cuda_plan_call", [](ACCL &a, operation op, uint32_t count, dataType dtype, communicatorId comm_id) {
    CCLO::Options o;
    o.scenario = op;
    o.count = count;
    o.comm = comm_id;
    o.arithcfg_addr = a.get_arithmetic_config_addr({dtype, dtype});
    WorkItem w;
    uint32_t err = 0;
    if (!cuda_device(a)->build_work_item(o, make_call_desc(o), w, err)) throw std::invalid_argument("cuda_plan_call: error " + std::to_string(err));
    return plan_dict(w);
  }, py::arg("accl"), py::arg("op"), py::arg("count"), py::arg("dtype"), py::arg("comm_id") = 0);
  m.def("cuda_set_tuning", [](ACCL &a, const std::string &name, long value) {
    if (!cuda_device(a)->set_tuning(name, value)) throw std::invalid_argument("unknown tuning knob '" + name + "'");
  });
  m.def("cuda_get_tuning", [](ACCL &a, const std::string &name) { return cuda_device(a)->get_tuning(name); });
  m.def("cuda_drain", [](ACCL &a) {
    auto *d = dynamic_cast<CudaDevice *>(a.device());
    if (d) d->drain();
  }, py::call_guard<py::gil_scoped_release>());
  // zero-copy operands for memory that already lives in the heap (torch tensors from the heap pool)
  m.def("cuda_wrap_device", [](ACCL &a, uintptr_t dev_ptr, size_t n, dataType t) {
    CudaDevice *d = cuda_device(a);
    const size_t bytes = n * dtype_bytes(t);
    return std::unique_ptr<BaseBuffer>(new BaseBuffer(d->wrap_device(reinterpret_cast<void *>(dev_ptr), bytes), 0, bytes, t));
  });
  m.def("cuda_heap_range", [](ACCL &a) {
    CudaDevice *d = cuda_device(a);
    return std::make_pair(reinterpret_cast<uintptr_t>(d->heap().local()), d->heap().bytes());
  });
  m.def("cuda_heap_pool_attach", [](ACCL &a) { heap_pool_attach(cuda_device(a)); });
  m.def("cuda_debug_state", [](ACCL &a) { return cuda_device(a)->debug_state(); });
  // out_shard[M/P, N] (heap buffer, bf16) = reduce_scatter_M( A[M,K] @ W[N,K]^T ), fused on tcgen05 + NVLink
  m.def("gemm_reduce_scatter", [](ACCL &a, uintptr_t a_ptr, uintptr_t w_ptr, BaseBuffer &out, uint32_t M, uint32_t N, uint32_t K,
                                  uintptr_t stream, int variant) {
    CudaDevice *d = cuda_device(a);
    GemmRsArgs g{reinterpret_cast<const void *>(a_ptr), reinterpret_cast<const void *>(w_ptr), out.address(), M, N, K, 0};
    g.variant = variant;
    g.out_f32 = out.type() == dataType::float32;
    if (!g.out_f32 && out.type() != dataType::bfloat16) throw std::invalid_argument("gemm_reduce_scatter: output shard must be bf16 or fp32");
    cudaError_t e = launch_gemm_rs(*d, g, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) throw std::runtime_error(std::string("gemm_reduce_scatter launch: ") + cudaGetErrorString(e));
  }, py::arg("accl"), py::arg("a_ptr"), py::arg("w_ptr"), py::arg("out"), py::arg("M"), py::arg("N"), py::arg("K"), py::arg("stream"),
        py::arg("variant") = 0, py::call_guard<py::gil_scoped_release>());
  // out = allreduce_sum(x + y): the kernel computes and then issues the collective itself (device API -> engine)
  m.def("vadd_allreduce", [](ACCL &a, BaseBuffer &x, BaseBuffer &y, BaseBuffer &tmp, BaseBuffer &out, uint32_t count,
                             uintptr_t status_dev_ptr, uintptr_t stream, uint32_t chunk_elems) {
    CudaDevice *d = cuda_device(a);
    cudaError_t e = launch_vadd_allreduce(*d, x.address(), y.address(), tmp.address(), out.address(), count, chunk_elems,
                                          static_cast<uint32_t>(a.get_communicator_addr(GLOBAL_COMM)),
                                          static_cast<uint32_t>(a.get_arithmetic_config_addr({dataType::float32, dataType::float32})),
                                          reinterpret_cast<uint32_t *>(status_dev_ptr), reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) throw std::runtime_error(std::string("vadd_allreduce launch: ") + cudaGetErrorString(e));
  }, py::arg("accl"), py::arg("x"), py::arg("y"), py::arg("tmp"), py::arg("out"), py::arg("count"), py::arg("status_dev_ptr"),
        py::arg("stream"), py::arg("chunk_elems") = 0, py::call_guard<py::gil_scoped_release>());
  // the reference's vadd_put example: src + 1 pushed into stream `stream_id` of rank dst while computing
  m.def("vadd_put", [](ACCL &a, BaseBuffer &src, uint32_t count, uint32_t dst_rank, uint32_t stream_id, uintptr_t status_dev_ptr,
                       uintptr_t stream) {
    CudaDevice *d = cuda_device(a);
    cudaError_t e = launch_vadd_put(*d, src.address(), count, dst_rank, stream_id, reinterpret_cast<uint32_t *>(status_dev_ptr),
                                    reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) throw std::runtime_error(std::string("vadd_put launch: ") + cudaGetErrorString(e));
  }, py::call_guard<py::gil_scoped_release>());
  m.def("stream_pull", [](ACCL &a, BaseBuffer &dst, uint32_t count, uint32_t stream_id, uintptr_t status_dev_ptr, uintptr_t stream) {
    CudaDevice *d = cuda_device(a);
    cudaError_t e = launch_stream_pull(*d, dst.address(), count, stream_id, reinterpret_cast<uint32_t *>(status_dev_ptr),
                                       reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) throw std::runtime_error(std::string("stream_pull launch: ") + cudaGetErrorString(e));
  }, py::call_guard<py::gil_scoped_release>());
  m.def("stream_loopback", [](ACCL &a, BaseBuffer &scratch, uint32_t count, bool add_one, uintptr_t status_dev_ptr,
                              uintptr_t stream) {
    CudaDevice *d = cuda_device(a);
    cudaError_t e = launch_loopback(*d, scratch.address(), count, add_one, reinterpret_cast<uint32_t *>(status_dev_ptr),
                                    reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) throw std::runtime_error(std::string("stream_loopback launch: ") + cudaGetErrorString(e));
  }, py::call_guard<py::gil_scoped_release>());
  m.def("cuda_probe", [](int device) { return probe_topology(device).describe(); });
  // N ranks in this process (threads), rank i on devices[i]
  m.def("make_cuda_world", [](std::vector<int> devices, const OptionMap &options) {
    std::vector<std::unique_ptr<ACCL>> out;
    for (auto &d : make_local_world(devices, config_from(options))) out.emplace_back(new ACCL(std::move(d)));
    return out;
  }, py::arg("devices"), py::arg("options"), py::call_guard<py::gil_scoped_release>());
  // one rank per process; bootstrap over a private TCP rendezvous on addr:port
  m.def("make_cuda_rank", [](int rank, int world, int device, const std::string &addr, int port, const OptionMap &options) {
    CudaConfig cfg = config_from(options);
    cfg.device = device;
    auto oob = std::make_shared<TcpOob>(rank, world, addr, port);
    return std::unique_ptr<ACCL>(new ACCL(std::unique_ptr<CCLO>(new CudaDevice(oob, cfg))));
  }, py::arg("rank"), py::arg("world_size"), py::arg("device"), py::arg("addr"), py::arg("port"), py::arg("options"),
        py::call_guard<py::gil_scoped_release>());
}

} // namespace cuda
} // namespace accl
