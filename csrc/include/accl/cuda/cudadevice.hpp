// CudaDevice: the B200 backend.  Owns the symmetric NVLink heap (control
// block + eager slots + user buffers), selects protocol/algorithm per call,
// and executes calls either by direct stream-ordered kernel launch or through
// the persistent engine kernel (command rings in device memory).
//
// Reference counterparts: XRTDevice / CoyoteDevice (driver/xrt/src/xrtdevice.cpp,
// coyotedevice.cpp) for the call path, XRTBuffer for storage, and the
// firmware's per-call decisions (ccl_offload_control.c:2308-2483) for
// `plan()`.
#pragma once
#include <cuda_runtime.h>

#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "accl/allocator.hpp"
#include "accl/bootstrap.hpp"
#include "accl/cclo.hpp"
#include "accl/cuda/devtypes.hpp"
#include "accl/cuda/launch.hpp"
#include "accl/cuda/plan.hpp"
#include "accl/cuda/symheap.hpp"
#include "accl/request.hpp"

namespace pybind11 {
class module_;
}

namespace accl {
namespace cuda {

constexpr size_t STREAM_FIFO_BYTES = 1u << 20; // capacity of one device-side stream FIFO (power of two; scaled down on small heaps)

struct CudaConfig {
  int device = 0;
  size_t heap_bytes = 1ull << 30;
  bool multicast = true;       // try to set up NVLS
  int max_ctas = 32;           // CTAs a single call may use (== sync channels used)
  int nvls_min_ranks = 3;      // below this, peer loads/stores beat the switch round trip
  size_t host_pipeline_chunk = 16u << 20; // chunk size of the pipelined host-operand path (0 = off)
  size_t oneshot_max_bytes = 2048 << 10; // allreduce: pull-everything one-shot while bytes x ranks <= this
  uint32_t nvls_ops = NVLS_OPS_DEFAULT;  // which operations may use multimem (bit = operation code)
  bool engine = false;         // route calls through the persistent engine kernel
  int engine_idle_us = 1000;   // engine kernel parks itself after this idle time (0 = never)
  int engine_workers = 0;      // worker CTAs of the engine (0: max_ctas, never more than SMs - 16)
  int nvls_ctas = 32;          // channel cap of the NVLS two-shot all-reduce
  size_t stage_bytes = 0;      // staging region per (bank, parity, source) of ALGO_STAGED (0: sized from the heap)
  size_t ll_bytes = 0;         // same for ALGO_LL
  size_t ll_max_bytes = 2u << 20;    // flag-in-data protocol while message x (P - 1) peers <= this (and it fits the LL area)
  size_t staged_max_bytes = 0;       // per-peer messages that do not fit LL use ALGO_STAGED up to this size (0: never)
  size_t ll_oneshot_max = 32u << 10; // all-reduce: one hop (everybody sends everything) up to this size
  size_t wire_min_bytes = 256u << 10; // compressed-wire collectives from this size on use the fused two-shot
  Tune tune{0, 4, 0, 0, 0, {0, 0, 0}};
  bool stream_loopback = true; // every stream id is served by FIFO 0 (the reference's loopback user kernel)
};

// The backend's options by name (construction arguments, Accl.set_tuning, ACCL_TUNE), defined by one table in
// cudadevice.cpp.  Applies `value` to `c` with the option's unit scaling (`*_kb`, `heap_mb`) and clamp.  `running`:
// the device already exists, so only the options that may change after construction are accepted.  Returns false
// for a name that is not accepted.
bool set_option(CudaConfig &c, const std::string &name, long value, bool running);

// What the planner (plan.hpp) is told about a device: its options plus the geometry it found at construction.
// `engine_workers`: worker CTAs of the persistent engine, which are the channels of its calls (0: direct launches).
PlanCfg make_plan_cfg(const CudaConfig &c, bool has_mc, uint32_t heap_world, size_t stg_bytes, size_t ll_bytes,
                      uint32_t engine_workers);

class CudaDevice;

struct CudaRequest : public BaseRequest {
  using BaseRequest::BaseRequest;
  ~CudaRequest() override;
  CudaDevice *dev = nullptr;
  cudaStream_t stream = nullptr; // stream the call was enqueued on (fallback for long waits)
  uint32_t slot = 0, seq = 0;
  bool immediate = false; // completed on the host (config calls)
  bool unordered = false; // engine call whose proxy does not hold the stream: completion is only visible in the record
  std::vector<std::shared_ptr<BufferStorage>> temps; // staging buffers that live as long as the call
  std::vector<std::pair<BaseBuffer *, std::shared_ptr<BufferStorage>>> copy_out;
  void wait() override;
  bool wait(std::chrono::milliseconds timeout) override;
  bool test() override;
  void finish();
};

class CudaDevice : public CCLO {
public:
  CudaDevice(std::shared_ptr<Oob> oob, const CudaConfig &cfg);
  ~CudaDevice() override;

  ACCLRequest *call(const Options &options) override;
  ACCLRequest *start(const Options &options) override;
  ACCLRequest *call_host_pipelined(const Options &options) override;
  val_t read(addr_t offset) override;
  void write(addr_t offset, val_t val) override;
  void wait(ACCLRequest *request) override;
  bool wait(ACCLRequest *request, std::chrono::milliseconds timeout) override;
  bool test(ACCLRequest *request) override;
  void free_request(ACCLRequest *request) override;
  val_t get_retcode(ACCLRequest *request) override;
  uint64_t get_duration(ACCLRequest *request) override;
  deviceType get_device_type() override { return deviceType::cuda; }
  std::string describe() override;
  void printDebug() override;
  std::string debug_state();
  std::shared_ptr<BufferStorage> allocate(size_t bytes, bufferKind kind) override;
  std::shared_ptr<BufferStorage> wrap_host(void *host_ptr, size_t bytes) override;
  // view of device memory that already lives inside this rank's heap (e.g. a torch tensor from the heap pool): zero-copy operand
  std::shared_ptr<BufferStorage> wrap_device(void *dev_ptr, size_t bytes);
  void attach(int world_size, int local_rank) override;

  // ---- CUDA specifics
  const DevWorld &world() const { return world_; }
  SymHeap &heap() { return *heap_; }
  const CudaConfig &config() const { return cfg_; }
  cudaStream_t stream() const { return stream_; }
  // stream of the current call sequence (user stream if one was set)
  cudaStream_t op_stream() const { return op_stream_ ? op_stream_ : stream_; }
  void set_stream(void *s) override { op_stream_ = static_cast<cudaStream_t>(s); }
  int device() const { return cfg_.device; }
  bool has_multicast() const { return heap_->has_multicast(); }
  RangeAllocator &allocator() { return *alloc_; }
  HostCompletion *host_completions() { return hc_host_; }
  struct PlanCfg plan_cfg() const;
  // the options that may change after construction (see set_option); must be set identically on every rank.
  // set_tuning returns false for a name it does not accept; get_tuning returns -1 for one it does not know, and also
  // reports the staging sizes "stage_bytes" / "ll_bytes".
  bool set_tuning(const std::string &name, long value);
  long get_tuning(const std::string &name) const;
  // wait until every call started so far has completed (engine quiesce before direct launches share its channels)
  void drain();
  bool build_work_item(const Options &o, const CallDesc &d, WorkItem &w, uint32_t &err);
  uint32_t timeout_us() const;
  Oob &oob() { return *oob_; }
  class Engine *engine() { return engine_.get(); }
  void *plugin_scratch(size_t bytes); // zero-initialised device memory for plugin kernels (grown on demand)
  // FIFO a stream id is served by: the id itself, or 0 while every id loops back through one FIFO (default)
  uint32_t stream_port_id(uint32_t id) const { return cfg_.stream_loopback ? 0u : id; }

private:
  uint32_t host_config(const CallDesc &d);
  void setup_eager_area();
  void sync_ctrl_word(uint32_t byte_off);
  void apply_env_tuning();
  void drain_locked();

  std::shared_ptr<Oob> oob_;
  CudaConfig cfg_;
  std::unique_ptr<SymHeap> heap_;
  std::unique_ptr<RangeAllocator> alloc_;
  DevWorld world_{};
  cudaStream_t stream_ = nullptr;
  cudaStream_t op_stream_ = nullptr;
  cudaStream_t h2d_stream_ = nullptr, d2h_stream_ = nullptr;
  std::vector<uint32_t> shadow_; // host copy of exchange memory
  HostCompletion *hc_host_ = nullptr, *hc_dev_ = nullptr;
  std::vector<std::shared_ptr<CudaRequest>> slot_owner_;
  uint32_t next_slot_ = 0, next_seq_ = 1;
  uint64_t egr_area_off_ = 0;
  std::mutex m_;
  RequestRegistry requests_;
  std::shared_ptr<BufferStorage> egr_area_;
  std::shared_ptr<BufferStorage> strm_area_;
  std::shared_ptr<BufferStorage> stg_area_, ll_area_; // staging of the one-way protocols (staged.cuh)
  std::shared_ptr<BufferStorage> scr_area_;           // scratch of the write-only rooted reduce
  friend struct CudaRequest;
  friend class Engine;
  std::unique_ptr<class Engine> engine_;
  void *plugin_scratch_ = nullptr;
  size_t plugin_scratch_bytes_ = 0;
};

// In-process world: N ranks as threads of this process, rank i on devices[i]
// (devices may repeat: several ranks share one GPU, without NVLS).
std::vector<std::unique_ptr<CudaDevice>> make_local_world(const std::vector<int> &devices, const CudaConfig &base);

void bind_cuda(pybind11::module_ &m);

// torch.cuda.MemPool over the heap (heap_pool.cpp): the backend that serves pool allocations of its CUDA device
void heap_pool_attach(CudaDevice *d);
void heap_pool_detach(CudaDevice *d);

} // namespace cuda
} // namespace accl
