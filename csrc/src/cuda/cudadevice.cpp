#include "accl/cuda/cudadevice.hpp"

#include <algorithm>
#include <atomic>
#include <cstring>
#include <map>
#include <sstream>
#include <thread>

#include "accl/common.hpp"
#include "accl/cuda/driver_api.hpp"
#include "accl/cuda/engine.hpp"
#include "accl/cuda/plan.hpp"

namespace accl {
namespace cuda {

// ------------------------------------------------------------------ storage
namespace {
// Process-wide cache of pinned host blocks.  cudaFreeHost synchronises the
// whole device: doing that while a peer rank's kernel on the same GPU spins on
// a flag this thread has yet to raise is a deadlock, so blocks are recycled
// instead of returned to the driver.
class PinnedPool {
public:
  static PinnedPool &get() {
    static PinnedPool *p = new PinnedPool(); // intentionally leaked: outlives every CUDA context user
    return *p;
  }
  void *alloc(size_t bytes, size_t &cap) {
    cap = 256;
    while (cap < bytes) cap <<= 1;
    {
      std::lock_guard<std::mutex> g(m_);
      auto &fl = free_[cap];
      if (!fl.empty()) {
        void *p = fl.back();
        fl.pop_back();
        return p;
      }
    }
    void *p = nullptr;
    ACCL_CUDART(cudaHostAlloc(&p, cap, cudaHostAllocPortable));
    return p;
  }
  void release(void *p, size_t cap) {
    std::lock_guard<std::mutex> g(m_);
    free_[cap].push_back(p);
  }

private:
  std::mutex m_;
  std::map<size_t, std::vector<void *>> free_;
};

class CudaStorage : public BufferStorage {
public:
  CudaStorage(CudaDevice *d, size_t bytes, bufferKind kind, void *wrap)
      : dev_(d), bytes_(bytes), kind_(kind), wrapped_(wrap) {
    if (kind != bufferKind::host_only) off_ = d->allocator().alloc(std::max<size_t>(bytes, 16), 256);
    else ensure_host();
    if (wrapped_ && bytes_ >= (64u << 10)) {
      // caller-owned host memory: page-lock it in place so H2D / D2H run at PCIe speed straight from / into the user's
      // array (no bounce through a pinned pool); best effort — pageable copies still work if the range cannot be locked
      cudaSetDevice(dev_->device());
      registered_ = cudaHostRegister(wrapped_, bytes_, cudaHostRegisterPortable) == cudaSuccess;
      if (!registered_) cudaGetLastError();
    }
  }
  // a view of memory that already lives inside this rank's heap (torch tensors allocated from the heap pool): not
  // owned, no host mirror unless somebody asks for one
  CudaStorage(CudaDevice *d, size_t bytes, uint64_t heap_off)
      : dev_(d), bytes_(bytes), kind_(bufferKind::p2p), off_(heap_off), owns_(false) {}
  ~CudaStorage() override {
    cudaSetDevice(dev_->device());
    if (kind_ != bufferKind::host_only && owns_) {
      // the engine may still be reading: drain the backend stream first
      cudaStreamSynchronize(dev_->stream());
      try {
        dev_->allocator().free(off_);
      } catch (...) {
      }
    }
    if (pinned_) PinnedPool::get().release(pinned_, pinned_cap_);
    if (registered_) cudaHostUnregister(wrapped_);
  }
  void *host_ptr() override {
    if (wrapped_) return wrapped_;
    ensure_host();
    return pinned_;
  }
  addr_t device_addr() const override { return kind_ == bufferKind::host_only ? 0 : off_; }
  void *device_ptr() const override {
    return kind_ == bufferKind::host_only ? nullptr : dev_->heap().local() + off_;
  }
  size_t bytes() const override { return bytes_; }
  bufferKind kind() const override { return kind_; }
  void to_device(size_t off, size_t len) override {
    if (kind_ == bufferKind::host_only || len == 0) return;
    cudaSetDevice(dev_->device());
    ACCL_CUDART(cudaMemcpyAsync(dev_->heap().local() + off_ + off, static_cast<char *>(host_ptr()) + off, len,
                                cudaMemcpyHostToDevice, dev_->op_stream()));
  }
  void from_device(size_t off, size_t len) override {
    if (kind_ == bufferKind::host_only || len == 0) return;
    cudaSetDevice(dev_->device());
    ACCL_CUDART(cudaMemcpyAsync(static_cast<char *>(host_ptr()) + off, dev_->heap().local() + off_ + off, len,
                                cudaMemcpyDeviceToHost, dev_->op_stream()));
    ACCL_CUDART(cudaStreamSynchronize(dev_->op_stream()));
  }
  bool is_simulated() const override { return false; }

private:
  void ensure_host() {
    if (wrapped_ || pinned_) return;
    cudaSetDevice(dev_->device());
    pinned_ = PinnedPool::get().alloc(std::max<size_t>(bytes_, 16), pinned_cap_);
    std::memset(pinned_, 0, bytes_);
  }
  CudaDevice *dev_;
  size_t bytes_;
  bufferKind kind_;
  uint64_t off_ = 0;
  void *pinned_ = nullptr;
  size_t pinned_cap_ = 0;
  void *wrapped_ = nullptr;
  bool registered_ = false;
  bool owns_ = true;
};
} // namespace

// ------------------------------------------------------------------ request
CudaRequest::~CudaRequest() {}

void CudaRequest::finish() {
  if (status() == operationStatus::COMPLETED) return;
  HostCompletion *hc = &dev->hc_host_[slot];
  const uint32_t rc = hc->seq == seq ? hc->retcode : static_cast<uint32_t>(DMA_INTERNAL_ERROR);
  const uint64_t dur = hc->duration_ns;
  for (auto &co : copy_out) { // results of host-resident operands
    co.second->from_device(0, co.second->bytes());
    if (co.first && co.first->byte_array()) std::memcpy(co.first->byte_array(), co.second->host_ptr(), co.first->size());
  }
  temps.clear();
  copy_out.clear();
  complete(rc, dur);
}

// Completion is detected on the pinned HostCompletion record the kernel writes last
// (retcode, timestamps, then seq after a system fence): no CUDA event per call.
static inline bool hc_done(const HostCompletion *hc, uint32_t seq) { return hc->seq == seq; }

void CudaRequest::wait() {
  if (status() == operationStatus::COMPLETED) return;
  if (!immediate) {
    const HostCompletion *hc = &dev->hc_host_[slot];
    // short spin for latency, then let the driver block on the stream
    const auto t0 = std::chrono::steady_clock::now();
    while (!hc_done(hc, seq)) {
      if (std::chrono::steady_clock::now() - t0 <= std::chrono::microseconds(200)) continue;
      if (unordered) {
        // engine call that does not hold its stream (asynchronous point to point): it may stay parked for as long
        // as the peer takes; the engine itself retires it with RECEIVE_TIMEOUT_ERROR when its wait budget is spent
        std::this_thread::sleep_for(std::chrono::microseconds(20));
        continue;
      }
      cudaSetDevice(dev->device());
      cudaError_t e = cudaStreamSynchronize(stream);
      if (e != cudaSuccess) {
        complete(DMA_INTERNAL_ERROR, 0);
        throw std::runtime_error(std::string("CUDA error while waiting for a call: ") + cudaGetErrorString(e));
      }
      // the stream has drained: the record must be there (engine mode: the proxy waited for it)
      const auto t1 = std::chrono::steady_clock::now();
      while (!hc_done(hc, seq) && std::chrono::steady_clock::now() - t1 < std::chrono::seconds(2)) std::this_thread::yield();
      break;
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  finish();
}

bool CudaRequest::wait(std::chrono::milliseconds timeout) {
  auto deadline = std::chrono::steady_clock::now() + timeout;
  while (!test()) {
    if (std::chrono::steady_clock::now() > deadline) return false;
    std::this_thread::sleep_for(std::chrono::microseconds(20));
  }
  return true;
}

bool CudaRequest::test() {
  if (status() == operationStatus::COMPLETED) return true;
  if (!immediate) {
    if (!hc_done(&dev->hc_host_[slot], seq)) return false;
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  finish();
  return true;
}

// ------------------------------------------------------------------- device
CudaDevice::CudaDevice(std::shared_ptr<Oob> oob, const CudaConfig &cfg) : oob_(std::move(oob)), cfg_(cfg) {
  ACCL_CUDART(cudaSetDevice(cfg_.device));
  heap_.reset(new SymHeap(*oob_, cfg_.device, cfg_.heap_bytes, cfg_.multicast));
  if (heap_->bytes() < CTRL_BYTES * 2) throw std::runtime_error("symmetric heap too small");
  alloc_.reset(new RangeAllocator(CTRL_BYTES, heap_->bytes() - CTRL_BYTES));
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  ACCL_CUDART(cudaStreamCreateWithPriority(&stream_, cudaStreamNonBlocking, prio_hi));
  world_.window = heap_->window();
  world_.mc = heap_->mc_base();
  world_.heap_bytes = heap_->bytes();
  world_.world = static_cast<uint32_t>(heap_->world());
  world_.rank = static_cast<uint32_t>(heap_->rank());
  shadow_.assign(exchmem::SIZE_WORDS, 0);
  uint32_t hwid = CAP_DMA | CAP_ARITH | CAP_COMPRESSION | CAP_RENDEZVOUS | CAP_FP8 | CAP_TCGEN05 | CAP_STREAMS;
  if (heap_->has_multicast()) hwid |= CAP_NVLS_MULTICAST;
  if (cfg_.engine) hwid |= CAP_PERSISTENT_ENGINE;
  shadow_[exchmem::HWID / 4] = hwid;
  ACCL_CUDART(cudaHostAlloc(reinterpret_cast<void **>(&hc_host_), sizeof(HostCompletion) * N_REQ_SLOTS,
                            cudaHostAllocMapped | cudaHostAllocPortable));
  std::memset(hc_host_, 0, sizeof(HostCompletion) * N_REQ_SLOTS);
  ACCL_CUDART(cudaHostGetDevicePointer(reinterpret_cast<void **>(&hc_dev_), hc_host_, 0));
  slot_owner_.assign(N_REQ_SLOTS, nullptr);
  // Symmetric infrastructure areas: allocated first and in the same order by every rank, so each sits at the same
  // offset in every heap.  Sizes derive from the heap size (identical everywhere) unless configured.
  {
    // device-side stream ports
    size_t cap = STREAM_FIFO_BYTES;
    while (cap > (4u << 10) && cap * N_STRM_PORTS > heap_->bytes() / 16) cap >>= 1;
    strm_area_ = allocate(cap * N_STRM_PORTS, bufferKind::p2p);
    world_.strm_off = strm_area_->device_addr();
    world_.strm_cap = cap;
    // staging of the one-way protocols: [bank][parity][source][region]; budget: a quarter of the heap
    const size_t regions = static_cast<size_t>(N_BANKS) * 2 * world_.world;
    const size_t budget = heap_->bytes() / 4 / regions;
    size_t ll = cfg_.ll_bytes ? cfg_.ll_bytes : std::min<size_t>(2u << 20, budget / 2);
    size_t stg = cfg_.stage_bytes ? cfg_.stage_bytes : std::min<size_t>(2u << 20, budget - std::min(budget, ll));
    ll &= ~static_cast<size_t>(4095);
    stg &= ~static_cast<size_t>(4095);
    if (ll >= (4u << 10) * STG_CH / 8 && stg >= (4u << 10)) {
      ll_area_ = allocate(stg_area_bytes(world_.world, ll), bufferKind::p2p);
      stg_area_ = allocate(stg_area_bytes(world_.world, stg), bufferKind::p2p);
      world_.ll_off = ll_area_->device_addr();
      world_.ll_bytes = ll;
      world_.stg_off = stg_area_->device_addr();
      world_.stg_bytes = stg;
    }
    // scratch of the write-only rooted reduce
    const size_t scr = std::min<size_t>(64u << 20, heap_->bytes() / 16) & ~static_cast<size_t>(4095);
    scr_area_ = allocate(scr, bufferKind::p2p);
    world_.scr_off = scr_area_->device_addr();
    world_.scr_bytes = scr;
  }
  apply_env_tuning();
  preload_engine_kernels();
  preload_gemm_rs_kernels();
  preload_vadd_kernels();
  (void)plugin_scratch(16u << 10); // allocate now: cudaMalloc later could stall behind a running engine kernel
  ACCL_CUDART(launch_reset_ctrl(world_, stream_));
  ACCL_CUDART(cudaStreamSynchronize(stream_));
  oob_->barrier(); // nobody signals a peer whose control block is not zeroed yet
  if (cfg_.engine) engine_.reset(new Engine(*this));
}

CudaDevice::~CudaDevice() {
  heap_pool_detach(this);
  cudaSetDevice(cfg_.device);
  engine_.reset();
  cudaStreamSynchronize(stream_);
  egr_area_.reset();
  strm_area_.reset();
  stg_area_.reset();
  ll_area_.reset();
  scr_area_.reset();
  slot_owner_.clear();
  if (hc_host_) cudaFreeHost(hc_host_);
  heap_.reset();
  if (h2d_stream_) cudaStreamDestroy(h2d_stream_);
  if (d2h_stream_) cudaStreamDestroy(d2h_stream_);
  if (stream_) cudaStreamDestroy(stream_);
}

void CudaDevice::attach(int world_size, int local_rank) {
  if (world_size > heap_->world()) throw std::invalid_argument("CudaDevice: more ranks than the heap was built for");
  (void)local_rank;
}

std::string CudaDevice::describe() {
  std::ostringstream o;
  o << "CudaDevice rank " << heap_->rank() << "/" << heap_->world() << " gpu " << cfg_.device << " heap "
    << (heap_->bytes() >> 20) << " MiB nvls=" << (heap_->has_multicast() ? "yes" : "no");
  if (!heap_->has_multicast()) o << " (" << heap_->multicast_note() << ")";
  o << " mode=" << (cfg_.engine ? "engine" : "direct") << " max_ctas=" << cfg_.max_ctas;
  if (engine_) o << " engine_workers=" << engine_->workers();
  o << " staging=" << (world_.stg_bytes >> 10) << "K ll=" << (world_.ll_bytes >> 10) << "K";
  return o.str();
}

void *CudaDevice::plugin_scratch(size_t bytes) {
  if (bytes > plugin_scratch_bytes_) {
    cudaSetDevice(cfg_.device);
    if (plugin_scratch_) throw std::runtime_error("plugin scratch cannot grow while in use");
    const size_t cap = std::max<size_t>(bytes, 16u << 10);
    ACCL_CUDART(cudaMalloc(&plugin_scratch_, cap));
    ACCL_CUDART(cudaMemset(plugin_scratch_, 0, cap));
    plugin_scratch_bytes_ = cap;
  }
  return plugin_scratch_;
}

void CudaDevice::printDebug() { ACCL_ERROR_LOG(debug_state()); }

// protocol counters of my control block, for post-mortems
std::string CudaDevice::debug_state() {
  cudaSetDevice(cfg_.device);
  std::vector<char> buf(sizeof(Ctrl));
  cudaMemcpy(buf.data(), heap_->local(), sizeof(Ctrl), cudaMemcpyDeviceToHost);
  const Ctrl *c = reinterpret_cast<const Ctrl *>(buf.data());
  std::ostringstream o;
  o << describe() << "\n";
  for (uint32_t p = 0; p < world_.world; ++p) {
    if (p == world_.rank) continue;
    o << " peer " << p << ":";
    for (int b = 0; b < N_BANKS; ++b) {
      const PadBank &pb = c->pad[b];
      const StageBank &sb = c->stg[b];
      if (!pb.sent[0][p] && !pb.sig[0][p] && !sb.sent[0][p] && !sb.recvd[0][p] && !pb.sent[MAX_CH - 2][p]) continue;
      o << " bank" << b << "[sync0 sent=" << pb.sent[0][p] << " exp=" << pb.expect[0][p] << " sig=" << pb.sig[0][p]
        << " | eng sent=" << pb.sent[MAX_CH - 2][p] << " exp=" << pb.expect[MAX_CH - 2][p] << " sig=" << pb.sig[MAX_CH - 2][p]
        << " | stg0 sent=" << sb.sent[0][p] << " recvd=" << sb.recvd[0][p] << " sig=" << sb.sig[0][p] << " ack=" << sb.ack[0][p] << "]";
    }
    o << " egr0[sent=" << c->egr_sent[0][p] << " ack=" << c->egr_ack[0][p] << " exp=" << c->egr_expect[0][p]
      << " sig=" << c->egr_sig[0][p] << "] notes[posted=" << c->note_posted[p] << "]\n";
  }
  o << " engine: cmd_tail=" << c->cmd_tail << " fetched=" << c->cmd_fetched << " moves=" << c->move_tail
    << " calls_done=" << c->eng_calls_done << " parks=" << c->eng_parks << "\n";
  return o.str();
}

uint32_t CudaDevice::timeout_us() const {
  // TIMEOUT register counts units of 32 µs on this backend (1e6 -> 32 s): GPU
  // ranks of different processes may reach their first call seconds apart
  const uint64_t t = static_cast<uint64_t>(shadow_[exchmem::TIMEOUT / 4]) * 32;
  return static_cast<uint32_t>(std::min<uint64_t>(t ? t : 32000000ull, 0xFFFFFFFFull));
}

val_t CudaDevice::read(addr_t off) {
  if (off >= exchmem::SIZE_BYTES || (off & 3)) throw std::out_of_range("exchange memory read out of range");
  // sequence counters live in the control block, not in the shadow
  if (off >= exchmem::COMM_BASE) {
    const uint32_t rel = static_cast<uint32_t>(off - exchmem::COMM_BASE);
    const uint32_t ci = rel / exchmem::COMM_STRIDE, w = (rel % exchmem::COMM_STRIDE) / 4;
    if (w >= 2) {
      const uint32_t r = (w - 2) / exchmem::COMM_RANK_WORDS, f = (w - 2) % exchmem::COMM_RANK_WORDS;
      if (f == exchmem::CR_INBOUND_SEQ || f == exchmem::CR_OUTBOUND_SEQ) {
        const uint32_t g = shadow_[exchmem::comm_rank_offset(ci, r, exchmem::CR_SESSION) / 4];
        if (g < static_cast<uint32_t>(ACCL_MAX_RANKS)) {
          std::lock_guard<std::mutex> lk(m_);
          cudaSetDevice(cfg_.device);
          Ctrl *c = reinterpret_cast<Ctrl *>(heap_->local());
          uint32_t v = 0;
          const uint32_t *src = f == exchmem::CR_INBOUND_SEQ ? &c->egr_expect[0][g] : &c->egr_sent[0][g];
          cudaMemcpy(&v, src, 4, cudaMemcpyDeviceToHost);
          return v;
        }
      }
    }
  }
  return shadow_[off / 4];
}

void CudaDevice::sync_ctrl_word(uint32_t off) {
  cudaSetDevice(cfg_.device);
  Ctrl *c = reinterpret_cast<Ctrl *>(heap_->local());
  ACCL_CUDART(cudaMemcpyAsync(&c->exch[off / 4], &shadow_[off / 4], 4, cudaMemcpyHostToDevice, stream_));
}

void CudaDevice::write(addr_t off, val_t val) {
  if (off >= exchmem::SIZE_BYTES || (off & 3)) throw std::out_of_range("exchange memory write out of range");
  std::lock_guard<std::mutex> lk(m_);
  shadow_[off / 4] = val;
  // device-side readers (plugins, engine) see the same block
  sync_ctrl_word(static_cast<uint32_t>(off));
}

std::shared_ptr<BufferStorage> CudaDevice::allocate(size_t bytes, bufferKind kind) {
  return std::make_shared<CudaStorage>(this, bytes, kind, nullptr);
}
std::shared_ptr<BufferStorage> CudaDevice::wrap_host(void *host_ptr, size_t bytes) {
  return std::make_shared<CudaStorage>(this, bytes, bufferKind::device, host_ptr);
}

std::shared_ptr<BufferStorage> CudaDevice::wrap_device(void *dev_ptr, size_t bytes) {
  const char *p = static_cast<const char *>(dev_ptr);
  if (!heap_->contains(p) || !heap_->contains(p + (bytes ? bytes - 1 : 0)))
    throw std::invalid_argument("wrap_device: the memory is not inside this rank's symmetric heap (allocate it from the heap pool)");
  return std::make_shared<CudaStorage>(this, bytes, static_cast<uint64_t>(heap_->offset_of(p)));
}

// (re)build the eager slot area from the geometry in exchange memory
void CudaDevice::setup_eager_area() {
  const uint32_t slot = std::max<uint32_t>(16, (shadow_[exchmem::EAGER_RX_BUF_SIZE / 4] + 15) & ~15u);
  const uint32_t depth = std::min<uint32_t>(std::max<uint32_t>(shadow_[exchmem::EAGER_RX_BUF_COUNT / 4], 2), EGR_DEPTH_MAX);
  egr_area_.reset();
  // fp8 block scaling appends scales: leave headroom of 1/8 + 16 bytes per slot
  const uint32_t slot_alloc = (slot + slot / 8 + 16 + 15) & ~15u;
  egr_area_ = allocate(egr_area_bytes(world_.world, depth, slot_alloc), bufferKind::p2p);
  world_.egr_off = egr_area_->device_addr();
  world_.egr_depth = depth;
  world_.egr_slot_bytes = slot_alloc;
}

uint32_t CudaDevice::host_config(const CallDesc &d) {
  switch (static_cast<cfgFunc>(d.function)) {
  case cfgFunc::reset_periph: {
    cudaSetDevice(cfg_.device);
    if (engine_) engine_->stop();
    cudaStreamSynchronize(stream_);
    launch_reset_ctrl(world_, stream_);
    cudaStreamSynchronize(stream_);
    if (engine_) engine_->clients_reset();
    for (auto &r : slot_owner_) r.reset();
    shadow_[exchmem::CFGRDY / 4] = 0;
    shadow_[exchmem::PKT_ENABLED / 4] = 0;
    return 0;
  }
  case cfgFunc::enable_pkt:
    if (engine_) engine_->stop(); // it restarts with the new slot geometry
    setup_eager_area();
    shadow_[exchmem::PKT_ENABLED / 4] = 1;
    return 0;
  case cfgFunc::set_timeout:
    shadow_[exchmem::TIMEOUT / 4] = d.count;
    return 0;
  case cfgFunc::set_max_eager_msg_size:
    if (d.count < shadow_[exchmem::EAGER_RX_BUF_SIZE / 4]) return EAGER_THRESHOLD_INVALID;
    shadow_[exchmem::MAX_EAGER_SIZE / 4] = d.count;
    return 0;
  case cfgFunc::set_max_rendezvous_msg_size:
    if (d.count <= shadow_[exchmem::MAX_EAGER_SIZE / 4]) return RENDEZVOUS_THRESHOLD_INVALID;
    shadow_[exchmem::MAX_RENDEZVOUS_SIZE / 4] = d.count;
    return 0;
  }
  return COLLECTIVE_NOT_IMPLEMENTED;
}

// ------------------------------------------------------------------ options
namespace {
struct Option {
  const char *name;
  bool runtime; // may change after construction (set_tuning / get_tuning / ACCL_TUNE)
  void (*set)(CudaConfig &c, long v, bool running);
  long (*get)(const CudaConfig &c); // run-time options only
};

// options stored as they are given
template <auto F> void put(CudaConfig &c, long v, bool) { c.*F = static_cast<std::decay_t<decltype(c.*F)>>(v); }
template <auto F> long get(const CudaConfig &c) { return static_cast<long>(c.*F); }
template <uint8_t Tune::*F> long get_tune(const CudaConfig &c) { return c.tune.*F; }

const Option OPTIONS[] = {
    {"heap_mb", false, [](CudaConfig &c, long v, bool) { c.heap_bytes = static_cast<size_t>(v) << 20; }, nullptr},
    {"multicast", false, put<&CudaConfig::multicast>, nullptr},
    {"engine", false, put<&CudaConfig::engine>, nullptr},
    {"engine_workers", false, put<&CudaConfig::engine_workers>, nullptr},
    {"engine_idle_us", false, put<&CudaConfig::engine_idle_us>, nullptr},
    {"oneshot_kb", false, [](CudaConfig &c, long v, bool) { c.oneshot_max_bytes = static_cast<size_t>(v) << 10; }, nullptr},
    {"nvls_ops", false, [](CudaConfig &c, long v, bool) { if (v >= 0) c.nvls_ops = static_cast<uint32_t>(v); }, nullptr}, // < 0: default
    {"stage_kb", false, [](CudaConfig &c, long v, bool) { c.stage_bytes = static_cast<size_t>(v) << 10; }, nullptr},
    {"ll_kb", false, [](CudaConfig &c, long v, bool) { c.ll_bytes = static_cast<size_t>(v) << 10; }, nullptr},
    {"host_pipeline_chunk_kb", false, [](CudaConfig &c, long v, bool) { c.host_pipeline_chunk = static_cast<size_t>(v) << 10; }, nullptr},
    // A live device keeps max_ctas below the sync channels of the engine and of the GEMM plugin (the two last ones);
    // construction accepts up to all of them, and the benchmarks run with 128.
    {"max_ctas", true, [](CudaConfig &c, long v, bool running) { c.max_ctas = static_cast<int>(running ? std::max(1l, std::min<long>(MAX_CH - 2, v)) : v); }, get<&CudaConfig::max_ctas>},
    {"nvls_min_ranks", true, put<&CudaConfig::nvls_min_ranks>, get<&CudaConfig::nvls_min_ranks>},
    {"nvls_ctas", true, put<&CudaConfig::nvls_ctas>, get<&CudaConfig::nvls_ctas>},
    {"hybrid_16ths", true, [](CudaConfig &c, long v, bool) { c.tune.hybrid_16ths = static_cast<uint8_t>(std::max(0l, std::min(15l, v))); }, get_tune<&Tune::hybrid_16ths>},
    {"nvls_unroll", true, [](CudaConfig &c, long v, bool) { c.tune.nvls_unroll = static_cast<uint8_t>(v == 2 || v == 8 || v == 16 ? v : 4); }, get_tune<&Tune::nvls_unroll>},
    {"reduce_push", true, [](CudaConfig &c, long v, bool) { c.tune.reduce_push = static_cast<uint8_t>(v < 0 || v > 2 ? 0 : v); }, get_tune<&Tune::reduce_push>},
    {"bcast_flags", true, [](CudaConfig &c, long v, bool) { c.tune.bcast_flags = static_cast<uint8_t>(v < 0 || v > 2 ? 0 : v); }, get_tune<&Tune::bcast_flags>},
    {"split_phases", true, [](CudaConfig &c, long v, bool) { c.tune.split_phases = v ? 1 : 0; }, get_tune<&Tune::split_phases>},
    {"ll_max_bytes", true, put<&CudaConfig::ll_max_bytes>, get<&CudaConfig::ll_max_bytes>},
    {"ll_oneshot_max", true, put<&CudaConfig::ll_oneshot_max>, get<&CudaConfig::ll_oneshot_max>},
    {"oneshot_max_bytes", true, put<&CudaConfig::oneshot_max_bytes>, get<&CudaConfig::oneshot_max_bytes>},
    {"wire_min_bytes", true, put<&CudaConfig::wire_min_bytes>, get<&CudaConfig::wire_min_bytes>},
    {"staged_max_bytes", true, put<&CudaConfig::staged_max_bytes>, get<&CudaConfig::staged_max_bytes>},
    {"stream_loopback", true, put<&CudaConfig::stream_loopback>, get<&CudaConfig::stream_loopback>},
};

const Option *find_option(const std::string &name) {
  for (const Option &o : OPTIONS) if (name == o.name) return &o;
  return nullptr;
}
} // namespace

bool set_option(CudaConfig &c, const std::string &name, long value, bool running) {
  const Option *o = find_option(name);
  if (!o || (running && !o->runtime)) return false;
  o->set(c, value, running);
  return true;
}

PlanCfg make_plan_cfg(const CudaConfig &cfg, bool has_mc, uint32_t heap_world, size_t stg_bytes, size_t ll_bytes,
                      uint32_t engine_workers) {
  PlanCfg c;
  std::memset(&c, 0, sizeof(c));
  c.max_ctas = static_cast<uint32_t>(cfg.max_ctas);
  if (engine_workers) c.max_ctas = std::min(c.max_ctas, engine_workers);
  c.nvls_min_ranks = static_cast<uint32_t>(cfg.nvls_min_ranks);
  c.has_mc = has_mc ? 1u : 0u;
  c.heap_world = heap_world;
  c.oneshot_max_bytes = cfg.oneshot_max_bytes;
  c.nvls_ops = cfg.nvls_ops;
  c.nvls_ctas = static_cast<uint32_t>(cfg.nvls_ctas);
  c.stg_bytes = static_cast<uint32_t>(stg_bytes);
  c.ll_bytes = static_cast<uint32_t>(ll_bytes);
  c.ll_max_bytes = static_cast<uint32_t>(cfg.ll_max_bytes);
  c.ll_oneshot_max = static_cast<uint32_t>(cfg.ll_oneshot_max);
  c.wire_min_bytes = static_cast<uint32_t>(cfg.wire_min_bytes);
  c.staged_max_bytes = static_cast<uint32_t>(cfg.staged_max_bytes);
  c.engine_mode = engine_workers ? 1u : 0u;
  c.tune = cfg.tune;
  return c;
}

PlanCfg CudaDevice::plan_cfg() const {
  return make_plan_cfg(cfg_, heap_->has_multicast(), static_cast<uint32_t>(heap_->world()), world_.stg_bytes,
                       world_.ll_bytes, engine_ ? static_cast<uint32_t>(engine_->workers()) : 0u);
}

bool CudaDevice::set_tuning(const std::string &name, long v) {
  std::lock_guard<std::mutex> lk(m_);
  return set_option(cfg_, name, v, true);
}

long CudaDevice::get_tuning(const std::string &name) const {
  if (name == "stage_bytes") return static_cast<long>(world_.stg_bytes);
  if (name == "ll_bytes") return static_cast<long>(world_.ll_bytes);
  const Option *o = find_option(name);
  return o && o->runtime ? o->get(cfg_) : -1;
}

// ACCL_TUNE="name=value,name=value": experiment without rebuilding (must be identical on every rank)
void CudaDevice::apply_env_tuning() {
  const char *e = std::getenv("ACCL_TUNE");
  if (!e) return;
  std::string str(e);
  size_t pos = 0;
  while (pos < str.size()) {
    size_t end = str.find(',', pos);
    if (end == std::string::npos) end = str.size();
    const std::string kv = str.substr(pos, end - pos);
    const size_t eq = kv.find('=');
    if (eq != std::string::npos && !set_tuning(kv.substr(0, eq), std::atol(kv.substr(eq + 1).c_str())))
      ACCL_ERROR_LOG("ACCL_TUNE: unknown knob '" + kv.substr(0, eq) + "'");
    pos = end + 1;
  }
}

void CudaDevice::drain_locked() {
  for (auto &r : slot_owner_)
    if (r && r->status() != operationStatus::COMPLETED) r->wait();
}
void CudaDevice::drain() {
  std::vector<std::shared_ptr<CudaRequest>> pending;
  {
    std::lock_guard<std::mutex> lk(m_);
    for (auto &r : slot_owner_)
      if (r && r->status() != operationStatus::COMPLETED) pending.push_back(r);
  }
  for (auto &r : pending) r->wait();
}

bool CudaDevice::build_work_item(const Options &o, const CallDesc &d, WorkItem &w, uint32_t &err) {
  (void)o;
  std::memset(&w, 0, sizeof(w));
  const uint32_t e = build_work_item_hd(shadow_.data(), plan_cfg(), world_.world, d, timeout_us(), w);
  err |= e;
  return e == 0;
}

ACCLRequest *CudaDevice::start(const Options &options) {
  for (ACCLRequest *dep : options.waitfor)
    if (dep) wait(dep);
  auto req = std::make_shared<CudaRequest>(options);
  req->dev = this;
  req->desc = make_call_desc(options);
  ACCLRequest *h = requests_.add(req);
  std::lock_guard<std::mutex> lk(m_);
  ACCL_CUDART(cudaSetDevice(cfg_.device));
  if (options.scenario == operation::config) {
    req->immediate = true;
    const uint32_t rc = host_config(req->desc);
    shadow_[exchmem::RETCODE / 4] = rc;
    req->complete(rc, 0);
    return h;
  }
  cudaStream_t s = options.stream ? static_cast<cudaStream_t>(options.stream) : op_stream();
  // ---- host-resident operands are staged through heap scratch
  Options o = options;
  std::unique_ptr<BaseBuffer> tmp_bufs[3];
  BaseBuffer **ops[3] = {&o.addr_0, &o.addr_1, &o.addr_2};
  const hostFlags hbits[3] = {hostFlags::OP0_HOST, hostFlags::OP1_HOST, hostFlags::RES_HOST};
  for (int i = 0; i < 3; ++i) {
    if (!any(options.host_flags & hbits[i]) || !*ops[i] || (*ops[i])->is_dummy()) continue;
    BaseBuffer *hb = *ops[i];
    auto st = allocate(hb->size(), bufferKind::device);
    req->temps.push_back(st);
    tmp_bufs[i].reset(new BaseBuffer(st, 0, hb->size(), hb->type()));
    if (i < 2) {
      ACCL_CUDART(cudaMemcpyAsync(st->device_ptr(), hb->byte_array(), hb->size(), cudaMemcpyHostToDevice, s));
    } else {
      req->copy_out.emplace_back(hb, st);
    }
    *ops[i] = tmp_bufs[i].get();
  }
  if (!req->temps.empty()) req->desc = make_call_desc(o);

  // ---- stream operands: lower onto the device-side FIFO (pop before / push after the call)
  const bool op0_strm = any(options.stream_flags & streamFlags::OP0_STREAM);
  const bool res_strm = any(options.stream_flags & streamFlags::RES_STREAM);
  std::unique_ptr<BaseBuffer> strm_bufs[2];
  uint64_t push_bytes = 0, push_src = 0;
  uint32_t push_rank = world_.rank;
  bool put_only = false;
  // stream id (TDEST) of a streamed result: the tag of stream_put / recv-to-stream when it is a user id
  const uint32_t res_strm_id = (!cfg_.stream_loopback && options.tag >= STREAM_ID_MIN && options.tag <= STREAM_ID_MAX) ? options.tag : 0;
  const bool lowered = op0_strm || res_strm;
  if (lowered && engine_) drain_locked(); // the lowering kernels below are direct launches: they take over the engine's channels
  if (op0_strm || res_strm) {
    const operation sop = options.scenario;
    if (sop != operation::copy && sop != operation::combine && sop != operation::send && sop != operation::recv &&
        sop != operation::reduce) {
      req->immediate = true;
      req->complete(COLLECTIVE_NOT_IMPLEMENTED, 0);
      return h;
    }
    if (op0_strm) {
      const size_t bytes = static_cast<size_t>(options.count) * dtype_bytes(options.data_type_io_0);
      auto st = allocate(bytes, bufferKind::p2p);
      req->temps.push_back(st);
      strm_bufs[0].reset(new BaseBuffer(st, 0, bytes, options.data_type_io_0));
      ACCL_CUDART(launch_stream_pop(world_, st->device_addr(), bytes, 0, timeout_us(), s));
      o.addr_0 = strm_bufs[0].get();
    }
    if (res_strm) {
      const uint32_t ci = o.comm;
      const uint32_t my_comm_rank = shadow_[exchmem::comm_offset(ci) / 4 + 1];
      push_bytes = static_cast<uint64_t>(options.count) * dtype_bytes(options.data_type_io_2 != dataType::none ? options.data_type_io_2 : options.data_type_io_0);
      if (sop == operation::send) {
        // stream_put: the payload goes straight into the destination rank's FIFO, no matching recv
        const uint32_t csize = shadow_[exchmem::comm_offset(ci) / 4];
        if (options.root_src_dst >= csize) {
          req->immediate = true;
          req->complete(CONFIG_SWITCH_ERROR, 0);
          return h;
        }
        push_rank = shadow_[exchmem::comm_rank_offset(ci, options.root_src_dst, exchmem::CR_SESSION) / 4];
        push_src = o.addr_0->address();
        put_only = true;
      } else if (sop == operation::reduce && options.root_src_dst != my_comm_rank) {
        push_bytes = 0; // only the root produces a result
      } else {
        auto st = allocate(push_bytes, bufferKind::p2p);
        req->temps.push_back(st);
        strm_bufs[1].reset(new BaseBuffer(st, 0, push_bytes, options.data_type_io_2));
        o.addr_2 = strm_bufs[1].get();
        push_src = st->device_addr();
      }
    }
    o.stream_flags = streamFlags::NO_STREAM;
    req->desc = make_call_desc(o);
  }

  WorkItem w;
  uint32_t err = 0;
  if (put_only) {
    CallDesc nd = req->desc;
    nd.scenario = static_cast<uint32_t>(operation::nop);
    if (!build_work_item(o, nd, w, err)) err |= CONFIG_SWITCH_ERROR;
  } else if (!build_work_item(o, req->desc, w, err)) {
    err |= CONFIG_SWITCH_ERROR;
  }
  if (err) {
    req->immediate = true;
    req->complete(err, 0);
    return h;
  }
  // ---- CUDA-graph capture: the launch is recorded, nothing executes now — no completion slot, no host-visible
  // record (a replayed kernel must not write a stale sequence number); the graph's own ordering is the completion
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (s != nullptr && s != cudaStreamLegacy) cudaStreamIsCapturing(s, &cap);
  if (cap == cudaStreamCaptureStatusActive) {
    if (push_bytes || engine_ || !req->temps.empty()) {
      req->immediate = true;
      req->complete(COLLECTIVE_NOT_IMPLEMENTED, 0); // only plain direct launches on device-resident operands are capturable
      return h;
    }
    w.req_slot = N_REQ_SLOTS - 1; // record reserved for captured launches (replays are stream ordered)
    w.req_seq = 0;
    ACCL_CUDART(launch_call(world_, w, nullptr, s));
    req->immediate = true;
    req->complete(0, 0);
    return h;
  }
  // ---- completion slot
  const uint32_t slot = next_slot_++ % (N_REQ_SLOTS - 1); // the last record belongs to captured launches
  if (slot_owner_[slot]) slot_owner_[slot]->wait(); // ring wrapped: the old occupant must be done
  slot_owner_[slot] = req;
  req->slot = slot;
  req->seq = next_seq_++;
  if (next_seq_ == 0) next_seq_ = 1;
  w.req_slot = slot;
  w.req_seq = req->seq;
  req->stream = s;
  if (push_bytes) {
    // lowered call: [op (chained)] -> push -> nop that publishes the completion of the whole chain
    if (!put_only) {
      WorkItem first = w;
      first.flags |= WF_CHAIN;
      ACCL_CUDART(launch_call(world_, first, &hc_dev_[slot], s));
    }
    ACCL_CUDART(launch_stream_push(world_, push_rank, push_src, push_bytes, res_strm_id, timeout_us(), s));
    WorkItem tail;
    CallDesc nd = req->desc;
    nd.scenario = static_cast<uint32_t>(operation::nop);
    uint32_t e2 = 0;
    build_work_item(o, nd, tail, e2);
    tail.req_slot = slot;
    tail.req_seq = req->seq;
    ACCL_CUDART(launch_call(world_, tail, &hc_dev_[slot], s));
  } else if (engine_ && !lowered) {
    // asynchronous point-to-point calls must not hold the stream: the matching call of the peer may be queued
    // behind them on ITS stream (send/send then recv/recv); everything else is stream ordered like a launch
    const bool p2p = options.scenario == operation::send || options.scenario == operation::recv;
    req->unordered = p2p;
    engine_->submit(w, &hc_dev_[slot], s, !p2p);
  } else {
    ACCL_CUDART(launch_call(world_, w, &hc_dev_[slot], s));
  }
  req->set_status(operationStatus::EXECUTING);
  return h;
}

// Blocking all-reduce on host-resident operands, software-pipelined: chunk i is copied in on
// the H2D engine while chunk i-1 is being reduced over NVLink and chunk i-2 is copied out on
// the D2H engine (PCIe is full duplex).  Same chunking on every rank by construction.
ACCLRequest *CudaDevice::call_host_pipelined(const Options &options) {
  if (options.scenario != operation::allreduce || cfg_.host_pipeline_chunk == 0) return nullptr;
  BaseBuffer *src = options.addr_0, *dst = options.addr_2;
  if (!src || !dst || src->is_dummy() || dst->is_dummy() || src->is_host_only() || dst->is_host_only()) return nullptr;
  if (options.compression_flags != compressionFlags::NO_COMPRESSION || !src->byte_array() || !dst->byte_array()) return nullptr;
  const size_t es = dtype_bytes(src->type());
  const size_t total = options.count;
  size_t chunk = cfg_.host_pipeline_chunk / es;
  if (total * es < 2 * cfg_.host_pipeline_chunk) return nullptr; // too small to be worth pipelining
  ACCL_CUDART(cudaSetDevice(cfg_.device));
  if (!h2d_stream_) {
    ACCL_CUDART(cudaStreamCreateWithFlags(&h2d_stream_, cudaStreamNonBlocking));
    ACCL_CUDART(cudaStreamCreateWithFlags(&d2h_stream_, cudaStreamNonBlocking));
  }
  cudaStream_t main = options.stream ? static_cast<cudaStream_t>(options.stream) : op_stream();
  const size_t nchunks = (total + chunk - 1) / chunk;
  std::vector<cudaEvent_t> ev_in(nchunks), ev_out(nchunks);
  std::vector<ACCLRequest *> reqs;
  cudaEvent_t ev_start;
  ACCL_CUDART(cudaEventCreateWithFlags(&ev_start, cudaEventDisableTiming));
  ACCL_CUDART(cudaEventRecord(ev_start, main)); // staging starts after whatever the caller queued before
  ACCL_CUDART(cudaStreamWaitEvent(h2d_stream_, ev_start, 0));
  uint32_t rc = 0;
  uint64_t dur = 0;
  for (size_t c = 0; c < nchunks; ++c) {
    const size_t e0 = c * chunk, n = std::min(chunk, total - e0);
    auto s = src->slice(e0, e0 + n);
    auto d = dst->slice(e0, e0 + n);
    ACCL_CUDART(cudaEventCreateWithFlags(&ev_in[c], cudaEventDisableTiming));
    ACCL_CUDART(cudaEventCreateWithFlags(&ev_out[c], cudaEventDisableTiming));
    ACCL_CUDART(cudaMemcpyAsync(s->device_ptr(), s->byte_array(), n * es, cudaMemcpyHostToDevice, h2d_stream_));
    ACCL_CUDART(cudaEventRecord(ev_in[c], h2d_stream_));
    ACCL_CUDART(cudaStreamWaitEvent(main, ev_in[c], 0));
    Options o = options;
    o.addr_0 = s.get();
    o.addr_2 = d.get();
    o.count = static_cast<unsigned int>(n);
    o.stream = main;
    reqs.push_back(start(o));
    ACCL_CUDART(cudaEventRecord(ev_out[c], main));
    ACCL_CUDART(cudaStreamWaitEvent(d2h_stream_, ev_out[c], 0));
    ACCL_CUDART(cudaMemcpyAsync(d->byte_array(), d->device_ptr(), n * es, cudaMemcpyDeviceToHost, d2h_stream_));
  }
  ACCL_CUDART(cudaStreamSynchronize(d2h_stream_));
  for (ACCLRequest *r : reqs) {
    wait(r);
    rc |= get_retcode(r);
    dur += get_duration(r);
    free_request(r);
  }
  for (size_t c = 0; c < nchunks; ++c) {
    cudaEventDestroy(ev_in[c]);
    cudaEventDestroy(ev_out[c]);
  }
  cudaEventDestroy(ev_start);
  auto req = std::make_shared<CudaRequest>(options);
  req->dev = this;
  req->immediate = true;
  req->complete(rc, dur);
  return requests_.add(req);
}

ACCLRequest *CudaDevice::call(const Options &options) {
  ACCLRequest *h = start(options);
  wait(h);
  return h;
}

void CudaDevice::wait(ACCLRequest *request) {
  auto r = requests_.find(request);
  if (!r) throw std::invalid_argument("wait: unknown request");
  r->wait();
}
bool CudaDevice::wait(ACCLRequest *request, std::chrono::milliseconds timeout) {
  auto r = requests_.find(request);
  if (!r) throw std::invalid_argument("wait: unknown request");
  return r->wait(timeout);
}
bool CudaDevice::test(ACCLRequest *request) {
  auto r = requests_.find(request);
  if (!r) throw std::invalid_argument("test: unknown request");
  return r->test();
}
void CudaDevice::free_request(ACCLRequest *request) {
  auto r = std::dynamic_pointer_cast<CudaRequest>(requests_.find(request));
  if (r) {
    std::lock_guard<std::mutex> lk(m_);
    if (r->status() != operationStatus::COMPLETED) {
      // still in flight: keep the slot owner alive, drop only the user handle
    } else {
      if (slot_owner_[r->slot] == r) slot_owner_[r->slot] = nullptr;
    }
  }
  requests_.erase(request);
}
val_t CudaDevice::get_retcode(ACCLRequest *request) {
  auto r = requests_.find(request);
  if (!r) throw std::invalid_argument("get_retcode: unknown request");
  return r->retcode();
}
uint64_t CudaDevice::get_duration(ACCLRequest *request) {
  auto r = requests_.find(request);
  if (!r) throw std::invalid_argument("get_duration: unknown request");
  return r->duration_ns();
}

std::vector<std::unique_ptr<CudaDevice>> make_local_world(const std::vector<int> &devices, const CudaConfig &base) {
  const int W = static_cast<int>(devices.size());
  auto oobs = LocalOob::create(W);
  std::vector<std::unique_ptr<CudaDevice>> out(static_cast<size_t>(W));
  std::vector<std::string> errs(static_cast<size_t>(W));
  std::vector<std::thread> ts;
  for (int r = 0; r < W; ++r)
    ts.emplace_back([&, r] {
      try {
        CudaConfig c = base;
        c.device = devices[static_cast<size_t>(r)];
        out[static_cast<size_t>(r)].reset(new CudaDevice(oobs[static_cast<size_t>(r)], c));
      } catch (const std::exception &e) {
        errs[static_cast<size_t>(r)] = e.what();
      }
    });
  for (auto &t : ts) t.join();
  for (auto &e : errs)
    if (!e.empty()) throw std::runtime_error("make_local_world: " + e);
  return out;
}

} // namespace cuda
} // namespace accl
