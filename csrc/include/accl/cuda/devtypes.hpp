// Structures shared by the CUDA backend's host code and its sm_100a kernels:
// geometry of the symmetric heap's control block, the work item a kernel
// executes, completion records and the persistent engine's rings.
//
// Mapping to the reference: `Ctrl` is the device-resident equivalent of the
// CCLO's exchange memory + RX-buffer metadata + rendezvous mailbox
// (kernels/cclo/fw/.../ccl_offload_control.h:85-98,292-323); `WorkItem` is the
// decoded 15-word call (ccl_offload_control.c:2319-2373); `Completion` is
// RETVAL + PERFCNT (:2291-2306).
//
// Protocol state is namespaced by *bank*: every communicator is bound to one of
// N_BANKS independent sets of sync pads / staging slots / counters (the bank is
// a hash of the member list, identical on all members), so calls on different
// communicators may be in flight at the same time — on different streams or
// parked side by side inside the engine — without sharing a counter.  The
// reference keeps per-communicator sequence numbers for the same reason
// (ccl_offload_control.h:297-304).
#pragma once
#include <cstdint>

#include "accl/cclo.hpp"
#include "accl/constants.hpp"
#include "accl/exchmem.hpp"

namespace accl {
namespace cuda {

constexpr int N_BANKS = 4;        // independent protocol-state sets (communicators hash onto them)
constexpr int MAX_CH = 128;       // rendezvous sync channels per bank == max CTAs cooperating on one call
constexpr int STG_CH = 32;        // channels of the staged (one-way) protocols per bank
constexpr int EGR_CH = 16;        // channels usable by eager (slot-based) transfers
constexpr int EGR_DEPTH_MAX = 16; // slots per (channel, src): the eager RX buffers
constexpr int N_REQ_SLOTS = 256;  // completion records
constexpr int RING_SLOTS = 128;   // command ring depth
constexpr int P2P_NOTES = 8;      // rendezvous address notes in flight per ordered pair of ranks
constexpr int MAX_ACTIVE = 16;    // calls the engine keeps in flight (running or parked)
constexpr int MOVE_SLOTS = 8;     // control -> worker move ring depth
constexpr int N_STRM_PORTS = 16;  // device-side stream FIFOs per rank
constexpr uint64_t CTRL_BYTES = 2ull << 20; // control block at the start of every heap
constexpr uint64_t INVALID_OFF = ~0ull;

enum Algo : uint32_t {
  ALGO_AUTO = 0,
  ALGO_LOCAL = 1,        // world == 1 / local-only primitive
  ALGO_EAGER = 2,        // push into the peers' eager slots, consume locally (segmented, any dtype / wire dtype)
  ALGO_NVLS = 3,         // multimem.ld_reduce / multimem.st through the NVSwitch
  ALGO_P2P = 4,          // peer loads/stores on the mapped heaps (one-shot or two-shot by op)
  ALGO_P2P_ONESHOT = 5,  // every rank pulls everything (small allreduce without slots)
  ALGO_LL = 6,           // staged one-way exchange, flag carried inside every 8 data bytes (no fence, one hop)
  ALGO_STAGED = 7,       // staged one-way exchange, payload then release-flag; consumer copies / reduces out of staging
  ALGO_WIRE = 8          // wire-compressed two-shot over the scratch area: cast fused into the NVLink stores / loads (compress.cuh)
};

struct SyncRec { // rendezvous "address exchange" record, written by a peer next to its signal
  uint64_t off0;
  uint64_t off2;
  uint32_t kind; // operation code of the sender's call | communicator signature << 8: mismatches are protocol errors
  uint32_t pad;
};

struct EgrHdr { // per-slot message header (the reference's eth_header, minus routing)
  uint32_t tag;
  uint32_t bytes;
  uint32_t elems;
  uint32_t kind; // scenario | wire dtype << 8
};

// rendezvous point-to-point: the receiver posts "write `count` elements tagged `tag` at `addr` of my heap" into
// the SENDER's control block (reference: rendezvous_send_addr, ccl_offload_control.c:142-150); the sender
// matches notes by tag, stores the payload and raises note_done at the receiver (RNDZVS_WR_DONE).
struct P2pNote {
  uint64_t addr;
  uint32_t count;
  uint32_t tag;
  uint32_t dtype;
  uint32_t seq; // written last: note sequence (1-based) of this (receiver -> sender) pair
};

struct Completion {
  uint32_t retcode;
  uint32_t done_ctas;
  unsigned long long t_start; // %globaltimer ns (min over CTAs)
  unsigned long long t_end;   // max over CTAs
  uint32_t seq;               // written last: request sequence this record belongs to
  uint32_t pad;
};

struct StrmPort {
  unsigned long long head;    // bytes published (readable by the consumer)
  unsigned long long tail;    // bytes consumed
  unsigned long long reserve; // bytes reserved by producers (local kernels or peers doing stream_put)
  unsigned long long pad;
};

struct PadBank { // rendezvous sync pads of one bank
  uint32_t sig[MAX_CH][ACCL_MAX_RANKS];    // written by peers
  SyncRec rec[MAX_CH][ACCL_MAX_RANKS];     // written by peers
  uint32_t sent[MAX_CH][ACCL_MAX_RANKS];   // local (single writer: the CTA owning the channel)
  uint32_t expect[MAX_CH][ACCL_MAX_RANKS]; // local
  // one-way "chunk landed" counters of the flag-driven pipelined broadcast
  uint32_t step_sig[MAX_CH][ACCL_MAX_RANKS];  // written by peers: chunks src has delivered to me on this channel
  uint32_t step_seen[MAX_CH][ACCL_MAX_RANKS]; // local: how many of them earlier calls already consumed
  uint32_t step_sent[MAX_CH][ACCL_MAX_RANKS]; // local: chunks I have delivered to dst
};

struct StageBank { // one-way staged exchanges of one bank
  uint32_t sig[STG_CH][ACCL_MAX_RANKS];    // written by peers: messages of src that have landed (ALGO_STAGED)
  uint32_t ack[STG_CH][ACCL_MAX_RANKS];    // written by peers: my messages consumed by dst (credits)
  uint32_t sent[STG_CH][ACCL_MAX_RANKS];   // local: messages pushed to dst
  uint32_t recvd[STG_CH][ACCL_MAX_RANKS];  // local: messages consumed from src
};

// Layout of the first CTRL_BYTES of every rank's heap (same offsets everywhere).
struct Ctrl {
  uint32_t exch[exchmem::SIZE_WORDS]; // exchange memory (host <-> engine configuration block)
  PadBank pad[N_BANKS];
  StageBank stg[N_BANKS];
  // ---- eager slot rings (point-to-point, compressed and rooted small messages)
  uint32_t egr_sig[EGR_CH][ACCL_MAX_RANKS]; // messages arrived from src on channel
  uint32_t egr_ack[EGR_CH][ACCL_MAX_RANKS]; // my messages consumed by dst (credits)
  EgrHdr egr_hdr[EGR_CH][EGR_DEPTH_MAX][ACCL_MAX_RANKS];
  uint32_t egr_sent[EGR_CH][ACCL_MAX_RANKS];
  uint32_t egr_expect[EGR_CH][ACCL_MAX_RANKS];
  // ---- rendezvous point-to-point mailbox
  P2pNote note[ACCL_MAX_RANKS][P2P_NOTES];        // written by receiver r: its pending recvs from me
  uint32_t note_done[ACCL_MAX_RANKS][P2P_NOTES];  // written by sender s: note seq whose payload has landed in my buffer
  uint32_t note_posted[ACCL_MAX_RANKS];           // local (as receiver): notes I posted to s
  uint32_t note_taken[ACCL_MAX_RANKS][P2P_NOTES]; // local (as sender): note seq of r already matched by one of my sends
  // ---- completion records (direct launches)
  Completion comp[N_REQ_SLOTS];
  // ---- persistent engine (engine.cu): configuration, command ring, doorbells
  uint32_t plan_cfg_words[24];    // PlanCfg image (plan.hpp) for device-side planning
  uint32_t engine_timeout_us;
  uint32_t engine_exit;           // workers leave when set
  unsigned long long cmd_tail;    // producers (host proxies, plugin kernels) take tickets here
  unsigned long long cmd_fetched; // entries consumed by the control CTA (survives relaunches)
  unsigned long long cmd_ready[RING_SLOTS];  // slot published: ticket + 1
  unsigned long long cmd_status[RING_SLOTS]; // slot finished: (ticket + 1) | retcode << 32
  unsigned long long move_tail;   // control -> workers: moves issued
  unsigned long long move_done[MOVE_SLOTS];  // worker CTAs that have passed the moves of this slot (monotonic)
  uint32_t move_err[MOVE_SLOTS];  // error bits raised by the workers of the slot's current move
  unsigned long long host_fetched; // commands of host proxies fetched so far (park handshake)
  unsigned long long eng_calls_done;  // statistics: calls retired by the engine
  unsigned long long eng_parks;       // statistics: NOT_READY returns (calls re-queued)
  // ---- device-side stream ports (OP0_STREAM / RES_STREAM operands, stream_put): one byte FIFO per port;
  // stream id s (9..246, the reference's TDEST) is served by port s % N_STRM_PORTS, id 0 (no id) by port 0
  StrmPort strm[N_STRM_PORTS];
  uint32_t strm_err;               // sticky error bits raised by stream helper kernels
  uint32_t clients_done;           // device-side clients (plugin kernels) that have finished, monotonic: the engine parks only
                                   // once this has caught up with the host's count of clients launched (HostRing::clients)
  // ---- opt-in instrumentation (channel 0 only): where a call's time goes.  Read with CudaDevice::debug_state().
  unsigned long long dbg_calls;      // calls executed
  unsigned long long dbg_kernel_ns;  // sum of kernel body durations (run_work entry -> exit)
  unsigned long long dbg_sync_ns;    // of which spent inside chan_sync / pair_sync (flag round trips)
  unsigned long long dbg_syncs;      // number of meetings
};
static_assert(sizeof(Ctrl) <= CTRL_BYTES / 2, "control block too large");

struct DevWorld {
  char *window;        // rank r's heap lives at window + r * heap_bytes
  char *mc;            // NVLS multicast alias of heap offset 0 on every rank (nullptr: none)
  uint64_t heap_bytes;
  uint32_t world;      // ranks sharing the heap
  uint32_t rank;       // my global rank
  uint64_t egr_off;    // heap offset of the eager slot area
  uint32_t egr_depth;  // slots per (channel, src)
  uint32_t egr_slot_bytes;
  uint64_t strm_off;   // heap offset of the device-side stream FIFOs (same on every rank), port p at strm_off + p * strm_cap
  uint64_t strm_cap;   // capacity of one FIFO in bytes (power of two)
  uint64_t stg_off;    // heap offset of the staging area of ALGO_STAGED (same on every rank)
  uint64_t stg_bytes;  // bytes per (bank, parity, source rank)
  uint64_t ll_off;     // heap offset of the staging area of ALGO_LL
  uint64_t ll_bytes;   // bytes per (bank, parity, source rank)
  uint64_t scr_off;    // heap offset of the collective scratch region (same on every rank)
  uint64_t scr_bytes;
};

// tuning knobs that travel with every call (set from CudaConfig / ACCL_TUNE="name=value,..." / Accl.set_tuning)
struct Tune {
  uint8_t hybrid_16ths;  // large NVLS all-reduce: 16ths of every shard handled by the peer two-shot body instead
  uint8_t nvls_unroll;   // 16-byte multimem accesses in flight per thread: 2, 4 (default), 8 or 16
  uint8_t reduce_push;   // rooted reduce: 1 = write-only chunked scheme for large messages, 2 = the root reduces through the switch at every size
  uint8_t bcast_flags;   // large bcast: 1 = one-way chunk flags instead of a meeting per step, 2 = never pipelined (single multicast pass)
  uint8_t split_phases;  // NVLS all-reduce: 1 = reduce-scatter and all-gather halves on disjoint CTA sets
  uint8_t pad[3];
};

struct WorkItem {
  CallDesc desc;
  uint32_t comm_size, comm_rank;
  uint8_t members[ACCL_MAX_RANKS]; // communicator rank -> global rank
  uint32_t algo;
  uint32_t n_ctas;
  uint32_t udtype, cdtype, ratio_log, arith_compressed;
  uint32_t req_slot, req_seq;
  uint32_t timeout_us;
  uint32_t flags;
  uint32_t bank;       // protocol-state bank of the communicator
  uint32_t comm_sig;   // signature of the member list (checked in rendezvous records)
  Tune tune;
  uint64_t scratch_off, scratch_bytes; // per-call scratch inside the heap (compression / staging)
  uint64_t hc_ptr;     // device-visible HostCompletion of a host-issued call (0: none)
};

enum WorkFlags : uint32_t {
  WF_USE_MC = 1u << 0,
  WF_ENGINE = 1u << 1,
  WF_CHAIN = 1u << 2,   // not the last kernel of a lowered call: park the error word instead of publishing completion
  WF_ONESHOT = 1u << 3, // staged all-reduce: every rank receives every block (one hop) instead of reduce-scatter + all-gather
  WF_PLANNED = 1u << 4  // command ring entry carries a planned WorkItem (host proxy); otherwise only `desc` is valid
};

// engine command ring entry: producers (the host's proxy kernels, plugin kernels using accl/device/api.cuh) take
// a ticket in Ctrl::cmd_tail, fill slot ticket % RING_SLOTS and publish it in Ctrl::cmd_ready (the reference's
// client_arbiter: any number of command sources, status routed back to the issuer through cmd_status)
struct CmdSlot {
  WorkItem item;
};

// One wait-free data-movement job handed by the control CTA to the worker CTAs — the reference's DMP move
// instruction (dma_mover.cpp:355-421): everything a mover needs is in the descriptor, nothing in it waits for a peer.
struct MoveDesc {
  WorkItem item;
  uint64_t off0[ACCL_MAX_RANKS], off2[ACCL_MAX_RANKS]; // exchanged buffer offsets by communicator rank
  uint32_t kind;   // MoveKind
  uint32_t n_ctas; // workers that take part
  uint64_t a, b, c; // kind-specific scalars (addresses / byte counts)
};
enum MoveKind : uint32_t {
  MV_BODY = 1, // the data phase of item.desc.scenario (between the entry and exit meetings)
  MV_COPY = 2, // plain copy a -> b of c bytes (absolute addresses; rendezvous send payload)
  MV_WORK = 3  // a whole one-way exchange (ALGO_LL / ALGO_STAGED / ALGO_EAGER collective): waits only for what the
               // peers push when they start the same collective
};

struct EngineArea { // at heap offset CTRL_BYTES / 2
  CmdSlot cmd_ring[RING_SLOTS];
  MoveDesc move_ring[MOVE_SLOTS];
};
static_assert(sizeof(EngineArea) <= CTRL_BYTES / 2, "engine area too large");

// eager slot addressing inside a heap
ACCL_HD uint64_t egr_slot_off(const DevWorld &w, uint32_t ch, uint32_t slot, uint32_t src) {
  return w.egr_off + ((static_cast<uint64_t>(ch) * w.egr_depth + slot) * w.world + src) * w.egr_slot_bytes;
}
ACCL_HD uint64_t egr_area_bytes(uint32_t world, uint32_t depth, uint32_t slot_bytes) {
  return static_cast<uint64_t>(EGR_CH) * depth * world * slot_bytes;
}
// staging areas: [bank][parity][source rank][region bytes]
ACCL_HD uint64_t stg_area_bytes(uint32_t world, uint64_t region_bytes) {
  return static_cast<uint64_t>(N_BANKS) * 2 * world * region_bytes;
}

} // namespace cuda
} // namespace accl
