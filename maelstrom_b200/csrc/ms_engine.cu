// ms_engine.cu -- host side of the C ABI declared in include/maelstrom_b200.h.
// Owns device memory, the endpoint registry, the fault knobs and the round
// loop; all simulation work happens in ms_kernels.cu.  There is no CPU
// fallback: without a usable CUDA device ms_create fails.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "ms_device.cuh"
#include "ms_tree.h"
#include "ms_fressian.h"
#include "ms_json.h"

using namespace msd;

extern "C" {
cudaError_t msk_round_smem_attr(size_t bytes);
size_t msk_round_smem_bytes(uint32_t cap);
int msk_round_occupancy(int threads, size_t smem);
void msk_launch_round(const msd::Params* p, int n_classes, const uint32_t* caps, const int* threads,
                      const int* grids, int with_release, cudaStream_t s, cudaEvent_t before_round,
                      cudaEvent_t after_round, int phases, const cudaStream_t* aux, const cudaEvent_t* aux_ev);
void msk_set_bit(uint32_t* words, size_t word, uint32_t bit, cudaStream_t s);
void msk_barrier(const msd::Params* p, cudaStream_t s);
void msk_journal_expand(const msd::Params* p, uint64_t r0, uint32_t n_rounds, uint64_t first, uint64_t count,
                        void* out_ev, void* out_body, int n_sms, cudaStream_t s);
size_t msk_stream_plan_bytes();
void msk_stream_batch(const msd::Params* p, void* plan, uint64_t cap_events, uint32_t cap_rounds, ms_jround* rows,
                      void* out, ms_jbatch* hdr, int format, int n_sms, cudaStream_t s, uint32_t parity);
void msk_stream_apply(const msd::Params* p, const void* plan, cudaStream_t s, uint32_t parity);
}

static thread_local std::string g_err;

// body.type names of the protocol (doc/workloads.md, doc/services.md; SURVEY.md appendix E)
static const struct { uint16_t code; const char* name; } kTypeNames[] = {
    {MS_T_INIT, "init"}, {MS_T_INIT_OK, "init_ok"}, {MS_T_ERROR, "error"}, {MS_T_ECHO, "echo"}, {MS_T_ECHO_OK, "echo_ok"},
    {MS_T_TOPOLOGY, "topology"}, {MS_T_TOPOLOGY_OK, "topology_ok"}, {MS_T_BROADCAST, "broadcast"},
    {MS_T_BROADCAST_OK, "broadcast_ok"}, {MS_T_READ, "read"}, {MS_T_READ_OK, "read_ok"}, {MS_T_ADD, "add"},
    {MS_T_ADD_OK, "add_ok"}, {MS_T_REPLICATE_ONE, "replicate_one"}, {MS_T_REPLICATE_FULL, "replicate_full"},
    {MS_T_WRITE, "write"}, {MS_T_WRITE_OK, "write_ok"}, {MS_T_CAS, "cas"}, {MS_T_CAS_OK, "cas_ok"}, {MS_T_TS, "ts"},
    {MS_T_TS_OK, "ts_ok"}, {MS_T_REQUEST_VOTE, "request_vote"}, {MS_T_REQUEST_VOTE_RES, "request_vote_res"},
    {MS_T_APPEND_ENTRIES, "append_entries"}, {MS_T_APPEND_ENTRIES_RES, "append_entries_res"}, {MS_T_TXN, "txn"},
    {MS_T_TXN_OK, "txn_ok"}};

static void set_err(const std::string& s) { g_err = s; }

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t e__ = (call);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      set_err(std::string(#call) + ": " + cudaGetErrorString(e__));                   \
      return MS_ERR_CUDA;                                                             \
    }                                                                                 \
  } while (0)

static uint32_t pow2_at_least(uint32_t x) {
  uint32_t p = 1;
  while (p < x) p <<= 1;
  return p;
}

// rows of per-round history: 24 B per (round, ticket), kept under ~2 GB; < 2^15 (entry tags)
static uint32_t history_rows(uint32_t wanted, uint32_t t_max) {
  uint32_t hist = wanted ? std::min<uint32_t>(pow2_at_least(wanted), 16384u) : 4096;
  while (hist > 64 && (uint64_t)hist * t_max * 24 > (2ull << 30)) hist >>= 1;
  return hist;
}

static const char* dev_error_text(uint32_t code) {
  switch (code) {
    case E_RING_OVERFLOW: return "inbox ring overflow (raise ms_config.ring_cap / server_ring_cap) at endpoint";
    case E_WINDOW_OVERFLOW: return "per-round window exceeds ms_config.max_window / server_max_window at endpoint";
    case E_JOURNAL_OVERFLOW: return "journal ring overflow (drain more often or raise journal_cap_log2)";
    case E_INVALID_DEST: return "Invalid dest for message (net.clj:174): endpoint";
    case E_HISTORY: return "message older than the round history (raise ms_config.reserved[0] = history rounds): round";
    case E_VALUE_RANGE: return "broadcast value out of range (raise ms_config.n_values): value";
    case E_MAIL_OVERFLOW: return "host mailbox overflow (raise ms_config.mailbox_cap) at endpoint";
    case E_CALENDAR_OVERFLOW: return "timing wheel out of blocks (raise calendar_cap; 4294967295 = pool empty, else the slot whose chain is full or a latency beyond 65535 turns):";
    case E_ID_RANGE: return "per-ticket count exceeds the table entry range at ticket";
    case E_BARRIER: return "cross-shard barrier timed out waiting for shard";
    case E_RAFT_CAPACITY: return "Raft node out of log / staging / payload-heap capacity (raise ms_config.reserved[3]) at node";
    case E_HISTORY_RING: return "history ring of the closed-loop clients is full (call ms_history_drain more often) at client";
    case E_SNAPSHOT: return "replicate_full names a set snapshot that is not resident (in flight longer than calendar_slots, or forged): sender";
  }
  return "unknown device error";
}

// workload/broadcast.clj:40-178, restated for the device neighbor table.
static void topo_neighbors(uint32_t topo, uint32_t n, uint32_t k, std::vector<uint32_t>& out) {
  out.clear();
  if (k >= n) return;
  if (topo == MS_TOPO_GRID) {
    uint32_t side = (uint32_t)ceil(sqrt((double)n));
    if (side == 0) side = 1;
    const int64_t i = k / side, j = k % side;
    const int64_t di[4] = {1, -1, 0, 0}, dj[4] = {0, 0, 1, -1};   // (i+1,j) (i-1,j) (i,j+1) (i,j-1), :60-63
    for (int d = 0; d < 4; d++) {
      const int64_t a = i + di[d], b = j + dj[d];
      if (a < 0 || b < 0 || b >= (int64_t)side) continue;
      const int64_t idx = a * side + b;
      if (idx < (int64_t)n) out.push_back((uint32_t)idx);
    }
  } else if (topo == MS_TOPO_LINE) {
    if (n < 2) return;
    if (k > 0 && k < n - 1) { out.push_back(k - 1); out.push_back(k + 1); }
    else if (k == 0) out.push_back(1);
    else out.push_back(n - 2);
  } else if (topo == MS_TOPO_TOTAL) {
    for (uint32_t i = 0; i < n; i++) if (i != k) out.push_back(i);
  } else {
    const uint32_t b = topo == MS_TOPO_TREE2 ? 2 : topo == MS_TOPO_TREE3 ? 3 : 4;
    if (k) out.push_back((k - 1) / b);
    for (uint32_t c = 1; c <= b; c++) {
      const uint64_t ch = (uint64_t)b * k + c;
      if (ch < n) out.push_back((uint32_t)ch);
    }
  }
}

struct ms_sim {
  std::mutex mu;
  ms_config cfg;
  int device = 0;
  cudaStream_t stream = nullptr;
  Params P;                 // by-value kernel parameters (pointers + sizing)
  NetParams np;             // host mirror of the device knobs
  DevState hs;              // host mirror of the device state (valid after sync_state)
  // window-size classes of the round kernel (ascending caps); exactly one runs per round
  int n_classes = 0;
  uint32_t class_cap[4] = {0, 0, 0, 0};
  int class_threads[4] = {0, 0, 0, 0};
  int class_grid[4] = {0, 0, 0, 0};
  int n_sms = 148;
  bool use_calendar = false;
  uint64_t launches = 0;
  // ms_run sizes its batches of rounds from what the previous call needed (rounds until `until` was reached):
  // a fixed batch wastes launches on rounds past the stop time and a blocking read-back per batch
  uint64_t run_hint = 0;
  bool mail_seen = false;          // host-visible deliveries happened: keep the batches short (mail_cap)

  std::vector<uint8_t> kinds;
  std::vector<std::string> names;
  std::unordered_map<std::string, uint32_t> by_name;
  std::vector<std::deque<ms_msg>> mailbox;
  std::vector<ms_msg> pending;      // host sends not yet staged
  std::vector<ms_op> sched;
  std::vector<uint32_t> tick_off;
  ms_op* d_sched = nullptr;
  uint32_t* d_tick_off = nullptr;
  size_t d_sched_cap = 0, d_tick_cap = 0;
  bool pair_alloc = false;
  // JSON data plane (ms_send_json / ms_recv_json): payloads the device does not interpret stay here,
  // keyed by the handle that travels in p1; types without a device handler get codes from 1000 up
  std::unordered_map<uint64_t, std::string> blobs;
  uint64_t next_blob = 0;
  std::unordered_map<std::string, uint16_t> dyn_types;
  std::vector<std::string> dyn_names;
  std::string type_name(uint16_t code) const {
    for (const auto& t : kTypeNames) if (t.code == code) return t.name;
    if (code >= 1000 && (size_t)(code - 1000) < dyn_names.size()) return dyn_names[code - 1000];
    return "type-" + std::to_string(code);
  }
  uint16_t type_code(const std::string& name) {
    for (const auto& t : kTypeNames) if (name == t.name) return t.code;
    auto it = dyn_types.find(name);
    if (it != dyn_types.end()) return it->second;
    const uint16_t code = (uint16_t)(1000 + dyn_names.size());
    dyn_types[name] = code;
    dyn_names.push_back(name);
    return code;
  }
  FILE* jfile = nullptr;
  msf::Writer* jfress = nullptr;    // non-null: the journal file is a Fressian stripe (net/journal.clj)
  // journal expansion (K3) staging
  void* stage_ev = nullptr;
  void* stage_body = nullptr;
  size_t stage_cap = 0;
  std::vector<RoundMeta> hmeta;
  // sharding
  ms_barrier_fn barrier = nullptr;     // optional user barrier; default = k_barrier over peer memory
  void* barrier_ctx = nullptr;
  void do_barrier() {
    if (barrier) barrier(barrier_ctx, (void*)stream);
    else msk_barrier(&P, stream);
  }
  // CUDA graph of a batch of rounds (the launch sequence of a round is always the same; what a
  // round does is decided on the device).  Re-captured whenever the kernel parameters change.
  cudaStream_t aux_streams[4] = {nullptr, nullptr, nullptr, nullptr};   // size classes run concurrently
  cudaEvent_t aux_events[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaGraphExec_t graph_exec = nullptr;
  uint64_t graph_rounds = 0;
  Params graph_P;
  bool use_graph = false;   // opt-in (ms_config.reserved[1] = 1): instantiating the forked graph costs more
                            // than it saves unless the kernel parameters stay fixed for many batches
  std::vector<void*> peer_ptrs;     // opened IPC mappings
  // journal streaming (ms_run_streamed): two pinned host buffers written by the packing kernel
  cudaStream_t jstream = nullptr;
  cudaEvent_t j_rounds_done[2] = {nullptr, nullptr}, j_copied[2] = {nullptr, nullptr};
  cudaEvent_t j_packed[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned char* jdev[2] = {nullptr, nullptr};    // device staging: [ms_jbatch | rows | events]
  unsigned char* jhost[2] = {nullptr, nullptr};   // pinned: events of a batch
  unsigned char* jhdr[4] = {nullptr, nullptr, nullptr, nullptr};   // pinned: [ms_jbatch | rows] of a batch
  size_t jhost_events = 0;
  int jhost_format = 0;
  void* jplan = nullptr;
  static constexpr uint32_t kStreamRows = 4096;   // rounds per batch at most
  // timing
  cudaEvent_t t0 = nullptr, t1 = nullptr;
  bool profiling = false;
  std::vector<cudaEvent_t> prof_ev;   // pairs
  size_t prof_used = 0;
  double prof_ms = 0;
  uint64_t prof_launches = 0;
  std::vector<void*> allocs;

  template <typename T>
  int dalloc(T** out, size_t count) {
    void* ptr = nullptr;
    const size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    CK(cudaMalloc(&ptr, bytes));
    CK(cudaMemsetAsync(ptr, 0, bytes, stream));
    allocs.push_back(ptr);
    *out = (T*)ptr;
    return MS_OK;
  }

  int push_np() {
    CK(cudaMemcpyAsync(P.np, &np, sizeof(np), cudaMemcpyHostToDevice, stream));
    return MS_OK;
  }

  int sync_state() {
    CK(cudaMemcpyAsync(&hs, P.st, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (prof_used) collect_profile();
    if (hs.mail_count) {
      mail_seen = true;
      const uint32_t n = std::min(hs.mail_count, P.mail_cap);
      std::vector<ms_msg> buf(n);
      CK(cudaMemcpy(buf.data(), P.mail, (size_t)n * sizeof(ms_msg), cudaMemcpyDeviceToHost));
      for (const ms_msg& m : buf)
        if (m.dest < mailbox.size()) mailbox[m.dest].push_back(m);
      const uint32_t zero = 0;
      CK(cudaMemcpy(&P.st->mail_count, &zero, sizeof(zero), cudaMemcpyHostToDevice));
      hs.mail_count = 0;
    }
    if (hs.error) {
      char buf[256];
      snprintf(buf, sizeof buf, "%s %u (round %llu)", dev_error_text(hs.error), hs.error_arg,
               (unsigned long long)hs.round);
      set_err(buf);
      return MS_ERR_SIM;
    }
    return MS_OK;
  }

  int stage_injections() {
    if (pending.empty()) return MS_OK;
    if (pending.size() > cfg.inject_cap) { set_err("too many host sends staged for one round (inject_cap)"); return MS_ERR_CAPACITY; }
    const uint32_t n = (uint32_t)pending.size();
    CK(cudaMemcpyAsync(P.inj_buf, pending.data(), (size_t)n * sizeof(ms_msg), cudaMemcpyHostToDevice, stream));
    CK(cudaMemcpyAsync(&P.st->inj_count, &n, sizeof(n), cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));   // `pending` is pageable host memory
    pending.clear();
    return MS_OK;
  }

  int set_stop(int64_t stop) {
    CK(cudaMemcpyAsync(&P.st->stop_ns, &stop, sizeof(stop), cudaMemcpyHostToDevice, stream));
    return MS_OK;
  }

  void launch_rounds(uint64_t n) {
    // batches of rounds are replayed from a CUDA graph: removes the per-launch host cost
    if (use_graph && !profiling && !barrier && n >= 8) {
      if (graph_exec && (graph_rounds != n || memcmp(&graph_P, &P, sizeof(Params)) != 0)) {
        cudaGraphExecDestroy(graph_exec);
        graph_exec = nullptr;
      }
      if (!graph_exec) {
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
          launch_rounds_direct(n);
          if (cudaStreamEndCapture(stream, &graph) == cudaSuccess && graph &&
              cudaGraphInstantiate(&graph_exec, graph, 0) == cudaSuccess) {
            graph_rounds = n;
            memcpy(&graph_P, &P, sizeof(Params));
          } else {
            graph_exec = nullptr;
            use_graph = false;          // fall back to direct launches for good
          }
          if (graph) cudaGraphDestroy(graph);
          cudaGetLastError();
        } else {
          use_graph = false;
          cudaGetLastError();
        }
      }
      if (graph_exec && cudaGraphLaunch(graph_exec, stream) == cudaSuccess) {
        launches += n * ((use_calendar ? 2 : 1) + n_classes + (P.n_shards > 1 ? (use_calendar ? 4 : 3) : 0));
        return;
      }
    }
    launch_rounds_direct(n);
  }

  void launch_rounds_direct(uint64_t n) {
    // sharded, no timing wheel, the engine's own barrier, few enough endpoints for one CTA: one glue launch between rounds
    const bool glue = P.n_shards > 1 && !use_calendar && !barrier && !P.cm_blk && P.n_ep <= 32768 && !getenv("MS_NO_GLUE");
    for (uint64_t i = 0; i < n; i++) {
      cudaEvent_t a = nullptr, b = nullptr;
      if (profiling) {
        if (prof_used + 2 > prof_ev.size()) {
          prof_ev.resize(prof_used + 2, nullptr);
          cudaEventCreate(&prof_ev[prof_used]);
          cudaEventCreate(&prof_ev[prof_used + 1]);
        }
        a = prof_ev[prof_used]; b = prof_ev[prof_used + 1];
        prof_used += 2;
      }
      // persistent grids: one CTA slot per resident block, never more CTAs than tickets
      const int T = (int)(P.n_inj_tickets + P.n_ep);
      int grids[4];
      for (int c = 0; c < n_classes; c++) grids[c] = std::max(1, std::min(class_grid[c], T));
      if (P.n_shards <= 1) {
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, use_calendar ? 1 : 0, stream, a, b, 15, aux_streams, aux_events);
        if (!capturing()) launches += (use_calendar ? 2 : 1) + n_classes + (P.split_commit ? (P.cm_blk ? 3 : 1) : 0);
      } else if (glue) {
        // sharded: glue (barrier | commit of the previous round | snapshot | barrier) | round kernels (peer writes)
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, a, b, 16, aux_streams, aux_events);
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, a, b, 2, aux_streams, aux_events);
        if (!capturing()) launches += 1 + n_classes;
      } else {
        // sharded: [release (peer writes) | barrier] snapshot | barrier | round kernels (peer writes) | barrier | commit
        if (use_calendar) {
          msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 1, stream, a, b, 1, aux_streams, aux_events);
          do_barrier();   // released messages must be in the owners' rings before they snapshot
        }
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, a, b, 8, aux_streams, aux_events);
        do_barrier();
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, a, b, 2, aux_streams, aux_events);
        do_barrier();
        msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, a, b, 4, aux_streams, aux_events);
        if (!capturing()) launches += (use_calendar ? 2 : 1) + n_classes + (use_calendar ? 4 : 3);
      }
    }
    if (glue && n) {     // close the batch: the last round's commit
      int grids[4] = {1, 1, 1, 1};
      msk_launch_round(&P, n_classes, class_cap, class_threads, grids, 0, stream, nullptr, nullptr, 32, aux_streams, aux_events);
      if (!capturing()) launches += 1;
    }
  }

  bool capturing() {
    cudaStreamCaptureStatus st_ = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &st_);
    return st_ != cudaStreamCaptureStatusNone;
  }

  void collect_profile() {   // call after the stream is synchronised
    for (size_t i = 0; i + 1 < prof_used; i += 2) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, prof_ev[i], prof_ev[i + 1]) == cudaSuccess) { prof_ms += ms; prof_launches++; }
    }
    prof_used = 0;
  }

  int maybe_flush_journal_file() {
    if (!jfile || cfg.journal_discard || cfg.journal_level == 0) return MS_OK;
    if (hs.jraw_cursor - hs.jraw_drained < (P.jmask + 1) / 4 && hs.round - hs.drain_round < P.hist / 4) return MS_OK;
    return flush_journal_file();
  }

  // Expands raw per-(round, ticket) chunks into events in event-id order
  // (k_journal_expand) in a device staging buffer, then copies them out.
  int drain(ms_event* ev, ms_jbody* bodies, size_t cap, size_t* n_out) {
    *n_out = 0;
    if (cfg.journal_level == 0 || cfg.journal_discard) return MS_OK;
    const uint64_t avail = hs.next_event - hs.journal_drained;
    const size_t n = (size_t)std::min<uint64_t>(avail, cap);
    if (n == 0) return MS_OK;
    if (!stage_ev) {
      stage_cap = (size_t)std::min<uint64_t>(P.jmask + 1, 1ull << 22);
      CK(cudaMalloc(&stage_ev, stage_cap * 32));
      if (cfg.journal_level >= 2) CK(cudaMalloc(&stage_body, stage_cap * 32));
    }
    hmeta.resize(P.hist);
    CK(cudaMemcpy(hmeta.data(), P.rmeta, (size_t)P.hist * sizeof(RoundMeta), cudaMemcpyDeviceToHost));
    auto meta = [&](uint64_t r) -> const RoundMeta& { return hmeta[(size_t)(r & P.hist_mask)]; };
    size_t done = 0;
    while (done < n) {
      const size_t piece = std::min(n - done, stage_cap);
      const uint64_t first = hs.journal_drained;
      // committed rounds [drain_round, hs.round) that intersect [first, first + piece)
      const uint64_t r0 = hs.drain_round;
      uint64_t r1 = r0;
      while (r1 < hs.round && meta(r1).round == r1 && meta(r1).ev_base < first + piece) r1++;
      if (r1 == r0) { set_err("journal drain: round history lost"); return MS_ERR_SIM; }
      const bool want_body = bodies && cfg.journal_level >= 2;
      if (P.n_shards > 1) {   // only this shard's events are produced; the rest stays 0xFF
        CK(cudaMemsetAsync(stage_ev, 0xFF, piece * 32, stream));
        if (want_body) CK(cudaMemsetAsync(stage_body, 0xFF, piece * 32, stream));
      }
      msk_journal_expand(&P, r0, (uint32_t)(r1 - r0), first, piece, stage_ev, want_body ? stage_body : nullptr, n_sms, stream);
      CK(cudaStreamSynchronize(stream));
      CK(cudaMemcpy(ev + done, stage_ev, piece * 32, cudaMemcpyDeviceToHost));
      if (want_body) CK(cudaMemcpy(bodies + done, stage_body, piece * 32, cudaMemcpyDeviceToHost));
      done += piece;
      hs.journal_drained += piece;
      while (hs.drain_round < hs.round && meta(hs.drain_round).ev_base + meta(hs.drain_round).ev_total <= hs.journal_drained)
        hs.drain_round++;
    }
    hs.jraw_drained = hs.drain_round < hs.round ? meta(hs.drain_round).raw_base : hs.jraw_cursor;
    CK(cudaMemcpy(&P.st->journal_drained, &hs.journal_drained, sizeof(uint64_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(&P.st->drain_round, &hs.drain_round, sizeof(uint64_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(&P.st->jraw_drained, &hs.jraw_drained, sizeof(uint64_t), cudaMemcpyHostToDevice));
    *n_out = n;
    return MS_OK;
  }

  int flush_journal_file() {
    if (!jfile) return MS_OK;
    std::vector<ms_event> ev(1 << 16);
    std::vector<ms_jbody> bd(cfg.journal_level >= 2 ? (1 << 16) : 0);
    for (;;) {
      size_t n = 0;
      const int rc = drain(ev.data(), bd.empty() ? nullptr : bd.data(), ev.size(), &n);
      if (rc) return rc;
      if (!n) break;
      for (size_t i = 0; i < n; i++) {
        if (jfress) { write_fressian_event(ev[i], bd[i]); continue; }
        fwrite(&ev[i], sizeof(ms_event), 1, jfile);
        if (!bd.empty()) fwrite(&bd[i], sizeof(ms_jbody), 1, jfile);
      }
    }
    fflush(jfile);
    return MS_OK;
  }

  // Event{id time type message} as maelstrom.net.journal writes it (journal.clj:70-92).  The body map
  // is rebuilt from the fixed-size record: reserved keys as they are (doc/protocol.md:36-45), the
  // payload under the key the workload's schema gives it (doc/workloads.md); what the device only
  // holds a handle or a size for is journaled as that handle / size.
  void write_fressian_event(const ms_event& e, const ms_jbody& b) {
    const std::string tname = type_name(b.type);
    std::vector<msf::Writer::KV> kv;
    kv.push_back({"type", true, 0, tname});
    if (b.flags & MS_F_MSG_ID) kv.push_back({"msg_id", false, (int64_t)b.msg_id, ""});
    if (b.flags & MS_F_REPLY) kv.push_back({"in_reply_to", false, (int64_t)b.in_reply_to, ""});
    const bool kv_peer = (e.src < kinds.size() && (kinds[e.src] & 0x7F) == MS_KIND_SERVICE) ||
                         (e.dest < kinds.size() && (kinds[e.dest] & 0x7F) == MS_KIND_SERVICE) || cfg.workload == MS_W_RAFT;
    const int64_t lo = (int64_t)(b.p1 & 0xFFFFFFFFull), hi = (int64_t)(b.p1 >> 32);
    switch (b.type) {
      case MS_T_BROADCAST: kv.push_back({"message", false, (int64_t)b.p0, ""}); break;
      case MS_T_ADD: case MS_T_REPLICATE_ONE: kv.push_back({"element", false, (int64_t)b.p0, ""}); break;
      case MS_T_ERROR: kv.push_back({"code", false, (int64_t)b.p0, ""}); break;
      case MS_T_ECHO: case MS_T_ECHO_OK: kv.push_back({"echo_handle", false, (int64_t)b.p1, ""}); break;
      case MS_T_READ: if (kv_peer) kv.push_back({"key", false, (int64_t)b.p0, ""}); break;
      case MS_T_READ_OK:
        if (kv_peer) kv.push_back({"value", false, (int64_t)b.p1, ""});
        else kv.push_back({"count", false, (int64_t)b.p0, ""});
        break;
      case MS_T_WRITE: kv.push_back({"key", false, (int64_t)b.p0, ""}); kv.push_back({"value", false, lo, ""}); break;
      case MS_T_CAS:
        kv.push_back({"key", false, (int64_t)b.p0, ""}); kv.push_back({"from", false, lo, ""}); kv.push_back({"to", false, hi, ""});
        break;
      case MS_T_TS_OK: kv.push_back({"ts", false, (int64_t)b.p1, ""}); break;
      case MS_T_REPLICATE_FULL: kv.push_back({"count", false, (int64_t)b.p0, ""}); kv.push_back({"snapshot", false, (int64_t)b.p1, ""}); break;
      case MS_T_REQUEST_VOTE:
        kv.push_back({"term", false, (int64_t)b.p0, ""}); kv.push_back({"last_log_index", false, lo, ""});
        kv.push_back({"last_log_term", false, hi, ""});
        break;
      case MS_T_REQUEST_VOTE_RES: kv.push_back({"term", false, (int64_t)b.p0, ""}); kv.push_back({"vote_granted", false, lo, ""}); break;
      case MS_T_APPEND_ENTRIES: kv.push_back({"term", false, (int64_t)b.p0, ""}); kv.push_back({"entries_handle", false, (int64_t)b.p1, ""}); break;
      case MS_T_APPEND_ENTRIES_RES: kv.push_back({"term", false, (int64_t)b.p0, ""}); kv.push_back({"success", false, lo, ""}); break;
      case MS_T_TXN: kv.push_back({"txn_handle", false, (int64_t)b.p1, ""}); break;
      case MS_T_TXN_OK: kv.push_back({"read_version", false, lo, ""}); kv.push_back({"written_version", false, hi, ""}); break;
      default: break;
    }
    auto name_of = [&](uint32_t i) { return i < names.size() ? names[i] : std::to_string(i); };
    jfress->write_event((int64_t)(e.event_id & ~MS_EVENT_RECV), e.time_ns, (e.event_id & MS_EVENT_RECV) != 0, (int64_t)e.msg_id,
                        name_of(e.src), name_of(e.dest), kv);
  }

  // Uploads only ops[first..) (the schedule is append-only) and refreshes tick_off.
  int upload_schedule(size_t first) {
    const size_t n = sched.size();
    if (n > d_sched_cap) {
      const size_t cap = std::max<size_t>(n, d_sched_cap * 2);
      ms_op* nd = nullptr;
      CK(cudaMalloc((void**)&nd, cap * sizeof(ms_op)));
      if (d_sched && first) CK(cudaMemcpy(nd, d_sched, first * sizeof(ms_op), cudaMemcpyDeviceToDevice));
      if (d_sched) cudaFree(d_sched);
      d_sched = nd;
      d_sched_cap = cap;
    }
    if (n > first)
      CK(cudaMemcpy(d_sched + first, sched.data() + first, (n - first) * sizeof(ms_op), cudaMemcpyHostToDevice));
    // tick_off[j] = number of ops whose injection tick ceil(time/tick) is < j.  The schedule is
    // append-only and sorted: count the new ops per tick, then one running sum from the first
    // tick they touch (entries below it are unchanged).
    const int64_t last = n ? sched.back().time_ns : 0;
    const size_t n_ticks = (size_t)((last + kTickNs - 1) / kTickNs) + 2;
    const size_t old_sz = tick_off.size();
    if (tick_off.size() < n_ticks + 1) tick_off.resize(n_ticks + 1, old_sz ? tick_off.back() : 0);
    if (n > first) {
      std::vector<uint32_t> add(tick_off.size() + 1, 0);
      size_t lo = tick_off.size();
      for (size_t i = first; i < n; i++) {
        const int64_t t = sched[i].time_ns <= 0 ? 0 : (sched[i].time_ns + kTickNs - 1) / kTickNs;
        add[(size_t)t + 1]++;
        lo = std::min(lo, (size_t)t + 1);
      }
      uint32_t run = 0;
      for (size_t j = lo; j < tick_off.size(); j++) { run += add[j]; tick_off[j] += run; }
    }
    if (tick_off.size() > d_tick_cap) {
      const size_t cap = std::max<size_t>(tick_off.size(), d_tick_cap * 2);
      uint32_t* nd = nullptr;
      CK(cudaMalloc((void**)&nd, cap * sizeof(uint32_t)));
      if (d_tick_off) cudaFree(d_tick_off);
      d_tick_off = nd;
      d_tick_cap = cap;
    }
    CK(cudaMemcpy(d_tick_off, tick_off.data(), tick_off.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    P.sched = d_sched;
    P.n_sched = (uint32_t)n;
    P.tick_off = d_tick_off;
    P.n_tick_off = (uint32_t)tick_off.size();
    return MS_OK;
  }
};

static int build_sim(ms_sim* s, const ms_config* in) {
  ms_config& c = s->cfg;
  c = *in;
  if (c.n_nodes == 0) { set_err("n_nodes must be positive (--node-count)"); return MS_ERR_ARG; }
  if (c.workload > MS_W_TXN_TREE || c.topology > MS_TOPO_TREE4 || c.latency_dist > MS_DIST_EXPONENTIAL) {
    set_err("bad workload/topology/latency_dist");
    return MS_ERR_ARG;
  }
  if (c.latency_dist != MS_DIST_CONSTANT && c.latency_mean_ms == 0) {
    // (exponential-distribution (/ 0)) divides by zero; (integer-distribution 0 0) is empty (net.clj:76-77)
    set_err("latency mean 0 is only valid with the constant distribution");
    return MS_ERR_ARG;
  }
  if (!c.n_values) c.n_values = 1u << 16;
  if (!c.max_endpoints) c.max_endpoints = c.n_nodes + 256;
  if (c.max_endpoints < c.n_nodes) { set_err("max_endpoints < n_nodes"); return MS_ERR_ARG; }
  c.ring_cap = pow2_at_least(c.ring_cap ? c.ring_cap : 1024);
  c.max_window = pow2_at_least(c.max_window ? c.max_window : std::min<uint32_t>(c.ring_cap, 1024));
  // 25 B of dynamic shared memory per window slot + ~3 KB static, 227 KB per CTA on sm_100a
  if (c.max_window > 8192) { set_err("max_window must be <= 8192 (25 B of shared memory per slot, 227 KB per CTA)"); return MS_ERR_ARG; }
  if (c.max_window > c.ring_cap) c.max_window = c.ring_cap;
  c.server_ring_cap = c.server_ring_cap ? pow2_at_least(c.server_ring_cap) : c.ring_cap;
  c.server_max_window = c.server_max_window ? pow2_at_least(c.server_max_window) : std::min(c.max_window, c.server_ring_cap);
  if (c.server_max_window > c.server_ring_cap) c.server_max_window = c.server_ring_cap;
  if (c.server_max_window > c.max_window) {   // the round kernel's size classes are cut for max_window
    set_err("server_max_window must not exceed max_window");
    return MS_ERR_ARG;
  }
  if (!c.journal_cap_log2) c.journal_cap_log2 = 22;
  if (c.journal_level > 2) c.journal_level = 2;
  if (!c.mailbox_cap) c.mailbox_cap = 1u << 16;
  if (!c.inject_cap) c.inject_cap = 1u << 16;
  if (!c.gset_interval_ms) c.gset_interval_ms = 5000;
  s->use_calendar = c.latency_mean_ms > 0;
  if (s->use_calendar) {
    c.calendar_slots = pow2_at_least(c.calendar_slots ? c.calendar_slots
                                                      : std::min<uint32_t>(16384u, std::max<uint32_t>(64u, 32u * c.latency_mean_ms)));
    // a record's order key is turned into its dense id when its slot first comes up, i.e. within
    // calendar_slots ticks of the send: keep that inside the round history (longer latencies
    // simply wait more turns, so the wheel's span is a tuning knob, not a limit)
    const uint32_t hist = history_rows(c.reserved[0], c.max_endpoints + 8u);
    while (c.calendar_slots > 4 && c.calendar_slots > hist / 4) c.calendar_slots >>= 1;
    if (!c.calendar_cap) c.calendar_cap = 1u << 16;
  }
  if (c.n_shards == 0) c.n_shards = 1;
  if (c.n_shards > 8 || c.shard_id >= c.n_shards) { set_err("n_shards must be <= 8 and shard_id < n_shards"); return MS_ERR_ARG; }
  if (c.threads_per_node && (c.threads_per_node % 32 || c.threads_per_node > 512)) {
    set_err("threads_per_node must be a multiple of 32 in [32,512]");
    return MS_ERR_ARG;
  }
  {
    const uint32_t* ladder = kClsLadder;
    // g-set: a node's step ORs whole bitmap rows (one word per thread and pass): wide CTAs even for short windows
    const int thr_gset[4] = {256, 256, 256, 512};
    const int* thr = c.workload == MS_W_GSET ? thr_gset : kClsThreads;
    s->n_classes = 0;
    for (int k = 0; k < 4; k++) {
      const uint32_t cap = std::min(ladder[k], c.max_window);
      s->class_cap[s->n_classes] = cap;
      s->class_threads[s->n_classes] = c.threads_per_node ? (int)c.threads_per_node : thr[k];
      s->n_classes++;
      if (cap == c.max_window) break;
    }
  }

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_err("no CUDA device: maelstrom_b200 has no CPU fallback");
    return MS_ERR_CUDA;
  }
  s->device = c.device;
  CK(cudaSetDevice(s->device));
  CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  for (int k = 0; k < 4; k++) CK(cudaStreamCreateWithFlags(&s->aux_streams[k], cudaStreamNonBlocking));
  for (int k = 0; k < 5; k++) CK(cudaEventCreateWithFlags(&s->aux_events[k], cudaEventDisableTiming));

  Params& P = s->P;
  memset(&P, 0, sizeof P);
  const uint32_t M = c.max_endpoints;
  int rc;
  if ((rc = s->dalloc(&P.st, 1))) return rc;
  if ((rc = s->dalloc(&P.np, 1))) return rc;
  if ((rc = s->dalloc(&P.kind, M))) return rc;
  if ((rc = s->dalloc(&P.tail, M))) return rc;
  if ((rc = s->dalloc(&P.limit, M))) return rc;
  if ((rc = s->dalloc(&P.head, M))) return rc;
  if ((rc = s->dalloc(&P.ep_born, M))) return rc;
  {
    void* ptr = nullptr;
    P.ring_slots = (size_t)c.n_nodes * c.server_ring_cap + (size_t)(M - c.n_nodes) * c.ring_cap;
    CK(cudaMalloc(&ptr, P.ring_slots * 48));   // key plane (16 B per slot), then body plane (32 B per slot)
    s->allocs.push_back(ptr);
    P.ring = (uint4*)ptr;
  }
  P.ring_cap = c.ring_cap;
  P.ring_cap_s = c.server_ring_cap;
  P.n_servers = c.n_nodes;
  P.n_ep = c.n_nodes;
  P.n_inj_tickets = 8;
  P.max_window = c.max_window;
  P.max_window_s = c.server_max_window;
  s->use_graph = c.reserved[1] == 1;
  P.n_shards = c.n_shards;
  P.shard_id = c.shard_id;
  {
    // per-round history: 16 B per (round, ticket); keep it under ~1 GB
    P.t_max = M + P.n_inj_tickets;
    const uint32_t hist = history_rows(c.reserved[0], P.t_max);
    P.hist = hist;
    P.hist_mask = hist - 1;
    if ((rc = s->dalloc(&P.rmeta, hist))) return rc;
    if ((rc = s->dalloc(&P.rt_em, (size_t)hist * P.t_max))) return rc;
    if ((rc = s->dalloc(&P.rt_ev, (size_t)hist * P.t_max))) return rc;
    if ((rc = s->dalloc(&P.rt_chunk, (size_t)hist * P.t_max))) return rc;
    if ((rc = s->dalloc(&P.rt_cnt, (size_t)hist * P.t_max))) return rc;
    std::vector<RoundMeta> init(hist);
    memset(init.data(), 0, init.size() * sizeof(RoundMeta));
    for (uint32_t i = 1; i < hist; i++) init[i].round = ~0ull;
    CK(cudaMemcpyAsync(P.rmeta, init.data(), init.size() * sizeof(RoundMeta), cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }
  P.jlevel = c.journal_level;
  P.jdiscard = c.journal_discard;
  if (c.journal_level) {
    const uint64_t J = 1ull << c.journal_cap_log2;
    void* ptr = nullptr;
    CK(cudaMalloc(&ptr, J * 16));
    s->allocs.push_back(ptr);
    P.jraw = (uint4*)ptr;
    P.jmask = J - 1;
    if (c.journal_level >= 2) {
      CK(cudaMalloc(&ptr, J * 32));
      s->allocs.push_back(ptr);
      P.jbody = (uint4*)ptr;
    }
  }
  if ((rc = s->dalloc(&P.comp, M))) return rc;
  P.seed_lo = c.seed_lo;
  P.seed_hi = c.seed_hi;
  P.workload = c.workload;
  P.topology = c.topology;
  P.n_values = c.n_values;
  P.bm_words = (c.n_values + 31) / 32;
  if (c.workload == MS_W_BROADCAST || c.workload == MS_W_GSET) {
    if ((rc = s->dalloc(&P.bitmap, (size_t)c.n_nodes * P.bm_words))) return rc;
    if ((rc = s->dalloc(&P.set_count, c.n_nodes))) return rc;
    if (c.topology != MS_TOPO_TOTAL) {
      std::vector<uint32_t> off(c.n_nodes + 1, 0), nbr, tmp;
      for (uint32_t k = 0; k < c.n_nodes; k++) {
        topo_neighbors(c.topology, c.n_nodes, k, tmp);
        nbr.insert(nbr.end(), tmp.begin(), tmp.end());
        off[k + 1] = (uint32_t)nbr.size();
      }
      if ((rc = s->dalloc(&P.nbr_off, off.size()))) return rc;
      if ((rc = s->dalloc(&P.nbr, nbr.size() + 1))) return rc;
      CK(cudaMemcpyAsync(P.nbr_off, off.data(), off.size() * 4, cudaMemcpyHostToDevice, s->stream));
      if (!nbr.empty()) CK(cudaMemcpyAsync(P.nbr, nbr.data(), nbr.size() * 4, cudaMemcpyHostToDevice, s->stream));
      CK(cudaStreamSynchronize(s->stream));
    }
  } else if (c.workload == MS_W_ECHO) {
    if ((rc = s->dalloc(&P.next_msg_id, c.n_nodes))) return rc;
  }
  P.family = c.workload == MS_W_GSET ? 1u : (c.workload >= MS_W_RAFT ? 4u : 0u);
  if (c.workload == MS_W_TXN_TREE) {
    // hash-tree txn-list-append (csrc/ms_tree.h): tree node records by pointer, per-node cache, lock queue
    if (c.n_shards > 1) { set_err("MS_W_TXN_TREE runs on one GPU (tree records are read across nodes)"); return MS_ERR_ARG; }
    const size_t N = c.n_nodes;
    P.tt_per_node = c.reserved[3] ? c.reserved[3] : 256u;
    P.tt_cache_mask = pow2_at_least(c.reserved[4] ? c.reserved[4] : 1024u) - 1u;
    const uint64_t n_ptrs = 2ull + (uint64_t)N * P.tt_per_node;
    if (n_ptrs > (1ull << 31)) { set_err("MS_W_TXN_TREE: n_nodes x reserved[3] pointers do not fit"); return MS_ERR_ARG; }
    if (!c.reserved[2]) c.reserved[2] = (uint32_t)n_ptrs;           // lww-kv is keyed by pointer
    if ((rc = s->dalloc(&P.tt_node, N)) || (rc = s->dalloc(&P.tt_recs, (size_t)n_ptrs * 64)) ||
        (rc = s->dalloc(&P.tt_cache, N * ((size_t)P.tt_cache_mask + 1))) || (rc = s->dalloc(&P.tt_queue, N * kTreeQueue)))
      return rc;
    mst::Rec empty{};                                               // Tree.empty: a leaf over the whole ring, no keys
    empty.type = 1; empty.lo = 0; empty.hi = (uint8_t)mst::kRing; empty.n = 0;
    CK(cudaMemcpyAsync(P.tt_recs + (size_t)(mst::kPtrEmpty - 1u) * 64, &empty, sizeof empty, cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }
  if (c.workload == MS_W_TXN || c.workload == MS_W_TXN_TREE) {
    // txn-list-append nodes: message ids, the table of pending RPC closures and the staging rows of
    // the sequential step (csrc/ms_raft.cuh)
    // (nothing here is read across nodes: sharded runs need no extra mapping)
    const size_t N = c.n_nodes;
    P.rf_stage_cap = c.workload == MS_W_TXN_TREE ? c.server_max_window * (mst::kMaxWrites + 2u) + 64u : c.server_max_window + 16u;
    P.rf_cb_mask = pow2_at_least(c.reserved[5] ? c.reserved[5] : kRaftCallbacks) - 1u;
    // one save! has up to mst::kMaxWrites writes in flight, each with its closure (the oracle applies the same floor)
    if (c.workload == MS_W_TXN_TREE && P.rf_cb_mask + 1u < 128u) P.rf_cb_mask = 127u;
    if ((rc = s->dalloc(&P.rf_node, N)) || (rc = s->dalloc(&P.rf_cb, N * ((size_t)P.rf_cb_mask + 1) * 2)) ||
        (rc = s->dalloc(&P.rf_stage, N * P.rf_stage_cap * 3)))
      return rc;
  }
  if (c.workload == MS_W_RAFT) {
    // Raft nodes (csrc/ms_raft.cuh): per-node log, KV store, leader tables, pending-RPC closures,
    // the staging rows of the sequential step and the heap of append_entries payloads
    const size_t N = c.n_nodes;
    P.rf_n_keys = c.reserved[2] ? c.reserved[2] : 4096u;
    P.rf_log_cap = c.reserved[3] ? c.reserved[3] : 4096u;
    // reserved[4] = g: independent Raft clusters of g consecutive servers (0 = one cluster of all)
    P.rf_group = (c.reserved[4] && c.reserved[4] < c.n_nodes) ? c.reserved[4] : 0u;
    P.rf_gmax = P.rf_group ? P.rf_group : c.n_nodes;
    P.rf_cb_mask = pow2_at_least(c.reserved[5] ? c.reserved[5] : kRaftCallbacks) - 1u;
    P.rf_stage_cap = c.server_max_window + 2u * P.rf_gmax + P.rf_log_cap + 16u;
    P.rf_vote_words = (P.rf_gmax + 31u) / 32u;
    // append_entries payloads live in one ring heap per shard until they are read: room for a
    // heartbeat wave of every cluster, a few times over
    const uint64_t heap_want = std::max<uint64_t>(std::max<uint64_t>(1u << 16, 8ull * P.rf_log_cap), 64ull * c.n_nodes);
    if (heap_want > (1ull << 30)) { set_err("Raft payload heap too large"); return MS_ERR_ARG; }
    const uint32_t heap_words = pow2_at_least((uint32_t)heap_want);
    P.rf_heap_mask = heap_words - 1u;
    if ((rc = s->dalloc(&P.rf_node, N)) || (rc = s->dalloc(&P.rf_log, N * P.rf_log_cap * 2)) ||
        (rc = s->dalloc(&P.rf_kv_val, N * P.rf_n_keys)) || (rc = s->dalloc(&P.rf_kv_has, N * P.rf_n_keys)) ||
        (rc = s->dalloc(&P.rf_next, N * P.rf_gmax)) || (rc = s->dalloc(&P.rf_match, N * P.rf_gmax)) ||
        (rc = s->dalloc(&P.rf_scratch, N * P.rf_gmax)) || (rc = s->dalloc(&P.rf_cb, N * ((size_t)P.rf_cb_mask + 1) * 2)) ||
        (rc = s->dalloc(&P.rf_votes, N * P.rf_vote_words)) || (rc = s->dalloc(&P.rf_stage, N * P.rf_stage_cap * 3)) ||
        (rc = s->dalloc(&P.rf_heap, (size_t)heap_words)) || (rc = s->dalloc(&P.rf_heap_cursor, 1)) ||
        (rc = s->dalloc(&P.rf_ext_off, N * kRaftExt + (N * kRaftExt + 1) / 2)))   // offsets, then the u32 tags
      return rc;
    P.rf_ext_tag = reinterpret_cast<uint32_t*>(P.rf_ext_off + N * kRaftExt);    // one allocation: one IPC handle
    P.rf_heap_sh[c.shard_id] = P.rf_heap;
    P.rf_ext_off_sh[c.shard_id] = P.rf_ext_off;
    P.rf_ext_tag_sh[c.shard_id] = P.rf_ext_tag;
    // fresh nodes: nascent, empty log but for the default entry {term 0, op None} (raft.py:121), last_applied 1
    std::vector<RaftDev> init(N);
    memset(init.data(), 0, N * sizeof(RaftDev));
    for (size_t i = 0; i < N; i++) { init[i].voted_for = -1; init[i].leader = -1; init[i].last_applied = 1; init[i].log_size = 1; }
    CK(cudaMemcpyAsync(P.rf_node, init.data(), N * sizeof(RaftDev), cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }
  for (int k = 0; k < 4; k++) P.sv_ep[k] = 0xFFFFFFFFu;
  if (c.workload == MS_W_GSET) {
    // replicate_full payloads: a snapshot stays resident while its messages can be in flight,
    // i.e. at most calendar_slots ticks; one run every gset_interval_ms (g_set.rb:34)
    P.gs_interval_ms = c.gset_interval_ms;
    // (the exponential law is unbounded: 48 means = a tail of e^-48; beyond that, e.g. after slow!, a
    // replicate_full that outlives its snapshot row is reported as E_SNAPSHOT)
    const uint32_t span_ms = !s->use_calendar ? 0u
        : std::max<uint32_t>(c.calendar_slots, c.latency_dist == MS_DIST_EXPONENTIAL ? 48u * c.latency_mean_ms : 2u * c.latency_mean_ms);
    P.gs_slots = std::min<uint32_t>(pow2_at_least(span_ms / c.gset_interval_ms + 2u), 1024u);
    const size_t rows = (size_t)c.n_nodes * P.gs_slots;
    if ((rc = s->dalloc(&P.gs_init, c.n_nodes))) return rc;
    if ((rc = s->dalloc(&P.gs_next_fire, c.n_nodes))) return rc;
    if ((rc = s->dalloc(&P.gs_fires, c.n_nodes))) return rc;
    if ((rc = s->dalloc(&P.gs_tag, rows))) return rc;
    if ((rc = s->dalloc(&P.gs_snap, rows * P.bm_words))) return rc;
    P.gs_snap_sh[c.shard_id] = P.gs_snap;
    P.gs_tag_sh[c.shard_id] = P.gs_tag;
  }
  if ((rc = s->dalloc(&P.inj_buf, c.inject_cap))) return rc;
  if ((rc = s->dalloc(&P.mail, c.mailbox_cap))) return rc;
  P.mail_cap = c.mailbox_cap;
  if (s->use_calendar) {
    // timing wheel = chains of pooled blocks (ms_device.cuh): calendar_cap is the AVERAGE number of
    // messages per slot the pool is sized for; a single slot may hold up to cal_tab_cap blocks
    const uint32_t cap_p2 = pow2_at_least(c.calendar_cap);
    uint32_t blk_log2 = 4;
    while ((1u << blk_log2) < cap_p2 / 16 && blk_log2 < 12) blk_log2++;
    const uint64_t blocks64 = (((uint64_t)c.calendar_slots * c.calendar_cap) >> blk_log2) + 2ull * c.calendar_slots + 64;
    if (blocks64 > (1ull << 30)) { set_err("timing wheel: calendar_slots x calendar_cap too large"); return MS_ERR_ARG; }
    P.cal_blk_log2 = blk_log2;
    P.cal_blocks = (uint32_t)blocks64;
    // chain table: 2 generations x slots x cal_tab_cap entries of 4 B, about 128 MB at most
    P.cal_tab_cap = std::min<uint32_t>(P.cal_blocks, std::max<uint32_t>(4096u, (1u << 24) / c.calendar_slots));
    P.cal_slots = c.calendar_slots;
    void* ptr = nullptr;
    CK(cudaMalloc(&ptr, ((size_t)P.cal_blocks << blk_log2) * 48));
    s->allocs.push_back(ptr);
    P.cal = (uint4*)ptr;
    if ((rc = s->dalloc(&P.cal_count, 2 * (size_t)c.calendar_slots))) return rc;
    if ((rc = s->dalloc(&P.cal_tab, 2 * (size_t)c.calendar_slots * P.cal_tab_cap))) return rc;
    if ((rc = s->dalloc(&P.cal_par, c.calendar_slots))) return rc;
    if ((rc = s->dalloc(&P.cal_free, P.cal_blocks))) return rc;
    if ((rc = s->dalloc(&P.cal_ret, P.cal_blocks))) return rc;
    std::vector<uint32_t> ids(P.cal_blocks);
    for (uint32_t i = 0; i < P.cal_blocks; i++) ids[i] = P.cal_blocks - 1 - i;   // block 0 is popped first
    CK(cudaMemcpyAsync(P.cal_free, ids.data(), ids.size() * 4, cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }

  // endpoints: servers n0..n{N-1} (core.clj:231-238)
  s->kinds.assign(M, kRemoved);
  s->names.resize(c.n_nodes);
  s->mailbox.resize(c.n_nodes);
  for (uint32_t i = 0; i < c.n_nodes; i++) {
    s->kinds[i] = MS_KIND_SERVER;
    s->names[i] = "n" + std::to_string(i);
    s->by_name[s->names[i]] = i;
  }
  CK(cudaMemcpyAsync(P.kind, s->kinds.data(), M, cudaMemcpyHostToDevice, s->stream));

  memset(&s->np, 0, sizeof s->np);
  s->np.dist = c.latency_dist;
  s->np.mean_ms = c.latency_mean_ms;
  s->np.scale = 1;
  s->np.exp_coeff = (uint64_t)llround((double)c.latency_mean_ms * 1.0 * 0.693147180559945309417232121458 * 4294967296.0);
  {
    const double p = c.p_loss;
    s->np.loss_thresh = !(p > 0.0) ? 0 : (p >= 1.0 ? (1ull << 32) : (uint64_t)(p * 4294967296.0));
  }
  if ((rc = s->push_np())) return rc;

  memset(&s->hs, 0, sizeof s->hs);
  s->hs.stop_ns = INT64_MAX;
  s->hs.cal_free_n = P.cal_blocks;
  CK(cudaMemcpyAsync(P.st, &s->hs, sizeof(DevState), cudaMemcpyHostToDevice, s->stream));

  CK(msk_round_smem_attr(msk_round_smem_bytes(c.max_window)));
  {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, s->device));
    s->n_sms = prop.multiProcessorCount;
    P.n_classes = (uint32_t)s->n_classes;
    for (int k = 0; k < 4; k++) P.cls_cap[k] = k < s->n_classes ? s->class_cap[k] : 0xFFFFFFFFu;
    for (int k = 0; k < s->n_classes; k++)
      s->class_grid[k] = s->n_sms * msk_round_occupancy(s->class_threads[k], msk_round_smem_bytes(s->class_cap[k]));
    if ((rc = s->dalloc(&P.cls_list, (size_t)2 * 4 * P.t_max))) return rc;
    // who commits a round: the last ticket inside k_round (one GPU, a few thousand tickets), or
    // launches of their own after the round kernels (sharded runs; tens of thousands of tickets)
    P.split_commit = (c.n_shards > 1 || P.t_max > 16384u) ? 1u : 0u;
    if (P.t_max > 16384u) {
      if ((rc = s->dalloc(&P.cm_blk, (size_t)(P.t_max + 1023) / 1024 + 1))) return rc;
      if ((rc = s->dalloc(&P.cm_flags, 4))) return rc;
    }
    for (int g = 0; g < 8; g++) { P.ring_sh[g] = nullptr; P.tail_sh[g] = nullptr; P.head_sh[g] = nullptr; P.rt_cnt_sh[g] = nullptr; }
    P.ring_sh[c.shard_id] = P.ring;
    P.tail_sh[c.shard_id] = P.tail;
    P.head_sh[c.shard_id] = P.head;
    P.rt_cnt_sh[c.shard_id] = P.rt_cnt;
    for (int g = 0; g < 8; g++) P.bar_sh[g] = nullptr;
    if ((rc = s->dalloc(&P.bar_sh[c.shard_id], 64))) return rc;
    CK(cudaStreamSynchronize(s->stream));
  }
  CK(cudaStreamSynchronize(s->stream));
  return MS_OK;
}

static void recompute_exp(ms_sim* s) {
  s->np.exp_coeff = (uint64_t)llround((double)s->np.mean_ms * (double)s->np.scale * 0.693147180559945309417232121458 * 4294967296.0);
}

extern "C" {

uint32_t ms_abi_version(void) { return MS_ABI_VERSION; }

const char* ms_last_error(ms_sim*) { return g_err.c_str(); }

ms_sim* ms_create(const ms_config* cfg) {
  if (!cfg) { set_err("null config"); return nullptr; }
  ms_sim* s = new ms_sim();
  if (build_sim(s, cfg) != MS_OK) {
    const std::string keep = g_err;
    ms_destroy(s);
    g_err = keep;
    return nullptr;
  }
  return s;
}

void ms_destroy(ms_sim* s) {
  if (!s) return;
  if (s->jfile) ms_journal_close(s);
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  for (void* p : s->peer_ptrs) cudaIpcCloseMemHandle(p);
  for (void* p : s->allocs) cudaFree(p);
  for (int k = 0; k < 2; k++) {
    if (s->jhost[k]) cudaFreeHost(s->jhost[k]);
    if (s->jdev[k]) cudaFree(s->jdev[k]);
    if (s->j_rounds_done[k]) cudaEventDestroy(s->j_rounds_done[k]);
    if (s->j_copied[k]) cudaEventDestroy(s->j_copied[k]);
  }
  for (int k = 0; k < 4; k++) {
    if (s->jhdr[k]) cudaFreeHost(s->jhdr[k]);
    if (s->j_packed[k]) cudaEventDestroy(s->j_packed[k]);
  }
  if (s->jstream) cudaStreamDestroy(s->jstream);
  if (s->stage_ev) cudaFree(s->stage_ev);
  if (s->stage_body) cudaFree(s->stage_body);
  if (s->d_sched) cudaFree(s->d_sched);
  if (s->d_tick_off) cudaFree(s->d_tick_off);
  if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
  for (int k = 0; k < 4; k++) if (s->aux_streams[k]) cudaStreamDestroy(s->aux_streams[k]);
  for (int k = 0; k < 5; k++) if (s->aux_events[k]) cudaEventDestroy(s->aux_events[k]);
  for (cudaEvent_t e : s->prof_ev) if (e) cudaEventDestroy(e);
  if (s->t0) cudaEventDestroy(s->t0);
  if (s->t1) cudaEventDestroy(s->t1);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int ms_start_nodes(ms_sim* s, uint32_t workload) {
  std::lock_guard<std::mutex> g(s->mu);
  if (workload != s->cfg.workload) {
    set_err("ms_start_nodes: workload differs from ms_config.workload (node state is sized at ms_create)");
    return MS_ERR_ARG;
  }
  return MS_OK;
}

int ms_stop_nodes(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  for (uint32_t i = 0; i < s->cfg.n_nodes; i++) {
    if (!(s->kinds[i] & kRemoved)) { s->by_name.erase(s->names[i]); s->kinds[i] |= kRemoved; }
  }
  CK(cudaMemcpy(s->P.kind, s->kinds.data(), s->cfg.n_nodes, cudaMemcpyHostToDevice));
  s->np.any_removed = 1;
  return s->push_np();
}

int ms_add_endpoint(ms_sim* s, const char* id, int kind) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (!id || kind < MS_KIND_CLIENT || kind > MS_KIND_SERVICE) { set_err("bad endpoint id/kind"); return MS_ERR_ARG; }
  if (s->by_name.count(id)) { set_err("endpoint already exists"); return MS_ERR_ARG; }
  // Slot of a removed non-server endpoint is recycled, lowest index first (Jepsen closes and reopens its
  // clients after every indefinite op, client.clj:55-59): the new endpoint starts with an empty
  // queue like any fresh one (net.clj:139-146).  Not while pairwise drop! entries exist: they
  // are keyed by index and must not leak onto another name.
  uint32_t idx = s->P.n_ep;
  bool reuse = false;
  if (kind != MS_KIND_SERVICE && !s->np.pair_active)
    for (uint32_t i = s->cfg.n_nodes; i < s->P.n_ep; i++)
      if ((s->kinds[i] & kRemoved) && (s->kinds[i] & 0x7F) != MS_KIND_SERVICE) { idx = i; reuse = true; break; }
  if (idx >= s->cfg.max_endpoints) { set_err("max_endpoints exhausted"); return MS_ERR_CAPACITY; }
  if (kind == MS_KIND_SERVICE) {
    // service/default-services (service.clj:290-296): the id names the service
    static const char* const names[4] = {"lin-kv", "seq-kv", "lww-kv", "lin-tso"};
    int svc = -1;
    for (int k = 0; k < 4; k++) if (!strcmp(id, names[k])) svc = k;
    if (svc < 0) { set_err("service endpoints are lin-kv, seq-kv, lww-kv or lin-tso (service.clj:290-296)"); return MS_ERR_ARG; }
    if (!s->P.sv_scalars) {
      int rc;
      Params& P = s->P;
      P.sv_n_keys = s->cfg.reserved[2] ? s->cfg.reserved[2] : 4096u;
      const size_t K = P.sv_n_keys;
      if ((rc = s->dalloc(&P.sv_lin_val, K)) || (rc = s->dalloc(&P.sv_lin_has, K)) ||
          (rc = s->dalloc(&P.sv_lww_val, 2 * K)) || (rc = s->dalloc(&P.sv_lww_has, 2 * K)) ||
          (rc = s->dalloc(&P.sv_scalars, 2)) || (rc = s->dalloc(&P.sv_seq_cli, s->cfg.max_endpoints)) ||
          (rc = s->dalloc(&P.sv_seq_vidx, K * kSeqHist)) || (rc = s->dalloc(&P.sv_seq_vval, K * kSeqHist)) ||
          (rc = s->dalloc(&P.sv_seq_vhas, K * kSeqHist)) || (rc = s->dalloc(&P.sv_seq_vcnt, K)))
        return rc;
      CK(cudaStreamSynchronize(s->stream));
    }
    s->P.sv_ep[svc] = idx;
    s->P.family |= 2u;   // from now on the round kernels with the service program compiled in
  }
  s->kinds[idx] = (uint8_t)kind;
  if (reuse) {
    // whatever was still queued for the old endpoint is gone with its queue: empty the ring, and
    // let the timing wheel drop what it still holds for the old name (sent before `born`)
    CK(cudaStreamSynchronize(s->stream));
    uint32_t tail = 0;
    CK(cudaMemcpy(&tail, s->P.tail + idx, 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(s->P.limit + idx, &tail, 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->P.head + idx, &tail, 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->P.ep_born + idx, &s->hs.next_id, 8, cudaMemcpyHostToDevice));
    if (s->P.sv_seq_cli) { const uint32_t zero = 0; CK(cudaMemcpy(s->P.sv_seq_cli + idx, &zero, 4, cudaMemcpyHostToDevice)); }
    s->names[idx] = id;
    s->mailbox[idx].clear();
  } else {
    s->names.push_back(id);
    s->mailbox.emplace_back();
    s->P.n_ep = idx + 1;
  }
  s->by_name[id] = idx;
  CK(cudaMemcpy(s->P.kind + idx, &s->kinds[idx], 1, cudaMemcpyHostToDevice));
  return (int)idx;
}

// Closed-loop clients: n endpoints "c<first_name>..", each bound to server k mod n_nodes, driven by
// gen_step inside the round kernel (csrc/ms_kernels.cu).
int ms_add_gen_clients(ms_sim* s, const ms_gen_config* gc, uint32_t first_name) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (!gc || gc->n_clients == 0 || gc->interval_ns <= 0 || gc->read_permille > 1000) { set_err("ms_add_gen_clients: bad configuration"); return MS_ERR_ARG; }
  if (s->P.gc) { set_err("ms_add_gen_clients: the generator's clients exist already"); return MS_ERR_ARG; }
  if (s->cfg.workload != MS_W_BROADCAST && s->cfg.workload != MS_W_GSET) {
    set_err("ms_add_gen_clients: the device generator drives the broadcast and g-set workloads");
    return MS_ERR_ARG;
  }
  if (s->P.n_shards > 1) { set_err("ms_add_gen_clients: single GPU only"); return MS_ERR_ARG; }
  if ((uint64_t)s->P.n_ep + gc->n_clients > s->cfg.max_endpoints) { set_err("max_endpoints exhausted"); return MS_ERR_CAPACITY; }
  Params& P = s->P;
  int rc;
  const uint32_t hist_cap = pow2_at_least(std::max<uint32_t>(1u << 16, 64u * gc->n_clients));
  if ((rc = s->dalloc(&P.gc, s->cfg.max_endpoints)) || (rc = s->dalloc(&P.gc_hist, (size_t)hist_cap * 2))) return rc;
  P.gc_hist_mask = hist_cap - 1u;
  P.gc_n = gc->n_clients;
  P.gc_read_permille = gc->read_permille;
  P.gc_interval_ns = gc->interval_ns;
  P.gc_timeout_ns = gc->timeout_ns > 0 ? gc->timeout_ns : 5000ll * kTickNs;      // client.clj:18-20
  P.gc_limit_ns = gc->time_limit_ns;
  P.gc_quiet_ns = gc->quiet_ns > 0 ? gc->quiet_ns : 10000ll * kTickNs;           // core.clj:75-78
  const uint32_t first = P.n_ep;
  std::vector<GenDev> init(gc->n_clients);
  memset(init.data(), 0, init.size() * sizeof(GenDev));
  for (uint32_t k = 0; k < gc->n_clients; k++) {
    const std::string id = "c" + std::to_string(first_name + k);
    if (s->by_name.count(id)) { set_err("endpoint already exists: " + id); return MS_ERR_ARG; }
    const uint32_t idx = first + k;
    s->kinds[idx] = MS_KIND_GEN_CLIENT;
    s->names.push_back(id);
    s->mailbox.emplace_back();
    s->by_name[id] = idx;
    init[k].node = k % s->cfg.n_nodes;
    init[k].ordinal = k;
  }
  P.n_ep = first + gc->n_clients;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaMemcpy(P.kind + first, s->kinds.data() + first, gc->n_clients, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(P.gc + first, init.data(), init.size() * sizeof(GenDev), cudaMemcpyHostToDevice));
  return (int)first;
}

int ms_history_drain(ms_sim* s, ms_hist* out, size_t cap, size_t* n_out) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (n_out) *n_out = 0;
  if (!s->P.gc_hist) return MS_OK;
  const uint64_t avail = s->hs.gc_hist_n - s->hs.gc_hist_drained;
  const size_t n = (size_t)std::min<uint64_t>(avail, cap);
  if (!n || !out) return MS_OK;
  static_assert(sizeof(ms_hist) == 32, "ms_hist is the device record");
  for (size_t k = 0; k < n;) {      // the ring may wrap
    const uint64_t pos = (s->hs.gc_hist_drained + k) & s->P.gc_hist_mask;
    const size_t piece = (size_t)std::min<uint64_t>(n - k, (uint64_t)s->P.gc_hist_mask + 1 - pos);
    CK(cudaMemcpy(out + k, s->P.gc_hist + pos * 2, piece * 32, cudaMemcpyDeviceToHost));
    k += piece;
  }
  // records of one round are appended in whatever order its CTAs ran: (time, round, client) is the order
  std::stable_sort(out, out + n, [](const ms_hist& a, const ms_hist& b) {
    return a.time_ns != b.time_ns ? a.time_ns < b.time_ns : a.order < b.order;
  });
  s->hs.gc_hist_drained += n;
  CK(cudaMemcpy(&s->P.st->gc_hist_drained, &s->hs.gc_hist_drained, 8, cudaMemcpyHostToDevice));
  if (n_out) *n_out = n;
  return MS_OK;
}

int ms_remove_endpoint(ms_sim* s, uint32_t idx) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (idx >= s->P.n_ep || (s->kinds[idx] & kRemoved)) { set_err("No such node in network"); return MS_ERR_NODE_NOT_FOUND; }
  s->by_name.erase(s->names[idx]);
  s->kinds[idx] |= kRemoved;   // the kind stays readable: a removed "c*" endpoint is still a client by name (util.clj:7-16)
  CK(cudaMemcpy(s->P.kind + idx, &s->kinds[idx], 1, cudaMemcpyHostToDevice));
  s->np.any_removed = 1;
  return s->push_np();
}

int ms_endpoint_index(ms_sim* s, const char* id) {
  std::lock_guard<std::mutex> g(s->mu);
  auto it = s->by_name.find(id ? id : "");
  if (it == s->by_name.end()) { set_err(std::string("No such node in network: ") + (id ? id : "")); return MS_ERR_NODE_NOT_FOUND; }
  return (int)it->second;
}

static int64_t send_locked(ms_sim* s, uint32_t src, uint32_t dest, const ms_body* b);

int64_t ms_send(ms_sim* s, uint32_t src, uint32_t dest, const ms_body* b) {
  std::lock_guard<std::mutex> g(s->mu);
  return send_locked(s, src, dest, b);
}

static int64_t send_locked(ms_sim* s, uint32_t src, uint32_t dest, const ms_body* b) {
  if (src >= s->P.n_ep || (s->kinds[src] & kRemoved)) { set_err("Invalid source for message"); return MS_ERR_NODE_NOT_FOUND; }
  if (dest >= s->P.n_ep || (s->kinds[dest] & kRemoved)) { set_err("Invalid dest for message"); return MS_ERR_NODE_NOT_FOUND; }
  if (!b) { set_err("null body"); return MS_ERR_ARG; }
  ms_msg m;
  memset(&m, 0, sizeof m);
  m.src = src; m.dest = dest; m.type = b->type; m.flags = b->flags;
  m.msg_id = b->msg_id; m.in_reply_to = b->in_reply_to; m.p0 = b->p0; m.p1 = b->p1;
  s->pending.push_back(m);
  return (int64_t)(s->hs.next_id + s->pending.size() - 1);
}

int ms_schedule_ops(ms_sim* s, const ms_op* ops, size_t n) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  const size_t first = s->sched.size();
  // validate the whole batch before anything is appended: a rejected batch leaves no orphans
  int64_t prev = first ? s->sched.back().time_ns : INT64_MIN;
  for (size_t i = 0; i < n; i++) {
    if (ops[i].time_ns < prev) { set_err("ops must be sorted by time"); return MS_ERR_ARG; }
    prev = ops[i].time_ns;
    if (ops[i].src >= s->P.n_ep || ops[i].dest >= s->P.n_ep || (s->kinds[ops[i].src] & kRemoved) ||
        (s->kinds[ops[i].dest] & kRemoved)) { set_err("scheduled op names an unknown endpoint"); return MS_ERR_NODE_NOT_FOUND; }
  }
  CK(cudaStreamSynchronize(s->stream));
  s->sched.insert(s->sched.end(), ops, ops + n);
  const int rc = s->upload_schedule(first);
  if (rc != MS_OK) s->sched.resize(first);   // keep host and device schedules identical
  return rc;
}

// true when the device refuses to run rounds until the host drains the journal
static bool journal_blocked(const ms_sim* s) {
  if (!s->cfg.journal_level || s->cfg.journal_discard) return false;
  // mirrors round_skipped(): after a sync no round is in flight, so the next round's raw_base == jraw_cursor
  if (s->hs.jraw_cursor - s->hs.jraw_drained > (s->P.jmask + 1) / 2) return true;
  return s->hs.round - s->hs.drain_round + 2 >= s->P.hist;
}

static int step_locked(ms_sim* s, uint64_t n_rounds, int64_t stop) {
  cudaSetDevice(s->device);
  int rc;
  if (s->P.n_shards > 1) {
    for (uint32_t g = 0; g < s->P.n_shards; g++)
      if (!s->P.ring_sh[g]) { set_err("sharded simulation: ms_shard_connect every peer first"); return MS_ERR_ARG; }
  }
  if ((rc = s->stage_injections())) return rc;
  if ((rc = s->set_stop(stop))) return rc;
  s->launch_rounds(n_rounds);
  {
    const cudaError_t le = cudaGetLastError();      // a launch that was refused never shows up in the stream
    if (le != cudaSuccess) { set_err(std::string("kernel launch: ") + cudaGetErrorString(le)); return MS_ERR_CUDA; }
  }
  if ((rc = s->sync_state())) return rc;
  return s->maybe_flush_journal_file();
}

// what the device state looks like when rounds stop advancing (appended to the error text)
static std::string stall_report(const ms_sim* s) {
  const DevState& h = s->hs;
  char buf[320];
  snprintf(buf, sizeof buf,
           " [round %llu now %lld stop %lld done %u slot_open %u rounds_run %llu drain_round %llu raw %llu/%llu events %llu/%llu "
           "lists %u+%u %u+%u %u+%u %u+%u]",
           (unsigned long long)h.round, (long long)h.now, (long long)h.stop_ns, h.done, h.slot_open,
           (unsigned long long)h.rounds_run, (unsigned long long)h.drain_round, (unsigned long long)h.jraw_drained,
           (unsigned long long)h.jraw_cursor, (unsigned long long)h.journal_drained, (unsigned long long)h.next_event,
           h.cls_count[h.round & 1][0], h.cls_small[h.round & 1][0], h.cls_count[h.round & 1][1], h.cls_small[h.round & 1][1],
           h.cls_count[h.round & 1][2], h.cls_small[h.round & 1][2], h.cls_count[h.round & 1][3], h.cls_small[h.round & 1][3]);
  return buf;
}

int ms_step(ms_sim* s, uint64_t n_rounds) {
  std::lock_guard<std::mutex> g(s->mu);
  // bounded batches so the journal file / mailbox keep up
  while (n_rounds) {
    if (journal_blocked(s)) { set_err("journal ring half full: drain it (ms_journal_drain) before stepping"); return MS_ERR_CAPACITY; }
    // one round at a time near the watermark so that "exactly n rounds" holds
    const bool near_full = s->cfg.journal_level && !s->cfg.journal_discard &&
                           (s->hs.jraw_cursor - s->hs.jraw_drained > (s->P.jmask + 1) / 4 ||
                            s->hs.round - s->hs.drain_round + 70 >= s->P.hist);
    const uint64_t b = near_full ? 1 : std::min<uint64_t>(n_rounds, 64);
    const uint64_t r0 = s->hs.rounds_run;
    const int rc = step_locked(s, b, INT64_MAX);
    if (rc) return rc;
    if (s->hs.rounds_run == r0) { set_err("simulation made no progress (device refuses to run rounds)" + stall_report(s)); return MS_ERR_SIM; }
    n_rounds -= std::min<uint64_t>(n_rounds, s->hs.rounds_run - r0);
  }
  return MS_OK;
}

// Virtual time only advances in a round that leaves nothing due "now" (DESIGN.md 2.3).  A node that
// sends zero-latency messages in every round forever (e.g. raft.py's replicate_log once a
// next_index has gone non-positive: it raises before recording the replication, so it replicates
// again in the next loop iteration) freezes it: report that instead of spinning.
static const uint64_t kMaxDeltaRounds = 1ull << 20;
static int time_stalled(ms_sim* s, int64_t now0, uint64_t round0) {
  if (s->hs.now != now0 || s->hs.rounds_run - round0 <= kMaxDeltaRounds) return 0;
  set_err("virtual time is not advancing: 2^20 delta rounds at the same instant (a node sends zero-latency "
          "messages in every round)");
  return 1;
}

int ms_run(ms_sim* s, int64_t until) {
  std::lock_guard<std::mutex> g(s->mu);
  int64_t stall_now = s->hs.now;
  uint64_t stall_round = s->hs.rounds_run;
  // batch sizing: nothing to hand to the host between rounds (no mailbox traffic, journal discarded or streamed
  // elsewhere) -> start from the previous call's round count, then grow while whole batches are productive
  // Sharded runs: every shard must issue the same launch sequence (the barriers pair up), so the decision may only
  // use what is identical on all shards -- the configuration, the endpoint table and the round counter -- and is
  // taken only when no endpoint has a host mailbox at all.
  bool adaptive = s->cfg.journal_discard || s->cfg.journal_level == 0;
  if (s->P.n_shards <= 1) {
    adaptive = adaptive && !s->mail_seen && s->pending.empty();
  } else {
    for (uint8_t k : s->kinds)
      if (!(k & kRemoved) && ((k & 0x7F) == MS_KIND_CLIENT || (k & 0x7F) == MS_KIND_HOST)) adaptive = false;
  }
  const uint64_t entry_rounds = s->hs.rounds_run;
  uint64_t batch = 32;
  if (adaptive) batch = s->run_hint > 36 ? std::min<uint64_t>(s->run_hint - 2, 1024) : 32;
  while (s->hs.now < until) {
    if (journal_blocked(s)) return 1;   // drain (ms_journal_drain) and call again
    const uint64_t r0 = s->hs.rounds_run;
    static const bool dbg_stall = getenv("MS_DEBUG_STALL") != nullptr;   // diagnostic: one round per batch, state on stderr
    if (dbg_stall) batch = 1;
    const int rc = step_locked(s, batch, until);
    if (rc) return rc;
    if (dbg_stall && (s->hs.rounds_run == r0 || s->hs.round < 4))
      fprintf(stderr, "MS_DEBUG_STALL advanced=%d%s cursors %u %u %u %u\n", (int)(s->hs.rounds_run - r0), stall_report(s).c_str(),
              s->hs.cls_cursor[s->hs.round & 1][0], s->hs.cls_cursor[s->hs.round & 1][1], s->hs.cls_cursor[s->hs.round & 1][2],
              s->hs.cls_cursor[s->hs.round & 1][3]);
    if (adaptive) {
      const bool full = s->hs.rounds_run - r0 == batch;
      batch = (s->mail_seen && s->P.n_shards <= 1) ? 32 : (full ? std::min<uint64_t>(std::max<uint64_t>(2 * batch, 4), 256) : 4);
      if (full && s->run_hint > 36 && s->hs.rounds_run - entry_rounds <= s->run_hint) batch = 4;   // the call's last rounds
    }
    if (s->hs.now != stall_now) { stall_now = s->hs.now; stall_round = s->hs.rounds_run; }
    else if (time_stalled(s, stall_now, stall_round)) return MS_ERR_SIM;
    if (s->hs.rounds_run == r0 && s->hs.now < until && !journal_blocked(s)) {
      set_err("simulation made no progress (device refuses to run rounds)" + stall_report(s));
      return MS_ERR_SIM;
    }
  }
  if (adaptive) s->run_hint = s->hs.rounds_run - entry_rounds;
  return MS_OK;
}

static int recv_locked(ms_sim* s, uint32_t e, int64_t timeout, ms_msg* out) {
  if (e >= s->P.n_ep || (s->kinds[e] & kRemoved)) { set_err("No such node in network"); return MS_ERR_NODE_NOT_FOUND; }
  const int64_t give_up = (timeout > INT64_MAX - s->hs.now) ? INT64_MAX : s->hs.now + timeout;
  int64_t stall_now = s->hs.now;
  uint64_t stall_round = s->hs.rounds_run;
  for (;;) {
    if (s->hs.now != stall_now) { stall_now = s->hs.now; stall_round = s->hs.rounds_run; }
    else if (time_stalled(s, stall_now, stall_round)) return MS_ERR_SIM;
    if (!s->mailbox[e].empty()) {
      *out = s->mailbox[e].front();
      s->mailbox[e].pop_front();
      return 1;
    }
    if (s->hs.now >= give_up) return 0;
    if (journal_blocked(s)) { set_err("journal ring half full: drain it (ms_journal_drain)"); return MS_ERR_CAPACITY; }
    const uint64_t r0 = s->hs.rounds_run;
    const int rc = step_locked(s, 1, INT64_MAX);
    if (!rc && s->hs.rounds_run == r0) { set_err("simulation made no progress (device refuses to run rounds)"); return MS_ERR_SIM; }
    if (rc) return rc;
  }
}

int ms_recv(ms_sim* s, uint32_t e, int64_t timeout, ms_msg* out) {
  std::lock_guard<std::mutex> g(s->mu);
  return recv_locked(s, e, timeout, out);
}

// ------------------------------------------------------------------ JSON data plane

// parse-msg + check-message (process.clj:26-66, net.clj:27-37), then the body's fixed-size encoding
int64_t ms_send_json(ms_sim* s, const char* line) {
  std::lock_guard<std::mutex> g(s->mu);
  if (!line) { set_err("null line"); return MS_ERR_ARG; }
  msj::Value m;
  std::string perr;
  if (!msj::Parser(line).parse(m, perr)) {
    set_err(std::string("Node printed a line to STDOUT which was not well-formed JSON (") + perr + "):\n" + line +
            "\nDid you mean to encode this line as JSON? Or was this line intended for STDERR? See doc/protocol.md for more guidance.");
    return MS_ERR_ARG;
  }
  // the Message schema: {:src NodeId, :dest NodeId, :body Any, (optional-key :id) Int}, nothing else
  std::string why;
  if (m.kind != msj::Value::Obj) why = "(not (map? message))";
  else {
    for (const auto& kv : m.obj)
      if (kv.first != "src" && kv.first != "dest" && kv.first != "body" && kv.first != "id") why += "{:" + kv.first + " disallowed-key} ";
    const msj::Value* v;
    if (!(v = m.get("src"))) why += "{:src missing-required-key} "; else if (v->kind != msj::Value::Str) why += "{:src (not (instance? java.lang.String))} ";
    if (!(v = m.get("dest"))) why += "{:dest missing-required-key} "; else if (v->kind != msj::Value::Str) why += "{:dest (not (instance? java.lang.String))} ";
    if (!m.get("body")) why += "{:body missing-required-key} ";
    if ((v = m.get("id")) && v->kind != msj::Value::Int) why += "{:id (not (integer? id))} ";
  }
  const msj::Value* body = why.empty() ? m.get("body") : nullptr;
  if (why.empty() && (body->kind != msj::Value::Obj || !body->get("type") || body->get("type")->kind != msj::Value::Str))
    why = "{:body (not a map with a string :type, doc/protocol.md:36-45)}";
  if (!why.empty()) {
    set_err(std::string("Malformed network message. Node tried to send the following message via STDOUT:\n\n") + line +
            "\n\nThis is malformed because:\n\n" + why + "\n\nSee doc/protocol.md for more guidance.");
    return MS_ERR_ARG;
  }
  auto idx = [&](const std::string& name, const char* what) -> int64_t {
    auto it = s->by_name.find(name);
    if (it == s->by_name.end()) { set_err(std::string("Invalid ") + what + " for message " + line); return MS_ERR_NODE_NOT_FOUND; }   // net.clj:172-175
    return it->second;
  };
  const int64_t src = idx(m.get("src")->s, "source"), dest = src < 0 ? src : idx(m.get("dest")->s, "dest");
  if (src < 0 || dest < 0) return MS_ERR_NODE_NOT_FOUND;
  const std::string t = body->get("type")->s;
  ms_body b;
  memset(&b, 0, sizeof b);
  b.type = s->type_code(t);
  std::map<std::string, std::string> rest;          // what no fixed field carries
  for (const auto& kv : body->obj) {
    const msj::Value& v = kv.second;
    const bool is_int = v.kind == msj::Value::Int;
    if (kv.first == "type") continue;
    if (kv.first == "msg_id" && is_int) { b.flags |= MS_F_MSG_ID; b.msg_id = (uint32_t)v.i; }
    else if (kv.first == "in_reply_to" && is_int) { b.flags |= MS_F_REPLY; b.in_reply_to = (uint32_t)v.i; }
    else if (t == "broadcast" && kv.first == "message" && is_int) b.p0 = (uint32_t)v.i;
    else if ((t == "add" || t == "replicate_one") && kv.first == "element" && is_int) b.p0 = (uint32_t)v.i;
    else if (t == "error" && kv.first == "code" && is_int) b.p0 = (uint32_t)v.i;
    else if ((t == "read" || t == "write" || t == "cas") && kv.first == "key" && is_int) b.p0 = (uint32_t)v.i;
    else if (t == "write" && kv.first == "value" && is_int) b.p1 = (b.p1 & ~0xFFFFFFFFull) | (uint32_t)v.i;
    else if (t == "cas" && kv.first == "from" && is_int) b.p1 = (b.p1 & ~0xFFFFFFFFull) | (uint32_t)v.i;
    else if (t == "cas" && kv.first == "to" && is_int) b.p1 = (b.p1 & 0xFFFFFFFFull) | ((uint64_t)(uint32_t)v.i << 32);
    else if (t == "cas" && kv.first == "create_if_not_exists") { if (v.kind == msj::Value::Bool && v.b) b.flags |= MS_F_CREATE; }
    else {
      if (t == "txn" && kv.first == "txn" && v.kind == msj::Value::Arr)
        for (const msj::Value& op : v.arr)
          if (op.kind == msj::Value::Arr && !op.arr.empty() && op.arr[0].kind == msj::Value::Str && op.arr[0].s == "append") b.flags |= MS_F_APPENDS;
      rest[kv.first] = v.text;
    }
  }
  if (!rest.empty()) {
    if (t == "write" || t == "cas") { set_err("write / cas bodies carry key, value / from, to only"); return MS_ERR_ARG; }
    b.p1 = ++s->next_blob;
    s->blobs[b.p1] = msj::object(rest);
  }
  return send_locked(s, (uint32_t)src, (uint32_t)dest, &b);
}

// the line a node process would read from STDIN (process.clj:162): {"id","src","dest","body"}
int ms_recv_json(ms_sim* s, uint32_t e, int64_t timeout, char* out, size_t cap) {
  std::lock_guard<std::mutex> g(s->mu);
  ms_msg m;
  const int rc = recv_locked(s, e, timeout, &m);
  if (rc != 1) return rc;
  std::map<std::string, std::string> body;
  const std::string t = s->type_name(m.type);
  body["type"] = msj::quote(t);
  if (m.flags & MS_F_MSG_ID) body["msg_id"] = std::to_string(m.msg_id);
  if (m.flags & MS_F_REPLY) body["in_reply_to"] = std::to_string(m.in_reply_to);
  const bool kv_peer = (m.src < s->kinds.size() && (s->kinds[m.src] & 0x7F) == MS_KIND_SERVICE) || s->cfg.workload == MS_W_RAFT;
  const uint32_t lo = (uint32_t)m.p1, hi = (uint32_t)(m.p1 >> 32);
  bool blob_ok = true;
  switch (m.type) {
    case MS_T_BROADCAST: body["message"] = std::to_string(m.p0); break;
    case MS_T_ADD: case MS_T_REPLICATE_ONE: body["element"] = std::to_string(m.p0); break;
    case MS_T_ERROR: {
      static const struct { uint32_t code; const char* text; } kErr[] = {   // resources/errors.edn
          {0, "timeout"}, {1, "node-not-found"}, {10, "not-supported"}, {11, "temporarily-unavailable"}, {12, "malformed-request"},
          {13, "crash"}, {14, "abort"}, {20, "key-does-not-exist"}, {21, "key-already-exists"}, {22, "precondition-failed"}, {30, "txn-conflict"}};
      body["code"] = std::to_string(m.p0);
      const char* text = "unknown";
      for (const auto& x : kErr) if (x.code == m.p0) text = x.text;
      body["text"] = msj::quote(text);
      break;
    }
    case MS_T_READ: if (kv_peer || (m.dest < s->kinds.size() && (s->kinds[m.dest] & 0x7F) == MS_KIND_SERVICE)) body["key"] = std::to_string(m.p0); break;
    case MS_T_WRITE: body["key"] = std::to_string(m.p0); body["value"] = std::to_string(lo); blob_ok = false; break;
    case MS_T_CAS:
      body["key"] = std::to_string(m.p0); body["from"] = std::to_string(lo); body["to"] = std::to_string(hi); blob_ok = false;
      if (m.flags & MS_F_CREATE) body["create_if_not_exists"] = "true";
      break;
    case MS_T_TS_OK: body["ts"] = std::to_string(m.p1); blob_ok = false; break;
    case MS_T_TXN_OK: body["versions"] = "[" + std::to_string(lo) + "," + std::to_string(hi) + "]"; blob_ok = false; break;
    case MS_T_READ_OK:
      if (kv_peer) { body["value"] = std::to_string(lo); blob_ok = false; }
      else if (m.src < s->cfg.n_nodes && s->P.bitmap) {
        // the device message carries the set size; the members are read back from the node
        // (broadcast: `messages`, workload/broadcast.clj:33-35; g-set: `value`, g_set.rb:14)
        std::vector<uint32_t> w(s->P.bm_words);
        if (cudaMemcpy(w.data(), s->P.bitmap + (size_t)m.src * s->P.bm_words, w.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
          set_err("ms_recv_json: cannot read the node's set"); return MS_ERR_CUDA;
        }
        std::string list = "[";
        uint32_t n = 0;
        for (uint32_t i = 0; i < s->P.bm_words && n < m.p0; i++)
          for (uint32_t bit = 0; bit < 32 && n < m.p0; bit++)
            if ((w[i] >> bit) & 1u) { list += (n ? "," : "") + std::to_string(i * 32 + bit); n++; }
        body[s->cfg.workload == MS_W_GSET ? "value" : "messages"] = list + "]";
        blob_ok = false;
      }
      break;
    default: break;
  }
  if (blob_ok && m.p1) {
    auto it = s->blobs.find(m.p1);
    if (it != s->blobs.end()) {                      // merge the stored object's members
      msj::Value v;
      std::string perr;
      if (msj::Parser(it->second).parse(v, perr) && v.kind == msj::Value::Obj)
        for (const auto& kv : v.obj) if (!body.count(kv.first)) body[kv.first] = kv.second.text;
    }
  }
  auto name_of = [&](uint32_t i) { return i < s->names.size() ? s->names[i] : std::to_string(i); };
  const std::string line = "{\"id\":" + std::to_string(m.id) + ",\"src\":" + msj::quote(name_of(m.src)) + ",\"dest\":" +
                           msj::quote(name_of(m.dest)) + ",\"body\":" + msj::object(body) + "}";
  if (!out || line.size() + 1 > cap) { set_err("ms_recv_json: buffer too small for " + std::to_string(line.size() + 1) + " bytes"); return MS_ERR_CAPACITY; }
  memcpy(out, line.c_str(), line.size() + 1);
  return 1;
}

int64_t ms_now(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return s->hs.now; }
uint64_t ms_round(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return s->hs.round; }

int ms_net_drop(ms_sim* s, uint32_t src, uint32_t dest) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  const uint32_t M = s->cfg.max_endpoints;
  if (src >= M || dest >= M) { set_err("drop!: endpoint out of range"); return MS_ERR_ARG; }
  if (!s->pair_alloc) {
    if (M > 65536) { set_err("pairwise drop! needs max_endpoints <= 65536; use ms_net_partition"); return MS_ERR_CAPACITY; }
    s->P.pair_words = (M + 31) / 32;
    int rc = s->dalloc(&s->P.pair_bits, (size_t)M * s->P.pair_words);
    if (rc) return rc;
    s->pair_alloc = true;
  }
  msk_set_bit(s->P.pair_bits, (size_t)dest * s->P.pair_words + (src >> 5), src & 31, s->stream);
  s->np.pair_active = 1;
  return s->push_np();
}

int ms_net_heal(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (s->pair_alloc && s->np.pair_active)
    CK(cudaMemsetAsync(s->P.pair_bits, 0, (size_t)s->cfg.max_endpoints * s->P.pair_words * 4, s->stream));
  s->np.pair_active = 0;
  s->np.comp_active = 0;
  return s->push_np();
}

int ms_net_slow(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  // scale stays a u32 and round(mean * scale * ln2 * 2^32) must fit the u64 exp_coeff
  if (s->np.scale > 100000000u || (double)s->np.mean_ms * (double)s->np.scale * 10.0 > 4.0e9) {
    set_err("slow!: latency scale overflow");
    return MS_ERR_ARG;
  }
  s->np.scale *= 10;
  recompute_exp(s);
  return s->push_np();
}

int ms_net_fast(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (s->np.scale >= 10) s->np.scale /= 10;
  recompute_exp(s);
  return s->push_np();
}

static int set_loss_locked(ms_sim* s, double p) {
  cudaSetDevice(s->device);
  s->np.loss_thresh = !(p > 0.0) ? 0 : (p >= 1.0 ? (1ull << 32) : (uint64_t)(p * 4294967296.0));
  return s->push_np();
}

int ms_net_flaky(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return set_loss_locked(s, 0.5); }
int ms_net_set_loss(ms_sim* s, double p) { std::lock_guard<std::mutex> g(s->mu); return set_loss_locked(s, p); }

int ms_net_partition(ms_sim* s, const uint32_t* comp, size_t n) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (n > s->cfg.max_endpoints) { set_err("partition vector longer than max_endpoints"); return MS_ERR_ARG; }
  std::vector<uint32_t> full(s->cfg.max_endpoints, 0);
  // endpoints not listed (index >= n) carry 0xFFFFFFFF = "never cut" (clients keep talking to every node)
  for (size_t i = 0; i < n; i++) full[i] = comp[i];
  for (size_t i = n; i < full.size(); i++) full[i] = 0xFFFFFFFFu;
  CK(cudaMemcpy(s->P.comp, full.data(), full.size() * 4, cudaMemcpyHostToDevice));
  s->np.comp_active = 1;
  return s->push_np();
}

int ms_journal_open(ms_sim* s, const char* path) {
  std::lock_guard<std::mutex> g(s->mu);
  if (s->jfile) { fclose(s->jfile); delete s->jfress; s->jfress = nullptr; }
  s->jfile = fopen(path, "wb");
  if (!s->jfile) { set_err(std::string("cannot open journal file ") + path); return MS_ERR_ARG; }
  const size_t plen = strlen(path);
  if (plen > 9 && !strcmp(path + plen - 9, ".fressian")) {
    // a stripe of net-journal/<stripe>.fressian (journal.clj:118-127): Fressian objects, no header
    if (s->cfg.journal_level < 2) {
      fclose(s->jfile); s->jfile = nullptr;
      set_err("a .fressian journal needs journal_level 2 (message bodies)");
      return MS_ERR_ARG;
    }
    s->jfress = new msf::Writer(s->jfile);
    return MS_OK;
  }
  const uint32_t hdr[4] = {0x314A534Du /* "MSJ1" */, s->cfg.journal_level, (uint32_t)sizeof(ms_event), (uint32_t)sizeof(ms_jbody)};
  fwrite(hdr, sizeof hdr, 1, s->jfile);
  return MS_OK;
}

int ms_journal_close(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  if (!s->jfile) return MS_OK;
  cudaSetDevice(s->device);
  const int rc = s->flush_journal_file();
  fclose(s->jfile);
  s->jfile = nullptr;
  delete s->jfress;
  s->jfress = nullptr;
  return rc;
}

int ms_journal_drain(ms_sim* s, ms_event* ev, ms_jbody* bodies, size_t cap, size_t* n_out) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  size_t n = 0;
  const int rc = s->drain(ev, bodies, cap, &n);
  if (n_out) *n_out = n;
  return rc;
}

uint64_t ms_journal_written(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return s->hs.next_event; }

static size_t stream_hdr_bytes() { return 256 + (size_t)ms_sim::kStreamRows * sizeof(ms_jround); }

int ms_run_streamed(ms_sim* s, int64_t until, int format, size_t buf_events, ms_journal_sink sink, void* ctx) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (format != MS_JFMT_EVENT && format != MS_JFMT_12 && format != MS_JFMT_8 && format != MS_JFMT_4) { set_err("ms_run_streamed: unknown format"); return MS_ERR_ARG; }
  if (!sink) { set_err("ms_run_streamed: null sink"); return MS_ERR_ARG; }
  if (s->cfg.journal_level == 0 || s->cfg.journal_discard) { set_err("ms_run_streamed: the journal is off (journal_level 0 or journal_discard)"); return MS_ERR_ARG; }
  if (!buf_events) buf_events = (size_t)1 << 24;
  const size_t hdr_bytes = stream_hdr_bytes();
  if (!s->jstream) {
    CK(cudaStreamCreateWithFlags(&s->jstream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++) {
      CK(cudaEventCreateWithFlags(&s->j_rounds_done[k], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&s->j_copied[k], cudaEventDisableTiming));
    }
    for (int k = 0; k < 4; k++) {
      CK(cudaEventCreateWithFlags(&s->j_packed[k], cudaEventDisableTiming));
      void* ptr = nullptr;
      CK(cudaHostAlloc(&ptr, hdr_bytes, cudaHostAllocPortable));
      s->jhdr[k] = (unsigned char*)ptr;
    }
    void* ptr = nullptr;
    CK(cudaMalloc(&ptr, msk_stream_plan_bytes()));
    s->allocs.push_back(ptr);
    s->jplan = ptr;
  }
  if (s->jhost_events < buf_events || s->jhost_format < format) {
    for (int k = 0; k < 2; k++) {
      if (s->jhost[k]) cudaFreeHost(s->jhost[k]);
      if (s->jdev[k]) cudaFree(s->jdev[k]);
      s->jhost[k] = nullptr; s->jdev[k] = nullptr;
      void* ptr = nullptr;
      const size_t rec = (s->P.n_shards > 1 && format < 16) ? 16 : (size_t)format;   // sharded: MS_JFMT_16 records
      CK(cudaHostAlloc(&ptr, buf_events * rec, cudaHostAllocPortable));
      s->jhost[k] = (unsigned char*)ptr;
      CK(cudaMalloc(&ptr, hdr_bytes + buf_events * rec));
      s->jdev[k] = (unsigned char*)ptr;
    }
    s->jhost_events = buf_events;
    s->jhost_format = format;
  }
  int rc;
  if ((rc = s->stage_injections())) return rc;
  if ((rc = s->set_stop(until))) return rc;
  // the shadow counters start from what has been drained so far
  {
    struct { uint64_t first, count, r0, n_rounds, jd, dr, jr; uint32_t ov, more; uint64_t local_n, hist[2][3], pad; } init =
        {0, 0, 0, 0, s->hs.journal_drained, s->hs.drain_round, s->hs.jraw_drained, 0, 0, 0,
         {{s->hs.journal_drained, s->hs.drain_round, s->hs.jraw_drained}, {s->hs.journal_drained, s->hs.drain_round, s->hs.jraw_drained}}, 0};
    static_assert(sizeof(init) == 128, "StreamPlan layout");
    CK(cudaMemcpyAsync(s->jplan, &init, sizeof init, cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
  }
  // Three batches are in flight: the rounds of batch i run (engine stream) while batch i-1 is packed
  // into device staging and copied out by the DMA engine (journal stream) and the caller's sink
  // looks at batch i-2 in pinned host memory.  The device skips rounds by itself when the raw ring is
  // half full, so a slow sink only slows the simulation down.
  // rounds launched per batch: 32 measured 9 % faster end to end than 8 on the broadcast bench (profiles/r2zz); three
  // batches are in flight, so stay well inside the round history
  // (sharded runs have no raw-ring back-pressure -- the ring must hold what three batches write -- so they keep 8)
  uint64_t batch_rounds = s->P.n_shards > 1 ? 8 : std::min<uint64_t>(32, std::max<uint64_t>(8, s->P.hist / 8));
  if (const char* br = getenv("MS_STREAM_BATCH_ROUNDS")) {            // tuning aid
    const long v = atol(br);
    if (v >= 1 && v <= 1024) batch_rounds = (uint64_t)v;
  }
  bool launching = true;
  int64_t stall_now = s->hs.now;
  uint64_t seen_round = s->hs.round, stall_round = s->hs.round;
  uint64_t idle_batches = 0, last_applied = 0;
  int result = MS_OK;
  for (uint64_t i = 0;; i++) {
    const int b = (int)(i & 1), hb = (int)(i & 3);
    if (launching) s->launch_rounds(batch_rounds);
    CK(cudaEventRecord(s->j_rounds_done[b], s->stream));
    CK(cudaStreamWaitEvent(s->jstream, s->j_rounds_done[b], 0));
    msk_stream_batch(&s->P, s->jplan, s->jhost_events, ms_sim::kStreamRows, (ms_jround*)(s->jdev[b] + 256),
                     s->jdev[b] + hdr_bytes, (ms_jbatch*)s->jdev[b], format, s->n_sms, s->jstream, (uint32_t)b);
    CK(cudaMemcpyAsync(s->jhdr[hb], s->jdev[b], hdr_bytes, cudaMemcpyDeviceToHost, s->jstream));
    CK(cudaEventRecord(s->j_packed[hb], s->jstream));
    if (i >= 1) {
      // batch i-1 is packed (its rounds ended a batch ago): now that its size is known, copy it out;
      // its drain counters reach the round kernels behind the rounds of batch i
      const uint64_t j = i - 1;
      CK(cudaEventSynchronize(s->j_packed[j & 3]));
      const ms_jbatch* hj = (const ms_jbatch*)s->jhdr[j & 3];
      if (hj->n_events)
        CK(cudaMemcpyAsync(s->jhost[j & 1], s->jdev[j & 1] + hdr_bytes, (size_t)hj->n_events * (size_t)hj->format,
                           cudaMemcpyDeviceToHost, s->jstream));
      CK(cudaEventRecord(s->j_copied[j & 1], s->jstream));
      CK(cudaStreamWaitEvent(s->stream, s->j_packed[j & 3], 0));
      msk_stream_apply(&s->P, s->jplan, s->stream, (uint32_t)(j & 1));
      last_applied = j;
    }
    if (i < 2) continue;
    const uint64_t k = i - 2;
    CK(cudaEventSynchronize(s->j_copied[k & 1]));
    const ms_jbatch* ph = (const ms_jbatch*)s->jhdr[k & 3];
    if (ph->overflow) { set_err("ms_run_streamed: MS_JFMT_4 / MS_JFMT_8 / MS_JFMT_12 cannot hold this batch (endpoint index or id range): use a wider format"); result = MS_ERR_CAPACITY; break; }
    if (ph->n_events && sink(ctx, ph, (const ms_jround*)(s->jhdr[k & 3] + 256), s->jhost[k & 1])) {
      set_err("ms_run_streamed: stopped by the sink");
      result = MS_ERR_ARG;
      break;
    }
    if (ph->error) break;                       // sync_state below reports it
    // (decisions below use what is the same on every shard of a sharded run: the range, not the local count)
    const bool progressed = ph->round != seen_round || ph->range_events != 0;
    seen_round = ph->round;
    if (ph->now != stall_now) { stall_now = ph->now; stall_round = seen_round; }
    else if (seen_round - stall_round > kMaxDeltaRounds) {
      set_err("virtual time is not advancing: 2^20 delta rounds at the same instant");
      result = MS_ERR_SIM;
      break;
    }
    if (ph->now >= until) launching = false;
    if (!launching && !ph->more && !progressed) break;      // nothing ran and nothing is left to pack
    idle_batches = progressed ? 0 : idle_batches + 1;
    if (idle_batches > 64) {
      char buf[384];
      snprintf(buf, sizeof buf, "simulation made no progress (device refuses to run rounds): streamed batch %llu now=%lld until=%lld "
               "round=%llu next_event=%llu first=%llu n=%llu more=%u err=%u launching=%d", (unsigned long long)k, (long long)ph->now,
               (long long)until, (unsigned long long)ph->round, (unsigned long long)ph->next_event, (unsigned long long)ph->first_event,
               (unsigned long long)ph->n_events, ph->more, ph->error, (int)launching);
      set_err(buf);
      result = MS_ERR_SIM;
      break;
    }
  }
  // everything packed is accounted for before the regular drain counters are trusted again
  CK(cudaStreamSynchronize(s->jstream));
  msk_stream_apply(&s->P, s->jplan, s->stream, (uint32_t)((last_applied + 1) & 1));
  msk_stream_apply(&s->P, s->jplan, s->stream, (uint32_t)(last_applied & 1));
  const std::string keep = g_err;
  rc = s->sync_state();
  if (!rc && result == MS_ERR_SIM) {
    char buf[256];
    snprintf(buf, sizeof buf, " [state: now=%lld stop=%lld round=%llu jraw_cursor=%llu jraw_drained=%llu drain_round=%llu journal_drained=%llu next_event=%llu slot_open=%u]",
             (long long)s->hs.now, (long long)s->hs.stop_ns, (unsigned long long)s->hs.round, (unsigned long long)s->hs.jraw_cursor,
             (unsigned long long)s->hs.jraw_drained, (unsigned long long)s->hs.drain_round, (unsigned long long)s->hs.journal_drained,
             (unsigned long long)s->hs.next_event, s->hs.slot_open);
    set_err(keep + buf);
  }
  return rc ? rc : result;
}

int ms_journal_decode(const ms_jbatch* b, const ms_jround* rounds, const void* events, ms_event* out) {
  if (!b || !rounds || !events || !out) return MS_ERR_ARG;
  if (b->n_events && !b->n_rounds) return MS_ERR_ARG;                     // every event belongs to a round row
  if (b->format == MS_JFMT_4) return MS_ERR_ARG;                         // needs the stream's history: ms_jdecoder_decode
  size_t r = 0;
  for (uint64_t k = 0; k < b->n_events; k++) {
    const uint64_t g = b->first_event + k;
    while (r + 1 < b->n_rounds && rounds[r + 1].ev_base <= g) r++;
    ms_event e;
    uint64_t id; uint32_t src, dest; bool recv;
    if (b->format == MS_JFMT_8) {
      const uint64_t w = ((const uint64_t*)events)[k];
      recv = (w >> 63) != 0; src = (uint32_t)(w >> 47) & 0xFFFFu; dest = (uint32_t)(w >> 31) & 0xFFFFu;
      id = rounds[r].id_ref + (w & 0x7FFFFFFFull);
    } else if (b->format == MS_JFMT_12) {
      const uint32_t* w = (const uint32_t*)events + 3 * k;
      id = (uint64_t)w[0] | ((uint64_t)(w[1] & 0x7FFFu) << 32);
      recv = (w[1] & 0x8000u) != 0;
      src = (w[1] >> 16) | ((w[2] & 0xFFu) << 16);
      dest = w[2] >> 8;
    } else if (b->format == MS_JFMT_16) {
      const uint64_t* w = (const uint64_t*)events + 2 * k;
      const uint64_t eid = w[0] & ~MS_EVENT_RECV;
      size_t rr = 0;
      while (rr + 1 < b->n_rounds && rounds[rr + 1].ev_base <= eid) rr++;
      e.event_id = w[0]; e.time_ns = rounds[rr].time_ns;
      e.msg_id = rounds[rr].id_ref + (w[1] & 0x7FFFFFFFull);
      e.src = (uint32_t)(w[1] >> 47) & 0xFFFFu; e.dest = (uint32_t)(w[1] >> 31) & 0xFFFFu;
      out[k] = e;
      continue;
    } else if (b->format == MS_JFMT_EVENT) {
      out[k] = ((const ms_event*)events)[k];
      continue;
    } else {
      return MS_ERR_ARG;
    }
    e.event_id = g | (recv ? MS_EVENT_RECV : 0ull);
    e.time_ns = rounds[r].time_ns;
    e.msg_id = id; e.src = src; e.dest = dest;
    out[k] = e;
  }
  return MS_OK;
}

// ------------------------------------------------------------------ ms_jdecoder (MS_JFMT_4 needs the stream's history)
struct ms_jdecoder {
  std::vector<uint64_t> tag, sd;     // per remembered send: its id + 1 (0 = empty), src | dest << 32
  uint64_t mask = 0;
  uint64_t next_send = 0;            // id of the next :send in stream order
  uint64_t expect_event = 0;         // event id right after the last event seen
  bool have = false;
  std::string err;
};

ms_jdecoder* ms_jdecoder_create(uint32_t log2_window) {
  if (log2_window < 4 || log2_window > 34) return nullptr;
  ms_jdecoder* d = new (std::nothrow) ms_jdecoder();
  if (!d) return nullptr;
  try {
    d->tag.assign((size_t)1 << log2_window, 0ull);
    d->sd.assign((size_t)1 << log2_window, 0ull);
  } catch (...) { delete d; return nullptr; }
  d->mask = ((uint64_t)1 << log2_window) - 1;
  return d;
}
void ms_jdecoder_destroy(ms_jdecoder* d) { delete d; }
const char* ms_jdecoder_error(const ms_jdecoder* d) { return d ? d->err.c_str() : "no decoder"; }

int ms_jdecoder_note(ms_jdecoder* d, const ms_event* ev, size_t n) {
  if (!d || (!ev && n)) return MS_ERR_ARG;
  for (size_t i = 0; i < n; i++) {
    const uint64_t g = ev[i].event_id & ~MS_EVENT_RECV;
    if (!(ev[i].event_id & MS_EVENT_RECV)) {
      d->tag[ev[i].msg_id & d->mask] = ev[i].msg_id + 1;
      d->sd[ev[i].msg_id & d->mask] = (uint64_t)ev[i].src | ((uint64_t)ev[i].dest << 32);
      d->next_send = ev[i].msg_id + 1;
    }
    d->expect_event = g + 1;
    d->have = true;
  }
  return MS_OK;
}

int ms_jdecoder_decode(ms_jdecoder* d, const ms_jbatch* b, const ms_jround* rounds, const void* events, ms_event* out) {
  if (!d || !b || !rounds || !events || !out) return MS_ERR_ARG;
  if (b->n_events && !b->n_rounds) { d->err = "ms_jdecoder: batch without round rows"; return MS_ERR_ARG; }
  if (b->format != MS_JFMT_4) {
    const int rc = ms_journal_decode(b, rounds, events, out);
    return rc ? rc : ms_jdecoder_note(d, out, (size_t)b->n_events);
  }
  const uint32_t* w = (const uint32_t*)events;
  size_t r = 0;
  for (uint64_t k = 0; k < b->n_events; k++) {
    const uint64_t g = b->first_event + k;
    while (r + 1 < b->n_rounds && rounds[r + 1].ev_base <= g) r++;
    if (g == rounds[r].ev_base) {
      d->next_send = rounds[r].id_ref;                   // a round starts: its sends count up from its first id
    } else if (k == 0 && (!d->have || d->expect_event != g)) {
      d->err = "ms_jdecoder: batch starts inside a round the decoder has not followed (event " + std::to_string(g) + ")";
      return MS_ERR_ARG;
    }
    ms_event e;
    e.time_ns = rounds[r].time_ns;
    if (w[k] & 0x80000000u) {
      const uint64_t id = rounds[r].id_ref - 1ull - (uint64_t)(w[k] & 0x7FFFFFFFu);
      if (d->tag[id & d->mask] != id + 1) {
        d->err = "ms_jdecoder: the :send of message " + std::to_string(id) + " is not in the decoder's window";
        return MS_ERR_ARG;
      }
      const uint64_t sd = d->sd[id & d->mask];
      e.event_id = g | MS_EVENT_RECV; e.msg_id = id; e.src = (uint32_t)sd; e.dest = (uint32_t)(sd >> 32);
    } else {
      const uint64_t id = d->next_send++;
      e.event_id = g; e.msg_id = id; e.src = (w[k] >> 16) & 0x7FFFu; e.dest = w[k] & 0xFFFFu;
      d->tag[id & d->mask] = id + 1;
      d->sd[id & d->mask] = (uint64_t)e.src | ((uint64_t)e.dest << 32);
    }
    out[k] = e;
  }
  d->expect_event = b->first_event + b->n_events;
  d->have = true;
  return MS_OK;
}

int ms_stats(ms_sim* s, uint64_t out[9]) {
  std::lock_guard<std::mutex> g(s->mu);
  // the device keeps {clients, servers} x {send, recv}; "all" is their sum
  const uint64_t snd[3] = {s->hs.stats[2] + s->hs.stats[4], s->hs.stats[2], s->hs.stats[4]};
  const uint64_t rcv[3] = {s->hs.stats[3] + s->hs.stats[5], s->hs.stats[3], s->hs.stats[5]};
  for (int c = 0; c < 3; c++) {
    out[c * 3 + 0] = snd[c];
    out[c * 3 + 1] = rcv[c];
    out[c * 3 + 2] = snd[c];   // every id has exactly one :send, so msg-count == send-count
  }
  return MS_OK;
}

size_t ms_node_set(ms_sim* s, uint32_t node, uint32_t* values, size_t cap) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (node >= s->cfg.n_nodes || !s->P.bitmap) return 0;
  std::vector<uint32_t> w(s->P.bm_words);
  if (cudaMemcpy(w.data(), s->P.bitmap + (size_t)node * s->P.bm_words, w.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess)
    return 0;
  size_t n = 0;
  for (uint32_t i = 0; i < s->P.bm_words; i++)
    for (uint32_t b = 0; b < 32; b++)
      if ((w[i] >> b) & 1u) { if (values && n < cap) values[n] = i * 32 + b; n++; }
  return n;
}

uint64_t ms_client_replies(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return s->hs.client_replies; }
uint64_t ms_undeliverable(ms_sim* s) { std::lock_guard<std::mutex> g(s->mu); return s->hs.undeliverable; }

int ms_raft_state(ms_sim* s, uint32_t node, uint64_t out[8]) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (!s->P.rf_node || node >= s->cfg.n_nodes) { set_err("ms_raft_state: not a Raft node"); return MS_ERR_ARG; }
  RaftDev r;
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaMemcpy(&r, s->P.rf_node + node, sizeof r, cudaMemcpyDeviceToHost));
  out[0] = (uint64_t)r.state; out[1] = r.term; out[2] = (uint64_t)(r.voted_for + 1); out[3] = r.commit_index;
  out[4] = r.last_applied; out[5] = (uint64_t)(r.leader + 1); out[6] = r.log_size; out[7] = r.kv_size;
  return MS_OK;
}

int ms_counters(ms_sim* s, uint64_t out[8]) {
  std::lock_guard<std::mutex> g(s->mu);
  out[0] = s->hs.rounds_run;
  out[1] = s->hs.stats[2] + s->hs.stats[4];
  out[2] = s->hs.stats[3] + s->hs.stats[5];
  out[3] = s->launches;
  out[4] = s->hs.lost;
  out[5] = s->hs.part_drops;
  out[6] = s->hs.max_window_seen;
  out[7] = s->hs.fallback_sorts;
  return MS_OK;
}

struct ShardBlob {   // MS_SHARD_BLOB_BYTES
  uint32_t magic, shard_id, n_shards, t_max;
  uint32_t max_endpoints, ring_cap, hist, pad;
  cudaIpcMemHandle_t ring, tail, head, rt_cnt, bar;
  cudaIpcMemHandle_t gs_snap, gs_tag;   // pad = 1: g-set snapshot rows, tags; pad = 2: Raft payload heap, handle table
  uint64_t ring_slots;                  // a peer's body plane starts ring_slots vectors into its ring
};
static_assert(sizeof(ShardBlob) <= MS_SHARD_BLOB_BYTES, "blob too large");

int ms_shard_handles(ms_sim* s, void* blob_out) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  ShardBlob b;
  memset(&b, 0, sizeof b);
  b.magic = 0x4253534Du;
  b.shard_id = s->P.shard_id; b.n_shards = s->P.n_shards; b.t_max = s->P.t_max;
  b.max_endpoints = s->cfg.max_endpoints; b.ring_cap = s->P.ring_cap ^ (s->P.ring_cap_s << 1); b.hist = s->P.hist;
  b.ring_slots = s->P.ring_slots;
  CK(cudaIpcGetMemHandle(&b.ring, s->P.ring));
  CK(cudaIpcGetMemHandle(&b.tail, s->P.tail));
  CK(cudaIpcGetMemHandle(&b.head, s->P.head));
  CK(cudaIpcGetMemHandle(&b.rt_cnt, s->P.rt_cnt));
  CK(cudaIpcGetMemHandle(&b.bar, s->P.bar_sh[s->P.shard_id]));
  if (s->P.gs_snap) {
    b.pad = 1;
    CK(cudaIpcGetMemHandle(&b.gs_snap, s->P.gs_snap));
    CK(cudaIpcGetMemHandle(&b.gs_tag, s->P.gs_tag));
  } else if (s->P.rf_heap) {
    b.pad = 2;
    CK(cudaIpcGetMemHandle(&b.gs_snap, s->P.rf_heap));
    CK(cudaIpcGetMemHandle(&b.gs_tag, s->P.rf_ext_off));
  }
  memset(blob_out, 0, MS_SHARD_BLOB_BYTES);
  memcpy(blob_out, &b, sizeof b);
  return MS_OK;
}

int ms_shard_connect(ms_sim* s, uint32_t peer, const void* blob) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  ShardBlob b;
  memcpy(&b, blob, sizeof b);
  if (b.magic != 0x4253534Du || b.shard_id != peer || peer >= s->P.n_shards || b.n_shards != s->P.n_shards ||
      b.t_max != s->P.t_max || b.max_endpoints != s->cfg.max_endpoints || b.ring_cap != (s->P.ring_cap ^ (s->P.ring_cap_s << 1)) ||
      b.hist != s->P.hist || b.ring_slots != s->P.ring_slots) {
    set_err("ms_shard_connect: peer blob does not match this simulation's configuration");
    return MS_ERR_ARG;
  }
  if (peer == s->P.shard_id) return MS_OK;
  void* ptr = nullptr;
  CK(cudaIpcOpenMemHandle(&ptr, b.ring, cudaIpcMemLazyEnablePeerAccess));
  s->peer_ptrs.push_back(ptr); s->P.ring_sh[peer] = (uint4*)ptr;
  CK(cudaIpcOpenMemHandle(&ptr, b.tail, cudaIpcMemLazyEnablePeerAccess));
  s->peer_ptrs.push_back(ptr); s->P.tail_sh[peer] = (uint32_t*)ptr;
  CK(cudaIpcOpenMemHandle(&ptr, b.head, cudaIpcMemLazyEnablePeerAccess));
  s->peer_ptrs.push_back(ptr); s->P.head_sh[peer] = (uint32_t*)ptr;
  CK(cudaIpcOpenMemHandle(&ptr, b.rt_cnt, cudaIpcMemLazyEnablePeerAccess));
  s->peer_ptrs.push_back(ptr); s->P.rt_cnt_sh[peer] = (uint64_t*)ptr;
  CK(cudaIpcOpenMemHandle(&ptr, b.bar, cudaIpcMemLazyEnablePeerAccess));
  s->peer_ptrs.push_back(ptr); s->P.bar_sh[peer] = (uint32_t*)ptr;
  if ((b.pad == 1) != (s->P.gs_snap != nullptr) || (b.pad == 2) != (s->P.rf_heap != nullptr)) {
    set_err("ms_shard_connect: peer runs another workload");
    return MS_ERR_ARG;
  }
  if (b.pad == 2) {
    const size_t N = s->cfg.n_nodes;
    CK(cudaIpcOpenMemHandle(&ptr, b.gs_snap, cudaIpcMemLazyEnablePeerAccess));
    s->peer_ptrs.push_back(ptr); s->P.rf_heap_sh[peer] = (uint4*)ptr;
    CK(cudaIpcOpenMemHandle(&ptr, b.gs_tag, cudaIpcMemLazyEnablePeerAccess));
    s->peer_ptrs.push_back(ptr); s->P.rf_ext_off_sh[peer] = (uint64_t*)ptr;
    s->P.rf_ext_tag_sh[peer] = reinterpret_cast<uint32_t*>((uint64_t*)ptr + N * kRaftExt);
  }
  if (b.pad == 1) {
    CK(cudaIpcOpenMemHandle(&ptr, b.gs_snap, cudaIpcMemLazyEnablePeerAccess));
    s->peer_ptrs.push_back(ptr); s->P.gs_snap_sh[peer] = (uint32_t*)ptr;
    CK(cudaIpcOpenMemHandle(&ptr, b.gs_tag, cudaIpcMemLazyEnablePeerAccess));
    s->peer_ptrs.push_back(ptr); s->P.gs_tag_sh[peer] = (uint32_t*)ptr;
  }
  return MS_OK;
}

int ms_set_barrier(ms_sim* s, ms_barrier_fn fn, void* ctx) {
  std::lock_guard<std::mutex> g(s->mu);
  s->barrier = fn;
  s->barrier_ctx = ctx;
  return MS_OK;
}

void* ms_stream(ms_sim* s) { return (void*)s->stream; }

uint32_t ms_shard_owner(uint32_t e, uint32_t n_servers, uint32_t n_shards) { return owner_of(e, n_servers, n_shards); }

int ms_timer_begin(ms_sim* s) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (!s->t0) { CK(cudaEventCreate(&s->t0)); CK(cudaEventCreate(&s->t1)); }
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaEventRecord(s->t0, s->stream));
  return MS_OK;
}

int ms_timer_end(ms_sim* s, double* elapsed_ms) {
  std::lock_guard<std::mutex> g(s->mu);
  cudaSetDevice(s->device);
  if (!s->t0) { set_err("ms_timer_end without ms_timer_begin"); return MS_ERR_ARG; }
  CK(cudaEventRecord(s->t1, s->stream));
  CK(cudaEventSynchronize(s->t1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, s->t0, s->t1));
  if (elapsed_ms) *elapsed_ms = ms;
  return MS_OK;
}

int ms_profile(ms_sim* s, int enable) {
  std::lock_guard<std::mutex> g(s->mu);
  s->profiling = enable != 0;
  return MS_OK;
}

int ms_debug_phase_cycles(ms_sim* s, int enable, uint64_t out[64]) {
  std::lock_guard<std::mutex> g(s->mu);
#ifndef MS_PHASE_TIMING
  if (enable) { set_err("this library was built without -DMS_PHASE_TIMING (the per-phase clock reads are compiled out of the product kernels)"); return MS_ERR_ARG; }
#endif
  cudaSetDevice(s->device);
  if (enable && !s->P.phase_cycles) {
    int rc = s->dalloc(&s->P.phase_cycles, 512);
    if (rc) return rc;
    CK(cudaStreamSynchronize(s->stream));
  }
  if (out) {
    if (s->P.phase_cycles) CK(cudaMemcpy(out, s->P.phase_cycles, 64 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    else memset(out, 0, 64 * sizeof(uint64_t));
  }
  if (s->P.phase_cycles && enable >= 0) CK(cudaMemset(s->P.phase_cycles, 0, 64 * sizeof(uint64_t)));
  if (enable == 2 && out) {   // diagnostic: first overlapping-block window, written to stderr
    std::vector<uint64_t> d(448);
    CK(cudaMemcpy(d.data(), s->P.phase_cycles + 64, 448 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (d[0]) {
      fprintf(stderr, "overlap window: e=%llu n=%llu R=%llu round=%llu\n", (unsigned long long)d[1], (unsigned long long)d[2],
              (unsigned long long)d[3], (unsigned long long)d[4]);
      for (uint64_t q = 0; q < d[3] && q < 64; q++)
        fprintf(stderr, "  block %llu: round=%llu ticket=%llu first_idx=%llu last_idx=%llu\n", (unsigned long long)q,
                (unsigned long long)(d[5 + 2 * q] >> 24), (unsigned long long)(d[5 + 2 * q] & 0xFFFFFF),
                (unsigned long long)(d[6 + 2 * q] >> 32), (unsigned long long)(d[6 + 2 * q] & 0xFFFFFFFFu));
    }
  }
  return MS_OK;
}

int ms_profile_read(ms_sim* s, double* ms, uint64_t* launches) {
  std::lock_guard<std::mutex> g(s->mu);
  if (ms) *ms = s->prof_ms;
  if (launches) *launches = s->prof_launches;
  s->prof_ms = 0;
  s->prof_launches = 0;
  return MS_OK;
}

size_t ms_topology(uint32_t topology, uint32_t n, uint32_t node, uint32_t* out, size_t cap) {
  std::vector<uint32_t> nb;
  topo_neighbors(topology, n, node, nb);
  for (size_t i = 0; i < nb.size() && i < cap; i++) out[i] = nb[i];
  return nb.size();
}

}  // extern "C"
