// ms_device.cuh -- device-side data layout and pure helpers of the sm_100a
// discrete-event engine.  Mirrors the deterministic spec in DESIGN.md section 2;
// reference citations are relative to /root/reference.
#pragma once
#include <stdint.h>
#include "../../include/maelstrom_b200.h"

#if defined(__CUDACC__)
#define MS_HD __host__ __device__ __forceinline__
#else
#define MS_HD inline
#endif

namespace msd {

constexpr int64_t  kTickNs   = 1000000;       // latencies are integer ms (net.clj:187,204)
constexpr uint32_t kInjector = 0xFFFFFFFFu;   // Philox "emitter" of host/scheduled sends
constexpr uint8_t  kRemoved  = 0x80;          // flag or-ed into the endpoint kind by remove-node!

// device-latched error codes (DevState.error)
enum : uint32_t {
  E_NONE = 0, E_RING_OVERFLOW = 1, E_WINDOW_OVERFLOW = 2, E_JOURNAL_OVERFLOW = 3,
  E_INVALID_DEST = 4, E_HISTORY = 5, E_VALUE_RANGE = 6, E_MAIL_OVERFLOW = 7,
  E_CALENDAR_OVERFLOW = 8, E_ID_RANGE = 9, E_BARRIER = 10, E_SNAPSHOT = 11,
  E_RAFT_CAPACITY = 12, E_HISTORY_RING = 13
};

// Mutable per-simulation scalars, resident in HBM, committed by the last CTA of
// every round (net.clj:92-103's atom, minus the queues).
// default CTA widths of the four window-size classes of k_round (windows <= 128 / 512 / 2048 / max_window);
// ms_engine.cu sizes the launches with them, ms_kernels.cu's shape-specialised instantiations assume them
#ifndef MS_CLS0_NT
#define MS_CLS0_NT 64
#endif
#ifndef MS_CLS1_NT
#define MS_CLS1_NT 128
#endif
constexpr int kClsThreads[4] = {MS_CLS0_NT, MS_CLS1_NT, 256, 512};
constexpr uint32_t kClsLadder[4] = {128u, 512u, 2048u, 32768u};

struct DevState {
  int64_t  now;              // virtual time, ns
  int64_t  stop_ns;          // rounds are no-ops once now >= stop_ns
  uint64_t round;            // round counter
  uint64_t next_id;          // next-message-id (net.clj:103,197): id base of the round in flight
  uint64_t next_event;       // journal next-id (journal.clj:195): event base of the round in flight
  uint64_t journal_drained;  // events the host has consumed
  uint64_t drain_round;      // first round whose events are not fully drained
  uint64_t jraw_cursor;      // raw journal claim cursor (16-B records)
  uint64_t jraw_drained;     // raw records below this are free
  uint64_t stats[6];         // {all,clients,servers} x {send,recv}  (net/checker.clj:28-41)
  uint64_t lost;             // sends dropped by the loss roll (net.clj:214-215)
  uint64_t part_drops;       // receives cut by a partition (net.clj:234)
  uint64_t client_replies;   // replies consumed by MS_KIND_SIM_CLIENT sinks
  uint64_t rounds_run;
  uint64_t fallback_sorts;   // windows that needed the full bitonic sort
  uint64_t undeliverable;    // sends whose src / dest was not a registered endpoint: journaled, then dropped
  uint64_t gc_hist_n;        // history records written
  uint64_t gc_hist_drained;  // ... and handed to the host
  uint32_t done;             // CTAs finished this round
  uint32_t zero_pending;     // messages sent this round that are due at `now`
  uint32_t error;            // first latched E_* code
  uint32_t error_arg;
  uint32_t inj_count;        // host sends staged for the next round
  uint32_t sched_cursor;     // next unscheduled op
  uint32_t mail_count;       // host-visible deliveries since the last sync
  uint32_t time_advanced;    // 1 when the last round moved `now`
  uint32_t max_window_seen;
  uint32_t cal_release;      // calendar slot to release before the next round (+1), 0 = none
  uint32_t cal_free_n;       // free blocks of the timing-wheel pool
  uint32_t cal_ret_n;        // entries of Params.cal_ret
  uint32_t slot_open;        // k_snapshot ran for this launch slot and the round has not been committed yet
  uint32_t bar_epoch;        // cross-shard barriers executed so far
  // per-round work lists of the k_round size classes, double-buffered by round parity
  uint32_t cls_count[2][4];   // tickets at the front of the class list (the longer windows)
  uint32_t cls_small[2][4];   // tickets at the back of the class list
  uint32_t cls_cursor[2][4];
};

// One row per round, kept in a ring of `hist` rounds: what is needed to turn an
// order key (round, ticket, idx) into the dense message id the reference's
// global counter would have produced, and raw journal chunks into events.
struct RoundMeta {
  uint64_t round;
  int64_t  now;
  uint64_t id_base;          // next-message-id at the start of the round
  uint64_t ev_base;          // journal next-id at the start of the round
  uint64_t raw_base;         // jraw_cursor at the start of the round
  uint32_t n_tickets;
  uint32_t pad;
  uint64_t ev_total, em_total;
};

// Fault / latency knobs mutated by jepsen-net calls between rounds (net.clj:105-122).
struct NetParams {
  uint64_t loss_thresh;      // (< (rand) p-loss), net.clj:214; x0 < loss_thresh
  uint64_t exp_coeff;        // round(mean*scale*ln2*2^32)
  uint32_t dist;             // MS_DIST_*
  uint32_t mean_ms;
  uint32_t scale;            // 10^k after k slow! calls
  uint32_t pair_active;      // any drop! since the last heal!
  uint32_t comp_active;      // bulk partition installed
  uint32_t any_removed;      // some endpoint has been removed (remove-node! / stop-node!): sends check their endpoints' kinds
};

struct Params {
  DevState* st;
  NetParams* np;
  // endpoints
  uint8_t*  kind;
  uint32_t* tail;            // claim counter per endpoint ring
  uint32_t* limit;           // snapshot of tail at the start of the round
  uint32_t* head;            // previous snapshot: window is [head, limit)
  uint64_t* ep_born;         // next-message-id when the endpoint slot was (re)registered: wheel records with a smaller id are not for it
  uint4*    ring;            // 48-B records in two planes (DESIGN.md 3.1): ring_slots 16-B order keys, then
                             // ring_slots 32-B bodies; slots: n_servers rings of ring_cap_s, then rings of ring_cap
  uint64_t  ring_slots;      // slots of all rings together (equal on every shard)
  uint32_t  ring_cap, ring_cap_s;      // per endpoint: others / servers (powers of two)
  uint32_t  n_ep, n_servers, n_inj_tickets, max_window, max_window_s;
  // per-round history (ring of `hist` rows, stride t_max entries)
  RoundMeta* rmeta;
  uint32_t* rt_em;           // emissions per ticket, exclusive prefix once the round is committed
  uint32_t* rt_ev;           // events per ticket, exclusive prefix once committed
  uint64_t* rt_chunk;        // raw journal position of the ticket's chunk
  uint64_t* rt_cnt;          // tagged per-ticket counts of the round in flight (see k_round epilogue)
  uint64_t* phase_cycles;    // diagnostic: [4 classes][16] cycle sums per k_round phase, or nullptr
  // sharding: arrays of every shard, reachable over NVLink peer memory (index = shard)
  uint32_t  n_shards, shard_id;
  uint4*    ring_sh[8];
  uint32_t* tail_sh[8];
  uint32_t* head_sh[8];
  uint64_t* rt_cnt_sh[8];
  uint32_t* bar_sh[8];       // bar_sh[g][s] = last barrier epoch shard s signalled to shard g
  uint32_t  hist, hist_mask, t_max, n_classes;
  uint32_t  split_commit;    // the round is committed by its own launch(es) after the round kernels (sharded runs, very many tickets)
  uint64_t* cm_blk;          // three-phase commit: per-block sums / offsets (nullptr = single-CTA k_commit)
  uint32_t* cm_flags;        // [0] zero-latency pending, [1] row being committed, [2] phase B committed
  uint32_t* cls_list;        // [2][4][t_max] tickets per size class
  uint32_t  cls_cap[4];      // ascending window capacities of the classes
  // raw journal: 16-B records, chunk per (round, ticket); bodies (level 2) 32 B at the same index
  uint4*    jraw;
  uint4*    jbody;
  uint64_t  jmask;
  uint32_t  jlevel, jdiscard;
  // partitions
  uint32_t* pair_bits;       // [dest][src] bitmap, row stride pair_words
  uint32_t  pair_words;
  uint32_t* comp;
  uint32_t  seed_lo, seed_hi;
  // workload state
  uint32_t  workload, topology, n_values, bm_words;
  uint32_t* bitmap;          // n_servers * bm_words
  uint32_t* nbr_off;         // CSR neighbor table (absent for MS_TOPO_TOTAL)
  uint32_t* nbr;
  uint32_t* next_msg_id;     // echo.rb:8
  uint32_t* set_count;
  // injection
  ms_msg*   inj_buf;
  const ms_op* sched;
  uint32_t  n_sched;
  const uint32_t* tick_off;  // tick_off[j] = #ops whose injection tick is < j
  uint32_t  n_tick_off;
  // host-visible deliveries
  ms_msg*   mail;
  uint32_t  mail_cap;
  // calendar (timing wheel) for latencies > 0
  // Slot s holds the messages whose deadline tick is == s (mod cal_slots).  A slot is a chain
  // of fixed-size blocks taken from one pool, so memory follows the messages in flight, not
  // slots x worst case; a latency of cal_slots ticks or more stays in its slot for `laps` more
  // turns of the wheel (kept in the record while it waits).  Two generations per slot: the one
  // being released and the one being filled (a release re-files the records with laps left).
  uint4*    cal;             // pool: cal_blocks blocks of (1 << cal_blk_log2) 48-B records
  uint32_t* cal_count;       // [2][cal_slots] records filed under (generation, slot)
  uint32_t* cal_tab;         // [2][cal_slots][cal_tab_cap] block id + 1 of the j-th block of the chain, 0 = none yet
  uint32_t* cal_par;         // [cal_slots] generation new records of the slot go to
  uint32_t* cal_free;        // stack of free block ids (DevState.cal_free_n entries): popped while rounds run
  uint32_t* cal_ret;         // blocks popped but not needed (lost a publish race); pushed back by k_snapshot
  uint32_t  cal_slots, cal_blk_log2, cal_blocks, cal_tab_cap;
  // g-set node program (demo/ruby/g_set.rb): the set is `bitmap`; replicate_full payloads are
  // snapshots of it, kept in gs_slots rotating rows per node (row = node * gs_slots + run % gs_slots)
  uint8_t*  gs_init;         // init received: the periodic task is running (node.rb:22-36,129-137)
  int64_t*  gs_next_fire;    // virtual time of the task's next run (g_set.rb:34)
  uint32_t* gs_fires;        // runs so far; run k (1-based) is the p1 of its replicate_full messages
  uint32_t* gs_tag;          // [row] run number whose snapshot the row holds
  uint32_t* gs_snap;         // [row][bm_words]
  uint32_t  gs_slots, gs_interval_ms;
  // services (service.clj): device-resident lin-kv / seq-kv / lww-kv / lin-tso endpoints
  uint32_t  family;          // node-program families compiled into the round kernel in use: bit 0 g-set, bit 1 services
  uint32_t  sv_ep[4];        // endpoint index of service MS_SVC_*, 0xFFFFFFFF = not started
  uint32_t  sv_n_keys;       // keys per store
  uint32_t* sv_lin_val;      // lin-kv: Linearizable(PersistentKV), service.clj:31-58,147-156
  uint8_t*  sv_lin_has;
  uint32_t* sv_lww_val;      // lww-kv: two replicas (service.clj:218-251; they never merge, see oracle)
  uint8_t*  sv_lww_has;
  uint64_t* sv_scalars;      // [0] lin-tso counter (service.clj:123-129), [1] seq-kv last-index
  uint32_t* sv_seq_cli;      // seq-kv: per client (endpoint) last observed state index (service.clj:162-166)
  uint32_t* sv_seq_vidx;     // seq-kv: per key a ring of kSeqHist versions {state index, value, present}
  uint32_t* sv_seq_vval;
  uint8_t*  sv_seq_vhas;
  uint32_t* sv_seq_vcnt;     // versions written per key
  // g-set snapshots of every shard (index = shard): a replicate_full is merged by reading the
  // sender's snapshot row where it lives, over NVLink peer memory when the sender is remote
  uint32_t* gs_snap_sh[8];
  uint32_t* gs_tag_sh[8];
  // Raft nodes (MS_W_RAFT, demo/python/raft.py); layouts in ms_raft.cuh
  struct RaftDev* rf_node;   // [n_servers] scalar state
  uint4*    rf_log;          // [n_servers][rf_log_cap] entries, 2 vectors each
  uint32_t* rf_kv_val;       // [n_servers][rf_n_keys] KVStore (raft.py:151-192)
  uint8_t*  rf_kv_has;
  int32_t*  rf_next;         // [n_servers][rf_gmax] next_index / match_index by cluster member (leader state)
  int32_t*  rf_match;
  int32_t*  rf_scratch;      // [n_servers][rf_gmax] median scratch
  uint4*    rf_cb;           // [n_servers][rf_cb_mask + 1] pending RPC closures, 2 vectors each
  uint32_t* rf_votes;        // [n_servers][rf_vote_words] by cluster member
  uint4*    rf_stage;        // [n_servers][rf_stage_cap] emissions of the node's step, 3 vectors each
  uint4*    rf_heap;         // append_entries payloads: ring of vectors
  unsigned long long* rf_heap_cursor;
  uint64_t* rf_ext_off;      // [n_servers][kRaftExt] heap offset of the sender's k-th append_entries
  uint32_t* rf_ext_tag;      // [n_servers][kRaftExt] k
  uint32_t  rf_log_cap, rf_n_keys, rf_stage_cap, rf_heap_mask, rf_vote_words;
  uint32_t  rf_group;        // servers per Raft cluster (0 = one cluster of all servers)
  uint32_t  rf_gmax;         // row stride of rf_next / rf_match / rf_scratch = largest cluster
  uint32_t  rf_cb_mask;      // pending-RPC table slots per node - 1 (power of two)
  // MS_W_TXN_TREE (csrc/ms_tree.h, tt_handle in csrc/ms_raft.cuh)
  struct TreeDev* tt_node;   // [n_servers]
  unsigned char* tt_recs;    // [1 + n_servers * tt_per_node] 64-B tree node records by pointer - 1
  uint32_t* tt_cache;        // [n_servers][tt_cache_mask + 1] pointers in the node's @@cache (open addressing, 0 = empty)
  uint4*    tt_queue;        // [n_servers][kTreeQueue] txn requests waiting for the node's txn_lock
  uint32_t  tt_per_node, tt_cache_mask;
  // closed-loop clients (ms_add_gen_clients)
  struct GenDev* gc;         // [max_endpoints], valid where kind == MS_KIND_GEN_CLIENT
  uint4*    gc_hist;         // ring of 32-B history records (ms_hist)
  uint32_t  gc_hist_mask, gc_n, gc_read_permille, gc_pad;
  int64_t   gc_interval_ns, gc_timeout_ns, gc_limit_ns, gc_quiet_ns;
  // append_entries payloads of every shard (index = shard): read where the sender wrote them
  uint4*    rf_heap_sh[8];
  uint64_t* rf_ext_off_sh[8];
  uint32_t* rf_ext_tag_sh[8];
};

constexpr uint32_t kRaftCallbacks = 4096;       // default pending-RPC table slots per node (ms_config.reserved[5]; oracle: same)
constexpr uint32_t kRaftExt = 1024;             // append_entries payload handles kept per sender
constexpr int64_t  kElectionTimeoutNs = 2000000000;   // raft.py:199
constexpr int64_t  kHeartbeatNs = 1000000000;         // raft.py:200
constexpr int64_t  kMinReplicationNs = 50000000;      // raft.py:201
enum : int32_t { RAFT_NASCENT = 0, RAFT_FOLLOWER = 1, RAFT_CANDIDATE = 2, RAFT_LEADER = 3 };

struct RaftDev {
  int32_t  state;
  uint32_t term;
  int32_t  voted_for, leader;          // -1 = none
  uint32_t commit_index, last_applied;
  int64_t  election_deadline, step_down_deadline, last_replication;
  uint32_t next_msg_id, log_size, appends, n_votes, kv_size;
  uint32_t busy;                       // leader with a follower behind its log (or a next_index <= 0): see rf_timer_due
};

// MS_W_TXN_TREE node (demo/ruby/datomic_list_append.rb DatomicListAppendNode, :322-417)
constexpr uint32_t kTreeQueue = 256;     // txn requests that can wait for one node's @txn_lock (more = capacity error)
struct TreeDev {
  uint32_t ptr_counter;                // @ptr (:355-358)
  uint32_t phase;                      // 0 idle, 1 root read out, 2 tree node read out, 3 writes out, 4 cas out
  uint32_t cur_src, cur_msg_id;        // the txn request holding @txn_lock
  uint64_t cur_ops;
  uint32_t root1, root2, start_counter, writes_left, write_failed, load_ptr;
  uint32_t q_head, q_tail;             // requests waiting for the lock
  uint32_t init_src, init_msg_id;      // the init request (first node: answered after the initial state is written)
  uint32_t init_phase;                 // 0 none, 1 the empty tree's write is out, 2 the root's write is out
  uint32_t gen;                        // transactions finished: a reply that belongs to an earlier one finds nobody waiting
  uint32_t first_write, first_write_ok, root_is_leaf;   // save!: tasks[0] and whether it was delivered; Leaf#save! vs Branch#save!
  uint32_t pad;
  int64_t  deadline, init_deadline;    // Promise#await gives up after 5 s (promise.rb:6,24-31); 0 = nobody waits
};
constexpr int64_t kPromiseTimeoutNs = 5000000000ll;

// closed-loop client (maelstrom.client + a Jepsen worker), one per MS_KIND_GEN_CLIENT endpoint
struct GenDev {
  uint32_t next_msg_id, waiting_for;   // client.clj:52,61-76
  int64_t  deadline_ns;                // when the outstanding request times out (client.clj:96-101)
  int64_t  next_op_ns;                 // stagger: earliest time of the next invocation
  uint32_t node;                       // the server this client talks to
  uint32_t ops, bcasts;                // ops invoked so far, broadcasts among them
  uint32_t phase;                      // 0 mix, 1 quiet period, 2 final read outstanding, 3 done
  uint32_t cur_f, cur_value;           // the op in flight
  uint32_t ordinal, pad;               // k of client k
};
enum : uint32_t { GEN_MIX = 0, GEN_QUIET = 1, GEN_FINAL = 2, GEN_DONE = 3 };

constexpr uint32_t kSeqBuffer = 32;             // (sequential 32 ...), service.clj:206-208
constexpr uint32_t kSeqHist = kSeqBuffer + 1;   // versions per key that can matter to a resident state

// ------------------------------------------------------------- Philox4x32-10
// Salmon et al. SC'11 (the generator cuRAND names Philox_4x32_10).  Stands in
// for the reference's unseeded (rand) / Incanter draws (net.clj:187,214).
MS_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                         uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int i = 0; i < 10; i++) {
    const uint64_t a = (uint64_t)0xD2511F53u * c0;
    const uint64_t b = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(b >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(a >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)b;
    c3 = (uint32_t)a;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

MS_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

MS_HD int clz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
  return __clzll((long long)x);
#else
  return __builtin_clzll(x);
#endif
}

// -log2(u) in Q32.32 for u = (X+1)/2^64; integer-only (DESIGN.md 2.5).
MS_HD uint64_t neg_log2_q32(uint64_t X) {
  if (X == ~0ull) return 0;
  const uint64_t Y = X + 1;
  const int n = 63 - clz64(Y);
  uint64_t m = Y << (63 - n);
  uint32_t frac = 0;
  for (int i = 31; i >= 0; i--) {
    const uint64_t hi = mulhi64(m, m);
    if (hi >> 63) { frac |= (1u << i); m = hi; }
    else          { m = hi << 1; }
  }
  return (64ull << 32) - (((uint64_t)n << 32) | frac);
}

// latency in ms for a server<->server message (net.clj:65-77,178-187)
MS_HD uint64_t latency_ms(const NetParams& np, const uint32_t x[4]) {
  if (np.dist == MS_DIST_CONSTANT) return (uint64_t)np.mean_ms * np.scale;
  if (np.dist == MS_DIST_UNIFORM)
    return (((uint64_t)x[1] * (2ull * np.mean_ms)) >> 32) * np.scale;
  const uint64_t X = ((uint64_t)x[2] << 32) | x[1];
  return mulhi64(neg_log2_q32(X), np.exp_coeff);
}

MS_HD bool kind_is_client(uint8_t k) { k &= 0x7F; return k == MS_KIND_CLIENT || k == MS_KIND_SIM_CLIENT || k == MS_KIND_GEN_CLIENT; }

// Shard that owns endpoint e: servers are split into G contiguous index ranges (rows of the
// grid stay together), every other endpoint round-robin.  Injector tickets belong to shard 0.
MS_HD uint32_t owner_of(uint32_t e, uint32_t n_servers, uint32_t G) {
  if (G <= 1) return 0;
  if (e < n_servers) return (uint32_t)(((uint64_t)e * G) / n_servers);
  return (e - n_servers) % G;
}
MS_HD uint32_t owner_of_ticket(uint32_t t, uint32_t n_inj, uint32_t n_servers, uint32_t G) {
  return t < n_inj ? 0u : owner_of(t - n_inj, n_servers, G);
}

}  // namespace msd
