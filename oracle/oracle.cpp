// oracle/oracle.cpp -- TEST INFRASTRUCTURE ONLY (see oracle/oracle.h header).
//
// Single-threaded, obviously-sequential restatement of maelstrom.net
// (/root/reference/src/maelstrom/net.clj) and the canonical node programs,
// under the deterministic refinement in DESIGN.md section 2.  Every rule cites
// the reference line it follows.  Nothing here is tuned for speed beyond what
// makes it usable as the measured "CPU restatement" baseline.
//
// Round structure (DESIGN.md 2.3):
//   round r runs at virtual time now_r.
//   (1) injector: host-queued sends (call order), then scheduled ops with
//       time <= now_r (schedule order) are sent.
//   (2) endpoints in ascending index: pop every envelope with deadline <= now_r
//       that was enqueued in a round < r, in (deadline, id) order
//       (net.clj:39-40,145 orders by deadline only; ties are unspecified in the
//       JDK heap, the spec breaks them by id); partition check at dequeue
//       (net.clj:234); journal :recv (net.clj:244); run the node program; the
//       node's emissions are sent right after its receives.
//   (3) messages sent in round r become visible to receivers in round r+1.
//   (4) if anything is due at now_r, the next round is a delta round at the same
//       time, otherwise time advances by one tick (1 ms).
#include "../maelstrom_b200/csrc/ms_tree.h"   // tree arithmetic of datomic_list_append.rb, shared with the engine (see its header)
#include "oracle.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <deque>
#include <map>
#include <queue>
#include <set>
#include <string>
#include <vector>

namespace {

constexpr int64_t kTickNs = 1000000;  // latencies are integer ms (net.clj:187,204)
constexpr uint32_t kInjector = 0xFFFFFFFFu;

// ---------------------------------------------------------------- Philox4x32-10
// Salmon et al., "Parallel random numbers: as easy as 1, 2, 3" (SC'11); the
// same generator cuRAND calls Philox_4x32_10.  Replaces the reference's
// unseeded (rand) (net.clj:214) and Incanter draws (net.clj:187).
inline void philox_round(uint32_t c[4], const uint32_t k[2]) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
  const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
  const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
  const uint32_t n0 = hi1 ^ c[1] ^ k[0];
  const uint32_t n1 = lo1;
  const uint32_t n2 = hi0 ^ c[3] ^ k[1];
  const uint32_t n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}

void philox(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
  uint32_t k[2] = {key[0], key[1]};
  for (int i = 0; i < 10; i++) {
    if (i) { k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u; }
    philox_round(c, k);
  }
  for (int i = 0; i < 4; i++) out[i] = c[i];
}

// ------------------------------------------------------------- latency (net.clj:65-77,178-187)
// Integer-only so CPU and GPU agree bit for bit (DESIGN.md 2.5).
//   constant     -> mean * scale                         (net.clj:42-49, 51-53)
//   uniform      -> scale * floor(u * 2*mean), u in [0,1) (integer-distribution 0 (* 2 mean))
//   exponential  -> floor(scale * mean * -ln(u)), u in (0,1]; (long (* scale (draw d)))
// -ln(u) is evaluated in fixed point: u = (X+1)/2^64 for 64 random bits X,
// log2 by normalise + 32 squarings (each squaring keeps the top 64 bits).
uint64_t neg_log2_q32(uint64_t X) {
  if (X == ~0ull) return 0;       // u == 1
  const uint64_t Y = X + 1;       // in [1, 2^64-1]
  const int n = 63 - __builtin_clzll(Y);
  uint64_t m = Y << (63 - n);     // Q1.63 in [1,2)
  uint32_t frac = 0;
  for (int i = 31; i >= 0; i--) {
    const uint64_t hi = (uint64_t)(((unsigned __int128)m * m) >> 64);  // Q2.62 in [1,4)
    if (hi >> 63) { frac |= (1u << i); m = hi; }
    else          { m = hi << 1; }
  }
  const uint64_t log2y = ((uint64_t)n << 32) | frac;
  return (64ull << 32) - log2y;   // -log2(u), Q32.32
}

uint64_t exp_coeff(uint32_t mean_ms, uint32_t scale) {
  // round(mean * scale * ln2 * 2^32); a double multiply and llround, done on
  // the host CPU by both the oracle and the engine's host side.
  const double c = (double)mean_ms * (double)scale * 0.693147180559945309417232121458 * 4294967296.0;
  return (uint64_t)std::llround(c);
}

uint64_t latency_draw(uint32_t dist, uint32_t mean_ms, uint32_t scale, const uint32_t x[4]) {
  switch (dist) {
    case OR_DIST_CONSTANT:
      return (uint64_t)mean_ms * scale;
    case OR_DIST_UNIFORM: {
      const uint64_t span = 2ull * mean_ms;
      return (((uint64_t)x[1] * span) >> 32) * scale;
    }
    case OR_DIST_EXPONENTIAL: {
      const uint64_t X = ((uint64_t)x[2] << 32) | x[1];
      const uint64_t L = neg_log2_q32(X);
      const uint64_t C = exp_coeff(mean_ms, scale);
      return (uint64_t)(((unsigned __int128)L * C) >> 64);
    }
  }
  return 0;
}

uint64_t loss_threshold(double p) {
  // (< (rand) p-loss), net.clj:214, with (rand) := x0 / 2^32.
  if (!(p > 0.0)) return 0;
  if (p >= 1.0) return 1ull << 32;
  return (uint64_t)(p * 4294967296.0);
}

// ------------------------------------------------------------- topologies (workload/broadcast.clj:40-178)
std::vector<uint32_t> topology_neighbors(uint32_t topo, uint32_t n, uint32_t k) {
  std::vector<uint32_t> out;
  if (k >= n) return out;
  switch (topo) {
    case OR_TOPO_GRID: {  // broadcast.clj:40-65
      const int64_t side = (int64_t)std::ceil(std::sqrt((double)n));
      const int64_t i = k / side, j = k % side;
      auto node = [&](int64_t a, int64_t b) -> int64_t {
        if (a > -1 && b > -1 && b < side) {        // (< -1 i) (< -1 j side)
          const int64_t idx = a * side + b;
          if (idx < (int64_t)n) return idx;
        }
        return -1;
      };
      const int64_t cand[4] = {node(i + 1, j), node(i - 1, j), node(i, j + 1), node(i, j - 1)};
      for (int64_t c : cand) if (c >= 0) out.push_back((uint32_t)c);
      break;
    }
    case OR_TOPO_LINE: {  // broadcast.clj:67-80
      if (n < 2) break;
      if (k == 0) out.push_back(1);
      else if (k == n - 1) out.push_back(n - 2);
      else { out.push_back(k - 1); out.push_back(k + 1); }
      break;
    }
    case OR_TOPO_TOTAL: {  // broadcast.clj:82-89
      for (uint32_t i = 0; i < n; i++) if (i != k) out.push_back(i);
      break;
    }
    case OR_TOPO_TREE2: case OR_TOPO_TREE3: case OR_TOPO_TREE4: {  // broadcast.clj:91-167
      const uint32_t b = topo == OR_TOPO_TREE2 ? 2 : topo == OR_TOPO_TREE3 ? 3 : 4;
      // tiers of size 1, b, b^2.. filled in order; children of the p-th node of a
      // tier are the next b nodes of the tier below => heap layout.
      if (k > 0) out.push_back((k - 1) / b);         // parent first (:163-165)
      for (uint32_t c = 0; c < b; c++) {
        const uint64_t ch = (uint64_t)b * k + 1 + c;
        if (ch < n) out.push_back((uint32_t)ch);
      }
      break;
    }
  }
  return out;
}

// ------------------------------------------------------------- simulator state
struct Envelope {           // {:deadline :message}, net.clj:219-220
  or_msg m;
  uint64_t sent_round;
};
struct EnvCmp {             // latency-compare (net.clj:39-40) + id tie-break
  bool operator()(const Envelope& a, const Envelope& b) const {
    if (a.m.deadline_ns != b.m.deadline_ns) return a.m.deadline_ns > b.m.deadline_ns;
    return a.m.id > b.m.id;
  }
};
typedef std::priority_queue<Envelope, std::vector<Envelope>, EnvCmp> Queue;

struct Emit {                 // one emission of a node program
  explicit Emit(const or_msg& mm) : m(mm) {}
  or_msg m;
  bool has_snap = false;
  std::vector<uint32_t> snap; // read_ok value list (the set as of the read)
};

// ------------------------------------------------------------- services (service.clj)
struct KVMap {                // PersistentKV's / LWWKV's :m (values only: timestamps never decide anything, see Service)
  std::map<uint32_t, uint32_t> m;
  bool operator==(const KVMap& o) const { return m == o.m; }
};

struct SvcReply {
  bool reply = false;         // false: `case` had no matching clause -> exception, logged, no reply (service.clj:262-263)
  uint16_t type = 0;
  uint32_t p0 = 0;
  uint64_t p1 = 0;
};

// PersistentKV/handle (service.clj:31-58); lww = LWWKV/handle (service.clj:66-95), whose cas has no
// create_if_not_exists branch.  Returns the new state.
static KVMap kv_handle(const KVMap& st, const or_body& q, bool lww, SvcReply& r) {
  KVMap out = st;
  const uint32_t k = q.p0;
  auto it = st.m.find(k);
  r = SvcReply();
  switch (q.type) {
    case OR_T_READ:
      r.reply = true;
      if (it != st.m.end()) { r.type = OR_T_READ_OK; r.p1 = it->second; }
      else { r.type = OR_T_ERROR; r.p0 = 20; }                           // key does not exist
      break;
    case OR_T_WRITE:
      r.reply = true; r.type = OR_T_WRITE_OK;
      out.m[k] = (uint32_t)q.p1;
      break;
    case OR_T_CAS: {
      const uint32_t from = (uint32_t)q.p1, to = (uint32_t)(q.p1 >> 32);
      r.reply = true;
      if (it != st.m.end()) {
        if (it->second == from) { out.m[k] = to; r.type = OR_T_CAS_OK; }
        else { r.type = OR_T_ERROR; r.p0 = 22; }                         // precondition failed
      } else if (!lww && (q.flags & OR_F_CREATE)) {
        out.m[k] = to; r.type = OR_T_CAS_OK;
      } else { r.type = OR_T_ERROR; r.p0 = 20; }
      break;
    }
    default: break;
  }
  return out;
}

struct Service {
  int type = OR_SVC_LIN_KV;
  KVMap lin;                               // Linearizable(PersistentKV): one state in an atom (service.clj:147-156)
  uint64_t ts = 0;                         // PersistentTSO (service.clj:123-129)
  // Sequential (service.clj:168-214): ring buffer of states, last index, per-client last observed index
  std::deque<KVMap> buffer;
  uint32_t buffer_size = 32;
  uint64_t last_index = 0;
  std::map<uint32_t, uint64_t> clients;
  // Eventual(2 x LWWKV) (service.clj:218-251).  The merged replica computed at :229-232 is
  // dropped: the second `replicas'` binding (:236) rebuilds from the unmerged vector.  So the
  // replicas never exchange state and LWW timestamps never decide anything; a request is
  // handled by replica (rand-int 2).
  KVMap replicas[2];

  SvcReply handle(uint32_t client, const or_body& q, uint32_t rnd) {
    SvcReply r;
    switch (type) {
      case OR_SVC_LIN_KV: {
        KVMap st2 = kv_handle(lin, q, false, r);
        if (r.reply) lin = st2;
        return r;
      }
      case OR_SVC_LIN_TSO:
        if (q.type == OR_T_TS) { r.reply = true; r.type = OR_T_TS_OK; r.p1 = ts++; }
        return r;
      case OR_SVC_LWW_KV: {
        const uint32_t i = rnd >> 31;                                    // (rand-int 2)
        KVMap st2 = kv_handle(replicas[i], q, true, r);
        if (r.reply) replicas[i] = st2;
        return r;
      }
      default: break;
    }
    // Sequential
    if (buffer.empty()) buffer.push_back(KVMap());
    auto ci_it = clients.find(client);
    const uint64_t ci = ci_it == clients.end() ? 0 : ci_it->second;
    uint64_t index = ci + (((uint64_t)rnd * (last_index - ci + 1)) >> 32);   // :182-186
    // states older than the ring buffer are gone; the reference indexes the buffer with a
    // negative offset (:190) whose out-of-range behaviour belongs to amalloy/ring-buffer
    // (third party, absent).  Spec: use the oldest resident state.
    const uint64_t oldest = last_index + 1 - buffer.size();
    if (index < oldest) index = oldest;
    const KVMap& st = buffer[(size_t)(index - oldest)];
    KVMap st2 = kv_handle(st, q, false, r);
    if (!r.reply) return r;                                             // exception inside swap!: nothing changes
    if (st2 == st) {                                                    // :195-199
      clients[client] = index;
      return r;
    }
    KVMap latest2 = kv_handle(buffer.back(), q, false, r);              // :203-209
    last_index++;
    clients[client] = last_index;
    buffer.push_back(latest2);
    if (buffer.size() > buffer_size) buffer.pop_front();
    return r;
  }
};

// ------------------------------------------------------------- Raft node (demo/python/raft.py)
constexpr uint32_t kRaftCallbacks = 4096;      // pending-RPC table slots (the reference's dict is unbounded)
constexpr int64_t kElectionTimeoutNs = 2000000000;     // raft.py:199
constexpr int64_t kHeartbeatNs = 1000000000;           // raft.py:200
constexpr int64_t kMinReplicationNs = 50000000;        // raft.py:201
enum { RAFT_NASCENT = 0, RAFT_FOLLOWER = 1, RAFT_CANDIDATE = 2, RAFT_LEADER = 3 };

struct RaftEntry {             // {'term': t, 'op': body + 'client'}  (raft.py:118-121,553-556)
  uint32_t term = 0;
  uint16_t type = 0, flags = 0;
  uint32_t key = 0, client = 0, msg_id = 0;
  uint64_t p1 = 0;
};
struct RaftCb {                // what the RPC's closure captured (raft.py:282-303, 413-432)
  uint32_t msg_id = 0;
  int kind = 0;                // 0 free, 1 request_vote, 2 append_entries
  uint32_t term = 0, node = 0;
  int64_t ni = 0;
  uint32_t n_entries = 0;
};
struct RaftAppend {            // body of one append_entries (raft.py:424-431)
  uint32_t prev_log_index = 0, prev_log_term = 0, leader_commit = 0;
  std::vector<RaftEntry> entries;
};
struct RaftNode {
  int state = RAFT_NASCENT;
  uint32_t term = 0;
  int64_t voted_for = -1, leader = -1;
  uint32_t commit_index = 0, last_applied = 1;                   // raft.py:214-215
  int64_t election_deadline = 0, step_down_deadline = 0, last_replication = 0;
  uint32_t next_msg_id = 0;                                      // raft.py:42
  std::vector<RaftEntry> log = std::vector<RaftEntry>(1);        // the default entry {term 0, op None} (raft.py:121)
  std::map<uint32_t, uint32_t> kv;
  std::vector<int64_t> next_index, match_index;
  std::vector<RaftCb> callbacks;                                 // sized by or_create (cfg.rpc_table)
  std::set<uint32_t> votes;
  uint64_t appends = 0;
  uint32_t draws = 0;                                            // random draws made in the current round
};

struct TreeNode {              // DatomicListAppendNode (datomic_list_append.rb:322-417)
  uint32_t ptr_counter = 0;                                      // @ptr
  int phase = 0;                                                 // 0 idle, 1 root read out, 2 tree node read out, 3 writes out, 4 cas out
  uint32_t cur_src = 0, cur_msg_id = 0;
  uint64_t cur_ops = 0;
  uint32_t root1 = 0, root2 = 0, start_counter = 0, writes_left = 0, write_failed = 0;
  std::deque<or_msg> waiting;                                    // threads blocked on @txn_lock, in arrival order
  std::set<uint32_t> cache;                                      // @@cache
  uint32_t init_src = 0, init_msg_id = 0;
  int init_phase = 0;                                            // 0 none, 1 the empty tree's write is out, 2 the root's write is out
  uint32_t gen = 0;                                              // transactions finished (a late reply finds a dead promise)
  uint32_t first_write = 0; bool first_write_ok = false, root_is_leaf = false;   // save!: tasks[0]; Leaf#save! vs Branch#save!
  int64_t deadline = 0, init_deadline = 0;                       // Promise#await gives up after 5 s (promise.rb:6,24-31)
};
static const int64_t kPromiseTimeoutNs = 5000000000ll;

struct Endpoint {
  std::string name;
  int kind = OR_KIND_SERVER;
  bool live = true;
  Queue q;                              // net.clj:145
  std::deque<or_msg> mailbox;           // delivered to a host-visible endpoint
  // node program state
  uint32_t next_msg_id = 0;             // echo.rb:8,12
  std::set<uint32_t> values;            // broadcast @messages / g-set @set
  std::vector<uint32_t> neighbors;      // broadcast @neighbors (topology)
  bool initialized = false;             // node.rb:22-36: periodic tasks start after init
  int64_t next_fire = 0;                // g-set: next run of the `every 5` task (g_set.rb:34)
  uint64_t fires = 0;                   // g-set: replication runs so far
  Service svc;                          // OR_KIND_SERVICE
  RaftNode rn;                          // OR_W_RAFT servers
  TreeNode tn;                          // OR_W_TXN_TREE servers
  // OR_KIND_GEN_CLIENT: maelstrom.client state (client.clj:41-64) + where the worker is in its generator
  struct Gen {
    uint32_t next_msg_id = 0, waiting_for = 0;
    int64_t deadline_ns = 0, next_op_ns = 0;
    uint32_t node = 0, ops = 0, bcasts = 0, phase = 0, cur_f = 0, cur_value = 0, ordinal = 0;
  } gen;
};

}  // namespace

struct or_sim {
  or_config cfg;
  std::vector<Endpoint> eps;
  int64_t now = 0;
  uint64_t round = 0;
  uint64_t next_id = 0;        // next-message-id starts at -1, first id 0 (net.clj:103,197)
  uint64_t next_event = 0;     // journal next-id (journal.clj:195,228)
  uint32_t scale = 1;          // slow!/fast! (net.clj:115-119)
  uint64_t loss_thresh = 0;
  std::set<std::pair<uint32_t, uint32_t>> partitions;  // (dest, src), net.clj:109-110
  std::vector<uint32_t> component;                     // bulk partition
  std::vector<or_event> journal;
  std::vector<or_body> bodies;                         // body of the message of each event
  std::deque<or_msg> host_queue;                       // pending host sends
  std::vector<or_op> schedule;
  size_t sched_cursor = 0;
  std::map<uint64_t, std::vector<uint32_t>> snapshots; // read_ok msg id -> set contents
  // replicate_full payloads: (sender, p1 = sender's replication run, 1-based) -> value list
  std::map<std::pair<uint32_t, uint64_t>, std::vector<uint32_t>> gset_snaps;
  uint64_t client_replies = 0;
  uint64_t undelivered = 0;    // sends whose src / dest was not a registered endpoint
  // nodes address a service by name: the index at which a service of that name was last added, live or
  // not (a send to a removed one is undeliverable, net.clj:166-176); -1 = never added
  int svc_last[4] = {-1, -1, -1, -1};
  or_gen_config gcfg = {0, 0, 0, 0, 0, 0};
  std::vector<or_hist> history;
  std::string error;
  uint64_t stats[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};

  // util.clj:7-10 goes by the name ("c..."): a removed client is still a client
  bool is_client(uint32_t e) const {
    return e < eps.size() && (eps[e].kind == OR_KIND_CLIENT || eps[e].kind == OR_KIND_SIM_CLIENT || eps[e].kind == OR_KIND_GEN_CLIENT);
  }
  bool involves_client(const or_msg& m) const {                                // util.clj:12-16
    return is_client(m.src) || is_client(m.dest);
  }
  bool partitioned(uint32_t src, uint32_t dest) const {                        // net.clj:234
    if (partitions.count(std::make_pair(dest, src))) return true;
    // bulk partition: endpoints beyond the list, or listed as 0xFFFFFFFF, are never cut
    if (!component.empty() && src < component.size() && dest < component.size() &&
        component[src] != component[dest] && component[src] != 0xFFFFFFFFu && component[dest] != 0xFFFFFFFFu)
      return true;
    return false;
  }

  void log_event(bool recv, const or_msg& m) {      // journal.clj:225-239
    or_event ev;
    ev.event_id = next_event++ | (recv ? (1ull << 63) : 0);
    ev.time_ns = now;
    ev.msg_id = m.id;
    ev.src = m.src;
    ev.dest = m.dest;
    journal.push_back(ev);
    or_body b;
    b.type = m.type; b.flags = m.flags; b.msg_id = m.msg_id;
    b.in_reply_to = m.in_reply_to; b.p0 = m.p0; b.p1 = m.p1;
    bodies.push_back(b);
    // net/checker.clj:28-41 folded on the fly
    const bool cl = involves_client(m);
    const int k = recv ? 1 : 0;
    stats[0 + k]++;
    stats[(cl ? 3 : 6) + k]++;
  }

  // net.clj:189-221
  bool send(uint32_t emitter, uint32_t emit_idx, or_msg m, std::vector<Envelope>& pending) {
    // :166-176: the asserts throw inside the sender's own thread (process.clj:148-150) after the id
    // was taken (:197); the network keeps running.  Spec (DESIGN.md 2.4): the id is consumed, the
    // :send is journaled, the message is dropped and counted.
    const bool undeliverable = m.src >= eps.size() || !eps[m.src].live || m.dest >= eps.size() || !eps[m.dest].live;
    m.id = next_id++;                                                             // :197
    const uint32_t ctr[4] = {emit_idx, emitter, (uint32_t)round, (uint32_t)(round >> 32)};
    const uint32_t key[2] = {cfg.seed_lo, cfg.seed_hi};
    uint32_t x[4];
    philox(ctr, key, x);
    const uint64_t lat_ms = involves_client(m) ? 0                                // :185-186
                                               : latency_draw(cfg.latency_dist, cfg.latency_mean_ms, scale, x);
    m.deadline_ns = now + (int64_t)lat_ms * kTickNs;                              // :202-205
    log_event(false, m);                                                          // :208 (always, before the loss roll)
    if (undeliverable) { undelivered++; return true; }
    if ((uint64_t)x[0] < loss_thresh) return true;                                // :214-215
    Envelope env; env.m = m; env.sent_round = round;
    pending.push_back(env);                                                       // :216-221 (visible next round)
    return true;
  }

  // ---- node programs: append emissions (src/dest/body filled) to `out`
  static or_msg reply_to(const or_msg& req, uint16_t type) {   // node.rb:88-91
    or_msg r; std::memset(&r, 0, sizeof r);
    r.src = req.dest; r.dest = req.src; r.type = type;
    r.flags = OR_F_REPLY; r.in_reply_to = req.msg_id;
    return r;
  }

  void node_echo(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    Endpoint& ep = eps[e];
    if (m.type == OR_T_INIT || m.type == OR_T_ECHO) {       // echo.rb:28-39
      or_msg r = reply_to(m, m.type == OR_T_INIT ? OR_T_INIT_OK : OR_T_ECHO_OK);
      r.flags |= OR_F_MSG_ID;
      r.msg_id = ++ep.next_msg_id;                          // echo.rb:12-13
      if (m.type == OR_T_ECHO) { r.p0 = m.p0; r.p1 = m.p1; }
      out.push_back(Emit(r));
    }
    // any other type: echo.rb's case has no else branch -> ignored
  }

  void node_common_unknown(const or_msg& m, std::vector<Emit>& out) {
    // Replies (in_reply_to present) with no callback are ignored (node.rb:159-164).
    // An unhandled request type gets error 10 "not-supported"
    // (resources/errors.edn; demo/go/node_test.go:51) when it carries a msg_id.
    if (m.flags & OR_F_REPLY) return;
    if (m.flags & OR_F_MSG_ID) {
      or_msg r = reply_to(m, OR_T_ERROR);
      r.p0 = 10;
      out.push_back(Emit(r));
    }
  }

  void node_broadcast(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    Endpoint& ep = eps[e];
    if (m.flags & OR_F_REPLY) return;                       // node.rb:159-164
    switch (m.type) {
      case OR_T_INIT:      out.push_back(Emit(reply_to(m, OR_T_INIT_OK))); break;      // node.rb:22-36
      case OR_T_TOPOLOGY:  out.push_back(Emit(reply_to(m, OR_T_TOPOLOGY_OK))); break;  // 01-broadcast.md:286-290
      case OR_T_READ: {                                                            // broadcast.rb:22-27
        or_msg r = reply_to(m, OR_T_READ_OK);
        r.p0 = (uint32_t)ep.values.size();
        Emit em(r);
        em.has_snap = true;
        em.snap.assign(ep.values.begin(), ep.values.end());
        out.push_back(em);
        break;
      }
      case OR_T_BROADCAST: {                                // 01-broadcast.md:527-544
        const uint32_t v = m.p0;
        if (v >= cfg.n_values) { error = "broadcast value out of range"; return; }
        if (!ep.values.count(v)) {
          ep.values.insert(v);
          for (uint32_t nb : ep.neighbors) {
            if (nb == m.src) continue;                      // 02-performance.md:61-67
            or_msg g; std::memset(&g, 0, sizeof g);
            g.src = e; g.dest = nb; g.type = OR_T_BROADCAST; g.p0 = v;
            out.push_back(Emit(g));                         // fire-and-forget, no msg_id
          }
        }
        if (m.flags & OR_F_MSG_ID) out.push_back(Emit(reply_to(m, OR_T_BROADCAST_OK)));
        break;
      }
      default: node_common_unknown(m, out);
    }
  }

  // g-set node (demo/ruby/g_set.rb:13-39)
  void node_gset(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    Endpoint& ep = eps[e];
    if (m.flags & OR_F_REPLY) return;                       // node.rb:159-164
    switch (m.type) {
      case OR_T_INIT:                                       // node.rb:22-36: reply, then start the periodic task,
        ep.initialized = true;                              // whose first run is immediate (node.rb:129-137)
        ep.next_fire = now;
        out.push_back(Emit(reply_to(m, OR_T_INIT_OK)));
        break;
      case OR_T_ADD:                                        // g_set.rb:17-21
        if (m.p0 >= cfg.n_values) { error = "g-set element out of range"; return; }
        ep.values.insert(m.p0);
        out.push_back(Emit(reply_to(m, OR_T_ADD_OK)));
        break;
      case OR_T_READ: {                                     // g_set.rb:13-15
        or_msg r = reply_to(m, OR_T_READ_OK);
        r.p0 = (uint32_t)ep.values.size();
        Emit em(r);
        em.has_snap = true;
        em.snap.assign(ep.values.begin(), ep.values.end());
        out.push_back(em);
        break;
      }
      case OR_T_REPLICATE_ONE:                              // g_set.rb:24-26
        if (m.p0 >= cfg.n_values) { error = "g-set element out of range"; return; }
        ep.values.insert(m.p0);
        break;
      case OR_T_REPLICATE_FULL: {                           // g_set.rb:29-31  @set |= value
        auto it = gset_snaps.find(std::make_pair(m.src, m.p1));
        if (it != gset_snaps.end()) ep.values.insert(it->second.begin(), it->second.end());
        break;
      }
      default: node_common_unknown(m, out);
    }
  }

  // g-set periodic task (g_set.rb:34-39): every interval, send the whole set to every other node.
  // Evaluated at the start of the node's step of a round, before its receives.
  void gset_timer(uint32_t e, std::vector<Emit>& out) {
    Endpoint& ep = eps[e];
    if (!ep.initialized || now < ep.next_fire) return;
    const uint64_t handle = ++ep.fires;
    gset_snaps[std::make_pair(e, handle)].assign(ep.values.begin(), ep.values.end());
    for (uint32_t other = 0; other < cfg.n_nodes; other++) {
      // node.rb:104-108 other_node_ids: every node named by init, alive or not -- a send to a
      // removed node trips net.clj:172-175 like any other
      if (other == e) continue;
      or_msg g; std::memset(&g, 0, sizeof g);
      g.src = e; g.dest = other; g.type = OR_T_REPLICATE_FULL;
      g.p0 = (uint32_t)ep.values.size(); g.p1 = handle;
      out.push_back(Emit(g));
    }
    ep.next_fire += (int64_t)cfg.gset_interval_ms * kTickNs;
  }

  // ------------------------------------------------------------- Raft (demo/python/raft.py)
  std::map<std::pair<uint32_t, uint64_t>, RaftAppend> raft_appends;   // (sender, k) -> append_entries payload

  uint32_t cb_slots = kRaftCallbacks;
  // the node's cluster = node_ids of its init (raft.py:447-459): [gbase, gbase + gn)
  uint32_t raft_gbase(uint32_t e) const { const uint32_t G = cfg.raft_group ? cfg.raft_group : cfg.n_nodes; return (e / G) * G; }
  uint32_t raft_gn(uint32_t e) const {
    const uint32_t G = cfg.raft_group ? cfg.raft_group : cfg.n_nodes;
    return std::min(G, cfg.n_nodes - raft_gbase(e));
  }
  uint32_t raft_majority(uint32_t e) const { return raft_gn(e) / 2 + 1; }        // raft.py:25-27
  // random.random() (raft.py:251): word 0 of Philox(0x80000000 | k, node, round), k-th draw of the node's step
  uint32_t raft_draw(uint32_t e) {
    RaftNode& r = eps[e].rn;
    const uint32_t ctr[4] = {0x80000000u | r.draws++, e, (uint32_t)round, (uint32_t)(round >> 32)};
    const uint32_t key[2] = {cfg.seed_lo, cfg.seed_hi};
    uint32_t x[4];
    philox(ctr, key, x);
    return x[0];
  }
  void raft_reset_election_deadline(uint32_t e) {                                 // raft.py:249-251
    const uint32_t x = raft_draw(e);
    eps[e].rn.election_deadline = now + kElectionTimeoutNs + (int64_t)(((uint64_t)x * (uint64_t)kElectionTimeoutNs) >> 32);
  }
  void raft_reset_step_down_deadline(uint32_t e) { eps[e].rn.step_down_deadline = now + kElectionTimeoutNs; }   // :253-255
  void raft_become_follower(uint32_t e) {                                         // :307-314
    RaftNode& r = eps[e].rn;
    r.state = RAFT_FOLLOWER;
    r.next_index.clear(); r.match_index.clear();
    r.leader = -1;
    raft_reset_election_deadline(e);
  }
  void raft_maybe_step_down(uint32_t e, uint32_t remote_term) {                   // :265-270 (+ advance_term :257-263)
    RaftNode& r = eps[e].rn;
    if (r.term < remote_term) {
      r.term = remote_term;
      r.voted_for = -1;
      raft_become_follower(e);
    }
  }
  // net.rpc (raft.py:77-82): fresh msg_id, remember the closure, send
  void raft_rpc(uint32_t e, uint32_t dest, or_msg m, const RaftCb& closure, std::vector<Emit>& out) {
    RaftNode& r = eps[e].rn;
    const uint32_t id = r.next_msg_id++;
    RaftCb cb = closure;
    cb.msg_id = id;
    r.callbacks[id % cb_slots] = cb;
    m.src = e; m.dest = dest; m.flags = OR_F_MSG_ID; m.msg_id = id;
    out.push_back(Emit(m));
  }
  void raft_request_votes(uint32_t e, std::vector<Emit>& out) {                   // :272-303
    RaftNode& r = eps[e].rn;
    r.votes.clear();
    r.votes.insert(e);
    for (uint32_t n = raft_gbase(e); n < raft_gbase(e) + raft_gn(e); n++) {       // brpc, :243-246
      if (n == e) continue;
      or_msg m; std::memset(&m, 0, sizeof m);
      m.type = OR_T_REQUEST_VOTE;
      m.p0 = r.term;
      m.p1 = (uint64_t)r.log.size() | ((uint64_t)r.log.back().term << 32);
      RaftCb cb; cb.kind = 1; cb.term = r.term;
      raft_rpc(e, n, m, cb, out);
    }
  }
  void raft_become_candidate(uint32_t e, std::vector<Emit>& out) {                // :316-325
    RaftNode& r = eps[e].rn;
    r.state = RAFT_CANDIDATE;
    r.term += 1; r.voted_for = -1;                                                // advance_term
    r.voted_for = e;
    r.leader = -1;
    raft_reset_election_deadline(e);
    raft_reset_step_down_deadline(e);
    raft_request_votes(e, out);
  }
  void raft_become_leader(uint32_t e) {                                           // :327-339
    RaftNode& r = eps[e].rn;
    r.state = RAFT_LEADER;
    r.leader = -1;
    r.last_replication = 0;
    r.next_index.assign(raft_gn(e), (int64_t)r.log.size() + 1);                   // by cluster member
    r.match_index.assign(raft_gn(e), 0);
    raft_reset_step_down_deadline(e);
  }
  // KVStore.apply (raft.py:158-192); the reply goes to op['client'] with in_reply_to = op['msg_id']
  or_msg raft_apply(uint32_t e, const RaftEntry& op) {
    RaftNode& r = eps[e].rn;
    or_msg res; std::memset(&res, 0, sizeof res);
    res.src = e; res.dest = op.client; res.flags = OR_F_REPLY; res.in_reply_to = op.msg_id;
    auto it = r.kv.find(op.key);
    if (op.type == OR_T_READ) {
      if (it != r.kv.end()) { res.type = OR_T_READ_OK; res.p1 = it->second; }
      else { res.type = OR_T_ERROR; res.p0 = 20; }
    } else if (op.type == OR_T_WRITE) {
      r.kv[op.key] = (uint32_t)op.p1;
      res.type = OR_T_WRITE_OK;
    } else {                                                                      // cas
      if (it == r.kv.end()) { res.type = OR_T_ERROR; res.p0 = 20; }
      else if (it->second != (uint32_t)op.p1) { res.type = OR_T_ERROR; res.p0 = 22; }
      else { it->second = (uint32_t)(op.p1 >> 32); res.type = OR_T_CAS_OK; }
    }
    return res;
  }

  // net.process_msg + the handlers (raft.py:84-111, 443-573).  An exception inside a handler is
  // caught by the main loop (raft.py:585-588): the message is consumed, nothing else happens.
  void node_raft(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    RaftNode& r = eps[e].rn;
    if (m.flags & OR_F_REPLY) {                                                   // :97-101 callback lookup
      RaftCb& slot = r.callbacks[m.in_reply_to % cb_slots];
      if (slot.kind == 0 || slot.msg_id != m.in_reply_to) return;                 // KeyError
      const RaftCb cb = slot;
      slot.kind = 0;                                                              // del self.callbacks[m]
      if (cb.kind == 1) {                                                         // request_votes' handle, :282-303
        raft_reset_step_down_deadline(e);
        raft_maybe_step_down(e, m.p0);
        if (r.state == RAFT_CANDIDATE && r.term == cb.term && m.p0 == r.term && m.p1 != 0 &&
            m.src >= raft_gbase(e) && m.src < raft_gbase(e) + raft_gn(e)) {
          r.votes.insert(m.src);
          if (raft_majority(e) <= r.votes.size()) raft_become_leader(e);
        }
      } else {                                                                    // replicate_log's handler, :413-426
        raft_maybe_step_down(e, m.p0);
        if (r.state == RAFT_LEADER && cb.term == r.term) {
          raft_reset_step_down_deadline(e);
          const uint32_t cn = cb.node - raft_gbase(e);                            // member index
          if (cn < raft_gn(e)) {
            if (m.p1 != 0) {
              r.next_index[cn] = std::max(r.next_index[cn], cb.ni + (int64_t)cb.n_entries);
              r.match_index[cn] = std::max(r.match_index[cn], cb.ni - 1 + (int64_t)cb.n_entries);
            } else {
              r.next_index[cn] -= 1;
            }
          }
        }
      }
      return;
    }
    switch (m.type) {
      case OR_T_INIT: {                                                           // :447-459
        if (r.state != RAFT_NASCENT) return;                                      // "Can't init twice!"
        raft_become_follower(e);
        out.push_back(Emit(reply_to(m, OR_T_INIT_OK)));
        return;
      }
      case OR_T_REQUEST_VOTE: {                                                   // :464-495
        raft_maybe_step_down(e, m.p0);
        bool grant = false;
        const uint32_t last_log_index = (uint32_t)m.p1, last_log_term = (uint32_t)(m.p1 >> 32);
        if (m.p0 < r.term) {
        } else if (r.voted_for >= 0) {
        } else if (last_log_term < r.log.back().term) {
        } else if (last_log_term == r.log.back().term && last_log_index < r.log.size()) {
        } else {
          grant = true;
          r.voted_for = m.src;                                                    // body['candidate_id']
          raft_reset_election_deadline(e);
        }
        or_msg res = reply_to(m, OR_T_REQUEST_VOTE_RES);
        res.p0 = r.term; res.p1 = grant ? 1 : 0;
        out.push_back(Emit(res));
        return;
      }
      case OR_T_APPEND_ENTRIES: {                                                 // :499-545
        raft_maybe_step_down(e, m.p0);
        or_msg res = reply_to(m, OR_T_APPEND_ENTRIES_RES);
        res.p0 = r.term; res.p1 = 0;
        if (m.p0 < r.term) { out.push_back(Emit(res)); return; }
        r.leader = m.src;                                                         // body['leader_id']
        raft_reset_election_deadline(e);
        auto it = raft_appends.find(std::make_pair(m.src, m.p1));
        if (it == raft_appends.end()) return;                                     // forged handle: KeyError
        const RaftAppend& a = it->second;
        if (a.prev_log_index == 0) return;                                        // "Out of bounds previous log index"
        if (a.prev_log_index > r.log.size() || r.log[a.prev_log_index - 1].term != a.prev_log_term) {
          out.push_back(Emit(res));                                               // we disagree on the previous term
          return;
        }
        r.log.resize(a.prev_log_index);                                           // truncate, :533
        r.log.insert(r.log.end(), a.entries.begin(), a.entries.end());
        if (r.commit_index < a.leader_commit)
          r.commit_index = std::min<uint32_t>(a.leader_commit, (uint32_t)r.log.size());
        res.p1 = 1;
        out.push_back(Emit(res));
        return;
      }
      case OR_T_READ: case OR_T_WRITE: case OR_T_CAS: {                           // kv_req, :550-570
        if (r.state == RAFT_LEADER) {
          RaftEntry en;
          en.term = r.term; en.type = m.type; en.flags = m.flags; en.key = m.p0; en.client = m.src;
          en.msg_id = m.msg_id; en.p1 = m.p1;
          r.log.push_back(en);
        } else if (r.leader >= 0) {
          or_msg f = m;                                                           // msg['dest'] = leader; send_msg(msg)
          f.dest = (uint32_t)r.leader;
          out.push_back(Emit(f));
        } else {
          or_msg res = reply_to(m, OR_T_ERROR);
          res.p0 = 11;                                                            // not a leader
          out.push_back(Emit(res));
        }
        return;
      }
      default: return;                                                            // 'No callback or handler'
    }
  }

  // One pass of the main loop's actions after the inbox is empty (raft.py:577-584), in the
  // loop's own priority order; every action is idle again right after it ran (time is frozen
  // inside a round), and the state machine catches up to the commit index.
  void raft_actions(uint32_t e, std::vector<Emit>& out) {
    RaftNode& r = eps[e].rn;
    if (r.state == RAFT_LEADER && r.step_down_deadline < now) raft_become_follower(e);    // :371-376
    {                                                                                      // replicate_log, :387-441
      const int64_t elapsed = now - r.last_replication;
      bool replicated = false, aborted = false;
      const uint32_t first_rpc = r.next_msg_id;            // RPCs of this pass: ids first_rpc .. next_msg_id - 1
      RaftCb last;                                          // what the pass's closures end up seeing (see below)
      if (r.state == RAFT_LEADER && kMinReplicationNs < elapsed) {
        for (uint32_t n = raft_gbase(e); n < raft_gbase(e) + raft_gn(e) && !aborted; n++) {
          if (n == e) continue;
          const int64_t ni = r.next_index[n - raft_gbase(e)];
          if (ni <= 0) { aborted = true; break; }                                          // from_index raises, :147-148
          const int64_t n_entries = (int64_t)r.log.size() - ni + 1 > 0 ? (int64_t)r.log.size() - ni + 1 : 0;
          if (0 < n_entries || kHeartbeatNs < elapsed) {
            RaftAppend a;
            a.prev_log_index = (uint32_t)(ni - 1);
            // log.get(ni - 1): entries[ni - 2]; Python's entries[-1] when ni == 1 is the last entry
            const int64_t pi = ni - 2;
            if (pi >= (int64_t)r.log.size()) { aborted = true; break; }                    // IndexError
            a.prev_log_term = pi < 0 ? r.log.back().term : r.log[(size_t)pi].term;
            a.leader_commit = r.commit_index;
            if (n_entries > 0) a.entries.assign(r.log.begin() + (ni - 1), r.log.end());
            const uint64_t k = ++r.appends;
            raft_appends[std::make_pair(e, k)] = a;
            or_msg m; std::memset(&m, 0, sizeof m);
            m.type = OR_T_APPEND_ENTRIES; m.p0 = r.term; m.p1 = k;
            RaftCb cb; cb.kind = 2; cb.term = r.term; cb.node = n; cb.ni = ni; cb.n_entries = (uint32_t)n_entries;
            raft_rpc(e, n, m, cb, out);
            last = cb;
            replicated = true;
          }
        }
      }
      // Python closures bind late: `handler` reads _ni / _entries / _node (raft.py:408-426) from the
      // frame of this replicate_log call when the reply arrives, i.e. the values of the LAST node the
      // pass sent to, for every RPC of the pass.  (A follower that is not last in other_nodes() only
      // advances in a pass where it alone has something to receive.)
      for (uint32_t id = first_rpc; id != r.next_msg_id; id++) {
        RaftCb& slot = r.callbacks[id % cb_slots];
        if (slot.kind == 2 && slot.msg_id == id) { slot.node = last.node; slot.ni = last.ni; slot.n_entries = last.n_entries; }
      }
      // an exception inside replicate_log ends this iteration of the main loop; every later
      // iteration raises again before it gets to the actions below (raft.py:577-588)
      if (aborted) return;
      if (replicated) r.last_replication = now;
    }
    if (r.election_deadline < now) {                                                       // election, :358-367
      if (r.state == RAFT_FOLLOWER || r.state == RAFT_CANDIDATE) raft_become_candidate(e, out);
      else raft_reset_election_deadline(e);
    }
    if (r.state == RAFT_LEADER) {                                                          // advance_commit_index, :378-385
      std::vector<int64_t> xs = r.match_index;
      xs[e - raft_gbase(e)] = (int64_t)r.log.size();
      std::sort(xs.begin(), xs.end());
      const int64_t n = xs[xs.size() - raft_majority(e)];                                 // median, :29-33
      if ((int64_t)r.commit_index < n && r.log[(size_t)n - 1].term == r.term) r.commit_index = (uint32_t)n;
    }
    while (r.last_applied < r.commit_index) {                                              // advance_state_machine, :343-354
      r.last_applied += 1;
      const or_msg res = raft_apply(e, r.log[r.last_applied - 1]);
      if (r.state == RAFT_LEADER) out.push_back(Emit(res));
    }
  }

  // ------------------------------------------------------------- txn-list-append on a hash tree (demo/ruby/datomic_list_append.rb)
  // Immutable tree nodes live in lww-kv under unique pointers, lin-kv key "root" (0) holds the root pointer.
  // handle txn (:340-353, one at a time under @txn_lock, arrival order): read root -> Tree.load lazily
  // (cache, else read lww-kv until read_ok, :83-101) -> apply_txn (ms_tree.h) -> if the tree changed: write all
  // new nodes, await every write_ok, cas root -> txn_ok | error 30.  Unreadable root -> error 14.
  std::vector<mst::Rec> tt_recs;                 // contents by pointer - 1 (immutable once made)
  uint32_t tt_per_node = 256;
  struct TreeStore {
    or_sim* s; uint32_t e;
    mst::Rec* rec(uint32_t ptr) const { return &s->tt_recs[ptr - 1]; }
    bool cached(uint32_t ptr) const { return s->eps[e].tn.cache.count(ptr) != 0; }
  };
  int svc_endpoint(int type) const { return svc_last[type]; }
  void tt_rpc(uint32_t e, int dest, uint16_t type, uint32_t p0, uint64_t p1, int kind, uint32_t arg, std::vector<Emit>& out) {
    if (dest < 0) { error = "txn-list-append (hash tree) needs the lin-kv and lww-kv services"; return; }
    RaftNode& r = eps[e].rn;
    RaftCb cb; cb.kind = kind; cb.node = arg; cb.term = eps[e].tn.gen;
    const uint32_t id = ++r.next_msg_id;                                          // node.rb:95-102
    cb.msg_id = id;
    r.callbacks[id % cb_slots] = cb;
    or_msg q; std::memset(&q, 0, sizeof q);
    q.type = type; q.p0 = p0; q.p1 = p1;
    q.src = e; q.dest = (uint32_t)dest; q.flags = OR_F_MSG_ID; q.msg_id = id;
    out.push_back(Emit(q));
  }
  void tt_start(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    TreeNode& t = eps[e].tn;
    t.cur_src = m.src; t.cur_msg_id = m.msg_id; t.cur_ops = m.p1;
    t.phase = 1;
    t.deadline = now + kPromiseTimeoutNs;
    tt_rpc(e, svc_endpoint(OR_SVC_LIN_KV), OR_T_READ, 0, 0, 10, 0, out);          // current_tree, :361-368
  }
  void tt_answer(uint32_t e, uint16_t type, uint32_t code, uint64_t p1, std::vector<Emit>& out) {
    TreeNode& t = eps[e].tn;
    or_msg req; std::memset(&req, 0, sizeof req);
    req.src = t.cur_src; req.dest = e; req.msg_id = t.cur_msg_id;
    or_msg a = reply_to(req, type);
    a.p0 = code; a.p1 = p1;
    out.push_back(Emit(a));
    t.phase = 0;                                                                  // the lock passes to the next waiter
    t.deadline = 0;
    t.gen++;
    if (!t.waiting.empty()) {
      const or_msg next = t.waiting.front();
      t.waiting.pop_front();
      tt_start(e, next, out);
    }
  }
  void tt_eval(uint32_t e, std::vector<Emit>& out) {
    TreeNode& t = eps[e].tn;
    TreeStore S{this, e};
    uint32_t counter = t.start_counter, root2 = 0, load_ptr = 0;
    const mst::Status st = mst::apply_txn(S, e, tt_per_node, t.root1, t.cur_ops, t.start_counter, counter, root2, load_ptr);
    if (st == mst::kCapacity) { error = "hash tree: out of pointers / leaf or depth capacity"; return; }
    if (st == mst::kNeedLoad) {                                                   // Tree.load, :83-101
      t.phase = 2;
      t.deadline = now + kPromiseTimeoutNs;
      tt_rpc(e, svc_endpoint(OR_SVC_LWW_KV), OR_T_READ, load_ptr, 0, 11, load_ptr, out);
      return;
    }
    t.ptr_counter = counter;
    t.root2 = root2;
    if (root2 == t.root1) { tt_answer(e, OR_T_TXN_OK, 0, (uint64_t)t.root1 | ((uint64_t)t.root1 << 32), out); return; }
    uint32_t order[mst::kMaxWrites], n = 0;
    if (!mst::save_order(S, e, tt_per_node, t.start_counter, root2, order, n)) { error = "hash tree: save walk too deep"; return; }
    t.phase = 3; t.writes_left = n; t.write_failed = 0;
    t.deadline = now + kPromiseTimeoutNs;
    t.first_write = order[0]; t.first_write_ok = false; t.root_is_leaf = S.rec(root2)->type == 1;
    for (uint32_t i = 0; i < n; i++)                                              // save_this!, :128-145
      tt_rpc(e, svc_endpoint(OR_SVC_LWW_KV), OR_T_WRITE, order[i], order[i], 12, order[i], out);
  }
  // Promise#await's 5 s (promise.rb:24-31), checked once per step after the step's messages.  A handler thread that
  // gives up raises RPCError.timeout: error 0 to the requester (node.rb:187-189), the lock is released.  Branch#save!
  // waits in a helper thread (:297-309): if its first write is still unanswered when the clocks run out, its "false"
  // is taken to reach the handler first (error 14), otherwise the handler's own time-out does (error 0).
  void tt_actions(uint32_t e, std::vector<Emit>& out) {
    TreeNode& t = eps[e].tn;
    if (t.init_phase != 0 && now >= t.init_deadline) {
      t.init_phase = 0;
      or_msg init_req; std::memset(&init_req, 0, sizeof init_req);
      init_req.src = t.init_src; init_req.dest = e; init_req.msg_id = t.init_msg_id;
      or_msg er = reply_to(init_req, OR_T_ERROR);
      er.p0 = 0;
      out.push_back(Emit(er));
    }
    if (t.phase != 0 && t.deadline != 0 && now >= t.deadline)
      tt_answer(e, OR_T_ERROR, (t.phase == 3 && !t.root_is_leaf && !t.first_write_ok) ? 14 : 0, 0, out);
  }
  void node_txn_tree(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    TreeNode& t = eps[e].tn;
    RaftNode& r = eps[e].rn;
    if (m.flags & OR_F_REPLY) {                                                  // node.rb:170-176
      RaftCb& slot = r.callbacks[m.in_reply_to % cb_slots];
      if (slot.kind == 0 || slot.msg_id != m.in_reply_to) return;                 // no callback
      const RaftCb cb = slot;
      slot.kind = 0;
      if (cb.kind >= 10 && cb.kind <= 13 && (cb.term != t.gen || t.phase == 0)) return;   // its transaction is over: a dead promise
      if ((cb.kind == 14 && t.init_phase != 1) || (cb.kind == 15 && t.init_phase != 2)) return;
      or_msg init_req; std::memset(&init_req, 0, sizeof init_req);
      init_req.src = t.init_src; init_req.dest = e; init_req.msg_id = t.init_msg_id;
      switch (cb.kind) {
        case 10:                                                                  // the root pointer
          if (m.type == OR_T_READ_OK) { t.root1 = (uint32_t)m.p1; t.start_counter = t.ptr_counter; tt_eval(e, out); }
          else tt_answer(e, OR_T_ERROR, 14, 0, out);                              // abort, :367
          return;
        case 11:                                                                  // a tree node
          if (m.type == OR_T_READ_OK) { t.cache.insert(cb.node); tt_eval(e, out); }
          else { t.deadline = now + kPromiseTimeoutNs; tt_rpc(e, svc_endpoint(OR_SVC_LWW_KV), OR_T_READ, cb.node, 0, 11, cb.node, out); }   // retry, :97-99
          return;
        case 12:                                                                  // one of save!'s writes
          if (m.type != OR_T_WRITE_OK) t.write_failed = 1;
          if (cb.node == t.first_write) t.first_write_ok = true;
          if (--t.writes_left == 0) {
            if (t.write_failed) { tt_answer(e, OR_T_ERROR, 14, 0, out); return; }  // "Couldn't save new tree"
            t.phase = 4;                                                          // advance_root!, :372-379
            t.deadline = now + kPromiseTimeoutNs;
            tt_rpc(e, svc_endpoint(OR_SVC_LIN_KV), OR_T_CAS, 0, (uint64_t)t.root1 | ((uint64_t)t.root2 << 32), 13, 0, out);
          }
          return;
        case 13:
          if (m.type == OR_T_CAS_OK) tt_answer(e, OR_T_TXN_OK, 0, (uint64_t)t.root1 | ((uint64_t)t.root2 << 32), out);
          else tt_answer(e, OR_T_ERROR, 30, 0, out);                              // txn_conflict, :378
          return;
        case 14:                                                                  // the first node's initial state, :330-338
          if (m.type == OR_T_WRITE_OK) {
            t.init_phase = 2; t.init_deadline = now + kPromiseTimeoutNs;
            tt_rpc(e, svc_endpoint(OR_SVC_LIN_KV), OR_T_WRITE, 0, mst::kPtrEmpty, 15, 0, out);
          } else {
            t.init_phase = 0;
            or_msg er = reply_to(init_req, OR_T_ERROR); er.p0 = 14; out.push_back(Emit(er));
          }
          return;
        case 15:
          t.init_phase = 0;
          out.push_back(Emit(reply_to(init_req, OR_T_INIT_OK)));                  // node.rb:31
          return;
      }
      return;
    }
    switch (m.type) {
      case OR_T_INIT:                                                             // node.rb:22-36 + :329-338
        if (e == 0) {                                                             // @node.node_ids.first == @node.node_id
          t.init_src = m.src; t.init_msg_id = m.msg_id;
          t.init_phase = 1; t.init_deadline = now + kPromiseTimeoutNs;
          tt_rpc(e, svc_endpoint(OR_SVC_LWW_KV), OR_T_WRITE, mst::kPtrEmpty, mst::kPtrEmpty, 14, 0, out);
        } else {
          out.push_back(Emit(reply_to(m, OR_T_INIT_OK)));
        }
        return;
      case OR_T_TXN:                                                              // :340-353
        if (t.phase == 0) tt_start(e, m, out);
        else t.waiting.push_back(m);
        return;
      default: {
        or_msg er = reply_to(m, OR_T_ERROR);
        er.p0 = 10;
        out.push_back(Emit(er));
        return;
      }
    }
  }

  // ------------------------------------------------------------- txn-list-append (demo/clojure/single_key_txn.clj)
  // The whole database is one value under key "root" (key 0 here) of lin-kv (:134-141).  A
  // database value is carried as a version id (see oracle.h); apply-txn (:115-127) is a pure
  // function of (value, txn), so the node only has to know whether the txn changes the value.
  void node_txn(uint32_t e, const or_msg& m, std::vector<Emit>& out) {
    RaftNode& r = eps[e].rn;                       // next_msg_id, callbacks, appends (= versions minted)
    const int lin_kv = svc_endpoint(OR_SVC_LIN_KV);
    if (m.flags & OR_F_REPLY) {                                                  // handle-reply!, :60-68
      RaftCb& slot = r.callbacks[m.in_reply_to % cb_slots];
      if (slot.kind == 0 || slot.msg_id != m.in_reply_to) return;                 // no such future
      const RaftCb cb = slot;
      slot.kind = 0;
      or_msg req; std::memset(&req, 0, sizeof req);                              // the txn request being served
      req.src = cb.node; req.dest = e; req.msg_id = cb.term;
      if (cb.kind == 3) {                                                         // read-service, :143-150
        uint32_t old_v;
        if (m.type == OR_T_READ_OK) old_v = (uint32_t)m.p1;
        else if (m.type == OR_T_ERROR && m.p0 == 20) old_v = 0;                   // not found: nil
        else { or_msg er = reply_to(req, OR_T_ERROR); er.p0 = m.p0; out.push_back(Emit(er)); return; }   // :99-103
        // apply-txn: an append makes a value nobody has seen; reads leave it as it is ({} for nil)
        uint32_t new_v;
        if (cb.n_entries) new_v = 2u + e + cfg.n_nodes * (uint32_t)(r.appends++);
        else new_v = old_v == 0 ? 1u : old_v;
        if (lin_kv < 0) { error = "txn-list-append needs the lin-kv service"; return; }
        or_msg c; std::memset(&c, 0, sizeof c);                                   // cas-service!, :152-161
        c.type = OR_T_CAS; c.p0 = 0; c.p1 = (uint64_t)old_v | ((uint64_t)new_v << 32);
        RaftCb n2; n2.kind = 4; n2.node = cb.node; n2.term = cb.term; n2.ni = (int64_t)old_v; n2.n_entries = new_v;
        const uint32_t id = ++r.next_msg_id;                                      // (swap! next-message-id inc), :54
        n2.msg_id = id;
        r.callbacks[id % cb_slots] = n2;
        c.src = e; c.dest = (uint32_t)lin_kv; c.flags = OR_F_MSG_ID | OR_F_CREATE; c.msg_id = id;
        out.push_back(Emit(c));
      } else if (cb.kind == 4) {                                                  // :168-173
        if (m.type == OR_T_CAS_OK) {
          or_msg ok = reply_to(req, OR_T_TXN_OK);
          ok.p1 = (uint64_t)(uint32_t)cb.ni | ((uint64_t)cb.n_entries << 32);
          out.push_back(Emit(ok));
        } else {
          or_msg er = reply_to(req, OR_T_ERROR);
          er.p0 = (m.type == OR_T_ERROR && m.p0 == 22) ? 30 : m.p0;              // "root altered"
          out.push_back(Emit(er));
        }
      }
      return;
    }
    switch (m.type) {
      case OR_T_INIT: out.push_back(Emit(reply_to(m, OR_T_INIT_OK))); return;     // :70-77
      case OR_T_TXN: {                                                            // handle-txn!, :163-173
        if (lin_kv < 0) { error = "txn-list-append needs the lin-kv service"; return; }
        or_msg q; std::memset(&q, 0, sizeof q);
        q.type = OR_T_READ; q.p0 = 0;
        RaftCb cb; cb.kind = 3; cb.node = m.src; cb.term = m.msg_id; cb.n_entries = (m.flags & OR_F_APPENDS) ? 1 : 0;
        const uint32_t id = ++r.next_msg_id;
        cb.msg_id = id;
        r.callbacks[id % cb_slots] = cb;
        q.src = e; q.dest = (uint32_t)lin_kv; q.flags = OR_F_MSG_ID; q.msg_id = id;
        out.push_back(Emit(q));
        return;
      }
      default: {                                                                  // "Unknown request type", :85-88
        or_msg er = reply_to(m, OR_T_ERROR);
        er.p0 = 10;
        out.push_back(Emit(er));
        return;
      }
    }
  }

  // ------------------------------------------------------------- closed-loop clients
  void gen_hist(uint32_t e, uint32_t op, uint8_t type, uint8_t f, uint16_t err, uint32_t value) {
    or_hist h;
    h.time_ns = now; h.order = (round << 24) | eps[e].gen.ordinal; h.client = e; h.op = op;
    h.type = type; h.f = f; h.error = err; h.value = value;
    history.push_back(h);
  }
  // a reply delivered to client e (client.clj:81-117): the awaited one completes the op, anything else is dropped
  void gen_reply(uint32_t e, const or_msg& m) {
    Endpoint::Gen& g = eps[e].gen;
    if (!g.waiting_for || !(m.flags & OR_F_REPLY) || m.in_reply_to != g.waiting_for) return;   // :106-107
    uint8_t outcome = 1; uint16_t err = 0; uint32_t value = g.cur_value;
    if (m.type == OR_T_ERROR) {                          // :165-172; definite = all codes but 0 and 13 (errors.edn)
      err = (uint16_t)m.p0;
      const bool definite = m.p0 != 0 && m.p0 != 13;
      outcome = (definite || g.cur_f == 1) ? 2 : 3;
    } else if (g.cur_f == 1) {
      value = m.p0;                                      // read_ok: the size of the set
    }
    gen_hist(e, g.ops, outcome, (uint8_t)g.cur_f, err, value);
    g.waiting_for = 0;
  }
  // after the replies of the round: timeout, then at most one invocation (the worker asks its generator)
  void gen_step(uint32_t e, std::vector<Emit>& out) {
    Endpoint::Gen& g = eps[e].gen;
    if (g.waiting_for && now >= g.deadline_ns) {         // :96-101,160-164
      gen_hist(e, g.ops, g.cur_f == 1 ? 2 : 3, (uint8_t)g.cur_f, 0xFFFF, g.cur_value);
      g.waiting_for = 0;
    }
    if (g.waiting_for) return;
    bool send = false;
    uint32_t f = 1, value = 0;
    if (g.phase == 0) {
      if (now >= gcfg.time_limit_ns) g.phase = 1;
      else if (now >= g.next_op_ns) {
        const uint32_t ctr[4] = {g.ops, e, 0xC11E47u, 0u};
        const uint32_t key[2] = {cfg.seed_lo, cfg.seed_hi};
        uint32_t x[4];
        philox(ctr, key, x);
        if ((((uint64_t)x[0] * 1000u) >> 32) >= gcfg.read_permille) { f = 0; value = g.ordinal + gcfg.n_clients * g.bcasts++; }
        g.next_op_ns = now + (int64_t)(((unsigned __int128)x[1] * (unsigned __int128)(2 * (uint64_t)gcfg.interval_ns)) >> 32);
        send = true;
      }
    }
    if (g.phase == 1 && now >= gcfg.time_limit_ns + gcfg.quiet_ns) { g.phase = 2; send = true; }   // broadcast.clj:237-240
    else if (g.phase == 2 && !send) g.phase = 3;
    if (!send) return;
    g.ops++;
    g.cur_f = f; g.cur_value = value;
    g.waiting_for = ++g.next_msg_id;                     // client.clj:61-64
    g.deadline_ns = now + gcfg.timeout_ns;
    gen_hist(e, g.ops, 0, (uint8_t)f, 0, value);
    or_msg m; std::memset(&m, 0, sizeof m);
    m.src = e; m.dest = g.node; m.flags = OR_F_MSG_ID; m.msg_id = g.waiting_for;
    m.type = f == 1 ? OR_T_READ : (cfg.workload == OR_W_GSET ? OR_T_ADD : OR_T_BROADCAST);
    m.p0 = value;
    out.push_back(Emit(m));
  }

  bool run_round() {
    std::vector<Envelope> pending;
    // (1) injector
    uint32_t inj = 0;
    while (!host_queue.empty()) {
      or_msg m = host_queue.front(); host_queue.pop_front();
      if (!send(kInjector, inj++, m, pending)) return false;
    }
    while (sched_cursor < schedule.size() && schedule[sched_cursor].time_ns <= now) {
      const or_op& op = schedule[sched_cursor++];
      or_msg m; std::memset(&m, 0, sizeof m);
      m.src = op.src; m.dest = op.dest; m.type = op.body.type; m.flags = op.body.flags;
      m.msg_id = op.body.msg_id; m.in_reply_to = op.body.in_reply_to;
      m.p0 = op.body.p0; m.p1 = op.body.p1;
      if (!send(kInjector, inj++, m, pending)) return false;
    }
    // (2) endpoints
    std::vector<Emit> out;
    for (uint32_t e = 0; e < eps.size(); e++) {
      Endpoint& ep = eps[e];
      if (!ep.live) continue;
      out.clear();
      if (cfg.workload == OR_W_GSET && ep.kind == OR_KIND_SERVER) gset_timer(e, out);
      if (cfg.workload == OR_W_RAFT && ep.kind == OR_KIND_SERVER) ep.rn.draws = 0;
      while (!ep.q.empty() && ep.q.top().m.deadline_ns <= now) {   // net.clj:228-229,236-238
        const or_msg m = ep.q.top().m;
        ep.q.pop();
        if (partitioned(m.src, e)) continue;                       // net.clj:234: consumed, no event
        log_event(true, m);                                        // net.clj:244
        switch (ep.kind) {
          case OR_KIND_CLIENT:
            ep.mailbox.push_back(m);
            break;
          case OR_KIND_SIM_CLIENT:      // simulated client sink: replies are counted, not mailed
            if (m.flags & OR_F_REPLY) client_replies++;
            break;
          case OR_KIND_HOST:
            ep.mailbox.push_back(m);
            break;
          case OR_KIND_GEN_CLIENT:
            gen_reply(e, m);
            break;
          case OR_KIND_SERVICE: {         // service-thread (service.clj:245-263)
            or_body q;
            q.type = m.type; q.flags = m.flags; q.msg_id = m.msg_id; q.in_reply_to = m.in_reply_to;
            q.p0 = m.p0; q.p1 = m.p1;
            // rand-int: word 3 of the Philox draw of the reply this request would emit
            const uint32_t ctr[4] = {(uint32_t)out.size(), e, (uint32_t)round, (uint32_t)(round >> 32)};
            const uint32_t key[2] = {cfg.seed_lo, cfg.seed_hi};
            uint32_t x[4];
            philox(ctr, key, x);
            const SvcReply r = ep.svc.handle(m.src, q, x[3]);
            if (r.reply) {
              or_msg rm = reply_to(m, r.type);          // body + :in_reply_to (service.clj:255-258)
              rm.p0 = r.p0; rm.p1 = r.p1;
              out.push_back(Emit(rm));
            }
            break;
          }
          default:
            if (cfg.workload == OR_W_ECHO) node_echo(e, m, out);
            else if (cfg.workload == OR_W_BROADCAST) node_broadcast(e, m, out);
            else if (cfg.workload == OR_W_GSET) node_gset(e, m, out);
            else if (cfg.workload == OR_W_RAFT) node_raft(e, m, out);
            else if (cfg.workload == OR_W_TXN) node_txn(e, m, out);
            else if (cfg.workload == OR_W_TXN_TREE) node_txn_tree(e, m, out);
            else { error = "workload not implemented in oracle"; return false; }
        }
        if (!error.empty()) return false;
      }
      if (cfg.workload == OR_W_RAFT && ep.kind == OR_KIND_SERVER) raft_actions(e, out);
      if (cfg.workload == OR_W_TXN_TREE && ep.kind == OR_KIND_SERVER) tt_actions(e, out);
      if (ep.kind == OR_KIND_GEN_CLIENT) gen_step(e, out);
      for (uint32_t j = 0; j < out.size(); j++) {
        if (out[j].has_snap) snapshots[next_id] = out[j].snap;   // keyed by the read_ok's net id
        if (!send(e, j, out[j].m, pending)) return false;
      }
    }
    // (3) visibility
    bool due_now = false;
    for (const Envelope& env : pending) {
      if (env.m.deadline_ns <= now) due_now = true;
      eps[env.m.dest].q.push(env);
    }
    // (4) time advance
    round++;
    if (!due_now) now += kTickNs;
    return true;
  }
};

extern "C" {

uint32_t or_tree_key_hash(uint32_t key) { return mst::key_hash(key); }

or_sim* or_create(const or_config* cfg) {
  or_sim* s = new or_sim();
  s->cfg = *cfg;
  if (s->cfg.n_values == 0) s->cfg.n_values = 1u << 20;
  if (s->cfg.gset_interval_ms == 0) s->cfg.gset_interval_ms = 5000;   // g_set.rb:34
  s->loss_thresh = loss_threshold(cfg->p_loss);
  s->eps.resize(cfg->n_nodes);
  if (s->cfg.rpc_table) { s->cb_slots = 1; while (s->cb_slots < s->cfg.rpc_table) s->cb_slots <<= 1; }
  if (s->cfg.raft_group >= s->cfg.n_nodes) s->cfg.raft_group = 0;
  if (cfg->workload == OR_W_TXN_TREE) {
    if (s->cb_slots < 128) s->cb_slots = 128;                          // one save! has up to mst::kMaxWrites closures in flight
    s->tt_per_node = s->cfg.tree_ptrs ? s->cfg.tree_ptrs : 256u;
    s->tt_recs.assign(1 + (size_t)cfg->n_nodes * s->tt_per_node, mst::Rec{});
    mst::Rec& empty = s->tt_recs[mst::kPtrEmpty - 1];                  // Tree.empty: a leaf over the whole ring
    empty.type = 1; empty.lo = 0; empty.hi = (uint8_t)mst::kRing; empty.n = 0;
  }
  for (uint32_t i = 0; i < cfg->n_nodes; i++) {
    if (cfg->workload == OR_W_RAFT || cfg->workload == OR_W_TXN || cfg->workload == OR_W_TXN_TREE) s->eps[i].rn.callbacks.resize(s->cb_slots);
    s->eps[i].name = "n" + std::to_string(i);          // core.clj:231-238
    s->eps[i].kind = OR_KIND_SERVER;
    s->eps[i].neighbors = topology_neighbors(cfg->topology, cfg->n_nodes, i);
  }
  return s;
}

void or_destroy(or_sim* s) { delete s; }
const char* or_last_error(or_sim* s) { return s->error.c_str(); }

int or_add_endpoint(or_sim* s, const char* name, int kind) {   // net.clj:139-146
  Endpoint ep;
  ep.name = name;
  ep.kind = kind;
  if (kind == OR_KIND_SERVICE) {                                  // service.clj:290-296
    if (ep.name == "lin-kv") ep.svc.type = OR_SVC_LIN_KV;
    else if (ep.name == "seq-kv") ep.svc.type = OR_SVC_SEQ_KV;
    else if (ep.name == "lww-kv") ep.svc.type = OR_SVC_LWW_KV;
    else if (ep.name == "lin-tso") ep.svc.type = OR_SVC_LIN_TSO;
    else return -2;
  }
  // the slot of a removed non-server, non-service endpoint is recycled, lowest index first, unless pairwise
  // drop! entries (keyed by index) exist; the newcomer starts with an empty queue (net.clj:139-146)
  if (kind != OR_KIND_SERVICE && s->partitions.empty())
    for (uint32_t i = s->cfg.n_nodes; i < s->eps.size(); i++)
      if (!s->eps[i].live && s->eps[i].kind != OR_KIND_SERVICE) {
        s->eps[i] = ep;
        for (Endpoint& other : s->eps) other.svc.clients.erase(i);   // seq-kv's per-client index (service.clj:162-166)
        return (int)i;
      }
  s->eps.push_back(ep);
  if (kind == OR_KIND_SERVICE) s->svc_last[ep.svc.type] = (int)s->eps.size() - 1;
  return (int)s->eps.size() - 1;
}

int or_remove_endpoint(or_sim* s, uint32_t idx) {               // net.clj:148-152
  if (idx >= s->eps.size() || !s->eps[idx].live) return -1;
  s->eps[idx].live = false;
  return 0;
}

int64_t or_send(or_sim* s, uint32_t src, uint32_t dest, const or_body* b) {
  if (src >= s->eps.size() || !s->eps[src].live) return -1;   // node-not-found, code 1 (net.clj:159-164)
  if (dest >= s->eps.size() || !s->eps[dest].live) return -1;
  or_msg m; std::memset(&m, 0, sizeof m);
  m.src = src; m.dest = dest; m.type = b->type; m.flags = b->flags;
  m.msg_id = b->msg_id; m.in_reply_to = b->in_reply_to; m.p0 = b->p0; m.p1 = b->p1;
  s->host_queue.push_back(m);
  return (int64_t)(s->next_id + s->host_queue.size() - 1);
}

int or_schedule(or_sim* s, const or_op* ops, size_t n) {
  for (size_t i = 0; i < n; i++) {
    if (!s->schedule.empty() && ops[i].time_ns < s->schedule.back().time_ns) return -2;
    s->schedule.push_back(ops[i]);
  }
  return 0;
}

int or_step(or_sim* s, uint64_t n_rounds) {
  for (uint64_t i = 0; i < n_rounds; i++) if (!s->run_round()) return -3;
  return 0;
}

int or_run(or_sim* s, int64_t until_ns) {
  // a node that sends zero-latency messages in every round freezes virtual time (DESIGN.md 2.3):
  // give up after 2^20 delta rounds at one instant, like the engine
  int64_t stall_now = s->now;
  uint64_t stall_round = s->round;
  while (s->now < until_ns) {
    if (!s->run_round()) return -3;
    if (s->now != stall_now) { stall_now = s->now; stall_round = s->round; }
    else if (s->round - stall_round > (1ull << 20)) { s->error = "virtual time is not advancing"; return -3; }
  }
  return 0;
}

int or_recv(or_sim* s, uint32_t e, int64_t timeout_ns, or_msg* out) {   // net.clj:223-247
  if (e >= s->eps.size() || !s->eps[e].live) return -1;
  // Poll; while nothing is deliverable advance the simulation one round at a
  // time until the virtual timeout has elapsed (the reference blocks on the
  // wall clock, net.clj:228-229).
  const int64_t give_up = s->now + timeout_ns;
  int64_t stall_now = s->now;
  uint64_t stall_round = s->round;
  for (;;) {
    if (s->now != stall_now) { stall_now = s->now; stall_round = s->round; }
    else if (s->round - stall_round > (1ull << 20)) { s->error = "virtual time is not advancing"; return -3; }
    if (!s->eps[e].mailbox.empty()) {
      *out = s->eps[e].mailbox.front();
      s->eps[e].mailbox.pop_front();
      return 1;
    }
    if (s->now >= give_up) return 0;
    if (!s->run_round()) return -3;
  }
}

int64_t or_now(or_sim* s) { return s->now; }
uint64_t or_round(or_sim* s) { return s->round; }

int or_net_drop(or_sim* s, uint32_t src, uint32_t dest) {        // net.clj:109-110
  s->partitions.insert(std::make_pair(dest, src));
  return 0;
}
int or_net_heal(or_sim* s) {                                     // net.clj:112-113
  s->partitions.clear();
  s->component.clear();
  return 0;
}
int or_net_slow(or_sim* s) { s->scale *= 10; return 0; }         // net.clj:115-116 (stackable)
int or_net_fast(or_sim* s) {                                     // net.clj:118-119; unwrap one level.
  if (s->scale >= 10) s->scale /= 10;                            // (nil on unscaled is a latent bug, not replicated)
  return 0;
}
int or_net_flaky(or_sim* s) { s->loss_thresh = loss_threshold(0.5); return 0; }  // net.clj:121-122
int or_net_set_loss(or_sim* s, double p) { s->loss_thresh = loss_threshold(p); return 0; }
int or_net_partition(or_sim* s, const uint32_t* c, size_t n) {
  s->component.assign(c, c + n);
  return 0;
}

size_t or_journal_size(or_sim* s) { return s->journal.size(); }
size_t or_journal_copy(or_sim* s, size_t first, or_event* ev, or_body* bodies, size_t cap) {
  size_t n = 0;
  for (size_t i = first; i < s->journal.size() && n < cap; i++, n++) {
    if (ev) ev[n] = s->journal[i];
    if (bodies) bodies[n] = s->bodies[i];
  }
  return n;
}

void or_stats(or_sim* s, uint64_t out[9]) {
  // {all,clients,servers} x {send-count, recv-count, msg-count}; msg-count = cardinality of message ids
  // over all events of the class (net/checker.clj:34-36).  The journal names the endpoints of a message
  // as they were when it was sent, so every id falls in the class of its one :send, taken when the :send
  // was logged: a recycled slot's new kind does not move messages of its old name.
  for (int c = 0; c < 3; c++) {
    out[c * 3 + 0] = s->stats[c * 3 + 0];
    out[c * 3 + 1] = s->stats[c * 3 + 1];
    out[c * 3 + 2] = s->stats[c * 3 + 0];
  }
}

size_t or_node_set(or_sim* s, uint32_t node, uint32_t* vals, size_t cap) {
  if (node >= s->eps.size()) return 0;
  size_t n = 0;
  for (uint32_t v : s->eps[node].values) { if (n < cap && vals) vals[n] = v; n++; }
  return n;
}

size_t or_read_snapshot(or_sim* s, uint64_t msg_id, uint32_t* vals, size_t cap) {
  auto it = s->snapshots.find(msg_id);
  if (it == s->snapshots.end()) return 0;
  size_t n = 0;
  for (uint32_t v : it->second) { if (n < cap && vals) vals[n] = v; n++; }
  return n;
}

int or_add_gen_clients(or_sim* s, const or_gen_config* gc, uint32_t first_name) {
  if (!gc || gc->n_clients == 0 || gc->interval_ns <= 0 || s->gcfg.n_clients) return -2;
  s->gcfg = *gc;
  if (s->gcfg.timeout_ns <= 0) s->gcfg.timeout_ns = 5000ll * kTickNs;      // client.clj:18-20
  if (s->gcfg.quiet_ns <= 0) s->gcfg.quiet_ns = 10000ll * kTickNs;         // core.clj:75-78
  const int first = (int)s->eps.size();
  for (uint32_t k = 0; k < gc->n_clients; k++) {
    Endpoint ep;
    ep.name = "c" + std::to_string(first_name + k);
    ep.kind = OR_KIND_GEN_CLIENT;
    ep.gen.node = k % s->cfg.n_nodes;
    ep.gen.ordinal = k;
    s->eps.push_back(ep);
  }
  return first;
}
size_t or_history_copy(or_sim* s, size_t first, or_hist* out, size_t cap) {
  size_t n = 0;
  for (size_t i = first; i < s->history.size() && n < cap; i++, n++) if (out) out[n] = s->history[i];
  return out ? n : s->history.size() - std::min(first, s->history.size());
}
uint64_t or_client_replies(or_sim* s) { return s->client_replies; }
uint64_t or_undeliverable(or_sim* s) { return s->undelivered; }

int or_raft_state(or_sim* s, uint32_t node, uint64_t out[8]) {
  if (node >= s->cfg.n_nodes) return -1;
  const RaftNode& r = s->eps[node].rn;
  out[0] = (uint64_t)r.state; out[1] = r.term; out[2] = (uint64_t)(r.voted_for + 1); out[3] = r.commit_index;
  out[4] = r.last_applied; out[5] = (uint64_t)(r.leader + 1); out[6] = r.log.size(); out[7] = r.kv.size();
  return 0;
}
int or_raft_append(or_sim* s, uint32_t sender, uint64_t k, uint32_t out[4]) {
  auto it = s->raft_appends.find(std::make_pair(sender, k));
  if (it == s->raft_appends.end()) return 0;
  out[0] = it->second.prev_log_index; out[1] = it->second.prev_log_term;
  out[2] = it->second.leader_commit; out[3] = (uint32_t)it->second.entries.size();
  return 1;
}

struct or_service { Service s; };
or_service* or_service_new(int svc_type, uint32_t buffer_size) {
  or_service* p = new or_service();
  p->s.type = svc_type;
  if (buffer_size) p->s.buffer_size = buffer_size;
  return p;
}
void or_service_free(or_service* p) { delete p; }
int or_service_handle(or_service* p, uint32_t client, const or_body* req, uint32_t rnd, or_body* reply) {
  const SvcReply r = p->s.handle(client, *req, rnd);
  if (!r.reply) return 0;
  std::memset(reply, 0, sizeof *reply);
  reply->type = r.type; reply->flags = OR_F_REPLY; reply->in_reply_to = req->msg_id;
  reply->p0 = r.p0; reply->p1 = r.p1;
  return 1;
}

size_t or_topology(uint32_t topo, uint32_t n, uint32_t node, uint32_t* out, size_t cap) {
  std::vector<uint32_t> nb = topology_neighbors(topo, n, node);
  for (size_t i = 0; i < nb.size() && i < cap; i++) out[i] = nb[i];
  return nb.size();
}

void or_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  philox(ctr, key, out);
}

uint64_t or_latency_draw(uint32_t dist, uint32_t mean_ms, uint32_t scale, const uint32_t x[4]) {
  return latency_draw(dist, mean_ms, scale, x);
}

uint64_t or_loss_threshold(double p) { return loss_threshold(p); }

}  // extern "C"
