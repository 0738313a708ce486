// ms_kernels.cu -- hand-written sm_100a kernels of the discrete-event engine.
//
// One *round* of the simulation (DESIGN.md section 2.3) is:
//   k_release   (only when a latency distribution can produce latency > 0):
//               scatters the timing-wheel slot that just became due into the
//               per-endpoint inbox rings;
//   k_snapshot  head <- limit, limit <- tail: freezes the window every endpoint
//               consumes this round (messages sent in round r are first visible
//               in round r+1) and finds the largest window of the round;
//   k_round     ONE fused kernel replacing process.clj's stdin/stdout pumps,
//               the node program, net/send! (net.clj:189-221) and net/recv!
//               (net.clj:223-247).  One CTA per endpoint ("ticket"), CTAs are
//               independent of each other:
//                 load window -> order it by (round, sender, emission index),
//                 which is the order of the reference's global message-id
//                 counter -> partition check at dequeue -> node transition
//                 -> block scan of (recv, emit, new) counts
//                 -> :recv records, emissions: Philox loss/latency, :send
//                    records, scatter into the destination rings.
//               Launched once per window-size class; exactly one class runs.
// No outbox exists: a message goes HBM ring -> registers -> HBM ring.
//
// Dense message ids / event ids (the reference's two global counters,
// net.clj:197 and journal.clj:228) are prefix sums over (round, ticket, idx).
// They are NOT computed on the critical path: every CTA records its counts in
// a per-round table, the last CTA of the round turns them into prefixes, and
// ids are resolved when a message is received (one table lookup per sender
// block) or when the journal is drained (k_journal_expand).
//
// HBM-bound integer work; tensor cores are deliberately idle.
#include <cuda_runtime.h>
#include <stdint.h>
#include "ms_device.cuh"

namespace msd {

#define FULL 0xFFFFFFFFu
// Kernel launches go through one macro so that tests/native/emul (a CPU SIMT emulator used by
// the CPU test-suite only) can run these same sources; under nvcc it is the plain <<<>>> launch.
#ifndef MS_EMUL
#define MS_LAUNCH(kern, grid, block, smem, stream, ...) kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif
constexpr int MAXB = 64;            // sender blocks handled by the fast ordering path
constexpr int MAXNB = 8;            // neighbor slots handled by per-(CTA, neighbor) claims
constexpr uint64_t RECV_BIT = 1ull << 63;
constexpr uint32_t kResolvedTicket = 0xFFFFFFu;   // order key of a record that carries its dense id: (id >> 32, this, id & 0xFFFFFFFF)

// ------------------------------------------------------------------ small PTX helpers
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t* p) { return __ldcg(p); }
// streaming 16-byte store: journal / ring records are written once and read by
// another SM (or the host) later, so keep them out of L1.
__device__ __forceinline__ void st_v4(uint4* p, uint4 v) {
#ifdef MS_EMUL
  *p = v;
#else
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
#endif
}
__device__ __forceinline__ uint4 ld_v4_stream(const uint4* p) {
  uint4 v;
#ifdef MS_EMUL
  v = *p;
#else
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
#endif
  return v;
}

// Bulk prefetch of `bytes` (a multiple of 16) at a 16-byte aligned global address into L2: one instruction for
// a whole ring window (cp.async.bulk.prefetch, the bulk-copy engine's path; a hint, nothing waits on it).
__device__ __forceinline__ void prefetch_l2_bulk(const void* gptr, uint32_t bytes) {
#ifndef MS_EMUL
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
#else
  (void)gptr; (void)bytes;
#endif
}

__device__ __forceinline__ void latch_error(DevState* st, uint32_t code, uint32_t arg) {
  if (atomicCAS(&st->error, 0u, code) == 0u) st->error_arg = arg;
}

// A round is skipped (by every kernel of the round alike) when the simulation has
// reached its stop time, an error is latched, or the host has to drain the
// journal first (raw ring half full / round history nearly exhausted).
__device__ __forceinline__ bool round_skipped(const Params& p, const DevState* st) {
  if (st->now >= st->stop_ns || st->error) return true;
  if (p.jlevel && !p.jdiscard) {
    // only values that are constant while a round is in flight may be used here:
    // raw_base of the round's row is jraw_cursor as of the START of the round
    // (sharded runs: a per-shard condition would desynchronise the shards, so only the
    // history test below, which is identical on every shard, applies; overflow is an error)
    const uint64_t raw_base = p.rmeta[(uint32_t)st->round & p.hist_mask].raw_base;
    if (p.n_shards <= 1 && raw_base - st->jraw_drained > ((p.jmask + 1) >> 1)) return true;
    if (st->round - st->drain_round + 2 >= p.hist) return true;
  }
  return false;
}

// DevState.slot_open: 0 = no round open (committed / not snapshotted yet), else the tag of the open round.
// k_round's CTAs may start at any time while their launch is alive -- also while, or after, another CTA commits
// the round -- so "is my round still open" must be ONE consistent decision per CTA: the tag names the round.
__device__ __forceinline__ uint32_t slot_tag(uint64_t round) { return 0x80000000u | (uint32_t)(round & 0x7FFFFFFFull); }

// ------------------------------------------------------------------ ring records
// 48-B record: v0 = order key {idx, ticket, round}, v1 = {src, dest,
// msg_id, in_reply_to}, v2 = {type | flags << 16, p0, p1}.
struct Rec {
  uint64_t round;
  uint32_t ticket, idx;
  uint32_t src, dest, msg_id, in_reply_to;
  uint32_t tf;
  uint32_t p0;
  uint64_t p1;
};

__device__ __forceinline__ void rec_pack(const Rec& r, uint4& a, uint4& b, uint4& c) {
  a = make_uint4(r.idx, r.ticket, (uint32_t)r.round, (uint32_t)(r.round >> 32));
  b = make_uint4(r.src, r.dest, r.msg_id, r.in_reply_to);
  c = make_uint4(r.tf, r.p0, (uint32_t)r.p1, (uint32_t)(r.p1 >> 32));
}
// timing-wheel slot: the three vectors side by side
__device__ __forceinline__ void rec_store(uint4* slot, const Rec& r) {
  uint4 a, b, c;
  rec_pack(r, a, b, c);
  st_v4(slot + 0, a); st_v4(slot + 1, b); st_v4(slot + 2, c);
}
__device__ __forceinline__ Rec rec_unpack(uint4 a, uint4 b, uint4 c) {
  Rec r;
  r.idx = a.x; r.ticket = a.y;
  r.round = (uint64_t)a.z | ((uint64_t)a.w << 32);
  r.src = b.x; r.dest = b.y; r.msg_id = b.z; r.in_reply_to = b.w;
  r.tf = c.x; r.p0 = c.y;
  r.p1 = (uint64_t)c.z | ((uint64_t)c.w << 32);
  return r;
}

// Inbox ring of endpoint e: servers have rings of ring_cap_s records, every other endpoint
// (clients, hosts, services -- a service hears from every node) of ring_cap records.
__device__ __forceinline__ uint32_t ring_cap_of(const Params& p, uint32_t e) { return e < p.n_servers ? p.ring_cap_s : p.ring_cap; }
__device__ __forceinline__ size_t ring_base(const Params& p, uint32_t e) {
  return e < p.n_servers ? (size_t)e * p.ring_cap_s
                         : (size_t)p.n_servers * p.ring_cap_s + (size_t)(e - p.n_servers) * p.ring_cap;
}
// Slot g of the rings: order key v0 at ring[g] (key plane), v1 and v2 at ring[ring_slots + 2g] (body plane).
// A window's keys are one contiguous run, so a reader that needs only the keys touches 16 B per message.
__device__ __forceinline__ size_t ring_index(const Params& p, uint32_t e, uint32_t pos) {
  return ring_base(p, e) + (pos & (ring_cap_of(p, e) - 1u));
}
__device__ __forceinline__ void ring_put(const Params& p, uint4* ring, size_t g, uint4 a, uint4 b, uint4 c) {
  uint4* body = ring + p.ring_slots + 2 * g;
  st_v4(ring + g, a); st_v4(body, b); st_v4(body + 1, c);
}
__device__ __forceinline__ void ring_store(const Params& p, uint4* ring, uint32_t e, uint32_t pos, const Rec& r) {
  uint4 a, b, c;
  rec_pack(r, a, b, c);
  ring_put(p, ring, ring_index(p, e, pos), a, b, c);
}
// Compact record: server -> neighbor gossip written by k_round's fast path is the key vector alone,
// {idx, ticket | kCompact, (uint32_t)round, value}; its body-plane slot is not written (it may hold a
// stale record of an earlier lap).  The rest is implied: src = ticket - n_inj_tickets, dest = the
// ring's owner, msg_id = in_reply_to = p1 = 0, tf = MS_T_BROADCAST.  Tickets fit in 24 bits
// (kResolvedTicket), so the flag never collides with one; every ticket read from a key is masked.
constexpr uint32_t kCompact = 1u << 31;
__device__ __forceinline__ void ring_store_gossip(uint4* ring, size_t g, uint32_t idx, uint32_t ticket, uint64_t round,
                                                  uint32_t value) {
  st_v4(ring + g, make_uint4(idx, ticket | kCompact, (uint32_t)round, value));
}
// The round a compact key was sent in: its low word is stored, and it lies fewer than `hist` rounds
// before the reader's round `cur`.
__device__ __forceinline__ uint64_t compact_round(uint64_t cur, uint32_t lo) { return cur - (uint32_t)((uint32_t)cur - lo); }
__device__ __forceinline__ Rec ring_expand(const Params& p, uint4 a, uint4 b, uint4 c, uint64_t cur, uint32_t owner) {
  if (!(a.y & kCompact)) return rec_unpack(a, b, c);
  Rec r;
  r.idx = a.x; r.ticket = a.y & 0xFFFFFFu;
  r.round = compact_round(cur, a.z);
  r.src = r.ticket - p.n_inj_tickets; r.dest = owner; r.msg_id = 0; r.in_reply_to = 0;
  r.tf = MS_T_BROADCAST; r.p0 = a.w; r.p1 = 0;
  return r;
}
// Full record of slot g of `owner`'s ring as seen in round `cur`; key and body are loaded together.
__device__ __forceinline__ Rec ring_load(const Params& p, const uint4* ring, size_t g, uint64_t cur, uint32_t owner) {
  const uint4* body = ring + p.ring_slots + 2 * g;
  return ring_expand(p, ring[g], body[0], body[1], cur, owner);
}
// The record of slot g without its order key, for a ring that never holds compact records (only a
// broadcast server's ring does): one fewer load on the reply paths of clients, services and Raft.
__device__ __forceinline__ Rec ring_load_body(const Params& p, const uint4* ring, size_t g) {
  const uint4* body = ring + p.ring_slots + 2 * g;
  return rec_unpack(make_uint4(0u, 0u, 0u, 0u), body[0], body[1]);
}

// dense id of (round, ticket, idx): id_base[round] + emit_prefix[round][ticket] + idx
__device__ __forceinline__ uint64_t dense_base(const Params& p, DevState* st, uint64_t round, uint32_t ticket) {
  if (ticket == kResolvedTicket) return round << 32;   // the record already carries its id (k_release)
  const uint32_t row = (uint32_t)round & p.hist_mask;
  const RoundMeta* m = p.rmeta + row;
  if (m->round != round || ticket >= p.t_max) {
    latch_error(st, E_HISTORY, (uint32_t)round);
    return 0;
  }
  return m->id_base + p.rt_em[(size_t)row * p.t_max + ticket];
}

// ------------------------------------------------------------------ block primitives
// Exclusive scan of a[0..n) in shared memory, total written to a[n] and returned.
__device__ uint64_t block_excl_scan(uint64_t* a, int n, uint64_t* wtmp /* >= 33 */) {
  const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (n + nt - 1) / nt;
  const int lo = min(tid * c, n), hi = min(lo + c, n);
  uint64_t sum = 0;
  for (int i = lo; i < hi; i++) sum += a[i];
  uint64_t incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) wtmp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int nw = nt >> 5;
    const uint64_t w = lane < nw ? wtmp[lane] : 0;
    uint64_t wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t y = __shfl_up_sync(FULL, wi, d);
      if (lane >= d) wi += y;
    }
    wtmp[lane] = wi - w;
    if (lane == 31) wtmp[32] = wi;
  }
  __syncthreads();
  uint64_t run = wtmp[warp] + incl - sum;
  for (int i = lo; i < hi; i++) {
    const uint64_t v = a[i];
    a[i] = run;
    run += v;
  }
  const uint64_t total = wtmp[32];
  if (tid == 0) a[n] = total;
  __syncthreads();
  return total;
}

// Fallback ordering: bitonic sort of the index array `ord` (np a power of two,
// pads = 0xFFFF) by (keyA, keyB) of the records they point to.
__device__ void block_bitonic_sort_idx(uint16_t* ord, const uint64_t* keyA, const uint32_t* keyB, int np) {
  const int nt = blockDim.x, tid = threadIdx.x;
  for (int k = 2; k <= np; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = tid; t < (np >> 1); t += nt) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = i | j;
        const bool asc = (i & k) == 0;
        const uint16_t a = ord[i], b = ord[l];
        bool gt;   // key(a) > key(b)
        if (a == 0xFFFF) gt = (b != 0xFFFF);
        else if (b == 0xFFFF) gt = false;
        else gt = keyA[a] > keyA[b] || (keyA[a] == keyA[b] && keyB[a] > keyB[b]);
        if (gt == asc) { ord[i] = b; ord[l] = a; }
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------ emission (net/send!, net.clj:189-221)
struct EmitCtx {
  int64_t now;
  uint64_t round;
  uint64_t chunk;    // raw journal position of this CTA's chunk
  uint32_t n_recv;   // :recv records precede the :send records in the chunk
  uint32_t ticket;
  uint32_t emitter;  // Philox stream: endpoint index or kInjector
  uint32_t idx_bias; // added to local_idx for the Philox counter (injector slices)
  bool need_rng;     // false: no loss and constant latency, the random draw is never looked at
  uint64_t const_lat;
  // per-thread counters, reduced at the end of the CTA
  uint32_t c_send_cl, c_send_sv, c_lost, c_zero;
};

__device__ __forceinline__ void journal_raw(const Params& p, uint64_t pos, uint64_t id_or_idx, bool recv,
                                            const Rec& r) {
  if (p.jlevel == 0) return;
  const uint64_t v = id_or_idx | (recv ? RECV_BIT : 0ull);
  st_v4(p.jraw + (pos & p.jmask), make_uint4((uint32_t)v, (uint32_t)(v >> 32), r.src, r.dest));
  if (p.jlevel >= 2) {
    uint4* b = p.jbody + (pos & p.jmask) * 2;
    st_v4(b + 0, make_uint4((uint32_t)v, (uint32_t)(v >> 32), r.msg_id, r.in_reply_to));
    st_v4(b + 1, make_uint4(r.tf, r.p0, (uint32_t)r.p1, (uint32_t)(r.p1 >> 32)));
  }
}

// ------------------------------------------------------------------ timing wheel (pooled chains)
// A word another thread publishes with an atomic (wheel block ids, slot_open): a relaxed atomic load.  On the GPU a
// volatile 32-bit load is exactly that; the emulator build says so in C++ terms (ThreadSanitizer checks it).
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
#ifdef MS_EMUL
  return __atomic_load_n(p, __ATOMIC_RELAXED);
#else
  return *reinterpret_cast<const volatile uint32_t*>(p);
#endif
}

// Block `j` of the chain of (generation, slot): its pool index, allocating it on first use.  The
// thread that filed the first record of the block is its designated allocator; everybody else
// polls briefly for the published id and then allocates too (whoever publishes first wins, the
// others hand their block back through cal_ret), so no thread ever waits on another one.
__device__ uint32_t wheel_block(const Params& p, DevState* st, uint32_t* entry, bool designated) {
  uint32_t b = ld_volatile_u32(entry);
  if (b) return b - 1;
  if (!designated) {
    for (int spin = 0; spin < 64; spin++) {
      __nanosleep(64);
      b = ld_volatile_u32(entry);
      if (b) return b - 1;
    }
  }
  const uint32_t n = atomicAdd(&st->cal_free_n, 0xFFFFFFFFu);          // pop
  if (n == 0 || n > p.cal_blocks) {                                     // pool exhausted
    atomicAdd(&st->cal_free_n, 1u);
    latch_error(st, E_CALENDAR_OVERFLOW, 0xFFFFFFFFu);
    return 0xFFFFFFFFu;
  }
  const uint32_t mine = p.cal_free[n - 1];
  const uint32_t old = atomicCAS(entry, 0u, mine + 1u);
  if (old == 0u) return mine;
  p.cal_ret[atomicAdd(&st->cal_ret_n, 1u)] = mine;                       // somebody else published first
  return old - 1u;
}

// Files record r into wheel slot `slot`.  Convergent: all 32 lanes call, `valid` selects.
__device__ __forceinline__ void wheel_file(const Params& p, DevState* st, bool valid, uint32_t slot, const Rec& r) {
  const int lane = threadIdx.x & 31;
  const uint32_t key = valid ? slot : (0x80000000u | (uint32_t)lane);
  const uint32_t mask = __match_any_sync(FULL, key);
  const int leader = __ffs(mask) - 1;
  const uint32_t rank = __popc(mask & ((1u << lane) - 1u));
  uint32_t gen = 0, base = 0;
  if (valid && lane == leader) {
    gen = p.cal_par[slot];
    base = atomicAdd(&p.cal_count[(size_t)gen * p.cal_slots + slot], (uint32_t)__popc(mask));
  }
  gen = __shfl_sync(FULL, gen, leader);
  base = __shfl_sync(FULL, base, leader);
  if (!valid) return;
  const uint32_t k = base + rank;
  const uint32_t j = k >> p.cal_blk_log2, off = k & ((1u << p.cal_blk_log2) - 1u);
  if (j >= p.cal_tab_cap) { latch_error(st, E_CALENDAR_OVERFLOW, slot); return; }
  const uint32_t b = wheel_block(p, st, p.cal_tab + ((size_t)gen * p.cal_slots + slot) * p.cal_tab_cap + j, off == 0);
  if (b == 0xFFFFFFFFu) return;
  rec_store(p.cal + (((size_t)b << p.cal_blk_log2) + off) * 3, r);
}

// Must be called convergently by all 32 lanes of a warp.  has_direct
// means ring space for this record was already claimed by the CTA (per-neighbor
// block claim); otherwise slots are claimed here, one atomic per destination
// per warp.
__device__ __forceinline__ void emit_one(const Params& p, DevState* st, const NetParams& np, EmitCtx& cx,
                                         bool valid, Rec& r, uint32_t local_idx, uint32_t direct_pos,
                                         bool has_direct) {
  const int lane = threadIdx.x & 31;
  bool push = false, wheel = false;
  uint32_t wslot = 0;
  // A message whose src or dest is not a registered endpoint (net.clj:166-176) never reaches a queue.
  // In the reference the assert only throws inside the sending node's stdout thread
  // (process.clj:148-150), after the id was taken (net.clj:197); the network keeps running.  Here
  // the id is consumed, the :send is journaled, the message is dropped and counted (DESIGN.md 2.4).
  const bool undeliverable = valid && (r.dest >= p.n_ep || r.src >= p.n_ep ||
                                       (np.any_removed && ((p.kind[r.dest] | p.kind[r.src]) & kRemoved)));
  if (valid) {
    r.round = cx.round; r.ticket = cx.ticket; r.idx = local_idx;     // order key == id order (net.clj:197)
    uint32_t x[4] = {0xFFFFFFFFu, 0, 0, 0};
    if (cx.need_rng)
      philox4x32_10(local_idx + cx.idx_bias, cx.emitter, (uint32_t)cx.round, (uint32_t)(cx.round >> 32),
                    p.seed_lo, p.seed_hi, x);
    // util.clj:12-16; servers are the endpoints below n_servers, so most lookups are avoided
    const bool cl = (r.src >= p.n_servers && r.src < p.n_ep && kind_is_client(p.kind[r.src])) ||
                    (r.dest >= p.n_servers && r.dest < p.n_ep && kind_is_client(p.kind[r.dest]));
    const uint64_t lat = cl ? 0ull : (cx.need_rng ? latency_ms(np, x) : cx.const_lat);   // net.clj:185-187
    journal_raw(p, cx.chunk + cx.n_recv + local_idx, local_idx, false, r);   // net.clj:208 (before the loss roll)
    if (cl) cx.c_send_cl++; else cx.c_send_sv++;
    if (undeliverable) {
      atomicAdd((unsigned long long*)&st->undeliverable, 1ull);
    } else if ((uint64_t)x[0] < np.loss_thresh) {                    // net.clj:214-215
      cx.c_lost++;
    } else if (lat == 0) {                                           // deadline == now: next delta round
      cx.c_zero++;
      if (has_direct) {
        ring_store(p, p.ring_sh[owner_of(r.dest, p.n_servers, p.n_shards)], r.dest, direct_pos, r);
      } else {
        push = true;
      }
    } else {
      // timing wheel: slot of the deadline tick (net.clj:202-205); a latency of cal_slots ticks or
      // more waits `laps` further turns in that slot
      const uint64_t tick = (uint64_t)(cx.now / kTickNs) + lat;
      const uint64_t laps = (lat - 1) / p.cal_slots;
      if (p.cal == nullptr || laps > 0xFFFFu) {
        latch_error(st, E_CALENDAR_OVERFLOW, (uint32_t)lat);
      } else {
        wheel = true;
        wslot = (uint32_t)tick & (p.cal_slots - 1);
        r.round |= laps << 48;
      }
    }
  }
  if (__any_sync(FULL, wheel)) wheel_file(p, st, wheel, wslot, r);
  if (!__any_sync(FULL, push)) return;
  // warp-aggregated claim of ring slots: one atomic per distinct destination
  const uint32_t key = push ? r.dest : (0x80000000u | (uint32_t)lane);
  const uint32_t mask = __match_any_sync(FULL, key);
  const int leader = __ffs(mask) - 1;
  const uint32_t rank = __popc(mask & ((1u << lane) - 1u));
  uint32_t base = 0;
  const uint32_t o = push ? owner_of(r.dest, p.n_servers, p.n_shards) : 0u;   // NVLink peer memory when o != shard_id
  if (push && lane == leader) base = atomicAdd(&p.tail_sh[o][r.dest], (uint32_t)__popc(mask));
  base = __shfl_sync(FULL, base, leader);
  if (push) {
    const uint32_t pos = base + rank;
    if ((uint32_t)(pos - p.head_sh[o][r.dest]) >= ring_cap_of(p, r.dest)) {
      latch_error(st, E_RING_OVERFLOW, r.dest);
    } else {
      ring_store(p, p.ring_sh[o], r.dest, pos, r);
    }
  }
}

__global__ void k_set_bit(uint32_t* words, size_t word, uint32_t bit) { atomicOr(words + word, 1u << bit); }

// ------------------------------------------------------------------ closed-loop clients (MS_KIND_GEN_CLIENT)
// maelstrom.client (client.clj:41-172) + what a Jepsen worker does with the workload's generator
// (workload/broadcast.clj:187-241, core.clj:67-80); the spec is in include/maelstrom_b200.h
// (ms_add_gen_clients) and DESIGN.md 2.10; the oracle's twin is or_sim::gen_step.
__device__ __forceinline__ void gen_hist(const Params& p, DevState* st, int64_t now, uint64_t round, uint32_t e,
                                         const GenDev& g, uint32_t op, uint32_t type, uint32_t f, uint32_t error, uint32_t value) {
  const unsigned long long pos = atomicAdd((unsigned long long*)&st->gc_hist_n, 1ull);
  if (pos - st->gc_hist_drained > p.gc_hist_mask) { latch_error(st, E_HISTORY_RING, e); return; }
  uint4* at = p.gc_hist + (pos & p.gc_hist_mask) * 2;
  const uint64_t order = (round << 24) | g.ordinal;
  at[0] = make_uint4((uint32_t)now, (uint32_t)((uint64_t)now >> 32), (uint32_t)order, (uint32_t)(order >> 32));
  at[1] = make_uint4(e, op, type | (f << 8) | (error << 16), value);
}

__device__ __forceinline__ bool gen_timer_due(const Params& p, const GenDev& g, int64_t now) {
  if (g.waiting_for) return now >= g.deadline_ns;
  if (g.phase == GEN_MIX) return now >= p.gc_limit_ns || now >= g.next_op_ns;
  if (g.phase == GEN_QUIET) return now >= p.gc_limit_ns + p.gc_quiet_ns;
  return g.phase == GEN_FINAL;            // the final read has completed or timed out: -> done
}

// One step of client e: its due replies in id order, then the timeout, then at most one invocation.
// Returns true and fills `out` when the step sends a request.
__device__ bool gen_step(const Params& p, DevState* st, uint32_t e, int64_t now, uint64_t round, size_t my0,
                         uint32_t head, uint32_t my_mask, uint32_t n, const uint16_t* ord, const uint32_t* vals, Rec& out) {
  GenDev g = p.gc[e];
  for (uint32_t pos = 0; pos < n; pos++) {
    const uint32_t i = ord[pos];
    if (!(vals[i] & (1u << 30))) continue;                                 // V_RECV: cut by a partition
    const Rec m = ring_load_body(p, p.ring, my0 + ((head + i) & my_mask));
    const uint32_t type = m.tf & 0xFFFFu, flags = m.tf >> 16;
    if (!g.waiting_for || !(flags & MS_F_REPLY) || m.in_reply_to != g.waiting_for) continue;   // client.clj:106-107
    uint32_t outcome = MS_H_OK, err = 0, value = g.cur_value;
    if (type == MS_T_ERROR) {                                              // client.clj:165-172, errors.edn
      err = m.p0;
      const bool definite = err != 0 && err != 13;
      outcome = (definite || g.cur_f == MS_HF_READ) ? MS_H_FAIL : MS_H_INFO;
    } else if (g.cur_f == MS_HF_READ) {
      value = m.p0;                                                        // read_ok: the size of the set
    }
    gen_hist(p, st, now, round, e, g, g.ops, outcome, g.cur_f, err, value);
    g.waiting_for = 0;
  }
  if (g.waiting_for && now >= g.deadline_ns) {                             // client.clj:96-101,160-164
    gen_hist(p, st, now, round, e, g, g.ops, g.cur_f == MS_HF_READ ? MS_H_FAIL : MS_H_INFO, g.cur_f, MS_H_TIMEOUT, g.cur_value);
    g.waiting_for = 0;
  }
  bool send = false;
  if (!g.waiting_for) {
    uint32_t f = MS_HF_READ, value = 0;
    if (g.phase == GEN_MIX) {
      if (now >= p.gc_limit_ns) g.phase = GEN_QUIET;
      else if (now >= g.next_op_ns) {
        uint32_t x[4];
        philox4x32_10(g.ops, e, 0xC11E47u, 0u, p.seed_lo, p.seed_hi, x);   // the client's own stream: op k
        if ((((uint64_t)x[0] * 1000u) >> 32) >= p.gc_read_permille) { f = MS_HF_BROADCAST; value = g.ordinal + p.gc_n * g.bcasts++; }
        g.next_op_ns = now + (int64_t)(((unsigned __int128)x[1] * (unsigned __int128)(2 * (uint64_t)p.gc_interval_ns)) >> 32);
        send = true;
      }
    }
    if (g.phase == GEN_QUIET && now >= p.gc_limit_ns + p.gc_quiet_ns) { g.phase = GEN_FINAL; send = true; }   // broadcast.clj:237-240
    else if (g.phase == GEN_FINAL && !send) g.phase = GEN_DONE;
    if (send) {
      g.ops++;
      g.cur_f = f; g.cur_value = value;
      g.waiting_for = ++g.next_msg_id;                                     // client.clj:61-64
      g.deadline_ns = now + p.gc_timeout_ns;
      gen_hist(p, st, now, round, e, g, g.ops, MS_H_INVOKE, f, 0, value);
      out.round = 0; out.ticket = 0; out.idx = 0;
      out.src = e; out.dest = g.node; out.msg_id = g.waiting_for; out.in_reply_to = 0;
      const uint32_t wtype = f == MS_HF_READ ? (uint32_t)MS_T_READ : (p.workload == MS_W_GSET ? (uint32_t)MS_T_ADD : (uint32_t)MS_T_BROADCAST);
      out.tf = wtype | ((uint32_t)MS_F_MSG_ID << 16);
      out.p0 = value; out.p1 = 0;
    }
  }
  p.gc[e] = g;
  return send;
}

#include "ms_tree.h"
#include "ms_raft.cuh"

// ------------------------------------------------------------------ k_barrier (sharded runs)
// Cross-GPU barrier over NVLink peer memory: every shard stores the epoch into its slot of
// every peer's flag array, then waits until all peers have stored it into its own.  Kernels
// of one shard are stream-ordered around it, so everything a shard wrote into peer inbox
// rings before the barrier is visible to the owner after it.
// Called by every thread of ONE CTA (the only CTA of its kernel); returns after a __syncthreads().
__device__ void barrier_body(const Params& p, uint32_t* s_epoch) {
  // the epoch lives on the device so that the launch sequence can be replayed from a CUDA graph;
  // all shards execute the same number of barriers, so their counters agree
  __syncthreads();                     // everything this CTA did before the barrier is done
  if (threadIdx.x == 0) *s_epoch = ++p.st->bar_epoch;
  __syncthreads();
  const uint32_t epoch = *s_epoch;
  const uint32_t g = threadIdx.x;
  if (g < p.n_shards) {
    __threadfence_system();
    *reinterpret_cast<volatile uint32_t*>(&p.bar_sh[g][p.shard_id]) = epoch;
    __threadfence_system();
    const volatile uint32_t* mine = p.bar_sh[p.shard_id] + g;
    uint32_t spins = 0;
    while ((int32_t)(*mine - epoch) < 0) {
      if (++spins > (1u << 27)) { latch_error(p.st, E_BARRIER, g); break; }   // a peer died: do not hang the GPU
      __nanosleep(40);
    }
    __threadfence_system();
  }
  __syncthreads();
}

__global__ void k_barrier(Params p) {
  __shared__ uint32_t s_epoch;
  barrier_body(p, &s_epoch);
}

// ------------------------------------------------------------------ k_snapshot
// head <- limit, limit <- tail, and sorts every ticket into the work list of the
// k_round size class its window fits (DESIGN.md 3.4).  Lists are double-buffered
// by round parity; the other parity's counters are cleared here.
__device__ __forceinline__ uint32_t class_of(const Params& p, uint32_t n) {
  uint32_t c = 0;
  while (c + 1 < p.n_classes && n > p.cls_cap[c]) c++;
  return c;
}

// The per-endpoint part of k_snapshot for the threads gid, gid + stride, ...: also run by the single CTA of
// k_glue (sharded runs), right after it has committed the previous round.
__device__ void snapshot_endpoints(const Params& p, DevState* st, uint32_t gid, uint32_t stride);

__global__ void k_snapshot(Params p) {
  DevState* st = p.st;
  if (round_skipped(p, st)) return;
  snapshot_endpoints(p, st, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
  const uint32_t par = (uint32_t)st->round & 1u;
  const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0) {
    // timing wheel housekeeping, one CTA (nothing pops blocks while this kernel runs): the chain
    // k_release has just emptied goes back to the pool, and so do blocks that lost a publish race
    if (p.cal && st->cal_release) {
      const uint32_t slot = st->cal_release - 1;
      const uint32_t gen = p.cal_par[slot] ^ 1u;                        // the generation that was released
      uint32_t* cnt = p.cal_count + (size_t)gen * p.cal_slots + slot;
      uint32_t* tab = p.cal_tab + ((size_t)gen * p.cal_slots + slot) * p.cal_tab_cap;
      const uint32_t nb = min((*cnt + (1u << p.cal_blk_log2) - 1u) >> p.cal_blk_log2, p.cal_tab_cap);
      for (uint32_t j = threadIdx.x; j < nb; j += blockDim.x) {
        const uint32_t b = tab[j];
        if (b) { p.cal_free[atomicAdd(&st->cal_free_n, 1u)] = b - 1u; tab[j] = 0; }
      }
      __syncthreads();
      if (threadIdx.x == 0) { *cnt = 0; st->cal_release = 0; }
    }
    if (p.cal) {
      const uint32_t nr = st->cal_ret_n;
      for (uint32_t i = threadIdx.x; i < nr; i += blockDim.x) p.cal_free[atomicAdd(&st->cal_free_n, 1u)] = p.cal_ret[i];
      __syncthreads();
      if (threadIdx.x == 0) st->cal_ret_n = 0;
    }
  }
  if (gid == 0) {
    for (int c = 0; c < 4; c++) { st->cls_count[par ^ 1u][c] = 0; st->cls_small[par ^ 1u][c] = 0; st->cls_cursor[par ^ 1u][c] = 0; }
    st->slot_open = slot_tag(st->round);
  }
}

__device__ void snapshot_endpoints(const Params& p, DevState* st, uint32_t gid, uint32_t stride) {
  const uint32_t par = (uint32_t)st->round & 1u;
  const uint32_t row = (uint32_t)st->round & p.hist_mask;
  const uint64_t empty_entry = (uint64_t)(((uint32_t)st->round & 0x7FFFu) + 1u) << 48;   // tag | 0 events | 0 emissions
  uint32_t n_empty = 0;
  for (uint32_t e = gid; e < p.n_ep; e += stride) {
    if (owner_of(e, p.n_servers, p.n_shards) != p.shard_id) continue;   // another shard's endpoint
    const uint32_t h = p.limit[e], l = p.tail[e];
    p.head[e] = h;
    p.limit[e] = l;
    const uint32_t n = ((p.kind[e] & kRemoved)) ? 0u : l - h;
    // g-set: a node whose periodic replication task is due emits even with an empty window
    // Raft: a node whose election / step-down / replication timers are due acts on an empty window too
    const bool timer_due = e < p.n_servers && p.kind[e] == MS_KIND_SERVER &&
                           ((p.workload == MS_W_GSET && p.gs_init[e] && st->now >= p.gs_next_fire[e]) ||
                            (p.workload == MS_W_RAFT && rf_timer_due(p.rf_node[e], st->now)) ||
                            (p.workload == MS_W_TXN_TREE && tt_timer_due(p.tt_node[e], st->now)));
    const bool gen_due = p.gc && p.kind[e] == MS_KIND_GEN_CLIENT && gen_timer_due(p, p.gc[e], st->now);
    if (n == 0 && !timer_due && !gen_due) {
      // nothing to receive, hence nothing to emit: the ticket is finished right here
      const uint32_t t = p.n_inj_tickets + e;
      p.rt_chunk[(size_t)row * p.t_max + t] = 0;
      __stcg(reinterpret_cast<unsigned long long*>(p.rt_cnt + (size_t)row * p.t_max + t), (unsigned long long)empty_entry);
      n_empty++;
      continue;
    }
    // longest windows first: a class's list is filled from the front by the windows in the upper half
    // of its size range and from the back by the others, and consumed front to back, so the tail of
    // a round is made of short tickets
    const uint32_t c = class_of(p, n);
    const uint32_t lo_cap = c ? p.cls_cap[c - 1] : 0u;
    uint32_t* list = p.cls_list + ((size_t)par * 4 + c) * p.t_max;
    // (k < t_max always holds for a round that is snapshotted once; the bound keeps a stuck round from writing wild)
    if (n > lo_cap + ((min(p.cls_cap[c], p.max_window) - lo_cap) >> 1)) {
      const uint32_t k = atomicAdd(&st->cls_count[par][c], 1u);
      if (k < p.t_max) list[k] = p.n_inj_tickets + e;
    } else {
      const uint32_t k = atomicAdd(&st->cls_small[par][c], 1u);
      if (k < p.t_max) list[p.t_max - 1u - k] = p.n_inj_tickets + e;
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) n_empty += __shfl_xor_sync(FULL, n_empty, d);
  // the injector tickets always run in k_round, so some ticket still finishes after this
  // kernel and commits the round once `done` reaches the ticket count
  if ((threadIdx.x & 31) == 0 && n_empty) atomicAdd(&st->done, n_empty);
  if (gid < p.n_inj_tickets && p.shard_id == 0) {   // injector slices run in the widest class (shard 0)
    const uint32_t c = p.n_classes - 1;
    const uint32_t k = atomicAdd(&st->cls_count[par][c], 1u);
    if (k < p.t_max) p.cls_list[((size_t)par * 4 + c) * p.t_max + k] = gid;
  }
}

// ------------------------------------------------------------------ k_release (timing wheel -> rings)
__global__ void k_release(Params p) {
  DevState* st = p.st;
  if (round_skipped(p, st) || st->cal_release == 0) return;
  const uint32_t slot = st->cal_release - 1;
  const uint32_t gen = p.cal_par[slot] ^ 1u;           // the commit that scheduled this release flipped the slot
  const uint32_t n = p.cal_count[(size_t)gen * p.cal_slots + slot];
  const uint32_t* tab = p.cal_tab + ((size_t)gen * p.cal_slots + slot) * p.cal_tab_cap;
  const uint32_t stride = gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const uint32_t n_round = (n + 31u) & ~31u;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
    bool valid = i < n;
    uint4 a = make_uint4(0, 0, 0, 0), b = a, c = a;
    if (valid) {
      const uint32_t j = i >> p.cal_blk_log2;
      const uint32_t blk = j < p.cal_tab_cap ? tab[j] : 0u;
      if (blk == 0) {
        valid = false;                                 // never filed: the overflow was latched by the sender
      } else {
        const uint4* src = p.cal + ((((size_t)(blk - 1u)) << p.cal_blk_log2) + (i & ((1u << p.cal_blk_log2) - 1u))) * 3;
        a = ld_v4_stream(src); b = ld_v4_stream(src + 1); c = ld_v4_stream(src + 2);
      }
    }
    // The sender's round is committed by now: turn the order key (round, ticket, idx) into the
    // dense message id once, here, so that a message may stay in flight for any number of rounds
    // without pinning the per-round history.  A released window holds only such records (time
    // advances only after a round without zero-latency sends, DESIGN.md 2.3), ordered by id.
    const uint32_t laps = a.w >> 16;
    if (valid && (a.y & 0xFFFFFFu) != kResolvedTicket) {
      const uint64_t id = dense_base(p, st, (uint64_t)a.z | ((uint64_t)(a.w & 0xFFFFu) << 32), a.y) + a.x;
      a = make_uint4((uint32_t)id, kResolvedTicket, (uint32_t)(id >> 32), laps << 16);
    }
    // a record with laps left stays in the slot for another turn of the wheel
    const bool again = valid && laps > 0;
    if (__any_sync(FULL, again)) {
      Rec r = rec_unpack(a, b, c);
      r.round = (r.round & 0xFFFFFFFFFFFFull) | ((uint64_t)(laps - 1u) << 48);
      wheel_file(p, st, again, slot, r);
    }
    if (again) valid = false;
    const uint32_t dest = b.y;
    // the endpoint slot was handed to a new endpoint after this message was sent: its queue went
    // with the old one (net.clj:148-152)
    if (valid && (((uint64_t)a.x | ((uint64_t)a.z << 32)) < p.ep_born[dest])) valid = false;
    const uint32_t key = valid ? dest : (0x80000000u | (uint32_t)lane);
    const uint32_t mask = __match_any_sync(FULL, key);
    const int leader = __ffs(mask) - 1;
    const uint32_t rank = __popc(mask & ((1u << lane) - 1u));
    uint32_t base = 0;
    const uint32_t o = valid ? owner_of(dest, p.n_servers, p.n_shards) : 0u;
    if (valid && lane == leader) base = atomicAdd(&p.tail_sh[o][dest], (uint32_t)__popc(mask));
    base = __shfl_sync(FULL, base, leader);
    if (valid) {
      const uint32_t pos = base + rank;
      // the previous window is fully consumed by now: the whole ring past `head` is writable
      if ((uint32_t)(pos - p.head_sh[o][dest]) >= ring_cap_of(p, dest)) {
        latch_error(st, E_RING_OVERFLOW, dest);
      } else {
        ring_put(p, p.ring_sh[o], ring_index(p, dest, pos), a, b, c);
      }
    }
  }
}

// ------------------------------------------------------------------ node programs
// Fields of a delivered message the node programs look at (from ring_load).
struct MsgView {
  uint32_t src, msg_id, p0;
  uint32_t tf;   // type | flags << 16
};

// vals[] bits
constexpr uint32_t V_FRESH = 1u << 31;  // broadcast value unseen so far (after PC: first sight = new)
constexpr uint32_t V_RECV = 1u << 30;   // passed the partition check
constexpr uint32_t V_CAND = 1u << 29;   // carries a broadcast value that needs the seen-set test
constexpr uint32_t V_MASK = (1u << 29) - 1u;


// neighbor list of the node held in shared memory when it is short (nl != nullptr)
struct NbrList {
  const uint32_t* nl;
  uint32_t deg;
};

__device__ __forceinline__ uint32_t nbr_count(const Params& p, uint32_t e) {
  if (p.topology == MS_TOPO_TOTAL) return p.n_servers - 1;
  return p.nbr_off[e + 1] - p.nbr_off[e];
}
__device__ __forceinline__ uint32_t nbr_at(const Params& p, uint32_t e, uint32_t j) {
  if (p.topology == MS_TOPO_TOTAL) return j < e ? j : j + 1;   // broadcast.clj:82-89
  return p.nbr[p.nbr_off[e] + j];
}
// position of `src` in e's neighbor list, or 0xFFFFFFFF
__device__ __forceinline__ uint32_t nbr_pos(const Params& p, uint32_t e, uint32_t src) {
  if (p.topology == MS_TOPO_TOTAL) {
    if (src >= p.n_servers || src == e) return 0xFFFFFFFFu;
    return src < e ? src : src - 1;
  }
  const uint32_t lo = p.nbr_off[e], hi = p.nbr_off[e + 1];
  for (uint32_t j = lo; j < hi; j++) if (p.nbr[j] == src) return j - lo;
  return 0xFFFFFFFFu;
}

// number of emissions of one delivered message (count phase)
__device__ __forceinline__ uint32_t nbr_pos_l(const Params& p, uint32_t e, uint32_t src, const NbrList& L) {
  if (L.nl == nullptr) return nbr_pos(p, e, src);
  for (uint32_t j = 0; j < L.deg; j++) if (L.nl[j] == src) return j;
  return 0xFFFFFFFFu;
}

__device__ __forceinline__ uint32_t node_emit_count(const Params& p, uint32_t e, const MsgView& w, bool is_new,
                                                    const NbrList& L) {
  const uint32_t type = w.tf & 0xFFFFu;
  const bool has_id = (w.tf >> 16) & MS_F_MSG_ID;
  const bool is_reply = (w.tf >> 16) & MS_F_REPLY;
  if (p.workload == MS_W_ECHO) {                       // demo/ruby/echo.rb:28-39
    return (type == MS_T_INIT || type == MS_T_ECHO) ? 1u : 0u;
  }
  // broadcast node (doc/03-broadcast/01-broadcast.md:527-544, 02-performance.md:61-67)
  if (is_reply) return 0;                              // node.rb:159-164
  switch (type) {
    case MS_T_INIT: case MS_T_TOPOLOGY: case MS_T_READ: return 1;
    case MS_T_BROADCAST: {
      uint32_t n = has_id ? 1u : 0u;
      if (is_new) {
        n += L.deg;
        if (nbr_pos_l(p, e, w.src, L) != 0xFFFFFFFFu) n -= 1;   // skip whoever sent it to us
      }
      return n;
    }
    default: return has_id ? 1u : 0u;                  // error 10 not-supported (errors.edn)
  }
}

// k-th emission of a delivered message (emit phase).  Returns the neighbor slot
// the emission goes to when it is gossip to a topology neighbor, else -1.
__device__ __forceinline__ int node_emit(const Params& p, uint32_t e, const MsgView& w, uint32_t k,
                                         uint32_t nemit, uint32_t emit_idx, uint32_t msg_id_base,
                                         uint32_t set_before, uint32_t new_before, uint64_t p1, Rec& r,
                                         const NbrList& L) {
  const uint32_t type = w.tf & 0xFFFFu;
  int slot = -1;
  r.src = e; r.dest = w.src; r.msg_id = 0; r.in_reply_to = w.msg_id;
  r.p0 = 0; r.p1 = 0;
  uint32_t otype = MS_T_ERROR, oflags = MS_F_REPLY;
  if (p.workload == MS_W_ECHO) {
    otype = (type == MS_T_INIT) ? MS_T_INIT_OK : MS_T_ECHO_OK;
    oflags |= MS_F_MSG_ID;
    r.msg_id = msg_id_base + 1 + emit_idx;             // echo.rb:12-13
    if (type == MS_T_ECHO) { r.p0 = w.p0; r.p1 = p1; }
  } else {
    switch (type) {
      case MS_T_INIT: otype = MS_T_INIT_OK; break;
      case MS_T_TOPOLOGY: otype = MS_T_TOPOLOGY_OK; break;
      case MS_T_READ: otype = MS_T_READ_OK; r.p0 = set_before + new_before; break;
      case MS_T_BROADCAST: {
        const bool has_id = (w.tf >> 16) & MS_F_MSG_ID;
        if (has_id && k == nemit - 1) { otype = MS_T_BROADCAST_OK; break; }
        // gossip to the k-th neighbor other than the sender, in topology order
        const uint32_t ps = nbr_pos_l(p, e, w.src, L);
        const uint32_t j = (ps != 0xFFFFFFFFu && k >= ps) ? k + 1 : k;
        r.dest = L.nl ? L.nl[j] : nbr_at(p, e, j);
        slot = (int)j;
        otype = MS_T_BROADCAST; oflags = 0; r.in_reply_to = 0; r.p0 = w.p0;
        break;
      }
      default: otype = MS_T_ERROR; r.p0 = 10; break;
    }
  }
  r.tf = otype | (oflags << 16);
  return slot;
}

// ------------------------------------------------------------------ round commit
// The scalar part of a round's commit (one thread): totals, next ids, time advance, next round's row.
__device__ void commit_scalars(const Params& p, DevState* st, uint64_t total, uint32_t zp_any, uint32_t T) {
  const int64_t now = st->now;
  const uint64_t round = st->round;
  const uint32_t row = (uint32_t)round & p.hist_mask;
  {
      const uint64_t ev_total = total >> 32, em_total = total & 0xFFFFFFFFull;
      RoundMeta* m = p.rmeta + row;
      m->ev_total = ev_total;
      m->em_total = em_total;
      m->n_tickets = T;
      st->next_event += ev_total;
      st->next_id += em_total;
      const uint64_t tick = (uint64_t)(now / kTickNs);
      uint32_t hi_s = (tick + 1 < p.n_tick_off) ? p.tick_off[tick + 1] : p.n_sched;
      if (hi_s > st->sched_cursor) st->sched_cursor = hi_s;
      st->inj_count = 0;
      int64_t next_now = now;
      if (zp_any == 0) {
        next_now = now + kTickNs;
        st->now = next_now;
        st->time_advanced = 1;
        if (p.cal) {
          // the slot of the new tick is released before the next round; what is filed into it from
          // now on (latencies of whole turns, re-filed laps) belongs to its next generation
          const uint32_t slot = ((uint32_t)(tick + 1)) & (p.cal_slots - 1);
          st->cal_release = slot + 1;
          p.cal_par[slot] ^= 1u;
        }
      } else {
        st->time_advanced = 0;
      }
      st->round = round + 1;
      st->rounds_run += 1;
      st->done = 0;
      st->slot_open = 0;
      const uint64_t raw_cur = *reinterpret_cast<volatile uint64_t*>(&st->jraw_cursor);
      if (p.jdiscard || !p.jlevel) {
        st->journal_drained = st->next_event;
        st->jraw_drained = raw_cur;
        st->drain_round = round + 1;
      }
      // open the next round's row
      RoundMeta* nx = p.rmeta + ((uint32_t)(round + 1) & p.hist_mask);
      nx->round = round + 1;
      nx->now = next_now;
      nx->id_base = st->next_id;
      nx->ev_base = st->next_event;
      nx->raw_base = raw_cur;
      nx->n_tickets = 0;
      nx->ev_total = 0;
      nx->em_total = 0;
      __threadfence();
  }
}


// Commit of a round (DESIGN.md 2.3 step 4), executed by one whole CTA: turn the per-ticket
// counts of every shard into exclusive prefixes, advance the id / event / time counters and
// open the next round's row.  Single GPU: called by the last ticket inside k_round; sharded:
// by k_commit on every shard (all shards compute the same values) after the barrier.
__device__ void commit_round(const Params& p, DevState* st, uint64_t* s_wtmp) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t now = st->now;
  const uint64_t round = st->round;
  const uint32_t T = p.n_inj_tickets + p.n_ep;
  const uint32_t row = (uint32_t)round & p.hist_mask;
  const uint32_t tag = ((uint32_t)round & 0x7FFFu) + 1u;
    uint32_t* em = p.rt_em + (size_t)row * p.t_max;
    uint32_t* ev = p.rt_ev + (size_t)row * p.t_max;
    // pass 1 (strided, loads batched 4 deep): validate the tags, unpack the counts
    uint32_t zp_any = 0;
    for (int base = 0; base < (int)T; base += 4 * nt) {
      uint64_t v[4];
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int i = base + q * nt + tid;
        v[q] = i < (int)T ? __ldcg(reinterpret_cast<const unsigned long long*>(p.rt_cnt_sh[owner_of_ticket((uint32_t)i, p.n_inj_tickets, p.n_servers, p.n_shards)] + (size_t)row * p.t_max + i)) : ((uint64_t)tag << 48);
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int i = base + q * nt + tid;
        if (i >= (int)T) continue;
        // every ticket has bumped `done`, so its entry store is in flight at worst: wait for the tag
        for (uint32_t spin = 0; (uint32_t)(v[q] >> 48) != tag && spin < (1u << 22); spin++)
          v[q] = __ldcg(reinterpret_cast<const unsigned long long*>(p.rt_cnt_sh[owner_of_ticket((uint32_t)i, p.n_inj_tickets, p.n_servers, p.n_shards)] + (size_t)row * p.t_max + i));
        if ((uint32_t)(v[q] >> 48) != tag) latch_error(st, E_HISTORY, (uint32_t)i);
        zp_any |= (uint32_t)(v[q] >> 47) & 1u;
        ev[i] = (uint32_t)(v[q] >> 24) & 0x7FFFFFu;
        em[i] = (uint32_t)v[q] & 0xFFFFFFu;
      }
    }
    zp_any = __syncthreads_or(zp_any);   // also makes ev[]/em[] visible to the whole CTA
    // pass 2 (one contiguous chunk per thread): exclusive prefix
    const int c = ((int)T + nt - 1) / nt;
    const int lo = min(tid * c, (int)T), hi = min(lo + c, (int)T);
    uint64_t sum = 0;   // ev << 32 | em  (per-round totals stay below 2^32)
    for (int i = lo; i < hi; i++) sum += ((uint64_t)ev[i] << 32) | em[i];
    uint64_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t y = __shfl_up_sync(FULL, incl, d);
      if (lane >= d) incl += y;
    }
    if (lane == 31) s_wtmp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const int nw = nt >> 5;
      const uint64_t w = lane < nw ? s_wtmp[lane] : 0;
      uint64_t wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint64_t y = __shfl_up_sync(FULL, wi, d);
        if (lane >= d) wi += y;
      }
      s_wtmp[lane] = wi - w;
      if (lane == 31) s_wtmp[32] = wi;
    }
    __syncthreads();
    uint64_t run = s_wtmp[warp] + incl - sum;
    for (int i = lo; i < hi; i++) {
      const uint32_t ve = ev[i], vm = em[i];   // written in pass 1, visible after the barrier
      ev[i] = (uint32_t)(run >> 32);
      em[i] = (uint32_t)run;
      run += ((uint64_t)ve << 32) | vm;
    }
    const uint64_t total = s_wtmp[32];
    __syncthreads();
    if (tid == 0) commit_scalars(p, st, total, zp_any, T);
}

__global__ void __launch_bounds__(512) k_commit(Params p) {
  __shared__ uint64_t s_wtmp[34];
  DevState* st = p.st;
  if (round_skipped(p, st) || !st->slot_open) return;
  commit_round(p, st, s_wtmp);
}

// Sharded runs, one launch between two rounds instead of four (k_barrier | k_commit | k_snapshot | k_barrier):
// barrier A -- every shard's round kernels are done and their peer writes visible; commit of the open round (all
// shards compute the same prefixes from all shards' counts); snapshot of this shard's endpoints for the next round
// unless it is skipped; barrier B -- nobody writes into a peer's ring before that peer has frozen its windows.
// open_next = 0 closes a batch of rounds: barrier A and the commit only.  Not used with the timing wheel (k_release
// and its barrier come between commit and snapshot) nor with many endpoints (one CTA walks them).
__global__ void __launch_bounds__(512) k_glue(Params p, uint32_t open_next) {
  __shared__ uint64_t s_wtmp[34];
  __shared__ uint32_t s_epoch;
  DevState* st = p.st;
  barrier_body(p, &s_epoch);
  if (!round_skipped(p, st) && st->slot_open) commit_round(p, st, s_wtmp);
  __syncthreads();
  if (!open_next) return;
  if (!round_skipped(p, st)) {                         // the state the commit has just left behind
    snapshot_endpoints(p, st, threadIdx.x, blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t par = (uint32_t)st->round & 1u;
      for (int c = 0; c < 4; c++) { st->cls_count[par ^ 1u][c] = 0; st->cls_small[par ^ 1u][c] = 0; st->cls_cursor[par ^ 1u][c] = 0; }
      st->slot_open = slot_tag(st->round);
    }
  }
  barrier_body(p, &s_epoch);
}

// Commit in three launches for simulations with very many endpoints (tens of thousands of tickets:
// one CTA walking all of them would dominate a round).  A: every block of kCommitBlk tickets
// validates and unpacks its entries and leaves its sum; B: one CTA scans the block sums and does the
// scalar commit; C: every block turns its counts into prefixes.  Same results as commit_round.
constexpr uint32_t kCommitBlk = 1024;

__global__ void __launch_bounds__(256) k_commit_a(Params p) {
  __shared__ uint64_t s_red[8];
  __shared__ uint32_t s_zp;
  DevState* st = p.st;
  if (round_skipped(p, st) || !st->slot_open) return;
  const uint32_t T = p.n_inj_tickets + p.n_ep;
  const uint32_t row = (uint32_t)st->round & p.hist_mask;
  const uint32_t tag = ((uint32_t)st->round & 0x7FFFu) + 1u;
  uint32_t* em = p.rt_em + (size_t)row * p.t_max;
  uint32_t* ev = p.rt_ev + (size_t)row * p.t_max;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_zp = 0;
  __syncthreads();
  uint64_t sum = 0;
  uint32_t zp = 0;
  uint64_t v[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint32_t i = blockIdx.x * kCommitBlk + q * 256 + tid;
    v[q] = i < T ? __ldcg(reinterpret_cast<const unsigned long long*>(p.rt_cnt_sh[owner_of_ticket(i, p.n_inj_tickets, p.n_servers, p.n_shards)] + (size_t)row * p.t_max + i)) : ((uint64_t)tag << 48);
  }
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint32_t i = blockIdx.x * kCommitBlk + q * 256 + tid;
    if (i >= T) continue;
    for (uint32_t spin = 0; (uint32_t)(v[q] >> 48) != tag && spin < (1u << 22); spin++)
      v[q] = __ldcg(reinterpret_cast<const unsigned long long*>(p.rt_cnt_sh[owner_of_ticket(i, p.n_inj_tickets, p.n_servers, p.n_shards)] + (size_t)row * p.t_max + i));
    if ((uint32_t)(v[q] >> 48) != tag) latch_error(st, E_HISTORY, i);
    zp |= (uint32_t)(v[q] >> 47) & 1u;
    const uint32_t ve = (uint32_t)(v[q] >> 24) & 0x7FFFFFu, vm = (uint32_t)v[q] & 0xFFFFFFu;
    ev[i] = ve; em[i] = vm;
    sum += ((uint64_t)ve << 32) | vm;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(FULL, sum, d);
  if (lane == 0) s_red[warp] = sum;
  if (zp) s_zp = 1;
  __syncthreads();
  if (tid == 0) {
    uint64_t t = 0;
    for (int w = 0; w < 8; w++) t += s_red[w];
    p.cm_blk[blockIdx.x] = t;
    if (s_zp) atomicOr(&p.cm_flags[0], 1u);
  }
}

__global__ void __launch_bounds__(512) k_commit_b(Params p, uint32_t nb) {
  __shared__ uint64_t s_wtmp[34];
  DevState* st = p.st;
  if (round_skipped(p, st) || !st->slot_open) {
    if (threadIdx.x == 0) p.cm_flags[2] = 0;
    return;
  }
  // exclusive scan of the block sums in place (block_excl_scan wants shared memory: do it by hand)
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int c = ((int)nb + nt - 1) / nt;
  const int lo = min(tid * c, (int)nb), hi = min(lo + c, (int)nb);
  uint64_t sum = 0;
  for (int i = lo; i < hi; i++) sum += p.cm_blk[i];
  uint64_t incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_wtmp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int nw = nt >> 5;
    const uint64_t w = lane < nw ? s_wtmp[lane] : 0;
    uint64_t wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint64_t y = __shfl_up_sync(FULL, wi, d);
      if (lane >= d) wi += y;
    }
    s_wtmp[lane] = wi - w;
    if (lane == 31) s_wtmp[32] = wi;
  }
  __syncthreads();
  uint64_t run = s_wtmp[warp] + incl - sum;
  for (int i = lo; i < hi; i++) {
    const uint64_t v = p.cm_blk[i];
    p.cm_blk[i] = run;
    run += v;
  }
  const uint64_t total = s_wtmp[32];
  __syncthreads();
  if (tid == 0) {
    const uint32_t T = p.n_inj_tickets + p.n_ep;
    p.cm_flags[1] = (uint32_t)st->round & p.hist_mask;      // phase C works on the row of the round being committed
    p.cm_flags[2] = 1;
    const uint32_t zp_any = p.cm_flags[0];
    p.cm_flags[0] = 0;
    commit_scalars(p, st, total, zp_any, T);
  }
}

__global__ void __launch_bounds__(256) k_commit_c(Params p) {
  __shared__ uint64_t s_w[9];
  if (!p.cm_flags[2]) return;
  const uint32_t T = p.n_inj_tickets + p.n_ep;
  const uint32_t row = p.cm_flags[1];
  uint32_t* em = p.rt_em + (size_t)row * p.t_max;
  uint32_t* ev = p.rt_ev + (size_t)row * p.t_max;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // thread t owns the 4 consecutive tickets base + 4t .. base + 4t + 3
  const uint32_t i0 = blockIdx.x * kCommitBlk + 4 * tid;
  uint64_t c[4], sum = 0;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint32_t i = i0 + q;
    c[q] = i < T ? (((uint64_t)ev[i] << 32) | em[i]) : 0ull;
    sum += c[q];
  }
  uint64_t incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (tid == 0) {
    uint64_t r = p.cm_blk[blockIdx.x];
    for (int w = 0; w < 8; w++) { const uint64_t v = s_w[w]; s_w[w] = r; r += v; }
  }
  __syncthreads();
  uint64_t run = s_w[warp] + incl - sum;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const uint32_t i = i0 + q;
    if (i < T) { ev[i] = (uint32_t)(run >> 32); em[i] = (uint32_t)run; }
    run += c[q];
  }
}

// ------------------------------------------------------------------ k_round
// Persistent CTAs; one ticket at a time: tickets [0, n_inj_tickets) are injector
// slices, ticket n_inj_tickets + e is endpoint e.  Dynamic shared memory, `cap` =
// window capacity of this size class (25 B / message):
//   reg1 u64[cap+1]  order keys (round << 24 | ticket)  ->  packed count scan
//   keyB u32[cap]    emission index of the key
//   vals u32[cap]    value | V_* flags        tab u16[2*cap]  first-sight table
//   meta u16[cap]    compact message class
//   ord  u16[cap]    sorted position -> window slot      blk u8[cap]  sorted position -> sender block
constexpr uint32_t M_SRCSLOT = 0xFu;      // meta bits 0-3: neighbor slot of src + 1, 15 = neighbor (slot unknown), 0 = none
constexpr uint32_t M_HAS_ID = 1u << 4;
constexpr uint32_t M_REPLY = 1u << 5;
constexpr uint32_t M_TC_SHIFT = 6;        // bits 6-8: type class
enum : uint32_t { TC_OTHER = 0, TC_INIT = 1, TC_TOPOLOGY = 2, TC_READ = 3, TC_BROADCAST = 4, TC_ECHO = 5 };

// emissions of one delivered message from its compact class (count phase, no global access)
__device__ __forceinline__ uint32_t emit_count_meta(uint32_t workload, uint32_t meta, bool is_new, uint32_t deg) {
  const uint32_t tc = (meta >> M_TC_SHIFT) & 7u;
  if (workload == MS_W_ECHO) return (tc == TC_INIT || tc == TC_ECHO) ? 1u : 0u;        // echo.rb:28-39
  if (meta & M_REPLY) return 0;                                                          // node.rb:159-164
  if (tc == TC_INIT || tc == TC_TOPOLOGY || tc == TC_READ) return 1;
  const uint32_t has_id = (meta & M_HAS_ID) ? 1u : 0u;
  if (tc == TC_BROADCAST) return has_id + (is_new ? deg - ((meta & M_SRCSLOT) ? 1u : 0u) : 0u);
  return has_id;                                                                         // error 10
}

// exclusive prefix of one u32 per thread over the CTA; total returned through *total
__device__ __forceinline__ uint32_t block_excl_scan_u32(uint32_t v, uint32_t* total, uint32_t* wcnt /* >= 17 */) {
  const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) wcnt[warp] = incl;
  __syncthreads();
  uint32_t before = 0, tot = 0;
  for (int w = 0; w < (nt >> 5); w++) {
    const uint32_t cw = wcnt[w];
    if (w < warp) before += cw;
    tot += cw;
  }
  __syncthreads();
  *total = tot;
  return before + incl - v;
}

// same for one u64 per thread (packed 4 x 16-bit counters)
__device__ __forceinline__ uint64_t block_excl_scan_u64v(uint64_t v, uint64_t* total, uint64_t* wtmp /* >= 17 */) {
  const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint64_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint64_t y = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) wtmp[warp] = incl;
  __syncthreads();
  uint64_t before = 0, tot = 0;
  for (int w = 0; w < (nt >> 5); w++) {
    const uint64_t cw = wtmp[w];
    if (w < warp) before += cw;
    tot += cw;
  }
  __syncthreads();
  *total = tot;
  return before + incl - v;
}

// g-set node program (demo/ruby/g_set.rb:13-39): message classes in meta bits 6-8
enum : uint32_t { GT_OTHER = 0, GT_INIT = 1, GT_ADD = 2, GT_READ = 3, GT_REPL_ONE = 4, GT_REPL_FULL = 5 };

__device__ __forceinline__ uint32_t gset_emit_count(uint32_t meta) {
  if (meta & M_REPLY) return 0;                                                          // node.rb:159-164
  const uint32_t tc = (meta >> M_TC_SHIFT) & 7u;
  if (tc == GT_INIT || tc == GT_ADD || tc == GT_READ) return 1;                          // g_set.rb:13-21
  if (tc == GT_REPL_ONE || tc == GT_REPL_FULL) return 0;                                 // g_set.rb:24-31: no reply
  return (meta & M_HAS_ID) ? 1u : 0u;                                                    // error 10
}

// sum of one u32 per thread over the CTA
__device__ __forceinline__ uint32_t block_sum_u32(uint32_t v, uint32_t* wcnt /* >= 17 */) {
  uint32_t total;
  (void)block_excl_scan_u32(v, &total, wcnt);
  return total;
}

// ------------------------------------------------------------------ services (service.clj)
struct SvReq {
  uint32_t type, flags, key, src;
  uint64_t p1;
};
struct SvRep {
  bool reply;          // false: no clause of the service's `case` matches -> exception, logged, no reply (service.clj:262-263)
  uint32_t otype, code, value;
};
// service reply kept in vals[] between the sequential pass and the emit phase
constexpr uint32_t SV_REPLY = 1u << 24;   // bits 0-15 reply type, 16-23 error code

// PersistentKV/handle (service.clj:31-58) on one key's binding; lww = LWWKV/handle (service.clj:66-95),
// whose cas has no create_if_not_exists branch
__device__ __forceinline__ void kv_eval(bool present, uint32_t cur, const SvReq& q, bool lww, SvRep& r,
                                        bool& n_present, uint32_t& n_val) {
  r.reply = false; r.otype = MS_T_ERROR; r.code = 0; r.value = 0;
  n_present = present; n_val = cur;
  if (q.type == MS_T_READ) {
    r.reply = true;
    if (present) { r.otype = MS_T_READ_OK; r.value = cur; } else r.code = 20;
  } else if (q.type == MS_T_WRITE) {
    r.reply = true; r.otype = MS_T_WRITE_OK;
    n_present = true; n_val = (uint32_t)q.p1;
  } else if (q.type == MS_T_CAS) {
    const uint32_t from = (uint32_t)q.p1, to = (uint32_t)(q.p1 >> 32);
    r.reply = true;
    if (present) {
      if (cur == from) { n_val = to; r.otype = MS_T_CAS_OK; } else r.code = 22;
    } else if (!lww && (q.flags & MS_F_CREATE)) {
      n_present = true; n_val = to; r.otype = MS_T_CAS_OK;
    } else r.code = 20;
  }
}

// seq-kv: the binding of `key` in state `index` = newest version written at or before it
__device__ __forceinline__ bool seq_lookup(const Params& p, uint32_t key, uint32_t index, uint32_t& v) {
  const uint32_t cnt = p.sv_seq_vcnt[key];
  const uint32_t m = cnt < kSeqHist ? cnt : kSeqHist;
  for (uint32_t j = 1; j <= m; j++) {
    const size_t sl = (size_t)key * kSeqHist + (cnt - j) % kSeqHist;
    if (p.sv_seq_vidx[sl] <= index) { v = p.sv_seq_vval[sl]; return p.sv_seq_vhas[sl] != 0; }
  }
  v = 0;
  return false;
}

// One request against service `svc` (MS_SVC_*), executed by one thread: requests of a service are
// handled one at a time (an atom, service.clj:147-156).  rnd = the draw behind rand-int.
__device__ void service_handle(const Params& p, uint32_t svc, const SvReq& q, uint32_t rnd, SvRep& r) {
  bool np_; uint32_t nv;
  if (svc == MS_SVC_LIN_TSO) {                                       // service.clj:123-129
    r.reply = q.type == MS_T_TS; r.otype = MS_T_TS_OK; r.code = 0; r.value = 0;
    if (r.reply) r.value = (uint32_t)(p.sv_scalars[0]++);
    return;
  }
  if (svc == MS_SVC_LIN_KV) {
    kv_eval(p.sv_lin_has[q.key] != 0, p.sv_lin_val[q.key], q, false, r, np_, nv);
    if (r.reply) { p.sv_lin_has[q.key] = np_ ? 1 : 0; p.sv_lin_val[q.key] = nv; }
    return;
  }
  if (svc == MS_SVC_LWW_KV) {                                        // replica (rand-int 2), never merged
    const size_t o = (size_t)(rnd >> 31) * p.sv_n_keys + q.key;
    kv_eval(p.sv_lww_has[o] != 0, p.sv_lww_val[o], q, true, r, np_, nv);
    if (r.reply) { p.sv_lww_has[o] = np_ ? 1 : 0; p.sv_lww_val[o] = nv; }
    return;
  }
  // Sequential (service.clj:168-214)
  const uint32_t last = (uint32_t)p.sv_scalars[1];
  const uint32_t ci = p.sv_seq_cli[q.src];
  uint32_t index = ci + (uint32_t)(((uint64_t)rnd * (uint64_t)(last - ci + 1u)) >> 32);
  const uint32_t resident = last + 1u < kSeqBuffer ? last + 1u : kSeqBuffer;
  const uint32_t oldest = last + 1u - resident;
  if (index < oldest) index = oldest;                                // states older than the ring buffer are gone
  uint32_t cur;
  const bool present = seq_lookup(p, q.key, index, cur);
  kv_eval(present, cur, q, false, r, np_, nv);
  if (!r.reply) return;
  if (np_ == present && (!np_ || nv == cur)) {                       // state unchanged: stay on that timeline point
    p.sv_seq_cli[q.src] = index;
    return;
  }
  uint32_t lcur;
  const bool lpresent = seq_lookup(p, q.key, last, lcur);            // redo on the newest state, append the result
  kv_eval(lpresent, lcur, q, false, r, np_, nv);
  const uint32_t li = last + 1u;
  p.sv_scalars[1] = li;
  p.sv_seq_cli[q.src] = li;
  if (np_ != lpresent || (np_ && nv != lcur)) {
    const uint32_t cnt = p.sv_seq_vcnt[q.key];
    const size_t sl = (size_t)q.key * kSeqHist + cnt % kSeqHist;
    p.sv_seq_vidx[sl] = li; p.sv_seq_vval[sl] = nv; p.sv_seq_vhas[sl] = np_ ? 1 : 0;
    p.sv_seq_vcnt[q.key] = cnt + 1u;
  }
}


// WL = node-program families compiled in: bit 0 g-set, bit 2 Raft (else echo / broadcast), bit 1 services.
// CTA width per window-size class (ms_engine.cu: 64 / 128 / 256 / 512 threads; the g-set family runs
// 256 wide) and the register budget that goes with it
#ifndef MS_ROUND_MINB2
#define MS_ROUND_MINB2 4
#endif
// Default shape of window-size class CLS (ms_engine.cu build_sim: ladder / thr_default).  The FIX instantiations
// assume it, which turns every shared-memory array base and every loop stride into an immediate; a simulation
// sized differently (max_window below the ladder, threads_per_node) runs the generic ones.
template <int CLS> struct ClsShape {
  static constexpr uint32_t cap = kClsLadder[CLS < 3 ? CLS : 2];
  static constexpr int nt = kClsThreads[CLS];
};

template <int CLS, int WL, bool FIX = false>
__global__ void __launch_bounds__(CLS == 3 ? 512 : 256, CLS == 3 ? 2 : MS_ROUND_MINB2) k_round(Params p, uint32_t cap_arg) {
  constexpr uint32_t cls = CLS;
  static_assert(!FIX || CLS < 3, "class 3 is sized by max_window");
  const uint32_t cap = FIX ? ClsShape<CLS>::cap : cap_arg;
  constexpr bool GS = (WL & 1) != 0;
  constexpr bool SV = (WL & 2) != 0;
  constexpr bool RF = (WL & 4) != 0;
  DevState* st = p.st;

#ifdef MS_EMUL
  unsigned char* smem_raw = simt::dyn_smem();
#else
  extern __shared__ __align__(16) unsigned char smem_raw[];
#endif
  uint64_t* reg1 = reinterpret_cast<uint64_t*>(smem_raw);          // cap+1 entries
  uint32_t* keyB = reinterpret_cast<uint32_t*>(reg1 + cap + 1);
  uint32_t* vals = keyB + cap;
  uint16_t* tab = reinterpret_cast<uint16_t*>(vals + cap);         // first-sight table, 2*cap entries
  uint16_t* meta = tab + 2 * (size_t)cap;
  uint16_t* ord = meta + cap;
  uint8_t* blk = reinterpret_cast<uint8_t*>(ord + cap);
  uint64_t* keyA = reg1;
  uint64_t* aux = reg1;                                            // packed counts (keyA is dead by then)

  __shared__ uint64_t s_wtmp[34];
  __shared__ NetParams s_np;
  __shared__ uint32_t s_wcnt[17];
  __shared__ uint32_t s_misc[8];       // 0: mail base, 1: use_blocks, 3: inj-server-src flag, 4: is_last, 5: next list index
  __shared__ uint32_t s_cnt[8];        // per-ticket counters
  __shared__ uint64_t s_chunk;
  // sender blocks of the window (fast ordering path)
  __shared__ uint16_t s_bstart[MAXB + 1];     // window offset of block r (arrival order)
  __shared__ uint16_t s_brank[MAXB];          // sorted rank of block r
  __shared__ uint16_t s_boff[MAXB + 1];       // sorted: first sorted position of block rho
  __shared__ uint64_t s_bkeyA[MAXB];          // sorted: (round << 24 | ticket)
  __shared__ uint64_t s_bbase[MAXB];          // sorted: dense id of the block's idx 0
  __shared__ uint16_t s_S[MAXB + 1][MAXNB];   // sorted: new messages from neighbor j in blocks < rho
  __shared__ uint32_t s_nbbase[MAXNB];        // ring position claimed for this CTA's gossip to neighbor j
  __shared__ uint32_t s_nbr[MAXNB];           // this node's neighbor list (topology order)
  __shared__ uint4 s_gen[2];                  // the request a closed-loop client sends in this step
  __shared__ uint64_t s_round0;               // the round this CTA works on (0: none, see below)
  __shared__ int64_t s_now0;
  __shared__ uint32_t s_go;

  const int tid = threadIdx.x, nt = FIX ? ClsShape<CLS>::nt : (int)blockDim.x, lane = tid & 31;
  if (tid == 0) {
    s_np = *p.np;
    // Is this launch's round still open?  Decided once per CTA, by one thread: a CTA of a persistent grid may
    // start late (its class queues behind the others for SM resources), even while the last ticket of the round
    // is committing it.  The commit stores round + 1 and then clears slot_open; reading slot_open first and
    // the round second, a CTA either sees the open round's tag with its own round, or leaves: it can never take
    // a ticket cursor of the NEXT round's parity, and its threads never disagree about leaving.
    const uint32_t so = ld_volatile_u32(&st->slot_open);
    __threadfence();
    const uint64_t r = *reinterpret_cast<const volatile uint64_t*>(&st->round);
    s_round0 = r;
    s_now0 = *reinterpret_cast<const volatile int64_t*>(&st->now);
    s_go = (so == slot_tag(r) && !round_skipped(p, st)) ? 1u : 0u;
  }
  __syncthreads();
  if (!s_go) return;
  const NetParams np = s_np;
  const int64_t now = s_now0;
  const uint64_t round = s_round0;
  const uint32_t T = p.n_inj_tickets + p.n_ep;
  const uint32_t row = (uint32_t)round & p.hist_mask;
  const uint32_t par = (uint32_t)round & 1u;
  const uint32_t my_big = st->cls_count[par][cls];                  // final: k_snapshot has completed
  const uint32_t my_count = my_big + st->cls_small[par][cls];
  const uint32_t* my_list = p.cls_list + ((size_t)par * 4 + cls) * p.t_max;
  const uint32_t tag = ((uint32_t)round & 0x7FFFu) + 1u;            // validates this round's table entries
  // with no loss and a constant latency nothing depends on the random draw: skip Philox
  const bool need_rng = np.loss_thresh != 0 || np.dist != MS_DIST_CONSTANT;
  const uint64_t const_lat = (uint64_t)np.mean_ms * np.scale;
  // optional per-phase cycle accounting (diagnostic, ms_debug_phase_cycles): only in builds with -DMS_PHASE_TIMING
  // (__graft_entry__.build_variant("timing", ["MS_PHASE_TIMING"])); the product library carries none of it
#ifdef MS_PHASE_TIMING
  const bool timing = p.phase_cycles != nullptr;
#else
  constexpr bool timing = false;
#endif
  long long t_prev = timing ? clock64() : 0;
#define PHASE_MARK(k)                                                                         \
  do {                                                                                        \
    if (timing && tid == 0) {                                                                 \
      const long long t_now = clock64();                                                      \
      atomicAdd((unsigned long long*)&p.phase_cycles[cls * 16 + (k)], (unsigned long long)(t_now - t_prev)); \
      t_prev = t_now;                                                                         \
    }                                                                                         \
  } while (0)
  if (tid == 0) s_misc[5] = atomicAdd(&st->cls_cursor[par][cls], 1u);

 // persistent CTA: take tickets of this size class until the list is exhausted
 for (;;) {
  __syncthreads();                     // the previous ticket is completely done with shared memory
  const uint32_t li = s_misc[5];
  if (tid < 5) s_misc[tid] = 0;
  if (tid < 8) s_cnt[tid] = 0;
  __syncthreads();
  if (li >= my_count) break;
  // fetch the index of the NEXT ticket now; it is consumed at the end of this one
  uint32_t next_li = 0;
  if (tid == 0) next_li = atomicAdd(&st->cls_cursor[par][cls], 1u);
  const uint32_t ticket = li < my_big ? my_list[li] : my_list[p.t_max - 1u - (li - my_big)];
  PHASE_MARK(0);
  if (timing && tid == 0) atomicAdd((unsigned long long*)&p.phase_cycles[cls * 16 + 15], 1ull);

  EmitCtx cx;
  cx.now = now;
  cx.round = round;
  cx.ticket = ticket;
  cx.idx_bias = 0;
  cx.chunk = 0;
  cx.n_recv = 0;
  cx.emitter = 0;
  cx.need_rng = need_rng;
  cx.const_lat = const_lat;
  cx.c_send_cl = cx.c_send_sv = cx.c_lost = cx.c_zero = 0;
  uint32_t c_recv_cl = 0, c_recv_sv = 0, c_part = 0, c_replies = 0;
  uint32_t n_ev_local = 0, n_em_local = 0;

  if (ticket < p.n_inj_tickets) {
    // ---------------------------------------------------------- injector slice
    // host sends staged by ms_send (call order), then scheduled ops whose time
    // has come (schedule order): DESIGN.md 2.3 step 1.
    const uint32_t n_host = st->inj_count;
    const uint64_t tick = (uint64_t)(now / kTickNs);
    const uint32_t cur = st->sched_cursor;
    uint32_t hi = (tick + 1 < p.n_tick_off) ? p.tick_off[tick + 1] : p.n_sched;
    if (hi < cur) hi = cur;
    const uint32_t K = n_host + (hi - cur);
    const uint32_t chunk = (K + p.n_inj_tickets - 1) / p.n_inj_tickets;
    const uint32_t lo = min(ticket * chunk, K), hi_s = min(lo + chunk, K);
    const uint32_t n_local = hi_s - lo;
    n_ev_local = n_local; n_em_local = n_local;
    if (tid == 0) {
      s_chunk = (n_local && p.jlevel)
                    ? atomicAdd((unsigned long long*)&st->jraw_cursor, (unsigned long long)n_local) : 0ull;
      if (n_local && p.jlevel && !p.jdiscard && s_chunk + n_local - st->jraw_drained > p.jmask + 1)
        latch_error(st, E_JOURNAL_OVERFLOW, ticket);
    }
    __syncthreads();
    cx.chunk = s_chunk;
    cx.emitter = kInjector;
    cx.idx_bias = lo;
    for (uint32_t base = 0; base < n_local; base += nt) {
      const uint32_t j = base + tid;
      const bool valid = j < n_local;
      Rec r;
      r.dest = 0; r.src = 0;
      if (valid) {
        const uint32_t g = lo + j;
        if (g < n_host) {
          const ms_msg m = p.inj_buf[g];
          r.src = m.src; r.dest = m.dest; r.msg_id = m.msg_id; r.in_reply_to = m.in_reply_to;
          r.tf = (uint32_t)m.type | ((uint32_t)m.flags << 16); r.p0 = m.p0; r.p1 = m.p1;
        } else {
          const ms_op op = p.sched[cur + (g - n_host)];
          r.src = op.src; r.dest = op.dest; r.msg_id = op.body.msg_id; r.in_reply_to = op.body.in_reply_to;
          r.tf = (uint32_t)op.body.type | ((uint32_t)op.body.flags << 16); r.p0 = op.body.p0; r.p1 = op.body.p1;
        }
      }
      emit_one(p, st, np, cx, valid, r, j, 0, false);
    }
  } else {
    // ---------------------------------------------------------- endpoint CTA
    const uint32_t e = ticket - p.n_inj_tickets;
    const uint8_t kind = p.kind[e];
    const uint32_t head = p.head[e];
    uint32_t n = ((kind & kRemoved)) ? 0u : (p.limit[e] - head);
    if (n > cap || n > (e < p.n_servers ? p.max_window_s : p.max_window)) {
      if (tid == 0) latch_error(st, E_WINDOW_OVERFLOW, e);
      n = 0;
    }
    const size_t my0 = ring_base(p, e);   // slot (head + i) & my_mask of the window is ring slot my0 + that
    const uint32_t my_mask = ring_cap_of(p, e) - 1u;
    const bool is_server = (kind == MS_KIND_SERVER);
    const bool bcast = !GS && is_server && p.workload == MS_W_BROADCAST;
    // g-set periodic task (g_set.rb:34-39), evaluated before the node's receives: when due, the
    // node snapshots its set and sends it to every other node (emissions 0 .. n_servers-2)
    uint32_t n_timer = 0, fire_seq = 0, fire_p0 = 0;
    if constexpr (GS) {
      if (is_server && p.gs_init[e] && now >= p.gs_next_fire[e]) {
        n_timer = p.n_servers - 1;
        fire_seq = p.gs_fires[e] + 1;
      }
    }
    const uint32_t* mybits = (is_server && p.bitmap) ? p.bitmap + (size_t)e * p.bm_words : nullptr;
    const uint32_t deg = bcast ? nbr_count(p, e) : 0;
    const bool nb_smem = bcast && p.topology != MS_TOPO_TOTAL && deg <= MAXNB;
    if (nb_smem && tid < (int)deg) s_nbr[tid] = p.nbr[p.nbr_off[e] + tid];
    __syncthreads();

    // PA1: one pass over the window in arrival order, loads 2 records deep: order keys,
    //      partition check at dequeue (net.clj:234), compact message class.  A broadcast server's
    //      window is nearly all compact gossip: it loads the keys first and a body only for a key
    //      without kCompact.  Other endpoints never receive compact records: key and body together.
    {
      uint32_t err_val = 0xFFFFFFFFu;
      uint32_t snap_gone = 0xFFFFFFFFu;
      bool inj_srv = false;
      // the node's (few) neighbors in registers: the source's slot is four compares, no shared-memory loop
      const bool nb4 = nb_smem && deg <= 4;
      const uint32_t nr0 = (nb4 && deg > 0) ? s_nbr[0] : 0xFFFFFFFFu, nr1 = (nb4 && deg > 1) ? s_nbr[1] : 0xFFFFFFFFu;
      const uint32_t nr2 = (nb4 && deg > 2) ? s_nbr[2] : 0xFFFFFFFFu, nr3 = (nb4 && deg > 3) ? s_nbr[3] : 0xFFFFFFFFu;
      const uint4* body = p.ring + p.ring_slots;
      // with a latency or loss nearly every record is full (compact gossip needs both to be zero): load
      // key and body together then, too, and still expand any compact key that is in the window
      const bool keys_first = bcast && !need_rng && const_lat == 0;
      for (int base = 0; base < (int)n; base += 2 * nt) {
        uint4 a[2];
        uint32_t q_src[2], q_tf[2], q_v[2], q_run[2];
#pragma unroll
        for (int q = 0; q < 2; q++) {
          const int i = base + q * nt + tid;
          if (i < (int)n) {
            const size_t g = my0 + ((head + i) & my_mask);
            a[q] = p.ring[g];
            if (!keys_first) {
              const uint4 b = body[2 * g], c = body[2 * g + 1];
              q_src[q] = b.x; q_tf[q] = c.x; q_v[q] = c.y; q_run[q] = c.z;
            }
          }
        }
        if (bcast) {
#pragma unroll
          for (int q = 0; q < 2; q++) {
            const int i = base + q * nt + tid;
            if (i >= (int)n) continue;
            if (a[q].y & kCompact) {
              q_src[q] = (a[q].y & 0xFFFFFFu) - p.n_inj_tickets; q_tf[q] = MS_T_BROADCAST; q_v[q] = a[q].w; q_run[q] = 0;
            } else if (keys_first) {
              const size_t g = my0 + ((head + i) & my_mask);
              const uint4 b = body[2 * g], c = body[2 * g + 1];
              q_src[q] = b.x; q_tf[q] = c.x; q_v[q] = c.y; q_run[q] = c.z;
            }
          }
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
          const int i = base + q * nt + tid;
          if (i >= (int)n) continue;
          const uint32_t tk = a[q].y & 0xFFFFFFu;
          const uint64_t rnd = (a[q].y & kCompact) ? compact_round(round, a[q].z) : ((uint64_t)a[q].z | ((uint64_t)a[q].w << 32));
          keyA[i] = (rnd << 24) | (uint64_t)tk;
          keyB[i] = a[q].x;
          const uint32_t src = q_src[q], tf = q_tf[q], v = q_v[q];
          if (tk < p.n_inj_tickets && src < p.n_servers) inj_srv = true;   // injected on behalf of a server
          bool cut = false;
          if (np.pair_active && p.pair_bits)
            cut = (p.pair_bits[(size_t)e * p.pair_words + (src >> 5)] >> (src & 31)) & 1u;
          if (!cut && np.comp_active) {
            // bulk partition: endpoints in different components are cut; 0xFFFFFFFF = not listed (never cut)
            const uint32_t cs = p.comp[src], ce = p.comp[e];
            cut = cs != ce && cs != 0xFFFFFFFFu && ce != 0xFFFFFFFFu;
          }
          const uint32_t type = tf & 0xFFFFu;
          const uint32_t fl = tf >> 16;
          uint32_t tc = TC_OTHER;
          if constexpr (GS) {
            if (type == MS_T_INIT) tc = GT_INIT;
            else if (type == MS_T_ADD) tc = GT_ADD;
            else if (type == MS_T_READ) tc = GT_READ;
            else if (type == MS_T_REPLICATE_ONE) tc = GT_REPL_ONE;
            else if (type == MS_T_REPLICATE_FULL) tc = GT_REPL_FULL;
          } else {
          if (type == MS_T_INIT) tc = TC_INIT;
          else if (type == MS_T_TOPOLOGY) tc = TC_TOPOLOGY;
          else if (type == MS_T_READ) tc = TC_READ;
          else if (type == MS_T_BROADCAST) tc = TC_BROADCAST;
          else if (type == MS_T_ECHO) tc = TC_ECHO;
          }
          uint32_t slot = 0;
          if (nb4) {
            slot = src == nr3 ? 4u : src == nr2 ? 3u : src == nr1 ? 2u : src == nr0 ? 1u : 0u;
          } else if (nb_smem) {
            for (uint32_t j = 0; j < deg; j++) if (s_nbr[j] == src) slot = j + 1;
          } else if (bcast && src < p.n_servers && src != e) {
            slot = 15;
          }
          meta[i] = (uint16_t)(slot | ((fl & MS_F_MSG_ID) ? M_HAS_ID : 0u) | ((fl & MS_F_REPLY) ? M_REPLY : 0u) |
                               (tc << M_TC_SHIFT));
          uint32_t val = cut ? 0u : V_RECV;
          if (bcast && !cut && tc == TC_BROADCAST && !(fl & MS_F_REPLY)) {
            if (v >= p.n_values || v > V_MASK) err_val = v;
            else val |= v | V_CAND;
          }
          if constexpr (GS) {
            if (is_server && !cut && !(fl & MS_F_REPLY)) {
              if (tc == GT_ADD || tc == GT_REPL_ONE) {           // the element (g_set.rb:17-26)
                if (v >= p.n_values || v > V_MASK) err_val = v;
                else val |= v;
              } else if (tc == GT_REPL_FULL) {                   // the snapshot row of (src, run p1)
                const uint32_t run = q_run[q];
                const uint32_t rowi = src * p.gs_slots + (run & (p.gs_slots - 1));
                if (src >= p.n_servers ||
                    __ldcg(p.gs_tag_sh[owner_of(src, p.n_servers, p.n_shards)] + rowi) != run) snap_gone = src;
                else val |= rowi;
              }
            }
          }
          vals[i] = val;
        }
      }
      if (err_val != 0xFFFFFFFFu) latch_error(st, E_VALUE_RANGE, err_val);
      if (snap_gone != 0xFFFFFFFFu) latch_error(st, E_SNAPSHOT, snap_gone);
      if (inj_srv) s_misc[3] = 1;
    }
    // PA2: seen-set test of the broadcast values (own slots only: no barrier needed in between)
    if (bcast) {
      for (int base = 0; base < (int)n; base += 4 * nt) {
        uint32_t w[4], vv[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int i = base + q * nt + tid;
          vv[q] = i < (int)n ? vals[i] : 0u;
          w[q] = (vv[q] & V_CAND) ? mybits[(vv[q] & V_MASK) >> 5] : 0xFFFFFFFFu;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int i = base + q * nt + tid;
          if (i < (int)n && (vv[q] & V_CAND) && !((w[q] >> (vv[q] & 31)) & 1u)) vals[i] = vv[q] | V_FRESH;
        }
      }
    }
    __syncthreads();
    PHASE_MARK(1);
    // this CTA's NEXT ticket: pull its window from HBM into L2 now, behind this ticket's remaining phases
    // (windows are frozen by k_snapshot, so head / limit are final; a window is contiguous up to the ring's wrap)
    if (tid == 0 && next_li < my_count) {
      const uint32_t t2 = next_li < my_big ? my_list[next_li] : my_list[p.t_max - 1u - (next_li - my_big)];
      if (t2 >= p.n_inj_tickets) {
        const uint32_t e2 = t2 - p.n_inj_tickets;
        const uint32_t h2 = p.head[e2], n2 = p.limit[e2] - h2, cap2 = ring_cap_of(p, e2);
        if (n2 > 0 && n2 <= cap2) {
          // keys always; bodies unless e2 is a broadcast server that loads its keys first (PA1)
          const size_t g2 = ring_base(p, e2);
          const uint32_t o2 = h2 & (cap2 - 1u), first = min(n2, cap2 - o2);
          prefetch_l2_bulk(p.ring + g2 + o2, first * 16u);
          if (n2 > first) prefetch_l2_bulk(p.ring + g2, (n2 - first) * 16u);
          if (GS || need_rng || const_lat != 0 || p.workload != MS_W_BROADCAST || p.kind[e2] != MS_KIND_SERVER) {
            const uint4* body2 = p.ring + p.ring_slots + 2 * g2;
            prefetch_l2_bulk(body2 + 2 * (size_t)o2, first * 32u);
            if (n2 > first) prefetch_l2_bulk(body2, (n2 - first) * 32u);
          }
        }
      }
    }

    // PB: order the due set by (round, ticket, idx) == message id order (all due
    //     deadlines equal `now`; the reference's PriorityBlockingQueue leaves ties
    //     unspecified, net.clj:39-40,145).  Senders claim ring space in blocks, so
    //     the window is a handful of internally ordered blocks: find them, sort
    //     the blocks, verify; anything else falls back to a bitonic sort.
    uint32_t R = 0;
    bool use_blocks = false;
    if (n > 0) {
      // block starts: each thread scans one contiguous segment of the window
      const int c = ((int)n + nt - 1) / nt;
      const int lo = min(tid * c, (int)n), hi = min(lo + c, (int)n);
      uint32_t nf = 0;
      uint32_t fmask = 0;                       // block starts of this thread's segment (when it has <= 32 slots)
      const bool use_mask = c <= 32;
      if (lo < hi) {
        uint64_t pa = lo ? keyA[lo - 1] : 0ull;
        uint32_t pb = lo ? keyB[lo - 1] : 0u;
        for (int i = lo; i < hi; i++) {
          const uint64_t ka = keyA[i];
          const uint32_t kb = keyB[i];
          if (i == 0 || ka != pa || kb <= pb) { nf++; fmask |= 1u << ((i - lo) & 31); }
          pa = ka; pb = kb;
        }
      }
      uint32_t off = block_excl_scan_u32(nf, &R, s_wcnt);
      if (R <= MAXB) {
        if (use_mask) {
          while (fmask) { s_bstart[off++] = (uint16_t)(lo + __ffs(fmask) - 1); fmask &= fmask - 1u; }
        } else {
          for (int i = lo; i < hi; i++)
            if (i == 0 || keyA[i] != keyA[i - 1] || keyB[i] <= keyB[i - 1]) s_bstart[off++] = (uint16_t)i;
        }
        if (tid == 0) s_bstart[R] = (uint16_t)n;
        __syncthreads();
        // rank blocks by their first key
        for (uint32_t b = tid; b < R; b += nt) {
          const uint32_t s0 = s_bstart[b];
          const uint64_t ka = keyA[s0];
          const uint32_t kb = keyB[s0];
          uint32_t rk = 0;
          for (uint32_t q = 0; q < R; q++) {
            const uint32_t sq = s_bstart[q];
            const uint64_t qa = keyA[sq];
            const uint32_t qb = keyB[sq];
            if (qa < ka || (qa == ka && (qb < kb || (qb == kb && q < b)))) rk++;
          }
          s_brank[b] = (uint16_t)rk;
          s_bkeyA[rk] = ka;
          // temporarily: length of the block, exclusive-scanned below
          s_boff[rk] = (uint16_t)(s_bstart[b + 1] - s0);
          // stash (first idx, last idx) of the block for the verification
          s_bbase[rk] = ((uint64_t)kb << 32) | keyB[s_bstart[b + 1] - 1];
        }
        __syncthreads();
        if (tid == 0) {
          uint32_t acc = 0;
          bool ok = true;
          for (uint32_t q = 0; q < R; q++) {
            const uint32_t len = s_boff[q];
            s_boff[q] = (uint16_t)acc;
            acc += len;
            if (q) {
              // previous block must end before this one begins
              const uint64_t pa = s_bkeyA[q - 1], ca = s_bkeyA[q];
              const uint32_t plast = (uint32_t)s_bbase[q - 1], cfirst = (uint32_t)(s_bbase[q] >> 32);
              if (!(pa < ca || (pa == ca && plast < cfirst))) ok = false;
            }
          }
          s_boff[R] = (uint16_t)acc;
          s_misc[1] = ok ? 1u : 0u;
          if (!ok && timing && atomicCAS((unsigned long long*)&p.phase_cycles[64], 0ull, 1ull) == 0ull) {
            // diagnostic dump of the first window whose blocks overlap
            unsigned long long* d = (unsigned long long*)p.phase_cycles + 65;
            d[0] = e; d[1] = n; d[2] = R; d[3] = round;
            for (uint32_t q = 0; q < R; q++) { d[4 + 2 * q] = s_bkeyA[q]; d[5 + 2 * q] = s_bbase[q]; }
          }
        }
        __syncthreads();
        use_blocks = s_misc[1] != 0;
      }
      if (use_blocks) {
        // sorted position of every slot of this thread's segment
        uint32_t bi = 0;
        if (lo < hi) {
          uint32_t l2 = 0, h2 = R;
          while (h2 - l2 > 1) { const uint32_t mid = (l2 + h2) >> 1; if (s_bstart[mid] <= (uint32_t)lo) l2 = mid; else h2 = mid; }
          bi = l2;
        }
        for (int i = lo; i < hi; i++) {
          while (bi + 1 < R && s_bstart[bi + 1] <= (uint32_t)i) bi++;
          const uint32_t rk = s_brank[bi];
          const uint32_t pos = s_boff[rk] + ((uint32_t)i - s_bstart[bi]);
          ord[pos] = (uint16_t)i;
          blk[pos] = (uint8_t)rk;
        }
        // dense-id base of each sender block (consumed in PE; issued early)
        for (uint32_t b = tid; b < R; b += nt) {
          const uint64_t ka = s_bkeyA[b];
          s_bbase[b] = dense_base(p, st, ka >> 24, (uint32_t)(ka & 0xFFFFFFu));
        }
      } else {
        int np2 = 1;
        while (np2 < (int)n) np2 <<= 1;
        for (int i = tid; i < np2; i += nt) ord[i] = i < (int)n ? (uint16_t)i : (uint16_t)0xFFFF;
        __syncthreads();
        if (n > 1) block_bitonic_sort_idx(ord, keyA, keyB, np2);
        if (tid == 0 && n > 1) atomicAdd((unsigned long long*)&st->fallback_sorts, 1ull);
        if (timing && tid == 0 && n > 1) atomicAdd((unsigned long long*)&p.phase_cycles[cls * 16 + (R > MAXB ? 9 : 10)], 1ull);
      }
    }
    __syncthreads();   // keyA (reg1) is dead from here on
    PHASE_MARK(2);

    // PC: first sight of a value among this round's copies: smallest sorted position wins
    int npad = 1;
    while (npad < (int)n) npad <<= 1;
    const int tsz = 2 * npad;
    const uint32_t hshift = (uint32_t)__clz(tsz) + 1u;          // 32 - log2(tsz); tsz >= 2
#define TAB_SLOT(v) (((v) * 0x9E3779B1u) >> hshift)
    if (bcast && n > 0) {
      if (tsz >= 4) {                                            // tab is 8-byte aligned (16 * cap + 8 bytes into the buffer)
        uint64_t* t8 = reinterpret_cast<uint64_t*>(tab);
        for (int i = tid; i < (tsz >> 2); i += nt) t8[i] = 0xFFFFFFFFFFFFFFFFull;
      } else {
        for (int i = tid; i < tsz; i += nt) tab[i] = 0xFFFF;
      }
      __syncthreads();
      for (int pos = tid; pos < (int)n; pos += nt) {
        const uint32_t val = vals[ord[pos]];
        if (val & V_FRESH) {
          const uint32_t v = val & V_MASK;
          uint32_t h = TAB_SLOT(v);
          for (int probe = 0; probe < tsz; probe++) {   // the table is at most half full
            uint32_t cur = *reinterpret_cast<volatile uint16_t*>(&tab[h]);
            if (cur == 0xFFFFu) {
              const uint32_t old = atomicCAS(&tab[h], (unsigned short)0xFFFF, (unsigned short)pos);
              if (old == 0xFFFFu) break;
              cur = old;
            }
            if ((vals[ord[cur]] & V_MASK) == v) {
              while ((uint32_t)pos < cur) {              // atomic min on a 16-bit slot
                const uint32_t old = atomicCAS(&tab[h], (unsigned short)cur, (unsigned short)pos);
                if (old == cur) break;
                cur = old;
              }
              break;
            }
            h = (h + 1) & (tsz - 1);
          }
        }
      }
      __syncthreads();
    }
    if constexpr (RF) {
      // ---- Raft / txn-list-append node: the step is sequential (ms_raft.cuh); its sends are staged and emitted below
      if (is_server) {
        if (tid == 0) {
          RaftCtx c{p, st, e, now, round, p.rf_node + e, p.rf_log + (size_t)e * p.rf_log_cap * 2,
                    p.rf_cb + (size_t)e * (p.rf_cb_mask + 1u) * 2, p.rf_stage + (size_t)e * p.rf_stage_cap * 3, 0u, 0u, 0u, 0u};
          rf_group_of(p, e, c.gbase, c.gn);
          for (uint32_t pos = 0; pos < n; pos++) {
            const uint32_t i = ord[pos];
            if (!(vals[i] & V_RECV)) continue;
            const Rec m = ring_load(p, p.ring, my0 + ((head + i) & my_mask), round, e);
            if (p.workload == MS_W_RAFT) rf_handle(c, m);
            else if (p.workload == MS_W_TXN_TREE) tt_handle(c, m);
            else txn_handle(c, m);
          }
          if (p.workload == MS_W_RAFT) { rf_actions(c); rf_note_busy(c); }
          if (p.workload == MS_W_TXN_TREE) tt_actions(c);
          s_misc[2] = c.n_stage;
        }
        __syncthreads();
        n_timer = s_misc[2];
      }
    }
    if (kind == MS_KIND_GEN_CLIENT) {
      // ---- closed-loop client: replies in id order, timeout, at most one new request (gen_step)
      if (tid == 0) {
        Rec q;
        const bool send = gen_step(p, st, e, now, round, my0, head, my_mask, n, ord, vals, q);
        if (send) {
          s_gen[0] = make_uint4(q.src, q.dest, q.msg_id, q.in_reply_to);
          s_gen[1] = make_uint4(q.tf, q.p0, 0u, 0u);
        }
        s_misc[2] = send ? 1u : 0u;
      }
      __syncthreads();
      n_timer = s_misc[2];
    }
    if constexpr (SV) {
      // ---- service endpoint: requests are handled one at a time in dequeue order (service.clj:147-156,
      //      245-263) by one thread; the reply is parked in vals[] / keyB[] for the emit phase
      if (kind == MS_KIND_SERVICE) {
        // the request fields the sequential walk needs, staged in sorted order by all threads (the
        // ordering keys are dead by now): p1 in reg1, the key in tab (as u32), type | flags << 8 in meta
        uint32_t* skey = reinterpret_cast<uint32_t*>(tab);
        for (uint32_t pos = tid; pos < n; pos += nt) {
          const uint32_t i = ord[pos];
          const Rec m = ring_load_body(p, p.ring, my0 + ((head + i) & my_mask));
          reg1[pos] = m.p1;
          skey[pos] = m.p0;
          const uint32_t ty = m.tf & 0xFFFFu;                       // types the device does not know (>= 256) stay unknown
          meta[i] = (uint16_t)((ty < 0xFFu ? ty : 0xFFu) | ((m.tf >> 8) & 0xFF00u));
        }
        __syncthreads();
        if (tid == 0) {
          uint32_t svc = 0;
          while (svc < 4 && p.sv_ep[svc] != e) svc++;
          uint32_t n_rep = 0;
          // lin-kv: the binding of the key last touched stays in registers (single_key_txn.clj has every
          // node hammer ONE key, the root): the walk is a dependent chain, keep memory out of it
          uint32_t ck = 0xFFFFFFFFu, cval = 0;
          bool chas = false, cdirty = false;
          for (uint32_t pos = 0; pos < n && svc < 4; pos++) {
            const uint32_t i = ord[pos];
            if (!(vals[i] & V_RECV)) continue;
            SvReq q;
            q.type = meta[i] & 0xFFu; q.flags = meta[i] >> 8; q.key = skey[pos];
            q.p1 = reg1[pos];
            q.src = 0;
            if (svc == MS_SVC_SEQ_KV)                               // per-client view (service.clj:162-166)
              q.src = ring_load_body(p, p.ring, my0 + ((head + i) & my_mask)).src;
            const bool keyed = q.type == MS_T_READ || q.type == MS_T_WRITE || q.type == MS_T_CAS;
            if (svc != MS_SVC_LIN_TSO && keyed && q.key >= p.sv_n_keys) { latch_error(st, E_VALUE_RANGE, q.key); continue; }
            if (svc != MS_SVC_LIN_TSO && !keyed) continue;   // no clause of the store's `case` matches: logged, no reply (service.clj:262-263)
            uint32_t x[4] = {0, 0, 0, 0};
            if (svc == MS_SVC_SEQ_KV || svc == MS_SVC_LWW_KV)      // rand-int = word 3 of the reply's own draw
              philox4x32_10(n_rep, e, (uint32_t)round, (uint32_t)(round >> 32), p.seed_lo, p.seed_hi, x);
            SvRep r;
            if (svc == MS_SVC_LIN_KV) {
              r.reply = false; r.otype = MS_T_ERROR; r.code = 0; r.value = 0;
              if (keyed) {
                if (q.key != ck) {
                  if (cdirty) { p.sv_lin_has[ck] = chas ? 1 : 0; p.sv_lin_val[ck] = cval; }
                  ck = q.key; chas = p.sv_lin_has[ck] != 0; cval = p.sv_lin_val[ck]; cdirty = false;
                }
                bool np_; uint32_t nv;
                kv_eval(chas, cval, q, false, r, np_, nv);
                if (r.reply) { cdirty = cdirty || np_ != chas || nv != cval; chas = np_; cval = nv; }
              }
            } else {
              service_handle(p, svc, q, x[3], r);
            }
            if (r.reply) {
              vals[i] |= SV_REPLY | (r.code << 16) | r.otype;
              keyB[pos] = r.value;
              n_rep++;
            }
          }
          if (cdirty) { p.sv_lin_has[ck] = chas ? 1 : 0; p.sv_lin_val[ck] = cval; }
        }
        __syncthreads();
      }
    }
    // resolve winners and publish packed counts in sorted order:
    //   emit (bits 0-31) | recv (32-47) | new (48-63)
    for (int pos = tid; pos < (int)n; pos += nt) {
      const uint32_t i = ord[pos];
      uint32_t val = vals[i];
      bool is_new = false;
      if (val & V_FRESH) {
        const uint32_t v = val & V_MASK;
        uint32_t h = TAB_SLOT(v);
        uint32_t win = tab[h];
        for (int probe = 0; probe < tsz && win != 0xFFFFu && (vals[ord[win]] & V_MASK) != v; probe++) {
          h = (h + 1) & (tsz - 1);   // the entry exists: probing ends on it
          win = tab[h];
        }
        if (win == (uint32_t)pos) {
          is_new = true;
          atomicOr(p.bitmap + (size_t)e * p.bm_words + (v >> 5), 1u << (v & 31));
        } else {
          vals[i] = val & ~V_FRESH;   // a lower-id copy of v is processed first this round
        }
      }
      uint64_t c = 0;
      if (val & V_RECV) {
        c = 1ull << 32;
        if constexpr (SV) {
          if (kind == MS_KIND_SERVICE && (val & SV_REPLY)) c |= 1;
        }
        if constexpr (RF) {
          // a Raft node's emissions are those staged by its sequential step
        } else if constexpr (GS) {
          if (is_server) {
            const uint32_t mt = meta[i];
            c |= gset_emit_count(mt);
            if (!(mt & M_REPLY)) {
              const uint32_t tc = (mt >> M_TC_SHIFT) & 7u;
              if (tc == GT_READ) c |= 1ull << 48;          // bits 48-63 count the reads (cut points of the merge)
              if (tc == GT_INIT) s_misc[2] = 1;            // node.rb:22-36: starts the periodic task
            }
          }
        } else {
        if (is_server) c |= emit_count_meta(p.workload, meta[i], is_new, deg);
        if (is_new) c |= 1ull << 48;
        }
      }
      aux[pos] = c;
    }
    __syncthreads();
    PHASE_MARK(3);
    const uint64_t tot = block_excl_scan(aux, (int)n, s_wtmp);
    const uint32_t n_emit_msgs = (uint32_t)tot;          // replies / gossip caused by the window
    const uint32_t n_emit = n_emit_msgs + n_timer;       // the periodic task's emissions come first
    const uint32_t n_recv = (uint32_t)(tot >> 32) & 0xFFFFu;
    const uint32_t n_new = (uint32_t)(tot >> 48);
    n_ev_local = n_recv + n_emit; n_em_local = n_emit;
    PHASE_MARK(4);

    if constexpr (GS) {
      if (is_server) {
        // ---- g-set state: snapshot for the periodic task, then the window in id order.  Unions
        //      commute, so the window is applied in segments cut at the reads; each read sees
        //      the set as of its place in the sequence (g_set.rb:13-15).
        uint32_t* myset = p.bitmap + (size_t)e * p.bm_words;
        const uint32_t n_reads = n_new;
        if (n_timer) {
          uint32_t* snap = p.gs_snap + (size_t)(e * p.gs_slots + (fire_seq & (p.gs_slots - 1))) * p.bm_words;
          uint32_t cnt = 0;
          for (uint32_t w = tid; w < p.bm_words; w += nt) {
            const uint32_t x = myset[w];
            snap[w] = x;
            cnt += __popc(x);
          }
          fire_p0 = block_sum_u32(cnt, s_wcnt);
        }
        for (uint32_t pos = tid; pos < n; pos += nt)       // sorted positions of the reads
          if ((uint32_t)(aux[pos + 1] >> 48) != (uint32_t)(aux[pos] >> 48)) tab[(uint32_t)(aux[pos] >> 48)] = (uint16_t)pos;
        __syncthreads();
        uint32_t seg_lo = 0;
        for (uint32_t k = 0; k <= n_reads; k++) {
          const uint32_t seg_hi = k < n_reads ? (uint32_t)tab[k] : n;
          bool any_full = false;
          for (uint32_t pos = seg_lo + tid; pos < seg_hi; pos += nt) {
            const uint32_t i = ord[pos];
            const uint32_t val = vals[i], mt = meta[i];
            if (!(val & V_RECV) || (mt & M_REPLY)) continue;
            const uint32_t tc = (mt >> M_TC_SHIFT) & 7u;
            if (tc == GT_ADD || tc == GT_REPL_ONE) atomicOr(myset + ((val & V_MASK) >> 5), 1u << (val & 31));
            else if (tc == GT_REPL_FULL) any_full = true;
          }
          if (__syncthreads_or(any_full ? 1 : 0)) {
            // @set |= value (g_set.rb:29-31): every thread owns a strided set of words
            for (uint32_t w = tid; w < p.bm_words; w += nt) {
              uint32_t acc = 0;
              // four snapshot rows at a time: the loads are independent, keep them all in flight
              for (uint32_t pos = seg_lo; pos < seg_hi; pos += 4) {
                uint32_t x[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (uint32_t q = 0; q < 4; q++) {
                  if (pos + q >= seg_hi) continue;
                  const uint32_t i = ord[pos + q];
                  const uint32_t val = vals[i], mt = meta[i];
                  if ((val & V_RECV) && !(mt & M_REPLY) && ((mt >> M_TC_SHIFT) & 7u) == GT_REPL_FULL) {
                    const uint32_t srow = val & V_MASK;    // sender = srow / gs_slots; its shard holds the row
                    const uint32_t* rows = p.gs_snap_sh[owner_of(srow / p.gs_slots, p.n_servers, p.n_shards)];
                    x[q] = __ldcg(rows + (size_t)srow * p.bm_words + w);
                  }
                }
                acc |= x[0] | x[1] | x[2] | x[3];
              }
              if (acc) myset[w] = __ldcg(myset + w) | acc;   // the adds above were atomics: read at L2
            }
            __syncthreads();
          }
          if (k < n_reads) {
            uint32_t cnt = 0;
            for (uint32_t w = tid; w < p.bm_words; w += nt) cnt += __popc(__ldcg(myset + w));
            const uint32_t total = block_sum_u32(cnt, s_wcnt);
            if (tid == 0) keyB[seg_hi] = total;            // keyB is free after the ordering phase
            seg_lo = seg_hi + 1;
          }
        }
        __syncthreads();
      }
    }

    // PD: claims: journal chunk, mailbox, per-neighbor ring blocks
    const bool mailed = (kind == MS_KIND_CLIENT || kind == MS_KIND_HOST);
    // per-(CTA, neighbor) ring claims need the rank of every gossip emission among this CTA's
    // emissions to that neighbor: mode 1 derives it from the sender blocks of the window
    // (table S), mode 2 (window was sorted the slow way) from a packed scan (deg <= 4)
    const bool agg_ok = nb_smem && n_new > 0 && !need_rng && const_lat == 0 && s_misc[3] == 0;
    const int agg_mode = !agg_ok ? 0 : (use_blocks ? 1 : (deg <= 4 ? 2 : 0));
    const bool agg = agg_mode != 0;
    uint32_t* F01 = keyB;                                   // mode 2: new-from-neighbor 0/1 before pos (2 x u16)
    uint32_t* F23 = reinterpret_cast<uint32_t*>(tab);       //         new-from-neighbor 2/3 before pos
    uint64_t f_total = 0;
    if (agg_mode == 2) {
      const int c = ((int)n + nt - 1) / nt;
      const int lo = min(tid * c, (int)n), hi = min(lo + c, (int)n);
      uint64_t acc = 0;
      for (int pos = lo; pos < hi; pos++) {
        const uint32_t i = ord[pos];
        const uint32_t ss = meta[i] & M_SRCSLOT;
        if ((vals[i] & V_FRESH) && ss >= 1 && ss <= 4) acc += 1ull << (16 * (ss - 1));
      }
      uint64_t run = block_excl_scan_u64v(acc, &f_total, s_wtmp);
      for (int pos = lo; pos < hi; pos++) {
        const uint32_t i = ord[pos];
        const uint32_t ss = meta[i] & M_SRCSLOT;
        F01[pos] = (uint32_t)run;
        F23[pos] = (uint32_t)(run >> 32);
        if ((vals[i] & V_FRESH) && ss >= 1 && ss <= 4) run += 1ull << (16 * (ss - 1));
      }
    }
    if (timing && tid == 0 && bcast && n_new > 0) atomicAdd((unsigned long long*)&p.phase_cycles[cls * 16 + (agg ? 11 : 12)], 1ull);
    if (timing && tid == 0 && n > 1) atomicAdd((unsigned long long*)&p.phase_cycles[cls * 16 + 13], (unsigned long long)R);
    if (tid == 32 % nt) {
      s_chunk = (n_ev_local && p.jlevel)
                    ? atomicAdd((unsigned long long*)&st->jraw_cursor, (unsigned long long)n_ev_local) : 0ull;
      if (n_ev_local && p.jlevel && !p.jdiscard && s_chunk + n_ev_local - st->jraw_drained > p.jmask + 1)
        latch_error(st, E_JOURNAL_OVERFLOW, ticket);
      if (mailed && n_recv) s_misc[0] = atomicAdd(&st->mail_count, n_recv);
    }
    if (agg && tid < (int)deg) {   // deg <= MAXNB <= 32 <= blockDim
      const uint32_t nb = s_nbr[tid];
      uint32_t acc = 0;
      if (agg_mode == 1) {
        // S[rho][j]: new messages, in blocks before rho, that came from neighbor j (they do not go back to j)
        for (uint32_t q = 0; q < R; q++) {
          s_S[q][tid] = (uint16_t)acc;
          const uint64_t ka = s_bkeyA[q];
          const uint32_t tk = (uint32_t)(ka & 0xFFFFFFu);
          if (tk >= p.n_inj_tickets && tk - p.n_inj_tickets == nb)
            acc += (uint32_t)(aux[s_boff[q + 1]] >> 48) - (uint32_t)(aux[s_boff[q]] >> 48);
        }
        s_S[R][tid] = (uint16_t)acc;
      } else {
        acc = (uint32_t)(f_total >> (16 * tid)) & 0xFFFFu;
      }
      const uint32_t total = n_new - acc;
      uint32_t base = 0;
      if (total) {
        const uint32_t o = owner_of(nb, p.n_servers, p.n_shards);
        base = atomicAdd(&p.tail_sh[o][nb], total);
        if ((uint32_t)(base + total - p.head_sh[o][nb]) > ring_cap_of(p, nb)) latch_error(st, E_RING_OVERFLOW, nb);
      }
      s_nbbase[tid] = base;
    }
    __syncthreads();
    cx.chunk = s_chunk;
    cx.n_recv = n_recv;
    cx.emitter = e;
    const bool cl_ep = kind_is_client(kind);
    const uint32_t msg_id_base = (is_server && p.next_msg_id) ? p.next_msg_id[e] : 0;
    const uint32_t set_before = (is_server && p.set_count) ? p.set_count[e] : 0;
    NbrList L;
    L.nl = nb_smem ? s_nbr : nullptr;
    L.deg = deg;
    PHASE_MARK(5);

    // PE1: :recv records (net.clj:244), one message per thread.  With journal level 1 and a
    //      neighbor as the source everything needed is already in shared memory.
    const bool full_recv = p.jlevel >= 2 || mailed || !use_blocks;
    for (uint32_t pos = tid; pos < n; pos += nt) {
      const uint32_t i = ord[pos];
      const uint32_t val = vals[i];
      if (!(val & V_RECV)) { c_part++; continue; }
      const uint32_t k = (uint32_t)(aux[pos] >> 32) & 0xFFFFu;
      const uint32_t mt = meta[i];
      const uint32_t sslot = mt & M_SRCSLOT;
      if (full_recv || !nb_smem || sslot == 0) {
        const Rec m = ring_load(p, p.ring, my0 + ((head + i) & my_mask), round, e);
        const uint64_t id = (use_blocks ? s_bbase[blk[pos]] : dense_base(p, st, m.round, m.ticket)) + m.idx;
        journal_raw(p, cx.chunk + k, id, true, m);
        const bool cl = cl_ep || (m.src >= p.n_servers && kind_is_client(p.kind[m.src]));
        if (cl) c_recv_cl++; else c_recv_sv++;
        if (kind == MS_KIND_SIM_CLIENT && ((m.tf >> 16) & MS_F_REPLY)) c_replies++;
        if (mailed) {
          const uint32_t mpos = s_misc[0] + k;
          if (mpos >= p.mail_cap) {
            latch_error(st, E_MAIL_OVERFLOW, e);
          } else {
            uint4* dst = reinterpret_cast<uint4*>(p.mail) + (size_t)mpos * 3;   // public ms_msg layout
            st_v4(dst + 0, make_uint4((uint32_t)id, (uint32_t)(id >> 32), (uint32_t)now, (uint32_t)((uint64_t)now >> 32)));
            st_v4(dst + 1, make_uint4(m.src, m.dest, m.msg_id, m.in_reply_to));
            st_v4(dst + 2, make_uint4(m.tf, m.p0, (uint32_t)m.p1, (uint32_t)(m.p1 >> 32)));
          }
        }
      } else {
        // server -> server gossip from topology neighbor sslot-1 (journal level 1)
        const uint64_t id = s_bbase[blk[pos]] + keyB[i];
        const uint64_t vrec = id | RECV_BIT;
        if (p.jlevel)
          st_v4(p.jraw + ((cx.chunk + k) & p.jmask),
                make_uint4((uint32_t)vrec, (uint32_t)(vrec >> 32), s_nbr[sslot - 1], e));
        c_recv_sv++;
      }
    }
    // PE2: emissions in id order, one emission per thread: emission j belongs to the last
    //      sorted position whose exclusive emit prefix is <= j.  When it fits, that map is
    //      materialised in the (now free) first-sight table instead of searched for.
    const bool own_map = agg_mode != 2 && n_emit_msgs <= 2u * cap;
    if (own_map) {
      for (uint32_t pos = tid; pos < n; pos += nt) {
        const uint32_t e0 = (uint32_t)aux[pos], e1 = (uint32_t)aux[pos + 1];
        for (uint32_t q = e0; q < e1; q++) tab[q] = (uint16_t)pos;
      }
      __syncthreads();
    }
    for (uint32_t base = 0; base < n_emit; base += nt) {
      const uint32_t j = base + tid;
      const bool valid = j < n_emit;
      Rec r;
      r.dest = 0; r.src = e;
      uint32_t direct = 0;
      bool has_direct = false;
      bool fast = false;
      bool timer_emission = false;
      if constexpr (GS) {
        if (valid && j < n_timer) {
          // replicate_full to the j-th other node (node.rb:104-108 other_node_ids, g_set.rb:36-38)
          timer_emission = true;
          r.dest = j < e ? j : j + 1;
          r.msg_id = 0; r.in_reply_to = 0; r.tf = MS_T_REPLICATE_FULL; r.p0 = fire_p0; r.p1 = fire_seq;
        }
      }
      if constexpr (RF) {
        if (valid && j < n_timer) {          // staged by the node's sequential step, in program order
          timer_emission = true;
          const uint4* at = p.rf_stage + ((size_t)e * p.rf_stage_cap + j) * 3;
          const uint4 a = at[0], b = at[1];
          r.src = a.x; r.dest = a.y; r.msg_id = a.z; r.in_reply_to = a.w;
          r.tf = b.x; r.p0 = b.y; r.p1 = (uint64_t)b.z | ((uint64_t)b.w << 32);
        }
      }
      if (kind == MS_KIND_GEN_CLIENT && valid && j < n_timer) {
        timer_emission = true;
        const uint4 a = s_gen[0], b = s_gen[1];
        r.src = a.x; r.dest = a.y; r.msg_id = a.z; r.in_reply_to = a.w;
        r.tf = b.x; r.p0 = b.y; r.p1 = 0;
      }
      if (valid && !timer_emission) {
        const uint32_t jm = j - n_timer;       // index among the emissions caused by messages
        uint32_t pos;
        if (own_map) {
          pos = tab[jm];
        } else {
          uint32_t lo = 0, hi = n;
          while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if ((uint32_t)aux[mid] <= jm) lo = mid; else hi = mid; }
          pos = lo;
        }
        const uint64_t a0 = aux[pos];
        const uint32_t k = jm - (uint32_t)a0;
        const uint32_t my_emit = (uint32_t)aux[pos + 1] - (uint32_t)a0;
        const uint32_t new_before = (uint32_t)(a0 >> 48);
        const uint32_t i = ord[pos];
        const uint32_t val = vals[i];
        const uint32_t mt = meta[i];
        const bool gossip = bcast && ((mt >> M_TC_SHIFT) & 7u) == TC_BROADCAST && !(mt & M_REPLY) &&
                            !((mt & M_HAS_ID) && k == my_emit - 1);
        if (gossip && nb_smem) {
          // k-th neighbor other than the sender, in topology order (02-performance.md:61-67)
          const uint32_t ss = mt & M_SRCSLOT;
          const uint32_t js = (ss && k >= ss - 1) ? k + 1 : k;
          r.dest = s_nbr[js];
          r.msg_id = 0; r.in_reply_to = 0; r.tf = MS_T_BROADCAST; r.p0 = val & V_MASK; r.p1 = 0;
          if (agg_mode == 1) {
            direct = s_nbbase[js] + new_before - s_S[blk[pos]][js];
            has_direct = true;
          } else if (agg_mode == 2) {
            const uint32_t f = js < 2 ? (F01[pos] >> (16 * js)) : (F23[pos] >> (16 * (js - 2)));
            direct = s_nbbase[js] + new_before - (f & 0xFFFFu);
            has_direct = true;
          }
          fast = has_direct && !np.any_removed;
        } else {
          const size_t g = my0 + ((head + i) & my_mask);
          const Rec m = bcast ? ring_load(p, p.ring, g, round, e) : ring_load_body(p, p.ring, g);
          MsgView w;
          w.src = m.src; w.msg_id = m.msg_id; w.tf = m.tf; w.p0 = m.p0;
          const uint64_t p1 = m.p1;
          bool svc_emission = false;
          if constexpr (SV) {
            if (kind == MS_KIND_SERVICE) {
              // the reply computed by the sequential pass + :in_reply_to (service.clj:255-258)
              svc_emission = true;
              r.src = e; r.dest = w.src; r.msg_id = 0; r.in_reply_to = w.msg_id;
              r.tf = (val & 0xFFFFu) | ((uint32_t)MS_F_REPLY << 16);
              r.p0 = (val >> 16) & 0xFFu;
              r.p1 = keyB[pos];
            }
          }
          if (svc_emission) {
          } else if constexpr (GS) {
            // g_set.rb:13-21: replies only; the set size a read reports was computed at its cut point
            const uint32_t tc = (mt >> M_TC_SHIFT) & 7u;
            r.src = e; r.dest = w.src; r.msg_id = 0; r.in_reply_to = w.msg_id; r.p0 = 0; r.p1 = 0;
            uint32_t otype = MS_T_ERROR;
            if (tc == GT_INIT) otype = MS_T_INIT_OK;
            else if (tc == GT_ADD) otype = MS_T_ADD_OK;
            else if (tc == GT_READ) { otype = MS_T_READ_OK; r.p0 = keyB[pos]; }
            else r.p0 = 10;                                  // not-supported (errors.edn)
            r.tf = otype | ((uint32_t)MS_F_REPLY << 16);
          } else {
          (void)node_emit(p, e, w, k, my_emit, jm, msg_id_base, set_before, new_before, p1, r, L);
          }
        }
      }
      if (fast) {
        // server -> neighbor gossip into ring space this CTA already claimed: what emit_one does for it, without
        // the general case's lookups (both ends are live servers, zero constant latency, no loss: agg_ok);
        // the record is compact, order key (round, ticket, j) == id order (net.clj:197)
        journal_raw(p, cx.chunk + n_recv + j, j, false, r);                    // net.clj:208
        cx.c_send_sv++;
        cx.c_zero++;
        ring_store_gossip(p.ring_sh[owner_of(r.dest, p.n_servers, p.n_shards)],
                          (size_t)r.dest * p.ring_cap_s + (direct & (p.ring_cap_s - 1u)), j, ticket, round, r.p0);
      }
      if (__any_sync(FULL, valid && !fast)) emit_one(p, st, np, cx, valid && !fast, r, j, direct, has_direct);
    }
    if (tid == 0 && is_server) {
      if (p.workload == MS_W_ECHO && p.next_msg_id && n_emit) p.next_msg_id[e] = msg_id_base + n_emit;
      if constexpr (!GS) {
      if (p.set_count && n_new) p.set_count[e] = set_before + n_new;
      } else {
        // periodic task bookkeeping: the run advances its schedule first, an init received this
        // round (re)starts it at `now` (oracle/oracle.cpp node_gset / gset_timer)
        int64_t nf = p.gs_next_fire[e];
        if (n_timer) {
          nf += (int64_t)p.gs_interval_ms * kTickNs;
          p.gs_fires[e] = fire_seq;
          p.gs_tag[e * p.gs_slots + (fire_seq & (p.gs_slots - 1))] = fire_seq;
        }
        if (s_misc[2]) { p.gs_init[e] = 1; nf = now; }
        p.gs_next_fire[e] = nf;
      }
      if (n > st->max_window_seen) atomicMax(&st->max_window_seen, n);
    }
  }

  PHASE_MARK(6);
  // ------------------------------------------------------------ ticket epilogue
  {
    uint32_t cnt[8] = {cx.c_send_cl, cx.c_send_sv, c_recv_cl, c_recv_sv, cx.c_lost, cx.c_zero, c_part, c_replies};
#pragma unroll
    for (int q = 0; q < 8; q++) {
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) cnt[q] += __shfl_xor_sync(FULL, cnt[q], d);
      if (lane == 0 && cnt[q]) atomicAdd(&s_cnt[q], cnt[q]);
    }
  }
  __syncthreads();
  if (tid < 8 && s_cnt[tid]) {
    // stats[2..5] = {clients send, clients recv, servers send, servers recv}; "all" is summed on the host
    const uint32_t v = s_cnt[tid];
    if (tid == 0) atomicAdd((unsigned long long*)&st->stats[2], (unsigned long long)v);
    else if (tid == 1) atomicAdd((unsigned long long*)&st->stats[4], (unsigned long long)v);
    else if (tid == 2) atomicAdd((unsigned long long*)&st->stats[3], (unsigned long long)v);
    else if (tid == 3) atomicAdd((unsigned long long*)&st->stats[5], (unsigned long long)v);
    else if (tid == 4) atomicAdd((unsigned long long*)&st->lost, (unsigned long long)v);
    else if (tid == 6) atomicAdd((unsigned long long*)&st->part_drops, (unsigned long long)v);
    else if (tid == 7) atomicAdd((unsigned long long*)&st->client_replies, (unsigned long long)v);
  }
  if (tid == 0) {
    // this ticket's table entry, validated by the round tag so that no fence is needed:
    // tag(16) | zero-latency pending(1) | events(23) | emissions(24); the last CTA turns
    // the counts into prefixes
    if (n_ev_local >= (1u << 23) || n_em_local >= (1u << 24)) latch_error(st, E_ID_RANGE, ticket);
    p.rt_chunk[(size_t)row * p.t_max + ticket] = cx.chunk;
    const uint64_t entry = ((uint64_t)tag << 48) | (s_cnt[5] ? (1ull << 47) : 0ull) |
                           ((uint64_t)(n_ev_local & 0x7FFFFFu) << 24) | (uint64_t)(n_em_local & 0xFFFFFFu);
    __stcg(reinterpret_cast<unsigned long long*>(p.rt_cnt + (size_t)row * p.t_max + ticket),
           (unsigned long long)entry);
    // single GPU: the last ticket commits the round right here; sharded: k_commit does it
    // after the cross-shard barrier
    s_misc[4] = (!p.split_commit && atomicAdd(&st->done, 1u) == T - 1) ? 1u : 0u;
    s_misc[5] = next_li;
  }
  __syncthreads();
  PHASE_MARK(7);
  if (s_misc[4]) {
    // ---------------------------------------------------------- last CTA: commit the round (DESIGN.md 2.3 step 4)
    commit_round(p, st, s_wtmp);
    PHASE_MARK(8);
  }
 }   // persistent loop
#undef PHASE_MARK
#undef TAB_SLOT
}

// ------------------------------------------------------------------ k_journal_expand (K3)
// Turns the raw per-(round, ticket) chunks of rounds [r0, r0 + n_rounds) into
// journal events in event-id order (journal.clj:225-239) for the event window
// [first, first + count): one warp per chunk.
__global__ void k_journal_expand(Params p, uint64_t r0, uint32_t n_rounds, uint64_t first, uint64_t count,
                                 uint4* out_ev, uint4* out_body) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t n_chunks = (uint64_t)n_rounds * p.t_max;
  for (uint64_t c = warp_global; c < n_chunks; c += n_warps) {
    const uint64_t r = r0 + c / p.t_max;
    const uint32_t t = (uint32_t)(c % p.t_max);
    const uint32_t row = (uint32_t)r & p.hist_mask;
    const RoundMeta* m = p.rmeta + row;
    if (m->round != r || t >= m->n_tickets) continue;
    if (owner_of_ticket(t, p.n_inj_tickets, p.n_servers, p.n_shards) != p.shard_id) continue;   // chunk lives on another shard
    const uint32_t* ev = p.rt_ev + (size_t)row * p.t_max;
    const uint64_t off = ev[t];
    const uint64_t end = (t + 1 < m->n_tickets) ? ev[t + 1] : m->ev_total;
    if (end == off) continue;
    const uint64_t g0 = m->ev_base + off;
    const uint64_t cnt = end - off;
    if (g0 + cnt <= first || g0 >= first + count) continue;
    const uint64_t chunk = p.rt_chunk[(size_t)row * p.t_max + t];
    const uint64_t send_base = m->id_base + p.rt_em[(size_t)row * p.t_max + t];
    const int64_t tnow = m->now;
    for (uint64_t k = lane; k < cnt; k += 32) {
      const uint64_t g = g0 + k;
      if (g < first || g >= first + count) continue;
      const uint4 raw = p.jraw[(chunk + k) & p.jmask];
      const uint64_t v = (uint64_t)raw.x | ((uint64_t)raw.y << 32);
      const bool recv = (v & RECV_BIT) != 0;
      const uint64_t id = recv ? (v & ~RECV_BIT) : send_base + v;
      const uint64_t eid = g | (recv ? MS_EVENT_RECV : 0ull);
      uint4* o = out_ev + (g - first) * 2;
      st_v4(o + 0, make_uint4((uint32_t)eid, (uint32_t)(eid >> 32), (uint32_t)tnow, (uint32_t)((uint64_t)tnow >> 32)));
      st_v4(o + 1, make_uint4((uint32_t)id, (uint32_t)(id >> 32), raw.z, raw.w));
      if (out_body) {
        const uint4* b = p.jbody + ((chunk + k) & p.jmask) * 2;
        const uint4 b0 = b[0], b1 = b[1];
        uint4* ob = out_body + (g - first) * 2;
        st_v4(ob + 0, make_uint4((uint32_t)id, (uint32_t)(id >> 32), b0.z, b0.w));
        st_v4(ob + 1, b1);
      }
    }
  }
}

// ------------------------------------------------------------------ journal streaming (ms_run_streamed)
// What has been packed so far lives in StreamPlan (a shadow of DevState's drain counters): the
// round kernels only ever see the counters k_stream_apply copies over between two rounds, so every
// kernel of a round takes the same back-pressure decision (round_skipped).
struct StreamPlan {
  uint64_t first, count, r0, n_rounds;
  uint64_t journal_drained, drain_round, jraw_drained;
  uint32_t overflow, more;
  unsigned long long local_n;   // sharded runs: events of this shard appended to the batch so far
  uint64_t hist[2][3];          // the drain counters as of batch i, slot i & 1: what k_stream_apply(i) hands over
  uint64_t pad;
};
static_assert(sizeof(StreamPlan) == 128, "StreamPlan is initialised from the host");

__global__ void k_stream_plan(Params p, StreamPlan* plan, uint64_t cap_events, uint32_t cap_rounds, ms_jround* rows, uint32_t format) {
  if (threadIdx.x || blockIdx.x) return;
  const DevState* st = p.st;
  const uint64_t first = plan->journal_drained;
  uint64_t count = st->next_event - first;
  if (count > cap_events) count = cap_events;
  const uint64_t r0 = plan->drain_round;
  uint64_t r1 = r0;
  while (r1 < st->round) {
    const RoundMeta* m = p.rmeta + ((uint32_t)r1 & p.hist_mask);
    if (m->round != r1 || m->ev_base >= first + count) break;
    if (r1 - r0 >= cap_rounds) { count = m->ev_base - first; break; }   // the rows table is full: cut at the round boundary
    ms_jround row;
    row.round = r1; row.time_ns = m->now; row.ev_base = m->ev_base;
    // MS_JFMT_4 (one GPU): the round's first message id -- its sends count up from it, its receives down from it
    row.id_ref = (format == MS_JFMT_4 && p.n_shards <= 1) ? m->id_base
                                                          : (m->id_base > (1ull << 30) ? m->id_base - (1ull << 30) : 0ull);
    rows[r1 - r0] = row;
    r1++;
  }
  plan->first = first; plan->count = count; plan->r0 = r0; plan->n_rounds = r1 - r0;
  plan->overflow = 0;
  plan->local_n = 0;
}

template <int FMT>
__global__ void k_journal_pack(Params p, StreamPlan* plan, unsigned char* out) {
  const uint64_t first = plan->first, count = plan->count, r0 = plan->r0;
  const uint32_t n_rounds = (uint32_t)plan->n_rounds;
  if (count == 0) return;
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t n_chunks = (uint64_t)n_rounds * p.t_max;
  bool bad = false;
  for (uint64_t c = warp_global; c < n_chunks; c += n_warps) {
    const uint64_t r = r0 + c / p.t_max;
    const uint32_t t = (uint32_t)(c % p.t_max);
    const uint32_t row = (uint32_t)r & p.hist_mask;
    const RoundMeta* m = p.rmeta + row;
    if (m->round != r || t >= m->n_tickets) continue;
    if (owner_of_ticket(t, p.n_inj_tickets, p.n_servers, p.n_shards) != p.shard_id) continue;
    const uint32_t* ev = p.rt_ev + (size_t)row * p.t_max;
    const uint64_t off = ev[t];
    const uint64_t end = (t + 1 < m->n_tickets) ? ev[t + 1] : m->ev_total;
    if (end == off) continue;
    const uint64_t g0 = m->ev_base + off;
    const uint64_t cnt = end - off;
    if (g0 + cnt <= first || g0 >= first + count) continue;
    const uint64_t chunk = p.rt_chunk[(size_t)row * p.t_max + t];
    const uint64_t send_base = m->id_base + p.rt_em[(size_t)row * p.t_max + t];
    const uint64_t id_ref = m->id_base > (1ull << 30) ? m->id_base - (1ull << 30) : 0ull;
    const int64_t tnow = m->now;
    // sharded runs: a shard holds only its own endpoints' events, so the batch is not positional: the
    // chunk's events in range are appended (one claim per chunk) with their event ids spelled out
    uint64_t slot0 = 0;
    const uint64_t k_lo = g0 < first ? first - g0 : 0, k_hi = g0 + cnt > first + count ? first + count - g0 : cnt;
    if (p.n_shards > 1) {
      if (lane == 0) slot0 = atomicAdd(&plan->local_n, (unsigned long long)(k_hi - k_lo));
      slot0 = __shfl_sync(FULL, slot0, 0);
    }
    for (uint64_t k = lane; k < cnt; k += 32) {
      const uint64_t g = g0 + k;
      if (g < first || g >= first + count) continue;
      const uint4 raw = p.jraw[(chunk + k) & p.jmask];
      const uint64_t v = (uint64_t)raw.x | ((uint64_t)raw.y << 32);
      const bool recv = (v & RECV_BIT) != 0;
      const uint64_t id = recv ? (v & ~RECV_BIT) : send_base + v;
      if (p.n_shards > 1) {
        const uint64_t at = slot0 + (k - k_lo);
        const uint64_t eid = g | (recv ? MS_EVENT_RECV : 0ull);
        if (FMT == 32) {
          uint4* o = reinterpret_cast<uint4*>(out) + at * 2;
          o[0] = make_uint4((uint32_t)eid, (uint32_t)(eid >> 32), (uint32_t)tnow, (uint32_t)((uint64_t)tnow >> 32));
          o[1] = make_uint4((uint32_t)id, (uint32_t)(id >> 32), raw.z, raw.w);
        } else {                                             // MS_JFMT_16: event id word + the MS_JFMT_8 word
          const uint64_t d = id - id_ref;
          if (id < id_ref || d >= (1ull << 31) || raw.z > 0xFFFFu || raw.w > 0xFFFFu) bad = true;
          const uint64_t w = (recv ? RECV_BIT : 0ull) | ((uint64_t)(raw.z & 0xFFFFu) << 47) |
                             ((uint64_t)(raw.w & 0xFFFFu) << 31) | (d & 0x7FFFFFFFull);
          reinterpret_cast<uint4*>(out)[at] = make_uint4((uint32_t)eid, (uint32_t)(eid >> 32), (uint32_t)w, (uint32_t)(w >> 32));
        }
        continue;
      }
      if (FMT == 8) {
        const uint64_t d = id - id_ref;
        if (id < id_ref || d >= (1ull << 31) || raw.z > 0xFFFFu || raw.w > 0xFFFFu) bad = true;
        const uint64_t w = (recv ? RECV_BIT : 0ull) | ((uint64_t)(raw.z & 0xFFFFu) << 47) |
                           ((uint64_t)(raw.w & 0xFFFFu) << 31) | (d & 0x7FFFFFFFull);
        reinterpret_cast<unsigned long long*>(out)[g - first] = w;
      } else if (FMT == 4) {
        // 32 bits per event.  A :send is {0, src (15), dest (16)}: sends appear in the journal in id order (both
        // counters are handed out in journal order, net.clj:197, journal.clj:228), so its id is implied by its
        // position.  A :recv is {1, id_base - 1 - id (31)}: src and dest are those of the :send with that id.
        uint32_t w;
        if (recv) {
          const uint64_t d = m->id_base - 1ull - id;
          if (id >= m->id_base || d >= (1ull << 31)) bad = true;
          w = 0x80000000u | (uint32_t)(d & 0x7FFFFFFFull);
        } else {
          if (raw.z > 0x7FFFu || raw.w > 0xFFFFu) bad = true;
          w = ((raw.z & 0x7FFFu) << 16) | (raw.w & 0xFFFFu);
        }
        reinterpret_cast<uint32_t*>(out)[g - first] = w;
      } else if (FMT == 12) {
        if (id >= (1ull << 47) || raw.z > 0xFFFFFFu || raw.w > 0xFFFFFFu) bad = true;
        uint32_t* o = reinterpret_cast<uint32_t*>(out) + (g - first) * 3;
        o[0] = (uint32_t)id;
        o[1] = (uint32_t)((id >> 32) & 0x7FFFu) | (recv ? 0x8000u : 0u) | ((raw.z & 0xFFFFu) << 16);
        o[2] = ((raw.z >> 16) & 0xFFu) | (raw.w << 8);
      } else {
        const uint64_t eid = g | (recv ? MS_EVENT_RECV : 0ull);
        uint4* o = reinterpret_cast<uint4*>(out) + (g - first) * 2;
        o[0] = make_uint4((uint32_t)eid, (uint32_t)(eid >> 32), (uint32_t)tnow, (uint32_t)((uint64_t)tnow >> 32));
        o[1] = make_uint4((uint32_t)id, (uint32_t)(id >> 32), raw.z, raw.w);
      }
    }
  }
  if (bad) atomicOr(&plan->overflow, 1u);
}

__global__ void k_stream_finish(Params p, StreamPlan* plan, ms_jbatch* hdr, uint32_t format, uint32_t parity) {
  if (threadIdx.x || blockIdx.x) return;
  const DevState* st = p.st;
  plan->journal_drained = plan->first + plan->count;
  uint64_t dr = plan->drain_round;
  while (dr < st->round) {
    const RoundMeta* m = p.rmeta + ((uint32_t)dr & p.hist_mask);
    if (m->round != dr || m->ev_base + m->ev_total > plan->journal_drained) break;
    dr++;
  }
  plan->drain_round = dr;
  plan->jraw_drained = dr < st->round ? p.rmeta[(uint32_t)dr & p.hist_mask].raw_base
                                      : *reinterpret_cast<const volatile uint64_t*>(&st->jraw_cursor);
  plan->more = st->next_event > plan->journal_drained ? 1u : 0u;
  plan->hist[parity][0] = plan->journal_drained;
  plan->hist[parity][1] = plan->drain_round;
  plan->hist[parity][2] = plan->jraw_drained;
  ms_jbatch b;
  b.first_event = plan->first; b.n_events = p.n_shards > 1 ? (uint64_t)plan->local_n : plan->count; b.n_rounds = plan->n_rounds;
  b.now = st->now; b.round = st->round; b.next_event = st->next_event;
  b.format = (p.n_shards > 1 && format != MS_JFMT_EVENT) ? (uint32_t)MS_JFMT_16 : format;
  b.overflow = plan->overflow; b.more = plan->more; b.error = st->error;
  b.range_events = plan->count;
  *hdr = b;
  __threadfence_system();
}

// on the engine's own stream, between two rounds: the round kernels now see what has been packed
__global__ void k_stream_apply(Params p, const StreamPlan* plan, uint32_t parity) {
  if (threadIdx.x || blockIdx.x) return;
  DevState* st = p.st;
  // the counters as of one given batch: every shard hands over the same drain_round at the same
  // place of its launch sequence, so all shards keep taking the same back-pressure decisions
  const uint64_t a = plan->hist[parity][0], b = plan->hist[parity][1], c = plan->hist[parity][2];
  if (a > st->journal_drained) st->journal_drained = a;
  if (b > st->drain_round) st->drain_round = b;
  if (c > st->jraw_drained) st->jraw_drained = c;
}

}  // namespace msd

// ------------------------------------------------------------------ host-callable launchers
extern "C" {

typedef void (*msk_round_fn)(msd::Params, uint32_t);
// round kernel of (node-program families: bit 0 g-set, bit 1 services; window-size class); fixed = the class has
// its default shape (ClsShape) and the family has a shape-specialised instantiation (echo / broadcast: family 0)
static msk_round_fn msk_round_kernel(uint32_t family, int cls, bool fixed = false) {
  if (fixed && (family & 7u) == 0 && cls < 3) {
    static const msk_round_fn fx[3] = {msd::k_round<0, 0, true>, msd::k_round<1, 0, true>, msd::k_round<2, 0, true>};
    return fx[cls];
  }
  static const msk_round_fn tab[8][4] = {
      {msd::k_round<0, 0>, msd::k_round<1, 0>, msd::k_round<2, 0>, msd::k_round<3, 0>},
      {msd::k_round<0, 1>, msd::k_round<1, 1>, msd::k_round<2, 1>, msd::k_round<3, 1>},
      {msd::k_round<0, 2>, msd::k_round<1, 2>, msd::k_round<2, 2>, msd::k_round<3, 2>},
      {msd::k_round<0, 3>, msd::k_round<1, 3>, msd::k_round<2, 3>, msd::k_round<3, 3>},
      {msd::k_round<0, 4>, msd::k_round<1, 4>, msd::k_round<2, 4>, msd::k_round<3, 4>},
      {nullptr, nullptr, nullptr, nullptr},     // g-set and Raft are different workloads
      {msd::k_round<0, 6>, msd::k_round<1, 6>, msd::k_round<2, 6>, msd::k_round<3, 6>},
      {nullptr, nullptr, nullptr, nullptr}};
  return tab[family & 7u][cls];
}

cudaError_t msk_round_smem_attr(size_t bytes) {
  cudaError_t e = cudaSuccess;
  for (uint32_t f = 0; f < 8 && e == cudaSuccess; f++)
    for (int c = 0; c < 4 && e == cudaSuccess; c++)
      if (msk_round_kernel(f, c))
        e = cudaFuncSetAttribute(msk_round_kernel(f, c), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  for (int c = 0; c < 3 && e == cudaSuccess; c++)
    e = cudaFuncSetAttribute(msk_round_kernel(0, c, true), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return e;
}

size_t msk_round_smem_bytes(uint32_t cap) { return (size_t)cap * 25 + 32; }

void msk_set_bit(uint32_t* words, size_t word, uint32_t bit, cudaStream_t s) {
  MS_LAUNCH(msd::k_set_bit, 1, 1, 0, s, words, word, bit);
}

int msk_round_occupancy(int threads, size_t smem) {
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, msk_round_kernel(0, 0), threads, smem) != cudaSuccess) return 1;
  return nb < 1 ? 1 : nb;
}

// One round = [k_release] k_snapshot | one persistent k_round grid per window-size class
// (caps ascending; every ticket is taken by exactly one class) | k_commit (sharded runs only;
// a single GPU commits inside k_round).  `phases` is a bit mask so that a sharded host can
// put its barriers in between: 1 = timing-wheel release, 8 = snapshot, 2 = round kernels, 4 = commit;
// 16 / 32 = k_glue opening the next round / closing a batch (sharded runs without the timing wheel).
void msk_launch_round(const msd::Params* p, int n_classes, const uint32_t* caps, const int* threads,
                      const int* grids, int with_release, cudaStream_t s, cudaEvent_t before_round,
                      cudaEvent_t after_round, int phases, const cudaStream_t* aux, const cudaEvent_t* aux_ev) {
  const uint32_t n_ep = p->n_ep;
  // two CTAs per SM on a B200 (the class-0 grid is SMs x occupancy >= 296 there)
  if (phases & 16) MS_LAUNCH(msd::k_glue, 1, 512, 0, s, *p, 1u);
  if (phases & 32) MS_LAUNCH(msd::k_glue, 1, 512, 0, s, *p, 0u);
  if ((phases & 1) && with_release) MS_LAUNCH(msd::k_release, grids[0] < 296 ? grids[0] : 296, 256, 0, s, *p);
  if (phases & 8) {
    const int sb = 256;
    int sg = (int)((n_ep + sb - 1) / sb);
    if (sg > 296) sg = 296;
    if (sg < 1) sg = 1;
    MS_LAUNCH(msd::k_snapshot, sg, sb, 0, s, *p);
  }
  if (phases & 2) {
    if (before_round) cudaEventRecord(before_round, s);
    // the size classes are independent of each other: run them concurrently (fork / join on
    // auxiliary streams; captured into the round graph as parallel branches)
    const bool fork = aux != nullptr && n_classes > 1;
    if (fork) cudaEventRecord(aux_ev[0], s);
    for (int c = n_classes - 1; c >= 0; c--) {   // big windows first
      const size_t sm = msk_round_smem_bytes(caps[c]);
      cudaStream_t sc = (fork && c != n_classes - 1) ? aux[c] : s;
      if (sc != s) cudaStreamWaitEvent(sc, aux_ev[0], 0);
      const int kc = c < 3 ? c : 3;
      const bool fixed = kc < 3 && caps[c] == msd::kClsLadder[kc] && threads[c] == msd::kClsThreads[kc];
      const msk_round_fn kern = msk_round_kernel(p->family, kc, fixed);
      MS_LAUNCH(kern, grids[c], threads[c], sm, sc, *p, caps[c]);
      if (sc != s) cudaEventRecord(aux_ev[1 + c], sc);
    }
    if (fork)
      for (int c = 0; c < n_classes - 1; c++) cudaStreamWaitEvent(s, aux_ev[1 + c], 0);
    if (after_round) cudaEventRecord(after_round, s);
  }
  if ((phases & 4) && p->split_commit) {
    const uint32_t T = p->n_inj_tickets + n_ep;
    if (p->cm_blk) {          // many tickets: three parallel phases
      const uint32_t nb = (T + msd::kCommitBlk - 1) / msd::kCommitBlk;
      MS_LAUNCH(msd::k_commit_a, nb, 256, 0, s, *p);
      MS_LAUNCH(msd::k_commit_b, 1, 512, 0, s, *p, nb);
      MS_LAUNCH(msd::k_commit_c, nb, 256, 0, s, *p);
    } else {
      MS_LAUNCH(msd::k_commit, 1, 512, 0, s, *p);
    }
  }
}

void msk_barrier(const msd::Params* p, cudaStream_t s) { MS_LAUNCH(msd::k_barrier, 1, 32, 0, s, *p); }

size_t msk_stream_plan_bytes() { return sizeof(msd::StreamPlan); }
// plan -> pack -> finish: one batch of the journal into (host-mapped) `out`, header into `hdr`
void msk_stream_batch(const msd::Params* p, void* plan, uint64_t cap_events, uint32_t cap_rounds, ms_jround* rows,
                      void* out, ms_jbatch* hdr, int format, int n_sms, cudaStream_t s, uint32_t parity) {
  msd::StreamPlan* pl = (msd::StreamPlan*)plan;
  MS_LAUNCH(msd::k_stream_plan, 1, 32, 0, s, *p, pl, cap_events, cap_rounds, rows, (uint32_t)format);
  const unsigned blocks = (unsigned)n_sms * 16;
  if (format == MS_JFMT_4) MS_LAUNCH(msd::k_journal_pack<4>, blocks, 256, 0, s, *p, pl, (unsigned char*)out);
  else if (format == MS_JFMT_8) MS_LAUNCH(msd::k_journal_pack<8>, blocks, 256, 0, s, *p, pl, (unsigned char*)out);
  else if (format == MS_JFMT_12) MS_LAUNCH(msd::k_journal_pack<12>, blocks, 256, 0, s, *p, pl, (unsigned char*)out);
  else MS_LAUNCH(msd::k_journal_pack<32>, blocks, 256, 0, s, *p, pl, (unsigned char*)out);
  MS_LAUNCH(msd::k_stream_finish, 1, 32, 0, s, *p, pl, hdr, (uint32_t)format, parity);
}
void msk_stream_apply(const msd::Params* p, const void* plan, cudaStream_t s, uint32_t parity) {
  MS_LAUNCH(msd::k_stream_apply, 1, 32, 0, s, *p, (const msd::StreamPlan*)plan, parity);
}

void msk_journal_expand(const msd::Params* p, uint64_t r0, uint32_t n_rounds, uint64_t first, uint64_t count,
                        void* out_ev, void* out_body, int n_sms, cudaStream_t s) {
  const uint64_t chunks = (uint64_t)n_rounds * p->t_max;
  uint64_t blocks = (chunks * 32 + 255) / 256;
  if (blocks > (uint64_t)n_sms * 16) blocks = (uint64_t)n_sms * 16;   // 2368 on a B200
  if (blocks < 1) blocks = 1;
  MS_LAUNCH(msd::k_journal_expand, (unsigned)blocks, 256, 0, s, *p, r0, n_rounds, first, count, (uint4*)out_ev,
            (uint4*)out_body);
}

}  // extern "C"
