#!/usr/bin/env python
"""bench.py -- simulated msgs/sec through the C ABI of maelstrom_b200.

Default (what the driver runs): BASELINE.json configs[1], the broadcast workload on 4096 nodes,
grid topology.  A "step" is one virtual tick (1 ms): V broadcast requests are injected by simulated
clients at Philox-random nodes and the engine runs delta rounds until the flood of every value has
died out (12 033 server messages per value on the 64x64 grid, BASELINE.md).

  value      delivered messages / second, inputs (the op schedule) resident in HBM, journal written
             to HBM, timed with CUDA events on the engine's stream (ms_timer_begin/end);
  e2e        the same metric through host buffers: every step uploads its ops from host memory
             (ms_schedule_ops) and the whole journal of the step streams back into pinned host memory
             (ms_run_streamed, 8 bytes per event) while the next rounds run;
  roofline   round kernel only: (128*sends + 144*recvs) algorithmic bytes (SURVEY.md 8d) / sum of
             its launch durations measured with CUDA events; `traffic` = bytes the kernel really
             moves, counted in-run from the record sizes of what it read and wrote;
  cpu_baseline  the CPU oracle (oracle/, a port of net.clj's rules) on a bounded sample of the same
             workload on the host cores.

--config selects the other BASELINE configs at full size: broadcast-lat1 (constant 1 ms latency:
the timing wheel is on), gset16k (configs[2]), raft64k (configs[3]), txn256k (configs[4]).
--verify adds a sharded parity run (256 nodes x 2000 values: merged journal digest vs the oracle).
--dump-outputs DIR writes what the timed steps computed (counters, clock, state of a seeded sample of
nodes; see dump_outputs) as .npy files, so that two builds can be compared output for output.
--impl reference times the CPU restatement instead (the JVM reference cannot run on this box: no
java/lein), on all host cores as independent replicas fed by one persistent worker pool.
"""
import argparse
import hashlib
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TICK_NS = 1_000_000
SEED = 0x4D41454C          # "MAEL"
ALG_SEND_B, ALG_RECV_B = 128, 144   # SURVEY.md section 8d


def philox_u32(n, stream, offset=0):
    """word 0 of Philox4x32-10(counter = (i, 0, 0, 0), key = (SEED, stream)), numpy restatement"""
    c0 = (np.arange(offset, offset + n, dtype=np.uint64)) & np.uint64(0xFFFFFFFF)
    c1 = np.zeros(n, dtype=np.uint64)
    c2 = np.zeros(n, dtype=np.uint64)
    c3 = np.zeros(n, dtype=np.uint64)
    k0 = np.full(n, SEED & 0xFFFFFFFF, dtype=np.uint64)
    k1 = np.full(n, stream, dtype=np.uint64)
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        a = M0 * c0
        b = M1 * c2
        n0 = (b >> np.uint64(32)) ^ c1 ^ k0
        n2 = (a >> np.uint64(32)) ^ c3 ^ k1
        c1 = b & mask
        c3 = a & mask
        c0, c2 = n0 & mask, n2 & mask
        k0 = (k0 + np.uint64(0x9E3779B9)) & mask
        k1 = (k1 + np.uint64(0xBB67AE85)) & mask
    return c0


# --------------------------------------------------------------------------- workloads
class Workload:
    """One BASELINE config: how to build the simulation, what a step injects, how bytes are counted."""
    name = ""
    label = ""
    n_nodes = 0
    n_clients = 64
    step_ticks = 1
    ramp_steps = 0                  # untimed steps before the warm-up (pipelines fill, leaders get elected)
    extra_recv_bytes = 0            # algorithmic payload bytes per delivered message on top of SURVEY 8d
    scaling = "strong"

    def __init__(self, args):
        self.args = args

    # engine -------------------------------------------------------------
    def sim_kwargs(self, n_steps, journal_discard):
        raise NotImplementedError

    def setup(self, sim, types):
        """add endpoints; returns the first client index"""
        from maelstrom_b200.engine import KIND_SIM_CLIENT
        c0 = None
        for i in range(self.n_clients):
            c = sim.add_endpoint("c%d" % i, KIND_SIM_CLIENT)
            c0 = c if c0 is None else c0
        return c0

    def prologue_ops(self, op_dtype, c0, types, flags):
        return None

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        raise NotImplementedError

    def between_steps(self, sim, step):
        """nemesis hook, called before step `step` runs (same on every rank)"""

    def dump_values(self, step):
        """--dump-outputs: the values whose presence in the sampled nodes' seen sets is written after step
        `step` (None: the workload keeps no seen sets)"""
        return None

    def alg_bytes(self, sends, recvs):
        return ALG_SEND_B * sends + (ALG_RECV_B + self.extra_recv_bytes) * recvs

    def real_bytes(self, sends, recvs):
        """what the fused round kernel moves per message by construction: 48-B ring record written +
        16-B raw journal record per send; 48-B record read + 16-B raw journal record + a 32-B seen-set
        sector read and its partial write-back (or the payload row) per receive"""
        return (48 + 16) * sends + (48 + 16 + 48 + self.extra_recv_bytes) * recvs

    # CPU oracle sample -----------------------------------------------------
    def cpu_sample(self, O, scale, seed):
        """run a bounded sample of the workload on the oracle; returns (messages, seconds, text)"""
        raise NotImplementedError


class Broadcast(Workload):
    name = "broadcast"
    n_nodes = 4096

    def __init__(self, args, latency_ms=0):
        Workload.__init__(self, args)
        self.latency_ms = latency_ms
        self.V = args.values_per_tick if args.values_per_tick else (32768 if latency_ms == 0 else 1024)
        # with latency L a flood lives ~126 L ticks: floods of consecutive ticks overlap, and the
        # pipeline is full after that many ticks
        self.step_ticks = 1 if latency_ms == 0 else 8
        self.ramp_steps = 0 if latency_ms == 0 else (130 * latency_ms) // self.step_ticks + 1
        self.label = "broadcast, 4096 nodes, grid 64x64 (BASELINE.json configs[1])"

    def sim_kwargs(self, n_steps, journal_discard):
        a = self.args
        kw = dict(workload="broadcast", topology="grid", latency_dist="constant",
                  latency_mean_ms=self.latency_ms, seed=SEED,
                  n_values=self.V * self.step_ticks * n_steps + 64,
                  max_endpoints=self.n_nodes + self.n_clients, ring_cap=a.ring_cap, max_window=a.max_window,
                  journal_level=1, journal_discard=1 if journal_discard else 0,
                  journal_cap_log2=a.journal_cap_log2, threads_per_node=a.threads)
        if self.latency_ms:
            # every message sent in a tick sits in ONE slot of the wheel until the next tick
            kw.update(calendar_slots=16, calendar_cap=self.V * 12033 // 8 + (1 << 16))
        return kw

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        per_tick = self.V
        n = n_steps * self.step_ticks * per_tick
        first_tick = first_step * self.step_ticks
        ops = np.zeros(n, dtype=op_dtype)
        g = np.arange(n, dtype=np.uint64) + np.uint64(first_tick * per_tick)     # global op index = value id
        ops["time_ns"] = ((g // np.uint64(per_tick)) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (g % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = (philox_u32(n, 1, offset=first_tick * per_tick) % np.uint64(self.n_nodes)).astype(np.uint32)
        ops["body"]["type"] = types["broadcast"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (g // np.uint64(self.n_clients) + np.uint64(1)).astype(np.uint32)
        ops["body"]["p0"] = g.astype(np.uint32)
        return ops

    def dump_values(self, step):
        first = step * self.step_ticks * self.V          # the values injected by this step
        return np.arange(first, first + self.step_ticks * self.V, dtype=np.uint64)

    def config_extra(self):
        return {"latency": "constant %d ms" % self.latency_ms, "values_per_tick": self.V,
                "l2_policy": "inputs larger than L2: inbox rings %.1f GB + seen bitmaps, streamed once per round"
                             % (self.n_nodes * self.args.ring_cap * 48 / 1e9)}

    def cpu_sample(self, O, scale, seed):
        per_tick = max(16, int(scale))
        s = O.Sim(self.n_nodes, workload=O.W_BROADCAST, topology="grid", n_values=per_tick + 1, seed=seed)
        c0 = None
        for i in range(self.n_clients):
            c = s.add_endpoint("c%d" % i, O.KIND_SIM_CLIENT)
            c0 = c if c0 is None else c0
        w = Broadcast(self.args, 0)
        w.V = per_tick
        s.schedule(w.ops(O.OP_DTYPE, 0, 1, c0, O.T, {"msg_id": O.F_MSG_ID}))
        t0 = time.perf_counter()
        s.run(TICK_NS)
        dt = time.perf_counter() - t0
        return s.stats()["all"]["recv-count"], dt, "%d values x 1 tick, latency 0" % per_tick


class GSet16k(Workload):
    """BASELINE configs[2]: g-set CRDT, 16384 nodes, 10 % loss + 100 ms (exponential) jitter.
    demo/ruby/g_set.rb:34-39: every node ships its whole set to every other node every 5 s."""
    name = "gset16k"
    n_nodes = 16384
    n_clients = 16
    interval_ms = 5000
    n_values = 16384                # universe of elements: a replicate_full payload is a 2-KB bitmap row
    adds_per_tick = 16

    def __init__(self, args, n_nodes=0, interval_ms=5000):
        Workload.__init__(self, args)
        self.n_nodes = n_nodes or args.nodes or 16384
        self.interval_ms = interval_ms
        self.step_ticks = self.interval_ms
        self.ramp_steps = 1                          # the staggered inits take one period
        self.extra_recv_bytes = self.n_values // 8   # the bitmap row a replicate_full names is read and OR-ed
        self.label = "g-set CRDT, %d nodes, 10 %% loss + exponential 100 ms latency (BASELINE.json configs[2])" % self.n_nodes

    def sim_kwargs(self, n_steps, journal_discard):
        n = self.n_nodes
        per_tick = n * (n - 1) // self.interval_ms + 1
        return dict(workload="g-set", topology="grid", latency_dist="exponential", latency_mean_ms=100, p_loss=0.1,
                    seed=SEED, n_values=self.n_values, gset_interval_ms=self.interval_ms,
                    max_endpoints=n + self.n_clients, ring_cap=2048, max_window=2048,
                    journal_level=1, journal_discard=1 if journal_discard else 0, journal_cap_log2=26,
                    calendar_slots=1024, calendar_cap=max(4096, 4 * per_tick))

    def prologue_ops(self, op_dtype, c0, types, flags):
        # db.clj:46-69 initialises the nodes one after the other: spread over the first period, so the
        # replication tasks of different nodes run at different ticks (as they do in a real run)
        n = self.n_nodes
        ops = np.zeros(n, dtype=op_dtype)
        i = np.arange(n, dtype=np.uint64)
        ops["time_ns"] = ((i * np.uint64(self.interval_ms)) // np.uint64(n) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (i % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = i.astype(np.uint32)
        ops["body"]["type"] = types["init"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (i // np.uint64(self.n_clients) + np.uint64(1)).astype(np.uint32)
        return ops

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        per_tick = self.adds_per_tick
        first_tick = max(first_step * self.step_ticks, 1)
        n_ticks = (first_step + n_steps) * self.step_ticks - first_tick
        n = n_ticks * per_tick
        ops = np.zeros(n, dtype=op_dtype)
        g = np.arange(n, dtype=np.uint64) + np.uint64(first_tick * per_tick)
        ops["time_ns"] = ((g // np.uint64(per_tick)) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (g % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = (philox_u32(n, 2, offset=first_tick * per_tick) % np.uint64(self.n_nodes)).astype(np.uint32)
        ops["body"]["type"] = types["add"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (np.uint64(1 << 20) + g // np.uint64(self.n_clients)).astype(np.uint32)
        ops["body"]["p0"] = (g % np.uint64(self.n_values)).astype(np.uint32)
        return ops

    def dump_values(self, step):
        return np.arange(self.n_values, dtype=np.uint64)

    def config_extra(self):
        return {"latency": "exponential, mean 100 ms", "p_loss": 0.1, "interval_ms": self.interval_ms,
                "step": "one replication period (5 s of virtual time): N x (N-1) replicate_full",
                "adds_per_tick": self.adds_per_tick,
                "l2_policy": "per step 2.7e8 distinct 48-B records through a 15-GB wheel pool and 1.6 GB of rings: larger than L2"}

    def cpu_sample(self, O, scale, seed):
        n, periods = 768, max(1, int(scale))
        w = GSet16k(self.args, n_nodes=n, interval_ms=500)
        w.n_clients, w.n_values, w.adds_per_tick = 4, 256, 1
        s = O.Sim(n, workload=O.W_GSET, latency_dist="exponential", latency_mean_ms=100, p_loss=0.1, seed=seed,
                  n_values=w.n_values, gset_interval_ms=w.interval_ms)
        cs = [s.add_endpoint("c%d" % i, O.KIND_SIM_CLIENT) for i in range(w.n_clients)]
        fl = {"msg_id": O.F_MSG_ID}
        ops = np.concatenate([w.prologue_ops(O.OP_DTYPE, cs[0], O.T, fl), w.ops(O.OP_DTYPE, 0, periods + 1, cs[0], O.T, fl)])
        s.schedule(ops[np.argsort(ops["time_ns"], kind="stable")])
        s.run(w.interval_ms * TICK_NS)                        # the staggered inits
        m0 = s.stats()["all"]["recv-count"]
        t0 = time.perf_counter()
        s.run((periods + 1) * w.interval_ms * TICK_NS)
        dt = time.perf_counter() - t0
        return s.stats()["all"]["recv-count"] - m0, dt, "g-set %d nodes x %d replication periods, 10 %% loss, exponential 100 ms" % (n, periods)


class Raft64k(Workload):
    """BASELINE configs[3]: lin-kv served by Raft (demo/python/raft.py), 65536 nodes in 5-node clusters
    (node_ids of a node's init = its cluster), partition nemesis re-rolled every virtual second."""
    name = "raft64k"
    n_nodes = 65536
    n_clients = 64
    group = 5
    ops_per_tick = 256
    n_keys = 16

    def __init__(self, args):
        Workload.__init__(self, args)
        self.n_nodes = args.nodes or 65536
        self.ops_per_tick = getattr(args, "ops_per_tick", 0) or 256
        self.step_ticks = 200
        self.ramp_steps = 23                         # 4.6 s: the first elections happen at 2-4 s (raft.py:249-251)
        self.label = "lin-kv on Raft, %d nodes in clusters of %d, partition nemesis (BASELINE.json configs[3])" % (self.n_nodes, self.group)
        self._rng = np.random.default_rng(SEED)

    def sim_kwargs(self, n_steps, journal_discard):
        n = self.n_nodes
        return dict(workload="lin-kv", topology="grid", latency_dist="constant", latency_mean_ms=0, seed=SEED,
                    max_endpoints=n + self.n_clients, ring_cap=8192, max_window=4096,
                    server_ring_cap=64, server_max_window=32, raft_group=self.group, rpc_table=64,
                    n_keys=self.n_keys, raft_log_cap=self.args.raft_log_cap,
                    journal_level=1, journal_discard=1 if journal_discard else 0, journal_cap_log2=24)

    def prologue_ops(self, op_dtype, c0, types, flags):
        n = self.n_nodes
        ops = np.zeros(n, dtype=op_dtype)
        i = np.arange(n, dtype=np.uint64)
        ops["src"] = (c0 + (i % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = i.astype(np.uint32)
        ops["body"]["type"] = types["init"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (i // np.uint64(self.n_clients) + np.uint64(1)).astype(np.uint32)
        return ops

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        per_tick = self.ops_per_tick
        first_tick = max(first_step * self.step_ticks, self.ramp_steps * self.step_ticks)   # clients start after the elections
        n_ticks = (first_step + n_steps) * self.step_ticks - first_tick
        if n_ticks <= 0:
            return np.zeros(0, dtype=op_dtype)
        n = n_ticks * per_tick
        ops = np.zeros(n, dtype=op_dtype)
        g = np.arange(n, dtype=np.uint64) + np.uint64(first_tick * per_tick)
        r = philox_u32(n, 3, offset=first_tick * per_tick)
        r2 = philox_u32(n, 4, offset=first_tick * per_tick)
        ops["time_ns"] = ((g // np.uint64(per_tick)) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (g % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = (r % np.uint64(self.n_nodes)).astype(np.uint32)
        kind = (r2 % np.uint64(3)).astype(np.int64)            # write / read / cas (workload/lin_kv.clj:12-38)
        ops["body"]["type"] = np.choose(kind, [types["write"], types["read"], types["cas"]]).astype(np.uint16)
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (np.uint64(1 << 20) + g // np.uint64(self.n_clients)).astype(np.uint32)
        ops["body"]["p0"] = ((r2 >> np.uint64(8)) % np.uint64(self.n_keys)).astype(np.uint32)
        v = (r2 >> np.uint64(16)) % np.uint64(5)
        ops["body"]["p1"] = np.where(kind == 2, v | (((r2 >> np.uint64(24)) % np.uint64(5)) << np.uint64(32)), v).astype(np.uint64)
        return ops

    def between_steps(self, sim, step):
        # nemesis: at every full virtual second the servers are split into two random components
        # (seeded: identical on every rank), one second later the partition is healed
        ticks = step * self.step_ticks
        if ticks % 1000 or ticks < self.ramp_steps * self.step_ticks:
            return
        if (ticks // 1000) % 2 == 0:
            sim.partition(self._rng.integers(0, 2, size=self.n_nodes).astype(np.uint32))
        else:
            sim.heal()

    def config_extra(self):
        return {"latency": "constant 0 ms", "ops_per_tick": self.ops_per_tick, "cluster_size": self.group,
                "step": "%d virtual ms" % self.step_ticks, "nemesis": "random halves for 1 s, healed for 1 s",
                "l2_policy": "node state (logs, KV, closure tables: > 1 GB) is touched once per round: larger than L2"}

    def cpu_sample(self, O, scale, seed):
        n = 3200
        s = O.Sim(n, workload=O.W_RAFT, seed=seed, raft_group=5, rpc_table=64)
        cs = [s.add_endpoint("c%d" % i, O.KIND_SIM_CLIENT) for i in range(4)]
        w = Raft64k(self.args)
        w.n_nodes, w.n_clients, w.ops_per_tick, w.ramp_steps = n, 4, 16, 23
        s.schedule(w.prologue_ops(O.OP_DTYPE, cs[0], O.T, {"msg_id": O.F_MSG_ID}))
        steps = 23 + max(1, int(scale))
        s.schedule(w.ops(O.OP_DTYPE, 0, steps, cs[0], O.T, {"msg_id": O.F_MSG_ID}))
        s.run(23 * 200 * TICK_NS)
        m0 = s.stats()["all"]["recv-count"]
        t0 = time.perf_counter()
        s.run(steps * 200 * TICK_NS)
        dt = time.perf_counter() - t0
        return s.stats()["all"]["recv-count"] - m0, dt, "Raft %d nodes (%d clusters of 5), 16 ops/tick x %d steps of 200 ms" % (n, n // 5, steps - 23)


class Txn256k(Workload):
    """BASELINE configs[4]: txn-list-append, 262144 nodes, every txn = read + cas of the root held by
    the lin-kv service (demo/clojure/single_key_txn.clj:134-173); the history is the journal."""
    name = "txn256k"
    n_nodes = 262144
    n_clients = 64
    txns_per_tick = 2048

    def __init__(self, args):
        Workload.__init__(self, args)
        self.n_nodes = args.nodes or 262144
        self.txns_per_tick = getattr(args, "ops_per_tick", 0) or 2048
        self.step_ticks = 50
        self.label = "txn-list-append, %d nodes, one lin-kv root (BASELINE.json configs[4])" % self.n_nodes

    def sim_kwargs(self, n_steps, journal_discard):
        n = self.n_nodes
        return dict(workload="txn-list-append", topology="grid", latency_dist="constant", latency_mean_ms=0, seed=SEED,
                    max_endpoints=n + self.n_clients + 4, ring_cap=8192, max_window=4096,
                    server_ring_cap=32, server_max_window=16, rpc_table=16,
                    journal_level=1, journal_discard=1 if journal_discard else 0, journal_cap_log2=24)

    def setup(self, sim, types):
        from maelstrom_b200.engine import KIND_SERVICE
        sim.add_endpoint("lin-kv", KIND_SERVICE)
        return Workload.setup(self, sim, types)

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        per_tick = self.txns_per_tick
        first_tick = first_step * self.step_ticks
        n = n_steps * self.step_ticks * per_tick
        ops = np.zeros(n, dtype=op_dtype)
        g = np.arange(n, dtype=np.uint64) + np.uint64(first_tick * per_tick)
        r = philox_u32(n, 5, offset=first_tick * per_tick)
        ops["time_ns"] = ((g // np.uint64(per_tick)) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (g % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = (r % np.uint64(self.n_nodes)).astype(np.uint32)
        ops["body"]["type"] = types["txn"]
        ops["body"]["flags"] = (flags["msg_id"] | np.where((r >> np.uint64(20)) % np.uint64(3) > 0, flags["appends"], 0)).astype(np.uint16)
        ops["body"]["msg_id"] = (g // np.uint64(self.n_clients) + np.uint64(1)).astype(np.uint32)
        ops["body"]["p1"] = g                                   # handle of the micro-op list (host side)
        return ops

    def config_extra(self):
        return {"latency": "constant 0 ms", "txns_per_tick": self.txns_per_tick, "step": "%d virtual ms" % self.step_ticks,
                "l2_policy": "per-node closure tables and staging rows (0.5 GB) + 0.4 GB of rings: larger than L2"}

    def cpu_sample(self, O, scale, seed):
        n = 2048
        s = O.Sim(n, workload=O.W_TXN, seed=seed, rpc_table=16)
        s.add_endpoint("lin-kv", O.KIND_SERVICE)
        cs = [s.add_endpoint("c%d" % i, O.KIND_SIM_CLIENT) for i in range(8)]
        w = Txn256k(self.args)
        w.n_nodes, w.n_clients, w.txns_per_tick = n, 8, 256
        steps = max(1, int(scale))
        s.schedule(w.ops(O.OP_DTYPE, 0, steps, cs[0], O.T, {"msg_id": O.F_MSG_ID, "appends": O.F_APPENDS}))
        t0 = time.perf_counter()
        s.run((steps * w.step_ticks + 2) * TICK_NS)
        dt = time.perf_counter() - t0
        return s.stats()["all"]["recv-count"], dt, "txn-list-append %d nodes, 256 txns/tick x %d ticks" % (n, steps * w.step_ticks)


class TxnTree(Txn256k):
    """txn-list-append on the persistent hash tree (demo/ruby/datomic_list_append.rb): tree nodes in lww-kv, the root
    pointer in lin-kv; 1-4 micro-ops per txn on a sliding window of keys.  Not a BASELINE config: a timing of the
    MS_W_TXN_TREE node program at a size that fits one GPU's tree-record table."""
    name = "txntree"

    def __init__(self, args):
        Txn256k.__init__(self, args)
        self.n_nodes = args.nodes or 16384
        self.txns_per_tick = getattr(args, "ops_per_tick", 0) or 256
        self.ramp_steps = 1                      # step 0 carries the inits (the first node writes the empty tree and the root)
        self.label = "txn-list-append on a persistent hash tree, %d nodes, lww-kv + lin-kv (datomic_list_append.rb)" % self.n_nodes

    def sim_kwargs(self, n_steps, journal_discard):
        n = self.n_nodes
        return dict(workload="txn-list-append-tree", topology="grid", latency_dist="constant", latency_mean_ms=0, seed=SEED,
                    max_endpoints=n + self.n_clients + 4, ring_cap=8192, max_window=4096,
                    server_ring_cap=64, server_max_window=32, rpc_table=64, tree_ptrs=1024, tree_cache=2048,
                    journal_level=1, journal_discard=1 if journal_discard else 0, journal_cap_log2=24)

    def setup(self, sim, types):
        from maelstrom_b200.engine import KIND_SERVICE
        sim.add_endpoint("lin-kv", KIND_SERVICE)
        sim.add_endpoint("lww-kv", KIND_SERVICE)
        return Workload.setup(self, sim, types)

    def prologue_ops(self, op_dtype, c0, types, flags):
        n = self.n_nodes
        ops = np.zeros(n, dtype=op_dtype)
        i = np.arange(n, dtype=np.uint64)
        ops["src"] = (c0 + (i % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = i.astype(np.uint32)
        ops["body"]["type"] = types["init"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (i // np.uint64(self.n_clients) + np.uint64(1)).astype(np.uint32)
        return ops

    def ops(self, op_dtype, first_step, n_steps, c0, types, flags):
        per_tick = self.txns_per_tick
        first_tick = max(first_step * self.step_ticks, self.step_ticks)          # clients start after the init step
        n_ticks = (first_step + n_steps) * self.step_ticks - first_tick
        if n_ticks <= 0:
            return np.zeros(0, dtype=op_dtype)
        n = n_ticks * per_tick
        ops = np.zeros(n, dtype=op_dtype)
        g = np.arange(n, dtype=np.uint64) + np.uint64(first_tick * per_tick)
        r = philox_u32(n, 6, offset=first_tick * per_tick)
        ops["time_ns"] = ((g // np.uint64(per_tick)) * np.uint64(TICK_NS)).astype(np.int64)
        ops["src"] = (c0 + (g % np.uint64(self.n_clients))).astype(np.uint32)
        ops["dest"] = (r % np.uint64(self.n_nodes)).astype(np.uint32)
        ops["body"]["type"] = types["txn"]
        ops["body"]["flags"] = flags["msg_id"]
        ops["body"]["msg_id"] = (g // np.uint64(self.n_clients) + np.uint64(1000)).astype(np.uint32)
        ops["body"]["p0"] = (g & np.uint64(0xFFFFFFFF)).astype(np.uint32)
        # 1-4 micro-ops, 2 of 3 appends, keys from a window of 64 that slides with time (Jepsen retires keys as it goes)
        base = (g // np.uint64(per_tick * 64)) * np.uint64(16)
        w = np.zeros(n, dtype=np.uint64)
        n_ops = np.uint64(1) + (r >> np.uint64(8)) % np.uint64(4)
        for j in range(4):
            rj = philox_u32(n, 7 + j, offset=first_tick * per_tick)
            key = (base + rj % np.uint64(64)) % np.uint64(16384)
            app = np.where((rj >> np.uint64(16)) % np.uint64(3) > 0, np.uint64(0x4000), np.uint64(0))
            w |= np.where(n_ops > np.uint64(j), (np.uint64(0x8000) | app | key) << np.uint64(16 * j), np.uint64(0))
        ops["body"]["p1"] = w
        return ops

    def config_extra(self):
        return {"latency": "constant 0 ms", "txns_per_tick": self.txns_per_tick, "step": "%d virtual ms" % self.step_ticks,
                "l2_policy": "tree records 0.5 GB + per-node caches and closure tables + lww-kv replicas: larger than L2"}

    def cpu_sample(self, O, scale, seed):
        n = 256                     # (the oracle visits every endpoint in every round: a sparse workload is slow on it)
        s = O.Sim(n, workload=O.W_TXN_TREE, seed=seed, rpc_table=64, tree_ptrs=512)
        s.add_endpoint("lin-kv", O.KIND_SERVICE)
        s.add_endpoint("lww-kv", O.KIND_SERVICE)
        cs = [s.add_endpoint("c%d" % i, O.KIND_SIM_CLIENT) for i in range(8)]
        w = TxnTree(self.args)
        w.n_nodes, w.n_clients, w.txns_per_tick = n, 8, 16
        steps = max(1, int(scale))
        flags = {"msg_id": O.F_MSG_ID, "appends": O.F_APPENDS}
        s.schedule(w.prologue_ops(O.OP_DTYPE, cs[0], O.T, flags))
        s.schedule(w.ops(O.OP_DTYPE, 0, steps + 1, cs[0], O.T, flags))
        t0 = time.perf_counter()
        s.run(((steps + 1) * w.step_ticks + 2) * TICK_NS)
        dt = time.perf_counter() - t0
        return s.stats()["all"]["recv-count"], dt, "hash-tree txn-list-append %d nodes, 16 txns/tick x %d ticks" % (n, (steps + 1) * w.step_ticks)


def make_workload(args):
    c = args.config
    if c == "broadcast":
        return Broadcast(args, args.latency_ms)
    if c == "broadcast-lat1":
        return Broadcast(args, 1)
    return {"gset16k": GSet16k, "raft64k": Raft64k, "txn256k": Txn256k, "txntree": TxnTree}[c](args)


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        threading.Thread.__init__(self, daemon=True)
        self.rows = []
        self.proc = None
        self.index = index

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = [nm for j, nm in enumerate(names)
                   if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- CPU restatement
class _Args:
    pass


def _oracle_worker(job):
    config, scale, seed, argd = job
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    a = _Args()
    a.__dict__.update(argd)
    a.config = config
    w = make_workload(a)
    msgs, dt, text = w.cpu_sample(O, scale, seed)
    return msgs, dt, text


def _arg_dict(args):
    return {k: getattr(args, k) for k in ("values_per_tick", "latency_ms", "ring_cap", "max_window", "journal_cap_log2",
                                          "threads", "nodes", "raft_log_cap", "config", "ops_per_tick")}


CPU_SCALE = {"broadcast": 1536, "broadcast-lat1": 1536, "gset16k": 4, "raft64k": 40, "txn256k": 400, "txntree": 5}


def cpu_baseline_single(args):
    """the oracle on one core, ~10-30 s of CPU work"""
    msgs, dt, text = _oracle_worker((args.config, CPU_SCALE[args.config], SEED, _arg_dict(args)))
    return {"value": msgs / dt, "unit": "msgs/s", "cores": 1, "kind": "port",
            "sample": "%s (%d msgs) in %.1f s, single-threaded oracle" % (text, msgs, dt)}


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    scale = max(1, CPU_SCALE[args.config] // 4)         # per replica and step: a step takes a few seconds
    argd = _arg_dict(args)
    ctx = mp.get_context("spawn")
    wl = make_workload(args)
    with ctx.Pool(cores) as pool:                       # ONE pool for the whole run: workers stay warm
        jobs = lambda k: [(args.config, scale, SEED + 1000 * k + i, argd) for i in range(cores)]
        for k in range(args.warmup):
            pool.map(_oracle_worker, jobs(k))
        per_step = []
        text = ""
        for k in range(args.steps):
            t0 = time.perf_counter()
            res = pool.map(_oracle_worker, jobs(args.warmup + k))
            wall = time.perf_counter() - t0
            per_step.append((sum(r[0] for r in res), wall))
            text = res[0][2]
    m_all = sum(p[0] for p in per_step)
    t_all = sum(p[1] for p in per_step)
    rates = [m / t for m, t in per_step]
    value = m_all / t_all
    line = {
        "impl": "reference", "metric": metric_name(wl), "value": value,
        "unit": "msgs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_all / max(args.steps, 1), "higher_is_better": True, "scaling": wl.scaling,
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": wl.label, "sample_per_replica": text,
                   "note": "CPU restatement of net.clj (oracle/), not the JVM: no java/lein on this box; %d independent "
                           "replicas (one per host core, different seeds) from one persistent worker pool; wall clock "
                           "around each step's map" % cores,
                   "step_rate_spread": (max(rates) - min(rates)) / value if rates else None},
        "cpu_baseline": {"value": value, "unit": "msgs/s", "cores": cores, "kind": "port",
                         "sample": "%d replicas x (%s) per step" % (cores, text)},
        "e2e": {"value": value, "unit": "msgs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def metric_name(wl):
    if wl.name == "broadcast":
        return "simulated msgs/sec (broadcast, 4096 nodes)"
    return "simulated msgs/sec (%s)" % wl.name


# --------------------------------------------------------------------------- outputs
DUMP_NODES = 128                 # seeded sample of nodes whose state --dump-outputs writes
DUMP_VALUES = 32768              # at most this many values (seeded sample) per node: seen.npy stays <= 16 MB
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, sim, wl, step):
    """--dump-outputs: what the timed path has computed once its last step (`step`) is done, as .npy files:
    stats.npy     send / recv / msg counts of all endpoints, clients, servers (Sim.stats order), float64
    clock.npy     virtual time (ns) and round, float64
    net.npy       messages lost, messages dropped by partitions, replies to clients, float64
    nodes.npy     the sampled node indices, float64
    seen.npy      seen-set workloads: [node, value] = 1.0 where the sampled node holds the value, float32;
    values.npy    its columns: the values the last step injected (g-set: every element), float64
    raft.npy      Raft workload: Sim.raft_state of each sampled node (Sim.RAFT_FIELDS order), float64
    The node and value samples are drawn from a fixed seed, so equal arguments give comparable files."""
    from maelstrom_b200.engine import Sim, WORKLOADS
    rng = np.random.default_rng(SEED)
    nodes = np.sort(rng.choice(wl.n_nodes, size=min(DUMP_NODES, wl.n_nodes), replace=False))
    st = sim.stats()
    c = sim.counters()
    out = {"stats": np.array([st[g][k] for g in ("all", "clients", "servers") for k in ("send-count", "recv-count", "msg-count")],
                             dtype=np.float64),
           "clock": np.array([sim.now, sim.round], dtype=np.float64),
           "net": np.array([c["lost"], c["partition_drops"], sim.client_replies()], dtype=np.float64),
           "nodes": nodes.astype(np.float64)}
    values = wl.dump_values(step)
    if values is not None:
        if len(values) > DUMP_VALUES:
            values = np.sort(rng.choice(values, size=DUMP_VALUES, replace=False))
        out["values"] = values.astype(np.float64)
        seen = np.zeros((len(nodes), len(values)), dtype=np.float32)
        for i, k in enumerate(nodes):
            held = np.zeros(sim.cfg.n_values, dtype=bool)
            held[sim.node_set(int(k))] = True
            seen[i] = held[values]
        out["seen"] = seen
    if sim.workload == WORKLOADS["lin-kv"]:
        out["raft"] = np.array([[sim.raft_state(int(k))[f] for f in Sim.RAFT_FIELDS] for k in nodes], dtype=np.float64)
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------- GPU arm
def make_sim(mb, wl, n_steps, journal_discard, device, world):
    kw = wl.sim_kwargs(n_steps, journal_discard)
    if world > 1:
        # one shard per rank; cross-shard messages go over NVLink peer memory (maelstrom_b200/sharded.py)
        from maelstrom_b200.sharded import ShardedSim
        sim = ShardedSim(wl.n_nodes, device=device, **kw)
    else:
        sim = mb.Sim(wl.n_nodes, device=device, **kw)
    from maelstrom_b200.engine import TYPES
    c0 = wl.setup(sim, TYPES)
    return sim, c0


def run_to(sim, t_ns):
    if sim.run_raw(t_ns) == 1:     # journal_discard runs never ask for a drain
        raise RuntimeError("device asked for a journal drain in a journal_discard run")


def sharded_verify(mb, world, rank, local_rank):
    """256 nodes x 2000 values, sharded over `world` GPUs: SHA-256 of the merged journal must equal
    the oracle's (computed on rank 0 on the host)."""
    from maelstrom_b200.engine import KIND_SIM_CLIENT, OP_DTYPE, TYPES, F_MSG_ID
    n, V = 256, 2000
    kw = dict(workload="broadcast", topology="grid", n_values=V + 8, ring_cap=4096, max_window=2048,
              journal_cap_log2=23, max_endpoints=n + 8, journal_level=1, seed=SEED)
    if world > 1:
        from maelstrom_b200.sharded import ShardedSim
        g = ShardedSim(n, device=local_rank, **kw)
    else:
        g = mb.Sim(n, device=local_rank, **kw)
    cs = [g.add_endpoint("c%d" % i, KIND_SIM_CLIENT) for i in range(4)]
    ops = np.zeros(V, dtype=OP_DTYPE)
    i = np.arange(V, dtype=np.uint64)
    ops["time_ns"] = ((i // np.uint64(250)) * np.uint64(TICK_NS)).astype(np.int64)
    ops["src"] = (cs[0] + i % np.uint64(4)).astype(np.uint32)
    ops["dest"] = (philox_u32(V, 9) % np.uint64(n)).astype(np.uint32)
    ops["body"]["type"] = TYPES["broadcast"]
    ops["body"]["flags"] = F_MSG_ID
    ops["body"]["msg_id"] = (i // np.uint64(4) + np.uint64(1)).astype(np.uint32)
    ops["body"]["p0"] = i.astype(np.uint32)
    g.schedule(ops)
    g.run(10 * TICK_NS)
    ev = g.gather_journal() if world > 1 else g.drain(bodies=False)[0]
    g.close()
    if rank != 0:
        return None
    digest = hashlib.sha256(np.ascontiguousarray(ev).tobytes()).hexdigest()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    o = O.Sim(n, workload=O.W_BROADCAST, topology="grid", n_values=V + 8, seed=SEED)
    for k in range(4):
        o.add_endpoint("c%d" % k, O.KIND_SIM_CLIENT)
    o.schedule(ops)
    o.run(10 * TICK_NS)
    ev_o, _ = o.journal()
    want = hashlib.sha256(np.ascontiguousarray(ev_o.astype(ev.dtype)).tobytes()).hexdigest()
    return {"parity_digest_ok": digest == want, "events": int(len(ev)), "sha256": digest[:16], "oracle_sha256": want[:16],
            "scenario": "broadcast, 256 nodes, 2000 values, %d shard(s): merged journal vs the oracle" % world}


class _NoCuda:
    """MS_BENCH_EMUL=1 (test infrastructure): dry-run of the harness on the CPU SIMT emulator; prints no
    usable number.  Never set on the GPU box."""
    class cuda:
        @staticmethod
        def synchronize():
            pass

        @staticmethod
        def set_device(i):
            pass


def gpu_arm(args, rank, world, local_rank):
    if os.environ.get("MS_BENCH_EMUL") == "1":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import emul_lib
        emul_lib.use().__enter__()
        torch = _NoCuda
    else:
        import torch
    import maelstrom_b200 as mb
    from maelstrom_b200.engine import TYPES, F_MSG_ID, F_APPENDS, OP_DTYPE
    from maelstrom_b200 import _lib

    flags = {"msg_id": F_MSG_ID, "appends": F_APPENDS}
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = make_workload(args)
    W, K, R = args.warmup, args.steps, wl.ramp_steps
    step_ns = wl.step_ticks * TICK_NS

    # ---- arm A: device-resident (value + roofline): ramp, W warm-up, K timed, K profiled steps
    total_a = R + W + 2 * K + 1
    sim, c0 = make_sim(mb, wl, total_a, True, local_rank, world)
    lstats = (lambda: sim.sim.stats()["all"]) if world > 1 else (lambda: sim.stats()["all"])   # this rank's endpoints
    pro = wl.prologue_ops(OP_DTYPE, c0, TYPES, flags)
    ops = wl.ops(OP_DTYPE, 0, total_a, c0, TYPES, flags)
    if pro is not None:
        ops = np.concatenate([pro, ops])
        ops = ops[np.argsort(ops["time_ns"], kind="stable")]
    sim.schedule(ops)
    step = 0

    def do_steps(n):
        nonlocal step
        for _ in range(n):
            wl.between_steps(sim, step)
            step += 1
            run_to(sim, step * step_ns)

    do_steps(R + W)
    if args.phase_cycles and world == 1:
        sim.phase_cycles(True)          # diagnostic: clock64() between the phases of every ticket (slows the kernels)
    before = lstats()
    c_before = sim.counters()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.25)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    sim.timer_begin()
    do_steps(K)
    ms_value = sim.timer_end()
    torch.cuda.synchronize()
    after = lstats()
    c_after = sim.counters()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sim, wl, R + W + K - 1)
    if args.phase_cycles and world == 1:
        pc = sim.phase_cycles(False)
        names = ["fetch", "load+seen (PA)", "order (PB)", "first-sight+counts (PC)", "scan", "claims (PD)", "records+emissions (PE)",
                 "epilogue", "commit"]
        for c in range(4):
            nt = int(pc[c][15])
            if not nt:
                continue
            tot = sum(int(pc[c][k]) for k in range(9))
            sys.stderr.write("class %d: %d tickets, %.0f cycles per ticket (thread 0's clock64 between phases)\n" % (c, nt, tot / nt))
            for k in range(9):
                sys.stderr.write("   %-26s %8.0f cycles/ticket  %5.1f %%\n" % (names[k], int(pc[c][k]) / nt, 100.0 * int(pc[c][k]) / max(tot, 1)))
    recvs = after["recv-count"] - before["recv-count"]
    sends = after["send-count"] - before["send-count"]
    launches = c_after["launches"] - c_before["launches"]
    rounds = c_after["rounds"] - c_before["rounds"]

    # roofline pass: the same work again (next K steps) with CUDA events around every round-kernel launch
    sim.profile(True)
    sim.profile_read()
    b2 = lstats()
    do_steps(K)
    a2 = lstats()
    k_ms, k_launches = sim.profile_read()
    sim.profile(False)
    # the sampler ran through the timed steps and the identical profiled steps; short multi-GPU runs can be over before
    # nvidia-smi's first row: the GPU is still under the same load pattern, wait for one
    t_wait = time.time()
    late = not sampler.rows
    while not sampler.rows and time.time() - t_wait < 3.0:
        time.sleep(0.05)
    clocks = sampler.stop()
    if late:
        clocks["note"] = "run shorter than nvidia-smi's start-up: first row taken right after the profiled steps"
    p_sends, p_recvs = a2["send-count"] - b2["send-count"], a2["recv-count"] - b2["recv-count"]
    alg_bytes = wl.alg_bytes(p_sends, p_recvs)
    real_bytes = wl.real_bytes(p_sends, p_recvs)
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    max_window = c_after["max_window"]
    fallback = c_after["fallback_sorts"] - c_before["fallback_sorts"]
    sim.close()

    # ---- arm B: end to end through host buffers (ops in from host memory, journal out to pinned host memory)
    e2e = None
    if not args.no_e2e:
        total_b = R + W + K + 1
        sim, c0 = make_sim(mb, wl, total_b, False, local_rank, world)
        lstats = (lambda: sim.sim.stats()["all"]) if world > 1 else (lambda: sim.stats()["all"])
        n_ep = wl.n_nodes + wl.n_clients + 8
        fmt = _lib.JFMT_4 if n_ep <= 32768 else _lib.JFMT_8 if n_ep <= 65536 else _lib.JFMT_12
        if args.stream_format:
            fmt = args.stream_format
        pro = wl.prologue_ops(OP_DTYPE, c0, TYPES, flags)
        host_ops = [wl.ops(OP_DTYPE, t, 1, c0, TYPES, flags) for t in range(total_b)]
        if pro is not None:                     # the inits belong to step 0
            m = np.concatenate([pro, host_ops[0]])
            host_ops[0] = m[np.argsort(m["time_ns"], kind="stable")]
        d2h = 0
        h2d = 0
        check = {"events": 0, "xor": 0}

        def sink(info, rnds, ev):
            # the consumer's work per batch: fold the packed records (the host touches every byte)
            check["events"] += len(ev)
            check["xor"] ^= int(np.bitwise_xor.reduce(ev.reshape(-1).view(np.uint32))) if len(ev) else 0

        st = 0
        for st in range(R + W):
            wl.between_steps(sim, st)
            sim.schedule(host_ops[st])
            sim.run_streamed((st + 1) * step_ns, None, fmt=fmt, buf_events=args.stream_events)
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        s0 = lstats()["recv-count"]
        t0 = time.perf_counter()
        for st in range(R + W, R + W + K):
            wl.between_steps(sim, st)
            sim.schedule(host_ops[st])                                 # host -> device: this step's ops
            h2d += host_ops[st].nbytes
            n_ev, n_b = sim.run_streamed((st + 1) * step_ns, sink if args.touch else None, fmt=fmt,
                                         buf_events=args.stream_events)   # device -> host: the step's journal
            d2h += n_b
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        t_e2e = time.perf_counter() - t0
        msgs_e2e = lstats()["recv-count"] - s0
        sim.close()
        e2e = {"seconds": t_e2e, "msgs": msgs_e2e, "h2d": h2d // max(K, 1), "d2h": d2h // max(K, 1), "fmt": fmt}

    verify = None
    if (args.verify or world > 1) and not args.no_verify:
        verify = sharded_verify(mb, world, rank, local_rank)

    # ---- aggregate over ranks (max time, sum of work)
    if dist:
        t = torch.tensor([ms_value, k_ms, e2e["seconds"] if e2e else 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        w = torch.tensor([recvs, sends, launches, alg_bytes, real_bytes, e2e["msgs"] if e2e else 0,
                          e2e["h2d"] if e2e else 0, e2e["d2h"] if e2e else 0], device="cuda", dtype=torch.float64)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        ms_value, k_ms = float(t[0]), float(t[1])
        recvs, sends, launches, alg_bytes, real_bytes = (int(x) for x in w.tolist()[:5])
        if e2e:
            e2e["seconds"] = float(t[2])
            e2e["msgs"], e2e["h2d"], e2e["d2h"] = (int(x) for x in w.tolist()[5:])
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9 / world if k_ms > 0 else 0.0     # per GPU

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    value = recvs / (ms_value * 1e-3)
    cfg = {"workload": wl.label, "step": "1 virtual tick (1 ms)" if wl.step_ticks == 1 else "%d virtual ms" % wl.step_ticks,
           "nodes": wl.n_nodes, "delivered_msgs_per_step": recvs // max(K, 1), "rounds_per_step": rounds / max(K, 1),
           "ramp_steps": R, "max_window_seen": max_window, "fallback_sorts": fallback,
           "parallelism": ("%d shards by endpoint range, cross-shard messages written into peer inbox rings over NVLink"
                           % world) if world > 1 else "single GPU",
           "published_reference": "6e4 msgs/s, 48-way Xeon (README.md:39-42), different hardware"}
    cfg.update(wl.config_extra())
    line = {
        "metric": metric_name(wl), "value": value, "unit": "msgs/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_value / K, "higher_is_better": True,
        "scaling": wl.scaling, "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": cfg,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     # bytes the round kernels moved per launch, from the sizes of the records they read and
                     # wrote in this very run (ring records, raw journal records, seen-set words)
                     "traffic": real_bytes / max(k_launches, 1) / (world if world > 1 else 1),
                     "traffic_unit": "bytes per round (one launch of each size class), counted in-run from record sizes",
                     "algorithmic_bytes_per_round": alg_bytes / max(k_launches, 1) / (world if world > 1 else 1),
                     "kernel": "msd::k_round", "launches": k_launches, "avg_launch_us": 1e3 * k_ms / max(k_launches, 1),
                     "algorithmic_bytes_per_msg": ALG_SEND_B + ALG_RECV_B + wl.extra_recv_bytes, "peak_source": peak_src,
                     "per_gpu": world > 1},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if e2e:
        line["e2e"] = {"value": e2e["msgs"] / e2e["seconds"], "unit": "msgs/s", "h2d_bytes_per_step": e2e["h2d"],
                       "d2h_bytes_per_step": e2e["d2h"],
                       "note": ("host op buffers in every step (ms_schedule_ops); the whole journal of the step streamed into "
                                "pinned host memory (ms_run_streamed, %d bytes per event, packed on the device, copied out by "
                                "the DMA engine behind the running rounds); lazily expandable with ms_journal_decode / ms_jdecoder"
                                % (e2e["fmt"] if world == 1 else 16)) +
                               ("" if world == 1 else "; every rank uploads the ops and streams its own shard's events (event id + "
                                "packed word each) over its own PCIe link: bytes are summed over the ranks")}
    if verify:
        line["verify"] = verify
        line["parity_digest_ok"] = verify["parity_digest_ok"]
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_single(args)
    print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="broadcast", choices=["broadcast", "broadcast-lat1", "gset16k", "raft64k", "txn256k", "txntree"])
    ap.add_argument("--values-per-tick", type=int, default=0)
    ap.add_argument("--latency-ms", type=int, default=0)
    ap.add_argument("--nodes", type=int, default=0, help="override the node count of gset16k / raft64k / txn256k")
    ap.add_argument("--ops-per-tick", type=int, default=0, help="override the client op rate of raft64k / txn256k")
    ap.add_argument("--ring-cap", type=int, default=8192)
    ap.add_argument("--max-window", type=int, default=4096)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--journal-cap-log2", type=int, default=28)
    ap.add_argument("--stream-events", type=int, default=1 << 26, help="events per host buffer of ms_run_streamed")
    ap.add_argument("--raft-log-cap", type=int, default=1024)
    ap.add_argument("--stream-format", type=int, default=0, choices=[0, 4, 8, 12, 32], help="e2e: bytes per journal event (0 = smallest that fits)")
    ap.add_argument("--touch", action="store_true", help="e2e: fold every streamed byte on the host inside the timed region")
    ap.add_argument("--verify", action="store_true", help="sharded parity digest (on by default when --gpus > 1)")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--phase-cycles", action="store_true", help="diagnostic: per-phase cycles per ticket on stderr; needs a -DMS_PHASE_TIMING build (MS_B200_LIB=...); not a bench run")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed steps computed into DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the GPU path on one GPU")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        reference_arm(args, rank, world)
    else:
        gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
