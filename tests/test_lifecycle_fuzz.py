"""Endpoints that come and go while traffic is in flight, engine against the oracle (DESIGN.md 2.1, 2.4, 2.7).

Jepsen closes and reopens a client after every indefinite op, so removal and slot recycling are on the
normal path.  Recycling a slot resets its ring, its birth id (the timing wheel drops mail for the old
name), its seq-kv client index and its host mailbox; once anything is removed the round kernels give
the removed endpoint an empty window, count sends to it as undeliverable and leave the compact gossip
path.  Two deterministic regression tests pin the service rules; the seeded fuzzer interleaves traffic
with every kind of removal and re-adding and compares everything both sides expose.  Each test runs
[emul] (kernel sources on the CPU SIMT emulator) in the CPU suite and [cuda] on a B200.
`MS_LIFECYCLE_SEEDS=a:b` and `MS_LIFECYCLE_SHARDED_SEEDS=a:b` widen the seed ranges."""
import os

import numpy as np
import pytest

import oracle_lib as O
from scenarios import assert_same_journal, both, make_pair
from test_emul_sharded import check_against_oracle, run_sharded_scenario
from test_fuzz_parity import random_ops
from test_txn_tree import pack_ops

pytestmark = pytest.mark.usefixtures("engine_backend")
SVC = ("lin-kv", "seq-kv", "lww-kv", "lin-tso")
USER_KINDS = (O.KIND_CLIENT, O.KIND_HOST, O.KIND_SIM_CLIENT)


def seed_range(var, default):
    a, b = (int(x) for x in os.environ.get(var, default).split(":"))
    return list(range(a, b))


def stop_nodes(s):
    """ms_stop_nodes on the engine; the oracle has no such call and removes every server instead"""
    if isinstance(s, O.Sim):
        for i in range(s.n_nodes):
            s.remove_endpoint(i)
    else:
        s._chk(s.L.ms_stop_nodes(s.h))


def test_readded_service_starts_empty():
    # service.clj:147-156, 290-296: a service added again is a new atom.  The old lin-kv held key 5 = 3 and
    # the old lin-tso had handed out 0 and 1; the new ones know nothing of either.
    g, o = make_pair(3, workload="echo", max_endpoints=32)

    def scenario(s, body):
        c = s.add_endpoint("c0")
        sv = {name: s.add_endpoint(name, O.KIND_SERVICE) for name in SVC}
        mids = iter(range(1, 100))

        def rpc(name, type, **kw):
            s.send(c, sv[name], body(type, msg_id=next(mids), **kw))
            r = s.recv(c, 1_000_000_000)
            return int(r["type"]), int(r["p0"]), int(r["p1"])

        before = [rpc(name, "write", p0=5, p1=3) for name in SVC[:3]]
        before += [rpc(name, "read", p0=5) for name in SVC[:2]]
        before += [rpc("lin-tso", "ts"), rpc("lin-tso", "ts")]
        for name in SVC:
            s.remove_endpoint(sv[name])
            sv[name] = s.add_endpoint(name, O.KIND_SERVICE)
        after = [rpc(name, "read", p0=5) for name in SVC[:3]] + [rpc("lin-tso", "ts")]
        return before, after, sorted(sv.values())

    rg, ro = both(g, o, scenario)
    assert rg == ro
    T = O.T
    before, after, idx = rg
    assert before == [(T["write_ok"], 0, 0)] * 3 + [(T["read_ok"], 0, 3)] * 2 + [(T["ts_ok"], 0, 0), (T["ts_ok"], 0, 1)]
    assert after == [(T["error"], 20, 0)] * 3 + [(T["ts_ok"], 0, 0)]
    assert idx == [8, 9, 10, 11]                              # services never recycle a slot
    assert_same_journal(g, o)


@pytest.mark.parametrize("workload", ["txn-list-append", "txn-list-append-tree"])
def test_txn_node_sends_to_a_removed_lin_kv_are_undeliverable(workload):
    # A node addresses lin-kv by name, i.e. the index where lin-kv was last added.  Once it is removed the
    # node's requests are journaled, dropped and counted (net.clj:166-176); the run goes on, and a lin-kv
    # added again (empty) serves the next txn.
    n = 3
    tree = workload.endswith("tree")
    sizing = dict(rpc_table=256, tree_ptrs=4096) if tree else {}
    g, o = make_pair(n, workload=workload, max_endpoints=32, **sizing)

    def scenario(s, body):
        kv = s.add_endpoint("lin-kv", O.KIND_SERVICE)
        if tree:
            s.add_endpoint("lww-kv", O.KIND_SERVICE)
        c = s.add_endpoint("c0")
        for i in range(n):
            s.send(c, i, body("init", msg_id=1 + i))
            assert int(s.recv(c, 1_000_000_000)["type"]) == O.T["init_ok"]
        txn = pack_ops([("append", 3), ("r", 3)]) if tree else 101

        def ask(node, mid, timeout):
            s.send(c, node, body("txn", msg_id=mid, p1=txn, appends=not tree))
            r = s.recv(c, timeout)
            return None if r is None else (int(r["type"]), int(r["in_reply_to"]), int(r["p0"]))

        out = [ask(0, 10, 1_000_000_000)]
        s.remove_endpoint(kv)
        out.append(ask(1, 11, 20_000_000))
        out.append(s.undeliverable())
        kv2 = s.add_endpoint("lin-kv", O.KIND_SERVICE)
        out.append(ask(2, 12, 1_000_000_000))
        return out, kv2

    rg, ro = both(g, o, scenario)
    assert rg == ro
    (first, lost, undeliverable, third), kv2 = rg
    assert first[:2] == (O.T["txn_ok"], 10) and lost is None and undeliverable >= 1
    assert third is not None and third[1] == 12 and kv2 > n
    assert_same_journal(g, o)
    assert g.undeliverable() == o.undeliverable()


def test_recycled_slot_starts_a_new_seq_kv_session():
    # seq-kv remembers, per client endpoint, the newest state the client has seen (service.clj:162-166).  A
    # client that takes over a recycled slot is a new client: it may be served any of the resident states,
    # including ones older than what the slot's previous owner had seen.
    g, o = make_pair(2, workload="echo", max_endpoints=16)

    def scenario(s, body):
        kv = s.add_endpoint("seq-kv", O.KIND_SERVICE)
        c = s.add_endpoint("c0")
        for v in range(1, 13):
            s.send(c, kv, body("write", msg_id=v, p0=1, p1=v))
            assert int(s.recv(c, 1_000_000_000)["type"]) == O.T["write_ok"]
        s.remove_endpoint(c)
        c2 = s.add_endpoint("c1")
        got = []
        for k in range(24):
            s.send(c2, kv, body("read", msg_id=k + 1, p0=1))
            r = s.recv(c2, 1_000_000_000)
            got.append((int(r["type"]), int(r["p0"]), int(r["p1"])))
        return c2 == c, got

    rg, ro = both(g, o, scenario)
    assert rg == ro
    recycled, got = rg
    assert recycled
    assert min(v for t, _, v in got if t == O.T["read_ok"]) < 12 or any(t == O.T["error"] for t, _, _ in got)
    assert_same_journal(g, o)


class Lifecycle:
    """One seeded run: traffic phases separated by lifecycle events and network faults.  The same object
    drives the engine and the oracle; every value a call returns is recorded in `seen` for comparison."""

    def __init__(self, seed, sharded=False):
        rng = np.random.default_rng(31000 + seed)
        self.seed = seed
        self.sharded = sharded
        wls = ("broadcast", "g-set", "txn-list-append", "broadcast") if sharded else (
            "broadcast", "g-set", "echo", "txn-list-append", "txn-list-append-tree", "lin-kv", "broadcast")
        self.workload = wls[seed % len(wls)]            # every workload within the first seeds
        self.world = int(rng.integers(2, 5)) if sharded else 1
        if self.workload == "lin-kv":
            self.n = int(rng.integers(3, 6))
        else:
            self.n = int(rng.integers(max(2, self.world), 24))
        dist = ("constant", "constant", "uniform", "exponential")[int(rng.integers(4))]
        mean = 0 if dist == "constant" and rng.integers(3) else int(rng.integers(1, 5))     # 0: compact gossip
        self.dist, self.mean = dist, mean
        self.kw = dict(latency_dist=dist, latency_mean_ms=mean, n_values=4096,
                       p_loss=float(rng.choice([0.0, 0.0, 0.03])), seed=int(rng.integers(1 << 40)))
        if self.workload in ("broadcast", "g-set"):
            self.kw["topology"] = ("grid", "line", "tree3", "total")[int(rng.integers(4))]
        if self.workload == "g-set":
            self.kw["gset_interval_ms"] = int(rng.integers(3, 10))
        self.gen = 0 if sharded or self.workload not in ("broadcast", "g-set") else (0, 4, 9)[seed % 3]
        self.services = self.workload.startswith("txn") or bool(rng.integers(2))
        self.sizing = dict(max_endpoints=self.n + self.gen + 40, ring_cap=1024, max_window=1024,
                           journal_cap_log2=20, calendar_slots=1024, calendar_cap=8192)
        if self.workload == "txn-list-append-tree":
            self.sizing.update(rpc_table=256, tree_ptrs=8192)
        self.phases = int(rng.integers(5, 10))
        self.events = [int(x) for x in rng.permutation(9)[:self.phases]]      # each event at most once
        self.faults = [int(x) for x in rng.integers(0, 8, size=self.phases)]
        self.stop_at_end = not sharded and bool(rng.integers(4) == 0)

    # traffic -------------------------------------------------------------------------------------
    def ops(self, s, r2, t_ms, ticks):
        st = self.st
        senders = [e for e, k in st["users"].items() if k == O.KIND_SIM_CLIENT or (k == O.KIND_CLIENT and r2.integers(2))]
        if not senders:
            return
        per_tick = int(r2.integers(1, 10))
        wl = self.workload
        if wl == "lin-kv":
            rows = np.zeros(ticks * per_tick, dtype=O.OP_DTYPE)
            for k in range(len(rows)):
                c = int(r2.integers(len(senders)))
                st["mids"][senders[c]] = st["mids"].get(senders[c], 0) + 1
                r = rows[k]
                r["time_ns"] = (t_ms + k // per_tick) * 1_000_000
                r["src"], r["dest"] = senders[c], int(r2.integers(self.n))
                b = r["body"]
                b["flags"], b["msg_id"], b["p0"] = O.F_MSG_ID, st["mids"][senders[c]], int(r2.integers(4))
                kind = int(r2.integers(3))
                b["type"] = (O.T["read"], O.T["write"], O.T["cas"])[kind]
                b["p1"] = int(r2.integers(4)) | ((int(r2.integers(4)) << 32) if kind == 2 else 0)
        else:
            mids = [st["mids"].get(e, 0) for e in senders]
            live_svc = {k: v for k, v in st["svc"].items() if v is not None} if wl != "txn-list-append-tree" else {}
            rows = random_ops(r2, self.n, senders, live_svc, "txn-list-append" if wl.startswith("txn") else wl,
                              t_ms, ticks, per_tick, mids)
            if wl == "txn-list-append-tree":
                for r in rows:
                    if r["body"]["type"] == O.T["txn"]:
                        r["body"]["p1"] = pack_ops([(("append", "r")[int(r2.integers(2))], int(r2.integers(30)))
                                                    for _ in range(int(r2.integers(1, 4)))])
            for e, m in zip(senders, mids):
                st["mids"][e] = m
        rows = rows[[int(d) not in st["dead"] for d in rows["dest"]]]     # ms_schedule_ops takes live endpoints only
        s.schedule(rows)

    def drain(self, s, everything):
        if self.sharded:
            return
        st = self.st
        for e, k in sorted(st["users"].items()):
            if k == O.KIND_SIM_CLIENT or (not everything and e % 2):
                continue
            while True:
                m = s.recv(e, 0)
                if m is None:
                    break
                st["seen"].append(("recv", e, int(m["id"]), int(m["type"]), int(m["src"]), int(m["in_reply_to"]),
                                   int(m["p0"]), int(m["p1"])))

    def add_user(self, s, kind):
        st = self.st
        st["names"] += 1
        name = ("h%d" if kind == O.KIND_HOST else "c%d") % (1000 + st["names"])
        e = s.add_endpoint(name, kind)
        st["seen"].append(("add", name, kind, e))
        st["users"][e] = kind
        return e

    def request(self, s, body, e, dest=None):
        st = self.st
        st["mids"][e] = st["mids"].get(e, 0) + 1
        dest = self.live_server(st["r2"]) if dest is None else dest
        if dest is None:
            return
        ty = {"echo": "echo", "lin-kv": "read", "g-set": "read"}.get(self.workload, "read")
        if self.workload == "broadcast" and st["r2"].integers(2):
            s.send(e, dest, body("broadcast", msg_id=st["mids"][e], p0=int(st["r2"].integers(4096))))
        else:
            s.send(e, dest, body(ty, msg_id=st["mids"][e], p0=3))

    def live_server(self, r2):
        live = [i for i in range(self.n) if i not in self.st["dead"]]
        return live[int(r2.integers(len(live)))] if live else None

    def step(self, s, k):
        for _ in range(k):
            s.step(1)

    # lifecycle events ----------------------------------------------------------------------------
    def event(self, s, body, ev):
        st, r2 = self.st, self.st["r2"]
        users = sorted(st["users"])
        if ev == 0 and users:                   # a request / reply in the removed endpoint's ring
            e = users[int(r2.integers(len(users)))]
            self.request(s, body, e)
            self.step(s, 1 + int(r2.integers(2)))
            self.remove(s, e)
            self.recycle(s)
        elif ev == 1:                           # server latency: the reply to a host is in the timing wheel
            hosts = [e for e in users if st["users"][e] == O.KIND_HOST] or [self.add_user(s, O.KIND_HOST)]
            e = hosts[int(r2.integers(len(hosts)))]
            self.request(s, body, e)
            self.step(s, 1 + int(r2.integers(2 + self.mean)))
            self.remove(s, e)
            self.recycle(s)
        elif ev == 2:
            self.recycle(s, True)
        elif ev == 3 and self.n > 1:            # pairwise drops suppress recycling until heal!
            a, b = int(r2.integers(self.n)), int(r2.integers(self.n))
            s.drop(a, b)
            if users:
                self.remove(s, users[int(r2.integers(len(users)))])
            self.add_user(s, USER_KINDS[int(r2.integers(3))])
            self.step(s, 2)
            s.heal()
            self.add_user(s, USER_KINDS[int(r2.integers(3))])
        elif ev == 4 and st["gen"]:             # one closed-loop client leaves
            self.remove(s, st["gen"].pop(int(r2.integers(len(st["gen"])))))
        elif ev == 5:                           # a server leaves mid-run
            if self.workload == "lin-kv":       # the leader, or a follower
                roles = [(s.raft_state(i)["state"], i) for i in range(self.n) if i not in st["dead"]]
                st["seen"].append(("roles", roles))
                leaders = [i for r, i in roles if r == 3]
                pick = leaders if leaders and r2.integers(2) else [i for _, i in roles]
                victim = pick[int(r2.integers(len(pick)))] if pick else None
            else:
                victim = self.live_server(r2)
            if victim is not None and len(st["dead"]) < max(1, self.n // 3):
                if self.workload == "broadcast" and users:     # gossip is under way when it goes
                    self.request(s, body, users[0], victim)
                    self.step(s, 1)
                self.remove(s, victim)
                st["dead"].add(victim)
        elif ev in (6, 7) and self.services:    # a service leaves with requests queued, and comes back
            # the hash tree's nodes live in lww-kv: a new, empty lww-kv loses them, and datomic_list_append.rb
            # retries a read that finds nothing at once, forever (at zero latency: 2^20 rounds at one instant)
            names = [k for k in SVC if k != "lww-kv"] if self.workload == "txn-list-append-tree" else SVC
            name = names[int(r2.integers(len(names)))]
            idx = st["svc"][name]
            if idx is None:
                st["svc"][name] = s.add_endpoint(name, O.KIND_SERVICE)
                st["seen"].append(("svc", name, st["svc"][name]))
                return
            for e in users:
                if st["users"][e] != O.KIND_SIM_CLIENT:
                    st["mids"][e] = st["mids"].get(e, 0) + 1
                    ty = "ts" if name == "lin-tso" else ("read", "write")[int(r2.integers(2))]
                    s.send(e, idx, body(ty, msg_id=st["mids"][e], p0=int(r2.integers(5)), p1=int(r2.integers(4))))
            self.step(s, 1)
            s.remove_endpoint(idx)
            st["svc"][name] = None
            if ev == 6 or self.workload.startswith("txn") and r2.integers(2):
                st["svc"][name] = s.add_endpoint(name, O.KIND_SERVICE)
            st["seen"].append(("svc", name, st["svc"][name]))

    def recycle(self, s, always=False):
        """mostly at once, before another round: the old endpoint's mail is still in the ring and the wheel"""
        st, r2 = self.st, self.st["r2"]
        if always or r2.integers(3):
            gone = st["gone_kinds"]                 # re-add into the freed slot under a different kind
            self.add_user(s, [k for k in USER_KINDS if k != (gone[-1] if gone else None)][int(r2.integers(2))])

    def remove(self, s, e):
        st = self.st
        st["seen"].append(("remove", e, s.remove_endpoint(e)))
        st["gone_kinds"].append(st["users"].pop(e, None))

    def fault(self, s, f, r2):
        if f == 1 and self.n > 1:
            s.drop(int(r2.integers(self.n)), int(r2.integers(self.n)))
        elif f == 2:
            s.partition([int(r2.integers(2)) for _ in range(self.n)])
        elif f == 3:
            s.heal()
        elif f == 4:                            # one level of slow! at most: x100 leaves the wheel
            if self.st["slow"]:
                s.fast()
                self.st["slow"] = False
            elif self.dist != "exponential":
                s.slow()
                self.st["slow"] = True
        elif f == 5:
            s.set_loss(float(r2.integers(0, 30)) / 100.0)
        elif f == 6:
            s.flaky()
            self.st["flaky"] = True
        if self.st.get("flaky") and f != 6:     # flaky! for one phase: half the messages lost
            s.set_loss(0.0)
            self.st["flaky"] = False

    # the run -------------------------------------------------------------------------------------
    def __call__(self, s, body):
        r2 = np.random.default_rng(self.seed)       # the same stream for both executions
        st = self.st = dict(r2=r2, users={}, mids={}, dead=set(), gen=[], gone_kinds=[], seen=[], names=0,
                            slow=False, svc={name: None for name in SVC})
        if self.services:
            for name in SVC:
                if self.workload != "txn-list-append-tree" or name in ("lin-kv", "lww-kv") or r2.integers(2):
                    st["svc"][name] = s.add_endpoint(name, O.KIND_SERVICE)
        for k in (O.KIND_CLIENT, O.KIND_SIM_CLIENT, O.KIND_HOST, O.KIND_SIM_CLIENT):
            self.add_user(s, k)
        t_ms = 0
        if self.gen:
            first = s.add_gen_clients(self.gen, interval_ns=int(r2.integers(1, 3_000_000)), time_limit_ns=40_000_000,
                                      read_permille=300, timeout_ns=30_000_000, quiet_ns=5_000_000, first_name=0)
            st["gen"] = list(range(first, first + self.gen))
        init = sorted(e for e, k in st["users"].items() if k == O.KIND_SIM_CLIENT)[0]
        if self.workload != "broadcast":
            for i in range(self.n):
                s.send(init, i, body("init", msg_id=9000 + i))
        if self.workload == "lin-kv":
            t_ms = 2500                             # a leader first (raft.py: election timeout 2 s)
            s.run(t_ms * 1_000_000)
        for ph in range(self.phases):
            self.fault(s, self.faults[ph], r2)
            ticks = int(r2.integers(2, 8))
            self.ops(s, r2, t_ms, ticks)
            s.run((t_ms + ticks // 2) * 1_000_000)
            self.event(s, body, self.events[ph])     # mid-phase: scheduled ops name removed and recycled slots
            self.drain(s, False)
            t_ms = max(t_ms + ticks, s.now // 1_000_000 + 1)
            s.run(t_ms * 1_000_000)
            if self.workload == "lin-kv" and ph % 2:
                t_ms += 300
                s.run(t_ms * 1_000_000)
        if self.stop_at_end:
            stop_nodes(s)
            st["dead"] = set(range(self.n))
            for e in sorted(st["users"]):
                if st["users"][e] != O.KIND_SIM_CLIENT:
                    self.request(s, body, e, 0)
        s.heal()
        if st["slow"]:
            s.fast()
        s.set_loss(0.0)
        s.run((t_ms + 60 + 12 * self.mean) * 1_000_000)
        self.drain(s, True)
        out = dict(seen=st["seen"], undeliverable=s.undeliverable(), replies=s.client_replies())
        if self.sharded:
            return out
        if self.workload == "lin-kv":
            out["raft"] = [s.raft_state(i) for i in range(self.n)]
        elif self.workload in ("broadcast", "g-set"):
            out["sets"] = [s.node_set(i).tolist() for i in range(self.n)]
        if self.gen:
            h = s.history()
            out["history"] = [h[f].tolist() for f in ("time_ns", "order", "client", "op", "type", "f", "error", "value")]
        return out


@pytest.mark.parametrize("seed", seed_range("MS_LIFECYCLE_SEEDS", "0:8"))
def test_lifecycle_scenario(seed):
    import maelstrom_b200 as mb
    run = Lifecycle(seed)
    g, o = make_pair(run.n, workload=run.workload, **run.kw, **run.sizing)
    rg, ro = both(g, o, run)
    assert rg == ro
    assert_same_journal(g, o)


@pytest.mark.parametrize("seed", seed_range("MS_LIFECYCLE_SHARDED_SEEDS", "0:4"))
def test_lifecycle_sharded(engine_backend, seed):
    # 2-4 emulated shards: every shard applies the same lifecycle calls; recycled client and host slots,
    # servers and services removed, against the single oracle (merged level-1 journal, stats, clock)
    if engine_backend != "emul":
        pytest.skip("emulated shards (one process): the CPU suite; multi-GPU runs are tests/test_gpu_sharded.py")
    run = Lifecycle(seed, sharded=True)
    wl = {"broadcast": O.W_BROADCAST, "g-set": O.W_GSET, "txn-list-append": O.W_TXN}[run.workload]
    sizing = dict(run.sizing, ring_cap=2048, journal_cap_log2=20)

    def scenario(s, body):                     # one Lifecycle per shard thread: each keeps its own state
        return Lifecycle(seed, sharded=True)(s, body)

    ev, st, now, rnd = run_sharded_scenario(run.world, run.n, dict(workload=run.workload, **run.kw, **sizing), scenario)
    check_against_oracle(O.Sim(run.n, workload=wl, **run.kw), scenario, ev, st, now, rnd)
