"""Pins the oracle's Raft restatement to the reference's own code.  tests/golden/
raft_reference_trace.json is every message sent by a 3-node cluster of the UNMODIFIED
demo/python/raft.py of jepsen-io/maelstrom, executed by tests/golden/raft_reference_harness.py under the
schedule of DESIGN.md section 2.8 (virtual clock, Philox draws).  The oracle, given the same
client operations, must send the same messages with the same ids at the same times, and end in
the same node states.  raft_reference_trace_partition.json and raft_reference_trace_random.json hold the
same for a partitioned 5-node cluster and for random scenarios; the harness regenerates all three
from a maelstrom checkout."""
import json
import os
import sys

import numpy as np
import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
FIXTURE = os.path.join(HERE, "golden", "raft_reference_trace.json")


def canonical_from_oracle(sim, ev, bd):
    names = {v: k for k, v in O.T.items()}
    out = []
    for e, b in zip(ev, bd):
        if int(e["event_id"]) >> 63:
            continue                                           # :recv events
        t = names[int(b["type"])]
        p0, p1, mid, irt = int(b["p0"]), int(b["p1"]), int(b["msg_id"]), int(b["in_reply_to"])
        if t == "request_vote":
            f = (p0, p1 & 0xFFFFFFFF, p1 >> 32, mid)
        elif t in ("request_vote_res", "append_entries_res"):
            f = (p0, p1, irt)
        elif t == "append_entries":
            a = np.zeros(4, dtype=np.uint32)
            assert sim.L.or_raft_append(sim.h, int(e["src"]), p1, a.ctypes.data) == 1
            f = (p0, int(a[0]), int(a[1]), int(a[3]), int(a[2]), mid)
        elif t == "init":
            f = (mid,)
        elif t in ("init_ok", "write_ok", "cas_ok"):
            f = (irt,)
        elif t == "read_ok":
            f = (p1, irt)
        elif t == "error":
            f = (p0, irt)
        elif t == "read":
            f = (p0, mid)
        elif t == "write":
            f = (p0, p1, mid)
        elif t == "cas":
            f = (p0, p1 & 0xFFFFFFFF, p1 >> 32, mid)
        else:
            raise AssertionError(t)
        out.append((int(e["msg_id"]), int(e["time_ns"]) // 1_000_000, int(e["src"]), int(e["dest"]), t) + f)
    return out


def run_oracle(fix, ops, events=()):
    n = fix["n"]
    s = O.Sim(n, workload=O.W_RAFT, seed=fix["seed"])
    clients = [s.add_endpoint("c%d" % i) for i in range(n)]
    rows = np.zeros(len(ops), dtype=O.OP_DTYPE)
    for r, (t_ms, src, dest, body) in zip(rows, ops):
        r["time_ns"] = t_ms * 1_000_000
        r["src"] = clients[int(src[1:])]
        r["dest"] = int(dest[1:])
        b = r["body"]
        b["type"] = O.T[body["type"]]
        b["flags"] = O.F_MSG_ID
        b["msg_id"] = body["msg_id"]
        if "key" in body:
            b["p0"] = body["key"]
            if body["type"] == "write":
                b["p1"] = body["value"]
            elif body["type"] == "cas":
                b["p1"] = (body["from"] & 0xFFFFFFFF) | (body["to"] << 32)
    s.schedule(rows)
    for t_ms, what in events:
        s.run(t_ms * 1_000_000)
        if what == "heal":
            s.heal()
        else:                                                  # cut whoever leads now off from the other nodes
            lead = [i for i in range(n) if s.raft_state(i)["state"] == 3]
            s.partition([1 if i in lead[:1] else 0 for i in range(n)])
    s.run(fix["until_ms"] * 1_000_000)
    return s


def check(fix, s):
    n = fix["n"]
    ev, bd = s.journal()
    want = [tuple(m) for m in fix["messages"]]
    got = canonical_from_oracle(s, ev, bd)
    for g, w in zip(got, want):
        assert g == w, (g, w)
    assert len(got) == len(want)
    assert s.round == fix["rounds"]
    state_code = {"nascent": 0, "follower": 1, "candidate": 2, "leader": 3}
    for i, f in enumerate(fix["final"]):
        st = s.raft_state(i)
        assert (st["state"], st["term"], st["commit_index"], st["log_size"], st["kv_size"]) == \
            (state_code[f["state"]], f["term"], f["commit_index"], f["log_size"], len(f["kv"]))
    return want


def test_oracle_sends_what_the_reference_raft_sends():
    import raft_reference_harness as H
    fix = json.load(open(FIXTURE))
    ops, until = H.scenario(None, fix["n"])
    assert until == fix["until_ms"]
    want = check(fix, run_oracle(fix, ops))
    types = {w[4] for w in want}
    assert {"request_vote", "request_vote_res", "append_entries", "append_entries_res", "read_ok", "write_ok",
            "cas_ok", "error", "init_ok"} <= types                          # the trace exercises every handler
    # ...and the proxy path: a follower re-sends the client's message, src unchanged, to the leader
    assert sum(1 for w in want if w[4] in ("read", "write", "cas")) > 24


def test_oracle_matches_the_reference_through_a_partition():
    # 5 nodes, the first leader isolated for 5 s: step-down, a second election, the old leader's
    # uncommitted entries truncated after the heal, late-bound closures slowing its catch-up
    import raft_reference_harness as H
    fix = json.load(open(FIXTURE.replace(".json", "_partition.json")))
    ops, events, until = H.partition_scenario(fix["n"])
    assert until == fix["until_ms"] and [list(e) for e in events] == fix["events"]
    want = check(fix, run_oracle(fix, ops, events))
    terms = {w[5] for w in want if w[4] == "request_vote"}
    assert len(terms) >= 2                                                   # more than one election
    assert any(w[4] == "append_entries_res" and w[6] == 0 for w in want)     # a follower rejected an append


def oracle_for(n, ops, seed):
    s = O.Sim(n, workload=O.W_RAFT, seed=seed)
    clients = [s.add_endpoint("c%d" % q) for q in range(n)]
    rows = np.zeros(len(ops), dtype=O.OP_DTYPE)
    for r, (t_ms, src, dest, body) in zip(rows, ops):
        r["time_ns"] = t_ms * 1_000_000
        r["src"] = clients[int(src[1:])]
        r["dest"] = int(dest[1:])
        b = r["body"]
        b["type"] = O.T[body["type"]]
        b["flags"] = O.F_MSG_ID
        b["msg_id"] = body["msg_id"]
        if "key" in body:
            b["p0"] = body["key"]
            if body["type"] == "write":
                b["p1"] = body["value"]
            elif body["type"] == "cas":
                b["p1"] = (body["from"] & 0xFFFFFFFF) | (body["to"] << 32)
    s.schedule(rows)
    return s


def run_events(s, events, until):
    for t_ms, what in events:
        s.run(t_ms * 1_000_000)
        s.heal()                                             # a new bulk partition replaces the old one
        if what != "heal":
            s.partition(list(what))
    s.run(until * 1_000_000)


def test_frozen_virtual_time_is_reported_not_spun_on():
    # seed 132 of the scenario generator drives a next_index non-positive: the reference's
    # replicate_log then raises before recording the replication and replicates again in every loop
    # iteration -- at latency 0 a message is always due "now" and virtual time stops (DESIGN.md 2.3)
    import raft_reference_harness as H
    n, ops, events, until = H.random_raft_scenario(132)
    s = oracle_for(n, ops, 0x4D41454C)
    with pytest.raises(RuntimeError, match="not advancing"):
        run_events(s, events, until)
    assert s.now < until * 1_000_000


RANDOM = {r["scenario_seed"]: r for r in json.load(open(FIXTURE.replace(".json", "_random.json")))["scenarios"]}


@pytest.mark.parametrize("seed", sorted(RANDOM))
def test_random_scenarios_against_the_executed_reference(seed):
    # random cluster size, client traffic and partitions (arbitrary sides, repeated, healed or not):
    # the oracle must send the messages the reference's raft.py sent under the harness
    import raft_reference_harness as H
    n, ops, events, until = H.random_raft_scenario(seed)
    fix = RANDOM[seed]
    assert (n, until) == (fix["n"], fix["until_ms"])
    want = [tuple(m) for m in fix["messages"]]

    s = oracle_for(n, ops, H.SEED)
    run_events(s, events, until)
    ev, bd = s.journal()
    got = canonical_from_oracle(s, ev, bd)
    for g, w in zip(got, want):
        assert g == w, (g, w)
    assert len(got) == len(want) and s.round == fix["rounds"]
    code = {"nascent": 0, "follower": 1, "candidate": 2, "leader": 3}
    for q, nd in enumerate(fix["final"]):
        st = s.raft_state(q)
        assert (st["state"], st["term"], st["commit_index"], st["log_size"], st["last_applied"]) == \
            (code[nd["state"]], nd["term"], nd["commit_index"], nd["log_size"], nd["last_applied"])
