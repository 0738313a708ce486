"""Runs the reference's own Raft node, demo/python/raft.py of jepsen-io/maelstrom, UNMODIFIED, as a
cluster inside this process and records every message it sends -- the trace the oracle's
restatement (oracle/oracle.cpp node_raft / raft_actions) is pinned to.

raft.py is a script: it ends with `RaftNode().main()`, an endless loop over stdin / wall clock /
random.  The harness execs its source once per node with that last line removed (nothing else is
touched) in a namespace whose `time`, `random`, `select` and `sys` are stand-ins, and then drives
each node with the reference's own methods under the schedule DESIGN.md section 2.8 specifies:
per round and node, every due message through `net.process_msg()`, then one pass of
`step_down_on_timeout`, `replicate_log`, `election`, `advance_commit_index`, and
`advance_state_machine` until the commit index is reached -- inside one try/except, like the
body of the reference's main loop (raft.py:577-588).  `time.time()` is the virtual clock
and `random.random()` the k-th Philox draw of the node's step (the oracle's raft_draw), both as
exact rationals so that the reference's comparisons are made without float rounding; messages get
ids in emission order and are delivered in id order in the next round (latency 0, no loss).

Needs a checkout of jepsen-io/maelstrom; what it produces is committed under tests/golden/
(python tests/golden/raft_reference_harness.py <maelstrom checkout>): raft_reference_trace.json,
raft_reference_trace_partition.json and raft_reference_trace_random.json (the random scenarios of
random_raft_scenario for seeds RANDOM_SEEDS).
"""
import json
import os
import sys
import types
from fractions import Fraction

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
RAFT_PY = None                                                       # set by main()
SEED = 0x4D41454C
RANDOM_SEEDS = range(8)


class Node:
    def __init__(self, cluster, index):
        self.cluster, self.index = cluster, index
        self.inbox, self.draws = [], 0
        src = open(RAFT_PY).read()
        assert src.rstrip().endswith("RaftNode().main()")
        src = src.rstrip()[:-len("RaftNode().main()")]                 # the only change: do not enter the loop
        node = self
        # exact rationals, not floats: the spec's clock arithmetic is exact (integer ns), and on a real
        # clock a float tie such as 4.121 - 3.121 == 1.0000000000000004 has probability zero
        fake_time = types.SimpleNamespace(time=lambda: Fraction(cluster.now_ns, 10 ** 9), sleep=lambda s: None)
        fake_random = types.SimpleNamespace(random=lambda: node.draw())
        stdin = types.SimpleNamespace(readline=lambda: node.inbox.pop(0))
        stdout = types.SimpleNamespace(write=lambda s: node.out(s), flush=lambda: None)
        stderr = types.SimpleNamespace(write=lambda s: None, flush=lambda: None)
        fake_sys = types.SimpleNamespace(stdin=stdin, stdout=stdout, stderr=stderr)
        fake_select = types.SimpleNamespace(select=lambda r, w, x, t: ([stdin] if node.inbox else [], [], []))
        ns = {"__name__": "raft_reference"}
        code = compile(src, RAFT_PY, "exec")
        exec(code, ns)                                                   # defines Net, Log, KVStore, RaftNode
        ns["time"], ns["random"], ns["select"], ns["sys"] = fake_time, fake_random, fake_select, fake_sys
        self.raft = ns["RaftNode"]()
        self.partial = ""

    def draw(self):
        import oracle_lib as O
        x = O.philox([0x80000000 | self.draws, self.index, self.cluster.round & 0xFFFFFFFF, self.cluster.round >> 32],
                     [SEED & 0xFFFFFFFF, SEED >> 32])[0]
        self.draws += 1
        return Fraction(x, 1 << 32)

    def out(self, s):                                                    # json.dump writes in pieces, then '\n'
        self.partial += s
        while "\n" in self.partial:
            line, self.partial = self.partial.split("\n", 1)
            if line.strip():
                self.cluster.send(json.loads(line))

    def step(self, due):
        self.draws = 0
        r = self.raft
        for msg in due:
            self.inbox.append(json.dumps(msg) + "\n")
            try:
                r.net.process_msg()
            except Exception:                                            # raft.py:585-588
                self.inbox.clear()
        try:
            r.step_down_on_timeout()
            r.replicate_log()
            r.election()
            r.advance_commit_index()
            while r.last_applied < r.commit_index:
                r.advance_state_machine()
        except Exception:
            pass


class Cluster:
    def __init__(self, n):
        self.n, self.now_ns, self.round, self.next_id = n, 0, 0, 0
        self.nodes = [Node(self, i) for i in range(n)]
        self.pending, self.trace, self.client_inbox = [], [], []
        self.host_queue = []
        self.component = None                                            # bulk partition: node index -> side

    def send(self, msg):
        msg = dict(msg)
        msg["id"] = self.next_id
        self.next_id += 1
        self.trace.append({"t_ms": self.now_ns // 1_000_000, "round": self.round, **msg})
        self.sent_this_round.append(msg)

    def client_send(self, src, dest, body):
        self.host_queue.append({"src": src, "dest": dest, "body": body})

    def run_round(self):
        self.sent_this_round = []
        for m in self.host_queue:                                        # injector first (DESIGN.md 2.3)
            self.send(m)
        self.host_queue = []
        due, self.pending = self.pending, []
        if self.component is not None:                                   # cut at dequeue, silently (net.clj:234)
            side = lambda name: self.component[int(name[1:])] if name[0] == "n" else None
            due = [m for m in due if side(m["src"]) is None or side(m["dest"]) is None or side(m["src"]) == side(m["dest"])]
        for i, node in enumerate(self.nodes):
            node.step([m for m in due if m["dest"] == "n%d" % i])
        self.client_inbox += [m for m in due if m["dest"].startswith("c")]
        self.pending = self.sent_this_round
        self.round += 1
        if not self.pending:
            self.now_ns += 1_000_000

    def run(self, until_ms):
        while self.now_ns < until_ms * 1_000_000:
            self.run_round()


def scenario(cluster_or_none, n=3):
    """The scripted run both sides execute: returns the list of (time_ms, client, dest, body) host sends."""
    ops = [(0, "c%d" % i, "n%d" % i, {"type": "init", "msg_id": 1, "node_id": "n%d" % i,
                                      "node_ids": ["n%d" % k for k in range(n)]}) for i in range(n)]
    t = 4300
    k = 1
    last = {}                                                            # what each key holds if every op commits in order
    for rep in range(8):
        for dest in range(n):
            k += 1
            kind = (rep + dest) % 3
            key = rep % 2
            body = {"msg_id": k, "key": key}
            if kind == 0:
                body.update(type="write", value=10 * rep + dest)
                last[key] = body["value"]
            elif kind == 1:
                body.update(type="read")
            else:                                                        # every other cas expects the right value
                frm = last.get(key, 7) if rep % 2 else 999
                body.update({"type": "cas", "from": frm, "to": 100 + rep})
                if frm == last.get(key):
                    last[key] = 100 + rep
            ops.append((t, "c%d" % dest, "n%d" % dest, body))
        t += 40
    return ops, t + 1300                                                 # a heartbeat after the last op


def partition_scenario(n=5):
    """5 nodes; whoever leads at 4.5 s is cut off from the others until 9.5 s; clients keep writing
    through every node.  Returns (ops, events, until_ms); events = [(time_ms, "isolate-leader" | "heal")]."""
    ops = [(0, "c%d" % i, "n%d" % i, {"type": "init", "msg_id": 1, "node_id": "n%d" % i,
                                      "node_ids": ["n%d" % k for k in range(n)]}) for i in range(n)]
    k = 1
    for rep in range(12):
        t = 4300 + 600 * rep
        for dest in range(n):
            k += 1
            body = {"msg_id": k, "key": dest % 3}
            if (rep + dest) % 2:
                body.update(type="write", value=100 * rep + dest)
            else:
                body.update(type="read")
            ops.append((t, "c%d" % dest, "n%d" % dest, body))
    return ops, [(4500, "isolate-leader"), (9500, "heal")], 12500


def run(n, ops, events, until):
    c = Cluster(n)
    i = j = 0
    while c.now_ns < until * 1_000_000:
        while j < len(events) and events[j][0] * 1_000_000 <= c.now_ns:
            if events[j][1] == "heal":
                c.component = None
            else:
                lead = [k for k, nd in enumerate(c.nodes) if nd.raft.state == "leader"]
                c.component = [1 if k in lead[:1] else 0 for k in range(n)]
            j += 1
        while i < len(ops) and ops[i][0] * 1_000_000 <= c.now_ns:
            c.client_send(ops[i][1], ops[i][2], ops[i][3])
            i += 1
        c.run_round()
    return c


def random_raft_scenario(seed):
    """(n, ops, events, until_ms): random cluster size, client traffic (with a second `init` now and
    then) and bulk partitions that come, change and sometimes heal."""
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 6))
    ops = [(0, "c%d" % i, "n%d" % i, {"type": "init", "msg_id": 1, "node_id": "n%d" % i,
                                      "node_ids": ["n%d" % k for k in range(n)]}) for i in range(n)]
    until = int(rng.integers(5000, 12000))
    k = 1
    times = sorted(int(t) for t in rng.integers(0, until, size=int(rng.integers(5, 60))))
    for t in times:
        k += 1
        dest = int(rng.integers(n))
        kind = int(rng.integers(4))
        body = {"msg_id": k, "key": int(rng.integers(3))}
        if kind == 0:
            body.update(type="read")
        elif kind == 1:
            body.update(type="write", value=int(rng.integers(5)))
        elif kind == 2:
            body.update({"type": "cas", "from": int(rng.integers(5)), "to": int(rng.integers(5))})
        else:
            body = {"msg_id": k, "type": "init", "node_id": "n%d" % dest, "node_ids": []}    # "Can't init twice!"
        ops.append((t, "c%d" % int(rng.integers(n)), "n%d" % dest, body))
    events = []
    for t in sorted(int(t) for t in rng.integers(2000, until, size=int(rng.integers(0, 5)))):
        events.append((t, "heal" if rng.integers(3) == 0 else [int(x) for x in rng.integers(0, 2, size=n)]))
    return n, ops, events, until


def run_random(n, ops, events, until):
    """A random_raft_scenario on the reference: bulk partitions with arbitrary sides, repeated, healed or
    not.  None when virtual time freezes: some next_index went non-positive, replicate_log now raises
    before it records the replication and so replicates again in every loop iteration; at latency 0
    that freezes virtual time (DESIGN.md 2.3).  The oracle gives up the same way (or_run)."""
    c = Cluster(n)
    i = j = 0
    while c.now_ns < until * 1_000_000:
        while j < len(events) and events[j][0] * 1_000_000 <= c.now_ns:
            c.component = None if events[j][1] == "heal" else list(events[j][1])
            j += 1
        while i < len(ops) and ops[i][0] * 1_000_000 <= c.now_ns:
            c.client_send(ops[i][1], ops[i][2], ops[i][3])
            i += 1
        c.run_round()
        if c.round > until + 30_000:
            return None
    return c


def canonical(m, n):
    """One sent message as a flat tuple: (id, time_ms, src, dest, type, fields...); endpoints as the
    engine numbers them (servers 0..n-1, then clients)."""
    def ep(name):
        return int(name[1:]) if name[0] == "n" else n + int(name[1:])
    b = m["body"]
    t = b["type"]
    if t == "request_vote":
        f = (b["term"], b["last_log_index"], b["last_log_term"], b["msg_id"])
    elif t == "request_vote_res":
        f = (b["term"], int(b["vote_granted"]), b["in_reply_to"])
    elif t == "append_entries":
        f = (b["term"], b["prev_log_index"], b["prev_log_term"], len(b["entries"]), b["leader_commit"], b["msg_id"])
    elif t == "append_entries_res":
        f = (b["term"], int(b["success"]), b["in_reply_to"])
    elif t == "init":
        f = (b["msg_id"],)
    elif t in ("init_ok", "write_ok", "cas_ok"):
        f = (b["in_reply_to"],)
    elif t == "read_ok":
        f = (b["value"], b["in_reply_to"])
    elif t == "error":
        f = (b["code"], b["in_reply_to"])
    elif t == "read":
        f = (b["key"], b["msg_id"])
    elif t == "write":
        f = (b["key"], b["value"], b["msg_id"])
    elif t == "cas":
        f = (b["key"], b["from"] & 0xFFFFFFFF, b["to"], b["msg_id"])
    else:
        raise AssertionError(t)
    return [m["id"], m["t_ms"], ep(m["src"]), ep(m["dest"]), t] + [int(x) for x in f]


def dump(c, n, until, name, extra=None):
    states = [{"state": nd.raft.state, "term": nd.raft.current_term, "commit_index": nd.raft.commit_index,
               "log_size": nd.raft.log.size(), "kv": {str(k): v for k, v in nd.raft.state_machine.state.items()}}
              for nd in c.nodes]
    out = {"reference": "demo/python/raft.py", "n": n, "seed": SEED, "until_ms": until, "rounds": c.round,
           "messages": [canonical(m, n) for m in c.trace], "final": states}
    out.update(extra or {})
    with open(os.path.join(HERE, name), "w") as f:                      # one message per line
        head = {k: v for k, v in out.items() if k != "messages"}
        f.write(json.dumps(head, sort_keys=True)[:-1] + ', "messages": [\n')
        f.write(",\n".join(json.dumps(m) for m in out["messages"]))
        f.write("\n]}\n")
    print(name, "messages", len(c.trace), "rounds", c.round, "final", [(x["state"], x["term"], x["log_size"]) for x in states])


def dump_random(name):
    with open(os.path.join(HERE, name), "w") as f:                      # one message per line
        f.write('{"reference": "demo/python/raft.py", "seed": %d, "scenarios": [\n' % SEED)
        for k, seed in enumerate(RANDOM_SEEDS):
            n, ops, events, until = random_raft_scenario(seed)
            c = run_random(n, ops, events, until)
            assert c is not None, "seed %d freezes virtual time: pick other seeds" % seed
            final = [{"state": nd.raft.state, "term": nd.raft.current_term, "commit_index": nd.raft.commit_index,
                      "log_size": nd.raft.log.size(), "last_applied": nd.raft.last_applied} for nd in c.nodes]
            head = {"scenario_seed": seed, "n": n, "until_ms": until, "rounds": c.round, "final": final}
            f.write(",\n" if k else "")
            f.write(json.dumps(head, sort_keys=True)[:-1] + ', "messages": [\n')
            f.write(",\n".join(json.dumps(canonical(m, n)) for m in c.trace))
            f.write("\n]}")
            print(name, "seed", seed, "messages", len(c.trace), "rounds", c.round)
        f.write("\n]}\n")


def main(maelstrom_checkout):
    global RAFT_PY
    RAFT_PY = os.path.join(maelstrom_checkout, "demo", "python", "raft.py")
    n = 3
    ops, until = scenario(None, n)
    dump(run(n, ops, [], until), n, until, "raft_reference_trace.json")
    ops, events, until = partition_scenario(5)
    dump(run(5, ops, events, until), 5, until, "raft_reference_trace_partition.json", {"events": events})
    dump_random("raft_reference_trace_random.json")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/raft_reference_harness.py <jepsen-io/maelstrom checkout>")
    main(sys.argv[1])
