"""Compact gossip records in the inbox rings (DESIGN.md 3.1): server -> neighbor gossip is written as its
16-byte order key alone, every other message as key + 32-byte body.  These scenarios put compact and
full records side by side in the situations a reader could get wrong, and compare the journal (bodies
included, journal level 2) with the oracle's.  Each runs [emul] in the CPU suite and [cuda] on the GPU."""
import numpy as np
import pytest

import oracle_lib as O
from scenarios import assert_same_journal, both, make_pair, random_broadcast_ops
from test_emul_sharded import check_against_oracle, run_sharded_scenario

pytestmark = pytest.mark.usefixtures("engine_backend")


def test_mixed_windows_wrapping_small_rings():
    # Closed-loop clients that re-send within the same tick (interval 1 ns: half of the next ops are due at
    # once) put full client requests into the windows that also carry the flood's compact gossip.  Server
    # rings of 128 slots wrap dozens of times, so the body plane under a compact key holds whatever full
    # record an earlier lap left there: a reader that took the body of a compact slot would journal it.
    n = 16
    g, o = make_pair(n, topology="grid", n_values=1 << 14, ring_cap=512, max_window=256,
                     server_ring_cap=128, server_max_window=128, journal_cap_log2=20)

    def scenario(s, body):
        s.add_gen_clients(48, interval_ns=1, time_limit_ns=12_000_000, read_permille=300, timeout_ns=50_000_000,
                          quiet_ns=2_000_000, first_name=0)
        s.run(16_000_000)
        return [s.node_set(k).tolist() for k in range(n)]

    sets_g, sets_o = both(g, o, scenario)
    assert sets_g == sets_o and len(sets_g[0]) > 0
    hg, ho = g.history(), o.history()
    assert len(hg) == len(ho) > 0
    for f in ("time_ns", "order", "client", "op", "type", "f", "error", "value"):
        assert np.array_equal(hg[f], ho[f]), f
    ev, _ = assert_same_journal(g, o)
    # a :send and a :recv per delivery: the server rings wrapped 10 times over on average
    assert np.count_nonzero(ev["dest"] < n) > 20 * 128 * n


def test_bitonic_fallback_windows_with_compact_gossip():
    # 72 closed-loop clients per node: a node's window holds one sender block per client that sent in the
    # previous round next to its neighbors' compact gossip, more than the 64 blocks of the fast ordering
    # path, so the window is ordered by the bitonic sort and every record is read back through ring_load.
    n = 9
    g, o = make_pair(n, topology="grid", n_values=1 << 15, ring_cap=2048, max_window=2048,
                     server_ring_cap=4096, server_max_window=2048, max_endpoints=n + 72 * n, journal_cap_log2=21)

    def scenario(s, body):
        s.add_gen_clients(72 * n, interval_ns=1, time_limit_ns=3_000_000, read_permille=250, timeout_ns=50_000_000,
                          quiet_ns=1_000_000, first_name=0)
        s.run(5_000_000)

    both(g, o, scenario)
    hg, ho = g.history(), o.history()
    assert len(hg) == len(ho) > 0
    for f in ("time_ns", "order", "client", "op", "type", "f", "error", "value"):
        assert np.array_equal(hg[f], ho[f]), f
    assert_same_journal(g, o)
    assert g.counters()["fallback_sorts"] > 0


def test_partition_in_force_while_gossip_queued():
    # Pair drops and a bulk partition cut compact gossip at dequeue: the receiver takes the sender from the
    # ticket in the key, not from a body.
    n = 16
    g, o = make_pair(n, topology="grid", n_values=1024, ring_cap=1024, max_window=512,
                     server_ring_cap=128, server_max_window=128)

    def scenario(s, body):
        cs = [s.add_endpoint("c%d" % i) for i in range(3)]
        ops, _ = random_broadcast_ops(n, cs, n_ticks=60, per_tick=6, seed=11)
        s.schedule(ops)
        s.run(8_000_000)
        for a in range(0, 8):
            for b in range(8, 16):
                s.drop(a, b)
        s.run(20_000_000)
        s.heal()
        s.run(30_000_000)
        s.partition([0, 0, 1, 1] * 4)
        s.run(45_000_000)
        s.heal()
        s.run(70_000_000)

    both(g, o, scenario)
    assert_same_journal(g, o)
    assert g.counters()["partition_drops"] > 0


def test_two_emulated_shards_small_rings(engine_backend):
    # gossip across the shard boundary lands as compact keys in the peer's ring, whose body plane starts
    # ring_slots vectors into that peer's allocation
    if engine_backend != "emul":
        pytest.skip("emulated shards (one process): the CPU suite; multi-GPU runs are tests/test_gpu_sharded.py")
    n = 16
    kw = dict(topology="grid", n_values=1024, max_endpoints=n + 8, ring_cap=512, max_window=256,
              server_ring_cap=64, server_max_window=64)

    def scenario(s, body):
        cs = [s.add_endpoint("c%d" % i) for i in range(2)]
        ops, _ = random_broadcast_ops(n, cs, n_ticks=40, per_tick=8, seed=5)
        s.schedule(ops)
        s.run(45_000_000)

    ev, st, now, rnd = run_sharded_scenario(2, n, kw, scenario)
    o = O.Sim(n, workload=O.W_BROADCAST, topology="grid", n_values=1024)
    check_against_oracle(o, scenario, ev, st, now, rnd)
    assert np.count_nonzero(ev["dest"] < n) > 2 * 8 * 64 * n     # a :send and a :recv per delivery: 8 laps
