"""Committed fixtures (tests/golden/): reference_vectors.json = known answers transcribed from the
reference's docs and resources (each with its file:line); journals.json = the oracle's journals
for the named scenarios of tests/golden_cases.py (regenerate: python tests/golden/make_golden.py).
Here the oracle must reproduce both; the engine is held to journals.json by
tests/test_sim_lifecycle.py and tests/test_workload_*.py ([emul] on the CPU emulator, [cuda] on a B200)."""
import json
import os

import numpy as np
import pytest

import golden_cases as G
import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
REF = json.load(open(os.path.join(HERE, "golden", "reference_vectors.json")))
JOURNALS = json.load(open(os.path.join(HERE, "golden", "journals.json")))


def _u32(x):
    return int(x, 16) if isinstance(x, str) else int(x)


# ------------------------------------------------------------------ oracle vs the reference's known answers
def test_oracle_topology_vector():
    want = REF["topology_grid_5"]["neighbors_1_based"]
    for node, nbrs in want.items():
        assert [x + 1 for x in O.topology("grid", 5, int(node) - 1)] == nbrs


@pytest.mark.parametrize("case", REF["flood_sends_per_value"]["cases"], ids=lambda c: "%s%d" % (c["topology"], c["nodes"]))
def test_oracle_flood_counts(case):
    s = O.Sim(case["nodes"], topology=case["topology"], n_values=4)
    c = s.add_endpoint("c0")
    s.send(c, 0, O.body("broadcast", msg_id=1, p0=1))
    s.run(5_000_000)
    assert s.stats()["servers"]["send-count"] == case["sends"]
    # the doc's msgs-per-op is over a 50/50 broadcast/read mix (and a few racing duplicates)
    assert abs(case["sends"] / 2 - case["doc_msgs_per_op"]) / case["doc_msgs_per_op"] < 0.05


def test_oracle_echo_count_and_first_id():
    o = G.make_oracle("echo_12_ops")
    G.CASES["echo_12_ops"][1](o, O.body)
    st = o.stats()
    assert st["all"]["send-count"] == REF["echo_message_count"]["all_sends"]
    assert st["servers"]["send-count"] == REF["echo_message_count"]["server_sends"]
    ev, _ = o.journal()
    assert int(ev["msg_id"][0]) == REF["first_message_id"]["id"]


def test_oracle_gset_replication_count():
    r = REF["gset_replication_count"]
    s = O.Sim(r["nodes"], workload=O.W_GSET, n_values=64, gset_interval_ms=r["interval_ms"])
    for i in range(r["nodes"]):
        c = s.add_endpoint("c%d" % i)
        s.send(c, i, O.body("init", msg_id=1))
    s.run(r["run_ms"] * 1_000_000)
    assert s.stats()["servers"]["msg-count"] == r["server_msgs"]


def test_oracle_philox_vectors():
    for v in REF["philox4x32_10"]["vectors"]:
        out = O.philox([_u32(x) for x in v["ctr"]], [_u32(x) for x in v["key"]])
        assert [int(x) for x in out] == [_u32(x) for x in v["out"]]


def test_error_registry_fixture():
    # error_codes is every {:code :name :definite?} entry of the reference's resources/errors.edn
    from maelstrom_b200 import errors
    want = {int(k): tuple(v) for k, v in REF["error_codes"]["codes"].items()}
    assert errors.ERRORS == want


# ------------------------------------------------------------------ journals
@pytest.mark.parametrize("name", sorted(G.CASES))
def test_oracle_reproduces_committed_journals(name):
    o = G.make_oracle(name)
    G.CASES[name][1](o, O.body)
    ev, bd = o.journal()
    assert G.digest(ev, bd, o.stats(), o.now, o.round) == JOURNALS[name]


# The engine is checked against journals.json in tests/test_sim_lifecycle.py (core cases) and in the
# tests/test_workload_*.py files (the later workloads).
