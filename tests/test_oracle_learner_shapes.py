"""The CPU restatement against whole reference runs away from the example config: 1..7 actions, gamma*lambda of 0, 0.96
and 1, an explicit trace_cap, memory_size 1, 2, 6002 and 8192..65536 (tests/golden/learner_shapes.json, tools/make_golden.py).

These runs are what tests/test_gpu_learner_shapes.py holds the CUDA learners to, so each case also checks that it still
covers the path it is there for: the longest trace list of the run stays inside the case's bounds.
"""
import pytest

import golden_util as G

CASES = G.learner_shapes()


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_learner_shape_runs_bitwise(oracle, case):
    cfg = G.case_config(case)
    port = oracle.run_port(cfg, case["env"], oracle.lib_generate(cfg, case["env"], case["ticks"]))
    gold = G.digests(case["name"])
    assert port["steps"] >= len(gold) == case["n_records"] > 500, (case["name"], port["steps"], len(gold))
    bad = [i for i in range(len(gold)) if G.record_digest(port["records"][i]) != gold[i]]
    assert not bad, "%s: steps %s differ from the reference's" % (case["name"], bad[:20])
    longest = max(r.n_traces for r in port["records"])
    assert longest >= case.get("min_traces", 1), (case["name"], longest)
    assert longest <= case.get("max_traces", longest), (case["name"], longest)


def test_cases_cover_the_learner_paths():
    """The cases are chosen for the branches they reach; this keeps the set from drifting away from them."""
    by = {c["name"]: c for c in CASES}
    assert sorted({c["yaml"]["learning"]["n_actions"] for c in CASES}) == [1, 2, 3, 4, 5, 7, 9]
    staged = [n for n, c in by.items() if "double" not in c["algo"] and c["M"] * 8 <= 65536 and c["M"] % 2 == 0]
    assert {"a1_q_m8192", "a2_sarsa_m2", "a5_q_m6002"} <= set(staged)
    assert by["a5_q_m6002"]["M"] & (by["a5_q_m6002"]["M"] - 1)  # staged, not a power of two: the mod_m path
    assert by["m1_q"]["M"] == 1
    assert all(by[n]["yaml"]["learning"]["lambda"] == 0.0 for n in ("lam0_q", "lam0_sarsa"))
    gl1 = by["gl1_sarsa_m8192"]
    assert gl1["yaml"]["learning"]["gamma"] * gl1["yaml"]["learning"]["lambda"] >= 1.0 and gl1["trace_cap"] >= gl1["M"]
    assert by["longtr_sarsa_m65536"]["min_traces"] > 4 * 512  # several drains of the 512-entry update table per step
