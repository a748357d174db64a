"""The CUDA learners away from the example config, bitwise against the reference and the CPU restatement.

The other parity tests run 9 actions, gamma*lambda ~ 0.83 (trace lists under ~800 entries) and a handful of table sizes.
The kernels branch on all three: the action count masks gathers, Q stores and the tile -> last-writer table, and it is
part of every tile hash; trace lists are drained through the one-warp learner's update table 512 entries at a time (and
skipped when the decay rate is 0); the learner itself is chosen per handle from the table size and the batch size.
Here every case of tests/golden/learner_shapes.json runs on a small batch on several kernel paths, its first env against
every record of the reference run and every env against the restatement (records, both weight tables, stats, counters).
Then the learner-selection boundaries at size, and the error flags of the trace lists.
"""
import ctypes as C

import numpy as np
import pytest

import golden_util as G
from rl_markets_b200 import abi, config

pytestmark = pytest.mark.gpu

CASES = {c["name"]: c for c in G.learner_shapes()}
N_ENVS = 6


def _staged(algo, M):
    """rlm_create's choice of the staged learner (whole table in shared memory) for independent policies."""
    return "double" not in algo and M * 8 <= 65536 and M % 2 == 0


def _matrix():
    out = []
    for name, c in CASES.items():
        paths = [("default", {}), ("agent3", {"RLM_AGENT_VARIANT": "3"}), ("agent1", {"RLM_AGENT_VARIANT": "1"})]
        if _staged(c["algo"], c["M"]):
            paths.append(("unstaged", {"RLM_STAGED": "0"}))
        if c["algo"] in ("q_learn", "sarsa", "double_q_learn"):
            paths += [("fused", {"RLM_ENGINE": "F"}), ("rounds_cap1", {"RLM_ROUNDS": "1", "RLM_ROUND_CAP": "1"}),
                      ("env_thread", {"RLM_ENV_VARIANT": "1"})]
        out += [pytest.param(name, env, id="%s-%s" % (name, label)) for label, env in paths]
    return out


def _port(oracle, cfg, env, n_ticks):
    """One env on the restatement: records, stats, sum of trace lengths, rho, and each weight table as (the indices the run
    touched, their bits) -- read in place through lobo_theta, so that tables of 2^27 weights are not copied whole."""
    L = oracle.lib()
    ticks = oracle.generate_ticks(cfg, env, n_ticks)
    h = L.lobo_create(C.byref(cfg), env)
    assert h, "lobo_create failed"
    try:
        recs = (abi.StepRecord * n_ticks)()
        used = C.c_int64(0)
        steps = L.lobo_run(h, ticks, n_ticks, -1, recs, n_ticks, C.byref(used))
        assert steps > 0, "lobo_run: %d" % steps
        st = abi.EnvStats()
        L.lobo_stats(h, C.byref(st))
        tables = []
        for t in (0, 1):
            p = L.lobo_theta(h, t)
            if not p:
                break
            w = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint64)), shape=(cfg.memory_size,))
            idx = np.flatnonzero(w)
            tables.append((idx, w[idx].copy()))
        return {"records": [recs[i] for i in range(steps)], "_keep": recs, "steps": steps, "stats": st,
                "sum_traces": L.lobo_sum_traces(h), "rho": L.lobo_rho(h), "tables": tables}
    finally:
        L.lobo_destroy(h)


_PORT_CACHE = {}


def _port_cached(oracle, case, cfg, b):
    key = (case["name"], b)
    if key not in _PORT_CACHE:
        _PORT_CACHE[key] = _port(oracle, cfg, cfg.env_index0 + b, case["ticks"])
    return _PORT_CACHE[key]


def _compare_records(got, want, label):
    assert len(got) == len(want), "%s: %d steps, the restatement %d" % (label, len(got), len(want))
    for i, (g, w) in enumerate(zip(got, want)):
        bad = abi.record_fields_equal(g, w)
        assert not bad, "%s step %d (cuda, restatement): %r" % (label, i, G.describe_diff(g, w, bad))


def _compare_env(m, b, port, label):
    """Records, every weight of every table, stats and rho of env b against the restatement, bitwise."""
    recs, _keep = m.records(b)
    _compare_records(recs, port["records"], label)
    assert len(port["tables"]) == (2 if m.cfg.algorithm in (abi.ALGO["double_q_learn"], abi.ALGO["double_r_learn"]) else 1)
    for t, (idx, bits) in enumerate(port["tables"]):
        assert idx.size > 0, "%s: the run wrote no weight" % label
        w = np.frombuffer(m.theta(b, t), dtype=np.uint64)
        assert np.count_nonzero(w) == idx.size, "%s table %d: %d weights written, the restatement %d" % (
            label, t, np.count_nonzero(w), idx.size)
        diff = np.flatnonzero(w[idx] != bits)
        assert diff.size == 0, "%s table %d: weights %s differ" % (label, t, idx[diff[:10]].tolist())
    got, want = m.stats(b, 1)[0], port["stats"]
    for f, _t in abi.EnvStats._fields_:
        assert getattr(got, f) == getattr(want, f), "%s stats.%s: cuda %r, restatement %r" % (label, f, getattr(got, f),
                                                                                            getattr(want, f))
    assert m.rho()[b] == port["rho"], label


@pytest.mark.parametrize("name,env_vars", _matrix())
def test_learner_shapes_match_reference_and_oracle(rlm, oracle, monkeypatch, name, env_vars):
    case = CASES[name]
    for k, v in env_vars.items():
        monkeypatch.setenv(k, v)
    cfg = G.case_config(case, n_envs=N_ENVS, env_index0=case["env"])  # local env 0 is the reference run's env
    cfg.record_envs = N_ENVS
    cfg.record_cap = case["ticks"]  # at most one step per tick
    m = rlm.BatchedMarket(cfg)
    m.run_ticks(case["ticks"])
    m.sync()  # also: no device error flag (a trace list outgrowing the derived or explicit trace_cap raises here)
    recs, _keep = m.records(0)
    gold = G.digests(name)
    assert len(recs) >= len(gold) == case["n_records"], (name, len(recs), len(gold))
    bad = [i for i in range(len(gold)) if G.record_digest(recs[i]) != gold[i]]
    assert not bad, "%s %r: steps %s differ from the reference's" % (name, env_vars, bad[:20])
    ports = [_port_cached(oracle, case, cfg, b) for b in range(N_ENVS)]
    for b, port in enumerate(ports):
        _compare_env(m, b, port, "%s %r env %d" % (name, env_vars, b))
    c = m.counters()
    assert c.steps == sum(p["steps"] for p in ports)
    assert c.ticks == N_ENVS * (case["ticks"] - 1)  # the first row only opens the market
    assert c.sum_traces == sum(p["sum_traces"] for p in ports)
    m.close()


def _mk(algo, M, n_envs, flow_seed, n_ticks, trace_cap=0, **over):
    y = config.example_dict(**{"learning.memory_size": M, "learning.algorithm": algo, **over})
    cfg = config.from_dict(y, n_envs=n_envs, flow_seed=flow_seed)
    cfg.trace_cap = trace_cap
    cfg.record_envs = n_envs
    cfg.record_cap = n_ticks
    return cfg


def _run_and_compare(rlm, oracle, cfg, n_ticks, check_envs, label):
    m = rlm.BatchedMarket(cfg)
    m.run_ticks(n_ticks)
    m.sync()
    for b in check_envs:
        port = _port(oracle, cfg, b, n_ticks)
        assert port["steps"] > 100
        _compare_env(m, b, port, "%s env %d" % (label, b))
        del port
    c = m.counters()
    assert c.ticks == cfg.n_envs * (n_ticks - 1)
    m.close()


@pytest.mark.parametrize("M", [8192, 8194, 8191])
def test_staged_learner_size_boundary(rlm, oracle, M):
    """8192 weights (64 KB) is the largest staged table; 8194 is even but too large, 8191 odd: both take the one-warp
    learner."""
    cfg = _mk("q_learn", M, 5, 41, 1500, **{"learning.n_actions": 5})
    _run_and_compare(rlm, oracle, cfg, 1500, range(5), "q_learn A=5 M=%d" % M)


def _mem_available_gb():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 2 ** 20
    return 0.0


@pytest.mark.parametrize("M", [1 << 27, (1 << 27) + 1])
def test_largest_tables_either_side_of_the_packed_tile_table(rlm, oracle, M):
    """The one-warp learners pack (feature << 4 | action) into one word, so memory_size above 2^27 is forced onto the
    three-warp learner (and off the fused engine).  2^27 is the largest table the one-warp learner takes."""
    # the restatement holds ~13 bytes per weight, the device table read back 8 more
    need_gb = 21 * M / 2 ** 30 + 2
    if _mem_available_gb() < need_gb:
        pytest.skip("needs %.1f GB of free host memory" % need_gb)
    cfg = _mk("q_learn", M, 2, 43, 1200)
    _run_and_compare(rlm, oracle, cfg, 1200, range(2), "q_learn M=%d" % M)


@pytest.mark.parametrize("n_envs", [16384, 16385])
def test_batch_size_boundary(rlm, oracle, n_envs):
    """Above 16 384 envs the thread-per-env tick kernel and the three-warp learner take over (unless the table is staged);
    envs at both ends of the batch, the last one included."""
    n_ticks = 700
    cfg = _mk("q_learn", 16384, n_envs, 47, n_ticks, **{"learning.n_actions": 5})
    cfg.record_cap = 400  # (~200 steps in 700 ticks; a longer run would show as a step count below the restatement's)
    _run_and_compare(rlm, oracle, cfg, n_ticks, [0, 1, 8191, n_envs - 2, n_envs - 1], "q_learn A=5 B=%d" % n_envs)


@pytest.mark.parametrize("M,env_vars", [
    (16384, {}),                          # one-warp learner
    (8192, {}),                           # staged learner
    (16384, {"RLM_AGENT_VARIANT": "3"}),  # three-warp learner
    (16384, {"RLM_AGENT_VARIANT": "1"}),  # one warp per env, round-1 kernel
    (16384, {"RLM_ENGINE": "F"}),         # fused persistent engine
], ids=["default", "staged", "agent3", "agent1", "fused"])
def test_trace_list_overflow_is_reported(rlm, oracle, monkeypatch, M, env_vars):
    """trace_cap = 64 against lists of ~800 entries: the lists are cut at the cap, the run goes on, and sync() reports it.
    Up to the first step whose list outgrows the cap, the records are still the restatement's."""
    for k, v in env_vars.items():
        monkeypatch.setenv(k, v)
    n_envs, n_ticks = 4, 1500
    cfg = _mk("sarsa", M, n_envs, 53, n_ticks, trace_cap=64)
    m = rlm.BatchedMarket(cfg)
    m.run_ticks(n_ticks)
    with pytest.raises(rlm.RlmError) as ei:
        m.sync()
    assert ei.value.code == abi.RLM_ERR_RUNTIME and "trace list overflow" in str(ei.value), str(ei.value)
    c = m.counters()
    assert c.ticks == n_envs * (n_ticks - 1)
    for b in range(n_envs):
        port = _port(oracle, cfg, b, n_ticks)
        recs, _keep = m.records(b)
        over = next(i for i, r in enumerate(port["records"]) if r.n_traces > 64)
        assert 0 < over < len(recs)
        _compare_records(recs[:over], port["records"][:over], "sarsa trace_cap 64 %r env %d" % (env_vars, b))
        assert recs[over].n_traces == 64
    m.close()


def test_gamma_lambda_of_one_needs_a_trace_cap(rlm):
    """No decay ever drops an entry: the list length cannot be derived from gamma*lambda."""
    cfg = _mk("sarsa", 8192, 2, 5, 100, **{"learning.gamma": 1.0, "learning.lambda": 1.0})
    with pytest.raises(rlm.RlmError) as ei:
        rlm.BatchedMarket(cfg)
    assert ei.value.code == abi.RLM_ERR_UNSUPPORTED and "trace_cap" in str(ei.value)
