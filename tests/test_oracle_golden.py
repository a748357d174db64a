"""The CPU restatement (oracle/liblob_oracle.so) against the reference's own outputs.

PINNING: tests/golden/* were produced by the UNMODIFIED reference compiled into oracle/_ref
(tools/make_golden.py).  Everything is compared bitwise.
"""
import ctypes as C

import pytest

import golden_util as G
from rl_markets_b200 import abi, config


def test_golden_step_records_bitwise(oracle):
    for case in G.manifest():
        cfg = G.case_config(case)
        ticks = oracle.lib_generate(cfg, case["env"], case["ticks"])
        port = oracle.run_port(cfg, case["env"], ticks)
        gold, _keep = G.records(case["name"])
        assert port["steps"] >= len(gold) > 100, case["name"]
        for i, g in enumerate(gold):
            bad = abi.record_fields_equal(g, port["records"][i])
            assert not bad, "%s step %d: %r" % (case["name"], i, G.describe_diff(g, port["records"][i], bad))


def test_golden_multi_episode_records_bitwise(oracle):
    """N episodes on one Intraday + one Learner (main.cpp:45-60): HandleTerminal(episode), the same day again, Initialise;
    the first transition of every later episode starts at the previous episode's stale State (serial.cpp:24-25,55,60)."""
    L = oracle.lib()
    for case in G.episode_manifest():
        cfg = G.case_config(case)
        cfg.flow.t0_ms = case["t0_ms"]
        ticks = oracle.lib_generate(cfg, case["env"], case["ticks"])
        h = L.lobo_create(C.byref(cfg), case["env"])
        got = []
        for ep in range(case["episodes"]):
            recs = (abi.StepRecord * case["ticks"])()
            used = C.c_int64()
            n = L.lobo_run(h, ticks, case["ticks"], -1, recs, case["ticks"], C.byref(used))
            assert n > 50 and L.lobo_is_terminal(h) == 1
            got += [recs[i] for i in range(n)]
            L.lobo_handle_terminal(h, ep)  # serial.cpp:79
            L.lobo_reset(h)
        gold, _k = G.records(case["name"])
        assert len(got) == len(gold) == case["n_records"]
        for i, g in enumerate(gold):
            bad = abi.record_fields_equal(g, got[i])
            assert not bad, "%s step %d: %r" % (case["name"], i, G.describe_diff(g, got[i], bad))
        L.lobo_destroy(h)


def test_golden_backtest_records_bitwise(oracle):
    """Train until the close, then main.cpp:216-241 (GoGreedy, a new Intraday, Backtester) -- vs the reference."""
    L = oracle.lib()
    for case in G.backtest_manifest():
        cfg = G.case_config(case)
        cfg.flow.t0_ms = case["t0_ms"]
        h = L.lobo_create(C.byref(cfg), case["env"])
        ticks = oracle.lib_generate(cfg, case["env"], case["ticks"])
        recs = (abi.StepRecord * case["ticks"])()
        used = C.c_int64()
        n1 = L.lobo_run(h, ticks, case["ticks"], -1, recs, case["ticks"], C.byref(used))
        gold, _k = G.records(case["name"])
        assert n1 == len(gold) > 100 and L.lobo_is_terminal(h) == 1
        for i, g in enumerate(gold):
            assert not abi.record_fields_equal(g, recs[i]), (case["name"], "train", i)
        L.lobo_handle_terminal(h, 0)      # Learner::RunEpisode, serial.cpp:79
        L.lobo_go_greedy(h)               # main.cpp:217
        L.lobo_set_backtest(h, 1)
        L.lobo_new_env(h)                 # main.cpp:219
        t = case["test"]
        cfg2 = config.from_dict(case["yaml"], flow_seed=t["flow_seed"])
        cfg2.flow.t0_ms = t["t0_ms"]
        ticks2 = oracle.lib_generate(cfg2, t["env"], t["ticks"])
        recs2 = (abi.StepRecord * t["ticks"])()
        n2 = L.lobo_run(h, ticks2, t["ticks"], -1, recs2, t["ticks"], C.byref(used))
        gold2, _k2 = G.records(case["name"] + "_test")
        assert n2 == len(gold2) > 100 and L.lobo_is_terminal(h) == 1
        for i, g in enumerate(gold2):
            bad = abi.record_fields_equal(g, recs2[i])
            assert not bad, "%s evaluation step %d: %r" % (case["name"], i, G.describe_diff(g, recs2[i], bad))
        st = abi.EnvStats()
        L.lobo_stats(h, C.byref(st))
        s = case["summary"]  # after Runner::RunEpisode's ClearInventory
        assert (st.position, st.episode_pnl, st.episode_reward, st.ask_transactions, st.bid_transactions, st.market_buys,
                st.market_sells) == (s["test_position"], s["test_ep_pnl"], s["test_ep_reward"], s["test_ask_tx"],
                                     s["test_bid_tx"], s["test_market_buys"], s["test_market_sells"])
        L.lobo_destroy(h)


def test_order_vectors(oracle):
    """test/test_Order.cpp scenarios + seeded scripts, values produced by market::Order itself."""
    L = oracle.lib()
    u = G.units()
    # the constants the reference's Catch tests assert (test/test_Order.cpp:193-263)
    by_ops = {(o["size"], o["q_head"], tuple(map(tuple, o["ops"]))): o["out"][-1][:2] for o in u["orders"]}
    assert by_ops[(100, 100, ((2, 500), (1, 50)))] == [91, 459]
    assert by_ops[(100, 100, ((2, 500), (1, 100)))] == [83, 417]
    assert by_ops[(100, 100, ((2, 500), (1, 600)))] == [0, 0]
    assert by_ops[(100, 100, ((2, 5000), (1, 50)))] == [99, 4951]
    assert by_ops[(100, 100, ((2, 5000), (1, 100)))] == [98, 4902]
    for o in u["orders"]:
        n = len(o["ops"])
        ops = (abi.OrderOp * n)(*[abi.OrderOp(op, 0, arg) for op, arg in o["ops"]])
        out = (abi.OrderState * n)()
        L.lobo_order_script(o["size"], o["q_head"], ops, n, out)
        got = [[out[i].q_head, out[i].q_tail, out[i].executed, out[i].ret] for i in range(n)]
        assert got == o["out"], o


def test_market_vectors(oracle):
    """test/test_Market.cpp: ToTicks / ToPrice / tick_size, reference values."""
    L = oracle.lib()
    for m in G.units()["market"]:
        y = config.example_dict()
        cfg = config.from_dict(y, ticker=m["symbol"])
        if m["symbol"] == "AAL.L":
            px = [G.hex_to_double(h) for h in m["px"]]
            assert m["ticks"][px.index(2750.0)] == 52500      # test_Market.cpp:26-27
            assert m["ticks"][px.index(702.1)] == 46021       # test_Market.cpp:42
        assert (cfg.open_ms, cfg.close_ms) == (m["open"], m["close"])
        for h, t, ts in zip(m["px"], m["ticks"], m["tick_size"]):
            p = G.hex_to_double(h)
            assert L.lobo_to_ticks(C.byref(cfg), p) == t, (m["symbol"], p)
            assert G.double_bits(L.lobo_tick_size(C.byref(cfg), p)) == int(ts, 16)
        for t, h in zip(m["tq"], m["price"]):
            assert G.double_bits(L.lobo_to_price(C.byref(cfg), t)) == int(h, 16), (m["symbol"], t)


def test_rolling_mean_vectors(oracle):
    """test/test_Accumulators.cpp: RollingMean<double> mean/var on sliding windows."""
    L = oracle.lib()
    u = G.units()["rolling"]
    # window 3 over 1..8: means 2,3,...; var 1 (test_Accumulators.cpp:8-22)
    mv = [[G.hex_to_double(a), G.hex_to_double(b)] for a, b in u[0]["mean_var"]]
    assert mv[2] == [2.0, 1.0] and mv[5] == [5.0, 1.0]
    for r in u:
        vals = [G.hex_to_double(h) for h in r["vals"]]
        n = len(vals)
        out = (C.c_double * (2 * n))()
        L.lobo_rolling_mean(r["window"], (C.c_double * n)(*vals), n, out)
        for i, (a, b) in enumerate(r["mean_var"]):
            assert G.double_bits(out[2 * i]) == int(a, 16), (r["window"], i)
            vb = G.double_bits(out[2 * i + 1])
            assert vb == int(b, 16) or (out[2 * i + 1] != out[2 * i + 1]), (r["window"], i)  # 0/0 at n==1 is NaN


def test_tile_vectors(oracle):
    """tiles()/hash_UNH through rl::State::populateFeatures: 9 x 96 indices per state."""
    L = oracle.lib()
    for t in G.units()["tiles"]:
        y = config.example_dict(**{"learning.memory_size": t["memory_size"]})
        cfg = config.from_dict(y)
        for c in t["cases"]:
            v = (C.c_float * 8)(*[C.c_float.from_buffer_copy(C.c_uint32(u)).value for u in c["vars"]])
            out = (C.c_int32 * (9 * 96))()
            L.lobo_tiles(C.byref(cfg), v, out)
            assert list(out) == c["features"], t["memory_size"]
    # SURVEY section 8c extra vector: tiles(T=32, M=20e6, {0.5,-100,-100}, int 0) -> 10174999, 12114698, ...
    t20 = [t for t in G.units()["tiles"] if t["memory_size"] == 20000000][0]["cases"][0]["features"]
    assert t20[:4] == [10174999, 12114698, 16498898, 12127300]


def test_generators(oracle):
    """std::mt19937_64 + libstdc++ distributions + glibc rand(), as consumed by policy.cpp / agent.cpp."""
    L = oracle.lib()
    for c in G.units()["rng"]["cases"]:
        s = c["seed"]
        for i in (0, 1, 2, 311, 312, 313, 319):
            assert L.lobo_mt19937_64(s, i) == int(c["mt"][i])
        for i in (0, 1, 17, 39):
            assert G.double_bits(L.lobo_uniform_real(s, i)) == int(c["real"][i], 16)
        for i in (0, 1, 2, 50, 199):
            assert L.lobo_uniform_int(s, 9, i) == c["int9"][i]
        for i in (0, 1, 2, 30, 31, 99):
            assert L.lobo_glibc_rand(s, i) == c["rand"][i]
    assert [c for c in G.units()["rng"]["cases"] if c["seed"] == 1994][0]["rand"][:3] == [1261852369, 322867519, 980044188]


# whole reference runs of 4000 ticks of flow seed 123, env 0: other seeds than the manifest's, the R-learning agents,
# Boltzmann, another venue's tick table and hours, random initial weights
FLOW_SEED_123 = [
    ("double_q_learn", 8192, 31, {}),
    ("online_r_learn", 5003, 7, {"policy.eps_init": 0.2, "learning.beta": 0.02}),
    ("r_learn", 4096, 11, {"policy.type": "boltzmann", "policy.tau_init": 0.08, "policy.tau_floor": 0.01, "policy.tau_T": 10}),
    ("sarsa", 8192, 5, {"reward.measure": "pnl", "data.symbols": ["NOKIA.HE"], "learning.random_init": True}),
]


def flow_seed_123_case(algo, M, seed, over):
    """(fixture name, reference yaml, config) of one FLOW_SEED_123 case."""
    y = config.example_dict(**{"learning.memory_size": M, "learning.algorithm": algo, "debug.random_seed": seed, **over})
    return "flow123_%s_m%d" % (algo, M), y, config.from_dict(y, flow_seed=123)


@pytest.mark.parametrize("algo,M,seed,over", FLOW_SEED_123)
def test_whole_reference_runs_bitwise(oracle, algo, M, seed, over):
    """The restatement against every record of a reference run (tests/golden/digests_flow123_*.bin, tools/make_golden.py)."""
    name, _y, cfg = flow_seed_123_case(algo, M, seed, over)
    ticks = oracle.lib_generate(cfg, 0, 4000)
    port = oracle.run_port(cfg, 0, ticks)
    gold = G.digests(name)
    n = min(len(gold), port["steps"])
    assert n > 800
    bad = [i for i in range(n) if G.record_digest(port["records"][i]) != gold[i]]
    assert not bad, "%s: steps %s differ from the reference's" % (algo, bad[:20])


def test_book_scenarios(oracle):
    """Ask/BidBook::ApplyTransactions, ApplyChanges/UpdateOrder, HandleAdverseSelection, PlaceOrder on
    seeded scenarios run through the reference's own Book classes (test/test_Book.cpp territory)."""
    L = oracle.lib()
    H = G.hex_to_double
    for sc in G.units()["book"]:
        ops, checks = [], []

        def add(op, side=0, px=(), vol=(), n=0, a=0.0, b=0):
            o = oracle.BookOp()
            o.op, o.side, o.n, o.a, o.b = op, side, n, a, b
            for i, p in enumerate(px):
                o.px[i] = p
            for i, v in enumerate(vol):
                o.vol[i] = v
            ops.append(o)
            return len(ops) - 1

        for st in sc["steps"]:
            tx = st.get("tx", [])
            txp, txv = [H(p) for p, _ in tx], [v for _, v in tx]
            if "ref" in st:
                i = add(2, 0, txp, txv, len(tx), H(st["ref"]))
                checks.append((i, "fill", st["au"]))
                i = add(2, 1, txp, txv, len(tx), H(st["ref"]))
                checks.append((i, "fill", st["bu"]))
            add(6, 0, txp, txv, len(tx))
            add(0, 0, [H(p) for p in st["ap"]], st["av"], 5)
            i = add(0, 1, [H(p) for p in st["bp"]], st["bv"], 5)
            if "as" in st:
                i = add(3)
                checks.append((i, "fill", st["as"]))
            if "place" in st:
                add(5, 0)
                add(1, 0, a=H(st["place"][0]), b=st["place"][2])
                add(5, 1)
                i = add(1, 1, a=H(st["place"][1]), b=st["place"][2])
            # order state is read from the last op touching each side
            checks.append((len(ops), "state", st))
            # sentinel no-op reads: op 6 with n=0 keeps `pending` empty for the next step and reports side state
            ia = add(6, 0)
            ib = add(6, 1)
            checks[-1] = (ia, ib, "state", st)
        n = len(ops)
        arr = (oracle.BookOp * n)(*ops)
        out = (oracle.BookResult * n)()
        L.lobo_book_script(arr, n, out)
        for chk in checks:
            if chk[1] == "fill":
                i, _, exp = chk
                assert out[i].r_volume == exp[0]
                assert G.double_bits(out[i].r_proxy) == int(exp[1], 16)
                assert G.double_bits(out[i].r_value) == int(exp[2], 16)
            else:
                ia, ib, _, st = chk
                for idx, key, ntr, tv in ((ia, "ask_o", st["ntr"][0], st["tv"][0]), (ib, "bid_o", st["ntr"][1], st["tv"][1])):
                    r = out[idx]
                    assert r.n_transacted == ntr and r.total_volume == tv
                    if st[key] is None:
                        assert r.order.exists == 0
                    else:
                        p, qa, qb, rem = st[key]
                        assert r.order.exists == 1 and G.double_bits(r.order.price) == int(p, 16)
                        assert (r.order.q_head, r.order.q_tail) == (qa, qb)
