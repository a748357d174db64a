#!/usr/bin/env python3
"""Generate tests/golden/* from the UNMODIFIED reference compiled into oracle/_ref (run in the
build container, where /root/reference exists; the fixtures are committed so that the GPU box,
which has no reference tree, can check against them).

  tests/golden/units.json          reference unit-level vectors (oracle/_ref/ref_units)
  tests/golden/steps_<name>.bin    first N rlm_step_record of a reference run (oracle/_ref/ref_driver)
  tests/golden/bt_*_{profit_log,test_stats}.csv   the reference's own evaluation logs for the backtest cases
  tests/golden/manifest.json       the configs that produced them
  (and, in tested_reference_runs, the fixtures single tests name themselves)
  tests/golden/learner_shapes.json + digests_<name>.bin   LEARNER_SHAPE_CASES (`make_golden.py learner_shapes`: only these)
"""
import ctypes as C
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as ol  # noqa: E402
from rl_markets_b200 import abi, config  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
N_RECORDS = 400
CASES = [
    dict(name="q_learn_m65536", algo="q_learn", M=65536, flow_seed=7, env=0, ticks=2500, over={}),
    dict(name="sarsa_m16384", algo="sarsa", M=16384, flow_seed=7, env=1, ticks=2500, over={}),
    dict(name="double_q_m65536", algo="double_q_learn", M=65536, flow_seed=9, env=2, ticks=2500, over={}),
    dict(name="q_learn_m5003_greedy", algo="q_learn", M=5003, flow_seed=11, env=3, ticks=2500,
         over={"policy.eps_init": 0.05}),
    dict(name="q_learn_m4096_random_init", algo="q_learn", M=4096, flow_seed=13, env=5, ticks=2500,
         over={"learning.random_init": True, "debug.random_seed": 77}),
    # SURVEY 8f rank 2: R-learning agents (agent.cpp:357-467) and the Boltzmann policy (policy.cpp:85-122)
    dict(name="r_learn_m16384", algo="r_learn", M=16384, flow_seed=15, env=6, ticks=2500, over={"policy.eps_init": 0.3}),
    dict(name="online_r_learn_m16384", algo="online_r_learn", M=16384, flow_seed=15, env=7, ticks=2500,
         over={"policy.eps_init": 0.3}),
    dict(name="double_r_learn_m8209", algo="double_r_learn", M=8209, flow_seed=17, env=8, ticks=2500,
         over={"policy.eps_init": 0.3, "learning.alpha_start": 0.01}),
    dict(name="sarsa_boltzmann_m8192", algo="sarsa", M=8192, flow_seed=19, env=9, ticks=2500,
         over={"policy.type": "boltzmann", "policy.tau_init": 0.05, "policy.tau_floor": 0.01, "policy.tau_T": 10}),
]


# SURVEY 8f rank 2, the rest: every reward measure (base.cpp:166-237), all 13 state variables (intraday.cpp:315-409),
# the Random policy (policy.cpp:27-30), and the other two target-price / quote rules (base.cpp:101-112, intraday.cpp:64-82).
# 150 records each keep the fixtures small.
_ALL_VARS = ["pos", "spd", "mpm", "imb", "svl", "vol", "rsi", "vwap", "a_dist", "a_queue", "b_dist", "b_queue", "last_action"]
F2_CASES = [
    dict(name="rew_none", algo="q_learn", M=8192, flow_seed=31, env=10, ticks=1200, over={"reward.measure": "none"}),
    dict(name="rew_pnl", algo="q_learn", M=8192, flow_seed=31, env=11, ticks=1200, over={"reward.measure": "pnl"}),
    dict(name="rew_spread", algo="sarsa", M=8192, flow_seed=31, env=12, ticks=1200, over={"reward.measure": "spread"}),
    dict(name="rew_normed", algo="q_learn", M=8192, flow_seed=31, env=13, ticks=1200,
         over={"reward.measure": "normed", "reward.pnl_lookback": 12}),
    dict(name="rew_lovol", algo="q_learn", M=8192, flow_seed=31, env=14, ticks=1200, over={"reward.measure": "lovol"}),
    dict(name="rew_mm_linear", algo="q_learn", M=8192, flow_seed=31, env=15, ticks=1200,
         over={"reward.measure": "mm_linear", "reward.pos_weight": 0.5, "reward.pnl_weight": 0.75}),
    dict(name="rew_mm_exp", algo="q_learn", M=8192, flow_seed=31, env=16, ticks=1200,
         over={"reward.measure": "mm_exp", "reward.pos_weight": 0.02, "reward.pnl_weight": 1.0}),
    dict(name="rew_mm_div", algo="double_q_learn", M=8192, flow_seed=31, env=17, ticks=1200, over={"reward.measure": "mm_div"}),
    dict(name="vars13", algo="q_learn", M=16384, flow_seed=33, env=18, ticks=1200,
         over={"state.variables": _ALL_VARS, "state.lookback.rsi": 10, "state.lookback.vwap": 20}),
    dict(name="vars13_sarsa_defaults", algo="sarsa", M=16384, flow_seed=33, env=19, ticks=1200,
         over={"state.variables": list(reversed(_ALL_VARS))}),  # rsi / vwap lookbacks 0 -> windows of 1
    dict(name="policy_random", algo="q_learn", M=8192, flow_seed=35, env=20, ticks=1200, over={"policy.type": "random"}),
    dict(name="policy_greedy", algo="sarsa", M=8192, flow_seed=35, env=21, ticks=1200, over={"policy.type": "greedy"}),
    dict(name="tp_microprice", algo="q_learn", M=8192, flow_seed=37, env=22, ticks=1200,
         over={"market.target_price.type": "microprice", "market.target_price.lookback": 5}),  # -> tp::MidPrice (A1)
    dict(name="tp_book", algo="q_learn", M=8192, flow_seed=37, env=23, ticks=1200, over={"market.target_price.type": "book"}),
]
N_F2_RECORDS = 150

# N training episodes on ONE Intraday and ONE Learner-equivalent (main.cpp:45-60, serial.cpp:72-95): the day ends
# `open_ticks` rows after the first one, HandleTerminal(episode), LoadData of the same day again, Initialise.
EPISODE_CASES = [
    dict(name="ep3_q_learn_m8192", algo="q_learn", M=8192, flow_seed=41, env=24, ticks=700, open_ticks=500, episodes=3,
         over={"learning.omega": 0.9, "learning.alpha_start": 0.01, "policy.eps_T": 3}),
    dict(name="ep3_double_q_m8192", algo="double_q_learn", M=8192, flow_seed=43, env=25, ticks=700, open_ticks=500, episodes=3,
         over={"learning.omega": 0.8, "learning.alpha_start": 0.01, "policy.eps_T": 2}),
    dict(name="ep2_sarsa_boltzmann_m8192", algo="sarsa", M=8192, flow_seed=45, env=26, ticks=700, open_ticks=500, episodes=2,
         over={"policy.type": "boltzmann", "policy.tau_init": 0.05, "policy.tau_floor": 0.01, "policy.tau_T": 2}),
]

# Real-data shapes (SURVEY 8f rank 1): a CSV pair with depth rows that share a timestamp (A21), a crossed book (the reference
# swallows the next row into the same tick), rows with a zero price (dropped) and bursts of 5..9 distinct print prices;
# the reference runs on the files, rlm_ingest_csv + the packed stream have to reproduce it.
INGEST_CASES = [
    dict(name="ingest_messy_q_learn", algo="q_learn", M=8192, flow_seed=51, env=27, ticks=1300, messy_seed=3,
         features=["dup", "zero", "cross", "burst"], over={}),
    dict(name="ingest_messy_sarsa", algo="sarsa", M=8192, flow_seed=53, env=28, ticks=1300, messy_seed=5,
         features=["dup", "zero", "cross", "burst"], over={}),
]

# train on one (short) synthetic day until the close, then main.cpp's evaluation phase (GoGreedy, a NEW Intraday,
# Backtester::RunEpisode) on another one: steps_<name>.bin = training records, steps_<name>_test.bin = evaluation
BACKTEST_CASES = [
    dict(name="bt_q_learn_m8192", algo="q_learn", M=8192, flow_seed=21, env=4, ticks=1200, train_open_ticks=900,
         test=dict(flow_seed=22, env=4, ticks=1000, open_ticks=700), over={"policy.eps_T": 3}),
    dict(name="bt_double_q_m8192", algo="double_q_learn", M=8192, flow_seed=23, env=5, ticks=1200, train_open_ticks=900,
         test=dict(flow_seed=24, env=5, ticks=1000, open_ticks=700), over={"learning.alpha_start": 0.01}),
]


# The learner away from the example config: other action counts, gamma*lambda of 0 and 1 and long trace lists, an explicit
# trace_cap, table sizes at the learner-selection boundaries (staged: single table, M*8 <= 64 KB, M even).  Every record of
# each run is kept as digests_<name>.bin, the cases as learner_shapes.json -- not in manifest.json, whose consumers build
# handles without a trace_cap.  min_traces / max_traces bound the longest trace list of the run, so that a case cannot
# silently stop covering its path (several update-table drains per step, the rate == 0 skip).
LEARNER_SHAPE_CASES = [
    dict(name="a1_q_m8192", algo="q_learn", M=8192, flow_seed=5, env=0, ticks=3000, over={"learning.n_actions": 1},
         min_traces=513),  # every action greedy: rate = gamma*lambda on every step; staged learner
    dict(name="a2_sarsa_m2", algo="sarsa", M=2, flow_seed=5, env=1, ticks=2000, over={"learning.n_actions": 2}),
    dict(name="a3_sarsa_m16384", algo="sarsa", M=16384, flow_seed=5, env=2, ticks=2000, over={"learning.n_actions": 3}),
    dict(name="a5_q_m6002", algo="q_learn", M=6002, flow_seed=5, env=3, ticks=2000, over={"learning.n_actions": 5}),
    dict(name="a7_dq_m4096", algo="double_q_learn", M=4096, flow_seed=5, env=4, ticks=2000, over={"learning.n_actions": 7}),
    dict(name="a4_drl_m8209", algo="double_r_learn", M=8209, flow_seed=5, env=5, ticks=2000,
         over={"learning.n_actions": 4, "policy.eps_init": 0.3, "learning.alpha_start": 0.01}),
    dict(name="lam0_q", algo="q_learn", M=8192, flow_seed=5, env=6, ticks=2000, over={"learning.lambda": 0.0}, max_traces=32),
    dict(name="lam0_sarsa", algo="sarsa", M=8192, flow_seed=5, env=7, ticks=2000, over={"learning.lambda": 0.0}, max_traces=32),
    dict(name="longtr_sarsa_m65536", algo="sarsa", M=65536, flow_seed=5, env=8, ticks=3000,
         over={"learning.gamma": 0.99, "learning.lambda": 0.97}, min_traces=2049),
    dict(name="gl1_sarsa_m8192", algo="sarsa", M=8192, flow_seed=5, env=9, ticks=3000,
         over={"learning.gamma": 1.0, "learning.lambda": 1.0}, trace_cap=8192, min_traces=513),
    dict(name="m1_q", algo="q_learn", M=1, flow_seed=5, env=10, ticks=2000, over={}),
]


def learner_shape_runs():
    import golden_util
    cases = []
    for c in LEARNER_SHAPE_CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = y["debug"]["random_seed"] + c["env"]
        ref = ol.run_ref(y_run, c["flow_seed"], c["env"], c["ticks"])
        recs = ref["records"]
        with open(os.path.join(GOLD, "digests_%s.bin" % c["name"]), "wb") as f:
            for r in recs:
                f.write(golden_util.record_digest(r))
        longest = max(r.n_traces for r in recs)
        assert longest >= c.get("min_traces", 0) and longest <= c.get("max_traces", longest), (c["name"], longest)
        cases.append(dict(c, yaml=y, trace_cap=c.get("trace_cap", 0), n_records=len(recs)))
        print(c["name"], len(recs), "records; longest trace list", longest)
    with open(os.path.join(GOLD, "learner_shapes.json"), "w") as f:
        json.dump(cases, f, indent=1)


def day_t0(cfg, open_ticks, dt_ms=250):
    """t0 such that the market closes (venue close - 30 min, market.cpp:67-70) `open_ticks` rows after the first one."""
    return int(cfg.close_ms) - 30 * 60000 - open_ticks * dt_ms


def main():
    os.makedirs(GOLD, exist_ok=True)
    units = subprocess.check_output([ol.REF_UNITS]).decode()
    json.loads(units)
    with open(os.path.join(GOLD, "units.json"), "w") as f:
        f.write(units)
    manifest = []
    for c in CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        # the reference seeds every generator with debug.random_seed (main.cpp:84-88); env b of a batch uses
        # random_seed + b, so the single-env reference run for env b gets that seed
        seed = y["debug"]["random_seed"] + c["env"]
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = seed
        ref = ol.run_ref(y_run, c["flow_seed"], c["env"], c["ticks"])
        recs = ref["records"][:N_RECORDS]
        with open(os.path.join(GOLD, "steps_%s.bin" % c["name"]), "wb") as f:
            for r in recs:
                f.write(bytes(r))
        manifest.append(dict(c, yaml=y, n_records=len(recs), summary=ref["summary"]))
        print(c["name"], len(recs), "records;", ref["summary"]["steps"], "reference steps")
    for c in F2_CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = y["debug"]["random_seed"] + c["env"]
        ref = ol.run_ref(y_run, c["flow_seed"], c["env"], c["ticks"])
        recs = ref["records"][:N_F2_RECORDS]
        assert len(recs) == N_F2_RECORDS, (c["name"], len(recs))
        with open(os.path.join(GOLD, "steps_%s.bin" % c["name"]), "wb") as f:
            for r in recs:
                f.write(bytes(r))
        manifest.append(dict(c, yaml=y, n_records=len(recs), summary=ref["summary"]))
        print(c["name"], len(recs), "records;", ref["summary"]["steps"], "reference steps")
    for c in EPISODE_CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = y["debug"]["random_seed"] + c["env"]
        cfg = config.from_dict(y)
        t0 = day_t0(cfg, c["open_ticks"])
        ref = ol.run_ref(y_run, c["flow_seed"], c["env"], c["ticks"], t0_ms=t0, episodes=c["episodes"])
        assert ref["summary"]["terminal"] == 1
        with open(os.path.join(GOLD, "steps_%s.bin" % c["name"]), "wb") as f:
            for r in ref["records"]:
                f.write(bytes(r))
        manifest.append(dict(c, yaml=y, multi_episode=True, t0_ms=t0, n_records=len(ref["records"]), summary=ref["summary"]))
        print(c["name"], len(ref["records"]), "records over", c["episodes"], "episodes")
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import messy_csv
    for c in INGEST_CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = y["debug"]["random_seed"] + c["env"]
        md_out, tas_out = os.path.join(GOLD, c["name"] + "_md.csv"), os.path.join(GOLD, c["name"] + "_tas.csv")
        with tempfile.TemporaryDirectory() as d:
            md, tas = os.path.join(d, "c_md_1.csv"), os.path.join(d, "c_tas_1.csv")
            subprocess.check_call([ol.FLOW_CSV, "--seed", str(c["flow_seed"]), "--env", str(c["env"]), "--ticks", str(c["ticks"]),
                                   "--md", md, "--tas", tas])
            messy_csv.make_messy(md, tas, md_out, tas_out, seed=c["messy_seed"], features=c["features"])
            cfgp, dump = os.path.join(d, "cfg.yaml"), os.path.join(d, "steps.bin")
            ol.write_ref_yaml(cfgp, y_run)
            out = subprocess.check_output([ol.REF_DRIVER, "--config", cfgp, "--symbol", "AAL.L", "--md", md_out, "--tas", tas_out,
                                           "--dump", dump, "--steps", "-1"])
            summary = json.loads(out.decode().strip().splitlines()[-1])
            raw = open(dump, "rb").read()
        with open(os.path.join(GOLD, "steps_%s.bin" % c["name"]), "wb") as f:
            f.write(raw)
        n = len(raw) // C.sizeof(abi.StepRecord)
        manifest.append(dict(c, yaml=y, ingest=True, n_records=n, summary=summary))
        print(c["name"], n, "records from the reference on the messy CSV pair")
    for c in BACKTEST_CASES:
        y = config.example_dict(**{"learning.memory_size": c["M"], "learning.algorithm": c["algo"], **c["over"]})
        seed = y["debug"]["random_seed"] + c["env"]
        y_run = json.loads(json.dumps(y))
        y_run["debug"]["random_seed"] = seed
        cfg = config.from_dict(y)
        t0 = day_t0(cfg, c["train_open_ticks"])
        test = dict(c["test"], t0_ms=day_t0(cfg, c["test"]["open_ticks"]))
        ref = ol.run_ref(y_run, c["flow_seed"], c["env"], c["ticks"], t0_ms=t0, test=dict(test, logs=True))
        # the evaluation logs as the reference itself writes them (Backtester's profit_log, Base::writeStats)
        for fname in ("profit_log.csv", "test_stats.csv"):
            with open(os.path.join(GOLD, "%s_%s" % (c["name"], fname)), "w") as f:
                f.write(ref["logs"][fname])
        assert ref["summary"]["terminal"] == 1
        for suffix, recs in (("", ref["records"]), ("_test", ref["test_records"])):
            with open(os.path.join(GOLD, "steps_%s%s.bin" % (c["name"], suffix)), "wb") as f:
                for r in recs:
                    f.write(bytes(r))
        manifest.append(dict(c, yaml=y, backtest=True, t0_ms=t0, test=test, n_records=len(ref["records"]),
                             n_test_records=len(ref["test_records"]), summary=ref["summary"]))
        print(c["name"], len(ref["records"]), "training records;", len(ref["test_records"]), "evaluation records")
    with open(os.path.join(GOLD, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    tested_reference_runs()
    learner_shape_runs()


def tested_reference_runs():
    """The reference outputs that single tests compare against, made with the tests' own cases and inputs:
      digests_flow123_<algo>_m<M>.bin  tests/test_oracle_golden.py FLOW_SEED_123, every record of each run
      digests_messy_flow77_*.bin       tests/test_ingest.py fresh_messy_pair, every record
      file_pairing.json                tests/test_file_pairing.py REF_CALLS on each DIR_NAMES tree, root written {root}
    Runs of a thousand records and more are kept as 8-byte digests per record (golden_util.record_digest)."""
    import tempfile
    import golden_util
    import test_file_pairing as tfp
    import test_ingest
    import test_oracle_golden as tog

    def write_digests(name, recs):
        with open(os.path.join(GOLD, "digests_%s.bin" % name), "wb") as f:
            for r in recs:
                f.write(golden_util.record_digest(r))
        print(name, len(recs), "records")
    for case in tog.FLOW_SEED_123:
        name, y, cfg = tog.flow_seed_123_case(*case)
        write_digests(name, ol.run_ref(y, 123, 0, 4000, t0_ms=cfg.flow.t0_ms)["records"])
    with tempfile.TemporaryDirectory() as d:
        md, tas, y = test_ingest.fresh_messy_pair(d, ol.FLOW_CSV)
        cfgp, dump = os.path.join(d, "cfg.yaml"), os.path.join(d, "steps.bin")
        ol.write_ref_yaml(cfgp, y)
        subprocess.check_output([ol.REF_DRIVER, "--config", cfgp, "--symbol", "AAL.L", "--md", md, "--tas", tas, "--dump", dump,
                                 "--steps", "-1"])
        raw = open(dump, "rb").read()
    recs = (abi.StepRecord * (len(raw) // C.sizeof(abi.StepRecord))).from_buffer_copy(raw)
    write_digests(test_ingest.FRESH_MESSY, recs)
    pairing = {}
    for md_name, tas_name in tfp.DIR_NAMES:
        with tempfile.TemporaryDirectory() as d:
            md, tas = tfp._tree(Path(d), md_name, tas_name)
            calls = {}
            for key, (verb, *rest) in tfp.REF_CALLS.items():
                r = subprocess.run([os.path.join(ol.REF_DIR, "ref_files"), verb, md, tas] + rest, capture_output=True, text=True)
                calls[key] = [r.returncode, [l.replace(d, "{root}").split("\t") for l in r.stdout.splitlines() if l]]
        pairing["%s,%s" % (md_name, tas_name)] = calls
    with open(os.path.join(GOLD, "file_pairing.json"), "w") as f:
        json.dump(pairing, f, indent=1)


if __name__ == "__main__":
    if sys.argv[1:] == ["learner_shapes"]:  # only digests_<learner shape>.bin and learner_shapes.json
        learner_shape_runs()
    else:
        main()
