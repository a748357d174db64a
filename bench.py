#!/usr/bin/env python3
"""bench.py -- env steps/sec of the batched LOB + tile-coded TD hot path on B200.

One bench "step" = `--ticks` market ticks for every one of the B environments of the workload (about TICKS/3.4 learner
steps per env).  The metric is BASELINE.json's: env steps/sec, one env step = one experiment::serial::Learner::_step
(src/experiment/serial.cpp:53-70).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C1..C4] [--no-extras]
                    [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); envs are sharded by rank, independent policies need no data-path
collective ("scaling": "weak").  The headline is C1 (BASELINE.json configs[1]) per GPU; the line also carries, under
"extra", short measurements of the other configs: C2 (the largest single-GPU config) at N = 1, C3 (shared policy, one
NCCL all-reduce per tick) and C4 at N > 1.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TICKS_PER_STEP = 1024  # device-resident leg: 20 driver steps = 20 480 ticks, a timed region of about a second at C1
E2E_TICKS = 64         # end-to-end leg: one upload chunk (32 MB of messages at C1)
WORKLOADS = {
    # BASELINE.json configs[1]: 4096 parallel LOBs, Q-learning tile coding, synthetic Poisson flow, 1xB200
    "C1": dict(envs=4096, algo="q_learn", memory_size=65536, shared=False, pretrain=108000, ticks=TICKS_PER_STEP),
    # configs[2]: 65536 LOBs, SARSA(lambda) with eligibility traces, 1xB200
    "C2": dict(envs=65536, algo="sarsa", memory_size=16384, shared=False, pretrain=20000, ticks=128),
    # configs[3]: 262144 LOBs over 8 GPUs (32768 per GPU), shared policy, per-tick NCCL all-reduce of dtheta
    "C3": dict(envs=32768, algo="q_learn", memory_size=1 << 22, shared=True, pretrain=4000, ticks=64),
    # configs[4]: 1M LOBs over 8 GPUs (131072 per GPU), independent policies, no collective
    "C4": dict(envs=131072, algo="q_learn", memory_size=4096, shared=False, pretrain=12000, ticks=64),
}
# tools/ubench/gather.cu on this pool's B200 (profiles/r2_ubench_gather.txt): independent 8-byte loads at random offsets
# inside a per-warp 512 KB window of a multi-GB array complete at 53.6 G loads/s whatever the parallelism (1.7 TB/s of
# 32-byte sectors = 26 % of the copy bandwidth): the DRAM ceiling of a tile-coded evaluation whose table does not fit
# on chip.  A coalesced 32 KB window per step streams at 6.6-7.0 TB/s instead.
DRAM_RANDOM_SECTORS_PER_S = 53.6e9
# --dump-outputs: per-env arrays and the weight-table sample each stay under these sizes, so that the whole dump, index
# arrays included, stays under 64 MB
DUMP_ENV_BYTES = 24 << 20
DUMP_THETA_BYTES = 16 << 20
DUMP_SEED = 2024


def engine_is_rounds(B, algo, shared, ticks_per_call):
    """Mirrors rlm_create / rlm_run_ticks (rlm_api.cu): the round-paced engine is the default for independent policies on the
    warp-per-env tick kernel (<= 16384 envs) and run calls of at least 128 ticks; RLM_ROUNDS / RLM_ENGINE override."""
    if shared or B > 16384 or os.environ.get("RLM_ENV_VARIANT", "0") not in ("0", ""):
        return False
    r = os.environ.get("RLM_ROUNDS")
    if r is not None:
        return r not in ("0", "")
    return "RLM_ENGINE" not in os.environ and algo in ("q_learn", "sarsa", "double_q_learn") and ticks_per_call >= 128


def workload_string(name, B, algo, M):
    """Identical in the `ours` and `reference` arms (the driver compares it)."""
    return "%s: %d parallel LOBs per GPU, %s + tile coding (32 tilings, memory_size %d per env), synthetic Poisson order flow" % (
        name, B, algo, M)


def algorithmic_bytes_per_step(k_ticks, z_traces, double_q=False):
    """SURVEY.md section 8d: B_step = 2*S_env + K*(B_msg + B_ring) + B_q + 28*Z with S_env=640,
    B_msg=96, B_ring=112, B_q = 8*A*G*T*2 = 13824 (doubled for Double-Q)."""
    return 1280.0 + 208.0 * k_ticks + (27648.0 if double_q else 13824.0) + 28.0 * z_traces


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def host_threads():
    """Threads this process may actually use: the affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                               "--format=csv,noheader,nounits"], timeout=5).decode().strip()
                self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.03)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        mx = max(int(s[1]) for s in self.samples if s[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


def make_cfg(workload, n_envs, env_index0, source, args):
    from rl_markets_b200 import config
    w = WORKLOADS[workload]
    y = config.example_dict(**{"learning.memory_size": args.memory_size or w["memory_size"],
                               "learning.algorithm": args.algo or w["algo"]})
    # dt_ms = 1: 27e6 ticks per synthetic trading day, so no env reaches the close inside a bench run
    cfg = config.from_dict(y, n_envs=n_envs, env_index0=env_index0, source=source, flow_seed=2024, dt_ms=1,
                           shared_policy=bool(w.get("shared")))
    return y, cfg


def _sample(rng, n, cap):
    """range(n) whole, or a fixed seeded sample of `cap` of its values in ascending order."""
    import numpy as np
    return np.arange(n) if n <= cap else np.sort(rng.choice(n, max(cap, 1), replace=False))


def dump_outputs(m, cfg, algo, out_dir):
    """Writes what a caller of the timed path can read back after its last step as out_dir/<name>.npy: every env's state
    vector, reward, action and EnvStats fields, and the weight tables of a fixed, seeded sample of policies (all of them
    are GBs at C1).  The same arguments give the same inputs, so two builds can be compared array by array."""
    import numpy as np
    from rl_markets_b200 import abi
    os.makedirs(out_dir, exist_ok=True)
    B, M, nv = cfg.n_envs, cfg.memory_size, cfg.n_state_vars
    rng = np.random.default_rng(DUMP_SEED)
    stat_names = [f for f, _ in abi.EnvStats._fields_]
    envs = _sample(rng, B, DUMP_ENV_BYTES // (4 * nv + 8 * (3 + len(stat_names))))
    out = {"env_index": envs.astype(np.float64),
           "state": np.ctypeslib.as_array(m.state()).reshape(B, nv)[envs].astype(np.float32),
           "reward": np.ctypeslib.as_array(m.rewards())[envs].astype(np.float64),
           "action": np.ctypeslib.as_array(m.actions())[envs].astype(np.float64)}
    st = np.ctypeslib.as_array(m.stats())[envs]
    for f in stat_names:
        out["stats_" + f] = st[f].astype(np.float64)
    tables = 2 if algo in ("double_q_learn", "double_r_learn") else 1
    policies = _sample(rng, 1 if cfg.shared_policy else B, DUMP_THETA_BYTES // (8 * tables * M))
    cols = _sample(rng, M, DUMP_THETA_BYTES // (8 * tables * len(policies)))
    theta = np.empty((len(policies), tables, len(cols)), dtype=np.float64)
    for i, p in enumerate(policies):
        for t in range(tables):
            theta[i, t] = np.ctypeslib.as_array(m.theta(int(p), t))[cols]
    out.update(theta=theta, theta_policy_index=policies.astype(np.float64), theta_column_index=cols.astype(np.float64))
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class Ctx:
    pass


def _setup():
    import torch
    ctx = Ctx()
    ctx.torch = torch
    ctx.rank = int(os.environ.get("RANK", "0"))
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(ctx.local)
    ctx.dist = None
    if ctx.world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", ctx.local))
        ctx.dist = dist
    ctx.stream = torch.cuda.Stream()
    return ctx


def _barrier(ctx):
    ctx.torch.cuda.synchronize()
    if ctx.dist is not None:
        ctx.dist.barrier()
    ctx.torch.cuda.synchronize()


def _allreduce(ctx, vals, op):
    if ctx.dist is None:
        return [float(v) for v in vals]
    t = ctx.torch.tensor([float(v) for v in vals], device="cuda", dtype=ctx.torch.float64)
    ctx.dist.all_reduce(t, op=getattr(ctx.dist.ReduceOp, op))
    return [float(x) for x in t]


def measure(ctx, name, args, steps, warmup, headline):
    """Device-resident measurement of one workload; returns (dict for rank 0, market, cfg)."""
    torch = ctx.torch
    from rl_markets_b200 import abi, lib, parallel
    w = WORKLOADS[name]
    B = (args.envs if (headline and args.envs) else w["envs"])
    M = (args.memory_size if (headline and args.memory_size) else w["memory_size"])
    algo = (args.algo if (headline and args.algo) else w["algo"])
    ticks = (args.ticks if (headline and args.ticks) else w["ticks"])
    pretrain = (args.pretrain_ticks if (headline and args.pretrain_ticks >= 0) else w["pretrain"])
    shared = bool(w.get("shared"))
    sub = argparse.Namespace(**vars(args))
    sub.memory_size, sub.algo = M, algo
    y, cfg = make_cfg(name, B, ctx.rank * B, abi.SOURCE_GENERATOR, sub)
    cfg.device = ctx.local
    m = lib.BatchedMarket(cfg)
    m.set_stream(ctx.stream.cuda_stream)

    def run_chunk(n):
        if shared and ctx.world > 1:
            with torch.cuda.stream(ctx.stream):
                parallel.run_shared_policy(m, n, ctx.dist)
        else:
            m.run_ticks(n)

    # ---- cold start (informational): the first steps of training from all-zero weight tables
    cold = None
    if headline and pretrain > 0:
        run_chunk(256)
        m.sync()
        cc_a = m.counters()
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _barrier(ctx)
        with torch.cuda.stream(ctx.stream):
            ev_a.record(ctx.stream)
            run_chunk(ticks)
            ev_b.record(ctx.stream)
        _barrier(ctx)
        m.sync()
        cold = {"ms": ev_a.elapsed_time(ev_b), "steps": m.counters().steps - cc_a.steps}
    # ---- pre-training (untimed) so that the timed region sees weight tables in their long-run state: the reference keeps
    # theta across ~1000 episodes (src/main.cpp:47-80).  C1: one LSE trading day of the reference's 250 ms rows.
    left = pretrain
    while left > 0:
        run_chunk(min(left, 512))
        left -= 512
    m.sync()
    occ = None
    if not shared:
        o = m.occupancy()
        occ = sum(o) / len(o) / float(M)
    for _ in range(max(warmup, 3)):
        run_chunk(ticks)
    m.sync()
    c0 = m.counters()
    sampler = ClockSampler(ctx.local) if headline else None
    if sampler:
        sampler.start()
    _barrier(ctx)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    with torch.cuda.stream(ctx.stream):
        evs[0].record(ctx.stream)
        for i in range(steps):
            run_chunk(ticks)
            evs[i + 1].record(ctx.stream)
    _barrier(ctx)
    if sampler:
        sampler.stop_flag = True
    m.sync()
    if headline and args.dump_outputs and ctx.rank == 0:
        dump_outputs(m, cfg, algo, args.dump_outputs)  # before the per-kernel pass below moves the state on
    c1 = m.counters()
    total_ms = evs[0].elapsed_time(evs[-1])
    steps_done, ticks_done, z_sum = c1.steps - c0.steps, c1.ticks - c0.ticks, c1.sum_traces - c0.sum_traces
    launches = c1.kernel_launches - c0.kernel_launches
    # ---- per-kernel pass (untimed, right after the timed region, same state): CUDA events on the launching stream around
    # every tick kernel and every learner kernel (direct launches; rlm_set_profiling) -> the dominant kernel's average
    # launch duration for the roofline block
    kt = None
    prof_ticks = 0 if (shared and ctx.world > 1) else min(ticks, 256)  # (>= 128: the same engine as the timed calls)
    if prof_ticks > 0 and os.environ.get("RLM_ENGINE", "s")[:1] == "s":
        try:
            m.set_profiling(True)
            cp0 = m.counters()
            m.run_ticks(prof_ticks)
            m.sync()
            cp1 = m.counters()
            kt = dict(m.kernel_times())
            kt.update({"steps": cp1.steps - cp0.steps, "z": cp1.sum_traces - cp0.sum_traces, "ticks": prof_ticks})
        except Exception:
            kt = None
        finally:
            m.set_profiling(False)
    total_ms = _allreduce(ctx, [total_ms], "MAX")[0]
    steps_all, ticks_all, z_all = _allreduce(ctx, [steps_done, ticks_done, z_sum], "SUM")
    if cold is not None:
        cold["ms"] = _allreduce(ctx, [cold["ms"]], "MAX")[0]
        cold["steps"] = _allreduce(ctx, [cold["steps"]], "SUM")[0]
    res = None
    if ctx.rank == 0:
        k_bar = ticks_all / max(steps_all, 1.0)
        z_bar = z_all / max(steps_all, 1.0)
        is_dq = algo == "double_q_learn"
        b_step = algorithmic_bytes_per_step(k_bar, z_bar, is_dq)
        value = steps_all / (total_ms * 1e-3)
        peak, peak_src = measured_peak_gbs()
        per_gpu = value / max(ctx.world, 1)
        achieved = per_gpu * b_step / 1e9
        engine = os.environ.get("RLM_ENGINE", "s")[:1]
        fused = engine == "F" and not shared
        rounds = engine_is_rounds(B, algo, shared, ticks)
        # DRAM sectors one env step touches at random when the table does not fit on chip: 864 gathers + Z re-reads of
        # updated weights that miss + 2 Z for the read-modify-write of theta (28 Z algorithmic bytes are trace-list traffic)
        sectors = (1728.0 if is_dq else 864.0) + 2.0 * z_bar
        res = {
            "workload": workload_string(name, B, algo, M), "value": value, "unit": "env_steps/s",
            "ms_per_step": total_ms / steps, "steps": steps, "ticks_per_bench_step": ticks, "envs_per_gpu": B,
            "mean_ticks_per_step": k_bar, "mean_nonzero_traces": z_bar, "ticks_per_s": ticks_all / (total_ms * 1e-3),
            "pretrain_ticks": pretrain, "theta_nonzero_fraction_at_start": occ, "gpu_launches": int(launches),
            "policy": "shared theta, one SUM all-reduce of dtheta per tick" if shared else "independent theta per env, no collective",
            "engine": ("round-paced (two launches per round; every live env runs up to %s ticks per round, until its step ends)" % os.environ.get("RLM_ROUND_CAP", "3")
                       if rounds else {"F": "fused persistent kernel (one launch per bench step)"}.get(engine, "tick-synchronous (two launches per market tick)")),
            "l2": ("working set (theta %.1f GB per GPU) is larger than L2; no flush needed" % (B * M * 8 / 1e9)) if not shared
                  else ("shared theta %.0f MB (L2-resident) + %.1f GB of env records, traces and generator state" % (M * 8 / 1e6, B * 8.0e3 / 1e9)),
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_nominal_8TBs": achieved / 8000.0, "traffic": None, "peak_source": peak_src,
                "kernel": ("rlm_fused2_kernel (market ticks + learner steps of all envs, one launch per bench step)" if fused else
                           ("whole round (tick kernel + learner kernel, two launches per round)" if rounds else
                            "whole tick (env tick kernel + learner kernel, two launches per market tick)")),
                "algorithmic_bytes_per_env_step": b_step,
                "env_steps_per_launch": (steps_all / max(ctx.world, 1)) / max(launches, 1),
                "avg_launch_ms": total_ms / max(launches, 1) if fused else None,
                "timing": "CUDA events on the launching stream around the timed region (max over ranks); per GPU",
                "dram_random_access_ceiling": {
                    "sectors_per_s": DRAM_RANDOM_SECTORS_PER_S, "random_sectors_per_env_step": sectors,
                    "env_steps_per_s": DRAM_RANDOM_SECTORS_PER_S / sectors, "frac_of_ceiling": per_gpu / (DRAM_RANDOM_SECTORS_PER_S / sectors),
                    "source": "tools/ubench/gather.cu, profiles/r2_ubench_gather.txt: random 8-byte gathers from a table larger than L2"
                              + ("" if M > 8192 else " (tables of <= 64 KB are staged whole by cp.async.bulk instead: this ceiling does not apply)")},
            },
        }
        if kt and kt["agent_launches"] > 0 and kt["env_launches"] > 0 and kt["steps"] > 0:
            # dominant kernel = the one with the larger share of a tick.  Algorithmic bytes per launch (SURVEY 8d):
            # learner kernel: steps x (B_q + 28 Z); tick kernel: envs x (B_msg + B_ring) + steps x 2 S_env
            spl = kt["steps"] / float(kt["agent_launches"])
            zpl = kt["z"] / float(max(kt["steps"], 1))
            learner = {"kernel": "learner kernel (%s)" % ("one launch per round: the learner steps of the envs whose step ended in the round"
                                                          if rounds else "one launch per market tick: the learner steps of the envs whose midprice moved"),
                       "avg_launch_ms": kt["agent_ms"] / kt["agent_launches"], "env_steps_per_launch": spl,
                       "algorithmic_bytes_per_launch": spl * ((27648.0 if is_dq else 13824.0) + 28.0 * zpl)}
            tpl = kt["ticks"] * float(B) / kt["env_launches"]  # env ticks per launch
            tick = {"kernel": "market tick kernel (%s)" % ("one launch per round: every live env runs up to round_cap ticks" if rounds
                                                           else "one launch per market tick, every env"),
                    "avg_launch_ms": kt["env_ms"] / kt["env_launches"], "env_ticks_per_launch": tpl,
                    "algorithmic_bytes_per_launch": tpl * 208.0 + spl * 1280.0}
            for k in (learner, tick):
                k["achieved"] = k["algorithmic_bytes_per_launch"] / (k["avg_launch_ms"] * 1e-3) / 1e9
                k["frac"] = k["achieved"] / peak
            dom, oth = (learner, tick) if learner["avg_launch_ms"] >= tick["avg_launch_ms"] else (tick, learner)
            share = dom["avg_launch_ms"] / (learner["avg_launch_ms"] + tick["avg_launch_ms"])
            rf = res["roofline"]
            rf["whole_path"] = {"achieved": rf["achieved"], "frac": rf["frac"], "frac_nominal_8TBs": rf["frac_nominal_8TBs"],
                                "algorithmic_bytes_per_env_step": rf["algorithmic_bytes_per_env_step"],
                                "note": "env steps/s of the timed region x B_step (SURVEY 8d), both kernels and the launch gaps"}
            rf.update({"kernel": dom["kernel"], "achieved": dom["achieved"], "frac": dom["frac"], "frac_nominal_8TBs": dom["achieved"] / 8000.0,
                       "avg_launch_ms": dom["avg_launch_ms"], "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"],
                       "share_of_tick_kernel_time": share,
                       "timing": "CUDA events on the launching stream around every launch of %d market ticks run right after the timed "
                                 "region in the same state (direct launches; rlm_set_profiling); per GPU, rank 0" % kt["ticks"],
                       "other_kernel": {k: oth[k] for k in ("kernel", "avg_launch_ms", "algorithmic_bytes_per_launch", "achieved", "frac")}})
            if dom is learner:
                rf["env_steps_per_launch"] = spl
        if cold is not None:
            res["cold_start"] = {"value": cold["steps"] / (cold["ms"] * 1e-3), "unit": "env_steps/s",
                                 "note": "first bench step of training from all-zero weight tables; informational"}
        if sampler:
            res["clocks"] = sampler.summary()
        try:
            with open(os.path.join(ROOT, "profiles", "r2_summary.json")) as f:
                prof = json.load(f).get(name)
            if prof:
                rf = res["roofline"]
                per_step = prof["dram_bytes_per_env_step"]
                spl_now = rf["env_steps_per_launch"]
                if "whole_path" in rf:  # the dominant kernel's own DRAM bytes per launch, scaled to this run's steps per launch
                    lk = [v for k, v in prof.get("kernels", {}).items() if ("learn" in k or "agent" in k) == rf["kernel"].startswith("learner")]
                    if lk:
                        per_step = (lk[0]["dram_read_bytes"] + lk[0]["dram_write_bytes"]) / float(prof["env_steps_in_captured_tick"])
                    spl_now = kt["steps"] / float(kt["agent_launches"])
                rf["traffic"] = per_step * spl_now
                rf["traffic_source"] = prof.get("source")
        except Exception:
            pass
    return res, m, cfg, (B, M, algo, ticks)


def e2e_leg(ctx, m, name, args, shape):
    """The same metric through the C ABI with HOST buffers: every step uploads its tick messages from pinned host memory
    (rlm_load_ticks) and reads the per-env rewards back (rlm_get_reward).  All B envs get their own stream."""
    torch = ctx.torch
    import numpy as np
    from rl_markets_b200 import abi, lib
    B, M, algo, _ticks = shape
    ticks = E2E_TICKS
    sub = argparse.Namespace(**vars(args))
    sub.memory_size, sub.algo = M, algo
    y2, cfg2 = make_cfg(name, B, ctx.rank * B, abi.SOURCE_STREAM, sub)
    cfg2.device = ctx.local
    m2 = lib.BatchedMarket(cfg2)
    m2.set_stream(ctx.stream.cuda_stream)
    m2.copy_theta_from(m)  # same long-run weight tables as the device-resident leg (a new data day, trained agent)
    n_warm, n_steps = 3, max(args.e2e_steps, 1)
    nbytes = ticks * B * C.sizeof(abi.TickMsg)
    gen_ticks = ticks * (n_warm + n_steps)
    # synthetic messages of every env, generated on the host cores and staged in pinned host memory BEFORE the timed
    # region (one pinned chunk per step); nothing host-side is excluded from the timing
    distinct = min(B, args.e2e_distinct) if args.e2e_distinct > 0 else B
    chunks = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(n_warm + n_steps)]
    views = [c.numpy().view(np.uint8).reshape(ticks, B, 128) for c in chunks]
    for b in range(distinct):
        pe = np.frombuffer(lib.flow_generate(cfg2.flow, ctx.rank * B + b, 0, gen_ticks), dtype=np.uint8).reshape(gen_ticks, 128)
        for k, v in enumerate(views):
            v[:, b, :] = pe[k * ticks:(k + 1) * ticks]
    for b in range(distinct, B):  # (only with --e2e-distinct: the remaining envs replay stream b mod distinct)
        for v in views:
            v[:, b, :] = v[:, b % distinct, :]
    rew = (C.c_double * B)()
    for ch in range(n_warm):
        m2.load_ticks(chunks[ch].data_ptr(), ticks)
        m2.run_ticks(ticks)
        m2.sync()
    cc0 = m2.counters()
    _barrier(ctx)
    t0 = time.perf_counter()
    # rlm_load_ticks double-buffers on a copy stream: the upload of step i+1 is issued before the result of step i is
    # read, so it overlaps step i's kernels; all uploads and all read-backs are inside the region
    m2.load_ticks(chunks[n_warm].data_ptr(), ticks)
    for i in range(n_steps):
        m2.run_ticks(ticks)
        if i + 1 < n_steps:
            m2.load_ticks(chunks[n_warm + i + 1].data_ptr(), ticks)  # H2D inside the timed region
        lib.check(m2.L.rlm_get_reward(m2.h, rew))                    # D2H inside the timed region (syncs)
    _barrier(ctx)
    wall = time.perf_counter() - t0
    cc1 = m2.counters()
    m2.close()
    secs = _allreduce(ctx, [wall], "MAX")[0]
    st = _allreduce(ctx, [cc1.steps - cc0.steps], "SUM")[0]
    return {"value": st / secs, "unit": "env_steps/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": B * 8,
            "steps": n_steps, "ticks_per_step": ticks, "distinct_streams": distinct,
            "engine": "round-paced" if engine_is_rounds(B, algo, False, ticks) else "tick-synchronous (run calls of %d ticks return at once, so that the next upload overlaps them)" % ticks,
            "note": "STREAM source: rlm_load_ticks from pinned host memory (double-buffered upload) + rlm_run_ticks + rlm_get_reward per step"}


def run_ours(args):
    ctx = _setup()
    res, m, cfg, shape = measure(ctx, args.workload, args, args.steps, args.warmup, headline=True)
    e2e = None
    if not args.no_e2e and not WORKLOADS[args.workload].get("shared"):
        e2e = e2e_leg(ctx, m, args.workload, args, shape)
    m.close()
    extras = {}
    if not args.no_extras:
        names = ["C2"] if ctx.world == 1 else ["C3", "C4"]
        for nm in names:
            if nm == args.workload:
                continue
            try:
                r, mx, _c, _s = measure(ctx, nm, args, steps=max(3, min(args.steps, 5)), warmup=3, headline=False)
                mx.close()
                if r is not None:
                    extras[nm] = r
            except Exception as ex:  # an extra must never cost the headline
                if ctx.rank == 0:
                    extras[nm] = {"error": str(ex)[:300]}
    if ctx.rank == 0:
        line = {
            "metric": "env steps/sec (batched LOBs)", "value": res["value"], "unit": "env_steps/s", "n_gpus": ctx.world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": res["workload"], "envs_per_gpu": res["envs_per_gpu"], "ticks_per_bench_step": res["ticks_per_bench_step"],
                       "mean_ticks_per_step": res["mean_ticks_per_step"], "mean_nonzero_traces": res["mean_nonzero_traces"],
                       "policy": res["policy"], "l2": res["l2"], "ticks_per_s": res["ticks_per_s"],
                       "flow": "in-kernel generator (device-resident leg); host-generated streams of every env (e2e leg)",
                       "engine": res["engine"],
                       "pretrain_ticks": res["pretrain_ticks"], "theta_nonzero_fraction_at_start": res["theta_nonzero_fraction_at_start"],
                       "state": "timed after %d ticks of training per env: long-run weight tables" % res["pretrain_ticks"]},
            "gpu_launches": res["gpu_launches"], "clocks": res.get("clocks"), "roofline": res["roofline"],
        }
        if "cold_start" in res:
            line["cold_start"] = res["cold_start"]
        if e2e:
            line["e2e"] = e2e
        if extras:
            line["extra"] = extras
        if ctx.world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_reference(args, n_procs=1, ticks=args.cpu_ticks)
        print(json.dumps(line))
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
def _ref_paths():
    ref = os.path.join(ROOT, "oracle", "_ref")
    return os.path.join(ref, "ref_driver"), os.path.join(ref, "flow_csv")


def cpu_baseline_reference(args, n_procs, ticks):
    """Times the reference's own CPU loop: oracle/_ref/ref_driver = the UNMODIFIED reference sources
    compiled in the build container (oracle/Makefile), one single-threaded process per env (the
    reference's only deterministic mode, src/main.cpp:196-209), CSV parsing included, files on tmpfs."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from rl_markets_b200 import config
    drv, flow = _ref_paths()
    w = WORKLOADS[args.workload]
    algo = args.algo or w["algo"]
    y = config.example_dict(**{"learning.memory_size": args.memory_size or w["memory_size"], "learning.algorithm": algo})
    if not os.path.exists(drv):
        # fall back to the CPU restatement ("port"), threads = n_procs
        cfg = config.from_dict(y, n_envs=n_procs, flow_seed=2024, dt_ms=1)
        L = oracle_lib.lib()
        tt, secs = C.c_int64(0), C.c_double(0)
        steps = L.lobo_run_batch(C.byref(cfg), n_procs, ticks, n_procs, C.byref(tt), C.byref(secs))
        return {"value": steps / secs.value, "unit": "env_steps/s", "cores": n_procs, "kind": "port",
                "sample": "%d env(s) x %d ticks through oracle/liblob_oracle.so (in-memory ticks)" % (n_procs, ticks)}
    tmp = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmp) as d:
        cfgp = _ref_prepare(d, y, flow, n_procs, ticks)
        res = _ref_run(d, cfgp, drv, n_procs)
    return _ref_result(res, n_procs, ticks, algo)


def _ref_prepare(d, y, flow, n_procs, ticks):
    """Config + one synthetic CSV pair per process (written in parallel, on tmpfs, outside any timed region)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    cfgp = os.path.join(d, "cfg.yaml")
    oracle_lib.write_ref_yaml(cfgp, y)
    gens = []
    for i in range(n_procs):
        md, tas = os.path.join(d, "e%d_md_1.csv" % i), os.path.join(d, "e%d_tas_1.csv" % i)
        gens.append(subprocess.Popen([flow, "--seed", "2024", "--env", str(i), "--ticks", str(ticks), "--dt-ms", "1", "--md", md, "--tas", tas]))
    for g in gens:
        if g.wait() != 0:
            raise RuntimeError("flow_csv failed")
    return cfgp


def _ref_run(d, cfgp, drv, n_procs):
    t0 = time.perf_counter()
    procs = []
    for i in range(n_procs):
        md, tas = os.path.join(d, "e%d_md_1.csv" % i), os.path.join(d, "e%d_tas_1.csv" % i)
        procs.append(subprocess.Popen([drv, "--config", cfgp, "--md", md, "--tas", tas], stdout=subprocess.PIPE))
    outs = [p.communicate()[0] for p in procs]
    wall = time.perf_counter() - t0
    steps, inner = 0, 0.0
    for o in outs:
        r = json.loads(o.decode().strip().splitlines()[-1])
        steps += r["steps"]
        inner = max(inner, r["seconds"])
    return steps, inner, wall


def _ref_result(res, n_procs, ticks, algo):
    steps, inner, wall = res
    return {"value": steps / inner, "unit": "env_steps/s", "cores": n_procs, "kind": "reference",
            "sample": "%d process(es) x %d synthetic ticks (%d learner steps), %s, CSV parsing included, "
                      "timed inside ref_driver (max over processes %.2fs; wall incl. process start %.2fs)"
                      % (n_procs, ticks, steps, algo, inner, wall)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_procs = host_threads()
    drv, flow = _ref_paths()
    n_runs = max(args.warmup, 0) + args.steps
    # one bench step = every usable host thread runs one single-env reference process over `ticks` ticks of the workload;
    # the sample is sized so that the whole --steps/--warmup run stays within a few minutes (~1e5 ticks/s per process)
    ticks = min(args.ref_ticks, max(10000, int(6e6 / max(n_runs, 1))))
    vals = []
    last = None
    if not os.path.exists(drv):
        for i in range(n_runs):
            last = cpu_baseline_reference(args, n_procs=n_procs, ticks=ticks)  # oracle port fallback
            if i >= args.warmup:
                vals.append(last)
    else:
        from rl_markets_b200 import config
        w0 = WORKLOADS[args.workload]
        algo = args.algo or w0["algo"]
        y = config.example_dict(**{"learning.memory_size": args.memory_size or w0["memory_size"], "learning.algorithm": algo})
        tmp = "/dev/shm" if os.path.isdir("/dev/shm") else None
        with tempfile.TemporaryDirectory(dir=tmp) as d:
            cfgp = _ref_prepare(d, y, flow, n_procs, ticks)
            for i in range(n_runs):
                last = _ref_result(_ref_run(d, cfgp, drv, n_procs), n_procs, ticks, algo)
                if i >= args.warmup:
                    vals.append(last)
    value = sum(v["value"] for v in vals) / len(vals)
    w = WORKLOADS[args.workload]
    line = {"impl": "reference", "metric": "env steps/sec (batched LOBs)", "value": value, "unit": "env_steps/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_string(args.workload, args.envs or w["envs"], args.algo or w["algo"], args.memory_size or w["memory_size"]),
                       "reference_arm": "%d independent single-threaded reference processes (one per usable host thread: affinity mask "
                                        "capped by the cgroup quota), each running ONE env of the workload" % n_procs},
            "cpu_baseline": {"value": value, "unit": "env_steps/s", "cores": n_procs, "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": value, "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C1", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0)
    ap.add_argument("--algo", default="")
    ap.add_argument("--memory-size", dest="memory_size", type=int, default=0)
    ap.add_argument("--ticks", type=int, default=0, help="market ticks per bench step (default: per workload, 1024 for C1)")
    ap.add_argument("--pretrain-ticks", dest="pretrain_ticks", type=int, default=-1,
                    help="untimed training before the timed region (default: per workload; C1 = one LSE day of 250 ms rows); 0 = cold start")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-steps", dest="e2e_steps", type=int, default=20)
    ap.add_argument("--e2e-distinct", type=int, default=0, help="0 = every env gets its own host-generated stream")
    ap.add_argument("--no-extras", action="store_true", help="skip the short measurements of the other configs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-ticks", type=int, default=1200000)
    ap.add_argument("--ref-ticks", type=int, default=100000)
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed (rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
