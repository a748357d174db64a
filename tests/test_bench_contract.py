"""The JSON line bench.py prints is a contract with the driver: check the committed round-2 lines against it, and
that the reference arm (which needs no GPU) still produces a conforming line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROF = os.path.join(ROOT, "profiles")

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def _line(name):
    return json.loads(open(os.path.join(PROF, name)).read().strip().splitlines()[-1])


def test_committed_headline_line_has_every_contract_key():
    d = _line("bench_r2b_c1.json")
    assert BASE_KEYS <= set(d) and {"roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches", "extra"} <= set(d)
    assert d["metric"].startswith("env steps/sec") and d["unit"] == "env_steps/s" and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert "workload" in d["config"] and d["config"]["workload"].startswith("C1") and "model" not in d["config"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["frac_nominal_8TBs"] - r["achieved"] / 8000.0) < 1e-12
    assert r["traffic"] is None or r["traffic"] > 0
    ceil = r["dram_random_access_ceiling"]  # tools/ubench/gather.cu: what random 8-byte gathers allow at all
    assert 0.0 < ceil["frac_of_ceiling"] < 1.0 and ceil["env_steps_per_s"] > d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 64 * 4096 * 128 and e["d2h_bytes_per_step"] == 4096 * 8
    assert e["distinct_streams"] == 4096, "every env gets its own host-generated stream"
    assert e["value"] != d["value"], "the end-to-end figure must be measured, not copied"
    ticks = d["config"]["ticks_per_bench_step"]
    # two kernels per market tick (tick-synchronous) or per round of at most three ticks (round-paced engine, long calls)
    assert d["gpu_launches"] >= 2 * ticks * d["steps"] // (3 if "round" in d["config"]["engine"] else 1)
    # the roofline block is on the dominant kernel, timed live with CUDA events around its launches
    assert r["avg_launch_ms"] > 0 and abs(r["achieved"] - r["algorithmic_bytes_per_launch"] / (r["avg_launch_ms"] * 1e-3) / 1e9) < 1e-6 * r["achieved"]
    assert 0.5 <= r["share_of_tick_kernel_time"] < 1.0 and r["other_kernel"]["avg_launch_ms"] > 0
    assert r["whole_path"]["achieved"] > 0 and abs(r["whole_path"]["achieved"] - d["value"] * r["whole_path"]["algorithmic_bytes_per_env_step"] / 1e9) < 1e-6 * r["whole_path"]["achieved"]
    assert d["ms_per_step"] * d["steps"] >= 1000.0, "the timed region is at least a second long"
    assert d["clocks"]["reasons"] == [] and d["clocks"]["sm_mhz"] >= 0.9 * d["clocks"]["sm_max_mhz"]
    assert d["config"]["pretrain_ticks"] > 0 and d["config"]["theta_nonzero_fraction_at_start"] > 0.5  # long-run tables
    c2 = d["extra"]["C2"]  # the largest single-GPU config rides along
    assert c2["workload"].startswith("C2: 65536") and c2["value"] > 0 and c2["roofline"]["frac"] > 0


def test_committed_scaling_and_reference_lines():
    two = _line("bench_r2b_c1_2gpu.json")
    one = _line("bench_r2b_c1.json")
    assert two["n_gpus"] == 2 and 1.8 < two["value"] / one["value"] < 2.2
    assert two["extra"]["C3"]["value"] > 0 and "shared theta" in two["extra"]["C3"]["policy"]
    assert two["extra"]["C4"]["value"] > 0 and two["extra"]["C4"]["workload"].startswith("C4: 131072")
    ref = _line("bench_r2b_c1_reference_arm.json")
    assert ref["impl"] == "reference" and BASE_KEYS <= set(ref)
    assert ref["config"]["workload"] == one["config"]["workload"], "both arms name the same workload"
    assert ref["e2e"]["value"] == ref["value"] and ref["e2e"]["h2d_bytes_per_step"] == 0
    assert ref["cpu_baseline"]["kind"] == "reference" and ref["cpu_baseline"]["cores"] >= 1


class _FakeMarket:
    """The read-back surface of lib.BatchedMarket that bench.dump_outputs uses, with values that name their origin."""

    def __init__(self, cfg):
        import numpy as np
        self.cfg, self.np = cfg, np

    def _arr(self, a):
        return self.np.ctypeslib.as_ctypes(self.np.ascontiguousarray(a))

    def state(self):
        return self._arr(self.np.arange(self.cfg.n_envs * self.cfg.n_state_vars, dtype=self.np.float32))

    def rewards(self):
        return self._arr(self.np.arange(self.cfg.n_envs, dtype=self.np.float64) * 0.5)

    def actions(self):
        return self._arr(self.np.arange(self.cfg.n_envs, dtype=self.np.int32) % 9)

    def stats(self):
        from rl_markets_b200 import abi
        st = (abi.EnvStats * self.cfg.n_envs)()
        self.np.ctypeslib.as_array(st)["position"][:] = self.np.arange(self.cfg.n_envs)
        return st

    def theta(self, policy, table):
        M = self.cfg.memory_size
        return self._arr(self.np.arange(M, dtype=self.np.float64) + (2 * policy + table) * M)


def test_dump_outputs_are_float_arrays_of_a_fixed_sample_under_64_mb(tmp_path):
    """bench.py --dump-outputs: float32/float64 .npy files only, at most 64 MB in all, the same sample on every run."""
    import types
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    shapes = [("double_q_learn", dict(n_envs=4096, memory_size=65536, n_state_vars=3, shared_policy=0)),      # C1, two tables
              ("q_learn", dict(n_envs=300000, memory_size=1 << 22, n_state_vars=13, shared_policy=1))]     # larger than the budget
    for algo, shape in shapes:
        cfg = types.SimpleNamespace(**shape)
        dirs = [tmp_path / ("%s_%d" % (algo, i)) for i in range(2)]
        for d in dirs:
            bench.dump_outputs(_FakeMarket(cfg), cfg, algo, str(d))
        files = sorted(os.listdir(dirs[0]))
        assert files == sorted(os.listdir(dirs[1])) and "theta.npy" in files and "reward.npy" in files
        assert sum(os.path.getsize(dirs[0] / f) for f in files) <= 64 << 20
        got = {f[:-4]: np.load(dirs[0] / f) for f in files}
        for f in files:
            assert got[f[:-4]].dtype in (np.float32, np.float64), f
            assert np.array_equal(got[f[:-4]], np.load(dirs[1] / f)), f
        envs = got["env_index"].astype(np.int64)
        assert np.array_equal(got["stats_position"], envs) and np.array_equal(got["reward"], envs * 0.5)
        pol, cols, th = got["theta_policy_index"].astype(np.int64), got["theta_column_index"].astype(np.int64), got["theta"]
        tables = 2 if algo == "double_q_learn" else 1
        assert th.shape == (len(pol), tables, len(cols)) and len(pol) >= 1
        M = cfg.memory_size
        assert np.array_equal(th[:, -1, :], cols[None, :] + (2 * pol[:, None] + tables - 1) * M)


def test_reference_arm_runs_without_a_gpu():
    """`bench.py --impl reference` times the reference's CPU loop (oracle/_ref when built, else the oracle port)."""
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                                   "--warmup", "0", "--ref-ticks", "10000"], timeout=600)
    d = json.loads(out.decode().strip().splitlines()[-1])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d) and d["value"] > 1e3
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
