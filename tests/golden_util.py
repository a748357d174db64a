"""Loaders for tests/golden (fixtures generated from the compiled reference by tools/make_golden.py)."""
import ctypes as C
import hashlib
import json
import os
import struct

from rl_markets_b200 import abi, config

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _all_cases():
    with open(os.path.join(GOLD, "manifest.json")) as f:
        return json.load(f)


def manifest():
    """Single-episode training cases."""
    return [c for c in _all_cases() if not c.get("backtest") and not c.get("multi_episode") and not c.get("ingest")]


def ingest_manifest():
    """Reference runs on CSV pairs with real-data irregularities (tools/messy_csv.py); the pair is committed beside them."""
    return [c for c in _all_cases() if c.get("ingest")]


def ingest_paths(case):
    return os.path.join(GOLD, case["name"] + "_md.csv"), os.path.join(GOLD, case["name"] + "_tas.csv")


def episode_manifest():
    """N training episodes on one Intraday + one Learner-equivalent (main.cpp:45-60)."""
    return [c for c in _all_cases() if c.get("multi_episode")]


def backtest_manifest():
    """Train-until-the-close, then evaluate (main.cpp:216-241) cases."""
    return [c for c in _all_cases() if c.get("backtest")]


def units():
    with open(os.path.join(GOLD, "units.json")) as f:
        return json.load(f)


def records(name):
    raw = open(os.path.join(GOLD, "steps_%s.bin" % name), "rb").read()
    n = len(raw) // C.sizeof(abi.StepRecord)
    arr = (abi.StepRecord * n).from_buffer_copy(raw)
    return [arr[i] for i in range(n)], arr


def record_digest(r):
    """8-byte BLAKE2b of the fields abi.record_fields_equal compares, field by field (alignment bytes left out): equal
    digests mean equal records.  Long reference runs are stored as digests_<name>.bin, one digest per record."""
    h = hashlib.blake2b(digest_size=8)
    for name, _t in abi.StepRecord._fields_:
        if name != "pad":
            f = getattr(abi.StepRecord, name)
            h.update(C.string_at(C.addressof(r) + f.offset, f.size))
    return h.digest()


def digests(name):
    raw = open(os.path.join(GOLD, "digests_%s.bin" % name), "rb").read()
    return [raw[i:i + 8] for i in range(0, len(raw), 8)]


def learner_shapes():
    """Whole reference runs at other action counts, gamma*lambda, trace caps and table sizes (digests_<name>.bin)."""
    with open(os.path.join(GOLD, "learner_shapes.json")) as f:
        return json.load(f)


def case_config(case, n_envs=1, env_index0=0, source=abi.SOURCE_GENERATOR):
    c = config.from_dict(case["yaml"], n_envs=n_envs, env_index0=env_index0, flow_seed=case["flow_seed"], source=source)
    c.trace_cap = case.get("trace_cap", 0)  # (the reference has no such key: it only sizes the device trace lists)
    return c


def hex_to_double(h):
    return struct.unpack("<d", struct.pack("<Q", int(h, 16)))[0]


def double_bits(d):
    return struct.unpack("<Q", struct.pack("<d", d))[0]


def describe_diff(a, b, fields):
    det = []
    for f in fields:
        x, y = getattr(a, f), getattr(b, f)
        if hasattr(x, "_fields_"):
            det.append((f, [(k, getattr(x, k), getattr(y, k)) for k, _ in x._fields_]))
        elif hasattr(x, "__len__"):
            det.append((f, list(x), list(y)))
        else:
            det.append((f, x, y))
    return det
