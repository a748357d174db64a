"""md/tas file pairing (include/utilities/files.h:39-108) of rl_markets_b200.ingest against what the reference's own
header returned for the same directory trees (tests/golden/file_pairing.json, written by tools/make_golden.py from
oracle/_ref/ref_files)."""
import json
import os

import pytest

import golden_util as G
from rl_markets_b200 import ingest

# directory names of equal and of different lengths, and one containing "md_" itself: the offset quirk
DIR_NAMES = [("depth", "trade"), ("md_data", "tas_data"), ("d", "trades_long")]
# ref_files <verb> <md_dir> <tas_dir> <arguments...> (oracle/ref_driver/ref_files.cpp), as recorded in the fixture
REF_CALLS = {"sample": ("sample", "AAL.L", "VOD.L"), "window": ("window", "AAL.L", "201001", "20100211"),
             "sample_missing": ("sample", "NONE.L")}


def _touch(path):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    open(path, "w").close()


def _tree(tmp_path, md_name, tas_name):
    md, tas = str(tmp_path / md_name), str(tmp_path / tas_name)
    for day in ("20100104", "20100105", "20100106", "20100211"):
        _touch("%s/AAL.L/xmd_%s.csv" % (md, day))
    for day in ("20100104", "20100106", "20100211"):  # the 5th has no partner
        _touch("%s/AAL.L/xmtas%s.csv" % (tas, day))
    _touch("%s/AAL.L/xmd_notes.txt" % md)
    for day in ("20100104",):
        _touch("%s/VOD.L/ymd_%s.csv" % (md, day))
        _touch("%s/VOD.L/ymtas%s.csv" % (tas, day))
    return md, tas


def test_pairing_rule_without_the_reference(tmp_path):
    md, tas = _tree(tmp_path, "depth", "trade")
    got = ingest.file_sample(md, tas, ["AAL.L", "VOD.L"])
    assert [os.path.basename(t[1]) for t in got] == ["xmd_20100104.csv", "xmd_20100106.csv", "xmd_20100211.csv", "ymd_20100104.csv"]
    assert all(os.path.basename(t[2]).startswith(("xmtas", "ymtas")) and os.path.exists(t[2]) for t in got)
    with pytest.raises(RuntimeError, match="No such directory"):
        ingest.file_sample(md, tas, ["NONE.L"])
    _touch("%s/BAD.L/depth_20100104.csv" % md)
    os.makedirs("%s/BAD.L" % tas)
    with pytest.raises(RuntimeError, match="Unexpected file name"):
        ingest.file_sample(md, tas, ["BAD.L"])


def reference_answers(root, md_name, tas_name):
    """The reference's (exit code, output rows) for each of REF_CALLS on _tree(root, md_name, tas_name)."""
    with open(os.path.join(G.GOLD, "file_pairing.json")) as f:
        calls = json.load(f)["%s,%s" % (md_name, tas_name)]
    return {k: (rc, [tuple(c.replace("{root}", str(root)) for c in r) for r in rows]) for k, (rc, rows) in calls.items()}


@pytest.mark.parametrize("md_name,tas_name", DIR_NAMES)
def test_file_sample_and_window_match_the_reference_header(tmp_path, md_name, tas_name):
    md, tas = _tree(tmp_path, md_name, tas_name)
    ref = reference_answers(tmp_path, md_name, tas_name)
    rc, rows = ref["sample"]
    assert rc == 0
    assert [tuple(r) for r in rows] == ingest.file_sample(md, tas, ["AAL.L", "VOD.L"])
    rc, rows = ref["window"]
    try:
        mine = ingest.sample_window(md, tas, "AAL.L", ["201001", "20100211"])
    except RuntimeError as e:
        assert rc == 1 and rows and rows[-1][0] == "ERROR" and str(e) in rows[-1][1]
    else:
        assert rc == 0 and [tuple(r) for r in rows] == mine
    rc, rows = ref["sample_missing"]
    assert rc == 1 and rows[-1][0] == "ERROR"
    with pytest.raises(RuntimeError) as ei:
        ingest.file_sample(md, tas, ["NONE.L"])
    assert str(ei.value) == rows[-1][1]
