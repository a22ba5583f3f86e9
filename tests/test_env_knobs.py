"""CRO_* knobs are validated the way the reference validates its environment
(internal/controller/composableresource_adapter.go:42-45, :64, :67): strict parse, legal range, one wording."""
import re

import pytest

REF_LINE = "the env variable DEVICE_RESOURCE_TYPE has an invalid value: '%s'"     # composableresource_adapter.go:44


def test_wording_is_the_references(cro, kats):
    # the reference's own sentence, as its controller tests expect it (tests/golden/reference_kats.json "env_errors")
    (ref,) = kats["env_errors"]
    assert ref["error"] == REF_LINE % ref["device_resource_type"]
    msg = cro.validate_env("CRO_USE_GRAPH", "yes")
    assert msg == REF_LINE.replace("DEVICE_RESOURCE_TYPE", "CRO_USE_GRAPH") % "yes"


@pytest.mark.parametrize("name,value,ok", [
    ("CRO_TMA_READ_TILE", "32768", True), ("CRO_TMA_READ_TILE", "32769", False), ("CRO_TMA_READ_TILE", "512", False),
    ("CRO_TMA_READ_TILE", "0x8000", False), ("CRO_TMA_READ_TILE", " 32768", False), ("CRO_TMA_READ_TILE", "-16", False),
    ("CRO_TMA_READ_STAGES", "4", True), ("CRO_TMA_READ_STAGES", "1", False), ("CRO_TMA_READ_STAGES", "17", False),
    ("CRO_FUSED_THREADS", "160", True), ("CRO_FUSED_THREADS", "150", False), ("CRO_EXPECT_CTAS", "2", True), ("CRO_EXPECT_CTAS", "0", False),
    ("CRO_P2P_READ_VARIANT", "2", True), ("CRO_P2P_READ_VARIANT", "0", False), ("CRO_USE_GRAPH", "", True),
    ("CRO_HELPER_TIMEOUT_MS", "99999999999999999999", False), ("CRO_USE_GRAPH", "1x", False),
])
def test_each_knob_has_a_range(cro, name, value, ok):
    msg = cro.validate_env(name, value)
    assert (msg == "") == ok, (name, value, msg)
    if not ok:
        assert msg == "the env variable %s has an invalid value: '%s'" % (name, value)


def test_process_environment_is_checked_as_a_whole(cro, monkeypatch):
    assert cro.validate_env() == ""
    monkeypatch.setenv("CRO_FUSED_TILE", "114688")
    monkeypatch.setenv("CRO_FUSED_STAGES", "4")                 # 448 KiB of ring: more shared memory than a CTA may own
    assert cro.validate_env() == "the env variable CRO_FUSED_TILE has an invalid value: '114688'"
    monkeypatch.setenv("CRO_FUSED_STAGES", "2")
    assert cro.validate_env() == ""


def test_no_raw_atoi_of_the_environment_is_left():
    import glob
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for path in glob.glob(os.path.join(root, "composable-resource-operator_b200", "csrc", "*.cu")):
        src = open(path).read()
        assert not re.search(r"atoi\s*\(\s*getenv", src) and "env_int(" not in src and "env_u32(" not in src, path


def test_chase_end_matches_the_golden_vectors(cro):
    """The product's restatement of the latency permutation (std::mt19937_64 + Sattolo) against the vectors the pure-Python
    generator wrote (tests/golden/make_pattern_kats.py)."""
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    g = json.load(open(os.path.join(root, "tests", "golden", "pattern_kats.json")))
    for c in g["chase_ends"]:
        assert cro.chase_end(c["minor_src"], c["minor_dst"], c["hops"]) == c["end"], c
