"""CPU: the oracle path that writes tests/golden/synth_large.json (oracle/gen_golden_large.py) reproduces what
the unmodified reference wrote into tests/golden/synth.json, and synth_large.json is consistent in itself."""
import json

import pytest

from conftest import GOLD

TIMING = ("reference_timing", "made_by")


@pytest.mark.parametrize("name", ["mid_50mbp", "largeN_260mbp"])
def test_oracle_case_reproduces_reference_record(oracle, name):
    """Plain and N-run variants: every field of the reference's record, timings aside, from the oracle."""
    from oracle.gen_golden_large import case
    want = json.loads((GOLD / "synth.json").read_text())[name]
    got = case(oracle, want["bases"], want["dna_size"], want["seed"], want["repeat_permille"], want["variant"],
               want["queries"])
    assert got["made_by"] == "oracle.c"
    got = {k: v for k, v in got.items() if k not in TIMING}
    want = {k: v for k, v in want.items() if k not in TIMING}
    assert got.keys() == want.keys()
    for k in want:
        assert got[k] == want[k], k


def test_synth_large_records_consistent():
    from oracle.gen_golden_large import CASES
    recs = json.loads((GOLD / "synth_large.json").read_text())
    assert list(recs) == list(CASES)
    fields = set(json.loads((GOLD / "synth.json").read_text())["mid_50mbp"]) - {"reference_timing"} | {"made_by"}
    for name, rec in recs.items():
        bases, S, seed, permille, variant, queries = CASES[name]
        assert set(rec) == fields, name
        assert rec["made_by"] == "oracle.c"
        assert (rec["bases"], rec["dna_size"], rec["seed"], rec["repeat_permille"], rec["variant"], rec["queries"]) == \
            (bases, S, seed, permille, variant, queries), name
        assert rec["width"] == bases // S, name
        counts = rec["layer_counts"]
        assert len(rec["pre_layer_sha256"]) == len(counts) == rec["depth"] - 1, name
        assert sum(counts) == rec["nodes"] and counts[-1] == 1, name
        # each level halves the positions (rounding up) and holds at most that many distinct nodes
        positions = rec["width"]
        for c in counts:
            positions = (positions + 1) // 2
            assert 1 <= c <= positions, name
        assert positions == 1, name
        assert rec["leaves"] <= rec["width"] and len(rec["query_first8"]) == 8, name
        assert rec["post_bytes"] <= rec["pre_bytes"], name
