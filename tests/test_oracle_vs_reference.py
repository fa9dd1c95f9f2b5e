"""CPU: the C restatement against what the unmodified reference returned on seeded fuzz inputs
(tests/golden/reference_fuzz.json, generator: oracle/gen_golden_fuzz.py).  Where the reference can be built
(oracle/_ref), its live answers are compared with the same records too."""
import json

import pytest

from conftest import GOLD
from oracle import gen_golden_fuzz as fuzz


@pytest.fixture(scope="module")
def want():
    return json.loads((GOLD / "reference_fuzz.json").read_text())


@pytest.fixture(scope="module")
def checkers(oracle):
    from oracle.pyoracle import Ref, build_ref
    return [oracle] + ([Ref()] if build_ref() is not None else [])


def test_leaf_fuzz(checkers, want):
    for checker in checkers:
        assert fuzz.leaf_fuzz(checker) == want["leaf_fuzz"], checker.kind


def test_node_fuzz(oracle, checkers, want):
    for checker in checkers:
        assert fuzz.node_fuzz(checker, oracle) == want["node_fuzz"], checker.kind


def test_random_trees(oracle, checkers, want):
    for checker in checkers:
        got = fuzz.random_trees(checker, oracle)
        for g, w in zip(got, want["random_trees"]):
            assert g == w, (checker.kind, w["dna_size"], w["n"])  # src/shared_tree.cpp:316 for the histograms
        assert len(got) == len(want["random_trees"])


def test_fasta_ingest_fuzz(checkers, want):
    for checker in checkers:
        got = fuzz.fasta_ingest_fuzz(checker)
        for g, w in zip(got, want["fasta_ingest_fuzz"]):
            assert g == w, (checker.kind, w["case"])
        assert len(got) == len(want["fasta_ingest_fuzz"])
