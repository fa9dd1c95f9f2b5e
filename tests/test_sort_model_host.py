"""CPU: tests/sort_model.py against the oracle.  The model's stream writer and reader on built trees, and the model's
histograms and sort on every constructed tree that tests/test_gpu_sort.py sorts on the device."""
import numpy as np
import pytest

import sort_model as M
from conftest import corpus_text


def as_model(tree):
    """An oracle tree as the model's dict."""
    return dict(S=tree.S, root=tree.root(), leaves=tree.leaves(), layers=[tree.layer(k) for k in range(tree.depth() - 1)])


def stored(tree):
    """What a stream keeps of a tree: no invariant bit, the null as the bare index."""
    strip = lambda p: np.where((p & np.uint32(M.KEY31)) == M.NULL_IDX, np.uint32(M.NULL_IDX), p & np.uint32(M.KEY31))
    return dict(S=tree["S"], root=int(strip(np.uint32(tree["root"]))), leaves=tree["leaves"],
                layers=[strip(nodes) for nodes in tree["layers"]])


def assert_same_tree(a, b):
    assert a["S"] == b["S"] and a["root"] == b["root"]
    assert np.array_equal(a["leaves"], b["leaves"])
    assert len(a["layers"]) == len(b["layers"])
    for x, y in zip(a["layers"], b["layers"]):
        assert np.array_equal(x, y)


def built_trees(oracle, golden):
    for name, S in (("humhbb", 12), ("humhbb", 5), ("humhbb", 16), ("merged", 12)):
        yield f"{name}:{S}", oracle.build(oracle.fasta_to_leaves(corpus_text(name), S), S)
    for name, rec in golden["small"].items():
        leaves = np.array([int(x, 16) for x in rec["input_leaves"]], dtype=np.uint64)
        yield name, oracle.build(leaves, rec["dna_size"])


def test_writer_and_reader_on_built_trees(oracle, golden):
    for name, ref in built_trees(oracle, golden):
        for sorted_ in (False, True):
            if sorted_:
                before = as_model(ref)
                ref.sort()
                assert M.write(M.sort(before)) == ref.serialize(), (name, "model sort")
            tree = as_model(ref)
            stream = ref.serialize()
            assert M.write(tree) == stream, (name, sorted_)
            back = M.read(stream, ref.S)
            assert_same_tree(back, stored(tree))
            assert M.write(back) == stream
            for c in range(len(tree["layers"])):
                assert np.array_equal(M.histogram(tree, c), ref.histogram(c)), (name, c)


def check_against_oracle(oracle, tree):
    stream = M.write(tree)
    ref = oracle.deserialize(stream, tree["S"])
    assert ref.serialize() == stream
    for c in range(len(tree["layers"])):
        assert np.array_equal(M.histogram(tree, c), ref.histogram(c)), c
    ref.sort()
    assert M.write(M.sort(tree)) == ref.serialize()
    return ref


@pytest.mark.parametrize("family", list(M.families()))
def test_families_sort_like_the_oracle(oracle, family):
    tree = M.families()[family]()
    check_against_oracle(oracle, tree)
    if len(tree["leaves"]) < 20_000:  # the reader walks pointer by pointer
        assert_same_tree(M.read(M.write(tree), tree["S"]), tree)


@pytest.mark.parametrize("span,m", M.LADDER)
def test_ladder(oracle, span, m):
    """Each rung has the span and pass count it was built for; below the 2^24 rungs (compared with the oracle on the
    GPU box, where the device sorts them), the model's sort equals the oracle's."""
    tree = M.ladder(span, m, seed=span + m)
    plan = M.radix_plan(tree)
    leaves = plan["layers"][0]
    freq = M.histogram(tree, 0)
    assert int(freq.min()) == m and leaves["span"] == span
    assert leaves["passes"] == M.ladder_passes(span) == [0, 1, 1, 2, 2, 3, 3, 4][M.LADDER_SPANS.index(span)]
    if span >= (1 << 24) - 1 and m <= 1:
        assert leaves["blocks"] > 1024 and len(np.unique(tree["leaves"])) == len(tree["leaves"])
    else:
        check_against_oracle(oracle, tree)


def test_pass_counts_across_families():
    """Together the families and the ladder run sorts of 0 to 4 passes, and every permute_rewire variant."""
    fam = {name: M.radix_plan(make()) for name, make in M.families().items()}
    assert fam["ties_two_pass"]["layers"][0]["passes"] == 2
    assert all(p["layers"][0]["n"] > 4096 * 256 for n, p in fam.items() if n.startswith("ties_1056"))
    # neighbours: child layer c permuted iff the pattern says so
    for name, plan in fam.items():
        if name.startswith("neighbours_"):
            assert [p["passes"] > 0 for p in plan["layers"][:3]] == [c == "1" for c in name.split("_")[1]]
    edges = M.families()["ptrlen_device"]()
    idx = edges["layers"][0].reshape(-1) & np.uint32(M.IDX_MASK)
    assert set(M.POINTER_EDGES) <= set(idx.tolist()) and len(edges["layers"][0]) > M.SMALL_LAYER
