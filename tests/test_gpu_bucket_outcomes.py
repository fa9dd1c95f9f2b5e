"""GPU: every outcome of the on-chip deduplication of a node level (csrc/bucket.cu), on inputs built for it.

Each case builds with bucket_min=1 (so the first node level is bucketed at oracle sizes) and profiling on, and
checks two things.  The outcome classes the device reports (stb_profile_read: dedup_on_chip, dedup_exact,
dedup_chunked, dedup_fallback_first_pass, dedup_fallback_distinct) must equal what tests/bucket_outcome_model.py
predicts from the oracle's pointer arrays.  The tree must equal the oracle's: layer counts, the stream before and
after sort_tree, and decode."""
import numpy as np
import pytest

import bucket_outcome_model as M

pytestmark = pytest.mark.gpu

# entry -> (dna_size, alphabet of the random leaves, options, build from packed leaves)
ENTRIES = {
    "acgt12": (12, M.ACGT, dict(leaf_prefix_log2=0), False),
    "acgt12_two_windows": (12, M.ACGT, dict(leaf_prefix_log2=10), False),  # the leaf kernel finishes most pointers
    "side_table12": (12, M.SIDE, dict(leaf_prefix_log2=10), False),
    "leaves12": (12, M.ACGT, {}, True),
    "direct5": (5, M.ACGT, {}, False),
    "hashed14": (14, M.ACGT, {}, False),  # level 0 reads finished leaf pointers (no LeafFinish)
}
SHAPES = [(p, d) for p in (512, 1024) for d in (256, 512, 1024)]


def reported(profile):
    return {name: v["launches"] for name, v in profile.items() if name.split("@")[0] in M.OUTCOMES}


def build_checked(stb, oracle, text, S, opts, from_leaves=False, tree=None):
    """Builds `text` with bucket_min=1 and `opts`; checks the outcomes against the model and the tree against the
    oracle.  Returns the profile of the build."""
    import torch
    leaves = oracle.fasta_to_leaves(text, S)
    tree = tree or stb.SharedTree(S)
    tree.set_option("bucket_min", 1)
    for name, value in opts.items():
        tree.set_option(name, value)
    tree.profile(True)
    tree.profile_reset()
    if from_leaves:
        tree.build_from_leaves(leaves)
    else:
        tree.build_from_body(torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda())
    profile = tree.profile_read()
    tree.profile(False)

    opt = M.options(bucket_min=1, **{k: v for k, v in opts.items() if k in M.DEFAULTS})
    predicted = M.build_outcomes(M.child_arrays(oracle, leaves, S), opt)
    if opts.get("profile_levels"):
        want = {f"{o['outcome']}@L{k + 1}": 1 for k, o in predicted.items()}
    else:
        want = M.outcome_counts(M.child_arrays(oracle, leaves, S), opt)
    assert reported(profile) == want, {k: (o["outcome"], o["max1"], o["cap1"], o["max2"], o["max_distinct"]) for k, o in predicted.items()}

    ref = oracle.build(leaves, S)
    assert tree.layer_counts() == ref.layer_counts()
    assert tree.leaf_count() == ref.leaf_count()
    assert tree.serialize() == ref.serialize(), "pre-sort stream"
    assert np.array_equal(tree.decode(), leaves)
    tree.sort()
    ref.sort()
    assert tree.serialize() == ref.serialize(), "post-sort stream"
    return profile


@pytest.mark.parametrize("entry", list(ENTRIES))
@pytest.mark.parametrize("name", M.INPUTS)
def test_each_outcome_under_each_entry(stb, oracle, name, entry):
    S, alphabet, opts, from_leaves = ENTRIES[entry]
    text, extra = M.outcome_input(name, oracle, S, alphabet)
    profile = build_checked(stb, oracle, text, S, {**opts, **extra}, from_leaves)
    assert reported(profile) == {M.expected_outcome(name): 1}
    if opts.get("leaf_prefix_log2") == 10:
        assert profile["leaf_insert"]["launches"] == 2, "the leaf level did not run in two windows"


@pytest.mark.parametrize("partition_threads,dedup_threads", SHAPES)
@pytest.mark.parametrize("case", ["heavy_chunked", "distinct_keys", "collapse_edge", "collapse_edge_shifted"])
def test_cta_shapes(stb, oracle, case, partition_threads, dedup_threads):
    opts = dict(partition_threads=partition_threads, dedup_threads=dedup_threads)
    if case == "heavy_chunked":
        text, extra = M.outcome_input("dedup_chunked", oracle, 12)
    elif case == "distinct_keys":
        text, extra = M.outcome_input("dedup_fallback_distinct", oracle, 12)
    else:
        # shift 0 at 1024 threads: the run fills one partition tile and its last position is COLLAPSE_WINDOW - 1
        # positions after its head, which is a later occurrence (the resolve kernel's second hop)
        text, extra = M.collapse_edge_text(21, 12, shift=int(case.endswith("shifted"))), {}
    build_checked(stb, oracle, text, 12, {**opts, **extra})


@pytest.mark.parametrize("child_filter", [1, 0])
def test_chunked_kernel_at_level_one(stb, oracle, child_filter):
    """Period 6: three heavy keys at node level 0 and three at level 1, both walked by the chunked kernel.  With the
    filter on, level 1 reads the multi bits the chunked kernel set at level 0."""
    text = M.heavy_text(17, 12, 20_000, 8_000, period=6)
    opts = dict(bucket_levels=2, child_filter=child_filter, bucket_headroom=1 << 16, profile_levels=1)
    profile = build_checked(stb, oracle, text, 12, opts)
    assert reported(profile) == {"dedup_chunked@L1": 1, "dedup_chunked@L2": 1}


def test_handle_reuse_across_outcomes(stb, oracle):
    """A fallback level, an on-chip level, then an exact level on one handle: counters, overflow words and the reset
    bitmaps must not leak from one build into the next."""
    tree = stb.SharedTree(12)
    plain = dict(bucket_cap=3072, bucket_slack_permille=125, bucket_headroom=1024)
    for name in ("dedup_fallback_distinct", "dedup_on_chip", "dedup_exact", "dedup_fallback_slack0", "dedup_chunked"):
        text, extra = M.outcome_input(name, oracle, 12)
        profile = build_checked(stb, oracle, text, 12, {**plain, **extra}, tree=tree)
        assert reported(profile) == {M.expected_outcome(name): 1}, name


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_build_falls_back_on_heavy_keys(stb, oracle, world):
    """The sharded build has no exact-size pass: heavy keys send the whole build to rank 0, and the tree is still
    the oracle's.  A random input of the same size stays sharded."""
    from genome_compression_b200 import shard
    heavy, _ = M.outcome_input("dedup_chunked", oracle, 12)
    rand = M.random_text(18, 12, len(heavy) // 12)
    for text, falls_back in ((heavy, True), (rand, False)):
        ranks = shard.create_local(world, device=0, dna_size=12)
        for r in ranks:
            r.set_option("cut", 1024)

        def work(rank):
            first, count = rank.range(len(text))
            rank.build_from_body(text[first:first + count], len(text))
            return rank.gather()
        tree = shard.run_local(ranks, work)[0]
        totals = ranks[0].layer_totals()
        for r in ranks:
            r.close()
        assert (all(t == 0 for t in totals[1:])) == falls_back, totals
        leaves = oracle.fasta_to_leaves(text, 12)
        ref = oracle.build(leaves, 12)
        assert tree.layer_counts() == ref.layer_counts()
        assert tree.serialize() == ref.serialize()
        assert np.array_equal(tree.decode(), leaves)
