"""GPU: node levels that finish their later occurrences in the assign pass (option fused_resolve).

With the option on, every node level that run_node_levels builds one kernel at a time finds the id of a later
occurrence's first occurrence q from the level's rank directory (tile bases, in-tile word prefixes and the bitmap)
instead of reading q's finished pointer in a separate resolve pass.  These tests push oracle-sized inputs through
that path (bucket_min, coop_max, bucket_levels and leaf_prefix_log2 lowered) and build each input with the option
on and off: both trees must equal the oracle's (layer counts, the stream before and after sort_tree, decode)."""
import hashlib

import numpy as np
import pytest

import bucket_outcome_model as M

pytestmark = pytest.mark.gpu

S = 12
TILE, CHUNK = 1024, 256 * 1024  # positions per tile of the level kernels; CHUNK_TILES tiles


def build(stb, text, opts, fused, tree=None):
    import torch
    tree = tree or stb.SharedTree(S)
    for name, value in {**opts, "fused_resolve": fused}.items():
        tree.set_option(name, value)
    tree.profile(True)
    tree.profile_reset()
    tree.build_from_body(torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda())
    profile = tree.profile_read()
    tree.profile(False)
    fused_launches = sum(v["launches"] for k, v in profile.items() if k.split("@")[0] == "assign_resolve")
    return tree, profile, fused_launches


def check(stb, oracle, text, opts, tree=None):
    """Builds `text` with fused_resolve 1 and 0 (on `tree` when given) against the oracle; returns the profiles."""
    leaves = oracle.fasta_to_leaves(text, S)
    ref = oracle.build(leaves, S)
    ref_pre = ref.serialize()
    ref.sort()
    ref_post = ref.serialize()
    profiles = []
    for fused in (1, 0):
        t, profile, launches = build(stb, text, opts, fused, tree)
        assert (launches > 0) == bool(fused), f"fused_resolve={fused}: {launches} assign_resolve launches"
        assert t.layer_counts() == ref.layer_counts(), f"fused_resolve={fused}"
        assert t.leaf_count() == ref.leaf_count()
        assert t.serialize() == ref_pre, f"pre-sort stream, fused_resolve={fused}"
        assert np.array_equal(t.decode(), leaves), f"decode, fused_resolve={fused}"
        t.sort()
        assert t.serialize() == ref_post, f"post-sort stream, fused_resolve={fused}"
        profiles.append(profile)
    return profiles


def synth_text(stb, n_leaves, seed, repeat_permille=500):
    import torch
    buf = torch.empty(n_leaves * S, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, buf.numel(), seed=seed, repeat_permille=repeat_permille)
    return buf.cpu().numpy().tobytes()


# every level above the small top runs one kernel at a time; the bucketed variants put the on-chip dedup below it
PER_LEVEL = {
    "table": dict(coop_max=0, bucket_min=1 << 22, bucket_levels=1, leaf_prefix_log2=25),
    "bucketed_layer0": dict(coop_max=0, bucket_min=1, bucket_levels=1, leaf_prefix_log2=0),
    "bucketed_layers0_3": dict(coop_max=0, bucket_min=1, bucket_levels=4, leaf_prefix_log2=12),
}


@pytest.mark.parametrize("paths", list(PER_LEVEL))
@pytest.mark.parametrize("n_leaves", [2 * CHUNK + 1, 4 * CHUNK - 1, 2 * CHUNK + 2 * TILE + 6, 300_007])
def test_level_sizes_across_tile_and_chunk_edges(stb, oracle, paths, n_leaves):
    """Node level 0 one position past a chunk, one short of two chunks, a tile past a chunk, and odd lengths above."""
    check(stb, oracle, synth_text(stb, n_leaves, seed=n_leaves % 97), PER_LEVEL[paths])


def run_text(kind, rng, n_leaves):
    """Random leaves with runs whose node positions straddle tile edges and whose heads repeat an earlier key."""
    rand = lambda n: np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n * S)].tobytes()
    if kind == "one_letter":
        run = b"A" * (S * 9000)
    elif kind == "period12":
        run = b"ACGTTGCAACGG" * 9000
    else:
        run = b"N" * (S * 9000)
    # leaf 1000: the run's key occurs first; node positions 1500 .. 6000 of level 0 hold the run, its head a later
    # occurrence, across the tile edges at 2048 .. 5120 (and level 1's at 1024 and 2048)
    return rand(1000) + run[:S * 40] + rand(1960) + run + rand(n_leaves - 1000 - 40 - 1960 - 9000) + b"GATTA"


@pytest.mark.parametrize("paths", list(PER_LEVEL))
@pytest.mark.parametrize("kind", ["one_letter", "period12", "n_run"])
def test_long_runs(stb, oracle, paths, kind):
    check(stb, oracle, run_text(kind, np.random.default_rng(len(kind)), 60_001), PER_LEVEL[paths])


@pytest.mark.parametrize("shift", [0, 1])
def test_collapsed_run_at_window_edge(stb, oracle, shift):
    """A run over one partition tile whose head is a later occurrence and whose last position is COLLAPSE_WINDOW - 1
    positions after the head: the second hop of the bucketed levels."""
    opts = dict(coop_max=0, bucket_min=1, bucket_levels=2, leaf_prefix_log2=0, partition_threads=1024)
    check(stb, oracle, M.collapse_edge_text(21, S, shift=shift), opts)


@pytest.mark.parametrize("name", ["dedup_fallback_first_pass", "dedup_fallback_slack0", "dedup_fallback_distinct"])
def test_bucketed_level_that_falls_back_to_the_table(stb, oracle, name):
    """The first node level gives up on chip: the fused pass then reads minimum positions from the table."""
    text, extra = M.outcome_input(name, oracle, S)
    opts = dict(bucket_min=1, coop_max=0, profile_levels=1, **extra)
    for profile in check(stb, oracle, text, opts):
        assert profile.get(f"{M.expected_outcome(name)}@L1", {}).get("launches") == 1


@pytest.mark.parametrize("child_filter", [1, 0])
@pytest.mark.parametrize("text_kind", ["synth", "period6"])
def test_table_levels_mark_repeated_first_occurrences(stb, oracle, child_filter, text_kind):
    """Table levels: the multi bits a level's later occurrences set decide which positions of the next level skip
    the table (the exact singleton filter)."""
    if text_kind == "synth":
        text = synth_text(stb, 400_003, seed=3, repeat_permille=700)
    else:
        text = M.heavy_text(17, S, 20_000, 8_000, period=6)
    check(stb, oracle, text, dict(coop_max=0, child_filter=child_filter))


def test_one_handle_rebuilds_different_inputs(stb, oracle):
    """The directory is reused by every build of a handle, larger and smaller, without a reset."""
    tree = stb.SharedTree(S)
    texts = [synth_text(stb, 2 * CHUNK + 1, seed=1), run_text("period12", np.random.default_rng(2), 30_001),
             synth_text(stb, 700_001, seed=3), M.collapse_edge_text(4, S)]
    for k, text in enumerate(texts):
        check(stb, oracle, text, list(PER_LEVEL.values())[k % 3], tree=tree)


def test_default_options_at_2_26_leaves(stb):
    """Default options: layer 0 on chip, the next levels through the table; the trees with the option on and off
    are the same."""
    import torch
    n = (1 << 26) * S
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=26, repeat_permille=500)
    results = []
    for fused in (1, 0):
        tree = stb.SharedTree(S).set_option("fused_resolve", fused)
        tree.profile(True)
        tree.build_from_body(buf)
        profile = tree.profile_read()
        assert ("assign_resolve" in profile) == bool(fused)
        pre = hashlib.sha256(tree.serialize()).hexdigest()
        probe = tree.decode(12_345_678, 4096)
        tree.sort()
        results.append((tree.layer_counts(), tree.leaf_count(), pre, hashlib.sha256(tree.serialize()).hexdigest(), probe))
        tree.close()
    assert results[0][:4] == results[1][:4]
    assert np.array_equal(results[0][4], results[1][4])
