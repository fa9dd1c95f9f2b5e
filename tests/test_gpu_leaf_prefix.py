"""GPU: the one-shot build's leaf level in two windows (option leaf_prefix_log2).

After the first 2^k leaves are inserted and their ids assigned, the ids of every code seen so far are
final; the leaf kernel then finishes the later occurrences of those codes itself and the first node
level's partition pass only finishes the rest.  These tests force the split onto inputs the oracle can
check (bucket_min=1 buckets the first node level, a small prefix makes n0 >= 2 * 2^k) and build the
inputs so that the boundary cases land on the prefix's edge."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

S = 12


def random_acgt(rng, n):
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, n)]


def leaf_launches(tree):
    return tree.profile_read().get("leaf_insert", {}).get("launches", 0)


def check(stb, oracle, body: bytes, prefix_log2: int, split_expected: bool):
    import torch
    dev = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    tree = stb.SharedTree(S).set_option("bucket_min", 1).set_option("leaf_prefix_log2", prefix_log2)
    tree.profile(True)
    tree.profile_reset()
    tree.build_from_body(dev)
    assert leaf_launches(tree) == (2 if split_expected else 1), "the leaf level did not take the expected path"
    tree.profile(False)
    leaves = oracle.fasta_to_leaves(body, S)
    want = oracle.build(leaves, S)
    assert tree.layer_counts() == want.layer_counts()
    assert tree.leaf_count() == want.leaf_count()
    pre = tree.serialize()
    assert hashlib.sha256(pre).hexdigest() == hashlib.sha256(want.serialize()).hexdigest(), "pre-sort stream"
    assert np.array_equal(tree.decode(), leaves)
    tree.sort()
    want.sort()
    assert tree.serialize() == want.serialize(), "post-sort stream"
    return tree


@pytest.mark.parametrize("prefix_log2", [0, 10, 14, 25])
def test_prefix_sizes_synthetic(stb, oracle, prefix_log2):
    """Off, one tile, a few windows' worth, and the default (too large to split at this size); odd n0."""
    import torch
    n0 = 150_001
    buf = torch.empty(n0 * S + 5, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, buf.numel(), seed=5, repeat_permille=500)
    body = buf.cpu().numpy().tobytes()
    check(stb, oracle, body, prefix_log2, split_expected=prefix_log2 in (10, 14))


@pytest.mark.parametrize("prefix_log2", [10, 12])
def test_low_complexity_prefix_random_suffix(stb, oracle, prefix_log2):
    """Nearly every suffix code is unseen by the prefix (pending), and runs of one unseen code share a warp."""
    rng = np.random.default_rng(prefix_log2)
    P = 1 << prefix_log2
    prefix = (b"A" * (P * S // 2) + b"ACCGTA" * (P * S // 12))[:P * S]
    run = b"CAGT" * 300  # period 4: the same unseen leaf at 100 consecutive positions
    suffix = run + random_acgt(rng, 40_001 * S).tobytes() + run + b"GATTACA"
    check(stb, oracle, prefix + suffix, prefix_log2, split_expected=True)


def test_first_occurrence_at_prefix_end(stb, oracle):
    """Position P is the first occurrence of its code; positions P-1 and P+1.. repeat prefix and suffix codes."""
    P = 1 << 11
    new = b"ACGTTGCAACGG"
    body = b"A" * (P * S) + new + b"C" * S + new * 37 + b"A" * (S * 50) + b"C" * S * (2 * P) + new + b"T" * (S * 3 + 7)
    check(stb, oracle, body, 11, split_expected=True)


def test_n_runs_and_soft_masking_straddling_prefix(stb, oracle):
    """Side-table leaves (symbols outside ACGT) on both sides of P: some first occur in the prefix, some in the suffix."""
    rng = np.random.default_rng(7)
    P = 1 << 12
    n0 = 3 * P + 333
    text = bytearray(random_acgt(rng, n0 * S + 11).tobytes())
    edge = P * S
    text[edge - 3000:edge + 3000] = bytes(text[edge - 3000:edge + 3000]).lower()  # soft-masked across P
    text[edge - 101:edge + 95] = b"N" * 196  # an N run across P
    text[edge + 5000:edge + 5000 + 61] = b"N" * 61  # an N run only in the suffix (other border leaves)
    text[1000:1013] = b"NNNNNNNNNNNNN"
    text[edge + 9000:edge + 9003] = b"RYK"  # IUPAC codes first seen in the suffix
    check(stb, oracle, bytes(text), 12, split_expected=True)


def test_masked_synthetic_with_small_prefix(stb, oracle):
    import torch
    n0 = 200_003
    buf = torch.empty(n0 * S, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, buf.numel(), seed=9, repeat_permille=300)
    stb.synth_mask(buf, seed=9)
    check(stb, oracle, buf.cpu().numpy().tobytes(), 13, split_expected=True)


def test_default_prefix_matches_one_window_at_scale(stb):
    """From 2 * 2^25 leaves on the default splits; the tree equals the single-window build's."""
    import torch
    n0 = (1 << 26) + 4097
    buf = torch.empty(n0 * S, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, buf.numel(), seed=3, repeat_permille=500)
    stb.synth_mask(buf, seed=3)
    digests = []
    for log2 in (25, 0):
        tree = stb.SharedTree(S)
        assert tree.get_option("leaf_prefix_log2") == 25
        tree.set_option("leaf_prefix_log2", log2)
        tree.profile(True)
        tree.profile_reset()
        tree.build_from_body(buf)
        assert leaf_launches(tree) == (2 if log2 else 1)
        tree.profile(False)
        pre = hashlib.sha256(tree.serialize()).hexdigest()
        tree.sort()
        digests.append((tree.layer_counts(), pre, hashlib.sha256(tree.serialize()).hexdigest()))
        del tree
    assert digests[0] == digests[1]
