"""CPU: the routing model of tests/bucket_outcome_model.py.  Its canonical_node must be the kernels' (stb_node_canonical)
and the oracle's, its leaf pointers must rebuild the oracle's first node level, and every input that
tests/test_gpu_bucket_outcomes.py builds for an outcome must have that outcome under the model."""
import numpy as np
import pytest

import bucket_outcome_model as M


def valid_pointers(rng, n):
    """Pointers this library makes: mirror is never set on an invariant target; null is 0x9fffffff."""
    p = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    p[(p >> 31) == 1] &= np.uint32(~M.MIRROR & 0xFFFFFFFF)
    p[rng.random(n) < 0.1] = M.NULL
    small = rng.random(n) < 0.3  # small indices: ties between the four variants are common
    p[small] = (p[small] & np.uint32(0xE0000000)) | rng.integers(0, 4, small.sum()).astype(np.uint32)
    p[(p >> 31) == 1] &= np.uint32(~M.MIRROR & 0xFFFFFFFF)
    return p


def test_canonical_node_matches_kernels_and_oracle(stb, oracle):
    rng = np.random.default_rng(1)
    l, r = valid_pointers(rng, 2000), valid_pointers(rng, 2000)
    cl, cr, f = M.canonical_node(l, r)
    for i in range(len(l)):
        want = stb.node_canonical(int(l[i]), int(r[i]))
        assert (int(cl[i]), int(cr[i]), int(f[i]) >> 29) == want, (hex(l[i]), hex(r[i]))
        assert oracle.node_canonical(int(l[i]), int(r[i]))[:2] == want[:2]


@pytest.mark.parametrize("S", [5, 12, 14])
def test_leaf_pointers_rebuild_the_first_node_level(oracle, S):
    """Node level 0 from the model's leaf pointers: first-occurrence ranks of canonical keys, with their flags."""
    text = M.random_text(3, S, 3001, M.SIDE) + M.heavy_text(4, S, 500, 300)
    leaves = oracle.fasta_to_leaves(text, S)
    arrays = M.child_arrays(oracle, leaves, S)
    cur = np.concatenate([arrays[0], [M.NULL] if len(leaves) % 2 else []]).astype(np.uint64)
    cl, cr, f = M.canonical_node(cur[0::2], cur[1::2])
    _, first, cls = np.unique(M.pair_key(cl, cr), return_index=True, return_inverse=True)
    rank = np.empty(len(first), dtype=np.uint64)
    rank[np.argsort(first)] = np.arange(len(first), dtype=np.uint64)
    inv = f >> np.uint64(31)
    mirror = np.where(inv == 1, np.uint64(0), f & np.uint64(M.MIRROR))
    got = rank[cls] | mirror | (f & np.uint64(M.TRANSPOSE)) | (inv << np.uint64(31))
    assert np.array_equal(got.astype(np.uint32), arrays[1])


def test_bucket_hash_and_plan_by_hand():
    k = 0x0000000500000007
    h = k ^ (k >> 33)
    h = (h * 0xFF51AFD7ED558CCD) & (2**64 - 1)
    h ^= h >> 33
    h = (h * 0xC4CEB9FE1A85EC53) & (2**64 - 1)
    assert int(M.bucket_hash(np.array([k], dtype=np.uint64))[0]) == h ^ (h >> 29)
    # 48001 positions: 5 hash bits (mean final bucket 1500 <= 2048), 3 in the first pass
    b1, b2, cap1, cap2, usable = M.bucket_plan(48001, M.DEFAULTS)
    assert (b1, b2, cap2, usable) == (3, 2, 3072, True)
    assert cap1 == (6001 + 6001 * 125 // 1000 + 1024 + 3) & ~3


@pytest.mark.parametrize("S,alphabet", [(12, M.ACGT), (12, M.SIDE), (5, M.ACGT), (14, M.ACGT)])
@pytest.mark.parametrize("name", M.INPUTS)
def test_outcome_inputs_have_their_outcome(oracle, name, S, alphabet):
    text, extra = M.outcome_input(name, oracle, S, alphabet)
    leaves = oracle.fasta_to_leaves(text, S)
    got = M.build_outcomes(M.child_arrays(oracle, leaves, S), M.options(bucket_min=1, **extra))
    assert list(got) == [0]
    assert got[0]["outcome"] == M.expected_outcome(name), got[0]
    if name == "dedup_chunked":
        assert got[0]["chunked_buckets"] >= 1 and got[0]["max_distinct"] <= M.DD_SLOTS
    if name == "dedup_fallback_distinct":
        assert got[0]["max2"] > M.DD_CAP and got[0]["max_distinct"] >= 4100


@pytest.mark.parametrize("partition_threads", [512, 1024])
@pytest.mark.parametrize("shift", [0, 1])
def test_collapse_edge_input(oracle, partition_threads, shift):
    """The run fills [4096, 8192) (shift 0: exactly one 1024-thread partition tile); its head is a later occurrence."""
    text = M.collapse_edge_text(21, 12, shift)
    leaves = oracle.fasta_to_leaves(text, 12)
    arrays = M.child_arrays(oracle, leaves, 12)
    nodes = arrays[1]
    run = nodes[4096 + shift:8192 + shift]
    assert (run == run[0]).all() and nodes[4095 + shift] != run[0] and nodes[8192 + shift] != run[0]
    assert (nodes[:4096 + shift] & M.IDX_MASK == run[0] & M.IDX_MASK).sum() == 1  # position 100
    opt = M.options(bucket_min=1, partition_threads=partition_threads)
    assert M.build_outcomes(arrays, opt)[0]["outcome"] == "dedup_on_chip"
    # records of the run: one per tile it touches
    tile = partition_threads * 4
    touched = len({p // tile for p in range(4096 + shift, 8192 + shift)})
    plain = M.level_records(arrays[0][:2 * (4096 + shift)], opt, False)
    assert len(M.level_records(arrays[0][:2 * (8192 + shift)], opt, False)) == len(plain) + touched


@pytest.mark.parametrize("child_filter", [1, 0])
def test_period_six_reaches_the_chunked_kernel_at_level_one(oracle, child_filter):
    text = M.heavy_text(17, 12, 20_000, 8_000, period=6)
    leaves = oracle.fasta_to_leaves(text, 12)
    opt = M.options(bucket_min=1, bucket_levels=2, child_filter=child_filter, bucket_headroom=1 << 16)
    got = M.build_outcomes(M.child_arrays(oracle, leaves, 12), opt)
    assert [got[k]["outcome"] for k in (0, 1)] == ["dedup_chunked", "dedup_chunked"]
    if child_filter:  # the filter drops every random position: level 1 keeps the stretch's records only
        assert got[1]["records"] <= 3 * 8_000 // 2 + 2
