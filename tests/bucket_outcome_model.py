"""A plain numpy restatement of how csrc/bucket.cu routes one on-chip (bucketed) node level, and the inputs that
tests/test_gpu_bucket_outcomes.py builds to drive each of its outcomes.

Given a level's child pointer array (child_arrays: arrays[k] holds the children of node level k) and the
handle's options, the model predicts what the device reports through the profile classes of stb_profile_read:

  dedup_on_chip              every final bucket fits its fixed region (cap2 records)
  dedup_exact                a final bucket holds more than cap2 records: the exact-size second pass runs
  dedup_chunked              ... and one holds more than DD_CAP = 3072: bucket_dedup_chunked_kernel walks it
  dedup_fallback_first_pass  a first-pass bucket holds more than cap1 records: the table in HBM redoes the level
  dedup_fallback_distinct    a chunked bucket holds more than DD_SLOTS = 4096 distinct keys: the same fallback

It restates bucket_plan, the partition tile (partition_threads * 4 positions; a position equal to its predecessor
makes no record, except at a tile's first position), the exact singleton filter of levels >= 1, canonical_node
and pair_key on 31-bit keys, mix64, bucket_hash (h ^ (h >> 29)) and the top b1, then the next b2 hash bits."""
from __future__ import annotations

import numpy as np

IDX_MASK, MIRROR, TRANSPOSE, KEY31, NULL = 0x1FFFFFFF, 1 << 29, 1 << 30, 0x7FFFFFFF, 0x9FFFFFFF
DD_CAP, DD_SLOTS, SMALL_MAX = 3072, 4096, 2048
DEFAULTS = dict(bucket_min=1 << 22, bucket_levels=1, bucket_cap=3072, partition_threads=512, dedup_threads=512,
                bucket_slack_permille=125, bucket_headroom=1024, child_filter=1)
OUTCOMES = ("dedup_on_chip", "dedup_exact", "dedup_chunked", "dedup_fallback_first_pass", "dedup_fallback_distinct")
U64 = np.uint64


def canonical_node(l, r):
    """canonical_node (csrc/common.cuh) on arrays of finished pointers: (left, right, flags), flags at bits 29..31."""
    l = np.asarray(l, dtype=U64)
    r = np.asarray(r, dtype=U64)
    tl = np.where((l & U64(KEY31)) == U64(IDX_MASK), U64(0), U64(TRANSPOSE))
    tr = np.where((r & U64(KEY31)) == U64(IDX_MASK), U64(0), U64(TRANSPOSE))
    ml = ((~l & U64(0xFFFFFFFF)) >> U64(2)) & U64(MIRROR)
    mr = ((~r & U64(0xFFFFFFFF)) >> U64(2)) & U64(MIRROR)
    lt, rt, lm, rm = l ^ tl, r ^ tr, l ^ ml, r ^ mr
    variants = [(l, r, 0), (lt, rt, TRANSPOSE), (rm, lm, MIRROR), (rm ^ tr, lm ^ tl, MIRROR | TRANSPOSE)]
    cl, cr = l.copy(), r.copy()
    flags = np.zeros(l.shape, dtype=U64)
    best = pair_key(l, r)
    for vl, vr, f in variants[1:]:
        k = pair_key(vl, vr)
        better = k < best  # the first minimum wins, as in the reference's variadic_min
        best = np.where(better, k, best)
        cl, cr, flags = np.where(better, vl, cl), np.where(better, vr, cr), np.where(better, U64(f), flags)
    flags |= np.where((l & U64(KEY31)) == (rm & U64(KEY31)), U64(1 << 31), U64(0))
    return cl, cr, flags


def pair_key(l, r):
    return ((np.asarray(l, dtype=U64) & U64(KEY31)) << U64(32)) | (np.asarray(r, dtype=U64) & U64(KEY31))


def mix64(k):
    k = np.asarray(k, dtype=U64).copy()
    with np.errstate(over="ignore"):
        k ^= k >> U64(33)
        k *= U64(0xFF51AFD7ED558CCD)
        k ^= k >> U64(33)
        k *= U64(0xC4CEB9FE1A85EC53)
    return k


def bucket_hash(k):
    h = mix64(k)
    return h ^ (h >> U64(29))


def options(**overrides):
    opt = dict(DEFAULTS)
    opt.update(overrides)
    return opt


def bucket_plan(n, opt):
    """bucket_plan (csrc/bucket.cu): (b1, b2, cap1, cap2, usable) for a level of n positions."""
    cap2 = min(max(opt["bucket_cap"], 16), DD_CAP)
    bits = 2
    while bits < 18 and (n >> bits) > cap2 * 2 // 3:
        bits += 1
    b1 = (bits + 1) // 2
    b2 = bits - b1
    mean1 = -(-n // (1 << b1))
    cap1 = (mean1 + mean1 * opt["bucket_slack_permille"] // 1000 + opt["bucket_headroom"] + 3) & ~3
    usable = (n >> bits) <= cap2 * 2 // 3 and n < (1 << 29)
    return b1, b2, cap1, cap2, usable


def level_records(cur, opt, child_filter):
    """Keys of the records the first partition pass makes from the child pointer array `cur`, in position order."""
    cur = np.asarray(cur, dtype=U64)
    if len(cur) % 2:
        cur = np.concatenate([cur, np.array([NULL], dtype=U64)])
    l, r = cur[0::2], cur[1::2]
    n = len(l)
    tile = opt["partition_threads"] * 4
    same = np.zeros(n, dtype=bool)
    same[1:] = (l[1:] == l[:-1]) & (r[1:] == r[:-1])
    same &= np.arange(n) % tile != 0  # every tile keeps a head
    keep = ~same
    if child_filter:
        # a child that never repeats in its level makes the node a certified singleton: no record
        idx = cur & U64(IDX_MASK)
        _, inverse, counts = np.unique(idx, return_inverse=True, return_counts=True)
        repeats = counts[inverse] >= 2
        repeats[cur == U64(NULL)] = True  # the odd tail's missing child: its bitmap bits are zero ("not first")
        keep &= repeats[0::2] & repeats[1::2]
    cl, cr, _ = canonical_node(l[keep], r[keep])
    return pair_key(cl, cr)


def level_outcome(cur, opt, child_filter=False):
    """The outcome class of one on-chip level and the numbers behind it, or None when bucket_plan is unusable."""
    n_next = (len(cur) + 1) // 2
    b1, b2, cap1, cap2, usable = bucket_plan(n_next, opt)
    if not usable:
        return None
    keys = level_records(cur, opt, child_filter)
    h = bucket_hash(keys)
    d1 = (h >> U64(64 - b1)).astype(np.int64)
    d2 = (h >> U64(64 - b1 - b2)).astype(np.int64)
    count1 = np.bincount(d1, minlength=1 << b1)
    count2 = np.bincount(d2, minlength=1 << (b1 + b2))
    big = np.nonzero(count2 > DD_CAP)[0]
    distinct = [len(np.unique(keys[d2 == b])) for b in big]
    if (count1 > cap1).any():
        outcome = "dedup_fallback_first_pass"
    elif not (count2 > cap2).any():
        outcome = "dedup_on_chip"
    elif not len(big):
        outcome = "dedup_exact"
    elif max(distinct) > DD_SLOTS:
        outcome = "dedup_fallback_distinct"
    else:
        outcome = "dedup_chunked"
    return dict(outcome=outcome, n_next=n_next, records=len(keys), b1=b1, b2=b2, cap1=cap1, cap2=cap2,
                max1=int(count1.max()), max2=int(count2.max()), chunked_buckets=len(big), max_distinct=max(distinct, default=0))


def leaf_pointers(oracle, leaves, S):
    """The leaf level's finished pointers: first-occurrence rank of the canonical leaf, with its flags."""
    values, inverse = np.unique(np.asarray(leaves, dtype=U64), return_inverse=True)
    canon = np.empty(len(values), dtype=U64)
    flags = np.empty(len(values), dtype=U64)
    for i, v in enumerate(values):
        c, f = oracle.leaf_canonical(int(v), S)
        canon[i], flags[i] = c, f
    uniq, first, cls = np.unique(canon[inverse], return_index=True, return_inverse=True)
    rank = np.empty(len(uniq), dtype=U64)
    rank[np.argsort(first)] = np.arange(len(uniq), dtype=U64)
    f = flags[inverse]
    m, t, inv = f & U64(1), (f >> U64(1)) & U64(1), (f >> U64(2)) & U64(1)
    return (rank[cls] | ((m & (inv ^ U64(1))) << U64(29)) | (t << U64(30)) | (inv << U64(31))).astype(np.uint32)


def child_arrays(oracle, leaves, S):
    """[leaf pointers, node level 0's pointers, node level 1's, ...]: arrays[k] holds the children of node level k."""
    return [leaf_pointers(oracle, leaves, S)] + oracle.build_levels(leaves, S)[1]


def build_outcomes(arrays, opt):
    """{node level: outcome dict} for every node level of a build that run_node_levels deduplicates on chip.
    arrays: child_arrays(...)."""
    out = {}
    for k in range(min(opt["bucket_levels"], len(arrays))):
        cur = arrays[k]
        n_next = (len(cur) + 1) // 2
        if len(cur) <= SMALL_MAX or n_next < opt["bucket_min"]:
            break  # the small top of the tree runs in one launch; no later level is bucketed either
        o = level_outcome(cur, opt, child_filter=k > 0 and opt["child_filter"] != 0)
        if o is None:
            break  # the level runs through the table (or the cooperative middle launch)
        out[k] = o
    return out


def outcome_counts(arrays, opt):
    """What profile_read() should report: {class name: number of levels}."""
    counts = {}
    for o in build_outcomes(arrays, opt).values():
        counts[o["outcome"]] = counts.get(o["outcome"], 0) + 1
    return counts


# ---- inputs built for each outcome --------------------------------------------------------------------------
# An input is text (bytes) of whole leaves of dna_size S.  SIDE adds symbols outside ACGT to the random leaves, which
# the direct leaf level keeps in its side table; those inputs also carry an N run across leaf 1024 (the end of a
# 2^10-leaf prefix).
ACGT = b"ACGT"
SIDE = b"ACGT" * 6 + b"NRYK"


def random_leaves(rng, n, S, alphabet=ACGT):
    """n random leaf strings (bytes of length S)."""
    a = np.frombuffer(alphabet, dtype=np.uint8)
    return [bytes(row) for row in a[rng.integers(0, len(a), size=(n, S))]]


def distinct_leaves(rng, n, S, alphabet=ACGT):
    seen, out = set(), []
    while len(out) < n:
        for leaf in random_leaves(rng, n, S, alphabet):
            if leaf not in seen and len(out) < n:
                seen.add(leaf)
                out.append(leaf)
    return out


def with_n_run(leaves, S, alphabet):
    """The leaves with an N run over leaves [900, 1200) when the input is one with side-table leaves."""
    if alphabet == ACGT or len(leaves) < 1200:
        return leaves
    return leaves[:900] + [b"N" * S] * 300 + leaves[1200:]


def random_text(seed, S, n_leaves, alphabet=ACGT):
    return b"".join(with_n_run(random_leaves(np.random.default_rng(seed), n_leaves, S, alphabet), S, alphabet))


def heavy_text(seed, S, flank, reps, period=3, alphabet=ACGT):
    """Random leaves around a stretch of `reps` repetitions of `period` distinct leaves.  With an odd period the
    node keys of the stretch alternate, so no position repeats its predecessor and nothing collapses: each of the
    `period` keys gets reps / 2 records at node level 0 (period 6: three keys at level 0, each reps times, and
    three at level 1, each reps / 2 times)."""
    rng = np.random.default_rng(seed)
    motif = distinct_leaves(rng, period, S)
    head = with_n_run(random_leaves(rng, flank, S, alphabet), S, alphabet)
    return b"".join(head + motif * reps + random_leaves(rng, flank + 1, S, alphabet))


def distinct_key_text(oracle, seed, S, keys=4200, pool=512, alphabet=ACGT):
    """A pool of distinct leaves, then `keys` node positions whose children are two pool leaves, chosen so that every
    node key is new and hashes into final bucket 0: that bucket then holds more distinct keys than the dedup table
    (the level has 4 final buckets, so the first pass needs more head-room than the default)."""
    rng = np.random.default_rng(seed)
    leaves = distinct_leaves(rng, pool, S, alphabet)
    head = b"".join(with_n_run(leaves + [b"A" * S] * 700, S, alphabet))  # N run: leaves 900..1199 of the head
    ptr = leaf_pointers(oracle, oracle.fasta_to_leaves(head, S), S).astype(U64)[:pool]
    n_next = len(head) // S // 2 + keys
    b1, b2, *_ = bucket_plan(n_next, DEFAULTS)
    chosen, seen = [], set()
    while len(chosen) < keys:
        a, b = rng.integers(0, pool, 4096), rng.integers(0, pool, 4096)
        cl, cr, _ = canonical_node(ptr[a], ptr[b])
        k = pair_key(cl, cr)
        hit = (bucket_hash(k) >> U64(64 - b1 - b2)) == U64(0)
        for i in np.nonzero(hit)[0]:
            if int(k[i]) not in seen and len(chosen) < keys:
                seen.add(int(k[i]))
                chosen.append((a[i], b[i]))
    return head + b"".join(leaves[a] + leaves[b] for a, b in chosen)


def collapse_edge_text(seed, S, shift=0, tile=4096):
    """A run of one node key over the partition tile [tile, 2 * tile) (shifted by `shift` positions), whose key first
    occurred at position 100: the run's head is a later occurrence, and the run's last position is tile - 1 positions
    after it, the edge of COLLAPSE_WINDOW."""
    rng = np.random.default_rng(seed)
    n_next = 3 * tile + 123
    x, y = distinct_leaves(rng, 2, S)
    nodes = [a + b for a, b in zip(*[iter(random_leaves(rng, 2 * n_next, S))] * 2)]
    nodes[100] = x + y
    for p in range(tile + shift, 2 * tile + shift):
        nodes[p] = x + y
    return b"".join(nodes)


# The inputs each outcome is built from: (text, options beyond bucket_min=1).  The first-pass overflow has two:
# from skew alone at the default slack, and from a random input with no slack at all.
def outcome_input(name, oracle, S, alphabet=ACGT):
    if name == "dedup_on_chip":
        return random_text(11, S, 40_000, alphabet), {}
    if name == "dedup_exact":
        return random_text(12, S, 40_000, alphabet), dict(bucket_cap=16)
    if name == "dedup_chunked":
        return heavy_text(13, S, 30_000, 12_000, alphabet=alphabet), dict(bucket_headroom=1 << 16)
    if name == "dedup_fallback_first_pass":
        return heavy_text(14, S, 30_000, 12_000, alphabet=alphabet), {}
    if name == "dedup_fallback_slack0":
        return random_text(15, S, 40_000, alphabet), dict(bucket_slack_permille=0, bucket_headroom=0)
    if name == "dedup_fallback_distinct":
        return distinct_key_text(oracle, 16, S, alphabet=alphabet), dict(bucket_headroom=4096)
    raise KeyError(name)


INPUTS = ("dedup_on_chip", "dedup_exact", "dedup_chunked", "dedup_fallback_first_pass", "dedup_fallback_slack0",
          "dedup_fallback_distinct")


def expected_outcome(name):
    return "dedup_fallback_first_pass" if name == "dedup_fallback_slack0" else name
