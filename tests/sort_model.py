"""A plain numpy restatement of sort_tree (csrc/sort.cu) and of the .dag stream, and the constructed trees that
tests/test_gpu_sort.py sorts on the device.

Built trees have small reference counts, so the frequency sort of a built tree runs one 8-bit radix pass per
layer.  The trees here are imported trees (written as streams, read back with stb_deserialize) whose child
layers are given a chosen frequency distribution, so that every pass count, every pass-to-pass hand-off and
every combination of permuted and unpermuted neighbouring layers runs.

A tree is a dict: S (dna_size), root (raw pointer), leaves (uint64), layers (list of (n, 2) uint32 arrays,
bottom-up).  Pointers are raw: index in bits 0..28, mirror bit 29, transpose bit 30, and the null read from a
stream is the bare index NULL_IDX (the stream does not keep the invariant bit).

All constructed trees have the build's shape: every node has two children, except that the root's node may
have a null as its logical right child (the right edge of a tree of odd width at that layer), which is what
width() assumes.
"""
from __future__ import annotations

import numpy as np

NULL_IDX = 0x1FFFFFFF
IDX_MASK, MIRROR, TRANSPOSE, KEY31 = 0x1FFFFFFF, 1 << 29, 1 << 30, 0x7FFFFFFF
SEG_START = (0, 16, 4112, 1052688)
SMALL_LAYER = 2048  # layers of at most this many nodes are parsed on the host by stb_deserialize
RS_TILE = 4096      # items per radix-sort CTA


# ---- the stream -------------------------------------------------------------------------------------------

def _be(values, width):
    """Big-endian bytes of uint64 values, `width` bytes each, as a flat uint8 array."""
    v = np.asarray(values, dtype=np.uint64).reshape(-1, 1)
    shifts = np.uint64(8) * np.arange(width - 1, -1, -1, dtype=np.uint64)
    return ((v >> shifts) & np.uint64(0xFF)).astype(np.uint8).reshape(-1)


def encode_pointers(raw):
    """The 1..4 byte encoding of every pointer, back to back (src/shared_tree.cpp:122-142)."""
    raw = np.asarray(raw, dtype=np.uint32).reshape(-1)
    idx = raw & np.uint32(IDX_MASK)
    null = idx == NULL_IDX
    seg = (idx >= 16).astype(np.uint32) + (idx >= 4112) + (idx >= 1052688)
    seg[null] = 3
    off = idx - np.array(SEG_START, dtype=np.uint32)[seg]
    off[null] = 0xFFFFFFF
    flags = ((raw >> 29) & 1) << 4 | ((raw >> 30) & 1) << 5 | seg << 6
    lens = seg + 1
    ends = np.cumsum(lens, dtype=np.int64)
    out = np.zeros(int(ends[-1]) if len(ends) else 0, dtype=np.uint8)
    starts = ends - lens
    out[starts] = ((off >> (8 * seg)) | flags).astype(np.uint8)
    for b in (1, 2, 3):
        has = seg >= b
        out[starts[has] + b] = (off[has] >> (8 * (seg[has] - b))).astype(np.uint8)
    return out


def write(tree) -> bytes:
    """The .dag stream: root pointer, u64 leaf count, leaves of ceil(S/2) bytes, per layer u64 count + pointers."""
    lb = (tree["S"] + 1) // 2
    leaves = np.ascontiguousarray(tree["leaves"], dtype=">u8").view(np.uint8).reshape(-1, 8)[:, 8 - lb:].reshape(-1)
    parts = [encode_pointers([tree["root"]]), _be([len(tree["leaves"])], 8), leaves]
    for nodes in tree["layers"]:
        parts += [_be([len(nodes)], 8), encode_pointers(nodes)]
    return np.concatenate(parts).tobytes()


def _decode_pointers(buf, o, count):
    """`count` pointers from byte o: (raw array, end offset).  The start of a pointer depends on the lengths before
    it, so the starts are walked one by one; the decoding is vectorised."""
    starts = np.empty(count, dtype=np.int64)
    seg_of = (np.frombuffer(buf, dtype=np.uint8) >> 6).tolist() if count else []
    for i in range(count):
        starts[i] = o
        o += 1 + seg_of[o]
    b = np.frombuffer(buf, dtype=np.uint8)
    seg = (b[starts] >> 6).astype(np.uint32)
    off = (b[starts] & 0xF).astype(np.uint32)
    for k in (1, 2, 3):
        has = seg >= k
        off[has] = (off[has] << 8) | b[starts[has] + k]
    idx = np.array(SEG_START, dtype=np.uint32)[seg] + off
    idx[(seg == 3) & (off == 0xFFFFFFF)] = NULL_IDX
    raw = idx | ((b[starts].astype(np.uint32) >> 4) & 1) << 29 | ((b[starts].astype(np.uint32) >> 5) & 1) << 30
    return raw.astype(np.uint32), o


def read(stream: bytes, S: int):
    """Inverse of write() for well-formed streams (no checks: the device's deserialize is what rejects)."""
    lb = (S + 1) // 2
    root, o = _decode_pointers(stream, 0, 1)
    n = int.from_bytes(stream[o:o + 8], "big")
    o += 8
    raw = np.frombuffer(stream, dtype=np.uint8, count=n * lb, offset=o).reshape(n, lb).astype(np.uint64)
    leaves = np.zeros(n, dtype=np.uint64)
    for b in range(lb):
        leaves = (leaves << np.uint64(8)) | raw[:, b]
    o += n * lb
    layers = []
    while o + 8 <= len(stream):
        count = int.from_bytes(stream[o:o + 8], "big")
        ptrs, o = _decode_pointers(stream, o + 8, 2 * count)
        layers.append(ptrs.reshape(count, 2))
    return dict(S=S, root=int(root[0]), leaves=leaves, layers=layers)


# ---- histogram and sort -----------------------------------------------------------------------------------

def child_count(tree, c):
    return len(tree["leaves"]) if c == 0 else len(tree["layers"][c - 1])


def histogram(tree, c):
    """References from node layer c into its child layer (the leaves for c = 0), nulls not counted."""
    p = tree["layers"][c].reshape(-1)
    p = p[(p & np.uint32(KEY31)) != NULL_IDX]
    return np.bincount(p & np.uint32(IDX_MASK), minlength=child_count(tree, c)).astype(np.uint64)


def new_positions(tree, c):
    """Rank of every child under (frequency descending, old index ascending)."""
    freq = histogram(tree, c)
    order = np.argsort(-freq.astype(np.int64), kind="stable")
    newpos = np.empty(len(freq), dtype=np.uint32)
    newpos[order] = np.arange(len(freq), dtype=np.uint32)
    return newpos


def _rewire(nodes, newpos):
    out = nodes.copy()
    keep = (out & np.uint32(KEY31)) != NULL_IDX
    out[keep] = (out[keep] & np.uint32(~IDX_MASK & 0xFFFFFFFF)) | newpos[out[keep] & np.uint32(IDX_MASK)]
    return out


def sort(tree):
    """shared_tree::sort_tree: every child layer ordered by its histogram (computed from the unsorted tree), parents
    rewired with their flags kept; the top layer keeps its order and the root is untouched."""
    L = len(tree["layers"])
    newpos = [new_positions(tree, c) for c in range(L)]
    leaves = np.empty_like(tree["leaves"])
    leaves[newpos[0]] = tree["leaves"]
    layers = []
    for k in range(L):
        nodes = _rewire(tree["layers"][k], newpos[k])
        if k + 1 < L:
            moved = np.empty_like(nodes)
            moved[newpos[k + 1]] = nodes
            nodes = moved
        layers.append(nodes)
    return dict(S=tree["S"], root=tree["root"], leaves=leaves, layers=layers)


def radix_plan(tree):
    """Per child layer: (items, span of the frequencies, radix passes), and the launch counts sort_tree makes."""
    L = len(tree["layers"])
    layers = []
    for c in range(L):
        f = histogram(tree, c)
        n = len(f)
        span = int(f.max() - f.min()) if n else 0
        passes = 0 if n < 2 or span == 0 else (span.bit_length() + 7) // 8
        layers.append(dict(n=n, span=span, passes=passes, blocks=-(-n // RS_TILE)))
    permuted = [p["passes"] > 0 for p in layers]
    total = sum(p["passes"] for p in layers)
    launches = dict(radix_scatter=total, radix_hist=total, permute_leaves=int(permuted[0]),
                    permute_rewire=sum(1 for k in range(L) if permuted[k] or (k + 1 < L and permuted[k + 1])))
    return dict(layers=layers, launches=launches)


# ---- constructed trees ------------------------------------------------------------------------------------

def acgt_leaves(n, S, seed):
    """n distinct leaves of S one-hot nucleotides (n <= 4^S), in a seeded order: code i * odd + seed mod 4^S."""
    assert n <= 4 ** S
    with np.errstate(over="ignore"):
        code = (np.arange(n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed)) % np.uint64(4 ** S)
    digits = np.arange(256, dtype=np.uint64)  # 4 nucleotides of the code -> 16 bits of one-hot nibbles
    spelled = sum(np.uint64(1) << (np.uint64(4 * i) + ((digits >> np.uint64(2 * i)) & np.uint64(3))) for i in range(4))
    out = np.zeros(n, dtype=np.uint64)
    for j in range(0, S, 4):
        out |= spelled[(code >> np.uint64(2 * j)) & np.uint64(0xFF)] << np.uint64(4 * j)
    return out & np.uint64((1 << (4 * S)) - 1)


def from_frequencies(S, freqs, top, seed, flags=False, root_index=None):
    """A tree whose child layer c is referenced freqs[c][i] times at item i (c = 0: the leaves).  Layer c has
    len(freqs[c + 1]) nodes, the top layer `top`; the references of each parent layer are dealt to its pointer
    slots in a seeded random order.  Every node has two children; only when the top layer's references are odd
    is the root's node given a null as its logical right child.  flags: random mirror and transpose bits on every
    non-null pointer, the root included."""
    rng = np.random.default_rng(seed)
    L = len(freqs)
    counts = [len(f) for f in freqs[1:]] + [top]
    root_index = top // 2 if root_index is None else root_index
    root = root_index
    if flags:
        root |= int(rng.integers(0, 4)) << 29
    layers = []
    for c in range(L):
        refs = np.repeat(np.arange(len(freqs[c]), dtype=np.uint32), np.asarray(freqs[c], dtype=np.int64))
        rng.shuffle(refs)
        slots = 2 * counts[c]
        nulls = slots - len(refs)
        assert nulls == 0 or (nulls == 1 and c == L - 1), (c, slots, len(refs))
        if flags:
            refs = refs | (rng.integers(0, 4, len(refs)).astype(np.uint32) << 29)
        if nulls:  # the root's node: its logical right child (the left slot when the root is mirrored)
            null_slot = 2 * root_index + (0 if root & MIRROR else 1)
            refs = np.insert(refs, null_slot, np.uint32(NULL_IDX))
        layers.append(refs.reshape(-1, 2))
    return dict(S=S, root=root, leaves=acgt_leaves(len(freqs[0]), S, seed), layers=layers)


def even_total(freq, rng):
    """Makes the sum even by moving one item one step inside [min, max] (the extremes stay present)."""
    freq = np.asarray(freq, dtype=np.int64)
    if freq.sum() % 2 == 0:
        return freq
    lo, hi = freq.min(), freq.max()
    for i in rng.permutation(len(freq)):
        f = freq[i]
        if f + 1 <= hi and (f != lo or (freq == lo).sum() > 1):
            freq[i] += 1
            return freq
        if f - 1 >= lo and (f != hi or (freq == hi).sum() > 1):
            freq[i] -= 1
            return freq
    raise ValueError("no item can move")


def halving_above(freq0, S, seed, flags=False, halve=True):
    """Child layer 0 as given (an even number of references); above it every node is referenced once, halving
    the layers while their size is even (halve=False: at once), up to a top layer whose root node has a null when
    the layer below is odd."""
    freqs = [np.asarray(freq0, dtype=np.int64)]
    n = int(freqs[0].sum()) // 2  # nodes of layer 0
    while halve and n > 1 and n % 2 == 0:
        freqs.append(np.ones(n, dtype=np.int64))
        n //= 2
    if n > 1:
        freqs.append(np.ones(n, dtype=np.int64))
        n = (n + 1) // 2
    return from_frequencies(S, freqs, n, seed, flags=flags)


LADDER_SPANS = (0, 1, 255, 256, 65535, 65536, (1 << 24) - 1, 1 << 24)
LADDER_MINS = (0, 1, 300)
# (span 0, m 0) has no references at all, so no layer 0: that stream is the empty-layer case, which is rejected
LADDER = [(span, m) for span in LADDER_SPANS for m in LADDER_MINS if (span, m) != (0, 0)]


def ladder(span, m, seed=0, flags=False):
    """Leaves referenced in [m, m + span] times, both ends present.  Spans below 2^16: 6000 leaves, most at m,
    some spread over the range.  From 2^16 up, a hub: one leaf referenced m + span times; with m <= 1 it shares
    layer-0 nodes with span + 1 leaves referenced once (m = 0 adds one unreferenced leaf), so that the 2^24 cases
    hold 2^24 + 2 leaves (dna_size 16 keeps them distinct) and sort in more than 1024 radix blocks.  There, 300
    items are also spread over m + [0, 2^16), so that the keys differ in every byte a pass before the last reads."""
    rng = np.random.default_rng(seed)
    if span < 1 << 16:
        n, S = 6000, 12
        freq = np.full(n, m, dtype=np.int64)
        some = rng.choice(n, n // 10, replace=False)
        freq[some] = m + rng.integers(0, min(span, 1000) + 1, len(some))
        hi, lo = rng.choice(n, 2, replace=False)
        freq[hi], freq[lo] = m + span, m
    elif m <= 1:
        S = 16
        others = span + m if m == 1 else span
        freq = np.concatenate([[m + span], np.ones(others, dtype=np.int64), [0] if m == 0 else []]).astype(np.int64)
        freq = np.roll(freq, int(rng.integers(0, len(freq))))
    else:
        n, S = 2000, 12
        freq = np.full(n, m, dtype=np.int64)
        freq[int(rng.integers(0, n))] = m + span
    if span >= 1 << 16:
        # without these every key but the hub's is 0, and all passes but the last would leave the order as it was:
        # 300 items spread over the low two bytes, so every pass moves items and hands a new order to the next
        spread = rng.choice(np.nonzero((freq < freq.max()) & (freq > 0))[0], 300, replace=False)
        freq[spread[:236]] = m + rng.integers(0, 1 << 12, 236)
        freq[spread[236:]] = m + rng.integers(0, 1 << 16, 64)
    freq = even_total(freq, rng)
    return halving_above(freq, S, seed, flags=flags, halve=span < 1 << 16)


def ladder_passes(span):
    return 0 if span == 0 else (span.bit_length() + 7) // 8


TIE_SIZES = (2, 3, 4095, 4096, 4097, 3 * 4096 - 1, 3 * 4096 + 1, 258 * 4096 - 1, 258 * 4096 + 1)


def ties(n, seed=0, hub=False):
    """n leaves referenced 1, 2 or 3 times (both ends present): long runs of equal keys across warps (512 items),
    tiles (4096) and CTAs.  hub: one more leaf referenced 300 times, so that the ties go through two passes."""
    rng = np.random.default_rng(seed)
    freq = rng.integers(1, 4, n).astype(np.int64)
    if n == 2:
        freq[:] = (1, 3)
    else:
        a, b = rng.choice(n, 2, replace=False)
        freq[a], freq[b] = 1, 3
    if hub:
        freq[int(rng.integers(0, n))] = 300
    return halving_above(even_total(freq, rng), 12, seed)


def neighbours(pattern, seed=0, flags=False):
    """Three node layers of 6000 nodes under a top layer of 5.  Child layer c (c = 0..2) is permuted when pattern[c]
    is set (frequencies 1..3) and keeps its order otherwise (every item referenced twice), so that permute_rewire
    runs with a child map only, a destination map only and both.  Child layer 3 (node layer 2, of which the top
    references 10 nodes) is always permuted."""
    rng = np.random.default_rng(seed)
    n = 6000
    freqs = [_with_total(rng, n, 2 * n, 1, 3) if on else np.full(n, 2, dtype=np.int64) for on in pattern]
    freqs.append(np.bincount(rng.choice(n, 10, replace=False), minlength=n))
    return from_frequencies(12, freqs, 5, seed, flags=flags)


def _with_total(rng, n, total, lo, hi):
    """n integers in [lo, hi] summing to `total`, both ends present."""
    assert n * lo + (hi - lo) <= total <= n * hi - (hi - lo)
    f = np.full(n, lo, dtype=np.int64)
    f[0] = hi
    extra = total - int(f.sum())
    while extra:
        room = np.nonzero(f[1:-1] < hi)[0] + 1
        pick = rng.choice(room, min(extra, len(room)), replace=False)
        f[pick] += 1
        extra -= len(pick)
    return f[rng.permutation(n)]


def top_layer(seed=0, flags=False, odd=True):
    """A top layer of 7 nodes with the root at index 3; the root's node has a null right child when odd."""
    rng = np.random.default_rng(seed)
    n1 = 13 if odd else 14  # node layer 0 items, referenced once each by the 7 top nodes (odd: one null)
    freq0 = _with_total(rng, 20, 2 * n1, 1, 3)
    return from_frequencies(12, [freq0, np.ones(n1, dtype=np.int64)], 7, seed, flags=flags)


POINTER_EDGES = (15, 16, 4111, 4112, 1052687, 1052688)


def pointer_lengths(nodes, seed=0):
    """1052700 leaves of which the edges between pointer lengths (15/16, 4111/4112, 1052687/1052688) and a seeded
    sample are referenced by a layer of `nodes` nodes (<= 2048: parsed on the host, more: on the device)."""
    rng = np.random.default_rng(seed)
    n = 1052700
    refs = np.concatenate([POINTER_EDGES, rng.choice(n, 2 * nodes - len(POINTER_EDGES), replace=False)])
    freq = np.bincount(refs, minlength=n).astype(np.int64)
    return halving_above(freq, 12, seed, flags=True)


def families():
    """name -> zero-argument constructor, for every constructed tree the tests use (the ladder is separate)."""
    out = {}
    for n in TIE_SIZES:
        out[f"ties_{n}"] = lambda n=n: ties(n, seed=n)
    out["ties_two_pass"] = lambda: ties(258 * 4096 + 1, seed=5, hub=True)
    for p in range(8):
        pattern = tuple((p >> c) & 1 for c in range(3))
        out["neighbours_" + "".join(map(str, pattern))] = lambda pattern=pattern, p=p: neighbours(pattern, seed=p)
    out["top_odd"] = lambda: top_layer(1, odd=True)
    out["top_even"] = lambda: top_layer(2, odd=False)
    out["top_flags"] = lambda: top_layer(3, flags=True, odd=True)
    out["flags_ladder"] = lambda: ladder(256, 1, seed=9, flags=True)
    out["flags_neighbours"] = lambda: neighbours((1, 0, 1), seed=11, flags=True)
    out["ptrlen_host"] = lambda: pointer_lengths(2000, seed=1)
    out["ptrlen_device"] = lambda: pointer_lengths(3000, seed=2)
    return out
