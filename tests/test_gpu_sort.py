"""GPU: sort_tree (csrc/sort.cu) on constructed trees, against tests/sort_model.py and the oracle.

Each tree is written as a stream by the model and read with stb_deserialize.  Before the sort, every histogram
(to host memory and to a CUDA tensor) equals the model's.  The sort runs with profiling on, and the launch counts
of radix_scatter, radix_hist, permute_leaves and permute_rewire must be the model's: that is what shows that the
1-, 2-, 3- and 4-pass sorts, the carry path of the row scan (more than 1024 radix blocks) and each permute_rewire
variant ran.  After it, the leaf table, every layer and the root equal the model's sorted tree, and the stream the
oracle's.  Also: serialize into device memory at every byte offset, decode and random access before and after,
handle reuse, the stream checks of stb_deserialize, and the pass counts of the full-size synthetic genomes."""
import numpy as np
import pytest

import sort_model as M

pytestmark = pytest.mark.gpu

SORT_CLASSES = ("radix_scatter", "radix_hist", "permute_leaves", "permute_rewire")
DECODE_MAX = 1 << 22  # widths up to this are decoded whole and compared with the oracle's decode


def launches(profile):
    return {name: profile.get(name, {}).get("launches", 0) for name in SORT_CLASSES}


def assert_tree(dev, want, what):
    assert dev.leaf_count() == len(want["leaves"]) and dev.depth() == len(want["layers"]) + 1, what
    assert np.array_equal(dev.leaves(), want["leaves"]), (what, "leaf table")
    for k, nodes in enumerate(want["layers"]):
        got = dev.layer(k)
        if not np.array_equal(got, nodes):
            bad = np.nonzero((got != nodes).any(axis=1))[0][:5]
            raise AssertionError(f"{what}: layer {k} differs at nodes {bad}: got {got[bad]}, want {nodes[bad]}")
    assert dev.root() == want["root"], what


def assert_serialize_into(stb, dev, stream):
    """serialize_into at byte offsets 0..3 (offset 0 is the aligned direct path) between guard bytes."""
    import torch
    want = torch.frombuffer(bytearray(stream), dtype=torch.uint8).cuda()
    n = len(stream)
    for off in range(4):
        buf = torch.full((n + 16,), 0xA5, dtype=torch.uint8, device="cuda")
        start = 4 + off
        assert dev.serialize_into(buf[start:start + n]) == n
        assert torch.equal(buf[start:start + n], want), off
        assert bool((buf[:start] == 0xA5).all()) and bool((buf[start + n:] == 0xA5).all()), (off, "wrote outside")


def check_sort(stb, oracle, tree, dev=None, what=""):
    """tree: a model tree.  Deserializes it into `dev` (a new handle when None), checks histograms, the sort and its
    launch counts, the sorted tables and stream, serialize_into, decode and random access.  Returns the handle."""
    import torch
    stream = M.write(tree)
    dev = dev or stb.SharedTree(tree["S"])
    dev.deserialize(stream)
    ref = oracle.deserialize(stream, tree["S"])
    L = len(tree["layers"])
    for k in range(L):
        want = M.histogram(tree, k)
        assert np.array_equal(dev.histogram(k), want), (what, "histogram", k)
        out = torch.full((len(want) + 1,), -1, dtype=torch.int64, device="cuda")
        dev.histogram(k, out=out)
        assert np.array_equal(out[:-1].cpu().numpy().astype(np.uint64), want), (what, "device histogram", k)
        assert int(out[-1]) == -1, (what, "device histogram wrote past its layer")
    width = ref.width()
    assert dev.width() == width, what
    rng = np.random.default_rng(width)
    idx = np.concatenate([rng.integers(0, width, 5000), [0, width - 1]]).astype(np.uint64)
    ra_before = dev.random_access(idx)
    assert np.array_equal(ra_before, ref.random_access(idx)), what
    dec_before = dev.decode() if width <= DECODE_MAX else None
    if dec_before is not None:
        assert np.array_equal(dec_before, ref.decode()), what

    plan = M.radix_plan(tree)
    dev.profile(True)
    dev.profile_reset()
    dev.sort()
    profile = dev.profile_read()
    dev.profile(False)
    assert launches(profile) == plan["launches"], (what, [(p["n"], p["span"], p["passes"]) for p in plan["layers"]])

    want = M.sort(tree)
    assert_tree(dev, want, what + " sorted")
    ref.sort()
    post = ref.serialize()
    assert M.write(want) == post, what
    assert dev.bytes() == len(post) and dev.serialize() == post, (what, "sorted stream")
    assert_serialize_into(stb, dev, post)
    assert dev.width() == width
    assert np.array_equal(dev.random_access(idx), ra_before), (what, "random access after the sort")
    if dec_before is not None:
        assert np.array_equal(dev.decode(), dec_before), (what, "decode after the sort")
    return dev


@pytest.mark.parametrize("span,m", M.LADDER)
def test_ladder(stb, oracle, span, m):
    tree = M.ladder(span, m, seed=span + m)
    leaves = M.radix_plan(tree)["layers"][0]
    assert leaves["passes"] == M.ladder_passes(span)
    if span >= (1 << 24) - 1 and m <= 1:
        assert leaves["blocks"] > 1024  # the row scan of the radix histogram carries across 1024-block rows
    check_sort(stb, oracle, tree, what=f"ladder span={span} m={m}")


@pytest.mark.parametrize("family", list(M.families()))
def test_family(stb, oracle, family):
    check_sort(stb, oracle, M.families()[family](), what=family)


def as_s16(tree, seed):
    return dict(tree, S=16, leaves=M.acgt_leaves(len(tree["leaves"]), 16, seed))


def test_handle_reuse(stb, oracle):
    """One handle: the sort arena and the spares grown by a 2^24-leaf sort, then reused by a small and a mid-size
    tree; two sorts in a row; a clone of an unsorted tree (no spares yet) sorted on its own."""
    dev = stb.SharedTree(16)
    check_sort(stb, oracle, M.ladder(1 << 24, 1, seed=3), dev, "hub")
    check_sort(stb, oracle, as_s16(M.ties(4097, seed=6), 6), dev, "small after the hub")
    check_sort(stb, oracle, as_s16(M.ladder(65535, 300, seed=5), 5), dev, "mid after small")
    check_sort(stb, oracle, as_s16(M.neighbours((1, 1, 1), seed=7, flags=True), 7), dev, "neighbours after mid")

    tree = as_s16(M.ties(3 * 4096 + 1, seed=8, hub=True), 8)
    stream = M.write(tree)
    dev.deserialize(stream)
    dev.sort()
    dev.sort()
    ref = oracle.deserialize(stream, 16)
    ref.sort()
    ref.sort()
    assert_tree(dev, M.sort(M.sort(tree)), "sorted twice")
    assert dev.serialize() == ref.serialize()

    fresh = stb.SharedTree(16).deserialize(stream)
    twin = fresh.clone()
    twin.sort()
    once = oracle.deserialize(stream, 16)
    once.sort()
    assert twin.serialize() == once.serialize()
    assert fresh.serialize() == stream, "the clone's sort changed the original"
    twin.close()
    fresh.close()
    dev.close()


# ---- streams stb_deserialize rejects ------------------------------------------------------------------------

FLAGGED_NULLS = (M.NULL_IDX | M.MIRROR, M.NULL_IDX | M.TRANSPOSE, M.NULL_IDX | M.MIRROR | M.TRANSPOSE)


def rejected(stb, tree):
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(tree["S"]).deserialize(M.write(tree))
    assert e.value.name == "STB_ERR_BAD_STREAM", str(e.value)
    return str(e.value)


def edited(tree, layer, node, side, value):
    layers = [nodes.copy() for nodes in tree["layers"]]
    layers[layer][node, side] = value
    return dict(tree, layers=layers)


@pytest.mark.parametrize("flagged", FLAGGED_NULLS)
def test_flagged_null_left_child_off_the_edge(stb, flagged):
    """A flagged null (first byte 0xDF / 0xEF / 0xFF, then ff ff ff) as the left child of a top-layer node the root
    does not lead to, in a layer parsed on the host.  Nothing but stb_deserialize touches the tree."""
    tree = M.top_layer(1, odd=True)  # 7 top nodes, the root at 3
    assert "flagged null" in rejected(stb, edited(tree, 1, 0, 0, flagged))


@pytest.mark.parametrize("flagged", FLAGGED_NULLS)
def test_flagged_null_in_device_parsed_layer(stb, flagged):
    tree = M.neighbours((1, 0, 1), seed=1)
    assert len(tree["layers"][1]) > M.SMALL_LAYER
    for node, side in ((0, 0), (1234, 1), (len(tree["layers"][1]) - 1, 1)):
        assert "flagged null" in rejected(stb, edited(tree, 1, node, side, flagged))


@pytest.mark.parametrize("flagged", FLAGGED_NULLS)
def test_flagged_null_on_the_right_edge(stb, flagged):
    """The root's node ends the right edge with a null; flagged, it is rejected before width() walks the edge."""
    tree = M.top_layer(1, odd=True)
    root = tree["root"] & M.IDX_MASK
    assert tree["layers"][1][root, 1] == M.NULL_IDX
    rejected(stb, edited(tree, 1, root, 1, flagged))
    for root_ptr in FLAGGED_NULLS + (M.NULL_IDX,):
        rejected(stb, dict(tree, root=root_ptr))


def test_both_children_null_on_the_right_edge(stb, oracle):
    """The width walk reaches a node whose children are both null: in the top layer, and in layer 0 (the second
    child of the root's node), each also through a mirrored pointer; and in layer 2 through a mirrored pointer."""
    tree = M.top_layer(1, odd=True)
    root = tree["root"] & M.IDX_MASK
    assert "both are null" in rejected(stb, edited(tree, 1, root, 0, M.NULL_IDX))
    even = M.top_layer(2, odd=False)
    second = even["layers"][1][even["root"] & M.IDX_MASK, 1] & M.IDX_MASK
    nulled = edited(edited(even, 0, second, 0, M.NULL_IDX), 0, second, 1, M.NULL_IDX)
    assert "both are null" in rejected(stb, nulled)
    # reached through a mirrored pointer: the walk reads the node's children swapped, and a null composed with the
    # mirror bit would no longer be null, so the check comes before composing.  The mirrored root, the top layer:
    mirrored = dict(edited(tree, 1, root, 0, M.NULL_IDX), root=root | M.MIRROR)
    assert "both are null" in rejected(stb, mirrored)
    # a mirrored pointer of the top layer (layer 3) into layer 2, whose node has no child; and the same into layer 0
    deep = M.neighbours((0, 0, 0), seed=3)
    top, root3 = len(deep["layers"]) - 1, deep["root"] & M.IDX_MASK
    b = deep["layers"][top][root3, 1] & M.IDX_MASK
    deep = edited(deep, top, root3, 1, b | M.MIRROR)
    deep = edited(edited(deep, top - 1, b, 0, M.NULL_IDX), top - 1, b, 1, M.NULL_IDX)
    assert "both are null" in rejected(stb, deep)
    to_leaves = edited(even, 1, even["root"] & M.IDX_MASK, 1, second | M.MIRROR)
    to_leaves = edited(edited(to_leaves, 0, second, 0, M.NULL_IDX), 0, second, 1, M.NULL_IDX)
    assert "both are null" in rejected(stb, to_leaves)
    # the same node off the edge stays readable: nulls away from the right edge are read as they are
    first = even["layers"][1][even["root"] & M.IDX_MASK, 0] & M.IDX_MASK
    off_edge = edited(edited(even, 0, first, 0, M.NULL_IDX), 0, first, 1, M.NULL_IDX)
    dev = stb.SharedTree(12).deserialize(M.write(off_edge))
    assert dev.serialize() == M.write(off_edge)


def test_empty_layers(stb):
    """No leaves, a node layer of no nodes in the middle, and an empty top layer are rejected; a stream with no
    node layer at all already was."""
    null = np.array([[M.NULL_IDX, M.NULL_IDX]], dtype=np.uint32)
    two = M.acgt_leaves(2, 12, 0)
    pair = np.array([[0, 1]], dtype=np.uint32)
    assert "no leaves" in rejected(stb, dict(S=12, root=0, leaves=two[:0], layers=[null]))
    assert "no nodes" in rejected(stb, dict(S=12, root=0, leaves=two, layers=[np.zeros((0, 2), np.uint32), null]))
    assert "no nodes" in rejected(stb, dict(S=12, root=0, leaves=two, layers=[pair, np.zeros((0, 2), np.uint32)]))
    rejected(stb, dict(S=12, root=0, leaves=two, layers=[]))
    ok = dict(S=12, root=0, leaves=two, layers=[pair])
    assert stb.SharedTree(12).deserialize(M.write(ok)).width() == 2


# ---- the full-size synthetic genomes ------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["config3_3100mbp", "config3N_3100mbp"])
def test_radix_passes_of_the_synthetic_genome(stb, name):
    """Builds the 3.1 Gbp genome (plain and with N runs), sorts it with profiling on, and checks that radix_scatter
    ran once per pass that the device histograms call for.  Prints the passes per child layer."""
    import torch
    from test_gpu_parity import _synth_record, build_memory_bound
    rec = _synth_record(name)
    if rec is None:
        pytest.skip(f"tests/golden has no synth record {name}")
    free, _ = torch.cuda.mem_get_info()
    if free < build_memory_bound(rec):
        pytest.skip("not enough free device memory for this size")
    n, S = rec["bases"], rec["dna_size"]
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=rec["seed"], repeat_permille=rec["repeat_permille"])
    if rec["variant"] == "nruns":
        stb.synth_mask(buf, seed=rec["seed"])
    tree = stb.SharedTree(S).build_from_body(buf)
    del buf
    passes = []
    for k in range(tree.depth() - 1):
        cnt = tree.leaf_count() if k == 0 else tree.layer_count(k - 1)
        h = tree.histogram(k, out=torch.empty(cnt, dtype=torch.int64, device="cuda"))
        span = int(h.max() - h.min())
        passes.append(0 if cnt < 2 or span == 0 else (span.bit_length() + 7) // 8)
        del h
    tree.profile(True)
    tree.profile_reset()
    tree.sort()
    scatter = tree.profile_read().get("radix_scatter", {}).get("launches", 0)
    tree.profile(False)
    print(f"{name}: radix passes per child layer {passes}, radix_scatter launches {scatter}")
    assert scatter == sum(passes)
    assert tree.bytes() == rec["post_bytes"]
    tree.close()


def test_histogram_out_must_be_an_integer_cuda_tensor(stb):
    """histogram(out=...) fills 8-byte counts: a float64 or CPU tensor is refused rather than filled with bit patterns."""
    import torch
    tree = M.top_layer(1)
    dev = stb.SharedTree(12).deserialize(M.write(tree))
    n = len(tree["leaves"])
    for bad in (torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.int64),
                torch.zeros(2 * n, dtype=torch.int64, device="cuda")[::2]):
        with pytest.raises(TypeError):
            dev.histogram(0, out=bad)
    got = dev.histogram(0, out=torch.zeros(n, dtype=torch.uint64, device="cuda"))
    assert np.array_equal(got.cpu().numpy(), M.histogram(tree, 0))
