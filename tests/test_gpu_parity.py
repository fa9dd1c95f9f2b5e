"""GPU: the CUDA path, called through the C ABI (ctypes), against the oracle and the
golden values.  Bit-exact everywhere: integer / byte / index work only."""
import hashlib

import numpy as np
import pytest

from conftest import CORPUS_CASES, corpus_text

pytestmark = pytest.mark.gpu


def hexs(a):
    return [f"{int(v):x}" for v in a]


def compare_trees(got, want, what=""):
    """got: genome_compression_b200.SharedTree, want: oracle tree. Reports the first differing table."""
    assert got.depth() == want.depth(), what
    assert got.leaf_count() == want.leaf_count(), what
    assert got.layer_counts() == want.layer_counts(), what
    assert np.array_equal(got.leaves(), want.leaves()), (what, "leaf table")
    for k in range(got.depth() - 1):
        a, b = got.layer(k), want.layer(k)
        if not np.array_equal(a, b):
            bad = np.nonzero((a != b).any(axis=1))[0][:5]
            raise AssertionError(f"{what}: layer {k} differs at nodes {bad}: got {a[bad]}, want {b[bad]}")
    assert got.root() == want.root(), what
    assert got.width() == want.width(), what


def full_check(stb, oracle, text_or_leaves, S, from_text=True, rec=None, what=""):
    tree = stb.SharedTree(S)
    if from_text:
        leaves = oracle.fasta_to_leaves(text_or_leaves, S)
        tree.build_from_fasta(text_or_leaves)
    else:
        leaves = np.asarray(text_or_leaves, dtype=np.uint64)
        tree.build_from_leaves(leaves)
    want = oracle.build(leaves, S)
    compare_trees(tree, want, what + " pre-sort")
    pre = tree.serialize()
    assert pre == want.serialize(), what + " pre-sort stream"
    for k in range(tree.depth() - 1):
        assert np.array_equal(tree.histogram(k), want.histogram(k)), (what, "histogram", k)
    assert np.array_equal(tree.decode(), leaves), what + " decode pre-sort"
    tree.sort()
    want.sort()
    compare_trees(tree, want, what + " post-sort")
    post = tree.serialize()
    assert tree.bytes() == len(post) == want.bytes()
    assert post == want.serialize(), what + " post-sort stream"
    if rec is not None:
        assert len(pre) == rec["pre_bytes"] and hashlib.sha256(pre).hexdigest() == rec["pre_sha256"]
        assert len(post) == rec["post_bytes"] and hashlib.sha256(post).hexdigest() == rec["post_sha256"]
        assert tree.layer_counts() == rec["layer_counts"] and tree.width() == rec["width"]
    n = len(leaves)
    assert np.array_equal(tree.decode(), leaves), what + " decode post-sort"
    text = tree.decode_ascii()
    assert text == b"".join(stb.leaf_to_str(v, S).encode() for v in leaves[:200]) + text[200 * S:]
    assert len(text) == n * S
    rng = np.random.default_rng(n)
    idx = np.concatenate([rng.integers(0, n, min(4 * n, 5000)), [0, n - 1]]).astype(np.uint64)
    assert np.array_equal(tree.random_access(idx), leaves[idx]), what + " random access"
    # sub-range decode
    for first, count in ((0, 1), (n - 1, 1), (n // 3, min(n - n // 3, 777)), (1, n - 1) if n > 1 else (0, 1)):
        assert np.array_equal(tree.decode(first, count), leaves[first:first + count]), (what, first, count)
    # ... as text, into device memory at odd byte offsets (the output kernel stages whole tiles)
    import torch
    whole = b"".join(stb.leaf_to_str(v, S).encode() for v in leaves[:min(n, 6000)])
    for first, count, off in ((0, min(n, 6000), 0), (min(n - 1, 5), min(n - min(n - 1, 5), 4100), 1), (min(n - 1, 2049), 1, 3),
                              (n // 2, min(n - n // 2, 9), 2)):
        if first + count > min(n, 6000):
            continue
        buf = torch.zeros(count * S + 8, dtype=torch.uint8, device="cuda")
        tree.decode_ascii(first, count, out=buf[off:])
        got = bytes(buf.cpu().numpy())
        assert got[off:off + count * S] == whole[first * S:(first + count) * S], (what, first, count, off)
        assert got[:off] == bytes(off) and got[off + count * S:] == bytes(8 - off), (what, "wrote outside the range")
    # deserialize round trip (invariant bits are not stored)
    back = stb.SharedTree(S).deserialize(post)
    assert back.width() == n and back.leaf_count() == tree.leaf_count()
    assert back.serialize() == post
    assert np.array_equal(back.decode(), leaves)
    assert np.array_equal(back.random_access(idx), leaves[idx])
    # copy (tests/test.cpp:275)
    twin = tree.clone()
    assert twin.serialize() == post
    return tree


@pytest.mark.parametrize("name,S", CORPUS_CASES)
def test_corpus(stb, oracle, golden, name, S):
    rec = golden["corpus"]["records"][f"{name}:{S}"]
    full_check(stb, oracle, corpus_text(name), S, rec=rec, what=f"{name}:{S}")


def test_small_vectors(stb, oracle, golden):
    for name, rec in golden["small"].items():
        S = rec["dna_size"]
        leaves = np.array([int(x, 16) for x in rec["input_leaves"]], dtype=np.uint64)
        tree = stb.SharedTree(S).build_from_leaves(leaves)
        assert tree.serialize().hex() == rec["pre_hex"], name
        assert hexs(tree.leaves()) == rec["stored_leaves"], name
        for k, want in enumerate(rec["layers"]):
            assert [f"{int(a):08x}" for a in tree.layer(k).reshape(-1)] == want, (name, k)
            assert [int(c) for c in tree.histogram(k)] == rec["histograms"][k], (name, k)
        tree.sort()
        assert tree.serialize().hex() == rec["post_hex"], name
        assert hexs(tree.decode()) == rec["input_leaves"], name
        full_check(stb, oracle, leaves, S, from_text=False, what=name)


def test_fasta_ingest(stb, oracle, golden):
    for key, rec in golden["fasta"].items():
        text = bytes.fromhex(rec["text_hex"])
        S = rec["dna_size"]
        got = stb.SharedTree(S).pack_fasta(text)
        assert hexs(got) == rec["leaves"], key
        if len(rec["leaves"]):
            full_check(stb, oracle, text, S, what=key)


def test_fasta_wrapped_large(stb, oracle):
    # multi-record, 60-column wrapped, lower/upper case, IUPAC codes, crossing many 64 KiB tiles
    rng = np.random.default_rng(3)
    parts = []
    for r in range(7):
        n = int(rng.integers(50_000, 400_000))
        seq = rng.choice(np.frombuffer(b"ACGTacgtNnRYKMSWBDHV-", dtype=np.uint8), size=n,
                         p=[.2, .2, .2, .2, .04, .04, .04, .04] + [.04 / 13] * 13)
        width = int(rng.choice([60, 70, 80, 61]))
        lines = [seq[i:i + width].tobytes() for i in range(0, n, width)]
        parts.append(b">record %d some description\n" % r + b"\n".join(lines) + b"\n")
    text = b"".join(parts)
    for S in (12, 7):
        want = oracle.fasta_to_leaves(text, S)
        got = stb.SharedTree(S).pack_fasta(text)
        assert np.array_equal(got, want)
    full_check(stb, oracle, text, 12, what="wrapped multi-record")


def test_fasta_line_state_machine(stb, oracle):
    # header/blank runs of every parity (src/fasta_reader.cpp:47-50): data lines that start
    # with '>' are packed as data by the reference (and abort); blank ones vanish.
    cases = [b">h\n\n\nACGTACGTACGTAAAA\n", b"\n\n\n\nACGTACGTACGTCCCC", b">a\n\n>b\nACGTACGTACGTGGGG\n\n\n>c\n\nTTTTACGTACGTGGGG",
             b"ACGTAC\n\nGTACGT\n\n\nACGTACGTACGT\n"]
    for text in cases:
        want = oracle.fasta_to_leaves(text, 4)
        got = stb.SharedTree(4).pack_fasta(text)
        assert np.array_equal(got, want), text
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(4).pack_fasta(b">a\n>b\nACGTACGT\n")  # second header is read as data
    assert e.value.name == "STB_ERR_UNKNOWN_SYMBOL" and "62" in str(e.value)


def test_errors(stb):
    t = stb.SharedTree(12)
    with pytest.raises(stb.StbError) as e:
        t.build_from_fasta(b"ACGTACGTACGTACGTACGTACGx")
    assert e.value.name == "STB_ERR_UNKNOWN_SYMBOL"
    assert str(e.value).endswith("Encountered unknown symbol: 88 (ASCII code 88)")
    # invalid byte inside the dropped tail is never looked at (src/fasta_reader.cpp:59-61)
    assert t.build_from_fasta(b"ACGTACGTACGTACx").width() == 1
    with pytest.raises(stb.StbError) as e:
        t.build_from_fasta(b"ACGTACGTACG\r\nACGTACGTACGTA")
    assert "13" in str(e.value)
    with pytest.raises(stb.StbError) as e:
        t.build_from_fasta(b"ACGT")
    assert e.value.name == "STB_ERR_EMPTY"
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(3).build_from_leaves(np.array([0x1111], dtype=np.uint64))
    assert e.value.name == "STB_ERR_BAD_LEAF"
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(12).width()
    assert e.value.name == "STB_ERR_NOT_BUILT"
    t.build_from_fasta(b"ACGTACGTACGT" * 5)
    with pytest.raises(stb.StbError) as e:
        t.random_access(np.array([5], dtype=np.uint64))
    assert e.value.name == "STB_ERR_OUT_OF_RANGE"
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(12).deserialize(t.serialize()[:9])
    assert e.value.name == "STB_ERR_BAD_STREAM"


def test_deserialize_on_device(stb, oracle):
    """Layers of more than 2048 nodes are parsed on the device (serialize.cu: a 4-state automaton per 32-byte
    chunk, maps composed by a scan): every pointer length, layer starts at every alignment, damaged streams."""
    rng = np.random.default_rng(77)
    for S, n in ((12, 300_000), (3, 200_001), (16, 70_000), (7, 99_999)):
        # 1-, 2- and 3-byte pointers (4-byte ones need more than 1 052 688 items in a layer: test_large_properties)
        nib = np.array([1, 2, 4, 8], dtype=np.uint64)[rng.integers(0, 4, size=(n, S))]
        leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
        if S == 12:
            leaves = np.concatenate([leaves, leaves[:50_000], leaves[::-1][:70_000]])
        want = oracle.build(leaves, S)
        for sort in (False, True):
            if sort:
                want.sort()
            stream = want.serialize()
            back = stb.SharedTree(S).deserialize(stream)
            assert back.layer_counts() == want.layer_counts() and back.leaf_count() == want.leaf_count()
            assert np.array_equal(back.leaves(), want.leaves())
            for k in range(back.depth() - 1):
                got_layer, want_layer = back.layer(k), want.layer(k)
                # the stream does not keep the invariant bit (src/shared_tree.cpp:162)
                assert np.array_equal(got_layer, want_layer & np.uint32(0x7fffffff)), (S, sort, k)
            assert back.serialize() == stream
            assert np.array_equal(back.decode(), leaves)
    # damaged streams: cut inside a large layer, and a pointer that indexes past the layer below
    tree = stb.SharedTree(12).build_from_leaves(leaves[:100_000])
    stream = tree.serialize()
    # (a cut inside the last few bytes is not an error by the format: layers are read "until the stream ends",
    # src/shared_tree.cpp:528-530, so a stream that lost its top layer is a shorter valid stream)
    for cut in (len(stream) // 2, len(stream) // 3, len(stream) - 40_000):
        with pytest.raises(stb.StbError) as e:
            stb.SharedTree(12).deserialize(stream[:cut])
        assert e.value.name == "STB_ERR_BAD_STREAM", cut
    head = 1 + 8 + tree.leaf_count() * 6 + 8  # root, leaf count, leaves, layer 0 count (the root of a tree this deep is a 1-byte pointer)
    bad = bytearray(stream)
    bad[head + 3000:head + 3004] = bytes([0xCF, 0xFF, 0xFF, 0x00])  # segment 3, offset 0xfffff00: far past the leaf table
    with pytest.raises(stb.StbError) as e:
        stb.SharedTree(12).deserialize(bytes(bad))
    assert e.value.name == "STB_ERR_BAD_STREAM"


def test_iupac_and_hash_leaf_path(stb, oracle):
    rng = np.random.default_rng(11)
    codes = np.array([1, 2, 4, 8, 3, 12, 7, 14, 0, 9, 5, 11, 13, 10, 6, 15], dtype=np.uint64)
    for S, n in ((12, 20000), (16, 9000), (13, 5000), (1, 3000), (5, 40000)):
        nib = codes[rng.integers(0, 16, size=(n, S))]
        leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
        leaves[n // 2:n // 2 + n // 4] = leaves[:n // 4]
        if S == 16:  # the leaf whose word equals the table's empty marker
            leaves[[5, 77, 78, n - 1]] = np.uint64(0xFFFFFFFFFFFFFFFF)
        full_check(stb, oracle, leaves, S, from_text=False, what=f"iupac S={S}")


def test_acgt_large_sizes(stb, oracle):
    rng = np.random.default_rng(12)
    for S in (14, 16, 9):  # ACGT-only but beyond / below the direct-table sizes
        n = 30000
        nib = np.array([1, 2, 4, 8], dtype=np.uint64)[rng.integers(0, 4, size=(n, S))]
        leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
        leaves[n // 2:n // 2 + 4096] = leaves[:4096]
        full_check(stb, oracle, leaves, S, from_text=False, what=f"acgt S={S}")


def test_synthetic_matches_oracle_generator(stb, oracle):
    import torch
    n = 3_000_000
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=42, repeat_permille=500)
    got = buf.cpu().numpy()
    want = oracle.synth(n, 42, 500)
    assert np.array_equal(got, want)
    part = torch.empty(100_001, dtype=torch.uint8, device="cuda")
    stb.synth_genome(part, n, first=1_234_567, seed=42, repeat_permille=500)
    assert np.array_equal(part.cpu().numpy(), want[1_234_567:1_234_567 + 100_001])
    reps = oracle.synth_repeats(n, 42, 500)
    covered = int(reps["len"].sum())
    assert 0.35 * n < covered < 0.65 * n
    # the "real genome" variant (N runs + soft-masking): device and CPU twins agree, whole and in parts
    stb.synth_mask(buf, seed=42)
    masked = oracle.synth_mask(want.copy(), 0, 42)
    assert np.array_equal(buf.cpu().numpy(), masked)
    stb.synth_mask(part, first=1_234_567, seed=42)
    assert np.array_equal(part.cpu().numpy(), masked[1_234_567:1_234_567 + 100_001])
    frac_n = float((masked == ord("N")).sum() + (masked == ord("n")).sum()) / n
    assert 0.002 < frac_n < 0.03 and 0.3 < float((masked >= ord("a")).sum()) / n < 0.7


def test_synthetic_tree_parity(stb, oracle):
    import torch
    n = 6_000_000
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=7, repeat_permille=500)
    text = buf.cpu().numpy().tobytes()
    leaves = oracle.fasta_to_leaves(text, 12)
    tree = stb.SharedTree(12).build_from_body(buf)
    want = oracle.build(leaves, 12)
    compare_trees(tree, want, "synthetic 6 Mbp")
    tree.sort()
    want.sort()
    assert tree.serialize() == want.serialize()
    assert tree.leaf_count() < tree.width() and tree.layer_count(0) < tree.width() // 2  # planted repeats dedup


def _synth_record(name):
    """A record of tests/golden/synth.json (made by the unmodified reference) or of synth_large.json (made by the
    oracle, at sizes the reference was not run at)."""
    import json
    from conftest import GOLD
    for f in ("synth.json", "synth_large.json"):
        rec = json.loads((GOLD / f).read_text()).get(name)
        if rec is not None:
            return rec
    return None


# Device workspace of a build, per leaf position. Measured on a B200 (1000 W limit) in a fresh process: the
# device-FASTA build of the 4.5 Gbp text (375 M positions) raised device use by 42.5 GiB. That figure includes
# the text and its FASTA copy (9.1 GB) and the extracted body (4.5 GB), which leaves about 85 B per position.
BUILD_BYTES_PER_POSITION = 96


def build_memory_bound(rec):
    """Free device memory a test that holds the text and builds it wants: text bytes + workspace per leaf
    position (which is what the build's tables follow, whatever the leaf size) + 4 GB."""
    return rec["bases"] + BUILD_BYTES_PER_POSITION * (rec["bases"] // rec["dna_size"]) + (4 << 30)


def check_record(stb, tree, rec, tables=True):
    """tree (built, not yet sorted) against a synth record: shape, optionally the leaf table and every raw node
    layer, the stream before and after sort(), and the answers to the record's seeded queries. Sorts the tree."""
    assert tree.width() == rec["width"] and tree.depth() == rec["depth"]
    assert tree.leaf_count() == rec["leaves"] and tree.node_count() == rec["nodes"]
    assert tree.layer_counts() == rec["layer_counts"]
    if tables:  # every table, word for word
        assert hashlib.sha256(tree.leaves().tobytes()).hexdigest() == rec["pre_leaves_sha256"]
        for k, want in enumerate(rec["pre_layer_sha256"]):
            assert hashlib.sha256(tree.layer(k).tobytes()).hexdigest() == want, f"node layer {k} differs from the record's"
    pre = tree.serialize()
    assert len(pre) == rec["pre_bytes"] and hashlib.sha256(pre).hexdigest() == rec["pre_sha256"]
    del pre
    tree.sort()
    assert tree.bytes() == rec["post_bytes"]
    post = tree.serialize()
    assert hashlib.sha256(post).hexdigest() == rec["post_sha256"]
    del post
    idx = stb.query_indices(rec["seed"], rec["queries"], rec["width"])
    ans = tree.random_access(idx)
    assert [f"{int(v):x}" for v in ans[:8]] == rec["query_first8"]
    assert hashlib.sha256(np.ascontiguousarray(ans, dtype="<u8").tobytes()).hexdigest() == rec["query_answers_sha256"]


LARGE_CASES = ("beyond4g_4500mbp", "beyond4gN_4500mbp", "ceiling_s1")


@pytest.mark.parametrize("name,entry", [("mid_50mbp", "device"), ("mid_50mbp", "host"), ("large_260mbp", "device"),
                                        ("large_260mbp", "host"), ("config3_3100mbp", "device"), ("config3_3100mbp", "host"),
                                        ("largeN_260mbp", "device"), ("largeN_260mbp", "host"),
                                        ("config3N_3100mbp", "device"), ("config3N_3100mbp", "host")] +
                         [(name, entry) for name in LARGE_CASES for entry in ("device", "host")])
def test_synth_reference_golden(stb, name, entry):
    """Full-size synthetic genomes against records of the same generated text: per-layer node counts, sha256 of the
    leaf table and of every raw node layer, of the stream before and after sort_tree (compress.cpp:183-200,
    src/shared_tree.cpp:488-513) and of the operator[] answers (:268-291).
    tests/golden/synth.json (BASELINE.json configs 3 / 5, up to 3.1 Gbp) was written by the UNMODIFIED reference
    (oracle/gen_golden_synth.py). tests/golden/synth_large.json was written by the oracle (oracle/gen_golden_large.py,
    "made_by": "oracle.c"): 4.5 Gbp at dna_size 12, past 2^32 text bytes, plain and with N runs, and 2^30 - 1 bases
    at dna_size 1, the largest input the build accepts. tests/test_golden_large_host.py checks that the oracle path
    reproduces the reference's records."""
    import torch
    rec = _synth_record(name)
    if rec is None:
        pytest.skip(f"tests/golden has no synth record {name} (oracle/gen_golden_synth.py, oracle/gen_golden_large.py)")
    n, S = rec["bases"], rec["dna_size"]
    free, _ = torch.cuda.mem_get_info()
    if free < build_memory_bound(rec):
        pytest.skip("not enough free device memory for this size")
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=rec["seed"], repeat_permille=rec["repeat_permille"])
    if rec["variant"] == "nruns":  # N runs (1 % of the bases) and soft-masked lower case: a real assembly's shape
        stb.synth_mask(buf, seed=rec["seed"])
    tree = stb.SharedTree(S)
    if entry == "host":  # stb_build_from_body(STB_HOST): the chunked build behind the copy
        host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        host.copy_(buf)
        torch.cuda.synchronize()
        del buf
        tree.build_from_body(host)
        del host
    else:
        tree.build_from_body(buf)
        del buf
    check_record(stb, tree, rec, tables=entry == "device")
    tree.close()


def test_large_properties(stb):
    """Sizes the oracle would not finish quickly: size-independent properties only."""
    import torch
    n = 260_000_000  # leaf level > 16384 CTA tiles: the two-level scan runs
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=1, repeat_permille=500)
    tree = stb.SharedTree(12).build_from_body(buf)
    w = tree.width()
    assert w == n // 12
    counts = tree.layer_counts()
    assert counts[-1] == 1 and len(counts) == int(np.ceil(np.log2(w)))
    tree.sort()
    out = torch.empty(w * 12, dtype=torch.uint8, device="cuda")
    tree.decode_ascii(out=out)
    assert torch.equal(out, buf[:w * 12])  # encode -> decode round trip
    idx = torch.randint(0, w, (1_000_000,), device="cuda", dtype=torch.int64)
    got = torch.empty(1_000_000, dtype=torch.int64, device="cuda")
    tree.random_access(idx, out=got)
    leaves = torch.empty(w, dtype=torch.int64, device="cuda")
    tree.decode(out=leaves)
    assert torch.equal(got, leaves[idx])
    # stream round trip: serialize -> deserialize -> identical stream and content
    stream = tree.serialize()
    assert len(stream) == tree.bytes()
    back = stb.SharedTree(12).deserialize(stream)
    assert back.width() == w
    out2 = torch.empty(w * 12, dtype=torch.uint8, device="cuda")
    back.decode_ascii(out=out2)
    assert torch.equal(out2, out)
    assert hashlib.sha256(back.serialize()).digest() == hashlib.sha256(stream).digest()
    # idempotence: sorting a sorted tree changes nothing
    tree.sort()
    assert hashlib.sha256(tree.serialize()).digest() == hashlib.sha256(stream).digest()


@pytest.mark.parametrize("options", [
    ["bucket_min=1"],
    ["bucket_min=1", "bucket_levels=9", "coop_max=0"],
    ["bucket_min=1", "bucket_cap=16", "bucket_levels=2"],
    ["bucket_min=1", "bucket_levels=3", "bucket_slack_permille=0", "bucket_headroom=0"],
    ["coop_max=0"],
    ["coop_max=0", "child_filter=0", "locality=0"],
    ["coop_max=65536"],
    ["stream_chunk_log2=12", "stream_min_chunks=2"],
    ["stream_chunk_log2=15", "stream_min_chunks=2", "bucket_min=1"],
])
def test_large_input_paths_forced_small(options):
    """The on-chip (bucketed) dedup, its overflow fallback, the cooperative middle launch and the
    streaming host build, forced onto inputs the oracle can check (tests/forced_paths_check.py)."""
    import subprocess
    import sys
    from conftest import ROOT
    res = subprocess.run([sys.executable, str(ROOT / "tests" / "forced_paths_check.py"), *options],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "forced_paths_check ok" in res.stdout, res.stdout[-2000:] + res.stderr[-3000:]
