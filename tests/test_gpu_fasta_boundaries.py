"""GPU: FASTA text -> body -> leaves and trees (csrc/ingest.cu, and the streaming build in csrc/build.cu) with lines,
headers and runs of header and blank lines placed on every boundary the kernels compose across: 16-byte thread
chunks, 512-byte warps, 4 KiB sub-tiles, 64 KiB tiles, the 16 MiB steps of the single-CTA scans and the text chunks
of the streaming build.  A wrong composition at one of them drops or keeps one line, which shifts the body and every
node id after it; everything here is compared with the oracle's sequential reading (oracle/oracle.c).

The texts come from tests/fasta_scan_model.py, whose restatement of the kernels is checked on the CPU by
tests/test_fasta_scan_model_host.py.  Streaming cases assert how many text chunks the line kernels ran on, so a
case that fell back to the one-shot path fails instead of passing untested."""
import gc
import hashlib
import json
import re

import numpy as np
import pytest

import fasta_scan_model as M
from conftest import GOLD

pytestmark = pytest.mark.gpu

R = M.REAL
KiB = 1 << 10
CLASS_LEN = {"chunk": 24 * KiB, "warp": 48 * KiB, "sub": 160 * KiB, "tile": 1200 * KiB}


@pytest.fixture(autouse=True)
def release_device_memory():
    yield
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def sha(b) -> str:
    return hashlib.sha256(b if isinstance(b, bytes) else np.ascontiguousarray(b).tobytes()).hexdigest()


def on_device(text: bytes, offset: int = 0):
    """The text in device memory, starting `offset` bytes into a 16-byte aligned allocation."""
    import torch
    buf = torch.zeros(len(text) + offset + 16, dtype=torch.uint8, device="cuda")
    if text:
        buf[offset:offset + len(text)] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    view = buf[offset:offset + len(text)]
    assert view.data_ptr() % 16 == offset % 16
    return view


def fasta_launches(tree) -> int:
    return tree.profile_read().get("fasta_lines", {}).get("launches", 0)


def leaf_launches(tree) -> int:
    return tree.profile_read().get("leaf_insert", {}).get("launches", 0)


def streaming_tree(stb, S, chunk_log2):
    tree = stb.SharedTree(S).set_option("stream_chunk_log2", chunk_log2).set_option("stream_min_chunks", 2)
    tree.profile(True)
    tree.profile_reset()
    return tree


def text_chunks(text, S, chunk_log2):
    return -(-len(text) // M.text_chunk_bytes(S, chunk_log2))


def check_tree(tree, oracle, leaves, S, what):
    want = oracle.build(leaves, S)
    assert tree.leaf_count() == want.leaf_count() and tree.width() == len(leaves), what
    assert tree.layer_counts() == want.layer_counts(), what
    assert tree.serialize() == want.serialize(), f"{what}: pre-sort stream"
    tree.sort()
    want.sort()
    assert tree.serialize() == want.serialize(), f"{what}: post-sort stream"


def build_streamed(stb, oracle, text, S, chunk_log2, what, leaves=None):
    """build_from_fasta from host bytes through the streaming build, checked against the oracle."""
    leaves = oracle.fasta_to_leaves(text, S) if leaves is None else leaves
    tree = streaming_tree(stb, S, chunk_log2)
    tree.build_from_fasta(text)
    assert fasta_launches(tree) == text_chunks(text, S, chunk_log2), f"{what}: not built chunk by chunk"
    check_tree(tree, oracle, leaves, S, what)
    return tree


def class_text(cls, rot):
    period = R.classes()[cls]
    n = CLASS_LEN[cls]
    rng = np.random.default_rng([11, period, rot])
    return M.adversarial_text(rng, R, M.boundary_targets(period, n, rot), n, large=0.3 if cls == "tile" else 0.0,
                              head=("", "nl", "gt")[rot % 3], tail=("", "nofinal", "header", "blanks")[rot % 4])


# ---- every boundary class, every entry -----------------------------------------------------------------------
@pytest.mark.parametrize("cls", ["chunk", "warp", "sub", "tile"])
def test_boundary_classes(stb, oracle, cls):
    """Seven texts per class, one per shift rotation.  Each is read at dna_size 1 (one leaf per body byte) from an
    aligned device tensor, from a device slice at an odd offset and from host bytes; then packed and built at one
    of dna_size 5, 12 (ACGT-12 leaf kernel) and 16 (hashed leaf level)."""
    k = list(CLASS_LEN).index(cls)
    for rot in range(7):
        text = class_text(cls, rot)
        what = f"{cls} rotation {rot}"
        body = oracle.fasta_to_leaves(text, 1)
        offset = (7 * k + rot) % 15 + 1
        for src in (on_device(text), on_device(text, offset), text):
            assert np.array_equal(stb.SharedTree(1).pack_fasta(src), body), (what, "body", type(src))
        S = (5, 12, 16)[(rot + k) % 3]
        leaves = oracle.fasta_to_leaves(text, S)
        assert np.array_equal(stb.SharedTree(S).pack_fasta(text), leaves), (what, S)
        src = (on_device(text), on_device(text, 16 - offset), text)[rot % 3]
        check_tree(stb.SharedTree(S).build_from_fasta(src), oracle, leaves, S, f"{what} dna_size {S}")


def test_past_one_scan_step(stb, oracle):
    """Over 32 MiB through the one-shot device path: both single-CTA scans loop three times, and events sit on
    every tile boundary, among them tiles 255 / 256 and 511 / 512."""
    for rot in (0, 4):
        rng = np.random.default_rng([12, rot])
        n = 2 * R.step + 5 * R.tile + 123
        targets = sorted(set(M.boundary_targets(R.tile, n, rot) + [b * R.tile + d for b in (255, 256, 511, 512) for d in (-3, 0, 3)]))
        text = M.adversarial_text(rng, R, targets, n, large=0.1, tail="nofinal")
        body = oracle.fasta_to_leaves(text, 1)
        dev = on_device(text)
        assert np.array_equal(stb.SharedTree(1).pack_fasta(dev), body), ("body", rot)
        del body
        leaves = oracle.fasta_to_leaves(text, 12)
        tree = stb.SharedTree(12)
        tree.profile(True)
        tree.build_from_fasta(dev)
        assert fasta_launches(tree) == 1
        check_tree(tree, oracle, leaves, 12, f"one-shot, rotation {rot}")
        if rot == 0:  # the same text streamed in 384 KiB text chunks
            build_streamed(stb, oracle, text, 12, 16, "streamed past one scan step", leaves)


# ---- the streaming build --------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,chunk_log2", [(1, 12), (5, 12), (12, 12), (5, 14), (12, 14), (12, 16)])
def test_streaming_chunk_boundaries(stb, oracle, S, chunk_log2):
    """Events on every text-chunk and tile boundary; leaf chunks of 2^chunk_log2 leaves."""
    step = M.text_chunk_bytes(S, chunk_log2)
    n = max(4 * step + 1000, int(2.6 * S * (1 << chunk_log2)))
    for rot in (0, 3):
        rng = np.random.default_rng([13, S, chunk_log2, rot])
        targets = sorted(set(M.boundary_targets(step, n, rot) + M.boundary_targets(R.tile, n, rot + 2)))
        text = M.adversarial_text(rng, R, targets, n, large=0.3, head=("gt", "nl")[rot % 2], tail=("header", "blanks")[rot % 2])
        assert text_chunks(text, S, chunk_log2) >= 4
        build_streamed(stb, oracle, text, S, chunk_log2, f"dna_size {S}, 2^{chunk_log2}-leaf chunks, rotation {rot}")


def exact_length(rng, text: bytes, n: int, last: bytes = b"A") -> bytes:
    """The text cut or padded with data lines to n bytes, ending in `last`."""
    text = text[:n - 1]
    gap = n - 1 - len(text)
    if gap == 1:
        text += b"C"
    elif gap:
        text += M.data_lines(rng, gap)
    return text + last


def test_streaming_edges(stb, oracle):
    """S = 12 in leaf chunks of 4096 leaves (49152 body bytes) and 64 KiB text chunks."""
    S, log2 = 12, 12
    chunk_body = S << log2
    rng = np.random.default_rng(14)
    cases = []
    # hardly any body next to the text: no leaf chunk fills, the stream's body is built in one shot
    cases.append(("no leaf chunk", M.header(rng, 150_000) + b"\n" + M.data_lines(rng, 30_000) + M.header(rng, 9)))
    # the body ends exactly on a leaf-chunk boundary; the text chunks after it hold only headers and blank lines
    for chunks in (1, 2, 3):
        body = M.letters(rng, chunk_body * chunks)
        text = b"".join(body[i:i + 61] + b"\n" for i in range(0, len(body), 61))
        text += (M.header(rng, 40) + b"\n\n") * 5000 + b"\n" * 70_001
        assert len(oracle.fasta_body(text)) == chunk_body * chunks
        cases.append((f"body ends on leaf chunk {chunks}", text))
    # the last text chunk is one byte long; the text is a multiple of 64 KiB
    base = M.adversarial_text(rng, R, M.boundary_targets(R.tile, 5 * R.tile, 1), 5 * R.tile, large=0.3)
    for n, last in ((4 * R.tile + 1, b"G"), (4 * R.tile + 1, b"\n"), (4 * R.tile, b"T"), (5 * R.tile, b"\n")):
        cases.append((f"{n} bytes ending in {last!r}", exact_length(rng, base, n, last)))
    # the dropped tail (body length mod dna_size) holds a byte outside the table; it is never looked at
    for tail in (b"X", b"ACGTACGTAC>", b"\x00"):
        body = M.letters(rng, 3 * chunk_body + 777)
        body = body[:len(body) - len(body) % S] + tail
        text = b">h\n" + b"\n".join(body[i:i + 61] for i in range(0, len(body), 61)) + b"\n>last header\n"
        cases.append((f"dropped tail {tail!r}", text))
    for what, text in cases:
        build_streamed(stb, oracle, text, S, log2, what)


# ---- errors ---------------------------------------------------------------------------------------------------
def header_as_data(rng, p, blank_run=0):
    """Data lines, then a '>' line read as data whose '>' is byte p: after a header, or after an odd run of blank
    lines.  None when no data lines fit in front (they need two bytes at least)."""
    lead = b"\n" * blank_run if blank_run else M.header(rng, int(rng.integers(1, 6))) + b"\n"
    if p - len(lead) == 1 and not blank_run:
        lead = b">" + lead
    gap = p - len(lead)
    if gap < 0 or gap == 1:
        return None
    return M.data_lines(rng, gap) + lead + M.header(rng, 8) + b"\n" + M.data_lines(rng, 600)


@pytest.mark.parametrize("period", [16, 512, 4096, 65536])
def test_header_read_as_data(stb, oracle, period):
    """A '>' line read as data on each boundary class: the reference exits with 'unknown symbol 62'."""
    rng = np.random.default_rng([15, period])
    for b in (1, 2):
        for d in range(-3, 4):
            p = b * period + d
            for blank_run in (0, 1, 3) if period < 65536 else (0, period + 1):
                text = header_as_data(rng, p, blank_run)
                if text is None:
                    continue
                assert text[p] == M.GT and text[p - 1] == M.NL
                with pytest.raises(ValueError, match="unknown symbol 62"):
                    oracle.fasta_to_leaves(text, 1)
                with pytest.raises(stb.StbError) as e:
                    stb.SharedTree(1).pack_fasta(on_device(text, (b + d) % 16))
                assert e.value.name == "STB_ERR_UNKNOWN_SYMBOL" and str(e.value).endswith("(ASCII code 62)"), (p, blank_run)


def test_all_headers_is_empty(stb):
    rng = np.random.default_rng(16)
    text = b"".join(M.header(rng, int(rng.integers(1, 90))) + b"\n\n" for _ in range(6000))
    assert len(text) > 3 * 65536
    assert len(stb.SharedTree(1).pack_fasta(text)) == 0
    for src in (on_device(text), text):
        with pytest.raises(stb.StbError) as e:
            stb.SharedTree(12).build_from_fasta(src)
        assert e.value.name == "STB_ERR_EMPTY"
    tree = streaming_tree(stb, 12, 12)
    with pytest.raises(stb.StbError) as e:
        tree.build_from_fasta(text)
    assert e.value.name == "STB_ERR_EMPTY"
    assert fasta_launches(tree) == text_chunks(text, 12, 12)


def oracle_bad_symbol(oracle, text, S) -> int:
    with pytest.raises(ValueError) as e:
        oracle.fasta_to_leaves(text, S)
    return int(re.fullmatch(r"unknown symbol (\d+)", str(e.value)).group(1))


def expect_unknown(stb, tree, build, want: int, what):
    with pytest.raises(stb.StbError) as e:
        build(tree)
    assert e.value.name == "STB_ERR_UNKNOWN_SYMBOL", what
    assert str(e.value).endswith(f"Encountered unknown symbol: {want} (ASCII code {want})"), (what, str(e.value))


# (first bad byte, offset in its leaf chunk), (later bad byte, offset in its leaf chunk): an offset counted from its
# own chunk's start picks the later byte in each of them
TWO_BAD = [((ord("X"), 3000), (ord("J"), 500)), ((ord("J"), 3000), (ord("X"), 500)), ((ord("X"), 1234), (ord("J"), 1234))]


def body_with_two_bad(rng, S, chunk_body, first, later, later_chunk=2, n_chunks=4):
    body = bytearray(M.letters(rng, n_chunks * chunk_body + 5))
    body[first[1]] = first[0]
    body[later_chunk * chunk_body + later[1]] = later[0]
    return bytes(body)


def as_fasta(body: bytes, width=60) -> bytes:
    return b">chr1 two bad bytes\n" + b"\n".join(body[i:i + width] for i in range(0, len(body), width)) + b"\n"


@pytest.mark.parametrize("S", [12, 5])
def test_first_unknown_symbol_streaming(stb, oracle, S):
    """Two bad bytes in different leaf chunks of the streaming build (host body and host FASTA): the error names
    the first in body order, as the reference does.  Then the same handle builds a clean input."""
    log2 = 12
    chunk_body = S << log2
    rng = np.random.default_rng([17, S])
    for first, later in TWO_BAD:
        body = body_with_two_bad(rng, S, chunk_body, first, later)
        want = oracle_bad_symbol(oracle, body, S)
        assert want == first[0]
        clean = body.replace(b"X", b"A").replace(b"J", b"C")
        tree = streaming_tree(stb, S, log2)
        expect_unknown(stb, tree, lambda t: t.build_from_body(body), want, ("host body", S, first, later))
        assert leaf_launches(tree) == -(-(len(body) // S) // (1 << log2)), "host body: not built chunk by chunk"
        tree.profile_reset()
        tree.build_from_body(clean)
        check_tree(tree, oracle, oracle.fasta_to_leaves(clean, S), S, "clean host body after the error")

        text, clean_text = as_fasta(body), as_fasta(clean)
        assert oracle_bad_symbol(oracle, text, S) == want
        tree = streaming_tree(stb, S, log2)
        expect_unknown(stb, tree, lambda t: t.build_from_fasta(text), want, ("host FASTA", S, first, later))
        assert fasta_launches(tree) == text_chunks(text, S, log2), "host FASTA: not built chunk by chunk"
        tree.profile_reset()
        tree.build_from_fasta(clean_text)
        assert fasta_launches(tree) == text_chunks(clean_text, S, log2)
        check_tree(tree, oracle, oracle.fasta_to_leaves(clean_text, S), S, "clean host FASTA after the error")


def test_first_unknown_symbol_split_leaf_level(stb, oracle):
    """The one-shot ACGT-12 leaf level in two launches (a 2^12-leaf prefix, then the rest in lookup mode): bad
    bytes on both sides of the split."""
    S, P = 12, 1 << 12
    rng = np.random.default_rng(18)
    for first, later in TWO_BAD:
        body = body_with_two_bad(rng, S, P * S, first, later, later_chunk=1, n_chunks=3)
        want = oracle_bad_symbol(oracle, body, S)
        tree = stb.SharedTree(S).set_option("bucket_min", 1).set_option("leaf_prefix_log2", 12)
        expect_unknown(stb, tree, lambda t: t.build_from_body(on_device(body)), want, ("split leaf level", first, later))
        clean = body.replace(b"X", b"A").replace(b"J", b"C")
        tree.profile(True)
        tree.build_from_body(on_device(clean))
        assert leaf_launches(tree) == 2, "the leaf level was not split"
        check_tree(tree, oracle, oracle.fasta_to_leaves(clean, S), S, "clean body after the error")


def test_first_unknown_symbol_1gb_host_body(stb):
    """About 1 GB of host body at default options (leaf chunks of 2^24 leaves): 'X' early in chunk 0, 'J' early in
    chunk 3 at a smaller in-chunk offset."""
    import torch
    S = 12
    n0 = 5 * (1 << 24) + 1001
    free, _ = torch.cuda.mem_get_info()
    if free < 8 * n0 * S:
        pytest.skip(f"needs {8 * n0 * S / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    dev = torch.empty(n0 * S, dtype=torch.uint8, device="cuda")
    stb.synth_genome(dev, dev.numel(), seed=19, repeat_permille=500)
    host = torch.empty(dev.numel(), dtype=torch.uint8, pin_memory=True)
    host.copy_(dev)
    torch.cuda.synchronize()
    chunk = (1 << 24) * S
    host[3000] = ord("X")
    host[3 * chunk + 500] = ord("J")
    tree = stb.SharedTree(S)
    tree.profile(True)
    expect_unknown(stb, tree, lambda t: t.build_from_body(host), ord("X"), "1 GB host body")
    assert leaf_launches(tree) == 6
    host[3000] = dev[3000].item()
    host[3 * chunk + 500] = dev[3 * chunk + 500].item()
    tree.build_from_body(host)
    want = stb.SharedTree(S).build_from_body(dev)  # the one-shot device build of the same body
    assert tree.layer_counts() == want.layer_counts()
    assert sha(tree.serialize()) == sha(want.serialize())


# ---- the texts certified against the reference -----------------------------------------------------------------
def test_reference_fuzz_replay(stb):
    """tests/golden/reference_fuzz.json's FASTA texts, regenerated: leaves and both streams, from device and host."""
    from oracle.gen_golden_fuzz import FASTA_CASES, random_fasta
    recs = json.loads((GOLD / "reference_fuzz.json").read_text())["fasta_ingest_fuzz"]
    rng = np.random.default_rng(10)
    done = 0
    for k, (S, n_bases, alphabet, width, records, blanks) in enumerate(FASTA_CASES):
        if n_bases < S:
            continue
        text = random_fasta(rng, n_bases, alphabet, width, records, blanks)
        rec = recs[done]
        done += 1
        assert rec["case"] == k and sha(text) == rec["inputs"], f"case {k}: the generator drifted"
        leaves = stb.SharedTree(S).pack_fasta(text)
        assert len(leaves) == rec["leaves"] and sha(leaves) == rec["leaves_sha256"], k
        if not rec["leaves"]:
            continue
        for src in (on_device(text), on_device(text, 1 + k), text):
            tree = stb.SharedTree(S).build_from_fasta(src)
            assert sha(tree.serialize()) == rec["pre_sha256"], k
            tree.sort()
            assert sha(tree.serialize()) == rec["post_sha256"], k
    assert done == len(recs)
