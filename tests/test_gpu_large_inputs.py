"""GPU: inputs past 2^32 text bytes and at the 2^30 leaf-position ceiling, against tests/golden/synth_large.json
(oracle/gen_golden_large.py) and the oracle.

A 32-bit truncation of a byte offset or a leaf position on these paths does not fault: it reads earlier text or
writes an earlier output slot of the same buffer. So every output here is compared in full (or by sha256 against a
record), and every partial write is checked for the bytes around it. One input is resident at a time and each is
freed before the next test: the device may be shared."""
import gc
import hashlib
import json

import numpy as np
import pytest

from conftest import GOLD
from test_gpu_parity import build_memory_bound, check_record

pytestmark = pytest.mark.gpu

B4G = 1 << 32
MiB = 1 << 20


def record(name):
    path = GOLD / "synth_large.json"
    rec = json.loads(path.read_text()).get(name) if path.exists() else None
    if rec is None:
        pytest.skip(f"tests/golden/synth_large.json has no record {name} (oracle/gen_golden_large.py {name})")
    return rec


def need_device(nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


def synth_text(stb, rec, n=None):
    """The record's text, generated on the device (n bytes: more than the record's for the size-limit tests)."""
    import torch
    buf = torch.empty(n or rec["bases"], dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf[:rec["bases"]], rec["bases"], seed=rec["seed"], repeat_permille=rec["repeat_permille"])
    if rec["variant"] == "nruns":
        stb.synth_mask(buf[:rec["bases"]], seed=rec["seed"])
    return buf


def pinned_copy(t):
    import torch
    host = torch.empty(t.numel(), dtype=torch.uint8, pin_memory=True)
    host.copy_(t)
    torch.cuda.synchronize()
    return host


@pytest.fixture(autouse=True)
def release_device_memory():
    yield
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("name", ["beyond4g_4500mbp", "beyond4gN_4500mbp"])
def test_generator_past_4g(stb, oracle, name):
    """The goldens assume the device generator and its CPU twin agree past byte 2^32 and at the end of the text."""
    import torch
    rec = record(name)
    n = rec["bases"]
    for first in (B4G - MiB, n - MiB):
        count = min(2 * MiB, n - first)
        part = torch.empty(count, dtype=torch.uint8, device="cuda")
        stb.synth_genome(part, n, first=first, seed=rec["seed"], repeat_permille=rec["repeat_permille"])
        want = oracle.synth(n, rec["seed"], rec["repeat_permille"], first=first, count=count)
        if rec["variant"] == "nruns":
            stb.synth_mask(part, first=first, seed=rec["seed"])
            oracle.synth_mask(want, first, rec["seed"])
        assert np.array_equal(part.cpu().numpy(), want), (name, first)


def test_fasta_past_4g(stb):
    """The 4.5 Gbp text wrapped as FASTA (a header, then 60-column lines): about 4.58 GB, so the line automaton's
    64-bit counts and the body offsets pass 2^32. Built from device memory (one-shot extraction) and from host
    memory (extraction and build chunk by chunk behind the copy)."""
    import torch
    rec = record("beyond4g_4500mbp")
    n, cols = rec["bases"], 60
    assert n % cols == 0
    header = b">beyond4g synthetic, 60 columns\n"
    need_device(2 * n + build_memory_bound(rec))
    body = synth_text(stb, rec)
    lines = n // cols
    fasta = torch.empty(len(header) + lines * (cols + 1), dtype=torch.uint8, device="cuda")
    fasta[:len(header)] = torch.frombuffer(bytearray(header), dtype=torch.uint8).cuda()
    grid = fasta[len(header):].view(lines, cols + 1)
    grid[:, :cols] = body.view(lines, cols)
    grid[:, cols] = ord("\n")
    del body, grid
    assert fasta.numel() > B4G
    for entry in ("device", "host"):
        tree = stb.SharedTree(12)
        if entry == "host":
            host = pinned_copy(fasta)
            del fasta
            tree.build_from_fasta(host)
            del host
        else:
            tree.build_from_fasta(fasta)
        assert tree.width() == rec["width"] and tree.layer_counts() == rec["layer_counts"], entry
        pre = tree.serialize()
        assert len(pre) == rec["pre_bytes"] and hashlib.sha256(pre).hexdigest() == rec["pre_sha256"], entry
        del pre
        tree.close()


def test_decode_past_4g(stb, oracle):
    """Decode output offsets past byte 2^32: the whole width as text into an aligned buffer (16-byte stores) and at
    byte offset 1 (every tile staged and written by bytes), to pinned host memory, a range straddling byte 2^32 at
    odd byte offsets, and packed leaves into a destination that is 8- but not 16-byte aligned."""
    import torch
    rec = record("beyond4g_4500mbp")
    n, S = rec["bases"], 12
    need_device(2 * n + build_memory_bound(rec))
    text = synth_text(stb, rec)
    tree = stb.SharedTree(S).build_from_body(text)
    tree.sort()
    w = tree.width()
    assert w * S == n

    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    assert out.data_ptr() % 16 == 0
    tree.decode_ascii(out=out)
    assert torch.equal(out, text), "whole-width decode into a 16-byte aligned buffer"
    del out
    guard = torch.full((n + 16,), 0xA5, dtype=torch.uint8, device="cuda")
    tree.decode_ascii(out=guard[1:1 + n])
    assert torch.equal(guard[1:1 + n], text), "whole-width decode at byte offset 1"
    assert int(guard[0]) == 0xA5 and bool((guard[1 + n:] == 0xA5).all()), "wrote outside [1, 1 + n)"
    del guard

    host = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    tree.decode_ascii_to_host(host)
    assert hashlib.sha256(host.numpy()).hexdigest() == rec["text_sha256"], "decode to pinned host memory"
    del host

    first, count = B4G // S - 3, 1_000_003
    assert first * S < B4G < (first + count) * S
    want = text[first * S:(first + count) * S]
    for off in (0, 1, 3):
        buf = torch.zeros(count * S + 8, dtype=torch.uint8, device="cuda")
        tree.decode_ascii(first, count, out=buf[off:])
        assert torch.equal(buf[off:off + count * S], want), ("range across byte 2^32", off)
        assert not bool(buf[:off].any()) and not bool(buf[off + count * S:].any()), ("wrote outside the range", off)

    for f in (first, first & ~7):  # a range start inside an 8-leaf group, and one on a group boundary
        exp = oracle.fasta_to_leaves(text[f * S:(f + count) * S].cpu().numpy(), S)
        leaves = torch.zeros(count + 2, dtype=torch.int64, device="cuda")
        view = leaves[1:1 + count]
        assert view.data_ptr() % 16 == 8
        tree.decode(f, count, out=view)
        got = leaves.cpu().numpy().view(np.uint64)
        assert np.array_equal(got[1:1 + count], exp), ("packed leaves into an 8-byte aligned view", f)
        assert got[0] == 0 and got[-1] == 0, ("wrote outside the view", f)
    tree.close()


@pytest.mark.parametrize("name", ["beyond4g_4500mbp", "ceiling_s1"])
def test_stream_round_trip(stb, name):
    """deserialize() of a multi-GB stream (copied in chunks, 4-byte pointers in the widest layers) gives the same
    stream back and decodes to the text."""
    import torch
    rec = record(name)
    n, S = rec["bases"], rec["dna_size"]
    need_device(2 * n + build_memory_bound(rec))
    text = synth_text(stb, rec)
    tree = stb.SharedTree(S).build_from_body(text)
    tree.sort()
    post = tree.serialize()
    tree.close()
    del tree
    assert hashlib.sha256(post).hexdigest() == rec["post_sha256"]
    back = stb.SharedTree(S).deserialize(post)
    del post
    assert back.width() == rec["width"] and back.layer_counts() == rec["layer_counts"]
    again = back.serialize()
    assert len(again) == rec["post_bytes"] and hashlib.sha256(again).hexdigest() == rec["post_sha256"]
    del again
    out = torch.empty(rec["width"] * S, dtype=torch.uint8, device="cuda")
    back.decode_ascii(out=out)
    assert torch.equal(out, text[:rec["width"] * S])
    back.close()


def test_unknown_symbol_past_4g(stb):
    """A byte outside the alphabet past 2^32 is found, and reported as the reference reports it."""
    rec = record("beyond4g_4500mbp")
    need_device(rec["bases"] + build_memory_bound(rec))
    text = synth_text(stb, rec)
    text[B4G + 7] = ord("X")
    tree = stb.SharedTree(12)
    with pytest.raises(stb.StbError) as e:
        tree.build_from_body(text)
    assert e.value.name == "STB_ERR_UNKNOWN_SYMBOL"
    assert str(e.value).endswith("Encountered unknown symbol: 88 (ASCII code 88)")
    tree.close()


def test_position_ceiling(stb):
    """2^30 leaf positions are refused by every build entry, before any kernel runs for the body entries; the
    handle stays usable and then builds 2^30 - 1 positions (the largest input accepted) to the record."""
    import torch
    rec = record("ceiling_s1")
    S, n = rec["dna_size"], rec["bases"] + 1
    assert n // S == 1 << 30
    need_device(3 * n + build_memory_bound(rec))
    text = synth_text(stb, rec, n)
    text[n - 1] = ord("A")
    tree = stb.SharedTree(S)
    host = pinned_copy(text)
    for what, body in (("device body", text), ("host body", host)):
        before = stb.kernel_launches()
        with pytest.raises(stb.StbError) as e:
            tree.build_from_body(body)
        assert e.value.name == "STB_ERR_TOO_LARGE", what
        assert stb.kernel_launches() == before, f"{what}: a kernel ran before the size check"
    del host
    header = b">ceiling\n"
    fasta = torch.empty(len(header) + n, dtype=torch.uint8, device="cuda")
    fasta[:len(header)] = torch.frombuffer(bytearray(header), dtype=torch.uint8).cuda()
    fasta[len(header):] = text
    for what, src in (("device FASTA", fasta), ("host FASTA", None)):
        if src is None:
            src = pinned_copy(fasta)
            del fasta
        with pytest.raises(stb.StbError) as e:
            tree.build_from_fasta(src)
        assert e.value.name == "STB_ERR_TOO_LARGE", what
        del src
    tree.build_from_body(text[:n - 1])
    del text
    check_record(stb, tree, rec)
    tree.close()


def test_side_table_limit(stb):
    """Leaves outside ACGT at more than 268 M positions with a side table too small for them: the hashed leaf level
    that would take over is not supported at that size, and the build says so instead of returning a tree."""
    rec = record("beyond4gN_4500mbp")
    need_device(rec["bases"] + build_memory_bound(rec))
    text = synth_text(stb, rec)
    tree = stb.SharedTree(12).set_option("side_table_slots", 1)
    with pytest.raises(stb.StbError) as e:
        tree.build_from_body(text)
    assert e.value.name == "STB_ERR_TOO_LARGE"
    tree.close()
