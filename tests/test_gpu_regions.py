"""GPU: stb_extract_regions (SharedTree.extract_regions, compress_b200 --decompress --regions=) against the tree's own
decode_ascii(), which the parity tests prove equal to the reference's sequence.

A forward region is a slice of that text; a reverse-strand region is the slice reversed with every letter mapped
through the 4-bit complement (dna::inverted): the bit reversal of the letter's index in "SACRGBNKTWVDYHM-"."""
import gc
import subprocess

import numpy as np
import pytest

from conftest import ROOT, corpus_text
from test_gpu_large_inputs import B4G, need_device, record, synth_text
from test_gpu_parity import build_memory_bound

pytestmark = pytest.mark.gpu

LETTERS = b"SACRGBNKTWVDYHM-"
COMPLEMENT = bytes.maketrans(LETTERS, bytes(LETTERS[int(f"{i:04b}"[::-1], 2)] for i in range(16)))
COMPRESS = ROOT / "genome-compression_b200" / "host" / "compress_b200"


def expected(text, start, end, strand):
    parts = []
    for s, e, r in zip(start, end, strand):
        piece = text[int(s):int(e)]
        parts.append(piece[::-1].translate(COMPLEMENT) if r else piece)
    return b"".join(parts)


def mixed_regions(n_bases, S, rng, count=400):
    """Seeded regions over [0, n_bases): empty and one-base regions, regions inside one leaf and across leaf and
    8-leaf-group boundaries, start = 0, end = n_bases, the whole sequence, overlapping and unsorted."""
    span = 8 * S
    reg = [(0, 0), (n_bases, n_bases), (n_bases // 2, n_bases // 2), (0, 1), (n_bases - 1, n_bases), (0, n_bases),
           (0, n_bases), (0, min(n_bases, S)), (max(0, n_bases - S), n_bases)]
    for k in range(1, min(n_bases // span, 6) + 1):  # around group boundaries and leaf boundaries next to them
        b = k * span
        reg += [(b - 1, b + 1), (b - S, b + S), (b, b + 1), (b - 1, b), (max(0, b - span - 3), min(n_bases, b + 5))]
        reg += [(b - S + 1, b - 1)] if S > 2 else []
    for _ in range(count):
        kind = rng.integers(0, 4)
        s = int(rng.integers(0, n_bases + 1))
        if kind == 0:
            e = s + int(rng.integers(0, 2 * S + 1))           # short: inside a leaf or across one boundary
        elif kind == 1:
            e = s + int(rng.integers(0, 3 * span + 1))        # a few groups
        elif kind == 2:
            e = s + int(rng.integers(0, max(1, n_bases // 3)))  # long
        else:
            e = int(rng.integers(s, n_bases + 1))
        reg.append((s, min(e, n_bases)))
    reg = [r for r in reg if 0 <= r[0] <= r[1] <= n_bases]
    rng.shuffle(reg)
    start = np.array([r[0] for r in reg], dtype=np.uint64)
    end = np.array([r[1] for r in reg], dtype=np.uint64)
    strand = rng.integers(0, 2, size=len(reg)).astype(np.uint8)
    return start, end, strand


def check_tree(stb, tree, rng, what, device=False, count=400):
    text = tree.decode_ascii()
    start, end, strand = mixed_regions(len(text), tree.dna_size, rng, count)
    want = expected(text, start, end, strand)
    got = tree.extract_regions(start, end, strand)
    assert got == want, what
    fwd = np.zeros_like(strand)
    assert tree.extract_regions(start, end) == expected(text, start, end, fwd), (what, "strand=None")
    if device:
        import torch
        ds, de = torch.from_numpy(start.view(np.int64)).cuda(), torch.from_numpy(end.view(np.int64)).cuda()
        dst = torch.from_numpy(strand).cuda()
        out = torch.zeros(len(want), dtype=torch.uint8, device="cuda")
        assert tree.extract_regions(ds, de, dst, out=out) == len(want)
        assert bytes(out.cpu().numpy()) == want, (what, "device")
    return text, (start, end, strand), want


CORPUS_SIZES = [("humhbb", S) for S in (1, 4, 11, 12, 13, 16)] + [("chmpxx", 12), ("vaccg", 13)]


@pytest.mark.parametrize("name,S", CORPUS_SIZES)
def test_corpus_regions(stb, name, S):
    tree = stb.SharedTree(S).build_from_fasta(corpus_text(name))
    check_tree(stb, tree, np.random.default_rng(S * 1000 + len(name)), f"{name}:{S}", device=True)


def test_small_vector_regions(stb, golden):
    rng = np.random.default_rng(3)
    for name, rec in golden["small"].items():
        S = rec["dna_size"]
        if S not in (1, 4, 11, 12, 13, 16):
            continue
        leaves = np.array([int(x, 16) for x in rec["input_leaves"]], dtype=np.uint64)
        tree = stb.SharedTree(S).build_from_leaves(leaves)
        check_tree(stb, tree, rng, name, count=100)


def test_iupac_letters_and_n_runs(stb):
    """Every one of the 16 letters (leaves outside ACGT go through the side table), and the synthetic "real genome"
    variant with runs of N and soft-masked stretches (folded to upper case by the build)."""
    import torch
    rng = np.random.default_rng(17)
    for S in (12, 13, 16):
        n = 6000
        nib = rng.integers(0, 16, size=(n, S)).astype(np.uint64)
        nib[n // 3:n // 3 + 40] = 6  # an N run
        leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
        leaves[n // 2:n // 2 + n // 4] = leaves[:n // 4]
        tree = stb.SharedTree(S).build_from_leaves(leaves)
        text, _, got = check_tree(stb, tree, rng, f"iupac S={S}", device=True)
        assert set(text) == set(LETTERS) and set(got) <= set(LETTERS)
    n = 2_000_000
    buf = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(buf, n, seed=9, repeat_permille=500)
    stb.synth_mask(buf, seed=9)
    tree = stb.SharedTree(12).build_from_body(buf)
    text = tree.decode_ascii()
    assert text == bytes(buf.cpu().numpy()).upper()[:len(text)]
    assert b"N" in text
    check_tree(stb, tree, rng, "synth_mask", device=True)


def test_same_answers_after_sort_stream_and_clone(stb):
    rng = np.random.default_rng(21)
    tree = stb.SharedTree(12).build_from_fasta(corpus_text("humdyst"))
    text, (start, end, strand), want = check_tree(stb, tree, rng, "built")
    tree.sort()
    assert tree.extract_regions(start, end, strand) == want, "after sort()"
    back = stb.SharedTree(12).deserialize(tree.serialize())
    assert back.extract_regions(start, end, strand) == want, "after serialize() / deserialize()"
    twin = tree.clone()
    assert twin.extract_regions(start, end, strand) == want, "on a clone()"
    assert twin.decode_ascii() == text


@pytest.mark.parametrize("S", [1, 3, 12])
def test_every_region_of_trees_up_to_20_leaves(stb, S):
    """Trees of 1 to 20 leaves: the ones of at most 4 leaves have fewer node layers than the 8-leaf groups need and
    descend to each leaf from the root.  Every (start, end) pair on both strands, in one call."""
    rng = np.random.default_rng(S)
    for w in range(1, 21):
        nib = np.array([1, 2, 4, 8, 5, 10], dtype=np.uint64)[rng.integers(0, 6, size=(w, S))]
        leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
        if w > 3:
            leaves[w // 2] = leaves[0]
        tree = stb.SharedTree(S).build_from_leaves(leaves)
        assert tree.width() == w
        text = tree.decode_ascii()
        n = len(text)
        pairs = np.array([(s, e) for s in range(n + 1) for e in range(s, n + 1)], dtype=np.uint64)
        for strand in (np.zeros(len(pairs), np.uint8), np.ones(len(pairs), np.uint8)):
            got = tree.extract_regions(pairs[:, 0], pairs[:, 1], strand)
            assert got == expected(text, pairs[:, 0], pairs[:, 1], strand), (S, w, int(strand[0]))


def test_device_path_matches_host_path_and_odd_offsets(stb):
    import torch
    rng = np.random.default_rng(5)
    tree = stb.SharedTree(12).build_from_fasta(corpus_text("humghcs"))
    text = tree.decode_ascii()
    start, end, strand = mixed_regions(len(text), 12, rng, 2000)
    host = tree.extract_regions(start, end, strand)
    ds, de = torch.from_numpy(start.view(np.int64)).cuda(), torch.from_numpy(end.view(np.int64)).cuda()
    dst = torch.from_numpy(strand).cuda()
    total = len(host)
    assert tree.extract_regions(ds, de, dst) == total, "query without out"
    for off in (0, 1, 3, 5):
        guard = torch.full((total + 16,), 0xA5, dtype=torch.uint8, device="cuda")
        assert tree.extract_regions(ds, de, dst, out=guard[off:off + total]) == total
        got = bytes(guard.cpu().numpy())
        assert got[off:off + total] == host, off
        assert got[:off] == b"\xa5" * off and got[off + total:] == b"\xa5" * (16 - off), ("wrote outside out", off)
    # uint64 device tensors and no strand
    us = torch.from_numpy(start.view(np.int64)).cuda().view(torch.uint64)
    ue = torch.from_numpy(end.view(np.int64)).cuda().view(torch.uint64)
    out = torch.zeros(int((end - start).sum()), dtype=torch.uint8, device="cuda")
    tree.extract_regions(us, ue, out=out)
    assert bytes(out.cpu().numpy()) == expected(text, start, end, np.zeros_like(strand))


# ---- errors: every check runs before anything is written ------------------------------------------------------

def small_tree(stb):
    return stb.SharedTree(12).build_from_fasta(corpus_text("humhbb"))


def raw_call(stb, tree, start, end, strand, out, cap, written=None):
    import ctypes as C
    s = np.ascontiguousarray(start, dtype=np.uint64)
    e = np.ascontiguousarray(end, dtype=np.uint64)
    st = None if strand is None else np.ascontiguousarray(strand, dtype=np.uint8)
    w = written if written is not None else C.c_uint64(0)
    status = stb.lib.stb_extract_regions(tree._h, s.ctypes.data if s.size else None, e.ctypes.data if e.size else None,
                                         None if st is None else st.ctypes.data, s.size,
                                         None if out is None else out.ctypes.data, cap, stb.HOST, C.byref(w))
    return status, int(w.value)


def test_error_start_after_end(stb):
    tree = small_tree(stb)
    with pytest.raises(stb.StbError) as e:
        tree.extract_regions([0, 10, 5], [4, 9, 6])
    assert e.value.name == "STB_ERR_INVALID_ARG"


def test_error_end_past_sequence(stb):
    tree = small_tree(stb)
    n = tree.width() * 12
    assert tree.extract_regions([n - 3], [n]) == tree.decode_ascii()[-3:]
    for bad in (n + 1, 1 << 40):
        with pytest.raises(stb.StbError) as e:
            tree.extract_regions([0, n - 3], [5, bad])
        assert e.value.name == "STB_ERR_OUT_OF_RANGE"


def test_error_strand_2(stb):
    tree = small_tree(stb)
    with pytest.raises(stb.StbError) as e:
        tree.extract_regions([0, 1], [4, 9], [1, 2])
    assert e.value.name == "STB_ERR_INVALID_ARG"


def test_error_cap_too_small(stb):
    tree = small_tree(stb)
    out = np.full(64, 0x5A, dtype=np.uint8)
    status, written = raw_call(stb, tree, [0, 100], [30, 130], [0, 1], out, 59)
    assert stb.STATUS[status] == "STB_ERR_BUFFER_TOO_SMALL"
    assert written == 60
    assert bool((out == 0x5A).all()), "out was written"
    status, written = raw_call(stb, tree, [0, 100], [30, 130], [0, 1], out, 60)
    assert status == 0 and written == 60
    text = tree.decode_ascii()
    assert out[:60].tobytes() == expected(text, [0, 100], [30, 130], [0, 1]) and bool((out[60:] == 0x5A).all())


def test_null_out_queries_the_total(stb):
    tree = small_tree(stb)
    status, written = raw_call(stb, tree, [0, 7, 50], [30, 7, 51], None, None, 0)
    assert status == 0 and written == 31


def test_no_regions(stb):
    tree = small_tree(stb)
    status, written = raw_call(stb, tree, [], [], None, None, 0, written=__import__("ctypes").c_uint64(99))
    assert status == 0 and written == 0
    assert tree.extract_regions([], []) == b""


def test_tree_not_built(stb):
    tree = stb.SharedTree(12)
    with pytest.raises(stb.StbError) as e:
        tree.extract_regions([0], [1])
    assert e.value.name == "STB_ERR_NOT_BUILT"


# ---- scale: against the generated text, on the device --------------------------------------------------------

def device_lut():
    import torch
    lut = torch.arange(256, dtype=torch.uint8)
    src = torch.frombuffer(bytearray(LETTERS), dtype=torch.uint8).long()
    lut[src] = torch.frombuffer(bytearray(LETTERS.translate(COMPLEMENT)), dtype=torch.uint8)
    return lut.cuda()


def check_on_device(text, start, end, strand, out, lut, chunk_bases=1 << 26):
    """out (device) against the text (device) for regions given as host arrays; one gather per chunk of regions."""
    import torch
    lengths = (end - start).astype(np.int64)
    offs = np.concatenate([[0], np.cumsum(lengths)])
    assert out.numel() == offs[-1]
    csum = np.concatenate([[0], np.cumsum(lengths)])
    long_idx = np.nonzero(lengths > chunk_bases // 4)[0]
    i = 0
    while i < len(start):
        if lengths[i] > chunk_bases // 4:  # a long region: slices
            s, e, o = int(start[i]), int(end[i]), int(offs[i])
            piece = text[s:e]
            if strand[i]:
                piece = lut[piece.flip(0).long()]
            assert torch.equal(out[o:o + e - s], piece), ("region", i, s, e, int(strand[i]))
            i += 1
            continue
        later_long = long_idx[np.searchsorted(long_idx, i):]
        j = min(int(later_long[0]) if later_long.size else len(start),
                int(np.searchsorted(csum, csum[i] + chunk_bases, "right")) - 1)
        acc = int(csum[j] - csum[i])
        ln = torch.from_numpy(lengths[i:j]).cuda()
        pos = torch.repeat_interleave(torch.arange(j - i, device="cuda"), ln)
        k = torch.arange(int(acc), device="cuda") - torch.from_numpy(offs[i:j] - offs[i]).cuda()[pos]
        s = torch.from_numpy(start[i:j].astype(np.int64)).cuda()[pos]
        rv = torch.from_numpy(strand[i:j].astype(bool)).cuda()[pos]
        e = torch.from_numpy(end[i:j].astype(np.int64)).cuda()[pos]
        src = torch.where(rv, e - 1 - k, s + k)
        want = text[src]
        want = torch.where(rv, lut[want.long()], want)
        assert torch.equal(out[int(offs[i]):int(offs[j])], want), ("regions", i, j)
        i = j


def run_device(stb, tree, start, end, strand):
    import torch
    ds = torch.from_numpy(start.astype(np.int64)).cuda()
    de = torch.from_numpy(end.astype(np.int64)).cuda()
    dst = torch.from_numpy(strand).cuda()
    total = tree.extract_regions(ds, de, dst)
    out = torch.empty(total, dtype=torch.uint8, device="cuda")
    assert tree.extract_regions(ds, de, dst, out=out) == total
    return out


@pytest.fixture(autouse=True)
def release_device_memory():
    yield
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def test_config3_genome(stb):
    """The 3.1 Gbp config-3 genome: 1 M random 150-bp regions on both strands, and long regions (50 Mbp and more,
    read from one level expansion over their hull) in one call with short ones (descending from the root)."""
    import torch
    n, S = 3_100_000_000, 12
    need_device(3 * n + 96 * (n // S) + (4 << 30))
    text = torch.empty(n, dtype=torch.uint8, device="cuda")
    stb.synth_genome(text, n, seed=42, repeat_permille=500)
    tree = stb.SharedTree(S).build_from_body(text)
    tree.sort()
    nb = tree.width() * S
    lut = device_lut()
    rng = np.random.default_rng(31)
    start = rng.integers(0, nb - 150 + 1, 1_000_000).astype(np.uint64)
    strand = rng.integers(0, 2, start.size).astype(np.uint8)
    out = run_device(stb, tree, start, start + 150, strand)
    check_on_device(text, start, start + 150, strand, out, lut)
    del out
    ls = np.array([0, 123_456_789, 5, nb - 60_000_001, 1_000_000_007, 7, nb - 150], dtype=np.uint64)
    le = np.array([50_000_000, 250_000_000, 1005, nb, 1_700_000_000, nb, nb], dtype=np.uint64)
    for strand in (np.zeros(7, np.uint8), np.ones(7, np.uint8), np.array([0, 1, 1, 1, 0, 1, 0], np.uint8)):
        out = run_device(stb, tree, ls, le, strand)
        check_on_device(text, ls, le, strand, out, lut)
        del out


def test_beyond_4g(stb):
    """Regions wholly above base 2^32 and straddling it, and one forward whole-sequence region: the output passes
    4 GiB."""
    import torch
    rec = record("beyond4g_4500mbp")
    n, S = rec["bases"], rec["dna_size"]
    need_device(3 * n + build_memory_bound(rec))
    text = synth_text(stb, rec)
    tree = stb.SharedTree(S).build_from_body(text)
    tree.sort()
    assert tree.width() * S == n
    rng = np.random.default_rng(44)
    above = rng.integers(B4G, n - 10_000, 2000).astype(np.uint64)
    a_end = above + rng.integers(0, 10_000, above.size).astype(np.uint64)
    across_s = np.array([B4G - 1, B4G - 7, B4G - 96, B4G - 5_000_001, B4G - 40_000_003], dtype=np.uint64)
    across_e = np.array([B4G + 1, B4G + 200, B4G + 96, B4G + 3_000_000, B4G + 50_000_000], dtype=np.uint64)
    start = np.concatenate([above, across_s, [0], across_s]).astype(np.uint64)
    end = np.concatenate([a_end, across_e, [n], across_e]).astype(np.uint64)
    strand = np.concatenate([rng.integers(0, 2, above.size), [0, 1, 0, 1, 0], [0], [1, 0, 1, 0, 1]]).astype(np.uint8)
    out = run_device(stb, tree, start, end, strand)
    assert out.numel() > B4G
    check_on_device(text, start, end, strand, out, device_lut())


def test_ceiling_s1(stb):
    """dna_size 1 at the 2^30 - 1 base ceiling: regions at the top of the range, on both strands, short and long."""
    rec = record("ceiling_s1")
    n, S = rec["bases"], rec["dna_size"]
    need_device(3 * n + build_memory_bound(rec))
    text = synth_text(stb, rec)
    tree = stb.SharedTree(S).build_from_body(text)
    assert tree.width() == n
    start = np.array([n - 1, n - 2, n - 1000, n - (1 << 20) - 3, (1 << 29) - 5, n - 1, n, n - (1 << 25) - 5, 0],
                     dtype=np.uint64)
    end = np.array([n, n, n, n, (1 << 29) + 5, n - 1, n, n, n], dtype=np.uint64)
    for strand in (np.zeros(start.size, np.uint8), np.ones(start.size, np.uint8)):
        out = run_device(stb, tree, start, end, strand)
        check_on_device(text, start, end, strand, out, device_lut())


# ---- command line --------------------------------------------------------------------------------------------

def test_cli_regions(stb, tmp_path):
    assert COMPRESS.exists(), "genome-compression_b200/host/compress_b200 missing: run __graft_entry__.build()"
    S = 12
    (tmp_path / "humhbb").write_bytes(corpus_text("humhbb"))
    dag = tmp_path / "humhbb.dag"
    res = subprocess.run([COMPRESS, f"--dna-size={S}", f"--output={dag}", tmp_path / "humhbb"], capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    text = stb.SharedTree(S).deserialize(dag.read_bytes()).decode_ascii()
    n = len(text)
    bed = tmp_path / "r.bed"
    bed.write_text("# comment\ntrack name=x\nbrowser position chr1\n\n"
                   "chr1\t0\t150\n"
                   "chr1 1000 1200 a 0 -\n"
                   "chrX\t5\t6\tb\t0\t+\n"
                   f"chr1 {n - 30} {n} c 0 .\n"
                   "chr2 77 77 d 0 -\n"
                   f"chr1\t0\t{n}\te\t0\t-\n")
    res = subprocess.run([COMPRESS, "--decompress", f"--dna-size={S}", f"--regions={bed}", dag], capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    rows = [("chr1", 0, 150, 0), ("chr1", 1000, 1200, 1), ("chrX", 5, 6, 0), ("chr1", n - 30, n, 0), ("chr2", 77, 77, 1),
            ("chr1", 0, n, 1)]
    want = b"".join(b">%s:%d-%d(%s)\n%s\n" % (c.encode(), s, e, b"-" if r else b"+", expected(text, [s], [e], [r]))
                    for c, s, e, r in rows)
    assert (tmp_path / "humhbb.fa").read_bytes() == want
    # an end past the sequence is reported once the tree is loaded, and nothing is written
    bad = tmp_path / "past.bed"
    bad.write_text(f"chr1 0 10\nchr1 5 {n + 1}\n")
    out = tmp_path / "past.fa"
    res = subprocess.run([COMPRESS, "--decompress", f"--dna-size={S}", f"--regions={bad}", f"--output={out}", dag],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 1 and res.stderr.startswith("line 2: "), res.stderr
    assert not out.exists()
