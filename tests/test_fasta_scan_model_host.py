"""CPU: tests/fasta_scan_model.py (csrc/ingest.cu's tile passes and scans, restated) against the oracle's sequential
reading of FASTA text.  At shrunken sizes (4-byte thread chunks, 2-lane warps, 16-byte sub-tiles, 64-byte tiles,
4 tiles per scan step, 128-byte stream chunks) the adversarial texts put line starts, headers, runs of header and
blank lines, whole tiles of blank lines and lines longer than a tile on every boundary of every composition."""
import hashlib

import numpy as np
import pytest

import fasta_scan_model as M

SMALL_LEN = 2000
CLASSES = dict(M.SMALL.classes(), step=M.SMALL.step, stream=M.SMALL.stream)


def small_texts(period, valid, seed):
    """Seven texts, one per shift rotation, with the head and tail variants spread over them."""
    for rot in range(7):
        rng = np.random.default_rng([seed, period, rot, valid])
        yield M.adversarial_text(rng, M.SMALL, M.boundary_targets(period, SMALL_LEN, rot), SMALL_LEN, valid=valid,
                                 large=0.25 if period >= M.SMALL.tile else 0.0, head=("", "nl", "gt")[rot % 3],
                                 tail=("", "nofinal", "header", "blanks")[rot % 4])


def check(oracle, text, sz):
    want = oracle.fasta_body(text)
    assert M.fasta_body(text, sz) == want, "one-shot extraction"
    assert M.fasta_body_streamed(text, sz) == want, "streaming extraction"


@pytest.mark.parametrize("valid", [True, False], ids=["valid", "headers_as_data"])
@pytest.mark.parametrize("boundary", sorted(CLASSES))
def test_small_sizes_every_boundary(oracle, boundary, valid):
    for text in small_texts(CLASSES[boundary], valid, 1):
        check(oracle, text, M.SMALL)


def test_generated_texts_are_what_they_claim(oracle):
    """Valid texts are accepted by the reader; the others read some header as data (the reference exits on it)."""
    rejected = 0
    for boundary, period in CLASSES.items():
        for text in small_texts(period, True, 1):
            oracle.fasta_to_leaves(text, 1)
        for text in small_texts(period, False, 1):
            try:
                oracle.fasta_to_leaves(text, 1)
            except ValueError as e:
                assert str(e) == "unknown symbol 62"
                rejected += 1
    assert rejected >= len(CLASSES) * 5


def test_real_sizes(oracle):
    """The kernel's own sizes: events on 16-byte, 512-byte and 4 KiB boundaries of the first tiles and on every tile
    boundary of a text of about five tiles, streamed in 64 KiB chunks; then the same with headers read as data."""
    R = M.REAL
    n = 5 * R.tile + 777
    for valid, seed in ((True, 2), (False, 3)):
        rng = np.random.default_rng(seed)
        targets = M.boundary_targets(16, 12_000, 0) + M.boundary_targets(512, 40_000, 2) + M.boundary_targets(4096, n, 4) + \
            M.boundary_targets(R.tile, n, 6)
        text = M.adversarial_text(rng, R, sorted(set(targets)), n, valid=valid, large=0.3, head="gt", tail="blanks")
        assert len(text) > 4 * R.tile
        check(oracle, text, R)


def test_reference_fuzz_texts(oracle):
    """The texts certified against the reference in tests/golden/reference_fuzz.json, regenerated."""
    import json

    from conftest import GOLD
    from oracle.gen_golden_fuzz import FASTA_CASES, random_fasta
    recs = json.loads((GOLD / "reference_fuzz.json").read_text())["fasta_ingest_fuzz"]
    rng = np.random.default_rng(10)
    done = 0
    for k, (S, n_bases, alphabet, width, records, blanks) in enumerate(FASTA_CASES):
        if n_bases < S:
            continue
        text = random_fasta(rng, n_bases, alphabet, width, records, blanks)
        rec = recs[done]
        assert rec["case"] == k and hashlib.sha256(text).hexdigest() == rec["inputs"], f"case {k}: the generator drifted"
        check(oracle, text, M.REAL)
        done += 1
    assert done == len(recs)


def wrong_run_no_all_hb(a, b):
    return (a[0] & b[0], b[1])


def wrong_scanb_one_state(a, b):
    return (a[0] | b[0], b[1] if b[0] else a[1], a[2] + b[2], a[3] + b[2])


def wrong_skip_first(a, b):
    return a if a[0] else b


@pytest.mark.parametrize("name,wrong", [("run_compose", wrong_run_no_all_hb), ("scanb_compose", wrong_scanb_one_state),
                                        ("skip_compose", wrong_skip_first)], ids=["run", "scanb", "skip"])
def test_wrong_composition_is_caught(oracle, monkeypatch, name, wrong):
    """The texts above are strong enough: a composition rule shrunk to a wrong one changes some body."""
    monkeypatch.setattr(M, name, wrong)
    caught = 0
    for boundary, period in CLASSES.items():
        for text in small_texts(period, False, 1):
            want = oracle.fasta_body(text)
            for extract in (M.fasta_body, M.fasta_body_streamed):
                try:
                    caught += extract(text, M.SMALL) != want
                except AssertionError:  # a tile emitted past its successor's offset
                    caught += 1
    assert caught > 0
