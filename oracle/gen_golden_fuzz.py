#!/usr/bin/env python3
"""Records what a checker returns on the seeded fuzz inputs of tests/test_oracle_vs_reference.py and writes
tests/golden/reference_fuzz.json.  TEST INFRASTRUCTURE ONLY.

    python oracle/gen_golden_fuzz.py [--checker reference|port]

Each function below rebuilds one test's inputs from its seed, in the order the test draws them, and returns
sha256 digests of everything the test compares (inputs included, so that a change in the input generation
shows as such).  The tests compute the same records with the C restatement, and with the unmodified
reference too where it can be built, and compare them with the stored ones.

The stored file says which checker wrote it.  `--checker port` exists for a machine without the reference's
sources: it is only valid while the tests have passed against the live reference on these exact inputs and
oracle/oracle.c has not changed since, because then the restatement's answers are the reference's.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
OUT = ROOT / "tests" / "golden" / "reference_fuzz.json"

NULL = 0x9FFFFFFF
TREE_CASES = ((12, 5000, 4), (12, 777, 2), (3, 4097, 4), (16, 1000, 16), (7, 2500, 16))
FASTA_CASES = [(12, 5000, b"ACGT", 60, 1, False), (12, 70001, b"ACGT", 70, 3, True), (5, 3333, b"ACGTRYKMSWBDHVN-", 50, 4, True),
               (16, 4096, b"ACGTRYKMSWBDHVN-", 61, 2, False), (1, 257, b"ACGT", 7, 2, True), (13, 999, b"ACGTRYKMSWBDHVN-", 1, 1, False),
               (12, 11, b"ACGT", 80, 1, False), (12, 12, b"ACGT", 5, 2, True), (8, 40000, b"ACGT", 100000, 1, False),
               (12, 25, b"ACGTRYKMSWBDHVN-", 3, 5, True)]


def sha(a, dtype=None) -> str:
    data = a if isinstance(a, bytes) else np.ascontiguousarray(a, dtype=dtype).tobytes()
    return hashlib.sha256(data).hexdigest()


def leaf_fuzz(checker) -> dict:
    """Leaf primitives on 300 random words per dna_size 1..16."""
    rng = np.random.default_rng(7)
    rows = []
    for S in range(1, 17):
        mask = (1 << (4 * S)) - 1
        for _ in range(300):
            v = int.from_bytes(rng.bytes(8), "little") & mask
            c, f = checker.leaf_canonical(v, S)
            rows.append((v, c, f, checker.mirrored(v, S), checker.inverted(v, S), checker.transposed(v, S)))
    rows = np.array(rows, dtype=np.uint64)
    return {"count": len(rows), "inputs": sha(rows[:, 0]), "results": sha(rows)}


def node_fuzz(checker, port) -> dict:
    """node::canonical on 20000 pairs of pointers (built with the port's pointer(), as inputs)."""
    rng = np.random.default_rng(8)

    def rp():
        if rng.integers(8) == 0:
            return NULL
        return port.pointer(int(rng.integers(5)), int(rng.integers(2)), int(rng.integers(2)), int(rng.integers(4) == 0))

    rows = []
    for _ in range(20000):
        l, r = rp(), rp()
        rows.append((l, r, *checker.node_canonical(l, r)))
    rows = np.array(rows, dtype=np.uint32)
    return {"count": len(rows), "inputs": sha(rows[:, :2]), "results": sha(rows)}


def tree_leaves(rng, S, n, alphabet):
    codes = np.array([1, 2, 4, 8, 3, 12, 7, 14, 0, 9, 5, 11, 13, 10, 6, 15], dtype=np.uint64)[:alphabet]
    nib = codes[rng.integers(0, alphabet, size=(n, S))]
    leaves = (nib << (4 * np.arange(S, dtype=np.uint64))).sum(axis=1).astype(np.uint64)
    leaves[n // 2:n // 2 + n // 8] = leaves[:n // 8]  # planted repeat
    return leaves


def random_trees(checker, port) -> list:
    """Whole trees: per-level pointer arrays, stored layers and histograms, the streams before and after
    sort_tree, decode and random access.  The port must parse the checker's sorted stream back to the input."""
    rng = np.random.default_rng(9)
    out = []
    for S, n, alphabet in TREE_CASES:
        leaves = tree_leaves(rng, S, n, alphabet)
        tree = checker.build(leaves, S)
        _, levels = checker.build_levels(leaves, S)
        pre = tree.serialize()
        assert tree.bytes() == len(pre), (S, n, "pre-sort bytes()")
        rec = {"dna_size": S, "n": n, "inputs": sha(leaves, np.uint64), "levels": [sha(lv, np.uint32) for lv in levels],
               "layers": [sha(tree.layer(k), np.uint32) for k in range(tree.depth() - 1)],
               "histograms": [sha(tree.histogram(k), np.uint64) for k in range(tree.depth() - 1)],
               "pre_bytes": len(pre), "pre_sha256": sha(pre)}
        tree.sort()
        post = tree.serialize()
        assert tree.bytes() == len(post), (S, n, "post-sort bytes()")
        back = port.deserialize(post, S)
        assert back.width() == n and np.array_equal(back.decode(), leaves), (S, n, "the port's parse of the stream")
        assert np.array_equal(tree.decode(), leaves), (S, n, "decode")
        idx = rng.integers(0, n, 500).astype(np.uint64)
        rec.update(post_bytes=len(post), post_sha256=sha(post), random_access=sha(tree.random_access(idx), np.uint64))
        out.append(rec)
    return out


def random_fasta(rng, n_bases, alphabet, width, records, blank_lines):
    """Valid FASTA text as the reference accepts it (src/fasta_reader.cpp:40-68): a header or a
    blank line is never followed directly by another one (the reference would parse the second
    as data and exit on '>'), no '\\r', symbols from its table only, mixed case."""
    letters = np.frombuffer(alphabet, dtype=np.uint8)
    body = letters[rng.integers(0, len(letters), n_bases)].copy()
    lower = rng.integers(0, 2, n_bases).astype(bool)
    body[lower] = np.char.lower(body[lower].view("S1")).view(np.uint8)
    body = body.tobytes()
    cuts = sorted(set(int(c) for c in rng.integers(1, max(2, n_bases), records - 1))) if records > 1 and n_bases > 2 else []
    pieces, start = [], 0
    for k, end in enumerate(cuts + [n_bases]):
        pieces.append(b">record %d some description\n" % k)
        chunk = body[start:end]
        lines = [chunk[i:i + width] for i in range(0, len(chunk), width)] or [b""]
        for j, line in enumerate(lines):
            pieces.append(line + b"\n")
            if blank_lines and line and j + 1 < len(lines) and rng.integers(0, 7) == 0:
                pieces.append(b"\n")  # a blank line between two data lines is skipped like a header
        start = end
    text = b"".join(pieces)
    return text if rng.integers(0, 2) else text.rstrip(b"\n")  # with and without the final newline


def fasta_ingest_fuzz(checker) -> list:
    """Body extraction + packing + whole build of FASTA text.  The reference reads it from a FILE through
    its own reader (fasta_reader + read_genome / shared_tree{path}); the port takes the same bytes."""
    rng = np.random.default_rng(10)
    out = []
    with tempfile.TemporaryDirectory() as tmp:
        for k, (S, n_bases, alphabet, width, records, blanks) in enumerate(FASTA_CASES):
            if n_bases < S:
                continue  # undefined in the reference (SIGFPE)
            text = random_fasta(rng, n_bases, alphabet, width, records, blanks)
            path = Path(tmp) / f"case{k}.fa"
            path.write_bytes(text)
            leaves = checker.read_genome(path, S) if checker.kind == "reference" else checker.fasta_to_leaves(text, S)
            rec = {"case": k, "dna_size": S, "inputs": sha(text), "leaves": len(leaves), "leaves_sha256": sha(leaves, np.uint64)}
            if len(leaves):
                tree = checker.build_file(path, S) if checker.kind == "reference" else checker.build(leaves, S)
                rec["pre_sha256"] = sha(tree.serialize())
                tree.sort()
                rec["post_sha256"] = sha(tree.serialize())
            out.append(rec)
    return out


def main() -> None:
    from oracle.pyoracle import Oracle, Ref
    ap = argparse.ArgumentParser()
    ap.add_argument("--checker", choices=["reference", "port"], default="reference")
    args = ap.parse_args()
    port = Oracle()
    checker = Ref() if args.checker == "reference" else port
    how = {"reference": "the unmodified reference (oracle/_ref/libref.so)",
           "port": "the C restatement (oracle/oracle.c) on a machine without the reference's sources; tests/test_oracle_vs_reference.py "
                   "had passed against the live reference on these inputs, and oracle.c has not changed since"}[args.checker]
    records = {"written_by": how, "leaf_fuzz": leaf_fuzz(checker), "node_fuzz": node_fuzz(checker, port),
               "random_trees": random_trees(checker, port), "fasta_ingest_fuzz": fasta_ingest_fuzz(checker)}
    OUT.write_text(json.dumps(records, indent=1) + "\n")
    print("written", OUT, OUT.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
