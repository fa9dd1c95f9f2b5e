#!/usr/bin/env python3
"""Generates tests/golden/synth.json: the UNMODIFIED reference (oracle/_ref/libref.so) executed on
the synthetic sequences of BASELINE.json configs 3 / 4 / 5 (DESIGN.md §6) at FULL size.

Run in the build container, where /root/reference exists (about 10 min and 16 GB for 3.1 Gbp):

    make -C oracle ref oracle && python oracle/gen_golden_synth.py [name ...]

Per case: the text is produced by the CPU twin of the device generator (oracle.c: orc_synth_*),
written to a file and built by the reference exactly as ./compress does (compress.cpp:183:
shared_tree{path} = loader thread + build thread), then sort_tree (compress.cpp:188), bytes
(src/shared_tree.cpp:488) and 10 M operator[] answers (src/shared_tree.cpp:268) for seeded indices.
Recorded: width, depth, per-layer node counts, leaf count, sha256 of every raw node layer and of the
leaf table before sort_tree, stream length + sha256 before and after sort_tree, sha256 of the
random-access answers, and the reference's own construct / sort seconds on this container's CPU.
"""
from __future__ import annotations

import hashlib
import json
import os
import platform
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle.pyoracle import Oracle, Ref  # noqa: E402

GOLD = ROOT / "tests" / "golden" / "synth.json"
DNA = 12

# name -> (bases, seed, repeat_permille, variant, queries)
CASES = {
    "config3_3100mbp": (3_100_000_000, 42, 500, "plain", 10_000_000),
    "large_260mbp": (260_000_000, 1, 500, "plain", 1_000_000),
    "mid_50mbp": (50_000_000, 3, 500, "plain", 1_000_000),
    "config3N_3100mbp": (3_100_000_000, 42, 500, "nruns", 10_000_000),
    "largeN_260mbp": (260_000_000, 1, 500, "nruns", 1_000_000),
}


def query_indices(seed: int, q: int, width: int) -> np.ndarray:
    """idx[i] = splitmix64(seed + (i + 1) * golden) mod width — the same closed form bench.py and
    the tests use (genome_compression_b200.query_indices)."""
    with np.errstate(over="ignore"):
        x = np.uint64(seed) + (np.arange(1, q + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15))
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return (x % np.uint64(width)).astype(np.uint64)


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return platform.processor()


def tree_record(tree, rec: dict, q: int) -> tuple[float, float]:
    """Adds the tree's fields to rec, in place: shape, sha256 of the leaf table and of every raw node layer,
    the stream before and after sort() (which this sorts the tree for), and the answers to q seeded queries.
    rec must already hold "seed" and "dna_size". Works on either checker's tree (oracle.pyoracle._Tree).
    Returns the seconds sort() and the queries took."""
    S = rec["dna_size"]
    rec.update({
        "width": int(tree.width()), "depth": int(tree.depth()), "leaves": int(tree.leaf_count()),
        "nodes": int(tree.node_count()), "layer_counts": [int(c) for c in tree.layer_counts()],
    })
    rec["pre_leaves_sha256"] = hashlib.sha256(tree.leaves().tobytes()).hexdigest()
    rec["pre_layer_sha256"] = [hashlib.sha256(tree.layer(k).tobytes()).hexdigest() for k in range(len(rec["layer_counts"]))]
    pre = tree.serialize()
    rec["pre_bytes"] = len(pre)
    rec["pre_sha256"] = hashlib.sha256(pre).hexdigest()
    del pre
    t0 = time.perf_counter()
    tree.sort()
    sort_s = time.perf_counter() - t0
    post = tree.serialize()
    assert tree.bytes() == len(post)
    rec["post_bytes"] = len(post)
    rec["post_sha256"] = hashlib.sha256(post).hexdigest()
    del post
    rec["bits_per_base"] = 8.0 * rec["post_bytes"] / (rec["width"] * S)
    idx = query_indices(rec["seed"], q, rec["width"])
    t0 = time.perf_counter()
    ans = tree.random_access(idx)
    ra_s = time.perf_counter() - t0
    rec["queries"] = q
    rec["query_answers_sha256"] = hashlib.sha256(np.ascontiguousarray(ans, dtype="<u8").tobytes()).hexdigest()
    rec["query_first8"] = [f"{int(v):x}" for v in ans[:8]]
    return sort_s, ra_s


def run_case(name: str, ref: Ref, orc: Oracle) -> dict:
    bases, seed, permille, variant, q = CASES[name]
    t0 = time.perf_counter()
    text = orc.synth(bases, seed, permille)
    if variant == "nruns":
        orc.synth_mask(text, 0, seed)
    path = Path(os.environ.get("TMPDIR", "/tmp")) / f"golden_{name}.txt"
    text.tofile(path)
    text_sha = hashlib.sha256(text).hexdigest()
    del text
    print(f"[{name}] text written in {time.perf_counter() - t0:.1f} s", flush=True)

    t0 = time.perf_counter()
    tree = ref.build_file(path, DNA)
    construct_s = time.perf_counter() - t0
    os.unlink(path)
    print(f"[{name}] reference build {construct_s:.1f} s", flush=True)
    rec = {"bases": bases, "seed": seed, "repeat_permille": permille, "variant": variant, "dna_size": DNA,
           "text_sha256": text_sha}
    sort_s, ra_s = tree_record(tree, rec, q)
    rec["reference_timing"] = {
        "construct_s": round(construct_s, 2), "sort_s": round(sort_s, 2), "random_access_s": round(ra_s, 3),
        "gbp_per_s": rec["width"] * DNA / construct_s / 1e9, "threads": 2,
        "host": f"{cpu_model()}, {os.cpu_count()} logical CPUs (the build container, not the GPU box)",
        "how": "oracle/_ref/libref.so: shared_tree{path} on the text file, as compress.cpp:183",
    }
    print(f"[{name}] {json.dumps({k: rec[k] for k in ('width', 'leaves', 'nodes', 'post_bytes', 'post_sha256')})}", flush=True)
    return rec


def main() -> None:
    names = sys.argv[1:] or list(CASES)
    ref, orc = Ref(), Oracle()
    out = json.loads(GOLD.read_text()) if GOLD.exists() else {}
    for name in names:
        out[name] = run_case(name, ref, orc)
        GOLD.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
