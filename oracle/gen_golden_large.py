#!/usr/bin/env python3
"""Generates tests/golden/synth_large.json: the oracle (oracle.c, the C restatement of the reference) run on
synthetic sequences past the sizes the unmodified reference was run at (tests/golden/synth.json):

* beyond4g_4500mbp / beyond4gN_4500mbp: 4.5 Gbp at dna_size 12, more than 2^32 text bytes and more than 2^28
  leaf positions (375 M), plain and with N runs + soft-masking (synth_mask);
* ceiling_s1: 2^30 - 1 bases at dna_size 1, the largest input the single-GPU build accepts (DESIGN.md §7).

    make -C oracle oracle && python oracle/gen_golden_large.py [name ...]

The records have the fields of synth.json (gen_golden_synth.tree_record, the same code that wrote those from the
reference's tree) and "made_by": "oracle.c". They hold no timings, so a second run writes an identical file.
tests/test_golden_large_host.py runs case() on the parameters of two synth.json cases and checks that it
reproduces the reference's records. Single-threaded; each 4.5 Gbp case needs about 20 GB of host memory.
"""
from __future__ import annotations

import fcntl
import hashlib
import json
import resource
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle.gen_golden_synth import tree_record  # noqa: E402
from oracle.pyoracle import Oracle  # noqa: E402

GOLD = ROOT / "tests" / "golden" / "synth_large.json"

# name -> (bases, dna_size, seed, repeat_permille, variant, queries)
CASES = {
    "beyond4g_4500mbp": (4_500_000_000, 12, 43, 500, "plain", 10_000_000),
    "beyond4gN_4500mbp": (4_500_000_000, 12, 43, 500, "nruns", 10_000_000),
    "ceiling_s1": ((1 << 30) - 1, 1, 5, 500, "plain", 1_000_000),
}


def case(orc: Oracle, bases: int, dna_size: int, seed: int, permille: int, variant: str, queries: int) -> dict:
    """One record: the synthetic text (orc_synth_*, the CPU twin of the device generator), its leaves
    (orc_fasta_to_leaves) and the oracle's tree of them."""
    text = orc.synth(bases, seed, permille)
    if variant == "nruns":
        orc.synth_mask(text, 0, seed)
    rec = {"bases": bases, "seed": seed, "repeat_permille": permille, "variant": variant, "dna_size": dna_size,
           "text_sha256": hashlib.sha256(text).hexdigest()}
    leaves = orc.fasta_to_leaves(text, dna_size)
    del text
    tree = orc.build(leaves, dna_size)
    del leaves
    tree_record(tree, rec, queries)
    rec["made_by"] = "oracle.c"
    return rec


def store(name: str, rec: dict) -> None:
    """Adds one record to the file, under a lock so that cases may run in parallel processes; the records are
    written in CASES order whatever order they finish in."""
    GOLD.touch()
    with open(GOLD, "r+") as f:
        fcntl.flock(f, fcntl.LOCK_EX)
        text = f.read()
        have = json.loads(text) if text.strip() else {}
        have[name] = rec
        out = {k: have[k] for k in CASES if k in have}
        f.seek(0)
        f.truncate()
        f.write(json.dumps(out, indent=1) + "\n")


def main() -> None:
    names = sys.argv[1:] or list(CASES)
    orc = Oracle()
    for name in names:
        t0 = time.perf_counter()
        rec = case(orc, *CASES[name])
        store(name, rec)
        peak_gb = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2**20
        print(f"[{name}] {time.perf_counter() - t0:.1f} s, peak RSS of this process {peak_gb:.1f} GB: "
              f"{json.dumps({k: rec[k] for k in ('width', 'leaves', 'nodes', 'post_bytes')})}", flush=True)


if __name__ == "__main__":
    main()
