"""Region extraction (stb_extract_regions) on the config-3 synthetic tree (3.1 Gbp, seed 42, f = 0.5), inputs and
outputs in device memory.  Prints one JSON line.

    python profiles/scripts/bench_regions.py [--reps 5] [--warmup 2]

W1  10 M regions of 150 bp, seeded uniform starts, random strand; baseline: stb_random_access of the covering leaves
    (what a caller does without extraction, before trimming and spelling).
W2  24 regions tiling [0, width*S) at seeded base offsets, forward and reverse; baseline: stb_decode_ascii of the
    whole width.  Whole-sequence-sized regions are what could favour decode_range's level expansion.
W3  100 K regions of 10 kbp, random strand.

Every timed output (baselines included) is compared with the generated text on the device, so each timing also
proves correctness.  Times: CUDA events around the call (which ends in a stream synchronise), median and every
repetition after the warm-up.  The outputs (1 to 3.1 GB) are larger than the L2."""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from __graft_entry__ import load_package  # noqa: E402

LETTERS = b"SACRGBNKTWVDYHM-"
COMPLEMENT = bytes.maketrans(LETTERS, bytes(LETTERS[int(f"{i:04b}"[::-1], 2)] for i in range(16)))


def card():
    """Name and power limit of the device the run uses, read in the same process as the timings."""
    props = torch.cuda.get_device_properties(0)
    info = {"name": props.name, "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id,name,power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60).stdout
        bus = f"{props.pci_domain_id:08X}:{props.pci_bus_id:02X}:{props.pci_device_id:02X}"
        for line in q.strip().splitlines():
            b, name, limit = [x.strip() for x in line.split(",")]
            if b.upper().startswith(bus) or len(q.strip().splitlines()) == 1:
                info = {"name": name, "power_limit_w": float(limit), "pci_bus_id": b}
    except (OSError, ValueError, AttributeError):
        pass
    return info


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": statistics.median(ms), "reps_ms": [round(x, 4) for x in ms]}


def complement_lut():
    lut = torch.arange(256, dtype=torch.uint8)
    lut[torch.frombuffer(bytearray(LETTERS), dtype=torch.uint8).long()] = torch.frombuffer(
        bytearray(LETTERS.translate(COMPLEMENT)), dtype=torch.uint8)
    return lut.cuda()


def verify_regions(text, start, end, strand, out, lut, chunk=1 << 26):
    """out == the regions of text, back to back (start/end/strand: device int64 / uint8 tensors)."""
    lengths = end - start
    offs = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), torch.cumsum(lengths, 0)])
    assert int(offs[-1]) == out.numel()
    n, i = start.numel(), 0
    host_len = lengths.cpu().numpy()
    csum = np.concatenate([[0], np.cumsum(host_len)])
    long_idx = np.nonzero(host_len > chunk // 4)[0]
    while i < n:
        if host_len[i] > chunk // 4:
            s, e, o = int(start[i]), int(end[i]), int(offs[i])
            piece = text[s:e]
            if int(strand[i]):
                piece = lut[piece.flip(0).long()]
            if not torch.equal(out[o:o + e - s], piece):
                raise SystemExit(f"bench_regions: region {i} differs from the text")
            i += 1
            continue
        later_long = long_idx[np.searchsorted(long_idx, i):]
        j = min(int(later_long[0]) if later_long.size else n, int(np.searchsorted(csum, csum[i] + chunk, "right")) - 1)
        acc = int(csum[j] - csum[i])
        pos = torch.repeat_interleave(torch.arange(j - i, device="cuda"), lengths[i:j])
        k = torch.arange(acc, device="cuda") - (offs[i:j] - offs[i])[pos]
        rv = strand[i:j].bool()[pos]
        src = torch.where(rv, end[i:j][pos] - 1 - k, start[i:j][pos] + k)
        want = text[src]
        want = torch.where(rv, lut[want.long()], want)
        if not torch.equal(out[int(offs[i]):int(offs[j])], want):
            raise SystemExit(f"bench_regions: regions {i}..{j} differ from the text")
        i = j


def verify_leaves(text, idx, leaves, S, chunk=1 << 24):
    """Packed leaves (random access answers) spelled against the text."""
    letters = torch.frombuffer(bytearray(LETTERS), dtype=torch.uint8).cuda()
    shifts = 4 * torch.arange(S, device="cuda", dtype=torch.int64)
    for a in range(0, idx.numel(), chunk):
        v = leaves[a:a + chunk]
        got = letters[(v[:, None] >> shifts) & 15]
        want = text[idx[a:a + chunk, None] * S + torch.arange(S, device="cuda")]
        if not torch.equal(got, want):
            raise SystemExit("bench_regions: random access answers differ from the text")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bases", type=int, default=3_100_000_000)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--repeat-permille", type=int, default=500)
    ap.add_argument("--dna-size", type=int, default=12)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    assert args.reps >= 5, "at least five repetitions"
    pkg = load_package()
    S = args.dna_size
    text = torch.empty(args.bases, dtype=torch.uint8, device="cuda")
    pkg.synth_genome(text, args.bases, seed=args.seed, repeat_permille=args.repeat_permille)
    tree = pkg.SharedTree(S).build_from_body(text)
    tree.sort()
    width = tree.width()
    nb = width * S
    lut = complement_lut()
    rng = np.random.default_rng(args.seed)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    res = {"script": "profiles/scripts/bench_regions.py", "card": card(), "torch": torch.__version__,
           "workload": {"bases": args.bases, "seed": args.seed, "repeat_permille": args.repeat_permille, "dna_size": S,
                        "width": width, "tree": "built from the device text, then sort_tree()"},
           "reps": args.reps, "warmup": args.warmup}

    def extraction(name, start, end, strand, what):
        ds, de, dst = dev(start.astype(np.int64)), dev(end.astype(np.int64)), dev(strand.astype(np.uint8))
        total = tree.extract_regions(ds, de, dst)
        out = torch.empty(total, dtype=torch.uint8, device="cuda")
        t = timed(lambda: tree.extract_regions(ds, de, dst, out=out), args.warmup, args.reps)
        verify_regions(text, ds, de, dst, out, lut)
        sec = t["median_ms"] / 1e3
        t.update({"what": what, "regions": int(start.size), "bases": int(total), "regions_per_s": start.size / sec,
                  "gbp_per_s": total / sec / 1e9})
        res[name] = t
        del out
        return ds, de

    # W1
    n1 = 10_000_000
    s1 = rng.integers(0, nb - 150 + 1, n1).astype(np.int64)
    ds, de = extraction("W1", s1, s1 + 150, rng.integers(0, 2, n1), "10 M regions of 150 bp, random strand")
    first, last = ds // S, (de - 1) // S
    idx = torch.repeat_interleave(first, last - first + 1)
    idx = idx + torch.arange(idx.numel(), device="cuda") - torch.repeat_interleave(
        torch.cumsum(last - first + 1, 0) - (last - first + 1), last - first + 1)
    ans = torch.empty(idx.numel(), dtype=torch.int64, device="cuda")
    t = timed(lambda: tree.random_access(idx, out=ans), args.warmup, args.reps)
    verify_leaves(text, idx, ans, S)
    t.update({"what": "baseline: stb_random_access of the covering leaves (no trimming, no spelling)",
              "queries": int(idx.numel()), "extraction_speedup": t["median_ms"] / res["W1"]["median_ms"]})
    res["W1_baseline_random_access"] = t
    del idx, ans, ds, de

    # W2
    cuts = np.sort(rng.choice(np.arange(1, nb, dtype=np.int64), 23, replace=False))
    s2 = np.concatenate([[0], cuts]).astype(np.int64)
    e2 = np.concatenate([cuts, [nb]]).astype(np.int64)
    extraction("W2_forward", s2, e2, np.zeros(24), "24 regions tiling the sequence, forward")
    extraction("W2_reverse", s2, e2, np.ones(24), "24 regions tiling the sequence, reverse complement")
    out = torch.empty(nb, dtype=torch.uint8, device="cuda")
    t = timed(lambda: tree.decode_ascii(0, width, out=out), args.warmup, args.reps)
    if not torch.equal(out, text[:nb]):
        raise SystemExit("bench_regions: decode_ascii differs from the text")
    del out
    t["what"] = "baseline: stb_decode_ascii(0, width)"
    res["W2_baseline_decode_ascii"] = t
    res["W2_ratio_forward"] = res["W2_forward"]["median_ms"] / t["median_ms"]
    res["W2_ratio_reverse"] = res["W2_reverse"]["median_ms"] / t["median_ms"]

    # W3
    n3 = 100_000
    s3 = rng.integers(0, nb - 10_000 + 1, n3).astype(np.int64)
    extraction("W3", s3, s3 + 10_000, rng.integers(0, 2, n3), "100 K regions of 10 kbp, random strand")
    res["verified"] = "every timed output equals the generated text"
    print(json.dumps(res))


if __name__ == "__main__":
    main()
