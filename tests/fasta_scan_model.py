"""A plain Python restatement of csrc/ingest.cu's FASTA text -> body extraction, and the adversarial texts that
tests/test_fasta_scan_model_host.py and tests/test_gpu_fasta_boundaries.py feed it.

The reference reads FASTA with a sequential getline loop (src/fasta_reader.cpp:40-68).  ingest.cu restates it as a
parallel automaton: a line that starts with '>' or is blank (an "hb" line) is skipped iff the run of hb lines just
before it has even length, every other line is data, and newlines are never data.  The run state and the skip
state are composed across 16-byte thread chunks, warps, 4 KiB sub-tiles and 64 KiB tiles, then carried across tiles
by two single-CTA scans, 256 tiles per loop step, and across the text chunks of the streaming build (FxStream).

The model runs the same three tile passes and two scans with the same composition operators, in the same order,
with every size a parameter: at shrunken sizes every composition path runs on a few KB of text.  Block-wide scans
compose as the kernel's do (a Hillis-Steele scan inside each warp, then the warp totals in order).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

NL, GT = 0x0A, 0x3E


@dataclass(frozen=True)
class Sizes:
    chunk: int = 16      # bytes per thread per sub-tile (FX_CHUNK)
    threads: int = 256   # threads per CTA (FX_THREADS); also the tiles per loop step of the single-CTA scans
    warp: int = 32       # lanes per warp
    subs: int = 16       # sub-tiles per tile (FX_SUBS_PER_TILE)
    stream: int = 65536  # text bytes per chunk of the streaming build (a multiple of the tile)

    @property
    def sub(self): return self.chunk * self.threads

    @property
    def tile(self): return self.sub * self.subs

    @property
    def step(self): return self.tile * self.threads

    def classes(self):
        """The boundary classes of the extraction: thread chunk, warp, sub-tile, tile."""
        return {"chunk": self.chunk, "warp": self.chunk * self.warp, "sub": self.sub, "tile": self.tile}


REAL = Sizes()
SMALL = Sizes(chunk=4, threads=4, warp=2, subs=4, stream=128)  # sub-tile 16 B, tile 64 B, scan step 256 B


# ---- composition operators (ingest.cu) ------------------------------------------------------------------------
# RunSum (all_hb, trail): every line start of the span is an hb line; hb line starts at the span's end
RUN_ID = (1, 0)


def run_compose(a, b):
    return (a[0] & b[0], a[1] + b[1] if b[0] else b[1])


# SkipSum (has_ls, last_skip): does the span hold a line start, is its last line skipped
SKIP_ID = (0, 0)


def skip_compose(a, b):
    return b if b[0] else a


def add(a, b):
    return a + b


# ScanB (has_ls, last_skip, cnt0, cnt1): kept bytes when the span is entered in skip state 0 / 1
SCANB_ID = (0, 0, 0, 0)


def scanb_compose(a, b):
    out0 = a[1] if a[0] else 0
    out1 = a[1] if a[0] else 1
    return (a[0] | b[0], b[1] if b[0] else a[1], a[2] + (b[3] if out0 else b[2]), a[3] + (b[3] if out1 else b[2]))


def block_exclusive(vals, ident, op, warp):
    """block_exclusive: (exclusive scan, total) of one value per thread, composed in the kernel's order."""
    n = len(vals)
    incl = []
    for w0 in range(0, n, warp):
        x = list(vals[w0:w0 + warp])
        d = 1
        while d < warp:
            x = [op(x[i - d], x[i]) if i >= d else x[i] for i in range(len(x))]
            d <<= 1
        incl += x
    warp_tot = [incl[min(w0 + warp, n) - 1] for w0 in range(0, n, warp)]
    prefix, acc = [], ident
    for t in warp_tot:
        prefix.append(acc)
        acc = op(acc, t)
    excl = [prefix[i // warp] if i % warp == 0 else op(prefix[i // warp], incl[i - 1]) for i in range(n)]
    return excl, acc


# ---- the tile passes (fasta_tile_kernel<PHASE>) --------------------------------------------------------------
def tile_pass(phase, sz, text, base, length, tile, run_state=RUN_ID, carry=None, body=None):
    """One CTA of fasta_tile_kernel over text[base : base + length] (the chunk; `text` is the whole text, so the byte
    before the chunk is real).  phase 0 returns the tile's RunSum, phase 1 its TileSum (has_ls, last_skip, cnt0,
    cnt1), phase 2 writes the kept bytes into `body` from carry's out_off and returns the offset after them."""
    tile_base = tile * sz.tile
    if phase == 2:
        run_state, in_skip, out_off = carry
        in_skip0 = in_skip1 = in_skip
    else:
        in_skip0, in_skip1, out_off = 0, 1, 0
    has_ls = last_skip = cnt0 = cnt1 = 0
    prev_sub_last = NL if base + tile_base == 0 else text[base + tile_base - 1]
    for sub in range(sz.subs):
        sub_base = tile_base + sub * sz.sub
        if sub_base >= length:
            break
        cs = []
        for t in range(sz.threads):
            my_base = sub_base + t * sz.chunk
            valid = max(0, min(sz.chunk, length - my_base))
            cs.append(text[base + my_base:base + my_base + valid])
        lasts = [c[-1] if c else 0 for c in cs]
        pbs = [prev_sub_last] + lasts[:-1]
        ls, hb, mine = [], [], []
        for c, pb in zip(cs, pbs):
            starts = [i for i in range(len(c)) if (pb if i == 0 else c[i - 1]) == NL]
            hbs = {i for i in starts if c[i] in (GT, NL)}
            r = RUN_ID
            for i in starts:
                r = (r[0], r[1] + 1) if i in hbs else (0, 0)
            ls.append(starts)
            hb.append(hbs)
            mine.append(r)
        before, total = block_exclusive(mine, RUN_ID, run_compose, sz.warp)
        before = [run_compose(run_state, b) for b in before]
        run_state = run_compose(run_state, total)
        prev_sub_last = lasts[-1]
        if phase == 0:
            continue
        skips, sks = [], []
        for starts, hbs, rb in zip(ls, hb, before):
            run, skip = rb[1], set()
            for i in starts:
                if i in hbs:
                    if run % 2 == 0:
                        skip.add(i)
                    run += 1
                else:
                    run = 0
            skips.append(skip)
            sks.append((1, int(starts[-1] in skip)) if starts else (0, 0))
        sk_before, sk_total = block_exclusive(sks, SKIP_ID, skip_compose, sz.warp)

        def kept(in_skip):
            out = []
            for c, starts, skip, skb in zip(cs, ls, skips, sk_before):
                cur = skb[1] if skb[0] else in_skip
                mine = bytearray()
                for i, ch in enumerate(c):
                    if i in starts:
                        cur = int(i in skip)
                    if ch != NL and not cur:
                        mine.append(ch)
                out.append(bytes(mine))
            return out

        keep0 = kept(in_skip0)
        if phase == 1:
            keep1 = kept(in_skip1)
            cnt0 += block_exclusive([len(k) for k in keep0], 0, add, sz.warp)[1]
            cnt1 += block_exclusive([len(k) for k in keep1], 0, add, sz.warp)[1]
            if sk_total[0]:
                has_ls, last_skip = 1, sk_total[1]
                in_skip0 = in_skip1 = sk_total[1]
        else:
            offs, total = block_exclusive([len(k) for k in keep0], 0, add, sz.warp)
            for off, k in zip(offs, keep0):
                body[out_off + off:out_off + off + len(k)] = k
            out_off += total
            if sk_total[0]:
                in_skip0 = in_skip1 = sk_total[1]
    if phase == 0:
        return run_state
    if phase == 1:
        return (has_ls, last_skip, cnt0, cnt1)
    return out_off


# ---- the single-CTA scans ------------------------------------------------------------------------------------
def scan_run(sz, sums, stream=None):
    """fasta_scan_run_kernel: the hb-run state before every tile."""
    state = stream["run"] if stream else RUN_ID
    carry = []
    for b in range(0, len(sums), sz.threads):
        v = [sums[i] if i < len(sums) else RUN_ID for i in range(b, b + sz.threads)]
        before, total = block_exclusive(v, RUN_ID, run_compose, sz.warp)
        carry += [run_compose(state, x) for x in before[:len(sums) - b]]
        state = run_compose(state, total)
    if stream:
        stream["run"] = state
    return carry


def scan_skip(sz, sums, run_carry, stream=None):
    """fasta_scan_skip_kernel: every tile's (run state, incoming skip state, body offset), and the body length."""
    state = SCANB_ID
    if stream:
        state = (1, stream["in_skip"], stream["out_off"], stream["out_off"])
    carry = []
    for b in range(0, len(sums), sz.threads):
        v = [sums[i] if i < len(sums) else SCANB_ID for i in range(b, b + sz.threads)]
        before, total = block_exclusive(v, SCANB_ID, scanb_compose, sz.warp)
        for i in range(b, min(b + sz.threads, len(sums))):
            upto = scanb_compose(state, before[i - b])
            carry.append((run_carry[i], upto[1] if upto[0] else 0, upto[2]))
        state = scanb_compose(state, total)
    if stream:
        stream["in_skip"] = state[1] if state[0] else 0
        stream["out_off"] = state[2]
    return carry, state[2]


def extract_chunk(sz, text, base, length, body, stream=None):
    """The five launches of fasta_extract_body (stream=None) or of fasta_stream_chunk; returns the body length."""
    tiles = -(-length // sz.tile)
    run_sums = [tile_pass(0, sz, text, base, length, k) for k in range(tiles)]
    run_carry = scan_run(sz, run_sums, stream)
    tile_sums = [tile_pass(1, sz, text, base, length, k, run_state=run_carry[k]) for k in range(tiles)]
    carry, body_len = scan_skip(sz, tile_sums, run_carry, stream)
    for k in range(tiles):
        end = tile_pass(2, sz, text, base, length, k, carry=carry[k], body=body)
        assert end == (carry[k + 1][2] if k + 1 < tiles else body_len), ("tile", k, "emitted up to", end)
    return body_len


def fasta_body(text: bytes, sz: Sizes = REAL) -> bytes:
    """The one-shot device extraction (fasta_extract_body)."""
    body = bytearray(len(text) + 16)
    n = extract_chunk(sz, text, 0, len(text), body) if text else 0
    return bytes(body[:n])


def fasta_body_streamed(text: bytes, sz: Sizes = REAL) -> bytes:
    """The streaming extraction (build_streaming_fasta): chunks of sz.stream bytes, FxStream carried between them."""
    assert sz.stream % sz.tile == 0
    body = bytearray(len(text) + 16)
    stream = {"run": RUN_ID, "in_skip": 0, "out_off": 0}
    n = 0
    for first in range(0, len(text), sz.stream):
        n = extract_chunk(sz, text, first, min(sz.stream, len(text) - first), body, stream)
        assert n == stream["out_off"]
    return bytes(body[:n])


def text_chunk_bytes(dna_size: int, chunk_log2: int) -> int:
    """The streaming build's text chunk for leaf chunks of 2^chunk_log2 leaves (build_streaming_fasta)."""
    return max(65536, ((1 << chunk_log2) * dna_size // 2) & ~65535)


# ---- adversarial texts --------------------------------------------------------------------------------------
ACGT = np.frombuffer(b"ACGTacgt", dtype=np.uint8)
IUPAC = np.frombuffer(b"RYKMSWBDHVryk-", dtype=np.uint8)


def letters(rng, n: int) -> bytes:
    """Mixed-case ACGT with a few IUPAC codes and runs of N / n."""
    out = ACGT[rng.integers(0, len(ACGT), n)]
    if n:
        pick = rng.random(n) < 0.004
        out[pick] = IUPAC[rng.integers(0, len(IUPAC), int(pick.sum()))]
        for start in rng.integers(0, n, max(1, n // 3000)):
            out[start:start + int(rng.integers(1, 60))] = ord("N") if rng.integers(2) else ord("n")
    return out.tobytes()


def header(rng, n: int) -> bytes:
    """'>' and n - 1 bytes of printable ASCII (a header line's text, without its newline)."""
    return b">" + rng.integers(0x20, 0x7F, max(0, n - 1)).astype(np.uint8).tobytes()


def data_lines(rng, n: int, width: int = 80) -> bytes:
    """n bytes of data lines (n != 1): no blank line, ends with a newline."""
    assert n != 1
    if n == 0:
        return b""
    out = np.frombuffer(letters(rng, n), dtype=np.uint8).copy()
    w = rng.integers(1, width + 1, n // 2 + 2)
    nl = np.cumsum(w + 1) - 1
    nl = nl[nl < n - 2]
    out[nl] = NL
    out[n - 1] = NL
    return out.tobytes()


def data_line(rng, lo=1, hi=12) -> bytes:
    return letters(rng, int(rng.integers(lo, hi))) + b"\n"


def hb_run(rng, k: int, valid: bool, first: int = 0) -> bytes:
    """k hb lines after a data line (or after `first` hb lines): the lines read as data are blank when valid."""
    lines = []
    for i in range(first, first + k):
        if (valid and i % 2) or rng.integers(2):
            lines.append(b"\n")
        else:
            lines.append(header(rng, int(rng.integers(1, 9))) + b"\n")
    return b"".join(lines)


SMALL_EVENTS = ("line_start", "newline", "header", "run")
LARGE_EVENTS = ("blank_tile", "long_header", "long_data")


def event(rng, kind: str, sz: Sizes, valid: bool):
    """(bytes, anchor): an event that starts at a line start and ends with a data line; its byte `anchor` is the one
    placed on the target offset."""
    if kind == "line_start":
        return data_line(rng), 0
    if kind == "newline":
        e = data_line(rng)
        return e, len(e) - 1
    if kind == "header":
        h = header(rng, int(rng.integers(1, 20))) + b"\n"
        return h + data_line(rng), (0 if rng.integers(2) else len(h) - 1)
    if kind == "run":
        r = hb_run(rng, int(rng.integers(1, 7)), valid)
        return r + data_line(rng), int(rng.integers(0, len(r) + 1))
    if kind == "blank_tile":  # a whole tile of blank lines (all_hb through a tile), then a header when it is skipped
        k = sz.tile + int(rng.integers(1, 300))
        r = b"\n" * k
        if not valid or k % 2 == 0:
            r += header(rng, int(rng.integers(1, 30))) + b"\n"
        return r + data_line(rng), int(rng.integers(0, k))
    if kind == "long_header":  # whole tiles without a line start, inside a skipped line
        h = header(rng, sz.tile + int(rng.integers(1, 2 * sz.tile)))
        return h + b"\n" + data_line(rng), int(rng.integers(0, len(h) + 1))
    if kind == "long_data":  # whole tiles without a line start, inside a kept line
        d = letters(rng, 3 * sz.tile + int(rng.integers(1, sz.tile)))
        return d + b"\n", int(rng.integers(0, len(d) + 1))
    raise ValueError(kind)


def adversarial_text(rng, sz: Sizes, targets, length: int, *, valid: bool = True, large: float = 0.0,
                     head: str = "", tail: str = "") -> bytes:
    """Data lines with an event placed on every target offset that the previous event has not passed.

    targets: sorted offsets (boundary + shift).  large: the share of events that span whole tiles.
    head: "" | "nl" (the text starts with a blank line) | "gt" (with a header).
    tail: "" | "nofinal" (no final newline) | "header" (ends inside a header) | "blanks" (in a run of blank lines).
    valid: every line read as data is blank or holds symbols only (the reference accepts the text)."""
    out = bytearray()
    if head:
        out += (b"\n" if head == "nl" else header(rng, 9) + b"\n") + data_line(rng)
    for pos in targets:
        kinds = LARGE_EVENTS if rng.random() < large else SMALL_EVENTS
        e, a = event(rng, kinds[int(rng.integers(len(kinds)))], sz, valid)
        gap = pos - a - len(out)
        if gap < 0 or gap == 1 or pos >= length:
            continue
        out += data_lines(rng, gap, int(rng.choice([3, 20, 80])))
        out += e
    gap = length - len(out)
    if gap > 1:
        out += data_lines(rng, gap)
    if tail == "nofinal":
        out = out.rstrip(b"\n")
    elif tail == "header":
        out += header(rng, int(rng.integers(1, 40)))
    elif tail == "blanks":
        out += b"\n" * int(rng.integers(1, 6))
    return bytes(out)


def boundary_targets(period: int, length: int, rotation: int, first: int = 1):
    """b + d for every multiple b of `period` below `length` (from the `first`-th), d cycling through -3..+3 from
    `rotation` on: seven rotations put every shift on every boundary."""
    return [b * period + ((b + rotation) % 7) - 3 for b in range(first, -(-length // period))]
