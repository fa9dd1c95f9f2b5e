"""ctypes access to the two CPU checkers.  TEST INFRASTRUCTURE ONLY.

* ``Oracle``  -> oracle/liboracle.so   (plain-C restatement, oracle/oracle.c)
* ``Ref``     -> oracle/_ref/libref.so (the unmodified reference behind
                 oracle/ref_shim.cpp; exists only where /root/reference was
                 available at build time, or travelled inside the snapshot)

Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline /
--impl reference) import this module.  The product package never does.
Both classes expose the same method names so tests can run one body against
either checker.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "liboracle.so"
REF_SO = HERE / "_ref" / "libref.so"
REF_COMPRESS = HERE / "_ref" / "compress"
REFERENCE_ROOT = Path(os.environ.get("REFERENCE_ROOT", "/root/reference"))

u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")

NULL = 0x9FFFFFFF
IDX_MASK = 0x1FFFFFFF


def build_oracle(force: bool = False) -> Path:
    src = [HERE / "oracle.c", HERE / "oracle.h"]
    if force or not ORACLE_SO.exists() or any(s.stat().st_mtime > ORACLE_SO.stat().st_mtime for s in src):
        subprocess.run(["make", "-C", str(HERE), "oracle"], check=True, capture_output=True)
    return ORACLE_SO


def build_ref(force: bool = False) -> Path | None:
    """Compiles the reference in place when its sources are reachable."""
    if REF_SO.exists() and REF_COMPRESS.exists() and not force:
        return REF_SO
    if not (REFERENCE_ROOT / "src" / "shared_tree.cpp").exists():
        return REF_SO if REF_SO.exists() else None
    subprocess.run(["make", "-C", str(HERE), "ref", f"REF={REFERENCE_ROOT}"], check=True, capture_output=True)
    return REF_SO


def build_dropin() -> bool:
    """Compiles the reference's unmodified compress.cpp / tests/test.cpp against the shim."""
    outs = [HERE / "_ref" / "ref_tests_on_b200", HERE / "_ref" / "ref_compress_on_b200"]
    if (REFERENCE_ROOT / "tests" / "test.cpp").exists():
        subprocess.run(["make", "-C", str(HERE), "dropin", f"REF={REFERENCE_ROOT}"], check=True, capture_output=True)
    return all(o.exists() for o in outs)


def have_ref() -> bool:
    return REF_SO.exists()


class _Tree:
    """Common python view of a built tree (either checker)."""

    def __init__(self, owner, handle, S):
        self._o, self._h, self.S = owner, handle, S

    def __del__(self):
        try:
            self._o._free(self._h)
        except Exception:
            pass

    # the methods below are filled in by the owners through small lambdas
    def depth(self): return self._o._depth(self._h)
    def width(self): return self._o._width(self._h)
    def leaf_count(self): return self._o._leaf_count(self._h)
    def node_count(self): return self._o._node_count(self._h)
    def layer_count(self, k): return self._o._layer_count(self._h, k)
    def layer_counts(self): return [self.layer_count(k) for k in range(self.depth() - 1)]
    def sort(self): self._o._sort(self._h)
    def bytes(self): return self._o._bytes(self._h)
    def serialize(self): return self._o._serialize(self._h)
    def leaves(self): return self._o._leaves(self._h)
    def layer(self, k): return self._o._layer(self._h, k)
    def histogram(self, k): return self._o._histogram(self._h, k)
    def decode(self): return self._o._decode(self._h)
    def random_access(self, idx): return self._o._random_access(self._h, np.ascontiguousarray(idx, dtype=np.uint64))
    def root(self): return self._o._root(self._h)


class Oracle:
    """oracle/oracle.c through ctypes."""

    kind = "port"

    def __init__(self):
        self.lib = L = C.CDLL(str(build_oracle()))
        L.orc_code.restype = C.c_int
        L.orc_pack.restype = C.c_uint64
        L.orc_pack.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_int)]
        for f in ("orc_transposed",):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_uint64]
        for f in ("orc_mirrored", "orc_inverted"):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_uint64, C.c_int]
        L.orc_leaf_canonical.restype = C.c_uint64
        L.orc_leaf_canonical.argtypes = [C.c_uint64, C.c_int, C.POINTER(C.c_int)]
        L.orc_ptr.restype = C.c_uint32
        L.orc_ptr.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int]
        L.orc_compose.restype = C.c_uint32
        L.orc_compose.argtypes = [C.c_uint32, C.c_int, C.c_int]
        L.orc_node_canonical.restype = C.c_int
        L.orc_node_canonical.argtypes = [C.c_uint32, C.c_uint32, u32p]
        L.orc_ptr_serialize.restype = C.c_int
        L.orc_ptr_serialize.argtypes = [C.c_uint32, u8p]
        L.orc_fasta_body.restype = C.c_uint64
        L.orc_fasta_body.argtypes = [C.c_char_p, C.c_uint64, u8p]
        L.orc_fasta_to_leaves.restype = C.c_uint64
        L.orc_fasta_to_leaves.argtypes = [C.c_char_p, C.c_uint64, C.c_int, u64p, C.c_uint64, C.POINTER(C.c_int)]
        L.orc_build.restype = C.c_void_p
        L.orc_build.argtypes = [u64p, C.c_uint64, C.c_int]
        L.orc_build_levels.restype = C.c_void_p
        L.orc_build_levels.argtypes = [u64p, C.c_uint64, C.c_int, u32p, C.c_uint64, u64p, C.c_int, C.POINTER(C.c_int)]
        L.orc_free.argtypes = [C.c_void_p]
        L.orc_sort.argtypes = [C.c_void_p]
        for f in ("orc_bytes", "orc_width", "orc_node_count", "orc_tree_leaf_count"):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_void_p]
        L.orc_tree_layers.restype = C.c_int
        L.orc_tree_layers.argtypes = [C.c_void_p]
        L.orc_tree_layer_size.restype = C.c_uint64
        L.orc_tree_layer_size.argtypes = [C.c_void_p, C.c_int]
        L.orc_tree_leaves.restype = C.POINTER(C.c_uint64)
        L.orc_tree_leaves.argtypes = [C.c_void_p]
        L.orc_tree_layer.restype = C.POINTER(C.c_uint32)
        L.orc_tree_layer.argtypes = [C.c_void_p, C.c_int]
        L.orc_tree_root.restype = C.c_uint32
        L.orc_tree_root.argtypes = [C.c_void_p]
        L.orc_serialize.restype = C.c_uint64
        L.orc_serialize.argtypes = [C.c_void_p, u8p, C.c_uint64]
        L.orc_deserialize.restype = C.c_void_p
        L.orc_deserialize.argtypes = [u8p, C.c_uint64, C.c_int]
        L.orc_decode.restype = C.c_uint64
        L.orc_decode.argtypes = [C.c_void_p, u64p, C.c_uint64]
        L.orc_random_access.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p]
        L.orc_histogram.argtypes = [C.c_void_p, C.c_int, u64p]
        L.orc_synth_repeats.restype = C.c_uint64
        L.orc_synth_repeats.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64]
        L.orc_synth_fill.argtypes = [u8p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64]
        L.orc_synth_mask.argtypes = [u8p, C.c_uint64, C.c_uint64, C.c_uint64]
        L.orc_synth_mask.restype = None

    # ---- primitives ----
    def pack(self, text: bytes, S: int):
        bad = C.c_int(-1)
        v = self.lib.orc_pack(text, S, C.byref(bad))
        return v, bad.value

    def transposed(self, v, S): return self.lib.orc_transposed(v)
    def mirrored(self, v, S): return self.lib.orc_mirrored(v, S)
    def inverted(self, v, S): return self.lib.orc_inverted(v, S)

    def leaf_canonical(self, v, S):
        f = C.c_int(0)
        c = self.lib.orc_leaf_canonical(v, S, C.byref(f))
        return c, f.value

    def pointer(self, index, m, t, inv): return self.lib.orc_ptr(index, m, t, inv)
    def compose(self, p, m, t): return self.lib.orc_compose(p, m, t)

    def node_canonical(self, l, r):
        out = np.zeros(2, dtype=np.uint32)
        f = self.lib.orc_node_canonical(l, r, out)
        return int(out[0]), int(out[1]), f

    def pointer_serialize(self, raw):
        out = np.zeros(4, dtype=np.uint8)
        n = self.lib.orc_ptr_serialize(raw, out)
        return bytes(out[:n])

    # ---- ingest ----
    def fasta_body(self, text: bytes) -> bytes:
        out = np.zeros(max(len(text), 1), dtype=np.uint8)
        n = self.lib.orc_fasta_body(text, len(text), out)
        return bytes(out[:n])

    def fasta_to_leaves(self, text, S: int):
        """text: bytes, or a contiguous uint8 array (read in place: no copy of a multi-GB text)."""
        size = len(text)
        cap = size // S + 1
        out = np.zeros(cap, dtype=np.uint64)
        bad = C.c_int(-1)
        ptr = text
        if isinstance(text, np.ndarray):  # `text` keeps the array alive during the call
            assert text.dtype == np.uint8 and text.flags.c_contiguous
            ptr = C.cast(text.ctypes.data, C.c_char_p)
        n = self.lib.orc_fasta_to_leaves(ptr, size, S, out, cap, C.byref(bad))
        if n == 0xFFFFFFFFFFFFFFFF:
            raise ValueError(f"unknown symbol {bad.value}")
        return out[:n].copy()

    # ---- tree ----
    def build(self, leaves, S):
        leaves = np.ascontiguousarray(leaves, dtype=np.uint64)
        h = self.lib.orc_build(leaves, len(leaves), S)
        if not h:
            raise ValueError("empty input")
        return _Tree(self, h, S)

    def build_levels(self, leaves, S):
        """Returns (tree, [pointer array per level])."""
        leaves = np.ascontiguousarray(leaves, dtype=np.uint64)
        cap = len(leaves) + 64
        out = np.zeros(cap, dtype=np.uint32)
        sizes = np.zeros(64, dtype=np.uint64)
        nl = C.c_int(0)
        h = self.lib.orc_build_levels(leaves, len(leaves), S, out, cap, sizes, 64, C.byref(nl))
        levels, o = [], 0
        for k in range(nl.value):
            levels.append(out[o:o + int(sizes[k])].copy())
            o += int(sizes[k])
        return _Tree(self, h, S), levels

    def deserialize(self, data: bytes, S):
        arr = np.frombuffer(data, dtype=np.uint8).copy()
        return _Tree(self, self.lib.orc_deserialize(arr, len(arr), S), S)

    def _free(self, h): self.lib.orc_free(h)
    def _depth(self, h): return self.lib.orc_tree_layers(h) + 1
    def _width(self, h): return self.lib.orc_width(h)
    def _leaf_count(self, h): return self.lib.orc_tree_leaf_count(h)
    def _node_count(self, h): return self.lib.orc_node_count(h)
    def _layer_count(self, h, k): return self.lib.orc_tree_layer_size(h, k)
    def _sort(self, h): self.lib.orc_sort(h)
    def _bytes(self, h): return self.lib.orc_bytes(h)
    def _root(self, h): return self.lib.orc_tree_root(h)

    def _serialize(self, h):
        n = self.lib.orc_bytes(h)
        out = np.zeros(n, dtype=np.uint8)
        w = self.lib.orc_serialize(h, out, n)
        assert w == n
        return out.tobytes()

    def _leaves(self, h):
        n = self.lib.orc_tree_leaf_count(h)
        return np.ctypeslib.as_array(self.lib.orc_tree_leaves(h), shape=(n,)).copy() if n else np.zeros(0, np.uint64)

    def _layer(self, h, k):
        n = self.lib.orc_tree_layer_size(h, k)
        return np.ctypeslib.as_array(self.lib.orc_tree_layer(h, k), shape=(n, 2)).copy() if n else np.zeros((0, 2), np.uint32)

    def _histogram(self, h, k):
        n = self.lib.orc_tree_leaf_count(h) if k == 0 else self.lib.orc_tree_layer_size(h, k - 1)
        out = np.zeros(n, dtype=np.uint64)
        self.lib.orc_histogram(h, k, out)
        return out

    def _decode(self, h):
        n = self.lib.orc_width(h)
        out = np.zeros(n, dtype=np.uint64)
        w = self.lib.orc_decode(h, out, n)
        assert w == n, (w, n)
        return out

    def _random_access(self, h, idx):
        out = np.zeros(len(idx), dtype=np.uint64)
        self.lib.orc_random_access(h, idx, len(idx), out)
        return out

    # ---- synthetic data ----
    REPEAT_DTYPE = np.dtype([("dst", "<u8"), ("src", "<u8"), ("len", "<u8"), ("rc", "<u4"), ("pad", "<u4")])

    def synth_repeats(self, n_bases, seed, permille):
        n = self.lib.orc_synth_repeats(n_bases, seed, permille, None, 0)
        out = np.zeros(max(n, 1), dtype=self.REPEAT_DTYPE)
        self.lib.orc_synth_repeats(n_bases, seed, permille, out.ctypes.data, n)
        return out[:n]

    def synth(self, n_bases, seed, permille, first=0, count=None):
        reps = self.synth_repeats(n_bases, seed, permille)
        count = n_bases - first if count is None else count
        out = np.zeros(count, dtype=np.uint8)
        self.lib.orc_synth_fill(out, first, count, seed, reps.ctypes.data if len(reps) else None, len(reps))
        return out


    def synth_mask(self, text, first, seed):
        """In place: N runs and soft-masking over bases [first, first + len(text)) (orc_synth_mask)."""
        self.lib.orc_synth_mask(text, first, len(text), seed)
        return text


class Ref:
    """The unmodified reference through oracle/ref_shim.cpp."""

    kind = "reference"

    def __init__(self):
        so = build_ref()
        if so is None or not so.exists():
            raise FileNotFoundError("oracle/_ref/libref.so is not built and /root/reference is absent")
        self.lib = L = C.CDLL(str(so))
        L.ref_dna_pack.restype = C.c_uint64
        L.ref_dna_pack.argtypes = [C.c_char_p, C.c_int]
        for f in ("ref_dna_transposed", "ref_dna_mirrored", "ref_dna_inverted"):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_uint64, C.c_int]
        L.ref_dna_canonical.restype = C.c_uint64
        L.ref_dna_canonical.argtypes = [C.c_uint64, C.c_int, C.POINTER(C.c_int)]
        L.ref_pointer_make.restype = C.c_uint32
        L.ref_pointer_make.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int]
        L.ref_pointer_null.restype = C.c_uint32
        L.ref_pointer_compose.restype = C.c_uint32
        L.ref_pointer_compose.argtypes = [C.c_uint32, C.c_int, C.c_int]
        L.ref_node_canonical.restype = C.c_int
        L.ref_node_canonical.argtypes = [C.c_uint32, C.c_uint32, u32p]
        L.ref_pointer_serialize.restype = C.c_int
        L.ref_pointer_serialize.argtypes = [C.c_uint32, u8p]
        L.ref_read_genome.restype = C.c_uint64
        L.ref_read_genome.argtypes = [C.c_char_p, C.c_int, u64p, C.c_uint64]
        L.ref_tree_from_file.restype = C.c_void_p
        L.ref_tree_from_file.argtypes = [C.c_char_p, C.c_int]
        L.ref_tree_from_leaves.restype = C.c_void_p
        L.ref_tree_from_leaves.argtypes = [u64p, C.c_uint64, C.c_int]
        L.ref_tree_deserialize.restype = C.c_void_p
        L.ref_tree_deserialize.argtypes = [u8p, C.c_uint64, C.c_int]
        L.ref_tree_free.argtypes = [C.c_void_p]
        for f in ("ref_tree_depth", "ref_tree_width", "ref_tree_leaf_count", "ref_tree_node_count", "ref_tree_bytes"):
            getattr(L, f).restype = C.c_uint64
            getattr(L, f).argtypes = [C.c_void_p]
        L.ref_tree_layer_count.restype = C.c_uint64
        L.ref_tree_layer_count.argtypes = [C.c_void_p, C.c_uint64]
        L.ref_tree_sort.argtypes = [C.c_void_p]
        L.ref_tree_serialize.restype = C.c_uint64
        L.ref_tree_serialize.argtypes = [C.c_void_p, u8p, C.c_uint64]
        L.ref_tree_leaves.restype = C.c_uint64
        L.ref_tree_leaves.argtypes = [C.c_void_p, u64p, C.c_uint64]
        L.ref_tree_layer.restype = C.c_uint64
        L.ref_tree_layer.argtypes = [C.c_void_p, C.c_uint64, u32p, C.c_uint64]
        L.ref_tree_histogram.restype = C.c_uint64
        L.ref_tree_histogram.argtypes = [C.c_void_p, C.c_uint64, u64p, C.c_uint64]
        L.ref_tree_decode.restype = C.c_uint64
        L.ref_tree_decode.argtypes = [C.c_void_p, u64p, C.c_uint64]
        L.ref_tree_random_access.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p]
        L.ref_build_levels.restype = C.c_uint64
        L.ref_build_levels.argtypes = [u64p, C.c_uint64, C.c_int, u32p, C.c_uint64, u64p, C.c_uint64]

    # ---- primitives ----
    def pack(self, text: bytes, S: int): return self.lib.ref_dna_pack(text, S), -1
    def transposed(self, v, S): return self.lib.ref_dna_transposed(v, S)
    def mirrored(self, v, S): return self.lib.ref_dna_mirrored(v, S)
    def inverted(self, v, S): return self.lib.ref_dna_inverted(v, S)

    def leaf_canonical(self, v, S):
        f = C.c_int(0)
        c = self.lib.ref_dna_canonical(v, S, C.byref(f))
        return c, f.value

    def pointer(self, index, m, t, inv): return self.lib.ref_pointer_make(index, m, t, inv)
    def compose(self, p, m, t): return self.lib.ref_pointer_compose(p, m, t)

    def node_canonical(self, l, r):
        out = np.zeros(2, dtype=np.uint32)
        f = self.lib.ref_node_canonical(l, r, out)
        return int(out[0]), int(out[1]), f

    def pointer_serialize(self, raw):
        out = np.zeros(4, dtype=np.uint8)
        n = self.lib.ref_pointer_serialize(raw, out)
        return bytes(out[:n])

    # ---- ingest ----
    def read_genome(self, path, S):
        cap = os.path.getsize(path) // S + 2
        out = np.zeros(cap, dtype=np.uint64)
        n = self.lib.ref_read_genome(str(path).encode(), S, out, cap)
        return out[:n].copy()

    # ---- tree ----
    def build(self, leaves, S):
        leaves = np.ascontiguousarray(leaves, dtype=np.uint64)
        return _Tree(self, self.lib.ref_tree_from_leaves(leaves, len(leaves), S), S)

    def build_file(self, path, S):
        return _Tree(self, self.lib.ref_tree_from_file(str(path).encode(), S), S)

    def build_levels(self, leaves, S):
        leaves = np.ascontiguousarray(leaves, dtype=np.uint64)
        cap = len(leaves) + 64
        out = np.zeros(cap, dtype=np.uint32)
        sizes = np.zeros(64, dtype=np.uint64)
        nl = self.lib.ref_build_levels(leaves, len(leaves), S, out, cap, sizes, 64)
        levels, o = [], 0
        for k in range(nl):
            levels.append(out[o:o + int(sizes[k])].copy())
            o += int(sizes[k])
        return None, levels

    def deserialize(self, data: bytes, S):
        arr = np.frombuffer(data, dtype=np.uint8).copy()
        return _Tree(self, self.lib.ref_tree_deserialize(arr, len(arr), S), S)

    def _free(self, h): self.lib.ref_tree_free(h)
    def _depth(self, h): return self.lib.ref_tree_depth(h)
    def _width(self, h): return self.lib.ref_tree_width(h)
    def _leaf_count(self, h): return self.lib.ref_tree_leaf_count(h)
    def _node_count(self, h): return self.lib.ref_tree_node_count(h)
    def _layer_count(self, h, k): return self.lib.ref_tree_layer_count(h, k)
    def _sort(self, h): self.lib.ref_tree_sort(h)
    def _bytes(self, h): return self.lib.ref_tree_bytes(h)

    def _root(self, h):
        # root is private in the reference; the first serialized pointer is it
        # (flags m/t only; the invariant bit is never stored).
        raise NotImplementedError

    def _serialize(self, h):
        n = self.lib.ref_tree_bytes(h)
        out = np.zeros(n, dtype=np.uint8)
        w = self.lib.ref_tree_serialize(h, out, n)
        assert w == n, (w, n)
        return out.tobytes()

    def _leaves(self, h):
        n = self.lib.ref_tree_leaf_count(h)
        out = np.zeros(n, dtype=np.uint64)
        self.lib.ref_tree_leaves(h, out, n)
        return out

    def _layer(self, h, k):
        n = self.lib.ref_tree_layer_count(h, k)
        out = np.zeros((n, 2), dtype=np.uint32)
        self.lib.ref_tree_layer(h, k, out.reshape(-1), n)
        return out

    def _histogram(self, h, k):
        n = self.lib.ref_tree_leaf_count(h) if k == 0 else self.lib.ref_tree_layer_count(h, k - 1)
        out = np.zeros(n, dtype=np.uint64)
        self.lib.ref_tree_histogram(h, k, out, n)
        return out

    def _decode(self, h):
        n = self.lib.ref_tree_width(h)
        out = np.zeros(n, dtype=np.uint64)
        w = self.lib.ref_tree_decode(h, out, n)
        assert w == n, (w, n)
        return out

    def _random_access(self, h, idx):
        out = np.zeros(len(idx), dtype=np.uint64)
        self.lib.ref_tree_random_access(h, idx, len(idx), out)
        return out
