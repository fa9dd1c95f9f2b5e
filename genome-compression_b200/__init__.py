"""genome-compression_b200 — B200-native shared_tree (hash-consed DNA tree) hot path.

Thin ctypes binding over the C ABI in include/shared_tree_b200.h.  The class mirrors
the reference's ``shared_tree`` surface (include/shared_tree.h:154-237): construct from
FASTA text or packed leaves, ``depth / width / leaf_count / node_count``,
``sort_tree``, ``bytes / serialize / deserialize``, iteration (decode) and
``operator[]`` (random access).

All computation runs in libshared_tree_b200.so (hand-written CUDA, sm_100a).  There is
no CPU path: importing works without a GPU (so symbols can be checked), but every
computing call raises ``StbError`` when no CUDA device is present, and the import
fails loudly when the library has not been built.
"""
from __future__ import annotations

import ctypes as C
import importlib.util
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libshared_tree_b200.so"
HEADER_PATH = _HERE.parent / "include" / "shared_tree_b200.h"

HOST, DEVICE = 0, 1
NULL = 0x9FFFFFFF
IDX_MASK = 0x1FFFFFFF
MIRROR, TRANSPOSE, INVARIANT = 0x20000000, 0x40000000, 0x80000000

STATUS = {
    0: "STB_OK", 1: "STB_ERR_CUDA", 2: "STB_ERR_INVALID_ARG", 3: "STB_ERR_UNKNOWN_SYMBOL", 4: "STB_ERR_EMPTY",
    5: "STB_ERR_BUFFER_TOO_SMALL", 6: "STB_ERR_NOT_BUILT", 7: "STB_ERR_INDEX_CEILING", 8: "STB_ERR_BAD_LEAF",
    9: "STB_ERR_OUT_OF_RANGE", 10: "STB_ERR_BAD_STREAM", 11: "STB_ERR_TOO_LARGE",
}


class StbError(RuntimeError):
    def __init__(self, status: int, detail: str = ""):
        self.status = status
        self.name = STATUS.get(status, str(status))
        super().__init__(f"{self.name}: {detail}" if detail else self.name)


def build_library(force: bool = False) -> Path:
    spec = importlib.util.spec_from_file_location("_stb_build", _HERE / "_build.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build(force=force)


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python genome-compression_b200/_build.py` "
            "(there is no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    u64, u32, i32, vp, cp = C.c_uint64, C.c_uint32, C.c_int, C.c_void_p, C.c_char_p
    P = C.POINTER
    sig = {
        "stb_create": [P(vp), i32, i32, vp],
        "stb_destroy": [vp],
        "stb_clone": [vp, P(vp)],
        "stb_release_workspace": [vp],
        "stb_set_option": [vp, cp, u64],
        "stb_get_option": [vp, cp, P(u64)],
        "stb_build_from_fasta": [vp, vp, u64, i32],
        "stb_build_from_body": [vp, vp, u64, i32],
        "stb_build_from_leaves": [vp, vp, u64, i32],
        "stb_pack_fasta": [vp, vp, u64, i32, vp, u64, i32, P(u64)],
        "stb_depth": [vp, P(u64)],
        "stb_width": [vp, P(u64)],
        "stb_leaf_count": [vp, P(u64)],
        "stb_node_count": [vp, P(u64)],
        "stb_layer_count": [vp, u64, P(u64)],
        "stb_root": [vp, P(u32)],
        "stb_dna_size": [vp, P(i32)],
        "stb_copy_leaves": [vp, vp, u64, i32],
        "stb_copy_layer": [vp, u64, vp, u64, i32],
        "stb_histogram": [vp, u64, vp, u64, i32],
        "stb_sort_tree": [vp],
        "stb_bytes": [vp, P(u64)],
        "stb_serialize": [vp, vp, u64, i32, P(u64)],
        "stb_deserialize": [vp, vp, u64],
        "stb_decode_leaves": [vp, u64, u64, vp, i32],
        "stb_decode_ascii": [vp, u64, u64, vp, i32],
        "stb_random_access": [vp, vp, u64, vp, i32],
        "stb_extract_regions": [vp, vp, vp, vp, u64, vp, u64, i32, P(u64)],
        "stb_profile_enable": [vp, i32],
        "stb_profile_reset": [vp],
        "stb_profile_read": [vp, P(cp), P(C.c_double), P(u64), u64, P(u64)],
        "stb_synth_genome": [i32, vp, vp, u64, u64, u64, u64, u32],
        "stb_synth_mask": [i32, vp, vp, u64, u64, u64],
        # include/shared_tree_b200_dist.h
        "stb_dist_pack_body": [vp, vp, u64, vp],
        "stb_dist_partition": [vp, i32, vp, u64, u64, i32, vp, vp, vp, vp],
        "stb_dist_owner": [vp, vp, vp, u64, vp, u32, vp, vp],
        "stb_dist_rank_index": [vp, vp, u64, vp, vp],
        "stb_dist_finish": [vp, i32, vp, u64, u64, vp, vp, u64, vp, vp, vp, vp, vp],
        "stb_dist_upper_levels": [vp, vp, u64, i32],
        "stb_dist_leaf_direct_minpos": [vp, vp, u64, u64, vp, vp, P(i32)],
        "stb_dist_leaf_direct_finish": [vp, vp, u64, vp, u64, vp, vp, vp, vp, vp, vp],
        "stb_assemble": [vp, vp, u64, u64, P(u64), P(vp), u32, u64],
        "stb_dist_peer_alloc": [vp, u64, P(vp), vp],
        "stb_dist_peer_open": [vp, vp, P(vp)],
        "stb_dist_peer_close": [vp, vp],
        "stb_dist_peer_free": [vp, vp],
        "stb_dist_peer_scatter": [vp, i32, vp, u64, u64, i32, i32, P(vp), u64, vp],
        "stb_dist_peer_owner": [vp, i32, i32, P(vp), u64, u64, vp, u64, u32, vp, vp, u64, vp],
        "stb_dist_peer_finish": [vp, i32, vp, u64, u64, vp, vp, u64, vp, vp, i32, u64, vp, vp, vp],
        "stb_dist_peer_put": [vp, vp, vp, u64],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = i32
    lib.stb_node_canonical.argtypes = [u32, u32, P(u32), P(u32), P(u32)]
    lib.stb_node_canonical.restype = None
    lib.stb_leaf_canonical.argtypes = [u64, i32, P(u32)]
    lib.stb_leaf_canonical.restype = u64
    lib.stb_pointer_compose.argtypes = [u32, i32, i32]
    lib.stb_pointer_compose.restype = u32
    lib.stb_status_string.argtypes = [i32]
    lib.stb_status_string.restype = cp
    lib.stb_last_error.argtypes = [vp]
    lib.stb_last_error.restype = cp
    lib.stb_dist_peer_arena_bytes.argtypes = [i32, u64]
    lib.stb_dist_peer_arena_bytes.restype = u64
    lib.stb_dist_peer_payload.argtypes = [vp, i32, u64]
    lib.stb_dist_peer_payload.restype = vp
    lib.stb_kernel_launches.argtypes = []
    lib.stb_kernel_launches.restype = u64
    return lib


lib = _load()


def kernel_launches() -> int:
    return int(lib.stb_kernel_launches())


def _is_device_tensor(x) -> bool:
    return hasattr(x, "data_ptr") and hasattr(x, "is_cuda") and bool(x.is_cuda)


def _as_input(x, dtype):
    """Returns (pointer, element count, memory kind, keepalive)."""
    if _is_device_tensor(x):
        assert x.is_contiguous()
        assert x.element_size() == np.dtype(dtype).itemsize, "device tensor has the wrong element size"
        return x.data_ptr(), x.numel(), DEVICE, x
    if hasattr(x, "data_ptr"):  # CPU torch tensor (possibly pinned)
        assert x.is_contiguous()
        return x.data_ptr(), x.numel() * x.element_size() // np.dtype(dtype).itemsize, HOST, x
    if isinstance(x, (bytes, bytearray, memoryview)):
        arr = np.frombuffer(x, dtype=np.uint8)
        if np.dtype(dtype) != np.uint8:
            arr = arr.view(dtype)
    else:
        arr = np.ascontiguousarray(x, dtype=dtype)
    return arr.ctypes.data, arr.size, HOST, arr


class SharedTree:
    """Device-resident shared tree; the reference's ``shared_tree`` (include/shared_tree.h:154)."""

    def __init__(self, dna_size: int = 12, device: int = 0, stream: int | None = None):
        self._h = C.c_void_p()
        self.dna_size = dna_size
        self.device = device
        st = lib.stb_create(C.byref(self._h), device, dna_size, C.c_void_p(stream or 0))
        if st != 0:
            self._h = C.c_void_p()
            raise StbError(st, lib.stb_status_string(st).decode())

    # -- plumbing -----------------------------------------------------------------
    def _check(self, st: int):
        if st != 0:
            raise StbError(st, lib.stb_last_error(self._h).decode() or lib.stb_status_string(st).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib.stb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _u64(self, fn, *args) -> int:
        out = C.c_uint64(0)
        self._check(fn(self._h, *args, C.byref(out)))
        return int(out.value)

    def set_option(self, name: str, value: int) -> "SharedTree":
        """Thresholds between the build's code paths (include/shared_tree_b200.h: stb_set_option)."""
        self._check(lib.stb_set_option(self._h, name.encode(), int(value)))
        return self

    def get_option(self, name: str) -> int:
        return self._u64(lib.stb_get_option, name.encode())

    # -- construction (shared_tree ctors, src/shared_tree.cpp:207-215) -----------------
    def build_from_fasta(self, text) -> "SharedTree":
        ptr, n, mem, _keep = _as_input(text, np.uint8)
        self._check(lib.stb_build_from_fasta(self._h, ptr, n, mem))
        return self

    def build_from_body(self, body) -> "SharedTree":
        ptr, n, mem, _keep = _as_input(body, np.uint8)
        self._check(lib.stb_build_from_body(self._h, ptr, n, mem))
        return self

    def build_from_leaves(self, leaves) -> "SharedTree":
        ptr, n, mem, _keep = _as_input(leaves, np.uint64)
        self._check(lib.stb_build_from_leaves(self._h, ptr, n, mem))
        return self

    def pack_fasta(self, text) -> np.ndarray:
        """read_genome (src/fasta_reader.cpp:108): FASTA text -> packed leaves (host array)."""
        ptr, n, mem, _keep = _as_input(text, np.uint8)
        count = C.c_uint64(0)
        self._check(lib.stb_pack_fasta(self._h, ptr, n, mem, None, 0, HOST, C.byref(count)))
        out = np.zeros(count.value, dtype=np.uint64)
        self._check(lib.stb_pack_fasta(self._h, ptr, n, mem, out.ctypes.data, out.size, HOST, C.byref(count)))
        return out

    def clone(self) -> "SharedTree":
        other = object.__new__(SharedTree)
        other.dna_size, other.device = self.dna_size, self.device
        other._h = C.c_void_p()
        self._check(lib.stb_clone(self._h, C.byref(other._h)))
        return other

    # -- queries (include/shared_tree.h:164-170) -----------------------------------------
    def depth(self) -> int: return self._u64(lib.stb_depth)
    def width(self) -> int: return self._u64(lib.stb_width)
    def leaf_count(self) -> int: return self._u64(lib.stb_leaf_count)
    def node_count(self) -> int: return self._u64(lib.stb_node_count)
    def layer_count(self, layer: int) -> int: return self._u64(lib.stb_layer_count, layer)
    def layer_counts(self): return [self.layer_count(k) for k in range(self.depth() - 1)]

    def root(self) -> int:
        out = C.c_uint32(0)
        self._check(lib.stb_root(self._h, C.byref(out)))
        return int(out.value)

    def leaves(self) -> np.ndarray:
        out = np.zeros(self.leaf_count(), dtype=np.uint64)
        self._check(lib.stb_copy_leaves(self._h, out.ctypes.data, out.size, HOST))
        return out

    def layer(self, k: int) -> np.ndarray:
        out = np.zeros((self.layer_count(k), 2), dtype=np.uint32)
        self._check(lib.stb_copy_layer(self._h, k, out.ctypes.data, out.shape[0], HOST))
        return out

    def histogram(self, k: int, out=None):
        """References from node layer k into its child layer.  out: a contiguous int64 or uint64 CUDA tensor of at
        least that many elements, filled on the device."""
        n = self.leaf_count() if k == 0 else self.layer_count(k - 1)
        if out is not None:
            import torch
            if not (_is_device_tensor(out) and out.is_contiguous() and out.dtype in (torch.int64, torch.uint64)):
                raise TypeError("histogram(out=...): a contiguous CUDA tensor of torch.int64 or torch.uint64")
            self._check(lib.stb_histogram(self._h, k, out.data_ptr(), out.numel(), DEVICE))
            return out
        out = np.zeros(n, dtype=np.uint64)
        self._check(lib.stb_histogram(self._h, k, out.ctypes.data, n, HOST))
        return out

    # -- sort / stream (src/shared_tree.cpp:443, :488-546) ----------------------------
    def sort(self) -> "SharedTree":
        self._check(lib.stb_sort_tree(self._h))
        return self

    sort_tree = sort

    def bytes(self) -> int: return self._u64(lib.stb_bytes)

    def serialize(self) -> bytes:
        n = self.bytes()
        out = np.zeros(n, dtype=np.uint8)
        written = C.c_uint64(0)
        self._check(lib.stb_serialize(self._h, out.ctypes.data, n, HOST, C.byref(written)))
        assert written.value == n
        return out.tobytes()

    def serialize_into(self, device_tensor) -> int:
        written = C.c_uint64(0)
        self._check(lib.stb_serialize(self._h, device_tensor.data_ptr(), device_tensor.numel(), DEVICE, C.byref(written)))
        return int(written.value)

    def serialize_to_host(self, host_tensor) -> int:
        """stb_serialize into caller-owned HOST memory (a pinned torch tensor or a numpy array)."""
        ptr, n, mem, _keep = _as_input(host_tensor, np.uint8)
        assert mem == HOST
        written = C.c_uint64(0)
        self._check(lib.stb_serialize(self._h, ptr, n, HOST, C.byref(written)))
        return int(written.value)

    def deserialize(self, data: bytes) -> "SharedTree":
        arr = np.frombuffer(data, dtype=np.uint8)
        self._check(lib.stb_deserialize(self._h, arr.ctypes.data, arr.size))
        return self

    # -- decode (iterator, operator[]) -------------------------------------------------
    def decode(self, first: int = 0, count: int | None = None, out=None):
        count = self.width() - first if count is None else count
        if out is not None:
            self._check(lib.stb_decode_leaves(self._h, first, count, out.data_ptr(), DEVICE))
            return out
        res = np.zeros(count, dtype=np.uint64)
        self._check(lib.stb_decode_leaves(self._h, first, count, res.ctypes.data, HOST))
        return res

    def decode_ascii(self, first: int = 0, count: int | None = None, out=None):
        count = self.width() - first if count is None else count
        if out is not None:
            self._check(lib.stb_decode_ascii(self._h, first, count, out.data_ptr(), DEVICE))
            return out
        res = np.zeros(count * self.dna_size, dtype=np.uint8)
        self._check(lib.stb_decode_ascii(self._h, first, count, res.ctypes.data, HOST))
        return res.tobytes()

    def decode_ascii_to_host(self, host_tensor, first: int = 0, count: int | None = None):
        """stb_decode_ascii into caller-owned HOST memory (a pinned torch tensor or a numpy array)."""
        count = self.width() - first if count is None else count
        ptr, n, mem, _keep = _as_input(host_tensor, np.uint8)
        assert mem == HOST and n >= count * self.dna_size
        self._check(lib.stb_decode_ascii(self._h, first, count, ptr, HOST))
        return host_tensor

    def random_access(self, index, out=None):
        if out is not None:
            self._check(lib.stb_random_access(self._h, index.data_ptr(), index.numel(), out.data_ptr(), DEVICE))
            return out
        idx = np.ascontiguousarray(index, dtype=np.uint64)
        res = np.zeros(idx.size, dtype=np.uint64)
        self._check(lib.stb_random_access(self._h, idx.ctypes.data, idx.size, res.ctypes.data, HOST))
        return res

    def extract_regions(self, start, end, strand=None, out=None):
        """Bases [start[i], end[i]) of the sequence (0-based, half-open as in BED), strand[i] = 1 for the reverse
        complement, back to back in input order (stb_extract_regions).  Host arrays: returns the letters as bytes.
        CUDA tensors (8-byte start / end, uint8 strand and out): fills out and returns the total length; without
        out, only returns the total length."""
        if _is_device_tensor(start):
            for x, size in ((start, 8), (end, 8), (strand, 1), (out, 1)):
                if x is not None:
                    assert _is_device_tensor(x) and x.is_contiguous() and x.element_size() == size, \
                        "device regions: contiguous CUDA tensors, 8-byte start / end, uint8 strand and out"
            assert end.numel() == start.numel() and (strand is None or strand.numel() == start.numel())
            written = C.c_uint64(0)
            self._check(lib.stb_extract_regions(self._h, start.data_ptr(), end.data_ptr(),
                                                None if strand is None else strand.data_ptr(), start.numel(),
                                                None if out is None else out.data_ptr(), 0 if out is None else out.numel(),
                                                DEVICE, C.byref(written)))
            return int(written.value)
        s = np.ascontiguousarray(start, dtype=np.uint64)
        e = np.ascontiguousarray(end, dtype=np.uint64)
        st = None if strand is None else np.ascontiguousarray(strand, dtype=np.uint8)
        assert e.size == s.size and (st is None or st.size == s.size)
        # sized here when the regions are ordered; otherwise the call reports them before writing anything
        total = int((e - s).sum(dtype=np.uint64)) if bool((e >= s).all()) else 0
        res = np.zeros(max(total, 1), dtype=np.uint8)
        written = C.c_uint64(0)
        self._check(lib.stb_extract_regions(self._h, s.ctypes.data, e.ctypes.data, None if st is None else st.ctypes.data,
                                            s.size, res.ctypes.data, total, HOST, C.byref(written)))
        return res[:written.value].tobytes()

    def __getitem__(self, i: int) -> int:
        return int(self.random_access(np.array([i], dtype=np.uint64))[0])

    def __iter__(self):
        return iter(self.decode())

    # -- profiling ------------------------------------------------------------------------
    def profile(self, on: bool = True): self._check(lib.stb_profile_enable(self._h, int(on)))
    def profile_reset(self): self._check(lib.stb_profile_reset(self._h))

    def profile_read(self) -> dict:
        cap = 64
        names = (C.c_char_p * cap)()
        ms = (C.c_double * cap)()
        launches = (C.c_uint64 * cap)()
        count = C.c_uint64(0)
        self._check(lib.stb_profile_read(self._h, names, ms, launches, cap, C.byref(count)))
        return {names[i].decode(): {"ms": ms[i], "launches": int(launches[i])} for i in range(min(cap, count.value))}


def synth_genome(out_device_tensor, n_bases: int, first: int = 0, count: int | None = None, seed: int = 42,
                 repeat_permille: int = 500, device: int = 0, stream: int | None = None):
    """Fills a uint8 CUDA tensor with bases [first, first+count) of the synthetic genome."""
    count = out_device_tensor.numel() if count is None else count
    st = lib.stb_synth_genome(device, C.c_void_p(stream or 0), out_device_tensor.data_ptr(), n_bases, first, count, seed,
                              repeat_permille)
    if st != 0:
        raise StbError(st, lib.stb_status_string(st).decode())
    return out_device_tensor


def synth_mask(text_device_tensor, first: int = 0, count: int | None = None, seed: int = 42, device: int = 0, stream: int | None = None):
    """Lays N runs (about 1 % of the bases) and soft-masked lower-case stretches over a generated text, in place."""
    count = text_device_tensor.numel() if count is None else count
    st = lib.stb_synth_mask(device, C.c_void_p(stream or 0), text_device_tensor.data_ptr(), first, count, seed)
    if st != 0:
        raise StbError(st, lib.stb_status_string(st).decode())
    return text_device_tensor


def node_canonical(left: int, right: int):
    """node::canonical as the kernels compute it: (left, right, flags >> 29)."""
    cl, cr, f = C.c_uint32(), C.c_uint32(), C.c_uint32()
    lib.stb_node_canonical(left, right, C.byref(cl), C.byref(cr), C.byref(f))
    return cl.value, cr.value, f.value >> 29


def leaf_canonical(leaf: int, dna_size: int):
    f = C.c_uint32()
    c = lib.stb_leaf_canonical(leaf, dna_size, C.byref(f))
    return int(c), f.value >> 29


def pointer_compose(pointer: int, mirror: int, transpose: int) -> int:
    return int(lib.stb_pointer_compose(pointer, mirror, transpose))


def query_indices(seed: int, queries: int, width: int) -> np.ndarray:
    """The seeded leaf indices of BASELINE.json config 5: idx[i] = splitmix64(seed + (i + 1) * golden) mod width.
    A closed form so that the reference's answers (tests/golden/synth.json, oracle/gen_golden_synth.py) can be
    compared on any machine."""
    with np.errstate(over="ignore"):
        x = np.uint64(seed) + (np.arange(1, queries + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15))
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return (x % np.uint64(width)).astype(np.uint64)


def leaf_to_str(v: int, dna_size: int) -> str:
    letters = "SACRGBNKTWVDYHM-"
    return "".join(letters[(int(v) >> (4 * i)) & 0xF] for i in range(dna_size))
