"""parallel-packed-csr_b200 -- B200-native Parallel Packed CSR edge-update engine.

Python is only the test/bench harness around the C-ABI in include/ppcsr_b200.h (the product boundary;
the reference-compatible C++ classes live in host/).  `Shard` mirrors reference PCSR
(src/pcsr/PCSR.h:64-124) one to one; `ShardedGraph` (router.py) mirrors PPPCSR with one shard per GPU.

There is NO CPU fallback: importing works anywhere, but creating a Shard without the compiled CUDA
library or without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = _build.LIB
SENT = 0xFFFFFFFF


class PpcsrError(RuntimeError):
    pass


class BatchStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "batch_size", "n_ignored", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found",
        "n_windows", "window_slots", "rebalance_bytes", "slots_before", "slots_after")] + [
        ("resized", C.c_uint32), ("whole_array", C.c_uint32)] + [(n, C.c_float) for n in (
            "ms_total", "ms_sort", "ms_locate", "ms_select", "ms_rebalance", "ms_rebalance_kernel")] + [
        ("kernel_launches", C.c_uint32), ("sparse_path", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Geometry(C.Structure):
    _fields_ = [("N", C.c_uint64), ("logN", C.c_uint32), ("H", C.c_uint32), ("n", C.c_uint64), ("items", C.c_uint64)]


class InvariantReport(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "bad_geometry", "bad_sentinel", "bad_order", "bad_leaf_layout", "bad_upper", "bad_lower", "bad_tree",
        "live_items", "edges", "full_leaves")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}

    def violations(self, check_lower=True):
        names = ["bad_geometry", "bad_sentinel", "bad_order", "bad_leaf_layout", "bad_upper", "bad_tree", "full_leaves"]
        if check_lower:
            names.append("bad_lower")
        return {n: getattr(self, n) for n in names if getattr(self, n)}


# every symbol include/ppcsr_b200.h declares: (restype, argtypes)
_vp, _u32, _u64, _i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
SYMBOLS = {
    "ppcsr_last_error": (C.c_char_p, []),
    "ppcsr_device_count": (_i, []),
    "ppcsr_create": (_i, [_u32, _u32, _i, C.POINTER(_vp)]),
    "ppcsr_destroy": (None, [_vp]),
    "ppcsr_set_stream": (_i, [_vp, _vp]),
    "ppcsr_sync": (_i, [_vp]),
    "ppcsr_reserve": (_i, [_vp, _u64, _u64]),
    "ppcsr_apply_batch": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_apply_batch_device": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_submit_batch": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(_u64)]),
    "ppcsr_wait": (_i, [_vp, _u64, C.POINTER(BatchStats)]),
    "ppcsr_apply_batch_pairs": (_i, [_vp, _vp, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_parse_edge_list": (_i, [_i, _vp, _u64, _u32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                   C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u32)]),
    "ppcsr_free_device": (_i, [_i, _vp]),
    "ppcsr_copy_to_host": (_i, [_i, _vp, _vp, _u64]),
    "ppcsr_group_create": (_i, [C.POINTER(_vp), _u32, _vp, _u64, _i, C.POINTER(_vp)]),
    "ppcsr_group_destroy": (None, [_vp]),
    "ppcsr_group_owner": (_u32, [_vp, _u64]),
    "ppcsr_group_apply": (_i, [_vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_add_edge": (_i, [_vp, _u32, _u32, _u32]),
    "ppcsr_remove_edge": (_i, [_vp, _u32, _u32, C.POINTER(_i)]),
    "ppcsr_add_nodes": (_i, [_vp, _u32]),
    "ppcsr_last_stats": (_i, [_vp, C.POINTER(BatchStats)]),
    "ppcsr_bin_by_owner": (_i, [_i, _vp, _vp, _u32, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp]),
    "ppcsr_bin_by_owner_packed": (_i, [_i, _vp, _vp, _u32, _vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "ppcsr_apply_batch_packed_device": (_i, [_vp, _vp, _vp, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_bin_to_peers": (_i, [_i, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _u64]),
    "ppcsr_apply_batch_segments_device": (_i, [_vp, _vp, _vp, _u64, _vp, _u32, _u64, _u32, C.POINTER(BatchStats)]),
    "ppcsr_geometry_of": (_i, [_vp, C.POINTER(Geometry)]),
    "ppcsr_edge_exists": (_i, [_vp, _u32, _u32, C.POINTER(_i), C.POINTER(_u32)]),
    "ppcsr_edges_exist": (_i, [_vp, _vp, _vp, _u64, _vp]),
    "ppcsr_neighbours": (_i, [_vp, _u32, _vp, _u64, C.POINTER(_u64)]),
    "ppcsr_read_neighbourhood": (_i, [_vp, _u32, C.POINTER(_u64)]),
    "ppcsr_num_neighbors": (_i, [_vp, _vp]),
    "ppcsr_node_ranges": (_i, [_vp, _vp, _vp]),
    "ppcsr_export_csr": (_i, [_vp, _vp, _vp, _vp, C.POINTER(_u64)]),
    "ppcsr_pagerank_step_f64": (_i, [_vp, _vp, _vp, _u64]),
    "ppcsr_pagerank_step_f32": (_i, [_vp, _vp, _vp, _u64]),
    "ppcsr_pagerank_push_device": (_i, [_vp, _vp, _vp, _u64]),
    "ppcsr_pagerank": (_i, [_vp, _u32, C.c_double, _vp]),
    "ppcsr_set_whole_array_policy": (_i, [_vp, _i]),
    "ppcsr_bfs": (_i, [_vp, _u32, _vp]),
    "ppcsr_check_invariants": (_i, [_vp, _i, C.POINTER(InvariantReport)]),
    "ppcsr_checksum": (_i, [_vp, _u64, _vp]),
    "ppcsr_snapshot": (_i, [_vp]),
    "ppcsr_restore": (_i, [_vp]),
    "ppcsr_debug_dump": (_i, [_vp, _vp, _vp, _vp]),
    "ppcsr_debug_sort_pairs": (_i, [_i, _vp, _vp, _u64, _i, _i]),
    "ppcsr_debug_exclusive_scan": (_i, [_i, _vp, _vp, _u64]),
}

_lib = None


def load_library(build_if_missing: bool = True) -> C.CDLL:
    """Load libppcsr_b200.so (building it in-tree with nvcc if it is missing). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PPCSR_B200_LIB", LIB_PATH)  # development knob: A/B a differently compiled build
    if not os.path.exists(path):
        if not build_if_missing or path != LIB_PATH:
            raise PpcsrError(f"{path} is missing: build it with `python parallel-packed-csr_b200/build.py`")
        _build.build_library()
    L = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        msg = load_library().ppcsr_last_error()
        raise PpcsrError(f"ppcsr status {rc}: {msg.decode() if msg else ''}")


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _u32_array(a, n=None):
    if a is None:
        return None
    a = np.asarray(a)
    if a.dtype == np.int32 and a.flags.c_contiguous:
        a = a.view(np.uint32)  # same bits, no copy (pinned buffers stay pinned)
    else:
        a = np.ascontiguousarray(a, dtype=np.uint32)
    if n is not None and a.shape != (n,):
        a = np.ascontiguousarray(np.broadcast_to(a, (n,)))
    return a


class Shard:
    """One PCSR instance in the HBM of one GPU (reference PCSR, src/pcsr/PCSR.h:64-124)."""

    def __init__(self, n: int, init_n: int | None = None, device: int = 0):
        self.L = load_library()
        if self.L.ppcsr_device_count() <= device:
            raise PpcsrError("no CUDA device: the B200 engine has no CPU fallback")
        h = C.c_void_p()
        _check(self.L.ppcsr_create(n if init_n is None else init_n, n, device, C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.ppcsr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- updates ----
    def apply(self, src, dst, val=None, default_val: int = 1) -> dict:
        """Host arrays. val: None (all default_val), scalar or array; 0 = remove."""
        src = _u32_array(src)
        dst = _u32_array(dst, src.shape[0])
        val = _u32_array(val, src.shape[0]) if val is not None else None
        st = BatchStats()
        _check(self.L.ppcsr_apply_batch(self.h, _np_ptr(src), _np_ptr(dst), _np_ptr(val), src.shape[0], default_val,
                                        C.byref(st)))
        return st.as_dict()

    def submit(self, src, dst, val=None, default_val: int = 1) -> int:
        """Pipelined host submit (ppcsr_submit_batch): starts the H2D copy, returns a ticket for wait().  The arrays
        must stay alive (and should be pinned) until wait() returns; they are kept referenced here."""
        src = _u32_array(src)
        dst = _u32_array(dst, src.shape[0])
        val = _u32_array(val, src.shape[0]) if val is not None else None
        t = C.c_uint64()
        _check(self.L.ppcsr_submit_batch(self.h, _np_ptr(src), _np_ptr(dst), _np_ptr(val), src.shape[0], default_val,
                                         C.byref(t)))
        if not hasattr(self, "_inflight"):
            self._inflight = {}
        self._inflight[t.value] = (src, dst, val)
        return t.value

    def wait(self, ticket: int) -> dict:
        st = BatchStats()
        _check(self.L.ppcsr_wait(self.h, ticket, C.byref(st)))
        self._inflight.pop(ticket, None)
        return st.as_dict()

    def apply_pairs(self, pairs, default_val: int = 1) -> dict:
        """Interleaved (src, dst) u32 pairs (an [n, 2] array or a flat one): the binary input path."""
        pairs = np.ascontiguousarray(pairs, dtype=np.uint32).reshape(-1)
        st = BatchStats()
        _check(self.L.ppcsr_apply_batch_pairs(self.h, _np_ptr(pairs), pairs.shape[0] // 2, default_val, C.byref(st)))
        return st.as_dict()

    def apply_device(self, d_src: int, d_dst: int, d_val: int | None, count: int, default_val: int = 1) -> dict:
        """Raw device pointers (e.g. torch tensor .data_ptr()) of uint32/int32 arrays."""
        st = BatchStats()
        _check(self.L.ppcsr_apply_batch_device(self.h, d_src, d_dst, d_val, count, default_val, C.byref(st)))
        return st.as_dict()

    def apply_packed_device(self, d_packed: int, d_val: int | None, count: int, default_val: int = 1) -> dict:
        """Device pointer to packed u64 records (src << 32 | dst), e.g. the all-to-all result."""
        st = BatchStats()
        _check(self.L.ppcsr_apply_batch_packed_device(self.h, d_packed, d_val, count, default_val, C.byref(st)))
        return st.as_dict()

    def apply_segments_device(self, d_packed: int, d_val: int | None, region_cap: int, d_counts: int, n_segments: int,
                              max_total: int = 0, default_val: int = 1) -> dict:
        """Records deposited by the peers: n_segments regions of region_cap records, region r holding d_counts[r]
        (device array).  The batch size comes back in the stats."""
        st = BatchStats()
        _check(self.L.ppcsr_apply_batch_segments_device(self.h, d_packed, d_val, region_cap, d_counts, n_segments,
                                                        max_total, default_val, C.byref(st)))
        return st.as_dict()

    def add_edge(self, s, d, v=1):
        _check(self.L.ppcsr_add_edge(self.h, s, d, v))

    def remove_edge(self, s, d) -> bool:
        f = C.c_int()
        _check(self.L.ppcsr_remove_edge(self.h, s, d, C.byref(f)))
        return bool(f.value)

    def add_nodes(self, k=1):
        _check(self.L.ppcsr_add_nodes(self.h, k))

    def reserve(self, max_slots=0, max_batch=0):
        _check(self.L.ppcsr_reserve(self.h, max_slots, max_batch))

    def set_stream(self, stream_ptr: int | None):
        """cudaStream_t handle; None / 0 = the shard's own stream (C-ABI convention)."""
        _check(self.L.ppcsr_set_stream(self.h, stream_ptr))

    def bind_torch_stream(self, stream=None):
        """Run the shard's work on a torch stream (default: the current one).  torch's default stream has the
        handle 0, which the C-ABI reads as "own stream": cudaStreamLegacy (0x1) names the same stream explicitly."""
        import torch

        stream = stream if stream is not None else torch.cuda.current_stream(self.device)
        self.set_stream(stream.cuda_stream or 1)

    def sync(self):
        _check(self.L.ppcsr_sync(self.h))

    def snapshot(self):
        _check(self.L.ppcsr_snapshot(self.h))

    def restore(self):
        _check(self.L.ppcsr_restore(self.h))

    # ---- reads ----
    @property
    def geometry(self) -> Geometry:
        g = Geometry()
        _check(self.L.ppcsr_geometry_of(self.h, C.byref(g)))
        return g

    @property
    def n(self) -> int:
        return self.geometry.n

    def edge_exists(self, s, d) -> bool:
        e = C.c_int()
        _check(self.L.ppcsr_edge_exists(self.h, s, d, C.byref(e), None))
        return bool(e.value)

    def edge_value(self, s, d):
        e, v = C.c_int(), C.c_uint32()
        _check(self.L.ppcsr_edge_exists(self.h, s, d, C.byref(e), C.byref(v)))
        return v.value if e.value else None

    def edges_exist(self, src, dst):
        src = _u32_array(src)
        dst = _u32_array(dst, src.shape[0])
        out = np.zeros(src.shape[0], dtype=np.uint8)
        _check(self.L.ppcsr_edges_exist(self.h, _np_ptr(src), _np_ptr(dst), src.shape[0], _np_ptr(out)))
        return out.astype(bool)

    def neighbours(self, v):
        cnt = C.c_uint64()
        _check(self.L.ppcsr_neighbours(self.h, v, None, 0, C.byref(cnt)))
        out = np.zeros(cnt.value, dtype=np.uint32)
        if cnt.value:
            _check(self.L.ppcsr_neighbours(self.h, v, _np_ptr(out), cnt.value, C.byref(cnt)))
        return out

    def read_neighbourhood(self, v) -> int:
        c = C.c_uint64()
        _check(self.L.ppcsr_read_neighbourhood(self.h, v, C.byref(c)))
        return c.value

    def num_neighbors(self):
        out = np.zeros(self.n, dtype=np.uint32)
        _check(self.L.ppcsr_num_neighbors(self.h, _np_ptr(out)))
        return out

    def node_ranges(self):
        n = self.n
        b, e = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
        _check(self.L.ppcsr_node_ranges(self.h, _np_ptr(b), _np_ptr(e)))
        return b, e

    def export(self, with_values=False):
        n = self.n
        E = C.c_uint64()
        rowptr = np.zeros(n + 1, dtype=np.uint64)
        _check(self.L.ppcsr_export_csr(self.h, _np_ptr(rowptr), None, None, C.byref(E)))
        col = np.zeros(E.value, dtype=np.uint32)
        val = np.zeros(E.value, dtype=np.uint32) if with_values else None
        _check(self.L.ppcsr_export_csr(self.h, None, _np_ptr(col), _np_ptr(val), C.byref(E)))
        return (rowptr, col, val) if with_values else (rowptr, col)

    def pagerank_step(self, values, dtype=np.float64, out_len=None):
        values = np.ascontiguousarray(values, dtype=dtype)
        out_len = self.n if out_len is None else out_len
        out = np.zeros(out_len, dtype=dtype)
        fn = self.L.ppcsr_pagerank_step_f64 if dtype == np.float64 else self.L.ppcsr_pagerank_step_f32
        _check(fn(self.h, _np_ptr(values), _np_ptr(out), out_len))
        return out

    def set_whole_array_policy(self, mode: int):
        """-1: always a window list; 0: cost model (default); 1: always one root window."""
        _check(self.L.ppcsr_set_whole_array_policy(self.h, int(mode)))

    def pagerank(self, iterations=20, damping=0.85):
        """Iterated PageRank with damping, all steps on the device (push semantics of reference pagerank.h:16-29)."""
        out = np.zeros(self.n, dtype=np.float64)
        _check(self.L.ppcsr_pagerank(self.h, iterations, float(damping), _np_ptr(out)))
        return out

    def bfs(self, start):
        out = np.zeros(self.n, dtype=np.uint32)
        _check(self.L.ppcsr_bfs(self.h, start, _np_ptr(out)))
        return out

    def check(self, check_lower=True) -> InvariantReport:
        r = InvariantReport()
        _check(self.L.ppcsr_check_invariants(self.h, 1 if check_lower else 0, C.byref(r)))
        return r

    def checksum(self, vertex_offset: int = 0) -> dict:
        """Order-independent checksum of the logical graph (edges, edge_hash, nn_hash), see ppcsr_checksum."""
        out = (C.c_uint64 * 3)()
        _check(self.L.ppcsr_checksum(self.h, vertex_offset, out))
        return {"edges": int(out[0]), "edge_hash": int(out[1]), "nn_hash": int(out[2])}

    def debug_dump(self):
        g = self.geometry
        dest = np.zeros(g.N, dtype=np.uint32)
        val = np.zeros(g.N, dtype=np.uint32)
        cnt = np.zeros(g.N // g.logN, dtype=np.uint32)
        _check(self.L.ppcsr_debug_dump(self.h, _np_ptr(dest), _np_ptr(val), _np_ptr(cnt)))
        return dest, val, cnt


def debug_sort_pairs(keys, payload=None, lo_bits=32, hi_bits=32, device=0):
    """ppcsr_debug_sort_pairs on copies; payload None sorts the keys alone (and returns None for it)."""
    L = load_library()
    keys = np.ascontiguousarray(keys, dtype=np.uint64).copy()
    if payload is not None:
        payload = np.ascontiguousarray(payload, dtype=np.uint32).copy()
    _check(L.ppcsr_debug_sort_pairs(device, _np_ptr(keys), _np_ptr(payload), keys.shape[0], lo_bits, hi_bits))
    return keys, payload


def debug_exclusive_scan(values, device=0):
    L = load_library()
    values = np.ascontiguousarray(values, dtype=np.uint32)
    out = np.zeros(values.shape[0] + 1, dtype=np.uint32)
    _check(L.ppcsr_debug_exclusive_scan(device, _np_ptr(values), _np_ptr(out), values.shape[0]))
    return out


def parse_edge_list(text: bytes, default_val: int = 1, device: int = 0):
    """The reference's text edge-list reader (src/main.cpp:29-62) on the GPU (ppcsr_parse_edge_list).  Returns host
    arrays (src, dst, val), the number of lines that parsed and the largest vertex id."""
    L = load_library()
    ds, dd, dv = C.c_void_p(), C.c_void_p(), C.c_void_p()
    cnt, ok, mx = C.c_uint64(), C.c_uint64(), C.c_uint32()
    buf = np.frombuffer(text, dtype=np.uint8)
    _check(L.ppcsr_parse_edge_list(device, _np_ptr(buf) if buf.size else None, buf.size, default_val, C.byref(ds),
                                   C.byref(dd), C.byref(dv), C.byref(cnt), C.byref(ok), C.byref(mx)))
    n = cnt.value
    out = [np.zeros(n, dtype=np.uint32) for _ in range(3)]
    for a, d in zip(out, (ds, dd, dv)):
        if n:
            _check(L.ppcsr_copy_to_host(device, _np_ptr(a), d, n * 4))
        _check(L.ppcsr_free_device(device, d))
    return out[0], out[1], out[2], ok.value, mx.value


class Group:
    """Several shards on several GPUs driven by one process (ppcsr_group_*): the data plane of reference PPPCSR."""

    def __init__(self, n: int, starts, devices, region_cap: int, with_values: bool = False):
        self.L = load_library()
        starts = np.ascontiguousarray(starts, dtype=np.uint64)
        assert starts[0] == 0 and starts[-1] == n and len(starts) == len(devices) + 1
        self.starts = starts
        self.shards = [Shard(int(starts[r + 1] - starts[r]), device=devices[r]) for r in range(len(devices))]
        arr = (C.c_void_p * len(devices))(*[s.h for s in self.shards])
        g = C.c_void_p()
        _check(self.L.ppcsr_group_create(arr, len(devices), _np_ptr(starts), region_cap, 1 if with_values else 0,
                                         C.byref(g)))
        self.g = g

    def apply(self, src, dst, val=None, default_val: int = 1):
        src = _u32_array(src)
        dst = _u32_array(dst, src.shape[0])
        val = _u32_array(val, src.shape[0]) if val is not None else None
        st = (BatchStats * len(self.shards))()
        _check(self.L.ppcsr_group_apply(self.g, _np_ptr(src), _np_ptr(dst), _np_ptr(val), src.shape[0], default_val, st))
        return [x.as_dict() for x in st]

    def owner(self, v: int) -> int:
        return int(self.L.ppcsr_group_owner(self.g, v))

    def close(self):
        if getattr(self, "g", None):
            self.L.ppcsr_group_destroy(self.g)
            self.g = None
            for s in self.shards:
                s.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
