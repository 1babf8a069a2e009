"""TEST INFRASTRUCTURE: ctypes front end for oracle/_build/libpcsr_oracle.so (the C restatement),
a reader for oracle/ref_driver dumps and a runner for oracle/_ref/ref_driver (the compiled,
unmodified reference).  Imported only by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never by the product package."""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "_build", "libpcsr_oracle.so")
REF_DRIVER = os.path.join(ORACLE_DIR, "_ref", "ref_driver")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "ppcsr_ref")
DUMP_MAGIC = 0x50504353524F5243


def build_oracle(with_ref: bool | None = None) -> None:
    """Compile the C restatement (always) and oracle/_ref from /root/reference (when it is there)."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "oracle"], check=True)
    if with_ref is None:
        with_ref = os.path.isdir("/root/reference/src")
    if with_ref:
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "ref"], check=True)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            build_oracle(with_ref=False)
        L = C.CDLL(ORACLE_SO)
        u32, u64, vp = C.c_uint32, C.c_uint64, C.c_void_p
        L.opcsr_create.restype = vp
        L.opcsr_create.argtypes = [u32, u32]
        L.opcsr_destroy.argtypes = [vp]
        L.opcsr_add_edge.argtypes = [vp, u32, u32, u32]
        L.opcsr_remove_edge.argtypes = [vp, u32, u32]
        L.opcsr_add_node.argtypes = [vp]
        L.opcsr_edge_exists.argtypes = [vp, u32, u32]
        L.opcsr_edge_exists.restype = C.c_int
        for name in ("opcsr_n", "opcsr_slots", "opcsr_not_found", "opcsr_resizes"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = u64
        for name in ("opcsr_leaf", "opcsr_height", "opcsr_check"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = C.c_int
        L.opcsr_num_neighbors.argtypes = [vp, u32]
        L.opcsr_num_neighbors.restype = u32
        L.opcsr_neighbourhood.argtypes = [vp, u32, vp, u64]
        L.opcsr_neighbourhood.restype = u64
        L.opcsr_export.argtypes = [vp, vp, vp, vp]
        L.opcsr_export.restype = u64
        L.opcsr_export_values.argtypes = [vp, vp]
        L.opcsr_export_values.restype = u64
        L.opcsr_apply.argtypes = [vp, vp, vp, vp, u64]
        L.opcsr_pagerank_f64.argtypes = [vp, vp, vp]
        L.opcsr_pagerank_f32.argtypes = [vp, vp, vp]
        L.opcsr_bfs.argtypes = [vp, u32, vp]
        L.opppcsr_table.argtypes = [u32, u32, vp, vp]
        L.opppcsr_owner.argtypes = [vp, u32, u64]
        L.opppcsr_owner.restype = u32
        L.opool_domain_table.argtypes = [C.c_int, C.c_int, vp, vp, vp]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class OraclePCSR:
    """Sequential reference semantics (reference src/pcsr/PCSR.h:64-124) via the C restatement."""

    def __init__(self, n: int, init_n: int | None = None):
        self.L = lib()
        self.h = self.L.opcsr_create(n if init_n is None else init_n, n)

    def __del__(self):
        try:
            self.L.opcsr_destroy(self.h)
        except Exception:
            pass

    def add_edge(self, s, d, v=1):
        self.L.opcsr_add_edge(self.h, s, d, v)

    def remove_edge(self, s, d):
        self.L.opcsr_remove_edge(self.h, s, d)

    def add_node(self):
        self.L.opcsr_add_node(self.h)

    def edge_exists(self, s, d) -> bool:
        return bool(self.L.opcsr_edge_exists(self.h, s, d))

    def apply(self, src, dst, val=None):
        src = np.ascontiguousarray(src, dtype=np.uint32)
        dst = np.ascontiguousarray(dst, dtype=np.uint32)
        if val is not None:
            val = np.ascontiguousarray(np.broadcast_to(np.asarray(val, dtype=np.uint32), src.shape))
        self.L.opcsr_apply(self.h, _ptr(src), _ptr(dst), _ptr(val), src.shape[0])

    @property
    def n(self):
        return self.L.opcsr_n(self.h)

    @property
    def geometry(self):
        return (self.L.opcsr_slots(self.h), self.L.opcsr_leaf(self.h), self.L.opcsr_height(self.h))

    @property
    def not_found(self):
        return self.L.opcsr_not_found(self.h)

    def check(self) -> int:
        return self.L.opcsr_check(self.h)

    def neighbourhood(self, v):
        k = self.L.opcsr_neighbourhood(self.h, v, None, 0)
        out = np.empty(k, dtype=np.uint32)
        self.L.opcsr_neighbourhood(self.h, v, _ptr(out), k)
        return out

    def export(self):
        n = self.n
        rowptr = np.zeros(n + 1, dtype=np.uint64)
        nn = np.zeros(n, dtype=np.uint32)
        E = self.L.opcsr_export(self.h, None, None, None)
        col = np.zeros(E, dtype=np.uint32)
        self.L.opcsr_export(self.h, _ptr(rowptr), _ptr(col), _ptr(nn))
        return rowptr, col, nn

    def export_values(self):
        """The stored values, aligned with export()'s col."""
        val = np.zeros(self.L.opcsr_export_values(self.h, None), dtype=np.uint32)
        self.L.opcsr_export_values(self.h, _ptr(val))
        return val

    def pagerank(self, values, dtype=np.float64):
        values = np.ascontiguousarray(values, dtype=dtype)
        out = np.zeros(self.n, dtype=dtype)
        with np.errstate(all="ignore"):
            (self.L.opcsr_pagerank_f64 if dtype == np.float64 else self.L.opcsr_pagerank_f32)(
                self.h, _ptr(values), _ptr(out))
        return out

    def bfs(self, start):
        out = np.zeros(self.n, dtype=np.uint32)
        self.L.opcsr_bfs(self.h, start, _ptr(out))
        return out


def partition_table(init_n: int, parts: int):
    starts = np.zeros(parts, dtype=np.uint64)
    sizes = np.zeros(parts, dtype=np.uint64)
    lib().opppcsr_table(init_n, parts, _ptr(starts), _ptr(sizes))
    return starts, sizes


def partition_owner(starts, vertex: int) -> int:
    starts = np.ascontiguousarray(starts, dtype=np.uint64)
    return lib().opppcsr_owner(_ptr(starts), starts.shape[0], vertex)


def domain_table(threads: int, domains: int):
    t2d = np.zeros(threads, dtype=np.int32)
    first = np.zeros(domains, dtype=np.int32)
    num = np.zeros(domains, dtype=np.int32)
    lib().opool_domain_table(threads, domains, _ptr(t2d), _ptr(first), _ptr(num))
    return t2d, first, num


# ------------------------------------------------------------------------------------------------
# compiled reference (oracle/_ref)
# ------------------------------------------------------------------------------------------------
def have_ref() -> bool:
    return os.path.exists(REF_DRIVER)


def read_dump(path: str) -> dict:
    raw = np.fromfile(path, dtype=np.uint8)
    hdr = raw[:48].view("<u8")
    assert int(hdr[0]) == DUMP_MAGIC, "bad dump magic"
    n, E = int(hdr[1]), int(hdr[2])
    off = 48
    rowptr = raw[off:off + 8 * (n + 1)].view("<u8").copy()
    off += 8 * (n + 1)
    col = raw[off:off + 4 * E].view("<u4").copy()
    off += 4 * E
    nn = raw[off:off + 4 * n].view("<u4").copy()
    off += 4 * n
    has_pr = int(raw[off:off + 8].view("<u8")[0])
    off += 8
    pr = raw[off:off + 8 * n].view("<f8").copy() if has_pr else None
    return {"n": n, "E": E, "N": int(hdr[3]), "logN": int(hdr[4]), "H": int(hdr[5]),
            "rowptr": rowptr, "col": col, "num_neighbors": nn, "pagerank": pr}


def write_triples(path, src, dst, val):
    src = np.asarray(src, dtype=np.uint32)
    out = np.empty((src.shape[0], 3), dtype="<u4")
    out[:, 0] = src
    out[:, 1] = np.asarray(dst, dtype=np.uint32)
    out[:, 2] = np.broadcast_to(np.asarray(val, dtype=np.uint32), src.shape)
    out.tofile(path)


def run_ref(n: int, core, updates, *, mode="ppcsr", api="direct", threads=1, ppd=1, pagerank=False,
            add_nodes=0, size=None, dump=True, workdir=None) -> dict:
    """Run the compiled reference on (core, updates), each a (src, dst, val) triple of arrays.
    Returns the dump (logical graph, geometry) plus the reference's own start()->stop() timings."""
    assert have_ref(), "oracle/_ref/ref_driver not built (needs /root/reference)"
    with tempfile.TemporaryDirectory(dir=workdir) as td:
        cpath, upath = os.path.join(td, "core.bin"), os.path.join(td, "upd.bin")
        write_triples(cpath, *core)
        write_triples(upath, *updates)
        dpath, tpath = os.path.join(td, "dump.bin"), os.path.join(td, "timing.json")
        cmd = [REF_DRIVER, "--mode", mode, "--api", api, "--threads", str(threads), "--ppd", str(ppd),
               "--n", str(n), "--core", cpath, "--updates", upath, "--timing", tpath]
        if dump:
            cmd += ["--dump", dpath]
        if pagerank:
            cmd += ["--pagerank"]
        if add_nodes:
            cmd += ["--add-nodes", str(add_nodes)]
        if size is not None:
            cmd += ["--size", str(size)]
        subprocess.run(cmd, stdout=subprocess.DEVNULL, check=True)
        out = read_dump(dpath) if dump else {}
        out["timing"] = json.load(open(tpath))
        return out
