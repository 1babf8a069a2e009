#!/usr/bin/env python
"""Vertex isolation (Shard.isolate_vertices / Group.isolate_vertices) against what a caller does without it.

Graphs: the C4 core (synth.rmat(scale, 0, 16 << scale, 42)) at scale 20, on one shard and on a group of 8 equal
vertex ranges (all on GPU 0, or one per GPU with --devices), and at scale 24 on one shard.  Id sets: one random
vertex, 1 K random vertices, the 1 K largest hubs by out-degree, 1 % of the vertices at random.

Each graph is built once and snapshotted; every call starts from ppcsr_restore of that snapshot, so each rep
isolates the same set in the same graph (the restore is not timed).  After --warmup untimed calls, --reps calls are
timed with the host clock (the call ends in a device synchronise) and their median is reported with the device times
of the median call's stats:
    filter_ms     ms_locate: the filter pass over the packed array (group: the slowest shard)
    bitmap_ms     ms_sort:   the copy of the ids and the bitmap build
    select_ms     ms_select: window selection
    rebalance_ms  ms_rebalance
and the filter pass's algorithmic bytes -- 4 B of dest per slot, 4 B of leaf_cnt and 4 B of del_cnt per leaf,
4 B per removed edge -- over filter_ms, against the HBM peak bench.py's roofline uses (MEASURED_PEAKS.json hbm_gbs,
else 6650 GB/s).  In a group the shards of one GPU run concurrently on their own streams: bytes are summed over the
shards and divided by the slowest shard's filter time.

Beside it, the route a caller has without the call, end to end on the host clock: ppcsr_export_csr of the whole graph
to the host, a numpy filter for the incident edges, and one remove batch through apply.  The checksums of both
results must be equal.  Prints one JSON line with the card's name and power limit read in the same run; exits
non-zero if a result differs.

    python benchmarks/isolate_vertices.py                 # scale 20 (shard + group of 8) and scale 24 (shard)
    python benchmarks/isolate_vertices.py --scales 20
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MASK64 = (1 << 64) - 1


def card() -> dict:
    """Name and power limit of GPU 0 (nvidia-smi query), read where the numbers are measured."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the numbers are still printed, marked as coming from an unnamed card
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def hbm_peak_gbs() -> float:
    """The peak bench.py's roofline uses (bench.measured_peak)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"])
        except Exception:
            pass
    return 6650.0


class Target:
    """One shard, or a group, behind the calls the benchmark makes."""

    def __init__(self, pp, n, parts, devices, core):
        self.n = n
        self.parts = parts
        if parts == 1:
            self.shards = [pp.Shard(n, device=devices[0])]
            self.starts = np.array([0, n], np.uint64)
            self.group = None
        else:
            self.starts = (np.arange(parts + 1, dtype=np.uint64) * (n // parts)).astype(np.uint64)
            self.starts[-1] = n
            cap = max(int(c[0].shape[0]) for c in core) // parts + 1
            self.group = pp.Group(n, self.starts, devices, region_cap=cap)
            self.shards = self.group.shards
        for cs, cd in core:
            self.apply(cs, cd, 1)
        for sh in self.shards:
            sh.snapshot()

    def apply(self, s, d, v):
        return (self.group or self.shards[0]).apply(s, d, default_val=v)

    def isolate(self, ids):
        st = (self.group or self.shards[0]).isolate_vertices(ids)
        return st if isinstance(st, list) else [st]

    def restore(self):
        for sh in self.shards:
            sh.restore()

    def export(self):
        rps, cols, off = [np.zeros(1, np.uint64)], [], 0
        for sh in self.shards:
            rp, c = sh.export()
            rps.append(rp[1:] + np.uint64(off))
            off += int(rp[-1])
            cols.append(c)
        return np.concatenate(rps), np.concatenate(cols)

    def checksum(self):
        out = [0, 0, 0]
        for r, sh in enumerate(self.shards):
            c = sh.checksum(int(self.starts[r]))
            out = [(out[0] + c["edges"]) & MASK64, (out[1] + c["edge_hash"]) & MASK64,
                   (out[2] + c["nn_hash"]) & MASK64]
        return tuple(out)

    def close(self):
        (self.group or self.shards[0]).close()


def incident(rowptr, col, ids):
    """The live edges (u, w) with u in ids or w in ids (w < n): the caller's numpy filter."""
    n = rowptr.size - 1
    mark = np.zeros(n, bool)
    mark[ids] = True
    src = np.repeat(np.arange(n, dtype=np.uint32), np.diff(rowptr).astype(np.int64))
    hit = mark[src] | ((col < n) & mark[np.minimum(col, n - 1).astype(np.int64)])
    return src[hit], col[hit]


def filter_bytes(st) -> int:
    N = int(st["slots_before"])
    leaves = N // (1 << ((2 * (N.bit_length() - 1) + 1).bit_length() - 1))
    return 4 * N + 8 * leaves + 4 * int(st["n_deleted"])


def measure(t: Target, name, ids, reps, warmup, peak):
    runs = []
    for i in range(warmup + reps):
        t.restore()
        t0 = time.perf_counter()
        sts = t.isolate(ids)
        ms = (time.perf_counter() - t0) * 1e3
        if i >= warmup:
            runs.append((ms, sts))
    runs.sort(key=lambda r: r[0])
    ms, sts = runs[len(runs) // 2]
    got = t.checksum()
    filt = max(st["ms_locate"] for st in sts)
    nbytes = sum(filter_bytes(st) for st in sts)
    out = {"ids": name, "count": int(ids.size), "removed": sum(int(st["n_deleted"]) for st in sts),
           "host_ms": round(ms, 3), "host_ms_all": [round(r[0], 3) for r in sorted(runs, key=lambda r: r[0])],
           "filter_ms": round(filt, 4), "bitmap_ms": round(max(st["ms_sort"] for st in sts), 4),
           "select_ms": round(max(st["ms_select"] for st in sts), 4),
           "rebalance_ms": round(max(st["ms_rebalance"] for st in sts), 4),
           "whole_array": [int(st["whole_array"]) for st in sts], "filter_bytes": nbytes,
           "filter_gbs": round(nbytes / (filt * 1e6), 1) if filt > 0 else None}
    out["filter_share_of_peak"] = round(out["filter_gbs"] / peak, 3) if out["filter_gbs"] else None
    # the caller's route without the call, from the same graph
    t.restore()
    t0 = time.perf_counter()
    rowptr, col = t.export()
    t1 = time.perf_counter()
    s, d = incident(rowptr, col, ids)
    t2 = time.perf_counter()
    t.apply(s, d, 0)
    t3 = time.perf_counter()
    out["export_filter_apply"] = {"ms": round((t3 - t0) * 1e3, 1), "export_ms": round((t1 - t0) * 1e3, 1),
                                  "filter_ms": round((t2 - t1) * 1e3, 1), "apply_ms": round((t3 - t2) * 1e3, 1),
                                  "exported_bytes": int(rowptr.nbytes + col.nbytes)}
    out["speedup"] = round((t3 - t0) * 1e3 / ms, 1)
    out["equal"] = bool(t.checksum() == got and s.size == out["removed"])
    return out


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scales", type=int, nargs="+", default=[20, 24], choices=(20, 22, 24))
    ap.add_argument("--parts", type=int, default=8, help="shards of the group (at the smallest scale only)")
    ap.add_argument("--devices", action="store_true", help="one part per GPU (parts on GPU p %% device count)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args(argv)
    import torch

    pp = importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    ndev = pp.load_library().ppcsr_device_count()
    if ndev < 1:
        print("no CUDA device: nothing to measure", file=sys.stderr)
        return 1
    peak = hbm_peak_gbs()
    result = {"bench": "isolate_vertices", **card(), "hbm_peak_gbs": peak, "configs": []}
    ok = True
    for scale in a.scales:
        n = 1 << scale
        E = 16 << scale
        chunk = 1 << 26  # the core is generated and applied in pieces: the host keeps one piece at a time
        pieces = [(lo, min(E, lo + chunk)) for lo in range(0, E, chunk)]

        def core():  # generated on GPU 0 (the host takes minutes at scale 24), handed over as host arrays
            for lo, hi in pieces:
                cs, cd = synth.rmat(scale, lo, hi, 42, device="cuda:0")
                yield (cs.to(torch.int32).cpu().numpy().view(np.uint32),
                       cd.to(torch.int32).cpu().numpy().view(np.uint32))

        configs = [1] + ([a.parts] if scale == min(a.scales) and a.parts > 1 else [])
        for parts in configs:
            devices = [p % ndev for p in range(parts)] if a.devices else [0] * parts
            t = Target(pp, n, parts, devices, list(core()) if parts > 1 else core())
            rowptr, _ = t.export()
            deg = np.diff(rowptr).astype(np.int64)
            rng = np.random.default_rng(scale)
            sets = [("1 random", rng.integers(0, n, 1)), ("1K random", rng.integers(0, n, 1024)),
                    ("1K hubs", np.argsort(deg, kind="stable")[-1024:]), ("1% random", rng.integers(0, n, n // 100))]
            del rowptr, deg
            cfg = {"scale": scale, "n": n, "parts": parts, "devices": sorted(set(devices)),
                   "slots": sum(int(sh.geometry.N) for sh in t.shards), "runs": []}
            for name, ids in sets:
                r = measure(t, name, ids.astype(np.uint32), a.reps, a.warmup, peak)
                ok &= r["equal"]
                cfg["runs"].append(r)
            result["configs"].append(cfg)
            t.close()
    result["equal"] = ok
    print(json.dumps(result))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
