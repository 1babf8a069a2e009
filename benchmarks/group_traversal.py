#!/usr/bin/env python
"""Traversals across the shards of a group against the single-shard traversals, on the same graph.

Builds the C4 core (synth.rmat(scale, 0, 16 << scale, 42); scale 20 by default, 22 and 24 as options) once in one
shard and once split over --parts vertex-range shards (equal vertex counts, the reference's distribution), all on
GPU 0 or, with --devices, one part per GPU.  Then times, after --warmup untimed calls and with each call ending in a
device synchronisation (every call copies its result to the host before it returns):

    Group.bfs / Shard.bfs     from the hub and from a seeded random vertex the hub reaches: ms, levels, and live
                              edges of the reached vertices scanned per second
    Group.pagerank(20) / Shard.pagerank(20)
                              ms of the call, and ms per iteration = the device time of all kernels of one
                              pagerank(20) call (torch.profiler, a run of its own) / 20

and checks in the same run that the group's results equal the single shard's (BFS exactly, PageRank to rtol 1e-9).
Prints one JSON line, with the card's name and power limit read in the same call.  Exits non-zero if a check fails.

    python benchmarks/group_traversal.py --scale 20 --parts 8
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    """Name and power limit of GPU 0 (nvidia-smi query), read where the numbers are measured."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the numbers are still printed, marked as coming from an unnamed card
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def timed(fn, reps: int, warmup: int):
    for _ in range(warmup):
        fn()
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def kernel_ms(fn) -> float:
    """Sum of the device time of the project's kernels fn launches (torch.profiler; copies excluded), in ms."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.self_device_time_total for e in prof.key_averages() if "k_" in e.key) / 1e3


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scale", type=int, default=20, choices=(20, 22, 24))
    ap.add_argument("--parts", type=int, default=8)
    ap.add_argument("--devices", action="store_true", help="one part per GPU (parts on GPU p %% device count)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args(argv)
    pp = importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    L = pp.load_library()
    ndev = L.ppcsr_device_count()
    if ndev < 1:
        print("no CUDA device: nothing to measure", file=sys.stderr)
        return 1
    n = 1 << a.scale
    cs, cd = synth.rmat(a.scale, 0, 16 << a.scale, 42)
    cs, cd = cs.astype(np.uint32), cd.astype(np.uint32)
    starts = (np.arange(a.parts + 1, dtype=np.uint64) * (n // a.parts)).astype(np.uint64)
    starts[-1] = n
    devices = [p % ndev for p in range(a.parts)] if a.devices else [0] * a.parts
    single = pp.Shard(n)
    single.apply(cs, cd, 1)
    group = pp.Group(n, starts, devices, region_cap=cs.size // a.parts + 1)
    group.apply(cs, cd)
    rowptr, _ = single.export()
    deg = np.diff(rowptr).astype(np.int64)
    hub = int(np.argmax(deg))

    result = {"bench": "group_traversal", "scale": a.scale, "n": n, "edges": int(rowptr[-1]), "parts": a.parts,
              "devices": sorted(set(devices)), **card()}
    ok = True
    d_hub = single.bfs(hub)
    reached = np.flatnonzero(d_hub != 0xFFFFFFFF)
    other = int(np.random.default_rng(1).choice(reached))
    for tag, s in (("hub", hub), ("random", other)):
        g_ms, g_d = timed(lambda: group.bfs(s), a.reps, a.warmup)
        s_ms, s_d = timed(lambda: single.bfs(s), a.reps, a.warmup)
        same = bool(np.array_equal(g_d, s_d))
        ok &= same
        hit = s_d != 0xFFFFFFFF
        scanned = int(deg[hit].sum())
        result[f"bfs_{tag}"] = {"start": s, "reached": int(hit.sum()), "levels": int(s_d[hit].max()) + 1,
                                "edges_scanned": scanned, "group_ms": round(g_ms, 3), "shard_ms": round(s_ms, 3),
                                "group_edges_per_s": scanned / (g_ms * 1e-3), "shard_edges_per_s": scanned / (s_ms * 1e-3),
                                "equal": same}
    it = 20
    g_ms, g_r = timed(lambda: group.pagerank(it), a.reps, a.warmup)
    s_ms, s_r = timed(lambda: single.pagerank(it), a.reps, a.warmup)
    g_k, s_k = kernel_ms(lambda: group.pagerank(it)) / it, kernel_ms(lambda: single.pagerank(it)) / it
    fin = np.isfinite(s_r)
    same = bool(np.array_equal(fin, np.isfinite(g_r)) and np.allclose(g_r[fin], s_r[fin], rtol=1e-9, atol=0))
    ok &= same
    result["pagerank"] = {"iterations": it, "group_ms": round(g_ms, 3), "shard_ms": round(s_ms, 3),
                          "group_kernel_ms_per_iteration": round(g_k, 4), "shard_kernel_ms_per_iteration": round(s_k, 4),
                          "group_over_shard": round(g_k / s_k, 3), "equal": same}
    result["equal"] = ok
    print(json.dumps(result))
    group.close()
    single.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
