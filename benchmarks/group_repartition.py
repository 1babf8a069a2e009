#!/usr/bin/env python
"""Repartitioning a live group: equal vertex counts -> edge-balanced boundaries, on the devices.

Builds the C4 core (synth.rmat(scale, 0, 16 << scale, 42); scale 20 by default, 24 as an option) in a group of --parts
vertex-range shards with equal vertex counts (the reference's distribution), all on GPU 0 or, with --devices, one part
per GPU, and recuts it at boundaries that balance the current out-degrees (the rule of the CLI's -repartition).
Reports:

    edges per shard before and after (max / mean)
    the wall time of Group.repartition (host clock, ends after a device synchronisation; every kernel was launched
        once before, on a small group)
    per rebuilt shard: the layout kernel's CUDA-event time and its algorithmic bandwidth -- reads 8 B per edge
        (col + val) + 8 B per vertex (rowptr), writes 8 B per slot (dest + val) + 4 B per vertex (beg) -- and its share
        of the HBM copy peak measured for this project (profiles/README.md)
    the max / mean per-shard ms_total of two successive batches of --batch skewed (R-MAT) inserts applied to a group
        with the equal split and to a repartitioned one (the same batches, the same core), and the wall time of each
        Group.apply; every shard first reserves slots and sort buffers for its worst case (ppcsr_reserve)

and checks in the same run that the summed checksums of the two groups agree (after the repartition and after the
batch).  Prints one JSON line with the card's name and power limit read in the same call.  Exits non-zero if a check
fails.  With every shard on one GPU the shards share that GPU's memory bandwidth: the max / mean balance of the batch
shows the per-shard work, not the multi-GPU speed-up, which was not measured.

    python benchmarks/group_repartition.py --scale 20 --parts 8
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

HBM_COPY_PEAK_GBS = 6550.0  # measured device-to-device copy peak of a B200 (profiles/README.md, first line)
SKEW_SEED = 7


def card() -> dict:
    """Name and power limit of GPU 0 (nvidia-smi query), read where the numbers are measured."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the numbers are still printed, marked as coming from an unnamed card
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def balanced_starts(deg, k):
    """First vertex of every part such that the parts hold about the same number of edges (main.cpp's rule)."""
    n = deg.size
    total = int(deg.sum())
    csum = np.cumsum(deg, dtype=np.int64)
    starts = [0]
    for p in range(1, k):
        v = int(np.searchsorted(csum * k, total * p, side="left")) + 1  # first v with run(v) * k >= total * p
        starts.append(min(max(v, starts[-1] + 1), n - (k - p)))
    return np.array(starts + [n], np.uint64)


def group_checksum(g):
    out = [0, 0, 0]
    for r, sh in enumerate(g.shards):
        c = sh.checksum(int(g.starts[r]))
        out = [(o + x) % (1 << 64) for o, x in zip(out, (c["edges"], c["edge_hash"], c["nn_hash"]))]
    return out


def edges_per_shard(g):
    return [sh.checksum(0)["edges"] for sh in g.shards]


def balance(x):
    return {"max": int(max(x)), "mean": float(np.mean(x)), "max_over_mean": round(max(x) / float(np.mean(x)), 3)}


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scale", type=int, default=20, choices=(20, 22, 24))
    ap.add_argument("--parts", type=int, default=8)
    ap.add_argument("--devices", action="store_true", help="one part per GPU (parts on GPU p %% device count)")
    ap.add_argument("--batch", type=int, default=10_000_000, help="skewed inserts of the batch applied afterwards")
    a = ap.parse_args(argv)
    pp = importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    L = pp.load_library()
    ndev = L.ppcsr_device_count()
    if ndev < 1:
        print("no CUDA device: nothing to measure", file=sys.stderr)
        return 1
    # launch every kernel once (module loading) on a small group
    ws, wd = synth.rmat(12, 0, 16 << 12, 42)
    warm = pp.Group(1 << 12, np.linspace(0, 1 << 12, 5).astype(np.uint64), [0] * 4, region_cap=ws.size // 4 + 1)
    warm.apply(ws, wd)
    warm.repartition(np.array([0, 100, 1000, 2000, 1 << 12], np.uint64))
    warm.close()
    n = 1 << a.scale
    total = 16 << a.scale
    cs, cd = synth.rmat(a.scale, 0, total, 42)
    starts = np.linspace(0, n, a.parts + 1).astype(np.uint64)
    devices = [p % ndev for p in range(a.parts)] if a.devices else [0] * a.parts
    cap = max(cs.size, a.batch) // a.parts + 1
    groups = [pp.Group(n, starts, devices, region_cap=cap) for _ in range(2)]
    for g in groups:
        g.apply(cs, cd)
    equal, moved = groups
    result = {"bench": "group_repartition", "scale": a.scale, "n": n, "parts": a.parts,
              "devices": sorted(set(devices)), **card()}
    ok = True
    before = edges_per_shard(moved)
    ck0 = group_checksum(moved)
    deg = np.concatenate([np.diff(sh.export()[0]).astype(np.int64) for sh in moved.shards])
    new = balanced_starts(deg, a.parts)
    st = moved.repartition(new)
    after = edges_per_shard(moved)
    ok &= group_checksum(moved) == ck0
    for sh in moved.shards:
        ok &= not sh.check(False).violations(False)
    layout = []
    for r, sh in enumerate(moved.shards):
        ls = pp.BatchStats()
        pp._check(L.ppcsr_last_stats(sh.h, ls))
        if int(new[r]) == int(starts[r]) and int(new[r + 1]) == int(starts[r + 1]):
            continue  # not rebuilt
        ms = ls.ms_rebalance_kernel
        gbs = ls.rebalance_bytes / (ms * 1e-3) / 1e9
        layout.append({"shard": r, "edges": after[r], "slots": int(ls.slots_after), "kernel_ms": round(ms, 4),
                       "algorithmic_bytes": int(ls.rebalance_bytes), "gb_per_s": round(gbs, 1),
                       "of_hbm_copy_peak": round(gbs / HBM_COPY_PEAK_GBS, 3), "ms_total": round(ls.ms_total, 4)})
    result["boundaries_before"] = [int(x) for x in starts]
    result["boundaries_after"] = [int(x) for x in new]
    result["edges_per_shard_before"] = balance(before)
    result["edges_per_shard_after"] = balance(after)
    result["repartition"] = {k: (round(v, 3) if isinstance(v, float) else v) for k, v in st.items()}
    result["layout_per_shard"] = layout
    # the same skewed batches on both groups: per-shard device time and wall time of each; the first batch after the
    # recut also sizes the per-update scratch of shards that now receive more updates than before
    batches = [synth.rmat(a.scale, total + i * a.batch, total + (i + 1) * a.batch, SKEW_SEED) for i in range(2)]
    res_b = {}
    for tag, g in (("equal_split", equal), ("repartitioned", moved)):
        for sh in g.shards:  # the worst case of a batch: every update lands on this shard
            geo = sh.geometry
            slots = 1 << int(2 * (geo.items + 2 * a.batch) - 1).bit_length()
            sh.reserve(min(slots, 1 << 31), a.batch)
        runs = []
        for bs, bd in batches:
            t0 = time.perf_counter()
            sts = g.apply(bs, bd)
            wall = (time.perf_counter() - t0) * 1e3
            t = [x["ms_total"] for x in sts]
            runs.append({"wall_ms": round(wall, 3), "max_ms": round(max(t), 3), "mean_ms": round(float(np.mean(t)), 3),
                         "max_over_mean": round(max(t) / float(np.mean(t)), 3), "per_shard_ms": [round(x, 3) for x in t],
                         "per_shard_updates": [int(x["batch_size"]) for x in sts]})
        res_b[tag] = {"first": runs[0], "second": runs[1]}
    result["skewed_batches"] = {"updates": a.batch, **res_b}
    ok &= group_checksum(equal) == group_checksum(moved)
    result["checksums_equal"] = bool(ok)
    print(json.dumps(result))
    for g in groups:
        g.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
