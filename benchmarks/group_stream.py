#!/usr/bin/env python
"""A stream of batches into a group: the Group.apply loop against the pipelined Group.submit / Group.wait.

Builds the C4 core (synth.rmat(scale, 0, 16 << scale, 42), scale 20 by default) and a stream of --batches batches of
--batch skewed R-MAT updates (synth.rmat with seed 99, the edge ids after the core's) in page-locked host buffers, and
runs it through groups of 1 and of 8 shards on GPU 0 (8 with equal vertex counts and with edge-balanced boundaries
from the core's out-degrees), and, when more than one GPU is present, through one shard per GPU.  For every group:

    loop     for b in batches: Group.apply(b)
    stream   submit(b0); for i: { submit(b[i+1]); wait(b[i]); }

each from the same starting state (every shard restores its snapshot of the core before a run), alternating the two
modes --reps times after one untimed run of each.  Reports the wall time of a run (host clock, ends after the last
wait, which synchronises every shard) per batch as the median over the repetitions, and updates/s.  A separate
torch.profiler run of the stream on the 8-shard equal group reports, for every batch i+1, the share of the device time
of its copies and routing kernels that falls inside the span of batch i's apply (from its first to its last kernel).

Checks in the same run that both modes give the summed checksum of a single shard fed the same batches; a mismatch
exits non-zero.  Prints one JSON line with the card's name and power limit read in the same call.

    python benchmarks/group_stream.py --scale 20 --batches 10 --batch 10000000
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SKEW_SEED = 99


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
        v = int(np.searchsorted(csum * k, total * p, side="left")) + 1
        starts.append(min(max(v, starts[-1] + 1), n - (k - p)))
    return np.array(starts + [n], np.uint64)


def group_checksum(g):
    out = [0, 0, 0]
    for r, sh in enumerate(g.shards):
        c = sh.checksum(int(g.starts[r]))
        out = [(o + x) % (1 << 64) for o, x in zip(out, (c["edges"], c["edge_hash"], c["nn_hash"]))]
    return out


def pinned(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, np.uint32)).pin_memory().numpy()


def run_loop(g, batches):
    for s, d in batches:
        g.apply(s, d)


def run_stream(g, batches, mark=None):
    """mark(tag) returns a context manager around every submit and wait (the profiler run labels them)."""
    from contextlib import nullcontext

    mark = mark or (lambda tag: nullcontext())
    pending = []
    for i, (s, d) in enumerate(batches):
        with mark(f"submit {i}"):
            pending.append((i, g.submit(s, d)))
        if len(pending) == 2:
            i0, t = pending.pop(0)
            with mark(f"wait {i0}"):
                g.wait(t)
    for i0, t in pending:
        with mark(f"wait {i0}"):
            g.wait(t)


def timed(g, fn, batches):
    for sh in g.shards:
        sh.restore()
        sh.sync()
    t0 = time.perf_counter()
    fn(g, batches)
    wall = time.perf_counter() - t0
    return wall, group_checksum(g)


def union_length(iv):
    total, end = 0.0, -1e300
    for a, b in sorted(iv):
        if b > end:
            total += b - max(a, end)
            end = b
    return total


def overlap_share(g, batches):
    """Profiler run of the stream: per batch i+1, the share of its copy + routing device time inside batch i's apply
    span.  GPU events are attributed to a batch by the host range (submit i / wait i) their launch call falls in."""
    import torch
    from torch.profiler import ProfilerActivity, profile, record_function

    for sh in g.shards:
        sh.restore()
        sh.sync()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        run_stream(g, batches, mark=record_function)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    ranges = [(e["name"], e["ts"], e["ts"] + e["dur"]) for e in events
              if e.get("cat") == "user_annotation" and e.get("name", "").split(" ")[0] in ("submit", "wait")]
    launch = {e["args"]["correlation"]: e["ts"] for e in events
              if e.get("cat") == "cuda_runtime" and "correlation" in e.get("args", {})}
    routing = {i: [] for i in range(len(batches))}
    apply_ = {i: [] for i in range(len(batches))}
    for e in events:
        if e.get("cat") not in ("kernel", "gpu_memcpy", "gpu_memset"):
            continue
        ts = launch.get(e.get("args", {}).get("correlation"))
        if ts is None:
            continue
        for name, a, b in ranges:
            if a <= ts <= b:
                kind, i = name.split(" ")
                (routing if kind == "submit" else apply_)[int(i)].append((e["ts"], e["ts"] + e["dur"]))
                break
    shares = []
    for i in range(len(batches) - 1):
        r, ap = routing[i + 1], apply_[i]
        if not r or not ap:
            continue
        lo, hi = min(a for a, _ in ap), max(b for _, b in ap)
        busy = union_length(r)
        inside = union_length([(max(a, lo), min(b, hi)) for a, b in r if min(b, hi) > max(a, lo)])
        shares.append(round(inside / busy, 3) if busy else 0.0)
    return shares


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--scale", type=int, default=20, choices=(16, 18, 20, 22))
    ap.add_argument("--batches", type=int, default=10)
    ap.add_argument("--batch", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args(argv)
    pp = importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    L = pp.load_library()
    ndev = L.ppcsr_device_count()
    if ndev < 1:
        print("no CUDA device: nothing to measure", file=sys.stderr)
        return 1
    n = 1 << a.scale
    total = 16 << a.scale
    cs, cd = synth.rmat(a.scale, 0, total, 42)
    batches = []
    for i in range(a.batches):
        s, d = synth.rmat(a.scale, total + i * a.batch, total + (i + 1) * a.batch, SKEW_SEED)
        batches.append((pinned(s), pinned(d)))
    single = pp.Shard(n)
    single.apply(cs, cd)
    for s, d in batches:
        single.apply(s, d)
    c = single.checksum(0)
    want = [c["edges"], c["edge_hash"], c["nn_hash"]]
    single.close()
    core_deg = np.bincount(cs[cs < n].astype(np.int64), minlength=n)  # R-MAT draws duplicates: an estimate, as in -balanced
    configs = [("1 shard", 1, [0]), ("8 equal", 8, [0] * 8), ("8 edge-balanced", 8, [0] * 8)]
    if ndev > 1:
        k = min(8, ndev)
        configs.append((f"{k} GPUs, one shard each", k, list(range(k))))
    result = {"bench": "group_stream", "scale": a.scale, "n": n, "core_edges": int(total), "batches": a.batches,
              "batch": a.batch, "reps": a.reps, "devices_present": ndev, **card()}
    ok = True
    rows = []
    for tag, k, devices in configs:
        starts = balanced_starts(core_deg, k) if "balanced" in tag else np.linspace(0, n, k + 1).astype(np.uint64)
        cap = max(cs.size, a.batch) // k + 1
        g = pp.Group(n, starts, devices, region_cap=cap)
        g.apply(cs, cd)
        for sh in g.shards:
            sh.snapshot()
        walls = {"loop": [], "stream": []}
        for rep in range(a.reps + 1):  # rep 0 warms both modes up (allocations, first submits)
            for mode, fn in (("loop", run_loop), ("stream", run_stream)):
                wall, ck = timed(g, fn, batches)
                if ck != want:
                    print(json.dumps({"error": "checksum mismatch", "config": tag, "mode": mode, "rep": rep,
                                      "got": ck, "want": want}))
                    ok = False
                if rep:
                    walls[mode].append(wall)
        row = {"config": tag, "shards": k, "devices": sorted(set(devices)), "boundaries": [int(x) for x in starts]}
        for mode in ("loop", "stream"):
            med = statistics.median(walls[mode])
            row[mode] = {"ms_per_batch": round(med * 1e3 / a.batches, 3),
                         "ms_per_batch_min": round(min(walls[mode]) * 1e3 / a.batches, 3),
                         "ms_per_batch_max": round(max(walls[mode]) * 1e3 / a.batches, 3),
                         "updates_per_s": round(a.batches * a.batch / med, 1)}
        row["stream_over_loop"] = round(row["stream"]["ms_per_batch"] / row["loop"]["ms_per_batch"], 3)
        if tag == "8 equal":
            row["routing_inside_previous_apply"] = overlap_share(g, batches[:4])
        rows.append(row)
        g.close()
    result["groups"] = rows
    result["checksums_match_single_shard"] = bool(ok)
    print(json.dumps(result))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
