#!/usr/bin/env python
"""Change capture (Shard.set_change_capture / last_changes): what it costs a batch.

Cases (bench.py's configs, one shard on GPU 0):
    C2     scale-20 core + 10 M uniform inserts (value 1: the insert-only locate)
    C3     scale-20 core + 10 M removes of core edges (the delete-only locate)
    mixed  scale-20 core with distinct values + 10 M updates of C5's op mix, every insert with its own value
           (payload sort, general locate)
    C4     scale-24 core + 100 M skewed inserts (--no-c4 skips it)

The core is built once per case and snapshotted; every timed batch starts from ppcsr_restore of it (not timed), with
the batch already in device memory (apply_device).  Capture off and on alternate, --warmup untimed pairs first, then
--reps pairs; the medians of ms_total and ms_locate (which with capture on includes the compaction pass) are
reported for both.  One more batch per mode runs under torch.profiler (a separate run, not in the medians) for the
kernel times of the locate kernel (k_locate vs k_locate_capture) and of the compaction scans (the kernels whose
functors are batch::InCap*).  The change lists are checked against the batch's stats.

Extra algorithmic bytes of capture, from the shapes (count updates, c changes of which w replace a value, p of them
carrying a payload, f misses):
    k_locate_capture   count (kind bytes) + 4 w (old values)
    compaction         2 count (kind bytes, once per scan) + 8 c (keys) + 4 w (old values) + 4 p (payload)
                       + 16 c (four change arrays) + 8 f (keys) + 8 f (two miss arrays)
Prints one JSON line with the card's name and power limit read in the same run.

    python benchmarks/change_capture.py                 # C2, C3, mixed, C4
    python benchmarks/change_capture.py --no-c4 --reps 5
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys

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


def workload(name, synth, rng):
    """(scale, core (src, dst, val), batch (src, dst, val or None), default_val)"""
    if name == "C4":
        scale, B = 24, 100_000_000
    else:
        scale, B = 20, 10_000_000
    total = 16 << scale
    cs, cd = synth.rmat(scale, 0, total, 42)
    cv = rng.integers(1, 1 << 30, cs.size).astype(np.uint32) if name == "mixed" else None
    if name == "C2":
        us, ud = synth.uniform(scale, 0, B, 7)
        return scale, (cs, cd, cv), (us, ud, None), 1
    if name == "C4":
        us, ud = synth.rmat(scale, 0, B, 99)
        return scale, (cs, cd, cv), (us, ud, None), 1
    idx = synth.sample_without_replacement(total, B, 7)
    if name == "C3":
        return scale, (cs, cd, cv), (cs[idx], cd[idx], None), 0
    ops = synth.mixed_ops(0, B, 11)
    us, ud = synth.uniform(scale, 0, B, 7)
    s, d = np.where(ops != 0, us, cs[idx]), np.where(ops != 0, ud, cd[idx])
    v = (ops != 0).astype(np.uint32) * rng.integers(1, 1 << 30, B).astype(np.uint32)
    return scale, (cs, cd, cv), (s, d, v), 1


def kernel_ms(prof, pred) -> float:
    import torch

    return sum(e.time_range.elapsed_us() for e in prof.events()
               if e.device_type == torch.autograd.DeviceType.CUDA and pred(e.name)) / 1000.0


def run_case(name, pp, synth, torch, warmup, reps):
    rng = np.random.default_rng(5)
    scale, (cs, cd, cv), (s, d, v), default = workload(name, synth, rng)
    n = 1 << scale
    sh = pp.Shard(n, device=0)
    sh.apply(cs, cd, cv)
    sh.snapshot()
    ts, td = (torch.from_numpy(x.astype(np.uint32).view(np.int32)).cuda() for x in (s, d))
    tv = torch.from_numpy(np.asarray(v, np.uint32).view(np.int32)).cuda() if v is not None else None
    B = int(s.size)

    def one(capture):
        sh.restore()
        sh.set_change_capture(capture)
        torch.cuda.synchronize()
        return sh.apply_device(ts.data_ptr(), td.data_ptr(), tv.data_ptr() if tv is not None else None, B, default)

    rows = {False: [], True: []}
    for i in range(warmup + reps):
        for capture in ((False, True) if i % 2 == 0 else (True, False)):
            st = one(capture)
            if i >= warmup:
                rows[capture].append((st["ms_total"], st["ms_locate"]))
    st = one(True)  # untimed: the lists of a capture-on batch, checked against its stats
    c = sh.last_changes()
    n_chg = st["n_inserted"] + st["n_overwritten"] + st["n_deleted"]
    assert c["src"].size == n_chg and c["nf_src"].size == st["n_not_found"], (name, c["src"].size, n_chg)
    assert int(np.sum(c["old_val"] == 0)) == st["n_inserted"]
    w = st["n_overwritten"] + st["n_deleted"]
    p = (st["n_inserted"] + st["n_overwritten"]) if v is not None else 0
    f = st["n_not_found"]
    locate_bytes = B + 4 * w
    compact_bytes = 2 * B + 8 * n_chg + 4 * w + 4 * p + 16 * n_chg + 16 * f
    # kernel times, one profiled batch per mode
    from torch.profiler import ProfilerActivity, profile

    prof_ms = {}
    for capture in (False, True):
        sh.restore()
        sh.set_change_capture(capture)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sh.apply_device(ts.data_ptr(), td.data_ptr(), tv.data_ptr() if tv is not None else None, B, default)
            torch.cuda.synchronize()
        prof_ms[capture] = {"locate_kernel_ms": kernel_ms(prof, lambda k: "k_locate" in k),
                            "compaction_ms": kernel_ms(prof, lambda k: "InCap" in k)}
    sh.close()
    med = lambda xs, j: float(np.median([x[j] for x in xs]))
    off_total, on_total = med(rows[False], 0), med(rows[True], 0)
    return {
        "case": name, "scale": scale, "batch": B,
        "n_changes": n_chg, "n_not_found": f,
        "ms_total_off": off_total, "ms_total_on": on_total,
        "overhead_pct": 100.0 * (on_total - off_total) / off_total,
        "ms_total_off_runs": [x[0] for x in rows[False]], "ms_total_on_runs": [x[0] for x in rows[True]],
        "ms_locate_off": med(rows[False], 1), "ms_locate_on": med(rows[True], 1),
        "profiled_off": prof_ms[False], "profiled_on": prof_ms[True],
        "extra_bytes_locate": locate_bytes, "extra_bytes_compaction": compact_bytes,
        "extra_bytes_per_update": (locate_bytes + compact_bytes) / B,
        "compaction_gbs": compact_bytes / (prof_ms[True]["compaction_ms"] * 1e6) if prof_ms[True]["compaction_ms"] else None,
    }


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--cases", default="C2,C3,mixed,C4")
    a = ap.parse_args(argv)
    import torch

    pp = importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    if pp.load_library().ppcsr_device_count() == 0:
        print("no CUDA device: nothing measured", file=sys.stderr)
        return 1
    cases = [c for c in a.cases.split(",") if c and not (a.no_c4 and c == "C4")]
    result = {"benchmark": "change_capture", **card(), "reps": a.reps, "warmup": a.warmup,
              "cases": [run_case(c, pp, synth, torch, a.warmup, a.reps) for c in cases]}
    print(json.dumps(result))
    return 0


if __name__ == "__main__":
    sys.exit(main())
