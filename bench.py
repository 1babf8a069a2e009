#!/usr/bin/env python
"""bench.py -- batched edge updates/s of the B200 Parallel Packed CSR engine (BASELINE.json metric).

A "step" is ONE pass of the hot path over one batch: the whole update batch is sorted, located and merged into the
packed edge array (window selection + rebalance, array doubling / halving folded in).

Default = BASELINE.json configs[3] ("C4", the config the >= 1e9 inserts/s target is quoted on):
  R-MAT scale-24 core graph (268 M raw edges, 2^29 slots) + ONE batch of 100 M skewed (R-MAT) edge insertions.
  --gpus 1 : one shard holds the whole graph.
  --gpus N : STRONG scaling -- the same graph and the same 100 M batch, vertex-range sharded over N GPUs (one process
             per GPU, edge-balanced contiguous ranges); every rank holds 1/N of the batch, routes it to the owners
             (fused bin+scatter over NVLink peer memory, NCCL all-to-all as the fallback) and applies what it owns.
The shard is restored from a device snapshot before every step, so every step is exactly that configuration.
At N = 1 the line also carries the other single-GPU configs as `other_configs` (C2: scale-20 + 10 M uniform inserts
with the 2^25 -> 2^26 doubling; C3: scale-20 + 10 M deletes; C5: 10 M mixed) and a PageRank push step over the C4 graph.

After the timed steps the logical graph of all shards is checksummed (ppcsr_checksum: edges, sum of mix64(src<<32|dst))
and compared with tests/golden/c4_checksum.json, which the UNMODIFIED reference produced for this exact workload
(tests/golden/make_c4_checksum.py): the scaling runs carry parity, not only invariants.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config C4|C2|C3|C5]
                  [--dump-outputs DIR]

--dump-outputs DIR (one GPU) writes what the timed steps computed as DIR/<name>.npy (float64, ~50 MB; see dump_graph):
the inputs are generated from fixed seeds, so two builds run with the same arguments can be compared file by file.

`--impl reference` times the reference's own CPU implementation (oracle/_ref/ref_driver: the unmodified reference
sources driven through ThreadPoolPPPCSR, -pppcsrnuma, all host threads) on the SAME workload, full size.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "edge_updates_per_sec"
UNIT = "updates/s"
SLOT_BYTES = 8  # this build: u32 dest + u32 value per slot (SoA)
CORE_SEED, UNIFORM_SEED, SKEW_SEED, OPS_SEED = 42, 7, 99, 11

# BASELINE.json configs (SURVEY.md §8d): name -> (scale, batch, workload)
CONFIGS = {
    "C4": (24, 100_000_000, "skewed"),
    "C2": (20, 10_000_000, "insert"),
    "C3": (20, 10_000_000, "delete"),
    "C5": (20, 10_000_000, "mixed"),
}
WORKLOAD_TEXT = {
    "insert": "uniform-random edge insertions",
    "delete": "edge deletions sampled from the core",
    "skewed": "skewed (R-MAT) edge insertions",
    "mixed": "mixed updates (3/4 uniform insertions, 1/4 deletions of core edges, per-update op)",
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS), help="BASELINE.json config (default C4)")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOAD_TEXT), help="override the config's stream")
    ap.add_argument("--scale", type=int, default=None, help="override the config's R-MAT scale")
    ap.add_argument("--batch", type=int, default=None, help="override the config's GLOBAL batch size")
    ap.add_argument("--weak", action="store_true",
                    help="weak scaling instead: scale + log2(N), --batch updates PER GPU (round-1 behaviour)")
    ap.add_argument("--strong", action="store_true", help="(the default now; kept so that older command lines still parse)")
    ap.add_argument("--pagerank", action="store_true", help="(kept for compatibility: the PageRank step is always timed)")
    ap.add_argument("--only-headline", action="store_true", help="skip other_configs / cpu_baseline at N = 1")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-sample", type=int, default=2_000_000, help="updates in the in-line cpu_baseline sample")
    ap.add_argument("--ref-budget-s", type=float, default=float(os.environ.get("PPCSR_REF_BUDGET_S", "200")),
                    help="--impl reference: full runs are repeated while they fit this wall-clock budget (>= 1 run)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the graph the last timed step left (a seeded sample) and the last PageRank step as "
                         "DIR/<name>.npy (one GPU)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    scale, batch, workload = CONFIGS[a.config]
    a.scale = a.scale if a.scale is not None else scale
    a.batch = a.batch if a.batch is not None else batch
    a.workload = a.workload or workload
    a.is_named = (a.scale, a.batch, a.workload) == CONFIGS[a.config] and not a.weak
    return a


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# workload description shared by both arms
# ------------------------------------------------------------------------------------------------
def global_shape(args, world):
    """(scale, GLOBAL batch) of the run: strong scaling keeps both fixed, --weak grows them with the ranks."""
    if args.weak:
        return args.scale + (world.bit_length() - 1), args.batch * world
    return args.scale, args.batch


def workload_config(args, world):
    scale, B = global_shape(args, world)
    name = args.config if args.is_named else "custom"
    return {
        "workload": f"{name}: R-MAT scale-{scale} core ({16 << scale} raw edges, a/b/c/d=.57/.19/.19/.05) + ONE batch of "
                    f"{B} {WORKLOAD_TEXT[args.workload]} per step" +
                    ("" if world == 1 else f", the same graph and batch split over {world} vertex-range shards"
                     if not args.weak else f" ({args.batch} per GPU, weak scaling)"),
        "config": name, "scale": scale, "global_batch": B, "batch_per_gpu": B // world, "slot_bytes": SLOT_BYTES,
        "parallelism": "1 shard" if world == 1 else f"{world} vertex-range shards (edge-balanced boundaries), updates "
                       "routed to their owner through NVLink peer memory (fused bin+scatter kernel; NCCL all-to-all "
                       "when unavailable)",
        "l2": "shard state is restored from a device snapshot (GBs of writes, far beyond the 126 MB L2) before every "
              "timed step; the working set also exceeds L2",
    }


def golden_checksum(args, world):
    """The reference's checksum for this exact workload, or None (tests/golden/c4_checksum.json)."""
    scale, B = global_shape(args, world)
    p = os.path.join(ROOT, "tests", "golden", "c4_checksum.json")
    if not os.path.exists(p):
        return None
    g = json.load(open(p))
    w = g.get("workload", {})
    if (w.get("scale"), w.get("batch"), w.get("stream")) == (scale, B, args.workload):
        return g
    return None


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ------------------------------------------------------------------------------------------------
def host_updates(scale, workload, lo, hi, synth, core=None):
    """Updates [lo, hi) of the workload's global stream on the host: (src, dst, value-or-array)."""
    total = 16 << scale
    if workload == "insert":
        us, ud = synth.uniform(scale, lo, hi, UNIFORM_SEED)
        return us, ud, 1
    if workload == "skewed":
        us, ud = synth.rmat(scale, lo, hi, SKEW_SEED)
        return us, ud, 1
    cs, cd = core if core is not None else synth.rmat(scale, 0, total, CORE_SEED)
    idx = synth.sample_without_replacement(total, hi, UNIFORM_SEED)[lo:hi]
    if workload == "delete":
        return cs[idx], cd[idx], 0
    ops = synth.mixed_ops(lo, hi, OPS_SEED)
    us, ud = synth.uniform(scale, lo, hi, UNIFORM_SEED)
    return np.where(ops != 0, us, cs[idx]), np.where(ops != 0, ud, cd[idx]), ops


def run_reference_once(scale, workload, count, threads, ppd, synth, tmp, checksum=False):
    """One run of the unmodified reference: core load, then `count` updates; returns ref_driver's timing dict.
    Insert streams are synthesised inside ref_driver (same counter hash as synth.py, pinned by tests/test_oracle.py);
    delete / mixed streams need the sampled core edges and travel as a file of triples."""
    import oracle_py as O

    n, total = 1 << scale, 16 << scale
    tpath, spath = os.path.join(tmp, "timing.json"), os.path.join(tmp, "sum.json")
    cmd = [O.REF_DRIVER, "--mode", "pppcsrnuma", "--api", "pool", "--threads", str(threads), "--ppd", str(ppd),
           "--n", str(n), "--synth-core", f"rmat:{scale}:0:{total}:{CORE_SEED}", "--timing", tpath]
    if workload == "insert":
        cmd += ["--synth-updates", f"uniform:{scale}:0:{count}:{UNIFORM_SEED}"]
    elif workload == "skewed":
        cmd += ["--synth-updates", f"rmat:{scale}:0:{count}:{SKEW_SEED}"]
    else:
        upd = os.path.join(tmp, "upd.bin")
        if not os.path.exists(upd):
            us, ud, v = host_updates(scale, workload, 0, count, synth)
            synth.write_triples(upd, us, ud, v)
        cmd += ["--updates", upd, "--size", str(count)]
    if checksum:
        cmd += ["--checksum", spath]
    subprocess.run(cmd, stdout=subprocess.DEVNULL, check=True)
    out = json.load(open(tpath))
    if checksum:
        out["checksum"] = json.load(open(spath))
    return out


def run_port_once(scale, workload, sample, synth):
    """No compiled reference on this box: time the C restatement (1 thread) instead."""
    import oracle_py as O

    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, CORE_SEED)
    g = O.OraclePCSR(n)
    g.apply(cs, cd, 1)
    us, ud, v = host_updates(scale, workload, 0, sample, synth, core=(cs, cd))
    t0 = time.perf_counter()
    g.apply(us, ud, v)
    return {"update_ms": (time.perf_counter() - t0) * 1e3, "update_ops": sample}


def host_description():
    threads = os.cpu_count() or 1
    nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]) \
        if os.path.isdir("/sys/devices/system/node") else 1
    return threads, nodes


def cpu_baseline_sample(args, synth):
    """In-line cpu_baseline of the B200 arm (N = 1): a BOUNDED sample so that the default run stays short -- the
    reference on a scale-20 core + the first --cpu-sample updates of the workload's stream (the full-size run is the
    reference arm, --impl reference)."""
    import oracle_py as O

    scale = min(args.scale, 20)
    sample = min(args.cpu_sample, args.batch)
    threads, nodes = host_description()
    what = (f"BOUNDED SAMPLE: R-MAT scale-{scale} core loaded through the reference, then the first {sample} "
            f"{WORKLOAD_TEXT[args.workload]}; time = start()->stop() of the update phase")
    if O.have_ref():
        with tempfile.TemporaryDirectory() as tmp:
            t = run_reference_once(scale, args.workload, sample, threads, 1, synth, tmp)
        kind, cores = "reference", threads
        what += (f"; -pppcsrnuma -threads={threads} -partitions_per_domain=1; host has {threads} hardware threads, "
                 f"{nodes} NUMA node(s); libnuma stubbed (the binary is built without libnuma => 1 domain)")
    else:
        t = run_port_once(scale, args.workload, sample, synth)
        kind, cores = "port", 1
    ms = float(t["update_ms"])
    return {"value": sample / (ms / 1e3), "unit": UNIT, "cores": cores, "kind": kind, "sample": what}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle_py as O

    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    world = max(1, args.gpus)
    scale, B = global_shape(args, world)
    threads, nodes = host_description()
    times, core_times, checksum = [], [], None
    t_start = time.perf_counter()
    if O.have_ref():
        kind, cores = "reference", threads
        with tempfile.TemporaryDirectory() as tmp:
            # FULL runs of the same workload (no sampling).  One run = core load + the whole batch; repeated up to
            # --steps times while the wall-clock budget lasts (the core load dominates a run, so warm-up runs are not
            # affordable at scale 24: the first run counts).
            for i in range(max(1, args.steps)):
                t = run_reference_once(scale, args.workload, B, threads, world, synth, tmp, checksum=(i == 0))
                times.append(t["update_ms"])
                core_times.append(t["core_ms"])
                checksum = t.get("checksum", checksum)
                elapsed = time.perf_counter() - t_start
                if elapsed + elapsed / (i + 1) > args.ref_budget_s:
                    break
        what = (f"FULL workload, no sampling: R-MAT scale-{scale} core ({16 << scale} raw edges) loaded through the "
                f"reference's ThreadPoolPPPCSR, then the whole batch of {B} {WORKLOAD_TEXT[args.workload]}; time = the "
                f"reference's own start()->stop() of the update phase; {len(times)} full run(s) (core load "
                f"{np.mean(core_times) / 1e3:.1f} s each); -pppcsrnuma -threads={threads} "
                f"-partitions_per_domain={world} (one partition per shard of the B200 arm); host has {threads} "
                f"hardware threads, {nodes} NUMA node(s); libnuma stubbed (the binary is built without libnuma => 1 "
                f"domain)")
    else:
        sample = min(args.cpu_sample, B)
        times.append(run_port_once(min(scale, 20), args.workload, sample, synth)["update_ms"])
        B, kind, cores = sample, "port", 1
        what = f"oracle port (1 thread), scale-{min(scale, 20)} core + first {sample} updates: oracle/_ref is missing"
    ms = float(np.mean(times))
    value = B / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": 0, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if args.weak else "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": what},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if checksum is not None:
        gold = golden_checksum(args, world)
        line["parity"] = {"checksum": checksum,
                          "matches_golden": None if gold is None else
                          (checksum["edges"] == gold["edges"] and checksum["edge_hash"] == gold["edge_hash"])}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed, for comparing two builds output for output
# ------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 20  # vertices and edges sampled: the C4 graph itself (16.8 M vertices, 360 M edges) is GBs
# the outcome of a batch; the window / byte counts are left out: they describe how a build did the work
BATCH_COUNTS = ("batch_size", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found", "slots_before",
                "slots_after", "resized")


def dump_graph(out_dir, shard, stats):
    """Writes the logical graph the last timed step left on the shard, as float64 arrays (ids < 2^32 are exact):
      checksum.npy       edges, edge_hash >> 32, edge_hash & 0xffffffff, nn_hash >> 32, nn_hash & 0xffffffff
      batch.npy          the last step's counts: BATCH_COUNTS, in that order
      vertices.npy       a seeded sample of vertex ids (sorted, unique), and for them
      degree.npy         out-degree in the logical graph (rowptr[v + 1] - rowptr[v])
      num_neighbors.npy  num_neighbors (call-count semantics of the reference)
      edge_src.npy       a seeded sample of positions of the exported CSR (sorted, unique): source of the edge there
      edge_dst.npy       and its destination
    Returns the vertex sample: run_config writes the last timed PageRank push step at those vertices as pagerank.npy."""
    os.makedirs(out_dir, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))

    cks = shard.checksum()
    save("checksum", [cks["edges"], cks["edge_hash"] >> 32, cks["edge_hash"] & 0xFFFFFFFF, cks["nn_hash"] >> 32,
                      cks["nn_hash"] & 0xFFFFFFFF])
    save("batch", [stats[k] for k in BATCH_COUNTS])
    rowptr, col = shard.export()
    rowptr = rowptr.astype(np.int64)
    n, E = rowptr.size - 1, col.size
    rng = np.random.default_rng(0)
    verts = np.unique(rng.integers(0, n, DUMP_SAMPLE)) if n else np.zeros(0, dtype=np.int64)
    save("vertices", verts)
    save("degree", (rowptr[verts + 1] - rowptr[verts]).astype(np.int64))
    save("num_neighbors", shard.num_neighbors()[verts])
    pos = np.unique(rng.integers(0, E, DUMP_SAMPLE)) if E else np.zeros(0, dtype=np.int64)
    save("edge_src", np.searchsorted(rowptr, pos, side="right") - 1)
    save("edge_dst", col[pos])
    return verts


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def make_updates(synth, torch, workload, scale, lo, hi, total_updates, dev):
    """This rank's slice [lo, hi) of the workload's global stream on the device: (src, dst, op-or-None, default_val)."""
    core_total = 16 << scale
    uv, default_val = None, 1
    if workload == "insert":
        us, ud = synth.uniform(scale, lo, hi, UNIFORM_SEED, device=dev)
    elif workload == "skewed":
        us, ud = synth.rmat(scale, lo, hi, SKEW_SEED, device=dev)
    else:
        # deletes: sampled without replacement from the raw core list; only the sampled edges are regenerated
        # (the stream is a pure function of the element index)
        idx = synth.sample_without_replacement(core_total, total_updates, UNIFORM_SEED, device=dev)[lo:hi]
        us, ud = synth.rmat_at(scale, idx, CORE_SEED)
        del idx
        if workload == "delete":
            default_val = 0
        else:
            uv = synth.mixed_ops(lo, hi, OPS_SEED, device=dev)
            fs, fd = synth.uniform(scale, lo, hi, UNIFORM_SEED, device=dev)
            us, ud = torch.where(uv != 0, fs, us), torch.where(uv != 0, fd, ud)
            uv = uv.to(torch.int32).contiguous()
            del fs, fd
    return us.to(torch.int32).contiguous(), ud.to(torch.int32).contiguous(), uv, default_val


def build_core(synth, torch, router, scale, rank, world, local_rank, dev, dist, workload, B_rank, chunk=1 << 26):
    """Generates this rank's slice of the R-MAT core (in pieces: the generator works in int64 lanes), computes the
    shard boundaries and loads the core through the normal batch path."""
    n, core_total = 1 << scale, 16 << scale
    lo, hi = rank * core_total // world, (rank + 1) * core_total // world
    cs = torch.empty(hi - lo, dtype=torch.int32, device=dev)
    cd = torch.empty(hi - lo, dtype=torch.int32, device=dev)
    for a in range(lo, hi, chunk):
        b = min(hi, a + chunk)
        s, d = synth.rmat(scale, a, b, CORE_SEED, device=dev)
        cs[a - lo:b - lo] = s.to(torch.int32)
        cd[a - lo:b - lo] = d.to(torch.int32)
        del s, d
    if world > 1:
        # Shard cost model measured at N=1/2: ~0.13 us per routed update (sort + locate) and ~0.016 us per stored
        # item (window selection + rebalance).  A uniform stream sends B/n updates to every vertex, so a vertex
        # weighs ~8 * B/n "edges"; skewed inserts and deletes follow the edge distribution instead.
        # Every vertex also stores one sentinel (an item like an edge), so it weighs at least 1: with weight 0 the shard
        # of the low-degree tail of an R-MAT graph holds millions of sentinels more than the others and is the one that
        # has to double its array (measured at 8 GPUs: 7.3 M vertices, 2^26 -> 2^27 slots, +0.13 ms on that rank).
        vw = 8.0 * B_rank * world / n + 1.0 if workload in ("insert", "mixed") else 1.0
        starts = router.edge_balanced_starts(cs, n, world, dist, vertex_weight=vw)
    else:
        starts = np.array([0, n], dtype=np.uint64)
    peer_cap = 0 if os.environ.get("PPCSR_NO_PEER") else max(B_rank, hi - lo)
    graph = router.ShardedGraph(n, starts, rank, world, local_rank, dist=dist, peer_cap=peer_cap,
                                peer_values=workload == "mixed")
    graph.shard.bind_torch_stream(torch.cuda.current_stream())
    graph.apply(cs, cd, None, default_val=1, global_max=-(-core_total // world))
    return graph, starts


def run_config(args, scale, B, workload, torch, dist, rank, world, local_rank, dev, steps, warmup, e2e_steps,
               with_clocks=False, with_pagerank=False, golden=None, dump_dir=None):
    """Builds the graph, times `steps` device-resident steps and `e2e_steps` host-buffer steps.  Returns a dict of
    results (rank 0 view; times are the max over ranks).  dump_dir (one shard): see dump_graph."""
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    router = importlib.import_module("parallel-packed-csr_b200.router")
    stream = torch.cuda.current_stream()
    n = 1 << scale
    Br = B // world  # this rank's slice of the global batch
    graph, starts = build_core(synth, torch, router, scale, rank, world, local_rank, dev, dist, workload, Br)
    core_geo = graph.shard.geometry
    us, ud, uv, default_val = make_updates(synth, torch, workload, scale, rank * Br, (rank + 1) * Br, Br * world, dev)
    # room for one doubling and for a received batch 1.5x the average (skewed streams, imperfect boundaries)
    graph.shard.reserve(max_slots=core_geo.N * 2, max_batch=int(Br * 1.5) + 1024)
    graph.shard.snapshot()
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing (value)
    stats_acc = []
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for _ in range(warmup):
        graph.shard.restore()
        graph.apply(us, ud, uv, default_val=default_val, global_max=Br)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0 and with_clocks:
        sampler.start()
    for k in range(steps):
        graph.shard.restore()
        barrier()  # the untimed restore takes a different time on every shard: start the step together
        ev0[k].record(stream)
        st = graph.apply(us, ud, uv, default_val=default_val, global_max=Br)
        ev1[k].record(stream)
        stats_acc.append(st)
    barrier()
    local_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
    total_ms = allmax(local_ms)
    value = Br * world * steps / (total_ms / 1e3)
    if world > 1 and os.environ.get("PPCSR_ROUTE_TIMING"):
        graph.route_timing = []
        for _ in range(3):
            graph.shard.restore()
            barrier()
            graph.apply(us, ud, uv, default_val=default_val, global_max=Br)
        print(f"[rank {rank}] routing stages ms ([bin, counts, all-to-all, apply] over NCCL, [exchange, apply] over "
              f"peer memory): {graph.route_timing}", file=sys.stderr)
        graph.route_timing = None
    if world > 1:  # per-rank view (stderr): how many updates each shard received and where its time went
        s0 = stats_acc[-1]
        print(f"[rank {rank}] local ms/step {local_ms / steps:.3f} received {s0['batch_size']} apply "
              f"{s0['ms_total']:.3f} ms (sort {s0['ms_sort']:.3f} locate {s0['ms_locate']:.3f} select "
              f"{s0['ms_select']:.3f} rebalance {s0['ms_rebalance']:.3f}) windows {s0['n_windows']} N "
              f"{s0['slots_before']}->{s0['slots_after']} vertices {graph.n_local}", file=sys.stderr)

    # ---- parity guard on the state after ONE application of the batch: invariants + checksum of the logical graph
    lower = workload in ("delete", "mixed")
    rep = graph.shard.check(check_lower=lower)
    if rep.violations(lower):
        raise SystemExit(f"bench.py: PMA invariants violated after the timed steps: {rep.as_dict()}")
    cs = graph.shard.checksum(int(starts[rank]))
    tot = torch.tensor([cs["edges"], cs["edge_hash"] - (1 << 64) if cs["edge_hash"] >= (1 << 63) else cs["edge_hash"],
                        cs["nn_hash"] - (1 << 64) if cs["nn_hash"] >= (1 << 63) else cs["nn_hash"]],
                       dtype=torch.int64, device=dev)
    if dist is not None:
        dist.all_reduce(tot)  # int64 sums wrap mod 2^64, like the checksum itself
    edges, edge_hash, nn_hash = (int(x) & ((1 << 64) - 1) for x in tot.tolist())
    parity = {"edges": edges, "edge_hash": f"{edge_hash:016x}", "nn_hash": f"{nn_hash:016x}",
              "invariants": "I1-I6 hold on every shard", "golden": None}
    if golden is not None:
        ok = edges == golden["edges"] and parity["edge_hash"] == golden["edge_hash"] and \
            parity["nn_hash"] == golden["nn_hash_call_count"]
        parity["golden"] = {"file": "tests/golden/c4_checksum.json", "produced_by": golden.get("produced_by"),
                            "edges_and_edge_hash": "reference run", "nn_hash": "call-count rule over the streams",
                            "match": ok}
        if not ok:
            raise SystemExit(f"bench.py: logical graph differs from the reference's: {parity} vs {golden}")
    dump_vertices = dump_graph(dump_dir, graph.shard, stats_acc[-1]) if dump_dir else None

    # ---- end to end through the public host-buffer call: pinned host inputs, H2D inside the timed region; the state
    # restore between the steps (a device-to-device copy) is inside the timed region as well
    hs = torch.empty(Br, dtype=torch.int32).pin_memory()
    hd = torch.empty(Br, dtype=torch.int32).pin_memory()
    hs.copy_(us)
    hd.copy_(ud)
    hv = None
    if uv is not None:
        hv = torch.empty(Br, dtype=torch.int32).pin_memory()
        hv.copy_(uv)
    hsn, hdn, hvn = hs.numpy(), hd.numpy(), hv.numpy() if hv is not None else None
    graph.shard.restore()
    graph.wait_host(graph.submit_host(hsn, hdn, hvn, default_val=default_val, global_max=Br))  # warm-up (allocates the staging slots)
    barrier()
    # Pipelined submit (ppcsr_submit_batch / ppcsr_wait): the copy of step k+1 runs under the compute of step k.  Every
    # step's H2D copy, its stats read-back and the restore of the state lie between t0 and the final synchronise.
    t0 = time.perf_counter()
    ticket = graph.submit_host(hsn, hdn, hvn, default_val=default_val, global_max=Br)
    for k in range(e2e_steps):
        nxt = graph.submit_host(hsn, hdn, hvn, default_val=default_val, global_max=Br) if k + 1 < e2e_steps else None
        graph.shard.restore()
        e2e_stats = graph.wait_host(ticket)
        ticket = nxt
    torch.cuda.synchronize()
    e2e_ms = allmax((time.perf_counter() - t0) * 1e3)
    # the same without the pipeline (one blocking ppcsr_apply_batch per step), for comparison
    barrier()
    t0 = time.perf_counter()
    for k in range(min(3, e2e_steps)):
        graph.shard.restore()
        graph.apply_host(hsn, hdn, hvn, default_val=default_val, global_max=Br)
    torch.cuda.synchronize()
    e2e_sync_ms = allmax((time.perf_counter() - t0) * 1e3) / min(3, e2e_steps)
    e2e_value = Br * world * e2e_steps / (e2e_ms / 1e3)

    # ---- edge scan: PageRank push steps over the updated graph (reference pagerank.h:16-29)
    pagerank = None
    if with_pagerank:
        vals = 1.0 + (torch.arange(n, device=dev, dtype=torch.float64) % 7)
        graph.pagerank_step(vals)
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        for _ in range(steps):
            pr = graph.pagerank_step(vals)
        p1.record(stream)
        barrier()
        if dump_vertices is not None:  # the last step's push result at the sampled vertices
            np.save(os.path.join(dump_dir, "pagerank.npy"), pr.cpu().numpy()[dump_vertices])
        geo = graph.shard.geometry
        pr_ms = allmax(p0.elapsed_time(p1) / steps)
        # SURVEY.md §8d: 12 n (node array) + slot bytes * N (every slot, gaps included) + 4 n (contribution) + 8 E
        pr_bytes = 12 * n + SLOT_BYTES * int(geo.N) * world + 4 * n + 8 * edges if world == 1 else None
        pagerank = {"ms_per_step": pr_ms, "slots_rank0": int(geo.N), "edges": edges,
                    "algorithmic_bytes": pr_bytes,
                    "achieved_gbs": (pr_bytes / (pr_ms / 1e3) / 1e9) if pr_bytes else None,
                    "note": "one push step over every shard (+ one all-reduce of the fp64 vector when sharded)"}

    clocks = sampler.stop() if (rank == 0 and with_clocks) else None

    def mean(key):
        return float(np.mean([s[key] for s in stats_acc]))

    peak, peak_src = measured_peak()
    reb_bytes, reb_ms = mean("rebalance_bytes"), mean("ms_rebalance_kernel")
    achieved = reb_bytes / (reb_ms / 1e3) / 1e9 if reb_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1:
        try:  # ncu DRAM bytes of the roofline kernel, captured per workload (null where there is no capture)
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch", {}).get(f"{workload}/scale{scale}/batch{B}")
        except Exception:
            traffic = None
    last = stats_acc[-1]
    out = {
        "value": value, "ms_per_step": total_ms / steps, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": (3 if hv is not None else 2) * 4 * Br * world,
                "d2h_bytes_per_step": 2 * 128 * world, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                "ms_per_step_unpipelined": e2e_sync_ms,
                "api": "ppcsr_submit_batch / ppcsr_wait (pinned host buffers; the copy of step k+1 runs under the "
                       "compute of step k); the device-to-device state restore between steps is inside the timed "
                       "region; ms_per_step_unpipelined = one blocking ppcsr_apply_batch per step"},
        "gpu_launches": int(sum(s["kernel_launches"] for s in stats_acc)),
        "roofline": {"bound": "hbm", "kernel": "reb::k_rebalance_m", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": reb_bytes, "kernel_ms": reb_ms,
                     "note": "rank 0's shard" if world > 1 else "the whole array streamed once"},
        "stages_ms": {k: mean(k) for k in ("ms_total", "ms_sort", "ms_locate", "ms_select", "ms_rebalance",
                                           "ms_rebalance_kernel")},
        "batch": {k: int(last[k]) for k in ("batch_size", "n_unique", "n_inserted", "n_overwritten", "n_deleted",
                                            "n_not_found", "n_windows", "window_slots", "slots_before", "slots_after",
                                            "resized", "whole_array")},
        "rebalance_bytes_per_update": reb_bytes / max(1, int(last["batch_size"])),
        "hbm_roofline_updates_per_sec": peak * 1e9 / (16 + reb_bytes / max(1, int(last["batch_size"]))),
        "parity": parity,
    }
    if pagerank is not None:
        out["pagerank"] = pagerank
    graph.shard.close()
    del graph, us, ud, uv, hs, hd, hv
    torch.cuda.empty_cache()
    return out


def main_b200(args):
    import torch

    importlib.import_module("parallel-packed-csr_b200")
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 engine has no CPU fallback)")
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs supports one GPU")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        # NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION/WARN; rank 0 must print ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    scale, B = global_shape(args, world)
    res = run_config(args, scale, B, args.workload, torch, dist, rank, world, local_rank, dev, args.steps, args.warmup,
                     args.e2e_steps, with_clocks=True, with_pagerank=True, golden=golden_checksum(args, world),
                     dump_dir=args.dump_outputs)
    others = {}
    if world == 1 and not args.only_headline and args.is_named:
        for name in ("C2", "C3", "C5"):
            if name == args.config:
                continue
            s2, b2, w2 = CONFIGS[name]
            try:
                r = run_config(args, s2, b2, w2, torch, None, 0, 1, local_rank, dev, args.steps, args.warmup,
                               min(args.e2e_steps, 5))
                others[name] = {"workload": f"R-MAT scale-{s2} core + {b2} {WORKLOAD_TEXT[w2]}", "value": r["value"],
                                "unit": UNIT, "ms_per_step": r["ms_per_step"], "e2e": r["e2e"]["value"],
                                "roofline_frac": r["roofline"]["frac"], "rebalance_kernel_ms": r["roofline"]["kernel_ms"],
                                "stages_ms": r["stages_ms"], "batch": r["batch"]}
            except Exception as e:  # the headline must survive a failing side config
                others[name] = {"failed": f"{type(e).__name__}: {e}"}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    line = {
        "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak" if args.weak else "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(args, world),
    }
    for k in ("clocks", "e2e", "gpu_launches", "roofline", "stages_ms", "batch", "rebalance_bytes_per_update",
              "hbm_roofline_updates_per_sec", "parity", "pagerank"):
        if k in res:
            line[k] = res[k]
    if others:
        line["other_configs"] = others
    if world == 1 and not args.no_cpu_baseline and not args.only_headline:
        try:
            line["cpu_baseline"] = cpu_baseline_sample(args, synth)
        except Exception as e:  # the baseline is reported context, never a reason to lose the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


def _claim_stdout():
    """Rank 0 must print exactly ONE JSON line on stdout, but libraries (NCCL's version banner) write to fd 1
    directly.  Point fd 1 at stderr for the whole run and keep the real stdout for the result line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real


if __name__ == "__main__":
    a = parse_args()
    _claim_stdout()
    rc = main_reference(a) if a.impl == "reference" else main_b200(a)
    sys.stdout.flush()
    sys.exit(rc)
