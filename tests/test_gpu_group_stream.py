"""Streaming batches into a group (ppcsr_group_submit / ppcsr_group_wait, Group.submit / Group.wait).

A stream `submit(b0); for i: { submit(b[i+1]); wait(b[i]); }` must leave exactly the graph that Group.apply of the same
batches leaves: exports with values, num_neighbors, the summed checksum and the per-shard batch counters, and a single
shard fed the same batches agrees.  Groups of 1 to 8 shards share GPU 0 here; the distinct-device case needs two GPUs
and skips otherwise."""
import importlib
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

pp = importlib.import_module("parallel-packed-csr_b200")
build = importlib.import_module("parallel-packed-csr_b200.build")
synth = importlib.import_module("parallel-packed-csr_b200.synth")

pytestmark = pytest.mark.gpu
MASK64 = (1 << 64) - 1
ERR_ARG, ERR_CAPACITY = -2, -3
COUNTERS = ("batch_size", "n_ignored", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found")


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def random_starts(n, k, seed):
    """k + 1 ascending boundaries; for k >= 2 one shard holds a single vertex."""
    if k == 1:
        return np.array([0, n], np.uint64)
    if k == 2:
        return np.array([0, n - 1, n], np.uint64)
    rng = np.random.default_rng(seed)
    c = int(rng.integers(1, n - 2))
    cuts = {c, c + 1}
    while len(cuts) < k - 1:
        cuts.add(int(rng.integers(1, n)))
    return np.array([0] + sorted(cuts) + [n], np.uint64)


def stream_batches(scale=14):
    """(src, dst, val or None, default_val): the R-MAT core, uniform inserts with default_val 7, edges with dst >= n,
    deletes of core edges and misses with default_val 0, a mixed batch with distinct values (0 = remove), an empty
    batch, and a batch of a prime size (no multiple of any shard count)."""
    n = 1 << scale
    rng = np.random.default_rng(11)
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, 20000, 7)
    xs, xd = rng.integers(0, n, 600), n + rng.integers(0, 4000, 600)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    ds = np.concatenate([cs[idx], rng.integers(0, n, 3000)])
    dd = np.concatenate([cd[idx], rng.integers(0, n, 3000)])
    ms, md = rng.integers(0, n, 30000), rng.integers(0, n + 50, 30000)
    mv = rng.integers(1, 1 << 24, 30000).astype(np.uint32)
    mv[rng.random(30000) < 0.3] = 0
    empty = np.zeros(0, np.uint32)
    ps, pd = rng.integers(0, n, 10007), rng.integers(0, n, 10007)
    batches = [(cs, cd, None, 1), (us, ud, None, 7), (xs, xd, None, 1), (ds, dd, None, 0), (ms, md, mv, 1),
               (empty, empty, None, 1), (ps, pd, None, 1)]
    return n, [(np.asarray(s, np.uint32), np.asarray(d, np.uint32), v, dv) for s, d, v, dv in batches]


def make_group(n, starts, batches, devices=None, with_values=True):
    k = len(starts) - 1
    cap = max(s.size for s, _, _, _ in batches) // k + 1
    return pp.Group(n, starts, devices or [0] * k, region_cap=cap, with_values=with_values)


def stream(g, batches):
    """Two ahead: submit(b0); for i: { submit(b[i+1]); wait(b[i]); }.  Returns the per-shard stats of every batch."""
    out, tickets = [], []
    for s, d, v, dv in batches:
        tickets.append(g.submit(s, d, v, dv))
        if len(tickets) == 2:
            out.append(g.wait(tickets.pop(0)))
    out += [g.wait(t) for t in tickets]
    return out


def apply_each(g, batches):
    return [g.apply(s, d, v, dv) for s, d, v, dv in batches]


def group_checksum(g):
    out = [0, 0, 0]
    for r, sh in enumerate(g.shards):
        c = sh.checksum(int(g.starts[r]))
        out = [(out[0] + c["edges"]) & MASK64, (out[1] + c["edge_hash"]) & MASK64, (out[2] + c["nn_hash"]) & MASK64]
    return tuple(out)


def group_export(g):
    """The global CSR (rowptr, col, val) and num_neighbors, concatenated over the shards."""
    rps, cols, vals, nns, off = [np.zeros(1, np.uint64)], [], [], [], 0
    for sh in g.shards:
        rp, c, v = sh.export(with_values=True)
        rps.append(rp[1:] + np.uint64(off))
        off += int(rp[-1])
        cols.append(c)
        vals.append(v)
        nns.append(sh.num_neighbors())
    return np.concatenate(rps), np.concatenate(cols), np.concatenate(vals), np.concatenate(nns)


def assert_same_graph(a, b, where=""):
    assert group_checksum(a) == group_checksum(b), where
    for x, y, name in zip(group_export(a), group_export(b), ("rowptr", "col", "val", "nn")):
        assert np.array_equal(x, y), (where, name)


def assert_same_counters(got, want, where=""):
    assert len(got) == len(want), where
    for i, (sg, sw) in enumerate(zip(got, want)):
        assert len(sg) == len(sw), (where, i)
        for r, (a, b) in enumerate(zip(sg, sw)):
            assert {c: a[c] for c in COUNTERS} == {c: b[c] for c in COUNTERS}, (where, i, r)


def assert_clean(g, where=""):
    for r, sh in enumerate(g.shards):
        assert not sh.check(False).violations(False), (where, r, sh.check(False).as_dict())


def assert_matches_single(g, single, where=""):
    rp, c, v, nn = group_export(g)
    srp, sc, sv = single.export(with_values=True)
    assert np.array_equal(rp, srp) and np.array_equal(c, sc) and np.array_equal(v, sv), where
    assert np.array_equal(nn, single.num_neighbors()), where
    s = single.checksum(0)
    assert group_checksum(g) == (s["edges"], s["edge_hash"], s["nn_hash"]), where


def raw_submit(g, s, d, v=None, dv=1):
    t = pp.C.c_uint64()
    s, d = pp._u32_array(s), pp._u32_array(d)
    v = pp._u32_array(v) if v is not None else None
    return g.L.ppcsr_group_submit(g.g, pp._np_ptr(s), pp._np_ptr(d), pp._np_ptr(v), s.size, dv, pp.C.byref(t)), t.value


# ------------------------------------------------------------------------------------------------
# scale-14 stream shared by the equivalence tests
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def graph14():
    n, batches = stream_batches()
    single = pp.Shard(n)
    for s, d, v, dv in batches:
        single.apply(s, d, v, dv)
    yield dict(n=n, batches=batches, single=single)
    single.close()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8])
def test_stream_equals_apply(graph14, k):
    n, batches = graph14["n"], graph14["batches"]
    starts = random_starts(n, k, seed=k)
    g, twin = make_group(n, starts, batches), make_group(n, starts, batches)
    got = stream(g, batches)
    want = apply_each(twin, batches)
    assert_same_counters(got, want, k)
    assert sum(st["n_not_found"] for st in got[3]) > 0 and sum(st["n_deleted"] for st in got[3]) > 0
    assert sum(st["batch_size"] for st in got[5]) == 0
    assert_same_graph(g, twin, k)
    assert_matches_single(g, graph14["single"], k)
    assert_clean(g, k)
    # the group keeps streaming after a drained stream, and Group.apply still works on it
    more = batches[1:3]
    stream(g, more)
    apply_each(twin, more)
    g.apply(*batches[4])
    twin.apply(*batches[4])
    assert_same_graph(g, twin, (k, "more"))
    g.close()
    twin.close()


def test_interleaving_with_apply_traversals_and_repartition(graph14):
    """apply -> stream -> apply -> BFS -> PageRank -> repartition -> stream, against the same sequence by Group.apply."""
    n, b = graph14["n"], graph14["batches"]
    starts = random_starts(n, 4, seed=3)
    g, twin = make_group(n, starts, b), make_group(n, starts, b)
    steps = [("apply", b[0:1]), ("stream", b[1:4]), ("apply", b[4:5])]
    for kind, part in steps:
        (stream if kind == "stream" else apply_each)(g, part)
        apply_each(twin, part)
    hub = int(np.argmax(np.diff(group_export(twin)[0].astype(np.int64))))
    assert np.array_equal(g.bfs(hub), twin.bfs(hub))
    got, want = g.pagerank(10, 0.85), twin.pagerank(10, 0.85)
    assert np.allclose(got, want, rtol=1e-9, atol=0.0)
    new = np.linspace(0, n, 5).astype(np.uint64)
    st_g, st_t = g.repartition(new), twin.repartition(new)
    assert st_g["vertices_moved"] == st_t["vertices_moved"] and st_g["edges_moved"] == st_t["edges_moved"]
    assert_same_counters(stream(g, b[5:7] + b[1:2]), apply_each(twin, b[5:7] + b[1:2]))
    assert_same_graph(g, twin)
    assert_clean(g)
    g.close()
    twin.close()


def test_misuse_leaves_the_group_usable():
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    rng = np.random.default_rng(5)
    b1 = (rng.integers(0, n, 4000).astype(np.uint32), rng.integers(0, n, 4000).astype(np.uint32))
    b2 = (rng.integers(0, n, 4000).astype(np.uint32), rng.integers(0, n, 4000).astype(np.uint32))
    starts = random_starts(n, 3, seed=9)
    cap = cs.size // 3 + 1
    g = pp.Group(n, starts, [0] * 3, region_cap=cap)  # no value buffers
    twin = pp.Group(n, starts, [0] * 3, region_cap=cap)
    for x in (g, twin):
        x.apply(cs, cd)
    before = group_checksum(g)
    L = g.L
    # values into a group created without values, a slice above region_cap: nothing in flight afterwards
    assert raw_submit(g, *b1, v=np.ones(4000, np.uint32))[0] == ERR_ARG
    big = np.zeros(3 * cap + 3, np.uint32)
    assert raw_submit(g, big, big)[0] == ERR_CAPACITY
    assert group_checksum(g) == before
    t1, t2 = g.submit(*b1), g.submit(*b2)
    assert raw_submit(g, *b1)[0] == ERR_ARG                    # a third batch
    assert L.ppcsr_group_wait(g.g, t2, None) == ERR_ARG         # the newer ticket first
    assert L.ppcsr_group_wait(g.g, t2 + 7, None) == ERR_ARG     # an unknown ticket
    # the calls that read or rewrite the shards refuse while batches are in flight
    h = np.zeros(n, np.uint32)
    s, d = pp._u32_array(b1[0]), pp._u32_array(b1[1])
    assert L.ppcsr_group_apply(g.g, pp._np_ptr(s), pp._np_ptr(d), None, s.size, 1, None) == ERR_ARG
    assert L.ppcsr_group_bfs(g.g, 0, pp._np_ptr(h)) == ERR_ARG
    assert L.ppcsr_group_pagerank(g.g, 3, 0.85, pp._np_ptr(np.zeros(n))) == ERR_ARG
    new = np.linspace(0, n, 4).astype(np.uint64)
    assert L.ppcsr_group_repartition(g.g, pp._np_ptr(new), None) == ERR_ARG
    assert group_checksum(g) == before and np.array_equal(g.starts, starts)
    g.wait(t1)
    g.wait(t2)
    assert L.ppcsr_group_wait(g.g, t1, None) == ERR_ARG         # already waited for
    twin.apply(*b1)
    twin.apply(*b2)
    assert_same_graph(g, twin)
    # usable: the stream, traversals and a repartition go on as on the twin
    assert_same_counters(stream(g, [(*b2, None, 0), (*b1, None, 1)]),
                         apply_each(twin, [(*b2, None, 0), (*b1, None, 1)]))
    assert np.array_equal(g.bfs(0), twin.bfs(0))
    g.repartition(new)
    twin.repartition(new)
    assert_same_graph(g, twin)
    assert_clean(g)
    twin.close()
    # close() with two batches in flight: synchronises and frees without applying them
    g.submit(*b1)
    g.submit(*b2)
    g.close()
    again = pp.Group(n, starts, [0] * 3, region_cap=cap)
    stream(again, [(cs, cd, None, 1)])
    assert group_checksum(again) == before
    again.close()


# The witness runs in a child process (see test_gpu_group_traversal.py).  It maps every kernel and copy of the trace to
# the cudaLaunchKernel / cudaMemcpyAsync call that enqueued it (same correlation id) for the launch timestamp.
WITNESS = r"""
import importlib, json, os, sys, tempfile
import numpy as np
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")
scale, P = 16, 4
n = 1 << scale
cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
rng = np.random.default_rng(1)
b = [(rng.integers(0, n, 400000).astype(np.uint32), rng.integers(0, n, 400000).astype(np.uint32)) for _ in range(2)]
g = pp.Group(n, np.linspace(0, n, P + 1).astype(np.uint64), [0] * P, region_cap=cs.size // P + 1)
g.apply(cs, cd)
for s, d in b:  # the first submits allocate
    g.wait(g.submit(s, d))
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    t0 = g.submit(*b[0])
    t1 = g.submit(*b[1])
    g.wait(t0)
    g.wait(t1)
    torch.cuda.synchronize()
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
launch = {e["args"]["correlation"]: e["ts"] for e in events
          if e.get("cat") == "cuda_runtime" and "correlation" in e.get("args", {})}
kernels, copies = [], []
for e in events:
    a = e.get("args", {})
    if e.get("cat") == "kernel" and a.get("correlation") in launch:
        kernels.append([e["name"], a.get("stream"), launch[a["correlation"]]])
    elif e.get("cat") == "gpu_memcpy" and "HtoD" in e["name"] and a.get("correlation") in launch:
        copies.append([int(a.get("bytes", 0)), a.get("stream"), launch[a["correlation"]]])
print(json.dumps({"P": P, "kernels": kernels, "copies": copies, "slice_bytes": 400000 // P * 4}))
g.close()
"""


def test_routing_runs_beside_the_apply():
    """torch.profiler (in a child process): the slices' H2D copies and k_bin_scatter_peers run on streams other than the
    shards' apply streams, and batch i+1's routing kernels are launched before batch i's first apply kernel."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", WITNESS, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    if not res["kernels"]:
        warnings.warn("torch.profiler recorded no kernels in the child process; stream witness skipped")
        return
    P = res["P"]
    routing = sorted((k for k in res["kernels"] if "k_bin_scatter_peers" in k[0]), key=lambda k: k[2])
    apply_k = [k for k in res["kernels"] if "k_bin_scatter_peers" not in k[0] and "k_publish_peer_counts" not in k[0]]
    assert len(routing) == 2 * P, [k[0] for k in res["kernels"]]
    assert apply_k
    apply_streams = {k[1] for k in apply_k}
    assert len(apply_streams) == P, apply_streams
    assert not {k[1] for k in routing} & apply_streams
    slices = [c for c in res["copies"] if c[0] == res["slice_bytes"]]
    assert len(slices) == 2 * 2 * P, res["copies"]  # src and dst of every sender, two batches
    assert not {c[1] for c in slices} & apply_streams
    second = routing[P:]
    assert max(k[2] for k in second) < min(k[2] for k in apply_k), (second, sorted(k[2] for k in apply_k)[:3])


def test_distinct_devices(graph14):
    L = pp.load_library()
    if L.ppcsr_device_count() < 2:
        pytest.skip("needs two GPUs: the shards on distinct devices")
    n, batches = graph14["n"], graph14["batches"]
    k = min(4, L.ppcsr_device_count())
    starts = random_starts(n, k, seed=21)
    g, twin = make_group(n, starts, batches, list(range(k))), make_group(n, starts, batches, list(range(k)))
    assert_same_counters(stream(g, batches), apply_each(twin, batches))
    assert_same_graph(g, twin)
    assert_matches_single(g, graph14["single"])
    g.close()
    twin.close()


def test_cli_batches(tmp_path):
    """-batches=5 prints the Graph checksum and not-found lines of -batches=1, for one shard and for a partitioned
    graph; -batches=0 and a non-number exit 1."""
    build.build_host()
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    rng = np.random.default_rng(3)
    idx = synth.sample_without_replacement(16 << scale, 15000, 7)
    us = np.concatenate([cs[idx], rng.integers(0, n, 5000)])
    ud = np.concatenate([cd[idx], rng.integers(0, n, 5000)])
    op = (rng.random(us.size) < 0.7).astype(np.uint32) ^ 1  # mostly deletes (op 0), some re-inserts
    core, upd = str(tmp_path / "core.bin"), str(tmp_path / "upd.bin3")
    np.stack([cs, cd], axis=1).astype("<u4").tofile(core)
    np.stack([us, ud, op], axis=1).astype("<u4").tofile(upd)
    pick = lambda lines, p: [l for l in lines if l.startswith(p)]
    for mode in (["-ppcsr"], ["-pppcsr", "-partitions_per_domain=4"]):
        out = []
        for k in (1, 5):
            cmd = [build.CLI, "-threads=8", "-size=20000", *mode, "-check", "-checksum", f"-batches={k}",
                   f"-core_graph={core}", f"-update_file={upd}"]
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
            out.append(r.stdout.splitlines())
        for p in ("Graph checksum: ", "not found ", "PMA invariants: ok"):
            assert pick(out[0], p) and pick(out[0], p) == pick(out[1], p), (mode, p)
        assert len(pick(out[1], "Elapsed wall clock time: ")) == 2
    for bad in ("-batches=0", "-batches=x", "-batches=3x"):
        r = subprocess.run([build.CLI, bad, f"-core_graph={core}", f"-update_file={upd}"], capture_output=True,
                           text=True, timeout=60)
        assert r.returncode == 1 and "batches" in r.stdout, (bad, r.stdout[-500:])
