"""Vertex isolation (ppcsr_isolate_vertices / ppcsr_group_isolate_vertices, csrc/isolate.cuh).

Isolating a set S must equal ONE remove batch of exactly the live edges (u, w) with u or w in S: against the oracle
(remove_edge per incident edge), against a twin shard that applies that remove batch (identical physical layout under
a forced window policy), and, across the shards of a group, against a single shard holding the whole graph."""
import importlib
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

import oracle_py as O

pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")

pytestmark = pytest.mark.gpu
MASK64 = (1 << 64) - 1


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def scale14_batches(scale=14):
    """R-MAT core with values, uniform inserts, edges with dst >= n, then a delete batch of core edges."""
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, 20000, 7)
    rng = np.random.default_rng(11)
    xs, xd = rng.integers(0, n, 600), n + rng.integers(0, 4000, 600)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    cv = rng.integers(1, 1 << 20, cs.size).astype(np.uint32)
    uv = rng.integers(1, 1 << 20, us.size).astype(np.uint32)
    return n, [(cs, cd, cv), (us, ud, uv), (xs, xd, 7), (cs[idx], cd[idx], 0)]


def apply_all(targets, batches):
    for s, d, v in batches:
        for t in targets:
            t.apply(s, d, np.broadcast_to(np.asarray(v, np.uint32), np.asarray(s).shape))


def incident(rowptr, col, ids):
    """The live edges (u, w) with u in ids or w in ids (w < n), in CSR order."""
    n = rowptr.size - 1
    mark = np.zeros(n, bool)
    mark[np.asarray(ids, np.int64)] = True
    src = np.repeat(np.arange(n, dtype=np.uint32), np.diff(rowptr).astype(np.int64))
    hit = mark[src] | ((col < n) & mark[np.minimum(col, n - 1).astype(np.int64)])
    return src[hit], col[hit]


def equal_starts(n, k):
    return np.linspace(0, n, k + 1).astype(np.uint64)


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


def balanced_starts(rowptr, k):
    """Partitions of about equal edge counts, every one non-empty."""
    n = rowptr.size - 1
    cum = rowptr[1:].astype(np.int64)
    starts = [0]
    for p in range(1, k):
        v = int(np.searchsorted(cum, cum[-1] * p // k)) + 1
        starts.append(min(max(v, starts[-1] + 1), n - (k - p)))
    return np.array(starts + [n], np.uint64)


def group_checksum(g):
    out = [0, 0, 0]
    for r, sh in enumerate(g.shards):
        c = sh.checksum(int(g.starts[r]))
        out = [(out[0] + c["edges"]) & MASK64, (out[1] + c["edge_hash"]) & MASK64, (out[2] + c["nn_hash"]) & MASK64]
    return tuple(out)


def shard_checksum(sh):
    c = sh.checksum()
    return (c["edges"], c["edge_hash"], c["nn_hash"])


def assert_matches_oracle(sh, o, where=""):
    rp, c, v = sh.export(with_values=True)
    orp, oc, onn = o.export()
    assert np.array_equal(rp, orp) and np.array_equal(c, oc), where
    assert np.array_equal(v, o.export_values()), where
    assert np.array_equal(sh.num_neighbors(), onn), where
    assert sh.n == o.n, where
    rep = sh.check(True)
    assert not rep.violations(True), (where, rep.as_dict())


# ------------------------------------------------------------------------------------------------
# one shard against the reference and against a twin remove batch
# ------------------------------------------------------------------------------------------------
def id_sets(rowptr, col, n):
    """leaf vertex, top hub, 1 % random with duplicates, 30 % random, every vertex"""
    outdeg = np.diff(rowptr).astype(np.int64)
    indeg = np.bincount(col[col < n].astype(np.int64), minlength=n)
    leaf = int(np.flatnonzero((outdeg == 1) & (indeg >= 1))[0])
    rng = np.random.default_rng(5)
    some = rng.integers(0, n, n // 100)
    some = np.concatenate([some, some[: some.size // 4]])
    return [("leaf", [leaf]), ("hub", [int(np.argmax(outdeg))]), ("1%", some),
            ("30%", rng.choice(n, int(n * 0.3), replace=False)), ("all", np.arange(n))]


@pytest.mark.parametrize("policy", [-1, 0, 1])
def test_isolation_matches_the_reference(policy):
    n, batches = scale14_batches()
    sh = pp.Shard(n)
    sh.set_whole_array_policy(policy)
    o = O.OraclePCSR(n)
    apply_all([sh, o], batches)
    assert_matches_oracle(sh, o, "before")
    rowptr, col = sh.export()
    resized = False
    for name, ids in id_sets(rowptr, col, n):
        rowptr, col = sh.export()
        s, d = incident(rowptr, col, ids)
        st = sh.isolate_vertices(ids)
        o.apply(s, d, 0)
        assert_matches_oracle(sh, o, (policy, name))
        assert st["batch_size"] == len(ids) and st["n_unique"] == np.unique(ids).size, (name, st)
        assert st["n_deleted"] == s.size and st["n_inserted"] == 0, (name, st)
        last = pp.BatchStats()
        pp._check(sh.L.ppcsr_last_stats(sh.h, pp.C.byref(last)))
        assert last.as_dict() == st, name
        if policy == 1 and s.size:
            assert st["whole_array"] == 1, st
        resized |= st["resized"] == 2
    rp, c = sh.export()
    assert rp[-1] == 0 and c.size == 0  # sentinels only
    assert resized, "the 30 % set should have shrunk the array"
    sh.close()


def test_isolation_equals_a_twin_remove_batch():
    """Under a forced policy the back half sees the same tombstones and counts as for the remove batch of the same
    edges: the physical layouts are identical (whenever the twin's batch did not take the small-batch path)."""
    n, batches = scale14_batches()
    paths = set()
    for policy in (-1, 1):
        a, b = pp.Shard(n), pp.Shard(n)
        for sh in (a, b):
            sh.set_whole_array_policy(policy)
        apply_all([a, b], batches)
        rowptr, col = a.export()
        for name, ids in id_sets(rowptr, col, n)[:4]:
            rowptr, col = a.export()
            s, d = incident(rowptr, col, ids)
            sa = a.isolate_vertices(ids)
            sb = b.apply(s, d, 0)
            assert sa["n_deleted"] == sb["n_deleted"] == s.size, (policy, name)
            assert shard_checksum(a) == shard_checksum(b), (policy, name)
            if sb["sparse_path"] == 0:
                for x, y in zip(a.debug_dump(), b.debug_dump()):
                    assert np.array_equal(x, y), (policy, name)
                assert (sa["whole_array"], sa["n_windows"], sa["resized"]) == \
                       (sb["whole_array"], sb["n_windows"], sb["resized"]), (policy, name, sa, sb)
                paths.add("whole" if sa["whole_array"] else "windows")
        a.close()
        b.close()
    assert paths == {"whole", "windows"}, paths


def test_updates_restore_and_misuse_after_isolation():
    n, batches = scale14_batches()
    sh = pp.Shard(n)
    o = O.OraclePCSR(n)
    apply_all([sh, o], batches)
    before = shard_checksum(sh)
    sh.snapshot()
    rowptr, col = sh.export()
    hub = int(np.argmax(np.diff(rowptr)))
    ids = [hub, 3, 77, 77]
    s, d = incident(rowptr, col, ids)
    sh.isolate_vertices(ids)
    o.apply(s, d, 0)
    assert_matches_oracle(sh, o, "isolated")
    # isolating them again finds nothing: the batch back half's "nothing moves" branch, stats included
    isolated = shard_checksum(sh)
    st = sh.isolate_vertices(ids)
    assert st["n_deleted"] == 0 and st["n_windows"] == 0 and st["whole_array"] == 0, st
    assert st["ms_total"] >= st["ms_rebalance_kernel"] >= 0.0, st
    assert shard_checksum(sh) == isolated
    assert_matches_oracle(sh, o, "isolated twice")
    # edges at the isolated vertices come back; more removes and inserts elsewhere
    rng = np.random.default_rng(3)
    rs = np.concatenate([np.full(500, hub), rng.integers(0, n, 3000), rng.integers(0, n, 200)])
    rd = np.concatenate([rng.integers(0, n, 500), np.full(3000, 77), rng.integers(0, n, 200)])
    rv = rng.integers(1, 1000, rs.size).astype(np.uint32)
    for bs, bd, bv in ((rs, rd, rv), (s[: s.size // 2], d[: d.size // 2], 9), (rs[::3], rd[::3], 0)):
        sh.apply(bs, bd, np.broadcast_to(np.asarray(bv, np.uint32), bs.shape))
        o.apply(bs, bd, bv)
        assert_matches_oracle(sh, o, "after")
    after = shard_checksum(sh)
    # an empty list changes nothing; an id >= n (or the sentinel marker) raises and changes nothing
    st = sh.isolate_vertices([])
    assert st["batch_size"] == 0 and st["n_deleted"] == 0
    assert shard_checksum(sh) == after
    for bad in ([n], [0, n + 5], [0xFFFFFFFF]):
        with pytest.raises(pp.PpcsrError):
            sh.isolate_vertices(bad)
        assert shard_checksum(sh) == after
    L = pp.load_library()
    assert L.ppcsr_isolate_vertices(None, None, 0, None) == -2
    assert L.ppcsr_isolate_vertices(sh.h, None, 3, None) == -2
    sh.restore()
    assert shard_checksum(sh) == before
    assert not sh.check(False).violations(False)
    sh.close()


# ------------------------------------------------------------------------------------------------
# groups
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def graph14():
    n, batches = scale14_batches()
    single = pp.Shard(n)
    apply_all([single], batches)
    rowptr, col = single.export()
    rng = np.random.default_rng(17)
    outdeg = np.diff(rowptr).astype(np.int64)
    ids = np.concatenate([rng.integers(0, n, n // 100), [int(np.argmax(outdeg)), n - 1]])
    st = single.isolate_vertices(ids)
    yield dict(n=n, batches=batches, rowptr=rowptr, ids=ids, single=single, st=st)
    single.close()


def make_group(n, starts, batches, devices=None):
    k = len(starts) - 1
    cap = max(int(np.asarray(s).size) for s, _, _ in batches) // k + 1
    return pp.Group(n, starts, devices or [0] * k, region_cap=cap, with_values=True)


def assert_group_equals_single(g, single, where=""):
    assert group_checksum(g) == shard_checksum(single), where
    assert np.array_equal(np.concatenate([sh.num_neighbors() for sh in g.shards]), single.num_neighbors()), where
    for start in (0, int(g.starts[-2])):
        assert np.array_equal(g.bfs(start), single.bfs(start)), (where, start)
    got, want = g.pagerank(10, 0.85), single.pagerank(10, 0.85)
    assert np.array_equal(np.isfinite(got), np.isfinite(want)), where
    fin = np.isfinite(want)
    assert np.allclose(got[fin], want[fin], rtol=1e-9, atol=0), where
    for sh in g.shards:
        assert not sh.check(True).violations(sh.n > 1), where


@pytest.mark.parametrize("k", [1, 2, 3, 8])
@pytest.mark.parametrize("cut", ["equal", "balanced", "random"])
def test_group_isolation_matches_a_single_shard(graph14, k, cut):
    n = graph14["n"]
    starts = {"equal": equal_starts(n, k), "balanced": balanced_starts(graph14["rowptr"], k),
              "random": random_starts(n, k, seed=k)}[cut]
    g = make_group(n, starts, graph14["batches"])
    apply_all([g], graph14["batches"])
    sts = g.isolate_vertices(graph14["ids"])
    assert len(sts) == k
    assert sum(st["n_deleted"] for st in sts) == graph14["st"]["n_deleted"] > 0
    for st in sts:
        assert st["batch_size"] == graph14["ids"].size and st["n_unique"] == graph14["st"]["n_unique"]
    assert_group_equals_single(g, graph14["single"], (k, cut))
    g.close()


def test_group_growth_misuse_and_streaming():
    n, batches = scale14_batches(12)
    starts = random_starts(n, 3, seed=4)
    g = make_group(n, starts, batches)
    single = pp.Shard(n)
    apply_all([g, single], batches)
    # a vertex grown onto the last shard, with edges in and out, can be isolated
    g.shards[-1].add_nodes(2)
    single.add_nodes(2)
    s = np.array([n, n, 5, 9, n + 1], np.uint32)
    d = np.array([3, 8, n, n, n], np.uint32)
    apply_all([g, single], [(s, d, 4)])
    sts, st = g.isolate_vertices([n, 17]), single.isolate_vertices([n, 17])
    assert sum(x["n_deleted"] for x in sts) == st["n_deleted"] >= 5
    assert_group_equals_single(g, single, "grown")
    # an id >= n_global is refused with nothing changed
    before = group_checksum(g)
    with pytest.raises(pp.PpcsrError):
        g.isolate_vertices([0, n + 2])
    assert group_checksum(g) == before
    st0 = g.isolate_vertices([])
    assert all(x["n_deleted"] == 0 and x["batch_size"] == 0 for x in st0) and group_checksum(g) == before
    # not while a submitted batch is in flight; submit, wait, isolate, submit, wait equals the single shard
    rng = np.random.default_rng(8)
    b1 = (rng.integers(0, n, 5000).astype(np.uint32), rng.integers(0, n, 5000).astype(np.uint32))
    b2 = (rng.integers(0, n, 5000).astype(np.uint32), rng.integers(0, n, 5000).astype(np.uint32))
    t = g.submit(*b1, default_val=3)
    with pytest.raises(pp.PpcsrError, match="in flight"):
        g.isolate_vertices([1])
    assert group_checksum(g) == before
    g.wait(t)
    single.apply(*b1, default_val=3)
    hub = int(np.argmax(single.export()[0][1:] - single.export()[0][:-1]))
    g.isolate_vertices([hub, 2])
    single.isolate_vertices([hub, 2])
    t = g.submit(*b2, default_val=0)
    g.wait(t)
    single.apply(*b2, default_val=0)
    assert_group_equals_single(g, single, "stream")
    L = pp.load_library()
    assert L.ppcsr_group_isolate_vertices(None, None, 0, None) == -2
    g.close()
    single.close()


def test_distinct_devices(graph14):
    L = pp.load_library()
    if L.ppcsr_device_count() < 2:
        pytest.skip("needs two GPUs: the shards on distinct devices")
    n = graph14["n"]
    k = min(4, L.ppcsr_device_count())
    g = make_group(n, random_starts(n, k, seed=21), graph14["batches"], devices=list(range(k)))
    apply_all([g], graph14["batches"])
    g.isolate_vertices(graph14["ids"])
    assert_group_equals_single(g, graph14["single"], "devices")
    g.close()


# ------------------------------------------------------------------------------------------------
# scale 20: the C4 core, its 1 K largest hubs
# ------------------------------------------------------------------------------------------------
def test_scale20_hubs_equal_export_filter_remove():
    scale = 20
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    one, twin = pp.Shard(n), pp.Shard(n)
    g = make_group(n, equal_starts(n, 8), [(cs, cd, 1)])
    apply_all([one, twin, g], [(cs, cd, 1)])
    rowptr, col = twin.export()
    hubs = np.argsort(np.diff(rowptr).astype(np.int64), kind="stable")[-1024:]
    s, d = incident(rowptr, col, hubs)
    st = one.isolate_vertices(hubs)
    sts = g.isolate_vertices(hubs)
    tw = twin.apply(s, d, 0)
    assert st["n_deleted"] == tw["n_deleted"] == s.size == sum(x["n_deleted"] for x in sts)
    assert shard_checksum(one) == shard_checksum(twin) == group_checksum(g)
    assert np.array_equal(one.num_neighbors(), twin.num_neighbors())
    assert np.array_equal(np.concatenate([sh.num_neighbors() for sh in g.shards]), twin.num_neighbors())
    assert not one.check(True).violations(True)
    for sh in g.shards:
        assert not sh.check(True).violations(True)
    for x in (one, twin, g):
        x.close()


# ------------------------------------------------------------------------------------------------
# kernel witness: the isolate kernels run, no sort pass and no k_locate, no edge data crosses to the host
# ------------------------------------------------------------------------------------------------
# In a child process for the reason test_gpu_group_traversal.py gives: later profiler sessions of the pytest process
# must see every kernel.
WITNESS = r"""
import importlib, json, os, sys, tempfile
sys.path.insert(0, sys.argv[1])
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")
n = 1 << 14
cs, cd = synth.rmat(14, 0, 16 << 14, 42)
ids = np.random.default_rng(1).integers(0, n, 2000).astype(np.uint32)
sh = pp.Shard(n)
sh.apply(cs, cd)
g = pp.Group(n, [0, 5000, 5001, n], [0, 0, 0], region_cap=cs.size // 3 + 1)
g.apply(cs, cd)
torch.cuda.synchronize()
out = {}
for name, call, copies in (("shard", lambda: sh.isolate_vertices(ids), 1),
                           ("group", lambda: g.isolate_vertices(ids), 3)):
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        st = call()
        torch.cuda.synchronize()
    path = os.path.join(tempfile.mkdtemp(), "trace.json")
    prof.export_chrome_trace(path)
    ev = json.load(open(path)).get("traceEvents", [])
    copied = sum(int(e.get("args", {}).get("bytes", 0)) for e in ev if e.get("cat") == "gpu_memcpy"
                 and ("HtoD" in e.get("name", "") or "DtoH" in e.get("name", "")))
    names = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "k_" in e.name})
    out[name] = dict(names=names, copied=copied, limit=copies * ids.nbytes + 65536,
                     deleted=int(st["n_deleted"]) if isinstance(st, dict) else sum(x["n_deleted"] for x in st))
print(json.dumps(out))
g.close()
sh.close()
"""


def test_isolate_kernels_run_and_no_edge_reaches_the_host():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", WITNESS, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    for name, w in out.items():
        assert w["deleted"] > 0, name
        if not w["names"]:
            warnings.warn(f"torch.profiler recorded no kernels in the child process ({name}); kernel witness skipped")
            continue
        for k in ("k_isolate_bitmap", "k_isolate_filter"):
            assert any(k in x for x in w["names"]), (name, k, w["names"])
        for k in ("k_os_pass", "k_os_hist", "k_sort_small", "k_locate", "k_build_keys"):
            assert not any(k in x for x in w["names"]), (name, k, w["names"])
        assert w["copied"] <= w["limit"], (name, w["copied"], w["limit"])
        if w["copied"] == 0:
            warnings.warn(f"the profiler trace gave no copy sizes ({name}); the traffic bound was not checked")
