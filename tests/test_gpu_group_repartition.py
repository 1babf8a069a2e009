"""Repartitioning a live group (ppcsr_group_repartition) and loading a shard from a CSR (ppcsr_load_csr).

A repartition changes the owners only, so everything that describes the logical graph must stay exactly as it was: the
summed checksum of the shards, the exports concatenated over the shards (rowptr, col, val) and num_neighbors, BFS, and
PageRank to rtol 1e-9.  The moved vertex and edge counts are checked against numpy's count from the exported rowptr.
Groups of 1 to 8 shards share GPU 0 here; the distinct-device case needs two GPUs and skips otherwise."""
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
RTOL = 1e-9
MASK64 = (1 << 64) - 1


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def scale14_batches(scale=14):
    """R-MAT core, uniform inserts, edges with dst >= n, then a delete batch of core edges."""
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, 20000, 7)
    rng = np.random.default_rng(11)
    xs, xd = rng.integers(0, n, 600), n + rng.integers(0, 4000, 600)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    return n, [(cs, cd, 1), (us, ud, 1), (xs, xd, 1), (cs[idx], cd[idx], 0)]


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
    """The cut rule of the CLI's -balanced / -repartition: partitions of about equal edge counts."""
    n = rowptr.size - 1
    deg = np.diff(rowptr.astype(np.int64))
    total, run, starts, p = int(deg.sum()), 0, [0] * k, 1
    for v in range(n):
        if p >= k:
            break
        run += int(deg[v])
        while p < k and run * k >= total * p:
            starts[p] = min(max(v + 1, starts[p - 1] + 1), n - (k - p))
            p += 1
    for q in range(p, k):
        starts[q] = min(starts[q - 1] + 1, n - (k - q))
    return np.array(starts + [n], np.uint64)


def disjoint_starts(cur, n):
    """New boundaries under which one shard (k >= 3) gets a range disjoint from its old one: shard 1 moves past its old
    end, or else shard k - 2 moves before its old start."""
    k = cur.size - 1
    cur = cur.astype(np.int64)
    if k == 1:
        return cur.astype(np.uint64)
    if k == 2:
        return np.array([0, int(cur[1]) // 2 + 1, n], np.uint64)
    if n - int(cur[2]) >= k:
        new = np.concatenate([[0], np.linspace(cur[2], n, k).astype(np.int64)])
        assert new[1] >= cur[2]
    else:
        new = np.concatenate([np.linspace(0, cur[k - 2], k).astype(np.int64), [n]])
        assert new[k - 1] <= cur[k - 2]
    assert np.all(np.diff(new) > 0)
    return new.astype(np.uint64)


def make_group(n, starts, batches, devices=None):
    k = len(starts) - 1
    cap = max(int(np.asarray(s).size) for s, _, _ in batches) // k + 1
    return pp.Group(n, starts, devices or [0] * k, region_cap=cap, with_values=True)


def apply_all(targets, batches):
    for s, d, v in batches:
        for t in targets:
            t.apply(s, d, np.broadcast_to(np.asarray(v, np.uint32), np.asarray(s).shape))


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


def expected_moves(rowptr, old, new):
    n = rowptr.size - 1
    v = np.arange(n)
    o_old = np.searchsorted(old[:-1].astype(np.int64), v, side="right") - 1
    o_new = np.searchsorted(new[:-1].astype(np.int64), v, side="right") - 1
    moved = o_old != o_new
    deg = np.diff(rowptr.astype(np.int64))
    return int(moved.sum()), int(deg[moved].sum())


def assert_clean(g, where=""):
    for r, sh in enumerate(g.shards):
        geo = sh.geometry
        dens = geo.items / geo.N
        lower = 0.25 <= dens < 0.75  # at the 32-slot floor the density may legitimately be lower
        assert not sh.check(True).violations(lower), (where, r, dens, sh.check(True).as_dict())


def last_stats(sh):
    st = pp.BatchStats()
    pp._check(sh.L.ppcsr_last_stats(sh.h, st))
    return st.as_dict()


def assert_same_ranks(got, want, where=""):
    assert got.shape == want.shape, where
    assert np.array_equal(np.isnan(got), np.isnan(want)), where
    fin = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), fin), where
    assert np.allclose(got[fin], want[fin], rtol=RTOL, atol=0.0), (where, np.max(np.abs(got[fin] - want[fin])))


def repartition_and_check(g, new, ref, where):
    """One step of a chain: the logical graph (ref) is unchanged, the stats count what numpy counts."""
    old = g.starts.copy()
    old[-1] = g.n
    changed = sum(int(old[r] != new[r] or old[r + 1] != new[r + 1]) for r in range(len(g.shards)))
    st = g.repartition(new)
    assert np.array_equal(g.starts, new), where
    assert [sh.n for sh in g.shards] == list(np.diff(new.astype(np.int64))), where
    assert st["shards_rebuilt"] == changed, (where, st)
    assert (st["vertices_moved"], st["edges_moved"]) == expected_moves(ref["rowptr"], old, new), (where, st)
    assert st["ms_total"] > 0, where
    assert group_checksum(g) == ref["checksum"], where
    got = group_export(g)
    for a, b, name in zip(got, (ref["rowptr"], ref["col"], ref["val"], ref["nn"]), ("rowptr", "col", "val", "nn")):
        assert np.array_equal(a, b), (where, name)
    assert_clean(g, where)
    for s in ref["bfs_starts"]:
        assert np.array_equal(g.bfs(s), ref["bfs"][s]), (where, s)
    assert_same_ranks(g.pagerank(20, 0.85), ref["pr"], where)
    return st


# The kernel witness runs in a child process: once torch.profiler has been started in a process, later profiler
# sessions there can miss the first kernels they should record (see test_gpu_group_traversal.py).  It reads the
# memcpy sizes from the exported trace.
WITNESS = r"""
import importlib, json, os, sys, tempfile
import numpy as np
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")
scale = 16
n = 1 << scale
cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
g = pp.Group(n, np.linspace(0, n, 5).astype(np.uint64), [0] * 4, region_cap=cs.size // 4 + 1)
g.apply(cs, cd)
torch.cuda.synchronize()
new = np.array([0, n // 8, n // 4, n // 2, n], np.uint64)
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    st = g.repartition(new)
    torch.cuda.synchronize()
names = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "k_" in e.name})
host = dev = 0
with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
for e in events:
    if e.get("cat") != "gpu_memcpy":
        continue
    b = int(e.get("args", {}).get("bytes", 0))
    if "HtoD" in e["name"] or "DtoH" in e["name"]:
        host += b
    else:
        dev += b
print(json.dumps({"names": names, "host_bytes": host, "device_bytes": dev, "stats": st}))
g.close()
"""


# ------------------------------------------------------------------------------------------------
# scale-14 graph shared by the chain tests
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def graph14():
    n, batches = scale14_batches()
    single = pp.Shard(n)
    apply_all([single], batches)
    rowptr, col, val = single.export(with_values=True)
    nn = single.num_neighbors()
    c = single.checksum(0)
    hub = int(np.argmax(np.diff(rowptr.astype(np.int64))))
    starts = (hub, n // 2, n - 1)
    ref = dict(n=n, batches=batches, rowptr=rowptr, col=col, val=val, nn=nn,
               checksum=(c["edges"], c["edge_hash"], c["nn_hash"]), bfs_starts=starts,
               bfs={s: single.bfs(s) for s in starts}, pr=single.pagerank(20, 0.85))
    assert (col >= n).any()  # edges with dst >= n move with their source
    single.close()
    return ref


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8])
def test_repartition_chain_keeps_the_logical_graph(graph14, k):
    """equal -> edge-balanced -> random with a one-vertex shard -> a shard's range disjoint from its old one -> back
    to the start."""
    n = graph14["n"]
    start = equal_starts(n, k)
    g = make_group(n, start, graph14["batches"])
    apply_all([g], graph14["batches"])
    assert group_checksum(g) == graph14["checksum"]
    chain = [balanced_starts(graph14["rowptr"], k), random_starts(n, k, seed=k)]
    chain.append(disjoint_starts(chain[-1], n))
    chain.append(start)
    moved_any = False
    for i, new in enumerate(chain):
        st = repartition_and_check(g, new, graph14, (k, i))
        moved_any |= st["vertices_moved"] > 0
        if st["shards_rebuilt"]:
            rebuilt = [sh for r, sh in enumerate(g.shards) if last_stats(sh)["whole_array"] == 1]
            assert rebuilt
            ls = last_stats(rebuilt[0])
            assert ls["rebalance_bytes"] > 0 and ls["slots_after"] == rebuilt[0].geometry.N
    assert moved_any == (k > 1)
    g.close()


def test_updates_after_repartition_match_a_single_shard(graph14):
    """Inserts and deletes on moved vertices, value overwrites and mixed batches after a repartition: the group keeps
    matching one shard fed the same batches."""
    n, batches = graph14["n"], graph14["batches"]
    start = equal_starts(n, 4)
    g = make_group(n, start, batches)
    single = pp.Shard(n)
    apply_all([g, single], batches)
    new = balanced_starts(graph14["rowptr"], 4)
    st = g.repartition(new)
    assert st["vertices_moved"] > 0
    old_owner = np.searchsorted(start[:-1].astype(np.int64), np.arange(n), side="right") - 1
    new_owner = np.searchsorted(new[:-1].astype(np.int64), np.arange(n), side="right") - 1
    moved = np.flatnonzero(old_owner != new_owner)
    rng = np.random.default_rng(5)
    rowptr, col = graph14["rowptr"], graph14["col"]
    src_all = np.repeat(np.arange(n), np.diff(rowptr.astype(np.int64)))
    on_moved = np.flatnonzero(np.isin(src_all, moved))
    pick = rng.choice(on_moved, 8000, replace=False)
    ins_s = rng.choice(moved, 20000)
    upd = [
        (ins_s, rng.integers(0, n + 100, 20000), 1),                                   # inserts on moved vertices
        (src_all[pick[:4000]], col[pick[:4000]], 0),                                   # deletes on moved vertices
        (src_all[pick[4000:]], col[pick[4000:]], rng.integers(1, 1 << 20, 4000)),       # value overwrites
        (rng.integers(0, n, 60000), rng.integers(0, n, 60000), rng.integers(0, 3, 60000)),  # mixed ops, 0 = remove
    ]
    for i, b in enumerate(upd):
        apply_all([g, single], [b])
        rp, c, v, nn = group_export(g)
        srp, sc, sv = single.export(with_values=True)
        assert np.array_equal(rp, srp) and np.array_equal(c, sc) and np.array_equal(v, sv), i
        assert np.array_equal(nn, single.num_neighbors()), i
        sc0 = single.checksum(0)
        assert group_checksum(g) == (sc0["edges"], sc0["edge_hash"], sc0["nn_hash"]), i
        for r, sh in enumerate(g.shards):
            assert not sh.check(False).violations(False), (i, r)
    g.close()
    single.close()


def test_growth_of_the_last_shard_is_spread_out():
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    g = make_group(n, equal_starts(n, 3), [(cs, cd, 1)])
    single = pp.Shard(n)
    apply_all([g, single], [(cs, cd, 1)])
    assert g.bfs(0).shape == (n,)  # traversal buffers exist for the old sizes
    extra = 600
    g.shards[-1].add_nodes(extra)
    single.add_nodes(extra)
    m = n + extra
    rng = np.random.default_rng(3)
    grow = [(rng.integers(0, n, 5000), rng.integers(n, m, 5000), 1), (rng.integers(n, m, 5000), rng.integers(0, m, 5000), 1)]
    apply_all([g, single], grow)
    assert g.n == m
    new = equal_starts(m, 3)
    st = g.repartition(new)
    assert st["shards_rebuilt"] == 3 and st["vertices_moved"] > 0
    assert [sh.n for sh in g.shards] == list(np.diff(new.astype(np.int64)))
    rp, c, v, nn = group_export(g)
    srp, sc, sv = single.export(with_values=True)
    assert np.array_equal(rp, srp) and np.array_equal(c, sc) and np.array_equal(v, sv)
    assert np.array_equal(nn, single.num_neighbors())
    for s in (0, n + 5, m - 1):
        assert np.array_equal(g.bfs(s), single.bfs(s)), s
    assert_same_ranks(g.pagerank(20, 0.85), single.pagerank(20, 0.85))
    assert_clean(g)
    g.close()
    single.close()


def test_identity_and_misuse():
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    starts = equal_starts(n, 4)
    g = make_group(n, starts, [(cs, cd, 1)])
    apply_all([g], [(cs, cd, 1)])
    dumps = [sh.debug_dump() for sh in g.shards]
    before = group_checksum(g)
    st = g.repartition(starts)
    assert st["shards_rebuilt"] == 0 and st["vertices_moved"] == 0 and st["edges_moved"] == 0
    for d0, sh in zip(dumps, g.shards):
        assert all(np.array_equal(a, b) for a, b in zip(d0, sh.debug_dump()))
    L = pp.load_library()
    bad = [
        np.array([1, 1000, 2000, 3000, n], np.uint64),        # first entry not 0
        np.array([0, 1000, 2000, 3000, n - 1], np.uint64),    # last entry not n
        np.array([0, 1000, 1000, 3000, n], np.uint64),        # not strictly increasing
        np.array([0, 2000, 1000, 3000, n], np.uint64),        # decreasing
    ]
    for b in bad:
        assert L.ppcsr_group_repartition(g.g, pp._np_ptr(b), None) == -2, b
        assert group_checksum(g) == before
        assert np.array_equal(g.starts, starts)
    assert L.ppcsr_group_repartition(None, pp._np_ptr(starts), None) == -2
    assert L.ppcsr_group_repartition(g.g, None, None) == -2
    g.shards[1].add_nodes(1)  # a shard other than the last no longer matches its range
    after_growth = [sh.checksum(0) for sh in g.shards]
    with pytest.raises(pp.PpcsrError, match="vertex range"):
        g.repartition(np.array([0, 500, 1500, 2500, n + 1], np.uint64))
    assert [sh.checksum(0) for sh in g.shards] == after_growth
    g.close()


def test_load_csr_round_trip_and_rejects_invalid_input(graph14):
    n = graph14["n"]
    src = pp.Shard(n)
    apply_all([src], graph14["batches"])
    rowptr, col, val = src.export(with_values=True)
    nn = src.num_neighbors()
    dst = pp.Shard(10)  # a different size: the content is replaced whole
    st = dst.load_csr(rowptr, col, val, nn)
    assert st["whole_array"] == 1 and st["ms_rebalance_kernel"] > 0
    assert dst.n == n
    got = dst.export(with_values=True)
    assert all(np.array_equal(a, b) for a, b in zip(got, (rowptr, col, val)))
    assert np.array_equal(dst.num_neighbors(), nn)
    assert dst.checksum(0) == src.checksum(0)
    assert not dst.check(True).violations(True), dst.check(True).as_dict()
    # defaults: every value 1, num_neighbors = row lengths; then updates keep working on the loaded layout
    small = pp.Shard(5)
    small.load_csr(np.array([0, 2, 2, 3], np.uint64), np.array([1, 7, 0], np.uint32))
    assert small.n == 3
    assert small.edge_value(0, 7) == 1 and list(small.num_neighbors()) == [2, 0, 1]
    small.apply([1, 0], [2, 1], [5, 0])
    r, c, v = small.export(with_values=True)
    assert list(r) == [0, 1, 2, 3] and list(c) == [7, 2, 0] and list(v) == [1, 5, 1]
    # invalid input: PpcsrError, shard untouched
    good_r, good_c = np.array([0, 2, 3, 5], np.uint64), np.array([1, 4, 2, 0, 3], np.uint32)
    invalid = [
        (np.array([1, 2, 3, 5], np.uint64), good_c, None),           # rowptr[0] != 0
        (np.array([0, 3, 2, 5], np.uint64), good_c, None),           # rowptr decreases
        (good_r, np.array([4, 1, 2, 0, 3], np.uint32), None),        # row not ascending
        (good_r, np.array([1, 4, 2, 3, 3], np.uint32), None),        # duplicate in a row
        (good_r, np.array([1, 4, 2, 0, pp.SENT], np.uint32), None),  # the sentinel marker
        (good_r, good_c, np.array([1, 1, 0, 1, 1], np.uint32)),      # a value 0
    ]
    before_ck, before_dump = dst.checksum(0), dst.debug_dump()
    for i, (r_, c_, v_) in enumerate(invalid):
        with pytest.raises(pp.PpcsrError):
            dst.load_csr(r_, c_, v_)
        assert dst.checksum(0) == before_ck, i
        assert all(np.array_equal(a, b) for a, b in zip(before_dump, dst.debug_dump())), i
    dst.load_csr(good_r, good_c)  # the same arrays pass once they are valid
    assert dst.n == 3 and dst.checksum(0)["edges"] == 5
    for sh in (src, dst, small):
        sh.close()


def test_scale20_over_eight_parts():
    """The C4 core at scale 20 over 8 shards: equal -> edge-balanced -> equal."""
    scale = 20
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    eq = equal_starts(n, 8)
    g = make_group(n, eq, [(cs, cd, 1)])
    apply_all([g], [(cs, cd, 1)])
    before = group_checksum(g)
    rowptr = group_export(g)[0]
    bal = balanced_starts(rowptr, 8)
    e_before = [sh.checksum(0)["edges"] for sh in g.shards]
    for new in (bal, eq):
        st = g.repartition(new)
        assert st["shards_rebuilt"] > 0 and st["edges_moved"] > 0
        assert group_checksum(g) == before
        assert_clean(g, "scale20")
        if new is bal:
            e = [sh.checksum(0)["edges"] for sh in g.shards]
            assert max(e) < max(e_before)
    g.close()


def test_cli_repartition(tmp_path):
    """-repartition keeps the checksum and BFS lines and PageRank to 1e-9, and prints its Repartition line."""
    build.build_host()
    scale = 12
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    core, upd = str(tmp_path / "core.bin"), str(tmp_path / "upd.bin")
    np.stack([cs, cd], axis=1).astype("<u4").tofile(core)
    np.stack([cs[idx], cd[idx]], axis=1).astype("<u4").tofile(upd)
    out = []
    for extra in ([], ["-repartition"]):
        cmd = [build.CLI, "-threads=8", "-delete", "-size=20000", "-pppcsr", "-partitions_per_domain=4", "-check",
               "-checksum", *extra, f"-core_graph={core}", f"-update_file={upd}", "-bfs=0", "-pagerank=5"]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        out.append(r.stdout.splitlines())
    pick = lambda lines, p: [l for l in lines if l.startswith(p)]
    for p in ("Graph checksum: ", "BFS from 0: reached ", "PMA invariants: ok"):
        assert pick(out[0], p) and pick(out[0], p) == pick(out[1], p), p
    pr = [pick(o, "PageRank 5 iterations: sum ")[0].split() for o in out]
    assert np.isclose(float(pr[1][4]), float(pr[0][4]), rtol=RTOL, atol=0)
    assert np.isclose(float(pr[1][6]), float(pr[0][6]), rtol=RTOL, atol=0)
    assert not pick(out[0], "Repartition: ")
    line = pick(out[1], "Repartition: moved ")
    assert line and int(line[0].split()[2]) > 0, out[1][-10:]


def test_edges_move_device_to_device():
    """torch.profiler (in a child process) sees the layout kernel, megabytes copied between device buffers and under
    64 KB copied between host and device during one repartition."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", WITNESS, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    st = res["stats"]
    assert st["edges_moved"] * 8 > 1 << 20, st  # col + val of the moved edges: megabytes
    if not res["names"]:
        warnings.warn("torch.profiler recorded no kernels in the child process; kernel witness skipped")
        return
    for k in ("k_layout_from_csr", "k_rebase_rowptr", "k_rowptr"):
        assert any(k in x for x in res["names"]), (k, res["names"])
    # a trace that recorded the kernels records the copies of the same CUDA activity: the moved edges must be there
    assert res["device_bytes"] >= st["edges_moved"] * 8, res
    assert res["host_bytes"] < 64 << 10, res


def test_distinct_devices(graph14):
    L = pp.load_library()
    if L.ppcsr_device_count() < 2:
        pytest.skip("needs two GPUs: the shards on distinct devices")
    n = graph14["n"]
    k = min(4, L.ppcsr_device_count())
    g = make_group(n, equal_starts(n, k), graph14["batches"], devices=list(range(k)))
    apply_all([g], graph14["batches"])
    repartition_and_check(g, balanced_starts(graph14["rowptr"], k), graph14, "devices")
    repartition_and_check(g, random_starts(n, k, seed=4), graph14, "devices")
    g.close()
