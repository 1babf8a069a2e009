"""Traversals across the shards of a group (ppcsr_group_bfs / ppcsr_group_pagerank, csrc/traverse.cuh).

BFS distances must equal, exactly, those of ppcsr_bfs on one shard fed the same batches, the oracle's queue BFS and
scipy's unweighted shortest paths on the exported CSR.  PageRank must equal Shard.pagerank and the numpy recurrence of
test_gpu_parity.py::test_iterated_pagerank_matches_numpy to rtol 1e-9, with the same NaN / +inf positions.  Groups of
1 to 8 shards share GPU 0 here; the distinct-device case needs two GPUs and skips otherwise."""
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
build = importlib.import_module("parallel-packed-csr_b200.build")
synth = importlib.import_module("parallel-packed-csr_b200.synth")

pytestmark = pytest.mark.gpu
UNREACHED = 0xFFFFFFFF
RTOL = 1e-9


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


def make_group(n, starts, batches, devices=None):
    k = len(starts) - 1
    cap = max(int(s.size) for s, _, _ in batches) // k + 1
    return pp.Group(n, starts, devices or [0] * k, region_cap=cap, with_values=True)


def apply_all(targets, batches):
    for s, d, v in batches:
        for t in targets:
            t.apply(s, d, np.broadcast_to(np.asarray(v, np.uint32), s.shape))


def scale14_batches(scale=14):
    """R-MAT core, uniform inserts, edges with dst >= n, then a delete batch of core edges."""
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, 20000, 7)
    rng = np.random.default_rng(11)
    xs, xd = rng.integers(0, n, 600), n + rng.integers(0, 4000, 600)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    return n, [(cs, cd, 1), (us, ud, 1), (xs, xd, 1), (cs[idx], cd[idx], 0)]


def scipy_bfs(rowptr, col, n, start):
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import shortest_path

    out = np.full(n, UNREACHED, np.uint32)
    if start >= n:
        return out
    src = np.repeat(np.arange(n), np.diff(rowptr).astype(np.int64))
    keep = col < n
    A = csr_matrix((np.ones(int(keep.sum())), (src[keep], col[keep].astype(np.int64))), shape=(n, n))
    d = shortest_path(A, method="D", unweighted=True, indices=start)
    fin = np.isfinite(d)
    out[fin] = d[fin].astype(np.uint32)
    return out


def numpy_pagerank(rowptr, col, nn, n, iterations, damping):
    src = np.repeat(np.arange(n), np.diff(rowptr).astype(np.int64))
    keep = col < n
    r = np.full(n, 1.0 / n)
    with np.errstate(divide="ignore", invalid="ignore"):
        for _ in range(iterations):
            contrib = r[src] / nn.astype(np.float64)[src]
            r = (1.0 - damping) / n + damping * np.bincount(col[keep].astype(np.int64), weights=contrib[keep],
                                                            minlength=n)
    return r


def assert_same_ranks(got, want, where=""):
    assert got.shape == want.shape, where
    assert np.array_equal(np.isnan(got), np.isnan(want)), where
    assert np.array_equal(np.isposinf(got), np.isposinf(want)), where
    fin = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), fin), where
    assert np.allclose(got[fin], want[fin], rtol=RTOL, atol=0.0), (where, np.max(np.abs(got[fin] - want[fin])))


def checksums(g):
    return [sh.checksum(int(g.starts[r])) for r, sh in enumerate(g.shards)]


# The kernel witness runs in a child process: once torch.profiler has been started in a process, later profiler
# sessions there can miss the first kernels they should record, and the branch witnesses of
# test_gpu_pipeline_branches.py, which run later in the same pytest process, rely on seeing every kernel.
WITNESS = r"""
import importlib, json, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")
n = 1 << 12
cs, cd = synth.rmat(12, 0, 16 << 12, 42)
g = pp.Group(n, [0, 1000, 1001, n], [0, 0, 0], region_cap=cs.size // 3 + 1)
g.apply(cs, cd)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    g.bfs(0)
    g.pagerank(3)
    torch.cuda.synchronize()
print(json.dumps(sorted({e.name for e in prof.events()
                         if e.device_type == torch.autograd.DeviceType.CUDA and "k_" in e.name})))
g.close()
"""


# ------------------------------------------------------------------------------------------------
# scale-14 graph shared by the equality tests
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def graph14():
    n, batches = scale14_batches()
    single = pp.Shard(n)
    o = O.OraclePCSR(n)
    apply_all([single], batches)
    for s, d, v in batches:
        o.apply(s, d, v)
    rowptr, col = single.export()
    nn = single.num_neighbors()
    orp, ocol, onn = o.export()
    assert np.array_equal(rowptr, orp) and np.array_equal(col, ocol) and np.array_equal(nn, onn)
    assert (col >= n).any()  # dst >= n is stored, and skipped by every traversal
    indeg = np.bincount(col[col < n].astype(np.int64), minlength=n)
    outdeg = np.diff(rowptr).astype(np.int64)
    no_in = np.flatnonzero((indeg == 0) & (outdeg > 0))
    assert no_in.size
    yield dict(n=n, batches=batches, single=single, oracle=o, rowptr=rowptr, col=col, nn=nn,
               hub=int(np.argmax(outdeg)), no_in=int(no_in[0]))
    single.close()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8])
def test_group_bfs_matches_single_shard(graph14, k):
    n = graph14["n"]
    starts = random_starts(n, k, seed=k)
    g = make_group(n, starts, graph14["batches"])
    apply_all([g], graph14["batches"])
    assert g.n == n
    for s in (graph14["hub"], int(starts[-2]) + (n - int(starts[-2])) // 2, graph14["no_in"], n - 1, n):
        got = g.bfs(s)
        want = graph14["single"].bfs(s)
        assert got.dtype == np.uint32 and got.shape == (n,)
        assert np.array_equal(got, want), (k, s, int(np.sum(got != want)))
        assert np.array_equal(got, graph14["oracle"].bfs(s)), (k, s)
        assert np.array_equal(got, scipy_bfs(graph14["rowptr"], graph14["col"], n, s)), (k, s)
        if s == n:
            assert np.all(got == UNREACHED)
        if s == graph14["hub"]:
            assert np.sum(got != UNREACHED) > n // 2
    g.close()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8])
def test_group_pagerank_matches_single_shard(graph14, k):
    n = graph14["n"]
    g = make_group(n, random_starts(n, k, seed=10 + k), graph14["batches"])
    apply_all([g], graph14["batches"])
    for it in (0, 1, 20):
        for d in (0.85, 1.0):
            got = g.pagerank(it, d)
            assert got.dtype == np.float64 and got.shape == (n,)
            if it == 0:
                assert np.all(got == 1.0 / n)
            assert_same_ranks(got, graph14["single"].pagerank(it, d), (k, it, d, "shard"))
            want = numpy_pagerank(graph14["rowptr"], graph14["col"], graph14["nn"], n, it, d)
            assert_same_ranks(got, want, (k, it, d, "numpy"))
    g.close()


def test_group_pagerank_zero_and_wrapped_num_neighbors():
    """Vertices with live edges whose num_neighbors is 0 (infinite contributions) or wrapped to 2^32 - 2, built as
    test_pagerank_step_edges does: the NaN and +inf positions equal the single shard's."""
    n = 3000
    rng = np.random.default_rng(9)
    s, d = rng.integers(0, n, 40000), rng.integers(0, n, 40000)
    deg = np.bincount(s, minlength=n)
    zero = np.flatnonzero(deg >= 3)[:20]
    wrap = np.flatnonzero(deg >= 3)[20:40]
    ms = np.concatenate([np.repeat(zero, deg[zero]), np.repeat(wrap, deg[wrap] + 2)])
    batches = [(s, d, 1), (ms, np.full(ms.size, n + 5), 0)]
    single = pp.Shard(n)
    g = make_group(n, random_starts(n, 4, seed=3), batches)
    apply_all([single, g], batches)
    nn = single.num_neighbors()
    assert np.all(nn[zero] == 0) and np.all(nn[wrap] == 0xFFFFFFFE)
    saw_inf = saw_nan = False
    for it in (1, 20):
        for damping in (0.85, 1.0):
            got, want = g.pagerank(it, damping), single.pagerank(it, damping)
            assert_same_ranks(got, want, (it, damping))
            saw_inf |= bool(np.isposinf(got).any())
            saw_nan |= bool(np.isnan(got).any())
    assert saw_inf
    if not saw_nan:
        warnings.warn("no NaN rank arose in this graph; only +inf positions were compared")
    single.close()
    g.close()


def test_interleaved_apply_and_traversals():
    """apply, traverse, apply, traverse on one group: every traversal matches a single shard, a traversal leaves
    every shard's checksum unchanged, and the group's updates still match the oracle afterwards."""
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, 8000, 5)
    idx = synth.sample_without_replacement(16 << scale, 8000, 3)
    batches = [(cs, cd, 1), (us, ud, 1), (cs[idx], cd[idx], 0)]
    starts = random_starts(n, 3, seed=7)
    g = make_group(n, starts, batches)
    single = pp.Shard(n)
    o = O.OraclePCSR(n)
    for s, d, v in batches:
        apply_all([g, single], [(s, d, v)])
        o.apply(s, d, v)
        before = checksums(g)
        for start in (0, int(starts[2])):
            assert np.array_equal(g.bfs(start), single.bfs(start))
        assert_same_ranks(g.pagerank(20, 0.85), single.pagerank(20, 0.85))
        assert checksums(g) == before
    rowptr, col, nn = o.export()
    for r, sh in enumerate(g.shards):
        lo, hi = int(starts[r]), int(starts[r + 1])
        rp, c = sh.export()
        assert np.array_equal(rp, rowptr[lo:hi + 1] - rowptr[lo]), r
        assert np.array_equal(c, col[int(rowptr[lo]):int(rowptr[hi])]), r
        assert np.array_equal(sh.num_neighbors(), nn[lo:hi]), r
        # a one-vertex shard sits in the minimum array, below the lower density bound by construction
        assert not sh.check(True).violations(sh.n > 1), r
    g.close()
    single.close()


def test_growth_of_the_last_shard_and_misuse():
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    batches = [(cs, cd, 1)]
    g = make_group(n, random_starts(n, 3, seed=5), batches)
    single = pp.Shard(n)
    apply_all([g, single], batches)
    assert np.array_equal(g.bfs(0), single.bfs(0))  # the traversal buffers exist for n
    g.shards[-1].add_nodes(5)
    single.add_nodes(5)
    assert g.n == n + 5
    dist = g.bfs(0)
    assert dist.shape == (n + 5,) and np.all(dist[n:] == UNREACHED)
    assert np.array_equal(dist, single.bfs(0))
    assert np.array_equal(g.bfs(n + 2), single.bfs(n + 2))
    for it in (0, 1, 20):
        r = g.pagerank(it, 0.85)
        assert r.shape == (n + 5,)
        base = 1.0 / (n + 5) if it == 0 else 0.15 / (n + 5)
        assert np.allclose(r[n:], base, rtol=1e-15, atol=0)
        assert_same_ranks(r, single.pagerank(it, 0.85), it)
    L = pp.load_library()
    assert L.ppcsr_group_bfs(None, 0, None) == -2 and L.ppcsr_group_pagerank(None, 1, 0.85, None) == -2
    assert L.ppcsr_group_bfs(g.g, 0, None) == -2 and L.ppcsr_group_pagerank(g.g, 1, 0.85, None) == -2
    g.shards[1].add_nodes(1)
    with pytest.raises(pp.PpcsrError, match="vertex range"):
        g.bfs(0)
    with pytest.raises(pp.PpcsrError, match="vertex range"):
        g.pagerank(3)
    g.close()
    single.close()


def test_scale20_over_eight_parts():
    """The C4 core at scale 20 over 8 parts on GPU 0: exact BFS, PageRank to rtol 1e-9, at a size where the inbox
    capacity bound matters."""
    scale = 20
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    batches = [(cs, cd, 1)]
    single = pp.Shard(n)
    g = make_group(n, np.linspace(0, n, 9).astype(np.uint64), batches)
    apply_all([single, g], batches)
    hub = int(np.argmax(np.bincount(cs, minlength=n)))
    for s in (hub, n - 1):
        assert np.array_equal(g.bfs(s), single.bfs(s)), s
    assert_same_ranks(g.pagerank(20, 0.85), single.pagerank(20, 0.85))
    g.close()
    single.close()


def test_new_kernels_are_launched():
    """torch.profiler sees the traversal kernels launched (in a child process, see WITNESS)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", WITNESS, root], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    names = json.loads(r.stdout.strip().splitlines()[-1])
    if not names:
        warnings.warn("torch.profiler recorded no kernels in the child process; kernel witness skipped")
        return
    for k in ("k_group_bfs_expand", "k_group_bfs_publish", "k_group_bfs_merge", "k_group_bfs_level_end",
              "k_group_pagerank_reduce", "k_pagerank_push"):
        assert any(k in x for x in names), (k, names)


def test_distinct_devices():
    L = pp.load_library()
    if L.ppcsr_device_count() < 2:
        pytest.skip("needs two GPUs: the shards on distinct devices")
    n, batches = scale14_batches()
    k = min(4, L.ppcsr_device_count())
    single = pp.Shard(n)
    g = make_group(n, random_starts(n, k, seed=21), batches, devices=list(range(k)))
    apply_all([single, g], batches)
    for s in (0, n - 1, n):
        assert np.array_equal(g.bfs(s), single.bfs(s)), s
    for it, d in ((0, 0.85), (20, 0.85), (20, 1.0)):
        assert_same_ranks(g.pagerank(it, d), single.pagerank(it, d), (it, d))
    g.close()
    single.close()


def test_cli_traversals_match_across_modes(tmp_path):
    """-bfs=0 -pagerank=20 print the same BFS line for -ppcsr and the partitioned modes, and PageRank sums and maxima
    within 1e-9 (the scale-12 inputs of test_cli_pppcsr_device_route_matches_ppcsr)."""
    build.build_host()
    scale = 12
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    idx = synth.sample_without_replacement(16 << scale, 20000, 7)
    core, upd = str(tmp_path / "core.bin"), str(tmp_path / "upd.bin")
    np.stack([cs, cd], axis=1).astype("<u4").tofile(core)
    np.stack([cs[idx], cd[idx]], axis=1).astype("<u4").tofile(upd)
    bfs_lines, prs = [], []
    for mode in (["-ppcsr"], ["-pppcsr", "-partitions_per_domain=3"], ["-pppcsr", "-partitions_per_domain=4", "-balanced"]):
        cmd = [build.CLI, "-threads=8", "-delete", "-size=20000", *mode, f"-core_graph={core}", f"-update_file={upd}",
               "-bfs=0", "-pagerank=20"]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        lines = r.stdout.splitlines()
        bfs_lines.append([l for l in lines if l.startswith("BFS from 0: reached ")][0])
        pr = [l for l in lines if l.startswith("PageRank 20 iterations: sum ")][0].split()
        prs.append((float(pr[4]), float(pr[6])))
    assert bfs_lines[0] == bfs_lines[1] == bfs_lines[2]
    assert int(bfs_lines[0].split()[4]) > 1000
    for s, m in prs[1:]:
        assert np.isclose(s, prs[0][0], rtol=RTOL, atol=0) and np.isclose(m, prs[0][1], rtol=RTOL, atol=0)
