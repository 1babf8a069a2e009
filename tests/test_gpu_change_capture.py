"""Change capture (ppcsr_set_change_capture / ppcsr_last_changes, batch::k_locate_capture + two compaction scans).

Every batch with capture on leaves, on the device, the keys whose state it changed (old and new value) and one entry per
remove call that missed.  Checked against a sequential Python model (a dict applied call by call), on every path of the
batch pipeline and every entry point, across groups, and by undoing a batch with its own change list."""
import importlib
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_py as O

pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")
build = importlib.import_module("parallel-packed-csr_b200.build")

pytestmark = pytest.mark.gpu
SENT = 0xFFFFFFFF
STAT_KEYS = ("batch_size", "n_ignored", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found",
             "n_windows", "window_slots", "rebalance_bytes", "slots_before", "slots_after", "resized", "whole_array",
             "sparse_path")


# ------------------------------------------------------------------------------------------------
# the sequential model
# ------------------------------------------------------------------------------------------------
class Model:
    """(src, dst) -> value, applied call by call as the reference does at -threads=1."""

    def __init__(self, n):
        self.n = n
        self.e = {}

    def apply(self, src, dst, val):
        src = np.asarray(src, np.uint32)
        dst = np.asarray(dst, np.uint32)
        val = np.broadcast_to(np.asarray(val, np.uint32), src.shape)
        before, nf = {}, []
        for s, d, v in zip(src.tolist(), dst.tolist(), val.tolist()):
            if s >= self.n or (v != 0 and d == SENT):
                continue  # ignored (n_ignored)
            k = (s, d)
            if k not in before:
                before[k] = self.e.get(k, 0)
            if v:
                self.e[k] = v
            elif k in self.e:
                del self.e[k]
            else:
                nf.append(k)
        ch = sorted((k, o, self.e.get(k, 0)) for k, o in before.items() if o or self.e.get(k, 0))
        u32 = lambda xs: np.array(xs, dtype=np.uint32)
        nf.sort()
        return {"src": u32([k[0] for k, _, _ in ch]), "dst": u32([k[1] for k, _, _ in ch]),
                "old_val": u32([o for _, o, _ in ch]), "new_val": u32([w for _, _, w in ch]),
                "nf_src": u32([k[0] for k in nf]), "nf_dst": u32([k[1] for k in nf])}


def assert_lists(got, exp, st=None, where=""):
    for k in ("src", "dst", "old_val", "new_val", "nf_src", "nf_dst"):
        assert np.array_equal(got[k], exp[k]), (where, k, got[k][:20], exp[k][:20], got[k].size, exp[k].size)
    if st is not None:
        old, new = got["old_val"], got["new_val"]
        assert int(np.sum(old == 0)) == st["n_inserted"], where
        assert int(np.sum(new == 0)) == st["n_deleted"], where
        assert int(np.sum((old != 0) & (new != 0))) == st["n_overwritten"], where
        assert got["nf_src"].size == st["n_not_found"], where


def assert_empty(sh, where=""):
    c = sh.last_changes()
    assert all(a.size == 0 for a in c.values()), (where, {k: a.size for k, a in c.items()})


def dup_stream(n, count, seed, kind, pool=None):
    """Batches with heavy duplication over a small key pool: ins/del/ins, del/del, ins/ins with other values, removes
    of absent keys, plus a few ignored updates.  kind: values | ops (one value + removes) | ins | del."""
    rng = np.random.default_rng(seed)
    pool = pool or max(8, count // 4)
    ks = rng.integers(0, pool, count)
    src = (ks * 2654435761 % n).astype(np.uint32)
    dst = (ks * 40503 % (2 * n)).astype(np.uint32)
    if kind == "values":
        val = rng.integers(0, 6, count).astype(np.uint32) * rng.integers(1, 1 << 20, count).astype(np.uint32)
    elif kind == "ops":
        val = (rng.random(count) < 0.55).astype(np.uint32) * 3
    else:
        val = None  # insert-only (default 1) or delete-only (default 0): no values, no op bit
    if kind in ("values", "ops") and count > 16:
        src[:2] = n + 5  # src >= n: ignored
        dst[2] = SENT  # an insert of the sentinel marker: ignored
        src[2] = 1
        val[2] = 3 if kind == "ops" else 9
    return src, dst, val


def fresh(n, policy=0, capture=True):
    sh = pp.Shard(n, device=0)
    sh.set_whole_array_policy(policy)
    if capture:
        sh.set_change_capture(True)
    return sh


def core(sh, m, n, seed=3, count=None):
    """An initial graph with distinct values, applied to shard and model alike."""
    rng = np.random.default_rng(seed)
    count = count or 6 * n
    s = rng.integers(0, n, count).astype(np.uint32)
    d = rng.integers(0, 2 * n, count).astype(np.uint32)
    v = rng.integers(1, 1 << 20, count).astype(np.uint32)
    sh.apply(s, d, v)
    m.apply(s, d, v)


# ------------------------------------------------------------------------------------------------
# mixed batches, every value form, all three window policies
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("policy", [-1, 0, 1])
@pytest.mark.parametrize("kind", ["values", "ops", "ins", "del"])
def test_mixed_batches_match_the_sequential_model(policy, kind):
    n = 1 << 12
    sh, m = fresh(n, policy), Model(n)
    core(sh, m, n)
    for i, count in enumerate((700, 5000, 40000)):
        s, d, v = dup_stream(n, count, 100 + i, kind)
        default = 1 if kind == "ins" else 0 if kind == "del" else 1
        exp = m.apply(s, d, v if v is not None else default)
        st = sh.apply(s, d, v, default)
        assert_lists(sh.last_changes(), exp, st, f"{kind} {policy} {count}")
    rp, col, val = sh.export(with_values=True)
    src = np.repeat(np.arange(n, dtype=np.uint32), np.diff(rp).astype(np.int64))
    assert dict(zip(zip(src.tolist(), col.tolist()), val.tolist())) == m.e


# ------------------------------------------------------------------------------------------------
# the small-batch path, its fall-through and the sparse_abort redo
# ------------------------------------------------------------------------------------------------
def test_small_batch_path_fallthrough_and_abort_redo():
    n = 1 << 14
    sh, m = fresh(n), Model(n)
    twin = fresh(n, capture=False)
    rng = np.random.default_rng(5)
    s = rng.integers(0, n, 20 * n).astype(np.uint32)
    d = rng.integers(0, n, 20 * n).astype(np.uint32)
    for g in (sh, twin):
        g.apply(s, d, 1)
    m.apply(s, d, 1)
    paths = set()
    # small batches on the small-batch path
    for i in range(4):
        bs, bd, bv = dup_stream(n, 300, 200 + i, "values", pool=120)
        bd %= n
        exp = m.apply(bs, bd, bv)
        st = sh.apply(bs, bd, bv)
        twin.apply(bs, bd, bv)
        paths.add(st["sparse_path"])
        assert_lists(sh.last_changes(), exp, st, f"small {i}")
    assert 1 in paths
    # a dst wider than any seen so far: k_locate leaves at once, the batch runs again the general way
    bs, bd, bv = dup_stream(n, 300, 300, "values", pool=120)
    bd = bd % n
    bd[7] = 1 << 27
    exp = m.apply(bs, bd, bv)
    st = sh.apply(bs, bd, bv)
    twin.apply(bs, bd, bv)
    assert st["sparse_path"] == 0
    assert_lists(sh.last_changes(), exp, st, "abort redo")
    # a dense burst into one vertex: a window too large for the small path, the general path takes over
    hub = np.full(2000, 17, np.uint32)
    hd = np.arange(2000, dtype=np.uint32) + 5
    exp = m.apply(hub, hd, 4)
    st = sh.apply(hub, hd, 4)
    twin.apply(hub, hd, 4)
    assert_lists(sh.last_changes(), exp, st, "fall-through")
    assert np.array_equal(sh.debug_dump()[0], twin.debug_dump()[0])


# ------------------------------------------------------------------------------------------------
# capture changes nothing else
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("policy", [-1, 0, 1])
def test_capture_off_and_on_leave_identical_shards(policy):
    n = 1 << 13
    on, off = fresh(n, policy, True), fresh(n, policy, False)
    rng = np.random.default_rng(9)
    batches = [(rng.integers(0, n, 8 * n), rng.integers(0, n, 8 * n), rng.integers(1, 99, 8 * n))]
    for i, kind in enumerate(("values", "ops", "ins", "del", "values")):
        s, d, v = dup_stream(n, (600, 30000)[i % 2], 400 + i, kind)
        batches.append((s, d % n, v if v is not None else 1))
    for s, d, v in batches:
        a, b = on.apply(s, d, v), off.apply(s, d, v)
        assert {k: a[k] for k in STAT_KEYS} == {k: b[k] for k in STAT_KEYS}
        for x, y in zip(on.debug_dump(), off.debug_dump()):
            assert np.array_equal(x, y)
        assert on.checksum() == off.checksum()
        assert np.array_equal(on.num_neighbors(), off.num_neighbors())
    with pytest.raises(pp.PpcsrError):
        off.last_changes()  # capture is off: no lists


# ------------------------------------------------------------------------------------------------
# every entry point
# ------------------------------------------------------------------------------------------------
def test_every_entry_point():
    import torch

    n = 1 << 12
    sh, m = fresh(n), Model(n)
    core(sh, m, n)
    s, d, v = dup_stream(n, 3000, 1, "values")
    exp = m.apply(s, d, v)
    ts, td, tv = (torch.from_numpy(x.astype(np.int32)).cuda() for x in (s, d, v))
    st = sh.apply_device(ts.data_ptr(), td.data_ptr(), tv.data_ptr(), s.size)
    assert_lists(sh.last_changes(), exp, st, "apply_device")
    s, d, v = dup_stream(n, 3000, 2, "ops")
    exp = m.apply(s, d, v)
    packed = torch.from_numpy(((s.astype(np.uint64) << np.uint64(32)) | d).view(np.int64)).cuda()
    tv = torch.from_numpy(v.astype(np.int32)).cuda()
    st = sh.apply_packed_device(packed.data_ptr(), tv.data_ptr(), s.size)
    assert_lists(sh.last_changes(), exp, st, "apply_packed_device")
    s, d, _ = dup_stream(n, 3000, 3, "del")
    exp = m.apply(s, d, 0)
    st = sh.apply_pairs(np.stack([s, d], 1), 0)
    assert_lists(sh.last_changes(), exp, st, "apply_pairs")
    # two batches in flight: the lists belong to the last wait
    b1, b2 = dup_stream(n, 4000, 4, "values"), dup_stream(n, 500, 5, "values")
    t1 = sh.submit(*b1)
    t2 = sh.submit(*b2)
    e1 = m.apply(*b1)
    st = sh.wait(t1)
    assert_lists(sh.last_changes(), e1, st, "wait 1")
    e2 = m.apply(*b2)
    st = sh.wait(t2)
    assert_lists(sh.last_changes(), e2, st, "wait 2")
    # batches of one
    k = next(iter(m.e))
    old = m.e[k]
    sh.add_edge(k[0], k[1], old + 1)
    m.apply([k[0]], [k[1]], [old + 1])
    c = sh.last_changes()
    assert (c["src"].tolist(), c["dst"].tolist(), c["old_val"].tolist(), c["new_val"].tolist()) == (
        [k[0]], [k[1]], [old], [old + 1])
    assert sh.remove_edge(*k)
    c = sh.last_changes()
    assert c["new_val"].tolist() == [0] and c["old_val"].tolist() == [old + 1] and c["nf_src"].size == 0
    assert not sh.remove_edge(*k)
    c = sh.last_changes()
    assert c["src"].size == 0 and (c["nf_src"].tolist(), c["nf_dst"].tolist()) == ([k[0]], [k[1]])
    sh.add_edge(1, 2, 0)  # a zero value is ignored: an empty batch
    assert_empty(sh, "add_edge value 0")


# ------------------------------------------------------------------------------------------------
# groups
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 8])
def test_group_lists_equal_a_single_shard(k):
    n = 1 << 12
    starts = np.linspace(0, n, k + 1).astype(np.uint64)
    grp = pp.Group(n, starts, [0] * k, region_cap=40000 // k + 1, with_values=True)
    grp.set_change_capture(True)
    one, m = fresh(n), Model(n)
    batches = [dup_stream(n, c, 600 + c, "values") for c in (5000, 700, 30000, 2000)]
    for s, d, v in batches[:2]:
        grp.apply(s, d, v)
        st = one.apply(s, d, v)
        exp = m.apply(s, d, v)
        got = grp.last_changes()
        assert_lists(got, exp, None, f"group {k} apply")
        assert_lists(one.last_changes(), got, st, f"single {k}")
    t1 = grp.submit(*batches[2])
    t2 = grp.submit(*batches[3])
    for t, b in ((t1, batches[2]), (t2, batches[3])):
        grp.wait(t)
        one.apply(*b)
        assert_lists(grp.last_changes(), one.last_changes(), None, f"group {k} wait")
    grp.close()


# ------------------------------------------------------------------------------------------------
# undo a batch with its own change list
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["values", "ops", "del"])
def test_undo_with_the_change_list_restores_the_export(kind):
    import torch

    n = 1 << 13
    sh, m = fresh(n), Model(n)
    core(sh, m, n)
    before = sh.export(with_values=True)
    s, d, v = dup_stream(n, 50000, 77, kind)
    sh.apply(s, d, v, 1)
    c = sh.last_changes_device()
    assert c.n_changes > 0
    # copied out first: the next batch of this shard may reuse the buffers the pointers name
    ch = sh.last_changes()
    lists = [torch.from_numpy(ch[k].view(np.int32)).cuda() for k in ("src", "dst", "old_val")]
    sh.apply_device(lists[0].data_ptr(), lists[1].data_ptr(), lists[2].data_ptr(), int(c.n_changes))
    after = sh.export(with_values=True)
    for a, b in zip(before, after):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------
# empty lists
# ------------------------------------------------------------------------------------------------
def test_lists_are_empty_after_failures_and_non_batch_calls():
    n = 1 << 12
    sh, m = fresh(n), Model(n)
    core(sh, m, n)

    def refill():
        s, d, v = dup_stream(n, 3000, 9, "values")
        sh.apply(s, d, v)
        assert sh.last_changes()["src"].size > 0

    refill()
    sh.apply(np.zeros(0, np.uint32), np.zeros(0, np.uint32))
    assert_empty(sh, "empty batch")
    refill()
    with pytest.raises(pp.PpcsrError):
        sh.wait(12345)  # no such batch
    assert_empty(sh, "bad argument")
    refill()
    with pytest.raises(pp.PpcsrError):  # a batch of 2^31 updates is refused before anything is read
        sh.apply_device(1, 1, None, 1 << 31)
    assert_empty(sh, "too large")
    refill()
    sh.snapshot()
    refill()
    sh.isolate_vertices([1, 2, 3])
    assert_empty(sh, "isolate_vertices")
    refill()
    rp, col, val = sh.export(with_values=True)
    sh.load_csr(rp, col, val)
    assert_empty(sh, "load_csr")
    refill()
    sh.add_nodes(3)
    assert_empty(sh, "add_nodes")
    refill()
    sh.restore()
    assert_empty(sh, "restore")
    refill()
    with pytest.raises(pp.PpcsrError):
        sh.load_csr(np.array([0, 2], np.uint64), np.array([5, 5], np.uint32))  # not strictly ascending
    assert_empty(sh, "load_csr refused")
    sh.set_change_capture(False)
    sh.set_change_capture(True)
    assert_empty(sh, "capture toggled")
    # repartition and group isolation
    starts = np.array([0, n // 2, n], np.uint64)
    grp = pp.Group(n, starts, [0, 0], region_cap=4000, with_values=True)
    grp.set_change_capture(True)
    s, d, v = dup_stream(n, 3000, 10, "values")
    grp.apply(s, d, v)
    assert grp.last_changes()["src"].size > 0
    grp.repartition(np.array([0, n // 4, n], np.uint64))
    assert all(a.size == 0 for a in grp.last_changes().values())
    grp.apply(s, d, v)
    grp.isolate_vertices([4, 5])
    assert all(a.size == 0 for a in grp.last_changes().values())
    grp.close()


def test_capacity_failure_leaves_the_lists_empty():
    """A batch whose worst-case buffers (capture scratch and lists included) do not fit is refused before anything is
    applied, and leaves no lists.  The batch's own arrays are real device arrays of its full length."""
    import torch

    n = 1 << 10
    sh, m = fresh(n), Model(n)
    core(sh, m, n)
    s, d, v = dup_stream(n, 500, 12, "values")
    sh.apply(s, d, v)
    assert sh.last_changes()["src"].size > 0
    before = (sh.checksum(), sh.num_neighbors())
    B = 50_000_000  # about 3 GB of worst-case buffers with capture on
    ts = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    td = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    free, _ = torch.cuda.mem_get_info(0)
    blocker = torch.empty(max(0, free - (256 << 20)), dtype=torch.uint8, device="cuda:0")
    try:
        with pytest.raises(pp.PpcsrError):
            sh.apply_device(ts.data_ptr(), td.data_ptr(), None, B)
    finally:
        del blocker, ts, td
        torch.cuda.empty_cache()
    assert_empty(sh, "capacity")
    assert sh.checksum() == before[0] and np.array_equal(sh.num_neighbors(), before[1])


# ------------------------------------------------------------------------------------------------
# scale 20, 10 M updates, against a vectorised model
# ------------------------------------------------------------------------------------------------
def vector_model(rp, col, val, n, src, dst, v):
    """The sequential rule for one batch, vectorised: returns the expected lists."""
    src = np.asarray(src, np.uint64)
    dst = np.asarray(dst, np.uint64)
    v = np.broadcast_to(np.asarray(v, np.uint32), src.shape)
    ok = (src < n) & ~((v != 0) & (dst == SENT))
    key = (src[ok] << np.uint64(32)) | dst[ok]
    v = v[ok]
    o = np.argsort(key, kind="stable")
    key, v = key[o], v[o]
    first = np.ones(key.size, bool)
    first[1:] = key[1:] != key[:-1]
    last = np.ones(key.size, bool)
    last[:-1] = key[1:] != key[:-1]
    esrc = np.repeat(np.arange(n, dtype=np.uint64), np.diff(rp).astype(np.int64))
    ekey = (esrc << np.uint64(32)) | col.astype(np.uint64)  # ascending already
    pos = np.searchsorted(ekey, key)
    pos_c = np.minimum(pos, max(ekey.size - 1, 0))
    present = (pos < ekey.size) & (ekey[pos_c] == key) if ekey.size else np.zeros(key.size, bool)
    preval = np.where(present, val[pos_c] if ekey.size else 0, 0).astype(np.uint32)
    prev_remove = np.zeros(key.size, bool)
    prev_remove[1:] = v[:-1] == 0
    miss = (v == 0) & np.where(first, ~present, prev_remove)
    kl, old, new = key[last], preval[last], v[last]
    keep = (old != 0) | (new != 0)
    mk = key[miss]
    return {"src": (kl[keep] >> np.uint64(32)).astype(np.uint32), "dst": kl[keep].astype(np.uint32),
            "old_val": old[keep], "new_val": new[keep],
            "nf_src": (mk >> np.uint64(32)).astype(np.uint32), "nf_dst": mk.astype(np.uint32)}


@pytest.mark.parametrize("workload", ["delete", "mixed"])
def test_scale20_ten_million_updates(workload):
    scale, B = 20, 10_000_000
    n, total = 1 << scale, 16 << scale
    cs, cd = synth.rmat(scale, 0, total, 42)
    sh = pp.Shard(n, device=0)
    sh.set_change_capture(True)
    rng = np.random.default_rng(1)
    sh.apply(cs, cd, rng.integers(1, 1 << 30, cs.size).astype(np.uint32))
    rp, col, val = sh.export(with_values=True)
    idx = synth.sample_without_replacement(total, B, 7)
    if workload == "delete":
        s, d, v = cs[idx], cd[idx], np.zeros(B, np.uint32)
    else:
        ops = synth.mixed_ops(0, B, 11)
        us, ud = synth.uniform(scale, 0, B, 7)
        s, d = np.where(ops != 0, us, cs[idx]), np.where(ops != 0, ud, cd[idx])
        v = (ops != 0).astype(np.uint32) * rng.integers(1, 1 << 30, B).astype(np.uint32)
    exp = vector_model(rp, col, val, n, s, d, v)
    st = sh.apply(s, d, v)
    assert_lists(sh.last_changes(), exp, st, workload)


# ------------------------------------------------------------------------------------------------
# the CLI
# ------------------------------------------------------------------------------------------------
NF_LINE = re.compile(r"^not found (\d+) (\d+)$")


def test_cli_not_found_lines():
    scale = 12
    n = 1 << scale
    cs, cd = synth.rmat(scale, 0, 8 << scale, 42)
    rng = np.random.default_rng(3)
    # removes of core edges, of absent edges and repeated removes of one edge
    idx = rng.integers(0, cs.size, 3000)
    us = np.concatenate([cs[idx], rng.integers(0, n, 1000).astype(np.uint32), np.full(5, cs[0], np.uint32)])
    ud = np.concatenate([cd[idx], rng.integers(n, 2 * n, 1000).astype(np.uint32), np.full(5, cd[0], np.uint32)])
    with tempfile.TemporaryDirectory() as td:
        core_f, upd_f = os.path.join(td, "core.txt"), os.path.join(td, "upd.txt")
        synth.write_text(core_f, cs, cd)
        synth.write_text(upd_f, us, ud)
        outs = {}
        for mode in ("-ppcsr", "-pppcsr"):
            base = [build.CLI, "-threads=1", "-delete", f"-size={us.size}", mode, "-partitions_per_domain=2",
                    f"-core_graph={core_f}", f"-update_file={upd_f}"]
            plain = subprocess.run(base, capture_output=True, text=True, timeout=300)
            r = subprocess.run(base + ["-not_found_lines"], capture_output=True, text=True, timeout=300)
            assert plain.returncode == 0 and r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
            lines = sorted(l for l in r.stdout.splitlines() if NF_LINE.match(l))
            count = [l for l in plain.stdout.splitlines() if l.startswith("not found ") and l.endswith(" edges")]
            assert count == [f"not found {len(lines)} edges"]
            assert not any(l.endswith(" edges") and l.startswith("not found") for l in r.stdout.splitlines())
            outs[mode] = lines
        assert outs["-ppcsr"] == outs["-pppcsr"]
        if os.path.exists(O.REF_CLI):
            ref = subprocess.run([O.REF_CLI, "-threads=1", "-delete", f"-size={us.size}", "-ppcsr",
                                  f"-core_graph={core_f}", f"-update_file={upd_f}"], capture_output=True, text=True,
                                 timeout=600)
            assert ref.returncode == 0
            expected = sorted(l for l in ref.stdout.splitlines() if NF_LINE.match(l))
        else:
            m = Model(n)
            m.apply(cs, cd, 1)
            e = m.apply(us, ud, 0)
            expected = sorted(f"not found {a} {b}" for a, b in zip(e["nf_src"].tolist(), e["nf_dst"].tolist()))
        assert outs["-ppcsr"] == expected
