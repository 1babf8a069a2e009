"""Differential tests of every dispatch branch of the batch pipeline against a numpy last-op-wins reference.

`ref_apply` below restates one batch (include/ppcsr_b200.h, "Conventions shared by the batch entry points") with
vectorised numpy, fast enough for batches of 40 M updates; `test_reference_matches_oracle` pins it to the sequential
C restatement (tests/oracle_py.py) on small streams.  Every GPU case applies ONE batch to a shard and compares the
exported graph with values, num_neighbors (mod 2^32), the batch counters and the PMA invariants with the reference.

Each case proves that it reached its branch: by a field of the batch stats, or by the kernel template instances
torch.profiler saw launched (names as demangled, `(bool)1` written `true`).  If the profiler records no kernels on a
machine, only that witness is skipped (with a warning); the comparison with the reference still runs.

Branch                                                        Case (test[id])                        Witness
------------------------------------------------------------  -------------------------------------  -----------------------------------------
apply_device_common
  host arrays (ppcsr_apply_batch -> k_build_keys)             matrix[host-*]                         k_build_keys
  device arrays (ppcsr_apply_batch_device)                    matrix[device-*]                       k_build_keys
  packed records (k_build_keys_packed, pairs = 0)             matrix[packed-*]                       k_build_keys_packed
  interleaved pairs (k_build_keys_packed, pairs = 1)          matrix[pairs-ins-*, pairs-del-*]       k_build_keys_packed
  submit / wait (ppcsr_wait)                                  matrix[submit-*]                       counters of the batch
  segments (k_build_keys_segments, never small-batch)         segments[*]                            k_build_keys_segments, sparse_path 0
    region count above region_cap (clamped)                   segments[over-cap-*]                   batch_size = clamped total
    deposited total above max_total -> PPCSR_ERR_CAPACITY     segments[max-total]                    error, checksum unchanged
    every region empty                                        segments[all-empty]                    batch_size 0
    n_segments > 64 -> PPCSR_ERR_ARG                          segments[too-many]                     error
  small-batch path (count <= 2^17, count*4 <= n_leaves)       matrix[*-1 .. *-16384], scale20[2^17]  sparse_path 1
    over SPARSE_MAX_BATCH                                     scale20[2^17+1]                        sparse_path 0
    over n_leaves / 4                                         matrix[host-ins-nl4], [host-ins-nl4+1] sparse_path 1 / 0
    k_locate<true, true> (no values, default != 0)            matrix[host-ins-1], [host-seven-1025]  k_locate<true,true,false>
    k_locate<true, false> (removes only, values, ops)         matrix[host-del-1024], [host-values-*]  k_locate<true,false,false>
    abort: dst wider than speculated, redone general          speculation                            k_locate<true,true,false> + sparse_path 0
  general path
    k_locate<false, true>  (no values, default != 0)          matrix[host-ins-16385], scale20[grow]  k_locate<false,true,false>
    k_locate<false, false, true> (no values, default 0)       matrix[host-del-16385], [pairs-del-*]  k_locate<false,false,true>
    k_locate<false, false> (values / op bit)                  matrix[packed-ops-*], [host-zeros-*]    k_locate<false,false,false>
    one locate tile (no scan, no gather) vs several           matrix[host-ins-512], [host-ins-513]   k_gather_inserts absent / present
    values all equal -> keys-only sort with the op bit        matrix[host-ops-20479-whole], [packed-ops-20000], scale20[mixed]
                                                                                                     k_os_pass<false,...>
    all-zero value array (removes only)                       matrix[host-zeros-*], [submit-zeros-*] counters
    rejected updates (src >= n, (v, SENT) inserts/removes)    rejected                               n_ignored
  whole-array policy -1 / 0 / 1                               matrix[*-win], [*-auto], [*-whole]     whole_array 0 / - / 1
  sort layout speculation: same layout (fused histograms)     speculation                            k_os_hist absent
    wider batch / one pass fewer (k_os_hist fallback)         speculation                            k_os_hist present
radix_sort_from / sort_small_dispatch
  k_sort_small ITEMS 1 (n <= 1024)                            matrix[host-ins-1], [host-del-1024]    k_sort_small<1,...>
  k_sort_small ITEMS 4 (n <= 4096)                            matrix[host-seven-1025], [...-4096]    k_sort_small<4,...>
  k_sort_small ITEMS 16 (n <= 16384)                          matrix[host-ins-4097], [...-16384]     k_sort_small<16,...>
  onesweep, payload; tail tile of 1 key                       matrix[host-values-20481-win]          k_os_pass<true,prim::KeyArray,true>
  onesweep, keys only, early counts; tail tile of 4095 keys   matrix[host-ops-20479-whole]           k_os_pass<false,prim::KeyArray,true>
  onesweep, keys only, late counts (n >= 2^25)                scale20[grow], scale20[mixed]          k_os_pass<false,prim::KeyArray,false>
  grown array (resize in the same pass)                       scale20[grow]                          resized 1
ppcsr_bin_to_peers
  with values: ordered k_bin_scatter_peers<true>              tests/test_gpu_host.py group test      -
  keys only: k_bin_scatter_peers<false,false> + publish       group[1, 3, 4 parts, default 1 and 0]  both kernels, k_build_keys_segments

The sort primitive itself (keys only and with payload, 2^25 +- 1, 40 M, lo_bits 32, 8 passes, equal and maximal
keys) is compared with np.argsort in tests/test_gpu_parity.py::test_primitives_scan_and_sort.
"""
import importlib
import warnings
import zlib

import numpy as np
import pytest

import oracle_py as O

pp = importlib.import_module("parallel-packed-csr_b200")
synth = importlib.import_module("parallel-packed-csr_b200.synth")

SENT = 0xFFFFFFFF
M32 = np.uint64(0xFFFFFFFF)
S32 = np.uint64(32)
COUNTERS = ("batch_size", "n_ignored", "n_unique", "n_inserted", "n_overwritten", "n_deleted", "n_not_found")


# ------------------------------------------------------------------------------------------------
# the reference
# ------------------------------------------------------------------------------------------------
class RefState:
    """A logical graph: sorted unique (src << 32 | dst) keys, their values, and num_neighbors as int64 (call counts,
    compared with the device's u32 modulo 2^32)."""

    def __init__(self, n, keys=None, vals=None, nn=None):
        self.n = n
        self.keys = np.zeros(0, np.uint64) if keys is None else keys
        self.vals = np.zeros(0, np.uint32) if vals is None else vals
        self.nn = np.zeros(n, np.int64) if nn is None else nn

    def nn_u32(self):
        return (self.nn % (1 << 32)).astype(np.uint32)

    def csr(self):
        src = (self.keys >> S32).astype(np.int64)
        rowptr = np.zeros(self.n + 1, np.uint64)
        np.cumsum(np.bincount(src, minlength=self.n), out=rowptr[1:])
        return rowptr, (self.keys & M32).astype(np.uint32)


def ref_apply(state, src, dst, val=None, default_val=1):
    """One batch with last-op-wins per (src, dst), the sequential `not found` rule and the header's rejection rules.
    Returns (new state, expected counters)."""
    n = state.n
    src = np.asarray(src).astype(np.uint64)
    dst = np.asarray(dst).astype(np.uint64)
    m = src.size
    v = np.full(m, default_val, np.uint32) if val is None else np.broadcast_to(np.asarray(val).astype(np.uint32), (m,))
    ins = v != 0
    # rejected: src >= n (inserts and removes), and inserts of the sentinel dst; a remove of (v, SENT) is a remove call
    # (num_neighbors -1) that can never find its edge
    ok = (src < n) & ~(ins & (dst == SENT))
    s, d, v, ins = src[ok], dst[ok], v[ok], ins[ok]
    si = s.astype(np.int64)
    nn = state.nn + np.bincount(si[ins], minlength=n) - np.bincount(si[~ins], minlength=n)
    order = np.argsort((s << S32) | d, kind="stable")  # equal keys keep submission order
    k, ins, v = ((s << S32) | d)[order], ins[order], v[order]
    first = np.ones(k.size, bool)
    first[1:] = k[1:] != k[:-1]
    last = np.ones(k.size, bool)
    last[:-1] = first[1:]
    uk = k[first]
    pos = np.searchsorted(state.keys, uk)
    present = np.zeros(uk.size, bool)
    if state.keys.size:
        present = (pos < state.keys.size) & (state.keys[np.minimum(pos, state.keys.size - 1)] == uk)
    w_ins, w_val = ins[last], v[last]
    # a remove misses if the previous op on its key in this batch was a remove, or, as the key's first op, if the
    # edge was absent before the batch
    prev_rm = np.zeros(k.size, bool)
    prev_rm[1:] = ~ins[:-1]
    run = np.cumsum(first) - 1
    miss = ~ins & np.where(first, ~present[run], prev_rm)
    want = {
        "batch_size": m, "n_ignored": int(m - ok.sum()), "n_unique": int(uk.size),
        "n_inserted": int((w_ins & ~present).sum()), "n_overwritten": int((w_ins & present).sum()),
        "n_deleted": int((~w_ins & present).sum()), "n_not_found": int(miss.sum()),
    }
    keep = np.ones(state.keys.size, bool)
    keep[pos[~w_ins & present]] = False
    vals = state.vals.copy()
    vals[pos[w_ins & present]] = w_val[w_ins & present]
    kept_k, kept_v = state.keys[keep], vals[keep]
    new = w_ins & ~present
    at = np.searchsorted(kept_k, uk[new])
    return RefState(n, np.insert(kept_k, at, uk[new]), np.insert(kept_v, at, w_val[new]), nn), want


def _oracle_stream(rng, n, m):
    """Duplicates, remove/insert/remove runs, misses, src >= n and removes of the sentinel dst."""
    pool = np.stack([rng.integers(0, n + 2, m // 4 + 1), rng.integers(0, n, m // 4 + 1)], 1)
    pick = pool[rng.integers(0, pool.shape[0], m)]
    src, dst = pick[:, 0].copy(), pick[:, 1].copy()
    sent = rng.integers(0, 40, m) == 0
    dst[sent] = SENT
    val = np.where(rng.integers(0, 3, m) == 0, 0, rng.integers(1, 1 << 31, m))
    return src, dst, val


def test_reference_matches_oracle():
    """ref_apply against the sequential C restatement on seeded streams: graph, values, num_neighbors, not found."""
    rng = np.random.default_rng(2024)
    for n, m, batch, one_value in ((300, 6000, 6000, False), (300, 6000, 257, True), (40, 3000, 1, False),
                                   (2000, 20000, 5000, True)):
        o, ref = O.OraclePCSR(n), RefState(n)
        src, dst, val = _oracle_stream(rng, n, m)
        if one_value:
            val = np.where(val != 0, 7, 0)
        misses = 0
        for lo in range(0, m, batch):
            sl = slice(lo, lo + batch)
            ref, want = ref_apply(ref, src[sl], dst[sl], val[sl])
            misses += want["n_not_found"]
            # inserts of the sentinel dst are rejected by the header's rule; the C restatement would store them
            keep = ~((val[sl] != 0) & (dst[sl] == SENT))
            o.apply(src[sl][keep], dst[sl][keep], val[sl][keep])
        rowptr, col, nn = o.export()
        erp, ecol = ref.csr()
        assert np.array_equal(erp, rowptr) and np.array_equal(ecol, col), (n, m, batch)
        assert np.array_equal(ref.vals, o.export_values()), (n, m, batch)
        assert np.array_equal(ref.nn_u32(), nn), (n, m, batch)
        assert misses == o.not_found, (n, m, batch)
    # default values: None with default 0 removes, with default 7 inserts 7
    o, ref = O.OraclePCSR(50), RefState(50)
    s, d = rng.integers(0, 52, 500), rng.integers(0, 50, 500)
    for default in (7, 0, 3):
        ref, _ = ref_apply(ref, s, d, None, default)
        o.apply(s, d, default)
    assert np.array_equal(ref.csr()[1], o.export()[1]) and np.array_equal(ref.vals, o.export_values())
    assert np.array_equal(ref.nn_u32(), o.export()[2])


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def _norm(name):
    return name.replace("(bool)1", "true").replace("(bool)0", "false").replace("(int)", "").replace(" ", "")


def launched(fn):
    """Runs fn under torch.profiler; returns (fn's result, normalised names of the kernels launched, or None if the
    profiler recorded none)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {_norm(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return out, ({k for k in names if "k_" in k} or None)


def assert_witness(names, present=(), absent=(), where=""):
    if names is None:
        warnings.warn(f"{where}: torch.profiler recorded no kernels in this process; branch witness skipped")
        return
    short = sorted(k.split("(")[0] for k in names)
    for p in present:
        assert any(_norm(p) in k for k in names), (where, "missing", p, short)
    for p in absent:
        assert not any(_norm(p) in k for k in names), (where, "unexpected", p, short)


def assert_matches(g, ref, st, want, where):
    for key in COUNTERS:
        assert st[key] == want[key], (where, key, st[key], want[key])
    rp, col, val = g.export(with_values=True)
    erp, ecol = ref.csr()
    assert np.array_equal(rp, erp), f"{where}: rowptr differs (first at {np.argmax(rp != erp)})"
    assert np.array_equal(col, ecol), f"{where}: adjacency differs"
    assert np.array_equal(val, ref.vals), f"{where}: values differ"
    assert np.array_equal(g.num_neighbors(), ref.nn_u32()), f"{where}: num_neighbors differs"
    lower = want["n_deleted"] > 0
    r = g.check(lower)
    assert not r.violations(lower), (where, r.as_dict())
    assert r.edges == ref.keys.size, where


class Core:
    """An R-MAT core (16 << scale inserts) on a shard, with its snapshot and reference state."""

    def __init__(self, scale):
        self.scale, self.n = scale, 1 << scale
        self.cs, self.cd = synth.rmat(scale, 0, 16 << scale, 42)
        self.ref, _ = ref_apply(RefState(self.n), self.cs, self.cd, None, 1)
        self.g = self.fresh()
        self.g.snapshot()

    def fresh(self):
        """A new shard holding the core: for cases that widen the speculated sort width (sticky per shard)."""
        g = pp.Shard(self.n)
        g.apply(self.cs, self.cd, 1)
        return g

    def restored(self, policy=0):
        self.g.restore()
        self.g.set_whole_array_policy(policy)
        return self.g


@pytest.fixture(scope="module")
def core16():
    c = Core(16)
    yield c
    c.g.close()


@pytest.fixture(scope="module")
def core20():
    c = Core(20)
    yield c
    c.g.close()


def make_batch(rng, core_keys, n, size, vmode):
    """`size` updates over a pool of about size/2 keys, half of them edges of the core: repeats, hits and misses."""
    half = max(1, size // 4)
    old = core_keys[rng.integers(0, core_keys.size, half)]
    new = (rng.integers(0, n, half).astype(np.uint64) << S32) | rng.integers(0, n, half).astype(np.uint64)
    pool = np.concatenate([old, new])
    k = pool[rng.integers(0, pool.size, size)]
    src, dst = (k >> S32).astype(np.uint32), (k & M32).astype(np.uint32)
    rm = rng.integers(0, 4, size) == 0
    if vmode == "ins":
        return src, dst, None, 1
    if vmode == "del":
        return src, dst, None, 0
    if vmode == "seven":
        return src, dst, None, 7
    if vmode == "values":
        return src, dst, np.where(rm, 0, rng.integers(1, 1 << 31, size)).astype(np.uint32), 1
    if vmode == "ops":
        return src, dst, np.where(rm, 0, 9).astype(np.uint32), 1
    if vmode == "zeros":
        return src, dst, np.zeros(size, np.uint32), 1
    raise ValueError(vmode)


def apply_entry(g, entry, src, dst, val, default):
    import torch

    m = src.size
    if entry == "host":
        return g.apply(src, dst, val, default)
    if entry == "submit":
        return g.wait(g.submit(src, dst, val, default))
    if entry == "pairs":
        assert val is None
        return g.apply_pairs(np.stack([src, dst], 1), default)
    tv = None if val is None else torch.from_numpy(np.ascontiguousarray(val, np.uint32).view(np.int32)).cuda()
    if entry == "device":
        ts = torch.from_numpy(np.ascontiguousarray(src, np.uint32).view(np.int32)).cuda()
        td = torch.from_numpy(np.ascontiguousarray(dst, np.uint32).view(np.int32)).cuda()
        torch.cuda.synchronize()
        return g.apply_device(ts.data_ptr(), td.data_ptr(), None if tv is None else tv.data_ptr(), m, default)
    if entry == "packed":
        packed = (src.astype(np.uint64) << S32) | dst.astype(np.uint64)
        tp = torch.from_numpy(packed.view(np.int64)).cuda()
        torch.cuda.synchronize()
        return g.apply_packed_device(tp.data_ptr(), None if tv is None else tv.data_ptr(), m, default)
    raise ValueError(entry)


# (id, entry, value mode, size, policy, kernels that must run, kernels that must not, stats)
# size "nl4" / "nl4+1": n_leaves / 4 (+ 1) of the core, the small-batch path's share limit
SMALL = {"sparse_path": 1}
GENERAL = {"sparse_path": 0}
MATRIX = [
    ("host-ins-1", "host", "ins", 1, 0, ["k_locate<true,true,false>", "k_sort_small<1,false,prim::KeyArray>"], [], SMALL),
    ("host-del-1024", "host", "del", 1024, 0, ["k_locate<true,false,false>", "k_sort_small<1,false,"], [], SMALL),
    ("host-seven-1025", "host", "seven", 1025, 0, ["k_locate<true,true,false>", "k_sort_small<4,false,"], [], SMALL),
    ("host-values-4096", "host", "values", 4096, 0, ["k_sort_small<4,true,"], [], SMALL),
    ("host-ins-4097", "host", "ins", 4097, 0, ["k_locate<true,true,false>", "k_sort_small<16,false,"], [], SMALL),
    # the small-batch path sorts the values along even when they are all equal
    ("host-ops-4097", "host", "ops", 4097, 0, ["k_locate<true,false,false>", "k_sort_small<16,true,"], [], SMALL),
    ("host-values-16384", "host", "values", 16384, 0, ["k_sort_small<16,true,"], ["k_os_pass"], SMALL),
    ("host-ins-512", "host", "ins", 512, 0, ["k_locate<true,true,false>"], ["k_gather_inserts"], SMALL),
    ("host-ins-513", "host", "ins", 513, 0, ["k_locate<true,true,false>", "k_gather_inserts"], [], SMALL),
    ("host-ins-512-whole", "host", "ins", 512, 1, ["k_locate<false,true,false>"], ["k_gather_inserts"],
     {"sparse_path": 0, "whole_array": 1}),
    ("host-values-513-whole", "host", "values", 513, 1, ["k_locate<false,false,false>", "k_gather_inserts"], [],
     {"sparse_path": 0, "whole_array": 1}),
    ("host-ins-16385", "host", "ins", 16385, 0, ["k_locate<false,true,false>", "k_os_pass<false,prim::KeyArray,true>"],
     ["k_sort_small"], GENERAL),
    ("host-del-16385-win", "host", "del", 16385, -1, ["k_locate<false,false,true>", "k_os_pass<false,"], [],
     {"sparse_path": 0, "whole_array": 0}),
    ("host-ops-20479-whole", "host", "ops", 5 * 4096 - 1, 1, ["k_os_pass<false,prim::KeyArray,true>", "k_locate<false,false,false>"],
     ["k_os_pass<true,"], {"whole_array": 1}),
    ("host-values-20481-win", "host", "values", 5 * 4096 + 1, -1, ["k_os_pass<true,prim::KeyArray,true>"], [],
     {"sparse_path": 0, "whole_array": 0}),
    ("host-seven-20000", "host", "seven", 20000, 0, ["k_locate<false,true,false>"], [], GENERAL),
    ("host-zeros-20000-whole", "host", "zeros", 20000, 1, ["k_locate<false,false,false>", "k_os_pass<false,"],
     ["k_os_pass<true,"], {"whole_array": 1}),
    ("host-ins-nl4", "host", "ins", "nl4", 0, ["k_locate<true,true,false>"], [], SMALL),
    ("host-ins-nl4+1", "host", "ins", "nl4+1", 0, ["k_locate<false,true,false>"], [], GENERAL),
    ("device-values-5000", "device", "values", 5000, 0, ["k_build_keys", "k_sort_small<16,true,"], [], SMALL),
    ("device-ins-20000-win", "device", "ins", 20000, -1, ["k_build_keys", "k_locate<false,true,false>"], [],
     {"sparse_path": 0, "whole_array": 0}),
    ("device-del-700", "device", "del", 700, 0, ["k_locate<true,false,false>"], [], SMALL),
    ("packed-ops-20000", "packed", "ops", 20000, 0, ["k_build_keys_packed", "k_os_pass<false,"], [], GENERAL),
    ("packed-del-3000-whole", "packed", "del", 3000, 1, ["k_build_keys_packed", "k_locate<false,false,true>"], [],
     {"whole_array": 1}),
    ("packed-values-2000", "packed", "values", 2000, 0, ["k_build_keys_packed", "k_sort_small<4,true,"], [], SMALL),
    ("pairs-ins-20000", "pairs", "ins", 20000, 0, ["k_build_keys_packed", "k_locate<false,true,false>"], [], GENERAL),
    ("pairs-del-20000-win", "pairs", "del", 20000, -1, ["k_build_keys_packed", "k_locate<false,false,true>"], [],
     {"sparse_path": 0, "whole_array": 0}),
    ("pairs-ins-300", "pairs", "ins", 300, 0, ["k_locate<true,true,false>"], [], SMALL),
    ("submit-values-20000", "submit", "values", 20000, 0, ["k_os_pass<true,"], [], GENERAL),
    ("submit-zeros-2000", "submit", "zeros", 2000, 0, ["k_locate<true,false,false>"], [], SMALL),
    ("submit-ins-3000-whole", "submit", "ins", 3000, 1, ["k_locate<false,true,false>"], [], {"whole_array": 1}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=[c[0] for c in MATRIX])
def test_branch_matrix(core16, case):
    name, entry, vmode, size, policy, present, absent, stats = case
    g = core16.restored(policy)
    geo = g.geometry
    nl = geo.N // geo.logN
    size = {"nl4": nl // 4, "nl4+1": nl // 4 + 1}.get(size, size)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    src, dst, val, default = make_batch(rng, core16.ref.keys, core16.n, size, vmode)
    ref, want = ref_apply(core16.ref, src, dst, val, default)
    st, names = launched(lambda: apply_entry(g, entry, src, dst, val, default))
    assert_matches(g, ref, st, want, name)
    for k, v in stats.items():
        assert st[k] == v, (name, k, st[k])
    assert_witness(names, present, absent, name)
    g.set_whole_array_policy(0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uneven", "uneven-values", "over-cap", "over-cap-values", "all-empty", "max-total",
                                  "too-many"])
def test_segments(core16, kind):
    """ppcsr_apply_batch_segments_device with regions built by torch: region r holds counts[r] records (clamped to
    region_cap); the batch is the regions' valid records in region order."""
    import torch

    g = core16.restored(0)
    n, cap = core16.n, 3000
    counts = {"uneven": [2500, 0, 3000, 17, 0, 1200], "uneven-values": [1, 2999, 0, 0, 3000, 40],
              "over-cap": [100, 9000, 0, 2000], "over-cap-values": [4000, 0, 3001, 5],
              "all-empty": [0, 0, 0, 0], "max-total": [3000, 3000, 3000], "too-many": [10] * 65}[kind]
    nseg = len(counts)
    rng = np.random.default_rng(nseg * 1000 + sum(counts))
    src, dst, val, default = make_batch(rng, core16.ref.keys, n, nseg * cap, "values" if "values" in kind else "ins")
    packed = (src.astype(np.uint64) << S32) | dst.astype(np.uint64)
    tp = torch.from_numpy(packed.view(np.int64)).cuda()
    tv = None if val is None else torch.from_numpy(val.view(np.int32)).cuda()
    tc = torch.tensor(counts, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    vp = None if tv is None else tv.data_ptr()
    if kind == "too-many":
        with pytest.raises(pp.PpcsrError):
            g.apply_segments_device(tp.data_ptr(), vp, cap, tc.data_ptr(), nseg)
        return
    if kind == "max-total":
        before = g.checksum()
        with pytest.raises(pp.PpcsrError, match="status -3"):
            g.apply_segments_device(tp.data_ptr(), vp, cap, tc.data_ptr(), nseg, max_total=sum(counts) - 1)
        assert g.checksum() == before
        assert_matches(g, core16.ref, {k: 0 for k in COUNTERS}, {k: 0 for k in COUNTERS}, kind)
        return
    take = np.concatenate([np.arange(r * cap, r * cap + min(c, cap)) for r, c in enumerate(counts)]).astype(np.int64)
    ref, want = ref_apply(core16.ref, src[take], dst[take], None if val is None else val[take], default)
    st, names = launched(lambda: g.apply_segments_device(tp.data_ptr(), vp, cap, tc.data_ptr(), nseg))
    assert_matches(g, ref, st, want, kind)
    assert st["sparse_path"] == 0
    if want["batch_size"]:
        assert_witness(names, ["k_build_keys_segments"], [], kind)


@pytest.mark.gpu
def test_rejected_updates(core16):
    """src >= n (inserts and removes) and inserts of the sentinel dst are ignored; removing (v, 0xFFFFFFFF) is a miss
    that leaves v's sentinel in place.  On a fresh shard: such a remove widens the speculated sort width for good."""
    n = core16.n
    for vmode, size, policy in (("values", 3000, 0), ("ops", 30000, 0), ("values", 30000, 1)):
        g = core16.fresh()
        g.set_whole_array_policy(policy)
        rng = np.random.default_rng(size + policy)
        src, dst, val, default = make_batch(rng, core16.ref.keys, n, size, vmode)
        src, dst = src.copy(), dst.copy()
        bad = rng.integers(0, 10, size)
        src[bad == 0] = n + rng.integers(0, 1000, (bad == 0).sum())
        dst[bad == 1] = SENT
        ref, want = ref_apply(core16.ref, src, dst, val, default)
        assert want["n_ignored"] > 0 and want["n_not_found"] > 0
        st = g.apply(src, dst, val, default)
        assert_matches(g, ref, st, want, f"rejected {vmode} {size} {policy}")  # check(): every sentinel in place
        g.close()


@pytest.mark.gpu
def test_speculation(core16):
    """The key builder takes the digit histograms of the speculated sort layout (widest dst seen, vertex ids); the
    fallback k_os_hist runs when a batch is wider or needs one pass fewer.  Then a small batch without values whose dst
    is wider than any seen: the small-batch path aborts and the batch is redone the general way."""
    g = core16.fresh()
    ref, n = core16.ref, core16.n
    rng = np.random.default_rng(11)

    def step(dst_bits, size, policy, present, absent, stats, where, val=None):
        nonlocal ref
        g.set_whole_array_policy(policy)
        src = rng.integers(0, n, size).astype(np.uint32)
        dst = rng.integers(0, 1 << dst_bits, size).astype(np.uint32)
        dst[0] = (1 << dst_bits) - 1  # the batch has exactly this width
        ref, want = ref_apply(ref, src, dst, val, 1)
        st, names = launched(lambda: g.apply(src, dst, val, 1))
        assert_matches(g, ref, st, want, where)
        for k, v in stats.items():
            assert st[k] == v, (where, k, st[k])
        assert_witness(names, present, absent, where)

    big = ["k_os_pass<"]
    step(16, 40000, 1, big, ["k_os_hist"], GENERAL, "same layout: fused histograms")
    step(8, 40000, 1, big + ["k_os_hist"], [], GENERAL, "one pass fewer: k_os_hist")
    step(20, 40000, 1, big + ["k_os_hist"], [], GENERAL, "wider: k_os_hist")
    step(20, 40000, 1, big, ["k_os_hist"], GENERAL, "the wider layout is now speculated")
    step(18, 40000, 1, big, ["k_os_hist"], GENERAL, "narrower, same number of passes: fused")
    step(25, 300, 0, ["k_locate<true,true,false>", "k_locate<false,true,false>"], [], GENERAL,
         "small batch wider than speculated: aborted")
    step(12, 300, 0, ["k_locate<true,true,false>"], ["k_locate<false,"], SMALL, "small batch again")
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("parts", [1, 3, 4])
def test_group_keys_only_route(parts):
    """ppcsr_group_apply without values on GPU 0: ppcsr_bin_to_peers claims places by atomics
    (k_bin_scatter_peers<false, false>) and publishes the counts afterwards (k_publish_peer_counts); the owners apply
    the regions keys-only (k_build_keys_segments).  Inserts (default 1), then removes (default 0)."""
    scale = 14
    n, m = 1 << scale, 60000
    rng = np.random.default_rng(parts)
    starts = np.array([0] + sorted(rng.choice(np.arange(1, n), parts - 1, replace=False).tolist()) + [n], np.uint64)
    grp = pp.Group(n, starts, [0] * parts, region_cap=m // parts + 1, with_values=False)
    s1, d1 = synth.rmat(scale, 0, m, 5)
    pick = rng.integers(0, m, m)
    s2 = np.where(pick % 5 == 0, rng.integers(0, n, m), s1[pick])  # removes: hits, repeats and misses
    d2 = np.where(pick % 5 == 0, rng.integers(0, n, m), d1[pick])
    ref = RefState(n)
    for s, d, default in ((s1, d1, 1), (s2, d2, 0)):
        ref, want = ref_apply(ref, s, d, None, default)
        sts, names = launched(lambda: grp.apply(s, d, None, default))
        for key in COUNTERS:
            assert sum(x[key] for x in sts) == want[key], (parts, default, key)
        rowptr, col = ref.csr()
        nn = ref.nn_u32()
        for r, sh in enumerate(grp.shards):
            lo, hi = int(starts[r]), int(starts[r + 1])
            rp, c, w = sh.export(with_values=True)
            assert np.array_equal(rp, rowptr[lo:hi + 1] - rowptr[lo]), (parts, default, r)
            assert np.array_equal(c, col[int(rowptr[lo]):int(rowptr[hi])]), (parts, default, r)
            assert np.array_equal(w, ref.vals[int(rowptr[lo]):int(rowptr[hi])]), (parts, default, r)
            assert np.array_equal(sh.num_neighbors(), nn[lo:hi]), (parts, default, r)
            assert not sh.check(default == 0).violations(default == 0), (parts, default, r)
        assert_witness(names, ["k_bin_scatter_peers<false,false>", "k_publish_peer_counts", "k_build_keys_segments"],
                       ["k_bin_scatter_peers<true"], f"group {parts} default {default}")
    grp.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["2^17", "2^17+1", "grow", "mixed"])
def test_scale20(core20, case):
    """The scale-20 core: the small-batch size limit (SPARSE_MAX_BATCH = 2^17), and batches of at least 2^25 updates,
    whose keys-only sort passes publish their tile counts late.  `grow`: 2^25 + 1 inserts without values double the
    array in the same pass.  `mixed`: 2^25 + 3 updates over a pool of 2^22 keys (about eight ops per key, random
    insert / remove, one insert value): last-op-wins and the `not found` count hold only if equal keys keep their
    submission order."""
    g = core20.restored(0)
    n = core20.n
    rng = np.random.default_rng(20)
    present, absent = [], []
    if case.startswith("2^17"):
        size = (1 << 17) + (case == "2^17+1")
        src, dst, val, default = make_batch(rng, core20.ref.keys, n, size, "ins")
        stats = {"sparse_path": int(case == "2^17")}
    elif case == "grow":
        size = (1 << 25) + 1
        src = rng.integers(0, n, size).astype(np.uint32)
        dst = rng.integers(0, n, size).astype(np.uint32)
        val, default = None, 1
        stats = {"resized": 1, "sparse_path": 0}
        present = ["k_os_pass<false,prim::KeyArray,false>", "k_locate<false,true,false>"]
    else:
        size = (1 << 25) + 3
        half = 1 << 21
        pool = np.concatenate([core20.ref.keys[rng.integers(0, core20.ref.keys.size, half)],
                               (rng.integers(0, n, half).astype(np.uint64) << S32) | rng.integers(0, n, half).astype(np.uint64)])
        k = pool[rng.integers(0, pool.size, size)]
        src, dst = (k >> S32).astype(np.uint32), (k & M32).astype(np.uint32)
        val, default = np.where(rng.integers(0, 2, size) == 0, 0, 5).astype(np.uint32), 1
        stats = {"sparse_path": 0}
        present, absent = ["k_os_pass<false,prim::KeyArray,false>", "k_locate<false,false,false>"], ["k_os_pass<true,"]
    ref, want = ref_apply(core20.ref, src, dst, val, default)
    st, names = launched(lambda: g.apply(src, dst, val, default))
    assert_matches(g, ref, st, want, case)
    for k, v in stats.items():
        assert st[k] == v, (case, k, st[k])
    assert_witness(names, present, absent, case)


# ------------------------------------------------------------------------------------------------
# PageRank step edges
# ------------------------------------------------------------------------------------------------
def _ulp_close(a, b, ulps):
    a, b = a.astype(np.float32), b.astype(np.float32)
    scale = np.spacing(np.maximum(np.abs(a), np.abs(b)))
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) <= ulps * scale.astype(np.float64)


@pytest.mark.gpu
def test_pagerank_step_edges():
    """ppcsr_pagerank_step_f64 / _f32 with out_len below, at and above n (the tail past n is zero, dsts >= out_len are
    skipped), on a graph where some vertices with live edges have num_neighbors 0 (infinite contributions) or wrapped
    below 0 (a divisor near 2^32)."""
    n = 3000
    rng = np.random.default_rng(9)
    s, d = rng.integers(0, n, 40000), rng.integers(0, n, 40000)
    g, o, ref = pp.Shard(n), O.OraclePCSR(n), RefState(n)
    batches = [(s, d, None, 1)]
    deg = np.bincount(s, minlength=n)
    zero = np.flatnonzero(deg >= 3)[:20]  # as many misses as calls: num_neighbors 0, edges still live
    wrap = np.flatnonzero(deg >= 3)[20:40]  # two misses more: num_neighbors wraps to 2^32 - 2
    ms = np.concatenate([np.repeat(zero, deg[zero]), np.repeat(wrap, deg[wrap] + 2)])
    batches.append((ms, np.full(ms.size, n + 5), None, 0))  # dst n + 5 is never inserted: every remove misses
    for src, dst, val, default in batches:
        ref, _ = ref_apply(ref, src, dst, val, default)
        g.apply(src, dst, val, default)
        o.apply(src, dst, default)
    nn = g.num_neighbors()
    assert np.all(nn[zero] == 0) and np.all(nn[wrap] == 0xFFFFFFFE) and np.array_equal(nn, ref.nn_u32())
    rowptr, col = ref.csr()
    esrc = np.repeat(np.arange(n), np.diff(rowptr).astype(np.int64))
    vals = 1.0 + (np.arange(n) % 7)
    with np.errstate(divide="ignore"):
        c64 = vals / nn.astype(np.float64)
        c32 = (vals.astype(np.float32) / nn.astype(np.float32)).astype(np.float64)
    opr32 = o.pagerank(vals, np.float32)
    for out_len in (n - 777, n, n + 500):
        keep = col < out_len
        for dtype, contrib in ((np.float64, c64), (np.float32, c32)):
            want = np.zeros(out_len, np.float64)
            w = contrib[esrc[keep]]
            fin_w = np.isfinite(w)
            want += np.bincount(col[keep][fin_w].astype(np.int64), weights=w[fin_w], minlength=out_len)
            inf_hit = np.zeros(out_len, bool)
            inf_hit[col[keep][~fin_w]] = True
            want[inf_hit] = np.inf  # every value is positive: an infinite contribution makes the sum +inf
            got = g.pagerank_step(vals, dtype, out_len)
            assert got.shape == (out_len,) and got.dtype == dtype
            assert np.array_equal(np.isfinite(got), np.isfinite(want)), (out_len, dtype)
            assert np.all(got[~np.isfinite(got)] == np.inf), (out_len, dtype)
            fin = np.isfinite(want)
            if dtype == np.float64:
                assert np.allclose(got[fin], want[fin], rtol=1e-6, atol=0.0), out_len
            else:
                assert np.all(_ulp_close(got[fin], want[fin].astype(np.float32), 2)), out_len
                m = min(out_len, n)
                assert np.array_equal(np.isfinite(got[:m]), np.isfinite(opr32[:m])), out_len
            if out_len > n:
                assert np.all(got[n:] == 0), (out_len, dtype)
    assert np.array_equal(np.isfinite(g.pagerank_step(vals, np.float32)), np.isfinite(opr32))
    g.close()
