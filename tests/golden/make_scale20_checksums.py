"""Generates tests/golden/scale20_checksums.json: the checksum (edges, edge_hash of ppcsr_checksum) of the logical graph
after the first 1 000 000 and after all 10 000 000 updates of three streams on the R-MAT scale-20 core (16 777 216 raw
edges, seed 42) -- uniform insertions (seed 7), skewed (R-MAT) insertions (seed 99) and deletions sampled without
replacement from the raw core list (seed 7).  tests/test_gpu_parity.py::test_full_size_vs_reference_dump compares the
device graph with these values.

For these streams the logical graph does not depend on the order of the updates: an insert stream gives the union of
the core's and the stream's (src, dst) keys, a delete stream the difference.  That is what the reference's dumps of
these runs hold, and what the C restatement (oracle/pcsr_oracle.c) gives applied sequentially (--check-oracle, ~6 min).

  python tests/golden/make_scale20_checksums.py [--check-oracle]
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCALE, N_UPD, CKPT, CORE_SEED, UNIFORM_SEED, SKEW_SEED = 20, 10_000_000, 1_000_000, 42, 7, 99


def streams(synth):
    """name -> (src, dst, value) of the update stream; (core src, core dst)."""
    cs, cd = synth.rmat(SCALE, 0, 16 << SCALE, CORE_SEED)
    idx = synth.sample_without_replacement(16 << SCALE, N_UPD, UNIFORM_SEED)
    return {"uniform": (*synth.uniform(SCALE, 0, N_UPD, UNIFORM_SEED), 1),
            "skewed": (*synth.rmat(SCALE, 0, N_UPD, SKEW_SEED), 1),
            "delete": (cs[idx], cd[idx], 0)}, (cs, cd)


def keys(s, d):
    return (np.asarray(s).astype(np.uint64) << np.uint64(32)) | np.asarray(d).astype(np.uint64)


def checksum(synth, k):
    with np.errstate(over="ignore"):
        return {"edges": int(k.size), "edge_hash": f"{int(synth.mix64(k).sum(dtype=np.uint64)):016x}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check-oracle", action="store_true", help="also apply the streams to the C restatement")
    a = ap.parse_args()
    synth = importlib.import_module("parallel-packed-csr_b200.synth")
    upd, (cs, cd) = streams(synth)
    core = np.unique(keys(cs, cd))
    out = {"workload": {"scale": SCALE, "core_edges": 16 << SCALE, "core_seed": CORE_SEED, "updates": N_UPD,
                        "checkpoint": CKPT, "uniform_seed": UNIFORM_SEED, "skewed_seed": SKEW_SEED,
                        "delete_sample_seed": UNIFORM_SEED},
           "produced_by": "tests/golden/make_scale20_checksums.py (keys of the core graph and the stream: union for "
                          "insertions, difference for deletions)"}
    for name, (s, d, v) in upd.items():
        for label, hi in (("checkpoint", CKPT), ("full", N_UPD)):
            k = np.unique(keys(s[:hi], d[:hi]))
            k = np.union1d(core, k) if v else np.setdiff1d(core, k, assume_unique=True)
            out[f"{name}_{label}"] = checksum(synth, k)
    if a.check_oracle:
        import oracle_py as O

        for name, (s, d, v) in upd.items():
            o = O.OraclePCSR(1 << SCALE)
            o.apply(cs, cd, 1)
            for label, lo, hi in (("checkpoint", 0, CKPT), ("full", CKPT, N_UPD)):
                o.apply(s[lo:hi], d[lo:hi], v)
                rowptr, col, _ = o.export()
                got = synth.graph_checksum(rowptr, col)
                want = out[f"{name}_{label}"]
                assert (got["edges"], f"{got['edge_hash']:016x}") == (want["edges"], want["edge_hash"]), (name, label)
            print(f"oracle agrees on {name}", file=sys.stderr)
        out["produced_by"] += "; the C restatement (oracle/pcsr_oracle.c) gives the same six checksums"
    with open(os.path.join(HERE, "scale20_checksums.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
