"""Cost of the nearest-partner search (hmk_nearest) on one GPU, next to the score graph's scoring pass.

For MUSI, the antibodies set (74 041), 100 000 and 1 000 000 synthetic 12-mers (BLOSUM62, T = round(1.7 x mean length),
default X, P = 0, input order), at k = 8 and 31:
* wall time of one hmk_nearest call over all rows into host arrays (option profile off; a host clock around a call that
  ends in a device synchronise), after a warm-up call on the first rows;
* device time of its scoring pass (profiles + the top-(k + 1) launch) and of its merge / score / shift pass (option
  profile on: hmk_get_section_ms slots 0 and 1 after a second full call), and that both calls give the same lists;
* entries, rows with more than k partners, and a checksum of the lists;
* the score graph's scoring passes on the same context (slot 0 after a full hmk_score_graph pull into one reused page
  buffer) as the reference point: nearest scores every ordered pair, the graph only i < j.
The card's name and power limit are read in the same process.

usage: python scripts/nearest_scale.py [--out profiles/r07_nearest.json] [--skip-1m]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hammock_b200 as hb                                                   # noqa: E402
from hammock_b200 import synth                                              # noqa: E402
from tests.golden.make_antibodies_clinkage_golden import input_arrays        # noqa: E402


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,power.max_limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit_max_limit_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_max_limit_max_sm_clock"] = f"unavailable: {e}"
    return out


def graph_scoring_ms(ctx, n, page=1 << 24):
    """full score-graph pull into one reused buffer -> (edges, slot-0 device ms)"""
    buf = np.zeros(page, dtype=hb.EDGE_DTYPE)
    cur = (C.c_int64 * 2)(0, 0)
    got = C.c_int64(0)
    err = C.create_string_buffer(512)
    edges = 0
    while not (cur[0] == n and cur[1] == 0):
        rc = ctx._L.hmk_score_graph(ctx._h, cur, buf.ctypes.data_as(C.c_void_p), page, C.byref(got), err, 512)
        if rc:
            raise RuntimeError(f"hmk_score_graph: status {rc} {err.value!r}")
        edges += got.value
    return edges, ctx.section_ms()["p1_select"]


def digest(lists):
    h = hashlib.sha256()
    for a in lists:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def measure(name, d, M, T, X):
    n = len(d["abundance"])
    rec = {"input": name, "n": n, "T": T, "X": X, "nearest": []}
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], M, T, X, 0, 0)
        for k in (8, 31):
            ctx.set_option("profile", 0)
            ctx.nearest(k, (0, min(n, 1024)))               # warm-up: modules, kernel attributes, buffers
            t0 = time.perf_counter()
            lists = ctx.nearest(k)
            wall = (time.perf_counter() - t0) * 1e3
            ctx.set_option("profile", 1)
            again = ctx.nearest(k)
            sec = ctx.section_ms()
            count, more = lists[3], lists[4]
            rec["nearest"].append({"k": k, "wall_ms": round(wall, 2), "scoring_device_ms": round(sec["p1_select"], 3),
                                   "merge_shift_device_ms": round(sec["p1_partner"], 3), "entries": int(count.sum()),
                                   "rows_with_more": int(more.sum()), "rows_empty": int((count == 0).sum()),
                                   "lists_digest": digest(lists),
                                   "profiled_call_equal": all(np.array_equal(a, b) for a, b in zip(lists, again)),
                                   "host_bytes": int(sum(a.nbytes for a in lists))})
            del lists, again
        ctx.set_option("profile", 1)
        edges, gms = graph_scoring_ms(ctx, n)
        rec["graph"] = {"edges": edges, "scoring_device_ms": round(gms, 3)}
        for r in rec["nearest"]:
            r["scoring_over_graph_scoring"] = round(r["scoring_device_ms"] / gms, 3) if gms else None
    finally:
        ctx.close()
    return rec


def synthetic(n):
    d = synth.generate(n, 12, 12, seed=20260101)
    T, X, _ = synth.default_params(d["lengths"])
    return d, T, X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_nearest.json"))
    ap.add_argument("--skip-1m", action="store_true")
    args = ap.parse_args()
    M = synth.blosum62()
    res = {"card": card(), "workloads": "BLOSUM62, T = round(1.7 x mean length), X = default, P = 0; synthetic: "
           "hammock_b200.synth.generate(n, 12, 12, seed=20260101) in generated order", "runs": []}

    def log(x):
        print(json.dumps(x), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)

    z = np.load(os.path.join(ROOT, "tests", "golden", "musi_clinkage.npz"))
    ab_res, ab_offs, ab_ab = input_arrays()
    inputs = [("musi", ({k: z[k] for k in ("residues", "offsets", "abundance")}, 20, 3)),
              ("antibodies", ({"residues": ab_res, "offsets": ab_offs, "abundance": ab_ab}, 20, 3)),
              ("synthetic_100000", synthetic(100_000))]
    if not args.skip_1m:
        inputs.append(("synthetic_1000000", synthetic(1_000_000)))
    for name, (d, T, X) in inputs:
        rec = measure(name, d, M, T, X)
        res["runs"].append(rec)
        log(rec)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
