"""Cost of the score graph export (hmk_score_graph) on one GPU, next to complete linkage's counting pass.

For MUSI, the antibodies set (74 041), 100 000 and 1 000 000 synthetic 12-mers (BLOSUM62, T = round(1.7 x mean length),
default X, P = 0, input order):
* edges, and whether they equal the valid pairs of hmk_clinkage_run on the same input (xhits_kept / 2);
* device time of the scoring passes and of the shift / sort / edge passes (option profile: hmk_get_section_ms slots 0
  and 1 after the pull);
* wall time of the full pull loop: hmk_score_graph pages of `--page` edges into one reused host buffer (the edges are
  not kept), from cursor {0, 0} to {n, 0};
* complete linkage's counting pass on the same input (slot 0 after hmk_clinkage_run) as the reference point.
The card's name and power limit are read in the same process.

usage: python scripts/score_graph_scale.py [--out profiles/r06_score_graph.json] [--skip-1m] [--page N]
"""
import argparse
import ctypes as C
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


def pull(ctx, n, page):
    """the whole graph in pages of `page` edges into one reused buffer -> (edges, pages, wall ms, checksum)"""
    buf = np.zeros(page, dtype=hb.EDGE_DTYPE)          # touched once, before the timed loop
    cur = (C.c_int64 * 2)(0, 0)
    got = C.c_int64(0)
    err = C.create_string_buffer(512)
    edges = pages = 0
    check = 0
    t0 = time.perf_counter()
    while not (cur[0] == n and cur[1] == 0):
        rc = ctx._L.hmk_score_graph(ctx._h, cur, buf.ctypes.data_as(C.c_void_p), page, C.byref(got), err, 512)
        if rc:
            raise RuntimeError(f"hmk_score_graph: status {rc} {err.value!r}")
        edges += got.value
        pages += 1
        if got.value:                                   # last edge of the page: the order is (seq, partner)
            check = (check * 1000003 + int(buf["seq"][got.value - 1]) * n + int(buf["partner"][got.value - 1])) % (1 << 61)
    wall = (time.perf_counter() - t0) * 1e3
    return edges, pages, wall, check


def measure(name, d, M, T, X, page):
    n = len(d["abundance"])
    rec = {"input": name, "n": n, "T": T, "X": X}
    ctx = hb.GreedyContext(0, profile=1)
    try:
        rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], M, T, X, 0)
        sec = ctx.section_ms()
        st = ctx.stats()
        rec["clinkage"] = {"status": rc, "counting_pass_ms": round(sec["p1_select"], 3), "total_ms": round(st["total_ms"], 3),
                           "valid_pairs": st["xhits_kept"] // 2 if n > 32768 else None,
                           "note": "dense path (n <= 32768): slot 0 is the n x n scoring" if n <= 32768 else "sparse path"}
        del G
        ctx.upload(d["residues"], d["offsets"], d["abundance"], M, T, X, 0, 0)
        before = ctx.stats()["bulk_pairs"]               # the stats still hold the clinkage call's count
        edges, pages, wall, check = pull(ctx, n, page)
        sec = ctx.section_ms()
        rec["graph"] = {"edges": edges, "pages": pages, "page_edges": page, "pull_wall_ms": round(wall, 2),
                        "scoring_device_ms": round(sec["p1_select"], 3), "shift_sort_device_ms": round(sec["p1_partner"], 3),
                        "pairs_scored": ctx.stats()["bulk_pairs"] - before, "copy_out_bytes": edges * 16, "order_checksum": check}
        if rec["clinkage"]["valid_pairs"] is not None:
            rec["graph"]["edges_equal_clinkage_valid_pairs"] = edges == rec["clinkage"]["valid_pairs"]
        edges2, _, wall2, check2 = pull(ctx, n, page)   # a second pull on the same context: repeatable
        rec["graph"]["second_pull_wall_ms"] = round(wall2, 2)
        rec["graph"]["second_pull_equal"] = edges2 == edges and check2 == check
    finally:
        ctx.close()
    return rec


def synthetic(n):
    d = synth.generate(n, 12, 12, seed=20260101)
    T, X, _ = synth.default_params(d["lengths"])
    return d, T, X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_score_graph.json"))
    ap.add_argument("--skip-1m", action="store_true")
    ap.add_argument("--page", type=int, default=1 << 24)
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
        rec = measure(name, d, M, T, X, args.page)
        res["runs"].append(rec)
        log(rec)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
