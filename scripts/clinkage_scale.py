"""Scaling of the exact complete-linkage clusterer (hmk_clinkage_run) on one GPU.

* dense against forced sparse (option clinkage_dense_max = 0), alternated in one process with the outputs compared, at
  MUSI, 10 000 and 32 768 synthetic 12-mers: the evidence for or against the dense path's 32 768 cutoff;
* the sparse path at antibodies (74 041), 100 000, 200 000 and 1 000 000 synthetic 12-mers: device time per stage
  (scoring = counting pass, row build = filling pass + row sort + twin index, chain), valid pairs, nearest searches, and
  the device memory the context holds after the call (its buffers only grow during a call, so this is its peak);
* the chain kernel's block size (option clinkage_threads) at antibodies, 100 000 and MCLA71 (rows of nearly n - 1
  entries).
The 1 000 000 run comes last; the output file is rewritten after every record.

usage: python scripts/clinkage_scale.py [--out profiles/r03_clinkage_scale.json] [--skip-1m]
"""
import argparse
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,power.max_limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"] = q
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit"] = f"unavailable: {e}"
    return out


def used_bytes():
    import torch
    free, total = torch.cuda.mem_get_info(0)
    return total - free


def run(d, M, T, X, dense_max, threads=0):
    """one hmk_clinkage_run on a fresh context -> (result or None, record)"""
    base = used_bytes()
    ctx = hb.GreedyContext(0, clinkage_dense_max=dense_max, clinkage_threads=threads, profile=1)
    try:
        t0 = time.perf_counter()
        rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], M, T, X, 0)
        wall = (time.perf_counter() - t0) * 1e3
        st, sec = ctx.stats(), ctx.section_ms()
        rec = {"status": rc, "message": err.decode(errors="replace"), "wall_ms": round(wall, 2),
               "total_ms": round(st["total_ms"], 3), "scoring_ms": round(sec["p1_select"], 3),
               "row_build_ms": round(sec["p1_partner"], 3), "chain_ms": round(sec["p1_cluster"], 3),
               "bulk_kernel_ms": round(st["bulk_kernel_ms"], 3), "pairs_scored": st["bulk_pairs"],
               "valid_pairs": st["xhits_kept"] // 2, "directed_entries": st["xhits_kept"],
               "nearest_searches": st["p1_steps"], "context_device_bytes": used_bytes() - base}
        if G is not None:
            rec.update(clusters=int(len(G.result_order)), multi=int(G.n_multi),
                       digest=hb.result_digest(G.cluster_id, G.member_rank, G.result_order))
        return G, rec
    finally:
        ctx.close()


def synthetic(n):
    d = synth.generate(n, 12, 12, seed=20260101)
    T, X, _ = synth.default_params(d["lengths"])
    return d, T, X


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_clinkage_scale.json"))
    ap.add_argument("--skip-1m", action="store_true")
    args = ap.parse_args()
    M = synth.blosum62()
    res = {"card": card(), "workloads": "BLOSUM62, T = round(1.7 x mean length), X = default, P = 0; synthetic: "
           "hammock_b200.synth.generate(n, 12, 12, seed=20260101) in generated order",
           "dense_vs_sparse": [], "sparse": [], "chain_threads": []}

    def log(x):                                            # the file is rewritten after every record
        print(json.dumps(x), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)

    z = np.load(os.path.join(ROOT, "tests", "golden", "musi_clinkage.npz"))
    musi = ({k: z[k] for k in ("residues", "offsets", "abundance")}, 20, 3)
    for name, (d, T, X) in (("musi", musi), ("synthetic_10000", synthetic(10000)), ("synthetic_32768", synthetic(32768))):
        row = {"input": name, "n": len(d["abundance"]), "dense": [], "sparse": []}
        for rep in range(3):                               # alternated in this process
            Gd, rd = run(d, M, T, X, 32768)
            Gs, rs = run(d, M, T, X, 0)
            row["dense"].append(rd)
            row["sparse"].append(rs)
            row["equal"] = bool(Gd is not None and Gs is not None and rd["digest"] == rs["digest"]
                                and rd["nearest_searches"] == rs["nearest_searches"]) and row.get("equal", True)
        res["dense_vs_sparse"].append(row)
        log(row)

    ab_res, ab_offs, ab_ab = input_arrays()
    ab = ({"residues": ab_res, "offsets": ab_offs, "abundance": ab_ab}, 20, 3)
    g = np.load(os.path.join(ROOT, "tests", "golden", "antibodies_clinkage.npz"))

    def sparse_at(name, d, T, X):
        G, rec = run(d, M, T, X, 32768)
        rec.update(input=name, n=len(d["abundance"]))
        if name == "antibodies":
            rec["equals_oracle_golden"] = bool(G is not None and (G.cluster_id == g["cluster_id"]).all()
                                               and (G.member_rank == g["member_rank"]).all()
                                               and (G.result_order == g["result_order"]).all()
                                               and rec["nearest_searches"] == int(g["nearest_searches"]))
        res["sparse"].append(rec)
        log(rec)

    for name, size in (("antibodies", None), ("synthetic_100000", 100_000), ("synthetic_200000", 200_000)):
        sparse_at(name, *(ab if size is None else synthetic(size)))

    zm = np.load(os.path.join(ROOT, "tests", "golden", "matrices.npz"))
    mc, T, X = synthetic(2000)
    for name, (d, M2, T2, X2) in (("antibodies", (ab[0], M, 20, 3)), ("synthetic_100000", (*synthetic(100_000)[:1], M, T, X)),
                                  ("mcla71_synthetic_2000", (mc, zm["mcla71"], T, X))):
        row = {"input": name, "runs": []}
        for threads in (64, 128, 256, 512, 1024, 0):
            _, rec = run(d, M2, T2, X2, 0, threads)
            row["runs"].append({"threads": threads or "auto", "chain_ms": rec["chain_ms"], "digest": rec["digest"],
                                "directed_entries": rec["directed_entries"]})
        res["chain_threads"].append(row)
        log(row)
    if not args.skip_1m:
        sparse_at("synthetic_1000000", *synthetic(1_000_000))
    print("wrote", args.out)


if __name__ == "__main__":
    main()
