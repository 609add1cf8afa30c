"""CPU model of the shared residue prefix in hmk_bulk_filter: how many warps of 32 consecutive database items share
residues 0..u-1, and the filter's shared-memory wavefronts per warp-query with and without the prefix sums.

Workload: the benchmark's 1 M 12-mer set (hammock_b200/synth.py, seed 20260101), walked in id order, which is the
clustering order the kernel's warps hold (abundance, then sequence, both descending).  Every item counts as scored.

Wavefronts are counted per warp-wide instruction as in scripts/filter_wavefronts.py (the most distinct 4-byte words any
one bank is asked for, bank = word mod 32):
  U = 0 block: 12 filter look-ups per query, each conflict free (one 24-word row per position);
  U = 3 block: 9 look-ups (rows 3..11), one broadcast LDS.128 of four queries' prefix sums (0.25 per query), and per
               item block the prefix sums themselves -- lane l sums rows 0..2 of queries l, l + 32 (profile stride 868
               words, so 32 lanes hit 8 banks) and stores them -- spread over the tile's queries.
The second part is a model, not a measurement.

usage: python scripts/prefix_share.py [n=1000000]   -> profiles/r05_prefix_share.json"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hammock_b200 import synth          # noqa: E402

FPW, SUB, ROW, QT, L, U = 868, 288, 24, 56, 12, 3


def share(res, order):
    r = res[order]
    m = len(r) // 32 * 32
    w = r[:m].reshape(-1, 32, L)
    return {u: float((w[:, :, :u] == w[:, :1, :u]).all(axis=(1, 2)).mean()) for u in range(1, 5)}


def lds_wavefronts(words):
    u = np.unique(words)
    return int(np.bincount(u % 32, minlength=32).max()) if len(u) else 0


def partial_wavefronts(qn, residues):
    """prefix sums of one item block: per lane round, HMK_PREFIX_RES look-ups and one store"""
    total = 0
    for t0 in range(0, qn, 32):
        t = np.arange(t0, min(qn, t0 + 32))
        for j in range(U):
            total += lds_wavefronts(t * FPW + 2 * SUB + j * ROW + residues[j])
        total += lds_wavefronts(t)                      # pfx[t]: consecutive words
    return total


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
    d = synth.generate(n, L, L, seed=20260101)
    res = np.asarray(d["residues"]).reshape(-1, L).astype(np.int64)
    by_id = share(res, np.arange(len(res)))
    key = ((res[:, 0] * 24 + res[:, 1]) * 24 + res[:, 2]) * 24 + res[:, 3]
    sorted_ = share(res, np.argsort(key, kind="stable"))
    f = by_id[U]
    part = partial_wavefronts(QT, [5, 9, 13]) / QT
    u3 = (L - U) + 0.25 + part
    weighted = f * u3 + (1 - f) * L
    out = {
        "workload": f"synth.generate({n}, 12, 12, seed=20260101), warps of 32 consecutive ids",
        "share_of_warps_with_common_residues_0_to_u_minus_1": {"id_order": by_id, "sorted_by_residues_0_3": sorted_},
        "model_wavefronts_per_warp_query": {
            "U0_block": L, "U3_block": round(u3, 3), "U3_partials_per_query_at_qn56": round(part, 3),
            "weighted": round(weighted, 3), "change": round(weighted / L - 1, 4)},
        "note": "model only; filter look-ups of the query loop, not the verify, hit or tile-load traffic",
    }
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    path = os.path.join(ROOT, "profiles", "r05_prefix_share.json")
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
        fh.write("\n")
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
