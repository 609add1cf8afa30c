"""Golden result of the EXACT complete-linkage clusterer on the antibodies fixture (74 041 sequences, above the dense
engine path's 32 768 limit), produced by the C oracle (oracle/clinkage_oracle.c).  PARITY UNPINNED: no JVM, no
reference outputs.

Hammock.runClinkageClustering does not sort, so the golden is in INPUT order.  antibodies.npz stores the clustering
(sorted) order: sorted position i holds input sequence input_perm[i].  With inv the inverse permutation, input sequence
j is sorted position inv[j].  input_arrays() rebuilds the input-order arrays; the golden holds no copy of the residues.

    python tests/golden/make_antibodies_clinkage_golden.py      (about 6 minutes on 8 cores, about 21 GB resident)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O      # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def input_arrays():
    """-> (residues u8, offsets i32[n+1], abundance i32[n]) of the antibodies fixture in input order"""
    z = np.load(os.path.join(GOLDEN, "antibodies.npz"))
    res, offs, ab, perm = z["residues"], z["offsets"].astype(np.int64), z["abundance"], z["input_perm"]
    n = len(ab)
    inv = np.empty(n, np.int64)
    inv[perm] = np.arange(n)
    lens = (offs[1:] - offs[:-1])[inv]
    o2 = np.zeros(n + 1, np.int32)
    o2[1:] = np.cumsum(lens)
    r2 = np.concatenate([res[offs[inv[j]]:offs[inv[j] + 1]] for j in range(n)]).astype(np.uint8)
    return r2, o2, np.ascontiguousarray(ab[inv]).astype(np.int32)


def main():
    res, offs, ab = input_arrays()
    M = np.load(os.path.join(GOLDEN, "matrices.npz"))["blosum62"]
    T, X, _ = O.default_params(offs)          # setClinkageThreshold == setGreedyThreshold: round(1.7 * mean length)
    R = O.clinkage_cluster(res, offs, ab, M, T, X, 0)
    assert R.status == 0, R.status
    np.savez_compressed(os.path.join(GOLDEN, "antibodies_clinkage.npz"), params=np.array([T, X, 0], np.int32),
                        cluster_id=R.cluster_id, member_rank=R.member_rank, result_order=R.result_order,
                        nearest_searches=np.int64(R.nearest_searches))
    sizes = np.bincount(R.cluster_id)
    print("n", len(ab), "T", T, "X", X, "clusters", len(R.result_order), "multi-member", int((sizes > 1).sum()),
          "largest", int(sizes.max()), "searches", R.nearest_searches, "first ids", R.result_order[:8].tolist())


if __name__ == "__main__":
    main()
