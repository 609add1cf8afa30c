"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(libhammock_b200.so) and is compared bit-exactly with the CPU oracle on the same inputs, with
the committed goldens, and -- at full BASELINE sizes -- through size-independent properties."""
import json
import os

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import _lib, synth
from oracle import oracle as O
from tests import kats

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mats(golden_dir):
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    return {k: z[k] for k in z.files}


def run_gpu(d, M, T, X, P, K, **opts):
    ctx = hb.GreedyContext(0, **opts)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K)
        rc, msg = ctx.run_status()
        st = ctx.stats()
        return rc, (ctx.download() if rc == 0 else None), st
    finally:
        ctx.close()


def assert_same(R, G, what=""):
    assert G is not None, what
    bad = np.nonzero(R.cluster_id != G.cluster_id)[0]
    assert len(bad) == 0, f"{what}: cluster_id differs at {bad[:10]} oracle={R.cluster_id[bad[:10]]} gpu={G.cluster_id[bad[:10]]}"
    assert (R.member_rank == G.member_rank).all(), what
    assert len(R.result_order) == len(G.result_order) and (R.result_order == G.result_order).all(), what
    assert R.n_multi == G.n_multi, what


def oracle_run(d, M, T, X, P, K, **kw):
    return O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K, nthreads=os.cpu_count() or 1, **kw)


def test_library_loads_on_gpu():
    L = _lib.load()
    assert L.hmk_abi_version() == 2


def test_scorer_kats_gpu(mats):
    for a, b, X, P, m, score, _ in kats.SCORER_KATS:
        sc = hb.ShiftedScorer(mats[m], P, X)
        assert sc.sequence_score(hb.UniqueSequence(a), hb.UniqueSequence(b)) == score, (a, b)


def test_shift_too_big_gpu(blosum62):
    sc = hb.ShiftedScorer(blosum62, 0, 3)
    with pytest.raises(hb.DataException):
        sc.sequence_score(hb.UniqueSequence("ACD"), hb.UniqueSequence("ACDEFG"))
    d = synth.generate(50, 7, 12, seed=3)
    rc, _, _ = run_gpu(d, blosum62, 16, 7, 0, 2)
    assert rc == _lib.STATUS_SHIFT_TOO_BIG
    R = oracle_run(d, blosum62, 16, 7, 0, 2)
    assert R.status == O.ERR_SHIFT_TOO_BIG


@pytest.mark.parametrize("generic", [0, 1])
@pytest.mark.parametrize("case", [("blosum62", 3, 0), ("blosum62", 2, -1), ("pam250", 3, 0), ("blosum100", 1, -3),
                                  ("blosum30", 3, 0)])
def test_score_block_vs_oracle(golden_dir, mats, generic, case):
    """every pair score of a MUSI block, both kernels, several matrices / shifts / penalties"""
    m, X, P = case
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    ctx = hb.GreedyContext(0, force_generic=generic)
    ctx.upload(z["residues"], z["offsets"], z["abundance"], mats[m], 20, X, P, 61)
    rng = np.random.default_rng(7)
    first = rng.choice(2457, 400, replace=False).astype(np.int32)
    second = rng.choice(2457, 300, replace=False).astype(np.int32)
    got = ctx.score_block(first, second)
    assert ctx.stats() is not None
    ctx.close()
    res, offs = z["residues"], z["offsets"]
    for ia in range(0, 400, 7):
        for ib in range(0, 300, 11):
            a, b = first[ia], second[ib]
            exp = O.score_with_shift(res[offs[a]:offs[a + 1]], res[offs[b]:offs[b + 1]], mats[m], X, P)[0]
            assert got[ia, ib] == exp, (a, b, got[ia, ib], exp)


def test_score_block_asymmetric_matrix(golden_dir, blosum62):
    """orientation M[shorter][longer] (ShiftedScorer.java:71,75): use a deliberately asymmetric matrix"""
    M = blosum62.copy()
    M[np.triu_indices(24, 1)] += 1
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    res, offs = z["residues"], z["offsets"]
    for generic in (0, 1):
        ctx = hb.GreedyContext(0, force_generic=generic)
        ctx.upload(res, offs, z["abundance"], M, 20, 3, 0, 61)
        ids = np.arange(0, 2457, 41, dtype=np.int32)
        got = ctx.score_block(ids, ids)
        ctx.close()
        for i, a in enumerate(ids):
            for j, b in enumerate(ids):
                exp = O.score_with_shift(res[offs[a]:offs[a + 1]], res[offs[b]:offs[b + 1]], M, 3, 0)[0]
                assert got[i, j] == exp


def _micro():
    strs = kats.MICRO_ORDER
    ab = dict(kats.MICRO)
    res, offs = O.pack(strs)
    return {"residues": res, "offsets": offs, "abundance": np.array([ab[s] for s in strs], np.int32)}


@pytest.mark.parametrize("K", [2, 5, 0, 1])
def test_micro_fixture_gpu(blosum62, K):
    d = _micro()
    rc, G, _ = run_gpu(d, blosum62, 24, 2, 0, K)
    assert rc == 0
    if K in kats.MICRO_EXPECT:
        assert kats.result_to_lists(G.cluster_id, G.member_rank, G.result_order, G.n_multi) == kats.MICRO_EXPECT[K]
    assert_same(oracle_run(d, blosum62, 24, 2, 0, K), G)


def test_null_cluster_gpu(blosum62):
    res, offs = O.pack(["WWWWWWWWWW", "AAAAAAAAAA", "CCCCCCCCCC"])
    d = {"residues": res, "offsets": offs, "abundance": np.array([3, 2, 1], np.int32)}
    rc, _, st = run_gpu(d, blosum62, 24, 2, 0, 2)
    assert rc == _lib.STATUS_NULL_CLUSTER and st["error_step"] == 0
    res, offs = O.pack(["WWWWWWWWWW"])
    rc, _, _ = run_gpu({"residues": res, "offsets": offs, "abundance": np.array([1], np.int32)}, blosum62, 24, 2, 0, 1)
    assert rc == _lib.STATUS_NULL_CLUSTER
    with pytest.raises(hb.NullClusterError):
        hb.LimitedGreedySequenceClusterer(hb.ShiftedScorer(blosum62, 0, 2), 24, 2).cluster(
            [hb.UniqueSequence(s, {"x": c}) for s, c in (("WWWWWWWWWW", 3), ("AAAAAAAAAA", 2), ("CCCCCCCCCC", 1))])


def test_empty_and_tiny_inputs(blosum62):
    d = {"residues": np.zeros(0, np.uint8), "offsets": np.zeros(1, np.int32), "abundance": np.zeros(0, np.int32)}
    rc, G, _ = run_gpu(d, blosum62, 20, 3, 0, 5)
    assert rc == 0 and len(G.result_order) == 0
    res, offs = O.pack(["WVTAPRSLPVLP", "WVTAPRSLPVLA"])
    d = {"residues": res, "offsets": offs, "abundance": np.array([2, 1], np.int32)}
    for K in (0, 1, 3):
        rc, G, _ = run_gpu(d, blosum62, 20, 3, 0, K)
        R = oracle_run(d, blosum62, 20, 3, 0, K)
        assert rc == R.status
        if rc == 0:
            assert_same(R, G)
    bad = {"residues": np.array([1, 2, 24, 3], np.uint8), "offsets": np.array([0, 2, 4], np.int32),
           "abundance": np.array([1, 1], np.int32)}
    rc, _, _ = run_gpu(bad, blosum62, 20, 1, 0, 1)
    assert rc == _lib.STATUS_BAD_RESIDUE


@pytest.mark.parametrize("opts", [{}, {"force_generic": 1}, {"batch": 7, "kb": 1}, {"batch": 64, "kb": 2, "qt": 16},
                                  {"batch": 512, "waves": 1}, {"p2_chunk": 1024, "hit_cap": 1024, "p2_window": 100, "capq": 1},
                                  {"lookahead": 0, "p2_window": 300}, {"lookahead": 1, "batch": 16, "p2_window": 64}])
def test_musi_golden_gpu(golden_dir, blosum62, opts):
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    T, X, P, K = (int(v) for v in z["params"])
    rc, G, st = run_gpu(z, blosum62, T, X, P, K, **opts)
    assert rc == 0
    assert (G.cluster_id == z["cluster_id"]).all() and (G.member_rank == z["member_rank"]).all()
    assert (G.result_order == z["result_order"]).all() and G.n_multi == int(z["n_multi"])
    assert (st["p1_steps"], st["p1_joins"], st["p1_new_clusters"], st["p2_queries"], st["p2_assigned"]) == (67, 6, 61, 2329, 574)
    assert st["fast_path"] == (0 if opts.get("force_generic") else 1)


def test_musi_reference_interface(golden_dir, blosum62):
    """the host mirror end to end: UniqueSequence list -> List<Cluster>"""
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    strs = synth.to_strings(z["residues"], z["offsets"])
    rng = np.random.default_rng(1)
    seqs = [hb.UniqueSequence(strs[i], {"no_label": int(z["abundance"][i])}) for i in rng.permutation(len(strs))]
    clusters = hb.run_greedy_clustering(seqs, blosum62)
    assert [c.get_id() for c in clusters] == z["result_order"].tolist()
    for c in clusters[:int(z["n_multi"])]:
        mem = np.nonzero(z["cluster_id"] == c.get_id())[0]
        mem = mem[np.argsort(z["member_rank"][mem])]
        assert [s.get_sequence_string() for s in c.get_sequences()] == [strs[m] for m in mem]
        assert c.size() == int(z["abundance"][mem].sum())


@pytest.mark.parametrize("opts", [{}, {"batch": 48, "kb": 2}, {"reuse": 0}])
def test_antibodies_golden_gpu(golden_dir, blosum62, opts):
    z = np.load(os.path.join(golden_dir, "antibodies.npz"))
    T, X, P, K = (int(v) for v in z["params"])
    rc, G, st = run_gpu(z, blosum62, T, X, P, K, **opts)
    assert rc == 0
    bad = np.nonzero(G.cluster_id != z["cluster_id"])[0]
    assert len(bad) == 0, (bad[:10], G.cluster_id[bad[:10]], z["cluster_id"][bad[:10]])
    assert (G.member_rank == z["member_rank"]).all() and (G.result_order == z["result_order"]).all()
    assert (st["p1_steps"], st["p1_joins"], st["p1_new_clusters"]) == (1923, 72, 1851)
    if opts.get("reuse") == 0:   # every founder x single pair is scored again in phase 2
        assert st["bulk_pairs"] + st["scalar_pairs"] >= 140546010 + 130649021   # >= the reference's early-exit count


SYNTH_CASES = [
    # n, min_len, max_len, matrix, P, K override, abundance shuffle, options
    (4000, 12, 12, "blosum62", 0, None, False, {}),
    (4000, 12, 12, "blosum62", -1, None, False, {"batch": 32}),
    (3000, 7, 12, "blosum62", 0, None, False, {}),                 # mixed lengths -> packed kernel per length bucket
    (3000, 7, 12, "blosum62", -2, None, False, {"batch": 16, "kb": 2}),
    (3000, 9, 9, "pam250", 0, None, False, {}),
    (3000, 12, 12, "blosum30", 0, None, False, {}),
    (2500, 12, 12, "blosum100", 0, None, False, {}),               # wide range: 16-bit lanes
    (3000, 12, 12, "blosum62", 0, 1000, False, {}),                # K large: phase 1 runs to exhaustion
    (3000, 12, 12, "blosum62", 0, None, True, {}),                 # abundance not sorted -> tie-rank path
    (1500, 16, 16, "blosum62", 0, None, False, {}),                # two packed words -> long packed kernel (s16 lanes)
    (1500, 30, 30, "blosum62", -1, None, False, {}),               # three packed words, 17 diagonals
    (2000, 13, 18, "blosum45", 0, None, False, {"batch": 40}),     # mixed lengths on the long kernel
    (1500, 20, 20, "blosum62", 0, None, False, {"force_generic": 1}),
    (2000, 7, 30, "blosum50", 0, None, False, {}),
    (4000, 12, 12, "blosum62", 0, None, False, {"filter": 0}),             # exact packed kernel instead of filter + verify
    (4000, 12, 12, "blosum62", 0, None, False, {"reuse": 0}),              # separate founder pass in phase 2
    (3000, 7, 12, "blosum62", 0, None, False, {"reuse": 0, "batch": 24}),
    (3000, 10, 10, "blosum62", -1, None, False, {"batch": 8, "kb": 1}),     # truncated partner lists -> restarts, hits of re-done batches
    (3000, 11, 11, "blosum62", 0, 200, True, {"batch": 20, "kb": 2}),
    (6000, 12, 12, "blosum62", 0, 60, False, {"p2_window": 256}),      # few clusters, many joiners per cluster and window
    (6000, 12, 12, "blosum62", 0, 60, False, {"p2_window": 100000, "hit_cap": 1024}),
    (5000, 12, 12, "blosum62", 0, None, False, {"batch": 32, "lookahead": 2, "hit_cap": 1024}),   # founder-hit buffer grows in the resolver
    (5000, 12, 12, "blosum62", 0, None, False, {"batch": 32, "lookahead": 1}),
    (5000, 12, 12, "blosum62", 0, None, False, {"batch": 32, "lookahead": 0}),
]


@pytest.mark.parametrize("case", SYNTH_CASES)
def test_synthetic_vs_oracle(mats, case):
    n, lo, hi, m, P, K, shuffle, opts = case
    d = synth.generate(n, lo, hi, seed=1000 + n + hi)
    if shuffle:
        rng = np.random.default_rng(5)
        d["abundance"] = np.ascontiguousarray(rng.permutation(d["abundance"]))
    T, X, K0 = synth.default_params(d["lengths"])
    K = K0 if K is None else K
    R = oracle_run(d, mats[m], T, X, P, K)
    rc, G, st = run_gpu(d, mats[m], T, X, P, K, **opts)
    assert rc == R.status
    if rc == 0:
        assert_same(R, G, str(case))
        assert st["p1_steps"] == R.counters["p1_steps"] and st["p2_assigned"] == R.counters["p2_assigned"]


def test_uniform_random_with_orphans(blosum62):
    """background-only data: many orphans in phase 1, high threshold"""
    rng = np.random.default_rng(11)
    n = 1500
    res = rng.integers(0, 20, size=n * 12, dtype=np.uint8)
    offs = np.arange(0, 12 * (n + 1), 12, dtype=np.int32)
    ab = np.sort(rng.integers(1, 50, size=n))[::-1].astype(np.int32)
    d = {"residues": res, "offsets": offs, "abundance": np.ascontiguousarray(ab)}
    # first make sure the first query has a partner (else NPE): low threshold
    for T, K in ((12, 40), (18, 200), (30, 10)):
        R = oracle_run(d, blosum62, T, 3, 0, K)
        rc, G, _ = run_gpu(d, blosum62, T, 3, 0, K, batch=50, kb=2)
        assert rc == R.status
        if rc == 0:
            assert_same(R, G, f"T={T}")


def test_s100k_vs_oracle(blosum62, golden_dir):
    """BASELINE config 1: synthetic 100k unique peptides, length 7-12, Zipf abundance, BLOSUM62"""
    d = synth.generate(100000, 7, 12)
    T, X, K = synth.default_params(d["lengths"])
    assert (T, X, K) == (16, 2, 2500)
    R = oracle_run(d, blosum62, T, X, 0, K)
    rc, G, st = run_gpu(d, blosum62, T, X, 0, K)
    assert rc == 0 and R.status == 0
    assert_same(R, G, "S100k")
    gold = json.load(open(os.path.join(golden_dir, "s100k_digest.json")))
    assert hb.result_digest(G.cluster_id, G.member_rank, G.result_order) == gold["sha256"]


def test_s1m_properties(blosum62, golden_dir):
    """BASELINE config 2 at full size (1M unique 12-mers): the oracle cannot finish, so check
    (a) a prefix of phase 1 against the bounded oracle, (b) complete linkage of every cluster,
    (c) maximality for sampled singletons, (d) independence from batch size."""
    d = synth.generate(1000000)
    T, X, K = synth.default_params(d["lengths"])
    assert (T, X, K) == (20, 3, 25000)
    ctx = hb.GreedyContext(0)
    ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, K)
    rc, _ = ctx.run_status()
    assert rc == 0
    G = ctx.download()
    st = ctx.stats()
    assert G.n_multi == K and st["p1_new_clusters"] == K
    # (0) bit-exact against the FULL oracle run on this input: tests/golden/s1m_digest.json
    # (scripts/make_s1m_digest.py; sha256 over cluster_id || member_rank || result_order)
    gold = json.load(open(os.path.join(golden_dir, "s1m_digest.json")))
    assert (gold["n"], gold["threshold"], gold["max_shift"], gold["max_clusters"]) == (1000000, T, X, K)
    assert hb.result_digest(G.cluster_id, G.member_rank, G.result_order) == gold["sha256"]
    assert (st["p1_steps"], st["p1_joins"], st["p1_orphans"], st["p2_assigned"]) == (
        gold["counters"]["p1_steps"], gold["counters"]["p1_joins"], gold["counters"]["p1_orphans"], gold["counters"]["p2_assigned"])
    assert st["flags"] & _lib.FLAG_P2_REUSED and not st["flags"] & _lib.FLAG_XHIT_OVERFLOW
    # (a) first 150 phase-1 steps of the oracle: same founders and partners
    R = oracle_run(d, blosum62, T, X, 0, K, max_p1_steps=150, max_p2_queries=1)
    founders = R.result_order[:R.n_multi]
    assert (G.result_order[:len(founders)] == founders).all()
    for f in founders:
        assert G.cluster_id[f] == f
        p = np.nonzero((R.cluster_id == f) & (R.member_rank == 1))[0][0]
        assert G.cluster_id[p] == f and G.member_rank[p] == 1
    # (b) complete linkage inside sampled clusters; ranks are a permutation
    rng = np.random.default_rng(3)
    order = np.argsort(G.cluster_id, kind="stable")
    cid_sorted = G.cluster_id[order]
    starts = np.nonzero(np.r_[True, cid_sorted[1:] != cid_sorted[:-1]])[0]
    ends = np.r_[starts[1:], len(order)]
    multi = [(s, e) for s, e in zip(starts, ends) if e - s > 1]
    assert len(multi) == K
    for s, e in [multi[i] for i in rng.choice(len(multi), 300, replace=False)]:
        mem = order[s:e].astype(np.int32)
        assert sorted(G.member_rank[mem].tolist()) == list(range(e - s))
        sc = ctx.score_block(mem, mem)
        assert (sc + np.eye(len(mem), dtype=np.int32) * 10 ** 6 >= T).all()
    # (c) sampled remaining singletons: no cluster accepts them (some member scores < T)
    singles = G.result_order[G.n_multi:]
    sample = rng.choice(singles, 64, replace=False).astype(np.int32)
    members = order[np.isin(cid_sorted, G.result_order[:G.n_multi])].astype(np.int32)
    sc = ctx.score_block(members, sample)                      # S(member, query)
    ok = sc >= T
    mcid = G.cluster_id[members]
    for j in range(len(sample)):
        bad_clusters = np.unique(mcid[~ok[:, j]])
        assert len(bad_clusters) == K, "a remaining singleton is accepted by some cluster"
    # (d) a different batching gives the identical clustering
    ctx.set_option("batch", 77)
    ctx.set_option("kb", 3)
    rc, _ = ctx.run_status()
    assert rc == 0
    G2 = ctx.download()
    assert (G2.cluster_id == G.cluster_id).all() and (G2.member_rank == G.member_rank).all()
    assert hb.result_digest(G2.cluster_id, G2.member_rank, G2.result_order) == gold["sha256"]
    ctx.close()


def test_bench_dump_outputs_match_the_oracle(tmp_path):
    """`bench.py --dump-outputs DIR` writes the clustering of the last timed step (float64 .npy): equal to the oracle's
    full run on the same seeded input, here on a small set"""
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "3", "--n", "20000",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["n_sequences"] == 20000
    d, M, (T, X, P, K) = bench.workload(20000)
    R = oracle_run(d, M, T, X, P, K)
    assert R.status == 0
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("cluster_id", "member_rank", "result_order", "n_multi")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert (got["cluster_id"] == R.cluster_id).all() and (got["member_rank"] == R.member_rank).all()
    assert (got["result_order"] == R.result_order).all() and got["n_multi"].tolist() == [R.n_multi]
    assert line["result_digest"] == hb.result_digest(R.cluster_id, R.member_rank, R.result_order)


def test_cpp_host_driver_end_to_end(tmp_path, golden_dir, blosum62):
    """hammock_greedy (C++ host side + C ABI): fasta in, the reference's result files out; compared with the
    Python mirror's writers on the same clustering and with the MUSI golden assignment."""
    import subprocess
    from hammock_b200 import build as hb_build
    exe = hb_build.build_host()
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    strs = synth.to_strings(z["residues"], z["offsets"])
    rng = np.random.default_rng(4)
    labs = ["rep1", "rep2", "ctrl"]
    fa = tmp_path / "in.fa"
    with open(fa, "w") as f:
        for k, i in enumerate(rng.permutation(len(strs))):
            f.write(f">s{k}|{int(z['abundance'][i])}|{labs[k % 3]}\n{strs[i]}\n")
    mp = tmp_path / "m.txt"
    with open(mp, "w") as f:
        f.write("# test copy of BLOSUM62\n   " + "  ".join(hb.ALPHABET) + "\n")
        for i in range(24):
            f.write(hb.ALPHABET[i] + " " + " ".join(f"{int(v):2d}" for v in blosum62[i]) + "\n")
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([exe, "greedy", "-i", str(fa), "-d", str(out), "-m", str(mp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    # same pipeline through the Python mirror
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    labels = hb.get_sorted_labels(seqs)
    ordered = hb.sort_sequences(seqs, "size", labels)
    clusters = hb.LimitedGreedySequenceClusterer(hb.ShiftedScorer(hb.load_scoring_matrix(str(mp)), 0, hb.get_max_shift(seqs)),
                                                 hb.set_greedy_threshold(seqs), hb.initial_clusters_limit(seqs)).cluster(ordered)
    ref = tmp_path / "ref"
    ref.mkdir()
    hb.save_cluster_sequences_to_csv(clusters, str(ref / "initial_clusters_sequences.tsv"), labels)
    hb.save_cluster_sequences_to_csv_ordered(clusters, str(ref / "initial_clusters_sequences_original_order.tsv"), labels, seqs)
    hb.save_clusters_to_csv(clusters, str(ref / "initial_clusters.tsv"), labels)
    hb.save_input_statistics(seqs, labels, str(ref / "input_statistics.tsv"))
    for fn in ("initial_clusters_sequences.tsv", "initial_clusters_sequences_original_order.tsv", "initial_clusters.tsv",
               "input_statistics.tsv"):
        assert (out / fn).read_text() == (ref / fn).read_text(), fn
    # ... and against the oracle's restatement of the reference writers (oracle/pyref_writers.py)
    from oracle import pyref_writers as W
    tup = lambda s: (s.get_sequence_string(), dict(s.labels_map))
    ct = [(c.get_id(), [tup(s) for s in c.get_sequences()]) for c in clusters]
    assert (out / "initial_clusters_sequences.tsv").read_text() == W.cluster_sequences_tsv(ct, labels)
    assert (out / "initial_clusters_sequences_original_order.tsv").read_text() == W.cluster_sequences_tsv_ordered(ct, labels, [tup(s) for s in seqs])
    assert (out / "initial_clusters.tsv").read_text() == W.clusters_tsv(ct, labels)
    assert (out / "input_statistics.tsv").read_text() == W.input_statistics([tup(s) for s in seqs], labels)
    # all abundances are 1 in MUSI and the clustering order is (abundance, string) -> same order as the golden
    got = {}
    for line in (out / "initial_clusters_sequences.tsv").read_text().splitlines()[1:]:
        cid, s = line.split("\t")[:2]
        got[s] = int(cid)
    assert [got[s] for s in strs] == z["cluster_id"].tolist()
