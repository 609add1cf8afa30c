"""Exact complete-linkage clustering beyond the dense n x n score matrix: the sparse path of hmk_clinkage_cluster /
hmk_clinkage_run (rows of the pairs scoring >= T, hmk_clinkage_chain_sparse).
CPU: a model of the sparse kernel's logic against the second restatement; sanity of the committed antibodies golden.
GPU (-m gpu): the sparse path forced on small inputs against the C oracle, against the dense path, and the default entry
on inputs above 32 768 sequences (antibodies golden, 100 000 synthetic 12-mers, status codes)."""
import os
import subprocess

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import _lib, build as hb_build, synth
from oracle import oracle as O, pyref_clinkage as PC
from tests.golden.make_antibodies_clinkage_golden import input_arrays as antibodies_input


def _input_order_case(n, lo, hi, seed):
    """a synthetic set in a shuffled (input) order: runClinkageClustering does not sort (Hammock.java:449-462)"""
    d = synth.generate(n, lo, hi, seed=seed)
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n)
    res, offs = d["residues"], d["offsets"]
    seqs = [res[offs[i]:offs[i + 1]] for i in perm]
    o = np.zeros(n + 1, np.int32)
    o[1:] = np.cumsum([len(s) for s in seqs])
    T, X, _ = synth.default_params(d["lengths"])
    return {"residues": np.concatenate(seqs), "offsets": o, "abundance": np.ascontiguousarray(d["abundance"][perm])}, seqs, T, X


def _well_formed(cid, rank, order):
    """singletons keep id i + 1 (<= n), merged clusters n + 2 .. 2n + 1; ranks 0 .. size - 1; the list holds every id once"""
    n = len(cid)
    ids = np.unique(cid)
    assert len(order) == len(ids) and (np.sort(order) == ids).all()
    sizes = np.bincount(cid, minlength=2 * n + 2)
    single = sizes[cid] == 1
    assert (cid[single] == np.nonzero(single)[0] + 1).all() and (rank[single] == 0).all()
    assert ((cid[~single] >= n + 2) & (cid[~single] <= 2 * n + 1)).all()
    key = cid.astype(np.int64) * (n + 1) + rank
    assert len(np.unique(key)) == n and (rank < sizes[cid]).all() and (rank >= 0).all()


def _member_lists(cid, rank):
    """cluster id -> members in getSequences() order, multi-member clusters only"""
    o = np.lexsort((rank, cid))
    c = cid[o]
    cuts = np.nonzero(np.diff(c))[0] + 1
    return {int(g[0]): m for g, m in zip(np.split(c, cuts), np.split(o, cuts)) if len(m) > 1}


# ------------------------------------------------------------------------------------------------ CPU model of the sparse kernel
def _sparse_chain_model(pair, ab, T):
    """The LOGIC of hmk_clinkage_chain_sparse (hmk_kernels.cuh), not its CUDA: rows hold only the entries scoring >= T,
    sorted by slot, with the position of every entry's mirror (twin); a merge intersects row(bs) into row(ts) IN PLACE
    (entries that leave the intersection are killed, not removed, so positions and twins stay valid) and writes the
    minimum into the mirror entries; inactive slots are skipped lazily; the chain restarts from a lowest-bin cursor."""
    n = len(ab)
    DEAD = -(2 ** 31)
    rows = [[[b, int(pair[a][b])] for b in range(n) if b != a and pair[a][b] >= T] for a in range(n)]
    twin = [[next(i for i, e in enumerate(rows[b]) if e[0] == a) for b, _ in rows[a]] for a in range(n)]
    hsh = lambda cid: ((553 + cid) & 0xFFFFFFFF) ^ (((553 + cid) & 0xFFFFFFFF) >> 16)
    acap = 16
    while n > int(acap * 0.75):
        acap *= 2
    bins = [[] for _ in range(acap)]
    id_of = [i + 1 for i in range(n)]
    slot_of = {i + 1: i for i in range(n)}
    size_of = [int(a) for a in ab]
    members = [[i] for i in range(n)]
    for cid in range(1, n + 1):
        bins[hsh(cid) & (acap - 1)].append(cid)
    cursor = min(hsh(cid) & (acap - 1) for cid in range(1, n + 1))
    nactive, cur_id, stack, ready = n, n + 1, [], []
    while True:
        if not stack:
            if nactive <= 1:
                break
            while not bins[cursor]:
                cursor += 1
            assert cursor == next(b for b in range(acap) if bins[b])     # the cursor is the lowest non-empty bin
            stack.append(bins[cursor][0])
        top = stack[-1]
        ts = slot_of[top]
        best = None                                    # (score, size, id) under score desc, size desc, id asc
        for k, sc in rows[ts]:
            if sc < T or id_of[k] < 0:
                continue
            cand = (sc, size_of[k], id_of[k])
            if best is None or (-cand[0], -cand[1], cand[2]) < (-best[0], -best[1], best[2]):
                best = cand
        if best is None:
            stack.pop()
            ready.append(top)
            bins[hsh(top) & (acap - 1)].remove(top)
            nactive -= 1
            id_of[ts] = -1
        elif len(stack) > 1 and stack[-2] == best[2]:
            bs = slot_of[best[2]]
            slots_bs = [e[0] for e in rows[bs]]
            assert slots_bs == sorted(slots_bs)
            for p, e in enumerate(rows[ts]):
                k, sc = e
                if sc < T:
                    continue
                m = DEAD
                live = k != bs and id_of[k] >= 0
                if live and k in slots_bs:
                    sb = rows[bs][slots_bs.index(k)][1]
                    if sb >= T:
                        m = min(sc, sb)
                e[1] = m
                if live:
                    mirror = rows[k][twin[ts][p]]
                    assert mirror[0] == ts
                    mirror[1] = m
            cur_id += 1
            stack.pop(); stack.pop()
            for cid in (top, best[2]):
                bins[hsh(cid) & (acap - 1)].remove(cid)
            members[ts] = members[ts] + members[bs]
            size_of[ts] = (size_of[ts] + size_of[bs] + 2 ** 31) % 2 ** 32 - 2 ** 31
            id_of[ts], id_of[bs] = cur_id, -1
            slot_of[cur_id] = ts
            b = hsh(cur_id) & (acap - 1)
            bins[b].append(cur_id)
            cursor = min(cursor, b)
            nactive -= 1
        else:
            stack.append(best[2])
    ready.append(next(bins[b] for b in range(cursor, acap) if bins[b])[0])
    rs = PC.JavaHashSet()
    for cid in ready:
        rs.add(cid)
    order = list(rs)
    cluster_id, member_rank = np.zeros(n, np.int32), np.zeros(n, np.int32)
    for cid in order:
        for r, m in enumerate(members[slot_of[cid]]):
            cluster_id[m], member_rank[m] = cid, r
    return cluster_id, member_rank, np.array(order, np.int32)


@pytest.mark.parametrize("n", [1, 2, 3, 11, 12, 13, 14, 24, 25, 26, 48, 49, 50, 96, 97, 130])
def test_sparse_chain_kernel_model(blosum62, n):
    """the sparse kernel's scheme against the second restatement around the HashMap growth points, at the default
    threshold, at T - 7 (dense rows) and at a threshold no pair reaches (every sequence isolated)"""
    from oracle.pyref import PyRef
    for seed in range(3):
        d, seqs, T, X = _input_order_case(n, 9, 12, 100 * n + seed)
        ref = PyRef(seqs, d["abundance"], blosum62, T, X, 0, 0)
        pair = np.empty((n, n), dtype=np.int64)
        for q in range(n):
            pair[:, q] = ref.scores(np.arange(n), q)
        for T2 in (T, T - 7, int(pair.max()) + 1):
            want = PC.clinkage_cluster(seqs, d["abundance"], blosum62, T2, X, 0)
            got = _sparse_chain_model(pair, d["abundance"], T2)
            for g, w in zip(got, want):
                assert (g == w).all(), (n, seed, T2)


def test_antibodies_clinkage_golden_sanity(golden_dir, blosum62):
    """the committed golden, checked independently of how it was made: well-formed ids and ranks, and every member pair
    of every multi-member cluster scores >= T (complete linkage) with the oracle's scorer"""
    z = np.load(os.path.join(golden_dir, "antibodies_clinkage.npz"))
    res, offs, ab = antibodies_input()
    n = len(ab)
    T, X, P = (int(v) for v in z["params"])
    assert n == 74041 and (T, X, P) == (20, 3, 0) and (T, X, P)[:2] == O.default_params(offs)[:2]
    cid, rank, order = z["cluster_id"], z["member_rank"], z["result_order"]
    assert len(cid) == len(rank) == n
    _well_formed(cid, rank, order)
    assert len(order) == len(np.unique(cid))
    pairs = 0
    for mem in _member_lists(cid, rank).values():
        for i in range(len(mem)):
            a = res[offs[mem[i]]:offs[mem[i] + 1]]
            for j in range(i + 1, len(mem)):
                assert O.score_with_shift(a, res[offs[mem[j]]:offs[mem[j] + 1]], blosum62, X, P)[0] >= T
                pairs += 1
    assert pairs > 29747


# ------------------------------------------------------------------------------------------------ GPU
CASES = [(2, 12, 12, 1), (3, 12, 12, 2), (40, 12, 12, 3), (700, 7, 12, 4), (1500, 12, 12, 5), (900, 9, 9, 6),
         (600, 16, 16, 7), (400, 7, 30, 8), (3000, 12, 12, 9),
         (12, 12, 12, 10), (13, 12, 12, 11), (25, 9, 12, 12), (49, 12, 12, 13)]   # those of test_clinkage_gpu_vs_oracle


def _sparse_ctx(**kw):
    return hb.GreedyContext(0, clinkage_dense_max=0, **kw)


def _check_vs_oracle(ctx, d, M, T, X, P):
    R = O.clinkage_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, P)
    rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], M, T, X, P)
    assert rc == R.status == 0, (rc, R.status, err)
    assert (G.cluster_id == R.cluster_id).all() and (G.member_rank == R.member_rank).all()
    assert (G.result_order == R.result_order).all()
    assert G.n_multi == int((np.bincount(R.cluster_id) > 1).sum())
    assert G.stats["p1_steps"] == R.nearest_searches
    return G


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_sparse_clinkage_gpu_vs_oracle(golden_dir, blosum62, case):
    n, lo, hi, seed = case
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    d, _, T, X = _input_order_case(n, lo, hi, seed)
    ctx = _sparse_ctx()
    try:
        for M, T2, P in ((blosum62, T, 0), (z["pam250"], T + 3, -1), (z["blosum100"], T - 5, 0)):
            G = _check_vs_oracle(ctx, d, M, T2, X, P)
            assert G.stats["xhits_kept"] % 2 == 0 and G.stats["xhits_capacity"] >= G.stats["xhits_kept"]
    finally:
        ctx.close()


@pytest.mark.gpu
def test_sparse_clinkage_musi_golden(golden_dir, blosum62):
    z = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
    T, X, P = (int(v) for v in z["params"])
    ctx = _sparse_ctx(profile=1)
    try:
        rc, G, err = ctx.clinkage(z["residues"], z["offsets"], z["abundance"], blosum62, T, X, P)
        assert rc == 0, err
        assert (G.cluster_id == z["cluster_id"]).all() and (G.member_rank == z["member_rank"]).all()
        assert (G.result_order == z["result_order"]).all()
        assert G.stats["p1_steps"] == int(z["nearest_searches"])
        sec = ctx.section_ms()
        assert sec["p1_select"] > 0 and sec["p1_partner"] > 0 and sec["p1_cluster"] > 0 and G.stats["total_ms"] > 0
    finally:
        ctx.close()


@pytest.mark.gpu
def test_sparse_clinkage_special_inputs(golden_dir, blosum62):
    """mixed lengths 7..30 (generic-kernel EMIT), MCLA71 where almost every 12-mer pair passes T (rows of nearly n - 1
    entries; the row storage holds exactly the pairs the oracle's scorer puts >= T), and a threshold no pair reaches
    (every sequence isolated), each with both chain block shapes"""
    from oracle.pyref import PyRef
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    ctx = _sparse_ctx()
    try:
        d, _, T, X = _input_order_case(2000, 7, 30, 21)
        G = _check_vs_oracle(ctx, d, blosum62, T, X, 0)
        assert G.stats["fast_path"] == 0
        d, seqs, T, X = _input_order_case(2000, 12, 12, 22)
        ref = PyRef(seqs, d["abundance"], z["mcla71"], T, X, 0, 0)
        valid = sum(int((ref.scores(np.arange(2000), q) >= T).sum()) - 1 for q in range(2000))   # minus the self pair
        assert valid > 0.99 * 2000 * 1999
        for threads in (0, 1024):
            ctx.set_option("clinkage_threads", threads)
            G = _check_vs_oracle(ctx, d, z["mcla71"], T, X, 0)
            assert G.stats["xhits_kept"] == valid
            G = _check_vs_oracle(ctx, d, blosum62, 200, X, 0)
            assert G.stats["xhits_kept"] == 0 and len(G.result_order) == 2000 and G.n_multi == 0
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [10000, 32768])
def test_sparse_equals_dense_on_gpu(blosum62, n):
    d, _, T, X = _input_order_case(n, 12, 12, 30 + n)
    outs = []
    for dense_max in (32768, 0):
        ctx = hb.GreedyContext(0, clinkage_dense_max=dense_max)
        try:
            rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0)
            assert rc == 0, err
            outs.append(G)
        finally:
            ctx.close()
    a, b = outs
    assert a.stats["xhits_kept"] == 0 and b.stats["xhits_kept"] > 0
    assert (a.cluster_id == b.cluster_id).all() and (a.member_rank == b.member_rank).all()
    assert (a.result_order == b.result_order).all() and a.n_multi == b.n_multi
    assert a.stats["p1_steps"] == b.stats["p1_steps"]


@pytest.fixture(scope="module")
def antibodies(golden_dir):
    res, offs, ab = antibodies_input()
    return res, offs, ab, np.load(os.path.join(golden_dir, "antibodies_clinkage.npz"))


@pytest.mark.gpu
def test_antibodies_clinkage_default_entry(antibodies, blosum62):
    """74 041 sequences, above the dense path's limit: the one-shot entry against the oracle golden"""
    res, offs, ab, z = antibodies
    T, X, P = (int(v) for v in z["params"])
    rc, G, err = hb.clinkage_cluster_arrays(res, offs, ab, blosum62, T, X, P)
    assert rc == 0, err
    assert (G.cluster_id == z["cluster_id"]).all() and (G.member_rank == z["member_rank"]).all()
    assert (G.result_order == z["result_order"]).all()
    assert G.n_multi == int((np.bincount(z["cluster_id"]) > 1).sum())


@pytest.mark.gpu
def test_antibodies_run_clinkage_clustering(antibodies, blosum62):
    res, offs, ab, z = antibodies
    strs = synth.to_strings(res, offs)
    seqs = [hb.UniqueSequence(s, {"x": int(a)}) for s, a in zip(strs, ab)]
    clusters = hb.run_clinkage_clustering(seqs, blosum62)
    assert [c.get_id() for c in clusters] == z["result_order"].tolist()
    big = max(clusters, key=lambda c: c.get_unique_size())
    mem = np.nonzero(z["cluster_id"] == big.get_id())[0]
    mem = mem[np.argsort(z["member_rank"][mem])]
    assert len(mem) == 174
    assert [s.get_sequence_string() for s in big.get_sequences()] == [strs[m] for m in mem]


@pytest.mark.gpu
def test_antibodies_cpp_driver_clinkage_mode(tmp_path, antibodies, blosum62):
    """hammock_greedy clinkage on a fasta of the antibodies set: the files against the oracle's writers fed with the golden"""
    from oracle import pyref_writers as W
    res, offs, ab, z = antibodies
    strs = synth.to_strings(res, offs)
    fa = tmp_path / "antibodies.fa"
    with open(fa, "w") as f:
        for j, (s, a) in enumerate(zip(strs, ab)):
            f.write(f">s{j}|{int(a)}|x\n{s}\n")
    mp = tmp_path / "m.txt"                                 # the matrix file in the reference's format
    with open(mp, "w") as f:
        f.write("# test copy of BLOSUM62\n   " + "  ".join(hb.ALPHABET) + "\n")
        for i in range(24):
            f.write(hb.ALPHABET[i] + " " + " ".join(f"{int(v):2d}" for v in blosum62[i]) + "\n")
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([hb_build.build_host(), "clinkage", "-i", str(fa), "-d", str(out), "-m", str(mp)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    assert [s.get_sequence_string() for s in seqs] == strs
    labels = hb.get_sorted_labels(seqs)
    n_multi = int((np.bincount(z["cluster_id"]) > 1).sum())
    clusters = hb.rebuild_clusters(seqs, hb.GreedyResult(z["cluster_id"], z["member_rank"], z["result_order"], n_multi, {}))
    tup = lambda s: (s.get_sequence_string(), dict(s.labels_map))
    ct = [(c.get_id(), [tup(s) for s in c.get_sequences()]) for c in clusters]
    assert (out / "initial_clusters_sequences.tsv").read_text() == W.cluster_sequences_tsv(ct, labels)
    assert (out / "initial_clusters_sequences_original_order.tsv").read_text() == W.cluster_sequences_tsv_ordered(ct, labels, [tup(s) for s in seqs])
    assert (out / "initial_clusters.tsv").read_text() == W.clusters_tsv(ct, labels)


@pytest.mark.gpu
def test_100k_synthetic_clinkage_without_oracle(blosum62):
    """100 000 synthetic 12-mers: repeatable, well formed, and complete linkage holds inside every cluster"""
    d = synth.generate(100_000, 12, 12, seed=20260101)
    T, X, _ = synth.default_params(d["lengths"])
    ctx = hb.GreedyContext(0)
    try:
        runs = []
        for _ in range(2):
            rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0)
            assert rc == 0, err
            runs.append(G)
        a, b = runs
        assert (a.cluster_id == b.cluster_id).all() and (a.member_rank == b.member_rank).all()
        assert (a.result_order == b.result_order).all() and a.stats["p1_steps"] == b.stats["p1_steps"]
        _well_formed(a.cluster_id, a.member_rank, a.result_order)
        assert a.n_multi > 0 and a.stats["xhits_kept"] > 0
        # intra-cluster scores, many clusters per hmk_score_block call
        ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, 1)
        groups = list(_member_lists(a.cluster_id, a.member_rank).values())
        i = 0
        while i < len(groups):
            batch, tot = [], 0
            while i < len(groups) and (not batch or tot + len(groups[i]) <= 2048):
                batch.append(groups[i]); tot += len(groups[i]); i += 1
            ids = np.concatenate(batch)
            S = ctx.score_block(ids, ids)
            o = 0
            for g in batch:
                blk = S[o:o + len(g), o:o + len(g)]
                assert (blk[~np.eye(len(g), dtype=bool)] >= T).all()
                o += len(g)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_clinkage_status_codes_above_the_dense_limit(blosum62):
    d = synth.generate(40_000, 12, 12, seed=7)
    asym = blosum62.copy()
    asym[0, 1] += 1
    assert hb.clinkage_cluster_arrays(d["residues"], d["offsets"], d["abundance"], asym, 20, 3, 0)[0] == _lib.STATUS_UNSUPPORTED
    res = np.concatenate([d["residues"], np.array([1, 2, 3], np.uint8)])
    offs = np.concatenate([d["offsets"], [d["offsets"][-1] + 3]]).astype(np.int32)
    ab = np.concatenate([d["abundance"], [1]]).astype(np.int32)
    assert hb.clinkage_cluster_arrays(res, offs, ab, blosum62, 20, 3, 0)[0] == _lib.STATUS_SHIFT_TOO_BIG
