"""Phase 1's per-batch inputs of the resolver against exact pair scores.

hmk_batch_probe writes a clustering state into a context and runs what a run runs for one batch: the partner search
(one launch, or one per length bucket on mixed lengths, merged once), the intra-batch table ib and its masks ibm / ibm2,
the partner ids pcand and their table pd, the founder filter, the linked member check and the candidate records.  Every
expected value comes from the definitions, with the exact scores of test_bulk_kernels.ref_scores (pinned to the oracle
there):
  qid      the first nq singletons with id >= cur;
  lists    per query, the kb best later singletons scoring >= T (test_bulk_kernels.expect_topk);
  ib       ib[b][b2] = S(member = qid[b2], query = qid[b]), every entry (the kernels write the whole nq x nq table);
  ibm      bit b2 = 32 w + k of word w set iff b2 < b and ib[b][b2] >= T;
  ibm2     those bits whose ib also reaches the lowest score of b's list; no bit when the list is empty;
  pcand    the ids of b's list, padded with qid[b];
  pd       pd[b][e] = S(pcand[e], qid[b]);
  founder  every (b, founder, S) with S >= T, in any order;
  members  cluster c is a candidate of b iff every member, founder included, scores >= T; its score is the minimum;
           with more candidates than capq the count is exact and the stored ones are a subset; the best record is the
           best of the stored ones under (score desc, size desc, founder id asc).
Each probe case asserts the kernels and paths that ran, so none passes on another path than the one it is named for.
Two whole runs against the oracle close the file: a run after probes on the same context, and a second input on one
context built so that a per-length profile kept from the first run would be taken for the second run's batch 2."""
import functools
import os
import zlib

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import synth
from oracle import oracle as O
from tests.test_bulk_kernels import B62, expect_topk, key_make, matrix, ref_scores, rows_sorted, tierank

FB_STRIDE = 1 << 16          # founders per slice of the mixed-length founder filter (HMK_FB_STRIDE)


# ---------------------------------------------------------------- expected values (CPU)
def key_score(keys):
    return (np.asarray(keys, dtype=np.uint64) >> np.uint64(32)).astype(np.int64) - (1 << 31)


def key_rank(keys):
    return 0xffffffff - (np.asarray(keys, dtype=np.uint64) & np.uint64(0xffffffff)).astype(np.int64)


def pack_bits(bits):
    """bool [nq, nq] -> uint32 [nq, nw]: column b2 is bit b2 % 32 of word b2 // 32"""
    nq = bits.shape[0]
    nw = (nq + 31) // 32
    padded = np.zeros((nq, nw * 32), dtype=np.uint64)
    padded[:, :bits.shape[1]] = bits
    return (padded.reshape(nq, nw, 32) << np.arange(32, dtype=np.uint64)).sum(axis=2).astype(np.uint32)


def expect_masks(ib, T, cnt, keys):
    """(ibm, ibm2) from the intra-batch table and the merged lists (keys[b, :cnt[b]] in descending order)"""
    nq = ib.shape[0]
    earlier = np.tri(nq, nq, -1, dtype=bool)
    thr = np.array([key_score(keys[b][cnt[b] - 1]) if cnt[b] > 0 else np.iinfo(np.int64).max for b in range(nq)])
    ok = earlier & (ib >= T)
    return pack_bits(ok), pack_bits(ok & (ib >= thr[:, None]))


def expect_pcand(qid, cnt, keys, kb, id_of_rank):
    out = np.repeat(np.asarray(qid, dtype=np.int64)[:, None], kb, axis=1)
    for b in range(len(qid)):
        out[b, :cnt[b]] = id_of_rank[key_rank(keys[b][:cnt[b]])]
    return out


def cluster_size(ab, members):
    """Cluster.size(): Java-int sum of the abundances"""
    return ((int(np.sum(np.asarray(ab, dtype=np.int64)[members])) + (1 << 31)) % (1 << 32)) - (1 << 31)


def expect_members(S, clusters, T):
    """per query b: {cluster: min score over its members} of the clusters whose every member scores >= T.
    S[id, b] = S(member = id, query = qid[b])"""
    nq = S.shape[1]
    out = [dict() for _ in range(nq)]
    if not clusters:
        return out
    flat = np.concatenate([np.asarray(c) for c in clusters])
    starts = np.cumsum([0] + [len(c) for c in clusters[:-1]])
    mins = np.minimum.reduceat(S[flat], starts, axis=0)
    for c, b in zip(*np.nonzero(mins >= T)):
        out[b][int(c)] = int(mins[c, b])
    return out


def expect_best(cands, clusters, ab):
    """the best of {cluster: score} under (score desc, size desc, founder id asc) as (score, size, founder, cluster)"""
    best = None
    for c, s in cands.items():
        k = (-s, -cluster_size(ab, clusters[c]), int(clusters[c][0]))
        if best is None or k < best[0]:
            best = (k, (s, -k[1], k[2], c))
    return best[1] if best else None


def singletons(n, clusters):
    single = np.ones(n, dtype=bool)
    for c in clusters:
        single[np.asarray(c)] = False
    return single


def expect_batch(d, M, X, P, T, kb, ab, clusters, cur, nq):
    n = len(d["abundance"])
    single = singletons(n, clusters)
    qid = (np.nonzero(single[cur:])[0] + cur)[:nq]
    S = ref_scores(d, M, X, P, np.arange(n), qid)                 # S[id, b]
    rank = tierank(ab)
    id_of_rank = np.argsort(rank)
    db = np.arange(cur, n)
    lists, cnt, ovf, _ = expect_topk(S[cur:], qid, db, T, kb, rank, ~single)
    keys = np.zeros((len(qid), kb), dtype=np.uint64)
    for b, l in enumerate(lists):
        keys[b, :len(l)] = l
    ib = S[qid].T
    ibm, ibm2 = expect_masks(ib, T, cnt, keys)
    pcand = expect_pcand(qid, cnt, keys, kb, id_of_rank)
    pd = S[pcand.reshape(-1)].T
    founders = np.array([c[0] for c in clusters], dtype=np.int64)
    if len(founders):
        a, b = np.nonzero(S[founders] >= T)
        fh = rows_sorted(np.stack([b, founders[a], S[founders[a], b]], axis=1))
    else:
        fh = np.zeros((0, 3), dtype=np.int64)
    return dict(qid=qid, S=S, keys=keys, cnt=cnt, ovf=ovf, ib=ib, ibm=ibm, ibm2=ibm2, pcand=pcand, pd=pd, fh=fh,
                members=expect_members(S, clusters, T))


# ---------------------------------------------------------------- CPU: the helpers against brute-force loops
def test_masks_match_loops():
    rng = np.random.default_rng(1)
    for nq in (1, 5, 31, 32, 33, 70):
        kb = int(rng.integers(1, 5))
        T = 5
        ib = rng.integers(0, 12, size=(nq, nq))
        cnt = rng.integers(0, kb + 1, size=nq)
        keys = np.zeros((nq, kb), dtype=np.uint64)
        for b in range(nq):
            sc = np.sort(rng.integers(T, 15, size=cnt[b]))[::-1]
            keys[b, :cnt[b]] = key_make(sc, rng.integers(0, 100, size=cnt[b]))
        ibm, ibm2 = expect_masks(ib, T, cnt, keys)
        nw = (nq + 31) // 32
        for b in range(nq):
            low = (int(keys[b, cnt[b] - 1] >> np.uint64(32)) - (1 << 31)) if cnt[b] else None
            for w in range(nw):
                m = m2 = 0
                for k in range(32):
                    b2 = 32 * w + k
                    if b2 < b and ib[b, b2] >= T:
                        m |= 1 << k
                        if low is not None and ib[b, b2] >= low:
                            m2 |= 1 << k
                assert ibm[b, w] == m and ibm2[b, w] == m2, (nq, b, w)


def test_pcand_matches_loop():
    rng = np.random.default_rng(2)
    ab = rng.integers(1, 5, size=50)
    rank = tierank(ab)
    id_of_rank = np.argsort(rank)
    qid = np.array([3, 7, 9])
    cnt = np.array([2, 0, 3])
    keys = np.zeros((3, 4), dtype=np.uint64)
    ids = {0: [20, 11], 2: [40, 12, 30]}
    for b, l in ids.items():
        keys[b, :len(l)] = key_make([9] * len(l), rank[l])
    got = expect_pcand(qid, cnt, keys, 4, id_of_rank)
    assert got.tolist() == [[20, 11, 3, 3], [7, 7, 7, 7], [40, 12, 30, 9]]


def test_member_check_matches_loop():
    rng = np.random.default_rng(3)
    T = 4
    S = rng.integers(0, 9, size=(40, 6))
    ab = rng.integers(1, 1 << 30, size=40)           # sizes wrap as Java ints
    clusters = [[0], [1, 2], [3, 4, 5, 6], [7, 8], [9, 10, 11]] + [[12 + 2 * i, 13 + 2 * i] for i in range(10)]
    got = expect_members(S, clusters, T)
    for b in range(6):
        want = {}
        for c, mem in enumerate(clusters):
            if all(S[m, b] >= T for m in mem):
                want[c] = min(S[m, b] for m in mem)
        assert got[b] == want, b
        best = None
        for c, s in want.items():
            size = sum(int(ab[m]) for m in clusters[c]) & 0xffffffff
            size -= (size >> 31) << 32
            if best is None or (s, size, -clusters[c][0]) > (best[0], best[1], -best[2]):
                best = (s, int(size), clusters[c][0], c)
        assert expect_best(got[b], clusters, ab) == best, b


# ---------------------------------------------------------------- GPU helpers
@functools.lru_cache(maxsize=None)
def data(name):
    if name == "u12":
        return synth.generate(3000, 12, 12, seed=21)
    if name == "mix":         # 7-12, with every 11-mer moved to the front: no later singleton of length 11
        d = synth.generate(3000, 7, 12, seed=22)
        lens = d["offsets"][1:] - d["offsets"][:-1]
        return reorder(d, np.argsort(lens != 11, kind="stable"))
    if name == "mixbig":
        return synth.generate(70000, 7, 12, seed=23)
    if name == "x1114":       # mixed lengths across one and two packed words
        return synth.generate(2000, 11, 14, seed=24)
    raise KeyError(name)


def reorder(d, order):
    off, res = d["offsets"], d["residues"]
    seqs = [res[off[i]:off[i + 1]] for i in order]
    new = np.zeros(len(seqs) + 1, dtype=np.int32)
    new[1:] = np.cumsum([len(x) for x in seqs])
    return {"residues": np.concatenate(seqs).astype(np.uint8), "offsets": new,
            "abundance": np.ascontiguousarray(d["abundance"][order]), "lengths": np.diff(new)}


def asym():
    M = B62.copy()
    M[np.triu_indices(24, 1)] -= 2
    M[3, 7] += 5
    return M


def mat(name):
    return asym() if name == "asym" else matrix(name)


def make_clusters(S, n, cur, qid, T, rng, big=50, many2=0, nrandom=20, ncl=None, avoid_len=None, lengths=None):
    """Clusters over ids < cur.  For each of the first queries b (S[id, b] = S(id, qid[b]) for the ids < cur): clusters
    of 2-6 members that all score >= T against it, and one whose last member scores below T; for the first query also
    one of up to `big` members and `many2` pairs.  Then `nrandom` random clusters of 2-5 members and two of 3 members
    behind the batch's last query (the partner search must skip them).  `ncl`: exactly that many, padded with
    founder-only clusters.  `avoid_len`: no member of that length."""
    free = np.ones(n, dtype=bool)
    if avoid_len is not None:
        free &= lengths != avoid_len
    late = free.copy()
    late[:int(qid[-1]) + 1] = False
    free[cur:] = False
    clusters = []

    def take(ids):
        clusters.append([int(x) for x in ids])
        free[ids] = False

    for b in range(S.shape[1]):
        good = np.nonzero(free[:cur] & (S[:cur, b] >= T))[0]
        bad = np.nonzero(free[:cur] & (S[:cur, b] < T))[0]
        rng.shuffle(good)
        if b == 0 and big and len(good) >= 2:
            take(good[:big])
            good = good[big:]
        if b == 0:
            for i in range(min(many2, len(good) // 2)):
                take(good[2 * i:2 * i + 2])
            good = good[2 * min(many2, len(good) // 2):]
        for k in (2, 4, 6):
            if len(good) >= k:
                take(good[:k])
                good = good[k:]
        if len(good) >= 2 and len(bad):
            take(np.r_[good[:2], bad[:1]])
    for _ in range(nrandom):
        pool = np.nonzero(free)[0]
        k = int(rng.integers(2, 6))
        if len(pool) < k:
            break
        take(rng.choice(pool, k, replace=False))
    pool = np.nonzero(late)[0]
    if len(pool) >= 6:
        pick = rng.choice(pool, 6, replace=False)
        clusters += [pick[:3].tolist(), pick[3:].tolist()]
    if ncl is not None:
        clusters = clusters[:ncl]
        pool = np.nonzero(free)[0]
        rng.shuffle(pool)
        clusters += [[int(i)] for i in pool[:ncl - len(clusters)]]
    return [[int(x) for x in c] for c in clusters]


def first_diff(got, want):
    bad = np.argwhere(np.asarray(got) != np.asarray(want))
    return [(tuple(int(v) for v in i), int(np.asarray(got)[tuple(i)]), int(np.asarray(want)[tuple(i)])) for i in bad[:5]]


def check(r, e, clusters, ab, capq, what):
    assert np.array_equal(r["qid"], e["qid"]), (what, r["qid"][:8], e["qid"][:8])
    nq = len(e["qid"])
    assert (r["cnt"] == e["cnt"]).all(), (what, "list counts", first_diff(r["cnt"], e["cnt"]))
    assert (r["ovf"] == e["ovf"]).all(), (what, "overflow flags", first_diff(r["ovf"], e["ovf"]))
    for b in range(nq):
        c = e["cnt"][b]
        assert np.array_equal(r["keys"][b, :c], e["keys"][b, :c]), (what, "list", b)
    assert np.array_equal(r["ib"], e["ib"]), (what, "ib [b, b2]", first_diff(r["ib"], e["ib"]))
    assert np.array_equal(r["ibm"], e["ibm"]), (what, "ibm [b, w]", first_diff(r["ibm"], e["ibm"]))
    assert np.array_equal(r["ibm2"], e["ibm2"]), (what, "ibm2 [b, w]", first_diff(r["ibm2"], e["ibm2"]))
    assert np.array_equal(r["pcand"], e["pcand"]), (what, "pcand", first_diff(r["pcand"], e["pcand"]))
    assert np.array_equal(r["pd"], e["pd"]), (what, "pd [b, e]", first_diff(r["pd"], e["pd"]))
    assert r["fhit_count"] == len(e["fh"]), (what, "founder hits", r["fhit_count"], len(e["fh"]))
    assert np.array_equal(rows_sorted(r["fhits"]), e["fh"]), (what, "founder hit rows")
    for b in range(nq):
        want = e["members"][b]
        assert r["ac_cnt"][b] == len(want), (what, "candidates of query", b, int(r["ac_cnt"][b]), len(want))
        k = min(len(want), capq)
        slots = r["ac_slot"][b, :k].tolist()
        assert len(set(slots)) == k and all(s in want for s in slots), (what, "candidate slots", b)
        assert [want[s] for s in slots] == r["ac_score"][b, :k].tolist(), (what, "candidate scores", b)
        best = expect_best({s: want[s] for s in slots}, clusters, ab)
        if best is None:
            assert r["ac_best"][b][3] == -1, (what, b)
        else:
            assert tuple(int(v) for v in r["ac_best"][b]) == best, (what, "best", b, r["ac_best"][b], best)


def run_case(dname, mname, T, X, P, opts, nq, kb, cur, capq=0, unsorted=False, K=None, kern=None, **cl):
    d, M = data(dname), mat(mname)
    n = len(d["abundance"])
    rng = np.random.default_rng(zlib.crc32(repr((dname, mname, T, nq, kb, cur, capq)).encode()))
    ab = rng.permutation(d["abundance"]) if unsorted else d["abundance"]
    cur = {"start": 0, "mid": n // 2, "end": n - max(1, nq // 2)}.get(cur, cur)
    qid0 = np.arange(cur, min(n, cur + nq))
    S0 = ref_scores(d, M, X, P, np.arange(cur), qid0[:8]) if cur > 0 else np.zeros((0, 0), np.int64)
    lengths = d["offsets"][1:] - d["offsets"][:-1]
    clusters = make_clusters(S0, n, cur, qid0, T, rng, lengths=lengths, **cl)
    e = expect_batch(d, M, X, P, T, kb, ab, clusters, cur, nq)
    ctx = hb.GreedyContext(0, kb=kb, **opts)
    try:
        ctx.upload(d["residues"], d["offsets"], ab, M, T, X, P, K or max(len(clusters), 1))
        cq = capq or 256
        for tail in (False, True):
            r = ctx.batch_probe(clusters, cur, nq, capq=cq, tail_stream=tail,
                                fhit_cap=len(e["fh"]) + 64)
            check(r, e, clusters, ab, cq, f"{dname}/{mname} nq={nq} kb={kb} cur={cur} tail={tail}")
            if kern:
                for k, v in kern.items():
                    assert r["kernel"][k] == v, (k, r["kernel"])
        return r, e, clusters
    finally:
        ctx.close()


# ---------------------------------------------------------------- GPU: uniform 12-mers
U12 = dict(kind="filter", filter_lt=12, lane_bits=8, search_launches=1, tables="fast", founder="filter",
           member_check="score12x3")


@pytest.mark.gpu
@pytest.mark.parametrize("nq,kb,cur", [(64, 8, "mid"), (1, 1, "mid"), (31, 2, "mid"), (32, 32, "mid"), (33, 8, "start"),
                                       (448, 8, "mid"), (512, 2, 700), (64, 8, "end")])
def test_u12_filter(nq, kb, cur):
    r, e, _ = run_case("u12", "blosum62", 15, 3, 0, {}, nq, kb, cur, kern=U12, many2=10)
    assert e["cnt"].sum() > 0


@pytest.mark.gpu
def test_u12_exact_kernel():
    r, e, cl = run_case("u12", "blosum62", 15, 3, 0, {"filter": 0}, 64, 8, "mid", unsorted=True,
                        kern=dict(U12, kind="fast", filter_lt=-1, nw=2, founder="fast"))
    assert sum(len(m) for m in e["members"]) > 0 and len(e["fh"]) > 0


@pytest.mark.gpu
def test_u12_x2_packed_member_check():
    run_case("u12", "blosum62", 18, 2, 0, {}, 96, 8, "mid", kern=dict(U12, member_check="packed"))


@pytest.mark.gpu
@pytest.mark.parametrize("mname,T,kern", [("asym", 16, dict(U12, kind="filter", founder="filter")),
                                          ("s300", 24000, dict(kind="fast", lane_bits=16, member_check="score12x3")),
                                          ("x700", 14000, dict(kind="generic", tables="generic", founder="generic",
                                                               member_check="packed"))])
def test_u12_matrices(mname, T, kern):
    r, e, _ = run_case("u12", mname, T, 3, 0, {}, 64, 8, "mid", kern=kern)
    if mname == "s300":
        assert e["S"].max() > 32767


@pytest.mark.gpu
@pytest.mark.parametrize("capq", [1, 4])
def test_capq_overflow_ties(capq):
    """0/1 matrix, heavy ties; the first query has more passing clusters than capq"""
    r, e, _ = run_case("u12", "ties", 6, 3, 0, {}, 40, 2, "mid", capq=capq, unsorted=True, many2=12, big=0, kern=U12)
    assert len(e["members"][0]) > capq


# ---------------------------------------------------------------- GPU: mixed lengths
MIX = dict(kind="fast", tables="dense_packed", table_launches=0, founder="fast", member_check="packed")


@pytest.mark.gpu
@pytest.mark.parametrize("nq,kb,cur,P,mname", [(64, 8, "mid", 0, "blosum62"), (33, 2, "mid", -1, "asym"),
                                               (512, 8, 900, 2, "blosum62"), (20, 32, "end", 0, "asym")])
def test_mixed_buckets(nq, kb, cur, P, mname):
    """one partner-search launch per length bucket with later singletons (none of length 11: every 11-mer comes
    first); founders of every length but 7, so that bucket 7 has none and bucket 11 builds its own profiles"""
    d = data("mix")
    lens = d["offsets"][1:] - d["offsets"][:-1]
    c = {"start": 0, "end": len(lens) - max(1, nq // 2), "mid": len(lens) // 2}.get(cur, cur)
    later = len(set(lens[c:].tolist()))
    assert 11 not in set(lens[c:].tolist())
    r, e, cl = run_case("mix", mname, 16, 2, P, {}, nq, kb, cur, avoid_len=7,
                        kern=dict(MIX, search_launches=later))
    assert not any(lens[x[0]] == 7 for x in cl)


@pytest.mark.gpu
@pytest.mark.parametrize("ncl", [0, 1, FB_STRIDE - 1, FB_STRIDE, FB_STRIDE + 1])
def test_mixed_founder_slices(ncl):
    """founder lists around the slice size of the per-length founder filter: every slice launches every bucket for
    the slice size and reads the bucket's real size on the device"""
    kern = dict(MIX, founder="fast" if ncl else "none", member_check="packed" if ncl else "none",
                founder_launches=-(-ncl // FB_STRIDE) * 6)
    r, e, cl = run_case("mixbig", "blosum62", 16, 2, 0, {}, 32, 8, 67000, K=70000, big=10, nrandom=5, ncl=ncl,
                        kern=kern)
    assert len(cl) == ncl


@pytest.mark.gpu
def test_mixed_across_words():
    """11-14: packed per-length partner search on the long layout, generic dense tables and founder filter, the
    byte-wise member check"""
    lens = data("x1114")["offsets"][1:] - data("x1114")["offsets"][:-1]
    later = len(set(lens[len(lens) // 2:].tolist()))
    assert later == 4
    run_case("x1114", "blosum62", 20, 2, 0, {}, 64, 8, "mid",
             kern=dict(kind="long", search_launches=later, tables="generic", founder="generic", member_check="state"))


# ---------------------------------------------------------------- GPU: a run after a probe; a second input
@pytest.mark.gpu
def test_run_after_probe_matches_oracle():
    """probes write a clustering state, a control block and batch buffer 0 into the context; the run resets them.  (A
    probe's per-length profile ids cannot outlive run batch 1, which is staged in buffer 0 and rebuilds every length.)"""
    d = synth.generate(1500, 12, 12, seed=5)
    T, X, K = synth.default_params(d["lengths"])
    R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], B62, T, X, 0, K, nthreads=os.cpu_count() or 1)
    assert R.status == 0
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], B62, T, X, 0, K)
        rng = np.random.default_rng(9)
        cl = [[int(x) for x in rng.choice(700, 3, replace=False)]]
        ctx.batch_probe(cl, 700, 128, tail_stream=True)
        ctx.batch_probe(cl, 100, 64)
        ctx.run()
        G = ctx.download()
        assert (G.cluster_id == R.cluster_id).all() and (G.member_rank == R.member_rank).all()
        assert (G.result_order == R.result_order).all() and G.n_multi == R.n_multi
    finally:
        ctx.close()


def family_input(region_b_first):
    """16 families over a +5 / -1 identity matrix, T = 40.  Family i: an 11-mer s (founder), s' (one substitution;
    S(s, s') = 49, so s takes s' as its partner), a 12-mer v (s with one other substitution plus one residue;
    S(v, s) = 49, S(v, s') = 43) and a 12-mer w (v with three more substitutions; S(v, w) = 42, S(w, s) = 31).  So v
    joins the family's cluster (43 > 42); without the founder hit (s, v) it would found {v, w} instead.  A 12-mer u
    (w with two more substitutions; S(u, w) = 48, S(u, v) = 30) is w's partner.  Region A (s, s' of every family: 32
    11-mers) is one batch of 32; region B (v, w, u, families in reverse order) follows."""
    rng = np.random.default_rng(77)
    A, B = [], []
    for i in range(16):
        s0 = rng.integers(0, 20, size=11)
        s1 = s0.copy()
        s1[5] = (s1[5] + 1 + rng.integers(0, 19)) % 20
        v = np.r_[s0, rng.integers(0, 20)]
        v[2] = (v[2] + 1 + rng.integers(0, 19)) % 20
        w = v.copy()
        for j in (0, 7, 9):
            w[j] = (w[j] + 1 + rng.integers(0, 19)) % 20
        u = w.copy()
        for j in (4, 11):
            u[j] = (u[j] + 1 + rng.integers(0, 19)) % 20
        A += [s0, s1]
        B = [v, w, u] + B
    seqs = B + A if region_b_first else A + B
    off = np.zeros(len(seqs) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(x) for x in seqs])
    return {"residues": np.concatenate(seqs).astype(np.uint8), "offsets": off,
            "abundance": np.ones(len(seqs), dtype=np.int32), "lengths": np.diff(off)}


def family_matrix():
    M = np.full((24, 24), -1, dtype=np.int32)
    M[np.arange(20), np.arange(20)] = 5
    return M


def test_family_input_scores():
    """the score relations family_input is built on, from the numpy restatement"""
    d, M = family_input(False), family_matrix()
    S = ref_scores(d, M, 2, 0, np.arange(80), np.arange(80))      # S[a, b] = S(member a, query b)
    for i in range(16):
        s0, s1, v = 2 * i, 2 * i + 1, 32 + 3 * (15 - i)
        w, u = v + 1, v + 2
        assert S[s1, s0] == 49 and S[s0, v] == 49 and S[s1, v] == 43 and S[w, v] == 42 and S[s0, w] == 31
        assert S[u, w] == 48 and S[u, v] == 30 and (S == S.T).all()
        fam = [s0, s1, v, w, u]
        assert S[np.setdiff1d(np.arange(80), fam)][:, fam].max() < 40


@pytest.mark.gpu
def test_second_input_on_one_context_matches_oracle():
    """Mixed lengths on one context, batches of 32, no look-ahead: batch i is staged in batch buffer (i - 1) % 3.  The
    first input puts the 11-mers second, so its batch 2 builds the length-11 profiles in buffer 1 for batch id 2.  The
    second input puts them first: its batch 2 has no later 11-mer, so only the founder filter needs length-11 profiles,
    and only a run that restarts the profile ids builds them for its own queries instead of taking the first run's."""
    M = family_matrix()
    ctx = hb.GreedyContext(0, lookahead=0, batch=32)
    try:
        for first in (True, False):
            d = family_input(first)
            R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, 40, 2, 0, 100, nthreads=1)
            assert R.status == 0 and R.n_multi >= 16
            ctx.upload(d["residues"], d["offsets"], d["abundance"], M, 40, 2, 0, 100)
            ctx.run()
            G = ctx.download()
            assert G.stats["fast_path"] == 2
            assert (G.cluster_id == R.cluster_id).all() and (G.member_rank == R.member_rank).all(), first
            assert (G.result_order == R.result_order).all() and G.n_multi == R.n_multi, first
    finally:
        ctx.close()
