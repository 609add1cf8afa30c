"""Every bulk scoring kernel against exact pair scores, in the three modes the clusterer uses.

The reference is a numpy restatement of ShiftedScorer.sequenceScore over all (member, query) pairs of a dataset, pinned to
the oracle on the CPU.  On the GPU, hmk_bulk_probe runs one bulk launch with a context's scheme and options:
  - TOPK (partner search): per query the kb best candidates under (score desc, tie-break rank asc), the count, the
    "more existed" flag, and every candidate kept for phase 2 exactly once with its exact score;
  - EMIT (founder filter, sparse complete linkage): every pair scoring >= T exactly once with its exact score, and the
    exact count when the buffer is too small;
  - DENSE: score_block on the same schemes.
Each case asserts the kernel that ran, so none passes on a fallback.  The last tests run whole clusterings with scaled
matrices whose pair scores exceed 32767 on 16-bit lanes."""
import functools
import os
import zlib

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import synth
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B62 = synth.blosum62()


def _mats():
    z = np.load(os.path.join(ROOT, "tests", "golden", "matrices.npz"))
    return {k: z[k].astype(np.int32) for k in z.files}


def _seqs(d, ids):
    off, res = d["offsets"], d["residues"]
    return [res[off[i]:off[i + 1]] for i in ids]


# ---------------------------------------------------------------- reference
def ref_scores(d, M, X, P, members, queries):
    """S[a, b] = sequenceScore(seq1 = members[a], seq2 = queries[b]) (ShiftedScorer.java:48-100): the shorter sequence
    slides over the longer one (equal lengths: seq2 is the shorter), shifts k = -X .. X + d, matrix M[shorter][longer],
    penalty P per unit of |d| plus 2 P per shift beyond the overlap.  int64, no wrap-around (no test gets near 2^31)."""
    off, res = d["offsets"], d["residues"]
    Mf = np.asarray(M, dtype=np.int64).reshape(-1)
    members, queries = np.asarray(members, dtype=np.int64), np.asarray(queries, dtype=np.int64)
    lm, lq = off[members + 1] - off[members], off[queries + 1] - off[queries]
    S = np.empty((len(members), len(queries)), dtype=np.int64)
    for a in np.unique(lm):
        ia = np.nonzero(lm == a)[0]
        A = res[off[members[ia]][:, None] + np.arange(a)].astype(np.int64)
        for b in np.unique(lq):
            ib = np.nonzero(lq == b)[0]
            B = res[off[queries[ib]][:, None] + np.arange(b)].astype(np.int64)
            q_short = a >= b                      # equal lengths: seq2 (the query) is the shorter one
            ls, ll = (b, a) if q_short else (a, b)
            dd = ll - ls
            best = None
            for k in range(-X, X + dd + 1):
                pen = dd * P + (-2 * k * P if k < 0 else 0) + (2 * (k - dd) * P if k > dd else 0)
                acc = np.full((len(ia), len(ib)), pen, dtype=np.int64)
                for j in range(max(k, 0), min(ls + k, ll)):
                    if q_short:
                        acc += Mf[B[:, j - k][None, :] * 24 + A[:, j][:, None]]
                    else:
                        acc += Mf[A[:, j - k][:, None] * 24 + B[:, j][None, :]]
                best = acc if best is None else np.maximum(best, acc)
            S[np.ix_(ia, ib)] = best
    return S


class Ref:
    """Exact scores of one dataset under one (M, X, P), computed once per block of (members, queries)."""

    def __init__(self, d, M, X, P, blocks):
        self.d, self.M, self.X, self.P = d, M, X, P
        self.blocks = [(np.asarray(m), np.asarray(q), ref_scores(d, M, X, P, m, q)) for m, q in blocks]

    def S(self, members, queries):
        members, queries = np.asarray(members), np.asarray(queries)
        for m, q, S in self.blocks:
            im, iq = np.searchsorted(m, members), np.searchsorted(q, queries)
            if (im < len(m)).all() and (iq < len(q)).all() and (m[np.minimum(im, len(m) - 1)] == members).all() and \
                    (q[np.minimum(iq, len(q) - 1)] == queries).all():
                return S[np.ix_(im, iq)]
        raise KeyError("no reference block holds these pairs")


def tierank(abundance):
    """rank under a stable sort by abundance, descending (the partner search's tie-break)"""
    order = np.argsort(-np.asarray(abundance, dtype=np.int64), kind="stable")
    r = np.empty(len(order), dtype=np.int64)
    r[order] = np.arange(len(order))
    return r


def key_make(score, rank):
    return ((np.asarray(score, dtype=np.int64) + (1 << 31)).astype(np.uint64) << np.uint64(32)) | \
        (np.uint64(0xffffffff) - np.asarray(rank, dtype=np.int64).astype(np.uint64))


def rows_sorted(a):
    a = np.asarray(a, dtype=np.int64).reshape(-1, 3)
    return a[np.lexsort(a.T[::-1])]


# ---------------------------------------------------------------- expected outputs
def expect_hits(S, queries, db, T, clustered=None):
    ok = S >= T
    if clustered is not None:
        ok &= ~clustered[db][:, None]
    a, b = np.nonzero(ok)
    return rows_sorted(np.stack([b, np.asarray(db)[a], S[a, b]], axis=1))


def expect_topk(S, queries, db, T, kb, rank, clustered=None):
    db, queries = np.asarray(db), np.asarray(queries)
    ok = (S >= T) & (db[:, None] > queries[None, :])
    if clustered is not None:
        ok &= ~clustered[db][:, None]
    lists, cnt, ovf, kept = [], [], [], []
    for b, q in enumerate(queries):
        a = np.nonzero(ok[:, b])[0]
        keys = np.sort(key_make(S[a, b], rank[db[a]]))[::-1]
        lists.append(keys[:kb])
        cnt.append(min(kb, len(a)))
        ovf.append(int(len(a) > kb))
        kept.append(np.stack([np.full(len(a), q), db[a], S[a, b]], axis=1))
    return lists, np.array(cnt), np.array(ovf), rows_sorted(np.concatenate(kept) if kept else np.zeros((0, 3)))


# ---------------------------------------------------------------- GPU helpers
def context(d, M, T, X, P, abundance=None, K=1, **opts):
    ctx = hb.GreedyContext(0, **opts)
    ab = d["abundance"] if abundance is None else abundance
    ctx.upload(d["residues"], d["offsets"], ab, M, T, X, P, K)
    return ctx


def first_wrong(got, want):
    w = {tuple(x) for x in want.tolist()}
    return [x for x in got.tolist() if tuple(x) not in w][:5]


def assert_kernel(got, want, persistent=None):
    for k, v in want.items():
        assert got[k] == v, (got, want)
    if persistent is not None:
        assert got["persistent"] == persistent, got


def check_topk(ctx, ref, queries, T, kb, rank, db=None, db_range=None, clustered=None, what=""):
    ids = np.asarray(db) if db is not None else np.arange(db_range[0], db_range[0] + db_range[1])
    S = ref.S(ids, queries)
    lists, cnt, ovf, kept = expect_topk(S, queries, ids, T, kb, rank, clustered)
    r = ctx.bulk_probe(0, queries, db=db, db_range=db_range, clustered=clustered, hit_cap=len(kept) + 64)
    assert r["hit_count"] == len(kept), (what, r["hit_count"], len(kept))
    got = rows_sorted(r["hits"])
    if not np.array_equal(got, kept):
        raise AssertionError(f"{what}: kept hits differ; {len(got)} vs {len(kept)}; first wrong (query id, id, score): "
                             f"{first_wrong(got, kept)}, first missing: {first_wrong(kept, got)}")
    assert (r["cnt"] == cnt).all(), (what, np.nonzero(r["cnt"] != cnt)[0][:8], r["cnt"][:8], cnt[:8])
    bad_ovf = np.nonzero(r["ovf"] != ovf)[0]
    assert len(bad_ovf) == 0, (what, "overflow flag", bad_ovf[:8].tolist(), r["ovf"][bad_ovf[:8]].tolist())
    for b in range(len(queries)):
        if not np.array_equal(r["keys"][b, :cnt[b]], lists[b]):
            gk = r["keys"][b, :cnt[b]]
            raise AssertionError(f"{what}: query {queries[b]}: list (score, rank) "
                                 f"{[(int(k >> np.uint64(32)) - (1 << 31), 0xffffffff - int(k & np.uint64(0xffffffff))) for k in gk]}"
                                 f" != {[(int(k >> np.uint64(32)) - (1 << 31), 0xffffffff - int(k & np.uint64(0xffffffff))) for k in lists[b]]}")
    return r, int(len(kept)), int(ovf.sum())


def check_emit(ctx, ref, queries, T, db=None, db_range=None, clustered=None, what=""):
    ids = np.asarray(db) if db is not None else np.arange(db_range[0], db_range[0] + db_range[1])
    want = expect_hits(ref.S(ids, queries), queries, ids, T, clustered)
    r = ctx.bulk_probe(1, queries, db=db, db_range=db_range, clustered=clustered, hit_cap=len(want) + 64)
    assert r["hit_count"] == len(want), (what, r["hit_count"], len(want))
    got = rows_sorted(r["hits"])
    if not np.array_equal(got, want):
        raise AssertionError(f"{what}: hits differ; first wrong (query index, id, score): {first_wrong(got, want)}, "
                             f"first missing: {first_wrong(want, got)}")
    return r, len(want)


# ---------------------------------------------------------------- datasets (CPU; seeded)
N12 = 20000
POOL = 1200          # members / thread side of the variant and query-count cases


@functools.lru_cache(maxsize=None)
def data(name):
    if name == "d12":
        return synth.generate(N12, 12, 12, seed=11)
    if name == "d10":
        return synth.generate(POOL, 10, 10, seed=12)
    if name == "d9":
        return synth.generate(POOL, 9, 9, seed=13)
    if name == "d16":
        return synth.generate(POOL, 16, 16, seed=14)
    if name == "d30":
        return synth.generate(POOL, 30, 30, seed=15)
    if name == "dmix":
        return synth.generate(POOL, 7, 12, seed=16)
    if name == "s12":
        return synth.generate(1500, 12, 12, seed=5)
    if name == "s9":
        return synth.generate(1500, 9, 9, seed=5)
    raise KeyError(name)


def scaled(f):
    return ((B62 + 4) * f).astype(np.int32)


def matrix(name):
    if name == "blosum62":
        return B62
    if name == "x700":
        return (B62 * 700).astype(np.int32)
    if name == "s300":
        return scaled(300)
    if name == "s375":
        return scaled(375)
    if name == "ties":                       # 0/1 entries: scores are small integers, heavy ties
        return (B62 > 0).astype(np.int32)
    return _mats()[name]


@functools.lru_cache(maxsize=None)
def ref(dname, mname, X, P, blocks="pool"):
    d = data(dname)
    n = len(d["abundance"])
    pool = np.arange(min(n, POOL))
    queries = np.unique(np.r_[0:min(n, 512), len(pool) - 4:len(pool)])
    if blocks == "pool":
        return Ref(d, matrix(mname), X, P, [(pool, queries)])
    # the 20 000 12-mers: besides, the 64 first and 16 last queries against everything
    return Ref(d, matrix(mname), X, P, [(pool, queries), (np.arange(n), np.r_[0:64, n - 16:n])])


# ---------------------------------------------------------------- CPU: the reference against the oracle
@pytest.mark.parametrize("mname,X,P,lo,hi", [("blosum62", 3, 0, 12, 12), ("asym", 2, -3, 5, 12), ("blosum30", 4, 2, 9, 20),
                                             ("asym", 0, 1, 6, 8), ("pam250", 5, -1, 13, 36)])
def test_reference_matches_oracle(mname, X, P, lo, hi):
    M = B62.copy() if mname == "asym" else matrix(mname)
    if mname == "asym":
        M[np.triu_indices(24, 1)] -= 2       # orientation M[shorter][longer] matters
        M[3, 7] += 5
    rng = np.random.default_rng(zlib.crc32(repr((mname, X, P, lo, hi)).encode()))
    d = synth.generate(300, lo, hi, seed=int(rng.integers(1, 1 << 30)))
    mem = rng.choice(300, 40, replace=False)
    qry = rng.choice(300, 30, replace=False)
    S = ref_scores(d, M, X, P, mem, qry)
    sm, sq = _seqs(d, mem), _seqs(d, qry)
    for a in range(len(mem)):
        for b in range(len(qry)):
            assert S[a, b] == O.score_with_shift(sm[a], sq[b], M, X, P)[0], (a, b)


def test_expected_topk_model():
    """the expected lists follow the key order of hmk_key_make: score desc, then tie-break rank asc"""
    S = np.array([[5], [7], [7], [3], [9]])
    rank = np.array([0, 4, 3, 2, 1, 0])
    lists, cnt, ovf, kept = expect_topk(S, np.array([0]), np.array([1, 2, 3, 4, 5]), 5, 2, rank)
    assert cnt.tolist() == [2] and ovf.tolist() == [1] and len(kept) == 4
    assert [(int(k >> np.uint64(32)) - (1 << 31), 0xffffffff - int(k & np.uint64(0xffffffff))) for k in lists[0]] == \
        [(9, 0), (7, 2)]


# ---------------------------------------------------------------- GPU: every kernel in every mode
F12 = dict(kind="filter", filter_lt=12, nw=2, lane_bits=8)
VARIANTS = {
    # name: dataset, matrix, T, X, P, options, kernel
    "filter12": ("d12", "blosum62", 20, 3, 0, {}, F12),
    "filter0_10mer_x2": ("d10", "blosum62", 17, 2, 0, {}, dict(kind="filter", filter_lt=0, nw=2, lane_bits=8)),
    "filter0_9mer_x3": ("d9", "blosum62", 15, 3, 0, {}, dict(kind="filter", filter_lt=0, nw=2, lane_bits=8)),
    "fast1_x0": ("d12", "blosum62", 12, 0, 0, {"filter": 0}, dict(kind="fast", nw=1, lane_bits=8)),
    "fast1_x1": ("d12", "blosum62", 16, 1, -1, {"filter": 0}, dict(kind="fast", nw=1, lane_bits=8)),
    "fast2_x2": ("d12", "blosum62", 20, 2, 0, {"filter": 0}, dict(kind="fast", nw=2, lane_bits=8)),
    "fast2_x3": ("d12", "blosum62", 20, 3, -1, {"filter": 0}, dict(kind="fast", nw=2, lane_bits=8)),
    "fast3_blosum30": ("d12", "blosum30", 20, 2, -2, {}, dict(kind="fast", nw=3, lane_bits=16)),
    "fast4_blosum30": ("d12", "blosum30", 20, 3, -2, {}, dict(kind="fast", nw=4, lane_bits=16)),
    "fast4_scaled12": ("s12", "s300", 24000, 3, 0, {}, dict(kind="fast", nw=4, lane_bits=16)),
    "fast3_scaled9": ("s9", "s375", 17858, 2, 0, {}, dict(kind="fast", nw=3, lane_bits=16)),
    "long16_u16": ("d16", "blosum62", 27, 4, 0, {}, dict(kind="long", nw=5, lane_bits=16)),
    "long16_u8": ("d16", "blosum62", 50, 4, 0, {}, dict(kind="long", nw=3, lane_bits=8)),
    "long30_u16": ("d30", "blosum62", 51, 8, -1, {}, dict(kind="long", nw=9, lane_bits=16)),
    "generic_forced": ("d12", "blosum62", 20, 3, 0, {"force_generic": 1}, dict(kind="generic", lane_bits=32)),
    "generic_x700": ("d12", "x700", 14000, 3, 0, {}, dict(kind="generic", lane_bits=32)),
    "generic_mixed": ("dmix", "blosum62", 16, 1, 0, {"force_generic": 1}, dict(kind="generic", lane_bits=32)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_variant_all_modes(name):
    dname, mname, T, X, P, opts, kern = VARIANTS[name]
    d, M = data(dname), matrix(mname)
    R = ref(dname, mname, X, P, "big" if (dname, mname, X, P) == ("d12", "blosum62", 3, 0) else "pool")
    n = len(d["abundance"])
    pool = np.arange(min(n, POOL))
    rng = np.random.default_rng(len(name))
    nq = 256 if name.startswith("fast") and "scaled" in name else 64
    queries = np.r_[0:nq - 4, len(pool) - 4:len(pool)]              # the last ones have (almost) empty candidate lists
    if "scaled" in name:             # the case this variant exists for: pair scores above 32767 with 16-bit lanes
        assert R.S(pool, np.arange(nq - 4)).max() > 32767
    ab = d["abundance"]
    if name in ("filter12", "fast4_blosum30", "long16_u16", "generic_forced"):
        ab = rng.permutation(ab)                                    # tie-break rank != id
    rank = tierank(ab)
    ctx = context(d, M, T, X, P, abundance=ab, **opts)
    try:
        # TOPK over an id range; with the length-sorted walk of the generic kernel over unequal lengths as an id list
        if name == "generic_mixed":
            db = np.argsort(d["offsets"][1:] - d["offsets"][:-1], kind="stable").astype(np.int32)
            r, nk, _ = check_topk(ctx, R, queries, T, 8, rank, db=db, what=name)
        else:
            r, nk, _ = check_topk(ctx, R, queries, T, 8, rank, db_range=(0, len(pool)), what=name)
        assert nk > 0
        assert_kernel(r["kernel"], kern, 1 if kern["kind"] == "filter" else 0)
        # EMIT over a shuffled id list (the founder filter's form)
        db = rng.permutation(len(pool))[:len(pool) * 3 // 4].astype(np.int32)
        r, nh = check_emit(ctx, R, queries, T, db=db, what=name)
        assert nh > 0
        assert_kernel(r["kernel"], kern)
        # DENSE: every score
        sub = pool[rng.permutation(len(pool))[:300]]
        got = ctx.score_block(sub, queries)
        assert np.array_equal(got, R.S(sub, queries)), name
    finally:
        ctx.close()


# ---------------------------------------------------------------- GPU: the filter kernel's edges
@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 7, 8, 9, 31, 32, 33, 56, 57, 100, 448, 512])
def test_filter_query_counts(nq):
    d = data("d12")
    R = ref("d12", "blosum62", 3, 0, "big")
    rank = tierank(d["abundance"])
    q = np.arange(nq)
    for persistent in (1, 0):
        ctx = context(d, B62, 20, 3, 0, persistent=persistent)
        try:
            r, _, _ = check_topk(ctx, R, q, 20, 8, rank, db_range=(0, POOL), what=f"nq={nq} persistent={persistent}")
            assert_kernel(r["kernel"], F12, persistent)
            check_emit(ctx, R, q, 20, db_range=(0, POOL), what=f"emit nq={nq} persistent={persistent}")
        finally:
            ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("qt,nq,ndb", [(2, 3, POOL), (2, 5, POOL), (8, 57, POOL), (4, 64, N12 - 64)])
def test_filter_small_tiles(qt, nq, ndb):
    """a full tile followed by a 1-query tile; many tiles, so that persistent CTAs change tiles"""
    d = data("d12")
    R = ref("d12", "blosum62", 3, 0, "big")
    rank = tierank(d["abundance"])
    q = np.arange(nq)
    for persistent in (1, 0):
        ctx = context(d, B62, 20, 3, 0, qt=qt, persistent=persistent)
        try:
            r, _, _ = check_topk(ctx, R, q, 20, 8, rank, db_range=(64, ndb), what=f"qt={qt} nq={nq}")
            assert_kernel(r["kernel"], F12, persistent)
            check_emit(ctx, R, q, 20, db_range=(64, ndb), what=f"emit qt={qt} nq={nq}")
        finally:
            ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ndb", [1, 31, 32, 33, 767, 768, 769, N12 - 64])
def test_filter_thread_counts(ndb):
    d = data("d12")
    R = ref("d12", "blosum62", 3, 0, "big")
    rank = tierank(d["abundance"])
    q = np.arange(64)
    for persistent in (1, 0):
        for T in (5, 20):
            ctx = context(d, B62, T, 3, 0, persistent=persistent)
            try:
                r, _, _ = check_topk(ctx, R, q, T, 8, rank, db_range=(64, ndb), what=f"ndb={ndb} T={T} p={persistent}")
                assert_kernel(r["kernel"], F12, persistent)
                check_emit(ctx, R, q, T, db_range=(64, ndb), what=f"emit ndb={ndb} T={T} p={persistent}")
            finally:
                ctx.close()


# T = 5: the lowest threshold with the filter (below, the lanes need 16 bits); 45: the filter passes pairs whose exact
# score fails; 80: the highest with u8 lanes, only a sequence against itself reaches it
@pytest.mark.gpu
@pytest.mark.parametrize("T,kb", [(5, 1), (5, 2), (5, 8), (5, 32), (20, 1), (20, 2), (20, 32), (45, 1), (45, 8),
                                  (80, 2), (80, 32)])
def test_filter_thresholds_and_options(T, kb):
    d = data("d12")
    R = ref("d12", "blosum62", 3, 0, "big")
    rng = np.random.default_rng(T * 100 + kb)
    unsorted = kb in (2, 32)
    ab = rng.permutation(d["abundance"]) if unsorted else d["abundance"]
    rank = tierank(ab)
    clustered = (rng.random(N12) < 0.3) if kb in (1, 32) else None
    q = np.arange(100)
    ctx = context(d, B62, T, 3, 0, abundance=ab, kb=kb)
    try:
        r, nk, novf = check_topk(ctx, R, q, T, kb, rank, db_range=(0, POOL), clustered=clustered, what=f"T={T} kb={kb}")
        assert_kernel(r["kernel"], F12, 1)
        if T == 5:
            assert novf > 50, novf                  # lists overflow
        if T == 80:
            assert nk == 0
        check_emit(ctx, R, q, T, db_range=(0, POOL), clustered=clustered, what=f"emit T={T}")
        # the far end: the last queries of the range have few or no later ids
        qe = np.arange(N12 - 16, N12)
        check_topk(ctx, R, qe, T, kb, rank, db_range=(0, N12), clustered=clustered, what=f"end T={T} kb={kb}")
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kb", [2, 8])
def test_filter_heavy_ties(kb):
    """0/1 matrix: thousands of equal scores per query, ordered by the tie-break rank only"""
    d = data("d12")
    R = ref("d12", "ties", 3, 0)
    ab = np.random.default_rng(kb).permutation(d["abundance"])
    rank = tierank(ab)
    q = np.arange(100)
    ctx = context(d, matrix("ties"), 6, 3, 0, abundance=ab, kb=kb)
    try:
        r, nk, novf = check_topk(ctx, R, q, 6, kb, rank, db_range=(0, POOL), what=f"ties kb={kb}")
        assert_kernel(r["kernel"], F12, 1)
        assert novf > 50
        check_emit(ctx, R, q, 6, db_range=(0, POOL), what="emit ties")
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("persistent", [1, 0])
def test_emit_capacity_below_count(persistent):
    """the count is exact past the capacity, and what was stored is a duplicate-free subset of the true hits"""
    d = data("d12")
    R = ref("d12", "blosum62", 3, 0, "big")
    q = np.arange(64)
    want = expect_hits(R.S(np.arange(POOL), q), q, np.arange(POOL), 5)
    ctx = context(d, B62, 5, 3, 0, persistent=persistent)
    try:
        cap = len(want) // 3
        r = ctx.bulk_probe(1, q, db_range=(0, POOL), hit_cap=cap)
        assert_kernel(r["kernel"], F12, persistent)
        assert r["hit_count"] == len(want) and len(r["hits"]) == cap
        got = rows_sorted(r["hits"])
        assert len(np.unique(got[:, :2], axis=0)) == cap
        wset = {tuple(x) for x in want.tolist()}
        assert all(tuple(x) in wset for x in got.tolist())
    finally:
        ctx.close()


# ---------------------------------------------------------------- GPU: whole clusterings with hit scores above 32767
SCALED = [("s12", 12, 12, 300, 24000, 3), ("s9", 9, 9, 375, 17858, 2), ("mix", 9, 12, 300, 24000, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SCALED, ids=[c[0] for c in SCALED])
def test_scaled_greedy_against_oracle(case):
    name, lo, hi, f, T, X = case
    d = synth.generate(1500, lo, hi, seed=5)
    M = scaled(f)
    K = synth.default_params(d["lengths"])[2]
    R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, 0, K, nthreads=os.cpu_count() or 1)
    assert R.status == 0
    ctx = context(d, M, T, X, 0, K=K)
    try:
        ctx.run()
        G = ctx.download()
        st = ctx.stats()
        assert st["lane_bits"] == 16 and st["fast_path"] == (2 if lo != hi else 1), st
        assert (G.cluster_id == R.cluster_id).all() and (G.member_rank == R.member_rank).all(), name
        assert (G.result_order == R.result_order).all() and G.n_multi == R.n_multi, name
    finally:
        ctx.close()


@pytest.mark.gpu
def test_scaled_sparse_clinkage_against_oracle_and_dense():
    d = synth.generate(1500, 12, 12, seed=5)
    M = scaled(300)
    R = O.clinkage_cluster(d["residues"], d["offsets"], d["abundance"], M, 24000, 3, 0)
    assert R.status == 0
    outs = []
    for dense_max in (0, 32768):
        ctx = hb.GreedyContext(0, clinkage_dense_max=dense_max)
        try:
            rc, G, err = ctx.clinkage(d["residues"], d["offsets"], d["abundance"], M, 24000, 3, 0)
            assert rc == 0, err
            assert G.stats["lane_bits"] == 16 and G.stats["fast_path"] == 1, G.stats
            assert (G.cluster_id == R.cluster_id).all() and (G.member_rank == R.member_rank).all(), dense_max
            assert (G.result_order == R.result_order).all(), dense_max
            outs.append(G)
        finally:
            ctx.close()
    assert outs[0].stats["xhits_kept"] > 0          # the sparse rows were built
    assert (outs[0].cluster_id == outs[1].cluster_id).all() and (outs[0].result_order == outs[1].result_order).all()
