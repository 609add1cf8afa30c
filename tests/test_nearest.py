"""Nearest partners (hmk_nearest, GreedyContext.nearest, nearest_partners, hammock_greedy nearest).

CPU: the numpy restatement the GPU tier compares with, pinned to the oracle's scoreWithShift (mixed lengths, an
asymmetric matrix, P != 0, a 0/1 matrix with ties everywhere, unsorted abundances); the C++ and Python
nearest_partners.tsv writers byte for byte; the driver's prepared parameters.
GPU: every list against that restatement, exactly -- per bulk kernel, tie-breaks by abundance, scores above 32 767,
T <= 0, tiny inputs, row ranges, statuses, the antibodies set against its score graph, clusterings on a context after
nearest calls, and the C++ driver."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import build as hb_build, synth
from oracle import oracle as O
from tests.test_score_graph import KERNEL_CASES, _mixed_case, _wrap32, ref_graph

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ references
def pair_scores(res, offs, M, X, P):
    """(S, K) int64 [n, n]: S[i, j], K[i, j] = ShiftedScorer.scoreWithShift(seq1 = j, seq2 = i) for every ordered pair,
    the per-length scoring of test_score_graph.ref_graph taken over all j"""
    offs = np.asarray(offs, np.int64)
    n = len(offs) - 1
    S = np.zeros((n, n), np.int64)
    K = np.zeros((n, n), np.int64)
    if n == 0:
        return S, K
    lens = np.diff(offs)
    Lmax = int(lens.max())
    R = np.zeros((n, Lmax), np.int64)
    for i in range(n):
        R[i, :lens[i]] = res[offs[i]:offs[i + 1]]
    M64 = np.asarray(M, np.int64)
    groups = {int(L): np.nonzero(lens == L)[0] for L in np.unique(lens)}
    for i in range(n):
        li = int(lens[i])
        q = R[i, :li]
        for L, js in groups.items():
            C = R[js, :L]
            query_short = L >= li                     # len1 >= len2: seq2 (the row) is the shorter one
            ls, ll = (li, L) if query_short else (L, li)
            d = ll - ls
            best = np.full(len(js), -2 ** 63, np.int64)
            bk = np.zeros(len(js), np.int64)
            for k in range(-X, X + d + 1):
                jj = np.arange(max(k, 0), min(ls + k, ll))
                if query_short:
                    v = M64[q[jj - k][None, :], C[:, jj]].sum(1) if len(jj) else np.zeros(len(js), np.int64)
                else:
                    v = M64[C[:, jj - k], q[jj][None, :]].sum(1) if len(jj) else np.zeros(len(js), np.int64)
                v = _wrap32(v + d * P + (-2 * k * P if k < 0 else 0) + (2 * (k - d) * P if k > d else 0))
                up = v > best
                best[up] = v[up]
                bk[up] = k
            S[i, js] = best
            K[i, js] = bk if query_short else -bk
    return S, K


def select_nearest(S, K, abundance, T, k):
    """the lists from full score tables: row i's candidates j != i with S[i, j] >= T sorted by (S desc, abundance desc,
    j asc), cut to k -> (partner, score, shift) int32 [n, k] (padding -1, 0, 0), count and more int32 [n]"""
    n = len(S)
    ab = np.asarray(abundance, np.int64)
    partner = np.full((n, k), -1, np.int32)
    score = np.zeros((n, k), np.int32)
    shift = np.zeros((n, k), np.int32)
    count = np.zeros(n, np.int32)
    more = np.zeros(n, np.int32)
    for i in range(n):
        js = np.nonzero(S[i] >= T)[0]
        js = js[js != i]
        sel = js[np.lexsort((js, -ab[js], -S[i, js]))][:k]
        c = len(sel)
        partner[i, :c], score[i, :c], shift[i, :c] = sel, S[i, sel], K[i, sel]
        count[i], more[i] = c, len(js) > k
    return partner, score, shift, count, more


def ref_nearest(res, offs, abundance, M, T, X, P, k):
    """numpy restatement of hmk_nearest over all rows"""
    S, K = pair_scores(res, offs, M, X, P)
    return select_nearest(S, K, abundance, T, k)


def oracle_scores(res, offs, M, X, P):
    """the tables of pair_scores, one O.score_with_shift call per ordered pair (small inputs only)"""
    n = len(offs) - 1
    S = np.zeros((n, n), np.int64)
    K = np.zeros((n, n), np.int64)
    for i in range(n):
        for j in range(n):
            S[i, j], K[i, j] = O.score_with_shift(res[offs[j]:offs[j + 1]], res[offs[i]:offs[i + 1]], M, X, P)
    return S, K


def _same(got, want, what=""):
    for name, g, w in zip(("partner", "score", "shift", "count", "more"), got, want):
        assert g.shape == w.shape and np.array_equal(g, w), (what, name, np.argwhere(g != w)[:5] if g.shape == w.shape else g.shape)


# ------------------------------------------------------------------------------------------------ CPU
def test_numpy_restatement_against_the_oracle(blosum62):
    """pair_scores == one oracle call per ordered pair, and select_nearest on them gives ref_nearest; mixed lengths, an
    asymmetric matrix, P != 0, a 0/1 matrix (score ties everywhere), unsorted abundances"""
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 2
    ident = np.eye(24, dtype=np.int32)
    rng = np.random.default_rng(8)
    for seed, (lo, hi), M, P, T in ((1, (7, 12), blosum62, 0, 15), (2, (5, 30), asym, -1, 10), (3, (12, 12), asym, -2, -5),
                                    (4, (6, 9), ident, 0, 3), (5, (6, 14), ident, -1, 2)):
        res, offs = _mixed_case(70, lo, hi, seed)
        if M is ident:
            res = (res % 3).astype(np.uint8)        # three letters: many equal scores, the abundances decide
        X = min(3, lo - 1)
        ab = rng.permutation(np.minimum(rng.zipf(1.6, 70), 50)).astype(np.int32)
        S, K = oracle_scores(res, offs, M, X, P)
        S2, K2 = pair_scores(res, offs, M, X, P)
        assert np.array_equal(S, S2) and np.array_equal(K, K2), seed
        for k in (1, 5, 31):
            want = select_nearest(S, K, ab, T, k)
            _same(ref_nearest(res, offs, ab, M, T, X, P, k), want, (seed, k))
            assert want[3].sum() > 0 and (k == 31 or want[4].any())
        if M is asym:
            assert (S != S.T).any()                  # rows follow the definition's argument order
        if M is ident:                               # ties on the score that the abundance (not the id) breaks
            p = select_nearest(S, K, ab, T, 5)[0]
            ties = sum(1 for i in range(70) for r in range(4) if p[i, r + 1] >= 0 and S[i, p[i, r]] == S[i, p[i, r + 1]]
                       and ab[p[i, r]] > ab[p[i, r + 1]] and p[i, r] > p[i, r + 1])
            assert ties > 0


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("nearest_shim") / "libnearestshim.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O1", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "nearest_shim.cpp")])
    L = ctypes.CDLL(out)
    i32p = ctypes.POINTER(ctypes.c_int32)
    L.shim_save_nearest.restype = ctypes.c_int
    L.shim_save_nearest.argtypes = [ctypes.c_char_p, ctypes.c_int32, i32p, i32p, i32p, i32p, ctypes.c_int32, ctypes.c_char_p]
    return L


def test_cpp_and_python_writers_are_byte_identical(shim, tmp_path, blosum62):
    res, offs = _mixed_case(150, 6, 14, 9)
    strs = synth.to_strings(res, offs)
    seqs = [hb.UniqueSequence(s) for s in strs]
    ab = np.ones(150, np.int32)
    k = 4
    near = ref_nearest(res, offs, ab, blosum62, 12, 2, -1, k)
    partner, score, shift, count, more = near
    assert count.sum() > 100 and (count == 0).any() and (count == k).any() and (shift < 0).any()
    py = tmp_path / "py.tsv"
    hb.save_nearest_partners(seqs, near, str(py))
    cp = tmp_path / "cpp.tsv"
    arrs = [np.ascontiguousarray(a, np.int32) for a in (partner, score, shift, count)]
    ptrs = [a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) for a in arrs]
    assert shim.shim_save_nearest("\n".join(strs).encode(), k, *ptrs, 61, str(cp).encode()) == 0    # rows [0, 61), [61, 150)
    assert py.read_bytes() == cp.read_bytes()
    lines = py.read_text().splitlines()
    assert lines[0] == "sequence\trank\tpartner\tscore\tshift" and len(lines) == count.sum() + 1
    i = int(np.argmax(count > 1))
    first = 1 + int(count[:i].sum())
    assert lines[first + 1] == f"{strs[i]}\t2\t{strs[partner[i, 1]]}\t{score[i, 1]}\t{shift[i, 1]}"


MULTI = """>a|3|x
ACDEFGHIKLMN
>b|1|x
ACDEFGHIKLMA
>c|5|y
WWDEFGHIKLMN
>d|2|y
ACDEFG
"""


def _dump(args):
    r = subprocess.run([hb_build.build_host(), "nearest"] + args + ["--dump-prepared"], capture_output=True, text=True)
    return r.returncode, r.stdout.splitlines(), r.stderr


def test_driver_prepares_like_the_python_defaults(tmp_path):
    """hammock_greedy nearest: input order, setClinkageThreshold, getMaxShift and k = 8, as nearest_partners"""
    p = tmp_path / "in.fa"
    p.write_text(MULTI)
    seqs = hb.load_unique_sequences_from_fasta(str(p))
    rc, out, err = _dump(["-i", str(p), "-R", "size"])
    assert rc == 0, err
    head = {l.split("\t")[0]: l.split("\t")[1:] for l in out[:5]}
    assert int(head["threshold"][0]) == hb.set_clinkage_threshold(seqs)
    assert int(head["max_shift"][0]) == hb.get_max_shift(seqs)
    assert head["k"] == ["8"]
    assert [tuple(l.split("\t")) for l in out[5:]] == [(s.get_sequence_string(), str(s.size())) for s in seqs]
    rc, out, _ = _dump(["-i", str(p), "-k", "31", "-g", "7", "-x", "2"])
    assert rc == 0 and out[4] == "k\t31" and out[0] == "threshold\t7" and out[1] == "max_shift\t2"
    for bad in ("0", "32"):
        rc, _, err = _dump(["-i", str(p), "-k", bad])
        assert rc == 2 and "-k" in err


# ------------------------------------------------------------------------------------------------ GPU
def _nearest(res, offs, ab, M, T, X, P, k, **opts):
    """-> (the five arrays of GreedyContext.nearest, the TOPK dispatch the nearest search runs)"""
    ctx = hb.GreedyContext(0, **opts)
    try:
        ctx.upload(res, offs, ab, M, T, X, P, 0)
        kern = ctx.bulk_probe(0, [0], db_range=(0, len(offs) - 1))["kernel"]
        return ctx.nearest(k), kern
    finally:
        ctx.close()


@pytest.mark.gpu
def test_musi(golden_dir, blosum62):
    z = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
    T, X, P = (int(v) for v in z["params"])
    res, offs, ab = z["residues"], z["offsets"], z["abundance"]
    S, K = pair_scores(res, offs, blosum62, X, P)
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(res, offs, ab, blosum62, T, X, P, 0)
        assert ctx.bulk_probe(0, [0], db_range=(0, len(ab)))["kernel"]["kind"] == "filter"
        for k in (1, 8, 31):
            want = select_nearest(S, K, ab, T, k)
            assert want[3].sum() > 1000 and want[4].any() and (want[3] < k).any()
            _same(ctx.nearest(k), want, k)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", KERNEL_CASES, ids=[c[0] for c in KERNEL_CASES])
def test_nearest_per_kernel(blosum62, case):
    name, n, (lo, hi), scale, T, opts, kind, lanes = case
    d = synth.generate(n, lo, hi, seed=40 + n + lo)
    T0, X, _ = synth.default_params(d["lengths"])
    T = T0 if T is None else T
    M = blosum62 * scale
    ab = d["abundance"]
    want = ref_nearest(d["residues"], d["offsets"], ab, M, T, X, 0, 8)
    got, kern = _nearest(d["residues"], d["offsets"], ab, M, T, X, 0, 8, **opts)
    assert want[3].sum() > 0
    _same(got, want, name)
    if kind:
        assert kern["kind"] == kind and (lanes is None or kern["lane_bits"] == lanes), kern
    for f in (0, 1):                      # the lists do not depend on the kernel
        for g in (0, 1):
            other, _ = _nearest(d["residues"], d["offsets"], ab, M, T, X, 0, 8, **{**opts, "filter": f, "force_generic": g})
            _same(other, want, (name, f, g))


@pytest.mark.gpu
def test_abundance_decides_ties(blosum62):
    """Zipf abundances in shuffled order: equal scores are ordered by abundance, then id (the tie-break rank of unsorted
    abundances); on BLOSUM62 and on a 0/1 matrix, where most of a row's scores tie"""
    d = synth.generate(2000, 12, 12, seed=12)
    rng = np.random.default_rng(3)
    ab = rng.permutation(np.minimum(rng.zipf(1.4, 2000), 100000)).astype(np.int32)
    T, X, _ = synth.default_params(d["lengths"])
    res = d["residues"]
    ident = np.eye(24, dtype=np.int32)
    low = (res % 4).astype(np.uint8)                  # four letters: 0/1 scores tie everywhere
    for r, M, t in ((res, blosum62, T), (low, ident, 7)):
        S, K = pair_scores(r, d["offsets"], M, X, 0)
        for k in (8, 31):
            want = select_nearest(S, K, ab, t, k)
            p = want[0]
            ties = ((p[:, 1:] >= 0) & (np.take_along_axis(S, np.maximum(p[:, :-1], 0), 1) ==
                                      np.take_along_axis(S, np.maximum(p[:, 1:], 0), 1)) & (p[:, :-1] > p[:, 1:])).sum()
            assert ties > 0                           # the abundance put a higher id first
            for opts in ({}, {"force_generic": 1}):
                got, _ = _nearest(r, d["offsets"], ab, M, t, X, 0, k, **opts)
                _same(got, want, (k, opts))


@pytest.mark.gpu
def test_asymmetric_penalty_scaled_and_complete(blosum62):
    res, offs = _mixed_case(700, 8, 14, 11)
    ab = np.random.default_rng(1).integers(1, 4, 700).astype(np.int32)
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 3
    asym[np.tril_indices(24, -1)] += 1
    got, _ = _nearest(res, offs, ab, asym, 22, 3, -1, 8)
    _same(got, ref_nearest(res, offs, ab, asym, 22, 3, -1, 8), "asymmetric")
    big = blosum62 * 5000                 # scores far above 32 767
    want = ref_nearest(res, offs, ab, big, 22 * 5000, 3, -2, 8)
    assert want[1].max() > 32767
    got, _ = _nearest(res, offs, ab, big, 22 * 5000, 3, -2, 8)
    _same(got, want, "scaled")
    rng = np.random.default_rng(9)                    # 16-bit lanes, hits above 32 767: W-rich 12-mers
    res = rng.choice([hb.ALPHABET.index(c) for c in "WCHY"], 1500 * 12, p=[0.7, 0.1, 0.1, 0.1]).astype(np.uint8)
    offs = np.arange(0, 1500 * 12 + 1, 12, dtype=np.int32)
    ab = rng.integers(1, 5, 1500).astype(np.int32)
    M = blosum62 * 300
    want = ref_nearest(res, offs, ab, M, 18000, 3, 0, 8)
    assert (want[1] > 32767).sum() > 1000
    got, kern = _nearest(res, offs, ab, M, 18000, 3, 0, 8)
    assert kern["kind"] == "fast" and kern["lane_bits"] == 16
    _same(got, want, "lane16")
    d = synth.generate(300, 12, 12, seed=3)           # T <= 0: every pair qualifies
    for k in (1, 31):
        want = ref_nearest(d["residues"], d["offsets"], d["abundance"], blosum62, -1000, 3, 0, k)
        assert (want[3] == k).all() and want[4].all()
        got, _ = _nearest(d["residues"], d["offsets"], d["abundance"], blosum62, -1000, 3, 0, k)
        _same(got, want, ("complete", k))


def _cyclic_families(n, seed):
    """12-mers over four letters in families of 1 .. 139: every member is the family's base with each residue moved on
    by the same step r (mod 4) and two point mutations, in shuffled order.  With cyclic_matrix a pair scores high in the
    direction where one member is the other moved on by one step, so the rows' candidate counts spread from 0 to ~40."""
    rng = np.random.default_rng(seed)
    seqs = []
    while len(seqs) < n:
        f = int(rng.integers(1, 140))
        b = rng.integers(0, 4, 12)
        for _ in range(min(f, n - len(seqs))):
            s = (b + rng.integers(0, 4)) % 4
            pos = rng.integers(0, 12, 2)
            s[pos] = rng.integers(0, 4, 2)
            seqs.append(s)
    res = np.concatenate([seqs[i] for i in rng.permutation(n)]).astype(np.uint8)
    return res, np.arange(0, 12 * n + 1, 12, dtype=np.int32)


def cyclic_matrix(diag):
    """an asymmetric matrix whose off-diagonal entries beat the diagonal: M[a][a + 1 mod 4] = 3, M[a][a] = diag"""
    M = np.zeros((24, 24), np.int32)
    for a in range(4):
        M[a, (a + 1) % 4] = 3
        M[a, a] = diag
    return M


@pytest.mark.gpu
def test_rows_whose_own_id_is_not_in_the_list():
    """The row's own id missing from the merged top-(k + 1) list: then count = min(c, k) and more = (c == k + 1).
    diag -1: no row's own score reaches T, and rows have more than k + 1, exactly k + 1, exactly k and fewer than k
    other candidates at every k, so both values of `more` and the uncut short list occur on this path.  diag 2: every
    row's own score (24) reaches T but most rows have more than k + 1 better partners, so it qualifies without being
    in the list; at k = 31 a few rows keep it in the list."""
    n = 1500
    res, offs = _cyclic_families(n, 5)
    rng = np.random.default_rng(6)
    ab = rng.permutation(np.minimum(rng.zipf(1.5, n), 1000)).astype(np.int32)
    T, X = 24, 3
    for diag in (-1, 2):
        M = cyclic_matrix(diag)
        S, K = pair_scores(res, offs, M, X, 0)
        own = np.diag(S).copy()
        others = S.copy()
        np.fill_diagonal(others, np.iinfo(np.int64).min)
        n_others = (others >= T).sum(1)
        # keys ahead of the row's own one: a higher score, or the same score with a better (abundance, id) rank
        rank = np.lexsort((np.arange(n), -ab.astype(np.int64)))
        pos = np.empty(n, np.int64)
        pos[rank] = np.arange(n)
        ahead = ((others > own[:, None]) | ((others == own[:, None]) & (pos[None, :] < pos[:, None]))).sum(1)
        for k in (1, 8, 31):
            want = select_nearest(S, K, ab, T, k)
            if diag < 0:
                assert (own < T).all()
                for c in (n_others > k + 1, n_others == k + 1, n_others == k, n_others < k):
                    assert c.sum() > 0, k
            else:
                assert (own >= T).all() and (ahead >= k + 1).sum() > 100 and (k < 31 or (ahead < k + 1).any()), k
            for opts in ({}, {"force_generic": 1}):
                got, _ = _nearest(res, offs, ab, M, T, X, 0, k, **opts)
                _same(got, want, (diag, k, opts))


@pytest.mark.gpu
def test_tiny_inputs(blosum62):
    ctx = hb.GreedyContext(0)
    try:
        for strs in ([], ["WVTAPRSLPVLP"], ["WVTAPRSLPVLP", "WVTAPRSLPVLA"], ["WVTAP"], ["WVTAPRSLPVLP", "AAAAAAAAAAAA"]):
            res, offs = O.pack(strs) if strs else (np.zeros(0, np.uint8), np.zeros(1, np.int32))
            ab = np.ones(len(strs), np.int32)
            ctx.upload(res, offs, ab, blosum62, 20, 6 if len(strs) == 1 else 3, 0, 0)
            for k in (1, 3):
                got = ctx.nearest(k)
                _same(got, ref_nearest(res, offs, ab, blosum62, 20, 3, 0, k), (strs, k))
                assert got[3].sum() == (2 if strs == ["WVTAPRSLPVLP", "WVTAPRSLPVLA"] else 0)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_row_ranges(blosum62):
    """any split of [0, n) into ranges concatenates to the full result, batches of 512 rows and all"""
    d = synth.generate(1300, 12, 12, seed=21)
    T, X, _ = synth.default_params(d["lengths"])
    n, k = 1300, 6
    want = ref_nearest(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, k)
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, 0)
        _same(ctx.nearest(k), want, "full")
        for cuts in ([1], [511, 512, 513, 1024], [7, 700, 1299], [0, 0, 650, 650]):
            b = [0] + cuts + [n]
            parts = [ctx.nearest(k, (lo, hi)) for lo, hi in zip(b[:-1], b[1:])]
            _same(tuple(np.concatenate([p[f] for p in parts]) for f in range(5)), want, cuts)
        got = ctx.nearest(k, (n, n))
        assert got[0].shape == (0, k) and len(got[3]) == 0
    finally:
        ctx.close()


@pytest.mark.gpu
def test_list_length_is_independent_of_option_kb(blosum62):
    """the nearest search keeps k + 1 keys per row whatever option kb is, and leaves the option to the partner search:
    after nearest(31), mode-0 probes on the context return lists of kb keys, equal to those of a context without nearest
    calls"""
    n = 1500
    d = synth.generate(n, 12, 12, seed=5)
    T, X, _ = synth.default_params(d["lengths"])
    res, offs, ab = d["residues"], d["offsets"], d["abundance"]
    want = ref_nearest(res, offs, ab, blosum62, T, X, 0, 31)
    assert want[4].any()                  # some rows have more than 31 partners
    q = np.arange(200)
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(res, offs, ab, blosum62, T, X, 0, 0)
        for kb in (1, 32):
            ctx.set_option("kb", kb)
            _same(ctx.nearest(31), want, kb)
            got = ctx.bulk_probe(0, q, db_range=(0, n))
            fresh = hb.GreedyContext(0, kb=kb)
            try:
                fresh.upload(res, offs, ab, blosum62, T, X, 0, 0)
                base = fresh.bulk_probe(0, q, db_range=(0, n))
            finally:
                fresh.close()
            assert got["keys"].shape == (len(q), kb) and got["cnt"].max() == kb
            assert np.array_equal(got["cnt"], base["cnt"]) and np.array_equal(got["ovf"], base["ovf"]), kb
            kept = np.arange(kb)[None, :] < got["cnt"][:, None]     # the slots past a list's count are not written
            assert np.array_equal(got["keys"][kept], base["keys"][kept]), kb
    finally:
        ctx.close()


@pytest.mark.gpu
def test_profile_sections(blosum62):
    """option profile: each call sets section slot 0 to the device time of its scoring passes and slot 1 to that of its
    merge, score and shift passes; the other slots stay 0"""
    d = synth.generate(3000, 12, 12, seed=8)
    T, X, _ = synth.default_params(d["lengths"])
    ctx = hb.GreedyContext(0, profile=1)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, 0)

        def slots():
            s = list(ctx.section_ms().values())
            assert s[0] > 0 and s[1] > 0 and not any(s[2:]), s
            return s[:2]

        ctx.nearest(8)                    # six batches of rows
        full = slots()
        ctx.nearest(8, (0, 10))           # one batch of ten rows: replaces the slots
        part = slots()
        assert part[0] < full[0] and part[1] < full[1], (full, part)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_statuses(blosum62):
    ctx = hb.GreedyContext(0)
    try:
        with pytest.raises(ValueError):               # status 5: before upload
            ctx.nearest(8)
        res, offs = O.pack(["WVTAPRSLPVLP", "RSLPVLP", "WVTAPRSLPVLA"])
        ab = np.ones(3, np.int32)
        ctx.upload(res, offs, ab, blosum62, 20, 7, 0, 0)
        with pytest.raises(hb.DataException):         # status 1: X >= the shortest length
            ctx.nearest(8)
        ctx.upload(res, offs, ab, blosum62, 20, 3, 0, 0)
        for k in (0, -1, 32):
            with pytest.raises(ValueError):
                ctx.nearest(k)
        for rows in ((-1, 2), (0, 4), (2, 1), (3, 4)):
            with pytest.raises(ValueError):
                ctx.nearest(8, rows)
        err = ctypes.create_string_buffer(512)
        one = np.zeros(8, np.int32)
        p = one.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
        assert ctx._L.hmk_nearest(ctx._h, 1, 0, 1, p, None, p, p, p, err, 512) == 5          # a null output
        assert ctx._L.hmk_nearest(ctx._h, 1, 0, 0, None, None, None, None, None, err, 512) == 0
        _same(ctx.nearest(31), ref_nearest(res, offs, ab, blosum62, 20, 3, 0, 31), "three")
        bad = res.copy()
        bad[3] = 24
        ctx.upload(bad, offs, ab, blosum62, 20, 3, 0, 0)
        with pytest.raises(hb.FileFormatException):   # status 3
            ctx.nearest(8)
    finally:
        ctx.close()


def _pull_graph(ctx):
    parts = list(ctx.score_graph(1 << 24))
    e = np.concatenate(parts) if parts else np.zeros(0, hb.EDGE_DTYPE)
    return e.view(np.int32).reshape(-1, 4).astype(np.int64)


@pytest.mark.gpu
def test_antibodies_lists_are_the_graph_neighbourhoods(blosum62):
    """74 041 sequences, symmetric BLOSUM62: each row's list is the top k, under (score desc, abundance desc, id asc), of
    its score-graph neighbours in both directions; shifts equal the graph's for j > i; more == degree > k"""
    from tests.golden.make_antibodies_clinkage_golden import input_arrays
    res, offs, ab = input_arrays()
    n = len(ab)
    T, X, P = 20, 3, 0
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(res, offs, ab, blosum62, T, X, P, 0)
        e = _pull_graph(ctx)
        got = {k: ctx.nearest(k) for k in (8, 31)}
    finally:
        ctx.close()
    assert len(e) > 5_000_000
    row = np.concatenate([e[:, 0], e[:, 1]])
    part = np.concatenate([e[:, 1], e[:, 0]])
    sc = np.concatenate([e[:, 2], e[:, 2]])
    sh = np.concatenate([e[:, 3], np.full(len(e), 1 << 40)])        # the graph's shift only where partner > row
    ab64 = np.asarray(ab, np.int64)
    o = np.lexsort((part, -ab64[part], -sc, row))
    row, part, sc, sh = row[o], part[o], sc[o], sh[o]
    deg = np.bincount(row, minlength=n)
    start = np.concatenate([[0], np.cumsum(deg)])
    pos = np.arange(len(row)) - start[row]
    for k, (partner, score, shift, count, more) in got.items():
        keep = pos < k
        wp = np.full((n, k), -1, np.int64)
        ws = np.zeros((n, k), np.int64)
        wh = np.full((n, k), 1 << 40, np.int64)
        wp[row[keep], pos[keep]], ws[row[keep], pos[keep]], wh[row[keep], pos[keep]] = part[keep], sc[keep], sh[keep]
        assert np.array_equal(partner, wp) and np.array_equal(score, ws), k
        later = partner > np.arange(n)[:, None]
        assert later.sum() > n and np.array_equal(shift[later], wh[later]), k
        assert np.array_equal(count, np.minimum(deg, k)) and np.array_equal(more, (deg > k).astype(np.int32)), k
        assert more.any()


@pytest.mark.gpu
def test_clusterings_after_nearest_calls(golden_dir, blosum62):
    """nearest calls, a greedy run, a complete-linkage run and a graph pull on one context: each matches its golden"""
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    T, X, P, K = (int(v) for v in z["params"])
    want = ref_nearest(z["residues"], z["offsets"], z["abundance"], blosum62, T, X, P, 31)
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(z["residues"], z["offsets"], z["abundance"], blosum62, T, X, P, K)
        _same(ctx.nearest(31), want, "before")
        ctx.nearest(3, (100, 900))
        ctx.run()
        G = ctx.download()
        assert (G.cluster_id == z["cluster_id"]).all() and (G.member_rank == z["member_rank"]).all()
        assert (G.result_order == z["result_order"]).all() and G.n_multi == int(z["n_multi"])
        _same(ctx.nearest(31), want, "after the run")
        zc = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
        Tc, Xc, Pc = (int(v) for v in zc["params"])
        rc, C, err = ctx.clinkage(zc["residues"], zc["offsets"], zc["abundance"], blosum62, Tc, Xc, Pc)
        assert rc == 0, err
        assert (C.cluster_id == zc["cluster_id"]).all() and (C.member_rank == zc["member_rank"]).all()
        assert (C.result_order == zc["result_order"]).all()
        ctx.upload(zc["residues"], zc["offsets"], zc["abundance"], blosum62, Tc, Xc, Pc, 0)
        ctx.nearest(8)
        assert np.array_equal(_pull_graph(ctx), ref_graph(zc["residues"], zc["offsets"], blosum62, Tc, Xc, Pc))
    finally:
        ctx.close()


@pytest.mark.gpu
def test_cpp_driver_nearest_mode_on_musi(tmp_path, golden_dir, blosum62):
    z = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
    strs = synth.to_strings(z["residues"], z["offsets"])
    fa = tmp_path / "musi.fa"
    with open(fa, "w") as f:
        for j, (s, a) in enumerate(zip(strs, z["abundance"])):
            f.write(f">s{j}|{int(a)}|x\n{s}\n")
    mp = tmp_path / "m.txt"
    with open(mp, "w") as f:
        f.write("# test copy of BLOSUM62\n   " + "  ".join(hb.ALPHABET) + "\n")
        for i in range(24):
            f.write(hb.ALPHABET[i] + " " + " ".join(f"{int(v):2d}" for v in blosum62[i]) + "\n")
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    assert [s.get_sequence_string() for s in seqs] == strs
    ab = np.array([s.size() for s in seqs], np.int32)
    T, X = hb.set_clinkage_threshold(seqs), hb.get_max_shift(seqs)
    S, K = pair_scores(z["residues"], z["offsets"], blosum62, X, 0)
    for k in (None, 5):
        out = tmp_path / f"out{k}"
        out.mkdir()
        r = subprocess.run([hb_build.build_host(), "nearest", "-i", str(fa), "-d", str(out), "-m", str(mp)] +
                           ([] if k is None else ["-k", str(k)]), capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        want = select_nearest(S, K, ab, T, k or 8)
        hb.save_nearest_partners(seqs, want, str(tmp_path / "py.tsv"))
        assert (out / "nearest_partners.tsv").read_bytes() == (tmp_path / "py.tsv").read_bytes()
        _same(hb.nearest_partners(seqs, blosum62, k=k or 8), want, k)
