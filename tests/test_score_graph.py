"""Score graph export (hmk_score_graph, hmk_score_pairs, GreedyContext.score_graph, hammock_greedy graph).

CPU: the host/device scorer with shift (hmk_common.h, built with g++) against the oracle's scoreWithShift; the numpy
restatement the GPU tier compares with, pinned to the oracle; the C++ and Python score_graph.tsv writers byte for byte.
GPU: every graph against that restatement or the oracle, exactly -- per bulk kernel, paging and cursors, statuses, the
antibodies set against complete linkage's row count, the C++ driver, and clusterings on a context after graph calls."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import _lib, build as hb_build, synth
from oracle import oracle as O
from tests import kats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ references
def _wrap32(v):
    return ((v + 2 ** 31) % 2 ** 32) - 2 ** 31


def ref_graph(res, offs, M, T, X, P):
    """numpy restatement of the score graph: for every i < j, (s, k) = ShiftedScorer.scoreWithShift(seq1 = j, seq2 = i)
    (ShiftedScorer.java:48-95; Java int arithmetic, the lowest winning diagonal, negated when seq1 is shorter); the
    edges with s >= T as an int64 array [m, 4] of (i, j, s, k) ordered by i, then j"""
    offs = np.asarray(offs, np.int64)
    n = len(offs) - 1
    if n < 2:
        return np.zeros((0, 4), np.int64)
    lens = np.diff(offs)
    Lmax = int(lens.max())
    S = np.zeros((n, Lmax), np.int64)
    for i in range(n):
        S[i, :lens[i]] = res[offs[i]:offs[i + 1]]
    M64 = np.asarray(M, np.int64)
    groups = {int(L): np.nonzero(lens == L)[0] for L in np.unique(lens)}
    out = []
    for i in range(n):
        li = int(lens[i])
        q = S[i, :li]
        rows = []
        for L, ids in groups.items():
            js = ids[ids > i]
            if not len(js):
                continue
            C = S[js, :L]
            query_short = L >= li                     # len1 >= len2: seq2 (the query) is the shorter one
            ls, ll = (li, L) if query_short else (L, li)
            d = ll - ls
            best = np.full(len(js), -2 ** 63, np.int64)
            bk = np.zeros(len(js), np.int64)
            for k in range(-X, X + d + 1):
                jj = np.arange(max(k, 0), min(ls + k, ll))      # longer index jj pairs with shorter index jj - k
                if query_short:
                    v = M64[q[jj - k][None, :], C[:, jj]].sum(1) if len(jj) else np.zeros(len(js), np.int64)
                else:
                    v = M64[C[:, jj - k], q[jj][None, :]].sum(1) if len(jj) else np.zeros(len(js), np.int64)
                v = v + d * P + (-2 * k * P if k < 0 else 0) + (2 * (k - d) * P if k > d else 0)
                v = _wrap32(v)
                up = v > best
                best[up] = v[up]
                bk[up] = k
            keep = best >= T
            sh = bk if query_short else -bk
            rows.append(np.stack([np.full(int(keep.sum()), i), js[keep], best[keep], sh[keep]], 1))
        if rows:
            r = np.concatenate(rows)
            out.append(r[np.argsort(r[:, 1], kind="stable")])
    return np.concatenate(out).astype(np.int64) if out else np.zeros((0, 4), np.int64)


def oracle_graph(res, offs, M, T, X, P):
    """the same edge list, one O.score_with_shift call per pair (small inputs only)"""
    n = len(offs) - 1
    out = []
    for i in range(n):
        for j in range(i + 1, n):
            s, k = O.score_with_shift(res[offs[j]:offs[j + 1]], res[offs[i]:offs[i + 1]], M, X, P)
            if s >= T:
                out.append((i, j, s, k))
    return np.array(out, np.int64).reshape(-1, 4)


def _mixed_case(n, lo, hi, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(lo, hi + 1, n)
    offs = np.zeros(n + 1, np.int32)
    offs[1:] = np.cumsum(lens)
    base = rng.integers(0, 20, int(offs[-1])).astype(np.uint8)
    for i in range(1, n):                         # relatives: copies of an earlier sequence with a few mutations
        if rng.random() < 0.5:
            a = int(rng.integers(0, i))
            m = min(lens[i], lens[a])
            base[offs[i]:offs[i] + m] = base[offs[a]:offs[a] + m]
            pos = rng.integers(0, lens[i], 2)
            base[offs[i] + pos] = rng.integers(0, 20, 2)
    return base, offs


# ------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("graph_shim") / "libgraphshim.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O1", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "graph_shim.cpp")])
    L = ctypes.CDLL(out)
    u8p, i32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int32)
    L.shim_score_with_shift.restype = ctypes.c_int32
    L.shim_score_with_shift.argtypes = [u8p, ctypes.c_int, u8p, ctypes.c_int, i32p, ctypes.c_int, ctypes.c_int,
                                        ctypes.POINTER(ctypes.c_int)]
    L.shim_save_score_graph.restype = ctypes.c_int
    L.shim_save_score_graph.argtypes = [ctypes.c_char_p, i32p, ctypes.c_int64, ctypes.c_char_p]
    return L


def _shim_sws(shim, a, b, M, X, P):
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    M = np.ascontiguousarray(M, np.int32)
    k = ctypes.c_int(12345)
    s = shim.shim_score_with_shift(a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), len(a),
                                   b.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), len(b),
                                   M.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), X, P, ctypes.byref(k))
    return int(s), int(k.value)


def _codes(s):
    return np.array([hb.ALPHABET.index(c) for c in s], np.uint8)


def test_device_scorer_with_shift_on_the_kats(shim, golden_dir):
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    for s1, s2, X, P, mat, score, shift in kats.SCORER_KATS:
        a, b, M = _codes(s1), _codes(s2), z[mat]
        got = _shim_sws(shim, a, b, M, X, P)
        assert got == O.score_with_shift(a, b, M, X, P)
        assert got[0] == score and (shift is None or got[1] == shift), (s1, s2)


def test_device_scorer_with_shift_random_pairs(shim, blosum62, golden_dir):
    """lengths 1..36, X up to the shorter length - 1, P in {0, -1, -2}; BLOSUM62, a 0/1 matrix (ties everywhere: the
    lowest diagonal wins, negated when seq1 is the shorter one) and an asymmetric matrix"""
    rng = np.random.default_rng(5)
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    ident = np.eye(24, dtype=np.int32)
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 3
    mats = [blosum62, ident, asym, z["pam250"]]
    ties = 0
    for it in range(6000):
        l1, l2 = int(rng.integers(1, 37)), int(rng.integers(1, 37))
        X = int(rng.integers(0, min(l1, l2)))
        P = int(rng.choice([0, -1, -2]))
        M = mats[it % len(mats)]
        alpha = 3 if M is ident else 24            # few letters: many equal diagonals on the 0/1 matrix
        a = rng.integers(0, alpha, l1).astype(np.uint8)
        b = rng.integers(0, alpha, l2).astype(np.uint8)
        want = O.score_with_shift(a, b, M, X, P)
        assert _shim_sws(shim, a, b, M, X, P) == want, (l1, l2, X, P, it % len(mats))
        ties += M is ident and l1 != l2 and want[1] != 0
    assert ties > 100


def test_numpy_restatement_against_the_oracle(blosum62):
    """ref_graph (the GPU tier's reference) == one oracle call per pair, mixed lengths, asymmetric matrix, P != 0"""
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 2
    for seed, (lo, hi), M, P in ((1, (7, 12), blosum62, 0), (2, (5, 30), asym, -1), (3, (12, 12), asym, -2)):
        res, offs = _mixed_case(90, lo, hi, seed)
        X = min(3, lo - 1)
        for T in (15, -5):
            a = ref_graph(res, offs, M, T, X, P)
            b = oracle_graph(res, offs, M, T, X, P)
            assert len(a) > 0 and np.array_equal(a, b), (seed, T)


def test_cpp_and_python_writers_are_byte_identical(shim, tmp_path, blosum62):
    res, offs = _mixed_case(150, 6, 14, 9)
    strs = synth.to_strings(res, offs)
    seqs = [hb.UniqueSequence(s) for s in strs]
    e = oracle_graph(res, offs, blosum62, 12, 2, -1)
    assert len(e) > 20 and (e[:, 3] != 0).any() and (e[:, 3] < 0).any()
    edges = np.zeros(len(e), hb.EDGE_DTYPE)
    for c, f in enumerate(("seq", "partner", "score", "shift")):
        edges[f] = e[:, c]
    py = tmp_path / "py.tsv"
    hb.save_score_graph(seqs, [edges[:7], edges[7:]], str(py))
    cp = tmp_path / "cpp.tsv"
    flat = np.ascontiguousarray(e.astype(np.int32))
    assert shim.shim_save_score_graph("\n".join(strs).encode(), flat.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                      len(e), str(cp).encode()) == 0
    assert py.read_bytes() == cp.read_bytes()
    lines = py.read_text().splitlines()
    assert lines[0] == "sequence\tpartner\tscore\tshift" and len(lines) == len(e) + 1
    i, j, s, k = e[0]
    assert lines[1] == f"{strs[i]}\t{strs[j]}\t{s}\t{k}"


# ------------------------------------------------------------------------------------------------ GPU
def _pull(ctx, chunk=1 << 22):
    parts = list(ctx.score_graph(chunk))
    e = np.concatenate(parts) if parts else np.zeros(0, hb.EDGE_DTYPE)
    return e.view(np.int32).reshape(-1, 4).astype(np.int64)


def _graph(res, offs, M, T, X, P, **opts):
    ctx = hb.GreedyContext(0, **opts)
    try:
        ctx.upload(res, offs, np.ones(len(offs) - 1, np.int32), M, T, X, P, 0)
        kern = ctx.bulk_probe(1, [0], db_range=(0, len(offs) - 1))["kernel"]    # the EMIT dispatch the graph runs
        return _pull(ctx), kern
    finally:
        ctx.close()


@pytest.mark.gpu
def test_musi_full_graph(golden_dir, blosum62):
    z = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
    T, X, P = (int(v) for v in z["params"])
    res, offs = z["residues"], z["offsets"]
    want = ref_graph(res, offs, blosum62, T, X, P)
    got, kern = _graph(res, offs, blosum62, T, X, P)
    assert len(want) > 1000 and np.array_equal(got, want)
    assert kern["kind"] == "filter"


# (name, n, lengths, matrix scale, threshold (None: default), options, kernel kind, lane bits or None)
KERNEL_CASES = [
    ("filter", 2000, (12, 12), 1, None, {}, "filter", 8),
    ("fast8", 2000, (12, 12), 1, None, {"filter": 0}, "fast", 8),
    ("fast16", 1500, (12, 12), 300, 7000, {}, "fast", 16),
    ("long", 1200, (14, 14), 1, None, {}, "long", None),
    ("generic_forced", 1500, (12, 12), 1, None, {"force_generic": 1}, "generic", 32),
    ("generic_beyond36", 500, (30, 40), 1, None, {}, "generic", 32),
    ("mixed_7_12", 1500, (7, 12), 1, None, {}, None, None),
    ("mixed_7_30", 800, (7, 30), 1, None, {}, None, None),
    ("mixed_11_14", 1200, (11, 14), 1, None, {}, None, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", KERNEL_CASES, ids=[c[0] for c in KERNEL_CASES])
def test_graph_per_kernel(blosum62, case):
    name, n, (lo, hi), scale, T, opts, kind, lanes = case
    d = synth.generate(n, lo, hi, seed=40 + n + lo)
    T0, X, _ = synth.default_params(d["lengths"])
    T = T0 if T is None else T
    M = blosum62 * scale
    want = ref_graph(d["residues"], d["offsets"], M, T, X, 0)
    got, kern = _graph(d["residues"], d["offsets"], M, T, X, 0, **opts)
    assert len(want) > 0 and np.array_equal(got, want), name
    if kind:
        assert kern["kind"] == kind and (lanes is None or kern["lane_bits"] == lanes), kern
    for f in (0, 1):                      # the graph does not depend on the kernel
        for g in (0, 1):
            other, _ = _graph(d["residues"], d["offsets"], M, T, X, 0, **{**opts, "filter": f, "force_generic": g})
            assert np.array_equal(other, want), (name, f, g)


@pytest.mark.gpu
def test_asymmetric_penalty_scaled_and_complete_graphs(blosum62):
    res, offs = _mixed_case(700, 8, 14, 11)
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 3
    asym[np.tril_indices(24, -1)] += 1
    T = 22
    want = ref_graph(res, offs, asym, T, 3, -1)
    got, _ = _graph(res, offs, asym, T, 3, -1)
    assert np.array_equal(got, want)
    flips = sum(O.score_with_shift(res[offs[i]:offs[i + 1]], res[offs[j]:offs[j + 1]], asym, 3, -1)[0] < T
                for i, j in want[:3000, :2])
    assert flips > 0                      # S(j, i) >= T > S(i, j): the graph follows the definition's argument order
    big = blosum62 * 5000                 # scores far above 32 767
    want = ref_graph(res, offs, big, 22 * 5000, 3, -2)
    got, _ = _graph(res, offs, big, 22 * 5000, 3, -2)
    assert want[:, 2].max() > 32767 and np.array_equal(got, want)
    d = synth.generate(300, 12, 12, seed=3)
    n = 300
    for cap in (0, 1, 5000):              # T <= 0: every pair; a small buffer splits the batches down to one row
        got, _ = _graph(d["residues"], d["offsets"], blosum62, -1000, 3, 0, graph_cap=cap)
        assert len(got) == n * (n - 1) // 2
        assert np.array_equal(got, ref_graph(d["residues"], d["offsets"], blosum62, -1000, 3, 0))


@pytest.mark.gpu
def test_tiny_inputs(blosum62):
    ctx = hb.GreedyContext(0)
    try:
        for strs in ([], ["WVTAPRSLPVLP"], ["WVTAPRSLPVLP", "WVTAPRSLPVLA"], ["WVTAP"]):
            res, offs = O.pack(strs) if strs else (np.zeros(0, np.uint8), np.zeros(1, np.int32))
            ctx.upload(res, offs, np.ones(len(strs), np.int32), blosum62, 20, 6 if len(strs) == 1 else 3, 0, 0)
            e, cur = ctx.graph_page((0, 0), 10)
            assert cur == (len(strs), 0)
            want = ref_graph(res, offs, blosum62, 20, 3, 0)
            assert np.array_equal(e.view(np.int32).reshape(-1, 4), want)
            assert len(e) == (1 if len(strs) == 2 else 0)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_paging_and_cursors(blosum62):
    d = synth.generate(1000, 12, 12, seed=77)
    T, X, _ = synth.default_params(d["lengths"])
    T -= 4
    n = 1000
    want = ref_graph(d["residues"], d["offsets"], blosum62, T, X, 0)
    rowlen = np.bincount(want[:, 0], minlength=n)
    row_start = np.concatenate([[0], np.cumsum(rowlen)])
    r0 = int(np.argmax(rowlen >= 3))
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, 0)
        full = _pull(ctx)
        assert np.array_equal(full, want) and len(want) > 2000
        for cap in (1, 7, int(rowlen[r0]) - 1, int(rowlen[r0]), len(want) + 5):
            cursor, got, saved = (0, 0), [], []
            while cursor != (n, 0):
                e, nxt = ctx.graph_page(cursor, cap)
                assert len(e) == min(cap, len(want) - sum(len(g) for g in got))
                i, r = nxt
                pos = sum(len(g) for g in got) + len(e)
                assert i == n or row_start[i] + r == pos           # the cursor names the next edge
                saved.append((cursor, pos - len(e)))
                got.append(e)
                cursor = nxt
                if cap == 1 and len(saved) == 400:
                    e, cursor = ctx.graph_page(cursor, len(want))   # the rest in one page
                    got.append(e)
            assert np.array_equal(np.concatenate(got).view(np.int32).reshape(-1, 4), want), cap
            for c, pos in saved[:: max(1, len(saved) // 6)]:      # restart from saved cursors (not continuing ones)
                e, end = ctx.graph_page(c, len(want))
                assert end == (n, 0) and np.array_equal(e.view(np.int32).reshape(-1, 4), want[pos:]), (cap, c)
        e, cur = ctx.graph_page((n, 0), 10)
        assert len(e) == 0 and cur == (n, 0)
        e, cur = ctx.graph_page((r0, int(rowlen[r0])), 3)       # after a whole row == the start of the next rows
        assert np.array_equal(e.view(np.int32).reshape(-1, 4), want[row_start[r0 + 1]:row_start[r0 + 1] + 3])
        for bad in ((-1, 0), (0, -1), (n + 1, 0), (n, 1), (r0, int(rowlen[r0]) + 1)):
            with pytest.raises(ValueError):
                ctx.graph_page(bad, 10)
        with pytest.raises(ValueError):
            ctx.graph_page((0, 0), -1)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_profile_sections(blosum62):
    """option profile: a pull adds the device time of the batches it computes to section slot 0 (scoring passes) and
    slot 1 (shift, sort and edge passes), and a pull from {0, 0} starts both at 0; the other slots stay 0"""
    n = 4000
    d = synth.generate(n, 12, 12, seed=8)
    T, X, _ = synth.default_params(d["lengths"])
    ctx = hb.GreedyContext(0, profile=1)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], blosum62, T, X, 0, 0)

        def slots():
            s = list(ctx.section_ms().values())
            assert s[0] > 0 and s[1] > 0 and not any(s[2:]), s
            return s[:2]

        _, cursor = ctx.graph_page((0, 0), 1)       # the first batch of rows
        first = slots()
        _, end = ctx.graph_page(cursor, 1 << 24)    # continues through the other seven batches
        assert end == (n, 0)
        total = slots()
        assert total[0] > first[0] and total[1] > first[1], (first, total)
        ctx.graph_page((0, 0), 1)                   # restarts: the first batch only
        again = slots()
        assert again[0] < total[0] and again[1] < total[1], (total, again)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_statuses(blosum62):
    ctx = hb.GreedyContext(0)
    try:
        with pytest.raises(ValueError):               # status 5: before upload
            ctx.graph_page((0, 0), 10)
        res, offs = O.pack(["WVTAPRSLPVLP", "RSLPVLP", "WVTAPRSLPVLA"])
        ab = np.ones(3, np.int32)
        ctx.upload(res, offs, ab, blosum62, 20, 7, 0, 0)
        with pytest.raises(hb.DataException):         # status 1: X >= the shortest length
            ctx.graph_page((0, 0), 10)
        with pytest.raises(hb.DataException):
            ctx.score_pairs([0], [1])
        assert ctx.score_pairs([0], [2])[0][0] == O.score_with_shift(res[0:12], res[19:31], blosum62, 7, 0)[0]
        bad = res.copy()
        bad[3] = 24
        ctx.upload(bad, offs, ab, blosum62, 20, 3, 0, 0)
        with pytest.raises(hb.FileFormatException):   # status 3
            ctx.graph_page((0, 0), 10)
        ctx.upload(res, offs, ab, blosum62, 20, 3, 0, 0)
        with pytest.raises(ValueError):
            ctx.score_pairs([0], [3])
    finally:
        ctx.close()


@pytest.mark.gpu
def test_score_pairs_against_the_oracle(golden_dir, blosum62):
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    for s1, s2, X, P, mat, score, shift in kats.SCORER_KATS:
        res, offs = O.pack([s1, s2])
        ctx = hb.GreedyContext(0)
        try:
            ctx.upload(res, offs, np.ones(2, np.int32), z[mat], 0, X, P, 0)
            sc, sh = ctx.score_pairs([0], [1])
        finally:
            ctx.close()
        assert sc[0] == score and (shift is None or sh[0] == shift)
        assert (int(sc[0]), int(sh[0])) == O.score_with_shift(res[:len(s1)], res[len(s1):], z[mat], X, P)
    sws = hb.ShiftedScorer(blosum62, -1, 2)
    assert sws.score_with_shift(hb.UniqueSequence("RSLPVLP"), hb.UniqueSequence("WVTAPRSLPVLP")) == \
        O.score_with_shift("RSLPVLP", "WVTAPRSLPVLP", blosum62, 2, -1)
    res, offs = _mixed_case(400, 4, 36, 17)
    rng = np.random.default_rng(2)
    a, b = rng.integers(0, 400, 5000).astype(np.int32), rng.integers(0, 400, 5000).astype(np.int32)
    for M, X, P in ((blosum62, 3, 0), (z["pam250"], 2, -2), (np.eye(24, dtype=np.int32), 3, -1)):
        ctx = hb.GreedyContext(0)
        try:
            ctx.upload(res, offs, np.ones(400, np.int32), M, 0, X, P, 0)
            sc, sh = ctx.score_pairs(a, b)
        finally:
            ctx.close()
        for e in range(0, 5000, 3):
            want = O.score_with_shift(res[offs[a[e]]:offs[a[e] + 1]], res[offs[b[e]]:offs[b[e] + 1]], M, X, P)
            assert (int(sc[e]), int(sh[e])) == want


@pytest.mark.gpu
def test_antibodies_graph_equals_clinkage_rows(blosum62):
    from tests.golden.make_antibodies_clinkage_golden import input_arrays
    res, offs, ab = input_arrays()
    n = len(ab)
    T, X, P = 20, 3, 0
    ctx = hb.GreedyContext(0)
    try:
        rc, G, err = ctx.clinkage(res, offs, ab, blosum62, T, X, P)
        assert rc == 0, err
        kept = G.stats["xhits_kept"]
        ctx.upload(res, offs, ab, blosum62, T, X, P, 0)
        e = _pull(ctx)
        assert len(e) == kept // 2 and len(e) > 5_000_000
        assert (e[:, 0] < e[:, 1]).all() and (e[:, 2] >= T).all()
        key = e[:, 0] * n + e[:, 1]
        assert (np.diff(key) > 0).all()
        sc, sh = ctx.score_pairs(e[:, 1].astype(np.int32), e[:, 0].astype(np.int32))
        assert np.array_equal(sc, e[:, 2]) and np.array_equal(sh, e[:, 3])
    finally:
        ctx.close()
    rng = np.random.default_rng(4)
    for r in rng.choice(len(e), 10000, replace=False):
        i, j, s, k = (int(v) for v in e[r])
        assert O.score_with_shift(res[offs[j]:offs[j + 1]], res[offs[i]:offs[i + 1]], blosum62, X, P) == (s, k)
    i = rng.integers(0, n, 30000)
    j = rng.integers(0, n, 30000)
    i, j = np.minimum(i, j), np.maximum(i, j)
    cand = np.unique((i * n + j)[i < j])
    non = cand[~np.isin(cand, key)][:10000]
    assert len(non) == 10000
    for c in non:
        a, b = int(c // n), int(c % n)
        assert O.score_with_shift(res[offs[b]:offs[b + 1]], res[offs[a]:offs[a + 1]], blosum62, X, P)[0] < T


@pytest.mark.gpu
def test_cpp_driver_graph_mode_on_musi(tmp_path, golden_dir, blosum62):
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
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([hb_build.build_host(), "graph", "-i", str(fa), "-d", str(out), "-m", str(mp)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    assert [s.get_sequence_string() for s in seqs] == strs
    T, X = hb.set_clinkage_threshold(seqs), hb.get_max_shift(seqs)
    want = ref_graph(z["residues"], z["offsets"], blosum62, T, X, 0)
    edges = np.zeros(len(want), hb.EDGE_DTYPE)
    for c, f in enumerate(("seq", "partner", "score", "shift")):
        edges[f] = want[:, c]
    hb.save_score_graph(seqs, edges, str(tmp_path / "py.tsv"))
    assert (out / "score_graph.tsv").read_bytes() == (tmp_path / "py.tsv").read_bytes()
    assert np.array_equal(hb.score_graph(seqs, blosum62).view(np.int32).reshape(-1, 4), want)


@pytest.mark.gpu
def test_clusterings_after_graph_calls(golden_dir, blosum62):
    """a graph pulled half-way, a greedy run and the rest of the graph on one context: the run matches its golden and
    the continued graph is complete; then complete linkage on the same context matches its golden"""
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    T, X, P, K = (int(v) for v in z["params"])
    want = ref_graph(z["residues"], z["offsets"], blosum62, T, X, P)
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(z["residues"], z["offsets"], z["abundance"], blosum62, T, X, P, K)
        first, cursor = ctx.graph_page((0, 0), len(want) // 2)
        ctx.run()
        G = ctx.download()
        assert (G.cluster_id == z["cluster_id"]).all() and (G.member_rank == z["member_rank"]).all()
        assert (G.result_order == z["result_order"]).all() and G.n_multi == int(z["n_multi"])
        rest, end = ctx.graph_page(cursor, len(want))
        assert end == (2457, 0)
        assert np.array_equal(np.concatenate([first, rest]).view(np.int32).reshape(-1, 4), want)
        zc = np.load(os.path.join(golden_dir, "musi_clinkage.npz"))
        Tc, Xc, Pc = (int(v) for v in zc["params"])
        rc, C, err = ctx.clinkage(zc["residues"], zc["offsets"], zc["abundance"], blosum62, Tc, Xc, Pc)
        assert rc == 0, err
        assert (C.cluster_id == zc["cluster_id"]).all() and (C.member_rank == zc["member_rank"]).all()
        assert (C.result_order == zc["result_order"]).all()
    finally:
        ctx.close()
