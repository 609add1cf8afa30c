"""CPU model of how hmk_bulk_filter hands its filter candidates out (hmk_kernels.cuh: hmk_transpose32, hmk_nth_bit and
the `octet`, `resolve` and `verify` lambdas).  Every lane keeps one bit per (query, exact word) that passed for its own item; at the
end of each group of HMK_FGROUP queries the warp lists the candidates query-major (lane minor) and moves them into a
round of 32, one per lane, that is verified when full and at the end of the chunk.  The model follows the kernel's
arithmetic step by step (transpose, scan, binary search, n-th set bit) and checks that every passed pair is verified
exactly once, with the exact words that passed, and that the pairs reaching the hit path are the ones the old
per-warp shared-memory queue produced."""
import numpy as np
import pytest

GROUP = 32       # HMK_FGROUP
KEEP = [0x0000FFFF, 0x00FF00FF, 0x0F0F0F0F, 0x33333333, 0x55555555]


def transpose32(rows):
    """hmk_transpose32 for the whole warp: rows[l] = lane l's word; returns the lanes' words afterwards"""
    x = [int(v) & 0xFFFFFFFF for v in rows]
    for i, s in enumerate((16, 8, 4, 2, 1)):
        k = KEEP[i]
        y = [x[lane ^ s] for lane in range(32)]
        x = [((x[l] & ~k) | ((y[l] & ~k) >> s)) & 0xFFFFFFFF if l & s else ((x[l] & k) | ((y[l] & k) << s)) & 0xFFFFFFFF
             for l in range(32)]
    return x


def nth_bit(m, n):
    pos = 0
    for s in (16, 8, 4, 2, 1):
        c = bin(m & ((1 << s) - 1)).count("1")
        if n >= c:
            n -= c
            m >>= s
            pos += s
    return pos


class Warp:
    """one warp's round (registers) and the candidates it verified, in order"""

    def __init__(self):
        self.fill = 0
        self.round = [None] * 32
        self.verified = []          # lists of (t, item, halves), one list per verify call

    def verify(self):
        assert 1 <= self.fill <= 32
        self.verified.append([self.round[l] for l in range(self.fill)])
        self.fill = 0
        self.round = [None] * 32

    def resolve(self, g0, qn, items, m0, m1, valid):
        pm = [(m0[l] | m1[l]) if valid[l] else 0 for l in range(32)]
        if not any(pm):
            return
        col = transpose32(pm)
        cnt = [bin(c).count("1") for c in col]
        incl = list(np.cumsum(cnt))
        n = incl[31]
        base = 0
        while base < n:
            take = min(32 - self.fill, n - base)
            new = list(self.round)
            for lane in range(32):
                g = base + lane - self.fill
                gq = min(max(g, 0), n - 1)
                k = 0
                for s in (16, 8, 4, 2, 1):
                    if incl[k + s - 1] <= gq:
                        k += s
                ck = col[k]
                first = incl[k] - cnt[k]
                src = nth_bit(ck, gq - first)
                h = ((m0[src] >> k) & 1) | (((m1[src] >> k) & 1) << 1)
                if lane >= self.fill and g < base + take:
                    assert k < GROUP and g0 + k < qn and (ck >> src) & 1 and h != 0
                    new[lane] = (g0 + k, items[src], h)
            self.round = new
            self.fill += take
            base += take
            if self.fill == 32:
                self.verify()


def run_rows(passed, valid_rows, items_rows, qn):
    """passed[row][lane][t] in {0, 1, 2, 3}: exact words whose filter bytes passed; returns the verify calls.
    All rows belong to one chunk: the round is flushed after the last one."""
    w = Warp()
    for P, valid, items in zip(passed, valid_rows, items_rows):
        for g0 in range(0, qn, GROUP):
            gend = min(qn, g0 + GROUP)
            m0 = [sum(1 << (t - g0) for t in range(g0, gend) if P[l][t] & 1) for l in range(32)]
            m1 = [sum(1 << (t - g0) for t in range(g0, gend) if P[l][t] & 2) for l in range(32)]
            w.resolve(g0, qn, items, m0, m1, valid)
    if w.fill:
        w.verify()
    return w.verified


def old_queue(passed, valid_rows, items_rows, qn):
    """the (t, item, halves) entries the removed per-warp queue received: per row, query by query, lanes in order"""
    out = []
    for P, valid, items in zip(passed, valid_rows, items_rows):
        for t in range(qn):
            for l in range(32):
                if valid[l] and P[l][t]:
                    out.append((t, items[l], int(P[l][t])))
    return out


def check(passed, valid_rows, qn):
    items_rows = [[1000 * r + l for l in range(32)] for r in range(len(passed))]
    calls = run_rows(passed, valid_rows, items_rows, qn)
    got = [c for call in calls for c in call]
    want = old_queue(passed, valid_rows, items_rows, qn)
    assert sorted(got) == sorted(want)
    assert len(set((t, i) for t, i, _ in got)) == len(got)          # each pair exactly once
    assert got == want                                               # and in query-major order within each row
    assert all(len(c) == 32 for c in calls[:-1])                     # only the last round of the chunk is part-filled
    return calls


@pytest.mark.parametrize("qn", [1, 5, 31, 32, 33, 56])
def test_random_masks(qn):
    rng = np.random.default_rng(qn)
    for rate in (0.02, 0.043, 0.3):
        rows = 4
        passed = (rng.random((rows, 32, qn)) < rate) * rng.integers(1, 4, (rows, 32, qn))
        valid = rng.random((rows, 32)) < 0.9
        check(passed, valid, qn)


def test_edge_masks():
    qn = 56
    full = np.full((1, 32, qn), 3)
    calls = check(full, np.ones((1, 32), bool), qn)
    assert len(calls) == qn and all([c[0] for c in call] == [t] * 32 for t, call in enumerate(calls))
    assert check(np.zeros((2, 32, qn), int), np.ones((2, 32), bool), qn) == []
    one = np.zeros((1, 32, qn), int)
    one[0, 17, :] = 2                                                 # one lane holds everything
    calls = check(one, np.ones((1, 32), bool), qn)
    assert [len(c) for c in calls] == [32, 24] and {c[1] for call in calls for c in call} == {17}
    invalid = np.full((1, 32, qn), 1)                                 # lanes without an item never hand out candidates
    assert check(invalid, np.zeros((1, 32), bool), qn) == []


def test_round_carries_across_groups_and_rows():
    qn = 56
    passed = np.zeros((3, 32, qn), int)
    passed[0, 0:20, 3] = 1          # 20 candidates in group 0 of row 0
    passed[0, 5:25, 40] = 3         # 20 more in group 1: the round fills at 32 across the group boundary
    passed[1, 31, 55] = 2           # the remaining 8 wait for the next row
    passed[2, 0, 0] = 1
    calls = check(passed, np.ones((3, 32), bool), qn)
    assert [len(c) for c in calls] == [32, 10]


def octet_masks(tops, gn):
    """the kernel's packing of one group: tops[q] = f & 0x80808080 of query q (gn <= 32 of them) -> (m0, m1)"""
    m0 = m1 = 0
    for o0 in range(0, gn, 8):
        c = min(8, gn - o0)
        x = 0
        for q in range(o0, o0 + c):
            x = (x >> 1) | tops[q]
        x >>= 8 - c
        y = x | (x >> 8)
        m0 = ((m0 >> 8) | ((y & 0xFF) << 24)) & 0xFFFFFFFF          # __funnelshift_r(m0, y, 8)
        m1 = ((m1 >> 8) | (((y >> 16) & 0xFF) << 24)) & 0xFFFFFFFF  # __funnelshift_r(m1, y >> 16, 8)
    octets = (gn + 7) // 8
    return m0 >> (8 * (4 - octets)), m1 >> (8 * (4 - octets))


@pytest.mark.parametrize("gn", [1, 7, 8, 9, 24, 31, 32])
def test_octet_packing(gn):
    rng = np.random.default_rng(gn)
    for _ in range(200):
        tops = [int(v) & 0x80808080 for v in rng.integers(0, 2 ** 32, gn, dtype=np.uint64)]
        tops[rng.integers(gn)] = 0x80808080
        m0, m1 = octet_masks(tops, gn)
        assert m0 == sum(1 << q for q in range(gn) if tops[q] & 0x00008080)
        assert m1 == sum(1 << q for q in range(gn) if tops[q] & 0x80800000)


def test_transpose_and_nth_bit():
    rng = np.random.default_rng(7)
    rows = [int(v) for v in rng.integers(0, 2 ** 32, 32, dtype=np.uint64)]
    cols = transpose32(rows)
    for c in range(32):
        assert cols[c] == sum(((rows[l] >> c) & 1) << l for l in range(32))
    for m in (1, 0x80000000, 0xFFFFFFFF, 0x12345678):
        bits = [b for b in range(32) if (m >> b) & 1]
        assert [nth_bit(m, n) for n in range(len(bits))] == bits
