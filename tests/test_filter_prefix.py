"""The filter kernel's shared residue prefix: where every scored item of a warp holds the same residues 0..2, their filter
rows are summed once per query (hmk_bulk_filter, hmk_prefix_* in hmk_common.h) instead of once per lane.

CPU: the warp's decision (tests/cpp/prefix_shim.cpp) against brute force.  GPU: hmk_bulk_probe over explicit id lists
whose warps share a prefix in every block, in none, or in every other block, with masked items that hide or expose a
differing residue, against exact pair scores."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from hammock_b200 import synth
from tests.test_bulk_kernels import B62, F12, Ref, check_emit, check_topk, context, assert_kernel, tierank

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PREFIX = 3


def pack(seqs):
    """5-bit packed words as the engine stores them (position j in bits 5j..5j+4, length in bits 60..63)"""
    seqs = np.asarray(seqs, dtype=np.uint64)
    w = np.zeros(len(seqs), dtype=np.uint64)
    for j in range(seqs.shape[1]):
        w |= seqs[:, j] << np.uint64(5 * j)
    return w | (np.uint64(seqs.shape[1]) << np.uint64(60))


def brute_prefix(seqs, scored):
    s = np.asarray(seqs)[np.asarray(scored, dtype=bool)]
    return PREFIX if len(s) and (s[:, :PREFIX] == s[:1, :PREFIX]).all() else 0


# ---------------------------------------------------------------- CPU: the warp's decision
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("prefix_shim") / "libprefix.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O1", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "prefix_shim.cpp")])
    L = ctypes.CDLL(out)
    L.shim_warp_prefix.restype = ctypes.c_int32
    L.shim_warp_prefix.argtypes = [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint8)]

    def decide(seqs, scored):
        w = pack(seqs)
        m = np.ascontiguousarray(scored, dtype=np.uint8)
        return L.shim_warp_prefix(w.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                  m.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    return decide


def test_prefix_constructed_warps(shim):
    rng = np.random.default_rng(1)
    base = np.tile(rng.integers(0, 24, 12), (32, 1))
    base[:, PREFIX:] = rng.integers(0, 24, (32, 12 - PREFIX))       # the residues after the prefix differ freely
    every = np.ones(32, dtype=bool)
    cases = {"all lanes scored": (base, every, PREFIX)}
    for pos, want in ((0, 0), (1, 0), (2, 0), (3, PREFIX), (11, PREFIX)):
        s = base.copy()
        s[17, pos] = (s[17, pos] + 5) % 24
        cases[f"lane 17 differs in residue {pos}"] = (s, every, want)
        hidden = every.copy()
        hidden[17] = False
        cases[f"lane 17 differs in residue {pos}, not scored"] = (s, hidden, PREFIX)
    s = base.copy()
    s[0, 2] = (s[0, 2] + 1) % 24
    lead_out = every.copy()
    lead_out[0] = False
    cases["lane 0 differs, not scored"] = (s, lead_out, PREFIX)
    cases["lane 0 differs, scored"] = (s, every, 0)
    z = s.copy()
    z[~lead_out] = 0                                                 # the kernel's unscored lanes carry word 0
    cases["lane 0 word 0, not scored"] = (z, lead_out, PREFIX)
    cases["no lane scored"] = (base, np.zeros(32, dtype=bool), 0)
    one = np.zeros(32, dtype=bool)
    one[31] = True
    cases["only lane 31 scored"] = (s, one, PREFIX)
    cases["key 0 in every scored lane"] = (np.zeros((32, 12), dtype=np.int64), lead_out, PREFIX)
    top = np.full((32, 12), 23)
    cases["key 23,23,23, lane 0 word 0 not scored"] = (np.where(lead_out[:, None], top, 0), lead_out, PREFIX)
    for name, (seqs, scored, want) in cases.items():
        assert brute_prefix(seqs, scored) == want, name
        assert shim(seqs, scored) == want, name


def test_prefix_random_warps(shim):
    rng = np.random.default_rng(2)
    seen = {0: 0, PREFIX: 0}
    for it in range(4000):
        alpha = int(rng.choice([1, 2, 3, 24]))                      # small alphabets make shared prefixes likely
        seqs = rng.integers(0, alpha, (32, 12))
        if it % 3 == 0:
            seqs[:, :PREFIX] = seqs[0, :PREFIX]
            seqs[rng.integers(32), rng.integers(12)] = rng.integers(24)
        scored = rng.random(32) < rng.choice([0.0, 0.05, 0.5, 1.0])
        want = brute_prefix(seqs, scored)
        seen[want] += 1
        assert shim(seqs, scored) == want, (it, seqs[:, :PREFIX].tolist(), scored.astype(int).tolist())
    assert min(seen.values()) > 500, seen


# ---------------------------------------------------------------- GPU: probes over constructed warps
NB = 48                  # blocks of 32 ids
T, X = 20, 3


def constructed():
    """12-mers in blocks of 32 ids.  Block kinds (by block index mod 6): 0 same prefix; 1 one lane differs in residue 3
    (still shared); 2 one lane differs in residue 2; 3 one lane differs in residue 0; 4 lane 0 differs in residue 1 and
    is masked; 5 one lane differs in residue 2 and is masked.  Returns the data, the clustered mask and the kinds."""
    d = synth.generate(NB * 32, 12, 12, seed=31)
    res = np.asarray(d["residues"]).reshape(-1, 12).copy()
    rng = np.random.default_rng(32)
    clustered = np.zeros(NB * 32, dtype=bool)
    kinds = np.arange(NB) % 6
    for b in range(NB):
        blk = res[32 * b:32 * b + 32]
        blk[:, :PREFIX] = blk[0, :PREFIX]
        k = kinds[b]
        if k == 0:
            continue
        lane = 0 if k == 4 else int(rng.integers(1, 32))
        pos = {1: 3, 2: 2, 3: 0, 4: 1, 5: 2}[k]
        blk[lane, pos] = (blk[lane, pos] + 1 + rng.integers(19)) % 20
        if k in (4, 5):
            clustered[32 * b + lane] = True
    d = dict(d, residues=np.ascontiguousarray(res.reshape(-1), dtype=np.uint8))
    for b in range(NB):
        sl = slice(32 * b, 32 * b + 32)
        assert brute_prefix(res[sl], ~clustered[sl]) == (0 if kinds[b] in (2, 3) else PREFIX), b
    return d, clustered, kinds


@pytest.fixture(scope="module")
def case():
    d, clustered, kinds = constructed()
    blocks = np.arange(NB)
    shared, differ = blocks[np.isin(kinds, (0, 1, 4, 5))], blocks[np.isin(kinds, (2, 3))]
    alt = np.ravel(np.stack([shared[:len(differ)], differ], axis=1))   # shared, differing, shared, ...
    lists = {name: np.concatenate([np.arange(32 * b, 32 * b + 32) for b in bl]).astype(np.int32)
             for name, bl in (("shared", shared), ("differ", differ), ("alternating", alt))}
    R = Ref(d, B62, X, 0, [(np.arange(NB * 32), np.arange(64))])
    return d, clustered, lists, R


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 31, 32, 33, 55, 56, 57])
def test_prefix_blocks_against_exact_scores(case, nq):
    d, clustered, lists, R = case
    rank = tierank(d["abundance"])
    q = np.arange(nq)
    found = 0
    for persistent in (1, 0):
        ctx = context(d, B62, T, X, 0, persistent=persistent)
        try:
            for name, db in lists.items():
                what = f"{name} nq={nq} persistent={persistent}"
                r, nk, _ = check_topk(ctx, R, q, T, 8, rank, db=db, clustered=clustered, what=what)
                assert_kernel(r["kernel"], F12, persistent)
                r, nh = check_emit(ctx, R, q, T, db=db, clustered=clustered, what="emit " + what)
                assert_kernel(r["kernel"], F12)
                found += nk + nh
                if name != "differ":            # without the mask, blocks of kinds 4 and 5 expose their differing lane
                    check_emit(ctx, R, q, T, db=db, what="emit unmasked " + what)
        finally:
            ctx.close()
    assert found > 0
