"""Phase-1 look-ahead pipeline: partner searches of prepared batches run on a side stream, their tails (merge, dense tables,
masks) on a tail stream, and a resolver exit that throws the prepared batches away bumps a discard counter at which their
persistent searches stop taking work (Engine::stage_partner_search / Engine::phase1, hmk_bulk_filter).

CPU: a cancelled search leaves an arbitrary part of its hits in the kept-hit buffer of phase 2.  The look-ahead model of
test_phase1_model.py gets discarded batches that contribute random subsets of their hits, with their batch tags; phase 2's
candidate pairs from the kept hits must still equal the separate founder pass, and must not without the tag test.

GPU: the resolver's discarding exits (DONE, RESTART, GROW, NPE) and the keeping one (GROWHITS) with prepared batches in
flight, against the oracle and against lookahead 0; two 1 M runs in one context (the counter restarts with every run)."""
import json
import os

import numpy as np
import pytest

from tests.test_phase1_model import CONTINUE, Model, _instance, sequential


class CancellingModel(Model):
    """A resolver exit other than CONTINUE throws away up to `depth` prepared batches.  Each got its batch id when it
    was staged and searched the sequences behind the batch before it, against a state older than the exit; its
    persistent search stopped at some chunk, so it appended an arbitrary subset of its qualifying hits."""

    def __init__(self, *args, keep_p=None, **kw):
        super().__init__(*args, **kw)
        self.keep_p = keep_p
        self.discarded = 0

    def resolve(self, bt, hook):
        seen = list(self.slot)
        st = super().resolve(bt, hook)
        if st != CONTINUE:
            last = bt["qid"][-1]
            for _ in range(self.depth):
                qid = self.select(seen, last + 1, self.B)
                if not qid:
                    break
                self.batch_id += 1
                p = self.rng.random() if self.keep_p is None else self.keep_p
                for q in qid:
                    for i in range(q + 1, self.n):
                        if seen[i] < 0 and self.S[i][q] >= self.T and self.rng.random() < p:
                            self.xhits.append((q, i, self.S[i][q], self.batch_id))
                self.discarded += 1
                last = qid[-1]
        return st


class _AnyTag:
    """qbatch stand-in for which every tag matches: the kept-hit filter without its batch-tag test"""
    class _Eq:
        def __eq__(self, other):
            return True

        def __ne__(self, other):
            return False

    def __getitem__(self, i):
        return self._Eq()


@pytest.mark.parametrize("keep_p", [None, 1.0])
def test_phase2_pairs_ignore_any_part_of_discarded_batches(keep_p):
    rng = np.random.default_rng(31 if keep_p is None else 32)
    discarded = runs = untagged_wrong = 0
    for trial in range(40):
        n = int(rng.integers(40, 140))
        S, ab, T = _instance(rng, n, int(rng.choice([12, 25])), bool(trial % 3 == 0), False)
        K = max(2, n // int(rng.choice([4, 6, 10])))
        m = CancellingModel(S, ab, T, K, int(rng.choice([8, 16, 32])), 1, int(rng.choice([0, 4])), 0,
                            int(rng.choice([1, 2])), rng, keep_p=keep_p)
        got = m.run()
        assert got == sequential(S, ab, T, K)
        if got["status"] != 0:
            continue
        runs += 1
        discarded += m.discarded
        kept = m.pairs_from_kept_hits()
        direct = sorted(m.pairs_direct())
        assert len(kept) == len(set(kept)) and sorted(kept) == direct, trial
        m.qbatch = _AnyTag()
        untagged_wrong += sorted(m.pairs_from_kept_hits()) != direct
    assert runs > 10 and discarded > runs      # DONE ends every run, and discards what is prepared behind it
    assert untagged_wrong > 0                  # the tag test is what drops them


# ---------------------------------------------------------------- GPU
def _oracle(d, M, T, X, P, K):
    from oracle import oracle as O
    return O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K, nthreads=os.cpu_count() or 1)


def _run(d, M, T, X, P, K, **opts):
    import hammock_b200 as hb
    ctx = hb.GreedyContext(0, **opts)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K)
        rc, msg = ctx.run_status()
        st = ctx.stats()
        if rc == 2:
            return {"npe": st["error_step"]}, st
        assert rc == 0, msg
        G = ctx.download()
        return {"cluster_id": G.cluster_id.copy(), "member_rank": G.member_rank.copy(),
                "result_order": G.result_order.copy(), "n_multi": G.n_multi}, st
    finally:
        ctx.close()


def _same(a, b):
    if "npe" in a or "npe" in b:
        return a == b
    return (a["n_multi"] == b["n_multi"] and np.array_equal(a["cluster_id"], b["cluster_id"])
            and np.array_equal(a["member_rank"], b["member_rank"]) and np.array_equal(a["result_order"], b["result_order"]))


# mid-size sets with full look-ahead batches (batch 64, two prepared behind each) and the resolver exit each case forces:
# (name, n, K as a fraction of n, options, batches phase 1 must at least resolve, stats field that shows the exit was taken)
CASES = [
    ("done_K_early", 4000, 0.004, {}, 1, None),
    ("restart_kb1", 5000, 0.2, {"kb": 1}, 8, "p1_restarts"),
    ("grow_capq1", 5000, 0.2, {"capq": 1}, 8, None),
    ("growhits_cap1024", 6000, 0.2, {"hit_cap": 1024}, 8, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_discarding_exits_with_batches_in_flight(case, blosum62):
    from hammock_b200 import synth
    name, n, kfrac, opts, min_batches, counter = case
    d = synth.generate(n, 12, 12, seed=4242 + n)
    T, X, _ = synth.default_params(d["lengths"])
    K = int(n * kfrac)
    R = _oracle(d, blosum62, T, X, 0, K)
    assert R.status == 0
    ref = {"cluster_id": R.cluster_id, "member_rank": R.member_rank, "result_order": R.result_order, "n_multi": R.n_multi}
    got, st = _run(d, blosum62, T, X, 0, K, batch=64, lookahead=2, **opts)
    assert _same(got, ref), name
    assert st["p1_batches"] >= min_batches, (name, st)
    if counter:
        assert st[counter] > 0, (name, st)
    got0, _ = _run(d, blosum62, T, X, 0, K, batch=64, lookahead=0, **opts)
    assert _same(got0, got), name


@pytest.mark.gpu
def test_npe_exit_with_batches_in_flight(blosum62):
    """an unlimited cluster count lets phase 1 of this input run into the reference's null-object step"""
    from hammock_b200 import synth
    d = synth.generate(3000, 12, 12, seed=77)
    T, X, _ = synth.default_params(d["lengths"])
    K = 10 ** 6
    R = _oracle(d, blosum62, T, X, 0, K)
    assert R.status == 2, "the input no longer reaches the null-object step"
    got, _ = _run(d, blosum62, T, X, 0, K, batch=64, lookahead=2)
    got0, _ = _run(d, blosum62, T, X, 0, K, batch=64, lookahead=0)
    assert got == {"npe": R.counters["npe_step"]} and got0 == got


@pytest.mark.gpu
def test_two_runs_in_one_context_match_the_1m_digest(golden_dir):
    import hammock_b200 as hb
    from hammock_b200 import synth
    gold = json.load(open(os.path.join(golden_dir, "s1m_digest.json")))
    d = synth.generate(1_000_000, 12, 12)
    T, X, K = synth.default_params(d["lengths"])
    ctx = hb.GreedyContext(0)
    try:
        ctx.upload(d["residues"], d["offsets"], d["abundance"], synth.blosum62(), T, X, 0, K)
        for _ in range(2):
            ctx.run()
            G = ctx.download()
            assert hb.result_digest(G.cluster_id, G.member_rank, G.result_order) == gold["sha256"]
    finally:
        ctx.close()
