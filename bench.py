#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 greedy-clustering stage (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference ...                     CPU arm (oracle port, see below)
    python bench.py ... --dump-outputs DIR                   also write the last timed step's clustering as DIR/*.npy

Workload (config.workload): synthetic 1M unique 12-mers, phage-display shape, Zipf abundance,
BLOSUM62, Hammock's automatic parameters (T=20, X=3, K=25000) -- BASELINE.json configs[2], the
configuration the metric is quoted on ("1M peptides"); it fits one GPU.  A "step" is one complete
greedy clustering of that set.  `value` = sequences clustered per second with the inputs already
resident in HBM (hmk_run only); `e2e` = the same through the C-ABI calls a host makes
(hmk_upload from pinned host buffers + hmk_run + hmk_download), copies inside the timed region.
All times are CUDA-event times on the library's stream, max over ranks.

The CPU arm times the oracle (C restatement of the reference's Java; the reference itself cannot
run: no JVM in the image) on all host cores over a BOUNDED sample of the same workload and
extrapolates with a lower bound of the pair scores the reference needs for the full job.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_SEQ = 1_000_000
SEED = 20260101
METRIC = "greedy_cluster_unique_seqs_per_sec"
UNIT = "seq/s"


def workload(n=N_SEQ):
    from hammock_b200 import synth
    d = synth.generate(n, 12, 12, seed=SEED)
    T, X, K = synth.default_params(d["lengths"])
    return d, synth.blosum62(), (T, X, 0, K)


def config(n, world):
    return {"workload": f"synthetic {n} unique 12-mers (phage-display families, Zipf abundance), BLOSUM62, "
                        f"T=20 X=3 P=0 K={int(np.floor(n * 0.025 + 0.5))} (BASELINE.json configs[2])",
            "n_sequences": n, "seed": SEED,
            "parallelism": "single GPU" if world == 1 else f"{world} GPUs: database striped (phase 1) / queries sharded "
                           "(phase 2), NCCL all-gather of best hits and candidates",
            "l2": "flushed between timed steps (256 MiB memset)"}


# ---------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------- CPU arm (oracle port)
ORACLE_BUILD = "gcc -O3 -march=x86-64-v3 -fopenmp (oracle/Makefile), scalar inner loop"


def cpu_sample(d, M, params, p1_steps, p2_queries):
    """Oracle on all host cores over a bounded sample: the first `p1_steps` phase-1 steps (each scores the
    query against every later singleton, like the reference) plus `p2_queries` phase-2 queries.
    BASELINE.md section 3 plans 2000 + 20000 for the 1 M set (used by the cpu_baseline leg); the reference arm
    repeats a quarter of that per step so that K steps + W warm-ups stay within minutes."""
    from oracle import oracle as O
    O.build()
    T, X, P, K = params
    cores = os.cpu_count() or 1
    t = time.time()
    R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K, nthreads=cores,
                         max_p1_steps=p1_steps, max_p2_queries=p2_queries)
    dt = time.time() - t
    pairs = R.counters["p1_pairs"] + R.counters["p2_pairs_early"]
    return {"seconds": dt, "pairs": pairs, "pairs_per_s": pairs / dt, "cores": cores, "p1_steps": p1_steps,
            "p2_queries": p2_queries, "status": R.status, "result": R}


DUMP_LIMIT_BYTES = 60_000_000


def dump_outputs(out_dir, r, limit=DUMP_LIMIT_BYTES):
    """Write the clustering a caller receives (cluster_id, member_rank, result_order, n_multi) as <out_dir>/<name>.npy in
    float64, which holds the int32 results exactly, so that two builds can be compared output for output.  If the whole
    set would exceed `limit` bytes, each array longer than its share is replaced by a fixed, seeded sample of its
    elements, and the sampled positions are written beside it as <name>_index.npy."""
    outputs = {"cluster_id": r.cluster_id, "member_rank": r.member_rank, "result_order": r.result_order,
               "n_multi": r.n_multi}
    os.makedirs(out_dir, exist_ok=True)
    whole = sum(np.size(a) for a in outputs.values()) * 8 <= limit
    cap = limit // (16 * len(outputs))             # 8 B per sampled value + 8 B per position
    for name, a in outputs.items():
        a = np.asarray(a, dtype=np.float64).reshape(-1)
        if not whole and a.size > cap:
            idx = np.sort(np.random.default_rng(SEED).choice(a.size, cap, replace=False))
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def golden_digest(name):
    try:
        with open(os.path.join(ROOT, "tests", "golden", f"{name}_digest.json")) as f:
            return json.load(f)
    except Exception:
        return None


def other_configs(hb, local_rank):
    """The other BASELINE.json configs, one clustering each AFTER the timed region (not bench lines: parity cases with a
    time beside them).  S100k (configs[1]) is checked against the committed digest of a full oracle run; the sweep
    points (configs[3]) against the oracle run right here on the host cores."""
    from hammock_b200 import synth
    from oracle import oracle as O
    out = []
    M62 = synth.blosum62()
    cases = [("S100k: 100000 unique peptides, length 7-12, BLOSUM62 (configs[1])", 100000, 7, 12, "s100k"),
             ("sweep: 50000 x length 30, BLOSUM62 (configs[3])", 50000, 30, 30, None),
             ("sweep: 50000 x length 7-30 mixed, BLOSUM62 (configs[3])", 50000, 7, 30, None)]
    for label, n, lo, hi, gold_name in cases:
        d = synth.generate(n, lo, hi)
        T, X, K = synth.default_params(d["lengths"])
        ctx = hb.GreedyContext(local_rank)
        try:
            ctx.upload(d["residues"], d["offsets"], d["abundance"], M62, T, X, 0, K)
            ctx.run()
            ctx.run()
            st = ctx.stats()
            G = ctx.download()
        finally:
            ctx.close()
        dg = hb.result_digest(G.cluster_id, G.member_rank, G.result_order)
        if gold_name:
            gold = golden_digest(gold_name)
            want, src = (gold or {}).get("sha256"), f"tests/golden/{gold_name}_digest.json (full oracle run)"
        else:
            R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M62, T, X, 0, K, nthreads=os.cpu_count() or 1)
            want, src = hb.result_digest(R.cluster_id, R.member_rank, R.result_order), "oracle run in this process"
        out.append({"workload": label, "T": T, "X": X, "K": K, "ms": round(st["total_ms"], 3),
                    "seq_per_s": round(n / (st["total_ms"] * 1e-3)), "kernel_path": {0: "generic", 1: "packed", 2: "packed per length"}[st["fast_path"]],
                    "lane_bits": st["lane_bits"], "result_digest": dg, "digest_matches_oracle": dg == want, "oracle": src})
    return out


def reference_pairs_lower_bound(n, p1_steps, p1_new, singles, ncl):
    """Pair scores the reference cannot avoid: phase 1 scores each query against every later singleton
    (LimitedGreedySequenceClusterer.java:93), phase 2 at least the founder of every cluster (:60)."""
    p1 = 0
    alive = n
    # step i sees (alive - 1) later singletons; each new cluster removes one partner
    removed_per_step = p1_new / max(p1_steps, 1)
    for i in range(p1_steps):
        p1 += max(alive - 1, 0)
        alive -= 1 + removed_per_step
    return int(p1 + singles * ncl)


# ---------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_SEQ, help="debug only: smaller synthetic set")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the clustering the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # the contract is ONE JSON line on stdout: libraries (NCCL prints its version) write to fd 1 too,
    # so everything but the final line is sent to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        if rank != 0:
            return 0
        d, M, params = workload(args.n)
        vals = []
        for i in range(args.warmup + args.steps):
            s = cpu_sample(d, M, params, 500, 5000)
            if i >= args.warmup:
                vals.append(s)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, vals[-1]["result"])
        # phase sizes of the full job (independent of who computes them)
        T, X, P, K = params
        p1_steps = K  # >= K steps are needed to open K clusters
        need = reference_pairs_lower_bound(args.n, p1_steps, K, args.n - 2 * K, K)
        pps = float(np.mean([v["pairs_per_s"] for v in vals]))
        value = args.n / (need / pps)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": float(np.mean([v["seconds"] for v in vals])) * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32",
                "data": "synthetic", "config": config(args.n, 1),
                "extrapolated": True,
                "note": "value is EXTRAPOLATED from a bounded sample of an extrapolated C port; ms_per_step is the time of one "
                        "sample, not of a whole clustering (a whole CPU clustering of this set takes tens of minutes: "
                        "tests/golden/s1m_digest.json oracle_seconds)",
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": vals[0]["cores"], "kind": "port",
                                 "nproc": os.cpu_count(), "build": ORACLE_BUILD,
                                 "sample": f"EXTRAPOLATED C PORT: C oracle (restatement of the reference Java; no JVM here), "
                                           f"OpenMP on {vals[0]['cores']} threads, first {vals[0]['p1_steps']} phase-1 steps + "
                                           f"{vals[0]['p2_queries']} phase-2 queries per step = {vals[0]['pairs']} pair scores in "
                                           f"{vals[0]['seconds']:.1f} s; extrapolated to the >= {need} pair scores "
                                           "the reference needs for the whole job"},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), file=real_stdout, flush=True)
        return 0

    # ------------------------------------------------------------ GPU arm
    import torch
    import hammock_b200 as hb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- hammock_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    d, M, params = workload(args.n)
    T, X, P, K = params

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = [pinned(d["residues"]), pinned(d["offsets"]), pinned(d["abundance"]), pinned(M.reshape(-1))]
    res, offs, ab, Mp = (k[1] for k in keep)
    ctx = hb.GreedyContext(local_rank, profile=1)
    if world > 1:
        ctx.init_distributed(dist, rank, world)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peaks = ctx.measure_peaks() if rank == 0 else None
    ctx.upload(res, offs, ab, Mp, T, X, P, K)

    def step_resident():
        flush.zero_()
        torch.cuda.synchronize()
        ctx.run()
        return ctx.stats()

    def step_e2e():
        flush.zero_()
        torch.cuda.synchronize()
        ctx.timer_begin()
        ctx.upload(res, offs, ab, Mp, T, X, P, K)
        ctx.run()
        out = ctx.download()
        return ctx.timer_end(), out

    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_wall = time.time()
    dev_ms, stats = [], None
    for _ in range(args.steps):
        stats = step_resident()
        dev_ms.append(stats["total_ms"])
    barrier()
    wall = time.time() - t_wall
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        last = ctx.download()          # every rank holds the whole clustering; rank 0 writes it
        if rank == 0:
            dump_outputs(args.dump_outputs, last)
    ms_per_step = max_over_ranks(float(np.mean(dev_ms)))
    sections = ctx.section_ms()

    # end-to-end through upload + run + download (same K, after one warm-up)
    step_e2e()
    barrier()
    e2e_ms = []
    out = None
    for _ in range(args.steps):
        ms, out = step_e2e()
        e2e_ms.append(ms)
    barrier()
    e2e_ms_per_step = max_over_ranks(float(np.mean(e2e_ms)))

    # Kernel-alone timings for the roofline: in the timed region the partner search of batch i+1 runs
    # concurrently with the resolver of batch i (look-ahead), which inflates per-launch CUDA-event
    # durations; two extra steps with the look-ahead off time every bulk launch on an otherwise idle GPU.
    ctx.set_option("lookahead", 0)
    ctx.upload(res, offs, ab, Mp, T, X, P, K)
    step_resident()
    alone = step_resident()
    ctx.set_option("lookahead", 1)
    barrier()

    # every rank returns the full clustering; the digest of rank 0's e2e result goes into the line, and all ranks
    # must agree on it
    digest = hb.result_digest(out.cluster_id, out.member_rank, out.result_order)
    digests_agree = True
    if dist is not None:
        mine = torch.tensor(list(bytes.fromhex(digest)), dtype=torch.uint8, device="cuda")
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        digests_agree = all(bool((e == mine).all().item()) for e in every)

    if rank == 0:
        n = args.n
        bulk_s = alone["bulk_kernel_ms"] * 1e-3
        ops_per_s = alone["bulk_ops"] / bulk_s
        gold = golden_digest("s1m") if n == N_SEQ else None
        ncu = None
        ncu_traffic = None
        for prof_name in ("r02_ncu_bulk_filter_full.json", "r01_ncu_bulk_filter_full.json"):
            try:
                with open(os.path.join(ROOT, "profiles", prof_name)) as f:
                    prof = json.load(f)
            except Exception:
                continue
            for l in prof["launches"]:
                if "hmk_bulk_filter<0" in l["Kernel Name"].replace("(int)", ""):
                    def _b(key):   # ncu picks a unit per column
                        u = prof["units"][key]
                        return float(l[key]) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[u]
                    ncu_traffic = {"bytes_per_launch": _b("dram__bytes_read.sum") + _b("dram__bytes_write.sum"),
                                   # 8 B packed word + 4 B singleton flag per database item, 16 B per kept hit (0.26 % of pairs)
                                   "algorithmic_bytes_per_launch": 12 * n + 16 * 0.0026 * n * stats["p1_steps"] / max(stats["p1_batches"], 1),
                                   "source": f"profiles/{prof_name} (ncu --set full, one partner-search launch)"}
                    ncu = {"source": f"profiles/{prof_name}",
                           "smem_wavefronts_pct_of_peak": float(l["l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"]),
                           "lsu_pipe_pct": float(l["sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active"]),
                           "alu_pipe_pct": float(l["sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active"]),
                           "issue_slots_pct": float(l["smsp__issue_active.avg.pct_of_peak_sustained_active"]),
                           "smem_wavefronts": float(l["l1tex__data_pipe_lsu_wavefronts_mem_shared.sum"]),
                           "smem_bank_conflicts": float(l["l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum"]),
                           "sm_cycles_active_avg_over_elapsed_max": float(l["sm__cycles_active.avg"]) / float(l["sm__cycles_elapsed.max"])}
                    break
            if ncu:
                break
        peak = peaks["int32_iadd3_per_s"]
        lds_bytes = alone["bulk_pairs"] * 12 * 4              # filter pass: L positions x one u32 word per pair (verify look-ups not counted)
        line = {
            "metric": METRIC, "value": n / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32 (u8x4 packed lanes)", "data": "synthetic",
            "config": config(n, world),
            "result_digest": digest,
            "digest_matches_golden": (digest == gold["sha256"]) if gold else None,
            "digest_golden": "tests/golden/s1m_digest.json: sha256(cluster_id || member_rank || result_order) of a FULL CPU-oracle run "
                             "on this input (scripts/make_s1m_digest.py)" if gold else None,
            "digests_agree_across_ranks": digests_agree,
            "gapless_gcups": alone["bulk_cells"] / bulk_s / 1e9,
            "e2e": {"value": n / (e2e_ms_per_step * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_per_step,
                    "h2d_bytes_per_step": int(res.nbytes + offs.nbytes + ab.nbytes + Mp.nbytes),
                    "d2h_bytes_per_step": int(out.cluster_id.nbytes + out.member_rank.nbytes + out.result_order.nbytes)},
            "gpu_launches": int(stats["total_launches"]) * args.steps,
            "roofline": {
                "kernel": "hmk_bulk_filter<*,12> (packed gapless scorer, filter + exact verify: partner search and cluster search; "
                          "the small dense tables use hmk_bulk_fast<2,2>)",
                # the pipe that binds the kernel: shared-memory loads of the query profiles.  Neither HBM (0.2 % of peak) nor
                # tensor cores (north_star rules them out) bound this path.
                "bound": "smem", "unit": "GB/s",
                "achieved": lds_bytes / bulk_s / 1e9, "peak": peaks["smem_lds_bytes_per_s"] / 1e9,
                "frac": lds_bytes / bulk_s / peaks["smem_lds_bytes_per_s"],
                "note": "achieved = ALGORITHMIC shared-memory bytes (48 B per pair: 12 positions x one u32 filter word; the exact "
                        "verify look-ups of the 2-3 % candidates and the queue traffic are overhead, not counted) / summed launch "
                        "time; peak = conflict-free LDS.32 stream measured live (hmk_measure_peaks)",
                "measured": "kernels timed alone: two extra steps with the phase-1 look-ahead switched off, CUDA events "
                            "around every bulk launch (in the timed region launches overlap the resolver)",
                "bytes_per_launch": lds_bytes / max(alone["bulk_launches"], 1),
                "launches_per_step": alone["bulk_launches"],
                "avg_launch_ms": alone["bulk_kernel_ms"] / max(alone["bulk_launches"], 1),
                "ncu": ncu,
                # SURVEY.md 8(d)'s figure, kept under its own name: algorithmic int ops (79 per pair: 72 cell adds + 7 shift
                # maxima) / launch time against the measured scalar IADD3 peak.  It exceeds 1 because one u32 add carries 4 u8
                # diagonals and the filter decides 97 % of the pairs with 12 look-ups + 6 adds: NOT a utilisation figure.
                "algorithmic_int_alu": {"unit": "Gop/s (int32)", "achieved": ops_per_s / 1e9, "peak": peak / 1e9,
                                        "algorithmic_frac": ops_per_s / peak,
                                        "peak_source": "measured live: dependent-free IADD3 stream; IADD3+IMAD dual-pipe stream reaches "
                                                       f"{peaks['int32_mix_per_s'] / 1e9:.0f} Gop/s",
                                        "ops_per_launch": alone["bulk_ops"] / max(alone["bulk_launches"], 1)},
                "overlapped": {"sum_launch_ms": stats["bulk_kernel_ms"],
                               "frac": stats["bulk_pairs"] * 48 / (stats["bulk_kernel_ms"] * 1e-3) / peaks["smem_lds_bytes_per_s"]},
                "traffic": ncu_traffic,
                "share_of_step": alone["bulk_kernel_ms"] / ms_per_step,
                "share_of_step_without_lookahead": alone["bulk_kernel_ms"] / alone["total_ms"],
                "step_ms_without_lookahead": alone["total_ms"]},
            "work": {"bulk_pairs": stats["bulk_pairs"], "scalar_pairs": stats["scalar_pairs"],
                     # phase 2 reuses the founder scores that the phase-1 partner searches already produced (symmetric
                     # matrix): the reference scores these (singleton, cluster) pairs a second time
                     "pairs_served_by_phase1_hits": (stats["p2_queries"] * stats["p1_new_clusters"]
                                                     if stats["flags"] & 1 else 0),
                     "reference_min_pairs": reference_pairs_lower_bound(n, stats["p1_steps"], stats["p1_new_clusters"],
                                                                        stats["p2_queries"], stats["p1_new_clusters"]),
                     "bulk_cells": stats["bulk_cells"], "p1_steps": stats["p1_steps"], "p1_batches": stats["p1_batches"],
                     "p1_restarts": stats["p1_restarts"],
                     "p2_queries": stats["p2_queries"], "p2_assigned": stats["p2_assigned"],
                     "multi_member_clusters": stats["p1_new_clusters"], "p2_iterations": stats["p2_rounds"],
                     "kept_hits": stats["xhits_kept"], "kept_hit_capacity": stats["xhits_capacity"], "flags": stats["flags"]},
            "sections_ms": {k: round(v, 2) for k, v in sections.items()},
            "wall_s_timed_region": wall,
            "clocks": clocks,
        }
        if not args.no_cpu_baseline and world == 1:
            s = cpu_sample(d, M, params, 2000, 20000)
            need = reference_pairs_lower_bound(n, stats["p1_steps"], stats["p1_new_clusters"], stats["p2_queries"],
                                               stats["p1_new_clusters"])
            v = n / (need / s["pairs_per_s"])
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": s["cores"], "kind": "port", "nproc": os.cpu_count(), "build": ORACLE_BUILD,
                "extrapolated": True,
                "sample": f"EXTRAPOLATED C PORT: C oracle (restatement of the reference Java; no JVM in the image), OpenMP on "
                          f"{s['cores']} threads: first {s['p1_steps']} phase-1 steps + {s['p2_queries']} phase-2 queries = "
                          f"{s['pairs']} pair scores in {s['seconds']:.1f} s ({s['pairs_per_s'] / 1e6:.1f} M pairs/s), extrapolated "
                          f"to the >= {need} pair scores the reference's early-exit evaluation needs for the whole job"}
            if gold and gold.get("oracle_seconds"):
                line["cpu_baseline"]["full_run_elsewhere"] = (
                    f"a FULL oracle clustering of this set took {gold['oracle_seconds']} s on {gold['oracle_threads']} threads of the "
                    "build container (tests/golden/s1m_digest.json)")
            if not args.no_other_configs:
                try:
                    line["other_configs"] = other_configs(hb, local_rank)
                except Exception as e:      # noqa: BLE001 -- the headline line must still be printed
                    line["other_configs"] = {"error": repr(e)}
        print(json.dumps(line), file=real_stdout, flush=True)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
