"""Device timeline of one clustering of the bench workload, from torch.profiler (CUPTI records every kernel, memset and
copy of the process, the library's included).  Attributes phase-1 time to streams and shows what the partner-search
stream does between two partner searches.

    python scripts/p1_timeline.py OUT_DIR [--n N] [--tag NAME]

Runs one warm-up clustering and one clustering under the profiler (same options as bench.py: profile=1), then writes
OUT_DIR/p1_timeline_<tag>.json:
  launches           per kernel name: count, total and mean µs over the profiled clustering
  phase1             window from the first hmk_select_queries to the end of the last hmk_p1_resolve_kernel; per stream the
                     busy time (union of its activities) and the idle time inside that window
  partner_gaps       on the stream that runs most hmk_bulk_filter<0,12> launches (the partner searches): the time between
                     the end of one search and the start of the next, split into what else ran on that stream in between
                     and the pure gap, as sums and per batch
  end_of_phase1      time from the end of the last resolver to the first phase-2 kernel (hmk_count_unassigned), and what
                     ran in between
  sections_ms, stats the library's own section timers of a separate, unprofiled clustering
Profiled kernel times are inflated; use this file to attribute time and bench.py for the headline number.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch                                   # noqa: E402
import hammock_b200 as hb                      # noqa: E402
from hammock_b200 import synth                 # noqa: E402

SEARCH = re.compile(r"hmk_bulk_filter<0, ?12>")
GPU_CATS = ("kernel", "gpu_memset", "gpu_memcpy")


def union_len(iv, lo=None, hi=None):
    """total length of the union of intervals [a, b), optionally clipped to [lo, hi)"""
    tot, end = 0.0, None
    for a, b in sorted(iv):
        if lo is not None:
            a, b = max(a, lo), min(b, hi)
        if b <= a:
            continue
        if end is None or a > end:
            tot += b - a
            end = b
        elif b > end:
            tot += b - end
            end = b
    return tot


def dist(xs):
    if not xs:
        return {}
    a = np.asarray(xs, dtype=np.float64)
    return {"n": int(a.size), "sum": round(float(a.sum()), 1), "mean": round(float(a.mean()), 2),
            "p10": round(float(np.percentile(a, 10)), 2), "p50": round(float(np.percentile(a, 50)), 2),
            "p90": round(float(np.percentile(a, 90)), 2), "max": round(float(a.max()), 2)}


def short(name):
    return re.sub(r"\(.*\)$", "", name.replace("void ", ""))


def analyse(events):
    ev = [e for e in events if e.get("ph") == "X" and e.get("cat") in GPU_CATS]
    for e in ev:
        e["t0"], e["t1"], e["s"], e["n"] = float(e["ts"]), float(e["ts"]) + float(e["dur"]), e["args"].get("stream"), short(e["name"])
    ev.sort(key=lambda e: e["t0"])
    launches = {}
    for e in ev:
        if e["cat"] != "kernel":
            continue
        r = launches.setdefault(e["n"], {"count": 0, "total_us": 0.0})
        r["count"] += 1
        r["total_us"] += e["t1"] - e["t0"]
    for r in launches.values():
        r["mean_us"] = round(r["total_us"] / r["count"], 2)
        r["total_us"] = round(r["total_us"], 1)
    launches = dict(sorted(launches.items(), key=lambda kv: -kv[1]["total_us"]))

    sel = [e for e in ev if e["n"].startswith("hmk_select_queries")]
    res = [e for e in ev if e["n"].startswith("hmk_p1_resolve_kernel")]
    p1_lo, p1_hi = sel[0]["t0"], res[-1]["t1"]
    streams = {}
    for e in ev:
        streams.setdefault(e["s"], []).append(e)
    main = res[-1]["s"]
    per_stream = {}
    for s, es in streams.items():
        inside = [e for e in es if e["t1"] > p1_lo and e["t0"] < p1_hi]
        if not inside:
            continue
        busy = union_len([(e["t0"], e["t1"]) for e in inside], p1_lo, p1_hi)
        names = {}
        for e in inside:
            names[e["n"]] = names.get(e["n"], 0) + 1
        per_stream[str(s)] = {"role": "main" if s == main else None, "activities": len(inside), "busy_us": round(busy, 1),
                              "idle_us": round(p1_hi - p1_lo - busy, 1),
                              "top": dict(sorted(names.items(), key=lambda kv: -kv[1])[:12])}

    searches = [e for e in ev if SEARCH.search(e["n"]) and p1_lo <= e["t0"] <= p1_hi]
    count = {}
    for e in searches:
        count[e["s"]] = count.get(e["s"], 0) + 1
    partner = max(count, key=count.get)
    per_stream[str(partner)]["role"] = "partner" + ("+main" if partner == main else "")
    ps = [e for e in searches if e["s"] == partner]
    gaps, between, pure, between_names = [], [], [], {}
    for a, b in zip(ps, ps[1:]):
        g = b["t0"] - a["t1"]
        mid = [e for e in streams[partner] if e["t0"] >= a["t1"] and e["t1"] <= b["t0"]]
        busy = union_len([(e["t0"], e["t1"]) for e in mid])
        for e in mid:
            r = between_names.setdefault(e["n"], {"count": 0, "total_us": 0.0})
            r["count"] += 1
            r["total_us"] = round(r["total_us"] + e["t1"] - e["t0"], 1)
        gaps.append(g); between.append(busy); pure.append(g - busy)

    p2 = [e for e in ev if e["n"].startswith("hmk_count_unassigned") and e["t0"] >= p1_hi]
    end = None
    if p2:
        mid = [e for e in ev if e["t1"] > p1_hi and e["t0"] < p2[0]["t0"]]
        names = {}
        for e in mid:
            k = f'{e["n"]} (stream {e["s"]})'
            names[k] = round(names.get(k, 0.0) + min(e["t1"], p2[0]["t0"]) - max(e["t0"], p1_hi), 1)
        end = {"wait_us": round(p2[0]["t0"] - p1_hi, 1), "ran_in_between_us": names}
    return {"launches": launches,
            "phase1": {"window_us": round(p1_hi - p1_lo, 1), "main_stream": main, "partner_stream": partner,
                       "partner_searches": len(searches), "partner_searches_on_partner_stream": len(ps),
                       "streams": per_stream},
            "partner_gaps": {"gap_us": dist(gaps), "ran_in_between_us": dist(between), "pure_gap_us": dist(pure),
                             "in_between_by_kernel": dict(sorted(between_names.items(), key=lambda kv: -kv[1]["total_us"])),
                             "per_batch_gap_us": [round(x, 1) for x in gaps],
                             "per_batch_pure_gap_us": [round(x, 1) for x in pure]},
            "end_of_phase1": end}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--tag", default="run")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("p1_timeline.py: no CUDA device")
    os.makedirs(args.out, exist_ok=True)
    d = synth.generate(args.n, 12, 12, seed=20260101)     # bench.py's workload
    T, X, K = synth.default_params(d["lengths"])
    M = synth.blosum62()
    ctx = hb.GreedyContext(0, profile=1)
    ctx.upload(d["residues"], d["offsets"], d["abundance"], M, T, X, 0, K)
    ctx.run()
    ctx.run()
    st, sec = ctx.stats(), ctx.section_ms()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.run()
        torch.cuda.synchronize()
    G = ctx.download()
    ctx.close()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    out = analyse(trace["traceEvents"] if isinstance(trace, dict) else trace)
    try:
        gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the numbers stay attributable only with the card beside them
        gpu = f"nvidia-smi failed: {e}"
    out = {"tag": args.tag, "gpu": gpu, "n": args.n, "digest": hb.result_digest(G.cluster_id, G.member_rank, G.result_order),
           "unprofiled": {"total_ms": round(st["total_ms"], 2), "phase1_ms": round(st["phase1_ms"], 2),
                          "phase2_ms": round(st["phase2_ms"], 2), "p1_batches": st["p1_batches"],
                          "sections_ms": {k: round(v, 2) for k, v in sec.items() if v}},
           **out}
    with open(os.path.join(args.out, f"p1_timeline_{args.tag}.json"), "w") as f:
        json.dump(out, f, indent=1)
    ph, g, e = out["phase1"], out["partner_gaps"], out["end_of_phase1"]
    print(json.dumps({"tag": args.tag, "gpu": gpu, "unprofiled": out["unprofiled"], "p1_window_us": ph["window_us"],
                      "partner_gap_sum_us": g["gap_us"].get("sum"), "pure_gap_sum_us": g["pure_gap_us"].get("sum"),
                      "in_between_sum_us": g["ran_in_between_us"].get("sum"), "end_wait_us": e and e["wait_us"],
                      "streams": {k: (v["role"], v["busy_us"], v["idle_us"]) for k, v in ph["streams"].items()}}), flush=True)


if __name__ == "__main__":
    main()
