"""Fit iterations at K = 256 (the reference point), 384 and 512 on 1 M x 512 S-mix rows generated on the device
(2 GB, larger than L2).  Per K: milliseconds per iteration split into score pass, auction and centroid update (CUDA
events around each stage, after a warm-up iteration), the auction's rounds / passes / window misses / list passes
per iteration, and the HIST kernel alone: the driver's HIST launch (`rqk_auction_pass` with which = 2 | 16) repeated
on one auction state, right after its window sampling.  The card's name and power limit are read in the same run.
Prints one JSON object; `--out` also writes it.

    python tools/wide_fit_probe.py [--rows 1000000] [--iters 3] [--hist-reps 50] [--out profiles/wide_fit_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from generative_ranking_recommender_b200 import engine  # noqa: E402


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def stage_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def hist_launch_us(scores_t, n, minmax, reps):
    """One auction state after init + window sampling; its HIST pass launched `reps` times (the pass leaves the state
    unchanged: the merge kernel that resolves it is not launched)."""
    sess = engine.AuctionSession(scores_t, n, n)
    sess.init(minmax)
    sess.do_pass(1 | 16)
    for _ in range(3):
        sess.do_pass(2 | 16)
    torch.cuda.synchronize()
    ms, _ = stage_ms(lambda: [sess.do_pass(2 | 16) for _ in range(reps)])
    return 1000.0 * ms / reps


def probe_k(x, k, iters, hist_reps):
    n = len(x)
    g = torch.Generator(device=x.device)
    g.manual_seed(k)
    c = x[torch.randperm(n, device=x.device, generator=g)[:k]].contiguous()
    rows = []
    for it in range(iters + 1):                                   # iteration 0 is the warm-up
        t_s, r = stage_ms(lambda: engine.score_pass(x, c, scores=True, argmin=True, counts=True))
        t_a, (a, st) = stage_ms(lambda: engine.auction(r.scores_t, n, r.minmax))
        def update():
            sums, counts = engine.centroid_accumulate(x, a, k)
            engine.centroid_finalize(sums, counts, c)
        t_u, _ = stage_ms(update)
        if it > 0:
            rows.append(dict(score_ms=t_s, auction_ms=t_a, update_ms=t_u, rounds=st.rounds, passes=st.passes,
                             window_misses=st.window_misses, list_passes=st.list_passes))
    hist_us = hist_launch_us(r.scores_t, n, r.minmax, hist_reps)
    mean = lambda key: sum(q[key] for q in rows) / len(rows)
    return dict(k=k, ms_per_iteration=mean("score_ms") + mean("auction_ms") + mean("update_ms"),
                score_ms=mean("score_ms"), auction_ms=mean("auction_ms"), update_ms=mean("update_ms"),
                hist_us_per_launch=hist_us, hist_bytes_per_launch=2 * k * n,
                per_iteration=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1000000)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--hist-reps", type=int, default=50)
    ap.add_argument("--ks", default="256,384,512")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wide_fit_probe: needs a CUDA device")
    dev = torch.device("cuda:0")
    x = bench.synth_device("mix", args.rows, dev)
    res = dict(card=card(), rows=args.rows, dim=bench.DIM, data="S-mix, generated on the device",
               iters=args.iters, results=[probe_k(x, int(k), args.iters, args.hist_reps) for k in args.ks.split(",")])
    base = res["results"][0]
    for q in res["results"]:
        q["hist_vs_first_k"] = q["hist_us_per_launch"] / base["hist_us_per_launch"]
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
