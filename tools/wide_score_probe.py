"""Score-pass throughput from K = 256 to K = 4096 (the wide kernel: phases of 256 columns) on 1 M x 512 S-mix rows
generated on the device (2 GB, larger than L2), in two modes: argmin only (KMeans.predict, the encode chain, a
3-layer model's last layer) and argmin + the fp32 distance matrix (pairwise_distance_full, the last layer's match
and reassignment).  Then predict() of a PROD-shaped model ([128, 1280, 1280] / [128, 128, 256], synthetic centres)
on the same rows, per layer.  Prints one JSON object; `--out` also writes it.

    python tools/wide_score_probe.py [--rows 1048576] [--reps 20] [--out profiles/wide_score_probe.json]
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

DIM = 512


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def prod_predict_layers(x, reps):
    """The three levels of HierarchicalRQKMeans._predict_chain for a [128, 1280, 1280] / [128, 128, 256] model, each
    timed on its own (CUDA events, after warm-up): layer 0 argmin + residual, the recursive middle layer (128
    blocks of 128 centres) + residual, the last layer's plain argmin over 2 x 1280 candidates."""
    from generative_ranking_recommender_b200.hierarchical_rq_kmeans import HierarchicalRQKMeans, HierarchicalRQKMeansConfig
    dev = x.device
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    n = len(x)
    c0 = x[torch.randint(0, n, (128,), device=dev, generator=g)].contiguous()
    unit = lambda t: (t / t.norm(dim=1, keepdim=True)).contiguous()
    c_mid = unit(torch.randn((128 * 128, DIM), device=dev, generator=g))
    c_last = unit(torch.randn((2560, DIM), device=dev, generator=g))
    cfg = HierarchicalRQKMeansConfig(layer_clusters=[128, 1280, 1280], need_clusters=[128, 128, 256], embedding_dim=DIM,
                                     group_dims=[DIM], hierarchical_weights=[[1.0]] * 3)
    m = HierarchicalRQKMeans(cfg, device=dev)
    m.cluster_centers_list, m.is_trained = [c0, c_mid, c_last], True
    state = {}

    def l0():
        state["ids0"] = engine.score_pass(x, c0, argmin=True).argmin
        state["r0"] = engine.residual_normalise(x, state["ids0"], c0, [DIM])

    def l1():
        prev = state["ids0"].long()
        order = torch.argsort(prev, stable=True)
        counts = torch.bincount(prev, minlength=128).cpu().tolist()
        ids = torch.empty(n, dtype=torch.int32, device=dev)
        start = 0
        for i in range(128):
            rows = order[start:start + counts[i]]
            start += counts[i]
            if counts[i]:
                ids[rows] = engine.score_pass(engine.gather_rows(state["r0"], rows),
                                              c_mid[i * 128:(i + 1) * 128].contiguous(), argmin=True).argmin
        state["r1"] = engine.residual_normalise(state["r0"], ids, c_mid, [DIM])

    def l2():
        engine.score_pass(state["r1"], c_last, argmin=True)

    out = {"layer0_ms": timed(l0, reps), "layer1_ms": timed(l1, max(3, reps // 4)), "layer2_ms": timed(l2, reps)}
    out["whole_predict_chain_ms"] = timed(lambda: m._predict_chain(x), 3, warmup=1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--ks", default="256,512,1280,2560,4096")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    n = args.rows
    x = bench.synth_device("mix", n, dev)
    peak = bench.tf32_peak(dev)
    res = {"card": card(), "rows": n, "dim": DIM, "tf32_peak_tflops": round(peak, 1), "score_pass": []}
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    for k in [int(v) for v in args.ks.split(",")]:
        c = x[torch.randint(0, n, (k,), device=dev, generator=g)].contiguous()
        kc = (k + 15) // 16 * 16                          # MMA N summed over the phases
        bound_ms = 6.0 * n * k * DIM / (peak * 1e12) * 1e3
        row = {"k": k, "bound_ms": round(bound_ms, 3)}
        for mode, kw in (("argmin", {}), ("argmin_dist", {"dist": True})):
            ms = timed(lambda: engine.score_pass(x, c, argmin=True, **kw), args.reps)
            row[f"{mode}_ms"] = round(ms, 3)
            row[f"{mode}_issued_tflops"] = round(6.0 * n * kc * DIM / (ms * 1e-3) / 1e12, 1)
            row[f"{mode}_of_bound"] = round(bound_ms / ms, 3)
        torch.cuda.empty_cache()
        res["score_pass"].append(row)
        print(json.dumps(row), flush=True)
    res["prod_predict_1m"] = {k: round(v, 3) for k, v in prod_predict_layers(x, args.reps).items()}
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
