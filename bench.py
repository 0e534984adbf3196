#!/usr/bin/env python
"""bench.py - RQ-KMeans vectors/sec per iteration (512-d, [128,128,256]) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows R] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): 1M x 512 fp32 synthetic vectors per GPU (weak scaling: the fit is
ONE balanced K-Means over all ranks' rows, sharded row-wise; per iteration only the K x 512 sums,
K counts and the auction's threshold histograms cross NVLink).  A step = one `fit_by_min_loss`
iteration of the reference (balancekmeans/__init__.py:304-362): fused score pass, balanced auction,
centroid update, loss/shift read-back; steps cycle over the three levels (K = 128 on X, 128 and 256 on
the normalised residuals).  value = rows of all ranks x steps / time (CUDA events, max over ranks).

Extra keys: `e2e` = the same metric through HierarchicalRQKMeans.train() on HOST arrays (H2D of X and
D2H of the ids inside the timed region); `roofline` = the auction's streaming pass kernels (one read of the K x N
fp16 score matrix per launch) against the measured HBM copy bandwidth; `cpu_baseline` = the CPU oracle
port of the reference (all host threads) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CLUSTERS = [128, 128, 256]
DIM = 512
METRIC = "RQ-KMeans vectors/sec per iteration (512-d, [128,128,256])"
UNIT = "vectors/s"


# --------------------------------------------------------------------------------------------
def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md's clocks line).  The timed region of
    a default run is ~0.1 s, shorter than nvidia-smi's start-up, so the sampler reads NVML directly (the same
    counters nvidia-smi prints) every 2 ms on a host thread; nvidia-smi -lms is the fallback without pynvml.
    Only samples taken between mark_begin() and mark_end() count."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        self.index = index
        self.samples = []          # (time, sm_mhz, reasons bitmask or set)
        self.max_mhz = None
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.t0 = self.t1 = None
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.source = "nvml"

            def loop():
                while not self.stop_flag:
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        try:
                            bits = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        except Exception:
                            bits = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.samples.append((time.perf_counter(), mhz, bits))
                    except Exception:
                        pass
                    time.sleep(0.002)

            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"

            def read():
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for line in self.proc.stdout:
                    f = [x.strip() for x in line.split(",")]
                    try:
                        mhz, self.max_mhz = float(f[0]), float(f[1])
                    except (ValueError, IndexError):
                        continue
                    bits = sum(self.REASONS[n] for n, v in zip(names, f[2:6]) if v.lower().startswith("active"))
                    self.samples.append((time.perf_counter(), mhz, bits))

            self.thread = threading.Thread(target=read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread:
            self.thread.join(timeout=2)
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        inside = [x for x in self.samples if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or x[0])]
        mhz = sorted(x[1] for x in inside)
        bits = 0
        for x in inside:
            bits |= x[2]
        reasons = sorted(n for n, b in self.REASONS.items() if bits & b)
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(mhz), "source": self.source}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


# --------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md section 8d).  S-mix is the primary one (song-like: 1024 modes, row norms ~1.1),
# S-iso (no structure) the stress case.  Device-side generation (throughput runs); the CPU arm uses the same formulas.
def synth_device(kind, n, dev, rank=0, chunk=1 << 20):
    import math
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + 1000003 * rank)
    x = torch.empty((n, DIM), dtype=torch.float32, device=dev)
    if kind == "iso":
        for i in range(0, n, chunk):
            m = min(chunk, n - i)
            x[i:i + m] = torch.randn((m, DIM), device=dev, generator=g)
        return x
    gc = torch.Generator(device=dev)
    gc.manual_seed(1234)                                       # the mode centres are the same on every rank
    c = torch.randn((1024, DIM), device=dev, generator=gc)
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        j = torch.randint(0, 1024, (m,), device=dev, generator=g)
        x[i:i + m] = (c[j] + 0.5 * torch.randn((m, DIM), device=dev, generator=g)) * (1.0 / math.sqrt(DIM))
    return x


def synth_host(kind, n, seed=1234):
    import numpy as np
    rng = np.random.default_rng(seed)
    if kind == "iso":
        return rng.standard_normal((n, DIM), dtype=np.float32)
    c = rng.standard_normal((1024, DIM), dtype=np.float32)
    j = rng.integers(0, 1024, n)
    return ((c[j] + np.float32(0.5) * rng.standard_normal((n, DIM), dtype=np.float32)) / np.float32(np.sqrt(DIM))).astype(np.float32)


def composite_bytes(n, k, rounds_executed):
    """SURVEY.md 8(d): algorithmic bytes of ONE fit iteration = (8*D + 2*K + 2*K*R) per vector: X read by the score
    pass and by the centroid accumulate, the fp16 scores written once, and one read of them per auction round."""
    return float(n) * (8 * DIM + 2 * k + 2 * k * rounds_executed)


# --------------------------------------------------------------------------------------------
class CpuWorkload:
    """The CPU arm: the oracle port of the reference (C/OpenMP auction + numpy) on a bounded S-mix sample of the
    workload, built exactly like the GPU arm's (level inputs prepared once, untimed; a step = ONE fit iteration of
    balancekmeans/__init__.py:304-362 at level step % 3).  N % K != 0 as in the full workload: the reference's
    1002-round regime, every round simulated."""

    def __init__(self, rows, kind="mix", seed=1234):
        import numpy as np
        from oracle import rqk_oracle as O
        O.set_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: use the box's cores anyway
        self.O, self.np, self.rows, self.kind = O, np, rows, kind
        rng = np.random.default_rng(seed)
        cur = synth_host(kind, rows, seed)
        self.levels = []
        for lvl, k in enumerate(CLUSTERS):
            c = cur[rng.choice(rows, k, replace=False)].copy()
            self.levels.append([k, cur, c])
            if lvl < len(CLUSTERS) - 1:
                c1, ids, _ = self.iterate(cur, c, k)
                self.levels[-1][2] = c1
                cur = O.residual_normalised(cur, ids, c1, [DIM])
        self.rounds, self.seconds = [], []

    def iterate(self, cur, c, k):
        O, np = self.O, self.np
        d = O.pairwise_distance_full(cur, c, 100000)                     # :308
        res = O.auction_lap_half(-d)                                     # :310
        c1 = O.update_centers(cur, res.assignment, c)                    # :314-324
        d2 = O.pairwise_distance_full(cur, c1, 100000)                   # :327
        ids = np.argmin(d2, axis=1)
        cnt = np.bincount(ids, minlength=k)                              # :328-329
        O.overflow_loss(cnt, 1 << 30)                                    # :333-336
        O.center_shift(c1, c)                                            # :343-346
        return c1, ids, res.rounds

    def step(self, i):
        lvl = i % len(self.levels)
        k, cur, c = self.levels[lvl]
        t0 = time.perf_counter()
        c1, _, r = self.iterate(cur, c, k)
        dt = time.perf_counter() - t0
        self.levels[lvl][2] = c1
        self.rounds.append(r)
        self.seconds.append(dt)
        return dt

    def record(self, first=0):
        sec, rounds = self.seconds[first:], self.rounds[first:]
        total = sum(sec)
        return {"value": self.rows * len(sec) / total, "unit": UNIT, "cores": self.O.num_threads(), "kind": "port",
                "sample": f"{self.rows} x {DIM} fp32 S-{self.kind} rows, {len(sec)} fit iterations (levels cycled over "
                          f"{CLUSTERS}), auction rounds {sorted(set(rounds))}, {total:.1f} s CPU",
                "sample_rows": self.rows, "seconds_per_step": [round(t, 2) for t in sec]}


def cpu_baseline_port(sample_rows):
    w = CpuWorkload(sample_rows)
    for i in range(len(CLUSTERS)):
        w.step(i)
    return w.record()


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; the reference itself is Python + torch CPU
    and does not exist on the GPU box) on the box's host cores, same metric/unit/config and the same step
    definition as the GPU arm; exactly --steps steps are timed after --warmup."""
    rank = _env_int("RANK", 0)
    if rank != 0:
        return
    rows = args.cpu_rows
    w = CpuWorkload(rows)
    dt = w.step(0) if args.warmup > 0 else None
    if dt is not None and dt * (args.warmup + args.steps) * 1.4 > 300 and rows > 4096:
        rows = max(4096, rows // 2 // 128 * 128 + 64)          # a slow box: keep the step COUNT, shrink the sample
        w = CpuWorkload(rows)
        w.step(0)
    for i in range(1, args.warmup):
        w.step(i)
    first = len(w.seconds)
    for i in range(args.steps):
        w.step(args.warmup + i)
    base = w.record(first)
    v = base["value"]
    cfg = workload_config(args, args.gpus)
    cfg["sample_rows"] = rows
    cfg["sample"] = "each step runs on a bounded sample of the workload (cpu_baseline.sample), not on all its rows"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * rows / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32 distance / fp16 auction (CPU)", "data": "synthetic",
            "config": cfg, "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"{args.rows} x {DIM} fp32 rows per GPU (S-mix: 1024-mode mixture, SURVEY.md 8d), 3-level RQ-KMeans "
                        f"{CLUSTERS} balanced fit iteration (score pass + auction + centroid update), levels cycled",
            "rows_per_gpu": args.rows, "rows_total": args.rows * world, "dim": DIM, "codebook": CLUSTERS,
            "input": "S-mix", "sharding": f"rows x{world}",
            "l2": "inputs (2 GB X + 256/512 MB scores per level) exceed the 126 MB L2"}


# --------------------------------------------------------------------------------------------
class Workload:
    """The three level inputs of one synthetic data set, resident in HBM, and the timed step over them."""

    def __init__(self, kind, n, world, rank, dev, shard, engine, KMeans):
        import numpy as np
        import torch
        self.n, self.n_global, self.shard, self.engine = n, n * world, shard, engine
        self.x0 = synth_device(kind, n, dev, rank)
        np.random.seed(42)
        torch.manual_seed(42)
        self.levels = []
        cur = self.x0
        for lvl, k in enumerate(CLUSTERS):
            km = KMeans(n_clusters=k, device=dev, balanced=True, shard=shard)
            km.cluster_centers = km.initialize(cur)
            self.levels.append((km, cur))
            if lvl < len(CLUSTERS) - 1:
                km._iterate(cur, self.n_global)                  # one real iteration to get sensible centroids
                ids = engine.score_pass(cur, km.cluster_centers, argmin=True).argmin
                cur = engine.residual_normalise(cur, ids, km.cluster_centers, [DIM])
        self.bufs = [None] * len(self.levels)
        self.stats = []
        self.last = None

    def step(self, i):
        import torch
        lvl = i % len(self.levels)
        km, xl = self.levels[lvl]
        score, assign, stats, shift = km._iterate(xl, self.n_global, self.bufs[lvl])
        self.last = (lvl, score, assign, shift)
        self.bufs[lvl] = score.scores_t
        c = score.counts.to(torch.int64)
        if self.shard is not None:
            self.shard.all_reduce(c, "sum")
        c.cpu()                                              # loss read-back of the fit loop (:333-341)
        if stats is not None:
            self.stats.append((CLUSTERS[lvl], stats))

    def timed(self, warmup, steps, barrier, sampler=None):
        import torch
        for i in range(warmup):
            self.step(i)
        self.stats.clear()
        barrier()
        if sampler:
            sampler.mark_begin()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            self.step(warmup + i)
        ev1.record()
        barrier()
        if sampler:
            sampler.mark_end()
        return ev0.elapsed_time(ev1)

    def composite(self, ms, peak, how):
        """Per-iteration composite roofline (SURVEY.md 8d): sum over the timed steps of (8D + 2K + 2K*R) * N bytes
        / time, with R = bidding rounds actually EXECUTED (the reference's count is 1002 in this regime; the exact
        fast-forward skips the rest).  Sharded runs: all ranks' bytes, against all ranks' peak."""
        r_exec = [st.passes - st.cold_passes for _, st in self.stats]
        by = [composite_bytes(self.n_global, k, r) for (k, _), r in zip(self.stats, r_exec)]
        world = self.n_global // self.n
        ach = sum(by) / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak * world, "unit": "GB/s", "frac": ach / (peak * world),
                "bytes_per_vector": "8*D + 2*K + 2*K*R (SURVEY.md 8d), R = bidding rounds executed",
                "rounds_executed_per_step": r_exec, "passes_per_step": [st.passes for _, st in self.stats],
                "list_rounds_per_step": [st.list_passes for _, st in self.stats],
                "window_misses_per_step": [st.window_misses for _, st in self.stats],
                "reference_rounds_per_step": [st.rounds for _, st in self.stats], "peak_source": how}

    def dump(self, out_dir, max_rows=1 << 20, score_rows=4096):
        """Writes what the last timed step returned to its caller as DIR/<name>.npy, so that two builds can be
        compared output for output: the updated centres, the balanced assignment, the argmin and counts of the
        step's input centres, the centre shift, and the fp16 scores of `score_rows` rows.  Per-row outputs of more
        than `max_rows` rows are a fixed sample (rows.npy holds its row indices); everything stays under 64 MB."""
        import numpy as np
        import torch
        lvl, score, assign, shift = self.last
        km = self.levels[lvl][0]
        n = self.n
        rows = np.arange(n) if n <= max_rows else np.sort(np.random.default_rng(0).choice(n, max_rows, replace=False))
        out = {"centers": km.cluster_centers.cpu().numpy().astype(np.float32),
               "assignment": assign.cpu().numpy()[rows].astype(np.float64),
               "argmin": score.argmin.cpu().numpy()[rows].astype(np.float64),
               "counts": score.counts.cpu().numpy().astype(np.float64),
               "shift": np.array([shift], dtype=np.float64)}
        if n > max_rows:
            out["rows"] = rows.astype(np.float64)
        if score.scores_t is not None:
            cols = np.sort(np.random.default_rng(1).choice(n, min(n, score_rows), replace=False))
            s = score.scores_t.index_select(1, torch.from_numpy(cols).to(score.scores_t.device))
            out["scores"] = s.t().float().cpu().numpy()
        os.makedirs(out_dir, exist_ok=True)
        for name, a in out.items():
            np.save(os.path.join(out_dir, f"{name}.npy"), a)


def fit_10m_record(dev, engine, KMeans, peak, how, rows=10000000, iters=3):
    """North-star size on ONE GPU: 10 M x 512 S-mix rows, K = 128 on the raw rows and K = 256 on their normalised
    level-0 residual; `iters` timed fit iterations each after one warm-up iteration (generated on the device)."""
    import numpy as np
    import torch
    out = {"rows": rows, "input": "S-mix (device-generated)", "iterations_timed": iters, "levels": []}
    x = synth_device("mix", rows, dev, 0)
    np.random.seed(42)
    torch.manual_seed(42)
    for k, what in ((128, "level 0 (raw rows)"), (256, "level 2 shape (normalised residual)")):
        km = KMeans(n_clusters=k, device=dev, balanced=True)
        km.cluster_centers = km.initialize(x)
        sc, _, _, _ = km._iterate(x, rows)
        buf = sc.scores_t
        stats = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            sc, _, st, _ = km._iterate(x, rows, buf)
            sc.counts.cpu()
            stats.append(st)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        r_exec = [st.passes - st.cold_passes for st in stats]
        by = sum(composite_bytes(rows, k, r) for r in r_exec)
        ach = by / (ms * 1e-3) / 1e9
        out["levels"].append({"k": k, "what": what, "ms_per_iteration": ms / iters, "vectors_per_s": rows * iters / (ms * 1e-3),
                              "rounds_executed": r_exec, "reference_rounds": [st.rounds for st in stats],
                              "passes": [st.passes for st in stats], "window_misses": [st.window_misses for st in stats],
                              "list_rounds": [st.list_passes for st in stats],
                              "composite": {"achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}})
        if k == 128:
            ids = engine.score_pass(x, km.cluster_centers, argmin=True).argmin
            engine.residual_normalise(x, ids, km.cluster_centers, [DIM], out=x)
        del buf, sc
    out["peak_source"] = how
    del x
    engine.SCRATCH.clear()
    torch.cuda.empty_cache()
    return out


def tf32_peak(dev):
    """Dense TF32 tensor throughput of this GPU (cuBLAS, 8192^3), the yardstick of the 3xTF32 score pass."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn((8192, 8192), device=dev)
        b = torch.randn((8192, 8192), device=dev)
        for _ in range(2):
            a @ b
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            a @ b
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1000000, help="rows per GPU")
    ap.add_argument("--cpu-rows", type=int, default=20032, help="rows of the CPU baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-10m", action="store_true", help="skip the 10 M-row single-GPU record")
    ap.add_argument("--no-extras", action="store_true", help="only the headline step timing (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the GPU step; it does not apply to --impl reference")
        return run_reference(args)
    if args.no_extras:
        args.no_e2e = args.no_cpu = args.no_10m = True

    import numpy as np
    import torch
    import torch.distributed as dist

    from generative_ranking_recommender_b200 import HierarchicalRQKMeans, HierarchicalRQKMeansConfig, engine
    from generative_ranking_recommender_b200.balancekmeans import KMeans

    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    shard = engine.ShardGroup() if world > 1 else None
    n = args.rows
    n_global = n * world
    peak, how = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- headline: S-mix level inputs resident in HBM before anything is timed ----
    wl = Workload("mix", n, world, rank, dev, shard, engine, KMeans)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                                      # before the warm-up: it is streaming when the timed region starts
    ms = wl.timed(args.warmup, args.steps, barrier, sampler if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        wl.dump(args.dump_outputs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = n_global * args.steps / (ms / 1e3)
    composite = wl.composite(ms, peak, how)
    passes = [st.passes for _, st in wl.stats]
    rounds = [st.rounds for _, st in wl.stats]

    # launches of our kernels inside the timed region: per step score pass (pad, minmax, split, tc) = 4,
    # auction init (memset + init) 2 + ROUND_LAUNCHES per enqueued round (rounds are enqueued two at a time, one
    # batch ahead of the host's look at the state) + finalize 1, centroid update 8
    ROUND_LAUNCHES = 5 if world == 1 else 7

    def auction_launches(st):
        rounds_ = st.passes - st.cold_passes
        return ROUND_LAUNCHES * 2 * (-(-rounds_ // 2) + 1)
    gpu_launches = int(sum(4 + 2 + auction_launches(st) + 1 + 8 for _, st in wl.stats))

    # ---- second record: the same step on S-iso (no structure; narrower windows, fewer survivors) ----
    s_iso = None
    if not args.no_extras:
        wl_iso = Workload("iso", n, world, rank, dev, shard, engine, KMeans)
        ms_iso = wl_iso.timed(args.warmup, args.steps, barrier)
        t = torch.tensor([ms_iso], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_iso = float(t.item())
        s_iso = {"input": "S-iso", "value": n_global * args.steps / (ms_iso / 1e3), "unit": UNIT,
                 "ms_per_step": ms_iso / args.steps, "composite": wl_iso.composite(ms_iso, peak, how)}
        del wl_iso
        torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel: the auction's streaming HIST pass at level 0 (K=128) ----
    # It reads the K x N fp16 score matrix exactly once: 2*K bytes per vector (SURVEY.md 8d).  The bidding half of
    # a round replays the HIST pass's survivor lists (L2-resident) and is reported beside it.
    roofline = None
    if rank == 0:
        km, xl = wl.levels[0]
        sc = engine.score_pass(xl, km.cluster_centers, scores=True, argmin=False)
        sess = engine.AuctionSession(sc.scores_t, n, n)
        sess.init(sc.minmax)
        # The kernels are launched one by one through the C-ABI step entry point in the flow rqk_auction chains
        # (which | 16): HIST dumps per CTA, the merge kernel (one CTA per worker) sums the dumps, resolves the thresholds
        # and takes the tie prefix, the bidding kernel's last CTA resolves the round.  A cycle runs whichever of them
        # the device-side state machine lets act; the others return at once.
        FLOW = 16
        t_hist, t_bid, t_merge = [], [], []
        prev = sess.poll()
        for cyc in range(60):
            sess.do_pass(1 | FLOW)                           # window sampling (early-exits unless needed), untimed
            e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
            e0.record()
            sess.do_pass(2 | FLOW)                           # streaming HIST kernel
            e1.record()
            sess.do_pass(8 | FLOW)                           # merge + resolve + tie prefix
            e2.record()
            sess.do_pass(4 | FLOW)                           # bid-list replay (+ the S-scanning fallback, which returns at once)
            e3.record()
            cur = sess.poll()
            if cur.done:
                break
            if cyc >= 4:                                     # past the cold start
                if cur.cold_passes > prev.cold_passes:
                    t_hist.append(e0.elapsed_time(e1))
                    t_merge.append(e1.elapsed_time(e2))
                if cur.passes - cur.cold_passes > prev.passes - prev.cold_passes:
                    t_bid.append(e2.elapsed_time(e3))
            prev = cur
        k0 = CLUSTERS[0]
        alg_bytes = 2.0 * k0 * n

        def line(name, ts):
            if not ts:
                return None
            t = sum(ts) / len(ts)
            ach = alg_bytes / (t * 1e-3) / 1e9
            return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": recorded_traffic(name.split("(")[0].strip()), "algorithmic_bytes_per_launch": alg_bytes,
                    "ms_per_launch": t, "launches_timed": len(ts), "peak_source": how}

        roofline = line("auction_hist_kernel (threshold select, K=128)", t_hist)
        if roofline is not None:
            if t_bid:
                roofline["other_kernel"] = {
                    "kernel": "auction_bidlist_kernel (bids replayed from the HIST pass's survivor lists, K=128)",
                    "ms_per_launch": sum(t_bid) / len(t_bid), "launches_timed": len(t_bid),
                    "note": "not a stream over S: reads ~2 % of it as L2-resident lists plus cost/owner of every job; "
                            "timed together with the early-exiting S-scanning fallback kernel"}
            if t_merge:
                roofline["merge_resolve_kernel"] = {
                    "kernel": "auction_merge_resolve_kernel (per-worker sum of the CTA histograms, threshold, tie prefix)",
                    "ms_per_launch": sum(t_merge) / len(t_merge), "launches_timed": len(t_merge)}
            roofline["composite"] = composite                # the per-ITERATION figure of SURVEY.md 8(d)
            try:
                tf = tf32_peak(dev)
                roofline["tensor"] = {"tf32_tflops_measured": tf, "how": "torch.matmul tf32 8192^3, best of 5 (cuBLAS)",
                                      "note": "the 3xTF32 score pass issues 3 MMAs per product: its floor is "
                                              "3*2*K*(D+2)*N / this"}
            except Exception as e:
                roofline["tensor"] = {"error": repr(e)}
        del sess, sc

    # ---- encode (the ids train() emits / predict() returns), rows resident in HBM ----
    # fused = the single tcgen05 kernel over all levels (csrc/encode_fused.cu); chain = score pass + residual per level
    encode = None
    if rank == 0 and not args.no_extras:
        try:
            cs = [km.cluster_centers for km, _ in wl.levels]

            def time_encode(fused):
                for _ in range(2):
                    engine.encode(wl.x0, cs, CLUSTERS, [DIM], mode=0, fused=fused)
                ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ee0.record()
                for _ in range(3):
                    engine.encode(wl.x0, cs, CLUSTERS, [DIM], mode=0, fused=fused)
                ee1.record()
                torch.cuda.synchronize()
                return ee0.elapsed_time(ee1) / 3
            t_enc = time_encode(True)
            redo = engine.encode_reevaluated_rows(dev)
            t_chain = time_encode(False)
            tf = (roofline or {}).get("tensor", {}).get("tf32_tflops_measured")
            flops = 3.0 * 2.0 * sum(CLUSTERS) * DIM * n          # three TF32 MMAs per product
            encode = {"value": n / (t_enc / 1e3), "unit": "vectors/s", "rows": n, "ms": t_enc, "gpus": 1,
                      "what": "3-level ids of resident fp32 rows, one tcgen05 kernel over all levels "
                              "(rqk_encode_fused, mode 0): X read once, no residual in memory",
                      "rows_reevaluated_exactly": redo,
                      "level_chain_ms": t_chain, "level_chain_vectors_per_s": n / (t_chain / 1e3),
                      "tensor_bound": ({"tflops_3xtf32_issued": flops / (t_enc / 1e3) / 1e12, "peak_tf32_tflops": tf,
                                        "frac": flops / (t_enc / 1e3) / 1e12 / tf} if tf else None),
                      "hbm_bytes_per_vector": 4 * DIM + 4 * len(CLUSTERS)}
        except Exception as e:      # never lose the bench line over the side metric
            encode = {"error": repr(e)}

    # ---- end to end through the public API: host array in, ids out ----
    # Headline e2e: a PAGEABLE np.ndarray, as train_semantic_ids.py:152 passes it (np.vstack of the CSV rows);
    # `pinned` repeats it from page-locked memory.  H2D of X and D2H of the ids are inside the timed region.
    e2e = None
    if not args.no_e2e:
        x_np = wl.x0.cpu().numpy()                           # pageable
        del wl
        engine.SCRATCH.clear()
        torch.cuda.empty_cache()
        cfg = HierarchicalRQKMeansConfig(layer_clusters=CLUSTERS, need_clusters=CLUSTERS, embedding_dim=DIM,
                                         group_dims=[DIM], hierarchical_weights=[[1.0]] * 3, iter_limit=20)

        def run_train(x_host):
            np.random.seed(42)
            torch.manual_seed(42)
            model = HierarchicalRQKMeans(cfg, device=dev, shard=shard)
            barrier()
            t0 = time.perf_counter()
            out = model.train(x_host, resume=False)
            barrier()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            iters = sum(len(s) for s in model.fit_stats)
            ids_bytes = sum(t.numel() * t.element_size() for t in out["cluster_ids"])
            return {"value": n_global * iters / dt, "unit": UNIT,
                    "h2d_bytes_per_step": x_host.nbytes * world / max(iters, 1),
                    "d2h_bytes_per_step": ids_bytes * world / max(iters, 1), "seconds": dt, "iterations": iters,
                    "iterations_per_level": [len(s) for s in model.fit_stats]}

        run_train(np.ascontiguousarray(x_np[:65536]))        # warm-up: a small fit through the same API (allocator, streams)
        e2e = run_train(x_np)
        e2e["host_memory"] = "pageable np.ndarray"
        e2e["api"] = "HierarchicalRQKMeans.train(np.ndarray) -> cluster_ids (int64, host), iter_limit=20"
        xh = torch.empty((n, DIM), dtype=torch.float32, pin_memory=True)
        xh.copy_(torch.from_numpy(x_np))
        del x_np
        pinned = run_train(xh.numpy())
        e2e["pinned"] = {"value": pinned["value"], "seconds": pinned["seconds"], "host_memory": "page-locked"}
        del xh
    else:
        del wl
    engine.SCRATCH.clear()
    torch.cuda.empty_cache()

    fit_10m = None
    if rank == 0 and world == 1 and not args.no_10m:
        try:
            fit_10m = fit_10m_record(dev, engine, KMeans, peak, how)
        except Exception as e:
            fit_10m = {"error": repr(e)}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline_port(args.cpu_rows)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "3xTF32 distance (fp32 accumulate), fp16 auction, fp32 centroids",
                "data": "synthetic", "config": workload_config(args, world), "clocks": clocks,
                "gpu_launches": gpu_launches, "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu,
                "auction": {"passes_per_step": passes, "reference_rounds_per_step": rounds,
                            "rounds_executed_per_step": composite["rounds_executed_per_step"]},
                "s_iso": s_iso, "fit_10m": fit_10m, "encode": encode}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
