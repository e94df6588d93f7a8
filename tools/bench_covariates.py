"""Known row covariates (PlateEngine(..., covariates=C), q free + k known) against a covariate-free engine at the same q' = q + k:
sweep time, alternating the two in one process, and the kernels the covariates add.

    python tools/bench_covariates.py [--part time,kernels] [--window 1.0] [--reps 3]
                                     [--out FILE (default profiles/r09_covariates_b200.jsonl)]

Parts (comma-separated, default all):
  time      ms per sweep of both engines, alternating, --reps rounds over windows of at least --window s (CUDA events around
            back-to-back iterate_async calls, after warm-up), on C2 (1M x 256, 20 % missing, q = 12 + k = 4 against q = 16: the
            INT8 path) and the C3 shard (1.25M x 1024, 30 % missing, q = 28 + k = 4 against q = 32)
  kernels   the kernels of 10 sweeps of each engine under torch.profiler (a separate pass): per kernel name, calls and total
            device time per sweep -- known_condition_kernel, known_finish_kernel and the statistics' rebuilt partials among them
One JSON line per measurement on stdout, also appended to --out ('' for stdout only), with the GPU's name, power limit and
maximum SM clock read in the same process.
"""
import argparse
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_wrows import gpu_info  # noqa: E402

SHAPES = [("C2", 1_000_000, 256, 12, 4, 0.2), ("C3-shard", 1_250_000, 1024, 28, 4, 0.3)]


def data(N, D, q, k, missing, seed, dev):
    """(X with NaN, C): x_n = W z_n + B c_n + mu + noise of precision 4."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    f64 = torch.float64
    W = torch.randn(D, q, generator=g, device=dev, dtype=f64)
    B = torch.randn(D, k, generator=g, device=dev, dtype=f64)
    mu = torch.randn(D, generator=g, device=dev, dtype=f64)
    C = torch.randn(N, k, generator=g, device=dev, dtype=f64)
    X = torch.empty(N, D, dtype=f64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        x = torch.randn(n, q, generator=g, device=dev, dtype=f64) @ W.T + C[lo:lo + n] @ B.T + mu
        x += 0.5 * torch.randn(n, D, generator=g, device=dev, dtype=f64)
        x[torch.rand(n, D, generator=g, device=dev) < missing] = float("nan")
        X[lo:lo + n] = x
    return X, C


def engines(name, N, D, q, k, missing, dev):
    from pyvb_b200 import PlateEngine
    X, C = data(N, D, q, k, missing, 7, dev)
    cov = PlateEngine(X, q, covariates=C)
    base = PlateEngine(X, q + k)
    for e in (cov, base):
        e.init_random(seed=3)
    return {"covariates": cov, "plain": base}


def time_sweeps(e, window):
    import torch
    for _ in range(3):
        e.iterate_async()
    torch.cuda.synchronize()
    n, t = 5, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            e.iterate_async()
        b.record()
        b.synchronize()
        t = a.elapsed_time(b) / 1e3
        if t >= window:
            return 1e3 * t / n, n
        n = max(n * 2, int(n * 1.2 * window / max(t, 1e-6)))


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def part_time(args, info, dev):
    for name, N, D, q, k, missing in SHAPES:
        es = engines(name, N, D, q, k, missing, dev)
        for r in range(args.reps):
            for mode, e in es.items():
                ms, n = time_sweeps(e, args.window)
                emit(dict(info, part="time", shape=name, N=N, D=D, q=q, k=k, qt=q + k, mode=mode, round=r, ms_per_sweep=ms,
                          sweeps=n, i8=bool(e.use_i8), i8_fallbacks=list(e.i8_fallbacks())), args.out)
        del es


def part_kernels(args, info, dev):
    import torch
    from torch.profiler import ProfilerActivity, profile
    for name, N, D, q, k, missing in SHAPES:
        es = engines(name, N, D, q, k, missing, dev)
        for mode, e in es.items():
            for _ in range(3):
                e.iterate_async()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(10):
                    e.iterate_async()
                torch.cuda.synchronize()
            per = collections.defaultdict(lambda: [0, 0.0])
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    per[ev.name][0] += 1
                    per[ev.name][1] += ev.device_time_total
            kernels = {n: {"calls_per_sweep": c / 10, "us_per_sweep": t / 10} for n, (c, t) in
                       sorted(per.items(), key=lambda kv: -kv[1][1])}
            emit(dict(info, part="kernels", shape=name, q=q, k=k, mode=mode, kernels=kernels), args.out)
        del es


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="time,kernels")
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_covariates_b200.jsonl"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_covariates: no CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    info = gpu_info()
    parts = args.part.split(",")
    if "time" in parts:
        part_time(args, info, dev)
    if "kernels" in parts:
        part_kernels(args, info, dev)


if __name__ == "__main__":
    main()
