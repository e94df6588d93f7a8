"""Cost of per-entry observation weights: the weighted sweep against the unweighted sweep on the same algorithm and against the
default (unweighted) path, alternating in one process.

    python tools/bench_weights.py [--window 1.0] [--reps 3] [--profile] [--out FILE (default profiles/r07_weights_b200.jsonl)]

Shapes: C2 (1M x 256, q = 16, 20 % missing), the C3 shard (1.25M x 1024, q = 32, 30 % missing) and sparse CSR 1M x 4096,
q = 16, 1 % observed.  Dense engines: "weighted" (weights log-uniform over three decades: the DMMA path), "dmma" (unweighted,
algo="dmma") and "default" (unweighted, algo="auto": the INT8 path where the shape allows it); sparse: "weighted" and
"default" (the CSR gathers either way).  Per engine and round: ms per sweep from CUDA events around back-to-back iterate_async
calls over a window of at least --window seconds, after warm-up.  --profile adds, in a separate pass, the per-kernel device
times of 5 sweeps of every engine from torch.profiler.  One JSON line per measurement on stdout, also appended to --out
('' for stdout only), with the GPU's name and power limit read in the same process.
"""
import argparse
import collections
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyvb_b200 import PlateEngine                         # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as ex:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % ex}


def dense(N, D, q, missing, seed, dev):
    """(X with NaN, S log-uniform over three decades)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    S = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        s = 10.0 ** (3.0 * torch.rand(n, D, generator=g, device=dev, dtype=torch.float64) - 1.5)
        x = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64) @ W.T
        x += torch.randn(n, D, generator=g, device=dev, dtype=torch.float64) / (4.0 * s).sqrt()
        x[torch.rand(n, D, generator=g, device=dev) < missing] = float("nan")
        X[lo:lo + n], S[lo:lo + n] = x, s
    return X, S


def sparse(N, D, dens, seed, dev):
    """(X, S): torch sparse CSR tensors with the same pattern."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    crow = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    cols = []
    for lo in range(0, N, 1 << 16):
        m = torch.rand(min(1 << 16, N - lo), D, generator=g, device=dev) < dens
        crow[lo + 1:lo + 1 + m.shape[0]] = m.sum(1)
        cols.append(m.nonzero(as_tuple=True)[1])
    crow = torch.cumsum(crow, 0)
    col = torch.cat(cols)
    val = torch.randn(col.numel(), generator=g, device=dev, dtype=torch.float64)
    s = 10.0 ** (3.0 * torch.rand(col.numel(), generator=g, device=dev, dtype=torch.float64) - 1.5)
    return (torch.sparse_csr_tensor(crow, col, val, size=(N, D)), torch.sparse_csr_tensor(crow, col, s, size=(N, D)))


def time_window(e, window):
    """ms per sweep over at least `window` seconds of back-to-back sweeps (the count from a 3-sweep probe)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def run(n):
        ev[0].record()
        for _ in range(n):
            e.iterate_async()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1])

    n = max(3, int(math.ceil(window * 1e3 / (run(3) / 3))))
    return run(n) / n, n


def kernel_times(e, sweeps=5):
    """Device time per sweep of every kernel name, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(sweeps):
            e.iterate_async()
        torch.cuda.synchronize()
    out = collections.defaultdict(float)
    for evt in prof.events():
        if evt.device_type == torch.autograd.DeviceType.CUDA:
            out[evt.name.replace("(anonymous namespace)::", "").split("(")[0][:90]] += evt.device_time / 1e3 / sweeps
    return {k: round(v, 4) for k, v in sorted(out.items(), key=lambda kv: -kv[1]) if v >= 0.002}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=1.0, help="seconds of sweeps per measurement")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="also report per-kernel times (separate pass)")
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "r07_weights_b200.jsonl"),
                    help="also append the JSON lines to this file ('' for none)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_weights.py measures on the GPU; there is none here")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    shapes = [("C2", lambda: dense(1_000_000, 256, 16, 0.2, 1, dev), 16, False),
              ("C3-shard", lambda: dense(1_250_000, 1024, 32, 0.3, 2, dev), 32, False),
              ("sparse-1M-4096-1%", lambda: sparse(1_000_000, 4096, 0.01, 3, dev), 16, True)]
    f = open(a.out, "a") if a.out else None

    def emit(rec):
        print(json.dumps(rec), flush=True)
        if f:
            f.write(json.dumps(rec) + "\n")
    try:
        for name, make, q, is_sparse in shapes:
            X, S = make()
            engines = {"weighted": PlateEngine(X, q, weights=S)}
            if not is_sparse:
                engines["dmma"] = PlateEngine(X, q, algo="dmma")
            engines["default"] = PlateEngine(X, q)
            del X, S
            for e in engines.values():
                e.init_random(seed=5)
                e.run(3)
                torch.cuda.synchronize()
            for rep in range(a.reps):
                for kind, e in engines.items():          # alternating: weighted, dmma, default, weighted, ...
                    ms, n = time_window(e, a.window)
                    e.check()
                    emit(dict(info, shape=name, N=e.N, D=e.D, q=e.q, engine=kind, rep=rep, sparse=e.sparse,
                              int8=bool(getattr(e, "use_i8", False)), sweeps=n, ms_per_sweep=round(ms, 4),
                              bound=float(e.elbo())))
            if a.profile:
                for kind, e in engines.items():
                    emit(dict(info, shape=name, engine=kind, kernel_ms_per_sweep=kernel_times(e)))
            del engines
            torch.cuda.empty_cache()
    finally:
        if f:
            f.close()


if __name__ == "__main__":
    main()
