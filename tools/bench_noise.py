"""Cost of per-dimension noise precisions: scalar against diagonal noise, alternating in one process, on three shapes.

    python tools/bench_noise.py [--sweeps 20] [--reps 3] [--out FILE]

Shapes: C2 (1M x 256, q = 16, 20 % missing: INT8 path), the C3 shard (1.25M x 1024, q = 32, 30 % missing: INT8 Z step, DMMA
statistics) and sparse CSR 1M x 4096, q = 16, 1 % observed.  Per shape and noise model: ms per sweep (CUDA events around
`sweeps` back-to-back iterate_async calls, after warm-up) and the second stage alone (the pyvb_global_f64 /
pyvb_global_nd_f64 call of a sweep, Mu + Alpha + Beta + bound, timed over 200 launches).  One JSON line per measurement on
stdout (and appended to --out), with the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyvb_b200 import PlateEngine                         # noqa: E402
from pyvb_b200._layout import OP_ALPHA, OP_BETA, OP_ELBO, OP_MU   # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as ex:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % ex}


def dense(N, D, q, missing, seed, dev):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    tau = torch.exp(torch.rand(D, generator=g, device=dev, dtype=torch.float64) * np.log(1e3))
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        x = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64) @ W.T
        x += torch.randn(n, D, generator=g, device=dev, dtype=torch.float64) / tau.sqrt()
        x[torch.rand(n, D, generator=g, device=dev) < missing] = float("nan")
        X[lo:lo + n] = x
    return X


def sparse(N, D, dens, seed, dev):
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
    return torch.sparse_csr_tensor(crow, col, val, size=(N, D))


def time_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_noise.py measures on the GPU; there is none here")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    shapes = [("C2", lambda: dense(1_000_000, 256, 16, 0.2, 1, dev), 16),
              ("C3-shard", lambda: dense(1_250_000, 1024, 32, 0.3, 2, dev), 32),
              ("sparse-1M-4096-1%", lambda: sparse(1_000_000, 4096, 0.01, 3, dev), 16)]
    ops = OP_MU | OP_ALPHA | OP_BETA | OP_ELBO
    f = open(a.out, "a") if a.out else None
    try:
        for name, make, q in shapes:
            X = make()
            engines = {noise: PlateEngine(X, q, noise=noise) for noise in ("scalar", "diagonal")}
            del X
            for e in engines.values():
                e.init_random(seed=5)
                e.run(3)
                e._global(ops)
                torch.cuda.synchronize()
            for rep in range(a.reps):
                for noise, e in engines.items():          # alternating: scalar, diagonal, scalar, ...
                    ms = time_ms(e.iterate_async, a.sweeps)
                    g_ms = time_ms(lambda: e._global(ops), 200)
                    e.check()
                    rec = dict(info, shape=name, N=e.N, D=e.D, q=e.q, noise=noise, rep=rep, sparse=e.sparse,
                               int8=bool(getattr(e, "use_i8", False)), ms_per_sweep=round(ms, 4),
                               second_stage_ms=round(g_ms, 4), i8_fallbacks=e.i8_fallbacks(),
                               bound=float(e.elbo()))
                    print(json.dumps(rec), flush=True)
                    if f:
                        f.write(json.dumps(rec) + "\n")
            del engines
            torch.cuda.empty_cache()
    finally:
        if f:
            f.close()


if __name__ == "__main__":
    main()
