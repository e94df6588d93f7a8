"""Row-wise against column-wise W posterior (PlateEngine(..., w_posterior="rows" | "columns")): sweep time, the W step alone and
convergence, alternating the two modes in one process.

    python tools/bench_wrows.py [--part time,wstep,converge,oracle] [--window 1.0] [--reps 3]
                                [--out FILE (default profiles/r08_wrows_b200.jsonl)]

Parts (comma-separated, default all):
  time      ms per sweep of both modes, alternating, --reps rounds over windows of at least --window s (CUDA events around
            back-to-back iterate_async calls, after warm-up), on C2 (1M x 256, q = 16, 20 % missing: the default INT8 path),
            the C3 shard (1.25M x 1024, q = 32, 30 % missing) and the C4 shape (400k x 512, q = 64, ARD, 30 % missing)
  wstep     the kernels of update_W alone under torch.profiler, 20 calls per mode on each shape (a separate pass):
            wupdate_kernel against wrows_assemble_kernel + the K2 kernel + wrows_finish_kernel
  converge  from the same seeded start (init_random) on C2-generated data and on a variant whose W_true has correlated columns
            of spread scales: sweeps until learn(tol=1e-3) would stop, sweeps until the bound's relative change falls below
            1e-7, and the largest principal angle between Wbar and W_true after k sweeps
  oracle    the same sweep counts from the CPU oracles at N = 2000, D = 32, q = 8 (no GPU needed)
One JSON line per measurement on stdout, also appended to --out ('' for stdout only); the GPU parts carry the GPU's name and power
limit read in the same process.
"""
import argparse
import collections
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [("C2", 1_000_000, 256, 16, 0.2, False), ("C3-shard", 1_250_000, 1024, 32, 0.3, False),
          ("C4-shape", 400_000, 512, 64, 0.3, True)]
MODES = ("columns", "rows")
REL_TOL = 1e-7
ANGLE_AT = (5, 10, 20, 50, 100, 1000)


def gpu_info():
    import torch
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as ex:  # pragma: no cover
        return {"gpu": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % ex}


def w_true(D, q, correlated, g, dev):
    """N(0, 1) loadings, or (correlated) W = G C^T diag(s): AR(1) column correlation 0.8, column scales log-spaced over 10x."""
    import torch
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    if correlated:
        idx = torch.arange(q, device=dev, dtype=torch.float64)
        C = torch.linalg.cholesky(0.8 ** (idx[:, None] - idx[None, :]).abs())
        W = (W @ C.T) * torch.logspace(0.0, -1.0, q, device=dev, dtype=torch.float64)[None, :]
    return W


def dense(N, D, q, missing, seed, dev, correlated=False):
    """(X with NaN, W_true): x_n = W z_n + mu + noise of precision 4."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    W = w_true(D, q, correlated, g, dev)
    mu = torch.randn(D, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        x = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64) @ W.T + mu
        x += 0.5 * torch.randn(n, D, generator=g, device=dev, dtype=torch.float64)
        x[torch.rand(n, D, generator=g, device=dev) < missing] = float("nan")
        X[lo:lo + n] = x
    return X, W.cpu().numpy()


def principal_angle(A, B):
    qa, _ = np.linalg.qr(A)
    qb, _ = np.linalg.qr(B)
    s = np.clip(np.linalg.svd(qa.T @ qb, compute_uv=False), -1.0, 1.0)
    return float(np.degrees(np.arccos(s.min())))


def convergence(bounds, angles=None):
    """Sweeps until learn(tol=1e-3) stops (the sweep whose bound gained < 1e-3) and until |db| < REL_TOL |b|."""
    b = np.asarray(bounds)
    d = np.diff(np.concatenate([[-np.inf], b]))
    learn = int(np.argmax(d < 1e-3)) + 1 if np.any(d < 1e-3) else None
    rel = np.abs(np.diff(b)) < REL_TOL * np.abs(b[1:])
    out = {"sweeps_learn_tol_1e-3": learn, "sweeps_rel_%g" % REL_TOL: int(np.argmax(rel)) + 2 if np.any(rel) else None,
           "sweeps_run": len(b), "final_bound": float(b[-1])}
    if angles is not None:
        out["max_principal_angle_deg"] = angles
    return out


def time_window(e, window):
    import torch
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


def wstep_kernels(e, calls=20):
    """Device time per update_W call of every kernel it launches, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    e.update_W()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            e.update_W()
        torch.cuda.synchronize()
    out = collections.defaultdict(float)
    for evt in prof.events():
        if evt.device_type == torch.autograd.DeviceType.CUDA:
            out[evt.name.replace("(anonymous namespace)::", "").split("(")[0][:90]] += evt.device_time / calls
    return {k: round(v, 2) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--part", default="time,wstep,converge,oracle")
    ap.add_argument("--window", type=float, default=1.0, help="seconds of sweeps per measurement")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sweeps", type=int, default=1000, help="sweeps of the convergence runs")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_wrows_b200.jsonl"),
                    help="also append the JSON lines to this file ('' for none)")
    a = ap.parse_args()
    parts = set(a.part.split(","))
    f = open(a.out, "a") if a.out else None

    def emit(rec):
        print(json.dumps(rec), flush=True)
        if f:
            f.write(json.dumps(rec) + "\n")
    try:
        if parts & {"time", "wstep", "converge"}:
            gpu_parts(a, parts, emit)
        if "oracle" in parts:
            oracle_part(emit)
    finally:
        if f:
            f.close()


def gpu_parts(a, parts, emit):
    import torch
    from pyvb_b200 import PlateEngine
    if not torch.cuda.is_available():
        raise SystemExit("bench_wrows.py measures on the GPU; there is none here (--part oracle runs on the CPU)")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    for name, N, D, q, missing, ard in SHAPES:
        if not parts & {"time", "wstep"}:
            break
        X, _ = dense(N, D, q, missing, 1, dev)
        engines = {m: PlateEngine(X, q, ard=ard, w_posterior=m) for m in MODES}
        del X
        for e in engines.values():
            e.init_random(seed=5)
            e.run(3)
            torch.cuda.synchronize()
        if "time" in parts:
            for rep in range(a.reps):
                for m, e in engines.items():                 # alternating: columns, rows, columns, ...
                    ms, n = time_window(e, a.window)
                    e.check()
                    emit(dict(info, part="time", shape=name, N=N, D=D, q=q, ard=ard, w_posterior=m, rep=rep,
                              int8=bool(e.use_i8), sweeps=n, ms_per_sweep=round(ms, 4), bound=float(e.elbo())))
        if "wstep" in parts:
            for m, e in engines.items():
                emit(dict(info, part="wstep", shape=name, N=N, D=D, q=q, w_posterior=m, kernel_us_per_update_W=wstep_kernels(e)))
        del engines
        torch.cuda.empty_cache()
    if "converge" in parts:
        N, D, q = 1_000_000, 256, 16
        for data in ("C2", "C2-correlated"):
            X, Wt = dense(N, D, q, 0.2, 7, dev, correlated=(data == "C2-correlated"))
            for m in MODES:
                e = PlateEngine(X, q, w_posterior=m)
                e.init_random(seed=3)
                bounds, angles = [], {}
                for k in range(1, a.sweeps + 1):
                    bounds.append(e.iterate())
                    if k in ANGLE_AT:
                        angles[k] = round(principal_angle(e.Wbar.cpu().numpy(), Wt), 6)
                e.check()
                emit(dict(info, part="converge", data=data, N=N, D=D, q=q, w_posterior=m, **convergence(bounds, angles)))
                del e
            del X
            torch.cuda.empty_cache()


def oracle_part(emit):
    from oracle.plate_oracle import PlateOracle
    from oracle.wrows_oracle import WRowsPlateOracle
    N, D, q = 2000, 32, 8
    for data in ("C2", "C2-correlated"):
        rng = np.random.RandomState(7)
        W = rng.randn(D, q)
        if data == "C2-correlated":
            idx = np.arange(q)
            W = (W @ np.linalg.cholesky(0.8 ** np.abs(idx[:, None] - idx[None, :])).T) * np.logspace(0.0, -1.0, q)[None, :]
        X = rng.randn(N, q) @ W.T + rng.randn(D)[None, :] + 0.5 * rng.randn(N, D)
        X[rng.rand(N, D) < 0.2] = np.nan
        init = {"Wbar": rng.randn(D, q), "Wvar": np.ones((D, q)), "mu": np.zeros(D), "muvar": np.ones(D),
                "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)), "qb": 0.5}
        for m, cls in (("columns", PlateOracle), ("rows", WRowsPlateOracle)):
            o = cls(X, q)
            o.load_state(init)
            bounds, angles = [], {}
            for k in range(1, 1001):
                bounds.append(o.iterate())
                if k in ANGLE_AT:
                    angles[k] = round(principal_angle(o.Wbar, W), 6)
            emit(dict(part="oracle", device="cpu (numpy oracle)", data=data, N=N, D=D, q=q, w_posterior=m,
                      **convergence(bounds, angles)))


if __name__ == "__main__":
    main()
