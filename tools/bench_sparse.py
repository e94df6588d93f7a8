"""Sparse-observation sweep benchmark (CSR input, kernels_sparse.cu) against the dense default path on the same data.

One process, JSON lines on stdout (and --out): first the card (name, power limit, max SM clock, read in this call), then
one line per (shape, density) with the median ms per sweep (CUDA events around every sweep after warm-up, timed window
>= --window seconds), the phase times (W update | Z step = K1-csr + K2 | statistics + globals), rows and stored entries per
second, the bytes the two gather kernels read (model: nnz * MZ/Gw pitch * 8 each) and the rate over their phase time, and
the HBM floor of a sweep (CSR / CSC streams, MZ passes, Sig, partials).  The dense default path (NaN-filled X) runs once
per shape where it fits (its time does not depend on the density).  Data: uniform random pattern, N(0, 1) values, from a
seeded device generator; state from init_random.

    python tools/bench_sparse.py [--quick] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = [  # (N, D, q, densities, run the dense default path)
    (1_000_000, 4096, 16, (0.005, 0.01, 0.02, 0.05, 0.10, 0.20), True),
    (1_000_000, 16384, 16, (0.005, 0.02), False),
    (400_000, 2048, 64, (0.02,), False),
]
QUICK = [(20_000, 512, 16, (0.01, 0.1), True), (5_000, 300, 64, (0.05,), False)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout
        name, pl, clk = [s.strip() for s in out.strip().splitlines()[0].split(",")]
    except Exception as ex:  # pragma: no cover
        name, pl, clk = torch.cuda.get_device_name(), "unknown (%s)" % ex, "unknown"
    return {"card": name, "power_limit": pl, "max_sm_clock": clk}


def make_csr(N, D, density, seed, dev):
    """Uniform random pattern (each entry stored with probability `density`), N(0,1) values: (crow, col int64, val)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    crow = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    cols, step = [], max(1, (1 << 28) // D)
    for lo in range(0, N, step):
        m = torch.rand(min(step, N - lo), D, generator=g, device=dev) < density
        crow[lo + 1:lo + 1 + m.shape[0]] = m.sum(1)
        cols.append(m.nonzero(as_tuple=True)[1])
        del m
    crow = torch.cumsum(crow, 0)
    col = torch.cat(cols)
    val = torch.randn(col.numel(), generator=g, device=dev, dtype=torch.float64)
    return crow, col, val


def time_sweeps(e, window):
    """Median / mean ms per sweep (CUDA events around each sweep), window >= `window` seconds after 2 warm-up sweeps."""
    for _ in range(2):
        e.iterate_async()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e.iterate_async()
    torch.cuda.synchronize()
    est = max(time.perf_counter() - t0, 1e-4)
    n = max(5, int(window / est) + 1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
    ev[0].record()
    for i in range(n):
        e.iterate_async()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(n))
    return ms[n // 2], ev[0].elapsed_time(ev[n]) / n, n


def time_phases(e, n=5):
    """Median ms of the three phases of a mode-B sweep: update_W | update_Z | statistics + Mu/Alpha/Beta/ELBO."""
    from pyvb_b200._layout import OP_ALPHA, OP_BETA, OP_ELBO, OP_MU
    out = {"w_ms": [], "z_ms": [], "stats_globals_ms": []}
    for _ in range(n):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        e.update_W()
        ev[1].record()
        e.update_Z()
        ev[2].record()
        slot = e.trace_pos % e.trace.numel()
        e._global(OP_MU | OP_ALPHA | OP_BETA | OP_ELBO, e.trace.data_ptr() + slot * 8)
        e.trace_pos += 1
        ev[3].record()
        torch.cuda.synchronize()
        for i, k in enumerate(("w_ms", "z_ms", "stats_globals_ms")):
            out[k].append(ev[i].elapsed_time(ev[i + 1]))
    return {k: sorted(v)[len(v) // 2] for k, v in out.items()}


def bytes_model(e, nnz):
    N, D, q, P = e.N, e.D, e.q, e.P
    pitch = e.ldmz * 8
    L = e.L.len * 8
    nblk = e.csc.nblk
    streams = 8 * (N + 1) + 12 * nnz + 8 * (nblk * D + 1) + 12 * nnz
    mz = 4 * N * pitch                       # K1 writes, K2 reads + writes, K3 reads (once, if the L2 held every block)
    sig = N * P * 8
    partials = 2 * nblk * L
    return {"k1_gather_bytes": nnz * pitch, "k3_gather_bytes": nnz * pitch,
            "hbm_floor_bytes": streams + mz + sig + partials, "row_blocks": nblk,
            "rows_per_block": e.csc.rows_per_block}


def run_sparse(N, D, q, dens, window, dev, out):
    from pyvb_b200 import PlateEngine
    crow, col, val = make_csr(N, D, dens, seed=1, dev=dev)
    nnz = int(col.numel())
    Xs = torch.sparse_csr_tensor(crow, col, val, size=(N, D))
    t0 = time.perf_counter()
    e = PlateEngine(Xs, q)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    del Xs, crow, col, val
    e.init_random(seed=5)
    med, mean, n = time_sweeps(e, window)
    ph = time_phases(e)
    bm = bytes_model(e, nnz)
    elbo = e.elbo()
    rec = {"path": "sparse", "N": N, "D": D, "q": q, "density": dens, "nnz": nnz, "ms_per_sweep": med,
           "ms_per_sweep_mean": mean, "timed_sweeps": n, **ph,
           "rows_it_per_s": N / (med * 1e-3), "entries_it_per_s": nnz / (med * 1e-3), **bm,
           "k1_gather_GBps_over_z_phase": bm["k1_gather_bytes"] / (ph["z_ms"] * 1e-3) / 1e9,
           "k3_gather_GBps_over_stats_phase": bm["k3_gather_bytes"] / (ph["stats_globals_ms"] * 1e-3) / 1e9,
           "hbm_floor_ms_at_7.7TBps": bm["hbm_floor_bytes"] / 7.7e12 * 1e3, "construct_s": build_s, "elbo": elbo}
    out(rec)
    del e
    torch.cuda.empty_cache()


def run_dense(N, D, q, dens, window, dev, out):
    from pyvb_b200 import PlateEngine
    crow, col, val = make_csr(N, D, dens, seed=1, dev=dev)
    X = torch.full((N, D), float("nan"), dtype=torch.float64, device=dev)
    rows = torch.repeat_interleave(torch.arange(N, device=dev), crow[1:] - crow[:-1])
    X[rows, col] = val
    nnz = int(col.numel())
    del rows, crow, col, val
    e = PlateEngine(X, q)
    path = "i8" if e.use_i8 else "dmma" if e.lib.pyvb_algo_supported(2, D, q) else "generic"
    del X
    e.init_random(seed=5)
    med, mean, n = time_sweeps(e, window)
    ph = time_phases(e)
    out({"path": "dense_default", "kernels": path, "N": N, "D": D, "q": q, "density": dens, "nnz": nnz,
         "ms_per_sweep": med, "ms_per_sweep_mean": mean, "timed_sweeps": n, **ph, "rows_it_per_s": N / (med * 1e-3),
         "elbo": e.elbo()})
    del e
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true", help="small shapes (a check of the script, not a measurement)")
    ap.add_argument("--window", type=float, default=1.0, help="seconds of timed sweeps per point (>= 1 for a measurement)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    f = open(a.out, "a") if a.out else None

    def out(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        if f:
            f.write(s + "\n")
            f.flush()

    out({"bench": "sparse", **card(), "window_s": a.window, "quick": a.quick})
    for N, D, q, dens_list, dense in (QUICK if a.quick else SHAPES):
        for dens in dens_list:
            run_sparse(N, D, q, dens, a.window, dev, out)
        if dense:
            run_dense(N, D, q, dens_list[1] if len(dens_list) > 1 else dens_list[0], a.window, dev, out)
    if f:
        f.close()


if __name__ == "__main__":
    main()
