#!/usr/bin/env python
"""Benchmark of the VB-PCA (missing data) hot path -- BASELINE.json's metric: rows*iterations/s.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA arm (one process per GPU)
    python bench.py --impl reference [--steps K] [--warmup W]      the reference's own CPU implementation
    python bench.py ... --dump-outputs DIR                          also write the headline's outputs as DIR/<name>.npy

Workload (config.workload): BASELINE.json configs[1] -- N=1M rows, D=256, q=16, 20% entries missing,
FP64, masked ("mode B") VB-PCA, synthetic data generated on the device.  With --gpus N every rank owns
its own 1M-row shard (weak scaling); the only exchange per sweep is one all-reduce of the packed
statistics buffer (fused into the statistics kernel over NVLink peer memory).  A "step" is one full VB
sweep (W columns, Z rows, Mu, Beta, ELBO) over the shard.

Besides the headline the line carries: `parity` (N = 1: the benchmarked kernels against the CPU oracle, ELBO and state
relative errors = BASELINE.json's "ELBO rel err vs ref"), `multi_gpu_check` (N > 1: a fixed global problem sharded over the
ranks against the oracle, both exchanges, bit-identity of the replicas), `c3_shard` (BASELINE.json configs[2] at one GPU's
share of its rows, 1.25M x 1024, q = 32: with --gpus 8 this is config 3 itself), `c4_shape` (N = 1: the shape of configs[3],
ARD, D = 512, q = 64, at 400k rows: the q = 64 kernels), `dmma_variant` / `f32_variant` /
`variant_elbo` (the all-FP64-tensor-core and the FP32 tcgen05 sweeps on the same shard, same sweep counts), `cpu_baseline`.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "VB-PCA missing-data rows*iters/sec"
UNIT = "rows*iters/s"


def workload_name(a):
    return "VB-PCA missing data N=%d (per GPU) D=%d q=%d %d%% missing FP64 mode=%s%s" % (
        a.N, a.D, a.q, int(round(a.missing * 100)), a.mode, " ARD" if getattr(a, "ard", False) else "")


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """Polls NVML (clocks, power, throttle reasons) every 20 ms from a thread; the samples that fall inside the timed
    region are reported.  It is created BEFORE the barrier that precedes the timed region: nvmlInit takes ~0.1 s, and
    when only rank 0 paid it after the barrier every other rank's first exchange waited for rank 0 inside ITS timed
    region (0.3-9 ms per sweep of apparent multi-GPU overhead, tools/comm_probe.sh)."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
               "hw_power_brake": 0x80, "sync_boost": 0x10}

    def __init__(self, index, interval=0.02):
        self.rows, self.ok, self._stop, self.interval = [], False, False, float(interval)
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop:
            try:
                fields = os.environ.get("PYVB_SAMPLER_FIELDS", "crp")      # diagnosis: which query disturbs
                rs, clk, pw = 0, 0, 0.0
                if "r" in fields:
                    try:
                        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if "c" in fields:
                    clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                if "p" in fields:
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.rows.append((time.time(), clk, pw, rs))
            except Exception:
                pass
            time.sleep(self.interval)

    def stop(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self._stop = True
        self.t.join(timeout=1.0)
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows[-3:]
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= int(r[3])
        reasons = sorted(n for n, bit in self.REASONS.items() if mask & bit)
        return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": float(self.max), "reasons": reasons,
                "power_w_max": max(r[2] for r in rows) if rows else None, "samples": len(rows)}


# ----------------------------------------------------------------------------- CPU baselines
def _synth_host(N, D, q, missing, seed):
    import numpy as np
    rng = np.random.RandomState(seed)
    W = rng.randn(D, q); Z = rng.randn(N, q); mu = rng.randn(D)
    X = Z @ W.T + mu[None, :] + rng.randn(N, D) * np.sqrt(1.0 / 20.0)
    X[rng.rand(N, D) < missing] = np.nan
    return X


def time_literal_reference(D, q, missing, rows, steps, warmup):
    """The UNMODIFIED reference (py3-translated copy in oracle/_ref), built exactly like
    examples/PCA_missing_data.py:31-42, one Network.learn(1) sweep per step."""
    import numpy as np
    from oracle.make_ref import import_ref
    pyvb = import_ref()
    if pyvb is None:
        return None
    X = _synth_host(rows, D, q, missing, seed=99)
    sink = io.StringIO()
    with contextlib.redirect_stdout(sink):
        np.random.seed(0)
        nodes = pyvb.nodes
        Ws = [nodes.Gaussian(D, np.zeros((D, 1)), np.eye(D) * 1e-3) for i in range(q)]
        W = nodes.hstack(Ws)
        Mu = nodes.Gaussian(D, np.zeros((D, 1)), np.eye(D) * 1e-3)
        Beta = nodes.Gamma(D, 1e-3, 1e-3)
        Zs = [nodes.Gaussian(q, np.zeros((q, 1)), np.eye(q)) for i in range(rows)]
        Xs = [nodes.Gaussian(D, W * z + Mu, Beta) for z in Zs]
        [xn.observe(xv.reshape(D, 1)) for xn, xv in zip(Xs, X)]
        net = pyvb.Network(); net.addnode(W); net.fetch_network()
        for _ in range(warmup):
            net.learn(1, tol=-np.inf)
        t0 = time.perf_counter()
        for _ in range(steps):
            net.learn(1, tol=-np.inf)
        dt = time.perf_counter() - t0
    return {"value": rows * steps / dt, "seconds": dt, "rows": rows, "steps": steps}


def time_port(D, q, missing, rows, steps, warmup):
    """The numpy restatement (oracle/plate_oracle.py, mode B), all host cores through BLAS."""
    import numpy as np
    from oracle.plate_oracle import PlateOracle
    X = _synth_host(rows, D, q, missing, seed=98)
    o = PlateOracle(X, q, mode="B")
    rng = np.random.RandomState(0)
    o.Wbar = rng.randn(D, q); o.Zbar = rng.randn(rows, q)
    for _ in range(warmup):
        o.iterate()
    t0 = time.perf_counter()
    for _ in range(steps):
        o.iterate()
    dt = time.perf_counter() - t0
    return {"value": rows * steps / dt, "seconds": dt, "rows": rows, "steps": steps}


def cpu_baseline(a, budget_s=25.0):
    cores = os.cpu_count() or 1
    lit = None
    try:
        lit = time_literal_reference(a.D, a.q, a.missing, rows=max(1, int(budget_s / 2 / 7.0)), steps=1, warmup=0)
    except Exception as e:  # pragma: no cover
        lit = None
        sys.stderr.write("literal reference failed: %r\n" % (e,))
    port = time_port(a.D, a.q, a.missing, rows=16384, steps=1, warmup=1)
    if lit is not None:
        out = {"value": lit["value"], "unit": UNIT, "cores": 1, "kind": "reference",
               "sample": "literal pyvb (py3-translated, single-threaded Python+numpy): %d rows x %d sweep of the same "
                         "D=%d q=%d %d%%-missing workload in %.1f s (its Z step allocates 8*q^2*D^2 bytes per row)"
                         % (lit["rows"], lit["steps"], a.D, a.q, int(a.missing * 100), lit["seconds"])}
    else:
        out = {"value": port["value"], "unit": UNIT, "cores": cores, "kind": "port", "sample": ""}
    out["port"] = {"value": port["value"], "cores": cores,
                   "sample": "numpy plate oracle (mode B, OpenBLAS on all cores): %d rows x %d sweep in %.1f s"
                             % (port["rows"], port["steps"], port["seconds"])}
    return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = max(1, a.steps + a.warmup)
    rows = max(1, min(16, int(240.0 / (total * 4.4))))         # ~4.4 s per row and sweep at D = 256, q = 16: a ~4 minute run
    res, kind, cores = None, "reference", 1
    try:
        res = time_literal_reference(a.D, a.q, a.missing, rows=rows, steps=a.steps, warmup=a.warmup)
    except Exception as e:  # pragma: no cover
        sys.stderr.write("literal reference failed: %r\n" % (e,))
    if res is None:
        kind, cores = "port", os.cpu_count() or 1
        res = time_port(a.D, a.q, a.missing, rows=16384, steps=a.steps, warmup=a.warmup)
    sample = "%d rows per step, %d steps (+%d warm-up) of the D=%d q=%d %d%%-missing workload, %.1f s" % (
        res["rows"], res["steps"], a.warmup, a.D, a.q, int(a.missing * 100), res["seconds"])
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * res["seconds"] / max(1, a.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "sample": sample},
            "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------- our arm
def make_data(torch, N, D, q, missing, seed, dev, rank=0):
    """Synthetic shard (SURVEY 8d): the model -- W_true, mu_true -- is drawn from `seed` alone, so every rank sees rows of
    the SAME subspace; the rows (Z, noise, erasures) come from a per-rank stream."""
    f64 = torch.float64
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    Wt = torch.randn(D, q, generator=g, device=dev, dtype=f64)
    mu = torch.randn(D, generator=g, device=dev, dtype=f64)
    g.manual_seed(seed + 7919 * (rank + 1))
    X = torch.empty(N, D, device=dev, dtype=f64)
    step = 1 << 16
    for lo in range(0, N, step):
        n = min(step, N - lo)
        Z = torch.randn(n, q, generator=g, device=dev, dtype=f64)
        x = Z @ Wt.t() + mu + torch.randn(n, D, generator=g, device=dev, dtype=f64) * (1.0 / 20.0) ** 0.5
        m = torch.rand(n, D, generator=g, device=dev) < missing
        x[m] = float("nan")
        X[lo:lo + n] = x
    return X


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def time_calls(torch, dev, fn, n):
    fn(); torch.cuda.synchronize(dev)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(n):
        fn()
    a1.record(); torch.cuda.synchronize(dev)
    return a0.elapsed_time(a1) / n


_DMMA_PEAK = {}


def dmma_peak_tflops(torch, dev, lib, _cabi):
    """FP64 tensor roofline of this box: a pure DMMA.8x8x4 loop (MEASURED_PEAKS.json has no FP64 figure)."""
    if dev not in _DMMA_PEAK:
        scratch = torch.empty(148 * 2 * 256, dtype=torch.float64, device=dev)
        iters = 20000
        st = torch.cuda.current_stream(dev).cuda_stream
        ms_p = min(time_calls(torch, dev, lambda: _cabi.check(lib.pyvb_bench_dmma_f64(148 * 2, iters, scratch.data_ptr(), st),
                                                             "bench_dmma"), 2) for _ in range(3))
        _DMMA_PEAK[dev] = 148 * 2 * 8 * iters * 8 * 512.0 / (ms_p * 1e-3) * 1e-12
    return _DMMA_PEAK[dev]


# launches of one mode-B sweep (engine.iterate_async), read off the C-ABI entry points in pyvb_b200/csrc/cabi.cu:
#   INT8 path: wupdate, pack_gw | pack_g_i8, zstep_i8, pack_weta, zstep_dmma<ETA>, zsolve, [zstep_dmma, zsolve: guard fall-back,
#              exit at once] | colmax_reduce, digitize, stats_i8, stats_dmma<XO>, stats_i8_check, [stats_dmma: guard fall-back],
#              stats_reduce(+exchange) | global                                                                = 17
#   all-DMMA path: wupdate, pack_gw, zstep_dmma, zsolve, stats_dmma, stats_reduce(+exchange), global              = 7
def launches_per_sweep(eng):
    if eng.use_i8:
        return 17 if eng.use_i8_stats else 14
    return 7


def kernel_breakdown(torch, dev, eng, lib, _cabi, rows):
    """Per-kernel times of one sweep (CUDA events on the launching stream, 5 calls each) and their algorithmic bytes."""
    tc = lambda fn, n: time_calls(torch, dev, fn, n)
    D, q = eng.D, eng.q
    P = q * (q + 1) // 2
    eng._ensure_gw()
    out = {"zstep_ms": tc(lambda: eng.update_Z(), 5)}
    stream = torch.cuda.current_stream(dev).cuda_stream
    zs = eng.zsums.data_ptr() if eng.zsums is not None else 0

    def k2_only():
        _cabi.check(lib.pyvb_zsolve_f64(eng.N, q, eng.MZ.data_ptr(), eng.ldmz, 0, eng.logdet.data_ptr(), eng.gl.data_ptr(),
                                        zs, stream), "zsolve")
    if eng.use_i8:
        def k1_phase(ph):
            _cabi.check(lib.pyvb_zstep_i8_f64(eng.N, D, q, eng.X.data_ptr(), D, eng.mask8.data_ptr(), eng.Wbar.data_ptr(),
                                              eng.Wvar.data_ptr(), eng.Gw.data_ptr(), eng.ldg, eng.P0.data_ptr(),
                                              eng.h0.data_ptr(), eng.gl.data_ptr(), eng.MZ.data_ptr(), eng.ldmz,
                                              eng.GI.data_ptr(), eng.gscale.data_ptr(), 0, eng.logdet.data_ptr(), 0, ph,
                                              stream), "zstep_i8")
        out["zstep_k1_i8_ms"] = tc(lambda: k1_phase(2), 5)
        out["zstep_k1_eta_ms"] = tc(lambda: k1_phase(3), 5)
        out["zstep_k1_ms"] = tc(lambda: k1_phase(1), 5)
        k1_phase(1)
        out["zsolve_k2_ms"] = tc(k2_only, 3)
        eng.update_Z()
    elif lib.pyvb_algo_supported(2, D, q):
        def k1_only():
            alg, eng.algo = eng.algo, 3          # PYVB_ALGO_DMMA_K1: contraction only
            eng.update_Z()
            eng.algo = alg
        out["zstep_k1_ms"] = tc(k1_only, 5)
        k1_only()
        out["zsolve_k2_ms"] = tc(k2_only, 3)
        eng.update_Z()

    def stats_call():
        eng._stats_fresh = False
        dflag, eng.distributed = eng.distributed, False
        eng._ensure_stats()
        eng.distributed = dflag
    out["stats_ms"] = tc(stats_call, 5)
    return out


def rooflines(eng, kt, rows, ms_sweep, hbm, peak_tf, traffic_json):
    """The dominant kernel's roofline entry (the contract's `roofline` object) + the per-kernel table."""
    D, q = eng.D, eng.q
    P = q * (q + 1) // 2
    fl_sweep = rows * (4.0 * D * P + 6.0 * D * q + q ** 3 + 2.0 * q * q)
    by_sweep = rows * (8.0 * D + 8.0 * q + 8.0 * P)
    table = None
    if eng.use_i8:
        ncz = (P + q + 31) // 32 * 32
        by = {"zstep_i8_kernel (INT8 mask contraction -> qprec)": (rows * (1.0 * D + 8.0 * P), kt["zstep_k1_i8_ms"]),
              "zstep_dmma_kernel<ETA> (eta = O.(X-mu) @ W, FP64 tensor cores)": (rows * (8.0 * D + 8.0 * q), kt["zstep_k1_eta_ms"]),
              "zsolve (K2: batched q x q SPD inverse / solve)": (rows * (16.0 * (P + q) + 8.0), kt["zsolve_k2_ms"]),
              "statistics (digitize + INT8 T1/Bst + DMMA Ast + guard + reduce)":
                  (rows * (8.0 * (P + q) + 7.0 * ncz + 1.0 * D + 7.0 * ncz + 8.0 * D + 8.0 * q), kt["stats_ms"])}
        table = {k: {"ms": v[1], "algorithmic_GB": v[0] * 1e-9, "GBps": v[0] / (v[1] * 1e-3) * 1e-9,
                     "frac_of_hbm_peak": v[0] / (v[1] * 1e-3) * 1e-9 / hbm} for k, v in by.items()}
        kname = ("zsolve (K2: batched q x q SPD inverse / solve, in place on the MZ rows; Gauss-Jordan in registers at q = 16, 32)"
                 if q != 64 else
                 "zsolve (K2: batched q x q SPD inverse / solve, in place on the MZ rows; blocked symmetric sweep on DMMA at q = 64)")
        by_dom, ms_dom = rows * (16.0 * (P + q) + 8.0), kt["zsolve_k2_ms"]
        traffic = None
        t = traffic_json.get("zsolve%d_dram_bytes_per_row" % q)
        if t is not None:
            traffic = t * rows
        ach = by_dom / (ms_dom * 1e-3) * 1e-9
        roof = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs",
                "bytes_per_launch": by_dom, "ms_per_launch": ms_dom, "fp64_tensor_peak_tflops": peak_tf,
                "sweep_fp64_equivalent_tflops": fl_sweep / (ms_sweep * 1e-3) * 1e-12,
                "sweep_algorithmic_GBps": by_sweep / (ms_sweep * 1e-3) * 1e-9,
                "sweep_frac_of_hbm_peak": by_sweep / (ms_sweep * 1e-3) * 1e-9 / hbm,
                "note": "the mask contractions run as exact integer GEMMs on the INT8 tensor cores: the sweep's FP64-equivalent "
                        "rate exceeds the FP64 tensor roof; every kernel is a stream over HBM (see kernels.i8_path)"}
    else:
        fl_k1 = rows * (2.0 * D * P + 2.0 * D * q)
        ms_k1 = kt.get("zstep_k1_ms")
        if ms_k1 is None:
            fl_k1, ms_k1 = fl_k1 + rows * (q ** 3 + 2.0 * q * q), kt["zstep_ms"]
        ach = fl_k1 / (ms_k1 * 1e-3) * 1e-12
        t = traffic_json.get("zstep_dmma%d_dram_bytes_per_row" % q)
        roof = {"bound": "tensor", "kernel": "zstep_dmma_kernel (K1: mask @ vec(G) contraction on the FP64 tensor cores)",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": t * rows if t is not None else None,
                "peak_source": "FP64 DMMA.8x8x4 loop measured in this run (MEASURED_PEAKS.json has no FP64 figure)",
                "flops_per_launch": fl_k1, "ms_per_launch": ms_k1,
                "sweep_algorithmic_tflops": fl_sweep / (ms_sweep * 1e-3) * 1e-12,
                "sweep_frac_of_fp64_tensor_peak": fl_sweep / (ms_sweep * 1e-3) * 1e-12 / peak_tf}
    return roof, table


def timed_sweeps(torch, dist, dev, eng, steps, warmup, sampler_local=None):
    """W warm-up sweeps, then exactly `steps` sweeps bracketed by barrier + synchronize; max over ranks (ms)."""
    def sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)
    for _ in range(max(warmup, 3)):
        eng.iterate_async()
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    slots = [eng.iterate_async() for _ in range(steps)]
    e1.record()
    sync()
    t1 = time.time()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), slots, (t0, t1)


def parity_vs_oracle(torch, dev, D, q, missing, ard, algo, rows, sweeps, seed=4242):
    """BASELINE.json's 'ELBO rel err vs ref': `sweeps` sweeps of a `rows`-row problem of the same shape through the SAME
    kernels (same algo) and through the CPU oracle (oracle/plate_oracle.py, pinned on the literal reference's goldens),
    from the same initial state.  Mode-B Gamma / ELBO under masking cannot be expressed in the literal reference
    (SURVEY 8c: 'parity unpinned' for those two terms): they are the reference formulas restricted to observed entries."""
    import numpy as np
    from pyvb_b200 import PlateEngine
    from oracle.plate_oracle import PlateOracle
    X = make_data(torch, rows, D, q, missing, seed, dev)
    e = PlateEngine(X, q, mode="B", algo=algo, keep_sigma=True, device=dev, ard=ard)
    e.init_random(seed=99)
    st0 = e.get_state()
    o = PlateOracle(X.cpu().numpy(), q, mode="B", ard=ard)
    o.load_state({k: st0[k] for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb", "al_qb")})
    t0 = time.perf_counter()
    elbo_err = state_err = 0.0
    for _ in range(sweeps):
        ref = o.iterate()
        got = e.iterate()
        elbo_err = max(elbo_err, abs(got - ref) / abs(ref))
        st = e.get_state()
        for k in ("Wbar", "Wvar", "mu", "Zbar", "Sig"):
            r = getattr(o, k)
            state_err = max(state_err, float(np.max(np.abs(st[k] - r)) / np.max(np.abs(r))))
        state_err = max(state_err, abs(st["qb"] - o.qb) / abs(o.qb))
    e.check()
    out = {"elbo_rel_err_max": elbo_err, "state_rel_err_max": state_err, "rows": rows, "sweeps": sweeps,
           "algo": "i8" if e.use_i8 else algo, "i8_guard_fallbacks": list(e.i8_fallbacks()),
           "oracle": "oracle/plate_oracle.py (numpy, mode B), pinned <= 3.4e-12 on the literal reference's goldens; mode-B "
                     "Gamma/ELBO terms 'parity unpinned' by construction (SURVEY 8c)",
           "state": "tensor-wise max|a-b|/max|b| over Wbar, Wvar, mu, Zbar, Sigma, qb after every sweep",
           "seconds": time.perf_counter() - t0}
    del e, X
    torch.cuda.empty_cache()
    return out


def multi_gpu_check(torch, dist, dev, rank, world, D, q, missing, rows_total, sweeps=3):
    """A fixed global problem sharded over the ranks, through both exchanges (fused NVLink peer kernel / NCCL all-reduce):
    the bound of every sweep against the oracle on the FULL data (rank 0, CPU) and bit-identity of the replicated W."""
    import numpy as np
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    # the same global data set on every rank (rank-independent seed), each rank keeps its row block
    Xg = make_data(torch, rows_total, D, q, missing, 2025, dev)
    lo, hi = shard_rows(rows_total, world, rank)
    out = {"rows_total": rows_total, "sweeps": sweeps, "D": D, "q": q}
    ref = None
    if rank == 0:
        from oracle.plate_oracle import PlateOracle
        o = PlateOracle(Xg.cpu().numpy(), q, mode="B")
    init_seed = 31
    for comm in ("peer", "nccl"):
        os.environ["PYVB_COMM"] = comm
        e = PlateEngine(Xg[lo:hi].clone(), q, mode="B", algo="auto", keep_sigma=True, device=dev, distributed=True,
                        row_offset=lo)
        # one global initial state: generated for all rows on every rank, sliced
        g = torch.Generator(device=dev); g.manual_seed(init_seed)
        Wb = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
        Zb = torch.randn(rows_total, q, generator=g, device=dev, dtype=torch.float64)
        st = {"Wbar": Wb.cpu().numpy(), "Wvar": np.ones((D, q)), "mu": np.zeros(D), "muvar": np.ones(D),
              "Zbar": Zb[lo:hi].cpu().numpy(), "Sig": np.tile(np.eye(q), (hi - lo, 1, 1)), "qb": 0.5}
        e.set_state(st)
        elbo = [e.iterate() for _ in range(sweeps)]
        e.check()
        W = e.Wbar.clone()
        Ws = [torch.empty_like(W) for _ in range(world)]
        dist.all_gather(Ws, W)
        same = all(torch.equal(Ws[0], w) for w in Ws)
        if rank == 0:
            if ref is None:
                st_full = dict(st, Zbar=Zb.cpu().numpy(), Sig=np.tile(np.eye(q), (rows_total, 1, 1)))
                o.load_state(st_full)
                ref = [o.iterate() for _ in range(sweeps)]
                ref_W = o.Wbar.copy()
            out[comm] = {"elbo_rel_err_max": max(abs(a - b) / abs(b) for a, b in zip(elbo, ref)),
                         "Wbar_rel_err": float(np.max(np.abs(W.cpu().numpy() - ref_W)) / np.max(np.abs(ref_W))),
                         "replicas_bit_identical": bool(same), "peer_kernel": e.peers is not None}
        e.close()
        del e
    os.environ.pop("PYVB_COMM", None)
    if rank == 0:
        out["rel_err"] = max(out["peer"]["elbo_rel_err_max"], out["nccl"]["elbo_rel_err_max"],
                             out["peer"]["Wbar_rel_err"], out["nccl"]["Wbar_rel_err"])
        out["ok"] = bool(out["rel_err"] <= 1e-9 and out["peer"]["replicas_bit_identical"]
                         and out["nccl"]["replicas_bit_identical"])
    del Xg
    torch.cuda.empty_cache()
    dist.barrier()
    return out


def variant_traces(torch, dev, X, q, ard, sweeps, want_f32):
    """The same `sweeps` sweeps from the same initial state on the three arithmetic variants of the path: INT8-assisted FP64
    (default), all-FP64-tensor (DMMA) and the FP32 tcgen05 variant; the bounds side by side."""
    from pyvb_b200 import PlateEngine
    out = {}
    for name, kw in (("i8", {"algo": "auto"}), ("dmma", {"algo": "dmma"}), ("f32", {"precision": "f32"})):
        if name == "f32" and not want_f32:
            continue
        e = PlateEngine(X, q, mode="B", keep_sigma=False, device=dev, ard=ard, **kw)
        e.init_random(seed=777)
        e.set_state({"qb": e.qa})                  # start from tau = 1 (the stand-in start of the timed runs is tau ~ 1e8)
        out[name] = [e.iterate() for _ in range(sweeps)]
        e.check()
        del e
        torch.cuda.empty_cache()
    return out


def bench_dmma_variant(torch, dev, X, q, ard, steps, lib, _cabi, hbm, peak_tf, traffic_json):
    """The all-FP64-tensor-core sweep (algo='dmma': K1 and K3 on DMMA.8x8x4) on the same shard."""
    from pyvb_b200 import PlateEngine
    e = PlateEngine(X, q, mode="B", algo="dmma", keep_sigma=False, device=dev, ard=ard)
    e.init_random(seed=4321, rank=0)
    ms, slots, _ = timed_sweeps(torch, None, dev, e, steps, 3)
    kt = kernel_breakdown(torch, dev, e, lib, _cabi, e.N)
    roof, _ = rooflines(e, kt, e.N, ms / steps, hbm, peak_tf, traffic_json)
    D, P = e.D, e.P
    fl_s = e.N * (2.0 * D * P + 4.0 * D * q)
    out = {"value": e.N * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
           "dtype": "f64 (mask contractions on the FP64 tensor cores, DMMA.8x8x4)", "kernels": kt, "roofline_k1": roof,
           "stats_tflops": fl_s / (kt["stats_ms"] * 1e-3) * 1e-12, "stats_frac_of_fp64_tensor_peak":
               fl_s / (kt["stats_ms"] * 1e-3) * 1e-12 / peak_tf}
    del e
    torch.cuda.empty_cache()
    return out


def bench_f32(torch, a, dev, X, lib, _cabi, steps, hbm):
    """The FP32 variant on the same data: sweeps/s and its three kernels (CUDA events)."""
    from pyvb_b200 import PlateEngine
    e = PlateEngine(X, a.q, mode="B", keep_sigma=False, device=dev, precision="f32")
    e.init_random(seed=4321, rank=0)
    ms, slots, _ = timed_sweeps(torch, None, dev, e, steps, 3)
    ms /= steps
    e.check()
    st = torch.cuda.current_stream(dev).cuda_stream
    e._ensure_gw()
    tc = lambda fn, n: time_calls(torch, dev, fn, n)

    def k1():
        _cabi.check(lib.pyvb_zstep_k1_f32(e.N, e.D, e.q, e.planes.data_ptr(), e.GT.data_ptr(), e.WT.data_ptr(),
                                          e.P0.data_ptr(), e.h0.data_ptr(), e.gl.data_ptr(), e.MZ.data_ptr(), st), "k1")
    ms_k1 = tc(k1, 5)
    ms_z = tc(lambda: e.update_Z(), 5)

    def stats_call():
        e._stats_fresh = False
        e._ensure_stats()
    ms_s = tc(stats_call, 5)
    ncp = e.ldmz
    by_k1 = e.N * (3.0 * 2 * e.D + 4.0 * ncp)           # the three bf16 planes once + the FP32 row out
    by_k3 = e.N * (3.0 * 2 * e.D + 3.0 * 2 * ncp)       # the planes + the bf16 x 3 rows once
    out = {"value": e.N / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
           "dtype": "f32 rows, bf16x3 tcgen05 contraction with FP32 TMEM accumulation, FP64 batched solve",
           "tolerance": "one sweep from a shared state: 5e-5 tensor-wise on W, mu, Z, Sigma; 5e-3 on qb; see tests/test_gpu_f32.py",
           "kernels": {"k1_ms": ms_k1, "zstep_ms": ms_z, "k2_ms": ms_z - ms_k1, "stats_ms": ms_s},
           "roofline_k1": {"bound": "hbm", "achieved": by_k1 / (ms_k1 * 1e-3) * 1e-9, "peak": hbm, "unit": "GB/s",
                           "frac": by_k1 / (ms_k1 * 1e-3) * 1e-9 / hbm, "bytes_per_launch": by_k1},
           "roofline_k3": {"bound": "hbm", "achieved": by_k3 / (ms_s * 1e-3) * 1e-9, "peak": hbm, "unit": "GB/s",
                           "frac": by_k3 / (ms_s * 1e-3) * 1e-9 / hbm, "bytes_per_launch": by_k3}}
    del e
    torch.cuda.empty_cache()
    return out


def numa_cpus_of_gpu(index):
    """CPUs of the NUMA node the GPU hangs off (for NUMA-local pinned staging buffers); None when unknown."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return node, sorted(cpus & os.sched_getaffinity(0)) or None
    except Exception:
        return None


def bench_e2e(torch, dist, dev, eng, local, steps):
    """End to end through the public API with HOST buffers: every step uploads the shard from pinned host memory (allocated
    NUMA-local to the GPU), runs one sweep (iterate_from_host: chunked upload overlapped with the Z step and the chunk's
    statistics) and reads the bound back."""
    old_aff, numa = None, numa_cpus_of_gpu(local)
    if numa is not None and numa[1]:
        try:                                   # first touch + cudaHostRegister from a thread on the GPU's NUMA node
            old_aff = os.sched_getaffinity(0)
            os.sched_setaffinity(0, numa[1])
        except Exception:
            old_aff = None
    Xh = torch.empty(eng.N, eng.D, dtype=torch.float64, pin_memory=True)
    Xh.copy_(eng.X)
    res_h = torch.empty(1, dtype=torch.float64, pin_memory=True)

    def sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)
    slot = eng.iterate_from_host(Xh)           # warm-up (copy stream, chunk buffers)
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        slot = eng.iterate_from_host(Xh)
        res_h.copy_(eng.trace[slot:slot + 1], non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
    e1.record()
    sync()
    ms2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms2 = float(ms2.item())
    if old_aff is not None:
        os.sched_setaffinity(0, old_aff)
    del Xh
    world = dist.get_world_size() if dist is not None else 1
    h2d = eng.N * eng.D * 8
    return {"value": world * eng.N * steps / (ms2 * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
            "steps": steps, "h2d_GBps_per_gpu": h2d * steps / (ms2 * 1e-3) * 1e-9,
            "bound": "PCIe: the 8-byte data of every sweep crosses the host link (Gen5 x16 ~ 55 GB/s usable per GPU); "
                     "no kernel work can move this number",
            "numa_node_of_pinned_buffer": numa[0] if numa is not None else None,
            "path": "iterate_from_host: 8 row chunks, Z step = INT8 path, per-chunk statistics on the FP64 tensor cores "
                    "(DMMA), summed; at N > 1 one NCCL all-reduce of the statistics"}


DUMP_ROW_BYTES = 32 << 20        # the sampled per-row outputs; the rest (W, mu, globals, bounds) is O(D q + steps)


def dump_outputs(eng, slots, out_dir, seed=0):
    """What a caller of the timed sweeps receives, as float64 .npy files: the bound of every timed sweep, the replicated
    state (PlateEngine.get_state_small) and, for a fixed seeded sample of rows (its indices in `rows`), the rows' posterior
    means and covariances in get_state()'s layout.  The sample keeps the files small at any N (about 32 MB of rows)."""
    import numpy as np
    import torch
    from pyvb_b200.engine import tril_pack_index
    os.makedirs(out_dir, exist_ok=True)
    out = {"elbo": eng.trace[slots].cpu().numpy()}
    out.update(eng.get_state_small())
    q = eng.q
    n = min(eng.N, DUMP_ROW_BYTES // (8 * (q + q * q)))
    rows = np.sort(np.random.RandomState(seed).choice(eng.N, n, replace=False))
    dev = eng.Zbar.device
    it = torch.as_tensor(rows, device=dev)
    z = eng.Zbar[it].to(torch.float64)
    ii, jj = tril_pack_index(q)
    if eng.Sig is not None:
        sp = eng.Sig[it]
    else:
        sp = eng.M2[it].to(torch.float64) - z[:, torch.as_tensor(ii, device=dev)] * z[:, torch.as_tensor(jj, device=dev)]
    sp = sp.cpu().numpy()
    Sig = np.zeros((n, q, q))
    Sig[:, ii, jj] = sp
    Sig[:, jj, ii] = sp
    out.update(rows=rows, Zbar=z.cpu().numpy(), Sig=Sig)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))
    return sorted(out)


def measure_config(torch, dist, dev, rank, world, local, lib, _cabi, cfg, steps, warmup, sampler, hbm, peak_tf, traffic_json,
                   dump_dir=None):
    """Build the engine of one configuration on this rank's shard, time `steps` sweeps, break the sweep down; with
    `dump_dir` (rank 0) the outputs of the timed sweeps are written there before anything else runs on the engine."""
    from pyvb_b200 import PlateEngine
    N, D, q = cfg["N"], cfg["D"], cfg["q"]
    X = make_data(torch, N, D, q, cfg["missing"], 1234, dev, rank=rank)
    eng = PlateEngine(X, q, mode=cfg.get("mode", "B"), algo=cfg.get("algo", "auto"), keep_sigma=False,
                      distributed=(world > 1), row_offset=rank * N, device=dev, ard=cfg.get("ard", False))
    del X
    eng.init_random(seed=4321, rank=rank)
    if os.environ.get("PYVB_NOCOMM"):          # diagnosis only: time the sweeps without the exchange
        eng.distributed = False
    ms, slots, win = timed_sweeps(torch, dist, dev, eng, steps, warmup)
    eng.check()
    if dump_dir is not None and rank == 0:
        dump_outputs(eng, slots, dump_dir)
    elbo = [float(v) for v in eng.trace[slots].cpu().tolist()]
    kt = kernel_breakdown(torch, dev, eng, lib, _cabi, N)
    roof, table = rooflines(eng, kt, N, ms / steps, hbm, peak_tf, traffic_json)
    kt["i8_path"] = table
    res = {"value": world * N * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
           "rows_per_gpu": N, "rows_total": world * N, "roofline": roof, "kernels": kt, "elbo_last": elbo[-1] if elbo else None,
           "elbo_first": elbo[0] if elbo else None, "algo": "i8" if eng.use_i8 else cfg.get("algo", "auto"),
           "i8_guard_fallbacks": list(eng.i8_fallbacks()), "gpu_launches": launches_per_sweep(eng) * steps,
           "stats_len": eng.L.len}
    return eng, res, win


def run_ours(a):
    # exactly ONE line on stdout: libraries (NCCL banner ...) get stderr, the JSON line gets the real stdout
    sys.stdout.flush()
    real_out = os.dup(1)
    os.dup2(2, 1)
    import torch
    from pyvb_b200 import _cabi
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _cabi.lib()
    peaks = load_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    traffic_json = {}
    try:
        traffic_json = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    peak_tf = dmma_peak_tflops(torch, dev, lib, _cabi)
    sampler = ClockSampler(local) if (rank == 0 and not os.environ.get("PYVB_NOSAMPLER")) else None

    # ---- headline: BASELINE.json configs[1] (or the --N/--D/--q override), one shard per GPU
    cfg = {"N": a.N, "D": a.D, "q": a.q, "missing": a.missing, "mode": a.mode, "algo": a.algo, "ard": a.ard}
    eng, head, win = measure_config(torch, dist, dev, rank, world, local, lib, _cabi, cfg, a.steps, a.warmup, sampler, hbm,
                                    peak_tf, traffic_json, dump_dir=a.dump_outputs)
    clocks = sampler.stop(*win) if sampler is not None else None
    e2e = bench_e2e(torch, dist, dev, eng, local, max(1, min(a.steps, 8))) if a.mode == "B" else None

    # ---- the other arithmetic variants on the same shard, same sweep counts (N = 1 only)
    extra = {}
    if world == 1 and a.mode == "B" and not a.quick:
        want_f32 = (a.q in (16, 32) and a.D % 32 == 0 and not a.no_f32)
        ksteps = max(3, min(a.steps, 10))
        try:
            extra["dmma_variant"] = bench_dmma_variant(torch, dev, eng.X, a.q, a.ard, ksteps, lib, _cabi, hbm, peak_tf,
                                                       traffic_json)
            if want_f32:
                extra["f32_variant"] = bench_f32(torch, a, dev, eng.X, lib, _cabi, ksteps, hbm)
            tr = variant_traces(torch, dev, eng.X, a.q, a.ard, 8, want_f32)
            rel = lambda x, y: abs(x - y) / abs(y)
            extra["variant_elbo"] = {"sweeps": 8, "same_initial_state": "init_random(seed=777), tau = 1", "i8": tr["i8"][-1],
                                     "dmma": tr["dmma"][-1],
                                     "i8_vs_dmma_elbo_rel_err": max(rel(x, y) for x, y in zip(tr["i8"], tr["dmma"]))}
            if "f32" in tr:
                extra["variant_elbo"]["f32"] = tr["f32"][-1]
                extra["variant_elbo"]["f32_vs_f64_elbo_rel_err"] = [rel(x, y) for x, y in zip(tr["f32"], tr["dmma"])]
        except Exception as ex:  # pragma: no cover
            extra["variant_error"] = repr(ex)
    eng.close()
    del eng
    torch.cuda.empty_cache()

    # ---- parity of the benchmarked path against the oracle (rank-0 CPU leg); multi-GPU consistency at N > 1
    if not a.quick:
        if world == 1:
            extra["parity"] = parity_vs_oracle(torch, dev, a.D, a.q, a.missing, a.ard, a.algo, 32768, 5)
        else:
            extra["multi_gpu_check"] = multi_gpu_check(torch, dist, dev, rank, world, a.D, a.q, a.missing, 65536)

    # ---- BASELINE.json configs[2] at one GPU's share of its rows (N = 10M over 8 GPUs = 1.25M rows per GPU, D = 1024, q = 32,
    # 30 % missing): at --gpus 8 this IS config 3; at fewer GPUs the same per-GPU shard (weak scaling)
    if not a.quick and not a.no_c3 and a.mode == "B":
        try:
            c3 = {"N": 1250000, "D": 1024, "q": 32, "missing": 0.3, "algo": a.algo}
            e3, r3, _ = measure_config(torch, dist, dev, rank, world, local, lib, _cabi, c3, max(3, min(a.steps, 10)), 3,
                                       None, hbm, peak_tf, traffic_json)
            r3["workload"] = ("VB-PCA missing data N=%d (=%d per GPU) D=1024 q=32 30%% missing FP64 mode=B"
                              % (world * c3["N"], c3["N"]))
            e3.close()
            del e3
            torch.cuda.empty_cache()
            if world == 1:
                r3["parity"] = parity_vs_oracle(torch, dev, 1024, 32, 0.3, False, a.algo, 16384, 3)
            else:
                r3["multi_gpu_check"] = multi_gpu_check(torch, dist, dev, rank, world, 1024, 32, 0.3, 32768)
            extra["c3_shard"] = r3
        except Exception as ex:  # pragma: no cover
            extra["c3_shard"] = {"error": repr(ex)}

    # ---- the shape of BASELINE.json configs[3] (ARD, D = 512, q = 64, 30 % missing) at 400k rows: the q = 64 kernels under the same clock
    if world == 1 and not a.quick and not a.no_c4 and a.mode == "B":
        try:
            c4 = {"N": 400000, "D": 512, "q": 64, "missing": 0.3, "algo": a.algo, "ard": True}
            e4, r4, _ = measure_config(torch, dist, dev, rank, world, local, lib, _cabi, c4, max(3, min(a.steps, 10)), 3,
                                       None, hbm, peak_tf, traffic_json)
            r4["workload"] = "VB-PCA missing data with ARD N=400000 D=512 q=64 30% missing FP64 mode=B"
            e4.close()
            del e4
            torch.cuda.empty_cache()
            extra["c4_shape"] = r4
        except Exception as ex:  # pragma: no cover
            extra["c4_shape"] = {"error": repr(ex)}

    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": max(a.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(a), "algo": head["algo"], "rows_total": head["rows_total"],
                           "l2": "inputs larger than L2 (X shard %.2f GB per GPU)" % (a.N * a.D * 8 / 1e9),
                           "parallelism": "rows sharded over %d GPU(s), one exchange of %d doubles per sweep fused into the "
                                          "statistics kernel over NVLink peer memory" % (world, head["stats_len"]),
                           "data": "W_true, mu_true from one seed on every rank; rows (Z, noise, erasures) per rank"},
                "clocks": clocks, "gpu_launches": head["gpu_launches"], "e2e": e2e, "roofline": head["roofline"],
                "kernels": head["kernels"], "elbo_last": head["elbo_last"], "i8_guard_fallbacks": head["i8_guard_fallbacks"]}
        line.update(extra)
        if world == 1 and not a.no_cpu and not a.quick:
            line["cpu_baseline"] = cpu_baseline(a)
        sys.stdout.flush()
        os.write(real_out, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--N", type=int, default=1000000)
    ap.add_argument("--D", type=int, default=256)
    ap.add_argument("--q", type=int, default=16)
    ap.add_argument("--missing", type=float, default=0.2)
    ap.add_argument("--mode", default="B", choices=["A", "B"])
    ap.add_argument("--algo", default="auto", choices=["auto", "generic", "dmma", "i8"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-f32", action="store_true", help="skip the FP32-variant leg")
    ap.add_argument("--no-c3", action="store_true", help="skip the config-3 shard leg")
    ap.add_argument("--quick", action="store_true", help="headline + e2e only (profiling runs)")
    ap.add_argument("--no-c4", dest="no_c4", action="store_true", help="skip the config-4-shape object (q = 64, ARD)")
    ap.add_argument("--ard", action="store_true", help="ARD Gamma precisions per latent column (config 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline's timed sweeps (last state, bounds) to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of our arm (--impl ours)")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
