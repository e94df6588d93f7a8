"""A/B of the INT8 statistics pass with the digit planes made in shared memory (stats_i8_fused_kernel) against
digitize_kernel + stats_i8_kernel (PYVB_I8_FUSED=0, read on every call), in ONE process on one GPU:

  * the card's name, power limit and maximum SM clock;
  * config 2 (N = 1M, D = 256, q = 16, 20 % missing, bench.py's data and seeds): the statistics pass (CUDA events, the
    call bench.py times as stats_ms) and whole sweeps, the two paths alternating for --rounds rounds;
  * bit-for-bit comparison of the two paths from the same initial state: the bound of every sweep, the state, the
    statistics;
  * the config-3 shard (1.25M rows, D = 1024, q = 32) and the config-4 shape (400k rows, D = 512, q = 64, ARD) once per
    setting: both stay on the two-kernel path, so their sweeps must not move.

usage: python tools/stats_fused_ab.py [--rounds 5] [--out DIR]   (prints one JSON document, also written to DIR)"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from pyvb_b200 import PlateEngine  # noqa: E402


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit, max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        out["power_limit, max_sm_clock"] = "unavailable: %s" % ex
    return out


def set_path(fused):
    os.environ["PYVB_I8_FUSED"] = "1" if fused else "0"


def stats_ms(dev, e, n=10):
    def call():
        e._stats_fresh = False
        e._ensure_stats()
    return bench.time_calls(torch, dev, call, n)


def sweep_ms(dev, e, n):
    for _ in range(2):
        e.iterate_async()
    torch.cuda.synchronize(dev)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(n):
        e.iterate_async()
    a1.record()
    torch.cuda.synchronize(dev)
    return a0.elapsed_time(a1) / n


def outputs(e, sweeps=3):
    e.init_random(seed=4321)
    slots = [e.iterate_async() for _ in range(sweeps)]
    torch.cuda.synchronize()
    return {"trace": e.trace[slots].clone(), "MZ": e.MZ.clone(), "logdet": e.logdet.clone(), "stats": e.stats.clone(),
            "Wbar": e.Wbar.clone(), "Wvar": e.Wvar.clone(), "mu": e.mu.clone(), "gl": e.gl.clone()}


def same_bits(a, b):
    return {k: bool(torch.equal(a[k].view(torch.int64), b[k].view(torch.int64))) for k in a}


def config(dev, N, D, q, missing, ard=False):
    X = bench.make_data(torch, N, D, q, missing, 1234, dev)
    e = PlateEngine(X, q, mode="B", algo="auto", keep_sigma=False, device=dev, ard=ard)
    del X
    e.init_random(seed=4321)
    return e


def summary(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=20, help="timed sweeps per round")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card()}

    set_path(True)
    e = config(dev, 1000000, 256, 16, 0.2)
    res["c2_zi_allocated_at_construction"] = e.ZI is not None
    for fused in (True, False):               # warm both paths (ZI is allocated at the first two-kernel call)
        set_path(fused)
        sweep_ms(dev, e, 3)
        stats_ms(dev, e, 3)
    t = {"fused": {"stats_ms": [], "sweep_ms": []}, "two_kernel": {"stats_ms": [], "sweep_ms": []}}
    for r in range(a.rounds):
        for fused in ((True, False) if r % 2 == 0 else (False, True)):
            set_path(fused)
            k = "fused" if fused else "two_kernel"
            t[k]["sweep_ms"].append(sweep_ms(dev, e, a.sweeps))
            t[k]["stats_ms"].append(stats_ms(dev, e))
    res["c2"] = {k: {m: summary(v) for m, v in d.items()} for k, d in t.items()}
    res["c2"]["sweep_speedup_median"] = (res["c2"]["two_kernel"]["sweep_ms"]["median"] /
                                         res["c2"]["fused"]["sweep_ms"]["median"])
    set_path(True)
    of = outputs(e)
    set_path(False)
    oo = outputs(e)
    res["c2_bit_identical"] = same_bits(of, oo)
    res["c2_guard_fallbacks"] = list(e.i8_fallbacks())
    del e, of, oo
    torch.cuda.empty_cache()

    for name, shape in (("c3_shard", (1250000, 1024, 32, 0.2, False)), ("c4_shape", (400000, 512, 64, 0.2, True))):
        set_path(True)
        e = config(dev, *shape)
        res[name] = {"zi_allocated": e.ZI is not None}
        for fused in (True, False):
            set_path(fused)
            res[name]["sweep_ms_" + ("fused_setting" if fused else "two_kernel_setting")] = sweep_ms(dev, e, 5)
        del e
        torch.cuda.empty_cache()
    os.environ.pop("PYVB_I8_FUSED", None)
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "stats_fused_ab.json"), "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
