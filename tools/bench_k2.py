"""Times pyvb_zsolve_f64 (K2 alone, the kernel of each q).  usage: python tools/bench_k2.py [q N]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from pyvb_b200 import _cabi

lib = _cabi.lib()
dev = torch.device("cuda", 0)
cases = [(16, 1000000), (32, 1000000), (64, 400000), (8, 1000000)]
if len(sys.argv) > 2:
    cases = [(int(sys.argv[1]), int(sys.argv[2]))]
for q, N in cases:
    P = q * (q + 1) // 2
    ld, zoff = int(lib.pyvb_mz_pitch(q)), int(lib.pyvb_gw_woff(q))
    g = torch.Generator(device=dev); g.manual_seed(1)
    ii, jj = np.tril_indices(q)
    diag = torch.as_tensor((ii == jj).astype(np.float64), device=dev)
    base = torch.zeros(N, ld, dtype=torch.float64, device=dev)
    base[:, :P] = 0.01 * torch.randn(N, P, generator=g, device=dev, dtype=torch.float64) + 3.0 * diag
    base[:, zoff:zoff + q] = torch.randn(N, q, generator=g, device=dev, dtype=torch.float64)
    logdet = torch.zeros(N, dtype=torch.float64, device=dev)
    gl = torch.zeros(144, dtype=torch.float64, device=dev)
    nz = int(lib.pyvb_zsums_len(N, q))
    zs = torch.zeros(max(nz, 1), dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    ts = []
    for rep in range(4):
        mz = base.clone()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _cabi.check(lib.pyvb_zsolve_f64(N, q, mz.data_ptr(), ld, 0, logdet.data_ptr(), gl.data_ptr(),
                                        zs.data_ptr() if nz else 0, st), "zsolve")
        e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = min(ts[1:])
    fl = N * (q ** 3 + 2.0 * q * q)
    by = N * 2.0 * (zoff + q) * 8
    print("q=%d N=%d %.3f ms  %.2f TF/s  %.0f GB/s  nonpd=%g" % (q, N, ms, fl / ms * 1e-9, by / ms * 1e-6, float(gl[11])),
          flush=True)
