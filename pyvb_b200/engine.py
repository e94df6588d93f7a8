"""Plate engine: device-resident state of the VB-PCA (missing data) model and the update
operators, each one a call into the CUDA C-ABI (include/pyvb_b200.h).

This is the host side of the hot path.  It mirrors, as batched "plate" operators, the
per-node methods of the reference (paths under /root/reference/src/pyvb):

    update_W(i0,i1)  <-  Gaussian.update on W_i          nodes/gaussian.py:102-123 + nodes/nodes_todo.py:43-62
    update_Z(lo,hi)  <-  Gaussian.update on Z_n          nodes/gaussian.py:102-123 + nodes/node.py:182-232
    update_X(lo,hi)  <-  Gaussian.update on partial X_n  nodes/gaussian.py:125-134           (mode A only)
    update_Mu()      <-  Gaussian.update on Mu           nodes/node.py:95-110
    update_Beta()    <-  Gamma.update                    nodes/nodes_todo.py:130-138
    update_Alpha()   <-  Gamma.update on ARD precisions  nodes/nodes_todo.py:130-138
    elbo()           <-  sum of log_lower_bound()        network.py:49
    iterate()        <-  one sweep in Network.learn order network.py:46-48 (SURVEY.md 0.6)

PyTorch is used for device memory, streams and torch.distributed only.  Rows shard across
ranks; the only exchange is one all-reduce(SUM) of the packed statistics buffer per sweep.
There is no CPU fallback: without the CUDA library or a GPU the constructor raises.
"""
import math

import numpy as np
import torch

from . import _cabi
from . import sparse as _sparse
import os

from .dist import PeerExchange, allreduce_stats
import functools

from ._layout import (ALGO_AUTO, ALGO_DMMA, ALGO_F32, ALGO_GENERIC, GL_ALPHA, GL_ALQB, GL_ELBO, GL_I8BAD, GL_I8FALL, GL_LEN,
                      GL_NONPD, GL_QA, GL_QB, GL_TAU, OP_ALPHA, OP_BETA, OP_ELBO, OP_MU, QMAX, StatLayout)

_ALGOS = {"auto": ALGO_AUTO, "generic": ALGO_GENERIC, "dmma": ALGO_DMMA}


def _digamma(x):
    try:
        from scipy import special
        return float(special.digamma(x))
    except Exception:  # pragma: no cover
        return float(torch.special.digamma(torch.tensor(x, dtype=torch.float64)))


def _on_device(fn):
    """Run a method with the engine's GPU as the current CUDA device: the C-ABI launches on the current device, while the
    tensors and the stream belong to self.device."""
    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapper


def tril_pack_index(q):
    ii, jj = np.tril_indices(q)
    return ii, jj


class PlateEngine(object):
    """VB-PCA plate on one GPU (one process per GPU; rows sharded when torch.distributed is up).

    Parameters
    ----------
    X : (N, D) array or tensor, NaN = missing.  The local row shard.
        Or a sparse matrix (scipy.sparse, any format; torch sparse CSR, host or device): the STORED entries are the
        observations (a stored zero is an observed 0), everything not stored is missing.  Sparse input runs the CSR
        gather kernels (kernels_sparse.cu): mode "B", precision "f64", q in {8, 16, 32, 64}, algo "auto", any D.
    q : latent dimension (<= 64)
    mode : "B" masked/marginalised (throughput path) or "A" reference-exact imputation
    distributed : all-reduce the statistics over torch.distributed's default group
    row_offset : global index of local row 0 (mode A treats global row 0 specially)
    """

    def __init__(self, X, q, mode="B", alpha0=1e-3, alpha_mu=1e-3, a0=1e-3, b0=1e-3, ard=False,
                 ard_a0=1e-3, ard_b0=1e-3, P0=None, m0=None, device=None, algo="auto",
                 keep_sigma=True, distributed=False, row_offset=0, trace_len=4096, precision="f64"):
        if not torch.cuda.is_available():
            raise RuntimeError("pyvb_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _cabi.lib()
        assert mode in ("A", "B")
        assert 1 <= q <= QMAX, "latent dimension must be in [1, %d]" % QMAX
        assert precision in ("f64", "f32")
        self.f32 = (precision == "f32")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(self.device):
            self._construct(X, q, mode, alpha0, alpha_mu, a0, b0, ard, ard_a0, ard_b0, P0, m0, algo, keep_sigma,
                            distributed, row_offset, trace_len)

    def _construct(self, X, q, mode, alpha0, alpha_mu, a0, b0, ard, ard_a0, ard_b0, P0, m0, algo, keep_sigma,
                   distributed, row_offset, trace_len):
        self.mode, self.q, self.ard = mode, int(q), bool(ard)
        self.sparse = _sparse.is_sparse(X)
        if self.sparse:
            if mode != "B":
                raise ValueError("sparse input needs mode='B' (mode A imputes every missing entry: pass a dense array)")
            if self.f32:
                raise ValueError("sparse input needs precision='f64'")
            if int(q) not in (8, 16, 32, 64):
                raise ValueError("sparse input needs q in (8, 16, 32, 64), got %d" % int(q))
            if algo != "auto":
                raise ValueError("sparse input needs algo='auto' (the CSR kernels are the only sparse path)")
        # algo "i8": the mask contraction of the Z step on the INT8 tensor cores (exact, kernels_i8.cu); the rest as "dmma".
        # "auto" picks it when the shape allows (PYVB_I8=0 keeps the all-DMMA path)
        self.use_i8 = (algo == "i8")
        if algo == "i8":
            algo = "dmma"
        elif algo == "auto" and mode == "B" and not self.f32 and os.environ.get("PYVB_I8", "1") != "0":
            self.use_i8 = None                                  # decided below, once D is known
        self.algo = _ALGOS[algo] if isinstance(algo, str) else int(algo)
        self.distributed = bool(distributed)
        self.row_offset = int(row_offset)
        f64 = torch.float64
        dev = self.device
        if self.sparse:
            self.csr = _sparse.to_csr(X, device=dev)         # validated: finite values, no duplicates, columns in [0, D)
            self.N, self.D = self.csr.N, self.csr.D
        else:
            Xt = torch.as_tensor(X)
            assert Xt.dim() == 2
            Xt = Xt.to(device=dev, dtype=f64).contiguous()
            self.N, self.D = int(Xt.shape[0]), int(Xt.shape[1])
        N, D = self.N, self.D
        self.P = q * (q + 1) // 2
        self.L = StatLayout(D, q)
        self.alpha0, self.alpha_mu = float(alpha0), float(alpha_mu)
        self.a0, self.b0 = float(a0), float(b0)
        self.ard_a0, self.ard_b0 = float(ard_a0), float(ard_b0)

        # ---- data
        obs = None if self.sparse else ~torch.isnan(Xt)
        n_obs_local = int(self.csr.values.numel()) if self.sparse else int(obs.sum().item())
        if self.sparse:
            # the statistics read the entries column-major per row block (K3-csc); the X-only sums are taken once, here
            self.csc = _sparse.block_csc(self.csr, int(self.lib.pyvb_csr_block_rows(N, D, q)))
            self.xcache_sparse = _sparse.x_cache(self.csr).to(dev)
            self.Xorig, self.X, self.V, self.qldX = None, None, None, None
            n_eff_local = n_obs_local
        elif self.f32:
            # FP32 variant (tcgen05): the data live as three bf16 planes (mask | x_h | x_m); the sums that depend on
            # X alone are taken once, here, in FP64
            if mode != "B" or not self.lib.pyvb_f32_supported(self.D, q) or q not in (16, 32):
                raise ValueError("precision='f32' needs mode B, q in (16, 32) and D % 32 == 0")
            x0 = torch.where(obs, Xt, torch.zeros((), dtype=f64, device=dev))
            self.xcache = torch.cat([obs.sum(0).to(f64), x0.sum(0), (x0 * x0).sum().reshape(1),
                                     torch.tensor([float(n_obs_local)], dtype=f64, device=dev)]).contiguous()
            del x0
            self.planes = torch.zeros(3, N, D, dtype=torch.bfloat16, device=dev)
            _cabi.check(self.lib.pyvb_prepare_x_f32(N, D, Xt.data_ptr(), D, self.planes.data_ptr(), self._stream()),
                        "pyvb_prepare_x_f32")
            torch.cuda.current_stream(dev).synchronize()
            self.Xorig, self.X, self.V, self.qldX = None, None, None, None
            n_eff_local = n_obs_local
        elif mode == "A":
            self.Xorig = Xt
            self.X = torch.where(obs, Xt, torch.zeros((), dtype=f64, device=dev)).contiguous()   # Xhat
            self.V = torch.where(obs, torch.zeros((), dtype=f64, device=dev),
                                 torch.ones((), dtype=f64, device=dev)).contiguous()
            self.qldX = torch.zeros(N, dtype=f64, device=dev)
            n_eff_local = N * D               # nodes_todo.py:125-128: every child counts dim/2
        else:
            self.Xorig = None
            self.X = Xt
            self.V = None
            self.qldX = None
            n_eff_local = n_obs_local
        del obs
        i8_ok = bool(self.lib.pyvb_i8_supported(D, q)) and mode == "B" and not self.f32 and not self.sparse
        if self.use_i8 is None:
            self.use_i8 = i8_ok
        elif self.use_i8 and not i8_ok:
            raise ValueError("algo='i8' needs mode B, FP64, q in (16, 32, 64), D % 64 == 0 and D <= ~1280")
        if self.use_i8:
            self.mask8 = torch.empty(int(self.lib.pyvb_i8_mask_bytes(N, D)), dtype=torch.int8, device=dev)
            self.GI = torch.empty(int(self.lib.pyvb_i8_digits_bytes(D, q)), dtype=torch.int8, device=dev)
            self.gscale = torch.empty(int(self.lib.pyvb_i8_ncols(q)), dtype=f64, device=dev)
        self._mask_valid = False
        # ... and the mask-type statistics (K3-i8): transposed mask + digit planes of the MZ rows
        self.use_i8_stats = bool(self.use_i8 and self.lib.pyvb_stats_i8_supported(D, q)
                                 and os.environ.get("PYVB_I8_STATS", "1") != "0")
        self._maskT_valid = False
        n_eff = self._allreduce_scalar(float(n_eff_local))
        self.n_rows_total = int(self._allreduce_scalar(float(N)))

        # ---- latent state
        # <zz^T> (packed) and <z> interleaved in one array: one TMA tile feeds the statistics GEMM
        if self.f32:
            # FP32 rows [zbar (q) | <zz^T> packed (P) | pad] + their three-way bf16 split (B operand of the statistics)
            self.ldmz = int(self.lib.pyvb_f32_pitch(q))
            self.zoff, self.poff = int(self.lib.pyvb_f32_zoff(q)), int(self.lib.pyvb_f32_poff(q))
            self.MZ = torch.zeros(N, self.ldmz, dtype=torch.float32, device=dev)
            self.MP = torch.zeros(3, N, self.ldmz, dtype=torch.bfloat16, device=dev)
            self.GT = torch.zeros(3, self.ldmz, D, dtype=torch.bfloat16, device=dev)
            self.WT = torch.zeros(3, q, D, dtype=torch.bfloat16, device=dev)
        else:
            self.ldmz = int(self.lib.pyvb_mz_pitch(q))
            self.zoff, self.poff = int(self.lib.pyvb_gw_woff(q)), 0
            self.MZ = torch.zeros(N, self.ldmz, dtype=f64, device=dev)
        self.M2 = self.MZ[:, self.poff:self.poff + self.P]
        self.Zbar = self.MZ[:, self.zoff:self.zoff + q]
        self.Sig = torch.zeros(N, self.P, dtype=f64, device=dev) if keep_sigma else None
        self.logdet = torch.ones(N, dtype=f64, device=dev)
        self.Wbar = torch.zeros(D, q, dtype=f64, device=dev)
        self.Wvar = torch.ones(D, q, dtype=f64, device=dev)
        self.mu = torch.zeros(D, dtype=f64, device=dev)
        self.muvar = torch.ones(D, dtype=f64, device=dev)
        self.ldg = int(self.lib.pyvb_gw_pitch(q))
        self.Gw = torch.zeros(D, self.ldg, dtype=f64, device=dev)
        self.stats = torch.zeros(self.L.len, dtype=f64, device=dev)
        assert self.L.len == int(self.lib.pyvb_stats_len(D, q))
        self.ws_bytes = int(self.lib.pyvb_stats_workspace_bytes(N, D, q, ALGO_F32 if self.f32 else self.algo))
        if self.sparse:
            self.ws_bytes = int(self.lib.pyvb_stats_csr_workspace_bytes(N, D, q, self.csc.nblk))
        if self.use_i8_stats:
            # the digit planes cost 7 bytes per MZ entry: when they would take more than 40 % of the free memory (config 4
            # at full size on one GPU) the statistics stay on the FP64 tensor cores.  At D <= 256 they are made in shared
            # memory (pyvb_stats_i8_fused) and only the transposed mask is allocated.
            fused = bool(self.lib.pyvb_stats_i8_fused(D, q))
            need = int(self.lib.pyvb_stats_i8_maskt_bytes(N, D)) + (0 if fused else int(self.lib.pyvb_stats_i8_digits_bytes(N, q)))
            if need > 0.4 * torch.cuda.mem_get_info(dev)[0]:
                self.use_i8_stats = False
        if self.use_i8_stats:
            try:
                self.npad = int(self.lib.pyvb_stats_i8_npad(N))
                self.maskT = torch.empty(int(self.lib.pyvb_stats_i8_maskt_bytes(N, D)), dtype=torch.int8, device=dev)
                self.ZI = None if fused else torch.empty(int(self.lib.pyvb_stats_i8_digits_bytes(N, q)), dtype=torch.int8,
                                                         device=dev)
                # (zeros: the tail of the scratch is the guard block -- counters of the accuracy check -- see the header)
                self.i8_scratch = torch.zeros(int(self.lib.pyvb_stats_i8_scratch_len(q)), dtype=f64, device=dev)
                self.ws_bytes = max(self.ws_bytes, int(self.lib.pyvb_stats_i8_workspace_bytes(N, D, q)))
            except torch.cuda.OutOfMemoryError:          # the digit planes are 7 bytes per MZ entry: DMMA statistics instead
                self.maskT = self.ZI = self.i8_scratch = None
                self.use_i8_stats = False
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        if self.sparse:
            self.xcache = self.xcache_sparse
            self._xcache_valid = True
            nz = int(self.lib.pyvb_zsums_len(N, q))
            self.zsums = torch.zeros(nz, dtype=f64, device=dev) if nz > 0 else None
        elif self.f32:
            self._xcache_valid = True
            nz = int(self.lib.pyvb_zsums_len_f32(N, q))
            self.zsums = torch.zeros(nz, dtype=f64, device=dev)
        else:
            self.xcache = torch.zeros(2 * D + 2, dtype=f64, device=dev) if mode == "B" else None
            self._xcache_valid = False
            # per-CTA column sums of the MZ rows left by the batched solve (K2) of a full-range Z update
            nz = int(self.lib.pyvb_zsums_len(N, q)) if self.lib.pyvb_algo_supported(ALGO_DMMA, D, q) else 0
            self.zsums = (torch.zeros(nz, dtype=f64, device=dev)
                          if nz > 0 and self.algo in (ALGO_AUTO, ALGO_DMMA) else None)
        self._zsums_valid = False
        # multi-GPU: the all-reduce happens inside the statistics kernel over NVLink peer memory
        # (PYVB_COMM=nccl: plain torch.distributed all_reduce instead, for comparison)
        self.peers = None
        if self.distributed and os.environ.get("PYVB_COMM", "peer") == "peer":
            import torch.distributed as dist
            if dist.get_world_size() > 1 and dist.get_backend() == "nccl":
                self.peers = PeerExchange(self.lib, self.L.len, dev)
        self.gl = torch.zeros(GL_LEN, dtype=f64, device=dev)
        self.trace = torch.zeros(int(trace_len), dtype=f64, device=dev)
        self.trace_pos = 0

        # ---- priors
        P0 = np.eye(q) if P0 is None else np.asarray(P0, dtype=np.float64).reshape(q, q)
        m0 = np.zeros(q) if m0 is None else np.asarray(m0, dtype=np.float64).reshape(q)
        self.P0 = torch.as_tensor(P0, dtype=f64).contiguous().to(dev)
        self.h0 = torch.as_tensor(P0 @ m0, dtype=f64).contiguous().to(dev)
        qa = self.a0 + 0.5 * n_eff
        al_qa = self.ard_a0 + 0.5 * D
        c = _cabi.Consts()
        c.alpha_mu, c.a0, c.b0 = self.alpha_mu, self.a0, self.b0
        c.psi_qa, c.lgam_qa, c.lgam_a0 = _digamma(qa), math.lgamma(qa), math.lgamma(self.a0)
        c.ard_a0, c.ard_b0, c.al_qa = self.ard_a0, self.ard_b0, al_qa
        c.psi_alqa, c.lgam_alqa, c.lgam_ard_a0 = _digamma(al_qa), math.lgamma(al_qa), math.lgamma(self.ard_a0)
        c.lndet_P0 = float(np.linalg.slogdet(P0)[1])
        c.m0P0m0 = float(m0 @ P0 @ m0)
        c.ard, c.mode_a = int(self.ard), int(mode == "A")
        self.consts = c
        self.qa, self.al_qa = qa, al_qa

        # deterministic stand-in initialisation (SURVEY 8d); parity runs call set_state()
        self.set_state({"qb": 0.5, "al_qb": np.ones(q)})
        self._stats_fresh = False
        self._gw_fresh = False

    @_on_device
    def close(self):
        """Release the peer exchange buffers (collective: every rank must call it)."""
        if self.peers is not None:
            self.peers.close()
            self.peers = None

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _allreduce_scalar(self, v):
        if self.distributed:
            import torch.distributed as dist
            t = torch.tensor([v], dtype=torch.float64, device=self.device)
            dist.all_reduce(t)
            return float(t.item())
        return v

    @staticmethod
    def _p(t):
        return 0 if t is None else t.data_ptr()

    # ------------------------------------------------------------------ state io
    @_on_device
    def set_state(self, st):
        """Inject state (numpy arrays in the oracle's layout: Sig is (N,q,q), qb scalar ...)."""
        f64, dev = torch.float64, self.device
        q = self.q

        def put(dst, src):
            dst.copy_(torch.as_tensor(np.ascontiguousarray(src), dtype=f64).reshape(dst.shape).to(dev))

        for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar"):
            if k in st:
                put(getattr(self, k), st[k])
        if "Xhat" in st and self.mode == "A":
            put(self.X, st["Xhat"])
        if "V" in st and self.mode == "A":
            put(self.V, st["V"])
        if "Sig" in st or "Zbar" in st:
            ii, jj = tril_pack_index(q)
            if "Sig" in st:
                sig = np.asarray(st["Sig"], dtype=np.float64)[:, ii, jj]
                sig_t = torch.as_tensor(np.ascontiguousarray(sig), dtype=f64).to(dev)
            elif self.Sig is not None:
                sig_t = self.Sig
            else:
                raise ValueError("Sig needed")
            if self.Sig is not None:
                self.Sig.copy_(sig_t)
            it, jt = torch.as_tensor(ii, device=dev), torch.as_tensor(jj, device=dev)
            zb = self.Zbar.to(f64)
            self.M2.copy_(sig_t + zb[:, it] * zb[:, jt])
        if self.f32:
            self._resplit()
        gl = self.gl.cpu()
        gl[GL_QA] = self.qa
        gl[GL_NONPD] = 0.0                      # a fresh state: earlier non-PD rows are history
        if "qb" in st:
            gl[GL_QB] = float(st["qb"])
        gl[GL_TAU] = gl[GL_QA] / gl[GL_QB]
        if self.ard:
            if "al_qb" in st:
                gl[GL_ALQB:GL_ALQB + q] = torch.as_tensor(np.asarray(st["al_qb"], dtype=np.float64).reshape(q))
            gl[GL_ALPHA:GL_ALPHA + q] = self.al_qa / gl[GL_ALQB:GL_ALQB + q]
        else:
            gl[GL_ALPHA:GL_ALPHA + q] = self.alpha0
        self.gl.copy_(gl.to(dev))
        self._stats_fresh = False
        self._gw_fresh = False
        self._zsums_valid = False

    def _resplit(self, step=1 << 16):
        """FP32 variant: refresh the bf16 x 3 planes after the FP32 rows were written from outside the kernels."""
        for lo in range(0, self.N, step):
            v = self.MZ[lo:lo + step]
            h = v.to(torch.bfloat16)
            r = v - h.float()
            m = r.to(torch.bfloat16)
            self.MP[0, lo:lo + step] = h
            self.MP[1, lo:lo + step] = m
            self.MP[2, lo:lo + step] = (r - m.float()).to(torch.bfloat16)

    def _zsums_from_state(self):
        """FP32 variant: the column sums K2 would have left, from an injected state (one partial, rest zero)."""
        kw = int(self.lib.pyvb_zsums_kw(self.q))
        z = self.zsums.view(-1, kw)
        z.zero_()
        pp = int(self.lib.pyvb_gw_woff(self.q))
        z[0, :self.P] = self.M2.to(torch.float64).sum(0)
        z[0, pp:pp + self.q] = self.Zbar.to(torch.float64).sum(0)
        z[0, pp + self.q] = (0.5 / self.logdet).sum()
        z[0, pp + self.q + 1] = self.logdet.sum()
        z[0, pp + self.q + 2] = float(self.N)
        self._zsums_valid = True

    @_on_device
    def init_random(self, seed=1234, rank=0):
        """Scale-run initialisation on the device (SURVEY 8d): Wbar ~ N(0,1) (same on every rank),
        Zbar ~ N(0,1) (per-rank stream), Wvar = 1, Sigma = I, mu = 0, qb = 0.5."""
        dev, q, P = self.device, self.q, self.P
        g = torch.Generator(device=dev)
        g.manual_seed(int(seed))
        self.Wbar.normal_(generator=g)
        self.Wvar.fill_(1.0)
        self.mu.zero_()
        self.muvar.fill_(1.0)
        g.manual_seed(int(seed) + 1 + int(rank))
        self.Zbar.normal_(generator=g)
        ii, jj = tril_pack_index(q)
        it, jt = torch.as_tensor(ii, device=dev), torch.as_tensor(jj, device=dev)
        eye = (it == jt).to(torch.float64)
        step = 1 << 16
        for lo in range(0, self.N, step):
            z = self.Zbar[lo:lo + step].to(torch.float64)
            self.M2[lo:lo + step] = (z[:, it] * z[:, jt] + eye).to(self.M2.dtype)
            if self.Sig is not None:
                self.Sig[lo:lo + step] = eye
        self.logdet.fill_(1.0)
        self.set_state({"qb": 0.5, "al_qb": np.ones(q)})

    @_on_device
    def set_X(self, X):
        """Replace the (mode B) data shard, e.g. from pinned host memory; invalidates the cached X sums."""
        if self.sparse:
            raise NotImplementedError("set_X: a sparse engine keeps its entries in the layouts built at construction; "
                                      "build a new engine for new data")
        assert self.mode == "B" and not self.f32
        self.X.copy_(X, non_blocking=True)
        self._xcache_valid = False
        self._mask_valid = False
        self._maskT_valid = False
        self._stats_fresh = False

    def get_state(self):
        """Host copy of the state in the oracle's layout."""
        q = self.q
        ii, jj = tril_pack_index(q)
        out = {k: getattr(self, k).contiguous().to(torch.float64).cpu().numpy()
               for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar")}
        N = self.N
        if self.Sig is not None:
            sp = self.Sig.cpu().numpy()
        else:
            z = out["Zbar"]
            sp = self.M2.contiguous().to(torch.float64).cpu().numpy() - z[:, ii] * z[:, jj]
        Sig = np.zeros((N, q, q))
        Sig[:, ii, jj] = sp
        Sig[:, jj, ii] = sp
        out["Sig"] = Sig
        if self.mode == "A":
            out["Xhat"] = self.X.cpu().numpy()
            out["V"] = self.V.cpu().numpy()
        gl = self.gl.cpu().numpy()
        out["qa"], out["qb"], out["tau"] = float(gl[GL_QA]), float(gl[GL_QB]), float(gl[GL_TAU])
        out["alpha"] = gl[GL_ALPHA:GL_ALPHA + q].copy()
        out["al_qb"] = gl[GL_ALQB:GL_ALQB + q].copy()
        return out

    def get_row(self, i):
        """Host copy of ONE row of the plate (O(q^2 + D), no pass over the other rows): zbar_i, Sigma_i and, in mode A,
        <x_i> and its variances."""
        q = self.q
        ii, jj = tril_pack_index(q)
        z = self.Zbar[i].contiguous().to(torch.float64).cpu().numpy()
        if self.Sig is not None:
            sp = self.Sig[i].cpu().numpy()
        else:
            sp = self.M2[i].contiguous().to(torch.float64).cpu().numpy() - z[ii] * z[jj]
        Sig = np.zeros((q, q))
        Sig[ii, jj] = sp
        Sig[jj, ii] = sp
        out = {"Zbar": z, "Sig": Sig}
        if self.mode == "A":
            out["Xhat"] = self.X[i].cpu().numpy()
            out["V"] = self.V[i].cpu().numpy()
        return out

    def get_state_small(self):
        """Host copy of the replicated (row-independent) state only."""
        gl = self.gl.cpu().numpy()
        return {"Wbar": self.Wbar.cpu().numpy(), "Wvar": self.Wvar.cpu().numpy(), "mu": self.mu.cpu().numpy(),
                "muvar": self.muvar.cpu().numpy(), "qa": float(gl[GL_QA]), "qb": float(gl[GL_QB]),
                "tau": float(gl[GL_TAU]), "alpha": gl[GL_ALPHA:GL_ALPHA + self.q].copy(),
                "al_qb": gl[GL_ALQB:GL_ALQB + self.q].copy()}

    def check(self):
        """Raise LinAlgError if any posterior precision was not positive definite (gaussian.py:118)."""
        bad = float(self.gl[GL_NONPD].item())
        if bad > 0:
            self.gl[GL_NONPD] = 0.0             # reported once; a state injected afterwards starts clean
            raise np.linalg.LinAlgError("posterior precision of %d row(s) is not positive definite" % int(bad))

    def i8_fallbacks(self):
        """How often the accuracy guard of the INT8 path sent a step to the FP64 tensor cores: (Z steps, statistics passes)."""
        z = float(self.gl[GL_I8FALL].item())
        s = 0.0
        if getattr(self, "i8_scratch", None) is not None:
            s = float(self.i8_scratch[int(self.lib.pyvb_stats_i8_guard_offset(self.q)) + 1].item())
        return int(z), int(s)

    # ------------------------------------------------------------------ operators
    @_on_device
    def _ensure_gw(self):
        if not self._gw_fresh and self.f32:
            rc = self.lib.pyvb_pack_gw_f32(self.D, self.q, self.Wbar.data_ptr(), self.Wvar.data_ptr(),
                                           self.mu.data_ptr(), self.GT.data_ptr(), self.WT.data_ptr(), self._stream())
            _cabi.check(rc, "pyvb_pack_gw_f32")
            self._gw_fresh = True
        if not self._gw_fresh:
            rc = self.lib.pyvb_pack_gw_f64(self.D, self.q, self.Wbar.data_ptr(), self.Wvar.data_ptr(),
                                           self.mu.data_ptr(), self.Gw.data_ptr(), self.ldg, self._stream())
            _cabi.check(rc, "pyvb_pack_gw_f64")
            self._gw_fresh = True

    @_on_device
    def _ensure_stats(self):
        if self._stats_fresh:
            return
        if self.sparse:
            c = self.csc
            rc = self.lib.pyvb_stats_csr_f64(self.N, self.D, self.q, c.nblk, c.colptr.data_ptr(), c.rows.data_ptr(),
                                             c.vals.data_ptr(), self.MZ.data_ptr(), self.ldmz, self.logdet.data_ptr(),
                                             self.stats.data_ptr(), self.ws.data_ptr(), self.ws_bytes,
                                             self.xcache.data_ptr(),
                                             self.zsums.data_ptr() if (self.zsums is not None and self._zsums_valid) else 0,
                                             self.peers.next() if (self.peers is not None and self.distributed) else None,
                                             self._stream())
            _cabi.check(rc, "pyvb_stats_csr_f64")
            if self.distributed and self.peers is None:
                allreduce_stats(self.stats)
            self._stats_fresh = True
            return
        if self.f32:
            if not self._zsums_valid and self.N > 0:
                self._zsums_from_state()
            rc = self.lib.pyvb_stats_f32(self.N, self.N, self.D, self.q, self.planes.data_ptr(), self.MP.data_ptr(),
                                         self.stats.data_ptr(), self.ws.data_ptr(), self.ws_bytes,
                                         self.xcache.data_ptr(), self.zsums.data_ptr(),
                                         self.peers.next() if (self.peers is not None and self.distributed) else None,
                                         self._stream())
            _cabi.check(rc, "pyvb_stats_f32")
            if self.distributed and self.peers is None:
                allreduce_stats(self.stats)
            self._stats_fresh = True
            return
        if self.use_i8_stats and self._xcache_valid and self.N > 0:
            if not self._maskT_valid:
                _cabi.check(self.lib.pyvb_prepare_maskt_i8(self.N, self.D, self.X.data_ptr(), self.D,
                                                           self.maskT.data_ptr(), self._stream()), "pyvb_prepare_maskt_i8")
                self._maskT_valid = True
            if self.ZI is None and not self.lib.pyvb_stats_i8_fused(self.D, self.q):    # PYVB_I8_FUSED=0 set since
                self.ZI = torch.empty(int(self.lib.pyvb_stats_i8_digits_bytes(self.N, self.q)), dtype=torch.int8,
                                      device=self.MZ.device)
            rc = self.lib.pyvb_stats_i8_f64(self.N, self.D, self.q, self.X.data_ptr(), self.D, self.maskT.data_ptr(),
                                            self.MZ.data_ptr(), self.ldmz, self.logdet.data_ptr(), self._p(self.ZI),
                                            self.i8_scratch.data_ptr(), self.stats.data_ptr(), self.ws.data_ptr(),
                                            self.ws_bytes, self.xcache.data_ptr(),
                                            self.zsums.data_ptr() if (self.zsums is not None and self._zsums_valid) else 0,
                                            self.peers.next() if (self.peers is not None and self.distributed) else None,
                                            self._stream())
            _cabi.check(rc, "pyvb_stats_i8_f64")
            self.i8_stats_calls = getattr(self, "i8_stats_calls", 0) + 1
            if self.distributed and self.peers is None:
                allreduce_stats(self.stats)
            self._stats_fresh = True
            return
        rc = self.lib.pyvb_stats_f64(self.N, self.D, self.q, self.X.data_ptr(), self.D, self._p(self.V),
                                     self._p(self.Xorig), self._p(self.qldX), self.Zbar.data_ptr(), self.ldmz,
                                     self.M2.data_ptr(), self.ldmz, self.logdet.data_ptr(), self.stats.data_ptr(),
                                     self.ws.data_ptr(), self.ws_bytes, self._p(self.xcache),
                                     int(self._xcache_valid), self._p(self.zsums), int(self._zsums_valid),
                                     self.peers.next() if (self.peers is not None and self.distributed) else None,
                                     self.algo, self._stream())
        _cabi.check(rc, "pyvb_stats_f64")
        self._xcache_valid = self.xcache is not None
        if self.distributed and self.peers is None:
            allreduce_stats(self.stats)          # fallback exchange: NCCL all-reduce
        self._stats_fresh = True

    @_on_device
    def update_W(self, col_lo=0, col_hi=None):
        col_hi = self.q if col_hi is None else col_hi
        self._ensure_stats()
        rc = self.lib.pyvb_wupdate_f64(self.D, self.q, col_lo, col_hi, self.stats.data_ptr(), self.mu.data_ptr(),
                                       self.gl.data_ptr(), self.Wbar.data_ptr(), self.Wvar.data_ptr(),
                                       self._stream())
        _cabi.check(rc, "pyvb_wupdate_f64")
        self._gw_fresh = False

    @_on_device
    def update_Z(self, lo=0, hi=None, _chunk_zsums=False):
        hi = self.N if hi is None else hi
        self._stats_fresh = False
        if hi <= lo:
            return
        self._ensure_gw()
        q, P, D = self.q, self.P, self.D
        sig = 0 if self.Sig is None else self.Sig.data_ptr() + lo * P * 8
        if self.sparse:
            # any row range: K1-csr owns whole rows, so [lo, hi) is a pointer offset into the row offsets
            full = (lo == 0 and hi == self.N and self.zsums is not None)
            self._zsums_valid = False
            rc = self.lib.pyvb_zstep_csr_f64(hi - lo, D, q, self.csr.indptr.data_ptr() + lo * 8,
                                             self.csr.indices.data_ptr(), self.csr.values.data_ptr(), self.Gw.data_ptr(),
                                             self.ldg, self.P0.data_ptr(), self.h0.data_ptr(), self.gl.data_ptr(),
                                             self.MZ.data_ptr() + lo * self.ldmz * 8, self.ldmz, sig,
                                             self.logdet.data_ptr() + lo * 8, self.zsums.data_ptr() if full else 0,
                                             self._stream())
            _cabi.check(rc, "pyvb_zstep_csr_f64")
            self._zsums_valid = full
            return
        if self.f32:
            full = (lo == 0 and hi == self.N)
            if not full and not self._zsums_valid:
                pass                                        # the sums are rebuilt from the state before the next statistics
            self._zsums_valid = False
            rc = self.lib.pyvb_zstep_f32(hi - lo, self.N, D, q, self.planes.data_ptr() + lo * D * 2, self.GT.data_ptr(),
                                         self.WT.data_ptr(), self.P0.data_ptr(), self.h0.data_ptr(), self.gl.data_ptr(),
                                         self.MZ.data_ptr() + lo * self.ldmz * 4, self.MP.data_ptr() + lo * self.ldmz * 2,
                                         sig, self.logdet.data_ptr() + lo * 8, self.zsums.data_ptr() if full else 0,
                                         self._stream())
            _cabi.check(rc, "pyvb_zstep_f32")
            self._zsums_valid = full
            return
        full = (lo == 0 and hi == self.N and self.zsums is not None and self.algo in (ALGO_AUTO, ALGO_DMMA))
        # (_chunk_zsums: iterate_from_host takes the K2 partials of a row chunk for that chunk's statistics)
        zs = self.zsums.data_ptr() if ((full or _chunk_zsums) and self.zsums is not None) else 0
        if zs and int(self.lib.pyvb_zsums_len(self.N, q)) > self.zsums.numel():
            # (PYVB_K2 picks the batched-solve kernel per call; its partial layout must be the one this buffer was sized for)
            raise RuntimeError("the K2 partial buffer was sized for another batched-solve kernel (PYVB_K2 changed?)")
        self._zsums_valid = False
        if self.use_i8 and lo % 128 == 0:                   # (the int8 mask is tiled by 128 rows: other offsets take the DMMA path)
            if not self._mask_valid:                        # the int8 mask follows X (static in mode B)
                rc = self.lib.pyvb_prepare_mask_i8(hi - lo, D, self.X.data_ptr() + lo * D * 8, D,
                                                   self.mask8.data_ptr() + lo * D, self._stream())
                _cabi.check(rc, "pyvb_prepare_mask_i8")
                self._mask_valid = (lo == 0 and hi == self.N)
            rc = self.lib.pyvb_zstep_i8_f64(hi - lo, D, q, self.X.data_ptr() + lo * D * 8, D,
                                            self.mask8.data_ptr() + lo * D, self.Wbar.data_ptr(), self.Wvar.data_ptr(),
                                            self.Gw.data_ptr(), self.ldg, self.P0.data_ptr(), self.h0.data_ptr(),
                                            self.gl.data_ptr(), self.MZ.data_ptr() + lo * self.ldmz * 8, self.ldmz,
                                            self.GI.data_ptr(), self.gscale.data_ptr(), sig,
                                            self.logdet.data_ptr() + lo * 8, zs, 0, self._stream())
            _cabi.check(rc, "pyvb_zstep_i8_f64")
            self._zsums_valid = full
            return
        rc = self.lib.pyvb_zstep_f64(hi - lo, D, q, self.X.data_ptr() + lo * D * 8, D, self.Gw.data_ptr(),
                                     self.ldg, self.P0.data_ptr(), self.h0.data_ptr(), self.gl.data_ptr(),
                                     self.Zbar.data_ptr() + lo * self.ldmz * 8, self.ldmz,
                                     self.M2.data_ptr() + lo * self.ldmz * 8, self.ldmz, sig,
                                     self.logdet.data_ptr() + lo * 8, zs, self.algo, self._stream())
        _cabi.check(rc, "pyvb_zstep_f64")
        self._zsums_valid = full
        self._stats_fresh = False

    @_on_device
    def update_X(self, lo=0, hi=None):
        """Mode A imputation of rows [lo,hi) that are not fully observed; no-op in mode B."""
        if self.mode != "A":
            return
        hi = self.N if hi is None else hi
        self._stats_fresh = False          # before the early return: every rank must redo the all-reduce
        if hi <= lo:
            return
        q, D = self.q, self.D
        rc = self.lib.pyvb_impute_f64(hi - lo, D, q, self.Xorig.data_ptr() + lo * D * 8, D, self.Wbar.data_ptr(),
                                      self.mu.data_ptr(), self.Zbar.data_ptr() + lo * self.ldmz * 8, self.ldmz,
                                      self.gl.data_ptr(),
                                      self.X.data_ptr() + lo * D * 8, self.V.data_ptr() + lo * D * 8,
                                      self.qldX.data_ptr() + lo * 8, self._stream())
        _cabi.check(rc, "pyvb_impute_f64")
        self._stats_fresh = False

    @_on_device
    def _global(self, ops, elbo_out=0, col_lo=0, col_hi=None):
        self._ensure_stats()
        col_hi = self.q if col_hi is None else col_hi
        rc = self.lib.pyvb_global_f64(self.D, self.q, ops, col_lo, col_hi, self.stats.data_ptr(), self.Wbar.data_ptr(),
                                      self.Wvar.data_ptr(), self.mu.data_ptr(), self.muvar.data_ptr(),
                                      self.gl.data_ptr(), self.P0.data_ptr(), self.h0.data_ptr(),
                                      _cabi.ctypes.byref(self.consts), elbo_out, self._stream())
        _cabi.check(rc, "pyvb_global_f64")
        if ops & OP_MU:
            self._gw_fresh = False

    def update_Mu(self):
        self._global(OP_MU)

    def update_Beta(self):
        self._global(OP_BETA)

    def update_Alpha(self, col_lo=0, col_hi=None):
        if self.ard:
            self._global(OP_ALPHA, 0, col_lo, col_hi)

    def elbo_async(self):
        """Evaluate the bound into the device trace; returns the trace slot (no host sync)."""
        slot = self.trace_pos % self.trace.numel()
        self._global(OP_ELBO, self.trace.data_ptr() + slot * 8)
        self.trace_pos += 1
        return slot

    def elbo(self):
        slot = self.elbo_async()
        return float(self.trace[slot].item())

    # ------------------------------------------------------------------ sweeps
    def iterate_async(self):
        """One sweep in the reference's order (SURVEY 0.6): W cols, Z rows, [Alpha], X_0, Mu, X_1.., Beta,
        then the ELBO -- with no host synchronisation.  Returns the trace slot of the bound."""
        self.update_W()
        self.update_Z()
        if self.mode == "A":
            self.update_Alpha()
            self.update_X(0, 1 if self.row_offset == 0 else 0)   # global row 0 lives on the first shard
            self.update_Mu()
            self.update_X(1 if self.row_offset == 0 else 0, self.N)
            slot = self.trace_pos % self.trace.numel()
            self._global(OP_BETA | OP_ELBO, self.trace.data_ptr() + slot * 8)
            self.trace_pos += 1
            return slot
        # mode B: one statistics pass feeds Mu, Alpha, Beta and the bound (and the next W update)
        slot = self.trace_pos % self.trace.numel()
        self._global(OP_MU | OP_ALPHA | OP_BETA | OP_ELBO, self.trace.data_ptr() + slot * 8)
        self.trace_pos += 1
        return slot

    @_on_device
    def iterate_from_host(self, Xh, nchunks=8):
        """One mode-B sweep whose data shard comes from (pinned) HOST memory: the upload is cut into row chunks on
        a copy stream and the Z step of chunk c (K1 + K2) runs while chunk c+1 is still on the PCIe bus.  The W
        update needs no data (it uses the statistics of the previous sweep), so it goes first.  The statistics are sums
        over rows: on the tensor-core paths every chunk's statistics are taken right behind its Z step and added up, so
        that only the last chunk's work is left when the upload ends.  Returns the trace slot of the bound (no host
        synchronisation)."""
        if self.sparse:
            raise NotImplementedError("iterate_from_host streams a dense host array; a sparse engine keeps its entries "
                                      "on the device")
        assert self.mode == "B"
        assert not self.f32, "iterate_from_host: the FP32 variant keeps X as bf16 planes; use precision='f64'"
        N = self.N
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        cs = self._copy_stream
        # first everything that may still read the resident X (stale statistics are rebuilt from it), THEN the copy
        # stream waits: the upload must not overwrite rows a queued kernel has yet to read
        self.update_W()
        self._ensure_gw()
        cs.wait_stream(cur)
        self._xcache_valid = False
        self._mask_valid = False
        self._maskT_valid = False
        step = (N + nchunks - 1) // nchunks
        step = (step + 127) // 128 * 128
        chunked = (not self.f32 and self.zsums is not None and self.algo in (ALGO_AUTO, ALGO_DMMA)
                   and bool(self.lib.pyvb_algo_supported(ALGO_DMMA, self.D, self.q)))
        if chunked:
            if getattr(self, "_acc", None) is None:
                self._acc, self._tmp = torch.zeros_like(self.stats), torch.zeros_like(self.stats)
            self._acc.zero_()
        for lo in range(0, N, step):
            hi = min(N, lo + step)
            with torch.cuda.stream(cs):
                self.X[lo:hi].copy_(Xh[lo:hi], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
            cur.wait_event(ev)
            self.update_Z(lo, hi, _chunk_zsums=chunked)
            if chunked:
                rc = self.lib.pyvb_stats_f64(hi - lo, self.D, self.q, self.X.data_ptr() + lo * self.D * 8, self.D, 0, 0, 0,
                                             self.Zbar.data_ptr() + lo * self.ldmz * 8, self.ldmz,
                                             self.M2.data_ptr() + lo * self.ldmz * 8, self.ldmz,
                                             self.logdet.data_ptr() + lo * 8, self._tmp.data_ptr(), self.ws.data_ptr(),
                                             self.ws_bytes, 0, 0, self.zsums.data_ptr(), 1, None, ALGO_DMMA, self._stream())
                _cabi.check(rc, "pyvb_stats_f64 (chunk)")
                self._acc += self._tmp
        if chunked:
            self.stats.copy_(self._acc)
            if self.distributed:
                allreduce_stats(self.stats)
            self._stats_fresh = True
            self._zsums_valid = False
        slot = self.trace_pos % self.trace.numel()
        self._global(OP_MU | OP_ALPHA | OP_BETA | OP_ELBO, self.trace.data_ptr() + slot * 8)
        self.trace_pos += 1
        return slot

    def iterate(self):
        slot = self.iterate_async()
        return float(self.trace[slot].item())

    def learn(self, niters, tol=1e-3, verbose=False):
        """Network.learn semantics (network.py:40-56): stop as soon as the bound improves by < tol."""
        old = -np.inf
        out = []
        for i in range(niters):
            llb = self.iterate()
            out.append(llb)
            if verbose:
                print(niters - i, llb)
            if not np.isfinite(llb):
                self.check()                     # a non-PD row poisons the bound: raise at once (gaussian.py:118)
            if llb - old < tol:
                if verbose:
                    print("Convergence!")
                break
            old = llb
        self.check()
        return out

    def run(self, niters):
        """niters sweeps back to back without host syncs; returns the bound trace as a device tensor view."""
        slots = [self.iterate_async() for _ in range(niters)]
        return self.trace[slots]
