"""ctypes binding of libpyvb_b200.so (the C-ABI declared in include/pyvb_b200.h).

There is NO fallback: if the library is missing, or a call fails, this raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpyvb_b200.so")

c_dp = ctypes.c_void_p          # device pointers travel as integers
c_ll = ctypes.c_longlong
c_int = ctypes.c_int
c_sz = ctypes.c_size_t


class Consts(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in (
        "alpha_mu", "a0", "b0", "psi_qa", "lgam_qa", "lgam_a0", "ard_a0", "ard_b0", "al_qa",
        "psi_alqa", "lgam_alqa", "lgam_ard_a0", "lndet_P0", "m0P0m0")] + [("ard", c_int), ("mode_a", c_int)]


class Peers(ctypes.Structure):
    _fields_ = [("bufs", ctypes.c_void_p), ("world", c_int), ("rank", c_int), ("epoch", ctypes.c_ulonglong)]


SIGNATURES = {
    "pyvb_version": (c_int, []),
    "pyvb_last_error": (ctypes.c_char_p, []),
    "pyvb_gw_pitch": (c_int, [c_int]),
    "pyvb_gw_woff": (c_int, [c_int]),
    "pyvb_mz_pitch": (c_int, [c_int]),
    "pyvb_stats_len": (c_sz, [c_int, c_int]),
    "pyvb_stats_workspace_bytes": (c_sz, [c_ll, c_int, c_int, c_int]),
    "pyvb_algo_supported": (c_int, [c_int, c_int, c_int]),
    "pyvb_pack_gw_f64": (c_int, [c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_int, c_dp]),
    "pyvb_zsums_len": (c_sz, [c_ll, c_int]),
    "pyvb_zsums_kw": (c_int, [c_int]),
    "pyvb_zsums_blocks": (c_int, [c_ll, c_int]),
    "pyvb_zstep_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_int, c_dp, c_dp, c_dp,
                               c_dp, c_ll, c_dp, c_ll, c_dp, c_dp, c_dp, c_int, c_dp]),
    "pyvb_zstep_w_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_ll, c_dp, c_int, c_dp, c_dp, c_dp,
                                 c_dp, c_ll, c_dp, c_ll, c_dp, c_dp, c_dp, c_int, c_dp]),
    "pyvb_stats_w_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_ll, c_dp, c_ll, c_dp, c_ll, c_dp,
                                 c_dp, c_dp, c_sz, c_dp, c_int, c_dp, c_int, ctypes.POINTER(Peers), c_int, c_dp]),
    "pyvb_global_w_f64": (c_int, [c_int, c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                  c_dp, ctypes.POINTER(Consts), c_dp, c_dp]),
    "pyvb_zsolve_f64": (c_int, [c_ll, c_int, c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_stats_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_ll, c_dp, c_ll, c_dp,
                               c_dp, c_dp, c_sz, c_dp, c_int, c_dp, c_int, ctypes.POINTER(Peers), c_int, c_dp]),
    "pyvb_i8_supported": (c_int, [c_int, c_int]),
    "pyvb_i8_digits_bytes": (c_sz, [c_int, c_int]),
    "pyvb_i8_ncols": (c_int, [c_int]),
    "pyvb_i8_mask_bytes": (c_sz, [c_ll, c_int]),
    "pyvb_prepare_mask_i8": (c_int, [c_ll, c_int, c_dp, c_ll, c_dp, c_dp]),
    "pyvb_zstep_i8_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_int, c_dp, c_dp, c_dp,
                                  c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_dp, c_int, c_dp]),
    "pyvb_stats_i8_supported": (c_int, [c_int, c_int]),
    "pyvb_stats_i8_npad": (c_ll, [c_ll]),
    "pyvb_stats_i8_digits_bytes": (c_sz, [c_ll, c_int]),
    "pyvb_stats_i8_fused": (c_int, [c_int, c_int]),
    "pyvb_stats_i8_maskt_bytes": (c_sz, [c_ll, c_int]),
    "pyvb_stats_i8_scratch_len": (c_sz, [c_int]),
    "pyvb_stats_i8_guard_offset": (c_sz, [c_int]),
    "pyvb_stats_i8_workspace_bytes": (c_sz, [c_ll, c_int, c_int]),
    "pyvb_prepare_maskt_i8": (c_int, [c_ll, c_int, c_dp, c_ll, c_dp, c_dp]),
    "pyvb_stats_i8_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_dp, c_sz,
                                  c_dp, c_dp, ctypes.POINTER(Peers), c_dp]),
    "pyvb_f32_pitch": (c_int, [c_int]),
    "pyvb_f32_zoff": (c_int, [c_int]),
    "pyvb_f32_poff": (c_int, [c_int]),
    "pyvb_f32_supported": (c_int, [c_int, c_int]),
    "pyvb_prepare_x_f32": (c_int, [c_ll, c_int, c_dp, c_ll, c_dp, c_dp]),
    "pyvb_pack_gw_f32": (c_int, [c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_zstep_k1_f32": (c_int, [c_ll, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_zsums_len_f32": (c_sz, [c_ll, c_int]),
    "pyvb_zstep_f32": (c_int, [c_ll, c_ll, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_stats_f32": (c_int, [c_ll, c_ll, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_sz, c_dp, c_dp, ctypes.POINTER(Peers), c_dp]),
    "pyvb_csr_supported": (c_int, [c_int, c_int]),
    "pyvb_csr_stats_blocks": (c_int, [c_ll, c_int, c_int]),
    "pyvb_csr_block_rows": (c_ll, [c_ll, c_int, c_int]),
    "pyvb_stats_csr_workspace_bytes": (c_sz, [c_ll, c_int, c_int, c_int]),
    "pyvb_zstep_csr_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_int, c_dp, c_dp, c_dp, c_dp, c_ll, c_dp,
                                   c_dp, c_dp, c_dp]),
    "pyvb_stats_csr_f64": (c_int, [c_ll, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_ll, c_dp, c_dp, c_dp, c_sz, c_dp,
                                   c_dp, ctypes.POINTER(Peers), c_dp]),
    "pyvb_zstep_csr_w_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_int, c_dp, c_dp, c_dp, c_dp, c_ll,
                                     c_dp, c_dp, c_dp, c_dp]),
    "pyvb_stats_csr_w_f64": (c_int, [c_ll, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_ll, c_dp, c_dp, c_dp, c_sz,
                                     c_dp, c_dp, ctypes.POINTER(Peers), c_dp]),
    "pyvb_lds_max_len": (c_int, []),
    "pyvb_lds_iterate_f64": (c_int, [c_int, c_int, c_int, c_int] + [c_dp] * 11 + [ctypes.c_double] * 3 + [c_int, c_dp, c_dp]),
    "pyvb_lds_iterate_known_f64": (c_int, [c_int, c_int, c_int, c_int] + [c_dp] * 12 + [ctypes.c_double] * 3 + [c_int, c_dp, c_dp]),
    "pyvb_peer_bytes": (c_sz, [c_sz]),
    "pyvb_peer_alloc": (c_int, [c_sz, ctypes.POINTER(ctypes.c_void_p)]),
    "pyvb_peer_free": (c_int, [c_dp]),
    "pyvb_peer_export": (c_int, [c_dp, ctypes.c_char_p]),
    "pyvb_peer_import": (c_int, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]),
    "pyvb_peer_close": (c_int, [c_dp]),
    "pyvb_wupdate_f64": (c_int, [c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_global_f64": (c_int, [c_int, c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                ctypes.POINTER(Consts), c_dp, c_dp]),
    "pyvb_nd_len": (c_sz, [c_int]),
    "pyvb_pack_gw_nd_f64": (c_int, [c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_int, c_dp]),
    "pyvb_wupdate_nd_f64": (c_int, [c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
    "pyvb_global_nd_f64": (c_int, [c_int, c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                   ctypes.POINTER(Consts), c_dp, c_dp]),
    "pyvb_bench_dmma_f64": (c_int, [c_int, c_int, c_dp, c_dp]),
    "pyvb_bench_umma": (c_int, [c_int, c_int, c_int, c_int, c_int, c_dp, c_dp, c_dp]),
    "pyvb_impute_f64": (c_int, [c_ll, c_int, c_int, c_dp, c_ll, c_dp, c_dp, c_dp, c_ll, c_dp, c_dp, c_dp, c_dp, c_dp]),
}

_lib = None


class PyvbError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library; raises ImportError when it was not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "pyvb_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().pyvb_last_error()
        raise PyvbError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else ""))
