"""In-tree build of libpyvb_b200.so (nvcc, sm_100a only).  Used by __graft_entry__.build().

Every .cu file is its own translation unit (no relocatable device code): the objects are compiled in parallel
into pyvb_b200/build/ (git-ignored), only the stale ones, and linked into pyvb_b200/libpyvb_b200.so."""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libpyvb_b200.so")
SOURCES = ["cabi.cu", "kernels_generic.cu", "kernels_dmma.cu", "kernels_k2.cu", "kernels_k2m.cu", "kernels_k2t.cu", "kernels_k2g.cu", "kernels_k2s.cu", "kernels_f32.cu",
           "kernels_i8.cu", "kernels_lds.cu", "kernels_sparse.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-diag-suppress", "177",
    "-Xcompiler", "-fPIC",
]


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))] + \
           [os.path.join(os.path.dirname(HERE), "include", "pyvb_b200.h")]


def _mtime(p):
    return os.path.getmtime(p) if os.path.isfile(p) else -1.0


def build(force=False, verbose=False):
    """Compile every CUDA source into pyvb_b200/libpyvb_b200.so (only what is stale unless force)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max(_mtime(h) for h in _headers())
    jobs = []
    for src in SOURCES:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src[:-3] + ".o")
        if force or _mtime(o) < max(_mtime(s), hdr_t):
            jobs.append([nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for r in ex.map(lambda c: subprocess.run(c, cwd=CSRC, capture_output=not verbose, text=True), jobs):
                if r.returncode != 0:
                    raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(r.args), (r.stderr or "") + (r.stdout or "")))
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in SOURCES]
    if jobs or _mtime(LIB) < max(_mtime(o) for o in objs):
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs, check=True)
    return LIB
