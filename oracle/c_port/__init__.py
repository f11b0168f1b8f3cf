"""ctypes glue for oracle/c_port/mg_port.c (plain C + OpenMP restatement of the solve loop) -- TEST INFRASTRUCTURE.
The hierarchy comes from the numpy oracle (oracle.mg_oracle); this module only runs the timed solve."""
from __future__ import annotations

import ctypes as C
import os
import stat
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_OUT = os.path.join(os.path.dirname(_HERE), "_ref")
_SO = os.path.join(_OUT, "libmgport.so")


class _Level(C.Structure):
    _fields_ = [("L", C.c_int), ("n", C.c_int), ("nc", C.c_int), ("D", C.c_void_p), ("mD0inv", C.c_void_p), ("P", C.c_void_p),
                ("phi", C.c_void_p), ("r", C.c_void_p), ("tmp", C.c_void_p)]


def build() -> str:
    """Path of an up-to-date libmgport.so: oracle/_ref/ of the tree, or a per-user temporary directory when the library there
    is missing or stale and the tree is read-only."""
    src = os.path.join(_HERE, "mg_port.c")
    fresh = lambda so: os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src)
    if fresh(_SO):
        return _SO
    out = _OUT if os.access(_OUT if os.path.isdir(_OUT) else os.path.dirname(_OUT), os.W_OK) else \
        os.path.join(tempfile.gettempdir(), f"mg2d_c_port_{os.getuid()}")
    if out != _OUT:
        os.makedirs(out, mode=0o700, exist_ok=True)
        st = os.lstat(out)          # a shared temporary directory: load nothing from a directory another account controls
        if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o022:
            raise RuntimeError(f"{out} is not a directory owned and writable only by this user")
    so = os.path.join(out, "libmgport.so")
    if not fresh(so):
        os.makedirs(out, exist_ok=True)
        # baseline x86-64 ISA on purpose: the built library travels with the repo snapshot to a different host CPU
        subprocess.check_call(["gcc", "-O3", "-fcx-limited-range", "-fopenmp", "-shared", "-fPIC", "-o", so, src, "-lm"])
    return so


def set_threads(n: int | None = None) -> int:
    """Use n OpenMP threads (None: every processor of the host, whatever OMP_NUM_THREADS says); returns the count in force."""
    lib = C.CDLL(build())
    lib.mgport_set_threads.restype = C.c_int
    return int(lib.mgport_set_threads(C.c_int(0 if n is None else n)))


def gcr_solve_arrays(levels, size, n_dof, pre, post, block, b, tol=1e-10, max_iters=1000, restart=8, threads=None):
    """levels: per level a dict(D=[S,5,n,n] reference layout, P=[S,nc,n] or None); the hierarchy may come from the numpy
    oracle or be exported from another setup.  Returns (x, info) with info['threads'] = OpenMP threads actually used."""
    lib = C.CDLL(build())
    lib.mgport_gcr_solve.restype = C.c_int
    assert lib.mgport_level_size() == C.sizeof(_Level)
    nthreads = set_threads(threads)
    nlevels = len(levels) - 1
    keep, lv_c = [], (_Level * (nlevels + 1))()
    for l, lv in enumerate(levels):
        S, n = size[l] ** 2, n_dof[l]
        D = np.ascontiguousarray(lv["D"], dtype=np.complex128)
        mD0inv = lv.get("mD0inv")
        if mD0inv is None:
            mD0inv = lv["mD0inv"] = np.ascontiguousarray(-np.linalg.inv(D[:, 0]), dtype=np.complex128)
        P = np.ascontiguousarray(lv["P"], dtype=np.complex128) if l < nlevels else None
        phi, r, tmp = (np.zeros((S, n), dtype=np.complex128) for _ in range(3))
        keep += [D, mD0inv, P, phi, r, tmp]
        lv_c[l] = _Level(size[l], n, n_dof[l + 1] if l < nlevels else 0, D.ctypes.data, mD0inv.ctypes.data,
                         P.ctypes.data if P is not None else None, phi.ctypes.data, r.ctypes.data, tmp.ctypes.data)
    pre_c = (C.c_int * (nlevels + 1))(*pre)
    post_c = (C.c_int * (nlevels + 1))(*post)
    b = np.ascontiguousarray(b, dtype=np.complex128)
    x = np.zeros_like(b)
    res = np.zeros(max_iters, dtype=np.float64)
    import time
    t0 = time.perf_counter()
    it = lib.mgport_gcr_solve(C.c_int(nlevels), lv_c, pre_c, post_c, C.c_int(block), C.c_void_p(b.ctypes.data),
                              C.c_void_p(x.ctypes.data), C.c_double(tol), C.c_int(max_iters), C.c_int(restart),
                              C.c_void_p(res.ctypes.data))
    info = {"iters": int(it), "resnorms": res[:it].tolist(), "converged": bool(it > 0 and res[it - 1] < tol),
            "seconds": time.perf_counter() - t0, "threads": nthreads}
    return x, info


def levels_from_oracle(LVL, p):
    return [{"D": lv.D, "P": lv.phi_null if l < p.nlevels else None} for l, lv in enumerate(LVL)]


def gcr_solve(LVL, p, b, tol=1e-10, max_iters=1000, restart=8, threads=None, cache=None):
    """Same contract as oracle.mg_oracle.gcr_MG for smoother 'rbgs', quad 1, telescoping cycle.  Returns (x, info).
    cache: a dict that keeps the converted level arrays (-D0^-1 ...) between calls on the same hierarchy."""
    assert p.smoother == "rbgs" and p.t_flag == 0 and p.quad == 1 and len(set(p.blocks)) <= 1
    levels = None if cache is None else cache.get("levels")
    if levels is None:
        levels = levels_from_oracle(LVL, p)
        if cache is not None:
            cache["levels"] = levels
    return gcr_solve_arrays(levels, p.size, p.n_dof, p.pre, p.post, p.block, b, tol, max_iters, restart, threads)
