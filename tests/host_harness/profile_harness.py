"""Host instantiation of the profile-likelihood task (profile_harness.cu) -- TEST INFRASTRUCTURE ONLY.  Built on demand with
g++ like the main harness and linked against the product library for the model flattening (``gf_build_dev_model``).  The
shared object goes next to the source, or to a per-user temporary directory when the tree is read-only."""

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from golemflavor_b200 import _lib, build

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'profile_harness.cu')
_h = None


def _so_path():
    where = HERE if os.access(HERE, os.W_OK) else os.path.join(tempfile.gettempdir(), 'gf_profile_harness_%d' % os.getuid())
    os.makedirs(where, exist_ok=True)
    return os.path.join(where, 'libgf_profile_harness.so')


def _load():
    global _h
    if _h is not None:
        return _h
    lib_path = build.build_library()
    so = _so_path()
    deps = [SRC, lib_path] + [os.path.join(build.CSRC, f) for f in build.HEADERS]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        cuda_inc = os.path.join(os.path.dirname(os.path.dirname(build.nvcc_path())), 'include')
        cmd = ['g++', '-x', 'c++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-I' + cuda_inc,
               '-o', so, SRC, '-L' + build.LIB_DIR, '-lgolemflavor_b200', '-Wl,-rpath,' + build.LIB_DIR]
        subprocess.run(cmd, check=True)
    _lib.load()
    _h = C.CDLL(so)
    return _h


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def profile(fm, scales, nstarts=64, seed=0, task0=0, max_evals=6000, ftol=1e-10, xtol=1e-7, spec=-1):
    """gf_profile_grid run sequentially on the host (spec: -1 as the library chooses, 2 = static 6-column layout, 1 = FIXED,
    0 = GENERIC).  Returns the dict of ``scan.scan_profile_grid``."""
    sc = np.ascontiguousarray(scales, dtype=np.float64).ravel()
    ns = sc.shape[0]
    best, argmax, fr = np.empty(ns), np.empty((ns, fm.ndim)), np.empty((ns, 3))
    st, counts = np.empty(ns, dtype=np.uint8), np.empty((ns, 2), dtype=np.int64)
    cfg = _lib.ProfileConfig(seed=int(seed), task0=int(task0), nstarts=int(nstarts), max_evals=int(max_evals), ftol=float(ftol), xtol=float(xtol))
    _lib.check(_load().hh_profile(fm.ref, C.byref(cfg), _p(sc), C.c_int32(ns), _p(best), _p(argmax), _p(fr), _p(st), _p(counts), C.c_int(spec)))
    return dict(best=best, argmax=argmax, fr=fr, status=st, nevals=counts[:, 0], nconverged=counts[:, 1])


def nm_box_quadratic(a, c, lo, hi, x0, ftol=1e-12, xtol=1e-8, max_evals=20000):
    """The Nelder-Mead core on sum_k a_k (x_k - c_k)^2 over [lo, hi]: (x_best, g_best, optimiser evaluations, objective
    calls, converged)."""
    arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (a, c, lo, hi, x0)]
    n = arrs[0].shape[0]
    xb, gb, nev, conv = np.empty(n), C.c_double(), np.empty(2, dtype=np.int64), C.c_int()
    _load().hh_nm_box_quadratic(C.c_int(n), *[_p(v) for v in arrs], C.c_double(ftol), C.c_double(xtol), C.c_int(max_evals), _p(xb),
                               C.byref(gb), _p(nev), C.byref(conv))
    return xb, gb.value, int(nev[0]), int(nev[1]), bool(conv.value)
