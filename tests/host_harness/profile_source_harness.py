"""Host instantiation of the task of gf_profile_sources (profile_source_harness.cu) -- TEST INFRASTRUCTURE ONLY.  Built on
demand with g++ like the main harness and linked against the product library for the model flattening
(``gf_build_dev_model``).  The shared object goes next to the source, or to a per-user temporary directory when the tree is
read-only."""

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from golemflavor_b200 import _lib, build

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'profile_source_harness.cu')
_h = None


def _so_path():
    where = HERE if os.access(HERE, os.W_OK) else os.path.join(tempfile.gettempdir(), 'gf_profile_source_harness_%d' % os.getuid())
    os.makedirs(where, exist_ok=True)
    return os.path.join(where, 'libgf_profile_source_harness.so')


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
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _rows(sources, injected):
    src = np.ascontiguousarray(sources, dtype=np.float64).reshape(-1, 3)
    inj = np.ascontiguousarray(np.broadcast_to(np.asarray(injected, dtype=np.float64).reshape(-1, 3), src.shape))
    return src, inj


def objective(fm, theta, scale, sources=None, injected=(1, 1, 1), spec=-1):
    """ln_prob at theta [n, ndim] with the scale frozen: (lnp[nsrc, n], fr[nsrc, n, 3], status[nsrc, n]) of the source objective of
    gf_profile_sources for each source, or ([1, n], ...) of gf_profile_grid's objective of the model itself (sources=None)."""
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    n = th.shape[0]
    src, inj = _rows(sources, injected) if sources is not None else (None, None)
    ns = 1 if src is None else src.shape[0]
    lnp, fr, st = np.empty((ns, n)), np.empty((ns, n, 3)), np.empty((ns, n), dtype=np.uint8)
    _lib.check(_load().hh_profile_objective(fm.ref, _p(th), C.c_int64(n), C.c_double(scale), _p(src), _p(inj), C.c_int(ns), C.c_int(spec),
                                            _p(lnp), _p(fr), _p(st)))
    return lnp, fr, st


def profile_sources(fm, scales, sources, injected, nstarts=64, seed=0, task0=0, max_evals=6000, ftol=1e-10, xtol=1e-7, spec=-1):
    """gf_profile_sources run sequentially on the host.  Returns the dict of ``scan.scan_profile_sources``."""
    sc = np.ascontiguousarray(scales, dtype=np.float64).ravel()
    src, inj = _rows(sources, injected)
    ns, nsrc = sc.shape[0], src.shape[0]
    best, argmax, fr = np.empty((nsrc, ns)), np.empty((nsrc, ns, fm.ndim)), np.empty((nsrc, ns, 3))
    st, counts = np.empty((nsrc, ns), dtype=np.uint8), np.empty((nsrc, ns, 2), dtype=np.int64)
    cfg = _lib.ProfileConfig(seed=int(seed), task0=int(task0), nstarts=int(nstarts), max_evals=int(max_evals), ftol=float(ftol), xtol=float(xtol))
    _lib.check(_load().hh_profile_sources(fm.ref, C.byref(cfg), _p(sc), C.c_int32(ns), _p(src), _p(inj), C.c_int32(nsrc), _p(best), _p(argmax),
                                          _p(fr), _p(st), _p(counts), C.c_int(spec)))
    return dict(best=best, argmax=argmax, fr=fr, status=st, nevals=counts[..., 0], nconverged=counts[..., 1])
