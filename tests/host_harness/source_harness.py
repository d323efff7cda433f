"""Host instantiation of the per-sample code of the source-grid evidence (source_harness.cu) -- TEST INFRASTRUCTURE ONLY.  Built
on demand with g++ like the main harness and linked against the product library for the model flattening
(``gf_build_dev_model``).  The shared object goes next to the source, or to a per-user temporary directory when the tree is
read-only."""

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from golemflavor_b200 import _lib, build

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'source_harness.cu')
_h = None


def _so_path():
    where = HERE if os.access(HERE, os.W_OK) else os.path.join(tempfile.gettempdir(), 'gf_source_harness_%d' % os.getuid())
    os.makedirs(where, exist_ok=True)
    return os.path.join(where, 'libgf_source_harness.so')


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


def transition_fr(fm, theta, sources, spec=-1):
    """(A[n, 3], fr[n, nsrc, 3], status[n]) of every point at its own logLam: the transition sums of
    ``gf_point_transition_scales`` and each source's composition from them (``gfp_transition_fr``)."""
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    src = np.ascontiguousarray(sources, dtype=np.float64).reshape(-1, 3)
    n, ns = th.shape[0], src.shape[0]
    A, fr, st = np.empty((n, 3)), np.empty((n, ns, 3)), np.empty(n, dtype=np.uint8)
    _lib.check(_load().hh_transition_fr(fm.ref, _p(th), C.c_int64(n), _p(src), C.c_int(ns), C.c_int(spec), _p(A), _p(fr), _p(st)))
    return A, fr, st


def evidence_sources(fm, scales, sources, injected, count, seed=26, first_index=0):
    """The task of ``gf_scan_evidence_sources`` run sequentially in sample order: ``lse[nsrc, ns, 2]`` (max, sum)."""
    sc = np.ascontiguousarray(scales, dtype=np.float64).ravel()
    src = np.ascontiguousarray(sources, dtype=np.float64).reshape(-1, 3)
    inj = np.ascontiguousarray(np.broadcast_to(np.asarray(injected, dtype=np.float64).reshape(-1, 3), src.shape))
    lse = np.zeros((src.shape[0], sc.shape[0], 2))
    lse[..., 0] = -np.inf
    _lib.check(_load().hh_evidence_sources(fm.ref, C.c_uint64(seed), C.c_uint64(first_index), C.c_int64(count), _p(sc), C.c_int(sc.shape[0]),
                                           _p(src), _p(inj), C.c_int(src.shape[0]), _p(lse)))
    return lse
