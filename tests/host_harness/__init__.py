"""Host instantiation of the kernels' per-point functions -- TEST INFRASTRUCTURE ONLY
(see harness.cu).  Built on demand with nvcc; links against the product library for the model
flattening (``gf_build_dev_model``)."""

import ctypes as C
import os
import subprocess

import numpy as np

from golemflavor_b200 import _lib, build

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, 'libgf_host_harness.so')
SRC = os.path.join(HERE, 'harness.cu')
_h = None


def load():
    global _h
    if _h is not None:
        return _h
    lib_path = build.build_library()
    deps = [SRC, lib_path] + [os.path.join(build.CSRC, f) for f in build.HEADERS]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        cuda_inc = os.path.join(os.path.dirname(os.path.dirname(build.nvcc_path())), 'include')
        cmd = ['g++', '-x', 'c++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-I' + cuda_inc,
               '-o', SO, SRC, '-L' + build.LIB_DIR, '-lgolemflavor_b200', '-Wl,-rpath,' + build.LIB_DIR]
        subprocess.run(cmd, check=True)
    _lib.load()
    _h = C.CDLL(SO)
    return _h


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def lnprob(fm, theta, spec=-1, rebuild=False):
    """rebuild=True: the refinement path recomputes H0 / T from the row (k_lnprob) instead of keeping them in memory."""
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    n = th.shape[0]
    lnp, fr, st = np.empty(n), np.empty((n, 3)), np.empty(n, dtype=np.uint8)
    fn = load().hh_lnprob_rebuild if rebuild else load().hh_lnprob
    rc = fn(fm.ref, _p(th), C.c_int64(n), _p(lnp), _p(fr), _p(st), C.c_int(spec))
    _lib.check(rc)
    return lnp, fr, st


def model_spec(fm):
    """(spec the log-posterior / sampler kernels launch, spec the column layout alone allows, Gaussian-dimension bit mask)."""
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    _lib.check(load().hh_model_spec(fm.ref, C.byref(a), C.byref(b), C.byref(c)))
    return a.value, b.value, c.value


def fr(fm, theta, spec=-1):
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    n = th.shape[0]
    out, st = np.empty((n, 3)), np.empty(n, dtype=np.uint8)
    _lib.check(load().hh_fr(fm.ref, _p(th), C.c_int64(n), _p(out), _p(st), C.c_int(spec)))
    return out, st


def lnprior(fm, theta):
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    out = np.empty(th.shape[0])
    _lib.check(load().hh_lnprior(fm.ref, _p(th), C.c_int64(th.shape[0]), _p(out)))
    return out


def philox(ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    out = np.empty_like(ctr)
    load().hh_philox(_p(ctr), C.c_int64(ctr.shape[0]), C.c_uint32(key[0]), C.c_uint32(key[1]), _p(out))
    return out


def draw(fm, seed, first, n):
    theta = np.empty((n, fm.ndim))
    _lib.check(load().hh_draw(fm.ref, C.c_uint64(seed), C.c_uint64(first), C.c_int64(n), _p(theta)))
    return theta


def hist(frs, nb):
    f = np.ascontiguousarray(frs, dtype=np.float64).reshape(-1, 3)
    h = np.zeros((nb + 1) ** 3, dtype=np.uint64)
    load().hh_hist(_p(f), C.c_int64(f.shape[0]), C.c_int(nb), _p(h))
    return h.reshape(nb + 1, nb + 1, nb + 1).astype(np.int64)


def eig(ham):
    h = np.ascontiguousarray(np.asarray(ham, dtype=np.complex128)).reshape(-1, 3, 3)
    n = h.shape[0]
    hv = h.view(np.float64).reshape(n, 18)
    lam, vec, xf, ok = np.empty((n, 3)), np.empty((n, 18)), np.empty((n, 4)), np.empty(n, dtype=np.uint8)
    load().hh_eig(_p(hv), C.c_int64(n), _p(lam), _p(vec), _p(xf), _p(ok))
    return lam, vec.view(np.complex128).reshape(n, 3, 3), xf.reshape(n, 2, 2), ok.astype(bool)


def deflate(ham):
    """gfp_herm3_x4_deflate on Hermitian matrices: ((n, 2, 2) = |V_ai|^2 for rows e, mu and columns
    (isolated eigenvalue, upper member of the remaining pair), status bits)."""
    h = np.ascontiguousarray(np.asarray(ham, dtype=np.complex128)).reshape(-1, 3, 3)
    n = h.shape[0]
    hv = h.view(np.float64).reshape(n, 18)
    x4, st = np.empty((n, 4)), np.empty(n, dtype=np.uint8)
    load().hh_deflate(_p(hv), C.c_int64(n), _p(x4), _p(st))
    return x4.reshape(n, 2, 2), st


def ensemble(fm, pos, lnp, nsteps, nwalkers, nchains=1, nfree=None, step0=0, thin=1, a=2.0, seed=0, chain0=0):
    """Sequential host replay of gf_ensemble_run.  Returns (pos, lnp, chain, lnp_chain, naccept)."""
    ndim = fm.ndim
    pos = np.array(pos, dtype=np.float64).reshape(nchains, nwalkers, ndim).copy()
    lnp = np.array(lnp, dtype=np.float64).reshape(nchains, nwalkers).copy()
    nstore = nsteps // thin
    chain = np.zeros((nchains, nwalkers, nstore, ndim))
    lchain = np.zeros((nchains, nwalkers, nstore))
    nacc = np.zeros((nchains, nwalkers), dtype=np.uint64)
    cfg = _lib.EnsembleConfig(nchains=nchains, nwalkers=nwalkers, nfree=nfree or ndim, nsteps=nsteps, step0=step0,
                              thin=thin, a=a, seed=seed, chain0=chain0, mode=0)
    _lib.check(load().hh_ensemble(fm.ref, C.byref(cfg), _p(pos), _p(lnp), _p(chain), _p(lchain), _p(nacc)))
    return pos, lnp, chain, lchain, nacc.astype(np.int64)


def cubic_w(delta):
    d = np.ascontiguousarray(delta, dtype=np.float64)
    w = np.empty_like(d)
    load().hh_cubic_w(_p(d), C.c_int64(d.size), _p(w))
    return w


def fr_scales(fm, theta, scales):
    """gf_point_fr_scales: compositions [n, ns, 3] of every point at each frozen scale, + status bytes."""
    th = np.ascontiguousarray(theta, dtype=np.float64).reshape(-1, fm.ndim)
    sc = np.ascontiguousarray(scales, dtype=np.float64)
    n, ns = th.shape[0], sc.shape[0]
    out, st = np.empty((n, ns, 3)), np.empty((n, ns), dtype=np.uint8)
    _lib.check(load().hh_fr_scales(fm.ref, _p(th), C.c_int64(n), _p(sc), C.c_int(ns), _p(out), _p(st)))
    return out, st


def ndtri(p):
    """gf_ndtri_table: (z, covered) of the table-based inverse normal CDF."""
    p = np.ascontiguousarray(p, dtype=np.float64).ravel()
    z, ok = np.empty_like(p), np.empty(p.shape[0], dtype=np.uint8)
    load().hh_ndtri(_p(p), C.c_int64(p.shape[0]), _p(z), _p(ok))
    return z, ok.astype(bool)


def fast_min_sin2():
    """(GFP_FAST_MIN_SIN2, the high word the device compares sin^2(phi/3) with)."""
    thr = C.c_double()
    fn = load().hh_fast_min_sin2
    fn.restype = C.c_uint
    hi = fn(C.byref(thr))
    return thr.value, hi
