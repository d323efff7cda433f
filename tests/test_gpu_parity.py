"""GPU parity tests (``-m gpu``): the CUDA path, called through the C ABI (via the Python mirror of
the reference interface), against the golden fixtures generated from the unmodified reference,
against the oracle on seeded inputs, and -- at full sizes -- through size-independent properties.

Tolerances (BASELINE.json north_star): flavor ratios within 1e-10 absolute on the unit-sum
composition (== 1e-10 relative to its norm), log-likelihood / log-posterior within 1e-10 relative;
histogram counts bit-exact given identical samples."""

import argparse
import ctypes as C
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from golemflavor_b200 import _lib, fr, llh, mcmc, model, scan  # noqa: E402
from golemflavor_b200.enums import Texture  # noqa: E402
from oracle import golem_oracle as go  # noqa: E402
from oracle import truth  # noqa: E402

import models  # noqa: E402

FR_TOL = 1e-10
LLH_RTOL = 1e-10


@pytest.fixture(scope='module')
def torch():
    import torch
    assert torch.cuda.is_available(), 'these tests need a CUDA device'
    return torch


def test_native_library_is_loaded(torch):
    lib = _lib.load()
    info = _lib.device_info()
    assert info['cc'][0] >= 9 and info['sm_count'] > 0
    before = lib.gf_launch_count()
    fr.angles_to_u((0.2, 0.3, 0.5, 1.5))
    assert lib.gf_launch_count() == before + 1
    maps = open('/proc/self/maps').read()
    assert 'libgolemflavor_b200.so' in maps


def test_device_math_helpers(torch):
    """The MUFU-seeded reciprocal / reciprocal square root used by the eigen stage (one cubic
    refinement step) must be accurate to a few ulp over the whole dynamic range it sees."""
    rng = np.random.default_rng(0)
    x = np.concatenate([10.0 ** rng.uniform(-250, 250, 200000), rng.uniform(0.5, 2.0, 200000),
                        [1.0, 2.0, 4.0, 1e-280, 1e280, 3.0, 0.1]])
    xt = torch.as_tensor(x).cuda()
    rs, rc = torch.empty_like(xt), torch.empty_like(xt)
    _lib.check(_lib.load().gf_selftest_math(_lib.ptr(xt), len(x), _lib.ptr(rs), _lib.ptr(rc), _lib.stream_ptr(torch)))
    xl = x.astype(np.longdouble)
    assert np.max(np.abs(rs.cpu().numpy() * np.sqrt(xl) - 1)) < 1e-15
    assert np.max(np.abs(rc.cpu().numpy() * xl - 1)) < 1e-15


def test_device_trig_helpers(torch):
    """The table-free sin / cos of the CP phase (Cody-Waite reduction + fdlibm polynomials with immediate
    coefficients) against x87 long-double NumPy: below 2 ulp of the unit scale on the prior box and far
    around it, library fallback for huge and non-finite arguments."""
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.uniform(0, 2 * np.pi, 400000), rng.uniform(-1000, 1000, 200000), rng.uniform(-99999, 99999, 100000),
                        np.arange(-64, 65) * (np.pi / 4), np.arange(-64, 65) * (np.pi / 2), [0.0, -0.0, 1e-300, 1e5, -1e5, 3e8, -7e15, 1e300]])
    xt = torch.as_tensor(x).cuda()
    sn, cs, co = torch.empty_like(xt), torch.empty_like(xt), torch.empty_like(xt)
    _lib.check(_lib.load().gf_selftest_trig(_lib.ptr(xt), len(x), _lib.ptr(sn), _lib.ptr(cs), _lib.ptr(co), _lib.stream_ptr(torch)))
    xl = x.astype(np.longdouble)
    small = np.abs(x) < 1e5
    assert np.max(np.abs(sn.cpu().numpy()[small] - np.sin(xl[small]))) < 4.5e-16
    assert np.max(np.abs(cs.cpu().numpy()[small] - np.cos(xl[small]))) < 4.5e-16
    assert np.max(np.abs(co.cpu().numpy()[small] - np.cos(xl[small]))) < 4.5e-16
    assert np.allclose(sn.cpu().numpy()[~small], np.sin(x[~small]), atol=1e-15) and np.allclose(co.cpu().numpy()[~small], np.cos(x[~small]), atol=1e-15)
    # the sampler's logarithm: below 2 ulp on (0, 1), on the stretch factors [1/2, 2] and on the whole normal range
    w = rng.integers(0, 1 << 32, 300000, dtype=np.uint64)
    xs = np.concatenate([(w.astype(np.float64) + 0.5) / 4294967296.0, rng.uniform(0.5, 2.0, 100000), 10.0 ** rng.uniform(-300, 300, 100000),
                         [1.0, 2.0, 0.5, np.e, 0.7071067811865476, 1.4142135623730951]])
    xt2 = torch.as_tensor(xs).cuda()
    lg = torch.empty_like(xt2)
    _lib.check(_lib.load().gf_selftest_log(_lib.ptr(xt2), len(xs), _lib.ptr(lg), _lib.stream_ptr(torch)))
    ref = np.log(xs.astype(np.longdouble))
    assert np.max(np.abs(lg.cpu().numpy() - ref) / np.maximum(np.abs(ref), 1e-300) * (ref != 0)) < 4.5e-16
    assert lg.cpu().numpy()[np.where(xs == 1.0)[0][0]] == 0.0
    bad = torch.as_tensor(np.array([np.nan, np.inf, -np.inf])).cuda()
    _lib.check(_lib.load().gf_selftest_trig(_lib.ptr(bad), 3, _lib.ptr(sn), _lib.ptr(cs), _lib.ptr(co), _lib.stream_ptr(torch)))
    assert np.all(np.isnan(sn.cpu().numpy()[:3])) and np.all(np.isnan(cs.cpu().numpy()[:3])) and np.all(np.isnan(co.cpu().numpy()[:3]))


# ------------------------------------------------------------------ docstring known answers (fr.py)
def test_kat_angles_to_u(torch):
    ref = np.array([[0.66195018 + 0.j, 0.33097509 + 0.j, 0.04757188 - 0.6708311j],
                    [-0.34631487 - 0.42427084j, 0.61741198 - 0.21213542j, 0.52331757 + 0.j],
                    [0.28614067 - 0.42427084j, -0.64749908 - 0.21213542j, 0.52331757 + 0.j]])
    got = fr.angles_to_u((0.2, 0.3, 0.5, 1.5))          # fr.py:131-135
    assert got.shape == (3, 3) and got.dtype == np.complex128
    assert np.abs(got - ref).max() < 1e-8


def test_kat_angles_to_fr_and_normalize(torch):
    ref = (0.38340579025361626, 0.16431676725154978, 0.45227744249483393)   # fr.py:97-98
    got = fr.angles_to_fr((0.3, 0.4))
    assert isinstance(got, tuple) and np.allclose(got, ref, rtol=0, atol=1e-15)
    assert np.allclose(fr.normalize_fr((1, 2, 3)), [1 / 6, 1 / 3, 0.5])     # fr.py:254-256
    assert fr.normalise_fr is fr.normalize_fr
    a = fr.fr_to_angles(got)
    assert np.allclose(a, (0.3, 0.4), atol=1e-12)


def test_kat_params_to_bsmu_and_u_to_fr(torch):
    v = fr.params_to_BSMu((0.2, 0.3, 0.5, 1.5, -20), dim=3, energy=1000)    # fr.py:354-358
    assert v.shape == (3, 3)
    assert np.abs(fr.test_unitarity(v) - np.eye(3)).max() < 1e-13
    got = fr.u_to_fr((1, 2, 0), v)                                          # fr.py:519-521
    assert np.allclose(got, [0.33740075, 0.33176584, 0.33083341], atol=1e-8)
    assert np.allclose(got, [0.3374007466, 0.3317658442, 0.3308334092], atol=2e-10)


def test_kat_docs_mappings_and_nufit(torch, golden):
    g = golden('ref_basic.npz')
    assert np.abs(np.asarray(fr.NUFIT_U) - g['nufit_u']).max() < 1e-15
    for src, ref, coarse in zip([(1, 0, 0), (0, 1, 0), (1, 2, 0)], g['fr_nufit'],
                                [(0.55, 0.18, 0.27), (0.18, 0.44, 0.38), (0.31, 0.35, 0.34)]):
        got = fr.u_to_fr(fr.normalize_fr(src), fr.NUFIT_U)
        assert np.abs(got - ref).max() < 1e-15
        assert np.allclose(got, coarse, atol=5e-3)       # docs/source/physics.rst:277-279
    with pytest.raises(ValueError):
        fr.u_to_fr((1, 2, 0), np.eye(2))                 # fr.py:198-202 style
    with pytest.raises(ValueError):
        fr.cardano_eqn(np.eye(4))


# ------------------------------------------------------------------ golden fixtures from the reference
def test_golden_basic(torch, golden):
    g = golden('ref_basic.npz')
    u = fr.angles_to_u(g['ang'])
    assert np.abs(u - g['u']).max() < 1e-14
    assert np.abs(fr.angles_to_fr(g['src_ang']) - g['src_fr']).max() < 1e-15
    got = fr.u_to_fr(g['srcs'], g['u'])
    assert np.abs(got - g['fr']).max() < 1e-14
    # cardano_eqn: eigenvectors agree with the reference up to column order and phase -> compare
    # the spectral projectors via |V|^2 sorted by eigenvalue
    lam, vec, st = fr.eigh3(g['herm'])
    w, vref = np.linalg.eigh(g['herm'])
    assert np.abs(lam - w).max() < 1e-13 and not st.any()
    assert np.abs(np.abs(vec) ** 2 - np.abs(vref) ** 2).max() < 1e-12
    ref_abs2 = np.abs(g['herm_vecs']) ** 2       # reference columns are unsorted
    for k in range(len(lam)):
        rk = ref_abs2[k]
        order = [int(np.argmin(np.abs(rk - (np.abs(vec[k]) ** 2)[:, [c]]).sum(axis=0))) for c in range(3)]
        assert sorted(order) == [0, 1, 2]
        assert np.abs(rk[:, order] - np.abs(vec[k]) ** 2).max() < 1e-10
    v1 = fr.cardano_eqn(g['herm'][0])
    resid = g['herm'][0] @ v1 - v1 * lam[0][None, :]
    assert np.abs(resid).max() < 1e-13


def test_golden_params_to_bsmu(torch, golden):
    g = golden('ref_bsm_u.npz')
    bsm = np.column_stack([g['npang'], g['loglam']])
    smu = fr.angles_to_u(g['sm'])
    worst_mp = 0.0
    worst_ref = 0.0
    for dim in range(3, 9):
        s = g['dim'] == dim
        v = fr.params_to_BSMu(bsm[s], dim, g['energy'][s], mass_eigenvalues=g['mass'][s], sm_u=smu[s])
        got = fr.u_to_fr(g['src'][s], v)
        worst_mp = max(worst_mp, np.abs(got - g['fr_mp'][s]).max())
        good = (g['resid'][s] < 1e-13) & (np.abs(g['fr'][s] - g['fr_mp'][s]).max(axis=1) < 1e-11)
        worst_ref = max(worst_ref, np.abs(got[good] - g['fr'][s][good]).max())
        eye = np.abs(np.einsum('nij,nkj->nik', v, v.conj())) - np.eye(3)
        assert np.abs(eye).max() < 1e-13
    assert worst_mp < FR_TOL and worst_ref < FR_TOL


def test_golden_flux_averaged(torch, golden):
    g = golden('ref_flux.npz')
    worst_mp = worst_ref = 0.0
    for dim in (3, 6):
        for src in ((1, 2, 0), (1, 0, 0), (0, 1, 0)):
            sel = (g['dim'] == dim) & np.all(g['src'] == np.array(src, float), axis=1)
            if not sel.any():
                continue
            got = fr.flux_averaged_BSMu(g['theta'][sel], models.bsm_args(dim, Texture.NONE, src), -2.0, models.bsm11_paramset(dim))
            worst_mp = max(worst_mp, np.abs(got - g['fr_mp'][sel]).max())
            ok = g['ok'][sel]
            good = np.abs(g['fr'][sel][ok] - g['fr_mp'][sel][ok]).max(axis=1) < 1e-11
            worst_ref = max(worst_ref, np.abs(got[ok][good] - g['fr'][sel][ok][good]).max())
    assert worst_mp < FR_TOL and worst_ref < FR_TOL
    # SURVEY 8c spot value, fixed-texture path, scalar call
    theta = [0.307, (1 - 0.02206) ** 2, 0.538, 4.08404, 7.40e-23, 2.494e-21, -43.0]
    got = fr.flux_averaged_BSMu(theta, models.bsm_args(6, Texture.OET), -2.5, models.bsm7_paramset(6))
    assert got.shape == (3,)
    assert np.abs(got - [0.17961929413794903, 0.6433699505955545, 0.17701075526649657]).max() < FR_TOL


def test_golden_notebook_lnprob(torch, golden):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    got = llh.ln_prob(g['theta'], args, asimov, pset)
    ref = g['lnprob']
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin) and np.all(np.isneginf(got[~fin]))
    assert np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL
    # scalar call returns a float, like the reference
    one = llh.ln_prob(list(g['theta'][0]), args, asimov, pset)
    assert isinstance(one, float) and abs(one - (-458.6843569885842)) < LLH_RTOL * 459
    lp = llh.lnprior(g['theta'], pset)
    f = np.isfinite(g['lnprior'])
    assert np.array_equal(np.isfinite(lp), f)
    assert np.max(np.abs(lp[f] - g['lnprior'][f]) / np.maximum(np.abs(g['lnprior'][f]), 1.0)) < 1e-12
    assert pset['s_12_2'].value == g['theta'][-1, 0]      # the Param.value side effect (llh.py:72-73)
    t = llh.triangle_llh(g['theta'][f], args, asimov, pset)
    tf = np.isfinite(t)
    assert np.max(np.abs((t + lp[f])[tf] - ref[f][tf]) / np.abs(ref[f][tf])) < LLH_RTOL
    lp7 = llh.lnprior(g['theta7'], models.bsm7_paramset())
    f7 = np.isfinite(g['lnprior7'])
    assert np.array_equal(np.isfinite(lp7), f7)
    assert np.max(np.abs(lp7[f7] - g['lnprior7'][f7]) / np.abs(g['lnprior7'][f7])) < 1e-12
    assert abs(llh.lnprior([0.31, 0.956, 0.5, 1.0, 0.5, 0.0], pset) - 10.572751418840092) < 1e-11


def test_golden_multi_gaussian(torch, golden):
    g = golden('ref_llh.npz')
    got = llh.multi_gaussian(g['mg_fr'], g['mg_bf'], 0.02)
    fin = np.isfinite(g['mg'])
    assert np.array_equal(np.isfinite(got), fin)
    deep = g['mg'] + 320 > -700      # above the sub-normal band of the reference's pdf (SURVEY 7.3)
    assert np.max(np.abs(got[fin & deep] - g['mg'][fin & deep]) / np.abs(g['mg'][fin & deep])) < LLH_RTOL
    wide = llh.multi_gaussian(g['mg_fr'], g['mg_bf'], 0.2, offset=0)
    assert np.max(np.abs(wide - g['mg_wide'])) < 1e-11
    assert abs(llh.multi_gaussian([.3, .35, .35], [.55, .18, .27], .02) - (-433.2707465833296)) < LLH_RTOL * 433
    rv = llh.GaussianBoundedRV(loc=0.3, sigma=0.1, lower=0.0, upper=1.0)
    from scipy.stats import truncnorm
    x = np.linspace(0.01, 0.99, 17)
    assert np.abs(rv.logpdf(x) - truncnorm(a=-3, b=7, loc=0.3, scale=0.1).logpdf(x)).max() < 1e-12


# ------------------------------------------------------------------ oracle on seeded inputs


def test_sm_only_column_layouts_agree(torch, golden):
    """The SM-only log-posterior has a register-resident specialisation for the reference's own column
    layout (4 mixing coordinates, then the 2 source angles) and a column-map path (theta staged in shared
    memory) for every other layout: the same model with its columns permuted must give the same values,
    in both theta layouts (row-major and SoA), and both must match the oracle."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    from golemflavor_b200.param import ParamSet
    perm = [4, 0, 1, 5, 2, 3]      # interleaved; the order within a tag is what identifies a parameter (param.py:185-199)
    pset_p = ParamSet([pset[k] for k in perm])
    fn, fn_p = llh.LnProb(args, asimov, pset), llh.LnProb(args, asimov, pset_p)
    rng = np.random.default_rng(12)
    theta = models.draw_in_ranges(pset, 5000, rng)
    theta[:50, 0] = rng.uniform(-0.2, 1.2, 50)            # some points outside the prior box
    a, fa, _ = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    b, fb, _ = (x.cpu().numpy() for x in fn_p.evaluate(theta[:, perm], want_fr=True, want_status=True))
    fin = np.isfinite(a)
    assert np.array_equal(fin, np.isfinite(b)) and 4000 < fin.sum() < 5000
    assert np.allclose(a[fin], b[fin], rtol=1e-13, atol=0) and np.array_equal(fa[fin], fb[fin])
    t = torch.as_tensor(theta).cuda()
    soa = t.t().contiguous().t()                           # same values, column-major storage
    assert np.array_equal(fn(soa).cpu().numpy()[fin], a[fin])
    tp = torch.as_tensor(np.ascontiguousarray(theta[:, perm])).cuda()
    assert np.array_equal(fn_p(tp.t().contiguous().t()).cpu().numpy()[fin], b[fin])
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    ref_fr = go.batch_u_to_fr(np.array(go.batch_angles_to_fr(theta[:, 4:6])).astype(float), go.batch_angles_to_u(theta[:, :4])).astype(float)
    ref = go.batch_lnprior(theta, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]) + \
        go.batch_multi_gaussian(ref_fr, go.angles_to_fr(g['asimov_angles']), 0.02)
    assert np.max(np.abs(a[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL


def test_prior_kind_specialisations_and_unnormalised_source_angles(torch, golden):
    """(i) The compile-time column layouts also fix the reference's own prior kinds at compile time; the same layout with
    other kinds must be served by the runtime-kind kernels with the right values (here: a Gaussian prior on dcp / flat
    priors on everything, against the oracle's lnprior + likelihood).  (ii) The SM-only path skips u_to_fr's division by
    sum(source) only while the source sums to one by construction: source angles beyond their natural box
    (sin^4 phi > 1, evaluated by flux_averaged_BSMu without a prior) are normalised like fr.py:535."""
    from golemflavor_b200.enums import PriorsCateg
    from golemflavor_b200.param import Param, ParamSet
    g = golden('ref_llh.npz')
    rng = np.random.default_rng(41)
    bf = go.angles_to_fr(g['asimov_angles'])

    def oracle_lnprob(pset, theta, ref_fr):
        lo, hi = np.array(pset.ranges).T
        kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
        return go.batch_lnprior(theta, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]) + \
            go.batch_multi_gaussian(ref_fr, bf, 0.02)

    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    theta = models.draw_in_ranges(pset, 4000, rng)
    ref_fr = go.batch_u_to_fr(np.array(go.batch_angles_to_fr(theta[:, 4:6])).astype(float), go.batch_angles_to_u(theta[:, :4])).astype(float)
    variants = [ParamSet([Param(name=p.name, value=p.value, seed=p.seed, ranges=p.ranges, std=p.std or 0.5,
                                prior=PriorsCateg.GAUSSIAN if p.name == 'dcp' else p.prior, tag=p.tag) for p in pset]),
                ParamSet([Param(name=p.name, value=p.value, seed=p.seed, ranges=p.ranges, std=p.std, prior=None, tag=p.tag) for p in pset])]
    for other in [pset] + variants:
        got = np.asarray(llh.LnProb(args, asimov, other)(theta))
        ref = oracle_lnprob(other, theta, ref_fr)
        fin = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), fin) and fin.sum() > 100
        assert np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL
    args3, asimov3, pset3 = models.bsm_model_c3(g['asimov_angles'])
    th3 = models.draw_in_ranges(pset3, 4000, rng)
    fr3 = truth.eigh_flux_averaged_fr(th3[:, :4], th3[:, 4:6], model.TEXTURE_ANGLES['OET'], th3[:, 6], 6, models.BINNING, args3.source_ratio)
    flat3 = ParamSet([Param(name=p.name, value=p.value, seed=p.seed, ranges=p.ranges, std=p.std, prior=None, tag=p.tag) for p in pset3])
    for other in (pset3, flat3):
        got = np.asarray(llh.LnProb(args3, asimov3, other)(th3))
        ref = oracle_lnprob(other, th3, fr3)
        fin = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), fin) and fin.sum() > 100
        assert np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL
    # (ii) through gf_flux_averaged_fr in the canonical (packed, 128-bit loads) and in a permuted layout
    theta[:2000, 4] = rng.uniform(1.0, 2.5, 2000)
    ref_fr = np.array([np.asarray(go.u_to_fr(go.angles_to_fr(t[4:6]), go.angles_to_u(t[:4])), dtype=np.float64) for t in theta[::10]])
    perm = [4, 0, 1, 5, 2, 3]
    fa = fr.flux_averaged_BSMu(theta, args, -2.0, pset)
    fb = fr.flux_averaged_BSMu(theta[:, perm], args, -2.0, ParamSet([pset[k] for k in perm]))
    fa, fb = np.asarray(fa), np.asarray(fb)
    assert np.abs(fa[::10] - ref_fr).max() < 1e-13 and np.array_equal(fa, fb)
    assert np.abs(fa.sum(axis=1) - 1).max() < 1e-14


def test_theta_memory_layouts_through_the_c_abi(torch, golden):
    """The compile-time column layouts pick their loads from the theta view: 128-bit loads for packed,
    16-byte aligned rows of an even length, scalar loads at constant offsets for contiguous rows, strided
    loads otherwise.  Same values from every view of the same data, straight through gf_lnprob."""
    g = golden('ref_llh.npz')
    lib = _lib.load()
    rng = np.random.default_rng(31)
    cases = [models.notebook_model(g['asimov_angles']),                                  # 6 columns (SM6)
             models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OUT)]       # 7 columns (FIXED7)
    for args, asimov, pset in cases:
        fn = llh.LnProb(args, asimov, pset)
        nd, n = fn.ndim, 3001
        theta = torch.as_tensor(models.draw_in_ranges(pset, n, rng)).cuda()

        def run(ptr_tensor, offset, ld_point, ld_dim):
            out = torch.empty(n, dtype=torch.float64, device='cuda')
            _lib.check(lib.gf_lnprob(fn.model.ref, C.c_void_p(ptr_tensor.data_ptr() + 8 * offset), n, ld_point, ld_dim, _lib.ptr(out),
                                     None, None, _lib.stream_ptr(torch)))
            return out.cpu().numpy()

        ref = run(theta, 0, nd, 1)                                  # packed rows, 256-byte aligned base
        buf = torch.zeros(nd * n + 1, dtype=torch.float64, device='cuda')
        buf[1:] = theta.reshape(-1)
        assert np.array_equal(run(buf, 1, nd, 1), ref)              # packed rows on an 8-byte boundary only
        wide = torch.zeros((n, nd + 3), dtype=torch.float64, device='cuda')
        wide[:, :nd] = theta
        assert np.array_equal(run(wide, 0, nd + 3, 1), ref)         # padded rows
        soa = theta.t().contiguous()
        assert np.array_equal(run(soa, 0, 1, n), ref)               # column-major
        assert np.isfinite(ref).mean() > 0.5 and not np.isnan(ref).any()


def test_largest_model_sixteen_columns(torch, golden):
    """GF_MAX_DIM = 16 columns: six SM parameters, five prior-only nuisances, four free new-physics mixing
    coordinates (Texture.NONE) and logLam -- the generic path at its limit, against the truth evaluator and the
    oracle's prior; a seventeenth column is refused."""
    from golemflavor_b200.enums import ParamTag
    from golemflavor_b200.param import Param, ParamSet
    g = golden('ref_llh.npz')
    args, asimov, _ = models.bsm_model_c3(g['asimov_angles'], dim=5, texture=Texture.NONE)
    p11 = models.bsm11_paramset(5)
    nuis = [Param(name='nuis%d' % k, value=1.0, ranges=[0., 2.], std=0.3, tag=ParamTag.NUISANCE) for k in range(5)]
    p16 = ParamSet(list(p11)[:6] + nuis + list(p11)[6:])
    for k in (6, 7, 8):                                      # Haar-flat NP coordinates inside the unit box
        p16[11 + k - 6].ranges = [0., 1.]
    fn = llh.LnProb(args, asimov, p16)
    assert fn.ndim == 16
    rng = np.random.default_rng(77)
    theta = models.draw_in_ranges(p16, 2000, rng)
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    ref_fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], theta[:, 11:15], theta[:, 15], 5, models.BINNING, args.source_ratio)
    assert np.abs(frs - ref_fr).max() < FR_TOL and not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
    lo, hi = np.array(p16.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in p16]
    ref = go.batch_lnprior(theta, lo, hi, kind, list(p16.nominal_values), [p.std or 1.0 for p in p16]) + \
        go.batch_multi_gaussian(ref_fr, go.angles_to_fr(g['asimov_angles']), 0.02)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp), fin) and fin.sum() > 1000
    assert np.max(np.abs(lnp[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL
    with pytest.raises(ValueError):
        llh.LnProb(args, asimov, ParamSet(list(p16) + [Param(name='one_too_many', value=0., ranges=[-1., 1.], std=1., tag=ParamTag.NUISANCE)]))


@pytest.mark.parametrize('nbins', [1, 3, 7, 22, 64])
def test_energy_bin_counts_and_interleave_remainders(torch, golden, nbins):
    """The energy-bin loop interleaves 2 bins (log-posterior, scans) or 4 (sampler) and finishes the remainder
    one at a time: every bin count -- one bin, odd counts, counts that are not multiples of four, the maximum
    of 64 -- against the truth evaluator, and the sampler's stored log-posterior against gf_lnprob."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OUT)
    args.binning = np.logspace(np.log10(6e4), np.log10(1e7), nbins + 1)
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(40 + nbins)
    theta = models.draw_in_ranges(pset, 3000, rng)
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OUT'], theta[:, 6], 6, args.binning,
                                      args.source_ratio)
    assert np.abs(frs - ref).max() < FR_TOL and not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
    # same model through the scan kernel (texture mode draws its own samples: compare on those)
    fm = scan.scan_model('texture', dimension=6, texture=Texture.OUT, binning=args.binning)
    th_s, fr_s, _ = scan.scan_samples(fm, 2000, seed=3)
    ref_s = truth.eigh_flux_averaged_fr(th_s[:, :4], th_s[:, 4:6], model.TEXTURE_ANGLES['OUT'], th_s[:, 6], 6, args.binning, np.array([1, 2, 0.]) / 3)
    assert np.abs(fr_s - ref_s).max() < FR_TOL
    h, kept = scan.scan_histogram(fm, 2000, nb=25, seed=3, distributed=False)
    assert kept == 2000 and np.array_equal(h, go.ternary_histogram(fr_s, 25))
    # sampler (four interleaved bins + remainder)
    np.random.seed(1)
    p0 = mcmc.flat_seed(pset, 64)
    smp = mcmc.DeviceEnsembleSampler(64, fn.ndim, fn, seed=3)
    smp.run_mcmc(p0, 6)
    assert np.allclose(fn(smp.chain[:, -1]), smp.lnprobability[:, -1], rtol=1e-11, atol=0)


def test_bsm_fixed_texture_column_layouts_agree(torch, golden):
    """Same for the fixed-texture BSM model: the scripts/fr.py column layout (4 mixing coordinates, 2 mass
    splittings, logLam) runs with compile-time theta indices, any other layout through the column map --
    identical compositions, log-posteriors equal up to the summation order of the prior terms."""
    from golemflavor_b200.param import ParamSet
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OUT)
    perm = [6, 0, 4, 1, 2, 5, 3]       # logLam first, masses interleaved; order within a tag preserved
    fn, fn_p = llh.LnProb(args, asimov, pset), llh.LnProb(args, asimov, ParamSet([pset[k] for k in perm]))
    rng = np.random.default_rng(13)
    theta = models.draw_in_ranges(pset, 20000, rng)
    a, fa, sa = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    b, fb, sb = (x.cpu().numpy() for x in fn_p.evaluate(theta[:, perm], want_fr=True, want_status=True))
    assert np.all(np.isfinite(a)) and np.array_equal(fa, fb) and np.array_equal(sa, sb)
    assert np.allclose(a, b, rtol=1e-13, atol=0)
    assert (sa & _lib.ST_REFINED).any()                  # the near-degenerate fallback is exercised on both paths


def test_production_paramset_of_fr_script_with_golemfit_nuisances(torch, golden):
    """scripts/fr.py:30-90 fits 12 parameters: six SM_ANGLES, five NUISANCE-tagged GolemFit normalisations
    and logLam.  The nuisances only enter the (proprietary) GolemFit likelihood; with the Gaussian stand-in
    they contribute their priors and nothing else: the 12-column model must equal the oracle's prior over all
    twelve columns plus the likelihood of the seven physical ones."""
    from golemflavor_b200.enums import ParamTag, PriorsCateg
    from golemflavor_b200.param import Param, ParamSet
    g = golden('ref_llh.npz')
    args, asimov, p7 = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
    lg, tag = PriorsCateg.LIMITEDGAUSS, ParamTag.NUISANCE
    nuis = [Param(name='convNorm', value=1., seed=[0.5, 2.], ranges=[0.1, 10.], std=0.4, prior=lg, tag=tag),
            Param(name='promptNorm', value=0., seed=[0., 6.], ranges=[0., 20.], std=2.4, prior=lg, tag=tag),
            Param(name='muonNorm', value=1., seed=[0.1, 2.], ranges=[0., 10.], std=0.1, tag=tag),
            Param(name='astroNorm', value=6.9, seed=[0., 5.], ranges=[0., 20.], std=1.5, tag=tag),
            Param(name='astroDeltaGamma', value=2.5, seed=[2.4, 3.], ranges=[-5., 5.], std=0.1, tag=tag)]
    p12 = ParamSet(list(p7)[:6] + nuis + [p7[6]])
    fn = llh.LnProb(args, asimov, p12)
    rng = np.random.default_rng(21)
    theta = models.draw_in_ranges(p12, 4000, rng, seeds=True)
    theta[:, 11] = rng.uniform(*model.SCALE_BOUNDARIES[6], 4000)
    theta[:40, 8] = rng.uniform(-1, 11, 40)                 # some nuisance values outside their box
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    phys = theta[:, [0, 1, 2, 3, 4, 5, 11]]
    ref_fr = truth.eigh_flux_averaged_fr(phys[:, :4], phys[:, 4:6], model.TEXTURE_ANGLES['OET'], phys[:, 6], 6,
                                         models.BINNING, args.source_ratio)
    lo, hi = np.array(p12.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in p12]
    ref = go.batch_lnprior(theta, lo, hi, kind, list(p12.nominal_values), [p.std or 1.0 for p in p12]) + \
        go.batch_multi_gaussian(ref_fr, go.angles_to_fr(g['asimov_angles']), 0.02)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp), fin) and 3900 < fin.sum() < 4000
    assert np.abs(frs[fin] - ref_fr[fin]).max() < FR_TOL
    assert np.max(np.abs(lnp[fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL
    # the nuisance columns do not touch the composition: same values through the 7-column model
    f7 = llh.LnProb(args, asimov, p7)
    _, fr7, _ = (x.cpu().numpy() for x in f7.evaluate(phys, want_fr=True, want_status=True))
    assert np.array_equal(fr7[fin], frs[fin])
    # ... and through the column-map path (this layout has its own compile-time specialisation): logLam first
    perm = [11] + list(range(11))
    fp = llh.LnProb(args, asimov, ParamSet([p12[k] for k in perm]))
    lp, frp, _ = (x.cpu().numpy() for x in fp.evaluate(theta[:, perm], want_fr=True, want_status=True))
    assert np.array_equal(frp[fin], frs[fin]) and np.allclose(lp[fin], lnp[fin], rtol=1e-13, atol=0)
    # the device sampler on the 12-parameter model: every launch shape gives the same chain
    np.random.seed(5)
    p0 = mcmc.flat_seed(p12, 64)
    ref = mcmc.DeviceEnsembleSampler(64, 12, fn, seed=2, mode=1)
    ref.run_mcmc(p0, 8)
    for mode in (0, 2):
        s = mcmc.DeviceEnsembleSampler(64, 12, fn, seed=2, mode=mode)
        s.run_mcmc(p0, 8)
        assert np.array_equal(s.chain, ref.chain)


@pytest.mark.parametrize('texture', ['OET', 'OUT', 'OEU'])
@pytest.mark.parametrize('dim', [3, 6, 8])
def test_bsm_lnprob_against_oracle(torch, golden, texture, dim):
    g = golden('ref_llh.npz')
    rng = np.random.default_rng(25 + dim)
    n = 20000
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=dim, texture=Texture[texture])
    theta = models.draw_in_ranges(pset, n, rng, seeds=True)
    theta[:, 6] = rng.uniform(*model.SCALE_BOUNDARIES[dim], n)
    theta[::97, 0] = -0.01                                   # outside the prior box
    fn = llh.LnProb(args, asimov, pset)
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    lp = go.batch_lnprior(theta, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset])
    inside = np.isfinite(lp)
    ti = theta[inside]
    ref_fr = np.full((n, 3), np.nan)
    ref_fr[inside] = truth.eigh_flux_averaged_fr(ti[:, :4], ti[:, 4:6], np.broadcast_to(model.TEXTURE_ANGLES[texture], (len(ti), 4)),
                                                 ti[:, 6], dim, models.BINNING, args.source_ratio)
    assert np.all(np.isneginf(lnp[~inside])) and np.all(st[~inside] & _lib.ST_OUT_OF_PRIOR)
    assert not np.any(st[inside] & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY | _lib.ST_OUT_OF_PRIOR))
    assert np.abs(frs[inside] - ref_fr[inside]).max() < FR_TOL
    assert np.abs(frs[inside].sum(axis=1) - 1).max() < 1e-14
    with np.errstate(invalid='ignore'):
        ref = np.where(inside, lp + go.batch_multi_gaussian(np.nan_to_num(ref_fr), go.angles_to_fr(g['asimov_angles']), 0.02), -np.inf)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp), fin)
    # LLH = -|d|^2/(2 s^2) + const amplifies an fr error of 1e-10 by |d|/s^2 ~ 2e3: bound the
    # comparison by the propagated fr tolerance as well as by the relative one
    tol = np.maximum(LLH_RTOL * np.abs(ref[fin]), 0.0) + 0
    d = np.linalg.norm(ref_fr[fin] - np.array(go.angles_to_fr(g['asimov_angles'])), axis=1)
    tol = np.maximum(tol, 2e-11 * d / 0.02 ** 2)
    assert np.all(np.abs(lnp[fin] - ref[fin]) <= tol)


def _prior_tables(pset):
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    return lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]


def _source_of(kind, cols):
    if kind == 'angles':
        return go.batch_angles_to_fr(cols)
    if kind == 'x':
        return np.column_stack([cols[:, 0], 1.0 - cols[:, 0], np.zeros(len(cols))])
    return cols


def test_golden_config1_and_sampled_source_models(torch, golden):
    """BASELINE config 1 (three raw source ratios, PMNS fixed at NUFIT_U: `col_src3`, SM specialisation) and the
    sampled-source compositions of llh.py:94-112 on the binned BSM path (GENERIC specialisation), through
    gf_lnprob and gf_flux_averaged_fr, against fixtures from the unmodified reference (make_golden_r2.py)."""
    g, gl = golden('ref_src.npz'), golden('ref_llh.npz')
    args, asimov, pset = models.sm_fit_c1(gl['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    assert list(fn.model.struct.col_src3) == [0, 1, 2] and fn.model.struct.no_bsm == 1
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(g['c1_theta'], want_fr=True, want_status=True))
    fin = np.isfinite(g['c1_lnprob'])
    inside = np.all((g['c1_theta'] >= 1e-6) & (g['c1_theta'] <= 1), axis=1)
    assert np.array_equal(np.isfinite(lnp), fin) and np.all(st[~inside] & _lib.ST_OUT_OF_PRIOR) and np.all(st[inside] == 0)
    assert np.abs(frs[inside] - g['c1_fr'][inside]).max() < 1e-14
    assert np.max(np.abs(lnp[fin] - g['c1_lnprob'][fin]) / np.abs(g['c1_lnprob'][fin])) < LLH_RTOL
    # the reference signature (scalar theta) and the flux-averaged entry point on the no-BSM branch (fr.py:437-438)
    assert abs(llh.ln_prob(list(g['c1_theta'][0]), args, asimov, pset) - g['c1_lnprob'][0]) < LLH_RTOL * abs(g['c1_lnprob'][0])
    a2 = argparse.Namespace(source_ratio=[1, 2, 0], no_bsm=True, binning=g['binning'], dimension=6, texture=Texture.OET)
    assert np.abs(fr.flux_averaged_BSMu(g['c1_theta'][inside], a2, -2.0, pset) - g['c1_fr'][inside]).max() < 1e-14
    for kind in ('angles', 'x', 'ratios'):
        nsrc = models.SOURCE_KINDS[kind]
        for tex, dim in (('OET', 6), ('OUT', 6), ('OEU', 3), ('OET', 8)):
            sel = (g['sb_kind'] == kind) & (g['sb_tex'] == tex) & (g['sb_dim'] == dim)
            theta = np.column_stack([g['sb_sm'][sel], g['sb_src'][sel][:, :nsrc], g['sb_loglam'][sel]])
            for first in (False, True):
                args, asimov, ps = models.bsm_sampled_source(gl['asimov_angles'], kind, dim, Texture[tex], source_first=first)
                th = np.column_stack([theta[:, 6:6 + nsrc], theta[:, :6], theta[:, -1:]]) if first else theta
                fn = llh.LnProb(args, asimov, ps)
                lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(th, want_fr=True, want_status=True))
                assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY | _lib.ST_OUT_OF_PRIOR))
                assert np.abs(frs - g['sb_fr'][sel]).max() < FR_TOL, (kind, tex, dim)
                assert np.abs(fr.flux_averaged_BSMu(th, args, -2.0, ps) - frs).max() == 0.0
                ref = go.batch_lnprior(th, *_prior_tables(ps)) + g['sb_llh'][sel]
                ok = np.isfinite(ref)
                assert np.array_equal(np.isfinite(lnp), ok)
                d = np.linalg.norm(g['sb_fr'][sel][ok] - g['bf'], axis=1)
                assert np.all(np.abs(lnp[ok] - ref[ok]) <= np.maximum(LLH_RTOL * np.abs(ref[ok]), 2e-10 * d / 0.02 ** 2))


@pytest.mark.parametrize('kind', ['angles', 'x', 'ratios'])
def test_sampled_source_bsm_lnprob_against_oracle(torch, golden, kind):
    """GF_SPEC_GENERIC with a sampled source AND a SCALE column (gf_model.cuh: per-point 1 / (S wsum)
    normalisation, one bin chain in the scans, two in k_lnprob) on 20 000 points per texture against the
    oracle: LAPACK-truth compositions + batch lnprior + batch multi_gaussian."""
    g = golden('ref_llh.npz')
    bf = np.array(go.angles_to_fr(g['asimov_angles']))
    nsrc = models.SOURCE_KINDS[kind]
    for tex, dim in (('OET', 6), ('OUT', 4)):
        rng = np.random.default_rng(31 + dim)
        n = 20000
        args, asimov, pset = models.bsm_sampled_source(g['asimov_angles'], kind, dim, Texture[tex])
        theta = models.draw_in_ranges(pset, n, rng, seeds=False)
        theta[:, :6] = models.draw_in_ranges(models.bsm7_paramset(dim), n, rng, seeds=True)[:, :6]
        theta[::89, 6] = 1.5                                   # source parameter outside its box
        fn = llh.LnProb(args, asimov, pset)
        assert fn.model.struct.col_scale == 6 + nsrc and fn.model.struct.no_bsm == 0
        lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
        lp = go.batch_lnprior(theta, *_prior_tables(pset))
        inside = np.isfinite(lp)
        ti = theta[inside]
        src = _source_of(kind, ti[:, 6:6 + nsrc])
        ref_fr = truth.eigh_flux_averaged_fr(ti[:, :4], ti[:, 4:6], np.broadcast_to(model.TEXTURE_ANGLES[tex], (len(ti), 4)),
                                             ti[:, -1], dim, models.BINNING, src)
        assert np.all(np.isneginf(lnp[~inside])) and np.all(st[~inside] & _lib.ST_OUT_OF_PRIOR)
        assert not np.any(st[inside] & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY | _lib.ST_OUT_OF_PRIOR))
        assert np.abs(frs[inside] - ref_fr).max() < FR_TOL
        with np.errstate(invalid='ignore'):
            ref = lp[inside] + go.batch_multi_gaussian(ref_fr, bf, 0.02)
        fin = np.isfinite(ref)
        assert np.array_equal(np.isfinite(lnp[inside]), fin)
        d = np.linalg.norm(ref_fr[fin] - bf, axis=1)
        assert np.all(np.abs(lnp[inside][fin] - ref[fin]) <= np.maximum(LLH_RTOL * np.abs(ref[fin]), 2e-11 * d / 0.02 ** 2))
        # the same model through the scan kernels (ILP 1 instantiation of the generic bin loop): draws + compositions
        fm = model.flatten(args, None, pset, likelihood='FLAT')
        th_s, fr_s, st_s = scan.scan_samples(fm, 4000, seed=7)
        src_s = _source_of(kind, th_s[:, 6:6 + nsrc])
        ref_s = truth.eigh_flux_averaged_fr(th_s[:, :4], th_s[:, 4:6], np.broadcast_to(model.TEXTURE_ANGLES[tex], (4000, 4)),
                                            th_s[:, -1], dim, models.BINNING, src_s)
        assert np.abs(fr_s - ref_s).max() < FR_TOL and not np.any(st_s & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
        h, kept = scan.scan_histogram(fm, 4000, nb=25, seed=7, distributed=False)
        assert kept == 4000 and np.array_equal(h, go.ternary_histogram(fr_s, 25))


def test_config1_lnprob_and_sampler_against_oracle(torch, golden):
    """BASELINE config 1 at scale and inside the device-resident sampler (`col_src3` on the SM specialisation):
    20 000 points against the oracle's u_to_fr(theta, NUFIT_U) + multi_gaussian; the sampler's chain is replayed by
    the NumPy stretch move scoring proposals with the ORACLE (longdouble) log-posterior."""
    import ref_sampler
    g = golden('ref_llh.npz')
    bf = np.array(go.angles_to_fr(g['asimov_angles']))
    args, asimov, pset = models.sm_fit_c1(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(41)
    theta = rng.uniform(1e-6, 1.0, (20000, 3))
    theta[::53, 2] = 1.2
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    inside = np.all((theta >= 1e-6) & (theta <= 1), axis=1)
    ref_fr = go.batch_u_to_fr(theta[inside], np.broadcast_to(go.NUFIT_U, (inside.sum(), 3, 3))).astype(np.float64)
    assert np.all(np.isneginf(lnp[~inside])) and np.abs(frs[inside] - ref_fr).max() < 1e-14
    ref = go.batch_multi_gaussian(ref_fr, bf, 0.02)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp[inside]), fin)
    assert np.max(np.abs(lnp[inside][fin] - ref[fin]) / np.abs(ref[fin])) < LLH_RTOL

    def oracle_lnprob(q):
        q = np.atleast_2d(q)
        ok = np.all((q >= 1e-6) & (q <= 1), axis=1)
        out = np.full(len(q), -np.inf)
        if ok.any():
            f = go.batch_u_to_fr(q[ok], np.broadcast_to(go.NUFIT_U, (ok.sum(), 3, 3))).astype(np.float64)
            out[ok] = go.batch_multi_gaussian(f, bf, 0.02)
        return out

    k = 100                                             # BASELINE config 1: 100 walkers
    p0 = np.array([1.0, 0.0, 0.0]) * rng.uniform(0.5, 0.9, (k, 1)) + rng.uniform(1e-3, 0.05, (k, 3))
    l0 = fn(p0)
    assert np.all(np.isfinite(l0)) and np.max(np.abs(l0 - oracle_lnprob(p0)) / np.abs(l0)) < LLH_RTOL
    chains = []
    for mode in (0, 1, 2, 3):
        s = mcmc.DeviceEnsembleSampler(k, 3, fn, seed=9, mode=mode)
        s.run_mcmc(p0, 200)
        chains.append((s.chain, s.lnprobability))
        assert np.array_equal(s.chain, chains[0][0]) and np.array_equal(s.lnprobability, chains[0][1]), mode
    _, _, rchain, racc = ref_sampler.run(oracle_lnprob, p0, oracle_lnprob(p0), 200, seed=9)
    # identical unless an acceptance test falls within the ~1e-13 difference between the fp64 kernel and the oracle
    assert np.mean(chains[0][0] == rchain) > 0.99
    assert 0.2 < np.mean(racc) / 200 < 0.8


def test_device_sampler_sampled_source_bsm_model(torch, golden):
    """SRCANGLES + SCALE inside the sampler (GENERIC specialisation, ILP 2): all launch shapes give the same chain, the
    stored log-posteriors are gf_lnprob's for the stored positions, and the chain replays under the NumPy stretch move."""
    import ref_sampler
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_sampled_source(g['asimov_angles'], 'angles', 6, Texture.OET)
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(17)
    k = 128
    p0 = models.draw_in_ranges(models.bsm7_paramset(6), k, rng, seeds=True)
    p0 = np.column_stack([p0[:, :6], rng.uniform(0.8, 1.0, k), rng.uniform(0.6, 1.0, k), rng.uniform(-50, -35, k)])
    ref = mcmc.DeviceEnsembleSampler(k, fn.ndim, fn, seed=21, mode=1)
    ref.run_mcmc(p0, 25)
    for mode, nc in ((0, 0), (2, 0), (3, 2)):
        s = mcmc.DeviceEnsembleSampler(k, fn.ndim, fn, seed=21, mode=mode, cluster_blocks=nc)
        s.run_mcmc(p0, 25)
        assert np.array_equal(s.chain, ref.chain) and np.array_equal(s.lnprobability, ref.lnprobability), (mode, nc)
    assert np.allclose(fn(ref.chain[:, -1]), ref.lnprobability[:, -1], rtol=1e-11, atol=0)
    _, _, rchain, _ = ref_sampler.run(lambda q: fn(q), p0, fn(p0), 25, seed=21)
    assert np.mean(ref.chain == rchain) > 0.99
    assert 0.02 < ref.acceptance_fraction.mean() < 0.9


def test_anarchic_free_np_angles_against_oracle(torch):
    rng = np.random.default_rng(9)
    n = 20000
    dim = 6
    pset = models.bsm11_paramset(dim)
    theta = models.draw_in_ranges(pset, n, rng, seeds=True)
    theta[:, 6:9] = rng.uniform(0, 1, (n, 3))
    theta[:, 9] = rng.uniform(0, 2 * np.pi, n)
    theta[:, 10] = rng.uniform(*model.SCALE_BOUNDARIES[dim], n)
    got = fr.flux_averaged_BSMu(theta, models.bsm_args(dim, Texture.NONE, (1, 0, 0)), -2.0, pset)
    ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], theta[:, 6:10], theta[:, 10], dim, models.BINNING, [1, 0, 0])
    assert np.abs(got - ref).max() < FR_TOL


def test_reference_cardano_restatement_where_well_conditioned(torch):
    """Parity against the float128 restatement of the reference's own Cardano path on the points
    where that path is well-conditioned (unitarity residual < 1e-13)."""
    rng = np.random.default_rng(4)
    n = 3000
    dim = 6
    pset = models.bsm7_paramset(dim)
    theta = models.draw_in_ranges(pset, n, rng, seeds=True)
    theta[:, 6] = rng.uniform(*model.SCALE_BOUNDARIES[dim], n)
    got = fr.flux_averaged_BSMu(theta, models.bsm_args(dim, Texture.OUT), -2.0, pset)
    ref, resid = go.batch_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OUT'], theta[:, 6], dim,
                                           models.BINNING, np.array([1, 2, 0.]) / 3)
    good = resid < 1e-13
    assert good.mean() > 0.3   # the reference's float128 Cardano is itself ill-conditioned on the rest (SURVEY 7.1)
    assert np.abs(got[good] - ref[good]).max() < FR_TOL


def test_ragged_sizes_around_the_block_boundaries_of_the_multi_point_kernels(torch, golden):
    """The compile-time-layout kernels evaluate two points per thread (rows i and i + 64 of a 128-point block; the SM-only
    kernel loads both rows up front and re-reads the last row for a slot past the end): every n around the 64- and
    128-point boundaries must give exactly the first n values of a larger batch, write nothing past n, and do so in every
    theta view (packed rows, padded rows, column-major)."""
    g = golden('ref_llh.npz')
    lib = _lib.load()
    rng = np.random.default_rng(77)
    for args, asimov, pset in (models.notebook_model(g['asimov_angles']), models.bsm_model_c3(g['asimov_angles'])):
        fn = llh.LnProb(args, asimov, pset)
        nd = fn.ndim
        theta = torch.as_tensor(models.draw_in_ranges(pset, 400, rng)).cuda()
        full = fn(theta)
        wide = torch.zeros((400, nd + 1), dtype=torch.float64, device='cuda')
        wide[:, :nd] = theta
        for n in (1, 2, 63, 64, 65, 127, 128, 129, 191, 193, 257):
            soa = theta[:n].t().contiguous()
            for ptr, ldp, ldd in ((theta, nd, 1), (wide, nd + 1, 1), (soa, 1, n)):
                out = torch.full((n + 3,), 7.0, dtype=torch.float64, device='cuda')
                frs = torch.full((n + 1, 3), 7.0, dtype=torch.float64, device='cuda')
                st = torch.full((n + 1,), 255, dtype=torch.uint8, device='cuda')
                _lib.check(lib.gf_lnprob(fn.model.ref, _lib.ptr(ptr), n, ldp, ldd, _lib.ptr(out), _lib.ptr(frs), _lib.ptr(st), _lib.stream_ptr(torch)))
                assert torch.equal(out[:n], full[:n]) and bool((out[n:] == 7.0).all()), (nd, n, ldp, ldd)
                assert bool((frs[n:] == 7.0).all()) and int(st[n]) == 255


def test_layouts_devices_and_edge_cases(torch, golden):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    th = torch.as_tensor(g['theta']).cuda()
    a = fn(th)
    assert a.is_cuda and a.shape == (300,)
    # SoA layout through the C ABI directly
    soa = th.t().contiguous()
    out = torch.empty(300, dtype=torch.float64, device='cuda')
    _lib.check(_lib.load().gf_lnprob(fn.model.ref, _lib.ptr(soa), 300, 1, 300, _lib.ptr(out), None, None, _lib.stream_ptr(torch)))
    assert torch.equal(out, a)
    # host-buffer pipeline: pageable and pinned, ragged sizes across the chunk boundary
    rng = np.random.default_rng(0)
    big = models.draw_in_ranges(pset, (1 << 18) * 2 + 12345, rng)
    ref = fn(big)
    assert np.array_equal(fn.evaluate_host(big), ref)
    pinned = torch.as_tensor(big).pin_memory()
    outp = torch.empty(len(big), dtype=torch.float64).pin_memory()
    fn.evaluate_host(pinned.numpy(), out=outp.numpy())
    assert np.array_equal(outp.numpy(), ref)
    # empty input
    assert fn(np.empty((0, 6))).shape == (0,)
    assert fr.angles_to_u(np.empty((0, 4))).shape == (0, 3, 3)
    # NaN theta fails the box test `lo <= v <= hi` exactly like the reference (llh.py:74-78): -inf, never NaN
    bad = g['theta'][:4].copy()
    bad[1, 2] = np.nan
    lnp, st = (x.cpu().numpy() for x in fn.evaluate(bad, want_status=True))
    assert np.isneginf(lnp[1]) and (st[1] & _lib.ST_OUT_OF_PRIOR) and not np.isnan(lnp).any()
    assert np.array_equal(lnp[[0, 2, 3]], g['lnprob'][[0, 2, 3]]) or np.allclose(lnp[[0, 2, 3]], g['lnprob'][[0, 2, 3]], rtol=1e-10)
    # degenerate Hamiltonians (exactly diagonal / zero) must not produce NaN (SURVEY 7.5)
    lam, vec, st = fr.eigh3(np.array([np.diag([1.0, 2.0, 3.0]), np.zeros((3, 3)), np.eye(3)], dtype=complex))
    assert np.isfinite(vec.view(float)).all() and np.allclose(lam[0], [1, 2, 3])
    assert np.abs(np.abs(np.einsum('nij,nkj->nik', vec, vec.conj())) - np.eye(3)).max() < 1e-14


# ------------------------------------------------------------------ scans and histograms
@pytest.mark.parametrize('mode', ['unitary', 'x', 'texture', 'anarchic'])
def test_scan_samples_against_oracle(torch, mode):
    from scipy.special import ndtri
    from scipy.stats import norm
    fm = scan.scan_model(mode, source_ratio=(1, 2, 0), dimension=6, texture=Texture.OET)
    pset = scan.scan_paramset(mode, 6)
    n, first, seed = 30000, (1 << 32) - 1000, 26
    theta, frs, st = scan.scan_samples(fm, n, seed=seed, first_index=first)
    # the draw convention of include/golemflavor_b200.h restated with the oracle's Philox
    ref_theta = np.empty_like(theta)
    for k, p in enumerate(pset):
        u = go.philox_uniforms(seed, first, n, block=k // 4)[:, k % 4]
        lo, hi = p.ranges
        if p.prior.name == 'UNIFORM':
            ref_theta[:, k] = lo + u * (hi - lo)
        else:
            a, b = norm.cdf((lo - p.nominal_value) / p.std), norm.cdf((hi - p.nominal_value) / p.std)
            ref_theta[:, k] = np.clip(p.nominal_value + p.std * ndtri(a + u * (b - a)), lo, hi)
    scale = np.maximum(np.abs(ref_theta), 1e-300)
    assert np.max(np.abs(theta - ref_theta) / scale) < 1e-11
    lo, hi = np.array(pset.ranges).T
    assert np.all(theta >= lo) and np.all(theta <= hi)
    # compositions from the oracle on the device-drawn theta
    if mode == 'unitary':
        ref = go.batch_u_to_fr(np.array([1, 2, 0.]) / 3, go.batch_angles_to_u(theta)).astype(float)
    elif mode == 'x':
        src = np.column_stack([theta[:, 4], 1 - theta[:, 4], np.zeros(n)])
        ref = go.batch_u_to_fr(src, go.batch_angles_to_u(theta[:, :4])).astype(float)
    elif mode == 'texture':
        ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], theta[:, 6], 6,
                                          models.BINNING, np.array([1, 2, 0.]) / 3)
    else:
        ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], theta[:, 6:10], theta[:, 10], 6,
                                          models.BINNING, np.array([1, 2, 0.]) / 3)
    assert np.abs(frs - ref).max() < FR_TOL
    assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
    # histogram: bit-exact np.histogramdd of the device compositions, and the fused scan kernel
    # must reproduce it exactly (same draws, same arithmetic), for smem-resident and global grids
    for nb in (25, 200):
        ref_h = go.ternary_histogram(frs, nb)
        assert np.array_equal(scan.ternary_histogram(frs, nb), ref_h)
        h, kept = scan.scan_histogram(fm, n, nb=nb, seed=seed, first_index=first, distributed=False)
        assert kept == ref_h.sum() == n
        assert np.array_equal(h, ref_h)


@pytest.mark.parametrize('mode', ['unitary', 'x', 'texture', 'anarchic'])
def test_scan_column_map_kernels_on_permuted_layouts(torch, mode):
    """The scan kernels have compile-time specialisations for the layouts scan.scan_paramset produces; any
    other column order runs the column-map kernels.  Same checks on a model with its columns rotated:
    compositions against the truth evaluator on the device-drawn sample, fused histogram bit-exact."""
    from golemflavor_b200.enums import ParamTag
    from golemflavor_b200.param import Param, ParamSet
    pset = scan.scan_paramset(mode, 6)
    n = len(pset)
    cnt, seed = 20000, 11
    if mode == 'unitary':      # one tag only (its order identifies the parameters): shift the columns by a spectator
        pp = ParamSet([Param(name='spectator', value=0.5, ranges=[0., 1.], std=0.1, tag=ParamTag.NUISANCE)] + list(pset))
        fm = scan.scan_model(mode, source_ratio=(1, 2, 0), paramset=pp)
        theta_p, frs, st = scan.scan_samples(fm, cnt, seed=seed)
        theta = theta_p[:, 1:]
    else:                      # logLam first: the relative order within each tag is kept
        perm = [n - 1] + list(range(n - 1))
        pp = ParamSet([pset[k] for k in perm])
        fm = scan.scan_model(mode, source_ratio=(1, 2, 0), dimension=6, texture=Texture.OET, paramset=pp)
        theta_p, frs, st = scan.scan_samples(fm, cnt, seed=seed)
        theta = np.empty_like(theta_p)
        theta[:, perm] = theta_p                            # back to the canonical column order
    lo, hi = np.array(pset.ranges).T
    assert np.all(theta >= lo) and np.all(theta <= hi)
    if mode == 'unitary':
        ref = go.batch_u_to_fr(np.array([1, 2, 0.]) / 3, go.batch_angles_to_u(theta)).astype(float)
    elif mode == 'x':
        src = np.column_stack([theta[:, 4], 1 - theta[:, 4], np.zeros(cnt)])
        ref = go.batch_u_to_fr(src, go.batch_angles_to_u(theta[:, :4])).astype(float)
    elif mode == 'texture':
        ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], theta[:, 6], 6,
                                          models.BINNING, np.array([1, 2, 0.]) / 3)
    else:
        ref = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], theta[:, 6:10], theta[:, 10], 6,
                                          models.BINNING, np.array([1, 2, 0.]) / 3)
    assert np.abs(frs - ref).max() < FR_TOL
    assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
    for nb in (25, 200):
        h, kept = scan.scan_histogram(fm, cnt, nb=nb, seed=seed, distributed=False)
        assert kept == cnt and np.array_equal(h, go.ternary_histogram(frs, nb))


def test_scan_is_shard_and_geometry_invariant(torch):
    fm = scan.scan_model('unitary')
    n = 3_000_000
    full, kept = scan.scan_histogram(fm, n, nb=25, seed=7, distributed=False)
    assert kept == n == full.sum()
    acc = np.zeros_like(full)
    for r in range(5):                       # 5 uneven shards == what 5 ranks would compute
        start, cnt = scan.shard_range(n, r, 5)
        h, _ = scan.scan_histogram(fm, cnt, nb=25, seed=7, first_index=start, distributed=False)
        acc += h
    assert np.array_equal(acc, full)
    other, _ = scan.scan_histogram(fm, n, nb=25, seed=8, distributed=False)
    assert not np.array_equal(other, full)
    # Haar-flat draws: every column of |U|^2 is uniform on the simplex -> mean composition for a
    # (1,0,0) source is (1/2, 1/4, 1/4) (docs/source/statistics.rst:373-385)
    fm1 = scan.scan_model('unitary', source_ratio=(1, 0, 0))
    _, frs, _ = scan.scan_samples(fm1, 400000, seed=1)
    assert np.allclose(frs.mean(axis=0), [0.5, 0.25, 0.25], atol=2e-3)


def test_histogram_edge_cases(torch):
    rng = np.random.default_rng(3)
    f = rng.dirichlet([1, 1, 1], 200000)
    f[:300, 0] = np.arange(300) / 26.0
    f[300:600, 1] = np.arange(300) * (1.0 / 26.0)
    f[600:900, 2] = np.nextafter(np.arange(300) / 201.0, 0)
    f[900:905] = [[1, 0, 0], [0, 1, 0], [0, 0, 1], [1.0000000001, 0, 0], [np.nan, 0.5, 0.5]]
    for nb in (0, 1, 25, 125, 200):
        assert np.array_equal(scan.ternary_histogram(f, nb), go.ternary_histogram(f, nb)), nb
    assert scan.ternary_histogram(np.empty((0, 3)), 25).sum() == 0


# ------------------------------------------------------------------ full-size properties
def test_full_size_properties(torch, golden):
    """BASELINE sizes: 4096-walker batches x many chains; properties that need no oracle."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(1)
    n = 4096 * 256
    theta = torch.as_tensor(models.draw_in_ranges(pset, n, rng)).cuda()
    lnp, frs, st = fn.evaluate(theta, want_fr=True, want_status=True)
    assert not bool((st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY)).any())
    assert float((frs.sum(dim=1) - 1).abs().max()) < 1e-14 and float(frs.min()) >= 0.0
    # determinism and batch-independence: any sub-batch gives bit-identical values
    lnp2 = fn(theta[12345:12345 + 4096])
    assert torch.equal(lnp2, lnp[12345:12345 + 4096])
    # the likelihood depends on theta only through fr: recompute it from fr with the stand-alone op
    mg = llh.multi_gaussian(frs, list(fn.model.struct.fr_bf), 0.02)
    lp = llh.lnprior(theta, pset)
    fin = torch.isfinite(lnp)
    assert torch.equal(torch.isfinite(mg + lp), fin)
    assert float(((mg + lp)[fin] - lnp[fin]).abs().max()) < 1e-9
    # source-linearity of the transition: fr(s1 + s2) ~ fr(s1) + fr(s2) before normalisation
    fa = fr.flux_averaged_BSMu(theta[:65536], models.bsm_args(6, Texture.OET, (1, 0, 0)), -2, pset)
    fb = fr.flux_averaged_BSMu(theta[:65536], models.bsm_args(6, Texture.OET, (0, 1, 0)), -2, pset)
    fc = fr.flux_averaged_BSMu(theta[:65536], models.bsm_args(6, Texture.OET, (1, 2, 0)), -2, pset)
    assert float((fc - (fa + 2 * fb) / 3).abs().max()) < 1e-13


def test_emcee_driver_on_gpu_lnprob(torch, golden, capsys):
    """Config 1/2-shaped end-to-end: the bundled stretch-move sampler scoring every half-ensemble
    with one kernel launch recovers the injected composition."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    np.random.seed(25)
    nwalkers = 128
    p0 = mcmc.flat_seed(pset, nwalkers)
    p0[:, 4] = np.random.uniform(0.9, 1.0, nwalkers)     # start near the injected (1,0,0) source
    p0[:, 5] = np.random.uniform(0.8, 1.0, nwalkers)
    lib = _lib.load()
    before = lib.gf_launch_count()
    samples = mcmc.mcmc(p0, fn, 6, nwalkers, burnin=300, nsteps=300, seed=2, device=False)   # host-loop sampler
    launches = lib.gf_launch_count() - before
    assert samples.shape == (nwalkers * 300, 6)
    assert launches == 2 * 600 + 2               # two half-ensembles per step + two initial full scores
    sampler = mcmc.mcmc.last_sampler
    assert isinstance(sampler, mcmc.EnsembleSampler)
    assert 0.1 < sampler.acceptance_fraction.mean() < 0.8
    measured = fr.u_to_fr(fr.angles_to_fr(samples[:, 4:6]), fr.angles_to_u(samples[:, :4]))
    bf = np.array(go.angles_to_fr(g['asimov_angles']))
    assert np.abs(np.median(measured, axis=0) - bf).max() < 0.03


# ------------------------------------------------------------------ device-resident ensemble sampler
def test_device_sampler_replays_numpy_stretch_move(torch, golden):
    """gf_ensemble_run against the NumPy stretch-move restatement, both scoring proposals with the
    CUDA log-posterior: identical chains (the acceptance test can only differ on a measure-zero tie)."""
    import ref_sampler
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(0)
    k = 64
    p0 = models.draw_in_ranges(pset, k, rng, seeds=True)
    p0[:, 4], p0[:, 5] = rng.uniform(.9, 1, k), rng.uniform(.8, 1, k)
    l0 = fn(p0)
    s = mcmc.DeviceEnsembleSampler(k, 6, fn, seed=5)
    lib = _lib.load()
    before = lib.gf_launch_count()
    pos, lnp, _ = s.run_mcmc(p0, 120)
    assert lib.gf_launch_count() - before == 2           # initial scoring + ONE launch for the whole chain
    rp, rl, rchain, racc = ref_sampler.run(lambda q: fn(q), p0, l0, 120, seed=5)
    same = np.mean(s.chain == rchain)
    assert same > 0.999, same
    assert s.chain.shape == (k, 120, 6) and s.lnprobability.shape == (k, 120)
    assert np.array_equal(s.lnprobability[:, -1], lnp)
    assert np.allclose(s.acceptance_fraction, racc / 120.0) and 0.2 < s.acceptance_fraction.mean() < 0.7
    # continue: pos0=None picks up where the run stopped, with fresh randomness
    s.run_mcmc(None, 30)
    _, _, rchain2, _ = ref_sampler.run(lambda q: fn(q), rp, rl, 30, seed=5, step0=120)
    assert np.mean(s.chain[:, 120:] == rchain2) > 0.999 and s.chain.shape[1] == 150


def test_device_sampler_many_chains_and_launch_paths(torch, golden):
    """Batched independent chains through the four launch shapes -- one cluster per chain (ensemble in
    distributed shared memory), one block per chain, one cooperative grid launch, one launch per
    half-step (batch too large for co-residency) -- must give identical chains, and a sub-set of chains
    must not depend on what else is in the batch."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(2)
    k, nchains, nsteps = 32, 24000, 6       # 3000 blocks of 128 threads: more than 148 SMs hold at once
    p0 = models.draw_in_ranges(pset, k * nchains, rng, seeds=True).reshape(nchains, k, 6)
    p0[:, :, 4], p0[:, :, 5] = rng.uniform(.9, 1, (nchains, k)), rng.uniform(.8, 1, (nchains, k))
    lib = _lib.load()
    big = mcmc.DeviceEnsembleSampler(k, 6, fn, nchains=nchains, seed=3, mode=1)    # grid barrier; not co-resident
    before = lib.gf_launch_count()
    big.run_mcmc(p0, nsteps)
    assert lib.gf_launch_count() - before == 1 + 3 * nsteps     # scoring + (2 half-steps + 1 store) per step
    for mode in (0, 2, 3):                                      # auto (= cluster per chain), block per chain, cluster per chain
        blk = mcmc.DeviceEnsembleSampler(k, 6, fn, nchains=nchains, seed=3, mode=mode)
        before = lib.gf_launch_count()
        blk.run_mcmc(p0, nsteps)
        assert lib.gf_launch_count() - before == 2              # scoring + ONE launch
        assert np.array_equal(blk.chain, big.chain) and np.array_equal(blk.acceptance_fraction, big.acceptance_fraction)
        assert np.array_equal(blk.lnprobability, big.lnprobability)
    sub = slice(4100, 4110)
    coop = mcmc.DeviceEnsembleSampler(k, 6, fn, nchains=10, seed=3, chain0=4100, mode=1)   # co-resident: cooperative launch
    before = lib.gf_launch_count()
    coop.run_mcmc(p0[sub], nsteps)
    assert lib.gf_launch_count() - before == 2
    assert np.array_equal(big.chain[sub], coop.chain)
    assert big.chain.shape == (nchains, k, nsteps, 6) and big.acceptance_fraction.shape == (nchains, k)
    # block mode with several walker pairs per thread (2 x 300 > 256 threads), clusters of every size with
    # partly filled CTAs, and ensembles too large for a cluster (auto falls back to the grid path)
    for kk, shapes in ((600, ((2, 0), (3, 0), (3, 2), (3, 8), (3, 16))), (4096, ((0, 0), (3, 8), (3, 16))), (10000, ((0, 0),))):
        q0 = models.draw_in_ranges(pset, kk, rng, seeds=True)
        q0[:, 4], q0[:, 5] = rng.uniform(.9, 1, kk), rng.uniform(.8, 1, kk)
        b = mcmc.DeviceEnsembleSampler(kk, 6, fn, seed=8, mode=1)
        b.run_mcmc(q0, 5)
        for mode, nc in shapes:
            a = mcmc.DeviceEnsembleSampler(kk, 6, fn, seed=8, mode=mode, cluster_blocks=nc)
            pa, la, _ = a.run_mcmc(q0, 5)
            assert np.array_equal(a.chain, b.chain), (kk, mode, nc)
            assert np.array_equal(pa, b.chain[:, -1]) and np.array_equal(la, b.lnprobability[:, -1])
    with pytest.raises(ValueError):
        mcmc.DeviceEnsembleSampler(20000, 6, fn, seed=8, mode=3).run_mcmc(models.draw_in_ranges(pset, 20000, rng, seeds=True), 1)


def test_device_sampler_thinning_small_ensembles_and_continuation(torch, golden):
    """Edge shapes of the device sampler in every launch shape: thinning with a step count that is not a
    multiple of the stride, the smallest ensemble emcee allows (2 ndim walkers), non-power-of-two half-ensembles, several
    chains, no stored log-posterior, and continuation of a run (global step counter) -- all compared with a
    single unthinned cooperative-grid run."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    rng = np.random.default_rng(4)
    for k, nchains in ((12, 3), (14, 2), (70, 5), (514, 1)):     # emcee rule: at least 2 ndim walkers
        p0 = models.draw_in_ranges(pset, k * nchains, rng, seeds=True).reshape(nchains, k, 6)
        p0[:, :, 4], p0[:, :, 5] = rng.uniform(.9, 1, (nchains, k)), rng.uniform(.8, 1, (nchains, k))
        up = (lambda x: x) if nchains > 1 else (lambda x: x[None])      # one chain: the sampler drops the chain axis
        full = mcmc.DeviceEnsembleSampler(k, 6, fn, nchains=nchains, seed=9, mode=1)
        full.run_mcmc(p0 if nchains > 1 else p0[0], 23)
        fc, fl = up(full.chain), up(full.lnprobability)
        for mode in (0, 2, 3):
            s = mcmc.DeviceEnsembleSampler(k, 6, fn, nchains=nchains, seed=9, mode=mode, store_lnprob=(mode != 2))
            s.run_mcmc(p0 if nchains > 1 else p0[0], 10, thin=3)   # stores steps 3, 6, 9
            s.run_mcmc(None, 13, thin=1)                             # continues at global step 10
            sc = up(s.chain)
            assert sc.shape == (nchains, k, 3 + 13, 6)
            assert np.array_equal(sc[:, :, :3], fc[:, :, 2:10:3]), (k, mode)
            assert np.array_equal(sc[:, :, 3:], fc[:, :, 10:]), (k, mode)
            assert np.array_equal(s.acceptance_fraction, full.acceptance_fraction)
            if mode != 2:
                assert np.array_equal(up(s.lnprobability)[:, :, 3:], fl[:, :, 10:])
    with pytest.raises(ValueError):
        mcmc.DeviceEnsembleSampler(7, 6, fn, seed=1).run_mcmc(models.draw_in_ranges(pset, 7, rng, seeds=True), 1)   # odd ensemble


def test_device_sampler_bsm_model_launch_shapes(torch, golden):
    """The BSM log-posterior (fixed-texture specialisation, two interleaved bin chains) inside the
    sampler: cluster, block and grid shapes give the same chain, and the stored log-posteriors are the
    ones gf_lnprob returns for the stored positions."""
    from golemflavor_b200.enums import Texture
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
    fn = llh.LnProb(args, asimov, pset)
    np.random.seed(3)
    k = 512
    p0 = mcmc.flat_seed(pset, k)
    ref = mcmc.DeviceEnsembleSampler(k, fn.ndim, fn, seed=11, mode=1)
    ref.run_mcmc(p0, 12)
    for mode, nc in ((0, 0), (2, 0), (3, 4), (3, 16)):
        s = mcmc.DeviceEnsembleSampler(k, fn.ndim, fn, seed=11, mode=mode, cluster_blocks=nc)
        s.run_mcmc(p0, 12)
        assert np.array_equal(s.chain, ref.chain), (mode, nc)
        assert np.array_equal(s.lnprobability, ref.lnprobability)
    assert 0.05 < ref.acceptance_fraction.mean() < 0.9
    # same per-point code, but a separate instantiation (four interleaved bins instead of two): FMA
    # contraction may differ in the last bits
    assert np.allclose(fn(ref.chain[:, -1]), ref.lnprobability[:, -1], rtol=1e-11, atol=0)


def test_mcmc_driver_uses_device_sampler_and_recovers_injection(torch, golden, capsys):
    """mcmc.mcmc with a partial of llh.ln_prob (the reference's calling pattern, scripts/fr.py:182-187)
    runs on the device-resident sampler; the BSM posterior sampled with logLam free stays inside the
    prior box and prefers compositions near the injected one."""
    from functools import partial
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    ln_prob = partial(llh.ln_prob, args=args, asimov_paramset=asimov, llh_paramset=pset)
    np.random.seed(25)
    k = 256
    p0 = mcmc.flat_seed(pset, k)
    p0[:, 4], p0[:, 5] = np.random.uniform(0.9, 1.0, k), np.random.uniform(0.8, 1.0, k)
    samples = mcmc.mcmc(p0, ln_prob, 6, k, burnin=400, nsteps=400, seed=4)
    assert isinstance(mcmc.mcmc.last_sampler, mcmc.DeviceEnsembleSampler)
    assert samples.shape == (k * 400, 6)
    lo, hi = np.array(pset.ranges).T
    assert np.all(samples >= lo) and np.all(samples <= hi)
    measured = fr.u_to_fr(fr.angles_to_fr(samples[:, 4:6]), fr.angles_to_u(samples[:, :4]))
    bf = np.array(go.angles_to_fr(g['asimov_angles']))
    assert np.abs(np.median(measured, axis=0) - bf).max() < 0.03
    assert 0.15 < mcmc.mcmc.last_sampler.acceptance_fraction.mean() < 0.7


def test_sens_sweep_small(torch):
    from golemflavor_b200 import sens
    out = sens.sweep(dimensions=(3, 6), segments=5, nwalkers=32, burnin=60, nsteps=60, injected_ratio=(1, 1, 1), distributed=False)
    assert len(out['scale']) == 10 and set(out['dimension']) == {3, 6}
    assert np.all(out['scale'][out['dimension'] == 3] == sens.scale_grid(3, 5))
    assert np.all(np.isfinite(out['mean_lnprob'])) and np.all((out['acceptance'] > 0.02) & (out['acceptance'] < 0.9))
    assert np.abs(out['mean_fr'].sum(axis=1) - 1).max() < 1e-12
    # the null point (logLam = -100: no new physics) and the smallest in-range scale agree; the largest scale differs
    d6 = out['dimension'] == 6
    assert np.abs(out['mean_fr'][d6][0] - out['mean_fr'][d6][1]).max() < 0.05


def test_coverage_mask_matches_reference_definition(torch):
    """plot.flavor_contour's coverage region (plot.py:372-384) restated with NumPy vs gf_coverage_mask."""
    fm = scan.scan_model('unitary', source_ratio=(1, 0, 0))
    for nb, n in ((25, 2_000_000), (100, 500_000)):
        hist, _ = scan.scan_histogram(fm, n, nb=nb, seed=3, distributed=False)
        for cov in (68.0, 90.0, 99.0, 99.9, 0.0):   # (at exactly 100 % the reference's answer is float-rounding noise)
            mask, (cstar, nmask, ntie) = scan.coverage_mask(hist, cov)
            H = hist / hist.sum()                         # plot.py:371; gaussian_filter(sigma=0.05) is a one-tap identity
            Hr = np.ravel(H)
            order = np.argsort(Hr)[::-1]
            thres = int(np.searchsorted(np.cumsum(Hr[order]), cov / 100.))
            ref = np.zeros(Hr.shape)
            ref[order[:thres]] = 1
            flat, m = hist.ravel(), mask.ravel()
            assert m.sum() == thres == nmask, (nb, cov, m.sum(), thres)
            if thres in (0, len(flat)):
                continue
            first_out = flat[order[thres]]
            assert cstar == first_out
            assert np.array_equal(m[flat > cstar], ref[flat > cstar]) and np.all(m[flat > cstar] == 1)
            assert np.all(m[flat < cstar] == 0) and m[flat == cstar].sum() == ntie == ref[flat == cstar].sum()
    full, (c100, n100, _) = scan.coverage_mask(hist, 100.0)
    assert n100 == np.count_nonzero(hist) - 1 and full.ravel()[hist.ravel() == 0].sum() == 0
    from scipy.ndimage import gaussian_filter
    assert np.array_equal(gaussian_filter(H, sigma=0.05), H)   # the reference's smoothing really is the identity


def test_smoothed_coverage_region_matches_scipy_and_the_reference_definition(torch):
    """hist_smooth beyond the one-tap identity (plot.py:372-384 with gaussian_filter(H, sigma=hist_smooth)): the device
    filter equals SciPy's bit for bit (separable, mode 'reflect', its accumulation order), and the region found on the
    smoothed field is the reference's `argsort / cumsum / searchsorted` set."""
    from scipy.ndimage import gaussian_filter
    fm = scan.scan_model('unitary', source_ratio=(1, 0, 0))
    for nb, n in ((25, 1_000_000), (60, 300_000)):
        hist, _ = scan.scan_histogram(fm, n, nb=nb, seed=5, distributed=False)
        H = hist / np.sum(hist)
        for sigma in (0.125, 0.4, 1.0, 3.0):
            Hs = gaussian_filter(H, sigma=sigma)
            got = scan.smooth_histogram(hist, sigma)
            assert got.shape == Hs.shape and np.array_equal(got, Hs), (nb, sigma, float(np.abs(got - Hs).max()))
            assert abs(got.sum() - 1.0) < 1e-12
            Hr = np.ravel(Hs)
            order = np.argsort(Hr)[::-1]
            crs = np.cumsum(Hr[order])
            for cov in (68.0, 90.0, 99.0, 0.0):
                thres = int(np.searchsorted(crs, cov / 100.))
                mask, (cstar, nmask, ntie) = scan.coverage_mask(hist, cov, hist_smooth=sigma)
                m = mask.ravel()
                # the cumulative sums of the two methods differ in their rounding: allow the boundary cell itself to move
                assert abs(int(m.sum()) - thres) <= 1 and nmask == int(m.sum()), (nb, sigma, cov, int(m.sum()), thres)
                if thres == 0:
                    continue
                assert np.all(m[Hr > cstar] == 1) and np.all(m[Hr < cstar] == 0)
                assert abs(cstar - Hr[order[min(thres, len(Hr) - 1)]]) <= 1e-12 * Hr.max()
                again, info = scan.coverage_mask(hist, cov, hist_smooth=sigma)
                assert np.array_equal(again, mask) and info == (cstar, nmask, ntie)      # deterministic
    # the default width stays on the integer path
    a, ia = scan.coverage_mask(hist, 90.0)
    b, ib = scan.coverage_mask(hist, 90.0, hist_smooth=0.05)
    assert np.array_equal(a, b) and ia == ib and isinstance(ia[0], int)
    with pytest.raises(ValueError):
        scan.smooth_histogram(np.zeros((3, 4, 3), dtype=np.int64), 0.4)


def test_scan_evidence_against_oracle(torch):
    """ln mean(L) over prior draws: device log-sum-exp vs the oracle's likelihood on the same draws."""
    from argparse import Namespace
    from golemflavor_b200.param import ParamSet
    args = Namespace(source_ratio=np.array([1, 2, 0.]) / 3, dimension=6, texture=Texture.OET, binning=models.BINNING, no_bsm=False,
                     injected_ratio=[1 / 3, 1 / 3, 1 / 3], smearing=0.02, fixed_scale=-42.0)
    fm = model.flatten(args, None, ParamSet(scan.sm_paramset(with_mass=True)))
    assert fm.struct.col_scale == -1 and fm.struct.fixed_loglam == -42.0 and fm.struct.no_bsm == 0
    n = 40000
    theta, frs, _ = scan.scan_samples(fm, n, seed=26)
    ref_fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], np.full(n, -42.0), 6,
                                         models.BINNING, args.source_ratio)
    assert np.abs(frs - ref_fr).max() < FR_TOL
    ll = go.batch_multi_gaussian(ref_fr, [1 / 3, 1 / 3, 1 / 3], 0.02)
    fin = np.isfinite(ll)
    mx = ll[fin].max()
    ref = mx + np.log(np.exp(ll[fin] - mx).sum()) - np.log(n)
    got = scan.scan_evidence(fm, n, seed=26, distributed=False)
    assert abs(got - ref) < 1e-9 * abs(ref), (got, ref)
    # shard invariance of the merge
    parts = [scan.scan_evidence(fm, c, seed=26, first_index=s, distributed=False) + np.log(c) for s, c in ((0, 15000), (15000, 25000))]
    both = np.logaddexp(parts[0], parts[1]) - np.log(n)
    assert abs(both - got) < 1e-12 * abs(got)
    # the null point (no new physics) has the same evidence for every dimension
    from golemflavor_b200 import sens
    ev = sens.evidence_grid(dimensions=(3, 6), segments=4, samples=20000)
    assert ev[3].shape == (4, 2) and ev[3][0, 0] == -100 and abs(ev[3][0, 1] - ev[6][0, 1]) < 1e-9


def test_evidence_grid_kernel_against_per_scale_launches_and_oracle(torch):
    """gf_scan_evidence_grid (one launch per dimension: every prior sample evaluated at all frozen scales) against
    (i) gf_scan_evidence launched once per scale on the same Philox draws and (ii) the oracle's likelihood on those
    draws; sample-shard invariance; the generic (sampled-source) specialisation; then the limit extraction on top."""
    from argparse import Namespace
    from golemflavor_b200 import sens
    from golemflavor_b200.param import ParamSet
    lib = _lib.load()
    n = 30000
    for dim, nsc in ((6, 23), (3, 7)):
        scales = sens.scale_grid(dim, nsc)
        args = Namespace(source_ratio=np.array([1, 2, 0.]) / 3, dimension=dim, texture=Texture.OET, binning=models.BINNING, no_bsm=False,
                         injected_ratio=[1 / 3, 1 / 3, 1 / 3], smearing=0.02, fixed_scale=-100.0)
        fm = model.flatten(args, None, ParamSet(scan.sm_paramset(with_mass=True)))
        before = lib.gf_launch_count()
        got = scan.scan_evidence_grid(fm, scales, n, seed=26, distributed=False)
        assert lib.gf_launch_count() - before == 1
        theta, _, _ = scan.scan_samples(fm, n, seed=26)
        for k, sc in enumerate(scales):
            fm.struct.fixed_loglam = float(sc)
            one = scan.scan_evidence(fm, n, seed=26, distributed=False)
            assert abs(got[k] - one) <= 1e-12 * abs(one), (dim, sc, got[k], one)
            if k in (0, 1, nsc // 2, nsc - 1):
                ref_fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], np.full(n, sc), dim,
                                                     models.BINNING, args.source_ratio)
                ll = go.batch_multi_gaussian(ref_fr, [1 / 3, 1 / 3, 1 / 3], 0.02)
                fin = np.isfinite(ll)
                mx = ll[fin].max()
                ref = mx + np.log(np.exp(ll[fin] - mx).sum()) - np.log(n)
                assert abs(got[k] - ref) < 1e-9 * abs(ref), (dim, sc, got[k], ref)
        parts = [scan.scan_evidence_grid(fm, scales, c, seed=26, first_index=s, distributed=False) + np.log(c) for s, c in ((0, 11000), (11000, 19000))]
        assert np.max(np.abs(np.logaddexp(parts[0], parts[1]) - np.log(n) - got) / np.abs(got)) < 1e-12
    # degenerate shapes: one scale is the single-scale entry point; no samples -> -inf; fewer samples than threads
    fm.struct.fixed_loglam = -40.0
    assert abs(scan.scan_evidence_grid(fm, [-40.0], 5000, seed=4, distributed=False)[0] - scan.scan_evidence(fm, 5000, seed=4, distributed=False)) < 1e-12 * 400
    assert np.all(np.isneginf(scan.scan_evidence_grid(fm, [-40.0, -35.0], 0, distributed=False)))
    few = scan.scan_evidence_grid(fm, scales, 37, seed=4, distributed=False)
    assert few.shape == (len(scales),) and np.all(np.isfinite(few))
    # sampled source (GENERIC specialisation, column-map path) + a model with a sampled scale is refused
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'ref_llh.npz'))
    a9, as9, ps9 = models.bsm_sampled_source(g['asimov_angles'], 'angles', 6, Texture.OUT)
    with pytest.raises(ValueError):
        scan.scan_evidence_grid(model.flatten(a9, as9, ps9), [-40.0], 100, distributed=False)
    a9.fixed_scale = -100.0
    fm8 = model.flatten(a9, as9, ParamSet([p for p in ps9 if p.name != 'logLam']))
    sc8 = np.array([-100.0, -44.0, -38.5, -33.0])
    got8 = scan.scan_evidence_grid(fm8, sc8, 8000, seed=3, distributed=False)
    for k, sc in enumerate(sc8):
        fm8.struct.fixed_loglam = float(sc)
        one = scan.scan_evidence(fm8, 8000, seed=3, distributed=False)
        assert abs(got8[k] - one) <= 1e-12 * abs(one)
    # the full grid through sens.evidence_grid and the limit extraction of plot.py:149-213 on top
    ev, mx = sens.evidence_grid(dimensions=(3, 6), segments=20, samples=50000, injected_ratio=(1, 1, 1), return_maxllh=True)
    assert ev[3].shape == (20, 2) and ev[3][0, 0] == -100 and abs(ev[3][0, 1] - ev[6][0, 1]) < 1e-9
    assert np.all(mx[6][:, 1] >= ev[6][:, 1]) and np.array_equal(mx[6][:, 0], ev[6][:, 0])
    lim = sens.limits(ev)
    for d in (3, 6):   # an injected (1:1:1) composition is compatible with the null: large scales are excluded
        lo, hi = model.SCALE_BOUNDARIES[d]
        assert lim[d] is not None and lo - 1 < lim[d] < hi, (d, lim[d])


def test_cli_scan_outputs(torch, tmp_path):
    from golemflavor_b200 import cli
    out = cli.main(['mc_unitary', '--nwalkers', '20', '--nsteps', '50', '--datadir', str(tmp_path)])
    assert out.endswith('mc_unitary_SRC_1_2_0.npy')
    frs = np.load(out)
    assert frs.shape == (1000, 3) and np.abs(frs.sum(axis=1) - 1).max() < 1e-14          # mc_unitary.py:189-193
    out = cli.main(['mc_texture', '--dimension', '6', '--texture', 'OET', '--nwalkers', '10', '--nsteps', '20', '--datadir', str(tmp_path)])
    arr = np.load(out)
    assert out.endswith('mc_texture_DIM6_SRC_1_2_0_OET.npy') and arr.shape == (200, 3 + 7)   # (frs, samples), mc_texture.py:222
    ref = truth.eigh_flux_averaged_fr(arr[:, 3:7], arr[:, 7:9], model.TEXTURE_ANGLES['OET'], arr[:, 9], 6, models.BINNING, np.array([1, 2, 0.]) / 3)
    assert np.abs(arr[:, :3] - ref).max() < FR_TOL
    out = cli.main(['fr', '--dimension', '6', '--texture', 'OET', '--nwalkers', '32', '--burnin', '20', '--nsteps', '30', '--datadir', str(tmp_path)])
    assert out.endswith('chain_DIM6_sfr_1_2_0_mfr_1_1_1_OET.npy') and np.load(out).shape == (32 * 30, 7)


def test_reference_call_variants(torch, golden):
    """Argument forms of the reference API: texture enums, no_bsm, tensors in / tensors out, host outputs."""
    g = golden('ref_bsm_u.npz')
    k = int(np.where(g['tex'] == 'OET')[0][0])
    smu = fr.angles_to_u(g['sm'][k])
    # texture given as enum + scalar scale == Texture.NONE with the explicit angle tuple (fr.py:367-378)
    v1 = fr.params_to_BSMu(g['loglam'][k], int(g['dim'][k]), g['energy'][k], mass_eigenvalues=g['mass'][k], sm_u=smu, texture=Texture.OET)
    v2 = fr.params_to_BSMu(tuple(model.TEXTURE_ANGLES['OET']) + (g['loglam'][k],), int(g['dim'][k]), g['energy'][k],
                           mass_eigenvalues=g['mass'][k], sm_u=smu)
    assert np.array_equal(v1, v2) and v1.shape == (3, 3)
    # no_bsm: eigenvectors of U diag(0, m21, m3x) U^+ are U's columns (ascending eigenvalue) up to phases
    v0 = fr.params_to_BSMu((0, 0, 0, 0, -30), 6, 1e5, sm_u=smu, no_bsm=True)
    assert np.abs(np.abs(v0) ** 2 - np.abs(smu) ** 2).max() < 1e-12
    assert np.abs(fr.u_to_fr((1, 2, 0), v0) - fr.u_to_fr((1, 2, 0), smu)).max() < 1e-13
    with pytest.raises(ValueError):
        fr.params_to_BSMu((0.1, 0.2, 0.3), 6, 1e5)          # Texture.NONE needs 5 entries
    with pytest.raises(ValueError):
        fr.params_to_BSMu((0, 0, 0, 0, -30), 6, 1e5, sm_u=np.eye(2))
    # tensors in -> tensors out, nothing leaves the device
    ang = torch.as_tensor(g['sm']).cuda()
    u = fr.angles_to_u(ang)
    assert u.is_cuda and u.dtype == torch.complex128 and u.shape == (len(g['sm']), 3, 3)
    f = fr.u_to_fr(torch.tensor([1., 2., 0.], device='cuda'), u)
    assert f.is_cuda and np.abs(f.cpu().numpy() - fr.u_to_fr((1, 2, 0), u.cpu().numpy())).max() == 0
    # host pipeline with the optional outputs
    gl = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(gl['asimov_angles'])
    fn = llh.LnProb(args, asimov, pset)
    th = models.draw_in_ranges(pset, 70000, np.random.default_rng(5))
    th[::13, 1] = 1.5
    lnp, frs, st = (x.cpu().numpy() for x in fn.evaluate(th, want_fr=True, want_status=True))
    h_fr, h_st = np.empty((70000, 3)), np.empty(70000, dtype=np.uint8)
    h_lnp = fn.evaluate_host(th, fr=h_fr, status=h_st)
    assert np.array_equal(h_lnp, lnp) and np.array_equal(h_st, st) and np.array_equal(np.isnan(h_fr), np.isnan(frs))
    assert np.array_equal(h_fr[~np.isnan(h_fr)], frs[~np.isnan(frs)])
    with pytest.raises(ValueError):
        fn.evaluate_host(th, fr=np.empty((5, 3)))


def test_host_pipeline_buffers_and_ring_geometry(torch, golden):
    """gf_lnprob_host on library-allocated page-locked buffers (plain and write-combined input), on pageable memory
    (internal staging ring) and across chunk boundaries: identical to the device path."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
    fn = llh.LnProb(args, asimov, pset)
    n = (1 << 18) * 2 + 12345                      # two full chunks of the default ring + a ragged third
    theta = models.draw_in_ranges(pset, n, np.random.default_rng(8))
    ref = fn.evaluate(theta).cpu().numpy()
    for wc in (False, True):
        hb_in, hb_out = _lib.HostBuffer((n, fn.ndim), write_combined=wc), _lib.HostBuffer((n,))
        hb_in.array[...] = theta
        out = fn.evaluate_host(hb_in.array, out=hb_out.array)
        assert out is hb_out.array and np.array_equal(out, ref, equal_nan=True)
    frs, st = np.empty((n, 3)), np.empty(n, dtype=np.uint8)
    out = fn.evaluate_host(theta, fr=frs, status=st)             # pageable in and out
    assert np.array_equal(out, ref, equal_nan=True)
    l2, f2, s2 = (x.cpu().numpy() for x in fn.evaluate(theta, want_fr=True, want_status=True))
    assert np.array_equal(frs, f2, equal_nan=True) and np.array_equal(st, s2)
    assert fn.evaluate_host(theta[:0]).shape == (0,)


def test_torch_ops_equal_the_c_abi(torch, golden):
    """`torch.ops.golemflavor.*` (csrc/gf_torch_ops.cpp) against the ctypes binding of the same entry points: identical
    bits, current-stream semantics, reference-style exceptions."""
    g = golden('ref_llh.npz')
    ops, lib = _lib.torch_ops(), _lib.load()
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OET)
    fn = llh.LnProb(args, asimov, pset)
    th = torch.as_tensor(models.draw_in_ranges(pset, 5000, np.random.default_rng(2))).cuda()
    lnp, frs, st = ops.lnprob(th, fn.model.blob, True, True)
    ref_l, ref_f = torch.empty(5000, dtype=torch.float64, device='cuda'), torch.empty((5000, 3), dtype=torch.float64, device='cuda')
    ref_s = torch.empty(5000, dtype=torch.uint8, device='cuda')
    _lib.check(lib.gf_lnprob(fn.model.ref, _lib.ptr(th), 5000, fn.ndim, 1, _lib.ptr(ref_l), _lib.ptr(ref_f), _lib.ptr(ref_s), _lib.stream_ptr(torch)))
    assert torch.equal(lnp, ref_l) and torch.equal(frs.nan_to_num(), ref_f.nan_to_num()) and torch.equal(st, ref_s)
    only, e1, e2 = ops.lnprob(th, fn.model.blob, False, False)
    assert torch.equal(only, ref_l) and e1.numel() == 0 and e2.numel() == 0
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                     # the operator runs on torch's CURRENT stream
        again = ops.lnprob(th, fn.model.blob, False, False)[0]
    side.synchronize()
    assert torch.equal(again, ref_l)
    f2, s2 = ops.flux_averaged_fr(th, fn.model.blob)
    inside = ~(st & _lib.ST_OUT_OF_PRIOR).bool()        # gf_lnprob leaves NaN compositions for out-of-prior points
    assert torch.equal(f2[inside], frs[inside]) and torch.equal(s2[inside], st[inside])
    assert np.allclose(ops.lnprior(th, fn.model.blob).cpu().numpy(), llh.lnprior(th, pset).cpu().numpy(), rtol=0, atol=0, equal_nan=True)
    ang = th[:, :4].contiguous()
    u = ops.angles_to_u(ang)
    assert u.dtype == torch.complex128 and np.array_equal(u.cpu().numpy(), fr.angles_to_u(ang).cpu().numpy())
    src = torch.tensor([1.0, 2.0, 0.0], dtype=torch.float64, device='cuda')
    assert np.array_equal(ops.u_to_fr(src, u).cpu().numpy(), fr.u_to_fr(src, u).cpu().numpy())
    hist, kept = torch.zeros(26 ** 3, dtype=torch.int64, device='cuda'), torch.zeros(1, dtype=torch.int64, device='cuda')
    fm = scan.scan_model('unitary')
    ops.scan_hist(fm.blob, 26, 0, 100000, 25, hist, kept)
    h2, k2 = scan.scan_histogram(fm, 100000, nb=25, seed=26, distributed=False)
    assert int(kept) == k2 == 100000 and np.array_equal(hist.cpu().numpy().reshape(26, 26, 26), h2)
    bad = model.FlatModel(model.physics_model(no_bsm=False, dimension=6, binning=models.BINNING, loglam=-40.0))
    bad.struct.dimension = 99                         # the blob shares memory with the struct
    with pytest.raises(ValueError):                   # GF_ERR_ARG -> ValueError, like the ctypes path and fr.py:198-202
        ops.lnprob(torch.zeros((4, 1), dtype=torch.float64, device='cuda'), bad.blob, False, False)
    with pytest.raises(RuntimeError):                 # wrong column count
        ops.lnprob(th[:, :5].contiguous(), fn.model.blob, False, False)


def test_multi_gpu_nccl_scan_evidence_and_sweep_are_rank_count_invariant(torch):
    """tests/dist_scan_check.py under torchrun on every GPU of the box (NCCL): sharded scan histograms bit-identical to
    the single-rank ones, evidence-grid merge and the sweep invariant.  Needs >= 2 GPUs (skipped on the 1-GPU test box;
    the 2- and 8-rank outputs of this round are committed under profiles/)."""
    import subprocess
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs at least two GPUs')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr', '127.0.0.1',
                          '--master-port', '29731', os.path.join(root, 'tests', 'dist_scan_check.py')], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    assert res.stdout.count('bit-identical=True') == 3 and 'ok=True' in res.stdout and 'sweep=True' in res.stdout


def test_bench_dumps_the_last_timed_step(torch, tmp_path):
    """`bench.py --dump-outputs DIR`: after exactly K timed launches, DIR/lnprob.npy holds the float64 log-posterior of every
    point of the seeded benchmark batch, in batch order -- the same values the public API computes for those rows -- and the
    dump stays within its 64 MB budget."""
    import json
    import subprocess

    import bench   # the repository root is on sys.path (conftest.py)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--steps', '2', '--warmup', '3', '--cpu-evals', '0',
                          '--scan-samples', '0', '--configs', '0', '--sustain-s', '0', '--dump-outputs', str(tmp_path / 'out')],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout)
    assert line['steps'] == 2 and line['gpu_launches'] == 2
    assert sorted(os.listdir(tmp_path / 'out')) == ['lnprob.npy']
    assert os.path.getsize(tmp_path / 'out' / 'lnprob.npy') <= 64 * 10 ** 6
    got = np.load(tmp_path / 'out' / 'lnprob.npy')
    n = bench.WALKERS * bench.CHAINS
    assert got.dtype == np.float64 and got.shape == (n,)
    (args, asimov, pset), models_ = bench.build_problem()
    sel = np.sort(np.random.default_rng(0).choice(n, 4096, replace=False))
    theta = bench.synth_theta(pset, n, 25, models_)[sel]
    want = llh.LnProb(args, asimov, pset).evaluate(theta).cpu().numpy()
    assert np.isfinite(want).mean() > 0.5
    np.testing.assert_allclose(got[sel], want, rtol=1e-12, atol=0)
