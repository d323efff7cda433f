"""Profile likelihood over the nuisance parameters on the (dimension, scale) grid (gf_profile_grid, scan.scan_profile_grid,
sens.profile_grid) and the frequentist limit (sens.get_limit with StatCateg.FREQUENTIST).

CPU tests run the optimiser through the host harness (the same per-task function, sequentially) against analytic minima,
SciPy's optimisers and the oracle; GPU tests hold the device to the harness, to LnProb, to the oracle and to the two
sampling stand-ins (evidence-grid prior samples, sweep chains)."""

import ctypes as C
import os
import sys
from argparse import Namespace

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import host_harness as hh  # noqa: E402
from host_harness import profile_harness as ph  # noqa: E402
import models  # noqa: E402
from golemflavor_b200 import _lib, build, llh, model, scan, sens  # noqa: E402
from golemflavor_b200.enums import StatCateg, Texture  # noqa: E402
from golemflavor_b200.param import ParamSet  # noqa: E402
from oracle import golem_oracle as go  # noqa: E402
from oracle import truth  # noqa: E402

INJ = np.array([1., 1., 1.]) / 3
SRC = np.array([1., 2., 0.]) / 3


def grid_model(dim, texture=Texture.OET):
    args = Namespace(source_ratio=SRC, dimension=dim, texture=texture, binning=models.BINNING, no_bsm=False, injected_ratio=INJ,
                     smearing=0.02, fixed_scale=-100.0)
    return args, model.flatten(args, None, ParamSet(scan.sm_paramset(with_mass=True)))


def study_scales(dim):
    return sens.scale_grid(dim, 100)[[0, 20, 40, 60, 80, 99]]


def units(fm):
    s = fm.struct
    return np.array([(s.prior[k].hi - s.prior[k].lo) / 10 if s.prior[k].kind == _lib.PRIOR_UNIFORM else s.prior[k].sigma for k in range(fm.ndim)])


def box(fm):
    s = fm.struct
    return np.array([[s.prior[k].lo, s.prior[k].hi] for k in range(fm.ndim)])


def oracle_lnprob(dim, theta, scale):
    """truth.eigh_flux_averaged_fr + batch_multi_gaussian + batch_lnprior at a frozen scale."""
    pset = ParamSet(scan.sm_paramset(with_mass=True))
    theta = np.atleast_2d(theta)
    fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], np.full(len(theta), scale), dim, models.BINNING, SRC)
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    return go.batch_lnprior(theta, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]) + go.batch_multi_gaussian(fr, INJ, 0.02)


# ------------------------------------------------------------------ CPU


def test_profile_config_abi():
    build.build_library()
    lib = _lib.load()
    assert lib.gf_sizeof(4) == C.sizeof(_lib.ProfileConfig) == 40
    assert 'gf_profile_grid' in _lib.EXPORTS
    assert 'gf_profile_dev.cuh' in build.HEADERS and 'gf_profile.cu' in build.SOURCES


@pytest.mark.parametrize('case', ['inside', 'face', 'edge'])
def test_nelder_mead_core_on_box_quadratic(case):
    """The optimiser core on sum a_k (x_k - c_k)^2 over [-1, 1]^6: the known minimum to 1e-10 in g."""
    a = np.array([1.0, 2.0, 3.0, 0.5, 5.0, 1.0])
    c = np.array([0.3, -0.2, 0.1, 0.7, 0.0, 0.5])
    if case in ('face', 'edge'):
        c[0] = 1.5
    if case == 'edge':
        c[4] = -2.0
    lo, hi = -np.ones(6), np.ones(6)
    xmin = np.clip(c, lo, hi)
    gmin = float(np.sum(a * (xmin - c) ** 2))
    xb, gb, nev, calls, conv = ph.nm_box_quadratic(a, c, lo, hi, np.full(6, -0.9), ftol=1e-12, xtol=1e-8, max_evals=20000)
    assert conv and nev < 20000 and calls == nev + 1            # + the final evaluation of the best vertex
    assert abs(gb - gmin) < 1e-10, (gb, gmin)
    assert np.all(xb >= lo) and np.all(xb <= hi)
    assert np.abs(xb - xmin).max() < 1e-4
    # a budget stops it: exactly max_evals optimiser evaluations, not converged
    _, _, nev, _, conv = ph.nm_box_quadratic(a, c, lo, hi, np.full(6, -0.9), max_evals=50)
    assert nev == 50 and not conv


@pytest.mark.parametrize('dim', [3, 6])
def test_harness_profile_against_scipy_and_oracle(dim):
    """The host-harness profile (default nstarts, max_evals, ftol) at six scales including the null point: at least the best
    of SciPy's Nelder-Mead and L-BFGS-B (same scaled coordinates, 20 starts) minus 1e-6; the value is hh_lnprob at the argmax
    (1e-12) and the oracle there (1e-10); every start converged before max_evals."""
    from scipy.optimize import minimize
    _, fm = grid_model(dim)
    scales = study_scales(dim)
    r = ph.profile(fm, scales, nstarts=scan.PROFILE_NSTARTS, seed=27, max_evals=scan.PROFILE_MAX_EVALS, ftol=scan.PROFILE_FTOL,
                   xtol=scan.PROFILE_XTOL)
    assert np.all(r['nconverged'] == scan.PROFILE_NSTARTS), r['nconverged']
    assert np.all(r['nevals'] < scan.PROFILE_NSTARTS * scan.PROFILE_MAX_EVALS)
    u, b = units(fm), box(fm)
    starts = hh.draw(fm, 99, 0, 20)
    for s, sc in enumerate(scales):
        fm.struct.fixed_loglam = float(sc)
        am = r['argmax'][s]
        assert np.all(am >= b[:, 0]) and np.all(am <= b[:, 1])
        at, fr_at, _ = hh.lnprob(fm, am)
        assert abs(at[0] - r['best'][s]) <= 1e-12 * abs(at[0]), (sc, at[0], r['best'][s])
        assert np.abs(fr_at[0] - r['fr'][s]).max() == 0.0
        ref = oracle_lnprob(dim, am, sc)[0]
        assert abs(ref - r['best'][s]) <= 1e-10 * abs(ref), (sc, ref, r['best'][s])

        def neg(x):
            v = hh.lnprob(fm, np.clip(x * u, b[:, 0], b[:, 1]))[0][0]
            return -v if np.isfinite(v) else 1e300
        sp = -np.inf
        bounds = list(zip(b[:, 0] / u, b[:, 1] / u))
        for x0 in starts / u:
            for method, opts in (('Nelder-Mead', dict(adaptive=True, maxfev=3000, xatol=1e-8, fatol=1e-11)), ('L-BFGS-B', {})):
                res = minimize(neg, x0, method=method, bounds=bounds, options=opts)
                sp = max(sp, -res.fun)
        assert r['best'][s] >= sp - 1e-6, (dim, sc, r['best'][s], sp)
    fm.struct.fixed_loglam = -100.0


def test_harness_profile_is_split_and_specialisation_invariant():
    """A scale's result depends on (seed, global scale index, nstarts) only: the run over all scales equals two runs split with
    task0 offsets bit for bit; the static 6-column and the runtime-layout FIXED paths agree bit for bit."""
    _, fm = grid_model(6)
    scales = sens.scale_grid(6, 9)
    kw = dict(nstarts=32, seed=5, max_evals=1500)
    full = ph.profile(fm, scales, **kw)
    parts = [ph.profile(fm, scales[:4], task0=0, **kw), ph.profile(fm, scales[4:], task0=4, **kw)]
    fixed = ph.profile(fm, scales, spec=1, **kw)
    for key in full:
        assert np.array_equal(full[key], np.concatenate([p[key] for p in parts])), key
        assert np.array_equal(full[key], fixed[key]), key
    generic = ph.profile(fm, scales, spec=0, **kw)
    assert np.all(np.abs(generic['best'] - full['best']) <= 1e-9 * np.abs(full['best']))


def test_frequentist_limit_is_the_bayesian_rule_with_the_wilks_threshold(golden):
    """get_limit(FREQUENTIST) on every ref_limit.npz curve equals get_limit(BAYESIAN) with ln 10^bayes_k = chi2.ppf(cl, 1) / 2,
    None and 'Discovered LV!' included; a hand-made curve crosses where it should."""
    from scipy.stats import chi2
    g = golden('ref_limit.npz')
    freq, bayes = Namespace(stat_method=StatCateg.FREQUENTIST), Namespace(stat_method=StatCateg.BAYESIAN)
    for cl in (sens.FREQ_CL, 0.68, 0.95):
        k_eq = np.log10(np.exp(chi2.ppf(cl, 1) / 2))
        for k in range(int(g['n'])):
            sc, st, mi = g['scales_%d' % k], g['stat_%d' % k], bool(g['mask_%d' % k])
            for stat in (st, st * 3.0):                                  # steeper curves move the crossings
                outs = []
                for a, kw in ((freq, dict(cl=cl)), (bayes, dict(bayes_k=k_eq))):
                    try:
                        outs.append(sens.get_limit(sc, stat, args=a, mask_initial=mi, **kw))
                    except AssertionError as e:
                        outs.append(str(e))
                assert outs[0] == outs[1], (cl, k, outs)
    with pytest.raises(NotImplementedError):
        sens.get_limit(np.array([-100., -40., -30.]), np.array([0., 0., 0.]), args=Namespace(stat_method='OTHER'))
    # profile flat up to -40, then falling by 1 per unit of log10 Lambda: the crossing of chi2.ppf(0.9, 1) / 2 = 1.353
    sc = np.concatenate([[-100.], np.linspace(-60, -20, 41)])
    st = -np.maximum(sc + 40.0, 0.0)
    lim = sens.get_limit(sc, st, args=freq)
    assert abs(lim + np.log10(2.) - (-40.0 + chi2.ppf(0.9, 1) / 2)) < 0.05, lim
    assert sens.FREQ_CL == 0.90


# ------------------------------------------------------------------ GPU


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


@pytest.mark.gpu
@pytest.mark.parametrize('dim', [3, 6])
def test_device_profile_against_harness_lnprob_and_oracle(torch, dim):
    """Device best >= harness best - 1e-6; best is LnProb(fixed_scale) at argmax (1e-12) and the oracle (1e-10); argmax inside
    the box; one launch."""
    args, fm = grid_model(dim)
    scales = study_scales(dim)
    lib = _lib.load()
    before = lib.gf_launch_count()
    d = scan.scan_profile_grid(fm, scales, seed=27)
    assert lib.gf_launch_count() - before == 1
    h = ph.profile(fm, scales, nstarts=scan.PROFILE_NSTARTS, seed=27, max_evals=scan.PROFILE_MAX_EVALS, ftol=scan.PROFILE_FTOL,
                   xtol=scan.PROFILE_XTOL)
    assert np.all(d['best'] >= h['best'] - 1e-6), (d['best'], h['best'])
    assert np.all(d['nconverged'] >= 1) and np.all(d['nevals'] > 0)
    b = box(fm)
    assert np.all(d['argmax'] >= b[:, 0]) and np.all(d['argmax'] <= b[:, 1])
    assert not np.any(d['status'] & (_lib.ST_NON_FINITE | _lib.ST_OUT_OF_PRIOR))
    for s, sc in enumerate(scales):
        a = Namespace(**vars(args))
        a.fixed_scale = float(sc)
        fn = llh.LnProb(a, None, ParamSet(scan.sm_paramset(with_mass=True)))
        lnp, fr = (x.cpu().numpy() for x in fn.evaluate(d['argmax'][s:s + 1], want_fr=True))
        assert abs(lnp[0] - d['best'][s]) <= 1e-12 * abs(lnp[0]), (sc, lnp[0], d['best'][s])
        assert np.abs(fr[0] - d['fr'][s]).max() < 1e-14
        ref = oracle_lnprob(dim, d['argmax'][s], sc)[0]
        assert abs(ref - d['best'][s]) <= 1e-10 * abs(ref), (sc, ref, d['best'][s])


@pytest.mark.gpu
def test_device_profile_split_and_specialisation_invariance(torch, monkeypatch):
    """Bit-identical outputs for one call over all scales and two calls split with task0, and for the static 6-column and the
    runtime-layout FIXED kernels; the GENERIC kernel agrees to 1e-9."""
    _, fm = grid_model(6)
    scales = sens.scale_grid(6, 12)
    kw = dict(nstarts=32, seed=8, max_evals=2000)
    full = scan.scan_profile_grid(fm, scales, **kw)
    parts = [scan.scan_profile_grid(fm, scales[:5], task0=0, **kw), scan.scan_profile_grid(fm, scales[5:], task0=5, **kw)]
    monkeypatch.setenv('GF_PROFILE_SPEC', 'fixed')
    fixed = scan.scan_profile_grid(fm, scales, **kw)
    monkeypatch.setenv('GF_PROFILE_SPEC', 'generic')
    generic = scan.scan_profile_grid(fm, scales, **kw)
    monkeypatch.setenv('GF_PROFILE_SPEC', 'nonsense')
    with pytest.raises(ValueError):
        scan.scan_profile_grid(fm, scales, **kw)
    monkeypatch.delenv('GF_PROFILE_SPEC')
    for key in full:
        assert np.array_equal(full[key], np.concatenate([p[key] for p in parts])), key
        assert np.array_equal(full[key], fixed[key]), key
    assert np.all(np.abs(generic['best'] - full['best']) <= 1e-9 * np.abs(full['best']))
    # a model in another column order runs the runtime-layout kernel and is refused the static one
    perm = [4, 5, 0, 1, 2, 3]
    args = Namespace(source_ratio=SRC, dimension=6, texture=Texture.OET, binning=models.BINNING, no_bsm=False, injected_ratio=INJ,
                     smearing=0.02, fixed_scale=-100.0)
    fmp = model.flatten(args, None, ParamSet([scan.sm_paramset(with_mass=True)[k] for k in perm]))
    monkeypatch.setenv('GF_PROFILE_SPEC', 'static6')
    with pytest.raises(ValueError):
        scan.scan_profile_grid(fmp, scales[:2], **kw)
    monkeypatch.delenv('GF_PROFILE_SPEC')
    rp = scan.scan_profile_grid(fmp, scales, **kw)
    assert np.all(rp['best'] >= full['best'] - 1e-6 * np.abs(full['best']))


@pytest.mark.gpu
def test_device_profile_beats_the_sampling_stand_ins(torch):
    """The profile is >= sweep()['max_lnprob'] - 1e-9 and >= the largest LnProb among 1e5 prior samples at each scale; at the
    null point it agrees across dimensions to 1e-9."""
    dims, seg = (3, 6), 6
    prof = sens.profile_grid(dimensions=dims, segments=seg, distributed=False)
    sw = sens.sweep(dimensions=dims, segments=seg, nwalkers=32, burnin=50, nsteps=100, distributed=False)
    null = [prof[d][0, 1] for d in dims]
    assert abs(null[0] - null[1]) <= 1e-9 * abs(null[0]), null
    for d in dims:
        args, fm = grid_model(d)
        theta, _, _ = scan.scan_samples(fm, 100000, seed=26)
        for s, sc in enumerate(prof[d][:, 0]):
            a = Namespace(**vars(args))
            a.fixed_scale = float(sc)
            fn = llh.LnProb(a, None, ParamSet(scan.sm_paramset(with_mass=True)))
            mx = float(fn.evaluate(theta).max().item())
            assert prof[d][s, 1] >= mx, (d, sc, prof[d][s, 1], mx)
            i = np.where((sw['dimension'] == d) & (sw['scale'] == sc))[0]
            assert len(i) == 1
            # the sweep's frozen logLam column has a flat prior: its ln_prob is the six-column one
            assert prof[d][s, 1] >= sw['max_lnprob'][i[0]] - 1e-9, (d, sc, prof[d][s, 1], sw['max_lnprob'][i[0]])


@pytest.mark.gpu
def test_profile_grid_frequentist_limit(torch):
    """sens.profile_grid + limits(FREQUENTIST) for injected (1:1:1): a limit inside SCALE_BOUNDARIES; one launch per dimension;
    return_argmax gives the maximising parameters."""
    lib = _lib.load()
    before = lib.gf_launch_count()
    prof, am = sens.profile_grid(dimensions=(3, 6), segments=20, distributed=False, return_argmax=True)
    assert lib.gf_launch_count() - before == 2
    lim = sens.limits(prof, args=Namespace(stat_method=StatCateg.FREQUENTIST))
    for d in (3, 6):
        assert prof[d].shape == (20, 2) and am[d].shape == (20, 6)
        assert np.array_equal(prof[d][:, 0], sens.scale_grid(d, 20))
        lo, hi = model.SCALE_BOUNDARIES[d]
        assert lim[d] is not None and lo <= lim[d] <= hi, (d, lim[d])


@pytest.mark.gpu
def test_profile_refusals(torch):
    _, fm = grid_model(6)
    with pytest.raises(ValueError, match='no BSM path'):
        scan.scan_profile_grid(scan.scan_model('unitary'), [-40.0])
    args, asimov, pset = models.bsm_model_c3([0.5, 0.5], dim=6)
    with pytest.raises(ValueError, match='sampled column'):
        scan.scan_profile_grid(model.flatten(args, asimov, pset), [-40.0])
    for bad in (48, 16, 512):
        with pytest.raises(ValueError, match='multiple of 32'):
            scan.scan_profile_grid(fm, [-40.0], nstarts=bad)
    # twelve columns (six with priors only) x 256 starts: 169 x 256 x 8 B of simplices do not fit in shared memory
    from golemflavor_b200.param import Param
    extra = [Param(name='nuis%d' % k, value=0.0, ranges=[-1., 1.], std=0.1) for k in range(6)]
    args = Namespace(source_ratio=SRC, dimension=6, texture=Texture.OET, binning=models.BINNING, no_bsm=False, injected_ratio=INJ,
                     smearing=0.02, fixed_scale=-100.0)
    fm12 = model.flatten(args, None, ParamSet(scan.sm_paramset(with_mass=True) + extra))
    with pytest.raises(ValueError, match='shared memory'):
        scan.scan_profile_grid(fm12, [-40.0], nstarts=256)
    r = scan.scan_profile_grid(fm12, [-40.0, -35.0], nstarts=32, max_evals=500)
    assert np.all(np.isfinite(r['best']))
