"""The profile likelihood over many source compositions (gf_profile_sources, scan.scan_profile_sources,
sens.profile_source_grid) and the frequentist limit table built from it.

CPU tests hold the source objective to gf_profile_grid's single-source objective on prior draws and on the fixture points,
the sequential profile of every (source, scale) to the existing profile harness of the single-source model, and the rows to
their own structure (permuted and repeated sources, task0 splits); they also check the export and the refusals that need no
device.  GPU tests hold the device to scan_profile_grid run once per source, to LnProb, to the oracle and to the harness,
check bit-identical rows across repeats, repeated and permuted sources, splits and specialisations, the launch count, every
refusal of the C entry point, and the frequentist limit table end to end."""

import ctypes as C
import os
import re
import sys
from argparse import Namespace

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import host_harness as hh  # noqa: E402
from host_harness import profile_harness as ph  # noqa: E402
from host_harness import profile_source_harness as psh  # noqa: E402
import models  # noqa: E402
from golemflavor_b200 import _lib, build, llh, model, scan, sens  # noqa: E402
from golemflavor_b200.enums import StatCateg, Texture  # noqa: E402
from golemflavor_b200.param import ParamSet  # noqa: E402
from oracle import golem_oracle as go  # noqa: E402
from oracle import truth  # noqa: E402

ROOT = os.path.dirname(HERE)
SMEARING = 0.02
SOURCES = np.array([(1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (1., 2., 0.), (0.31, 0.52, 0.17)])
INJECTED = np.array([(1., 1., 1.), (1., 0., 0.), (1., 2., 0.), (0., 1., 0.), (2., 1., 1.)])
FREQ = Namespace(stat_method=StatCateg.FREQUENTIST)


def grid_model(dim, src=(1., 2., 0.), inj=(1., 1., 1.), texture=Texture.OET, binning=scan.DEFAULT_BINNING):
    """sens._grid_model: the frozen-scale model of the sensitivity grid with source `src` and injected composition `inj`."""
    return sens._grid_model(dim, texture, np.asarray(src, dtype=np.float64), np.asarray(inj, dtype=np.float64), SMEARING, binning)


def box(fm):
    s = fm.struct
    return np.array([[s.prior[k].lo, s.prior[k].hi] for k in range(fm.ndim)])


def oracle_lnprob(dim, theta, scale, src, inj):
    """truth.eigh_flux_averaged_fr + batch_multi_gaussian + batch_lnprior at a frozen scale for source `src`."""
    pset = ParamSet(scan.sm_paramset(with_mass=True))
    theta = np.atleast_2d(theta)
    src, inj = np.asarray(src, dtype=np.float64), np.asarray(inj, dtype=np.float64)
    fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES['OET'], np.full(len(theta), scale), dim, scan.DEFAULT_BINNING,
                                     src / src.sum())
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    return go.batch_lnprior(theta, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]) + \
        go.batch_multi_gaussian(fr, inj / inj.sum(), SMEARING)


def assert_rel(got, ref, rtol, what=''):
    got, ref = np.asarray(got), np.asarray(ref)
    f = np.isfinite(ref)
    assert np.array_equal(f, np.isfinite(got)) and np.array_equal(got[~f], ref[~f], equal_nan=True), what
    err = np.abs(got[f] - ref[f]) / np.abs(ref[f])
    assert err.size == 0 or err.max() <= rtol, (what, err.max())


# ------------------------------------------------------------------ CPU


def test_abi_and_build():
    build.build_library()
    lib = _lib.load()
    assert 'gf_profile_sources' in _lib.EXPORTS and hasattr(lib, 'gf_profile_sources')
    header = open(os.path.join(ROOT, 'include', 'golemflavor_b200.h')).read()
    assert re.search(r'int gf_profile_sources\(', header)
    assert 'scan_profile_sources' in scan.__all__ and 'profile_source_grid' in sens.__all__


def _objective_pairs(fm_src, fm_j, theta, scale, j):
    got, gfr, gst = psh.objective(fm_src, theta, scale, SOURCES[j], INJECTED[j])
    ref, rfr, rst = psh.objective(fm_j, theta, scale)
    return got[0], gfr[0], gst[0], ref[0], rfr[0], rst[0]


def test_source_objective_equals_single_source_objective_on_prior_draws():
    """gf_profile_src_obj with source j == gf_profile_obj of the model whose source and injected composition are source j:
    ln_prob to 1e-12 relative and fr to 1e-14 at 400 prior draws per scale, static6 / FIXED / GENERIC, dims 3 and 6 (-inf
    where the Gaussian pdf underflows, as llh.multi_gaussian)."""
    finite = 0
    for dim in (3, 6):
        fm = grid_model(dim)
        theta = hh.draw(fm, 31, 0, 400)
        for scale in sens.scale_grid(dim, 10)[[0, 3, 6, 9]]:
            for j in range(len(SOURCES)):
                fmj = grid_model(dim, SOURCES[j], INJECTED[j])
                for spec in (2, 1, 0):
                    got, gfr, gst = psh.objective(fm, theta, scale, SOURCES[j], INJECTED[j], spec=spec)
                    ref, rfr, rst = psh.objective(fmj, theta, scale, spec=spec)
                    finite += int(np.isfinite(ref).sum())
                    assert_rel(got, ref, 1e-12, (dim, scale, j, spec))
                    assert np.abs(gfr - rfr).max() <= 1e-14
                    flags = _lib.ST_REFINED | _lib.ST_ILL_COND | _lib.ST_NON_FINITE | _lib.ST_OUT_OF_PRIOR
                    assert np.array_equal(gst & flags, rst & flags)
    assert finite > 10000, finite


def test_source_objective_equals_single_source_objective_on_the_fixtures(golden):
    """The same identity at the points of ref_flux.npz (fixed textures) and ref_resonance.npz (one bin's eigenvalue pair at
    relative gaps down to 1e-10: the refinement path), each at its own logLam."""
    npts, refined = 0, 0
    g = golden('ref_flux.npz')
    r = golden('ref_resonance.npz')
    points = [(str(g['tex'][i]), int(g['dim'][i]), g['theta'][i, :6], float(g['theta'][i, 10]), g['binning']) for i in range(len(g['dim']))]
    points += [(str(r['texture'][i]), int(r['dim'][i]), r['theta'][i, :6], float(r['theta'][i, 6]), r['binning']) for i in range(len(r['dim']))]
    for tex, dim, th, scale, binning in points:
        if tex == 'NONE':
            continue
        fm = grid_model(dim, texture=Texture[tex], binning=binning)
        for j in range(len(SOURCES)):
            fmj = grid_model(dim, SOURCES[j], INJECTED[j], texture=Texture[tex], binning=binning)
            got, gfr, gst, ref, rfr, rst = _objective_pairs(fm, fmj, th, scale, j)
            assert_rel(got, ref, 1e-12, (tex, dim, scale, j))
            if np.isfinite(ref[0]):
                assert np.abs(gfr - rfr).max() <= 1e-14
            flags = _lib.ST_REFINED | _lib.ST_ILL_COND | _lib.ST_NON_FINITE | _lib.ST_OUT_OF_PRIOR
            assert (gst[0] & flags) == (rst[0] & flags), (tex, dim, j, gst[0], rst[0])
        refined += bool(gst[0] & _lib.ST_REFINED)
        npts += 1
    assert npts > 200 and refined > 20, (npts, refined)


@pytest.mark.parametrize('dim', [3, 6])
def test_harness_profile_sources_against_the_single_source_profile(dim):
    """The sequential profile of (scale, source j) == profile_harness.profile (hh_profile) of the source-j model to 1e-9
    relative, five sources including the pure ones, at the null point and two scales inside SCALE_BOUNDARIES."""
    scales = sens.scale_grid(dim, 100)[[0, 60, 99]]
    kw = dict(nstarts=32, seed=27, max_evals=scan.PROFILE_MAX_EVALS, ftol=scan.PROFILE_FTOL, xtol=scan.PROFILE_XTOL)
    r = psh.profile_sources(grid_model(dim), scales, SOURCES, INJECTED, **kw)
    for j in range(len(SOURCES)):
        ref = ph.profile(grid_model(dim, SOURCES[j], INJECTED[j]), scales, **kw)
        assert_rel(r['best'][j], ref['best'], 1e-9, (dim, j))
        assert np.all(r['nconverged'][j] == 32)
        assert not np.any(r['status'][j] & (_lib.ST_NON_FINITE | _lib.ST_OUT_OF_PRIOR))


def test_harness_rows_are_independent_of_the_other_sources_and_of_splits():
    """Permuted sources give permuted rows, a repeated source repeats its row, and two task0 splits of the scales give the
    same rows: all bit for bit."""
    fm = grid_model(6)
    scales = sens.scale_grid(6, 6)
    kw = dict(nstarts=32, seed=5, max_evals=600)
    src, inj = SOURCES[:4], INJECTED[:4]
    full = psh.profile_sources(fm, scales, src, inj, **kw)
    perm = [2, 0, 3, 1]
    p = psh.profile_sources(fm, scales, src[perm], inj[perm], **kw)
    rep = psh.profile_sources(fm, scales, np.concatenate([src, src[1:2]]), np.concatenate([inj, inj[1:2]]), **kw)
    parts = [psh.profile_sources(fm, scales[:2], src, inj, task0=0, **kw), psh.profile_sources(fm, scales[2:], src, inj, task0=2, **kw)]
    for key in full:
        assert np.array_equal(p[key], full[key][perm]), key
        assert np.array_equal(rep[key][:4], full[key]) and np.array_equal(rep[key][4], full[key][1]), key
        assert np.array_equal(np.concatenate([q[key] for q in parts], axis=1), full[key]), key


def test_python_argument_checks_need_no_device():
    for bad_src, bad_inj, msg in (
            (np.ones((2, 4)), (1, 1, 1), 'sources must be'),
            (np.zeros((0, 3)), (1, 1, 1), 'sources must be'),
            (SOURCES, np.ones((3, 3)), 'injected must be'),
            ([(1, -1e-9, 1)], (1, 1, 1), 'source 0'),
            ([(1, 1, 1), (0, 0, 0)], (1, 1, 1), 'source 1'),
            ([(1, np.nan, 1)], (1, 1, 1), 'source 0'),
            (SOURCES, (0, 0, 0), 'injected composition 0')):
        with pytest.raises(ValueError, match=msg):
            scan.scan_profile_sources(None, [-40.0], bad_src, bad_inj)
        with pytest.raises(ValueError, match=msg):
            sens.profile_source_grid(bad_src, dimensions=(3,), segments=4, injected_ratio=bad_inj)


def _caller(lib, fm, nscales=5, nsrc=2, nstarts=64, stream=None, **ptrs):
    """gf_profile_sources with defaults that pass; keyword overrides replace one argument."""
    P = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    src = np.ascontiguousarray(SOURCES[:2])
    inj = np.ascontiguousarray(INJECTED[:2])
    cfg = _lib.ProfileConfig(seed=27, task0=0, nstarts=nstarts, max_evals=500, ftol=1e-10, xtol=1e-7)

    def call(model=fm.ref, cfg_=cfg, ns=nscales, s=src, i=inj, n=nsrc, **kw):
        a = dict(ptrs)
        a.update(kw)
        return lib.gf_profile_sources(model, C.byref(cfg_) if cfg_ is not None else None, a.get('scales'), ns, P(s) if s is not None else None,
                                      P(i) if i is not None else None, n, a.get('best'), a.get('argmax'), a.get('fr'), a.get('status'),
                                      a.get('counts'), stream)
    return call, cfg


def _refusals(lib, fm, call, cfg, refused):
    """Every refusal that is decided before anything touches the device."""
    refused('null pointer', model=None)
    refused('null pointer', cfg_=None)
    refused('null pointer', scales=None)
    refused('null pointer', s=None)
    refused('null pointer', i=None)
    refused('null pointer', best=None)
    refused(r'nscales = -1 outside \[0, 2\^30\]', ns=-1)
    refused(r'nsrc = 0 outside \[1, %d\]' % _lib.GF_SRC_MAX, n=0)
    refused(r'nsrc = %d outside' % (_lib.GF_SRC_MAX + 1), n=_lib.GF_SRC_MAX + 1)
    refused('no BSM path', model=scan.scan_model('unitary').ref)
    args, asimov, pset = models.bsm_model_c3([0.5, 0.5], dim=6)
    refused('sampled column', model=model.flatten(args, asimov, pset).ref)
    args, asimov, pset = models.bsm_sampled_source([0.5, 0.5], kind='angles')
    pset = ParamSet([p for p in pset if p.name != 'logLam'])
    args.fixed_scale = -40.0
    refused('samples the source', model=model.flatten(args, asimov, pset).ref)
    flat_args = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=6, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                          fixed_scale=-100.0)
    refused('Gaussian likelihood', model=model.flatten(flat_args, None, ParamSet(scan.sm_paramset(with_mass=True)), likelihood='FLAT').ref)
    for bad in ([(1, -1, 0), (1, 1, 1)], [(1, 1, 1), (0, 0, 0)], [(np.nan, 1, 1), (1, 1, 1)], [(1, np.inf, 1), (1, 1, 1)]):
        refused('source 0|source 1', s=np.ascontiguousarray(bad, dtype=np.float64))
        refused('injected', i=np.ascontiguousarray(bad, dtype=np.float64))
    for field, value, msg in (('nstarts', 48, 'multiple of 32'), ('nstarts', 512, 'multiple of 32'), ('nstarts', 0, 'multiple of 32'),
                              ('max_evals', 0, 'max_evals = 0 must be positive'), ('ftol', -1.0, 'must be non-negative'),
                              ('xtol', -1e-3, 'must be non-negative'), ('task0', -1, 'task0 = -1 is negative')):
        bad = _lib.ProfileConfig.from_buffer_copy(cfg)
        setattr(bad, field, value)
        refused(msg, cfg_=bad)
    from golemflavor_b200.param import Param
    a = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=6, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                  injected_ratio=np.ones(3) / 3, smearing=SMEARING, fixed_scale=-100.0)
    unbounded = model.flatten(a, None, ParamSet(scan.sm_paramset(with_mass=True) + [Param(name='u', value=0.0, ranges=[0., np.inf])]))
    refused('finite box', model=unbounded.ref)


def test_refusals_that_need_no_device():
    """The refusals of gf_profile_sources decided on the host: GF_ERR_ARG with the message, nothing launched (the device
    pointers are never touched, so placeholders stand in for them)."""
    build.build_library()
    lib = _lib.load()
    fm = grid_model(6)
    dummy = C.c_void_p(256)
    call, cfg = _caller(lib, fm, scales=dummy, best=dummy)

    def refused(msg, **kw):
        before = lib.gf_launch_count()
        assert call(**kw) == _lib.GF_ERR_ARG, msg
        assert re.search(msg, lib.gf_last_error().decode()), (msg, lib.gf_last_error())
        assert lib.gf_launch_count() == before

    _refusals(lib, fm, call, cfg, refused)


# ------------------------------------------------------------------ GPU


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


@pytest.mark.gpu
@pytest.mark.parametrize('dim', [3, 6])
def test_device_rows_against_the_single_source_profile(torch, dim):
    """Row j == scan_profile_grid of the source-j model (best to 1e-9); best is LnProb of the source-j frozen-scale model at
    argmax (1e-12, fr 1e-14) and the oracle (1e-10); argmax inside the box; no NON_FINITE / OUT_OF_PRIOR; best >= the
    harness - 1e-6; one launch.  A row whose Gaussian pdf underflows in the whole box is -inf in both."""
    scales = sens.scale_grid(dim, 100)[[0, 20, 40, 60, 80, 99]]
    lib = _lib.load()
    before = lib.gf_launch_count()
    d = scan.scan_profile_sources(grid_model(dim), scales, SOURCES, INJECTED, seed=27)
    assert lib.gf_launch_count() - before == 1
    assert d['best'].shape == (5, 6) and d['argmax'].shape == (5, 6, 6) and d['fr'].shape == (5, 6, 3) and d['nevals'].shape == (5, 6)
    b = box(grid_model(dim))
    assert np.all(d['argmax'] >= b[:, 0]) and np.all(d['argmax'] <= b[:, 1])
    assert not np.any(d['status'] & (_lib.ST_NON_FINITE | _lib.ST_OUT_OF_PRIOR))
    assert np.all(d['nconverged'] >= 1) and np.all(d['nevals'] > 0)
    sub = [0, 3, 5]
    finite = 0
    h = np.stack([psh.profile_sources(grid_model(dim), scales[k:k + 1], SOURCES, INJECTED, seed=27, task0=k)['best'][:, 0] for k in sub], axis=1)
    for j, (s, i) in enumerate(zip(SOURCES, INJECTED)):
        fmj = grid_model(dim, s, i)
        ref = scan.scan_profile_grid(fmj, scales, seed=27)
        assert_rel(d['best'][j], ref['best'], 1e-9, (dim, j))
        args = Namespace(source_ratio=s / s.sum(), dimension=dim, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                         injected_ratio=i / i.sum(), smearing=SMEARING)
        for k, sc in enumerate(scales):
            a = Namespace(**vars(args))
            a.fixed_scale = float(sc)
            fn = llh.LnProb(a, None, ParamSet(scan.sm_paramset(with_mass=True)))
            lnp, fr = (x.cpu().numpy() for x in fn.evaluate(d['argmax'][j, k:k + 1], want_fr=True))
            if d['best'][j, k] == -np.inf:       # the Gaussian pdf underflows everywhere in the box (source far from injected)
                assert lnp[0] == -np.inf and ref['best'][k] == -np.inf
                continue
            finite += 1
            assert abs(lnp[0] - d['best'][j, k]) <= 1e-12 * abs(lnp[0]), (dim, j, sc, lnp[0], d['best'][j, k])
            assert np.abs(fr[0] - d['fr'][j, k]).max() < 1e-14
            o = oracle_lnprob(dim, d['argmax'][j, k], sc, s, i)[0]
            assert abs(o - d['best'][j, k]) <= 1e-10 * abs(o), (dim, j, sc, o, d['best'][j, k])
    assert finite >= 15, finite
    assert np.all(d['best'][:, sub] >= h - 1e-6), (d['best'][:, sub], h)


@pytest.mark.gpu
def test_device_determinism_and_structure(torch, monkeypatch):
    """Bit-identical rows for a repeated launch, repeated and permuted sources, a task0 split of the scales, more than 256
    sources over two launches, and static6 against FIXED; GENERIC agrees to 1e-9."""
    fm = grid_model(6)
    scales = sens.scale_grid(6, 8)
    rng = np.random.default_rng(11)
    src = np.concatenate([SOURCES, rng.uniform(size=(25, 3))])
    inj = np.concatenate([INJECTED, rng.uniform(0.1, 1, size=(25, 3))])
    kw = dict(nstarts=32, seed=8, max_evals=1500)
    a = scan.scan_profile_sources(fm, scales, src, inj, **kw)
    b = scan.scan_profile_sources(fm, scales, src, inj, **kw)
    rep = scan.scan_profile_sources(fm, scales, np.concatenate([src, src[3:4]]), np.concatenate([inj, inj[3:4]]), **kw)
    perm = rng.permutation(30)
    p = scan.scan_profile_sources(fm, scales, src[perm], inj[perm], **kw)
    parts = [scan.scan_profile_sources(fm, scales[:3], src, inj, task0=0, **kw), scan.scan_profile_sources(fm, scales[3:], src, inj, task0=3, **kw)]
    monkeypatch.setenv('GF_PROFILE_SPEC', 'fixed')
    fixed = scan.scan_profile_sources(fm, scales, src, inj, **kw)
    monkeypatch.setenv('GF_PROFILE_SPEC', 'generic')
    generic = scan.scan_profile_sources(fm, scales, src, inj, **kw)
    monkeypatch.setenv('GF_PROFILE_SPEC', 'nonsense')
    with pytest.raises(ValueError, match='GF_PROFILE_SPEC'):
        scan.scan_profile_sources(fm, scales, src, inj, **kw)
    monkeypatch.delenv('GF_PROFILE_SPEC')
    for key in a:
        assert np.array_equal(a[key], b[key]), key
        assert np.array_equal(rep[key][:30], a[key]) and np.array_equal(rep[key][30], a[key][3]), key
        assert np.array_equal(p[key], a[key][perm]), key
        assert np.array_equal(np.concatenate([q[key] for q in parts], axis=1), a[key]), key
        assert np.array_equal(fixed[key], a[key]), key
    assert_rel(generic['best'], a['best'], 1e-9, 'generic')
    # 270 sources: two launches of at most 256, rows equal to the 30-source launch
    lib = _lib.load()
    few = dict(nstarts=32, seed=8, max_evals=200)
    ref = scan.scan_profile_sources(fm, scales[:2], src, inj, **few)
    before = lib.gf_launch_count()
    many = scan.scan_profile_sources(fm, scales[:2], np.concatenate([src] * 9), np.concatenate([inj] * 9), **few)
    assert lib.gf_launch_count() - before == 2
    for key in ref:
        assert np.array_equal(many[key], np.concatenate([ref[key]] * 9)), key


@pytest.mark.gpu
def test_device_refusals(torch):
    """Every refusal of gf_profile_sources: GF_ERR_ARG, the message in gf_last_error(), nothing launched and d_best
    untouched; nscales = 0 is a no-op and a valid call then runs."""
    lib = _lib.load()
    fm = grid_model(6)
    sc = torch.as_tensor(sens.scale_grid(6, 5)).cuda()
    best = torch.full((2, 5), 7.0, dtype=torch.float64, device='cuda')
    call, cfg = _caller(lib, fm, scales=_lib.ptr(sc), best=_lib.ptr(best), stream=_lib.stream_ptr(torch))

    def refused(msg, **kw):
        before = lib.gf_launch_count()
        assert call(**kw) == _lib.GF_ERR_ARG, msg
        assert re.search(msg, lib.gf_last_error().decode()), (msg, lib.gf_last_error())
        assert lib.gf_launch_count() == before

    _refusals(lib, fm, call, cfg, refused)
    # twelve columns (six with priors only) x 256 starts: 169 x 256 x 8 B of simplices do not fit in shared memory
    from golemflavor_b200.param import Param
    extra = [Param(name='nuis%d' % k, value=0.0, ranges=[-1., 1.], std=0.1) for k in range(6)]
    a = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=6, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                  injected_ratio=np.ones(3) / 3, smearing=SMEARING, fixed_scale=-100.0)
    fm12 = model.flatten(a, None, ParamSet(scan.sm_paramset(with_mass=True) + extra))
    call12, _ = _caller(lib, fm12, nstarts=256, scales=_lib.ptr(sc), best=_lib.ptr(best), stream=_lib.stream_ptr(torch))
    before = lib.gf_launch_count()
    assert call12() == _lib.GF_ERR_ARG and 'shared memory' in lib.gf_last_error().decode()
    assert lib.gf_launch_count() == before
    torch.cuda.synchronize()
    assert torch.equal(best, torch.full_like(best, 7.0))
    assert call(ns=0) == _lib.GF_OK
    torch.cuda.synchronize()
    assert torch.equal(best, torch.full_like(best, 7.0))
    assert call() == _lib.GF_OK
    torch.cuda.synchronize()
    assert not torch.isnan(best).any() and torch.isfinite(best[0]).all()   # source 1 (0:1:0) against (1:0:0) underflows: -inf


@pytest.mark.gpu
def test_limit_table_of_the_profile_source_grid_end_to_end(torch):
    """limit_table(profile_source_grid(S, dims 3 and 6, 20 segments), FREQUENTIST) against get_limit of per-source
    profile_grid results: identical NaN and discovered masks, limits equal to 1e-6; one launch per dimension."""
    lib = _lib.load()
    before = lib.gf_launch_count()
    prof, am = sens.profile_source_grid(SOURCES, dimensions=(3, 6), segments=20, distributed=False, return_argmax=True)
    assert lib.gf_launch_count() - before == 2
    lim, disc = sens.limit_table(prof, args=FREQ)
    assert lim.shape == disc.shape == (2, len(SOURCES))
    for i, d in enumerate((3, 6)):
        assert prof[d].shape == (len(SOURCES), 20, 2) and am[d].shape == (len(SOURCES), 20, 6)
    ref_lim, ref_disc = np.full_like(lim, np.nan), np.zeros_like(disc)
    for j, s in enumerate(SOURCES):
        ref = sens.profile_grid(dimensions=(3, 6), segments=20, source_ratio=s, injected_ratio=(1, 1, 1), distributed=False)
        for i, d in enumerate((3, 6)):
            assert np.array_equal(prof[d][j][:, 0], ref[d][:, 0])
            assert_rel(prof[d][j][:, 1], ref[d][:, 1], 1e-9, (d, j))
            try:
                r = sens.get_limit(ref[d][:, 0], ref[d][:, 1], args=FREQ)
            except AssertionError:
                ref_disc[i, j] = True
                continue
            if r is not None:
                ref_lim[i, j] = r
    assert np.array_equal(np.isnan(lim), np.isnan(ref_lim)) and np.array_equal(disc, ref_disc)
    f = np.isfinite(ref_lim)
    assert np.all(np.abs(lim[f] - ref_lim[f]) <= 1e-6), (lim, ref_lim)
    assert f.any()


@pytest.mark.gpu
def test_multi_gpu_nccl_profile_source_grid_is_rank_count_invariant(torch):
    """tests/dist_profile_source_check.py under torchrun on every GPU of the box (NCCL): the sharded profile source grid
    against one rank alone.  Needs >= 2 GPUs."""
    import subprocess
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs at least two GPUs')
    res = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr', '127.0.0.1',
                          '--master-port', '29737', os.path.join(HERE, 'dist_profile_source_check.py')], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    assert 'ok=True' in res.stdout
