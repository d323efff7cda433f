"""The eigen stage near level crossings.

Points of ``golden/ref_resonance.npz`` (``make_golden_resonance.py``) put the closest eigenvalue pair of one energy bin
at a chosen relative gap (splitting / spectral spread) from 1e-1 down to 1e-10, across the fast-path cut and the
ILL_COND edge, in every bin position, with 50-digit truth.  Every kernel family with a bin loop or an eigen solver is
run on them (``-m gpu``); the host harness runs the same per-point code on the CPU.

Tolerance, stated once here (``fr_bound``): where the smallest relative gap of the model's bins is >= 1e-4 the
composition is held to FR_TOL with no exception; below, a result can only be as good as the inputs' conditioning,
eps / relgap, and is held to 1e-14 + 4e-15 / relgap -- the constant of the harness's deflation test
(``test_host_logic.py::test_harness_deflation_refinement_on_near_degenerate_pairs``).
"""

import ctypes as C
import os
import struct

import numpy as np
import pytest

from golemflavor_b200 import _lib
from golemflavor_b200.enums import ParamTag, Texture
from golemflavor_b200.param import Param, ParamSet
from oracle import golem_oracle as go
from oracle import truth

import models

HERE = os.path.dirname(os.path.abspath(__file__))
FR_TOL = 1e-10
LLH_RTOL = 1e-10
SMEARING = 0.02
FAST_MIN_SIN2 = 4.7e-6                                   # gf_physics.cuh GFP_FAST_MIN_SIN2
CUT = 2.0 / np.sqrt(3.0) * np.sqrt(FAST_MIN_SIN2)        # the same cut as a relative gap, 2.5e-3
ILL_GAP = 1e-6                                           # GFP_ILL_GAP
SPEC_GENERIC, SPEC_FIXED, SPEC_NPFREE, SPEC_FIXED7, SPEC_FIXED12 = 0, 1, 3, 5, 6   # gf_model.cuh GF_SPEC_*


def fr_bound(relgap_min):
    rg = np.asarray(relgap_min, dtype=np.float64)
    return np.where(rg >= 1e-4, FR_TOL, 1e-14 + 4e-15 / rg)


def expected_flags(relgaps):
    """(REFINED expected, ILL_COND expected, decidable) for the relative gaps of a model's bins: a flag is only asserted
    when no bin lies within a factor 1.5 of its threshold."""
    rg = np.atleast_2d(relgaps)
    near = lambda t: np.any((rg > t / 1.5) & (rg < t * 1.5), axis=1)
    return np.any(rg < CUT, axis=1), np.any(rg < ILL_GAP, axis=1), ~near(CUT), ~near(ILL_GAP)


def check_fr(fr, st, ref, relgaps, what):
    rmin = np.atleast_2d(relgaps).min(axis=1)
    err = np.abs(fr - ref).max(axis=1)
    bad = err > fr_bound(rmin)
    assert not bad.any(), (what, err[bad], rmin[bad])
    assert np.abs(fr.sum(axis=1) - 1).max() < 1e-14, what
    assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY | _lib.ST_OUT_OF_PRIOR)), what
    ref_on, ill_on, dec_ref, dec_ill = expected_flags(relgaps)
    got_ref, got_ill = (st & _lib.ST_REFINED) != 0, (st & _lib.ST_ILL_COND) != 0
    assert np.array_equal(got_ref[dec_ref], ref_on[dec_ref]), (what, np.nonzero(got_ref[dec_ref] != ref_on[dec_ref]))
    assert np.array_equal(got_ill[dec_ill], ill_on[dec_ill]), (what, np.nonzero(got_ill[dec_ill] != ill_on[dec_ill]))
    return int((got_ref & dec_ref & ref_on).sum()), int((got_ill & dec_ill & ill_on).sum())


# ------------------------------------------------------------------------------------------------ fixture and models

@pytest.fixture(scope='module')
def res():
    return np.load(os.path.join(HERE, 'golden', 'ref_resonance.npz'))


@pytest.fixture(scope='module')
def asimov():
    return np.load(os.path.join(HERE, 'golden', 'ref_llh.npz'))['asimov_angles']


def window(res, i, nbins):
    """(first bin, edges, truth fr, truth relgaps) of point i in the 20-, 7- or 1-bin model."""
    b = {20: 0, 7: int(res['b7'][i]), 1: int(res['bin'][i])}[nbins]
    return b, res['binning'][b:b + nbins + 1], res['fr%d' % nbins][i], res['relgap'][i][b:b + nbins]


def theta_of(res, i, layout):
    """The point in a model's column layout: 'fixed7' (scripts/fr.py), 'fixed12' (with five nuisances), 'perm' (logLam
    first, masses interleaved: the column map), 'none11' (Texture.NONE: NP coordinates before logLam)."""
    t = res['theta'][i]
    if layout == 'fixed7':
        return t.copy()
    if layout == 'fixed12':
        return np.concatenate([t[:6], [1.0, 0.0, 1.0, 6.9, 2.5], t[6:]])
    if layout == 'perm':
        return t[PERM]
    return np.concatenate([t[:6], res['np'][i], t[6:]])


PERM = [6, 0, 4, 1, 2, 5, 3]


def lnprob_model(res, i, nbins, layout, asimov):
    from golemflavor_b200 import llh
    dim, tex = int(res['dim'][i]), str(res['texture'][i])
    args, asi, p7 = models.bsm_model_c3(asimov, dim=dim, texture=Texture[tex])
    args.binning = window(res, i, nbins)[1]
    if layout == 'none11':
        pset = models.bsm11_paramset(dim, res['np'][i])
    elif layout == 'fixed12':
        nuis = [Param(name='nuis%d' % k, value=v, ranges=[-10., 10.], std=1.0, tag=ParamTag.NUISANCE)
                for k, v in enumerate([1.0, 0.0, 1.0, 6.9, 2.5])]
        pset = ParamSet(list(p7)[:6] + nuis + [p7[6]])
    elif layout == 'perm':
        pset = ParamSet([p7[k] for k in PERM])
    else:
        pset = p7
    return llh.LnProb(args, asi, pset), pset


def truth_lnprob(pset, theta, fr_ref, asimov):
    lo, hi = np.array(pset.ranges).T
    kind = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in pset]
    th = np.atleast_2d(theta)
    return go.batch_lnprior(th, lo, hi, kind, list(pset.nominal_values), [p.std or 1.0 for p in pset]) + \
        go.batch_multi_gaussian(np.atleast_2d(fr_ref), go.angles_to_fr(asimov), SMEARING)


def lnprob_tol(ref, fr_ref, bound, bf):
    """The propagated bound of test_bsm_lnprob_against_oracle with the conditioning-aware fr bound: LLH = -|d|^2/(2 s^2)
    turns an fr error e into |d| e sqrt(3) / s^2."""
    d = np.linalg.norm(np.atleast_2d(fr_ref) - np.asarray(bf), axis=1)
    return np.maximum(LLH_RTOL * np.abs(ref), np.sqrt(3.0) * bound * d / SMEARING ** 2 + 1e-12 * np.abs(ref))


# ------------------------------------------------------------------------------------------------ host tests

def test_fixture_covers_the_strata(res):
    b, rg = res['bin'], res['relgap']
    assert set(b.tolist()) == set(range(20))
    rmin = rg.min(axis=1)
    own = rg[np.arange(len(b)), b]
    assert np.all(np.abs(np.log(own / res['target'])) < 0.05)             # the chosen bin sits at its target gap
    for lo, hi in ((CUT / 1.5, CUT), (CUT, CUT * 1.5), (1e-4, 1e-3), (ILL_GAP / 1.5, ILL_GAP), (1e-11, 1e-7), (1e-2, 1)):
        assert np.any((rmin > lo) & (rmin < hi)), (lo, hi)
    for tex in ('OET', 'OUT', 'NONE'):                       # OEU: no crossing inside the prior box (make_golden_resonance.py)
        for dim in (3, 6, 8):
            sel = (res['texture'] == tex) & (res['dim'] == dim)
            assert sel.sum() >= 4, (tex, dim)


def test_fixture_truth_at_60_digits(res):
    for i in range(0, len(res['bin']), max(1, len(res['bin']) // 6)):
        t = res['theta'][i]
        args = (t[:4], t[4:6], res['np'][i], t[6], int(res['dim'][i]))
        fr = truth.mp_flux_averaged_fr(*args, res['binning'], res['source'], dps=60)
        assert np.abs(fr - res['fr20'][i]).max() < 1e-15
        rg = truth.mp_bin_relgaps(*args, res['binning'], dps=60)
        assert np.all(np.abs(rg / res['relgap'][i] - 1) < 1e-12)


@pytest.mark.parametrize('nbins', [20, 7, 1])
def test_harness_bin_loop_on_the_fixture(res, asimov, nbins):
    """The kernels' per-point code on the host: fast path, cut, deflation, both matrix sources of the refinement (kept /
    rebuilt from the row), the FIXED, FIXED7 and GENERIC specialisations."""
    import host_harness as hh
    nref = nill = 0
    for i in range(len(res['bin'])):
        layout = 'none11' if res['texture'][i] == 'NONE' else 'fixed7'
        fn, pset = lnprob_model(res, i, nbins, layout, asimov)
        _, _, ref, rg = window(res, i, nbins)
        th = theta_of(res, i, layout)
        lp_ref = truth_lnprob(pset, th, ref, asimov)
        tol = lnprob_tol(lp_ref, ref, fr_bound(rg.min()), go.angles_to_fr(asimov))
        fixed = layout == 'fixed7'
        assert hh.model_spec(fn.model)[0] == (SPEC_FIXED7 if fixed else SPEC_NPFREE)   # NPFREE runs as GENERIC here
        runs = [(spec, rebuild) for spec in ((SPEC_FIXED7, SPEC_FIXED, SPEC_GENERIC) if fixed else (-1,)) for rebuild in (False, True)
                if not (rebuild and spec == SPEC_FIXED7)]
        for spec, rebuild in runs:
            lnp, fr, st = hh.lnprob(fn.model, th, spec=spec, rebuild=rebuild)
            a, b = check_fr(fr, st, ref[None], rg[None], (i, nbins, spec, rebuild))
            nref, nill = nref + a, nill + b
            assert abs(lnp[0] - lp_ref[0]) <= tol[0], (i, nbins, spec, rebuild, lnp[0], lp_ref[0])
        fr, st = hh.fr(fn.model, th)
        check_fr(fr, st, ref[None], rg[None], (i, nbins, 'fr'))
    assert nref > 0 and nill > 0


def test_harness_closed_form_error_at_the_fast_path_cut():
    """Haar-random unitaries Q, spectrum (t, -t/2 +- 3/4 g) s + shift (relative gap g): every matrix the closed form
    accepts must be within half the fr tolerance of the deflation refinement (accurate to ~1e-13 here), and below the
    cut the closed form must refuse."""
    from host_harness import deflate, eig
    rng = np.random.default_rng(7)
    n = 40000
    for g in (1.2e-3, 1.37e-3, 1.6e-3, 2e-3, 2.4e-3, 2.6e-3, 3e-3, 1e-2):
        z = rng.normal(size=(n, 3, 3)) + 1j * rng.normal(size=(n, 3, 3))
        q, r = np.linalg.qr(z)
        q = q * (np.diagonal(r, axis1=1, axis2=2) / np.abs(np.diagonal(r, axis1=1, axis2=2)))[:, None, :]
        top = np.where(rng.uniform(size=n) < 0.5, 1.0, -1.0)
        sc, sh = 0.3 + 2.7 * rng.uniform(size=n), 4 * rng.uniform(size=n) - 2
        lam = np.stack([top, -0.5 * top + 0.75 * g, -0.5 * top - 0.75 * g], axis=1) * sc[:, None] + sh[:, None]
        h = np.einsum('nai,ni,nbi->nab', q, lam, q.conj())
        _, _, xf, ok = eig(h)
        xd, _ = deflate(h)
        if g < CUT / 1.02:
            assert not ok.any(), g
        if g > CUT * 1.02:
            assert ok.all(), g
        if ok.any():
            err = np.abs(xf[ok] - xd[ok]).max()
            assert err < 0.5 * FR_TOL, (g, err)


def test_harness_fast_path_threshold_high_word():
    """The device compares sin^2(phi/3) with the threshold's high word: it must be the high word of the fp64 constant."""
    from host_harness import fast_min_sin2
    thr, hi = fast_min_sin2()
    assert thr == FAST_MIN_SIN2
    assert hi == struct.unpack('>II', struct.pack('>d', thr))[0]


SCALE_MATRIX = np.array([[0.5, 0.3125 + 0.125j, 0.1875 - 0.0625j],
                         [0.3125 - 0.125j, 1.0, 0.4375 + 0.0625j],
                         [0.1875 + 0.0625j, 0.4375 - 0.0625j, 1.5]])   # entries k/16: exact down to 2^-1070


def _scale_sweep(eigfun):
    exps = list(range(-1070, 1024, 7)) + [-1070, -1060, -1023, -1022, 1000, 1023]
    lam1, vec1 = eigfun(SCALE_MATRIX[None])[:2]
    hs = np.stack([np.ldexp(SCALE_MATRIX.real, e) + 1j * np.ldexp(SCALE_MATRIX.imag, e) for e in exps])
    lam, vec = eigfun(hs)[:2]
    assert np.all(np.isfinite(lam)) and np.all(np.isfinite(vec))
    for k, e in enumerate(exps):
        assert np.array_equal(vec[k], vec1[0]), e
        assert np.array_equal(lam[k], np.ldexp(lam1[0], e)), e


def test_harness_jacobi_scale_sweep():
    """gfp_herm3_jacobi at scales 2^-1070 ... 2^1023: power-of-two scaling is exact, so the eigenvectors are the same
    bits and the eigenvalues scale exactly -- no overflow of the squares, no reciprocal of a subnormal."""
    from host_harness import eig
    _scale_sweep(eig)


# ------------------------------------------------------------------------------------------------ device tests

@pytest.fixture(scope='module')
def torch():
    import torch
    assert torch.cuda.is_available(), 'these tests need a CUDA device'
    return torch


class _Counts(object):
    def __init__(self):
        self.refined = self.ill = 0

    def add(self, pair):
        self.refined += pair[0]
        self.ill += pair[1]

    def check(self, what):
        assert self.refined > 0 and self.ill > 0, (what, self.refined, self.ill)


def _groups(res, nbins, layouts):
    """Points grouped by (texture, dim, window) -- one model per group -- for each layout that applies."""
    out = {}
    for i in range(len(res['bin'])):
        none = res['texture'][i] == 'NONE'
        for layout in layouts:
            if (layout == 'none11') != none:
                continue
            key = (str(res['texture'][i]), int(res['dim'][i]), window(res, i, nbins)[0], layout)
            if none:
                key += (tuple(res['np'][i]),)
            out.setdefault(key, []).append(i)
    return out


def _block_rows(theta_pts, rng, pset):
    """A batch in which point j occupies rows 128 j + (j mod 64) and that + 64 -- both points of one thread of the
    two-points-per-thread kernel -- and benign prior draws fill the rest."""
    m = len(theta_pts)
    batch = models.draw_in_ranges(pset, 128 * m, rng)
    rows = np.array([128 * j + (j % 64) for j in range(m)])
    batch[rows] = theta_pts
    batch[rows + 64] = theta_pts
    return batch, rows


@pytest.mark.gpu
@pytest.mark.parametrize('nbins', [20, 7, 1])
def test_lnprob_kernel_on_the_fixture(torch, res, asimov, nbins):
    """gf_lnprob in the FIXED7, FIXED12, FIXED (column map) and GENERIC specialisations, theta packed, padded and SoA,
    every constructed point in both slots of a thread; the composition, status bits and log-posterior against truth."""
    from host_harness import model_spec
    lib = _lib.load()
    rng = np.random.default_rng(nbins)
    want_spec = {'fixed7': SPEC_FIXED7, 'fixed12': SPEC_FIXED12, 'perm': SPEC_FIXED, 'none11': SPEC_NPFREE}   # k_lnprob runs NPFREE as GENERIC
    cnt = _Counts()
    for key, idx in _groups(res, nbins, ('fixed7', 'fixed12', 'perm', 'none11')).items():
        layout = key[3]
        fn, pset = lnprob_model(res, idx[0], nbins, layout, asimov)
        assert model_spec(fn.model)[0] == want_spec[layout], key
        pts = np.stack([theta_of(res, i, layout) for i in idx])
        batch, rows = _block_rows(pts, rng, pset)
        n, nd = batch.shape
        th = torch.as_tensor(batch).cuda()

        def run(buf, ld_point, ld_dim):
            lnp = torch.empty(n, dtype=torch.float64, device='cuda')
            fr = torch.empty((n, 3), dtype=torch.float64, device='cuda')
            st = torch.empty(n, dtype=torch.uint8, device='cuda')
            _lib.check(lib.gf_lnprob(fn.model.ref, _lib.ptr(buf), n, ld_point, ld_dim, _lib.ptr(lnp), _lib.ptr(fr), _lib.ptr(st),
                                     _lib.stream_ptr(torch)))
            return lnp.cpu().numpy(), fr.cpu().numpy(), st.cpu().numpy()

        lnp, fr, st = run(th, nd, 1)
        wide = torch.zeros((n, nd + 3), dtype=torch.float64, device='cuda')
        wide[:, :nd] = th
        for other in (run(wide, nd + 3, 1), run(th.t().contiguous(), 1, n)):
            for a, b in zip((lnp, fr, st), other):
                assert np.array_equal(a[rows], b[rows]) and np.array_equal(a[rows + 64], b[rows + 64]), key
        ref = np.stack([window(res, i, nbins)[2] for i in idx])
        rg = np.stack([window(res, i, nbins)[3] for i in idx])
        for r in (rows, rows + 64):
            cnt.add(check_fr(fr[r], st[r], ref, rg, key))
        lp_ref = truth_lnprob(pset, pts, ref, asimov)
        tol = lnprob_tol(lp_ref, ref, fr_bound(rg.min(axis=1)), go.angles_to_fr(asimov))
        assert np.all(np.abs(lnp[rows] - lp_ref) <= tol) and np.array_equal(lnp[rows], lnp[rows + 64]), key
    cnt.check(('lnprob', nbins))


def _pinned(pset, values):
    """The ParamSet with every range [v, v]: each prior draw of a scan is exactly the point."""
    ps = ParamSet([Param(name=p.name, value=float(v), ranges=[float(v), float(v)], tag=p.tag) for p, v in zip(pset, values)])
    return ps


@pytest.mark.gpu
def test_scan_kernels_pinned_to_the_fixture(torch, res):
    """gf_scan_samples and gf_scan_hist (texture and anarchic modes) with prior boxes [v, v]: every draw is the
    constructed point, so the returned composition is compared with truth and the histogram has one cell."""
    from golemflavor_b200 import scan
    cnt = {'texture': _Counts(), 'anarchic': _Counts()}
    src = res['source']
    for i in range(len(res['bin'])):
        mode = 'anarchic' if res['texture'][i] == 'NONE' else 'texture'
        dim = int(res['dim'][i])
        base = scan.scan_paramset(mode, dim)
        vals = theta_of(res, i, 'none11' if mode == 'anarchic' else 'fixed7')
        tex = Texture.NONE if mode == 'anarchic' else Texture[str(res['texture'][i])]
        fm = scan.scan_model(mode, dimension=dim, texture=tex, binning=res['binning'], paramset=_pinned(base, vals))
        th, fr, st = scan.scan_samples(fm, 130, seed=5)
        assert np.array_equal(th, np.broadcast_to(vals, th.shape)), i
        assert np.array_equal(fr, np.broadcast_to(fr[0], fr.shape)) and np.all(st == st[0])
        cnt[mode].add(check_fr(fr[:1], st[:1], res['fr20'][i][None], res['relgap'][i][None], (mode, i)))
        h, kept = scan.scan_histogram(fm, 130, nb=25, seed=5, distributed=False)
        assert kept == 130 and np.array_equal(h, go.ternary_histogram(np.repeat(fr[:1], 130, axis=0), 25))
        assert np.abs(src.sum() - 1) < 1e-15
    for mode, c in cnt.items():
        c.check(mode)


@pytest.mark.gpu
def test_evidence_kernels_pinned_to_the_fixture(torch, res):
    """gf_scan_evidence_grid and gf_scan_evidence with the SM columns pinned to a constructed point: lnZ at the
    constructed logLam is the truth log-likelihood of that point, at two neighbouring scales that of LAPACK truth."""
    from argparse import Namespace
    from golemflavor_b200 import model, scan
    cnt = _Counts()
    inj = np.array([1., 1., 1.]) / 3
    for i in range(len(res['bin'])):
        if res['texture'][i] == 'NONE':
            continue
        dim, t = int(res['dim'][i]), res['theta'][i]
        args = Namespace(source_ratio=res['source'], dimension=dim, texture=Texture[str(res['texture'][i])], binning=res['binning'],
                         no_bsm=False, injected_ratio=list(inj), smearing=SMEARING, fixed_scale=-100.0)
        for perm in ([0, 1, 2, 3, 4, 5], [4, 0, 5, 1, 2, 3]):
            sm = scan.sm_paramset(with_mass=True, gaussian=False)
            fm = model.flatten(args, None, _pinned([sm[k] for k in perm], t[:6][perm]))
            scales = np.array([t[6] - 0.7, t[6], t[6] + 0.7])
            got = scan.scan_evidence_grid(fm, scales, 300, seed=2, distributed=False)
            fm.struct.fixed_loglam = float(t[6])
            one = scan.scan_evidence(fm, 300, seed=2, distributed=False)
            th, fr, st = scan.scan_samples(fm, 1, seed=2)
            cnt.add(check_fr(fr, st, res['fr20'][i][None], res['relgap'][i][None], ('evidence', i)))
            ll = go.batch_multi_gaussian(res['fr20'][i][None], inj, SMEARING)[0]
            tol = lnprob_tol(np.array([ll]), res['fr20'][i][None], fr_bound(res['relgap'][i].min()), inj)[0]
            assert abs(got[1] - ll) <= tol and abs(one - ll) <= tol, (i, got[1], one, ll)
            nb = truth.eigh_flux_averaged_fr(np.tile(t[:4], (2, 1)), np.tile(t[4:6], (2, 1)), res['np'][i], scales[[0, 2]], dim,
                                             res['binning'], res['source'])
            llb = go.batch_multi_gaussian(nb, inj, SMEARING)
            assert np.all(np.abs(got[[0, 2]] - llb) <= 1e-9 * np.abs(llb) + 1e-6), (i, got, llb)
    cnt.check('evidence')


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(1, 0), (2, 0), (3, 0), (3, 2)])
def test_device_sampler_on_the_fixture(torch, res, asimov, shape):
    """gf_ensemble_run with all walkers of a chain on one constructed point (one chain per point): every stretch
    proposal c - z (c - c) is the point itself, so every stored log-posterior after an accept is the sampler's own
    evaluation (two lanes per point, interleaved bins) and must equal truth."""
    from golemflavor_b200 import mcmc
    mode, blocks = shape
    cnt = _Counts()
    for layout in ('fixed7', 'none11'):
        for key, idx in _groups(res, 20, (layout,)).items():
            fn, pset = lnprob_model(res, idx[0], 20, layout, asimov)
            pts = np.stack([theta_of(res, i, layout) for i in idx])
            nw = 8
            p0 = np.repeat(pts[:, None, :], nw, axis=1)
            smp = mcmc.DeviceEnsembleSampler(nw, fn.ndim, fn, nchains=len(idx), seed=11, nfree=1, mode=mode, cluster_blocks=blocks)
            smp.run_mcmc(p0, 3)
            assert np.array_equal(np.asarray(smp.chain).reshape(len(idx), nw, 3, -1), np.broadcast_to(p0[:, :, None, :], (len(idx), nw, 3, fn.ndim)))
            assert np.asarray(smp.acceptance_fraction).min() > 0
            lnp = np.asarray(smp.lnprobability).reshape(len(idx), -1)
            ref = np.stack([res['fr20'][i] for i in idx])
            rg = res['relgap'][idx]
            lp_ref = truth_lnprob(pset, pts, ref, asimov)
            tol = lnprob_tol(lp_ref, ref, fr_bound(rg.min(axis=1)), go.angles_to_fr(asimov))
            assert np.all(np.abs(lnp - lp_ref[:, None]) <= tol[:, None]), key
            st = fn.evaluate(pts, want_fr=True, want_status=True)[2].cpu().numpy()
            ref_on, ill_on, dec_ref, dec_ill = expected_flags(rg)
            cnt.add((int((ref_on & dec_ref).sum()), int((ill_on & dec_ill).sum())))
            assert np.array_equal(((st & _lib.ST_REFINED) != 0)[dec_ref], ref_on[dec_ref])
    cnt.check(('sampler', shape))


def _constructed_spectra(rng):
    """Hermitian matrices Q diag(l) Q^+ with pair gaps 1e-2 ... 1e-12 and exact two- and threefold degeneracies."""
    hs = []
    for g in (1e-2, 1e-3, 1e-4, 1e-6, 1e-8, 1e-10, 1e-12, 0.0):
        for _ in range(6):
            z = rng.normal(size=(3, 3)) + 1j * rng.normal(size=(3, 3))
            q, _ = np.linalg.qr(z)
            lam = np.array([1.0, -0.5 + 0.75 * g, -0.5 - 0.75 * g]) * rng.uniform(0.3, 3) + rng.uniform(-2, 2)
            hs.append(q @ np.diag(lam) @ q.conj().T)
    hs.append(np.eye(3) * 1.7)
    hs.append(np.diag([2.0, 2.0, -1.0]).astype(complex))
    return np.array(hs)


def _mp_eig(h, dps=50):
    import mpmath as mp
    mp.mp.dps = dps
    m = mp.matrix([[mp.mpc(complex(h[a, b])) for b in range(3)] for a in range(3)])
    m = (m + m.H) / 2
    lam, v = mp.eighe(m)
    order = sorted(range(3), key=lambda k: lam[k])
    return np.array([float(lam[k]) for k in order]), np.array([[float(abs(v[a, k]) ** 2) for k in order] for a in range(3)])


@pytest.mark.gpu
def test_eigh3_on_constructed_spectra_and_scale_sweep(torch):
    from golemflavor_b200 import fr
    hs = _constructed_spectra(np.random.default_rng(3))
    lam, vec, st = fr.eigh3(hs)
    nill = 0
    for k, h in enumerate(hs):
        l_ref, v_ref = _mp_eig(h)
        spread = l_ref[2] - l_ref[0]
        rg = np.diff(l_ref).min() / spread if spread > 0 else 0.0
        assert np.abs(lam[k] - l_ref).max() <= 4 * 2.2e-16 * np.abs(h).max() * 3, k
        if rg > 0:
            assert np.abs(np.abs(vec[k]) ** 2 - v_ref).max() <= 1e-14 + 4e-15 / rg, (k, rg)
        if not (ILL_GAP / 1.5 < rg < ILL_GAP * 1.5):
            assert bool(st[k] & _lib.ST_ILL_COND) == (rg < ILL_GAP), (k, rg)
        nill += bool(st[k] & _lib.ST_ILL_COND)
        assert not st[k] & _lib.ST_NON_FINITE
    assert nill > 0
    _scale_sweep(lambda h: fr.eigh3(h)[:2])


@pytest.mark.gpu
def test_params_to_bsmu_on_the_fixture(torch, res):
    """gf_params_to_bsmu (the Jacobi solver on the rebuilt bin Hamiltonian) at the constructed bin of every point: |V|^2
    per bin against mpmath within the conditioning bound."""
    from golemflavor_b200 import fr
    edges = res['binning']
    centers = np.sqrt(edges[:-1] * edges[1:])
    nill = 0
    for i in range(len(res['bin'])):
        t, b, dim = res['theta'][i], int(res['bin'][i]), int(res['dim'][i])
        u = np.asarray(fr.angles_to_u(t[:4]))
        bsm = np.concatenate([res['np'][i], [t[6]]])
        v = np.asarray(fr.params_to_BSMu(bsm, dim, centers[b], mass_eigenvalues=t[4:6], sm_u=u, texture=Texture.NONE))
        import mpmath as mp
        mp.mp.dps = 50
        h = truth._mp_bin_hamiltonian(t[:4], t[4:6], res['np'][i], t[6], dim, centers[b], mp)
        lam, vm = mp.eighe(h)
        order = sorted(range(3), key=lambda k: lam[k])
        v_ref = np.array([[float(abs(vm[a, k]) ** 2) for k in order] for a in range(3)])
        rg = res['relgap'][i][b]
        assert np.abs(np.abs(v) ** 2 - v_ref).max() <= max(1e-13, 1e-14 + 4e-15 / rg), (i, rg)
        nill += rg < ILL_GAP
    assert nill > 0
