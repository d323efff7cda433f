"""Evidence grids with Monte-Carlo error bars: the grouped evidence kernels (gf_scan_evidence_grid_groups,
gf_scan_evidence_sources_groups), the leave-one-group-out lnZ of scan / sens, the jackknife errors of lnZ
(sens.evidence_error) and of the limits (sens.limit_table(..., loo=...)).

Sample i (global Philox index) is in group i mod R.  lnZ = LSE over all groups - ln N, lnZ_(-r) = LSE over the groups != r -
ln(N - n_r), sigma = sqrt((R - 1) / R * sum_r (x_(-r) - mean)^2) for lnZ and for the limit alike."""

import ctypes as C
import os
import re
import sys
from argparse import Namespace

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import models  # noqa: E402
from golemflavor_b200 import _lib, model, scan, sens  # noqa: E402
from golemflavor_b200.enums import StatCateg, Texture  # noqa: E402
from golemflavor_b200.param import ParamSet  # noqa: E402
from oracle import golem_oracle as go  # noqa: E402
from oracle import truth  # noqa: E402

SMEARING = 0.02
SOURCES = np.array([(1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (1., 2., 0.), (0.31, 0.52, 0.17)])
INJECTED = np.array([(1., 1., 1.), (1., 0., 0.), (1., 2., 0.), (0., 1., 0.), (2., 1., 1.)])
FREQ = Namespace(stat_method=StatCateg.FREQUENTIST)


# ------------------------------------------------------------------ NumPy restatement of the definitions

def np_lse(ll):
    """(max, sum exp(ll - max)) over the last axis; -inf / NaN carry no weight."""
    ll = np.where(np.isnan(ll), -np.inf, ll)
    m = ll.max(axis=-1)
    with np.errstate(invalid='ignore'):
        s = np.where(np.isfinite(m), np.exp(ll - np.where(np.isfinite(m), m, 0.0)[..., None]).sum(axis=-1), 0.0)
    return m, s


def np_ln(m, s, n):
    with np.errstate(divide='ignore'):
        return np.where(s > 0, m + np.log(np.where(s > 0, s, 1.0)) - np.log(n), -np.inf)


def np_jackknife(h, n_r):
    """(lnZ, lnZ_(-r) [R], sigma) of one set of group pairs h [R, 2] by the formulas, group by group."""
    R, N = len(h), int(np.sum(n_r))
    w = [h[r, 1] * np.exp(h[r, 0]) if h[r, 1] > 0 else 0.0 for r in range(R)]   # synthetic pairs keep exp() in range
    lnz = np.log(sum(w)) - np.log(N) if sum(w) > 0 else -np.inf
    loo = np.array([np.log(sum(w) - w[r]) - np.log(N - n_r[r]) if sum(w) - w[r] > 0 else -np.inf for r in range(R)])
    if not np.isfinite(lnz):
        sig = np.nan
    elif not np.all(np.isfinite(loo)):
        sig = np.inf
    else:
        sig = np.sqrt((R - 1) / R * np.sum((loo - loo.mean()) ** 2))
    return lnz, loo, sig


def np_limit_sigma(L, Lr):
    R = len(Lr)
    if np.isnan(L):
        return np.nan
    if np.any(np.isnan(Lr)):
        return np.inf
    return np.sqrt((R - 1) / R * np.sum((Lr - Lr.mean()) ** 2))


# ------------------------------------------------------------------ CPU


def test_group_sizes():
    for first, count, R in ((0, 100, 16), (1237, 5003, 32), (5, 3, 2), (31, 1, 32), (7, 0, 4)):
        i = np.arange(first, first + count)
        assert np.array_equal(scan.group_sizes(count, R, first), np.bincount(i % R, minlength=R))


def test_jackknife_against_the_formulas():
    """scan._group_lnz + sens.evidence_error on synthetic (max, sum) groups: ordinary groups, -inf (empty) groups, all the
    weight in one group (sigma = +inf), no weight at all (lnZ = -inf, sigma NaN)."""
    rng = np.random.default_rng(3)
    R, N, first = 16, 1000, 3
    n_r = scan.group_sizes(N, R, first)
    h = np.empty((5, R, 2))
    h[..., 0] = rng.normal(-5.0, 2.0, size=(5, R))
    h[..., 1] = rng.uniform(1.0, 40.0, size=(5, R))
    h[1, [2, 7], 0], h[1, [2, 7], 1] = -np.inf, 0.0                                  # empty groups
    h[2, 1:, 0], h[2, 1:, 1] = -np.inf, 0.0                                          # all the weight in group 0
    h[3, :, 0], h[3, :, 1] = -np.inf, 0.0                                            # no weight anywhere
    h[4, :, 0] += 700.0                                                              # large ln L
    lnz, loo = scan._group_lnz(h, N, first)
    assert lnz.shape == (5,) and loo.shape == (R, 5)
    scales = np.linspace(-40, -30, 5)
    ev = {3: np.column_stack([scales, lnz])}
    lo = {3: np.stack([np.broadcast_to(scales, (R, 5)), loo], axis=-1)}
    sig = sens.evidence_error(ev, lo)[3]
    for k in range(5):
        hk = h[k].copy()
        if k == 4:
            hk[:, 0] -= 700.0
        rl, rloo, rs = np_jackknife(hk, n_r)
        off = 700.0 if k == 4 else 0.0
        assert (np.isneginf(lnz[k]) and np.isneginf(rl)) or abs(lnz[k] - (rl + off)) <= 1e-12 * max(1.0, abs(rl + off)), k
        f = np.isfinite(rloo)
        assert np.array_equal(np.isfinite(loo[:, k]), f), k
        assert np.allclose(loo[f, k], rloo[f] + off, rtol=1e-12, atol=1e-12), k
        if np.isnan(rs):
            assert np.isnan(sig[k])
        else:
            assert sig[k] == rs or abs(sig[k] - rs) <= 1e-9 * rs, (k, sig[k], rs)
    assert np.isinf(sig[2]) and sig[2] > 0 and np.isnan(sig[3]) and np.all(np.isfinite(sig[[0, 1, 4]]))
    # the source layout: {d: [nsrc, segments, 2]} with {d: [nsrc, R, segments, 2]}
    ev2 = {3: np.stack([ev[3], ev[3]])}
    lo2 = {3: np.stack([lo[3], lo[3]])}
    s2 = sens.evidence_error(ev2, lo2)[3]
    assert s2.shape == (2, 5) and np.array_equal(s2[0], sig, equal_nan=True) and np.array_equal(s2[1], sig, equal_nan=True)


def test_jackknife_calibration_on_log_normal_weights():
    """The jackknife sigma of lnZ = ln mean(w) against the spread of lnZ over repeated synthetic experiments: ln w ~ N(0, 1.5),
    N = 4000 samples in R = 16 groups, 400 experiments from a fixed seed.  The RMS of sigma agrees with the standard deviation
    of lnZ within 10 % (the standard deviation of 400 draws alone is uncertain to ~3.5 %)."""
    rng = np.random.default_rng(2024)
    R, N, E = 16, 4000, 400
    n_r = scan.group_sizes(N, R)
    lnz, sig = np.empty(E), np.empty(E)
    for e in range(E):
        ll = rng.normal(0.0, 1.5, size=N)
        m, s = np_lse(ll.reshape(N // R, R).T)                    # sample i in group i mod R
        h = np.stack([m, s], axis=-1)
        z, loo = scan._group_lnz(h[None], N)
        lnz[e] = z[0]
        sig[e] = sens._jackknife_sigma(z, loo.T)[0]
        assert np.all(n_r == N // R)
    ratio = np.sqrt(np.mean(sig ** 2)) / np.std(lnz, ddof=1)
    assert 0.9 < ratio < 1.1, ratio


def _curves():
    """Synthetic (scale, statistic) curves: a limit that moves with the curve's slope, a flat one (no limit) and one whose
    null point is disfavoured with a negative threshold ('Discovered LV!')."""
    sc = np.concatenate([[-100.], np.linspace(-60, -20, 41)])
    lim = lambda x0, a: np.column_stack([sc, -np.maximum(sc - x0, 0.0) * a])   # noqa: E731
    return sc, lim


def test_limit_table_with_loo_is_get_limit_on_every_curve():
    """limit_table(ev, loo=...) == a hand-written loop of get_limit over the curve and its R leave-one-out curves, for both
    statistics; the limit error and the undefined count by the rules of the jackknife."""
    sc, lim = _curves()
    rng = np.random.default_rng(5)
    R = 4
    flat = np.column_stack([sc, np.zeros_like(sc)])
    ev = {3: np.stack([lim(-40.0, 3.0), lim(-45.0, 1.0), flat, lim(-35.0, 2.0)]), 6: np.stack([lim(-50.0, 2.0), flat, lim(-42.0, 0.5), lim(-38.0, 3.0)])}
    loo = {}
    for d, curves in ev.items():
        lo = np.repeat(curves[:, None], R, axis=1).copy()
        lo[..., 1] *= 1.0 + rng.normal(0.0, 0.1, size=lo.shape[:2] + (1,))        # each leave-one-out curve: another slope
        loo[d] = lo
    loo[3][3, 2] = flat                                           # one leave-one-out curve without a limit: +inf, counted
    loo[6][0, 1:3] = flat
    for kw in (dict(), dict(args=FREQ), dict(args=Namespace(stat_method=StatCateg.BAYESIAN)), dict(bayes_k=-1.0)):
        L, disc, err, nund = sens.limit_table(ev, loo=loo, **kw)
        L0, disc0 = sens.limit_table(ev, **kw)
        assert np.array_equal(L, L0, equal_nan=True) and np.array_equal(disc, disc0)
        assert L.shape == disc.shape == err.shape == nund.shape == (2, 4)
        for i, d in enumerate(ev):
            for j in range(4):
                def one(c):
                    try:
                        v = sens.get_limit(c[:, 0], c[:, 1], **kw)
                    except AssertionError:
                        return np.nan
                    return np.nan if v is None else v
                Lr = np.array([one(c) for c in loo[d][j]])
                assert np.array_equal(L[i, j], one(ev[d][j]), equal_nan=True)
                assert nund[i, j] == np.sum(np.isnan(Lr))
                ref = np_limit_sigma(L[i, j], Lr)
                assert np.array_equal(err[i, j], ref, equal_nan=True) or abs(err[i, j] - ref) <= 1e-12 * abs(ref), (kw, d, j, err[i, j], ref)
    L, disc, err, nund = sens.limit_table(ev, loo=loo)
    assert np.isinf(err[0, 3]) and nund[0, 3] >= 1 and np.isinf(err[1, 0]) and nund[1, 0] >= 2
    assert np.isnan(err[0, 2]) and np.isnan(L[0, 2]) and np.isfinite(err[0, 0])
    # a single-source evidence_grid result wrapped as one source
    one = {3: ev[3][0]}
    L1, _, e1, n1 = sens.limit_table({d: one[d][None] for d in one}, loo={3: loo[3][0][None]})
    assert L1[0, 0] == L[0, 0] and e1[0, 0] == err[0, 0] and n1[0, 0] == nund[0, 0]


def test_python_refusals_need_no_device():
    for bad in (0, 1, 3, 6, 64, 2.5, -2):
        with pytest.raises(ValueError, match='power of two'):
            sens.evidence_grid(dimensions=(3,), segments=5, samples=1000, groups=bad)
        with pytest.raises(ValueError, match='power of two'):
            sens.evidence_source_grid(SOURCES, dimensions=(3,), segments=5, samples=1000, groups=bad)
        with pytest.raises(ValueError, match='power of two'):
            scan.scan_evidence_grid(None, [-40.0], 1000, groups=bad)
        with pytest.raises(ValueError, match='power of two'):
            scan.scan_evidence_sources(None, [-40.0], SOURCES, (1, 1, 1), 1000, groups=bad)
    with pytest.raises(ValueError, match='at least one sample'):
        sens.evidence_grid(dimensions=(3,), segments=5, samples=15, groups=16)
    with pytest.raises(ValueError, match='at least one sample'):
        sens.evidence_source_grid(SOURCES, dimensions=(3,), segments=5, samples=1, groups=2)
    sc, lim = _curves()
    ev = {3: np.stack([lim(-40.0, 3.0)] * 2)}
    with pytest.raises(ValueError, match='do not match'):
        sens.limit_table(ev, loo={3: np.stack([lim(-40.0, 3.0)] * 2)})                 # no group axis
    with pytest.raises(ValueError, match='do not match'):
        sens.limit_table(ev, loo={3: np.zeros((3, 4, len(sc), 2))})                    # a different number of sources
    with pytest.raises(ValueError, match='dimensions'):
        sens.limit_table(ev, loo={6: np.zeros((2, 4, len(sc), 2))})
    with pytest.raises(ValueError, match='do not match'):
        sens.evidence_error({3: ev[3][0]}, {3: np.zeros((4, 7, 2))})
    with pytest.raises(ValueError, match='dimensions'):
        sens.evidence_error({3: ev[3][0], 6: ev[3][0]}, {3: np.zeros((4, len(sc), 2))})
    # an empty table: empty results, no error
    L, disc, err, nund = sens.limit_table({}, loo={})
    assert L.shape == disc.shape == err.shape == nund.shape == (0, 0)
    assert sens.evidence_error({}, {}) == {}


def test_abi_declares_the_grouped_entry_points():
    for name in ('gf_scan_evidence_grid_groups', 'gf_scan_evidence_grid_groups_workspace', 'gf_scan_evidence_sources_groups',
                 'gf_scan_evidence_sources_groups_workspace'):
        assert name in _lib.EXPORTS
    header = open(os.path.join(os.path.dirname(HERE), 'include', 'golemflavor_b200.h')).read()
    assert 'gf_scan_evidence_sources_groups(' in header and 'd_lse /*[nsrc][nscales][groups][2]*/' in header


# ------------------------------------------------------------------ GPU


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


def grid_model(dim, texture=Texture.OET, source=(1., 2., 0.), injected=(1., 1., 1.)):
    return sens._grid_model(dim, texture, np.array(source), np.array(injected), SMEARING, scan.DEFAULT_BINNING)


def fixed_model(dim, texture=Texture.OET):
    """The grid model with the mass columns first: not the six-column head of sens.py, so the FIXED specialisation."""
    args = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=dim, texture=texture, binning=scan.DEFAULT_BINNING, no_bsm=False,
                     injected_ratio=np.array([1., 1., 1.]) / 3, smearing=SMEARING, fixed_scale=-100.0)
    ps = scan.sm_paramset(with_mass=True)
    return model.flatten(args, None, ParamSet(ps[4:] + ps[:4]))


def generic_model():
    """A sampled-source model with the scale frozen (GENERIC specialisation)."""
    g = np.load(os.path.join(HERE, 'golden', 'ref_llh.npz'))
    a9, as9, ps9 = models.bsm_sampled_source(g['asimov_angles'], 'angles', 6, Texture.OUT)
    a9.fixed_scale = -100.0
    return model.flatten(a9, as9, ParamSet([p for p in ps9 if p.name != 'logLam']))


def grid_lse(torch, fm, scales, first, count, R, seed=26):
    """Raw (max, sum) pairs [ns, R, 2] of one gf_scan_evidence_grid_groups call."""
    lib = _lib.load()
    sc = torch.as_tensor(np.asarray(scales, dtype=np.float64)).cuda()
    lse = torch.empty((len(scales), R, 2), dtype=torch.float64, device='cuda')
    lse[..., 0], lse[..., 1] = -np.inf, 0.0
    nbytes = int(lib.gf_scan_evidence_grid_groups_workspace(len(scales), R))
    work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=seed, first_index=first, count=count, nb=0)
    _lib.check(lib.gf_scan_evidence_grid_groups(fm.ref, C.byref(cfg), _lib.ptr(sc), len(scales), R, _lib.ptr(lse), _lib.ptr(work), nbytes,
                                                _lib.stream_ptr(torch)))
    return lse.cpu().numpy()


def sources_lse(torch, fm, scales, src, inj, first, count, R, seed=26):
    """Raw (max, sum) pairs [nsrc, ns, R, 2] of one gf_scan_evidence_sources_groups call."""
    lib = _lib.load()
    src, inj = scan.source_rows(src, inj)
    sc = torch.as_tensor(np.asarray(scales, dtype=np.float64)).cuda()
    lse = torch.empty((len(src), len(scales), R, 2), dtype=torch.float64, device='cuda')
    lse[..., 0], lse[..., 1] = -np.inf, 0.0
    nbytes = int(lib.gf_scan_evidence_sources_groups_workspace(len(scales), len(src), R))
    work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=seed, first_index=first, count=count, nb=0)
    _lib.check(lib.gf_scan_evidence_sources_groups(fm.ref, C.byref(cfg), _lib.ptr(sc), len(scales), src.ctypes.data_as(C.c_void_p),
                                                   inj.ctypes.data_as(C.c_void_p), len(src), R, _lib.ptr(lse), _lib.ptr(work), nbytes,
                                                   _lib.stream_ptr(torch)))
    return lse.cpu().numpy()


def group_lnz(h, first, count):
    """per-(..., group) lnZ_r = LSE_r - ln n_r of raw pairs h[..., R, 2]"""
    return np_ln(h[..., 0], h[..., 1], scan.group_sizes(count, h.shape[-2], first))


def assert_close(got, ref, rtol, what=''):
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)), what
    f = np.isfinite(ref)
    assert np.all(np.isfinite(got[f])), what
    err = np.abs(got[f] - ref[f]) / np.maximum(1.0, np.abs(ref[f]))
    assert err.size == 0 or err.max() <= rtol, (what, err.max())


def truth_ll(theta, dim, texture, sc, source, injected, mass_first=False):
    sm, mass = (theta[:, 2:6], theta[:, 0:2]) if mass_first else (theta[:, :4], theta[:, 4:6])
    fr = truth.eigh_flux_averaged_fr(sm, mass, model.TEXTURE_ANGLES[texture.name], np.full(len(theta), sc), dim, scan.DEFAULT_BINNING,
                                     np.asarray(source) / np.sum(source))
    return go.batch_multi_gaussian(fr, np.asarray(injected) / np.sum(injected), SMEARING)


FIRST, COUNT = 1237, 5003          # first index not a multiple of 32; count not a multiple of R or of 256


@pytest.mark.gpu
@pytest.mark.parametrize('spec', ['static6', 'fixed', 'generic'])
def test_per_group_truth_merge_identity_and_shards(torch, spec):
    """Every (scale, group) lnZ of the grid kernel against the host grouping of per-sample likelihoods (truth physics for
    static6 / FIXED, the per-point kernel's compositions for the sampled-source GENERIC model), 1e-9; lnZ merged from the
    groups against the ungrouped kernel, 1e-12; two sample shards, one starting at an index that is not a multiple of R,
    merged per group against one call, 1e-12."""
    cases = {'static6': [(3, grid_model(3)), (6, grid_model(6, Texture.OUT))], 'fixed': [(3, fixed_model(3)), (6, fixed_model(6, Texture.OUT))],
             'generic': [(6, generic_model())]}[spec]
    for dim, fm in cases:
        texture = Texture.OUT if (dim == 6 and spec != 'generic') else Texture.OET
        scales = sens.scale_grid(dim, 12)[[0, 3, 6, 9, 11]]
        theta, _, _ = scan.scan_samples(fm, COUNT, seed=26, first_index=FIRST)
        ll = np.empty((len(scales), COUNT))
        for k, sc in enumerate(scales):
            if spec == 'generic':
                fm.struct.fixed_loglam = float(sc)
                _, fr, _ = scan.scan_samples(fm, COUNT, seed=26, first_index=FIRST)
                ll[k] = go.batch_multi_gaussian(fr, np.array(fm.struct.fr_bf), fm.struct.smearing)
            else:
                ll[k] = truth_ll(theta, dim, texture, sc, (1, 2, 0), (1, 1, 1), mass_first=spec == 'fixed')
        grp = (FIRST + np.arange(COUNT))
        for R in (2, 16, 32):
            h = grid_lse(torch, fm, scales, FIRST, COUNT, R)
            got = group_lnz(h, FIRST, COUNT)
            ref = np.empty_like(got)
            for r in range(R):
                m, s = np_lse(ll[:, grp % R == r])
                ref[:, r] = np_ln(m, s, np.sum(grp % R == r))
            assert np.isfinite(ref).sum() >= ref.size // 3, (spec, dim, R)
            assert_close(got, ref, 1e-9, (spec, dim, R, 'per group'))
            lnz, loo = scan.scan_evidence_grid(fm, scales, COUNT, seed=26, first_index=FIRST, distributed=False, groups=R)
            one = scan.scan_evidence_grid(fm, scales, COUNT, seed=26, first_index=FIRST, distributed=False)
            assert lnz.shape == one.shape and loo.shape == (R, len(scales))
            assert_close(lnz, one, 1e-12, (spec, dim, R, 'merge'))
            n1 = 2001                                                                        # 2001 mod R != 0
            a, b = grid_lse(torch, fm, scales, FIRST, n1, R), grid_lse(torch, fm, scales, FIRST + n1, COUNT - n1, R)
            with np.errstate(divide='ignore'):
                merged = np.logaddexp(np.log(a[..., 1]) + a[..., 0], np.log(b[..., 1]) + b[..., 0]) - np.log(scan.group_sizes(COUNT, R, FIRST))
            assert_close(merged, got, 1e-12, (spec, dim, R, 'shards'))


@pytest.mark.gpu
def test_source_grid_per_group_truth_and_identities(torch):
    """The grouped source grid: per-(source, scale, group) truth, 1e-9; lnZ merged against the ungrouped source grid, 1e-12;
    row j against the grouped evidence grid of the source-j model, 1e-12; repeated and permuted sources bit-identical; two
    shards merged per group, 1e-12; a one-source launch (several threads per unit)."""
    for dim, texture in ((3, Texture.OET), (6, Texture.OUT)):
        fm = grid_model(dim, texture)
        scales = sens.scale_grid(dim, 12)[[0, 2, 5, 8, 11]]
        theta, _, _ = scan.scan_samples(fm, COUNT, seed=26, first_index=FIRST)
        grp = FIRST + np.arange(COUNT)
        for R in (2, 16, 32):
            h = sources_lse(torch, fm, scales, SOURCES, INJECTED, FIRST, COUNT, R)
            got = group_lnz(h, FIRST, COUNT)
            if R != 2 or dim == 3:
                ref = np.empty_like(got)
                for j, (s, inj) in enumerate(zip(SOURCES, INJECTED)):
                    for k, sc in enumerate(scales):
                        ll = truth_ll(theta, dim, texture, sc, s, inj)
                        for r in range(R):
                            m, ss = np_lse(ll[grp % R == r][None])
                            ref[j, k, r] = np_ln(m, ss, np.sum(grp % R == r))[0]
                assert_close(got, ref, 1e-9, (dim, R, 'sources per group'))
            lnz, loo = scan.scan_evidence_sources(fm, scales, SOURCES, INJECTED, COUNT, seed=26, first_index=FIRST, distributed=False, groups=R)
            assert lnz.shape == (len(SOURCES), len(scales)) and loo.shape == (len(SOURCES), R, len(scales))
            one = scan.scan_evidence_sources(fm, scales, SOURCES, INJECTED, COUNT, seed=26, first_index=FIRST, distributed=False)
            assert_close(lnz, one, 1e-12, (dim, R, 'merge'))
            for j in (0, 3, 4):
                fj = grid_model(dim, texture, SOURCES[j], INJECTED[j])
                gz, gl = scan.scan_evidence_grid(fj, scales, COUNT, seed=26, first_index=FIRST, distributed=False, groups=R)
                assert_close(lnz[j], gz, 1e-12, (dim, R, j, 'vs grid'))
                assert_close(loo[j], gl, 1e-12, (dim, R, j, 'vs grid loo'))
            n1 = 2001
            a = sources_lse(torch, fm, scales, SOURCES, INJECTED, FIRST, n1, R)
            b = sources_lse(torch, fm, scales, SOURCES, INJECTED, FIRST + n1, COUNT - n1, R)
            with np.errstate(divide='ignore'):
                merged = np.logaddexp(np.log(a[..., 1]) + a[..., 0], np.log(b[..., 1]) + b[..., 0]) - np.log(scan.group_sizes(COUNT, R, FIRST))
            assert_close(merged, got, 1e-12, (dim, R, 'shards'))
            single = sources_lse(torch, fm, scales, SOURCES[4:5], INJECTED[4:5], FIRST, COUNT, R)
            assert_close(group_lnz(single, FIRST, COUNT)[0], got[4], 1e-12, (dim, R, 'one source'))
    # repeated and permuted sources: bit-identical rows (30 sources, several slots per thread)
    fm = grid_model(6)
    scales = sens.scale_grid(6, 23)
    rng = np.random.default_rng(7)
    src = np.concatenate([SOURCES, rng.uniform(size=(25, 3))])
    inj = np.concatenate([INJECTED, rng.uniform(0.1, 1, size=(25, 3))])
    a = sources_lse(torch, fm, scales, src, inj, 0, 100_003, 16)
    rep = sources_lse(torch, fm, scales, np.concatenate([src, src[3:4]]), np.concatenate([inj, inj[3:4]]), 0, 100_003, 16)
    assert np.array_equal(rep[30], rep[3]) and np.array_equal(rep[:30], a)
    perm = rng.permutation(30)
    p = sources_lse(torch, fm, scales, src[perm], inj[perm], 0, 100_003, 16)
    assert np.array_equal(p, a[perm])


@pytest.mark.gpu
def test_launch_count_and_source_splits(torch):
    """One launch per dimension; a source list longer than one grouped launch takes 4096 / R per launch (128 at R = 32); the
    split result equals the unsplit rows."""
    lib = _lib.load()
    before = lib.gf_launch_count()
    ev, loo = sens.evidence_grid(dimensions=(3, 6), segments=10, samples=20_000, groups=16)
    assert lib.gf_launch_count() - before == 2
    assert ev[3].shape == (10, 2) and loo[3].shape == (16, 10, 2) and np.array_equal(loo[6][5, :, 0], ev[6][:, 0])
    ev2, mx, loo2 = sens.evidence_grid(dimensions=(3, 6), segments=10, samples=20_000, groups=16, return_maxllh=True)
    assert np.array_equal(ev2[3], ev[3]) and np.array_equal(loo2[6], loo[6]) and mx[3].shape == (10, 2)
    ref_mx = sens.evidence_grid(dimensions=(3, 6), segments=10, samples=20_000, return_maxllh=True)[1]
    assert np.array_equal(mx[3], ref_mx[3]) and np.array_equal(mx[6], ref_mx[6])
    rng = np.random.default_rng(9)
    src = np.concatenate([SOURCES, rng.uniform(size=(125, 3))])                    # 130 sources: 128 + 2 at R = 32
    before = lib.gf_launch_count()
    ev, loo = sens.evidence_source_grid(src, dimensions=(3, 6), segments=10, samples=20_000, groups=32)
    assert lib.gf_launch_count() - before == 4
    assert ev[3].shape == (130, 10, 2) and loo[6].shape == (130, 32, 10, 2)
    part, ploo = sens.evidence_source_grid(src[120:], dimensions=(3, 6), segments=10, samples=20_000, groups=32)
    for d in (3, 6):
        assert_close(ev[d][120:, :, 1], part[d][:, :, 1], 1e-12, 'split')
        assert_close(loo[d][120:, ..., 1], ploo[d][..., 1], 1e-12, 'split loo')
    before = lib.gf_launch_count()
    sens.evidence_source_grid(src, dimensions=(3,), segments=10, samples=20_000, groups=16)
    assert lib.gf_launch_count() - before == 1


@pytest.mark.gpu
def test_c_abi_refusals(torch):
    """Every refusal of the grouped entry points: GF_ERR_ARG, the message, no launch and the output untouched."""
    lib = _lib.load()
    fm = grid_model(6)
    sc = torch.as_tensor(sens.scale_grid(6, 5)).cuda()
    R = 16
    lse = torch.full((2, 5, R, 2), 7.0, dtype=torch.float64, device='cuda')
    gb = int(lib.gf_scan_evidence_grid_groups_workspace(5, R))
    sb = int(lib.gf_scan_evidence_sources_groups_workspace(5, 2, R))
    assert gb > int(lib.gf_scan_evidence_grid_workspace(5)) and sb > int(lib.gf_scan_evidence_sources_workspace(5, 2))
    for bad in (0, 1, 3, 64, -2):
        assert lib.gf_scan_evidence_grid_groups_workspace(5, bad) == 0 and lib.gf_scan_evidence_sources_groups_workspace(5, 2, bad) == 0
    assert lib.gf_scan_evidence_sources_groups_workspace(5, 129, 32) == 0 and lib.gf_scan_evidence_sources_groups_workspace(5, 128, 32) > 0
    assert lib.gf_scan_evidence_sources_groups_workspace(5, 256, 16) > 0
    work = torch.empty(max(gb, sb), dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=26, first_index=0, count=1000, nb=0)
    src, inj = np.ascontiguousarray(SOURCES[:2]), np.ascontiguousarray(INJECTED[:2])
    P = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    stream = _lib.stream_ptr(torch)

    def grid(model=fm.ref, cfg_=cfg, scales=_lib.ptr(sc), ns=5, groups=R, out=_lib.ptr(lse), w=_lib.ptr(work), wb=gb):
        return lib.gf_scan_evidence_grid_groups(model, C.byref(cfg_) if cfg_ is not None else None, scales, ns, groups, out, w, wb, stream)

    def sources(model=fm.ref, cfg_=cfg, scales=_lib.ptr(sc), ns=5, s=src, i=inj, nsrc=2, groups=R, out=_lib.ptr(lse), w=_lib.ptr(work), wb=sb):
        return lib.gf_scan_evidence_sources_groups(model, C.byref(cfg_) if cfg_ is not None else None, scales, ns, P(s) if s is not None else None,
                                                   P(i) if i is not None else None, nsrc, groups, out, w, wb, stream)

    def refused(fn, msg, **kw):
        before = lib.gf_launch_count()
        assert fn(**kw) == _lib.GF_ERR_ARG, msg
        assert re.search(msg, lib.gf_last_error().decode()), (msg, lib.gf_last_error())
        assert lib.gf_launch_count() == before

    unitary = scan.scan_model('unitary').ref
    args, asimov, pset = models.bsm_model_c3([0.5, 0.5], dim=6)
    sampled_scale = model.flatten(args, asimov, pset).ref
    for fn in (grid, sources):
        refused(fn, 'null pointer', cfg_=None)
        refused(fn, 'null pointer', scales=None)
        refused(fn, 'null pointer', out=None)
        refused(fn, r'nscales = 0 outside \[1, 65535\]', ns=0)
        for bad in (0, 1, 3, 48, 64, -16):
            refused(fn, r'groups = %d is not a power of two in \[2, 32\]' % bad, groups=bad)
        refused(fn, 'no BSM path', model=unitary)
        refused(fn, 'sampled column', model=sampled_scale)
        refused(fn, 'workspace of 0 B is too small', w=None, wb=0)
        refused(fn, 'too small', wb=16)
    # 1000 samples take 4 blocks in x: 1000 B hold the ungrouped partials of this call (5 x 4 x 16 B) but not the grouped ones
    refused(grid, 'workspace of 1000 B is too small', wb=1000)
    refused(sources, 'null pointer', model=None)
    refused(sources, 'null pointer', s=None)
    refused(sources, r'nsrc = 0 outside \[1, %d\]' % _lib.GF_SRC_MAX, nsrc=0)
    refused(sources, r'nsrc = 129 with 32 groups: one launch takes at most 128 sources', nsrc=129, groups=32)
    refused(sources, 'source', s=np.ascontiguousarray([(1, -1, 0), (1, 1, 1)], dtype=np.float64))
    refused(sources, 'injected', i=np.ascontiguousarray([(1, 1, 1), (0, 0, 0)], dtype=np.float64))
    flat_args = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=6, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                          fixed_scale=-100.0)
    refused(sources, 'Gaussian likelihood', model=model.flatten(flat_args, None, ParamSet(scan.sm_paramset(with_mass=True)), likelihood='FLAT').ref)
    refused(sources, 'samples the source', model=generic_model().ref)
    refused(sources, 'workspace of 1000 B is too small', wb=1000)
    torch.cuda.synchronize()
    assert torch.equal(lse, torch.full_like(lse, 7.0))
    lse[..., 0], lse[..., 1] = -np.inf, 0.0
    assert grid(out=_lib.ptr(lse[0])) == _lib.GF_OK and sources() == _lib.GF_OK
    torch.cuda.synchronize()
    assert torch.isfinite(lse[..., 0]).any()


@pytest.mark.gpu
def test_statistical_calibration_over_seeds(torch):
    """64 fixed seeds x 2e4 samples, R = 16, dims 3 and 6 at 12 scales: at every scale where lnZ is finite for every seed
    and the RMS sigma is below 1, the jackknife's RMS sigma over the seeds and the standard deviation of lnZ over the seeds
    agree within a factor of [0.7, 1.4] (the standard deviation of 64 draws alone is uncertain to ~9 %).  Scales where sigma is at
    the rounding level (the composition does not depend on the sampled parameters there) are skipped."""
    seeds = range(1000, 1064)
    lnz, sig = {3: [], 6: []}, {3: [], 6: []}
    for s in seeds:
        ev, loo = sens.evidence_grid(dimensions=(3, 6), segments=12, samples=20_000, seed=s, groups=16)
        err = sens.evidence_error(ev, loo)
        for d in (3, 6):
            lnz[d].append(ev[d][:, 1])
            sig[d].append(err[d])
    checked = 0
    for d in (3, 6):
        z, e = np.array(lnz[d]), np.array(sig[d])
        for k in range(z.shape[1]):
            if not np.all(np.isfinite(z[:, k])) or not np.all(np.isfinite(e[:, k])):
                continue
            rms = np.sqrt(np.mean(e[:, k] ** 2))
            if rms >= 1.0 or rms < 1e-9:   # below 1e-9: the composition no longer depends on the samples, lnZ varies by rounding only
                continue
            spread = np.std(z[:, k], ddof=1)
            assert 0.7 <= rms / spread <= 1.4, (d, k, rms, spread)
            checked += 1
    assert checked >= 6, checked


@pytest.mark.gpu
def test_limit_table_with_errors_end_to_end(torch):
    """evidence_source_grid(..., groups=16) -> limit_table(..., loo=...): the limits are the ungrouped table's -- the same cells
    defined and discovered, the values to 1e-9 (the grouped lnZ is the ungrouped one summed in another order, equal to 1e-12
    relative, and the spline carries that rounding into the limit) -- and the errors are finite where every leave-one-out limit
    exists, +inf where some does not and NaN where there is no limit."""
    kw = dict(dimensions=(3, 6), segments=20, samples=50_000)
    ev, loo = sens.evidence_source_grid(SOURCES, injected_ratio=(1, 1, 1), groups=16, **kw)
    ref = sens.evidence_source_grid(SOURCES, injected_ratio=(1, 1, 1), **kw)
    L, disc, err, nund = sens.limit_table(ev, loo=loo)
    L0, disc0 = sens.limit_table(ref)
    assert np.array_equal(np.isnan(L), np.isnan(L0)) and np.array_equal(disc, disc0)
    assert np.isfinite(L).any() and np.max(np.abs(L - L0)[~np.isnan(L)]) <= 1e-9
    assert np.all(np.isnan(err[np.isnan(L)]))
    defined = ~np.isnan(L)
    assert np.all(np.isfinite(err[defined & (nund == 0)])) and np.all(np.isposinf(err[defined & (nund > 0)]))
    assert np.all(err[defined & (nund == 0)] >= 0)
    sig = sens.evidence_error(ev, loo)
    for d in (3, 6):
        assert sig[d].shape == (len(SOURCES), 20)
        fin = np.isfinite(ev[d][..., 1])
        assert np.all(np.isnan(sig[d][~fin])) and np.all(sig[d][fin] >= 0)
    Lf, _, ef, _ = sens.limit_table(ev, loo=loo, args=FREQ)                       # the other threshold on the same curves
    assert np.all(np.isnan(ef[np.isnan(Lf)]))


@pytest.mark.gpu
def test_multi_gpu_nccl_grouped_grids_are_rank_count_invariant(torch):
    """tests/dist_jackknife_check.py under torchrun on every GPU of the box (NCCL): the sharded grouped grids against one rank
    alone.  Needs >= 2 GPUs."""
    import subprocess
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs at least two GPUs')
    res = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr', '127.0.0.1',
                          '--master-port', '29741', os.path.join(HERE, 'dist_jackknife_check.py')], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    assert 'ok=True' in res.stdout
