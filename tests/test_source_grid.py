"""The evidence grid over many source compositions (gf_scan_evidence_sources, scan.scan_evidence_sources,
sens.evidence_source_grid) and the limit table (sens.limit_table).

CPU tests check the transition identity (fr of any source from the bin-width-weighted transition sums equals the per-bin
composition of gf_point_fr), the whole per-sample task run sequentially on the host against the oracle, limit_table against
get_limit, the ABI and the argument checks that need no device.  GPU tests hold the device to sens.evidence_grid run once per
source, to the oracle, and to its own structure (repeats, repeated and permuted sources, splits over launches and samples,
ranks), and check every refusal of the C entry point."""

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
from host_harness import source_harness as sh  # noqa: E402
import models  # noqa: E402
from golemflavor_b200 import _lib, build, model, scan, sens  # noqa: E402
from golemflavor_b200.enums import StatCateg, Texture  # noqa: E402
from golemflavor_b200.param import ParamSet  # noqa: E402
from oracle import golem_oracle as go  # noqa: E402
from oracle import truth  # noqa: E402

ROOT = os.path.dirname(HERE)
SMEARING = 0.02
SOURCES = np.array([(1., 0., 0.), (0., 1., 0.), (0., 0., 1.), (1., 2., 0.), (0.31, 0.52, 0.17)])
INJECTED = np.array([(1., 1., 1.), (1., 0., 0.), (1., 2., 0.), (0., 1., 0.), (2., 1., 1.)])


def grid_model(dim, texture=Texture.OET):
    """The model of sens.evidence_grid / evidence_source_grid (its own source and injected composition are ignored by the
    source-grid kernel)."""
    return sens._grid_model(dim, texture, np.array([1., 2., 0.]), np.array([1., 1., 1.]), SMEARING, scan.DEFAULT_BINNING)


def lse_of(ll):
    """(max, sum exp(ll - max)) over the last axis; -inf / NaN carry no weight."""
    ll = np.where(np.isnan(ll), -np.inf, ll)
    m = ll.max(axis=-1)
    with np.errstate(invalid='ignore'):
        s = np.where(np.isfinite(m), np.exp(ll - np.where(np.isfinite(m), m, 0.0)[..., None]).sum(axis=-1), 0.0)
    return m, s


def lnz_of(m, s, n):
    with np.errstate(divide='ignore'):
        return np.where(s > 0, m + np.log(np.where(s > 0, s, 1.0)) - np.log(n), -np.inf)


def oracle_lnz(dim, texture, theta, scales, sources, injected):
    """lnZ[nsrc, ns] of prior samples theta (six SM columns) from truth.eigh_flux_averaged_fr + batch_multi_gaussian."""
    out = np.empty((len(sources), len(scales)))
    for j, (s, inj) in enumerate(zip(sources, injected)):
        for k, sc in enumerate(scales):
            fr = truth.eigh_flux_averaged_fr(theta[:, :4], theta[:, 4:6], model.TEXTURE_ANGLES[texture.name], np.full(len(theta), sc), dim,
                                             scan.DEFAULT_BINNING, s / s.sum())
            ll = go.batch_multi_gaussian(fr, inj / inj.sum(), SMEARING)
            m, ssum = lse_of(ll[None])
            out[j, k] = lnz_of(m, ssum, len(theta))[0]
    return out


def assert_lnz_close(got, ref, rtol, what=''):
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)), what
    f = np.isfinite(ref)
    assert np.all(np.isfinite(got[f])), what
    err = np.abs(got[f] - ref[f]) / np.maximum(1.0, np.abs(ref[f]))
    assert err.size == 0 or err.max() <= rtol, (what, err.max())


# ------------------------------------------------------------------ CPU


def test_transition_identity_on_the_flux_fixture():
    """fr of a source from (A00, A01, A11) == gf_point_fr with that source as the model's, for the ref_flux.npz points
    (textures OET, OUT, OEU and Haar-random NP mixing), FIXED and GENERIC code paths."""
    g = np.load(os.path.join(HERE, 'golden', 'ref_flux.npz'))
    rng = np.random.default_rng(3)
    srcs = np.concatenate([SOURCES[:4], rng.uniform(size=(1, 3))])
    worst, npts = 0.0, 0
    for tex in ('OET', 'OUT', 'OEU', 'NONE'):
        for dim in sorted(set(g['dim'].tolist())):
            sel = (g['tex'] == tex) & (g['dim'] == dim)
            if not sel.any():
                continue
            th = g['theta'][sel]
            fm = model.flatten(models.bsm_args(dim, Texture.NONE, (1, 2, 0)), None, models.bsm11_paramset(dim), likelihood='FLAT')
            _, fr, st = sh.transition_fr(fm, th, srcs)
            assert not np.any(st & _lib.ST_NON_FINITE)
            for j, s in enumerate(srcs):
                fmj = model.flatten(models.bsm_args(dim, Texture.NONE, s), None, models.bsm11_paramset(dim), likelihood='FLAT')
                ref, _ = hh.fr(fmj, th)
                worst = max(worst, np.abs(fr[:, j] - ref).max())
                if tex != 'NONE':   # the fixed-texture model: FIXED specialisation and the generic path
                    fm7 = model.flatten(models.bsm_args(dim, Texture[tex], s), None, models.bsm7_paramset(dim), likelihood='FLAT')
                    th7 = np.delete(th, [6, 7, 8, 9], axis=1)
                    ref7, _ = hh.fr(fm7, th7)
                    for spec in (1, 0):
                        _, fr7, _ = sh.transition_fr(fm7, th7, s, spec=spec)
                        worst = max(worst, np.abs(fr7[:, 0] - ref7).max())
            npts += len(th)
    assert npts > 100
    assert worst <= 1e-14, worst


def test_transition_identity_near_level_crossings():
    """The same identity on ref_resonance.npz, whose points put one bin's closest eigenvalue pair at relative gaps down to
    1e-10 -- the refinement path of the bin loop -- and whose flags must agree with gf_point_fr's."""
    res = np.load(os.path.join(HERE, 'golden', 'ref_resonance.npz'))
    rng = np.random.default_rng(5)
    srcs = np.concatenate([SOURCES[:4], rng.uniform(size=(1, 3))])
    worst, refined = 0.0, 0
    for i in range(len(res['bin'])):
        dim, tex = int(res['dim'][i]), str(res['texture'][i])
        t = res['theta'][i]
        if tex == 'NONE':
            pset, th = models.bsm11_paramset(dim, res['np'][i]), np.concatenate([t[:6], res['np'][i], t[6:]])
            texture = Texture.NONE
        else:
            pset, th, texture = models.bsm7_paramset(dim), t, Texture[tex]
        _, fr, st = sh.transition_fr(model.flatten(models.bsm_args(dim, texture, (1, 2, 0)), None, pset, likelihood='FLAT'), th, srcs)
        for j, s in enumerate(srcs):
            ref, rst = hh.fr(model.flatten(models.bsm_args(dim, texture, s), None, pset, likelihood='FLAT'), th)
            worst = max(worst, np.abs(fr[0, j] - ref[0]).max())
            flags = _lib.ST_REFINED | _lib.ST_ILL_COND
            assert (st[0] & flags) == (rst[0] & flags), (i, st[0], rst[0])
        refined += bool(st[0] & _lib.ST_REFINED)
    assert refined > 20
    assert worst <= 1e-14, worst


@pytest.mark.parametrize('dim,texture', [(3, Texture.OET), (6, Texture.OUT)])
def test_harness_task_against_the_oracle(dim, texture):
    """The kernel's per-sample code run sequentially on 3000 draws: lnZ per (source, scale) against a NumPy log-sum-exp of
    truth.eigh_flux_averaged_fr + batch_multi_gaussian, 1e-10 relative."""
    fm = grid_model(dim, texture)
    scales = sens.scale_grid(dim, 12)[[0, 3, 6, 9, 11]]
    n = 3000
    lse = sh.evidence_sources(fm, scales, SOURCES, INJECTED, n, seed=26)
    got = lnz_of(lse[..., 0], lse[..., 1], n)
    theta = hh.draw(fm, 26, 0, n)
    ref = oracle_lnz(dim, texture, theta, scales, SOURCES, INJECTED)
    assert np.isfinite(ref).sum() >= ref.size // 2
    assert_lnz_close(got, ref, 1e-10, (dim, texture))


def test_limit_table_is_get_limit_row_by_row(golden):
    """limit_table == get_limit on every curve: the ref_limit.npz rows (as one source each) and synthetic curves that give a
    limit, None and 'Discovered LV!'; NaN exactly where there is no limit, discovered exactly where get_limit raises; both
    statistics' thresholds."""
    g = golden('ref_limit.npz')
    by_len = {}
    for k in range(int(g['n'])):
        by_len.setdefault((len(g['scales_%d' % k]), bool(g['mask_%d' % k])), []).append(k)
    for (_, mi), ks in by_len.items():
        ev = {0: np.stack([np.column_stack([g['scales_%d' % k], g['stat_%d' % k]]) for k in ks])}
        for kw in (dict(), dict(args=Namespace(stat_method=StatCateg.FREQUENTIST)), dict(args=Namespace(stat_method=StatCateg.BAYESIAN))):
            lim, disc = sens.limit_table(ev, mask_initial=mi, **kw)
            assert lim.shape == disc.shape == (1, len(ks))
            for j, k in enumerate(ks):
                try:
                    ref = sens.get_limit(g['scales_%d' % k], g['stat_%d' % k], mask_initial=mi, **kw)
                except AssertionError as e:
                    assert str(e) == 'Discovered LV!'
                    assert disc[0, j] and np.isnan(lim[0, j])
                    continue
                assert not disc[0, j]
                assert (np.isnan(lim[0, j]) if ref is None else lim[0, j] == ref), (k, lim[0, j], ref)
    # synthetic curves over two "dimensions": a limit, a flat curve (None) and, with a negative threshold (the only way the
    # null point, part of the maximum, can be disfavoured), 'Discovered LV!'
    sc = np.concatenate([[-100.], np.linspace(-60, -20, 41)])
    curves = np.stack([np.column_stack([sc, -np.maximum(sc + 40.0, 0.0) * 3]), np.column_stack([sc, np.zeros_like(sc)]),
                       np.column_stack([sc, np.where(sc < -90, -10.0, 0.0)])])
    seen = set()
    for kw in (dict(), dict(bayes_k=-1.0), dict(args=Namespace(stat_method=StatCateg.FREQUENTIST))):
        ev = {3: curves, 6: curves[::-1]}
        lim, disc = sens.limit_table(ev, **kw)
        for i, d in enumerate(ev):
            for j, c in enumerate(ev[d]):
                try:
                    ref = sens.get_limit(c[:, 0], c[:, 1], **kw)
                except AssertionError:
                    assert disc[i, j] and np.isnan(lim[i, j])
                    seen.add('discovered')
                    continue
                assert not disc[i, j]
                assert (np.isnan(lim[i, j]) if ref is None else lim[i, j] == ref)
                seen.add('none' if ref is None else 'limit')
    assert seen == {'discovered', 'none', 'limit'}
    with pytest.raises(ValueError, match='numbers of sources'):
        sens.limit_table({3: curves, 6: curves[:2]})


def test_abi_and_build():
    assert 'gf_sources.cu' in build.SOURCES and 'gf_sources_dev.cuh' in build.HEADERS
    build.build_library()
    lib = _lib.load()
    for name in ('gf_scan_evidence_sources', 'gf_scan_evidence_sources_workspace'):
        assert name in _lib.EXPORTS and hasattr(lib, name)
    header = open(os.path.join(ROOT, 'include', 'golemflavor_b200.h')).read()
    assert re.search(r'nsrc outside \[1, GF_SRC_MAX = %d\]' % _lib.GF_SRC_MAX, header)
    assert _lib.GF_SRC_MAX >= 64
    assert {'scan_evidence_sources'} <= set(scan.__all__) and {'evidence_source_grid', 'limit_table'} <= set(sens.__all__)


def test_python_argument_checks_need_no_device():
    good, inj = SOURCES, (1, 1, 1)
    src, i = scan.source_rows((1, 2, 0), inj)
    assert src.shape == i.shape == (1, 3)
    src, i = scan.source_rows(good, INJECTED)
    assert src.shape == i.shape == (5, 3)
    for bad_src, bad_inj, msg in (
            (np.ones((2, 4)), inj, 'sources must be'),
            (np.ones((2, 2, 3)), inj, 'sources must be'),
            (np.zeros((0, 3)), inj, 'sources must be'),
            (good, np.ones((3, 3)), 'injected must be'),
            (good, np.ones(4), 'injected must be'),
            ([(1, -1e-9, 1)], inj, 'source 0'),
            ([(1, 1, 1), (0, 0, 0)], inj, 'source 1'),
            ([(1, np.nan, 1)], inj, 'source 0'),
            ([(1, np.inf, 1)], inj, 'source 0'),
            (good, (0, 0, 0), 'injected composition 0'),
            (good, (1, -1, 1), 'injected composition 0')):
        with pytest.raises(ValueError, match=msg):
            scan.scan_evidence_sources(None, [-40.0], bad_src, bad_inj, 10)
        with pytest.raises(ValueError, match=msg):
            sens.evidence_source_grid(bad_src, dimensions=(3,), segments=4, injected_ratio=bad_inj, samples=10)


# ------------------------------------------------------------------ GPU


@pytest.fixture(scope='module')
def torch():
    t = pytest.importorskip('torch')
    if not t.cuda.is_available():
        pytest.skip('needs a CUDA device')
    return t


@pytest.mark.gpu
@pytest.mark.parametrize('texture', [Texture.OET, Texture.OUT])
def test_device_against_the_evidence_grid_per_source(torch, texture):
    """evidence_source_grid row j == evidence_grid(source_ratio=s_j, injected_ratio=inj_j): same samples, same layout,
    |dlnZ| <= 1e-12 max(1, |lnZ|); shared and per-source injected compositions, unnormalised inputs."""
    kw = dict(dimensions=(3, 6), segments=20, texture=texture, samples=200_000, seed=26)
    for inj in ((1, 1, 1), INJECTED):
        ev = sens.evidence_source_grid(SOURCES, injected_ratio=inj, **kw)
        assert sorted(ev) == [3, 6]
        injs = np.broadcast_to(np.asarray(inj, dtype=np.float64), SOURCES.shape)
        for j, (s, i) in enumerate(zip(SOURCES, injs)):
            ref = sens.evidence_grid(source_ratio=s, injected_ratio=i, **kw)
            for d in (3, 6):
                assert ev[d].shape == (len(SOURCES), 20, 2)
                assert np.array_equal(ev[d][j][:, 0], ref[d][:, 0])
                assert_lnz_close(ev[d][j][:, 1], ref[d][:, 1], 1e-12, (texture, d, j, inj is INJECTED))
        assert np.isfinite(ev[3][:, :, 1]).any()


@pytest.mark.gpu
def test_device_against_the_oracle(torch):
    """<= 5000 samples: the drawn theta of scan_samples -> per-source truth fr -> host log-sum-exp, 1e-10 relative."""
    for dim, texture in ((3, Texture.OET), (6, Texture.OUT)):
        fm = grid_model(dim, texture)
        scales = sens.scale_grid(dim, 12)[[0, 2, 5, 8, 11]]
        n = 4000
        got = scan.scan_evidence_sources(fm, scales, SOURCES, INJECTED, n, seed=31)
        theta, _, _ = scan.scan_samples(fm, n, seed=31)
        ref = oracle_lnz(dim, texture, theta, scales, SOURCES, INJECTED)
        assert np.isfinite(ref).sum() >= ref.size // 2
        assert_lnz_close(got, ref, 1e-10, (dim, texture))


@pytest.mark.gpu
def test_device_determinism_and_structure(torch):
    fm = grid_model(6)
    scales = sens.scale_grid(6, 37)
    n = 300_001
    rng = np.random.default_rng(11)
    src = np.concatenate([SOURCES, rng.uniform(size=(25, 3))])             # 30 sources: several slots per thread
    inj = np.concatenate([INJECTED, rng.uniform(0.1, 1, size=(25, 3))])
    a = scan.scan_evidence_sources(fm, scales, src, inj, n)
    assert a.shape == (30, 37) and np.isfinite(a).any()
    b = scan.scan_evidence_sources(fm, scales, src, inj, n)
    assert np.array_equal(a, b)                                           # a repeated launch is bit-identical
    rep = scan.scan_evidence_sources(fm, scales, np.concatenate([src, src[3:4]]), np.concatenate([inj, inj[3:4]]), n)
    assert np.array_equal(rep[30], rep[3])                                # a repeated source: the same row
    perm = rng.permutation(30)
    p = scan.scan_evidence_sources(fm, scales, src[perm], inj[perm], n)
    assert np.array_equal(p, a[perm])                                     # permuted sources: permuted rows
    split = np.concatenate([scan.scan_evidence_sources(fm, scales, src[:7], inj[:7], n),
                            scan.scan_evidence_sources(fm, scales, src[7:], inj[7:], n)])
    assert_lnz_close(split, a, 1e-12, 'split over launches')
    one = scan.scan_evidence_sources(fm, scales, src[4], inj[4], n)       # one source: several threads per pair
    assert_lnz_close(one[0], a[4], 1e-12, 'one source')
    n1 = 123_457                                                          # two sample shards merged on the host
    z1 = scan.scan_evidence_sources(fm, scales, src, inj, n1)
    z2 = scan.scan_evidence_sources(fm, scales, src, inj, n - n1, first_index=n1)
    merged = np.logaddexp(z1 + np.log(n1), z2 + np.log(n - n1)) - np.log(n)
    assert_lnz_close(merged, a, 1e-12, 'sample shards')
    many = np.concatenate([src] * 9)                                      # 270 sources: two launches of at most 256
    m = scan.scan_evidence_sources(fm, scales[:4], many, np.concatenate([inj] * 9), 20_000)
    ref = scan.scan_evidence_sources(fm, scales[:4], src, inj, 20_000)
    assert_lnz_close(m, np.concatenate([ref] * 9), 1e-12, 'more sources than one launch takes')
    ev = sens.evidence_grid(dimensions=(6,), segments=37, source_ratio=src[5], injected_ratio=inj[5], samples=n)
    assert_lnz_close(a[5], ev[6][:, 1], 1e-12, 'evidence grid')


@pytest.mark.gpu
def test_device_refusals(torch):
    """Every refusal of gf_scan_evidence_sources: GF_ERR_ARG, a message in gf_last_error(), nothing launched and d_lse
    untouched."""
    lib = _lib.load()
    fm = grid_model(6)
    sc = torch.as_tensor(sens.scale_grid(6, 5)).cuda()
    lse = torch.full((2, 5, 2), 7.0, dtype=torch.float64, device='cuda')
    nbytes = int(lib.gf_scan_evidence_sources_workspace(5, 2))
    assert nbytes > 0
    assert lib.gf_scan_evidence_sources_workspace(0, 2) == 0 and lib.gf_scan_evidence_sources_workspace(5, _lib.GF_SRC_MAX + 1) == 0
    work = torch.empty(nbytes, dtype=torch.uint8, device='cuda')
    cfg = _lib.ScanConfig(seed=26, first_index=0, count=1000, nb=0)
    src = np.ascontiguousarray(SOURCES[:2])
    inj = np.ascontiguousarray(INJECTED[:2])
    P = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    stream = _lib.stream_ptr(torch)

    def call(model=fm.ref, cfg_=cfg, scales=_lib.ptr(sc), ns=5, s=src, i=inj, nsrc=2, out=_lib.ptr(lse), w=_lib.ptr(work), wb=nbytes):
        return lib.gf_scan_evidence_sources(model, C.byref(cfg_) if cfg_ is not None else None, scales, ns,
                                            P(s) if s is not None else None, P(i) if i is not None else None, nsrc, out, w, wb, stream)

    def refused(msg, **kw):
        before = lib.gf_launch_count()
        assert call(**kw) == _lib.GF_ERR_ARG, msg
        assert re.search(msg, lib.gf_last_error().decode()), (msg, lib.gf_last_error())
        assert lib.gf_launch_count() == before

    refused('null pointer', model=None)
    refused('null pointer', cfg_=None)
    refused('null pointer', scales=None)
    refused('null pointer', s=None)
    refused('null pointer', i=None)
    refused('null pointer', out=None)
    refused(r'nscales = 0 outside \[1, 65535\]', ns=0)
    refused(r'nscales = 65536 outside', ns=65536)
    refused(r'nsrc = 0 outside \[1, %d\]' % _lib.GF_SRC_MAX, nsrc=0)
    refused(r'nsrc = %d outside' % (_lib.GF_SRC_MAX + 1), nsrc=_lib.GF_SRC_MAX + 1)
    refused('no BSM path', model=scan.scan_model('unitary').ref)
    args, asimov, pset = models.bsm_model_c3([0.5, 0.5], dim=6)
    refused('sampled column', model=model.flatten(args, asimov, pset).ref)
    args, asimov, pset = models.bsm_sampled_source([0.5, 0.5], kind='angles')
    pset = ParamSet([p for p in pset if p.name != 'logLam'])
    args.fixed_scale = -40.0
    refused('samples the source', model=model.flatten(args, asimov, pset).ref)
    flat_args = Namespace(source_ratio=np.array([1., 2., 0.]) / 3, dimension=6, texture=Texture.OET, binning=scan.DEFAULT_BINNING, no_bsm=False,
                          fixed_scale=-100.0)
    flat = model.flatten(flat_args, None, ParamSet(scan.sm_paramset(with_mass=True)), likelihood='FLAT')
    refused('Gaussian likelihood', model=flat.ref)
    for bad in ([(1, -1, 0), (1, 1, 1)], [(1, 1, 1), (0, 0, 0)], [(np.nan, 1, 1), (1, 1, 1)], [(1, np.inf, 1), (1, 1, 1)]):
        refused('source', s=np.ascontiguousarray(bad, dtype=np.float64))
        refused('injected', i=np.ascontiguousarray(bad, dtype=np.float64))
    refused('workspace of 0 B is too small', w=None, wb=0)
    refused('too small', wb=16)
    assert torch.equal(lse, torch.full_like(lse, 7.0))
    # count = 0 is a no-op; a valid call then runs
    cfg0 = _lib.ScanConfig(seed=26, first_index=0, count=0, nb=0)
    assert call(cfg_=cfg0) == _lib.GF_OK
    torch.cuda.synchronize()
    assert torch.equal(lse, torch.full_like(lse, 7.0))
    lse.fill_(0.0)
    lse[..., 0] = -np.inf
    assert call() == _lib.GF_OK
    torch.cuda.synchronize()
    assert torch.isfinite(lse[..., 0]).any()


@pytest.mark.gpu
def test_multi_gpu_nccl_source_grid_is_rank_count_invariant(torch):
    """tests/dist_source_check.py under torchrun on every GPU of the box (NCCL): the sharded source grid against one rank
    alone.  Needs >= 2 GPUs."""
    import subprocess
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip('needs at least two GPUs')
    res = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr', '127.0.0.1',
                          '--master-port', '29733', os.path.join(HERE, 'dist_source_check.py')], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:]
    assert 'ok=True' in res.stdout


@pytest.mark.gpu
def test_limit_table_end_to_end(torch):
    """limit_table(evidence_source_grid(...)) == limits(evidence_grid(...)) source by source: dims 3 and 6, 20 segments,
    5e4 samples, five sources including (1, 2, 0)."""
    kw = dict(dimensions=(3, 6), segments=20, samples=50_000)
    ev = sens.evidence_source_grid(SOURCES, injected_ratio=(1, 1, 1), **kw)
    lim, disc = sens.limit_table(ev)
    assert lim.shape == disc.shape == (2, len(SOURCES))
    for j, s in enumerate(SOURCES):
        ref = sens.evidence_grid(source_ratio=s, injected_ratio=(1, 1, 1), **kw)
        for i, d in enumerate((3, 6)):
            try:
                r = sens.get_limit(ref[d][:, 0], ref[d][:, 1])
            except AssertionError:
                assert disc[i, j] and np.isnan(lim[i, j])
                continue
            assert not disc[i, j]
            if r is None:
                assert np.isnan(lim[i, j])
            else:
                assert abs(lim[i, j] - r) < 1e-9, (d, j, lim[i, j], r)
    assert np.isfinite(lim).any()
