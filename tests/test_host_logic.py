"""CPU-side tests (no GPU): the C-ABI library loads and exports every declared symbol, the host
logic (ParamSet flattening, argument checking, sharding) behaves like the reference, and the
kernels' per-point arithmetic -- instantiated on the host by tests/host_harness -- agrees with
the golden fixtures / the oracle.  The GPU parity tests proper are in test_gpu_*.py."""

import argparse
import ctypes as C
import os
import re

import numpy as np
import pytest

from golemflavor_b200 import _lib, build, enums, llh, mcmc, model, scan
from golemflavor_b200.enums import ParamTag, PriorsCateg, Texture
from golemflavor_b200.param import Param, ParamSet
from oracle import golem_oracle as go
from oracle import truth

import host_harness as hh
import models

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ library / ABI
def test_library_builds_and_exports_every_declared_symbol():
    build.build_library()
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'golemflavor_b200.h')).read()
    declared = set(re.findall(r'^\s*(?:int|uint64_t|const char\*)\s+(gf_\w+)\s*\(', header, flags=re.M))
    assert declared, 'no prototypes found in the header'
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.gf_abi_version() == 1
    assert lib.gf_sizeof(0) == C.sizeof(_lib.Model)


def test_torch_ops_library_builds_and_registers_every_operator():
    """The `torch.ops.golemflavor.*` registration of the C ABI (csrc/gf_torch_ops.cpp) builds in-tree, loads and
    defines every operator `_lib.TORCH_OPS` names (no compute call without a GPU)."""
    import torch
    path = build.build_torch_ops()
    assert os.path.exists(path) and path == _lib.TORCH_OPS_PATH
    ops = _lib.torch_ops()
    assert int(ops.abi_version()) == 1
    for name in _lib.TORCH_OPS:
        assert hasattr(ops, name), name
    schema = str(torch.ops.golemflavor.lnprob.default._schema)
    assert 'Tensor theta' in schema and 'bool want_fr' in schema
    # argument validation happens before any CUDA call: a CPU theta is refused
    fm = model.physics_model(ndim=1)
    with pytest.raises(RuntimeError):
        ops.lnprob(torch.zeros((2, 1), dtype=torch.float64), model.FlatModel(fm).blob, False, False)


def test_no_oracle_or_cpu_fallback_in_product():
    """The product package must not import the oracle or the host harness."""
    pkg = os.path.join(ROOT, 'golemflavor_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            src = open(os.path.join(pkg, fn)).read()
            assert 'oracle' not in src.replace('golem_oracle', 'oracle') or fn == '__none__', fn
            assert 'host_harness' not in src, fn


def test_compute_without_gpu_raises():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from golemflavor_b200 import fr
    with pytest.raises(_lib.GolemFlavorError):
        fr.angles_to_u((0.2, 0.3, 0.5, 1.5))
    with pytest.raises(_lib.GolemFlavorError):
        llh.multi_gaussian([.3, .35, .35], [.55, .18, .27], .02)


def test_model_check_rejects_bad_models():
    m = model._new_struct()
    m.ndim = 0
    with pytest.raises(ValueError):
        model.FlatModel(m)
    m = model._new_struct()
    m.ndim = 2
    m.prior[0].lo, m.prior[0].hi = 1.0, 0.0
    with pytest.raises(ValueError):
        model.FlatModel(m)
    m = model._new_struct()
    m.ndim = 3
    m.col_scale = 5
    with pytest.raises(ValueError):
        model.FlatModel(m)
    m = model._new_struct()
    m.ndim = 1
    m.prior[0].lo, m.prior[0].hi, m.prior[0].kind, m.prior[0].sigma = 0., 1., _lib.PRIOR_GAUSSIAN, 0.0
    with pytest.raises(ValueError):
        model.FlatModel(m)
    m = model._new_struct()
    m.ndim, m.no_bsm, m.nbins, m.dimension = 1, 0, 20, 9
    with pytest.raises(ValueError):
        model.FlatModel(m)


# ------------------------------------------------------------------ host containers
def test_paramset_mirrors_reference_api():
    ps = ParamSet([Param('a', 1., [0, 2], tag=ParamTag.SCALE, std=0.1),
                   Param('b', 2., [0, 3], seed=[1, 2], prior=PriorsCateg.GAUSSIAN, std=0.5)])
    assert ps.names == ('a', 'b') and ps.values == (1., 2.) and ps.ranges == ((0, 2), (0, 3))
    assert ps.seeds == ((0, 2), (1, 2)) and ps.stds == (0.1, 0.5)
    assert ps['b'].prior is PriorsCateg.GAUSSIAN and ps[0].prior is PriorsCateg.UNIFORM
    assert ps.from_tag(ParamTag.SCALE, values=True) == (1.,)
    assert ps.from_tag(ParamTag.SCALE, index=True, invert=True) == (1,)
    assert len(ps.from_tag([ParamTag.SCALE, ParamTag.NONE])) == 2
    assert ps[1].tag is ParamTag.NONE and ps[1].nominal_value == 2.
    with pytest.raises(ValueError):
        ParamSet([Param('a', 1., [0, 2]), Param('a', 1., [0, 2])])
    assert len(ps.extend(Param('c', 0., [0, 1]))) == 3
    assert ps.remove_params(ParamSet([ps[0]])).names == ('b',)
    assert enums.Texture.OET.value == 2 and enums.ParamTag.BESTFIT.value == 6  # enums.py:28-63


def test_flatten_resolves_columns_like_the_reference(golden):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    s = fm.struct
    assert s.ndim == 6 and s.no_bsm == 1 and list(s.col_sm) == [0, 1, 2, 3] and list(s.col_src) == [4, 5]
    assert [s.prior[k].kind for k in range(6)] == [2, 2, 2, 0, 0, 0]
    assert np.allclose(list(s.fr_bf), go.angles_to_fr(g['asimov_angles']), atol=1e-15) and s.smearing == 0.02
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'])
    s = model.flatten(args, asimov, pset).struct
    assert s.no_bsm == 0 and s.col_scale == 6 and list(s.col_mass) == [4, 5] and s.nbins == 20 and s.dimension == 6
    assert np.allclose(list(s.fixed_np), model.TEXTURE_ANGLES['OET']) and list(s.col_np) == [-1] * 4
    assert [s.prior[k].kind for k in range(7)] == [2, 2, 2, 0, 1, 1, 0]
    # only four of the six SM names present -> NuFIT defaults on the BSM path (fr.py:425-435)
    pset4 = ParamSet(scan.sm_paramset(with_mass=False) + [pset['logLam']])
    s = model.flatten(args, asimov, pset4).struct
    assert list(s.col_sm) == [-1] * 4 and list(s.col_mass) == [-1, -1] and s.col_scale == 4
    # Texture.NONE needs the four MMANGLES
    s = model.flatten(models.bsm_args(texture=Texture.NONE), asimov, models.bsm11_paramset()).struct
    assert list(s.col_np) == [6, 7, 8, 9] and s.col_scale == 10
    with pytest.raises(ValueError):
        model.flatten(models.bsm_args(texture=Texture.NONE), asimov, pset)
    with pytest.raises(ValueError):
        model.flatten(argparse.Namespace(likelihood=enums.Likelihood.GOLEMFIT, source_ratio=[1, 2, 0]), asimov, pset)
    assert np.allclose(model.binning_edges([6e4, 1e7, 20]), models.BINNING)


def test_length_mismatch_raises_assertion_like_reference(golden):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    with pytest.raises(AssertionError):
        llh.lnprior([0.1, 0.2], pset)          # llh.py:67-71
    with pytest.raises(AssertionError):
        llh.ln_prob([0.1] * 5, args, asimov, pset)
    with pytest.raises(AssertionError):
        llh.triangle_llh([0.1] * 7, args, asimov, pset)


def test_shard_range_partitions_exactly():
    for count in (0, 1, 7, 10 ** 10 + 3):
        for world in (1, 2, 3, 8):
            parts = [scan.shard_range(count, r, world, first_index=5) for r in range(world)]
            assert parts[0][0] == 5 and sum(n for _, n in parts) == count
            for (a, n), (b, _) in zip(parts, parts[1:]):
                assert a + n == b
            assert max(n for _, n in parts) - min(n for _, n in parts) <= 1


def test_ensemble_sampler_recovers_gaussian():
    rng = np.random.RandomState(5)
    mu, sig = np.array([1.0, -2.0, 0.5]), np.array([0.5, 2.0, 1.0])
    calls = []

    def lnp(t):
        calls.append(t.shape)
        return -0.5 * np.sum(((t - mu) / sig) ** 2, axis=-1)
    s = mcmc.EnsembleSampler(40, 3, lnp, seed=11)
    pos = None
    for pos, lp, _ in s.sample(mu + rng.randn(40, 3), iterations=300):
        pass
    s.reset()
    for _ in s.sample(pos, iterations=1500):
        pass
    assert s.chain.shape == (40, 1500, 3) and s.lnprobability.shape == (40, 1500)
    flat = s.chain.reshape(-1, 3)   # walker-major, mcmc.py:44
    assert np.allclose(flat.mean(0), mu, atol=0.15) and np.allclose(flat.std(0), sig, rtol=0.1)
    assert 0.4 < s.acceptance_fraction.mean() < 0.8 and s.acor.shape == (3,)
    # one vectorised call per half-ensemble (+ one full-ensemble call at the start of each sample())
    assert calls.count((40, 3)) == 2 and calls.count((20, 3)) == 2 * 1800 and len(calls) == 3602
    with pytest.raises(ValueError):
        mcmc.EnsembleSampler(5, 3, lnp)
    bad = mcmc.EnsembleSampler(8, 2, lambda t: np.full(len(t), np.nan))
    with pytest.raises(ValueError):
        next(bad.sample(np.zeros((8, 2)), iterations=1))


def test_seeds_and_save_chains(tmp_path):
    pset = models.bsm7_paramset()
    np.random.seed(3)
    p0 = mcmc.flat_seed(pset, 32)
    box = np.array(pset.seeds)
    assert p0.shape == (32, 7) and np.all(p0 >= box[:, 0]) and np.all(p0 <= box[:, 1])
    assert mcmc.gaussian_seed(pset, 8).shape == (8, 7)
    out = str(tmp_path / 'sub' / 'chain')
    mcmc.save_chains(p0, out)
    assert np.array_equal(np.load(out + '.npy'), p0)


# ------------------------------------------------------------------ kernel arithmetic on the host harness
def test_harness_notebook_lnprob_matches_reference_fixture(golden):
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    lnp, fr, st = hh.lnprob(fm, g['theta'])
    ref = g['lnprob']
    inside = np.isfinite(g['lnprior'])
    assert np.array_equal(np.isneginf(lnp[~inside]), np.ones((~inside).sum(), bool))
    assert np.all((st[~inside] & _lib.ST_OUT_OF_PRIOR) != 0) and np.all(st[inside] == 0)
    assert np.abs(fr[inside] - g['fr'][inside]).max() < 1e-12
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp), fin)          # incl. the pdf-underflow -> -inf emulation
    assert np.max(np.abs(lnp[fin] - ref[fin]) / np.abs(ref[fin])) < 1e-10
    assert abs(lnp[0] - (-458.6843569885842)) < 1e-9 * 458   # SURVEY 8c spot value


def test_harness_lnprior_matches_scipy_fixture(golden):
    g = golden('ref_llh.npz')
    fm = model.flatten(argparse.Namespace(source_ratio=[1, 2, 0], dimension=6, texture=Texture.OET,
                                          binning=models.BINNING, no_bsm=False), None, models.bsm7_paramset(),
                       likelihood='FLAT')
    got = hh.lnprior(fm, g['theta7'])
    ref = g['lnprior7']
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin)
    assert np.max(np.abs(got[fin] - ref[fin]) / np.abs(ref[fin])) < 1e-12


def test_harness_flux_averaged_fr_matches_reference_and_mpmath(golden):
    g = golden('ref_flux.npz')
    worst_mp, worst_ref = 0.0, 0.0
    for tex in ('OET', 'OUT', 'OEU', 'NONE'):
        for dim in (3, 6):
            for src in ((1, 2, 0), (1, 0, 0), (0, 1, 0)):
                sel = (g['tex'] == tex) & (g['dim'] == dim) & np.all(g['src'] == np.array(src, float), axis=1)
                if not sel.any():
                    continue
                fm = model.flatten(models.bsm_args(dim, Texture.NONE, src), None, models.bsm11_paramset(dim), likelihood='FLAT')
                fr, st = hh.fr(fm, g['theta'][sel])
                assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
                worst_mp = max(worst_mp, np.abs(fr - g['fr_mp'][sel]).max())
                ok = g['ok'][sel]   # points where the reference passed its own unitarity assertion
                # the reference's own error vs mpmath on those points bounds what can be asked of parity
                ref_err = np.abs(g['fr'][sel][ok] - g['fr_mp'][sel][ok]).max(axis=1)
                good = ref_err < 1e-11
                worst_ref = max(worst_ref, np.abs(fr[ok][good] - g['fr'][sel][ok][good]).max())
                if tex != 'NONE':  # same answer through the fixed-texture (constant T) path
                    fm7 = model.flatten(models.bsm_args(dim, Texture[tex], src), None, models.bsm7_paramset(dim), likelihood='FLAT')
                    th7 = np.delete(g['theta'][sel], [6, 7, 8, 9], axis=1)
                    fr7, _ = hh.fr(fm7, th7)            # FIXED specialisation (texture + source in constants)
                    fr7g, _ = hh.fr(fm7, th7, spec=0)   # same model through the generic path
                    assert np.abs(fr7 - fr).max() < 1e-13 and np.abs(fr7g - fr7).max() < 1e-13
    assert worst_mp < 1e-10, worst_mp     # vs mpmath truth, everywhere (abs. error on a unit-sum composition)
    assert worst_ref < 1e-10, worst_ref   # vs the reference where the reference itself is accurate


def test_harness_eigen_stage_against_lapack_on_random_bsm_points():
    rng = np.random.default_rng(7)
    n = 4000
    worst = 0.0
    nfast = 0
    for texname in ('OET', 'OUT', 'OEU', 'NONE'):
        for dim in (3, 5, 6, 8):
            pset = models.bsm11_paramset(dim)
            th = models.draw_in_ranges(pset, n, rng, seeds=True)
            lo, hi = model.SCALE_BOUNDARIES[dim]
            th[:, 10] = rng.uniform(lo, hi, n)
            if texname == 'NONE':
                th[:, 6:9] = rng.uniform(0, 1, (n, 3))
                th[:, 9] = rng.uniform(0, 2 * np.pi, n)
            else:
                th[:, 6:10] = model.TEXTURE_ANGLES[texname]
            fm = model.flatten(models.bsm_args(dim, Texture.NONE), None, pset, likelihood='FLAT')
            fr, st = hh.fr(fm, th)
            ref = truth.eigh_flux_averaged_fr(th[:, :4], th[:, 4:6], th[:, 6:10], th[:, 10], dim, models.BINNING,
                                              np.array([1, 2, 0.]) / 3)
            assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY))
            err = np.abs(fr - ref).max(axis=1)
            worst = max(worst, err.max())
            nfast += np.count_nonzero((st & _lib.ST_REFINED) == 0)
    assert worst < 1e-10, worst
    assert nfast > 0.5 * 16 * n   # the closed-form path must carry the bulk of the points


def test_harness_deflation_refinement_on_near_degenerate_pairs():
    """gfp_herm3_x4_deflate (the fallback of the energy-bin loop) against mpmath on Hermitian matrices with
    a prescribed eigenvalue pair splitting from 1e-2 down to 1e-9 of the spectral scale: |V_ai|^2 to
    ~eps / gap (the conditioning of the eigenvectors themselves), at every matrix scale the pencil reaches."""
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(11)
    worst = {}
    for gap in (1e-2, 1e-4, 1e-6, 1e-9):
        hams, truth_x = [], []
        for trial in range(12):
            z = rng.normal(size=(3, 3)) + 1j * rng.normal(size=(3, 3))
            q, _ = np.linalg.qr(z)
            top = rng.choice([-1.0, 1.0])                      # isolated eigenvalue above or below the pair
            lam = np.array([top * 1.0, -0.5 * top + gap, -0.5 * top - gap]) * rng.uniform(0.3, 3.0) + rng.uniform(-2, 2)
            scale = 10.0 ** rng.uniform(-30, 30)
            h = (q * lam) @ q.conj().T * scale
            h = (h + h.conj().T) / 2
            hams.append(h)
            hm = mp.matrix(3, 3)
            for a in range(3):
                for b in range(3):
                    hm[a, b] = mp.mpc(float(h[a, b].real), float(h[a, b].imag)) if a != b else mp.mpf(float(h[a, a].real))
            ev, vec = mp.eighe(hm)
            ev = [float(e) for e in ev]
            iso = 0 if abs(ev[0] - ev[1]) > abs(ev[1] - ev[2]) else 2     # sorted ascending: the pair is adjacent
            upper = 2 if iso == 0 else 1
            truth_x.append([[float(abs(vec[a, iso]) ** 2), float(abs(vec[a, upper]) ** 2)] for a in range(2)])
        x, st = hh.deflate(np.array(hams))
        assert np.all(st & _lib.ST_REFINED) and not np.any(st & _lib.ST_NON_FINITE)
        worst[gap] = float(np.abs(x - np.array(truth_x)).max())
        assert worst[gap] < 4e-15 / gap + 1e-14, worst
        assert np.all(((st & _lib.ST_ILL_COND) != 0) == (gap < 1e-7))      # relative gap below 1e-6 is flagged
    # exactly degenerate pair: flagged, and the (arbitrary) split of the pair stays a valid one
    x, st = hh.deflate(np.diag([2.0, -1.0, -1.0]).astype(complex)[None])
    assert (st[0] & _lib.ST_ILL_COND) and np.allclose(x[0, 0], [1.0, 0.0], atol=1e-15) and abs(x[0, 1, 0]) < 1e-15 and 0.0 <= x[0, 1, 1] <= 1.0
    # zero / non-finite matrices hand over to Jacobi
    _, st = hh.deflate(np.zeros((1, 3, 3), dtype=complex))
    assert st[0] & _lib.ST_NON_FINITE


def test_harness_prior_draws_follow_philox_convention():
    fm = scan.scan_model('unitary')
    th = hh.draw(fm, 26, 12345, 1000)
    u = go.philox_uniforms(26, 12345, 1000, block=0)
    assert np.array_equal(th[:, :3], u[:, :3])                      # U(0,1) ranges: theta == uniform
    assert np.allclose(th[:, 3], 2 * np.pi * u[:, 3], rtol=1e-15)
    th2 = hh.draw(fm, 26, 12345 + 500, 500)
    assert np.array_equal(th2, th[500:])                            # counter = global index: shard-invariant
    big = hh.draw(fm, 26, (1 << 32) - 2, 4)                         # index crosses 2^32
    assert np.array_equal(big[:, :3], go.philox_uniforms(26, (1 << 32) - 2, 4)[:, :3])


def test_harness_histogram_is_bit_exact_np_histogramdd():
    rng = np.random.default_rng(3)
    fr = rng.dirichlet([1, 1, 1], 100000)
    fr[:300, 0] = np.arange(300) / 26.0
    fr[300:600, 1] = np.arange(300) * (1.0 / 26.0)
    fr[600:900, 2] = np.nextafter(np.arange(300) / 201.0, 0)
    fr[900:905] = [[1, 0, 0], [0, 1, 0], [0, 0, 1], [1.0000000001, 0, 0], [np.nan, 0.5, 0.5]]
    for nb in (0, 1, 25, 125, 200):
        assert np.array_equal(hh.hist(fr, nb), go.ternary_histogram(fr, nb)), nb


# ------------------------------------------------------------------ ensemble sampler update on the host harness
def test_harness_ensemble_update_is_the_numpy_stretch_move(golden):
    """The kernel's per-walker update (RNG convention, proposal, acceptance rule, in-place half-step
    semantics), replayed on the host, must reproduce an independent NumPy stretch-move sampler
    bit-for-bit when both score proposals with the same log-posterior."""
    import ref_sampler
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    rng = np.random.default_rng(0)
    k = 32
    p0 = models.draw_in_ranges(pset, k, rng, seeds=True)
    p0[:, 4], p0[:, 5] = rng.uniform(.9, 1, k), rng.uniform(.8, 1, k)
    l0 = hh.lnprob(fm, p0)[0]
    pos, lnp, chain, lch, nacc = hh.ensemble(fm, p0, l0, 150, k, seed=5)
    rp, rl, rchain, racc = ref_sampler.run(lambda q: hh.lnprob(fm, q)[0], p0, l0, 150, seed=5)
    assert np.array_equal(chain[0], rchain) and np.array_equal(nacc[0], racc) and np.array_equal(lnp[0], rl)
    assert 0.2 < nacc.mean() / 150 < 0.7
    assert np.array_equal(lch[0][:, -1], lnp[0])
    # continuing with step0 = 150 equals one 300-step run; thinning stores every other step
    pos2, lnp2, chain2, _, _ = hh.ensemble(fm, pos, lnp, 150, k, seed=5, step0=150)
    _, _, chain_all, _, _ = hh.ensemble(fm, p0, l0, 300, k, seed=5)
    assert np.array_equal(chain_all[0][:, 150:], chain2[0])
    _, _, thin, _, _ = hh.ensemble(fm, p0, l0, 300, k, seed=5, thin=2)
    assert np.array_equal(thin[0], chain_all[0][:, 1::2])
    # two chains in one call are independent and shard-invariant (chain0 offsets the RNG counter)
    q0 = np.stack([p0, p0[::-1]])
    lq = np.stack([l0, l0[::-1]])
    _, _, both, _, _ = hh.ensemble(fm, q0, lq, 40, k, nchains=2, seed=9)
    _, _, second, _, _ = hh.ensemble(fm, q0[1], lq[1], 40, k, nchains=1, seed=9, chain0=1)
    assert np.array_equal(both[1], second[0]) and not np.array_equal(both[0], both[1])


def test_harness_ensemble_frozen_column_and_posterior(golden):
    """BSM model with log10(Lambda) frozen (the sens sweep): the frozen column never moves and the
    free-dimension count enters the acceptance factor."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.bsm_model_c3(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    np.random.seed(3)
    k = 28
    p0 = mcmc.flat_seed(pset, k)
    p0[:, 6] = -40.0
    l0 = hh.lnprob(fm, p0)[0]
    pos, lnp, chain, _, nacc = hh.ensemble(fm, p0, l0, 60, k, nfree=6, seed=1)
    assert np.all(chain[0][:, :, 6] == -40.0) and nacc.sum() > 0
    assert np.allclose(hh.lnprob(fm, pos[0])[0], lnp[0], rtol=0, atol=0)
    assert lnp.mean() > l0.mean()    # the ensemble climbs towards the posterior bulk


def test_sens_grid_matches_reference_definition():
    from golemflavor_b200 import sens
    g = sens.scale_grid(6, 10)       # sens.py:199-201
    assert g[0] == -100 and len(g) == 10 and np.allclose(g[1:], np.linspace(-56, -30, 9))
    ps = sens.sweep_paramset(3)
    assert ps.names[-1] == 'logLam' and ps['logLam'].ranges[0] < -100


def test_harness_config1_three_source_ratios_fixed_pmns(golden):
    """BASELINE config 1 (the CPU-runnable case): 3 raw source ratios, fixed NuFIT PMNS."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.sm_fit_c1(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    assert list(fm.struct.col_src3) == [0, 1, 2] and list(fm.struct.col_sm) == [-1] * 4 and fm.struct.no_bsm == 1
    rng = np.random.default_rng(1)
    theta = rng.uniform(0.01, 1, (500, 3))
    lnp, fr, st = hh.lnprob(fm, theta)
    ref_fr = np.array([np.asarray(go.u_to_fr(t, go.NUFIT_U), dtype=float) for t in theta])
    assert np.abs(fr - ref_fr).max() < 1e-14
    ref = go.batch_multi_gaussian(ref_fr, go.angles_to_fr(g['asimov_angles']), 0.02)
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(lnp), fin) and np.max(np.abs(lnp[fin] - ref[fin]) / np.abs(ref[fin])) < 1e-10
    # scale invariance of the raw ratios
    assert np.abs(hh.lnprob(fm, theta * 0.5)[1] - fr).max() < 1e-15


def _sampled_source_cases(g):
    """(kind, texture, dim, theta rows in the product's column order, reference fr, reference llh) per group of ref_src.npz."""
    for kind in ('angles', 'x', 'ratios'):
        nsrc = models.SOURCE_KINDS[kind]
        for tex, dim in (('OET', 6), ('OUT', 6), ('OEU', 3), ('OET', 8)):
            sel = (g['sb_kind'] == kind) & (g['sb_tex'] == tex) & (g['sb_dim'] == dim)
            theta = np.column_stack([g['sb_sm'][sel], g['sb_src'][sel][:, :nsrc], g['sb_loglam'][sel]])
            yield kind, tex, dim, theta, g['sb_fr'][sel], g['sb_llh'][sel]


def test_harness_sampled_source_models_match_reference_fixture(golden):
    """The GENERIC specialisation with a sampled source (two angles / x / three raw ratios) on the binned
    BSM path and BASELINE config 1, against fixtures from the unmodified reference (make_golden_r2.py)."""
    g, gl = golden('ref_src.npz'), golden('ref_llh.npz')
    args, asimov, pset = models.sm_fit_c1(gl['asimov_angles'])
    lnp, fr, st = hh.lnprob(model.flatten(args, asimov, pset), g['c1_theta'])
    fin = np.isfinite(g['c1_lnprob'])
    assert np.array_equal(np.isfinite(lnp), fin)
    assert np.abs(fr[fin] - g['c1_fr'][fin]).max() < 1e-14
    assert np.max(np.abs(lnp[fin] - g['c1_lnprob'][fin]) / np.abs(g['c1_lnprob'][fin])) < 1e-10
    for kind, tex, dim, theta, ref_fr, ref_llh in _sampled_source_cases(g):
        for first in (False, True):
            args, asimov, ps = models.bsm_sampled_source(gl['asimov_angles'], kind, dim, Texture[tex], source_first=first)
            fm = model.flatten(args, asimov, ps)
            assert model_spec_name(fm) == 'GENERIC'
            nsrc = models.SOURCE_KINDS[kind]
            th = np.column_stack([theta[:, 6:6 + nsrc], theta[:, :6], theta[:, -1:]]) if first else theta
            lnp, fr, st = hh.lnprob(fm, th)
            assert not np.any(st & (_lib.ST_NON_FINITE | _lib.ST_NON_UNITARY | _lib.ST_OUT_OF_PRIOR))
            # the reference's float128 Cardano is itself only good to ~1e-11 on part of these points (SURVEY 7.1)
            assert np.abs(fr - ref_fr).max() < 1e-10, (kind, tex, dim)
            lo, hi = np.array(ps.ranges).T
            kinds = [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in ps]
            lp = go.batch_lnprior(th, lo, hi, kinds, list(ps.nominal_values), [p.std or 1.0 for p in ps])
            ref = lp + ref_llh
            fin = np.isfinite(ref)
            assert np.array_equal(np.isfinite(lnp), fin)
            d = np.linalg.norm(ref_fr[fin] - g['bf'], axis=1)
            assert np.all(np.abs(lnp[fin] - ref[fin]) <= np.maximum(1e-10 * np.abs(ref[fin]), 2e-10 * d / 0.02 ** 2))


def model_spec_name(fm):
    s = fm.struct
    fixed_source = s.col_src[0] < 0 and s.col_x < 0 and s.col_src3[0] < 0
    if s.no_bsm:
        return 'SM'
    return 'GENERIC' if not fixed_source else 'NPFREE' if any(c >= 0 for c in s.col_np) else 'FIXED'


def test_cli_identifiers_match_reference_naming():
    from argparse import Namespace
    from golemflavor_b200 import cli
    assert cli.solve_ratio([1 / 3, 2 / 3, 0]) == '1_2_0' and cli.solve_ratio([1, 0, 0]) == '1_0_0'   # misc.py:34-41
    assert cli.solve_ratio([0.3, 0.3, 0.4]) == '0.30_0.30_0.40'
    a = Namespace(dimension=6, source_ratio=[1, 2, 0], injected_ratio=[1, 1, 1], texture=Texture.OET)
    assert cli.gen_identifier(a, 'fr') == '_DIM6_sfr_1_2_0_mfr_1_1_1_OET'                              # misc.py:44-51
    assert cli.gen_identifier(a, 'mc_texture') == '_DIM6_SRC_1_2_0_OET' and cli.gen_identifier(a, 'mc_unitary') == '_SRC_1_2_0'
    ns = cli._parser().parse_args(['mc_texture', '--dimension', '6', '--texture', 'out', '--nwalkers', '10'])
    assert ns.texture is Texture.OUT and ns.nwalkers == 10 and ns.binning == [6e4, 1e7, 20]


def test_harness_cubic_root_seeded_newton_is_full_precision():
    """w = 1 - cos(acos(1 - delta)/3) from the fp32-seeded Newton iteration: RELATIVE error below 2e-13
    over the whole range with the single fp64 step the kernels take (a few ulp with
    GFP_CUBIC_NEWTON_STEPS=2), including delta -> 0 (where the eigen-gap lives)."""
    import mpmath as mp
    mp.mp.dps = 40
    delta = np.concatenate([10.0 ** np.linspace(-14, 0, 600), np.linspace(0, 1, 401)[1:]])
    w = hh.cubic_w(delta)
    ref = np.array([float(1 - mp.cos(mp.acos(1 - mp.mpf(float(d))) / 3)) for d in delta])
    assert np.max(np.abs(w / ref - 1)) < 2e-13
    assert hh.cubic_w(np.array([0.0]))[0] == 0.0 and np.isnan(hh.cubic_w(np.array([np.nan]))[0])


def test_harness_prior_kind_specialisations_and_their_fallback(golden):
    """GF_SPEC_SM6 / GF_SPEC_FIXED7 fix the reference's own prior kinds at compile time (examples/inference.ipynb: three
    LIMITEDGAUSS mixing coordinates, flat dcp and source angles; scripts/fr.py:30-104: the same four, two GAUSSIAN masses,
    flat logLam).  On those models they give what the runtime-kind code gives; a model in the same column layout but with
    other prior kinds is routed to the runtime-layout sibling (gf_model_spec), never to the wrong mask."""
    SM, FIXED, SM6, FIXED7 = 2, 1, 4, 5          # GF_SPEC_* of gf_model.cuh
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    assert hh.model_spec(fm) == (SM6, SM6, 0b000111)
    a = hh.lnprob(fm, g['theta'], spec=SM6)
    b = hh.lnprob(fm, g['theta'], spec=SM)
    c = hh.lnprob(fm, g['theta'])                # the generic specialisation
    for x, y in ((a, b), (a, c)):
        assert np.array_equal(x[0], y[0], equal_nan=True) and np.array_equal(x[1], y[1], equal_nan=True) and np.array_equal(x[2], y[2])
    # same layout, dcp with a Gaussian prior: the mask differs, the layout does not
    other = ParamSet([Param(name=p.name, value=p.value, seed=p.seed, ranges=p.ranges, std=p.std or 0.5,
                            prior=PriorsCateg.GAUSSIAN if p.name == 'dcp' else p.prior, tag=p.tag) for p in pset])
    fo = model.flatten(args, asimov, other)
    assert hh.model_spec(fo) == (SM, SM6, 0b001111)
    ref = go.batch_lnprior(g['theta'], np.array(other.ranges)[:, 0], np.array(other.ranges)[:, 1],
                           [0 if p.prior.name == 'UNIFORM' else 1 if p.prior.name == 'GAUSSIAN' else 2 for p in other],
                           list(other.nominal_values), [p.std or 1.0 for p in other])
    got = hh.lnprior(fo, g['theta'])
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(got), fin) and np.max(np.abs(got[fin] - ref[fin]) / np.maximum(1.0, np.abs(ref[fin]))) < 1e-12
    # config 3 (scripts/fr.py layout)
    args3, asimov3, pset3 = models.bsm_model_c3(g['asimov_angles'])
    f3 = model.flatten(args3, asimov3, pset3)
    assert hh.model_spec(f3) == (FIXED7, FIXED7, 0b0110111)
    th = models.draw_in_ranges(pset3, 400, np.random.default_rng(3))
    th[::7, 4] = 9e-23                           # out of the prior box
    a = hh.lnprob(f3, th, spec=FIXED7)
    b = hh.lnprob(f3, th, spec=FIXED)
    assert np.array_equal(a[0], b[0], equal_nan=True) and np.array_equal(a[1], b[1], equal_nan=True) and np.array_equal(a[2], b[2])
    flat = ParamSet([Param(name=p.name, value=p.value, seed=p.seed, ranges=p.ranges, std=p.std, prior=None, tag=p.tag) for p in pset3])
    assert hh.model_spec(model.flatten(args3, asimov3, flat)) == (FIXED, FIXED7, 0)


def test_harness_source_angles_outside_their_natural_box(golden):
    """fr.py:101-113 takes |cos^2 phi|: for sin^4 phi > 1 the source built from the angles no longer sums to one and
    u_to_fr's division by sum(source) (fr.py:535) matters.  The SM-only path skips that division only while the source is
    unit-sum by construction."""
    g = golden('ref_llh.npz')
    args, asimov, pset = models.notebook_model(g['asimov_angles'])
    fm = model.flatten(args, asimov, pset)
    rng = np.random.default_rng(11)
    th = models.draw_in_ranges(pset, 200, rng)
    th[:100, 4] = rng.uniform(1.0, 2.5, 100)     # sin^4 phi beyond one (no prior is evaluated by flux_averaged_fr)
    th[100, 4], th[101, 4] = 1.0, 0.0
    fr, st = hh.fr(fm, th)
    ref = np.array([np.asarray(go.u_to_fr(go.angles_to_fr(t[4:6]), go.angles_to_u(t[:4])), dtype=np.float64) for t in th])
    assert np.abs(fr - ref).max() < 1e-14 and np.abs(fr.sum(axis=1) - 1).max() < 1e-15
    assert not st.any()


def test_gaussian_weights_are_scipys():
    """scan.gaussian_weights restates SciPy's kernel construction (the device filter is handed these weights): same radius
    rule int(4 sigma + 0.5) and bit-identical values; the reference's default hist_smooth = 0.05 is a one-tap identity."""
    from scipy.ndimage import _filters, gaussian_filter
    for sigma in (0.05, 0.1249, 0.125, 0.4, 1.0, 2.5, 16.0):
        radius, w = scan.gaussian_weights(sigma)
        assert radius == int(4.0 * sigma + 0.5) and len(w) == 2 * radius + 1
        assert np.array_equal(w, _filters._gaussian_kernel1d(sigma, 0, radius))
    assert scan.gaussian_weights(0.05)[0] == 0
    h = np.random.default_rng(1).random((5, 5, 5))
    assert np.array_equal(gaussian_filter(h, sigma=0.05), h)


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on
    stdout with the contract's keys, timing the oracle port on the host cores; the GPU arm refuses to run
    without a device instead of falling back."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['metric'] == 'log-posterior evals/sec' and d['value'] > 10
    installed = os.path.isdir(os.path.join(root, 'baseline', '_ref', 'golemflavor'))
    assert d['cpu_baseline']['kind'] == ('reference' if installed else 'port') and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['value'] == d['value']
    gpu = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--steps', '1'], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, env=env, timeout=600)
    assert gpu.returncode != 0 and 'no CUDA device' in (gpu.stderr + gpu.stdout)


def test_bench_refuses_no_timed_steps_and_a_dump_of_the_reference_arm(tmp_path):
    """`--steps` is the number of timed steps, so 0 is refused rather than rounded up; `--dump-outputs` belongs to the GPU
    arm (the reference arm keeps no outputs) and is refused before any work or any file is written."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    for extra in (['--steps', '0'], ['--impl', 'reference', '--steps', '0'],
                  ['--impl', 'reference', '--dump-outputs', str(tmp_path / 'out')]):
        res = subprocess.run([sys.executable, os.path.join(root, 'bench.py')] + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                             text=True, env=env, timeout=600)
        assert res.returncode == 2 and not res.stdout.strip(), (extra, res.stderr[-500:])
    assert not os.path.exists(tmp_path / 'out')


def test_installed_reference_agrees_with_the_oracle_on_the_headline_model():
    """`baseline/_ref` (the unmodified reference, pip-installed by `__graft_entry__.build()`; absent on boxes without
    /root/reference and then skipped): the ln_prob composition that `bench.py --impl reference` times equals the oracle's
    `ln_prob` on the headline model -- the same x87 arithmetic, bit for bit -- so either CPU arm measures the same work."""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    ref = bench._reference_problem()
    if ref is None:
        pytest.skip('baseline/_ref not installed')
    ln_prob, pset = ref
    go, args, asimov, ps = bench._cpu_problem()
    theta = bench.synth_theta(pset, 24, 77, sys.modules['models'])
    theta[0, 0] = 1.5    # out of the prior box: -inf before any physics (llh.py:125-126)
    for t in theta:
        with np.errstate(all='ignore'):
            try:
                a = float(ln_prob(t))
            except AssertionError:
                a = np.nan
            try:
                b = float(go.ln_prob(list(t), args, asimov, ps))
            except AssertionError:
                b = np.nan
        assert a == b or (a != a and b != b), (a, b)
    assert float(ln_prob(theta[0])) == -np.inf


def test_mcmc_driver_probes_scalar_callables(capsys):
    """A reference-style scalar ln_prob(theta[ndim]) (mcmc.py:29-31 hands such a callable to emcee) is mapped over the
    walkers; a batched callable is called once per half-ensemble."""
    calls = {'scalar': 0, 'batch': 0}

    def scalar(theta):
        calls['scalar'] += 1
        x, y = theta            # raises for a batch
        return -0.5 * (x * x + y * y)

    def batch(theta):
        calls['batch'] += 1
        theta = np.atleast_2d(theta)
        return -0.5 * (theta ** 2).sum(axis=1)

    np.random.seed(1)
    p0 = np.random.normal(size=(8, 2))
    s1 = mcmc.mcmc(p0, scalar, 2, 8, 5, 10, seed=3)
    s2 = mcmc.mcmc(p0, batch, 2, 8, 5, 10, seed=3)
    capsys.readouterr()
    assert s1.shape == s2.shape == (80, 2) and np.allclose(s1, s2)
    assert calls['scalar'] > 8 * 15 and calls['batch'] < 2 * 15 + 5


def test_get_limit_matches_reference_fixture(golden):
    """sens.get_limit against plot.get_limit of the unmodified reference (tests/golden/make_golden_limit.py): the same
    limit / None outcome and the same splined reduced-evidence curve on every fixture curve."""
    from golemflavor_b200 import sens
    g = golden('ref_limit.npz')
    assert float(g['bayes_k']) == sens.BAYES_K
    nlim = 0
    for k in range(int(g['n'])):
        sc, st, ref, mi = g['scales_%d' % k], g['stat_%d' % k], float(g['limit_%d' % k]), bool(g['mask_%d' % k])
        got = sens.get_limit(sc, st, mask_initial=mi)
        if np.isnan(ref):
            assert got is None, (k, got)
            continue
        nlim += 1
        assert got is not None and abs(got - ref) < 1e-12, (k, got, ref)
        isc, iev = sens.get_limit(sc, st, mask_initial=mi, return_interp=True)
        assert np.allclose(isc, g['interp_sc_%d' % k], rtol=0, atol=1e-12) and np.allclose(iev, g['interp_ev_%d' % k], rtol=0, atol=1e-10)
    assert nlim >= 10
    ev = {6: np.column_stack([g['scales_0'], g['stat_0']])}
    assert sens.limits(ev)[6] == sens.get_limit(g['scales_0'], g['stat_0'])


def test_harness_inverse_normal_cdf_table_against_scipy():
    """The table-based Phi^-1 of the truncated-Gaussian prior draws (csrc/gf_ndtri_table.h, gf_scan_dev.cuh) against
    scipy.special.ndtri: 1e-13 absolute wherever the table applies (min(p, 1-p) in [2^-17, 1/2)), and it declines
    everything else (deep tails, p = 1/2, p outside (0, 1), NaN) so that the library routine takes over."""
    from scipy.special import ndtri
    rng = np.random.default_rng(5)
    p = np.concatenate([rng.uniform(0, 1, 200000), 2.0 ** -rng.uniform(1, 17, 50000), 1 - 2.0 ** -rng.uniform(1, 17, 50000),
                        np.nextafter(2.0 ** -np.arange(1, 18), 0), 2.0 ** -np.arange(2, 18), [0.5 - 1e-17, np.nextafter(0.5, 0), np.nextafter(0.5, 1)]])
    z, ok = hh.ndtri(p)
    t = np.minimum(p, 1 - p)
    assert np.array_equal(ok, (t >= 2.0 ** -17) & (t < 0.5))
    assert ok.mean() > 0.99
    assert np.abs(z[ok] - ndtri(p[ok])).max() < 1e-13
    for bad in (0.5, 0.0, 1.0, -0.1, 1.1, 1e-6, 1 - 1e-6, np.nan, np.inf):
        assert not hh.ndtri([bad])[1][0], bad
    # exact antisymmetry (1 - q is exact for multiples of 2^-40) and monotonicity across the row boundaries
    q = rng.integers(1 << 24, 1 << 39, 100000).astype(np.float64) * 2.0 ** -40
    assert np.array_equal(hh.ndtri(q)[0], -hh.ndtri(1 - q)[0])
    edges = (2.0 ** -np.arange(2, 18)[:, None] * (1 + np.arange(8) / 8)).ravel()
    grid = np.sort(np.concatenate([q, edges, np.nextafter(edges, 0), np.nextafter(edges, 1)]))
    zz, cov = hh.ndtri(grid)
    assert np.all(np.diff(zz[cov]) >= -2e-13)
    # a scan model with LIMITEDGAUSS / GAUSSIAN priors now draws on the host as well (away from the deep tails)
    fm = scan.scan_model('texture')
    th = hh.draw(fm, 26, 0, 2000)
    ps = scan.scan_paramset('texture', 6)
    from scipy.stats import norm
    for k, prm in enumerate(ps):
        u = go.philox_uniforms(26, 0, 2000, block=k // 4)[:, k % 4]
        lo, hi_ = prm.ranges
        if prm.prior.name == 'UNIFORM':
            ref = lo + u * (hi_ - lo)
        else:
            a, b = norm.cdf((lo - prm.nominal_value) / prm.std), norm.cdf((hi_ - prm.nominal_value) / prm.std)
            ref = np.clip(prm.nominal_value + prm.std * ndtri(a + u * (b - a)), lo, hi_)
        good = np.isfinite(th[:, k])
        assert good.mean() > 0.999 and np.max(np.abs(th[good, k] - ref[good]) / np.abs(ref[good])) < 1e-12


def test_harness_refinement_rebuilds_identical_matrices(golden):
    """k_lnprob keeps neither H0 nor T for the rare refinement path: it re-reads the row and rebuilds them
    (gf_mats_rebuild).  Same bits as the variant that keeps them in memory, on a batch with refined points, for the
    fixed-texture, the free-NP and the sampled-source specialisations."""
    g = golden('ref_llh.npz')
    rng = np.random.default_rng(12)
    cases = [models.bsm_model_c3(g['asimov_angles'], dim=3, texture=Texture.OET),
             models.bsm_model_c3(g['asimov_angles'], dim=6, texture=Texture.OUT),
             models.bsm_sampled_source(g['asimov_angles'], 'angles', 6, Texture.OET)]
    a11 = models.bsm_args(6, Texture.NONE)
    a11.injected_ratio, a11.smearing = [1 / 3, 1 / 3, 1 / 3], 0.02
    cases.append((a11, None, models.bsm11_paramset(6)))
    refined = 0
    for args, asimov, pset in cases:
        fm = model.flatten(args, asimov, pset)
        theta = models.draw_in_ranges(pset, 40000, rng)
        l0, f0, s0 = hh.lnprob(fm, theta)
        l1, f1, s1 = hh.lnprob(fm, theta, rebuild=True)
        assert np.array_equal(l0, l1, equal_nan=True) and np.array_equal(f0, f1, equal_nan=True) and np.array_equal(s0, s1)
        refined += int(np.count_nonzero(s0 & _lib.ST_REFINED))
    assert refined > 20
