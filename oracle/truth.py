"""Independent "truth" evaluators for the eigen stage -- TEST INFRASTRUCTURE ONLY.

The reference's float128 Cardano (golemflavor/fr.py:170-237) is itself
ill-conditioned on part of the scan range (SURVEY.md section 7, hard part 1): it
fails its own unitarity assertion on a few per cent of uniformly drawn BSM points
and is wrong by up to 1e-8 on some points it accepts.  Parity of the CUDA path is
therefore reported twice: against the reference restatement where the reference
is well-conditioned, and against the evaluators below everywhere.

* ``mp_flux_averaged_fr``: mpmath (dps = 50) Hermitian eigendecomposition of the
  same Hamiltonian built from the same double-precision inputs.
* ``eigh_absv2`` / ``eigh_flux_averaged_fr``: LAPACK ``zheev`` (NumPy ``eigh``) on
  the norm-scaled fp64 Hamiltonian; agrees with mpmath to a few 1e-16/gap and is
  fast enough for 1e5-point parity sets.
"""

from __future__ import annotations

import numpy as np

from . import golem_oracle as go


def eigh_absv2(h):
    """|V|^2 of Hermitian h[..., 3, 3] by LAPACK after scaling to unit norm."""
    h = np.asarray(h, dtype=np.complex128)
    nrm = np.sqrt((np.abs(h) ** 2).sum(axis=(-1, -2)))
    nrm = np.where(nrm > 0, nrm, 1.0)
    _, v = np.linalg.eigh(h / nrm[..., None, None])
    return np.abs(v) ** 2


def eigh_vectors(h):
    """Adapter with the batch_cardano calling convention (eigenvector matrices)."""
    h = np.asarray(h)
    nrm = np.sqrt((np.abs(h) ** 2).sum(axis=(-1, -2))).astype(np.float64)
    nrm = np.where(nrm > 0, nrm, 1.0)
    hs = (h / nrm[..., None, None]).astype(np.complex128)
    _, v = np.linalg.eigh(hs)
    return v


def eigh_flux_averaged_fr(sm_angles, mass, np_angles, loglam, dim, binning, source):
    """flux_averaged_BSMu with the eigen stage replaced by scaled fp64 LAPACK."""
    fr, _ = go.batch_flux_averaged_fr(sm_angles, mass, np_angles, loglam, dim,
                                      binning, source, eig=eigh_vectors)
    return fr


def _mp_u(ang, mp):
    s12_2, c13_4, s23_2, dcp = [mp.mpf(float(a)) for a in ang]
    s12, c12 = mp.sqrt(s12_2), mp.sqrt(1 - s12_2)
    c13_2 = mp.sqrt(c13_4)
    c13, s13 = mp.sqrt(c13_2), mp.sqrt(1 - c13_2)
    s23, c23 = mp.sqrt(s23_2), mp.sqrt(1 - s23_2)
    ep = mp.e ** (1j * dcp)
    em = mp.e ** (-1j * dcp)
    return mp.matrix([
        [c13 * c12, c13 * s12, s13 * em],
        [-c23 * s12 - s23 * s13 * ep * c12, c23 * c12 - s23 * s13 * ep * s12, s23 * c13],
        [s23 * s12 - c23 * s13 * ep * c12, -s23 * c12 - c23 * s13 * ep * s12, c23 * c13]])


def _mp_bin_hamiltonian(sm_angles, mass, np_angles, loglam, dim, energy, mp):
    u = _mp_u(sm_angles, mp)
    n = _mp_u(np_angles, mp)
    m = mp.diag([0, mp.mpf(float(mass[0])), mp.mpf(float(mass[1]))])
    sc2 = mp.mpf(10) ** mp.mpf(float(loglam))
    s = mp.diag([0, sc2 / 100, sc2])
    e = mp.mpf(float(energy))
    h = (u * m * u.H) / (2 * e) + (e ** (dim - 3)) * (n * s * n.H)
    return (h + h.H) / 2


def mp_bsm_fr_bin(sm_angles, mass, np_angles, loglam, dim, energy, source, dps=50):
    """u_to_fr(source, eigvecs(H)) for one energy, all in mpmath."""
    import mpmath as mp
    mp.mp.dps = dps
    _, v = mp.eighe(_mp_bin_hamiltonian(sm_angles, mass, np_angles, loglam, dim, energy, mp))
    p = [[abs(v[a, i]) ** 2 for i in range(3)] for a in range(3)]
    src = [mp.mpf(float(x)) for x in source]
    tot = sum(src)
    out = []
    for b in range(3):
        acc = mp.mpf(0)
        for a in range(3):
            for i in range(3):
                acc += p[a][i] * p[b][i] * src[a]
        out.append(acc / tot)
    return out


def mp_flux_averaged_fr(sm_angles, mass, np_angles, loglam, dim, binning, source, dps=50):
    """flux_averaged_BSMu (golemflavor/fr.py:413-457) in mpmath for one point."""
    import mpmath as mp
    mp.mp.dps = dps
    binning = np.asarray(binning, dtype=np.float64)
    centers = np.sqrt(binning[:-1] * binning[1:])
    widths = np.abs(np.diff(binning))
    acc = [mp.mpf(0)] * 3
    for ec, w in zip(centers, widths):
        f = mp_bsm_fr_bin(sm_angles, mass, np_angles, loglam, dim, ec, source, dps)
        acc = [a + mp.mpf(float(w)) * x for a, x in zip(acc, f)]
    tot = sum(acc)
    return np.array([float(a / tot) for a in acc])


def mp_bin_relgaps(sm_angles, mass, np_angles, loglam, dim, binning, dps=50):
    """Relative gap of every energy bin's Hamiltonian in mpmath: the closest eigenvalue pair's splitting divided by
    the spectral spread (the quantity the kernels' ILL_COND flag and fast-path cut refer to)."""
    import mpmath as mp
    mp.mp.dps = dps
    binning = np.asarray(binning, dtype=np.float64)
    out = []
    for ec in np.sqrt(binning[:-1] * binning[1:]):
        lam = sorted(mp.eighe(_mp_bin_hamiltonian(sm_angles, mass, np_angles, loglam, dim, ec, mp), eigvals_only=True))
        out.append(float(min(lam[1] - lam[0], lam[2] - lam[1]) / (lam[2] - lam[0])))
    return np.array(out)
