#!/usr/bin/env python
"""Parameter points whose energy-bin Hamiltonian sits near a level crossing, with 50-digit truth.

Writes ``ref_resonance.npz`` next to this file.  Seeded and deterministic; about 70 s on one core
(most of it the mpmath truth).

Construction.  With the CP phases at zero (SM ``dcp`` and, for Texture.NONE, the NP phase) the Hamiltonian
H = U diag(0, m21, m3x) U^+ + rho N diag(0, 1/100, 1) N^+, rho = 2 E^(d-2) 10^logLam, is real symmetric, and a
level crossing is codimension 2: an exact crossing is bracketed in (logLam, s_23^2) by minimising the LAPACK
relative gap of one energy bin (s_23^2, else s_12^2 or c_13^4, whichever reaches deeper).  The fixed textures carry NP phases of 1e-9 (``model.TEXTURE_ANGLES``), so there
the SM ``dcp`` is a third coordinate of the search.  |V|^2 depends on rho alone, so shifting logLam by
-(d-2) log10(E_b / E_0) moves the crossing from bin 0 to bin b.  That coordinate is then offset from the crossing until the
bin's relative gap (closest pair's splitting / spectral spread) is the target.  Points outside the prior box, or
whose target gap the search could not reach, are dropped.  The OEU texture keeps a relative gap of ~1e-2 everywhere the
search went inside the prior box, so it contributes no points.

Truth: ``oracle.truth.mp_flux_averaged_fr`` (mpmath, dps 50) from the exact double inputs for the 20-bin model
(``models.BINNING``), the 1-bin model of bin b alone and the 7-bin window starting at bin b0 (a remainder case of
every interleave), and ``truth.mp_bin_relgaps`` for the relative gap of every bin.

    python tests/golden/make_golden_resonance.py
"""
import os
import sys

import numpy as np
from scipy.optimize import minimize

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from golemflavor_b200.model import SCALE_BOUNDARIES, TEXTURE_ANGLES  # noqa: E402
from oracle import truth  # noqa: E402

import models  # noqa: E402

TEXTURES = ('OET', 'OUT', 'OEU', 'NONE')
DIMS = (3, 6, 8)
# relative gaps: wide, a band around the fast-path cut (relgap 2.5e-3) and around its former place (1.37e-3), the
# ILL_COND edge (1e-6) and deep in the refinement
STRATA = (1e-1, 1e-2, 3e-3, 2.7e-3, 2.4e-3, 2e-3, 1.6e-3, 1.45e-3, 1.4e-3, 1.37e-3, 1.3e-3, 1.2e-3, 1e-4, 2e-6, 1e-6, 5e-7, 1e-8,
          1e-10)
NP_FREE = (0.3, 0.6, 0.45, 0.0)        # Texture.NONE: Haar-flat NP coordinates with zero NP phase
SM0 = (0.307, (1 - 0.02206) ** 2, 0.538, 0.0)
MASS = (7.40e-23, 2.494e-21)
EDGES = models.BINNING
CENTERS = np.sqrt(EDGES[:-1] * EDGES[1:])


def mix(ang):
    s12_2, c13_4, s23_2, d = ang
    s12, c12 = np.sqrt(s12_2), np.sqrt(1 - s12_2)
    c13_2 = np.sqrt(c13_4)
    c13, s13 = np.sqrt(c13_2), np.sqrt(1 - c13_2)
    s23, c23 = np.sqrt(s23_2), np.sqrt(1 - s23_2)
    ep, em = np.exp(1j * d), np.exp(-1j * d)
    return np.array([[c13 * c12, c13 * s12, s13 * em],
                     [-c23 * s12 - s23 * s13 * ep * c12, c23 * c12 - s23 * s13 * ep * s12, s23 * c13],
                     [s23 * s12 - c23 * s13 * ep * c12, -s23 * c12 - c23 * s13 * ep * s12, c23 * c13]])


def relgap(sm, npa, loglam, dim, energy):
    """LAPACK relative gap of the bin Hamiltonian (times 2E, norm-scaled)."""
    u, n = mix(sm), mix(npa)
    h0 = (u * np.array([0, MASS[0], MASS[1]])) @ u.conj().T
    t = (n * np.array([0, 0.01, 1.0])) @ n.conj().T
    h = h0 + 2 * energy ** (dim - 2) * 10.0 ** loglam * t
    lam = np.linalg.eigvalsh(h / np.abs(h).max())
    d = np.diff(lam)
    return d.min() / (lam[2] - lam[0])


def find_crossing(npa, dim, complex_search):
    """(logLam, SM coordinates, coordinate index, depth) of the deepest relative-gap minimum of bin 0 found from a
    logLam grid, searching in (logLam, one mixing coordinate[, dcp])."""
    lo, hi = SCALE_BOUNDARIES[dim]
    grid = np.linspace(lo, hi, 2000)
    g = np.array([relgap(SM0, npa, x, dim, CENTERS[0]) for x in grid])
    minima = [i for i in range(1, len(g) - 1) if g[i] < g[i - 1] and g[i] < g[i + 1]] or [int(np.argmin(g))]
    best = None
    for ci in (2, 0, 1):
        for i in sorted(minima, key=lambda i: g[i])[:3]:
            x0 = [grid[i], SM0[ci]] + ([0.3] if complex_search else [])

            def f(x):
                if not (0 < x[1] < 1 and lo <= x[0] <= hi):
                    return 10.0
                sm = list(SM0)
                sm[ci] = x[1]
                sm[3] = x[2] if complex_search else 0.0
                return np.log10(relgap(sm, npa, x[0], dim, CENTERS[0]) + 1e-300)

            simplex = np.array([x0] + [np.add(x0, 0.05 * np.eye(len(x0))[k]) for k in range(len(x0))])
            r = minimize(f, x0, method='Nelder-Mead', options={'xatol': 1e-15, 'fatol': 1e-6, 'maxiter': 20000, 'maxfev': 20000,
                                                                'initial_simplex': simplex})
            if best is None or r.fun < best[0]:
                sm = list(SM0)
                sm[ci] = r.x[1]
                sm[3] = (r.x[2] if complex_search else 0.0) % (2 * np.pi)
                best = (r.fun, r.x[0], sm, ci)
    return best[1], best[2], best[3], 10.0 ** best[0]


def offset_to_gap(loglam, sm, ci, npa, dim, b, target):
    """SM coordinates with sm[ci] offset from the crossing until the bin's relative gap is the target (bisection on
    the log of the offset)."""
    for sign in (1.0, -1.0):
        def at(dl):
            out = list(sm)
            out[ci] = sm[ci] + sign * 10.0 ** dl
            return out

        f = lambda dl: relgap(at(dl), npa, loglam, dim, CENTERS[b]) - target
        room = 1.0 - sm[ci] if sign > 0 else sm[ci]
        a, c = -16.0, min(-0.5, np.log10(0.99 * room))
        if not (c > a and f(a) < 0 < f(c)):
            continue
        for _ in range(80):
            m = 0.5 * (a + c)
            a, c = (m, c) if f(m) < 0 else (a, m)
        return at(c)
    return None


def main():
    import time
    t0 = time.time()
    rows = []
    k = 0
    for tex in TEXTURES:
        npa = np.array(NP_FREE if tex == 'NONE' else TEXTURE_ANGLES[tex], dtype=np.float64)
        for dim in DIMS:
            lam0, smc, ci, depth = find_crossing(npa, dim, tex != 'NONE')
            print('%s dim %d: crossing depth %.2e at logLam %.6f, SM %s, coordinate %d' % (tex, dim, depth, lam0, smc, ci), flush=True)
            lo, hi = SCALE_BOUNDARIES[dim]
            for target in STRATA:
                b = k % 20
                k += 1
                loglam = lam0 - (dim - 2) * np.log10(CENTERS[b] / CENTERS[0])
                if not lo <= loglam <= hi or target < 30 * depth:
                    continue
                sm = offset_to_gap(loglam, smc, ci, npa, dim, b, target)
                if sm is not None:
                    rows.append((tex, dim, b, target, sm, loglam, npa))
    print('%d points, construction %.0f s' % (len(rows), time.time() - t0), flush=True)
    n = len(rows)
    out = {k: [] for k in ('texture', 'dim', 'bin', 'target', 'theta', 'np', 'fr20', 'fr1', 'fr7', 'b7', 'relgap')}
    src = np.array([1., 2., 0.]) / 3
    for i, (tex, dim, b, target, sm, loglam, npa) in enumerate(rows):
        theta = np.array(list(sm) + list(MASS) + [loglam])
        b7 = min(max(b - 3, 0), 13)
        out['texture'].append(tex)
        out['dim'].append(dim)
        out['bin'].append(b)
        out['target'].append(target)
        out['theta'].append(theta)
        out['np'].append(npa)
        out['b7'].append(b7)
        args = (theta[:4], theta[4:6], npa, theta[6], dim)
        out['fr20'].append(truth.mp_flux_averaged_fr(*args, EDGES, src))
        out['fr1'].append(truth.mp_flux_averaged_fr(*args, EDGES[b:b + 2], src))
        out['fr7'].append(truth.mp_flux_averaged_fr(*args, EDGES[b7:b7 + 8], src))
        out['relgap'].append(truth.mp_bin_relgaps(*args, EDGES))
    arrays = {k: np.array(v) for k, v in out.items()}
    arrays['source'] = src
    arrays['binning'] = EDGES
    np.savez_compressed(os.path.join(HERE, 'ref_resonance.npz'), **arrays)
    print('wrote %d points in %.0f s' % (n, time.time() - t0))


if __name__ == '__main__':
    main()
