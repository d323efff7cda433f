/*
 * gf_profile_dev.cuh -- the profile likelihood of one (scale, start) task: bounded Nelder-Mead over the nuisance
 * parameters of a model whose new-physics scale is frozen (see gf_profile_grid and gf_profile_sources in the C header and
 * gf_profile.cu).
 *
 * The optimiser core is templated on the objective, so the host harness runs it on an analytic function as well
 * as on the model.  It is written as a STATE MACHINE that makes exactly one objective evaluation per iteration:
 * reflection, expansion, the two contractions and every vertex of a shrink are candidate points chosen by the
 * state, followed by the same single call of the objective.  In a warp whose threads sit in different states only
 * the bookkeeping diverges; the ~1 900-instruction log-posterior runs once per iteration for the whole warp.
 */
#ifndef GF_PROFILE_DEV_CUH
#define GF_PROFILE_DEV_CUH

#include "gf_ensemble_dev.cuh" /* GF_*_RN, gf_draw_theta */
#include "gf_sources_dev.cuh"  /* gf_src_rec, gf_src_llh */

/* the starting simplex: vertex j = x0 + GF_NM_STEP e_(j-1) in scaled coordinates (one sigma of a Gaussian prior, a tenth of a
 * uniform box), stepping inwards when the outward step would leave the box */
#define GF_NM_STEP 1.0

struct gf_nm_opts {
    double ftol, xtol;
    int32_t max_evals;
};

struct gf_nm_out {
    int32_t nevals; /* optimiser evaluations (the final re-evaluation of the best vertex is not counted) */
    int32_t best;   /* slot of the best vertex */
    bool converged; /* stopped by the restart rule, not by max_evals */
};

/*
 * Minimise g over the box [obj.lo(k), obj.hi(k)] from x0 with the dimension-adaptive coefficients of Gao & Han (2012)
 * (SciPy's `adaptive=True`): reflection 1, expansion 1 + 2/n, contraction 3/4 - 1/(2n), shrink 1 - 1/n; every candidate is
 * projected onto the box.  Converged when max |g_v - g_best| <= ftol and max |x_v - x_best| <= xtol (SciPy's fatol / xatol);
 * then the simplex restarts from the best vertex, and the run stops when a restart gains less than ftol, or after
 * max_evals evaluations.  Finally the best vertex is evaluated once more, so that the objective's side outputs (the
 * composition, the status) describe it.
 *
 * S holds the simplex of this task, element e at S[e * ld]: vertex v at elements v*n .. v*n+n-1, its value at (n+1)*n + v:
 * (n+1)^2 doubles.  g = NaN or -inf counts as +inf.  The simplex is never sorted: best, worst and second-worst vertices are
 * found by a scan (ties: lowest index is best, highest index is worst), identically on the host and the device.
 * All simplex arithmetic is GF_*_RN (no FMA contraction).  NDIM > 0: the dimension count at compile time.
 */
template <int NDIM, class Obj>
GF_HD gf_nm_out gf_nm_minimize(Obj& obj, int n_rt, const double* x0, double* S, int ld, const gf_nm_opts& o) {
    constexpr int NMAX = NDIM > 0 ? NDIM : GF_MAX_DIM;
    const int n = NDIM > 0 ? NDIM : n_rt;
    auto X = [&](int v, int k) -> double& { return S[(int64_t)(v * n + k) * ld]; };
    auto F = [&](int v) -> double& { return S[(int64_t)((n + 1) * n + v) * ld]; };
    const double dn = (double)n;
    const double chi = GF_ADD_RN(1.0, GF_DIV_RN(2.0, dn));
    const double psi = GF_SUB_RN(0.75, GF_DIV_RN(1.0, GF_MUL_RN(2.0, dn)));
    const double sig = GF_SUB_RN(1.0, GF_DIV_RN(1.0, dn));
    enum { INIT, REFLECT, EXPAND, CONT_OUT, CONT_IN, SHRINK, FINAL };
    for (int v = 0; v <= n; ++v) F(v) = INFINITY;
    int state = INIT, j = 0, b = 0, w = 0, s2 = 0, nev = 0, restarts = 0;
    double fr = INFINITY, g_restart = INFINITY;
    bool conv = false;
    double xc[NMAX], xbar[NMAX];
    for (;;) {
        /* ---- the candidate of this iteration */
        if (state == INIT) {
            for (int k = 0; k < n; ++k) {
                double x = j == 0 ? x0[k] : X(0, k);
                if (k == j - 1) {
                    const double up = GF_ADD_RN(x, GF_NM_STEP);
                    x = up <= obj.hi(k) ? up : GF_SUB_RN(x, GF_NM_STEP);
                }
                xc[k] = x;
            }
        } else if (state == SHRINK) {
            for (int k = 0; k < n; ++k) xc[k] = GF_ADD_RN(X(b, k), GF_MUL_RN(sig, GF_SUB_RN(X(j, k), X(b, k))));
        } else if (state == FINAL) {
            for (int k = 0; k < n; ++k) xc[k] = X(b, k);
        } else {
            /* centroid of every vertex but the worst, then a point on the line through the worst vertex */
            const double c = state == REFLECT ? 1.0 : state == EXPAND ? chi : state == CONT_OUT ? psi : -psi;
            for (int k = 0; k < n; ++k) {
                double sum = 0.0;
                for (int v = 0; v <= n; ++v)
                    if (v != w) sum = GF_ADD_RN(sum, X(v, k));
                xbar[k] = GF_DIV_RN(sum, dn);
                xc[k] = GF_ADD_RN(xbar[k], GF_MUL_RN(c, GF_SUB_RN(xbar[k], X(w, k))));
            }
        }
        for (int k = 0; k < n; ++k) xc[k] = fmin(fmax(xc[k], obj.lo(k)), obj.hi(k));
        /* ---- the one evaluation */
        double g = obj(xc);
        if (!(g > -INFINITY)) g = INFINITY;
        if (state == FINAL) break;
        ++nev;
        /* ---- transition */
        auto put = [&](int v, const double* x, double gv) {
            for (int k = 0; k < n; ++k) X(v, k) = x[k];
            F(v) = gv;
        };
        bool top = false;
        if (state == INIT) {
            put(j, xc, g);
            top = ++j > n;
        } else if (state == REFLECT) {
            if (g < F(b)) {
                fr = g;
                state = EXPAND;
            } else if (g < F(s2)) {
                put(w, xc, g);
                top = true;
            } else {
                fr = g;
                state = g < F(w) ? CONT_OUT : CONT_IN;
            }
        } else if (state == EXPAND) {
            if (!(g < fr)) /* keep the reflected point: rebuild it from the unchanged simplex (xbar is this iteration's) */
                for (int k = 0; k < n; ++k) xc[k] = fmin(fmax(GF_ADD_RN(xbar[k], GF_SUB_RN(xbar[k], X(w, k))), obj.lo(k)), obj.hi(k));
            put(w, xc, g < fr ? g : fr);
            top = true;
        } else if (state == CONT_OUT || state == CONT_IN) {
            if (state == CONT_OUT ? g <= fr : g < F(w)) {
                put(w, xc, g);
                top = true;
            } else {
                state = SHRINK;
                j = b == 0 ? 1 : 0;
            }
        } else { /* SHRINK */
            put(j, xc, g);
            if (++j == b) ++j;
            top = j > n;
        }
        if (top) {
            b = 0;
            w = 0;
            for (int v = 1; v <= n; ++v) {
                if (F(v) < F(b)) b = v;
                if (F(v) >= F(w)) w = v;
            }
            if (w == b) w = b == 0 ? n : 0; /* n >= 1 */
            s2 = w == 0 ? 1 : 0;
            for (int v = 0; v <= n; ++v)
                if (v != w && F(v) >= F(s2)) s2 = v;
            double dx = 0.0, df = 0.0;
            for (int v = 0; v <= n; ++v) {
                if (v == b) continue;
                df = fmax(df, fabs(GF_SUB_RN(F(v), F(b)))); /* inf - inf = NaN is ignored: an all-invalid simplex is flat */
                for (int k = 0; k < n; ++k) dx = fmax(dx, fabs(GF_SUB_RN(X(v, k), X(b, k))));
            }
            state = REFLECT;
            if (dx <= o.xtol && df <= o.ftol) {
                if (restarts == 0 || GF_SUB_RN(g_restart, F(b)) >= o.ftol) {
                    ++restarts;
                    g_restart = F(b);
                    if (b != 0) {
                        for (int k = 0; k < n; ++k) X(0, k) = X(b, k);
                        F(0) = F(b);
                    }
                    b = 0;
                    j = 1;
                    state = INIT;
                } else {
                    conv = true;
                    state = FINAL;
                }
            }
        }
        if (state != FINAL && nev >= o.max_evals) state = FINAL;
        if (state == FINAL) {
            b = 0;
            for (int v = 1; v <= n; ++v)
                if (F(v) < F(b)) b = v;
        }
    }
    return gf_nm_out{nev, b, conv};
}

/* ------------------------------------------------------------------ the model's objective */

GF_HD double gf_exp10(double x) {
#ifdef __CUDA_ARCH__
    return exp10(x); /* the same exp10 the per-point kernels apply to logLam */
#else
    return pow(10.0, x);
#endif
}

/* Scaled coordinate of dimension k: x = theta / unit, unit = sigma for Gaussian kinds, a tenth of the box for uniform ones
 * (the parameters span 23 orders of magnitude: m21^2 ~ 7e-23). */
GF_HD double gf_profile_unit(const gf_dev_model& m, int k) {
    return m.kind[k] == GF_PRIOR_UNIFORM ? GF_DIV_RN(GF_SUB_RN(m.hi[k], m.lo[k]), 10.0) : m.sigma[k];
}

/* The nominal start: the prior mean clipped to the box; the centre of the box for uniform kinds (which carry no mean). */
GF_HD double gf_profile_nominal(const gf_dev_model& m, int k) {
    if (m.kind[k] == GF_PRIOR_UNIFORM) return GF_ADD_RN(m.lo[k], GF_MUL_RN(0.5, GF_SUB_RN(m.hi[k], m.lo[k])));
    return fmin(fmax(m.mu[k], m.lo[k]), m.hi[k]);
}

/* The point of the physics at theta: the layout of sens.py for STATIC6 (columns 0-3 mixing coordinates, 4-5 mass
 * splittings), the model's column map otherwise. */
template <int SPEC, bool STATIC6>
GF_HD void gf_profile_point(const gf_dev_model& m, const double* th, gf_point& q) {
    if constexpr (STATIC6) {
        q.sm[0] = th[0]; q.sm[1] = th[1]; q.sm[2] = th[2]; q.sm[3] = th[3];
        q.mass[0] = th[4]; q.mass[1] = th[5];
        q.src_unit = false;
    } else {
        gf_resolve_point<SPEC>(m, [&](int k) { return th[k]; }, q);
    }
}

/* -ln_prob of an objective at scaled coordinates x: theta_k = x_k unit_k clipped to the prior box; NaN and +inf ln_prob count
 * as -inf and set GFP_ST_NON_FINITE in obj.st and obj.nonfinite. */
template <class Obj>
GF_HD double gf_profile_neg(Obj& obj, const double* x) {
    constexpr int NDIM = Obj::NDIM;
    double th[NDIM > 0 ? NDIM : GF_MAX_DIM];
    for (int k = 0; k < (NDIM > 0 ? NDIM : obj.m.ndim); ++k) th[k] = obj.theta(x[k], k);
    const double f = obj.lnprob(th);
    if (f != f || f == INFINITY) {
        obj.st |= GFP_ST_NON_FINITE;
        obj.nonfinite |= GFP_ST_NON_FINITE;
        return INFINITY;
    }
    return -f;
}

/*
 * -ln_prob at log10 Lambda = log10(lam) of a frozen-scale model (col_scale < 0), on scaled coordinates.  The point is
 * theta_k = x_k unit_k clipped to the prior box; ln_prob is llh.ln_prob as gf_point_lnprob computes it, with the scale
 * substituted through gf_point_fr_scales (ns = 1).  Non-finite values count as -inf and set GF_ST_NON_FINITE in
 * `nonfinite`.  The last evaluation's composition and status stay in fr / st.
 */
template <int SPEC, bool STATIC6, int ILP>
struct gf_profile_obj {
    static constexpr int NDIM = STATIC6 ? 6 : 0;
    const gf_dev_model& m;
    double lam;
    unsigned nonfinite = 0u, st = 0u;
    double fr[3] = {0.0, 0.0, 0.0};

    GF_HD double lo(int k) const { return GF_DIV_RN(m.lo[k], gf_profile_unit(m, k)); }
    GF_HD double hi(int k) const { return GF_DIV_RN(m.hi[k], gf_profile_unit(m, k)); }
    GF_HD double theta(double x, int k) const { return fmin(fmax(GF_MUL_RN(x, gf_profile_unit(m, k)), m.lo[k]), m.hi[k]); }

    /* ln prior at th; where it is not finite, fr is NaN and st says why (as gf_point_lnprob) */
    GF_HD double lnprior(const double* th) {
        const double lp = gf_point_lnprior<NDIM>(m, [&](int k) { return th[k]; });
        if (!(lp > -INFINITY)) {
            fr[0] = fr[1] = fr[2] = NAN;
            st = (lp != lp) ? (GFP_ST_NON_FINITE | GFP_ST_OUT_OF_PRIOR) : GFP_ST_OUT_OF_PRIOR;
        }
        return lp;
    }

    GF_HD double lnprob(const double* th) {
        const double lp = lnprior(th);
        if (!(lp > -INFINITY)) return (lp != lp) ? NAN : -INFINITY;
        gf_point q;
        gf_profile_point<SPEC, STATIC6>(m, th, q);
        gf_point_fr_scales<SPEC, ILP>(
            m, q, 1, [&](int) { return lam; },
            [&](int, const double* f, unsigned s) {
                fr[0] = f[0]; fr[1] = f[1]; fr[2] = f[2];
                st = s;
            });
        if (m.llh_kind == GF_LLH_FLAT) return lp + m.llh_const;
        return lp + gf_multi_gaussian(fr, m.fr_bf, m.half_inv_s2, m.lognorm3, m.offset, m.emulate_underflow, m.underflow_logpdf);
    }

    GF_HD double operator()(const double* x) { return gf_profile_neg(*this, x); }
};

/*
 * The objective of gf_profile_sources: gf_profile_obj with source record *r substituted for the model's source and injected
 * composition (the Gaussian likelihood only).  The eigen stage gives the transition sums of gf_point_transition_scales
 * (ns = 1), and r's composition and likelihood follow from them (gf_src_llh).  st carries the bits gf_point_fr_scales sets:
 * the eigen stage's, NON_UNITARY and NON_FINITE of the composition.
 */
template <int SPEC, bool STATIC6, int ILP>
struct gf_profile_src_obj : gf_profile_obj<SPEC, STATIC6, ILP> {
    const gf_src_rec* r;

    GF_HD double lnprob(const double* th) {
        const gf_dev_model& m = this->m;
        const double lp = this->lnprior(th);
        if (!(lp > -INFINITY)) return (lp != lp) ? NAN : -INFINITY;
        gf_point q;
        gf_profile_point<SPEC, STATIC6>(m, th, q);
        double ll = NAN;
        gf_point_transition_scales<SPEC, ILP>(
            m, q, 1, [&](int) { return this->lam; },
            [&](int, const double* A, unsigned s) {
                double* f = this->fr;
                ll = gf_src_llh(m, *r, A, f);
                if (!(fmin(f[0], fmin(f[1], f[2])) >= -m.epsilon)) s |= GFP_ST_NON_UNITARY;
                if (!(fabs(f[0]) + fabs(f[1]) + fabs(f[2]) < 1e300)) s |= GFP_ST_NON_FINITE;
                this->st = s;
            });
        return lp + ll;
    }

    GF_HD double operator()(const double* x) { return gf_profile_neg(*this, x); }
};

/*
 * One task: start `k` of the scale whose global index is `task` (start 0: the nominal point; start k >= 1: a prior draw of
 * the scans, gf_draw_theta(m, seed, task * nstarts + k)), optimised in place in S (see gf_nm_minimize).  On return
 * obj.fr / obj.st describe the best vertex, whose ln_prob is -S[((n+1) n + out.best) ld].  Obj: gf_profile_obj or
 * gf_profile_src_obj (Obj::NDIM = 6: the static 6-column layout).
 */
template <class Obj>
GF_HD gf_nm_out gf_profile_task(Obj& obj, uint64_t seed, uint64_t task, int32_t nstarts, int32_t k, const gf_nm_opts& o, double* S, int ld) {
    constexpr int NDIM = Obj::NDIM;
    const gf_dev_model& m = obj.m;
    double x0[NDIM > 0 ? NDIM : GF_MAX_DIM];
    if (k == 0) {
        for (int d = 0; d < (NDIM > 0 ? NDIM : m.ndim); ++d) x0[d] = gf_profile_nominal(m, d);
    } else if constexpr (NDIM == 6) {
        gf_draw_theta<true, 6>(m, seed, task * (uint64_t)nstarts + (uint64_t)k, x0);
    } else {
        gf_draw_theta(m, seed, task * (uint64_t)nstarts + (uint64_t)k, x0);
    }
    for (int d = 0; d < (NDIM > 0 ? NDIM : m.ndim); ++d) x0[d] = GF_DIV_RN(x0[d], gf_profile_unit(m, d));
    return gf_nm_minimize<NDIM>(obj, m.ndim, x0, S, ld, o);
}

#endif /* GF_PROFILE_DEV_CUH */
