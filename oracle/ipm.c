/*
 * oracle/ipm.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.  See ipm.h.
 *
 * Restates Algorithm A of Waechter & Biegler (2006) -- the algorithm
 * Ipopt 3.12.8 runs when the reference calls app->OptimizeTNLP
 * (mpc_ros/include/cppad/ipopt/solve.hpp:586) with only print_level and
 * max_cpu_time overridden (mpc_ros/src/mpc_planner.cpp:358,368):
 * monotone barrier update, gradient-based NLP scaling, least-squares
 * multiplier start, filter line search with second-order correction,
 * inertia-correcting regularisation.  Ipopt's restoration phase is replaced
 * by a plain feasibility (min-norm Gauss-Newton) fallback.
 */
#include "ipm.h"
#include "ldl.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define IPM_INF 1e19

void ipm_default_options(ipm_options *o)
{
    o->tol = 1e-8;
    o->max_iter = 3000;
    o->max_cpu_time = 1e6;
    o->dual_inf_tol = 1.0;
    o->constr_viol_tol = 1e-4;
    o->compl_inf_tol = 1e-4;
    o->acceptable_tol = 1e-6;
    o->acceptable_iter = 15;
    o->mu_init = 0.1;
    o->bound_push = 0.01;
    o->bound_frac = 0.01;
    o->bound_relax_factor = 1e-8;
    o->nlp_scaling_max_gradient = 100.0;
    o->max_soc = 4;
    o->print_level = 0;
    o->use_dense_ldl = 0;
}

typedef struct {
    const ipm_nlp *nlp;
    const ipm_options *opt;
    int n, m, ns, N, NK;
    int *slack_of;      /* m: slack index (0..ns) or -1 for equality rows */
    double *gl, *gu;    /* m, scaled */
    double *XL, *XU;    /* N, relaxed, scaled where slack */
    char *hasL, *hasU;
    int nbL, nbU;
    double sf;          /* objective scaling */
    double *sc;         /* m constraint scaling */
    int *jr, *jc;       /* Jacobian structure */
    int *hr, *hc;       /* Hessian structure */
    double *jv, *hv;    /* values (scaled) */
    double *graw;       /* m: unscaled g(x) */
    double *lam_tmp;    /* m */
    /* KKT */
    int *pos;           /* NK: position of original index in factor ordering */
    ldl_fact *F;
    int nfact;
} ipm_ws;

static double cpu_now(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* ---- scaled function evaluations on the augmented variable X = [x; s] ---- */
static int ev_fc(ipm_ws *w, const double *X, double *f, double *c)
{
    const ipm_nlp *p = w->nlp;
    double fr;
    if (!p->eval_f(p->user, X, &fr)) return 0;
    if (!p->eval_g(p->user, X, w->graw)) return 0;
    *f = w->sf * fr;
    for (int i = 0; i < w->m; i++) {
        double gi = w->sc[i] * w->graw[i];
        if (w->slack_of[i] < 0) c[i] = gi - w->gl[i];
        else c[i] = gi - X[w->n + w->slack_of[i]];
    }
    if (!isfinite(*f)) return 0;
    for (int i = 0; i < w->m; i++) if (!isfinite(c[i])) return 0;
    return 1;
}

static int ev_grad(ipm_ws *w, const double *X, double *g)
{
    const ipm_nlp *p = w->nlp;
    if (!p->eval_grad_f(p->user, X, g)) return 0;
    for (int i = 0; i < w->n; i++) g[i] *= w->sf;
    for (int i = w->n; i < w->N; i++) g[i] = 0.0;
    return 1;
}

static int ev_jac(ipm_ws *w, const double *X)
{
    const ipm_nlp *p = w->nlp;
    if (!p->eval_jac(p->user, X, w->jv)) return 0;
    for (int k = 0; k < p->nnz_jac; k++) w->jv[k] *= w->sc[w->jr[k]];
    return 1;
}

static int ev_hess(ipm_ws *w, const double *X, const double *lam)
{
    const ipm_nlp *p = w->nlp;
    for (int i = 0; i < w->m; i++) w->lam_tmp[i] = lam[i] * w->sc[i];
    return p->eval_hess(p->user, X, w->sf, w->lam_tmp, w->hv);
}

/* y = J^T lam over the augmented variables */
static void jt_mul(const ipm_ws *w, const double *lam, double *y)
{
    for (int i = 0; i < w->N; i++) y[i] = 0.0;
    for (int k = 0; k < w->nlp->nnz_jac; k++) y[w->jc[k]] += w->jv[k] * lam[w->jr[k]];
    for (int i = 0; i < w->m; i++)
        if (w->slack_of[i] >= 0) y[w->n + w->slack_of[i]] -= lam[i];
}

/* y = J d */
static void j_mul(const ipm_ws *w, const double *d, double *y)
{
    for (int i = 0; i < w->m; i++) y[i] = 0.0;
    for (int k = 0; k < w->nlp->nnz_jac; k++) y[w->jr[k]] += w->jv[k] * d[w->jc[k]];
    for (int i = 0; i < w->m; i++)
        if (w->slack_of[i] >= 0) y[i] -= d[w->n + w->slack_of[i]];
}

/* Assemble and factor  [W + Sigma + dw I, J^T; J, -dc I]  (W may be NULL => identity-free
 * "restoration" matrix with Wdiag on the diagonal).  Returns inertia through F. */
static void kkt_factor(ipm_ws *w, const double *Sigma, int use_hess, double dw, double dc)
{
    const int NK = w->NK, N = w->N, n = w->n;
    double *A = w->F->A;
    memset(A, 0, sizeof(double) * (size_t)NK * NK);
    const int *pos = w->pos;
    if (use_hess) {
        for (int k = 0; k < w->nlp->nnz_hess; k++) {
            int i = pos[w->hr[k]], j = pos[w->hc[k]];
            A[(size_t)i * NK + j] += w->hv[k];
            if (i != j) A[(size_t)j * NK + i] += w->hv[k];
        }
    }
    for (int i = 0; i < N; i++) {
        int p = pos[i];
        A[(size_t)p * NK + p] += Sigma[i] + dw;
    }
    for (int k = 0; k < w->nlp->nnz_jac; k++) {
        int i = pos[N + w->jr[k]], j = pos[w->jc[k]];
        A[(size_t)i * NK + j] += w->jv[k];
        A[(size_t)j * NK + i] += w->jv[k];
    }
    for (int r = 0; r < w->m; r++) {
        int i = pos[N + r];
        if (w->slack_of[r] >= 0) {
            int j = pos[n + w->slack_of[r]];
            A[(size_t)i * NK + j] -= 1.0;
            A[(size_t)j * NK + i] -= 1.0;
        }
        A[(size_t)i * NK + i] -= dc;
    }
    ldl_factor(w->F, w->opt->use_dense_ldl);
    w->nfact++;
}

/* Solve KKT * [dx; dl] = [r1; r2]  (rhs given in original ordering, result too). */
static void kkt_solve(ipm_ws *w, const double *r1, const double *r2, double *dx, double *dl, double *tmp)
{
    const int N = w->N, m = w->m;
    for (int i = 0; i < N; i++) tmp[w->pos[i]] = r1[i];
    for (int i = 0; i < m; i++) tmp[w->pos[N + i]] = r2[i];
    ldl_solve(w->F, tmp);
    for (int i = 0; i < N; i++) dx[i] = tmp[w->pos[i]];
    for (int i = 0; i < m; i++) dl[i] = tmp[w->pos[N + i]];
}

static double barrier_terms(const ipm_ws *w, const double *X, double mu, int *ok)
{
    double s = 0.0;
    *ok = 1;
    for (int i = 0; i < w->N; i++) {
        if (w->hasL[i]) { double d = X[i] - w->XL[i]; if (!(d > 0.0)) { *ok = 0; return 0.0; } s -= log(d); }
        if (w->hasU[i]) { double d = w->XU[i] - X[i]; if (!(d > 0.0)) { *ok = 0; return 0.0; } s -= log(d); }
    }
    return mu * s;
}

static double norm1(const double *v, int n) { double s = 0; for (int i = 0; i < n; i++) s += fabs(v[i]); return s; }
static double norminf(const double *v, int n) { double s = 0; for (int i = 0; i < n; i++) if (fabs(v[i]) > s) s = fabs(v[i]); return s; }

typedef struct { double theta, phi; } filt_entry;

static int filter_ok(const filt_entry *flt, int nf, double theta_max, double theta, double phi)
{
    if (!(theta < theta_max)) return 0;
    for (int i = 0; i < nf; i++)
        if (theta >= flt[i].theta && phi >= flt[i].phi) return 0;
    return 1;
}

int ipm_solve(const ipm_nlp *nlp, const ipm_options *opt, ipm_result *res)
{
    return ipm_solve_from(nlp, opt, NULL, res);
}

int ipm_solve_from(const ipm_nlp *nlp, const ipm_options *opt, const ipm_start *start, ipm_result *res)
{
    const double t_start = cpu_now();
    ipm_ws W; memset(&W, 0, sizeof(W));
    ipm_ws *w = &W;
    w->nlp = nlp; w->opt = opt;
    const int n = nlp->n, m = nlp->m;
    w->n = n; w->m = m;

    /* Ipopt defaults (Waechter & Biegler 2006, Sec. 3 and Table of constants) */
    const double kappa_eps = 10.0, kappa_mu = 0.2, theta_mu = 1.5, tau_min = 0.99;
    const double s_max = 100.0;
    const double gamma_theta = 1e-5, gamma_phi = 1e-8, delta_sw = 1.0, s_theta = 1.1, s_phi = 2.3;
    const double eta_phi = 1e-8, gamma_alpha = 0.05, kappa_soc = 0.99, kappa_sigma = 1e10;
    const double dw_min = 1e-20, dw_0 = 1e-4, dw_max = 1e40, dc_bar = 1e-8, kw_minus = 1.0 / 3.0,
                 kw_plus = 8.0, kw_plus_bar = 100.0, kappa_c = 0.25;
    const double lam_max = 1e3;
    const double eps_mach = 2.220446049250313e-16;

    double *xl = (double *)malloc(sizeof(double) * n), *xu = (double *)malloc(sizeof(double) * n);
    double *glr = (double *)malloc(sizeof(double) * (m + 1)), *gur = (double *)malloc(sizeof(double) * (m + 1));
    nlp->get_bounds(nlp->user, xl, xu, glr, gur);
    w->slack_of = (int *)malloc(sizeof(int) * (m + 1));
    int ns = 0;
    for (int i = 0; i < m; i++) {
        if (glr[i] == gur[i]) w->slack_of[i] = -1; else w->slack_of[i] = ns++;
    }
    w->ns = ns;
    const int N = n + ns, NK = N + m;
    w->N = N; w->NK = NK;

    w->jr = (int *)malloc(sizeof(int) * (nlp->nnz_jac + 1)); w->jc = (int *)malloc(sizeof(int) * (nlp->nnz_jac + 1));
    w->hr = (int *)malloc(sizeof(int) * (nlp->nnz_hess + 1)); w->hc = (int *)malloc(sizeof(int) * (nlp->nnz_hess + 1));
    w->jv = (double *)calloc(nlp->nnz_jac + 1, sizeof(double)); w->hv = (double *)calloc(nlp->nnz_hess + 1, sizeof(double));
    nlp->jac_struct(nlp->user, w->jr, w->jc);
    nlp->hess_struct(nlp->user, w->hr, w->hc);
    w->graw = (double *)calloc(m + 1, sizeof(double));
    w->lam_tmp = (double *)calloc(m + 1, sizeof(double));
    w->sc = (double *)malloc(sizeof(double) * (m + 1));
    w->gl = (double *)malloc(sizeof(double) * (m + 1)); w->gu = (double *)malloc(sizeof(double) * (m + 1));
    w->XL = (double *)malloc(sizeof(double) * N); w->XU = (double *)malloc(sizeof(double) * N);
    w->hasL = (char *)calloc(N, 1); w->hasU = (char *)calloc(N, 1);

    double *X = (double *)calloc(N, sizeof(double)), *Xt = (double *)calloc(N, sizeof(double));
    double *lam = (double *)calloc(m + 1, sizeof(double));
    double *zL = (double *)calloc(N, sizeof(double)), *zU = (double *)calloc(N, sizeof(double));
    double *gradf = (double *)calloc(N, sizeof(double)), *c = (double *)calloc(m + 1, sizeof(double)), *ct = (double *)calloc(m + 1, sizeof(double));
    double *Sigma = (double *)calloc(N, sizeof(double));
    double *r1 = (double *)calloc(N, sizeof(double)), *r2 = (double *)calloc(m + 1, sizeof(double));
    double *dx = (double *)calloc(N, sizeof(double)), *dl = (double *)calloc(m + 1, sizeof(double));
    double *dxs = (double *)calloc(N, sizeof(double)), *dls = (double *)calloc(m + 1, sizeof(double));
    double *dzL = (double *)calloc(N, sizeof(double)), *dzU = (double *)calloc(N, sizeof(double));
    double *tmpN = (double *)calloc(N, sizeof(double)), *tmpK = (double *)calloc(NK, sizeof(double));
    double *csoc = (double *)calloc(m + 1, sizeof(double));
    int filt_cap = 64, nfilt = 0;
    filt_entry *filt = (filt_entry *)malloc(sizeof(filt_entry) * filt_cap);

    int status = IPM_INTERNAL_ERROR;
    int iter = 0;
    double mu = start ? start->mu0 : opt->mu_init;
    int n_inertia = 0, n_resto = 0;
    double E0 = INFINITY;

    /* ---- starting point, pushed into the relaxed bounds ---- */
    nlp->get_start(nlp->user, X);
    w->sf = 1.0;
    for (int i = 0; i < m; i++) w->sc[i] = 1.0;
    for (int i = 0; i < n; i++) {
        w->hasL[i] = xl[i] > -IPM_INF; w->hasU[i] = xu[i] < IPM_INF;
        w->XL[i] = w->hasL[i] ? xl[i] - opt->bound_relax_factor * fmax(1.0, fabs(xl[i])) : -INFINITY;
        w->XU[i] = w->hasU[i] ? xu[i] + opt->bound_relax_factor * fmax(1.0, fabs(xu[i])) : INFINITY;
    }
    /* push x (bound_push / bound_frac, W&B Sec. 3.6) */
    for (int i = 0; i < n; i++) {
        if (w->hasL[i] && w->hasU[i]) {
            double pl = fmin(opt->bound_push * fmax(1.0, fabs(w->XL[i])), opt->bound_frac * (w->XU[i] - w->XL[i]));
            double pu = fmin(opt->bound_push * fmax(1.0, fabs(w->XU[i])), opt->bound_frac * (w->XU[i] - w->XL[i]));
            if (X[i] < w->XL[i] + pl) X[i] = w->XL[i] + pl;
            if (X[i] > w->XU[i] - pu) X[i] = w->XU[i] - pu;
        } else if (w->hasL[i]) {
            double pl = opt->bound_push * fmax(1.0, fabs(w->XL[i]));
            if (X[i] < w->XL[i] + pl) X[i] = w->XL[i] + pl;
        } else if (w->hasU[i]) {
            double pu = opt->bound_push * fmax(1.0, fabs(w->XU[i]));
            if (X[i] > w->XU[i] - pu) X[i] = w->XU[i] - pu;
        }
    }

    /* ---- gradient-based scaling at the (pushed) start point ---- */
    if (opt->nlp_scaling_max_gradient > 0.0) {
        const double gmax = opt->nlp_scaling_max_gradient;
        if (!nlp->eval_grad_f(nlp->user, X, gradf)) { status = IPM_INVALID_NUMBER_DETECTED; goto done; }
        double gn = norminf(gradf, n);
        if (gn > gmax) w->sf = gmax / gn;
        if (!nlp->eval_jac(nlp->user, X, w->jv)) { status = IPM_INVALID_NUMBER_DETECTED; goto done; }
        double *rowmax = (double *)calloc(m + 1, sizeof(double));
        for (int k = 0; k < nlp->nnz_jac; k++) {
            double v = fabs(w->jv[k]);
            if (v > rowmax[w->jr[k]]) rowmax[w->jr[k]] = v;
        }
        for (int i = 0; i < m; i++) if (rowmax[i] > gmax) w->sc[i] = gmax / rowmax[i];
        free(rowmax);
    }
    /* a given start: the scaling stays the cold start's, the iterate is the given one (not pushed) */
    if (start) {
        if (start->sf > 0.0) w->sf = start->sf;
        memcpy(X, start->x0, sizeof(double) * n);
    }
    for (int i = 0; i < m; i++) {
        w->gl[i] = (glr[i] > -IPM_INF) ? w->sc[i] * glr[i] : -INFINITY;
        w->gu[i] = (gur[i] < IPM_INF) ? w->sc[i] * gur[i] : INFINITY;
    }
    /* slack bounds + start */
    if (!nlp->eval_g(nlp->user, X, w->graw)) { status = IPM_INVALID_NUMBER_DETECTED; goto done; }
    for (int i = 0; i < m; i++) {
        int s = w->slack_of[i];
        if (s < 0) continue;
        int j = n + s;
        w->hasL[j] = isfinite(w->gl[i]); w->hasU[j] = isfinite(w->gu[i]);
        w->XL[j] = w->hasL[j] ? w->gl[i] - opt->bound_relax_factor * fmax(1.0, fabs(w->gl[i])) : -INFINITY;
        w->XU[j] = w->hasU[j] ? w->gu[i] + opt->bound_relax_factor * fmax(1.0, fabs(w->gu[i])) : INFINITY;
        double v = w->sc[i] * w->graw[i];
        if (w->hasL[j] && w->hasU[j]) {
            double pl = fmin(opt->bound_push * fmax(1.0, fabs(w->XL[j])), opt->bound_frac * (w->XU[j] - w->XL[j]));
            double pu = fmin(opt->bound_push * fmax(1.0, fabs(w->XU[j])), opt->bound_frac * (w->XU[j] - w->XL[j]));
            if (v < w->XL[j] + pl) v = w->XL[j] + pl;
            if (v > w->XU[j] - pu) v = w->XU[j] - pu;
        } else if (w->hasL[j]) {
            double pl = opt->bound_push * fmax(1.0, fabs(w->XL[j]));
            if (v < w->XL[j] + pl) v = w->XL[j] + pl;
        } else if (w->hasU[j]) {
            double pu = opt->bound_push * fmax(1.0, fabs(w->XU[j]));
            if (v > w->XU[j] - pu) v = w->XU[j] - pu;
        }
        X[j] = v;
    }
    w->nbL = w->nbU = 0;
    for (int i = 0; i < N; i++) { w->nbL += w->hasL[i]; w->nbU += w->hasU[i]; }
    for (int i = 0; i < N; i++) { zL[i] = w->hasL[i] ? 1.0 : 0.0; zU[i] = w->hasU[i] ? 1.0 : 0.0; }
    if (start) {
        for (int i = 0; i < n; i++) {
            if (w->hasL[i]) zL[i] = start->zl0[i];
            if (w->hasU[i]) zU[i] = start->zu0[i];
        }
        memcpy(lam, start->lambda0, sizeof(double) * m);
    }

    /* ---- KKT ordering (RCM on the pattern of the augmented system) ---- */
    {
        int nnz = nlp->nnz_hess + nlp->nnz_jac + ns;
        int *ri = (int *)malloc(sizeof(int) * (nnz + 1)), *ci = (int *)malloc(sizeof(int) * (nnz + 1));
        int q = 0;
        for (int k = 0; k < nlp->nnz_hess; k++) { ri[q] = w->hr[k]; ci[q] = w->hc[k]; q++; }
        for (int k = 0; k < nlp->nnz_jac; k++) { ri[q] = N + w->jr[k]; ci[q] = w->jc[k]; q++; }
        for (int i = 0; i < m; i++) if (w->slack_of[i] >= 0) { ri[q] = N + i; ci[q] = n + w->slack_of[i]; q++; }
        int *order = (int *)malloc(sizeof(int) * NK);
        w->pos = (int *)malloc(sizeof(int) * NK);
        if (opt->use_dense_ldl) for (int i = 0; i < NK; i++) order[i] = i;
        else rcm_order(NK, q, ri, ci, order);
        for (int p = 0; p < NK; p++) w->pos[order[p]] = p;
        free(ri); free(ci); free(order);
        w->F = ldl_alloc(NK);
    }

    double f;
    if (!ev_fc(w, X, &f, c) || !ev_grad(w, X, gradf) || !ev_jac(w, X)) { status = IPM_INVALID_NUMBER_DETECTED; goto done; }

    /* ---- least-squares multiplier start (W&B eq. (36)); a given start brings its own ---- */
    if (m > 0 && !start) {
        for (int i = 0; i < N; i++) Sigma[i] = 1.0;
        kkt_factor(w, Sigma, 0, 0.0, 0.0);
        for (int i = 0; i < N; i++) r1[i] = -(gradf[i] - zL[i] + zU[i]);
        for (int i = 0; i < m; i++) r2[i] = 0.0;
        kkt_solve(w, r1, r2, dx, lam, tmpK);
        int bad = w->F->nzero > 0;
        for (int i = 0; i < m; i++) if (!isfinite(lam[i])) bad = 1;
        if (bad || norminf(lam, m) > lam_max) for (int i = 0; i < m; i++) lam[i] = 0.0;
    }

    double theta0 = norm1(c, m);
    const double theta_max = 1e4 * fmax(1.0, theta0), theta_min = 1e-4 * fmax(1.0, theta0);
    double tau = fmax(tau_min, 1.0 - mu);
    double dw_last = 0.0;
    int n_acceptable = 0;
    int tiny_prev = 0, force_mu = 0;

    for (;;) {
        /* ---- optimality error (W&B eq. (5)) ---- */
        jt_mul(w, lam, tmpN);
        double dual_inf = 0.0, compl0 = 0.0, complmu = 0.0;
        for (int i = 0; i < N; i++) {
            double r = gradf[i] + tmpN[i] - zL[i] + zU[i];
            if (fabs(r) > dual_inf) dual_inf = fabs(r);
            if (w->hasL[i]) { double v = (X[i] - w->XL[i]) * zL[i]; compl0 = fmax(compl0, fabs(v)); complmu = fmax(complmu, fabs(v - mu)); }
            if (w->hasU[i]) { double v = (w->XU[i] - X[i]) * zU[i]; compl0 = fmax(compl0, fabs(v)); complmu = fmax(complmu, fabs(v - mu)); }
        }
        double pr_inf = norminf(c, m);
        double zsum = norm1(zL, N) + norm1(zU, N);
        int nb = w->nbL + w->nbU;
        double s_d = fmax(s_max, (norm1(lam, m) + zsum) / fmax(1, m + nb)) / s_max;
        double s_c = nb ? fmax(s_max, zsum / nb) / s_max : 1.0;
        E0 = fmax(fmax(dual_inf / s_d, pr_inf), compl0 / s_c);
        double Emu = fmax(fmax(dual_inf / s_d, pr_inf), complmu / s_c);

        /* unscaled measures for the absolute tolerances */
        double u_dual = dual_inf / w->sf, u_compl = compl0 / w->sf, u_pr = 0.0;
        for (int i = 0; i < m; i++) u_pr = fmax(u_pr, fabs(c[i]) / w->sc[i]);
        res->dual_inf = u_dual; res->constr_viol = u_pr; res->compl_inf = u_compl;

        if (opt->print_level > 0)
            fprintf(stderr, "it %3d f %.10e pr %.2e du %.2e cmp %.2e mu %.2e E0 %.2e\n", iter, f / w->sf, pr_inf, dual_inf, compl0, mu, E0);

        if (E0 <= opt->tol && u_dual <= opt->dual_inf_tol && u_pr <= opt->constr_viol_tol && u_compl <= opt->compl_inf_tol) {
            status = IPM_SUCCESS; break;
        }
        if (E0 <= opt->acceptable_tol && u_pr <= 1e-2 && u_compl <= 1e-2) n_acceptable++; else n_acceptable = 0;
        if (n_acceptable >= opt->acceptable_iter) { status = IPM_STOP_AT_ACCEPTABLE_POINT; break; }
        if (iter >= opt->max_iter) { status = IPM_MAXITER_EXCEEDED; break; }
        if (cpu_now() - t_start > opt->max_cpu_time) { status = 15; break; }

        /* ---- barrier update (W&B eq. (7), A-3), possibly several times ---- */
        int mu_changed = 0;
        while (Emu <= kappa_eps * mu || force_mu) {
            force_mu = 0;
            double mu_floor = fmin(opt->tol, opt->compl_inf_tol) / (kappa_eps + 1.0);
            double mu_new = fmax(mu_floor, fmin(kappa_mu * mu, pow(mu, theta_mu)));
            if (mu_new >= mu) break;
            mu = mu_new; tau = fmax(tau_min, 1.0 - mu); mu_changed = 1;
            complmu = 0.0;
            for (int i = 0; i < N; i++) {
                if (w->hasL[i]) complmu = fmax(complmu, fabs((X[i] - w->XL[i]) * zL[i] - mu));
                if (w->hasU[i]) complmu = fmax(complmu, fabs((w->XU[i] - X[i]) * zU[i] - mu));
            }
            Emu = fmax(fmax(dual_inf / s_d, pr_inf), complmu / s_c);
        }
        if (mu_changed) nfilt = 0;

        /* ---- search direction (W&B eq. (13)) with inertia correction (Alg. IC) ---- */
        if (!ev_hess(w, X, lam)) { status = IPM_INVALID_NUMBER_DETECTED; break; }
        for (int i = 0; i < N; i++) {
            double s = 0.0;
            if (w->hasL[i]) s += zL[i] / (X[i] - w->XL[i]);
            if (w->hasU[i]) s += zU[i] / (w->XU[i] - X[i]);
            Sigma[i] = s;
        }
        double dw = 0.0, dc = 0.0;
        int ic_fail = 0;
        kkt_factor(w, Sigma, 1, 0.0, 0.0);
        if (!(w->F->npos == N && w->F->nneg == m && w->F->nzero == 0)) {
            n_inertia++;
            if (w->F->nzero > 0) dc = dc_bar * pow(mu, kappa_c);
            dw = (dw_last == 0.0) ? dw_0 : fmax(dw_min, kw_minus * dw_last);
            for (;;) {
                kkt_factor(w, Sigma, 1, dw, dc);
                if (w->F->npos == N && w->F->nneg == m && w->F->nzero == 0) break;
                dw = (dw_last == 0.0) ? kw_plus_bar * dw : kw_plus * dw;
                if (dw > dw_max) { ic_fail = 1; break; }
            }
            if (!ic_fail) dw_last = dw;
        }
        if (ic_fail) { status = IPM_ERROR_IN_STEP_COMPUTATION; break; }

        /* rhs: -(grad phi_mu + J^T lam), -c */
        double gphi_d = 0.0;
        for (int i = 0; i < N; i++) {
            double gp = gradf[i];
            if (w->hasL[i]) gp -= mu / (X[i] - w->XL[i]);
            if (w->hasU[i]) gp += mu / (w->XU[i] - X[i]);
            tmpN[i] = gp;                       /* grad phi_mu */
        }
        {
            double *jtl = dxs; /* scratch */
            jt_mul(w, lam, jtl);
            for (int i = 0; i < N; i++) r1[i] = -(tmpN[i] + jtl[i]);
            for (int i = 0; i < m; i++) r2[i] = -c[i];
        }
        kkt_solve(w, r1, r2, dx, dl, tmpK);
        {
            int bad = 0;
            for (int i = 0; i < N; i++) if (!isfinite(dx[i])) bad = 1;
            for (int i = 0; i < m; i++) if (!isfinite(dl[i])) bad = 1;
            if (bad) { status = IPM_ERROR_IN_STEP_COMPUTATION; break; }
        }
        for (int i = 0; i < N; i++) {
            gphi_d += tmpN[i] * dx[i];
            dzL[i] = w->hasL[i] ? mu / (X[i] - w->XL[i]) - zL[i] - zL[i] / (X[i] - w->XL[i]) * dx[i] : 0.0;
            dzU[i] = w->hasU[i] ? mu / (w->XU[i] - X[i]) - zU[i] + zU[i] / (w->XU[i] - X[i]) * dx[i] : 0.0;
        }

        /* tiny step (W&B Sec. 3.9): relative step below 10 eps */
        int tiny = 1;
        for (int i = 0; i < N; i++) if (fabs(dx[i]) / (1.0 + fabs(X[i])) > 10.0 * eps_mach) { tiny = 0; break; }

        /* ---- fraction to the boundary (W&B eq. (15)) ---- */
        double a_max = 1.0, a_z = 1.0;
        for (int i = 0; i < N; i++) {
            if (w->hasL[i] && dx[i] < 0.0) a_max = fmin(a_max, -tau * (X[i] - w->XL[i]) / dx[i]);
            if (w->hasU[i] && dx[i] > 0.0) a_max = fmin(a_max, tau * (w->XU[i] - X[i]) / dx[i]);
            if (w->hasL[i] && dzL[i] < 0.0) a_z = fmin(a_z, -tau * zL[i] / dzL[i]);
            if (w->hasU[i] && dzU[i] < 0.0) a_z = fmin(a_z, -tau * zU[i] / dzU[i]);
        }

        /* ---- filter line search (A-5) ---- */
        int okb;
        double theta = norm1(c, m);
        double phi = f + barrier_terms(w, X, mu, &okb);
        double a_min;
        if (gphi_d < 0.0 && theta <= theta_min)
            a_min = gamma_alpha * fmin(fmin(gamma_theta, gamma_phi * theta / (-gphi_d)), delta_sw * pow(theta, s_theta) / pow(-gphi_d, s_phi));
        else if (gphi_d < 0.0)
            a_min = gamma_alpha * fmin(gamma_theta, gamma_phi * theta / (-gphi_d));
        else
            a_min = gamma_alpha * gamma_theta;

        double alpha = a_max;
        int accepted = 0, first = 1, armijo_step = 0;
        if (tiny) {
            if (tiny_prev) {
                double mu_floor = fmin(opt->tol, opt->compl_inf_tol) / (kappa_eps + 1.0);
                if (mu <= mu_floor * (1.0 + 1e-12)) { status = IPM_STOP_AT_TINY_STEP; break; }
                force_mu = 1;
            }
            tiny_prev = 1;
            accepted = 1; armijo_step = 1; /* take the step without a filter test */
        } else tiny_prev = 0;
        double f_t = f, theta_t = theta;
        const double *dacc = dx;
        double alpha_acc = alpha;
        while (!accepted && (alpha >= a_min || first) && alpha > 1e-40) {
            for (int i = 0; i < N; i++) Xt[i] = X[i] + alpha * dx[i];
            int ok = ev_fc(w, Xt, &f_t, ct);
            double phi_t = INFINITY;
            if (ok) { double b = barrier_terms(w, Xt, mu, &okb); if (okb) phi_t = f_t + b; else ok = 0; }
            theta_t = ok ? norm1(ct, m) : INFINITY;
            int sw = (gphi_d < 0.0) && (alpha * pow(-gphi_d, s_phi) > delta_sw * pow(theta, s_theta));
            int acc = 0;
            if (ok && filter_ok(filt, nfilt, theta_max, theta_t, phi_t)) {
                if (theta <= theta_min && sw) {
                    if (phi_t - phi - 10.0 * eps_mach * fabs(phi) <= eta_phi * alpha * gphi_d) { acc = 1; armijo_step = 1; }
                } else {
                    if (theta_t <= (1.0 - gamma_theta) * theta || phi_t - 10.0 * eps_mach * fabs(phi) <= phi - gamma_phi * theta) { acc = 1; armijo_step = 0; }
                }
            }
            if (acc) { accepted = 1; dacc = dx; alpha_acc = alpha; break; }

            /* ---- second-order correction (A-5.5 .. A-5.9) ---- */
            if (first && ok && theta_t >= theta && opt->max_soc > 0) {
                double theta_soc_old = theta;
                for (int i = 0; i < m; i++) csoc[i] = alpha * c[i] + ct[i];
                for (int p = 0; p < opt->max_soc; p++) {
                    for (int i = 0; i < m; i++) r2[i] = -csoc[i];
                    kkt_solve(w, r1, r2, dxs, dls, tmpK);
                    double a_soc = 1.0;
                    for (int i = 0; i < N; i++) {
                        if (w->hasL[i] && dxs[i] < 0.0) a_soc = fmin(a_soc, -tau * (X[i] - w->XL[i]) / dxs[i]);
                        if (w->hasU[i] && dxs[i] > 0.0) a_soc = fmin(a_soc, tau * (w->XU[i] - X[i]) / dxs[i]);
                    }
                    for (int i = 0; i < N; i++) Xt[i] = X[i] + a_soc * dxs[i];
                    double f_s; int oks = ev_fc(w, Xt, &f_s, ct);
                    if (!oks) break;
                    double bs = barrier_terms(w, Xt, mu, &okb);
                    if (!okb) break;
                    double phi_s = f_s + bs, theta_s = norm1(ct, m);
                    int accs = 0;
                    if (filter_ok(filt, nfilt, theta_max, theta_s, phi_s)) {
                        if (theta <= theta_min && sw) {
                            if (phi_s - phi - 10.0 * eps_mach * fabs(phi) <= eta_phi * alpha * gphi_d) { accs = 1; armijo_step = 1; }
                        } else {
                            if (theta_s <= (1.0 - gamma_theta) * theta || phi_s - 10.0 * eps_mach * fabs(phi) <= phi - gamma_phi * theta) { accs = 1; armijo_step = 0; }
                        }
                    }
                    if (accs) { accepted = 1; dacc = dxs; alpha_acc = a_soc; f_t = f_s; theta_t = theta_s; break; }
                    if (theta_s > kappa_soc * theta_soc_old) break;
                    theta_soc_old = theta_s;
                    for (int i = 0; i < m; i++) csoc[i] = a_soc * csoc[i] + ct[i];
                }
                if (accepted) break;
            }
            first = 0;
            alpha *= 0.5;
        }

        if (!accepted) {
            /* ---- stand-in for Ipopt's restoration phase: reduce theta by
             * min-norm Gauss-Newton steps until the point is acceptable to the
             * filter and theta dropped by 10 % (kappa_resto = 0.9). ---- */
            n_resto++;
            if (theta <= 1e-13 * fmax(1.0, theta0)) { status = IPM_STOP_AT_TINY_STEP; break; }
            /* augment filter with current point first (W&B A-9) */
            if (nfilt == filt_cap) { filt_cap *= 2; filt = (filt_entry *)realloc(filt, sizeof(filt_entry) * filt_cap); }
            filt[nfilt].theta = (1.0 - gamma_theta) * theta; filt[nfilt].phi = phi - gamma_phi * theta; nfilt++;
            int resto_ok = 0;
            double theta_r = theta;
            for (int rit = 0; rit < 50 && !resto_ok; rit++) {
                for (int i = 0; i < N; i++) Sigma[i] = 1.0;
                kkt_factor(w, Sigma, 0, 0.0, 1e-10);
                for (int i = 0; i < N; i++) r1[i] = 0.0;
                for (int i = 0; i < m; i++) r2[i] = -c[i];
                kkt_solve(w, r1, r2, dx, dl, tmpK);
                double a = 1.0;
                for (int i = 0; i < N; i++) {
                    if (w->hasL[i] && dx[i] < 0.0) a = fmin(a, -tau * (X[i] - w->XL[i]) / dx[i]);
                    if (w->hasU[i] && dx[i] > 0.0) a = fmin(a, tau * (w->XU[i] - X[i]) / dx[i]);
                }
                int moved = 0;
                for (int bt = 0; bt < 30; bt++, a *= 0.5) {
                    for (int i = 0; i < N; i++) Xt[i] = X[i] + a * dx[i];
                    double ft; if (!ev_fc(w, Xt, &ft, ct)) continue;
                    double th = norm1(ct, m);
                    if (th < (1.0 - 1e-4 * a) * theta_r) {
                        memcpy(X, Xt, sizeof(double) * N); memcpy(c, ct, sizeof(double) * m);
                        f = ft; theta_r = th; moved = 1; break;
                    }
                }
                if (!moved) break;
                if (!ev_jac(w, X)) break;
                double b = barrier_terms(w, X, mu, &okb);
                if (theta_r <= 0.9 * theta && okb && filter_ok(filt, nfilt, theta_max, theta_r, f + b)) resto_ok = 1;
            }
            if (!resto_ok) { status = (theta_r > 1e-6) ? IPM_LOCAL_INFEASIBILITY : IPM_RESTORATION_FAILURE; break; }
            if (!ev_grad(w, X, gradf) || !ev_jac(w, X)) { status = IPM_INVALID_NUMBER_DETECTED; break; }
            /* reset bound multipliers as Ipopt does after restoration */
            for (int i = 0; i < N; i++) {
                if (w->hasL[i]) zL[i] = fmax(fmin(zL[i], kappa_sigma * mu / (X[i] - w->XL[i])), mu / (kappa_sigma * (X[i] - w->XL[i])));
                if (w->hasU[i]) zU[i] = fmax(fmin(zU[i], kappa_sigma * mu / (w->XU[i] - X[i])), mu / (kappa_sigma * (w->XU[i] - X[i])));
            }
            iter++;
            continue;
        }

        /* ---- accept (A-6, A-7) ---- */
        if (dacc == dxs) {
            /* Ipopt replaces the whole primal-dual step by the corrected one (actual_delta = delta_soc in
             * TrySecondOrderCorrection) before it computes the dual step size: dz and alpha_z follow dxs. */
            a_z = 1.0;
            for (int i = 0; i < N; i++) {
                dzL[i] = w->hasL[i] ? mu / (X[i] - w->XL[i]) - zL[i] - zL[i] / (X[i] - w->XL[i]) * dxs[i] : 0.0;
                dzU[i] = w->hasU[i] ? mu / (w->XU[i] - X[i]) - zU[i] + zU[i] / (w->XU[i] - X[i]) * dxs[i] : 0.0;
                if (w->hasL[i] && dzL[i] < 0.0) a_z = fmin(a_z, -tau * zL[i] / dzL[i]);
                if (w->hasU[i] && dzU[i] < 0.0) a_z = fmin(a_z, -tau * zU[i] / dzU[i]);
            }
        }
        if (!armijo_step) {
            if (nfilt == filt_cap) { filt_cap *= 2; filt = (filt_entry *)realloc(filt, sizeof(filt_entry) * filt_cap); }
            filt[nfilt].theta = (1.0 - gamma_theta) * theta; filt[nfilt].phi = phi - gamma_phi * theta; nfilt++;
        }
        for (int i = 0; i < N; i++) X[i] += alpha_acc * dacc[i];
        {
            const double *dlacc = (dacc == dx) ? dl : dls;
            for (int i = 0; i < m; i++) lam[i] += alpha_acc * dlacc[i];
        }
        for (int i = 0; i < N; i++) {
            if (w->hasL[i]) {
                zL[i] += a_z * dzL[i];
                double s = X[i] - w->XL[i];
                zL[i] = fmax(fmin(zL[i], kappa_sigma * mu / s), mu / (kappa_sigma * s));
            }
            if (w->hasU[i]) {
                zU[i] += a_z * dzU[i];
                double s = w->XU[i] - X[i];
                zU[i] = fmax(fmin(zU[i], kappa_sigma * mu / s), mu / (kappa_sigma * s));
            }
        }
        if (!ev_fc(w, X, &f, c) || !ev_grad(w, X, gradf) || !ev_jac(w, X)) { status = IPM_INVALID_NUMBER_DETECTED; break; }
        iter++;
    }

done:
    res->status = status;
    res->iters = iter;
    res->kkt_error = E0;
    res->mu = mu;
    res->n_inertia_corrections = n_inertia;
    res->n_restorations = n_resto;
    res->n_factorizations = w->nfact;
    {
        double fr = NAN;
        nlp->eval_f(nlp->user, X, &fr);
        res->obj = fr;
        if (res->g) { nlp->eval_g(nlp->user, X, w->graw); memcpy(res->g, w->graw, sizeof(double) * m); }
        if (res->x) memcpy(res->x, X, sizeof(double) * n);
        /* unscale multipliers: lambda_i * sc_i / sf, z / sf */
        if (res->lambda) for (int i = 0; i < m; i++) res->lambda[i] = lam[i] * w->sc[i] / w->sf;
        if (res->zl) for (int i = 0; i < n; i++) res->zl[i] = zL[i] / w->sf;
        if (res->zu) for (int i = 0; i < n; i++) res->zu[i] = zU[i] / w->sf;
    }
    free(xl); free(xu); free(glr); free(gur);
    free(w->slack_of); free(w->jr); free(w->jc); free(w->hr); free(w->hc); free(w->jv); free(w->hv);
    free(w->graw); free(w->lam_tmp); free(w->sc); free(w->gl); free(w->gu); free(w->XL); free(w->XU);
    free(w->hasL); free(w->hasU); free(w->pos); ldl_free(w->F);
    free(X); free(Xt); free(lam); free(zL); free(zU); free(gradf); free(c); free(ct); free(Sigma);
    free(r1); free(r2); free(dx); free(dl); free(dxs); free(dls); free(dzL); free(dzU); free(tmpN); free(tmpK);
    free(csoc); free(filt);
    return status;
}
