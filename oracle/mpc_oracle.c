/*
 * oracle/mpc_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.  See mpc_oracle.h.
 *
 * Variable layout follows mpc_ros/src/mpc_planner.cpp:232-239 (component
 * major): x[0,N) y[N,2N) theta[2N,3N) v[3N,4N) cte[4N,5N) etheta[5N,6N)
 * w[6N,7N-1) a[7N-1,8N-2).  Constraint row i = fg index 1+i (:153-158, :208-215).
 */
#include "mpc_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

void mpc_oracle_params_yaml_default(mpc_oracle_params *p)
{
    /* mpc_ros/params/mpc_params.yaml:9-25 */
    p->mpc_steps = 20;
    p->dt = 0.1;            /* 1 / controller_freq */
    p->ref_cte = 0.0; p->ref_vel = 0.5; p->ref_etheta = 0.0;
    p->w_cte = 100.0; p->w_etheta = 0.0; p->w_vel = 1000.0;
    p->w_angvel = 100.0; p->w_angvel_d = 0.0; p->w_accel = 50.0; p->w_accel_d = 0.0;
    p->max_angvel = 1.5; p->max_throttle = 1.0; p->bound_value = 1.0e3;
}

int mpc_oracle_nvars(int N) { return 6 * N + 2 * (N - 1); }   /* mpc_planner.cpp:281 */
int mpc_oracle_ncons(int N) { return 6 * N; }                 /* mpc_planner.cpp:284 */

/* CppAD::pow(x, int) is repeated multiplication (cppad/utility/pow_int.hpp:115-137) */
static double powi(double x, int e) { double r = 1.0; for (int i = 0; i < e; i++) r *= x; return r; }

static double poly(const double *c, int nc, double x)      /* mpc_planner.cpp:186-190 */
{ double s = 0.0; for (int i = 0; i < nc; i++) s += c[i] * powi(x, i); return s; }
static double dpoly(const double *c, int nc, double x)
{ double s = 0.0; for (int i = 1; i < nc; i++) s += i * c[i] * powi(x, i - 1); return s; }
static double ddpoly(const double *c, int nc, double x)
{ double s = 0.0; for (int i = 2; i < nc; i++) s += i * (i - 1) * c[i] * powi(x, i - 2); return s; }

#define LAYOUT(N) \
    const int xs = 0, ys = N, ts = 2 * N, vs = 3 * N, cs = 4 * N, es = 5 * N, ws = 6 * N, as = 7 * N - 1; \
    (void)xs; (void)ys; (void)ts; (void)vs; (void)cs; (void)es; (void)ws; (void)as;

void mpc_oracle_eval_fg(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                        const double *z, double *f, double *g)
{
    const int N = p->mpc_steps; LAYOUT(N)
    const double dt = p->dt;
    if (f) {
        double s = 0.0;
        for (int i = 0; i < N; i++) {                       /* mpc_planner.cpp:122-127 */
            s += p->w_cte * powi(z[cs + i] - p->ref_cte, 2);
            s += p->w_etheta * powi(z[es + i] - p->ref_etheta, 2);
            s += p->w_vel * powi(z[vs + i] - p->ref_vel, 2);
        }
        for (int i = 0; i < N - 1; i++) {                   /* :137-140 */
            s += p->w_angvel * powi(z[ws + i], 2);
            s += p->w_accel * powi(z[as + i], 2);
        }
        for (int i = 0; i < N - 2; i++) {                   /* :144-147 */
            s += p->w_angvel_d * powi(z[ws + i + 1] - z[ws + i], 2);
            s += p->w_accel_d * powi(z[as + i + 1] - z[as + i], 2);
        }
        *f = s;
    }
    if (g) {
        g[xs] = z[xs]; g[ys] = z[ys]; g[ts] = z[ts];        /* :153-158 */
        g[vs] = z[vs]; g[cs] = z[cs]; g[es] = z[es];
        for (int i = 0; i < N - 1; i++) {                   /* :161-216 */
            const double x0 = z[xs + i], y0 = z[ys + i], th0 = z[ts + i], v0 = z[vs + i], e0 = z[es + i];
            const double w0 = z[ws + i], a0 = z[as + i];
            const double f0 = poly(coeffs, ncoef, x0);
            g[xs + 1 + i] = z[xs + i + 1] - (x0 + v0 * cos(th0) * dt);
            g[ys + 1 + i] = z[ys + i + 1] - (y0 + v0 * sin(th0) * dt);
            g[ts + 1 + i] = z[ts + i + 1] - (th0 + w0 * dt);
            g[vs + 1 + i] = z[vs + i + 1] - (v0 + a0 * dt);
            g[cs + 1 + i] = z[cs + i + 1] - ((f0 - y0) + (v0 * sin(e0) * dt));
            g[es + 1 + i] = z[es + i + 1] - (e0 + w0 * dt);
        }
    }
}

void mpc_oracle_eval_grad(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                          const double *z, double *gr)
{
    (void)coeffs; (void)ncoef;
    const int N = p->mpc_steps; LAYOUT(N)
    const int n = mpc_oracle_nvars(N);
    for (int i = 0; i < n; i++) gr[i] = 0.0;
    for (int i = 0; i < N; i++) {
        gr[cs + i] += 2.0 * p->w_cte * (z[cs + i] - p->ref_cte);
        gr[es + i] += 2.0 * p->w_etheta * (z[es + i] - p->ref_etheta);
        gr[vs + i] += 2.0 * p->w_vel * (z[vs + i] - p->ref_vel);
    }
    for (int i = 0; i < N - 1; i++) {
        gr[ws + i] += 2.0 * p->w_angvel * z[ws + i];
        gr[as + i] += 2.0 * p->w_accel * z[as + i];
    }
    for (int i = 0; i < N - 2; i++) {
        const double dw = z[ws + i + 1] - z[ws + i], da = z[as + i + 1] - z[as + i];
        gr[ws + i + 1] += 2.0 * p->w_angvel_d * dw; gr[ws + i] -= 2.0 * p->w_angvel_d * dw;
        gr[as + i + 1] += 2.0 * p->w_accel_d * da;  gr[as + i] -= 2.0 * p->w_accel_d * da;
    }
}

int mpc_oracle_nnz_jac(int N) { return 22 * (N - 1) + 6; }

/* COO Jacobian, fixed order: 6 initial rows, then per interval the 22 entries of SURVEY section 0. */
static void jac_coo(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                    const double *z, int *ir, int *jc, double *val)
{
    const int N = p->mpc_steps; LAYOUT(N)
    const double dt = p->dt;
    int q = 0;
#define PUT(r, c, v) do { if (ir) { ir[q] = (r); jc[q] = (c); } if (val) val[q] = (v); q++; } while (0)
    const int comp[6] = { xs, ys, ts, vs, cs, es };
    for (int k = 0; k < 6; k++) PUT(comp[k], comp[k], 1.0);
    for (int i = 0; i < N - 1; i++) {
        double x0 = 0, th0 = 0, v0 = 0, e0 = 0;
        if (z) { x0 = z[xs + i]; th0 = z[ts + i]; v0 = z[vs + i]; e0 = z[es + i]; }
        const double s = sin(th0), c = cos(th0), se = sin(e0), ce = cos(e0);
        const double dp = z ? dpoly(coeffs, ncoef, x0) : 0.0;
        PUT(xs + 1 + i, xs + i + 1, 1.0); PUT(xs + 1 + i, xs + i, -1.0);
        PUT(xs + 1 + i, vs + i, -c * dt); PUT(xs + 1 + i, ts + i, v0 * s * dt);
        PUT(ys + 1 + i, ys + i + 1, 1.0); PUT(ys + 1 + i, ys + i, -1.0);
        PUT(ys + 1 + i, vs + i, -s * dt); PUT(ys + 1 + i, ts + i, -v0 * c * dt);
        PUT(ts + 1 + i, ts + i + 1, 1.0); PUT(ts + 1 + i, ts + i, -1.0); PUT(ts + 1 + i, ws + i, -dt);
        PUT(vs + 1 + i, vs + i + 1, 1.0); PUT(vs + 1 + i, vs + i, -1.0); PUT(vs + 1 + i, as + i, -dt);
        PUT(cs + 1 + i, cs + i + 1, 1.0); PUT(cs + 1 + i, xs + i, -dp); PUT(cs + 1 + i, ys + i, 1.0);
        PUT(cs + 1 + i, vs + i, -se * dt); PUT(cs + 1 + i, es + i, -v0 * ce * dt);
        PUT(es + 1 + i, es + i + 1, 1.0); PUT(es + 1 + i, es + i, -1.0); PUT(es + 1 + i, ws + i, -dt);
    }
#undef PUT
}

int mpc_oracle_nnz_hess(const mpc_oracle_params *p)
{
    const int N = p->mpc_steps;
    /* diag: cte N, etheta N, v N, w N-1, a N-1, x N-1, theta N-1; off: (v,theta),(etheta,v) N-1 each; rate N-2 each */
    return 3 * N + 4 * (N - 1) + 2 * (N - 1) + 2 * (N - 2);
}

/* COO lower-triangular Hessian of sigma f + lambda^T g. */
static void hess_coo(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                     const double *z, double sigma, const double *lam, int *ir, int *jc, double *val)
{
    const int N = p->mpc_steps; LAYOUT(N)
    const double dt = p->dt;
    int q = 0;
#define PUT(r, c, v) do { if (ir) { ir[q] = (r); jc[q] = (c); } if (val) val[q] = (v); q++; } while (0)
    for (int i = 0; i < N; i++) {
        double hee = 2.0 * sigma * p->w_etheta;
        if (i < N - 1 && z) hee += lam[cs + 1 + i] * z[vs + i] * sin(z[es + i]) * dt;
        PUT(cs + i, cs + i, 2.0 * sigma * p->w_cte);
        PUT(es + i, es + i, hee);
        PUT(vs + i, vs + i, 2.0 * sigma * p->w_vel);
    }
    for (int i = 0; i < N - 1; i++) {
        double rw = 2.0 * sigma * p->w_angvel, ra = 2.0 * sigma * p->w_accel;
        /* each control appears in the rate terms (i-1,i) and (i,i+1), indices within [0, N-2] */
        int cnt = 0;
        if (i >= 1) cnt++;
        if (i <= N - 3) cnt++;
        rw += 2.0 * sigma * p->w_angvel_d * cnt; ra += 2.0 * sigma * p->w_accel_d * cnt;
        PUT(ws + i, ws + i, rw);
        PUT(as + i, as + i, ra);
        double hxx = 0, htt = 0, hvt = 0, hev = 0;
        if (z) {
            const double x0 = z[xs + i], th0 = z[ts + i], v0 = z[vs + i], e0 = z[es + i];
            const double lx = lam[xs + 1 + i], ly = lam[ys + 1 + i], lc = lam[cs + 1 + i];
            hxx = -lc * ddpoly(coeffs, ncoef, x0);
            htt = lx * v0 * cos(th0) * dt + ly * v0 * sin(th0) * dt;
            hvt = lx * sin(th0) * dt - ly * cos(th0) * dt;
            hev = -lc * cos(e0) * dt;
        }
        PUT(xs + i, xs + i, hxx);
        PUT(ts + i, ts + i, htt);
        PUT(vs + i, ts + i, hvt);
        PUT(es + i, vs + i, hev);
    }
    for (int i = 0; i < N - 2; i++) {
        PUT(ws + i + 1, ws + i, -2.0 * sigma * p->w_angvel_d);
        PUT(as + i + 1, as + i, -2.0 * sigma * p->w_accel_d);
    }
#undef PUT
}

void mpc_oracle_eval_jac_dense(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                               const double *z, double *J)
{
    const int N = p->mpc_steps, n = mpc_oracle_nvars(N), m = mpc_oracle_ncons(N), nnz = mpc_oracle_nnz_jac(N);
    int *ir = (int *)malloc(sizeof(int) * nnz), *jc = (int *)malloc(sizeof(int) * nnz);
    double *v = (double *)malloc(sizeof(double) * nnz);
    jac_coo(p, coeffs, ncoef, z, ir, jc, v);
    memset(J, 0, sizeof(double) * (size_t)m * n);
    for (int k = 0; k < nnz; k++) J[(size_t)ir[k] * n + jc[k]] += v[k];
    free(ir); free(jc); free(v);
}

void mpc_oracle_eval_hess_dense(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                                const double *z, double sigma, const double *lambda, double *H)
{
    const int N = p->mpc_steps, n = mpc_oracle_nvars(N), nnz = mpc_oracle_nnz_hess(p);
    int *ir = (int *)malloc(sizeof(int) * nnz), *jc = (int *)malloc(sizeof(int) * nnz);
    double *v = (double *)malloc(sizeof(double) * nnz);
    hess_coo(p, coeffs, ncoef, z, sigma, lambda, ir, jc, v);
    memset(H, 0, sizeof(double) * (size_t)n * n);
    for (int k = 0; k < nnz; k++) {
        H[(size_t)ir[k] * n + jc[k]] += v[k];
        if (ir[k] != jc[k]) H[(size_t)jc[k] * n + ir[k]] += v[k];
    }
    free(ir); free(jc); free(v);
}

/* ---- NLP adapter for oracle/ipm.c ---- */
typedef struct {
    const mpc_oracle_params *p;
    const double *coeffs; int ncoef;
    const double *state;
} nlp_ctx;

static int cb_bounds(void *u, double *xl, double *xu, double *gl, double *gu)
{
    nlp_ctx *c = (nlp_ctx *)u; const mpc_oracle_params *p = c->p;
    const int N = p->mpc_steps; LAYOUT(N)
    const int n = mpc_oracle_nvars(N), m = mpc_oracle_ncons(N);
    for (int i = 0; i < ws; i++) { xl[i] = -p->bound_value; xu[i] = p->bound_value; }     /* :308-312 */
    for (int i = ws; i < as; i++) { xl[i] = -p->max_angvel; xu[i] = p->max_angvel; }       /* :315-319 */
    for (int i = as; i < n; i++) { xl[i] = -p->max_throttle; xu[i] = p->max_throttle; }    /* :321-325 */
    for (int i = 0; i < m; i++) { gl[i] = 0.0; gu[i] = 0.0; }                              /* :332-336 */
    const int comp[6] = { xs, ys, ts, vs, cs, es };
    for (int k = 0; k < 6; k++) { gl[comp[k]] = c->state[k]; gu[comp[k]] = c->state[k]; } /* :337-348 */
    return 1;
}
static int cb_start(void *u, double *x0)
{
    nlp_ctx *c = (nlp_ctx *)u; const int N = c->p->mpc_steps; LAYOUT(N)
    const int n = mpc_oracle_nvars(N);
    for (int i = 0; i < n; i++) x0[i] = 0.0;                                               /* :288-292 */
    const int comp[6] = { xs, ys, ts, vs, cs, es };
    for (int k = 0; k < 6; k++) x0[comp[k]] = c->state[k];                                 /* :295-300 */
    return 1;
}
static int cb_f(void *u, const double *x, double *f)
{ nlp_ctx *c = (nlp_ctx *)u; mpc_oracle_eval_fg(c->p, c->coeffs, c->ncoef, x, f, NULL); return 1; }
static int cb_grad(void *u, const double *x, double *g)
{ nlp_ctx *c = (nlp_ctx *)u; mpc_oracle_eval_grad(c->p, c->coeffs, c->ncoef, x, g); return 1; }
static int cb_g(void *u, const double *x, double *g)
{ nlp_ctx *c = (nlp_ctx *)u; mpc_oracle_eval_fg(c->p, c->coeffs, c->ncoef, x, NULL, g); return 1; }
static int cb_jstruct(void *u, int *ir, int *jc)
{ nlp_ctx *c = (nlp_ctx *)u; jac_coo(c->p, c->coeffs, c->ncoef, NULL, ir, jc, NULL); return 1; }
static int cb_jac(void *u, const double *x, double *v)
{ nlp_ctx *c = (nlp_ctx *)u; jac_coo(c->p, c->coeffs, c->ncoef, x, NULL, NULL, v); return 1; }
static int cb_hstruct(void *u, int *ir, int *jc)
{ nlp_ctx *c = (nlp_ctx *)u; hess_coo(c->p, c->coeffs, c->ncoef, NULL, 1.0, NULL, ir, jc, NULL); return 1; }
static int cb_hess(void *u, const double *x, double sigma, const double *lam, double *v)
{ nlp_ctx *c = (nlp_ctx *)u; hess_coo(c->p, c->coeffs, c->ncoef, x, sigma, lam, NULL, NULL, v); return 1; }

static int solve_from(const mpc_oracle_params *p, const double *state6, const double *coeffs, int ncoef,
                      const ipm_options *opt_in, const ipm_start *start, double *u0, double *pred, double *sol,
                      double *lambda, double *zl, double *zu, mpc_oracle_result *out)
{
    const int N = p->mpc_steps; LAYOUT(N)
    const int n = mpc_oracle_nvars(N), m = mpc_oracle_ncons(N);
    nlp_ctx ctx = { p, coeffs, ncoef, state6 };
    ipm_nlp nlp;
    nlp.n = n; nlp.m = m; nlp.nnz_jac = mpc_oracle_nnz_jac(N); nlp.nnz_hess = mpc_oracle_nnz_hess(p);
    nlp.user = &ctx;
    nlp.get_bounds = cb_bounds; nlp.get_start = cb_start; nlp.eval_f = cb_f; nlp.eval_grad_f = cb_grad;
    nlp.eval_g = cb_g; nlp.jac_struct = cb_jstruct; nlp.eval_jac = cb_jac; nlp.hess_struct = cb_hstruct;
    nlp.eval_hess = cb_hess;
    ipm_options opt;
    if (opt_in) opt = *opt_in; else ipm_default_options(&opt);
    ipm_result r; memset(&r, 0, sizeof(r));
    double *x = (double *)malloc(sizeof(double) * n);
    r.x = x; r.lambda = lambda; r.zl = zl; r.zu = zu; r.g = NULL;
    int st = ipm_solve_from(&nlp, &opt, start, &r);
    if (u0) { u0[0] = x[ws]; u0[1] = x[as]; }                                              /* :399-400 */
    if (pred) for (int i = 0; i < N; i++) { pred[i] = x[xs + i]; pred[N + i] = x[ys + i]; pred[2 * N + i] = x[ts + i]; } /* :391-396 */
    if (sol) memcpy(sol, x, sizeof(double) * n);
    if (out) {
        out->status = r.status; out->iters = r.iters; out->obj = r.obj; out->kkt_error = r.kkt_error;
        out->dual_inf = r.dual_inf; out->constr_viol = r.constr_viol; out->compl_inf = r.compl_inf;
        out->n_inertia_corrections = r.n_inertia_corrections; out->n_restorations = r.n_restorations;
    }
    free(x);
    return st;
}

int mpc_oracle_solve(const mpc_oracle_params *p, const double *state6, const double *coeffs, int ncoef,
                     const ipm_options *opt, double *u0, double *pred, double *sol, double *lambda,
                     double *zl, double *zu, mpc_oracle_result *out)
{
    return solve_from(p, state6, coeffs, ncoef, opt, NULL, u0, pred, sol, lambda, zl, zu, out);
}

int mpc_oracle_solve_warm(const mpc_oracle_params *p, const double *state6, const double *coeffs, int ncoef,
                          const ipm_options *opt_in, const double *rec, double warm_mu,
                          double *u0, double *pred, double *sol, double *lambda, double *zl, double *zu,
                          mpc_oracle_result *out)
{
    if (!(p->bound_value >= 1e19)) return -1;      /* the record carries no state-bound multipliers */
    const int N = p->mpc_steps; LAYOUT(N)
    const int n = mpc_oracle_nvars(N), m = mpc_oracle_ncons(N), nu = N - 1;
    const int rl = n, rz = n + m;                   /* record: primal, lambda, zL_w, zL_a, zU_w, zU_a */
    ipm_options opt;
    if (opt_in) opt = *opt_in; else ipm_default_options(&opt);
    double *x = (double *)calloc(n, sizeof(double)), *gr = (double *)malloc(sizeof(double) * n);
    double *lam = (double *)malloc(sizeof(double) * m);
    double *zl0 = (double *)calloc(n, sizeof(double)), *zu0 = (double *)calloc(n, sizeof(double));

    /* objective scaling of the cold start (cb_start's point; no state bounds, so nothing is pushed) */
    const int comp[6] = { xs, ys, ts, vs, cs, es };
    for (int k = 0; k < 6; k++) x[comp[k]] = state6[k];
    mpc_oracle_eval_grad(p, coeffs, ncoef, x, gr);
    double gn = 0.0;
    for (int i = 0; i < n; i++) gn = fmax(gn, fabs(gr[i]));
    const double sf = (opt.nlp_scaling_max_gradient > 0.0 && gn > opt.nlp_scaling_max_gradient)
                      ? opt.nlp_scaling_max_gradient / gn : 1.0;

    /* controls from the record, clipped 1e-3 U inside the relaxed bounds U */
    const double Uw = p->max_angvel + opt.bound_relax_factor * fmax(1.0, p->max_angvel);
    const double Ua = p->max_throttle + opt.bound_relax_factor * fmax(1.0, p->max_throttle);
    for (int k = 0; k < nu; k++) {
        x[ws + k] = fmax(fmin(rec[ws + k], Uw - 1e-3 * Uw), -Uw + 1e-3 * Uw);
        x[as + k] = fmax(fmin(rec[as + k], Ua - 1e-3 * Ua), -Ua + 1e-3 * Ua);
    }
    /* states: the model rolled out from state6 with those controls, as eval_fg writes the dynamics */
    for (int i = 0; i < N - 1; i++) {
        const double x0 = x[xs + i], y0 = x[ys + i], th0 = x[ts + i], v0 = x[vs + i], e0 = x[es + i];
        const double w0 = x[ws + i], a0 = x[as + i];
        const double f0 = poly(coeffs, ncoef, x0);
        x[xs + i + 1] = x0 + v0 * cos(th0) * p->dt;
        x[ys + i + 1] = y0 + v0 * sin(th0) * p->dt;
        x[ts + i + 1] = th0 + w0 * p->dt;
        x[vs + i + 1] = v0 + a0 * p->dt;
        x[cs + i + 1] = (f0 - y0) + (v0 * sin(e0) * p->dt);
        x[es + i + 1] = e0 + w0 * p->dt;
    }
    /* multipliers in the solver's scaled units, lambda_i = sf lambda_i(record) / sc_i: refused where the cold start
     * scales a constraint row (sc_i != 1), which the record's rule does not provide for; z at least mu / slack */
    {
        const int nnz = mpc_oracle_nnz_jac(N);
        int *ir = (int *)malloc(sizeof(int) * nnz), *jc = (int *)malloc(sizeof(int) * nnz);
        double *jv = (double *)malloc(sizeof(double) * nnz), *x_cold = (double *)calloc(n, sizeof(double));
        for (int k = 0; k < 6; k++) x_cold[comp[k]] = state6[k];
        jac_coo(p, coeffs, ncoef, x_cold, ir, jc, jv);
        int scaled = 0;
        for (int k = 0; k < nnz; k++) scaled |= opt.nlp_scaling_max_gradient > 0.0 && fabs(jv[k]) > opt.nlp_scaling_max_gradient;
        free(ir); free(jc); free(jv); free(x_cold);
        if (scaled) { free(x); free(gr); free(lam); free(zl0); free(zu0); return -1; }
    }
    for (int i = 0; i < m; i++) lam[i] = sf * rec[rl + i];
    for (int k = 0; k < nu; k++) {
        const double w = x[ws + k], a = x[as + k];
        zl0[ws + k] = fmax(sf * rec[rz + k], warm_mu / (w + Uw));
        zl0[as + k] = fmax(sf * rec[rz + nu + k], warm_mu / (a + Ua));
        zu0[ws + k] = fmax(sf * rec[rz + 2 * nu + k], warm_mu / (Uw - w));
        zu0[as + k] = fmax(sf * rec[rz + 3 * nu + k], warm_mu / (Ua - a));
    }
    ipm_start start = { x, lam, zl0, zu0, warm_mu, sf };
    const int st = solve_from(p, state6, coeffs, ncoef, &opt, &start, u0, pred, sol, lambda, zl, zu, out);
    free(x); free(gr); free(lam); free(zl0); free(zu0);
    return st;
}

/* ---- pre-step ---- */

/* polyfit (driving_state.cpp:283-300): Vandermonde by running products, then
 * unpivoted Householder QR least squares (what Eigen's householderQr().solve does). */
int mpc_oracle_polyfit(const double *xs_, const double *ys_, int M, int order, double *coeffs)
{
    const int nc = order + 1;
    if (!(order >= 1 && order <= M - 1)) return -1;
    double *A = (double *)malloc(sizeof(double) * (size_t)M * nc);
    double *b = (double *)malloc(sizeof(double) * M);
    for (int j = 0; j < M; j++) {
        A[j * nc] = 1.0;
        for (int i = 0; i < order; i++) A[j * nc + i + 1] = A[j * nc + i] * xs_[j];
        b[j] = ys_[j];
    }
    for (int k = 0; k < nc; k++) {
        double nrm = 0.0;
        for (int i = k; i < M; i++) nrm += A[i * nc + k] * A[i * nc + k];
        nrm = sqrt(nrm);
        if (nrm == 0.0) { free(A); free(b); return -2; }
        const double alpha = (A[k * nc + k] > 0.0) ? -nrm : nrm;
        /* v = a_k - alpha e_k, stored in place; beta = 2 / v'v */
        A[k * nc + k] -= alpha;
        double vtv = 0.0;
        for (int i = k; i < M; i++) vtv += A[i * nc + k] * A[i * nc + k];
        const double beta = 2.0 / vtv;
        for (int j = k + 1; j < nc; j++) {
            double s = 0.0;
            for (int i = k; i < M; i++) s += A[i * nc + k] * A[i * nc + j];
            s *= beta;
            for (int i = k; i < M; i++) A[i * nc + j] -= s * A[i * nc + k];
        }
        double s = 0.0;
        for (int i = k; i < M; i++) s += A[i * nc + k] * b[i];
        s *= beta;
        for (int i = k; i < M; i++) b[i] -= s * A[i * nc + k];
        A[k * nc + k] = alpha; /* R_kk; the reflector below the diagonal is no longer needed */
    }
    for (int k = nc - 1; k >= 0; k--) {
        double s = b[k];
        for (int j = k + 1; j < nc; j++) s -= A[k * nc + j] * coeffs[j];
        coeffs[k] = s / A[k * nc + k];
    }
    free(A); free(b);
    return 0;
}

void mpc_oracle_prestep(const double *wx, const double *wy, int M,
                        double px, double py, double theta,
                        double *coeffs4, double *cte, double *etheta)
{
    const double ct = cos(theta), st = sin(theta);            /* driving_state.cpp:197-198 */
    double *xv = (double *)malloc(sizeof(double) * M), *yv = (double *)malloc(sizeof(double) * M);
    for (int i = 0; i < M; i++) {                             /* :202-207 */
        const double dx = wx[i] - px, dy = wy[i] - py;
        xv[i] = dx * ct + dy * st;
        yv[i] = dy * ct - dx * st;
    }
    mpc_oracle_polyfit(xv, yv, M, 3, coeffs4);                /* :210 */
    *cte = coeffs4[0];                                        /* polyeval(coeffs, 0.0), :211 */
    double eth = atan(coeffs4[1]);                            /* :212 (overwritten below) */
    double gx = 0.0, gy = 0.0;
    const int n_sample = (int)(M * 0.3);                      /* :217 */
    for (int i = 1; i < n_sample; i++) { gx += wx[i] - wx[i - 1]; gy += wy[i] - wy[i - 1]; } /* :218-221 */
    double temp_theta = theta;
    const double traj_deg = atan2(gy, gx);                    /* :224 */
    if (temp_theta <= -M_PI + traj_deg) temp_theta += 2.0 * M_PI;    /* :228-229 */
    if (gx != 0.0 && gy != 0.0 && temp_theta - traj_deg < 1.8 * M_PI) /* :232-235 */
        eth = temp_theta - traj_deg;
    else
        eth = 0.0;
    *etheta = eth;
    free(xv); free(yv);
}

/* Tracking::deceleration, driving_state.cpp:121-141 */
double mpc_oracle_decel(double px, double py, double gx, double gy, double v,
                        double max_throttle, double max_speed, double min_speed, double ref_v)
{
    const double dist_to_goal = hypot(px - gx, py - gy);                 /* :125-126 */
    if (dist_to_goal <= pow(v, 2) / max_throttle) {                      /* :127 */
        const double speed = max_throttle * dist_to_goal;                /* :129 */
        if (speed > ref_v) ref_v = max_speed;                            /* :130-132 */
        else if (speed < min_speed) ref_v = min_speed;                   /* :133-135 */
        else ref_v = speed;                                              /* :136-138 */
    }
    return ref_v;
}

/* State assembly, driving_state.cpp:242-256 */
void mpc_oracle_state(int delay_mode, double v, double w_prev, double throttle_prev, double dt,
                      double cte, double etheta, double *state6)
{
    if (delay_mode) {
        const double px_act = v * dt;                                    /* :245 */
        const double py_act = 0;                                         /* :246 */
        const double theta_act = w_prev * dt;                            /* :247 */
        const double v_act = v + throttle_prev * dt;                     /* :248 */
        const double cte_act = cte + v * sin(etheta) * dt;               /* :250 */
        const double etheta_act = etheta - theta_act;                    /* :251 */
        state6[0] = px_act; state6[1] = py_act; state6[2] = theta_act; state6[3] = v_act;
        state6[4] = cte_act; state6[5] = etheta_act;                     /* :253 */
    } else {
        state6[0] = 0; state6[1] = 0; state6[2] = 0; state6[3] = v; state6[4] = cte; state6[5] = etheta;   /* :255 */
    }
}

/* driving_state.cpp:266-269 */
double mpc_oracle_poststep_speed(double v, double throttle, double dt, double ref_v)
{
    double speed = v + throttle * dt;
    if (speed >= ref_v) speed = ref_v;
    return speed;
}

/* MPCPlannerROS::getCutOffPlan, mpc_planner_ros.cpp:266-291 */
int mpc_oracle_cutoff(int n, const double *px, const double *py, int first, int ring, int max_erase,
                      double rx, double ry)
{
    double max_distance_sq = 10e5;                                       /* :273 */
    int erased = 0;
    while (erased < max_erase) {                                         /* :276 while (it != end) */
        int i = first + erased;
        if (ring) i %= n; else if (i >= n) break;
        const double x_diff = rx - px[i], y_diff = ry - py[i];           /* :278-279 */
        const double distance_sq = x_diff * x_diff + y_diff * y_diff;    /* :280 */
        if (max_distance_sq < distance_sq) break;                        /* :282-284 */
        erased++;                                                        /* :285 erase(it) */
        max_distance_sq = distance_sq;                                   /* :286 */
    }
    return erased;
}

/* mpc_planner_ros.cpp:374 */
int mpc_oracle_downsample_step(double path_length, double waypoints_dist)
{
    return (int)(path_length / 10.0 / waypoints_dist);
}

/* MPCPlannerROS::downSamplePlan, mpc_planner_ros.cpp:365-391 */
int mpc_oracle_downsample(int n, const double *px, const double *py, int first, int ring, int win, int step,
                          int cap, double *wx, double *wy)
{
    int m = 0;
    int sampling = step;                                                 /* :376 */
    int last = first;
    for (int i = 0; i < win; i++) {                                      /* :379 */
        int q = first + i;
        if (ring) q %= n; else if (q >= n) break;
        last = q;
        if (sampling == step) {                                          /* :381-386 */
            if (m < cap) { wx[m] = px[q]; wy[m] = py[q]; }
            m++;
            sampling = 0;
        }
        sampling += 1;                                                   /* :388 */
    }
    if (m < cap) { wx[m] = px[last]; wy[m] = py[last]; }                 /* :390 cutoff_plan.back() */
    m++;
    return m;
}
