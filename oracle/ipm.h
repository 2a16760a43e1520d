/*
 * oracle/ipm.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Generic dense-storage primal-dual interior-point filter line-search NLP
 * solver: a from-scratch CPU restatement of the published Ipopt algorithm
 * (Waechter & Biegler, Math. Prog. 106 (2006) 25-57) with Ipopt 3.12's
 * default option values.  It stands in for the Ipopt 3.12.8 library that
 * the reference links by name (mpc_ros/CMakeLists.txt:101, call site
 * mpc_ros/include/cppad/ipopt/solve.hpp:586) and that is absent from this
 * image.  "Parity unpinned" against real Ipopt: pinned instead on the HS071
 * known answer the reference ships (assets/document/example/CppAD_Ipopt.cpp
 * :146-150) and on SciPy SLSQP (tests/test_oracle.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may link or call this.
 */
#ifndef ORACLE_IPM_H
#define ORACLE_IPM_H

#ifdef __cplusplus
extern "C" {
#endif

/* Status values = CppAD::ipopt::solve_result<>::status_type
 * (mpc_ros/include/cppad/ipopt/solve_result.hpp:30-46). */
enum {
    IPM_NOT_DEFINED = 0,
    IPM_SUCCESS = 1,
    IPM_MAXITER_EXCEEDED = 2,
    IPM_STOP_AT_TINY_STEP = 3,
    IPM_STOP_AT_ACCEPTABLE_POINT = 4,
    IPM_LOCAL_INFEASIBILITY = 5,
    IPM_USER_REQUESTED_STOP = 6,
    IPM_FEASIBLE_POINT_FOUND = 7,
    IPM_DIVERGING_ITERATES = 8,
    IPM_RESTORATION_FAILURE = 9,
    IPM_ERROR_IN_STEP_COMPUTATION = 10,
    IPM_INVALID_NUMBER_DETECTED = 11,
    IPM_TOO_FEW_DOF = 12,
    IPM_INTERNAL_ERROR = 13,
    IPM_UNKNOWN = 14
};

/* NLP in Ipopt's TNLP form:  min f(x)  s.t.  gl <= g(x) <= gu, xl <= x <= xu.
 * |bound| >= 1e19 means "no bound".  Sparse COO Jacobian / lower-triangular
 * Hessian of  sigma*f + sum_i lambda_i g_i.  Callbacks return nonzero on ok. */
typedef struct ipm_nlp {
    int n, m, nnz_jac, nnz_hess;
    void *user;
    int (*get_bounds)(void *user, double *xl, double *xu, double *gl, double *gu);
    int (*get_start)(void *user, double *x0);
    int (*eval_f)(void *user, const double *x, double *f);
    int (*eval_grad_f)(void *user, const double *x, double *grad);
    int (*eval_g)(void *user, const double *x, double *g);
    int (*jac_struct)(void *user, int *irow, int *jcol);
    int (*eval_jac)(void *user, const double *x, double *vals);
    int (*hess_struct)(void *user, int *irow, int *jcol);
    int (*eval_hess)(void *user, const double *x, double sigma,
                     const double *lambda, double *vals);
} ipm_nlp;

typedef struct ipm_options {
    double tol;               /* 1e-8 */
    int max_iter;             /* 3000 */
    double max_cpu_time;      /* 1e6 s; the reference sets 0.5 (mpc_planner.cpp:368) */
    double dual_inf_tol;      /* 1 */
    double constr_viol_tol;   /* 1e-4 */
    double compl_inf_tol;     /* 1e-4 */
    double acceptable_tol;    /* 1e-6 */
    int acceptable_iter;      /* 15 */
    double mu_init;           /* 0.1 */
    double bound_push;        /* 0.01 */
    double bound_frac;        /* 0.01 */
    double bound_relax_factor;/* 1e-8 */
    double nlp_scaling_max_gradient; /* 100; <=0 disables scaling */
    int max_soc;              /* 4 */
    int print_level;          /* 0 */
    int use_dense_ldl;        /* 0: sparsity-aware LDL^T after RCM; 1: plain dense */
} ipm_options;

typedef struct ipm_result {
    int status;
    int iters;
    double obj;        /* unscaled f(x*) */
    double kkt_error;  /* final scaled E_0 (Ipopt eq. (5)) */
    double dual_inf, constr_viol, compl_inf; /* unscaled inf-norms at exit */
    double mu;         /* final barrier parameter */
    int n_inertia_corrections;
    int n_restorations;
    int n_factorizations;
    /* caller-allocated, may be NULL: */
    double *x;      /* n */
    double *zl;     /* n */
    double *zu;     /* n */
    double *g;      /* m */
    double *lambda; /* m */
} ipm_result;

/* A given starting iterate (warm start).  Multipliers are in the solver's scaled units:
 * lambda_i = sf * lambda_i(unscaled) / sc_i, z = sf * z(unscaled).  The NLP scaling is the cold solve's:
 * computed at the NLP's own (pushed) starting point, so a warm solve differs from a cold one in its
 * starting iterate only; sf > 0 overrides the objective factor.  With a start the solver takes x0 as
 * given (no bound_push), sets mu = mu0 and tau = max(0.99, 1 - mu0), skips the least-squares
 * multiplier solve, and uses zL0 / zU0 for the bounds of x (slacks keep z = 1). */
typedef struct ipm_start {
    const double *x0;       /* n */
    const double *lambda0;  /* m */
    const double *zl0;      /* n */
    const double *zu0;      /* n */
    double mu0;
    double sf;              /* > 0: objective scaling factor; <= 0: computed as for the cold start */
} ipm_start;

void ipm_default_options(ipm_options *o);
int ipm_solve(const ipm_nlp *nlp, const ipm_options *opt, ipm_result *res);
/* start == NULL: ipm_solve */
int ipm_solve_from(const ipm_nlp *nlp, const ipm_options *opt, const ipm_start *start, ipm_result *res);

#ifdef __cplusplus
}
#endif
#endif
