/*
 * oracle/mpc_oracle.h -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement of the reference's MPC::Solve hot path
 * (mpc_ros/src/mpc_planner.cpp:102-217 problem definition, :265-402 solve)
 * and of its pre-step (mpc_ros/src/driving_state.cpp:196-256, :273-300),
 * with hand-written analytic derivatives, solved by oracle/ipm.c.
 *
 * Pinning: derivatives are checked against the reference's own FG_eval +
 * vendored CppAD (oracle/_ref, tests/golden/fg_eval_*.json); the solver is
 * checked on HS071 and against SciPy.  Real Ipopt is absent from this image,
 * so solver parity with Ipopt itself is "unpinned" (see DESIGN.md).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may
 * use this.
 */
#ifndef MPC_ORACLE_H
#define MPC_ORACLE_H
#include "ipm.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct mpc_oracle_params {
    int mpc_steps;
    double dt, ref_cte, ref_etheta, ref_vel;
    double w_cte, w_etheta, w_vel, w_angvel, w_accel, w_angvel_d, w_accel_d;
    double max_angvel, max_throttle, bound_value;
} mpc_oracle_params;

/* YAML defaults of mpc_ros/params/mpc_params.yaml:9-25 (dt = 1/controller_freq). */
void mpc_oracle_params_yaml_default(mpc_oracle_params *p);

/* Sizes: n = 8N-2, m = 6N (mpc_planner.cpp:281,284). */
int mpc_oracle_nvars(int N);
int mpc_oracle_ncons(int N);

/* f and g in the reference's fg layout (fg[0]=f, fg[1+i]=g_i; mpc_planner.cpp:102-217). */
void mpc_oracle_eval_fg(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                        const double *vars, double *f, double *g);
void mpc_oracle_eval_grad(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                          const double *vars, double *grad);
/* Dense Jacobian (m x n, row-major) and dense symmetric Hessian of
 * sigma*f + sum lambda_i g_i (n x n); for golden-vector comparison. */
void mpc_oracle_eval_jac_dense(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                               const double *vars, double *J);
void mpc_oracle_eval_hess_dense(const mpc_oracle_params *p, const double *coeffs, int ncoef,
                                const double *vars, double sigma, const double *lambda, double *H);
int mpc_oracle_nnz_jac(int N);
int mpc_oracle_nnz_hess(const mpc_oracle_params *p);

typedef struct mpc_oracle_result {
    int status, iters;
    double obj, kkt_error, dual_inf, constr_viol, compl_inf;
    int n_inertia_corrections, n_restorations;
} mpc_oracle_result;

/* MPC::Solve restated (mpc_planner.cpp:265-402): cold start at zeros except
 * stage 0, bounds of :303-325, equality constraints of :330-348.
 * u0[2] = {w_0, a_0}; pred (3*N) = x_k, y_k, theta_k; sol (n), lambda (m), zl/zu (n) optional. */
int mpc_oracle_solve(const mpc_oracle_params *p, const double *state6, const double *coeffs, int ncoef,
                     const ipm_options *opt /* NULL = Ipopt defaults */,
                     double *u0, double *pred, double *sol, double *lambda, double *zl, double *zu,
                     mpc_oracle_result *res);

/* The same solve from a warm-start record in the layout of the GPU path's mpc_b200_warm_size (no reference
 * counterpart: primal 8N-2, lambda 6N, then zL_w, zL_a, zU_w, zU_a of N-1 each; multipliers unscaled).
 * Restates the record's rule: controls from the record clipped 1e-3 U inside the relaxed bounds U; states
 * rolled out from state6 with this file's model (the record's states are ignored); lambda (lambda_0
 * included) times the cold start's objective scaling sf; z = max(sf z, warm_mu / slack); mu = warm_mu,
 * no least-squares multipliers.  The NLP scaling is the cold start's.  Returns -1 without solving where
 * p->bound_value < 1e19 (the record has no state-bound multipliers) or where the cold start would scale a
 * constraint row. */
int mpc_oracle_solve_warm(const mpc_oracle_params *p, const double *state6, const double *coeffs, int ncoef,
                          const ipm_options *opt, const double *warm_record, double warm_mu,
                          double *u0, double *pred, double *sol, double *lambda, double *zl, double *zu,
                          mpc_oracle_result *res);

/* Pre-step (driving_state.cpp:196-235): waypoints (global frame) -> robot frame,
 * cubic least-squares fit by Householder QR, cte = c[0], etheta by the
 * reference's atan2 rule.  Returns 0 on success. */
int mpc_oracle_polyfit(const double *xs, const double *ys, int M, int order, double *coeffs);
void mpc_oracle_prestep(const double *wx, const double *wy, int M,
                        double px, double py, double theta,
                        double *coeffs4, double *cte, double *etheta);

/* Reference-speed schedule near the goal (Tracking::deceleration, driving_state.cpp:121-141): returns the
 * new REF_V (the map entry persists from tick to tick, so the caller passes the previous value in).
 * max_throttle is the context member floored at 0.1 (driving_state.cpp:61-63). */
double mpc_oracle_decel(double px, double py, double gx, double gy, double v,
                        double max_throttle, double max_speed, double min_speed, double ref_v);

/* State handed to MPC::Solve (Tracking::findBestPath, driving_state.cpp:242-256): with delay_mode the kinematic
 * model predicts the state one dt ahead using the previous w / throttle, else (0, 0, 0, v, cte, etheta). */
void mpc_oracle_state(int delay_mode, double v, double w_prev, double throttle_prev, double dt,
                      double cte, double etheta, double *state6);

/* Result post-step (driving_state.cpp:263-269): speed = v + throttle dt, clamped ABOVE at REF_V only. */
double mpc_oracle_poststep_speed(double v, double throttle, double dt, double ref_v);

/* Plan windowing (SURVEY 8f-2).
 * mpc_oracle_cutoff: MPCPlannerROS::getCutOffPlan, mpc_ros/src/mpc_planner_ros.cpp:266-291 -- plan points are erased
 * from the front while the squared distance to the robot does not grow (start value 10e5); returns how many were
 * erased, at most max_erase (the reference walks the whole plan: pass n).  Indices wrap modulo n when ring != 0
 * (closed tracks; the reference's plan is open).
 * mpc_oracle_downsample: MPCPlannerROS::downSamplePlan, :365-391 -- of a window of `win` points starting at `first`
 * keep every `step`-th one, beginning with the first, then append the window's last point; the reference derives
 * step = int(path_length / 10 / waypoints_dist) from the spacing of the first two points (:369-375) -- here the
 * caller passes it (mpc_oracle_downsample_step).  Returns the number of waypoints written (capacity cap). */
int mpc_oracle_cutoff(int n, const double *px, const double *py, int first, int ring, int max_erase,
                      double rx, double ry);
int mpc_oracle_downsample_step(double path_length, double waypoints_dist);
int mpc_oracle_downsample(int n, const double *px, const double *py, int first, int ring, int win, int step,
                          int cap, double *wx, double *wy);

#ifdef __cplusplus
}
#endif
#endif
