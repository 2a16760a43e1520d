/*
 * mpc_b200.h -- C ABI of the B200-native batched NMPC solver that drops in
 * behind mpc_ros's MPC::Solve hot path.
 *
 * Every entry point names the reference interface it replaces (paths relative
 * to the OkDoky/mpc_ros tree).  Plain C: pointers and sizes only, no C++ or
 * torch types.  All batch buffers are SoA, component-major with the problem
 * index fastest: element (c, i) of a "C x batch" buffer is buf[c*batch + i].
 * Buffers may live in host or device memory (auto-detected per pointer; host
 * buffers are staged through the handle's pinned memory).
 *
 * There is no CPU fallback: every solve runs the sm_100a CUDA kernels and the
 * calls fail with MPC_B200_ERR_CUDA when no usable device is present.
 */
#ifndef MPC_B200_H
#define MPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPC_B200_VERSION 100

/* ---- error codes (return values) ---- */
enum {
    MPC_B200_OK = 0,
    MPC_B200_ERR_INVALID = -1,      /* bad argument (NULL, batch > max_batch, ...) */
    MPC_B200_ERR_CUDA = -2,         /* CUDA runtime error / no device; see mpc_b200_last_cuda_error */
    MPC_B200_ERR_UNSUPPORTED = -3,  /* parameter combination outside the GPU path (see DESIGN.md) */
    MPC_B200_ERR_IO = -4,           /* params file unreadable */
    MPC_B200_ERR_NOMEM = -5
};

/* ---- per-problem status: numeric values of CppAD::ipopt::solve_result<>::status_type
 *      (mpc_ros/include/cppad/ipopt/solve_result.hpp:30-46), which MPC::Solve reads at
 *      mpc_ros/src/mpc_planner.cpp:378 ---- */
enum {
    MPC_B200_STATUS_NOT_DEFINED = 0,
    MPC_B200_STATUS_SUCCESS = 1,
    MPC_B200_STATUS_MAXITER_EXCEEDED = 2,
    MPC_B200_STATUS_STOP_AT_TINY_STEP = 3,
    MPC_B200_STATUS_STOP_AT_ACCEPTABLE_POINT = 4,
    MPC_B200_STATUS_LOCAL_INFEASIBILITY = 5,
    MPC_B200_STATUS_RESTORATION_FAILURE = 9,
    MPC_B200_STATUS_ERROR_IN_STEP_COMPUTATION = 10,
    MPC_B200_STATUS_INVALID_NUMBER_DETECTED = 11,
    /* Not a solve_result value.  The reference bounds every state variable by +-bound_value
     * (mpc_ros/src/mpc_planner.cpp:303-312, cfg range 0.01 .. 1000, cfg/MPCPlanner.cfg:37).  The GPU path carries
     * barrier terms for the control bounds only: a point all of whose states lie strictly inside the state bounds
     * is a KKT point of the bounded problem as well and is returned as SUCCESS; a point with some |state| within
     * 0.1 % of bound_value (or beyond) would have been shaped by the bounds and is returned with THIS status -- the
     * iterate is still written out (mpc_planner.cpp:378 ignores the status), but it is never counted as converged. */
    MPC_B200_STATUS_BOUND_ACTIVE = 64
};

/*
 * Parameters of one MPC instance.  Replaces the string-keyed map of
 * MPC::LoadParams / FG_eval::LoadParams (mpc_ros/src/mpc_planner.cpp:71-97,
 * :243-262; keys written at mpc_ros/src/driving_state.cpp:65-79) and the
 * mpc_* keys of mpc_ros/params/mpc_params.yaml:12-25.
 */
typedef struct mpc_b200_params {
    int32_t mpc_steps;      /* STEPS  / mpc_steps        (horizon N) */
    double dt;              /* DT     / 1/controller_freq */
    double ref_cte;         /* REF_CTE    / mpc_ref_cte   */
    double ref_etheta;      /* REF_ETHETA / mpc_ref_etheta */
    double ref_vel;         /* REF_V      / mpc_ref_vel   */
    double w_cte;           /* W_CTE      / mpc_w_cte     */
    double w_etheta;        /* W_EPSI     / mpc_w_etheta  */
    double w_vel;           /* W_V        / mpc_w_vel     */
    double w_angvel;        /* W_ANGVEL   / mpc_w_angvel  */
    double w_accel;         /* W_A        / mpc_w_accel   */
    double w_angvel_d;      /* W_DANGVEL  / mpc_w_angvel_d */
    double w_accel_d;       /* W_DA       / mpc_w_accel_d */
    double max_angvel;      /* ANGVEL     / mpc_max_angvel */
    double max_throttle;    /* MAXTHR     / mpc_max_throttle */
    double bound_value;     /* BOUND      / mpc_bound_value */
    /* solver controls; the reference leaves these at Ipopt's defaults
     * (only print_level and max_cpu_time are set, mpc_planner.cpp:358,368) */
    double tol;             /* Ipopt tol, 1e-8 */
    int32_t max_iter;       /* iteration cap per problem (Ipopt: 3000; default here 100) */
    /* non-solver keys of mpc_params.yaml:2-9, carried for the callers above MPC::Solve */
    int32_t delay_mode;     /* delay_mode */
    double max_speed;       /* max_speed */
    double path_length;     /* path_length */
    double waypoints_dist;  /* waypoints_dist */
    double goal_radius;     /* goal_radius */
    double controller_freq; /* controller_freq */
    /* warm start (no reference counterpart): barrier parameter a warm-started solve begins with */
    double warm_mu_init;    /* default 1e-3 */
} mpc_b200_params;

/* Defaults = the constructor defaults of MPC::MPC (mpc_planner.cpp:223-241) and
 * FG_eval::FG_eval (:42-68) as MPC::Solve sees them before any LoadParams. */
void mpc_b200_params_default(mpc_b200_params *p);
/* The values of mpc_ros/params/mpc_params.yaml:1-25 (the benchmark configuration). */
void mpc_b200_params_yaml_default(mpc_b200_params *p);
/* Parse a flat "key: value" YAML file with the keys of mpc_params.yaml; unknown keys are
 * ignored, missing keys keep the value already in *p.  Returns MPC_B200_OK / _ERR_IO. */
int mpc_b200_params_from_yaml(const char *path, mpc_b200_params *p);
/* One key of the LoadParams map (DT STEPS REF_CTE REF_ETHETA REF_V W_CTE W_EPSI W_V W_ANGVEL
 * W_A W_DANGVEL W_DA ANGVEL MAXTHR BOUND).  Unknown key: MPC_B200_ERR_INVALID, *p untouched. */
int mpc_b200_params_set(mpc_b200_params *p, const char *key, double value);

typedef struct mpc_b200_handle mpc_b200_handle;

/* Creates a solver bound to one CUDA device with scratch for max_batch problems.
 * One handle per host thread / per GPU; a handle is not re-entrant. */
int mpc_b200_create(mpc_b200_handle **h, const mpc_b200_params *p, int32_t max_batch, int32_t device);
void mpc_b200_destroy(mpc_b200_handle *h);
/* Replaces MPC::LoadParams between solves (mpc_planner.cpp:243; called per tick from
 * Tracking::deceleration, driving_state.cpp:121-141).  Cheap: no rebuild. */
int mpc_b200_set_params(mpc_b200_handle *h, const mpc_b200_params *p);
int mpc_b200_get_params(const mpc_b200_handle *h, mpc_b200_params *p);
/* Launch tuning, no reference counterpart.  "max_ctas": cap on the persistent grid (0 = one CTA per SM;
 * smaller values leave SMs to batches in flight on other streams and make each lane work through
 * several problems); "problems_per_cta": 0 = auto (up to 32); "hard_first": 1 (default) serves the work queue
 * in descending order of |c1|+|c2|+|c3| so that the slow problems of a batch start first (results do not
 * depend on it).  "poly_coeffs": rows of the coeffs arrays of mpc_b200_solve_batch = order of the path
 * polynomial + 1, 4 (default, the cubic of driving_state.cpp:210) .. 8; FG_eval takes any order
 * (mpc_planner.cpp:186-190: coeffs.size()); the pre-step entry points then fit that order (polyfit(x, y, order),
 * driving_state.cpp:283-300) and write as many rows (they need M >= poly_coeffs waypoints).
 * "dual_groups": 1 (default) runs full CTAs (32 lanes, 28 with rate penalties; horizons 11..20) as two lane groups
 * out of phase on shared stage threads (nmpc_kernel_dual.cuh); "narrow_one_stage": 1 (default) gives every stage thread
 * of a narrow CTA (16 / 8 / 4 / 1 lanes: small batches, a single MPC::Solve) one stage instead of two (latency mode).
 * Both only choose between kernels that run the same phase functions; results agree to rounding.
 * Unknown name or value: MPC_B200_ERR_INVALID. */
int mpc_b200_set_option(mpc_b200_handle *h, const char *name, double value);

/* Size in doubles of one problem's warm-start record: primal (8N-2, the reference's variable
 * layout, mpc_planner.cpp:232-239) + equality multipliers (6N) + control-bound multipliers
 * zL, zU (2(N-1) each). */
int32_t mpc_b200_warm_size(int32_t mpc_steps);

/*
 * Batched MPC::Solve (mpc_ros/src/mpc_planner.cpp:265-402): `batch` independent problems.
 *   state    6 x batch   [x, y, theta, v, cte, etheta]        (:270-275)
 *   coeffs   4 x batch   cubic reference-path coefficients    (:186-190; driving_state.cpp:210)
 *   ref_vel  batch       optional per-problem REF_V override (NULL = params.ref_vel); the reference
 *                        rewrites REF_V per tick (driving_state.cpp:127-139)
 *   warm_in  warm_size x batch, optional, device or host memory (NULL = the reference's cold start, :288-300):
 *            controls, equality and bound multipliers are taken from it, the states are re-derived
 *            by a roll-out of the model from `state` (the record's state rows are not read).  Controls
 *            are clipped 1e-3 U inside the relaxed bounds U, so a NaN control is read as U - 1e-3 U;
 *            z = max(sf z, warm_mu_init / slack), so a NaN bound multiplier is read as the floor and an
 *            infinite one ends the problem at once with status 11.  A non-finite equality multiplier
 *            (lambda_0 included) ends it after the start point's evaluation with status 10 and 0
 *            iterations, as Ipopt's first step would (at mpc_steps = 2, where no multiplier enters a
 *            Newton system, with status 11 at that evaluation): it is never carried into a status-1 result.
 *   u0       2 x batch   {w_0, throttle_0} = MPC::Solve's return value (:398-401)
 *   pred     3N x batch  mpc_x, mpc_y, mpc_theta (:388-396)
 *   obj      batch       objective value (solution.obj_value, :381), optional
 *   status   batch       per-problem status (:378), optional
 *   iters    batch       interior-point iterations, optional
 *   kkt_res  batch       final scaled optimality error E_0 (Ipopt's `tol` measure), optional
 *   warm_out warm_size x batch, optional, device or host memory (host records are staged)
 *   stream   cudaStream_t, or NULL for the handle's own stream.  The call returns after the
 *            results are in the caller's buffers (synchronous, like MPC::Solve) unless every
 *            buffer is device memory AND a stream is given, in which case it only enqueues; one handle
 *            may have max(16, min(1024, 4M / max_batch)) such launches in flight on different streams.
 */
int mpc_b200_solve_batch(mpc_b200_handle *h, int32_t batch,
                         const double *state, const double *coeffs, const double *ref_vel,
                         const double *warm_in,
                         double *u0, double *pred, double *obj, int32_t *status, int32_t *iters,
                         double *kkt_res, double *warm_out, void *stream);

/*
 * Plan windowing for a device-resident closed loop (all pointers DEVICE memory): cut the plan at the
 * first plan point past the one nearest to the robot (MPCPlannerROS::getCutOffPlan, mpc_ros/src/mpc_planner_ros.cpp:266-291)
 * and down-sample the next params.path_length metres (downSamplePlan, :365-391; waypoint spacing =
 * params.waypoints_dist, or 0.05 m when that is <= 0).  Plans are closed tracks stored back to back:
 * track t occupies path_x/path_y[track_off[t] .. track_off[t] + track_len[t]).
 *   track_id  batch      track of each robot          idx_inout  batch   plan index of the cut (updated)
 *   pose      3 x batch                               wx_out, wy_out   mpc_b200_num_waypoints(params) x batch
 */
int mpc_b200_window_batch(mpc_b200_handle *h, int32_t batch, const double *path_x, const double *path_y,
                          const int32_t *track_off, const int32_t *track_len, const int32_t *track_id,
                          int32_t *idx_inout, const double *pose, double *wx_out, double *wy_out, void *stream);
int mpc_b200_num_waypoints(const mpc_b200_params *p);

/*
 * Reference-speed schedule near the goal (Tracking::deceleration, mpc_ros/src/driving_state.cpp:121-141),
 * device memory: inside the braking distance v^2 / max_throttle of its goal a robot's REF_V becomes
 * max_throttle * distance (not below min_speed; the reference's `speed > REF_V -> max_speed` branch is kept).
 * pose 3 x batch, goal 2 x batch, vel 3 x batch (row 0 = feedback speed), ref_vel_inout batch: the value
 * persists from tick to tick and is what solve_batch / poststep_batch take as `ref_vel`.
 * max_throttle (floored at 0.1, :61-63) and max_speed come from the handle's params; min_speed is the
 * reference's context member (0.05, :29).
 */
int mpc_b200_decel_batch(mpc_b200_handle *h, int32_t batch, const double *pose, const double *goal, const double *vel,
                         double min_speed, double *ref_vel_inout, void *stream);

/*
 * Plant step for closed-loop simulation (SURVEY 8d config 5; the reference has no plant, the robot is):
 * unicycle x += v cos(theta) dt, y += v sin(theta) dt, theta += w dt wrapped to [-pi, pi), with
 * {v, w} = cmd (2 x batch, from poststep_batch); vel_inout row 0 becomes the new feedback speed.  Device memory.
 */
int mpc_b200_plant_step_batch(mpc_b200_handle *h, int32_t batch, const double *cmd, double *pose_inout, double *vel_inout,
                              void *stream);

/*
 * Result post-step of Tracking::findBestPath (mpc_ros/src/driving_state.cpp:263-269), device memory:
 * speed = v + throttle * dt clamped above at REF_V; cmd_out (2 x batch) = {linear.x, angular.z}
 * (:115-116); vel_inout (3 x batch: v, previous w, previous throttle) gets the new w and throttle for the
 * next tick's delay compensation (the caller supplies the new feedback speed v).
 */
int mpc_b200_poststep_batch(mpc_b200_handle *h, int32_t batch, const double *u0, double *vel_inout,
                            const double *ref_vel, double *cmd_out, void *stream);

/* Next tick's warm start from this tick's solution (device buffers): every block of the record moves
 * one stage forward, the last entry is repeated. */
int mpc_b200_warm_shift(mpc_b200_handle *h, int32_t batch, const double *warm_prev, double *warm_next, void *stream);

/*
 * Batched waypoint transform + cubic polyfit + (cte, etheta): the reference pre-step
 * Tracking::findBestPath (mpc_ros/src/driving_state.cpp:196-235) with polyfit (:283-300).
 *   wx, wy   M x batch   waypoints in the global frame
 *   pose     3 x batch   px, py, theta
 *   coeffs_out      4 x batch
 *   cte_etheta_out  2 x batch (cte = c[0], :211; etheta by the atan2 rule, :215-235), optional
 */
int mpc_b200_polyfit_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                           const double *wx, const double *wy, const double *pose,
                           double *coeffs_out, double *cte_etheta_out, void *stream);

/*
 * The whole reference pre-step in one call: polyfit_batch plus the 6-state assembly of
 * Tracking::findBestPath (mpc_ros/src/driving_state.cpp:242-256), including the delay-compensated
 * state when params.delay_mode is set (:243-254).
 *   vel        3 x batch   v (feedback_vel.linear.x, :191), previous w (:192), previous throttle (:193)
 *   state_out  6 x batch   ready for mpc_b200_solve_batch
 */
int mpc_b200_prestep_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                           const double *wx, const double *wy, const double *pose, const double *vel,
                           double *coeffs_out, double *state_out, void *stream);

/*
 * CUDA streams for hosts that do not link the CUDA runtime themselves (cgo / JNI / ctypes callers): the
 * `stream` argument of the *_batch calls takes what _stream_create returns (a cudaStream_t, non-blocking).
 * Independent batches issued on different streams overlap on the device.
 */
int mpc_b200_stream_create(int32_t device, void **stream_out);
int mpc_b200_stream_destroy(void *stream);
int mpc_b200_stream_synchronize(void *stream);

/*
 * The whole control tick of Tracking::findBestPath (mpc_ros/src/driving_state.cpp:175-271) for `batch` robots,
 * HOST buffers in and out, one synchronous call: pre-step (:196-256) -> MPC::Solve (:260) -> post-step
 * (:263-269).  The fitted coefficients and the assembled state never leave the device.
 *   wx, wy  M x batch; pose 3 x batch; vel_inout 3 x batch (v, previous w, previous throttle; w and
 *   throttle are updated); ref_vel batch or NULL; u0 2 x batch; pred 3N x batch;
 *   cmd_out 2 x batch {linear.x, angular.z} (:115-116), optional; obj/status/iters/kkt_res optional.
 */
int mpc_b200_track_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                         const double *wx, const double *wy, const double *pose, double *vel_inout,
                         const double *ref_vel, double *u0, double *pred, double *cmd_out,
                         double *obj, int32_t *status, int32_t *iters, double *kkt_res);
/*
 * The same tick split in two so that one host thread can keep several handles busy: _submit enqueues the
 * copies and kernels on the handle's own stream and returns; _wait blocks until the results are in the
 * caller's buffers.  Page-locked buffers are read and written by DMA while the tick is in flight; pageable
 * ones are staged (inputs copied inside _submit, outputs inside _wait).  One tick in flight per handle:
 * a second _submit before _wait returns MPC_B200_ERR_INVALID.  track_batch == _submit followed by _wait.
 */
int mpc_b200_track_submit(mpc_b200_handle *h, int32_t batch, int32_t M,
                          const double *wx, const double *wy, const double *pose, double *vel_inout,
                          const double *ref_vel, double *u0, double *pred, double *cmd_out,
                          double *obj, int32_t *status, int32_t *iters, double *kkt_res);
int mpc_b200_track_wait(mpc_b200_handle *h);

/*
 * The same tick over ONE caller buffer: a single host-to-device and a single device-to-host copy per tick instead
 * of one per array (the arrays are small; per-copy overhead is what a host thread feeding several GPUs pays).
 * _layout returns the buffer size in BYTES and the byte offset of each block, in this order:
 *   0 wx (M x batch)  1 wy  2 pose (3 x batch)  3 ref_vel (batch; -1 when with_ref_vel == 0)
 *   4 vel (3 x batch, in AND out)  5 u0 (2 x batch)  6 pred (3N x batch)  7 cmd (2 x batch)  8 obj  9 kkt_res
 *   10 status (int32 x batch)  11 iters (int32 x batch)
 * Blocks 0-4 are read, blocks 4-11 written; the caller fills the inputs in place, calls _packed_submit, and reads the
 * outputs in place after mpc_b200_track_wait.  Page-locked buffers (mpc_b200_host_alloc) are copied by DMA directly.
 */
int64_t mpc_b200_track_packed_layout(const mpc_b200_handle *h, int32_t batch, int32_t M, int32_t with_ref_vel,
                                     int64_t *offsets_bytes12);
int mpc_b200_track_packed_submit(mpc_b200_handle *h, int32_t batch, int32_t M, int32_t with_ref_vel, void *io);
/*
 * Multi-GPU sharding of ONE batch (SURVEY 8e: contiguous slices, no collective, host gather): the caller's SoA arrays
 * hold the whole batch (`ld` columns); the handle -- one per GPU and host thread -- takes columns
 * [offset, offset + batch).  Arrays must be page-locked (mpc_b200_host_alloc; else MPC_B200_ERR_UNSUPPORTED): every
 * array moves by one strided DMA copy straight between the caller's memory and the device, and each slice's results
 * land in their own sub-range of the caller's output arrays -- that is the whole "gather".  Arguments as
 * mpc_b200_track_submit; finish with mpc_b200_track_wait.
 */
int mpc_b200_track_slice_submit(mpc_b200_handle *h, int32_t ld, int32_t offset, int32_t batch, int32_t M,
                                const double *wx, const double *wy, const double *pose, double *vel_inout,
                                const double *ref_vel, double *u0, double *pred, double *cmd_out,
                                double *obj, int32_t *status, int32_t *iters, double *kkt_res);
/* Page-locked host memory for callers that do not link the CUDA runtime (cgo / JNI / ctypes). */
void *mpc_b200_host_alloc(size_t bytes);
void mpc_b200_host_free(void *p);

/* Seconds spent on the device by the last solve_batch / polyfit_batch on this handle
 * (CUDA events on the launching stream around the kernel only; no copies). */
double mpc_b200_last_kernel_seconds(const mpc_b200_handle *h);
/* Number of kernels this handle has launched so far. */
int64_t mpc_b200_launch_count(const mpc_b200_handle *h);

const char *mpc_b200_strerror(int code);
const char *mpc_b200_last_cuda_error(const mpc_b200_handle *h);
int mpc_b200_version(void);
/* Number of usable CUDA devices (0 when none / no driver). */
int mpc_b200_device_count(void);

/* FP64 FMA microbenchmark used to fix the roofline denominator (MEASURED_PEAKS.json has
 * no FP64 entry): independent DFMA chains on every SM.  Returns measured TFLOP/s, <0 on error. */
double mpc_b200_measure_fp64_peak(int32_t device, int32_t iters);
/* Diagnostics.  _debug_profile: per-phase SM-cycle counters of the last solve (libraries built with
 * -DNMPC_PROFILE only; returns 0 otherwise; out = 1024 values, see bench/gpu_sat.py).  _debug_fp64_probe: SM cycles per
 * warp-level DFMA of a single warp with `ilp` independent chains and `active_lanes` lanes (profiles/r1_fp64_probe.md). */
int mpc_b200_debug_profile(mpc_b200_handle *h, long long *out1024);
double mpc_b200_debug_fp64_probe(int32_t device, int32_t ilp, int32_t active_lanes, int32_t iters);

#ifdef __cplusplus
}
#endif
#endif /* MPC_B200_H */
