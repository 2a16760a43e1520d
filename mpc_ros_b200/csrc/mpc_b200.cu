// mpc_b200.cu -- C ABI (include/mpc_b200.h) + kernel launches.  sm_100a only; no CPU path.
#include "../../include/mpc_b200.h"
#include "nmpc_kernel.cuh"
#include "nmpc_kernel_dual.cuh"

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <string>

using nmpc::SolveArgs;

// NVTX range around every batch entry point (SURVEY section 5: tracing): shows up in nsys / ncu timelines
namespace { struct NvtxRange { explicit NvtxRange(const char *n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } }; }

#define MAX_WAYPOINTS 64
#define QUEUE_RING 1024
// stages per stage thread: at N = 20, 2 control warps + 10 stage warps = 384 threads at 168 registers (the whole
// register file; the serial Riccati sweep keeps ~70 doubles live)
#define SPT 2
#define STAGE_THREADS 320

// ================================================================ K1: transform + polyfit
// Reference: Tracking::findBestPath, mpc_ros/src/driving_state.cpp:196-235, polyfit :283-300
// (Vandermonde by running products + unpivoted Householder QR, what Eigen's
// householderQr().solve() does).  One thread per problem: M ~ 11 waypoints, a 11x4 QR.
// NC = order + 1 columns (polyfit(x, y, order), driving_state.cpp:283-300, takes any order; the caller fits 3).
// MAXM: rows the per-thread scratch is sized for -- 16 covers the reference's ~11 down-sampled waypoints (640 B of stack
// at NC = 4), 64 is the general case.
template <int NC, int MAXM>
__global__ void prestep_kernel(int batch, int M, const double *__restrict__ wx, const double *__restrict__ wy,
                               const double *__restrict__ pose, double *__restrict__ coeffs_out,
                               double *__restrict__ cte_eth_out, const double *__restrict__ vel,
                               double *__restrict__ state_out, int delay_mode, double dt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const double px = pose[i], py = pose[(size_t)batch + i], th = pose[2 * (size_t)batch + i];
    double st, ct;
    sincos(th, &st, &ct);
    double A[MAXM][NC];
    double b[MAXM];
    for (int j = 0; j < M; j++) {
        const double dx = wx[(size_t)j * batch + i] - px, dy = wy[(size_t)j * batch + i] - py;
        const double xv = dx * ct + dy * st;      // driving_state.cpp:205
        b[j] = dy * ct - dx * st;                 // :206
        A[j][0] = 1.0;
#pragma unroll
        for (int q = 1; q < NC; q++) A[j][q] = A[j][q - 1] * xv;                  // :292-296
    }
    double c[NC];
    bool ok = true;
    for (int k = 0; k < NC; k++) {
        double nrm = 0.0;
        for (int r = k; r < M; r++) nrm += A[r][k] * A[r][k];
        nrm = sqrt(nrm);
        if (nrm == 0.0) { ok = false; break; }
        const double alpha = (A[k][k] > 0.0) ? -nrm : nrm;
        A[k][k] -= alpha;
        double vtv = 0.0;
        for (int r = k; r < M; r++) vtv += A[r][k] * A[r][k];
        const double beta = 2.0 / vtv;
        for (int j = k + 1; j < NC; j++) {
            double s = 0.0;
            for (int r = k; r < M; r++) s += A[r][k] * A[r][j];
            s *= beta;
            for (int r = k; r < M; r++) A[r][j] -= s * A[r][k];
        }
        double s = 0.0;
        for (int r = k; r < M; r++) s += A[r][k] * b[r];
        s *= beta;
        for (int r = k; r < M; r++) b[r] -= s * A[r][k];
        A[k][k] = alpha;
    }
    if (ok) {
        for (int k = NC - 1; k >= 0; k--) {
            double s = b[k];
            for (int j = k + 1; j < NC; j++) s -= A[k][j] * c[j];
            c[k] = s / A[k][k];
        }
    } else {
        const double nanv = nan("");
        for (int k = 0; k < NC; k++) c[k] = nanv;
    }
    for (int k = 0; k < NC; k++) coeffs_out[(size_t)k * batch + i] = c[k];
    if (cte_eth_out || state_out) {
        // cte = polyeval(coeffs, 0) = c[0] (:211); etheta by the reference's atan2 rule (:215-235)
        double gx = 0.0, gy = 0.0;
        const int ns = (int)(M * 0.3);
        for (int j = 1; j < ns; j++) {
            gx += wx[(size_t)j * batch + i] - wx[(size_t)(j - 1) * batch + i];
            gy += wy[(size_t)j * batch + i] - wy[(size_t)(j - 1) * batch + i];
        }
        double tt = th;
        const double traj = atan2(gy, gx);
        const double PI = 3.14159265358979323846;
        if (tt <= -PI + traj) tt += 2.0 * PI;
        double eth;
        if (gx != 0.0 && gy != 0.0 && tt - traj < 1.8 * PI) eth = tt - traj; else eth = 0.0;
        if (cte_eth_out) {
            cte_eth_out[i] = c[0];
            cte_eth_out[(size_t)batch + i] = eth;
        }
        if (state_out) {
            // state assembly, driving_state.cpp:242-256
            const double v = vel[i];
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = v, s4 = c[0], s5 = eth;
            if (delay_mode) {
                const double w = vel[(size_t)batch + i], thr = vel[2 * (size_t)batch + i];
                s0 = v * dt;                       // px_act   (:245)
                s1 = 0.0;                          // py_act   (:246)
                s2 = w * dt;                       // theta_act (:247)
                s3 = v + thr * dt;                 // v_act    (:248)
                s4 = c[0] + v * sin(eth) * dt;     // cte_act  (:250)
                s5 = eth - s2;                     // etheta_act (:251)
            }
            state_out[i] = s0; state_out[(size_t)batch + i] = s1; state_out[2 * (size_t)batch + i] = s2;
            state_out[3 * (size_t)batch + i] = s3; state_out[4 * (size_t)batch + i] = s4;
            state_out[5 * (size_t)batch + i] = s5;
        }
    }
}

// Launch for nc = order + 1 coefficient rows (4 .. NMPC_MAX_COEFFS).
static void launch_prestep(int nc, cudaStream_t st, int batch, int M, const double *wx, const double *wy, const double *pose,
                           double *coeffs_out, double *cte_eth_out, const double *vel, double *state_out, int delay_mode,
                           double dt)
{
    const int grid = (batch + 127) / 128;
#define PRESTEP_ARGS batch, M, wx, wy, pose, coeffs_out, cte_eth_out, vel, state_out, delay_mode, dt
#define PRESTEP_CASE(K) case K: if (M <= 16) prestep_kernel<K, 16><<<grid, 128, 0, st>>>(PRESTEP_ARGS); \
                                else prestep_kernel<K, MAX_WAYPOINTS><<<grid, 128, 0, st>>>(PRESTEP_ARGS); break
    switch (nc) {
        PRESTEP_CASE(5); PRESTEP_CASE(6); PRESTEP_CASE(7); PRESTEP_CASE(8);
        default:
            if (M <= 16) prestep_kernel<4, 16><<<grid, 128, 0, st>>>(PRESTEP_ARGS);
            else prestep_kernel<4, MAX_WAYPOINTS><<<grid, 128, 0, st>>>(PRESTEP_ARGS);
            break;
    }
#undef PRESTEP_CASE
#undef PRESTEP_ARGS
}

// ================================================================ hard-first queue order
// Iteration counts range from 5 to the cap; the few slow problems are almost always the ones whose fitted
// path polynomial is wild (a 5 m window wrapped around a sharp corner gives |c2|, |c3| in the tens or
// thousands).  The work queue is therefore served in descending order of |c1|+|c2|+|c3| (bucketed by binary
// exponent): slow problems start first and the tail of a launch is filled with quick ones.  Results do not
// depend on the order (lanes are independent).  One CTA, counting sort with shared-memory atomics.
// Small on purpose (128 threads, few registers): it has to fit on an SM NEXT TO a resident solve CTA, or every
// launch would wait for an SM to drain completely before its solve kernel could even be queued.  Also resets the
// launch's work-queue head.
__global__ void __launch_bounds__(128) queue_order_kernel(int batch, const double *__restrict__ coeffs, int *__restrict__ order,
                                                          int *__restrict__ queue)
{
    __shared__ int hist[32], offs[32];
    if (threadIdx.x == 0) *queue = 0;
    if (threadIdx.x < 32) hist[threadIdx.x] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < batch; i += blockDim.x) {
        const double s = fabs(coeffs[(size_t)batch + i]) + fabs(coeffs[2 * (size_t)batch + i]) + fabs(coeffs[3 * (size_t)batch + i]);
        int b = 0;
        if (s == s) { int e; frexp(s + 1e-12, &e); b = min(31, max(0, e + 12)); } else b = 31;
        atomicAdd(&hist[b], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int b = 31; b >= 0; b--) { offs[b] = acc; acc += hist[b]; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < batch; i += blockDim.x) {
        const double s = fabs(coeffs[(size_t)batch + i]) + fabs(coeffs[2 * (size_t)batch + i]) + fabs(coeffs[3 * (size_t)batch + i]);
        int b = 0;
        if (s == s) { int e; frexp(s + 1e-12, &e); b = min(31, max(0, e + 12)); } else b = 31;
        order[atomicAdd(&offs[b], 1)] = i;
    }
}

// ================================================================ plan windowing (SURVEY 8f-2)
// Reference: MPCPlannerROS::getCutOffPlan (mpc_ros/src/mpc_planner_ros.cpp:266-291) erases plan points from the
// front while the squared distance to the robot does not grow (start value 10e5, :273): the plan then begins at the
// first point that is farther away than its predecessor, i.e. one past the nearest point.  downSamplePlan
// (:365-391) keeps every `step`-th point of the window, beginning with its first, and appends its last point (with
// path_length / waypoints_dist taken from the parameters instead of the reference's uninitialised members).
// Closed tracks: indices wrap; at most max_advance points are erased per tick.  One thread per robot.
// Checked against oracle/mpc_oracle.c (mpc_oracle_cutoff / _downsample), the restatement of the reference's code.
__global__ void window_kernel(int batch, const double *__restrict__ px, const double *__restrict__ py,
                              const int *__restrict__ track_off, const int *__restrict__ track_len,
                              const int *__restrict__ track_id, int *__restrict__ idx_io,
                              const double *__restrict__ pose, int win, int step, int max_advance,
                              double *__restrict__ wx, double *__restrict__ wy)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const int t = track_id[i], off = track_off[t], n = track_len[t];
    const double rx = pose[i], ry = pose[(size_t)batch + i];
    int j = idx_io[i] % n;
    double max_distance_sq = 10e5;                          // :273
    int erased = 0;
    while (erased < max_advance) {
        const int q = (j + erased) % n;
        const double dx = rx - px[off + q], dy = ry - py[off + q];
        const double d2 = dx * dx + dy * dy;
        if (max_distance_sq < d2) break;                    // :282-284: this point stays, it is the new plan start
        erased++;                                           // :285
        max_distance_sq = d2;                               // :286
    }
    j = (j + erased) % n;
    idx_io[i] = j;
    int m = 0;
    for (int a = 0; a < win; a += step, m++) {
        const int q = (j + a) % n;
        wx[(size_t)m * batch + i] = px[off + q]; wy[(size_t)m * batch + i] = py[off + q];
    }
    const int q = (j + win - 1) % n;
    wx[(size_t)m * batch + i] = px[off + q]; wy[(size_t)m * batch + i] = py[off + q];
}

// ================================================================ result post-step (SURVEY 8a last row, 8f-1)
// Reference: Tracking::findBestPath after the solve, mpc_ros/src/driving_state.cpp:263-269:
//   w = res[0]; throttle = res[1]; speed = v + throttle * dt, clamped ABOVE at REF_V only.
// vel (3 x batch: v, previous w, previous throttle) is updated in place for the next tick's delay
// compensation (:191-193, :245-251); cmd (2 x batch) = {linear.x, angular.z} (:115-116).
__global__ void poststep_kernel(int batch, const double *__restrict__ u0, double *__restrict__ vel,
                                const double *__restrict__ ref_vel, double ref_vel_all, double dt,
                                double *__restrict__ cmd)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const double w = u0[i], thr = u0[(size_t)batch + i];
    const double v = vel[i];
    const double rv = ref_vel ? ref_vel[i] : ref_vel_all;
    double speed = v + thr * dt;
    if (speed >= rv) speed = rv;
    vel[(size_t)batch + i] = w;
    vel[2 * (size_t)batch + i] = thr;
    cmd[i] = speed;
    cmd[(size_t)batch + i] = w;
}

// ================================================================ reference-speed schedule near the goal (8f-1)
// Reference: Tracking::deceleration, mpc_ros/src/driving_state.cpp:121-141.  Inside the braking distance
// v^2 / max_throttle of the goal REF_V becomes max_throttle * distance, limited below at min_speed; the
// reference's first branch (speed > REF_V -> max_speed) is kept as it is written.  REF_V persists per robot.
__global__ void decel_kernel(int batch, const double *__restrict__ pose, const double *__restrict__ goal,
                             const double *__restrict__ vel, double max_throttle, double max_speed, double min_speed,
                             double *__restrict__ ref_vel)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const double dist = hypot(pose[i] - goal[i], pose[(size_t)batch + i] - goal[(size_t)batch + i]);
    const double v = vel[i];
    if (dist <= v * v / max_throttle) {
        const double speed = max_throttle * dist;
        double rv = ref_vel[i];
        if (speed > rv) rv = max_speed;
        else if (speed < min_speed) rv = min_speed;
        else rv = speed;
        ref_vel[i] = rv;
    }
}

// ================================================================ plant step (SURVEY 8d config 5, 8f-1)
// Not in the reference (there the robot or Gazebo is the plant): unicycle driven by the command,
//   x += v cos(theta) dt, y += v sin(theta) dt, theta += w dt (wrapped to [-pi, pi)), v = commanded speed.
__global__ void plant_kernel(int batch, const double *__restrict__ cmd, double *__restrict__ pose, double *__restrict__ vel,
                             double dt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const double speed = cmd[i], w = cmd[(size_t)batch + i];
    double th = pose[2 * (size_t)batch + i];
    double sn, cs;
    sincos(th, &sn, &cs);
    pose[i] += speed * cs * dt;
    pose[(size_t)batch + i] += speed * sn * dt;
    const double kPi = 3.14159265358979323846;
    th += w * dt + kPi;
    th -= 2.0 * kPi * floor(th / (2.0 * kPi));
    pose[2 * (size_t)batch + i] = th - kPi;
    vel[i] = speed;
}

// ================================================================ warm-start shift
// Next tick's warm start from this tick's solution: every block of the record (6 state components,
// 2 controls, 6 multiplier components, 4 bound multipliers) moves one stage forward, the last entry is
// repeated.  (The solver re-derives the states by a roll-out; they are shifted only for completeness.)
__global__ void warm_shift_kernel(int batch, int N, const double *__restrict__ in, double *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    size_t off = 0;
    for (int blk = 0; blk < 18; blk++) {
        const int len = (blk < 6) ? N : (blk < 8) ? N - 1 : (blk < 14) ? N : N - 1;
        for (int j = 0; j < len; j++) {
            const int src = (j + 1 < len) ? j + 1 : len - 1;
            out[(off + j) * (size_t)batch + i] = in[(off + src) * (size_t)batch + i];
        }
        off += len;
    }
}

// ================================================================ FP64 probes
// mode 0: throughput -- 8 independent DFMA chains per thread, every SM busy
// mode 1..: single-warp issue/latency probes (see mpc_b200_debug_fp64_probe)
template <int ILP>
__global__ void dfma_kernel(double *out, int iters, int active_lanes, long long *cycles)
{
    double acc[ILP];
    const double a = 1.0000001, b = 1e-9;
#pragma unroll
    for (int j = 0; j < ILP; j++) acc[j] = 1.0 + 1e-3 * (threadIdx.x + j);
    const bool act = (threadIdx.x & 31) < active_lanes;
    long long t0 = clock64();
    if (act) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int j = 0; j < ILP; j++) acc[j] = fma(acc[j], a, b);
        }
    }
    long long t1 = clock64();
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < ILP; j++) s += acc[j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (cycles && threadIdx.x == 0 && blockIdx.x == 0) cycles[0] = t1 - t0;
}

// ================================================================ solve-kernel specialisations
// Every compiled solve kernel.  enqueue_solve launches the entry whose key (kind, spt, warm, rate, nc) matches and whose
// lanes per CTA equal the launch's, else the run-time generic entry (cpb 0) of that key; mpc_b200_create raises the
// dynamic shared-memory limit of each.
struct SolveKernel {
    bool dual;        // nmpc_kernel_dual.cuh: full CTAs as two lane groups out of phase
    int spt, cpb;     // stages per stage thread; lanes per CTA (0: chosen at run time)
    bool warm, rate;  // warm start; rate-penalty variant (w_angvel_d / w_accel_d != 0, 44 slots per stage)
    int nc;           // coefficient rows: 4, or NMPC_MAX_COEFFS for a path polynomial of order 4..7
    const void *fn;
};
#define SK(S, C, W, R, NC) { false, S, C, W, R, NC, (const void *)nmpc::nmpc_solve_kernel<S, C, W, R, NC> }
#define SK_DUAL(W, R) { true, SPT, (R) ? 28 : 32, W, R, 4, (const void *)nmpc::nmpc_solve_kernel_dual<W, 4, R> }
static const SolveKernel kSolveKernels[] = {
    SK(SPT, 0, false, false, 4), SK(SPT, 32, false, false, 4), SK(SPT, 16, false, false, 4), SK(SPT, 8, false, false, 4),
    SK(SPT, 4, false, false, 4), SK(SPT, 1, false, false, 4),
    SK(SPT, 6, false, false, 4),                                  // N = 100 (BASELINE config 4)
    SK(SPT, 0, true, false, 4), SK(SPT, 32, true, false, 4),
    // 28 lanes: what the 44-slot stages of the rate-penalty variant leave room for at N = 20, the cfg defaults
    SK(SPT, 0, false, true, 4), SK(SPT, 0, true, true, 4), SK(SPT, 28, false, true, 4), SK(SPT, 28, true, true, 4),
    // narrow CTAs, one stage per stage thread (the closed loop of BASELINE config 5: 1,024 robots = 8 lanes per CTA)
    SK(1, 16, false, false, 4), SK(1, 8, false, false, 4), SK(1, 4, false, false, 4), SK(1, 1, false, false, 4),
    SK(1, 16, true, false, 4), SK(1, 8, true, false, 4), SK(1, 4, true, false, 4), SK(1, 1, true, false, 4),
    SK_DUAL(false, false), SK_DUAL(true, false), SK_DUAL(false, true), SK_DUAL(true, true),
    SK(SPT, 0, false, false, NMPC_MAX_COEFFS), SK(SPT, 0, true, false, NMPC_MAX_COEFFS),
    SK(SPT, 0, false, true, NMPC_MAX_COEFFS), SK(SPT, 0, true, true, NMPC_MAX_COEFFS),
};
#undef SK
#undef SK_DUAL

static const SolveKernel *find_solve_kernel(bool dual, int spt, int pb, bool warm, bool rate, int nc)
{
    const SolveKernel *generic = NULL;
    for (const SolveKernel &k : kSolveKernels) {
        if (k.dual != dual || k.spt != spt || k.warm != warm || k.rate != rate || k.nc != nc) continue;
        if (k.cpb == pb) return &k;
        if (k.cpb == 0) generic = &k;
    }
    return generic;
}

// ================================================================ handle
// Host-buffer results of a call whose D2H copies are enqueued: the copies that went through the staging area h_out
// (the destination was not page-locked), moved to their destination by fetch_finish.
struct Fetch {
    bool active = false;
    int n = 0;
    struct { void *dst; const void *src; size_t bytes; } staged[8];
};

struct mpc_b200_handle {
    mpc_b200_params params;
    int device = 0;
    int max_batch = 0;
    int num_sms = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = NULL;
    cudaEvent_t ev0 = NULL, ev1 = NULL;
    // device scratch
    double *d_state = NULL, *d_coeffs = NULL, *d_refv = NULL, *d_u0 = NULL, *d_pred = NULL, *d_obj = NULL, *d_kkt = NULL,
           *d_warm_out = NULL;
    int *d_status = NULL, *d_iters = NULL;
    double *d_wx = NULL, *d_wy = NULL, *d_pose = NULL, *d_cte = NULL, *d_vel = NULL;
    // pinned staging
    double *h_in = NULL, *h_out = NULL;
    size_t h_in_bytes = 0, h_out_bytes = 0;
    int pred_steps = 0;        // horizon the scratch was sized for
    double last_kernel_s = 0.0;
    long long launches = 0;    // API calls that launched work (also drives the queue / order rings)
    long long kernels = 0;     // kernels launched by this handle
    long long *d_prof = NULL;
    int opt_dual = 1;
    int opt_spt1 = 1;
    int *d_queue = NULL;       // ring of work-queue heads, one per in-flight launch
    int *d_order = NULL;       // ring of hard-first queue orders (order_ring x max_batch)
    int order_ring = 0;        // launches that may be in flight on this handle at once (16 .. 1024)
    int opt_order = 1;         // option: serve the queue hard-first (default on)
    int max_ctas = 0;          // option: cap on the persistent grid (0 = one CTA per SM)
    int opt_pb = 0;            // option: problems per CTA (0 = auto)
    int opt_nc = 4;            // option: rows of the coeffs arrays = polynomial order + 1 (4 .. NMPC_MAX_COEFFS; default 4)
    double *d_io = NULL;       // packed tick buffer (mpc_b200_track_packed_*), allocated on first use
    size_t d_io_doubles = 0;
    double *d_warm_stage_in = NULL, *d_warm_stage_out = NULL;   // device staging of HOST warm-start records, allocated on first use
    const void *pin_ptr[8] = {}; bool pin_val[8] = {}; int pin_next = 0;   // small cache of cudaPointerGetAttributes answers
    cudaEvent_t *slot_ev = NULL;   // one event per queue / order ring slot: a slot is reused only after its launch has finished
    Fetch pending;         // the tick in flight (mpc_b200_track_*_submit / _wait)
    std::string last_err;
};

static bool is_device_ptr(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. a pinned torch tensor): copies can go
// straight from / to the caller's buffer without the handle's staging area
static bool is_pinned_host(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

// The tick entry points see the same caller buffers every tick: remember the answers (a buffer's kind does not
// change while it is allocated; a freed-and-reallocated address of another kind would be a caller bug either way).
static bool is_pinned_cached(mpc_b200_handle *h, const void *p)
{
    if (!p) return false;
    for (int i = 0; i < 8; i++) if (h->pin_ptr[i] == p) return h->pin_val[i];
    const bool v = is_pinned_host(p);
    h->pin_ptr[h->pin_next] = p; h->pin_val[h->pin_next] = v; h->pin_next = (h->pin_next + 1) & 7;
    return v;
}

static int cuda_fail(mpc_b200_handle *h, cudaError_t e, const char *what)
{
    if (h) h->last_err = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();
    return MPC_B200_ERR_CUDA;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(h, e_, #call); } while (0)

// last_kernel_seconds from the events around the last timed launch (once the stream has been synchronised)
static void read_kernel_time(mpc_b200_handle *h)
{
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) == cudaSuccess) h->last_kernel_s = 1e-3 * ms; else cudaGetLastError();
}

// End of a device-only entry point that launched one kernel: count it; without a caller stream, return once it has run.
static int finish_device_call(mpc_b200_handle *h, cudaStream_t st, void *stream_v)
{
    CK(cudaGetLastError());
    h->launches++; h->kernels++;
    if (!stream_v) CK(cudaStreamSynchronize(st));
    return MPC_B200_OK;
}

static void free_scratch(mpc_b200_handle *h)
{
    cudaFree(h->d_state); cudaFree(h->d_coeffs); cudaFree(h->d_refv); cudaFree(h->d_u0); cudaFree(h->d_pred);
    cudaFree(h->d_obj); cudaFree(h->d_kkt); cudaFree(h->d_status); cudaFree(h->d_iters); cudaFree(h->d_warm_out);
    cudaFree(h->d_wx); cudaFree(h->d_wy); cudaFree(h->d_pose); cudaFree(h->d_cte); cudaFree(h->d_vel);
    cudaFreeHost(h->h_in); cudaFreeHost(h->h_out);
    if (h->d_io) { cudaFree(h->d_io); h->d_io = NULL; h->d_io_doubles = 0; }
    if (h->d_warm_stage_in) { cudaFree(h->d_warm_stage_in); h->d_warm_stage_in = NULL; }
    if (h->d_warm_stage_out) { cudaFree(h->d_warm_stage_out); h->d_warm_stage_out = NULL; }
    h->d_state = h->d_coeffs = h->d_refv = h->d_u0 = h->d_pred = h->d_obj = h->d_kkt = h->d_warm_out = NULL;
    h->d_status = h->d_iters = NULL; h->d_wx = h->d_wy = h->d_pose = h->d_cte = h->d_vel = NULL;
    h->h_in = h->h_out = NULL;
}

// what does not depend on the horizon: the work-queue heads, the queue orders and their per-slot events
static void free_rings(mpc_b200_handle *h)
{
    if (h->d_prof) { cudaFree(h->d_prof); h->d_prof = NULL; }
    if (h->d_queue) { cudaFree(h->d_queue); h->d_queue = NULL; }
    if (h->d_order) { cudaFree(h->d_order); h->d_order = NULL; }
    if (h->slot_ev) {
        for (int i = 0; i < h->order_ring; i++) if (h->slot_ev[i]) cudaEventDestroy(h->slot_ev[i]);
        free(h->slot_ev); h->slot_ev = NULL;
    }
}

static int alloc_rings(mpc_b200_handle *h)
{
    const size_t B = (size_t)h->max_batch;
    CK(cudaMalloc(&h->d_queue, sizeof(int) * QUEUE_RING));
    h->order_ring = (int)((size_t)(1 << 22) / B);
    if (h->order_ring < 16) h->order_ring = 16;
    if (h->order_ring > QUEUE_RING) h->order_ring = QUEUE_RING;
    CK(cudaMalloc(&h->d_order, sizeof(int) * (size_t)h->order_ring * B));
    h->slot_ev = (cudaEvent_t *)calloc((size_t)h->order_ring, sizeof(cudaEvent_t));
    if (!h->slot_ev) return MPC_B200_ERR_NOMEM;
    return MPC_B200_OK;
}

static int alloc_scratch(mpc_b200_handle *h, int steps)
{
    const size_t B = (size_t)h->max_batch, N = (size_t)steps;
    h->pred_steps = (int)N;
    CK(cudaMalloc(&h->d_state, sizeof(double) * 6 * B));
    CK(cudaMalloc(&h->d_coeffs, sizeof(double) * NMPC_MAX_COEFFS * B));
    CK(cudaMalloc(&h->d_refv, sizeof(double) * B));
    CK(cudaMalloc(&h->d_u0, sizeof(double) * 2 * B));
    CK(cudaMalloc(&h->d_pred, sizeof(double) * 3 * N * B));
    CK(cudaMalloc(&h->d_obj, sizeof(double) * B));
    CK(cudaMalloc(&h->d_kkt, sizeof(double) * B));
    CK(cudaMalloc(&h->d_status, sizeof(int) * B));
    CK(cudaMalloc(&h->d_iters, sizeof(int) * B));
    CK(cudaMalloc(&h->d_wx, sizeof(double) * MAX_WAYPOINTS * B));
    CK(cudaMalloc(&h->d_wy, sizeof(double) * MAX_WAYPOINTS * B));
    CK(cudaMalloc(&h->d_pose, sizeof(double) * 3 * B));
    CK(cudaMalloc(&h->d_cte, sizeof(double) * 2 * B));
    CK(cudaMalloc(&h->d_vel, sizeof(double) * 3 * B));
    h->d_warm_out = NULL;
    h->h_in_bytes = sizeof(double) * (2 * MAX_WAYPOINTS + 3 + 11) * B;
    h->h_out_bytes = sizeof(double) * (2 + 3 * N + 2 + 2 + 3 + 1 + 6) * B;   // u0 pred obj kkt cmd vel status/iters + slack
    CK(cudaMallocHost(&h->h_in, h->h_in_bytes));
    CK(cudaMallocHost(&h->h_out, h->h_out_bytes));
    return MPC_B200_OK;
}

static int check_params(const mpc_b200_params *p)
{
    if (!p) return MPC_B200_ERR_INVALID;
    if (p->mpc_steps < 2 || p->mpc_steps > 600) return MPC_B200_ERR_INVALID;
    if (!(p->dt > 0.0) || !(p->max_angvel > 0.0) || !(p->max_throttle > 0.0)) return MPC_B200_ERR_INVALID;
    if (p->w_angvel_d < 0.0 || p->w_accel_d < 0.0) return MPC_B200_ERR_INVALID;
    return MPC_B200_OK;
}

extern "C" {

int mpc_b200_version(void) { return MPC_B200_VERSION; }

int mpc_b200_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *mpc_b200_strerror(int code)
{
    switch (code) {
        case MPC_B200_OK: return "ok";
        case MPC_B200_ERR_INVALID: return "invalid argument";
        case MPC_B200_ERR_CUDA: return "CUDA error or no usable device (this library has no CPU path)";
        case MPC_B200_ERR_UNSUPPORTED: return "parameter combination not supported by the GPU path";
        case MPC_B200_ERR_IO: return "cannot read parameter file";
        case MPC_B200_ERR_NOMEM: return "out of memory";
        default: return "unknown error";
    }
}

const char *mpc_b200_last_cuda_error(const mpc_b200_handle *h) { return h ? h->last_err.c_str() : ""; }

int32_t mpc_b200_warm_size(int32_t N) { return (8 * N - 2) + 6 * N + 4 * (N - 1); }

int mpc_b200_create(mpc_b200_handle **out, const mpc_b200_params *p, int32_t max_batch, int32_t device)
{
    if (!out || max_batch < 1) return MPC_B200_ERR_INVALID;
    *out = NULL;
    int rc = check_params(p);
    if (rc != MPC_B200_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return MPC_B200_ERR_CUDA;
    }
    mpc_b200_handle *h = new (std::nothrow) mpc_b200_handle();
    if (!h) return MPC_B200_ERR_NOMEM;
    h->params = *p; h->device = device; h->max_batch = max_batch;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    int sms = 0, optin = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e != cudaSuccess) { cudaGetLastError(); delete h; return MPC_B200_ERR_CUDA; }
    h->num_sms = sms; h->smem_optin = (size_t)optin;
    for (const SolveKernel &k : kSolveKernels)
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e != cudaSuccess) { cudaGetLastError(); delete h; return MPC_B200_ERR_CUDA; }
    rc = alloc_scratch(h, h->params.mpc_steps);
    if (rc == MPC_B200_OK) rc = alloc_rings(h);
    if (rc != MPC_B200_OK) { free_scratch(h); free_rings(h); delete h; return rc; }
    *out = h;
    return MPC_B200_OK;
}

void mpc_b200_destroy(mpc_b200_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();          // launches given caller streams may still be using the rings
    free_scratch(h);
    free_rings(h);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int mpc_b200_stream_create(int32_t device, void **stream_out)
{
    if (!stream_out) return MPC_B200_ERR_INVALID;
    cudaStream_t s = NULL;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        return MPC_B200_ERR_CUDA;
    }
    *stream_out = (void *)s;
    return MPC_B200_OK;
}

int mpc_b200_stream_destroy(void *stream)
{
    if (!stream) return MPC_B200_ERR_INVALID;
    if (cudaStreamDestroy((cudaStream_t)stream) != cudaSuccess) { cudaGetLastError(); return MPC_B200_ERR_CUDA; }
    return MPC_B200_OK;
}

int mpc_b200_stream_synchronize(void *stream)
{
    if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) { cudaGetLastError(); return MPC_B200_ERR_CUDA; }
    return MPC_B200_OK;
}

int mpc_b200_set_params(mpc_b200_handle *h, const mpc_b200_params *p)
{
    if (!h) return MPC_B200_ERR_INVALID;
    int rc = check_params(p);
    if (rc != MPC_B200_OK) return rc;
    if (h->pending.active) return MPC_B200_ERR_INVALID;      // a submitted tick must be waited for first
    const bool regrow = p->mpc_steps > h->pred_steps;
    if (regrow) {
        // A longer horizon needs larger result / staging buffers.  Launches enqueued with CALLER streams may still be
        // running: wait for the whole device, not just the handle's stream.  The queue / order rings do not depend on
        // the horizon and are kept.  The new parameters are adopted only once the new scratch exists.
        CK(cudaSetDevice(h->device));
        CK(cudaDeviceSynchronize());
        free_scratch(h);
        rc = alloc_scratch(h, p->mpc_steps);
        if (rc != MPC_B200_OK) {
            // back to a usable handle with the OLD parameters
            free_scratch(h);
            if (alloc_scratch(h, h->params.mpc_steps) != MPC_B200_OK) free_scratch(h);
            return rc;
        }
    }
    h->params = *p;
    return MPC_B200_OK;
}

int mpc_b200_get_params(const mpc_b200_handle *h, mpc_b200_params *p)
{
    if (!h || !p) return MPC_B200_ERR_INVALID;
    *p = h->params;
    return MPC_B200_OK;
}

int mpc_b200_set_option(mpc_b200_handle *h, const char *name, double value)
{
    if (!h || !name) return MPC_B200_ERR_INVALID;
    if (!strcmp(name, "max_ctas")) h->max_ctas = value > 0 ? (int)value : 0;
    else if (!strcmp(name, "problems_per_cta")) h->opt_pb = value > 0 ? (int)value : 0;
    else if (!strcmp(name, "hard_first")) h->opt_order = value != 0.0;
    else if (!strcmp(name, "narrow_one_stage")) h->opt_spt1 = value != 0.0;   // narrow CTAs: one stage per stage thread (latency mode)
    else if (!strcmp(name, "dual_groups")) h->opt_dual = value != 0.0;   // full CTAs as two lane groups out of phase (nmpc_kernel_dual.cuh)
    else if (!strcmp(name, "poly_coeffs")) {
        // rows of the coeffs arrays of mpc_b200_solve_batch: order of the path polynomial + 1 (mpc_planner.cpp:186-190
        // takes any order; the pre-step entry points always fit and write a cubic, 4 rows)
        if (value < 4 || value > NMPC_MAX_COEFFS) return MPC_B200_ERR_INVALID;
        h->opt_nc = (int)value;
    }
    else return MPC_B200_ERR_INVALID;
    return MPC_B200_OK;
}

double mpc_b200_last_kernel_seconds(const mpc_b200_handle *h) { return h ? h->last_kernel_s : 0.0; }
int64_t mpc_b200_launch_count(const mpc_b200_handle *h) { return h ? h->kernels : 0; }

// Problems per CTA: as many as shared memory and the thread budget allow, but spread a small
// batch over all SMs (the CTA's latency does not depend on how many lanes are active).
static int choose_pb(const mpc_b200_handle *h, int N, int batch, int nslots)
{
    const int NG = (N + SPT - 1) / SPT;
    int pb = 32;
    if (pb > STAGE_THREADS / NG) pb = STAGE_THREADS / NG;
    while (pb > 1 && nmpc::smem_bytes(N, NG, pb, nslots) > h->smem_optin) pb--;
    if (h->opt_pb > 0) return h->opt_pb < pb ? h->opt_pb : pb;
    // a small batch is spread over all SMs; snap to the lane counts that have a compiled specialisation
    const int spread = (batch + h->num_sms - 1) / h->num_sms;
    if (spread < pb) {
        int want = spread < 1 ? 1 : spread;
        if (nslots == nmpc::NSLOTS) {
            if (want > 16) want = 32; else if (want > 8) want = 16; else if (want > 4) want = 8;
            else if (want > 1) want = 4;
        }
        if (want < pb) pb = want;
    }
    return pb;
}

// Enqueue one batched solve on `st`; every pointer is DEVICE memory.
static int enqueue_solve(mpc_b200_handle *h, int32_t batch, const double *d_state, const double *d_coeffs,
                         const double *d_refv, const double *d_warm_in, double *d_u0, double *d_pred, double *d_obj,
                         int32_t *d_status, int32_t *d_iters, double *d_kkt, double *d_warm_out, cudaStream_t st,
                         bool timed = true)
{
    const mpc_b200_params &P = h->params;
    const int N = P.mpc_steps;
    SolveArgs a;
    a.prm.N = N; a.prm.dt = P.dt; a.prm.ref_cte = P.ref_cte; a.prm.ref_etheta = P.ref_etheta; a.prm.ref_vel = P.ref_vel;
    a.prm.w_cte = P.w_cte; a.prm.w_etheta = P.w_etheta; a.prm.w_vel = P.w_vel; a.prm.w_angvel = P.w_angvel;
    a.prm.w_accel = P.w_accel; a.prm.max_angvel = P.max_angvel; a.prm.max_throttle = P.max_throttle;
    a.prm.tol = P.tol > 0.0 ? P.tol : 1e-8;
    a.prm.max_iter = P.max_iter > 0 ? P.max_iter : 100;
    a.prm.grp = SPT;     // (adjusted below once the lanes per CTA are known)
    a.prm.idt = 1.0 / P.dt;
    a.prm.i_mnb = 1.0 / (double)(6 * N + 4 * (N - 1)); a.prm.i_nb = 1.0 / (double)(4 * (N - 1));
    a.prm.warm_mu = P.warm_mu_init > 0.0 ? P.warm_mu_init : 1e-3;
    // +-bound_value on the states (mpc_planner.cpp:303-312) carries no barrier term here: a point within 0.1 % of
    // it is reported as MPC_B200_STATUS_BOUND_ACTIVE instead of success (nmpc_phases.cuh, ctrl_decide)
    a.prm.bound_chk = (P.bound_value > 0.0 ? P.bound_value : 1e3) * (1.0 - 1e-3);
    a.batch = batch;
    a.ncoef = h->opt_nc;
    const bool rate = P.w_angvel_d != 0.0 || P.w_accel_d != 0.0;
    const int nslots = rate ? nmpc::NSLOTS_RATE : nmpc::NSLOTS;
    a.prm.w_angvel_d = P.w_angvel_d; a.prm.w_accel_d = P.w_accel_d;
    a.PB = choose_pb(h, N, batch, nslots);
    a.prof = h->d_prof;
    a.state = d_state; a.coeffs = d_coeffs; a.ref_vel = d_refv; a.warm_in = d_warm_in;
    a.u0 = d_u0; a.pred = d_pred; a.obj = d_obj; a.status = d_status; a.iters = d_iters; a.kkt = d_kkt; a.warm_out = d_warm_out;

    // Narrow CTAs (small batches spread over the SMs, a single MPC::Solve) are latency-bound: one stage per stage thread
    // instead of two halves the stage phases (plain variant, the compiled lane counts).
    const int spt1_threads = NMPC_CTRL_THREADS + ((N * a.PB + 31) / 32) * 32;
    const int spt = (h->opt_spt1 && !rate && a.ncoef <= 4 && (a.PB == 16 || a.PB == 8 || a.PB == 4 || a.PB == 1) &&
                     spt1_threads <= NMPC_MAX_THREADS(1, a.PB)) ? 1 : SPT;
    a.prm.grp = spt;
    const int NG = (N + spt - 1) / spt;
    // full CTAs: two lane groups out of phase, one stage per stage thread and group
    const bool dual = h->opt_dual && a.ncoef <= 4 && a.PB == (rate ? 28 : 32) && N > 10 && N <= NMPC_DUAL_MAX_N;
    const SolveKernel *kern = find_solve_kernel(dual, spt, a.PB, a.warm_in != NULL, rate, a.ncoef > 4 ? NMPC_MAX_COEFFS : 4);
    if (!kern) {
        h->last_err = "no compiled solve kernel for this configuration";
        return MPC_B200_ERR_UNSUPPORTED;
    }
    const int threads = NMPC_CTRL_THREADS + ((dual ? 16 * N : NG * a.PB) + 31) / 32 * 32;
    // persistent grid: at most one CTA per SM (or the max_ctas option); lanes refill from the queue
    int grid = (batch + a.PB - 1) / a.PB;
    const int cap = h->max_ctas > 0 ? h->max_ctas : h->num_sms;
    if (grid > cap) grid = cap;
    const size_t smem = nmpc::smem_bytes(N, NG, a.PB, nslots);
    // Ring slot of this launch (work-queue head + queue order).  A slot is reused only when the launch that had it
    // last has finished: more than order_ring launches in flight is refused, not silently aliased.
    const int slot = (int)(h->launches % h->order_ring);
    if (h->slot_ev[slot]) {
        const cudaError_t q = cudaEventQuery(h->slot_ev[slot]);
        if (q == cudaErrorNotReady) {
            h->last_err = "too many launches in flight on this handle (see mpc_b200_solve_batch, `stream`)";
            return MPC_B200_ERR_INVALID;
        }
        if (q != cudaSuccess) return cuda_fail(h, q, "cudaEventQuery(slot)");
    } else {
        CK(cudaEventCreateWithFlags(&h->slot_ev[slot], cudaEventDisableTiming));
    }
    a.queue = h->d_queue + slot;
    a.order = NULL;
    if (h->opt_order && batch > grid * a.PB) {      // only matters when lanes work through several problems
        a.order = h->d_order + (size_t)slot * h->max_batch;
        queue_order_kernel<<<1, 128, 0, st>>>(batch, a.coeffs, (int *)a.order, a.queue);
        CK(cudaGetLastError());
        h->kernels++;
    } else {
        CK(cudaMemsetAsync(a.queue, 0, sizeof(int), st));
    }
    if (timed) CK(cudaEventRecord(h->ev0, st));
    void *args[] = {&a};
    CK(cudaLaunchKernel(kern->fn, dim3(grid), dim3(threads), args, smem, st));
    if (timed) CK(cudaEventRecord(h->ev1, st));
    CK(cudaEventRecord(h->slot_ev[slot], st));
    h->launches++; h->kernels++;
    return MPC_B200_OK;
}

// D2H of results into host buffers: straight into `dst` when it is page-locked, else into the staging area at `stage`,
// from where fetch_finish moves it once the stream has run.
static cudaError_t fetch_copy(Fetch &f, void *dst, void *stage, const void *src, size_t bytes, bool pinned, cudaStream_t st)
{
    if (!pinned) f.staged[f.n++] = {dst, stage, bytes};
    return cudaMemcpyAsync(pinned ? dst : stage, src, bytes, cudaMemcpyDeviceToHost, st);
}

// the solve results (and a tick's cmd / vel) from the handle's scratch; h_out: u0 pred obj kkt cmd vel status iters
static int fetch_enqueue(mpc_b200_handle *h, Fetch &f, int32_t batch, double *u0, double *pred, double *obj, double *kkt,
                         int32_t *status, int32_t *iters, double *cmd, double *vel, cudaStream_t st)
{
    const size_t B = (size_t)batch, N = (size_t)h->params.mpc_steps;
    double *ho = h->h_out, *ho_obj = ho + (2 + 3 * N) * B, *ho_cmd = ho_obj + 2 * B, *ho_vel = ho_cmd + 2 * B;
    int *ho_status = reinterpret_cast<int *>(ho_vel + 3 * B);
    f = Fetch();
    CK(fetch_copy(f, u0, ho, h->d_u0, sizeof(double) * 2 * B, is_pinned_cached(h, u0), st));
    CK(fetch_copy(f, pred, ho + 2 * B, h->d_pred, sizeof(double) * 3 * N * B, is_pinned_cached(h, pred), st));
    if (obj) CK(fetch_copy(f, obj, ho_obj, h->d_obj, sizeof(double) * B, is_pinned_cached(h, obj), st));
    if (kkt) CK(fetch_copy(f, kkt, ho_obj + B, h->d_kkt, sizeof(double) * B, is_pinned_cached(h, kkt), st));
    if (status) CK(fetch_copy(f, status, ho_status, h->d_status, sizeof(int) * B, is_pinned_cached(h, status), st));
    if (iters) CK(fetch_copy(f, iters, ho_status + B, h->d_iters, sizeof(int) * B, is_pinned_cached(h, iters), st));
    if (cmd) CK(fetch_copy(f, cmd, ho_cmd, h->d_cte, sizeof(double) * 2 * B, is_pinned_cached(h, cmd), st));
    if (vel) CK(fetch_copy(f, vel, ho_vel, h->d_vel, sizeof(double) * 3 * B, is_pinned_cached(h, vel), st));
    f.active = true;
    return MPC_B200_OK;
}

static int fetch_finish(mpc_b200_handle *h, Fetch &f, cudaStream_t st)
{
    if (!f.active) return MPC_B200_OK;
    f.active = false;
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < f.n; i++) memcpy(f.staged[i].dst, f.staged[i].src, f.staged[i].bytes);
    read_kernel_time(h);
    return MPC_B200_OK;
}

int mpc_b200_solve_batch(mpc_b200_handle *h, int32_t batch,
                         const double *state, const double *coeffs, const double *ref_vel,
                         const double *warm_in,
                         double *u0, double *pred, double *obj, int32_t *status, int32_t *iters,
                         double *kkt_res, double *warm_out, void *stream_v)
{
    NvtxRange nv("mpc_b200_solve_batch");
    if (!h || batch < 0 || batch > h->max_batch || !state || !coeffs || !u0 || !pred) return MPC_B200_ERR_INVALID;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    const size_t B = (size_t)batch;
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;

    const bool dev_in = is_device_ptr(state);
    const bool dev_out = is_device_ptr(u0);
    if (is_device_ptr(coeffs) != dev_in || (ref_vel && is_device_ptr(ref_vel) != dev_in)) return MPC_B200_ERR_INVALID;
    // Warm-start records are large and meant to stay on the device between ticks; HOST records are accepted too
    // (SURVEY 8b "ownership": any buffer may be host memory) and staged through device buffers the handle keeps.
    const size_t wsz = (size_t)mpc_b200_warm_size(h->params.mpc_steps);
    double *host_warm_out = NULL;
    if (warm_in && !is_device_ptr(warm_in)) {
        if (!h->d_warm_stage_in) CK(cudaMalloc(&h->d_warm_stage_in, sizeof(double) * (size_t)mpc_b200_warm_size(h->pred_steps) * h->max_batch));
        CK(cudaMemcpyAsync(h->d_warm_stage_in, warm_in, sizeof(double) * wsz * B, cudaMemcpyHostToDevice, st));
        warm_in = h->d_warm_stage_in;
    }
    if (warm_out && !is_device_ptr(warm_out)) {
        if (!h->d_warm_stage_out) CK(cudaMalloc(&h->d_warm_stage_out, sizeof(double) * (size_t)mpc_b200_warm_size(h->pred_steps) * h->max_batch));
        host_warm_out = warm_out;
        warm_out = h->d_warm_stage_out;
    }
    if (is_device_ptr(pred) != dev_out || (obj && is_device_ptr(obj) != dev_out) ||
        (status && is_device_ptr(status) != dev_out) || (iters && is_device_ptr(iters) != dev_out) ||
        (kkt_res && is_device_ptr(kkt_res) != dev_out))
        return MPC_B200_ERR_INVALID;

    const double *ds = state, *dc = coeffs, *dr = ref_vel;
    if (!dev_in) {
        double *hi = h->h_in;
        const double *src_s = state, *src_c = coeffs, *src_r = ref_vel;
        if (!is_pinned_host(state)) { memcpy(hi, state, sizeof(double) * 6 * B); src_s = hi; }
        const size_t nc = (size_t)h->opt_nc;
        if (!is_pinned_host(coeffs)) { memcpy(hi + 6 * B, coeffs, sizeof(double) * nc * B); src_c = hi + 6 * B; }
        if (ref_vel && !is_pinned_host(ref_vel)) { memcpy(hi + (6 + nc) * B, ref_vel, sizeof(double) * B); src_r = hi + (6 + nc) * B; }
        // state and coeffs scratch are separate allocations: two copies (three with ref_vel)
        CK(cudaMemcpyAsync(h->d_state, src_s, sizeof(double) * 6 * B, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(h->d_coeffs, src_c, sizeof(double) * nc * B, cudaMemcpyHostToDevice, st));
        if (ref_vel) CK(cudaMemcpyAsync(h->d_refv, src_r, sizeof(double) * B, cudaMemcpyHostToDevice, st));
        ds = h->d_state; dc = h->d_coeffs; dr = ref_vel ? h->d_refv : NULL;
    }
    int rc;
    if (dev_out)
        rc = enqueue_solve(h, batch, ds, dc, dr, warm_in, u0, pred, obj, status, iters, kkt_res, warm_out, st,
                           !(dev_in && stream_v));      // asynchronous calls are not timed (last_kernel_seconds)
    else
        rc = enqueue_solve(h, batch, ds, dc, dr, warm_in, h->d_u0, h->d_pred, h->d_obj, h->d_status, h->d_iters, h->d_kkt,
                           warm_out, st);
    if (rc != MPC_B200_OK) return rc;
    if (host_warm_out) {
        CK(cudaMemcpyAsync(host_warm_out, warm_out, sizeof(double) * wsz * B, cudaMemcpyDeviceToHost, st));
        if (dev_out) CK(cudaStreamSynchronize(st));      // a host buffer is filled when the call returns
    }

    if (!dev_out) {
        Fetch f;
        rc = fetch_enqueue(h, f, batch, u0, pred, obj, kkt_res, status, iters, NULL, NULL, st);
        if (rc != MPC_B200_OK) return rc;
        return fetch_finish(h, f, st);
    }
    if (!(dev_in && stream_v)) {
        CK(cudaStreamSynchronize(st));
        read_kernel_time(h);
    }
    return MPC_B200_OK;
}

// One control tick on `st` once its inputs are on the device: pre-step into the handle's state / coeffs scratch, solve,
// post-step (cmd, and w / throttle back into vel for the next tick's delay compensation).
static int enqueue_tick(mpc_b200_handle *h, cudaStream_t st, int32_t batch, int32_t M, const double *d_wx, const double *d_wy,
                        const double *d_pose, double *d_vel, const double *d_refv, double *d_u0, double *d_pred,
                        double *d_obj, int32_t *d_status, int32_t *d_iters, double *d_kkt, double *d_cmd)
{
    launch_prestep(h->opt_nc, st, batch, M, d_wx, d_wy, d_pose, h->d_coeffs, NULL, d_vel, h->d_state, h->params.delay_mode,
                   h->params.dt);
    CK(cudaGetLastError());
    h->kernels++;
    const int rc = enqueue_solve(h, batch, h->d_state, h->d_coeffs, d_refv, NULL, d_u0, d_pred, d_obj, d_status, d_iters, d_kkt,
                                 NULL, st);
    if (rc != MPC_B200_OK) return rc;
    poststep_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, d_u0, d_vel, d_refv, h->params.ref_vel, h->params.dt, d_cmd);
    CK(cudaGetLastError());
    h->kernels++;
    return MPC_B200_OK;
}

int mpc_b200_track_submit(mpc_b200_handle *h, int32_t batch, int32_t M,
                          const double *wx, const double *wy, const double *pose, double *vel_inout,
                          const double *ref_vel, double *u0, double *pred, double *cmd_out,
                          double *obj, int32_t *status, int32_t *iters, double *kkt_res)
{
    NvtxRange nv("mpc_b200_track_submit");
    if (!h || batch < 0 || batch > h->max_batch || !wx || !wy || !pose || !vel_inout || !u0 || !pred) return MPC_B200_ERR_INVALID;
    if (M < 4 || M > MAX_WAYPOINTS) return MPC_B200_ERR_INVALID;
    if (is_device_ptr(wx) || is_device_ptr(u0)) return MPC_B200_ERR_UNSUPPORTED;   // host entry point; device callers chain the
                                                                                 // prestep / solve / poststep calls themselves
    if (h->pending.active) return MPC_B200_ERR_INVALID;                         // one tick in flight per handle
    if (M < h->opt_nc) return MPC_B200_ERR_INVALID;                             // fewer waypoints than coefficients
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    const size_t B = (size_t)batch;
    cudaStream_t st = h->stream;
    double *hi = h->h_in;
    const double *sx = wx, *sy = wy, *sp = pose, *sv = vel_inout, *sr = ref_vel;
    if (!is_pinned_cached(h, wx)) { memcpy(hi, wx, sizeof(double) * M * B); sx = hi; }
    if (!is_pinned_cached(h, wy)) { memcpy(hi + (size_t)M * B, wy, sizeof(double) * M * B); sy = hi + (size_t)M * B; }
    if (!is_pinned_cached(h, pose)) { memcpy(hi + 2 * (size_t)M * B, pose, sizeof(double) * 3 * B); sp = hi + 2 * (size_t)M * B; }
    if (!is_pinned_cached(h, vel_inout)) { memcpy(hi + 2 * (size_t)M * B + 3 * B, vel_inout, sizeof(double) * 3 * B); sv = hi + 2 * (size_t)M * B + 3 * B; }
    if (ref_vel && !is_pinned_cached(h, ref_vel)) { memcpy(hi + 2 * (size_t)M * B + 6 * B, ref_vel, sizeof(double) * B); sr = hi + 2 * (size_t)M * B + 6 * B; }
    CK(cudaMemcpyAsync(h->d_wx, sx, sizeof(double) * M * B, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_wy, sy, sizeof(double) * M * B, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_pose, sp, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->d_vel, sv, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, st));
    if (ref_vel) CK(cudaMemcpyAsync(h->d_refv, sr, sizeof(double) * B, cudaMemcpyHostToDevice, st));
    const int rc = enqueue_tick(h, st, batch, M, h->d_wx, h->d_wy, h->d_pose, h->d_vel, ref_vel ? h->d_refv : NULL, h->d_u0,
                                h->d_pred, h->d_obj, h->d_status, h->d_iters, h->d_kkt, h->d_cte);
    if (rc != MPC_B200_OK) return rc;
    // previous w / throttle for the next tick's delay compensation go back into the caller's vel buffer
    return fetch_enqueue(h, h->pending, batch, u0, pred, obj, kkt_res, status, iters, cmd_out, vel_inout, st);
}

// ---- packed tick: ONE caller buffer, one H2D and one D2H copy per tick
// Layout in doubles for (batch B, M waypoints, horizon N), blocks in this order:
//   wx M*B | wy M*B | pose 3B | [ref_vel B] | vel 3B | u0 2B | pred 3N*B | cmd 2B | obj B | kkt B | status | iters
// (status, iters: int32 arrays, each padded to a whole number of doubles).  Inputs = [wx .. vel], outputs = [vel .. iters]:
// the in/out block vel sits where the two ranges meet.
static size_t packed_layout(int N, size_t B, size_t M, int with_refv, int64_t *off /* 12, doubles */)
{
    size_t o = 0;
    off[0] = (int64_t)o; o += M * B;            // wx
    off[1] = (int64_t)o; o += M * B;            // wy
    off[2] = (int64_t)o; o += 3 * B;            // pose
    if (with_refv) { off[3] = (int64_t)o; o += B; } else off[3] = -1;
    off[4] = (int64_t)o; o += 3 * B;            // vel (in / out)
    off[5] = (int64_t)o; o += 2 * B;            // u0
    off[6] = (int64_t)o; o += 3 * (size_t)N * B;   // pred
    off[7] = (int64_t)o; o += 2 * B;            // cmd
    off[8] = (int64_t)o; o += B;                // obj
    off[9] = (int64_t)o; o += B;                // kkt
    off[10] = (int64_t)o; o += (B + 1) / 2;     // status (int32)
    off[11] = (int64_t)o; o += (B + 1) / 2;     // iters (int32)
    return o;
}

int64_t mpc_b200_track_packed_layout(const mpc_b200_handle *h, int32_t batch, int32_t M, int32_t with_ref_vel,
                                     int64_t *offsets_bytes12)
{
    if (!h || batch < 1 || M < 1) return MPC_B200_ERR_INVALID;
    int64_t off[12];
    const size_t n = packed_layout(h->params.mpc_steps, (size_t)batch, (size_t)M, with_ref_vel, off);
    if (offsets_bytes12) for (int i = 0; i < 12; i++) offsets_bytes12[i] = off[i] < 0 ? -1 : off[i] * (int64_t)sizeof(double);
    return (int64_t)(n * sizeof(double));
}

int mpc_b200_track_packed_submit(mpc_b200_handle *h, int32_t batch, int32_t M, int32_t with_ref_vel, void *io)
{
    NvtxRange nv("mpc_b200_track_packed_submit");
    if (!h || batch < 0 || batch > h->max_batch || !io) return MPC_B200_ERR_INVALID;
    if (M < 4 || M > MAX_WAYPOINTS || M < h->opt_nc) return MPC_B200_ERR_INVALID;
    if (h->pending.active) return MPC_B200_ERR_INVALID;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    const size_t B = (size_t)batch;
    const int N = h->params.mpc_steps;
    int64_t off[12];
    const size_t total = packed_layout(N, B, (size_t)M, with_ref_vel, off);
    if (h->d_io_doubles < total) {
        // sized for the largest tick this handle can see, so that it is allocated once
        int64_t o2[12];
        const size_t cap = packed_layout(h->pred_steps, (size_t)h->max_batch, MAX_WAYPOINTS, 1, o2);
        CK(cudaStreamSynchronize(h->stream));
        if (h->d_io) { cudaFree(h->d_io); h->d_io = NULL; h->d_io_doubles = 0; }
        CK(cudaMalloc(&h->d_io, sizeof(double) * cap));
        h->d_io_doubles = cap;
    }
    cudaStream_t st = h->stream;
    double *d = h->d_io;
    const size_t in_bytes = sizeof(double) * (size_t)off[5], out_off = sizeof(double) * (size_t)off[4],
                 out_bytes = sizeof(double) * total - out_off;
    if (is_device_ptr(io)) return MPC_B200_ERR_UNSUPPORTED;
    const bool pinned = is_pinned_cached(h, io);
    if (in_bytes > h->h_in_bytes || out_bytes > h->h_out_bytes) return MPC_B200_ERR_INVALID;
    const void *src = io;
    if (!pinned) { memcpy(h->h_in, io, in_bytes); src = h->h_in; }
    CK(cudaMemcpyAsync(d, src, in_bytes, cudaMemcpyHostToDevice, st));
    double *d_wx = d + off[0], *d_wy = d + off[1], *d_pose = d + off[2], *d_refv = off[3] >= 0 ? d + off[3] : NULL, *d_vel = d + off[4];
    double *d_u0 = d + off[5], *d_pred = d + off[6], *d_cmd = d + off[7], *d_obj = d + off[8], *d_kkt = d + off[9];
    int *d_status = reinterpret_cast<int *>(d + off[10]), *d_iters = reinterpret_cast<int *>(d + off[11]);
    const int rc = enqueue_tick(h, st, batch, M, d_wx, d_wy, d_pose, d_vel, d_refv, d_u0, d_pred, d_obj, d_status, d_iters, d_kkt,
                                d_cmd);
    if (rc != MPC_B200_OK) return rc;
    Fetch &f = h->pending;
    f = Fetch();
    CK(fetch_copy(f, (char *)io + out_off, h->h_out, (const char *)d + out_off, out_bytes, pinned, st));
    f.active = true;
    return MPC_B200_OK;
}

// ---- one GPU's contiguous slice of a batch held in the caller's SoA arrays (SURVEY 8e)
// The arrays have `ld` columns (the whole batch); this handle takes columns [offset, offset + batch).  Every array
// is moved by ONE strided copy (cudaMemcpy2DAsync: `rows` rows of batch doubles, pitch ld doubles) straight between
// the caller's page-locked arrays and the device: no staging, no host-side scatter / gather.
int mpc_b200_track_slice_submit(mpc_b200_handle *h, int32_t ld, int32_t offset, int32_t batch, int32_t M,
                                const double *wx, const double *wy, const double *pose, double *vel_inout,
                                const double *ref_vel, double *u0, double *pred, double *cmd_out,
                                double *obj, int32_t *status, int32_t *iters, double *kkt_res)
{
    NvtxRange nv("mpc_b200_track_slice_submit");
    if (!h || batch < 0 || batch > h->max_batch || ld < batch || offset < 0 || offset + batch > ld) return MPC_B200_ERR_INVALID;
    if (!wx || !wy || !pose || !vel_inout || !u0 || !pred) return MPC_B200_ERR_INVALID;
    if (M < 4 || M > MAX_WAYPOINTS || M < h->opt_nc) return MPC_B200_ERR_INVALID;
    if (h->pending.active) return MPC_B200_ERR_INVALID;
    if (batch == 0) return MPC_B200_OK;
    // DMA needs page-locked memory on both ends of a tick that is in flight
    if (!is_pinned_cached(h, wx) || !is_pinned_cached(h, wy) || !is_pinned_cached(h, pose) || !is_pinned_cached(h, vel_inout) ||
        !is_pinned_cached(h, u0) || !is_pinned_cached(h, pred) || (ref_vel && !is_pinned_cached(h, ref_vel)) ||
        (cmd_out && !is_pinned_cached(h, cmd_out)) || (obj && !is_pinned_cached(h, obj)) || (status && !is_pinned_cached(h, status)) ||
        (iters && !is_pinned_cached(h, iters)) || (kkt_res && !is_pinned_cached(h, kkt_res)))
        return MPC_B200_ERR_UNSUPPORTED;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    const size_t B = (size_t)batch, N = (size_t)h->params.mpc_steps;
    const size_t hp = sizeof(double) * (size_t)ld, dp = sizeof(double) * B, w = sizeof(double) * B;
#define H2D2(dst, src, rows) CK(cudaMemcpy2DAsync(dst, dp, (src) + offset, hp, w, (size_t)(rows), cudaMemcpyHostToDevice, st))
#define D2H2(dst, src, rows) CK(cudaMemcpy2DAsync((dst) + offset, hp, src, dp, w, (size_t)(rows), cudaMemcpyDeviceToHost, st))
    H2D2(h->d_wx, wx, M); H2D2(h->d_wy, wy, M); H2D2(h->d_pose, pose, 3); H2D2(h->d_vel, vel_inout, 3);
    if (ref_vel) H2D2(h->d_refv, ref_vel, 1);
    const int rc = enqueue_tick(h, st, batch, M, h->d_wx, h->d_wy, h->d_pose, h->d_vel, ref_vel ? h->d_refv : NULL, h->d_u0,
                                h->d_pred, h->d_obj, h->d_status, h->d_iters, h->d_kkt, h->d_cte);
    if (rc != MPC_B200_OK) return rc;
    D2H2(u0, h->d_u0, 2); D2H2(pred, h->d_pred, 3 * N); D2H2(vel_inout, h->d_vel, 3);
    if (cmd_out) D2H2(cmd_out, h->d_cte, 2);
    if (obj) D2H2(obj, h->d_obj, 1);
    if (kkt_res) D2H2(kkt_res, h->d_kkt, 1);
    if (status) CK(cudaMemcpyAsync(status + offset, h->d_status, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    if (iters) CK(cudaMemcpyAsync(iters + offset, h->d_iters, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
#undef H2D2
#undef D2H2
    h->pending = Fetch();      // nothing staged: the copies go straight into the caller's arrays
    h->pending.active = true;
    return MPC_B200_OK;
}

void *mpc_b200_host_alloc(size_t bytes)
{
    void *p = NULL;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return NULL; }
    return p;
}

void mpc_b200_host_free(void *p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) cudaGetLastError();
}

int mpc_b200_track_wait(mpc_b200_handle *h)
{
    if (!h) return MPC_B200_ERR_INVALID;
    if (!h->pending.active) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    return fetch_finish(h, h->pending, h->stream);
}

int mpc_b200_track_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                         const double *wx, const double *wy, const double *pose, double *vel_inout,
                         const double *ref_vel, double *u0, double *pred, double *cmd_out,
                         double *obj, int32_t *status, int32_t *iters, double *kkt_res)
{
    const int rc = mpc_b200_track_submit(h, batch, M, wx, wy, pose, vel_inout, ref_vel, u0, pred, cmd_out, obj, status, iters,
                                         kkt_res);
    if (rc != MPC_B200_OK) return rc;
    return mpc_b200_track_wait(h);
}

// The pre-step kernel with one of its optional outputs: cte / etheta (cte_eth_out), or the solver's initial state
// (state_out, from vel).  Inputs and outputs are each either all device or all host memory; host arrays are staged.
static int prestep_call(mpc_b200_handle *h, int32_t batch, int32_t M, const double *wx, const double *wy, const double *pose,
                        const double *vel, double *coeffs_out, double *cte_eth_out, double *state_out, void *stream_v)
{
    if (M < h->opt_nc || M > MAX_WAYPOINTS) return MPC_B200_ERR_INVALID;   // polyfit asserts order <= M-1 (driving_state.cpp:286)
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    const size_t B = (size_t)batch, nc = (size_t)h->opt_nc;
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    const bool dev_in = is_device_ptr(wx), dev_out = is_device_ptr(coeffs_out);
    if (is_device_ptr(wy) != dev_in || is_device_ptr(pose) != dev_in || (vel && is_device_ptr(vel) != dev_in))
        return MPC_B200_ERR_INVALID;
    if ((cte_eth_out && is_device_ptr(cte_eth_out) != dev_out) || (state_out && is_device_ptr(state_out) != dev_out))
        return MPC_B200_ERR_INVALID;
    const double *dwx = wx, *dwy = wy, *dpose = pose, *dvel = vel;
    if (!dev_in) {
        double *hi = h->h_in;
        memcpy(hi, wx, sizeof(double) * M * B);
        memcpy(hi + (size_t)M * B, wy, sizeof(double) * M * B);
        memcpy(hi + 2 * (size_t)M * B, pose, sizeof(double) * 3 * B);
        if (vel) memcpy(hi + 2 * (size_t)M * B + 3 * B, vel, sizeof(double) * 3 * B);
        CK(cudaMemcpyAsync(h->d_wx, hi, sizeof(double) * M * B, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(h->d_wy, hi + (size_t)M * B, sizeof(double) * M * B, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(h->d_pose, hi + 2 * (size_t)M * B, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, st));
        if (vel) CK(cudaMemcpyAsync(h->d_vel, hi + 2 * (size_t)M * B + 3 * B, sizeof(double) * 3 * B, cudaMemcpyHostToDevice, st));
        dwx = h->d_wx; dwy = h->d_wy; dpose = h->d_pose; dvel = vel ? h->d_vel : NULL;
    }
    double *dco = dev_out ? coeffs_out : h->d_coeffs;
    double *dce = cte_eth_out ? (dev_out ? cte_eth_out : h->d_cte) : NULL;
    double *dso = state_out ? (dev_out ? state_out : h->d_state) : NULL;
    CK(cudaEventRecord(h->ev0, st));
    launch_prestep(h->opt_nc, st, batch, M, dwx, dwy, dpose, dco, dce, dvel, dso, h->params.delay_mode, h->params.dt);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev1, st));
    h->launches++; h->kernels++;
    if (!dev_out) {
        // h_out: coeffs, then cte / etheta or the state
        Fetch f;
        CK(fetch_copy(f, coeffs_out, h->h_out, dco, sizeof(double) * nc * B, false, st));
        if (dce) CK(fetch_copy(f, cte_eth_out, h->h_out + nc * B, dce, sizeof(double) * 2 * B, false, st));
        if (dso) CK(fetch_copy(f, state_out, h->h_out + nc * B, dso, sizeof(double) * 6 * B, false, st));
        f.active = true;
        return fetch_finish(h, f, st);
    }
    if (!(dev_in && stream_v)) {
        CK(cudaStreamSynchronize(st));
        read_kernel_time(h);
    }
    return MPC_B200_OK;
}

int mpc_b200_polyfit_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                           const double *wx, const double *wy, const double *pose,
                           double *coeffs_out, double *cte_etheta_out, void *stream_v)
{
    NvtxRange nv("mpc_b200_polyfit_batch");
    if (!h || batch < 0 || batch > h->max_batch || !wx || !wy || !pose || !coeffs_out) return MPC_B200_ERR_INVALID;
    return prestep_call(h, batch, M, wx, wy, pose, NULL, coeffs_out, cte_etheta_out, NULL, stream_v);
}

int mpc_b200_prestep_batch(mpc_b200_handle *h, int32_t batch, int32_t M,
                           const double *wx, const double *wy, const double *pose, const double *vel,
                           double *coeffs_out, double *state_out, void *stream_v)
{
    NvtxRange nv("mpc_b200_prestep_batch");
    if (!h || batch < 0 || batch > h->max_batch || !wx || !wy || !pose || !vel || !coeffs_out || !state_out)
        return MPC_B200_ERR_INVALID;
    return prestep_call(h, batch, M, wx, wy, pose, vel, coeffs_out, NULL, state_out, stream_v);
}

int mpc_b200_window_batch(mpc_b200_handle *h, int32_t batch, const double *path_x, const double *path_y,
                          const int32_t *track_off, const int32_t *track_len, const int32_t *track_id,
                          int32_t *idx_inout, const double *pose, double *wx_out, double *wy_out, void *stream_v)
{
    if (!h || batch < 0 || !path_x || !path_y || !track_off || !track_len || !track_id || !idx_inout || !pose ||
        !wx_out || !wy_out) return MPC_B200_ERR_INVALID;
    if (!is_device_ptr(path_x) || !is_device_ptr(idx_inout) || !is_device_ptr(pose) || !is_device_ptr(wx_out))
        return MPC_B200_ERR_UNSUPPORTED;     // device-resident closed loop only
    const mpc_b200_params &P = h->params;
    const double wd = P.waypoints_dist > 0.0 ? P.waypoints_dist : 0.05;
    const int win = (int)lround(P.path_length / wd);
    const int step = (int)(P.path_length / 10.0 / wd);     // mpc_planner_ros.cpp:374
    if (win < 4 || step < 1 || (win + step - 1) / step + 1 > MAX_WAYPOINTS) return MPC_B200_ERR_INVALID;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    window_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, path_x, path_y, track_off, track_len, track_id, idx_inout,
                                                        pose, win, step, 64, wx_out, wy_out);
    return finish_device_call(h, st, stream_v);
}

int mpc_b200_poststep_batch(mpc_b200_handle *h, int32_t batch, const double *u0, double *vel_inout,
                            const double *ref_vel, double *cmd_out, void *stream_v)
{
    if (!h || batch < 0 || !u0 || !vel_inout || !cmd_out) return MPC_B200_ERR_INVALID;
    if (!is_device_ptr(u0) || !is_device_ptr(vel_inout) || !is_device_ptr(cmd_out) || (ref_vel && !is_device_ptr(ref_vel)))
        return MPC_B200_ERR_UNSUPPORTED;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    poststep_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, u0, vel_inout, ref_vel, h->params.ref_vel, h->params.dt, cmd_out);
    return finish_device_call(h, st, stream_v);
}

int mpc_b200_decel_batch(mpc_b200_handle *h, int32_t batch, const double *pose, const double *goal, const double *vel,
                         double min_speed, double *ref_vel_inout, void *stream_v)
{
    if (!h || batch < 0 || !pose || !goal || !vel || !ref_vel_inout) return MPC_B200_ERR_INVALID;
    if (!is_device_ptr(pose) || !is_device_ptr(goal) || !is_device_ptr(vel) || !is_device_ptr(ref_vel_inout))
        return MPC_B200_ERR_UNSUPPORTED;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    const double thr = h->params.max_throttle < 0.1 ? 0.1 : h->params.max_throttle;      // driving_state.cpp:63
    decel_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, pose, goal, vel, thr, h->params.max_speed, min_speed, ref_vel_inout);
    return finish_device_call(h, st, stream_v);
}

int mpc_b200_plant_step_batch(mpc_b200_handle *h, int32_t batch, const double *cmd, double *pose_inout, double *vel_inout,
                              void *stream_v)
{
    if (!h || batch < 0 || !cmd || !pose_inout || !vel_inout) return MPC_B200_ERR_INVALID;
    if (!is_device_ptr(cmd) || !is_device_ptr(pose_inout) || !is_device_ptr(vel_inout)) return MPC_B200_ERR_UNSUPPORTED;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    plant_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, cmd, pose_inout, vel_inout, h->params.dt);
    return finish_device_call(h, st, stream_v);
}

int mpc_b200_num_waypoints(const mpc_b200_params *p)
{
    if (!p) return MPC_B200_ERR_INVALID;
    const double wd = p->waypoints_dist > 0.0 ? p->waypoints_dist : 0.05;
    const int win = (int)lround(p->path_length / wd);
    const int step = (int)(p->path_length / 10.0 / wd);
    if (step < 1) return MPC_B200_ERR_INVALID;
    return (win + step - 1) / step + 1;
}

int mpc_b200_warm_shift(mpc_b200_handle *h, int32_t batch, const double *warm_prev, double *warm_next, void *stream_v)
{
    if (!h || batch < 0 || !warm_prev || !warm_next || warm_prev == warm_next) return MPC_B200_ERR_INVALID;
    if (!is_device_ptr(warm_prev) || !is_device_ptr(warm_next)) return MPC_B200_ERR_UNSUPPORTED;
    if (batch == 0) return MPC_B200_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = stream_v ? (cudaStream_t)stream_v : h->stream;
    warm_shift_kernel<<<(batch + 127) / 128, 128, 0, st>>>(batch, h->params.mpc_steps, warm_prev, warm_next);
    return finish_device_call(h, st, stream_v);
}

double mpc_b200_measure_fp64_peak(int32_t device, int32_t iters)
{
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return -1.0; }
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int blocks = sms * 8, threads = 256;
    double *out = NULL;
    if (cudaMalloc(&out, sizeof(double) * blocks * threads) != cudaSuccess) { cudaGetLastError(); return -1.0; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    dfma_kernel<8><<<blocks, threads>>>(out, 64, 32, NULL);   // warm-up
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0);
        dfma_kernel<8><<<blocks, threads>>>(out, iters, 32, NULL);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
        const double tf = flops / (1e-3 * ms) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    if (cudaGetLastError() != cudaSuccess) return -1.0;
    return best;
}

// NMPC_PROFILE builds: per-phase SM-cycle counters of CTA 0's control thread for the last solve
// (0 residual phase, 1 check, 2 coeff phase, 3 backward sweep, 4 forward sweep, 5 step phase,
//  6 ctrl_step + adjoint, 7 trial phase, 8 line-search decision, 9 accept phase).  Returns 0 if
// the library was built without NMPC_PROFILE.
int mpc_b200_debug_profile(mpc_b200_handle *h, long long *out12)
{
#ifdef NMPC_PROFILE
    if (!h) return 0;
    if (!h->d_prof) {
        if (cudaMalloc(&h->d_prof, sizeof(long long) * 1024) != cudaSuccess) { cudaGetLastError(); return 0; }
        cudaMemset(h->d_prof, 0, sizeof(long long) * 1024);
        return 1;
    }
    if (out12) {
        cudaMemcpy(out12, h->d_prof, sizeof(long long) * 1024, cudaMemcpyDeviceToHost);
        cudaMemcpyFromSymbol(out12 + 1020, nmpc::nmpc_dec_acc, sizeof(long long) * 4);      // ctrl_decide sub-phases
    }
    return 1;
#else
    (void)h; (void)out12;
    return 0;
#endif
}

// Single-warp DFMA probe: returns SM cycles per warp-level DFMA instruction for `ilp`
// independent chains (1, 2, 4 or 8) with `active_lanes` lanes enabled.
double mpc_b200_debug_fp64_probe(int32_t device, int32_t ilp, int32_t active_lanes, int32_t iters)
{
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return -1.0; }
    double *out = NULL; long long *cyc = NULL;
    cudaMalloc(&out, sizeof(double) * 32); cudaMalloc(&cyc, sizeof(long long));
    for (int rep = 0; rep < 2; rep++) {
        if (ilp == 1) dfma_kernel<1><<<1, 32>>>(out, iters, active_lanes, cyc);
        else if (ilp == 2) dfma_kernel<2><<<1, 32>>>(out, iters, active_lanes, cyc);
        else if (ilp == 4) dfma_kernel<4><<<1, 32>>>(out, iters, active_lanes, cyc);
        else dfma_kernel<8><<<1, 32>>>(out, iters, active_lanes, cyc);
    }
    long long c = 0;
    cudaMemcpy(&c, cyc, sizeof(c), cudaMemcpyDeviceToHost);
    cudaFree(out); cudaFree(cyc);
    if (cudaGetLastError() != cudaSuccess) return -1.0;
    const int chains = (ilp == 1 || ilp == 2 || ilp == 4) ? ilp : 8;
    return (double)c / ((double)iters * chains);
}

}  // extern "C"
