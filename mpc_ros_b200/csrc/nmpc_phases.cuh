// nmpc_phases.cuh -- the per-(problem, stage) and per-problem phases of the batched
// structure-exploiting interior-point NMPC solver.
//
// What it replaces in the reference (OkDoky/mpc_ros):
//   * FG_eval's CppAD-taped cost / dynamics and taped Jacobian / Hessian
//     (mpc_ros/src/mpc_planner.cpp:102-217, cppad/ipopt/solve_callback.hpp:625-1020)
//     -> closed-form stage derivatives (stage_eval / stage_apply_coeffs below);
//   * Ipopt's primal-dual interior-point loop (call site cppad/ipopt/solve.hpp:586)
//     -> the same published algorithm (Waechter & Biegler 2006, Ipopt 3.12 defaults: monotone
//     barrier, filter line search, inertia-correcting regularisation) with the stage-wise
//     block-tridiagonal KKT system solved by a sparsity-exploiting Riccati recursion.
//
// Execution model (see nmpc_kernel.cuh): a CTA has PB problem lanes.  "Stage threads" own a few
// (lane, stage) pairs each in the stage-parallel phases; one "control thread" per lane (16 lanes per
// control warp) runs the per-problem logic and the serial Riccati sweeps.  All cross-thread data
// goes through the CTA's shared memory, indexed [stage][slot][lane] so that a warp touches 32
// consecutive doubles.  Every lane is a small state machine (enum Mode); one global cycle runs the six
// phases P1..P6 once and each lane does the work its state asks for, so a lane that needs an extra
// factorisation (inertia correction) or a shorter trial step repeats on the next cycle without stalling
// the other lanes.  Phases are separated by CTA barriers, which is also what lets tests/emu run the
// identical phase functions sequentially on the host as a logic check (test-only; the product has no
// CPU path).
#pragma once

#include <math.h>
#include <string.h>

#if defined(__CUDACC__)
#define MPC_HD __host__ __device__ __forceinline__
#define MPC_HD_RARE __host__ __device__ __noinline__     /* rare paths: kept out of the hot phases' register allocation */
#else
#define MPC_HD inline
#define MPC_HD_RARE inline
#endif

namespace nmpc {

// ---------------------------------------------------------------- shared-memory layout
enum Slot {
    S_X = 0, S_Y, S_T, S_V, S_C, S_E,          // state s_k = [x y theta v cte etheta]
    L_X, L_Y, L_T, L_V, L_C, L_E,              // lambda_{k+1}: multiplier of  s_{k+1} - phi(s_k,u_k) = 0
    A_13, A_14, A_23, A_24, A_51, A_54, A_56,  // non-trivial entries of A_k = d phi / d s
    D_X, D_Y, D_T, D_V, D_C, D_E,              // d_k = -(s_{k+1} - phi_k); after the forward sweep: ds_{k+1}
    W_0, W_1, W_2, W_3, W_4, W_5, W_6, W_7, W_8, W_9, W_10, W_11,  // work slots (see phases)
    NSLOTS,
    // only in the rate-penalty variant (w_angvel_d / w_accel_d != 0 couple u_k and u_{k+1}):
    U_W = NSLOTS, U_A,          // controls of the stage, published for the neighbouring stages
    DU_W, DU_A,                 // their Newton step
    RI_11, RI_12, RI_22,        // inverse of the Riccati pivot R~_k (forward sweep: gain on the previous control step)
    NSLOTS_RATE
};
// partial sums, one set per group of stages: [group][NPART][lane]
enum PartSlot { PT_0 = 0, PT_1, PT_2, PT_3, PT_4, PT_5, PT_6, PT_7, PT_8, NPART };

// per-lane scalars shared between the control thread and the stage threads
enum PSlot {
    PS_MU = 0,     // barrier parameter of the Newton system being built / solved
    PS_MU_STEP,    // barrier parameter the pending step was computed with (for the z update, W&B eq. (16))
    PS_TAU, PS_SF, PS_REFV, PS_ALPHA, PS_ALPHA_Z, PS_DW,
    PS_L0X, PS_L0Y, PS_L0T, PS_L0V, PS_L0C, PS_L0E,       // lambda_0 (initial-condition rows)
    PS_N0X, PS_N0Y, PS_N0T, PS_N0V, PS_N0C, PS_N0E,       // its Newton target lambda_0^+
    PS_AP_ALPHA, PS_AP_AZ, PS_AP_MU, PS_AP_SF,            // the step to apply in P3 (copied in P2: the lane may
                                                          // already have been re-initialised for its next problem)
    PS_NX0, PS_NX1, PS_NX2, PS_NX3, PS_NX4, PS_NX5,       // staged inputs of the lane's next problem: state (6),
    PS_NX6, PS_NX7, PS_NX8, PS_NX9, PS_NX10,              // coeffs (4), ref_vel -- written at refill, read in P3a
    PS_NXC4, PS_NXC5, PS_NXC6, PS_NXC7,                   // coefficients 4..7 of a path polynomial of order > 3
    PS_ALPHA_LS,   // second-order correction: length of the rejected first trial step (Armijo / switching tests, resume)
    PS_SOC_THETA,  // second-order correction: constraint violation of the previous attempt (kappa_soc test)
    NPS
};
enum PISlot {
    PI_MODE = 0,   // lane state (enum Mode)
    PI_FLAGS,      // enum Flag bits
    PI_PROB,       // index of the problem in this lane
    PI_NEXT,       // refill: index of the problem the lane takes over in P3, or -1
    PI_SOC,        // line search of the pending step: 0 = first trial not yet judged, k >= 1 = k-th second-order
                   // correction in progress, -1 = plain backtracking (no correction any more)
    NPI
};

// Lane state, written by the control thread, read by the stage threads.
enum Mode {
    MODE_IDLE = 0,   // no problem in this lane
    MODE_EVAL,       // P1: evaluate the point iterate + alpha * step (alpha may be 0); P2: decide
    MODE_NEWTON,     // P3: (apply the accepted step and) write the Newton-system coefficients; P4: sweeps
    MODE_STEP,       // P5: step-dependent stage work; P6: multipliers + step-size limits
    MODE_FAIL,       // the Newton system could not be regularised: flushed at the next P2
    MODE_ROLLOUT     // warm start: P4 rolls the model out from the given state with the warm controls
};
enum Flag {
    FL_LSQ = 1,      // the system being solved is the least-squares multiplier start (W&B eq. (36))
    FL_APPLY = 2,    // P3 must first apply the step accepted in P2
    FL_ADOPT = 4,    // P1 must first adopt the least-squares multipliers (or zero them)
    FL_LS = 8,       // the point evaluated in P1 is a line-search trial (else it is accepted as is)
    FL_FLUSH = 16,   // P3 must write this lane's finished problem out
    FL_KEEP = 32,    // with FL_ADOPT: keep the least-squares multipliers (else reset to zero)
    FL_WARM = 64,    // P3a initialises the lane from a warm-start record instead of the cold start
    FL_SOC = 128,    // the Newton system / the trial point is a second-order correction (W&B A-5.5 .. A-5.9): same matrix,
                     // constraint right-hand side c_soc kept in the stage threads' trial sin/cos registers
    FL_RESUME = 256, // the Newton step is recomputed after a failed correction: the line search resumes at alpha / 2
    FL_RESTO = 512   // feasibility restoration (stand-in for Ipopt's restoration phase, as in the oracle: min-norm Gauss-Newton
                     // steps on the constraint violation): the system is  [I J'; J 0] (dx, .) = (0, -c),  only the primal moves
};
// What the Newton machinery is asked to solve: 0 = the primal-dual Newton step, 1 = the least-squares multiplier start
// (identity Hessian, right-hand side (grad, 0)), 2 = a restoration step (identity Hessian, right-hand side (0, -c)).
MPC_HD int sys_kind(int flags) { return (flags & FL_LSQ) ? 1 : ((flags & FL_RESTO) ? 2 : 0); }

struct Params {
    int N;
    double dt, ref_cte, ref_etheta, ref_vel;
    double w_cte, w_etheta, w_vel, w_angvel, w_accel;
    double max_angvel, max_throttle;
    double tol;
    int max_iter;
    int grp;      // stages per stage thread: partial sums are pre-reduced over groups of grp stages
    double warm_mu;   // initial barrier parameter of a warm-started problem
    double w_angvel_d, w_accel_d;   // rate penalties (mpc_planner.cpp:144-147); both 0 in the plain variant
    double idt;       // 1 / dt
    double i_mnb, i_nb;   // 1 / (6N + 4(N-1)), 1 / (4(N-1)): reciprocal counts of all / of the bound multipliers
    double bound_chk;     // a returned point with some |state| >= this would feel the +-bound_value state bounds
                          // (mpc_planner.cpp:303-312), which this kernel leaves out: flagged NMPC_STATUS_BOUND_ACTIVE
                          // when the finished problem is written out (stage_bound_hit)
};

// A batch to solve: inputs, outputs (SoA over the batch) and the work queue.
struct SolveArgs {
    Params prm;
    int PB;
    int batch;
    int ncoef;              // rows of coeffs: 4 (cubic) .. NMPC_MAX_COEFFS
    const double *state;    // 6 x batch
    const double *coeffs;   // ncoef x batch
    const double *ref_vel;  // batch or NULL
    double *u0;             // 2 x batch
    double *pred;           // 3N x batch
    double *obj;            // batch or NULL
    int *status;            // batch or NULL
    int *iters;             // batch or NULL
    double *kkt;            // batch or NULL
    double *warm_out;       // warm_size x batch or NULL
    const double *warm_in;  // warm_size x batch or NULL (cold start)
    int *queue;             // work-queue head (zeroed by the host before the launch)
    const int *order;       // queue position -> problem index (hard-first order) or NULL (identity)
    long long *prof;        // NMPC_PROFILE builds only: per-phase cycle counters of CTA 0
};

#define NMPC_MAX_FILTER 8
// per-problem status outside the solve_result::status_type values: see Params::bound_chk (= MPC_B200_STATUS_BOUND_ACTIVE)
#define NMPC_STATUS_BOUND_ACTIVE 64

// View of the CTA's shared-memory block.  CPB > 0 fixes the lanes-per-CTA at compile time so that
// every access is base + lane*8 + immediate (no index arithmetic in the sweeps).
template <int CPB, int NS = NSLOTS>
struct SmemT {
    double *st;   // [N][NS][PB]
    double *pt;   // [NG][NPART][PB]
    double *ps;   // [NPS][PB]
    double *fl;   // [2*NMPC_MAX_FILTER][PB]  filter entries (theta, phi)
    int *pi;      // [NPI][PB]
    int PB;
    MPC_HD int pb() const { return CPB > 0 ? CPB : PB; }
    MPC_HD double &at(int k, int slot, int p) const { return st[(k * NS + slot) * pb() + p]; }
    MPC_HD double &part(int g, int slot, int p) const { return pt[(g * NPART + slot) * pb() + p]; }
    MPC_HD double &P(int slot, int p) const { return ps[slot * pb() + p]; }
    MPC_HD double &F(int slot, int p) const { return fl[slot * pb() + p]; }
    MPC_HD int &I(int slot, int p) const { return pi[slot * pb() + p]; }
    MPC_HD void carve(double *base, int N, int NG)
    {
        st = base;
        pt = st + (size_t)N * NS * pb();
        ps = pt + (size_t)NG * NPART * pb();
        fl = ps + (size_t)NPS * pb();
        pi = reinterpret_cast<int *>(fl + (size_t)2 * NMPC_MAX_FILTER * pb());
    }
};
typedef SmemT<0> Smem;

MPC_HD size_t smem_bytes(int N, int NG, int PB, int nslots = NSLOTS)
{
    return sizeof(double) * ((size_t)N * nslots + (size_t)NG * NPART + NPS + 2 * NMPC_MAX_FILTER) * PB +
           sizeof(int) * (size_t)NPI * PB;
}

// Ipopt 3.12 default constants (Waechter & Biegler 2006)
#define NMPC_KAPPA_EPS 10.0
#define NMPC_KAPPA_MU 0.2
#define NMPC_TAU_MIN 0.99
#define NMPC_S_MAX 100.0
#define NMPC_GAMMA_THETA 1e-5
#define NMPC_GAMMA_PHI 1e-8
#define NMPC_S_THETA 1.1
#define NMPC_S_PHI 2.3
#define NMPC_ETA_PHI 1e-8
#define NMPC_GAMMA_ALPHA 0.05
#define NMPC_KAPPA_SIGMA 1e10
#define NMPC_MU_INIT 0.1
#define NMPC_BOUND_RELAX 1e-8
#define NMPC_DW_MIN 1e-20
#define NMPC_DW_0 1e-4
#define NMPC_DW_MAX 1e40
#define NMPC_KW_MINUS (1.0 / 3.0)
#define NMPC_KW_PLUS 8.0
#define NMPC_KW_PLUS_BAR 100.0
#define NMPC_EPS_MACH 2.220446049250313e-16
#define NMPC_MAX_SOC 4
#define NMPC_KAPPA_SOC 0.99

// Roles of the work slots between the sweeps and the next coefficient phase:
//   W_LAM..+5  g_k (P5), then lambda_{k+1}^+ (adjoint sweep, in place);
//   W_ISL..+3  reciprocal slacks of the control bounds at the iterate (P5), read by P1 / P3a;
//   W_DU, +1   Newton step of the controls (forward sweep), read by P5 / P1 / P3a.
enum { W_LAM = W_0, W_ISL = W_6, W_DU = W_10 };

// ---------------------------------------------------------------- per-(lane, stage) registers
struct StageRegs {
    double uw, ua;              // controls of this stage (k <= N-2)
    double zlw, zuw, zla, zua;  // bound multipliers of the controls (scaled problem)
    double sn, cs, se, ce;      // sin/cos(theta_k), sin/cos(etheta_k) at the iterate
    double tsn, tcs, tse, tce;  // the same at the last evaluated point
};

MPC_HD double fmax2(double a, double b) { return a > b ? a : b; }
MPC_HD double fmin2(double a, double b) { return a < b ? a : b; }

// sin and cos together, branch-free (so that the evaluations of a thread's stages interleave):
// Cody-Waite reduction by pi/2 in three parts, then the classical minimax kernels on [-pi/4, pi/4].
// Accurate to about 1 ulp for |a| < 1e5 (heading angles here are a few radians); beyond that the
// reduction loses bits gradually, NaN / Inf propagate as NaN.
MPC_HD void sincos_d(double a, double *s, double *c)
{
    const double TWO_OVER_PI = 6.36619772367581382433e-01;
    const double PIO2_1 = 1.57079632673412561417e+00;   // first 33 bits of pi/2
    const double PIO2_2 = 6.07710050630396597660e-11;   // next 33 bits
    const double PIO2_3 = 2.02226624871116645580e-21;   // next 33 bits
    const double PIO2_3T = 8.47842766036889956997e-32;  // tail
    const double MAGIC = 6755399441055744.0;            // 1.5 * 2^52: round to nearest integer
    const double qd = (a * TWO_OVER_PI + MAGIC) - MAGIC;
    double r = fma(-qd, PIO2_1, a);
    r = fma(-qd, PIO2_2, r);
    r = fma(-qd, PIO2_3, r);
    r = fma(-qd, PIO2_3T, r);
    const int q = (int)qd;
    const double z = r * r;
    // sin kernel
    const double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03, S3 = -1.98412698298579493134e-04,
                 S4 = 2.75573137070700676789e-06, S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
    const double ps = S1 + z * (S2 + z * (S3 + z * (S4 + z * (S5 + z * S6))));
    const double sr = fma(r * z, ps, r);
    // cos kernel
    const double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03, C3 = 2.48015872894767294178e-05,
                 C4 = -2.75573143513906633035e-07, C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
    const double pc = z * (C1 + z * (C2 + z * (C3 + z * (C4 + z * (C5 + z * C6)))));
    const double cr = fma(z, pc, fma(-0.5, z, 1.0));
    // quadrant
    const bool swap = (q & 1) != 0;
    double ss = swap ? cr : sr, cc = swap ? sr : cr;
    if (q & 2) ss = -ss;
    if ((q + 1) & 2) cc = -cc;
    *s = ss; *c = cc;
}

// natural logarithm of a positive normal number, branch-free (the caller has checked x > 0).
MPC_HD double log_pos(double x)
{
#if defined(__CUDA_ARCH__)
    long long ix = __double_as_longlong(x);
#else
    long long ix; { double t_ = x; memcpy(&ix, &t_, sizeof(ix)); }
#endif
    // split x = 2^k * m with m in [sqrt(1/2), sqrt(2))
    int hx = (int)(ix >> 32);
    hx += 0x3ff00000 - 0x3fe6a09e;
    const int k = (hx >> 20) - 0x3ff;
    hx = (hx & 0x000fffff) + 0x3fe6a09e;
    const long long im = ((long long)hx << 32) | (ix & 0xffffffffLL);
#if defined(__CUDA_ARCH__)
    const double m = __longlong_as_double(im);
#else
    double m; memcpy(&m, &im, sizeof(m));
#endif
    const double f = m - 1.0;
    const double hfsq = 0.5 * f * f;
    const double sden = 2.0 + f;
#if defined(__CUDA_ARCH__)
    double inv; asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(inv) : "d"(sden));
    double e_ = fma(-sden, inv, 1.0); inv = fma(inv, e_, inv);
    e_ = fma(-sden, inv, 1.0); inv = fma(inv, e_, inv);
#else
    const double inv = 1.0 / sden;
#endif
    const double s_ = f * inv;
    const double z = s_ * s_, w = z * z;
    const double Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                 Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                 Lg7 = 1.479819860511658591e-01;
    const double t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    const double t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    const double R = t2 + t1;
    const double dk = (double)k;
    const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10;
    return dk * ln2_hi - ((hfsq - (s_ * (hfsq + R) + dk * ln2_lo)) - f);
}

// Reciprocal for the 2x2 Riccati pivot: hardware seed + Newton steps (no special-case branch; the
// caller has already checked the argument is a positive finite number).
MPC_HD double fast_rcp(double x)
{
#if defined(__CUDA_ARCH__)
    double y;
    // (the seed is good to ~2^-20: two Newton steps reach 2^-80, i.e. the last bit; a third one was measured to change nothing)
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0); y = fma(y, e, y);
    e = fma(-x, y, 1.0); y = fma(y, e, y);
    return y;
#else
    return 1.0 / x;
#endif
}

// relaxed control bounds (Ipopt bound_relax_factor, W&B Sec. 3.5)
MPC_HD double relaxed(double b) { return b + NMPC_BOUND_RELAX * fmax2(1.0, b); }
// keep a bound multiplier within kappa_Sigma of mu / slack (W&B eq. (16))
MPC_HD double zclamp(double z, double mu, double islack)
{
    const double c = mu * islack;
    return fmax2(fmin2(z, NMPC_KAPPA_SIGMA * c), (1.0 / NMPC_KAPPA_SIGMA) * c);
}

// Partial sums of one group of stages at an evaluated point.
struct EvalPart { double prinf, pr1, duinf, vmax, vmin, l1, z1, f, lnsum; int inside; };
struct StepPart { double rmax, rzmax, gd; };
MPC_HD void part_reset(EvalPart &a) { a.prinf = 0; a.pr1 = 0; a.duinf = 0; a.vmax = -1e300; a.vmin = 1e300; a.l1 = 0; a.z1 = 0; a.f = 0; a.lnsum = 0; a.inside = 1; }
MPC_HD void part_reset(StepPart &a) { a.rmax = 0.0; a.rzmax = 0.0; a.gd = 0.0; }
template <class SM> MPC_HD void part_store(const SM &sm, int g, int p, const EvalPart &a)
{
    sm.part(g, PT_0, p) = a.prinf; sm.part(g, PT_1, p) = a.pr1; sm.part(g, PT_2, p) = a.duinf;
    sm.part(g, PT_3, p) = a.vmax; sm.part(g, PT_4, p) = a.vmin; sm.part(g, PT_5, p) = a.l1;
    sm.part(g, PT_6, p) = a.z1; sm.part(g, PT_7, p) = a.f; sm.part(g, PT_8, p) = a.inside ? a.lnsum : -1e300;
}
template <class SM> MPC_HD void part_store(const SM &sm, int g, int p, const StepPart &a)
{
    sm.part(g, PT_0, p) = a.rmax; sm.part(g, PT_1, p) = a.rzmax; sm.part(g, PT_2, p) = a.gd;
}

// The reference bounds every state by +-bound_value (mpc_planner.cpp:303-312); this solver carries no barrier for those
// bounds.  A point strictly inside them is a KKT point of the bounded problem as well (zero multipliers); one that is not
// would have been shaped by them.  Checked per stage when a finished problem is written out: a success / acceptable
// status is then replaced by NMPC_STATUS_BOUND_ACTIVE -- reported, never passed off as a solution.
template <class SM>
MPC_HD bool stage_bound_hit(const Params &prm, const SM &sm, int k, int p)
{
    const double m = fmax2(fmax2(fmax2(fabs(sm.at(k, S_X, p)), fabs(sm.at(k, S_Y, p))), fmax2(fabs(sm.at(k, S_T, p)), fabs(sm.at(k, S_V, p)))),
                           fmax2(fabs(sm.at(k, S_C, p)), fabs(sm.at(k, S_E, p))));
    return !(m < prm.bound_chk);
}

// ---------------------------------------------------------------- init (new problem in a lane)
// Reference cold start (mpc_planner.cpp:288-300): zeros except stage 0 = state; z = 1; lambda = 0.
template <bool RATE = false, class SM>
MPC_HD void stage_init(const Params &prm, const SM &sm, StageRegs &r, int k, int p,
                       const double *state6, const double *coef4)
{
    if (RATE) { sm.at(k, U_W, p) = 0.0; sm.at(k, U_A, p) = 0.0; sm.at(k, DU_W, p) = 0.0; sm.at(k, DU_A, p) = 0.0; }
    for (int c = 0; c < 6; c++) sm.at(k, S_X + c, p) = (k == 0) ? state6[c] : 0.0;
    for (int c = 0; c < 6; c++) sm.at(k, L_X + c, p) = 0.0;
    // the step slots are read (times a zero step length) by plain evaluations before any sweep wrote them
    for (int c = 0; c < 6; c++) { sm.at(k, D_X + c, p) = 0.0; sm.at(k, W_0 + c, p) = 0.0; sm.at(k, W_6 + c, p) = 0.0; }
    r.uw = 0.0; r.ua = 0.0;
    r.zlw = r.zuw = r.zla = r.zua = 1.0;      // bound_mult_init_val
    (void)coef4;
    if (k == 0) {
        sincos_d(state6[2], &r.sn, &r.cs);
        sincos_d(state6[5], &r.se, &r.ce);
    } else {
        r.sn = 0.0; r.cs = 1.0; r.se = 0.0; r.ce = 1.0;
    }
    r.tsn = r.sn; r.tcs = r.cs; r.tse = r.se; r.tce = r.ce;
}

// Warm start (new capability; the reference cold-starts every call, solve_callback.hpp:595-597).
// Record layout (mpc_b200_warm_size doubles per problem, SoA over the batch): primal in the reference's
// variable layout (mpc_planner.cpp:232-239), equality multipliers in its row layout (:153-158), then
// zL_w, zL_a, zU_w, zU_a.  Controls and multipliers are taken from the record (controls pushed into the
// interior of their bounds); the states are NOT taken from it: the control thread rolls the model out
// from the given state (ctrl_rollout), so the start point satisfies the dynamics exactly.
// Rows of the blocks: state c of stage k at c*N + k; controls of stage k < N-1 at warm_uw + k, warm_ua + k; lambda_k,
// component c, at warm_lam + c*N + k (lambda_0: the initial-condition rows); zL_w, zL_a, zU_w, zU_a of stage k < N-1 at
// warm_z + j*(N-1) + k, j = 0..3.
MPC_HD size_t warm_uw(int N) { return (size_t)6 * N; }
MPC_HD size_t warm_ua(int N) { return (size_t)7 * N - 1; }
MPC_HD size_t warm_lam(int N) { return (size_t)(8 * N - 2); }
MPC_HD size_t warm_z(int N) { return warm_lam(N) + (size_t)6 * N; }
MPC_HD size_t warm_size(int N) { return warm_z(N) + (size_t)4 * (N - 1); }

template <bool RATE = false, class SM>
MPC_HD void stage_init_warm(const Params &prm, const SM &sm, StageRegs &r, int k, int p,
                            const double *state6, const double *coef4, const double *warm, size_t stride, size_t idx)
{
    const int N = prm.N;
    stage_init<RATE>(prm, sm, r, k, p, state6, coef4);
    if (k < N - 1) {
        const double sf = sm.P(PS_SF, p), mu = prm.warm_mu;
        const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
        double uw = warm[(warm_uw(N) + k) * stride + idx], ua = warm[(warm_ua(N) + k) * stride + idx];
        const double pw = 1e-3 * Uw, pa = 1e-3 * Ua;       // warm_start_bound_push
        uw = fmax2(fmin2(uw, Uw - pw), -Uw + pw); ua = fmax2(fmin2(ua, Ua - pa), -Ua + pa);
        r.uw = uw; r.ua = ua;
        sm.at(k, W_10, p) = uw; sm.at(k, W_11, p) = ua;    // for the roll-out
        if (RATE) { sm.at(k, U_W, p) = uw; sm.at(k, U_A, p) = ua; }
        const size_t offl = warm_lam(N), offz = warm_z(N);
        // A non-finite equality multiplier must not end in a "success": the max of the dual residuals drops a NaN, and only
        // the x, y and cte components of lambda_{k+1} at a free stage (k >= 1) enter a Newton system, through the Hessian.
        // bad is +0 when the entries it sums are finite, else NaN (0 * |l|, one term per entry, so that finite entries
        // cannot overflow).  A non-finite component of lambda_{k+1} is spread over all six, and stage 1 also takes in
        // lambda_0 and lambda_1, which enter no Newton system: the first Newton step then fails with status 10, as the
        // oracle's does.  At N = 2 no multiplier enters a Newton system; there stage 0 takes in lambda_0 and lambda_1 and
        // makes z_L,w NaN, which ends the problem with status 11 at its first evaluation.  Finite records are read
        // unchanged: l - (+0) is l bit for bit, -0 included, and z_L,w > 0.
        double bad = 0.0;
        for (int c = 0; c < 6; c++) bad += 0.0 * fabs(warm[(offl + (size_t)c * N + k + 1) * stride + idx]);
        if (k == 1 || N == 2)
            for (int c = 0; c < 6; c++) bad += 0.0 * fabs(warm[(offl + (size_t)c * N) * stride + idx]) + 0.0 * fabs(warm[(offl + (size_t)c * N + 1) * stride + idx]);
        for (int c = 0; c < 6; c++) sm.at(k, L_X + c, p) = sf * warm[(offl + (size_t)c * N + k + 1) * stride + idx] - bad;
        const int nu = N - 1;
        // multipliers of the control bounds: at least on the central path of the starting mu
        r.zlw = fmax2(sf * warm[(offz + k) * stride + idx], mu / (uw + Uw));
        if (N == 2) r.zlw += bad;
        r.zla = fmax2(sf * warm[(offz + nu + k) * stride + idx], mu / (ua + Ua));
        r.zuw = fmax2(sf * warm[(offz + 2 * nu + k) * stride + idx], mu / (Uw - uw));
        r.zua = fmax2(sf * warm[(offz + 3 * nu + k) * stride + idx], mu / (Ua - ua));
    }
}

// Path polynomial p(x) = sum_i cf[i] x^i (mpc_planner.cpp:186-190; the order is coeffs.size() - 1 there) with its
// first two derivatives, by Horner's rule.  NC = 4 is the cubic the reference's only caller fits
// (driving_state.cpp:210); the forms below then reduce to the closed cubic expressions.
#define NMPC_MAX_COEFFS 8
template <int NC>
MPC_HD void path_poly(const double *cf, double x, double &p0, double &p1, double &p2)
{
    double a = cf[NC - 1], b = (double)(NC - 1) * cf[NC - 1], c = (double)((NC - 1) * (NC - 2)) * cf[NC - 1];
#pragma unroll
    for (int i = NC - 2; i >= 0; i--) a = cf[i] + x * a;
#pragma unroll
    for (int i = NC - 2; i >= 1; i--) b = (double)i * cf[i] + x * b;
#pragma unroll
    for (int i = NC - 2; i >= 2; i--) c = (double)(i * (i - 1)) * cf[i] + x * c;
    p0 = a; p1 = b; p2 = c;
}

// Roll-out of the model from s_0 with the controls left in W_10/W_11 (control thread).
template <int NC = 4, class SM>
MPC_HD void ctrl_rollout(const Params &prm, const SM &sm, int p, const double *coef4)
{
    const int N = prm.N;
    const double dt = prm.dt;
    double x = sm.at(0, S_X, p), y = sm.at(0, S_Y, p), th = sm.at(0, S_T, p), v = sm.at(0, S_V, p), e = sm.at(0, S_E, p);
    for (int k = 0; k < N - 1; k++) {
        const double uw = sm.at(k, W_10, p), ua = sm.at(k, W_11, p);
        double sn, cs, se, ce;
        sincos_d(th, &sn, &cs);
        sincos_d(e, &se, &ce);
        double poly, d1_unused, d2_unused;
        path_poly<NC>(coef4, x, poly, d1_unused, d2_unused);
        (void)d1_unused; (void)d2_unused;
        const double nc = (poly - y) + v * se * dt;
        const double nx = x + v * cs * dt, ny = y + v * sn * dt;
        th += uw * dt; e += uw * dt; v += ua * dt; x = nx; y = ny;
        sm.at(k + 1, S_X, p) = x; sm.at(k + 1, S_Y, p) = y; sm.at(k + 1, S_T, p) = th;
        sm.at(k + 1, S_V, p) = v; sm.at(k + 1, S_C, p) = nc; sm.at(k + 1, S_E, p) = e;
        sm.at(k, W_10, p) = 0.0; sm.at(k, W_11, p) = 0.0;
    }
}

// trial bound multipliers  z + alpha_z dz (dz from W&B eq. (12)), kept within kappa_Sigma of mu / slack
// (W&B eq. (16)).  The safeguard almost never binds, so it is tested on the complementarity product
// z * slack (needed anyway) and the division only happens on the rare path.
MPC_HD double zsafe(double z, double mu, double slack)
{
    const double prod = z * slack;
    if (prod > NMPC_KAPPA_SIGMA * mu || prod < (1.0 / NMPC_KAPPA_SIGMA) * mu) z = zclamp(z, mu, 1.0 / slack);
    return z;
}
template <class SM>
MPC_HD void trial_z(const Params &prm, const SM &sm, const StageRegs &r, int k, int p, double az, double mu, double uw, double ua,
                    double &zlw, double &zuw, double &zla, double &zua)
{
    const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
    const double duw = sm.at(k, W_DU, p), dua = sm.at(k, W_DU + 1, p);
    const double ilw = sm.at(k, W_ISL, p), iuw = sm.at(k, W_ISL + 1, p), ila = sm.at(k, W_ISL + 2, p), iua = sm.at(k, W_ISL + 3, p);
    // az == 0 (plain evaluation) leaves the multipliers bit-for-bit unchanged and skips the safeguard
    zlw = r.zlw + az * (mu * ilw - r.zlw - r.zlw * ilw * duw);
    zuw = r.zuw + az * (mu * iuw - r.zuw + r.zuw * iuw * duw);
    zla = r.zla + az * (mu * ila - r.zla - r.zla * ila * dua);
    zua = r.zua + az * (mu * iua - r.zua + r.zua * iua * dua);
    const double slw = uw + Uw, suw = Uw - uw, sla = ua + Ua, sua = Ua - ua;
    const double hi = NMPC_KAPPA_SIGMA * mu, lo = (1.0 / NMPC_KAPPA_SIGMA) * mu;
    const double p1 = zlw * slw, p2 = zuw * suw, p3 = zla * sla, p4 = zua * sua;
    const bool out = (fmax2(fmax2(p1, p2), fmax2(p3, p4)) > hi) || (fmin2(fmin2(p1, p2), fmin2(p3, p4)) < lo);
    if (az != 0.0 && out) {
        zlw = zsafe(zlw, mu, slw); zuw = zsafe(zuw, mu, suw);
        zla = zsafe(zla, mu, sla); zua = zsafe(zua, mu, sua);
    }
}

// P1, before the evaluation, lanes with FL_ADOPT: adopt the least-squares multipliers left in W_6..W_11 by
// the adjoint sweep (or zero them).  Kept apart from stage_eval so that the evaluations of a thread's
// stages contain no shared-memory stores and can be interleaved by the compiler.
template <class SM>
MPC_HD void stage_adopt(const Params &prm, const SM &sm, int k, int p, int flags)
{
    const bool keep = (flags & FL_KEEP) != 0;
    if (k < prm.N - 1)
        for (int c = 0; c < 6; c++) sm.at(k, L_X + c, p) = keep ? sm.at(k, W_LAM + c, p) : 0.0;
}

// Rate penalty  sum_j w_d (u_{j+1} - u_j)^2  (mpc_planner.cpp:144-147): gradient wrt u_k given its neighbours.
// The pair (u_{k-1}, u_k) exists for 1 <= k <= N-2, the pair (u_k, u_{k+1}) for k <= N-3.
MPC_HD double rate_grad(double wd2, double u, double up, double un, bool has_prev, bool has_next)
{
    double g = 0.0;
    if (has_prev) g += wd2 * (u - up);
    if (has_next) g -= wd2 * (un - u);
    return g;
}

// ---------------------------------------------------------------- P1: evaluate  iterate + alpha * step
// Everything the control thread needs to (a) run the filter line search on this point and (b), if it
// becomes the iterate, test convergence and update mu: sum|c|, max|c|, scaled objective, log-barrier
// sum, max|dual residual| and the extreme complementarity products with the trial multipliers
// lambda + alpha (lambda^+ - lambda), z + alpha_z dz, plus the multiplier norms.
template <bool RATE = false, int NC = 4, class SM>
MPC_HD void stage_eval(const Params &prm, const SM &sm, StageRegs &r, int k, int p, int flags, EvalPart &acc,
                       const double *cf)
{
    // Written without lane-dependent branches (one rare one excepted) so that the compiler sees one long
    // basic block per stage: a plain evaluation is a trial point with alpha = 0 (the step slots always hold
    // finite numbers: stage_init zeroes them), and the multipliers to adopt after the least-squares solve
    // are the trial multipliers with base 0 and step length 1.
    const int N = prm.N;
    const double sf = sm.P(PS_SF, p), refv = sm.P(PS_REFV, p), dt = prm.dt;
    const bool ls = (flags & FL_LS) != 0;
    const bool adopt = (flags & FL_ADOPT) != 0;
    const double alpha = ls ? sm.P(PS_ALPHA, p) : 0.0;
    const double az = ls ? sm.P(PS_ALPHA_Z, p) : 0.0;
    const double al = (flags & FL_RESTO) ? 0.0 : alpha;      // step length of the equality multipliers (restoration: primal only)
    const double lcoef = adopt ? (((flags & FL_KEEP) != 0) ? 1.0 : 0.0) : al;   // step length of lambda_k
    const double mu = sm.P(PS_MU_STEP, p);
    const int km = k > 0 ? k - 1 : 0;
    const double dmask = k > 0 ? alpha : 0.0;        // ds_0 = 0
    const double x = sm.at(k, S_X, p) + dmask * sm.at(km, D_X, p), y = sm.at(k, S_Y, p) + dmask * sm.at(km, D_Y, p);
    const double th = sm.at(k, S_T, p) + dmask * sm.at(km, D_T, p), v = sm.at(k, S_V, p) + dmask * sm.at(km, D_V, p);
    const double ct = sm.at(k, S_C, p) + dmask * sm.at(km, D_C, p), e = sm.at(k, S_E, p) + dmask * sm.at(km, D_E, p);
    sincos_d(th, &r.tsn, &r.tcs);
    sincos_d(e, &r.tse, &r.tce);
    // objective part of this stage (mpc_planner.cpp:122-140) and its gradient
    const double ec = ct - prm.ref_cte, ee = e - prm.ref_etheta, ev = v - refv;
    double f = prm.w_cte * ec * ec + prm.w_etheta * ee * ee + prm.w_vel * ev * ev;
    const double qv = 2.0 * sf * prm.w_vel * ev, qc = 2.0 * sf * prm.w_cte * ec, qe = 2.0 * sf * prm.w_etheta * ee;
    // lambda_k (multiplier of the rows that define s_k) lives with stage k-1 (lambda_0: per-lane scalars):
    // current value in L (PS_L0*), the Newton / least-squares value in W_LAM.. (PS_N0*)
    const double *lcur = (k == 0) ? &sm.P(PS_L0X, p) : &sm.at(k - 1, L_X, p);
    const double *lnew = (k == 0) ? &sm.P(PS_N0X, p) : &sm.at(k - 1, W_LAM, p);
    const int ld = sm.pb();
    double lk[6];
#pragma unroll
    for (int c = 0; c < 6; c++) {
        const double b = adopt ? 0.0 : lcur[c * ld];
        lk[c] = b + lcoef * (lnew[c * ld] - b);
    }
    const double lkx = lk[0], lky = lk[1], lkt = lk[2], lkv = lk[3], lkc = lk[4], lke = lk[5];
    double l1 = 0.0;
    if (k == 0) l1 = fabs(lkx) + fabs(lky) + fabs(lkt) + fabs(lkv) + fabs(lkc) + fabs(lke);
    double prinf = 0.0, pr1 = 0.0, duinf, vmax = -1e300, vmin = 1e300, z1 = 0.0, lnsum = 0.0;
    if (k < N - 1) {
        const double uw = r.uw + alpha * sm.at(k, W_DU, p), ua = r.ua + alpha * sm.at(k, W_DU + 1, p);
        f += prm.w_angvel * uw * uw + prm.w_accel * ua * ua;
        double poly, dpoly, ddpoly_unused;
        path_poly<NC>(cf, x, poly, dpoly, ddpoly_unused);
        (void)ddpoly_unused;
        const double nx = sm.at(k + 1, S_X, p) + alpha * sm.at(k, D_X, p), ny = sm.at(k + 1, S_Y, p) + alpha * sm.at(k, D_Y, p);
        const double nt = sm.at(k + 1, S_T, p) + alpha * sm.at(k, D_T, p), nv = sm.at(k + 1, S_V, p) + alpha * sm.at(k, D_V, p);
        const double nc = sm.at(k + 1, S_C, p) + alpha * sm.at(k, D_C, p), ne = sm.at(k + 1, S_E, p) + alpha * sm.at(k, D_E, p);
        // defect of the dynamics interval k -> k+1 (mpc_planner.cpp:208-215)
        const double cx = nx - (x + v * r.tcs * dt);
        const double cy = ny - (y + v * r.tsn * dt);
        const double cth = nt - (th + uw * dt);
        const double cv = nv - (v + ua * dt);
        const double cc = nc - ((poly - y) + v * r.tse * dt);
        const double ce_ = ne - (e + uw * dt);
        prinf = fmax2(fmax2(fmax2(fabs(cx), fabs(cy)), fmax2(fabs(cth), fabs(cv))), fmax2(fabs(cc), fabs(ce_)));
        pr1 = fabs(cx) + fabs(cy) + fabs(cth) + fabs(cv) + fabs(cc) + fabs(ce_);
        // trial lambda_{k+1} (after an adoption stage_adopt has already put it into L)
        double mx = sm.at(k, L_X, p), my = sm.at(k, L_Y, p), mt = sm.at(k, L_T, p);
        double mv = sm.at(k, L_V, p), mc = sm.at(k, L_C, p), me = sm.at(k, L_E, p);
        mx += al * (sm.at(k, W_LAM, p) - mx); my += al * (sm.at(k, W_LAM + 1, p) - my);
        mt += al * (sm.at(k, W_LAM + 2, p) - mt); mv += al * (sm.at(k, W_LAM + 3, p) - mv);
        mc += al * (sm.at(k, W_LAM + 4, p) - mc); me += al * (sm.at(k, W_LAM + 5, p) - me);
        // stationarity wrt s_k:  grad f + lambda_k - A_k^T lambda_{k+1}
        const double a13 = -v * r.tsn * dt, a14 = r.tcs * dt, a23 = v * r.tcs * dt, a24 = r.tsn * dt;
        const double a51 = dpoly, a54 = r.tse * dt, a56 = v * r.tce * dt;
        const double rx = lkx - (mx + a51 * mc);
        const double ry = lky - (my - mc);
        const double rt = lkt - (a13 * mx + a23 * my + mt);
        const double rv = qv + lkv - (a14 * mx + a24 * my + mv + a54 * mc);
        const double rc = qc + lkc;
        const double re = qe + lke - (a56 * mc + me);
        // stationarity wrt u_k:  grad f - B^T lambda_{k+1} - zL + zU
        double zlw, zuw, zla, zua;
        trial_z(prm, sm, r, k, p, az, mu, uw, ua, zlw, zuw, zla, zua);
        double rw = 2.0 * sf * prm.w_angvel * uw - dt * (mt + me) - zlw + zuw;
        double ra = 2.0 * sf * prm.w_accel * ua - dt * mv - zla + zua;
        if (RATE) {
            const bool hp = k >= 1, hn = k <= N - 3;
            double upw = 0, upa = 0, unw = 0, una = 0;
            if (hp) { upw = sm.at(k - 1, U_W, p) + alpha * sm.at(k - 1, DU_W, p); upa = sm.at(k - 1, U_A, p) + alpha * sm.at(k - 1, DU_A, p); }
            if (hn) { unw = sm.at(k + 1, U_W, p) + alpha * sm.at(k + 1, DU_W, p); una = sm.at(k + 1, U_A, p) + alpha * sm.at(k + 1, DU_A, p); }
            rw += rate_grad(2.0 * sf * prm.w_angvel_d, uw, upw, unw, hp, hn);
            ra += rate_grad(2.0 * sf * prm.w_accel_d, ua, upa, una, hp, hn);
            if (hp) f += prm.w_angvel_d * (uw - upw) * (uw - upw) + prm.w_accel_d * (ua - upa) * (ua - upa);
        }
        duinf = fmax2(fmax2(fmax2(fabs(rx), fabs(ry)), fmax2(fabs(rt), fabs(rv))),
                      fmax2(fmax2(fabs(rc), fabs(re)), fmax2(fabs(rw), fabs(ra))));
        l1 += fabs(mx) + fabs(my) + fabs(mt) + fabs(mv) + fabs(mc) + fabs(me);
        z1 = zlw + zuw + zla + zua;
        const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
        const double slw = uw + Uw, suw = Uw - uw, sla = ua + Ua, sua = Ua - ua;
        const double p1 = slw * zlw, p2 = suw * zuw, p3 = sla * zla, p4 = sua * zua;
        vmax = fmax2(fmax2(p1, p2), fmax2(p3, p4));
        vmin = fmin2(fmin2(p1, p2), fmin2(p3, p4));
        const bool in_ = slw > 0.0 && suw > 0.0 && sla > 0.0 && sua > 0.0;
        lnsum = log_pos(in_ ? (slw * suw) * (sla * sua) : 1.0);      // log_pos(1) == 0 exactly
        if (!in_) acc.inside = 0;
    } else {
        // last stage: no dynamics, no control
        const double rv = qv + lkv, rc = qc + lkc, re = qe + lke;
        duinf = fmax2(fmax2(fmax2(fabs(lkx), fabs(lky)), fmax2(fabs(lkt), fabs(rv))), fmax2(fabs(rc), fabs(re)));
    }
    acc.prinf = fmax2(acc.prinf, prinf); acc.pr1 += pr1; acc.duinf = fmax2(acc.duinf, duinf);
    acc.vmax = fmax2(acc.vmax, vmax); acc.vmin = fmin2(acc.vmin, vmin); acc.l1 += l1;
    acc.z1 += z1; acc.f += sf * f; acc.lnsum += lnsum;
}

#define NMPC_AZ_RESTO (-1.0)
#define NMPC_AZ_RESTO_END (-2.0)
#define NMPC_RESTO_MAX_IT 50
#define NMPC_RESTO_MAX_BT 30

// ---------------------------------------------------------------- P3: apply the accepted step, write coefficients
// With FL_APPLY: s += alpha ds, lambda += alpha (lambda^+ - lambda), u, z updated (W&B A-6); the sin/cos of
// the point evaluated in P1 become the iterate's.  Then writes A_k, d_k and the work slots
//   W_0 qv, W_1 qc, W_2 qe, W_3 qw, W_4 qa, W_5 hxx, W_6 htt, W_7 htv, W_8 hee, W_9 hev, W_10 rw, W_11 ra
// for the Riccati sweep.  FL_LSQ: the least-squares multiplier system (identity Hessian, zero defect).
// Must be called for ALL stages of a lane before any stage's coefficients are written when FL_APPLY is
// set (stage k reads stage k-1's D slots and stage k+1's S slots): the caller runs apply for its whole
// group first (apply==1), synchronises the CTA, then calls again with apply==0.
template <bool RATE = false, class SM>
MPC_HD void stage_apply(const Params &prm, const SM &sm, StageRegs &r, int k, int p)
{
    const int N = prm.N;
    // PS_AP_AZ < 0 marks a restoration step: only the primal moves (NMPC_AZ_RESTO), and when restoration ends the bound
    // multipliers are brought back within kappa_Sigma of mu / slack as Ipopt does (NMPC_AZ_RESTO_END)
    const double alpha = sm.P(PS_AP_ALPHA, p), azm = sm.P(PS_AP_AZ, p), mu = sm.P(PS_AP_MU, p);
    const bool resto = azm < 0.0;
    const double az = resto ? 0.0 : azm, al = resto ? 0.0 : alpha;
    if (k > 0)
        for (int c = 0; c < 6; c++) sm.at(k, S_X + c, p) += alpha * sm.at(k - 1, D_X + c, p);
    if (k < N - 1) {
        for (int c = 0; c < 6; c++) {
            const double l = sm.at(k, L_X + c, p);
            sm.at(k, L_X + c, p) = l + al * (sm.at(k, W_LAM + c, p) - l);
        }
        const double uw = r.uw + alpha * sm.at(k, W_DU, p), ua = r.ua + alpha * sm.at(k, W_DU + 1, p);
        double zlw, zuw, zla, zua;
        trial_z(prm, sm, r, k, p, az, mu, uw, ua, zlw, zuw, zla, zua);
        if (azm == NMPC_AZ_RESTO_END) {
            const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
            zlw = zclamp(zlw, mu, 1.0 / (uw + Uw)); zuw = zclamp(zuw, mu, 1.0 / (Uw - uw));
            zla = zclamp(zla, mu, 1.0 / (ua + Ua)); zua = zclamp(zua, mu, 1.0 / (Ua - ua));
        }
        r.uw = uw; r.ua = ua; r.zlw = zlw; r.zuw = zuw; r.zla = zla; r.zua = zua;
        if (RATE) { sm.at(k, U_W, p) = uw; sm.at(k, U_A, p) = ua; }
    }
    r.sn = r.tsn; r.cs = r.tcs; r.se = r.tse; r.ce = r.tce;
}

// Second-order correction (W&B A-5.5 .. A-5.9; Ipopt TrySecondOrderCorrection): the rejected trial point
// iterate + a * step (a = PS_ALPHA; the step is still in the D / W_DU slots) gives the next right-hand side
//   c_soc <- a * c_soc + c(trial),   first attempt: c_soc = c(iterate).
// The right-hand side the pending step was computed with is recovered from the step itself, which satisfies the
// linearised dynamics:  c_old = A_k ds_k + B du_k - ds_{k+1}  (A_k is still in its slots: the iterate has not moved).
// The rows of theta, v, etheta are linear, so their c_soc equals c(iterate) at every attempt (stage_coeffs writes
// them as usual); the rows of x, y, cte are handed to stage_coeffs in r.tsn, r.tcs, r.tse (free until the next
// evaluation).  Runs in P3a, before stage_coeffs of any stage overwrites the step slots.
template <int NC = 4, class SM>
MPC_HD void stage_soc_rhs(const Params &prm, const SM &sm, StageRegs &r, int k, int p, const double *cf)
{
    if (k >= prm.N - 1) return;
    const double a = sm.P(PS_ALPHA, p), dt = prm.dt;
    double dsx = 0, dsy = 0, dst = 0, dsv = 0, dse = 0;
    if (k > 0) {
        dsx = sm.at(k - 1, D_X, p); dsy = sm.at(k - 1, D_Y, p); dst = sm.at(k - 1, D_T, p);
        dsv = sm.at(k - 1, D_V, p); dse = sm.at(k - 1, D_E, p);
    }
    const double nsx = sm.at(k, D_X, p), nsy = sm.at(k, D_Y, p), nsc = sm.at(k, D_C, p);
    const double bx = (dsx + sm.at(k, A_13, p) * dst + sm.at(k, A_14, p) * dsv) - nsx;
    const double by = (dsy + sm.at(k, A_23, p) * dst + sm.at(k, A_24, p) * dsv) - nsy;
    const double bc = (sm.at(k, A_51, p) * dsx - dsy + sm.at(k, A_54, p) * dsv + sm.at(k, A_56, p) * dse) - nsc;
    const double x = sm.at(k, S_X, p) + a * dsx, y = sm.at(k, S_Y, p) + a * dsy;
    const double th = sm.at(k, S_T, p) + a * dst, v = sm.at(k, S_V, p) + a * dsv, e = sm.at(k, S_E, p) + a * dse;
    const double nx = sm.at(k + 1, S_X, p) + a * nsx, ny = sm.at(k + 1, S_Y, p) + a * nsy, nc = sm.at(k + 1, S_C, p) + a * nsc;
    double sn, cs, se, ce, poly, d1, d2;
    sincos_d(th, &sn, &cs);
    sincos_d(e, &se, &ce);
    path_poly<NC>(cf, x, poly, d1, d2);
    (void)ce; (void)d1; (void)d2;
    r.tsn = a * bx + (nx - (x + v * cs * dt));
    r.tcs = a * by + (ny - (y + v * sn * dt));
    r.tse = a * bc + (nc - ((poly - y) + v * se * dt));
}

// Diagonal of the stage Hessian that is constant over the horizon: {x, y, theta, v, cte, etheta}, u.
struct HessDiag { double dx, dy, dt_, dv, dc, de, du; double rw, ra; /* 2 sf w_angvel_d, 2 sf w_accel_d */ };
MPC_HD HessDiag hess_diag(const Params &prm, double sf, double dw, int lsq)
{
    HessDiag h;
    h.rw = 0.0; h.ra = 0.0;
    if (lsq) { h.dx = h.dy = h.dt_ = h.dv = h.dc = h.de = 1.0; h.du = 0.0; return h; }
    h.rw = 2.0 * sf * prm.w_angvel_d; h.ra = 2.0 * sf * prm.w_accel_d;
    h.dx = dw; h.dy = dw; h.dt_ = dw; h.du = dw;
    h.dv = 2.0 * sf * prm.w_vel + dw;
    h.dc = 2.0 * sf * prm.w_cte + dw;
    h.de = 2.0 * sf * prm.w_etheta + dw;
    return h;
}

template <bool RATE = false, int NC = 4, class SM>
MPC_HD void stage_coeffs(const Params &prm, const SM &sm, StageRegs &r, int k, int p, int lsq, const double *cf, int soc = 0)
{
    const int N = prm.N;
    const double sf = sm.P(PS_SF, p), mu = sm.P(PS_MU, p), refv = sm.P(PS_REFV, p), dt = prm.dt;
    const double x = sm.at(k, S_X, p), y = sm.at(k, S_Y, p), th = sm.at(k, S_T, p);
    const double v = sm.at(k, S_V, p), ct = sm.at(k, S_C, p), e = sm.at(k, S_E, p);
    const double qv = 2.0 * sf * prm.w_vel * (v - refv);
    const double qc = 2.0 * sf * prm.w_cte * (ct - prm.ref_cte);
    const double qe = 2.0 * sf * prm.w_etheta * (e - prm.ref_etheta);
    if (k < N - 1) {
        double poly, dpoly, ddpoly;
        path_poly<NC>(cf, x, poly, dpoly, ddpoly);
        sm.at(k, A_13, p) = -v * r.sn * dt; sm.at(k, A_14, p) = r.cs * dt;
        sm.at(k, A_23, p) = v * r.cs * dt;  sm.at(k, A_24, p) = r.sn * dt;
        sm.at(k, A_51, p) = dpoly; sm.at(k, A_54, p) = r.se * dt; sm.at(k, A_56, p) = v * r.ce * dt;
        const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
        const double ilw = fast_rcp(r.uw + Uw), iuw = fast_rcp(Uw - r.uw);
        const double ila = fast_rcp(r.ua + Ua), iua = fast_rcp(Ua - r.ua);
        double gw = 2.0 * sf * prm.w_angvel * r.uw, ga = 2.0 * sf * prm.w_accel * r.ua;
        double rdw = 0.0, rda = 0.0;     // diagonal Hessian contribution of the rate terms this control is part of
        if (RATE) {
            const bool hp = k >= 1, hn = k <= N - 3;
            const double upw = hp ? sm.at(k - 1, U_W, p) : 0.0, upa = hp ? sm.at(k - 1, U_A, p) : 0.0;
            const double unw = hn ? sm.at(k + 1, U_W, p) : 0.0, una = hn ? sm.at(k + 1, U_A, p) : 0.0;
            gw += rate_grad(2.0 * sf * prm.w_angvel_d, r.uw, upw, unw, hp, hn);
            ga += rate_grad(2.0 * sf * prm.w_accel_d, r.ua, upa, una, hp, hn);
            const double cnt = (hp ? 1.0 : 0.0) + (hn ? 1.0 : 0.0);
            rdw = 2.0 * sf * prm.w_angvel_d * cnt; rda = 2.0 * sf * prm.w_accel_d * cnt;
        }
        double hxx = 0.0, htt = 0.0, htv = 0.0, hee = 0.0, hev = 0.0;
        // the constant diagonal of the stage Hessian (hess_diag) is added here, not in the backward sweep
        const HessDiag hd = hess_diag(prm, sf, sm.P(PS_DW, p), lsq);
        // plain variant: the sweeps work with the control step scaled by dt (riccati_backward): q_u / dt, R / dt^2
        const double su = RATE ? 1.0 : prm.idt, su2 = su * su;
        if (lsq) {
            // least-squares multipliers (1): right-hand side (gradient, 0); restoration step (2): right-hand side (0, defect)
            sm.at(k, W_3, p) = lsq == 2 ? 0.0 : (gw - r.zlw + r.zuw) * su;
            sm.at(k, W_4, p) = lsq == 2 ? 0.0 : (ga - r.zla + r.zua) * su;
            sm.at(k, W_10, p) = (1.0 + hd.du) * su2; sm.at(k, W_11, p) = (1.0 + hd.du) * su2;
            if (lsq == 2) {
                sm.at(k, D_X, p) = (x + v * r.cs * dt) - sm.at(k + 1, S_X, p);
                sm.at(k, D_Y, p) = (y + v * r.sn * dt) - sm.at(k + 1, S_Y, p);
                sm.at(k, D_T, p) = (th + r.uw * dt) - sm.at(k + 1, S_T, p);
                sm.at(k, D_V, p) = (v + r.ua * dt) - sm.at(k + 1, S_V, p);
                sm.at(k, D_C, p) = ((poly - y) + v * r.se * dt) - sm.at(k + 1, S_C, p);
                sm.at(k, D_E, p) = (e + r.uw * dt) - sm.at(k + 1, S_E, p);
            } else {
                for (int c = 0; c < 6; c++) sm.at(k, D_X + c, p) = 0.0;
            }
        } else {
            // d_k = -(s_{k+1} - phi(s_k, u_k))  (mpc_planner.cpp:208-215)
            sm.at(k, D_X, p) = (x + v * r.cs * dt) - sm.at(k + 1, S_X, p);
            sm.at(k, D_Y, p) = (y + v * r.sn * dt) - sm.at(k + 1, S_Y, p);
            sm.at(k, D_T, p) = (th + r.uw * dt) - sm.at(k + 1, S_T, p);
            sm.at(k, D_V, p) = (v + r.ua * dt) - sm.at(k + 1, S_V, p);
            sm.at(k, D_C, p) = ((poly - y) + v * r.se * dt) - sm.at(k + 1, S_C, p);
            sm.at(k, D_E, p) = (e + r.uw * dt) - sm.at(k + 1, S_E, p);
            if (soc) { sm.at(k, D_X, p) = -r.tsn; sm.at(k, D_Y, p) = -r.tcs; sm.at(k, D_C, p) = -r.tse; }   // -c_soc (stage_soc_rhs)
            const double mx = sm.at(k, L_X, p), my = sm.at(k, L_Y, p), mc = sm.at(k, L_C, p);
            // second derivatives of the constraint rows weighted by lambda_{k+1} (SURVEY section 0)
            // (stage_step recomputes these five instead of keeping them in registers across the cycle)
            hxx = -mc * ddpoly;
            htt = (mx * r.cs + my * r.sn) * v * dt;
            htv = (mx * r.sn - my * r.cs) * dt;
            hee = mc * v * r.se * dt;
            hev = -mc * r.ce * dt;
            sm.at(k, W_3, p) = (gw - mu * ilw + mu * iuw) * su;     // gradient of the barrier objective
            sm.at(k, W_4, p) = (ga - mu * ila + mu * iua) * su;
            sm.at(k, W_10, p) = ((2.0 * sf * prm.w_angvel + rdw + r.zlw * ilw + r.zuw * iuw) + hd.du) * su2;   // R + Sigma + delta
            sm.at(k, W_11, p) = ((2.0 * sf * prm.w_accel + rda + r.zla * ila + r.zua * iua) + hd.du) * su2;
        }
        sm.at(k, W_5, p) = hxx + hd.dx; sm.at(k, W_6, p) = htt + hd.dt_; sm.at(k, W_7, p) = htv;
        sm.at(k, W_8, p) = hee + hd.de; sm.at(k, W_9, p) = hev;
    }
    sm.at(k, W_0, p) = qv; sm.at(k, W_1, p) = qc; sm.at(k, W_2, p) = qe;
    if (lsq == 2) { sm.at(k, W_0, p) = 0.0; sm.at(k, W_1, p) = 0.0; sm.at(k, W_2, p) = 0.0; }      // (rare: restoration step)
}

// ---------------------------------------------------------------- Riccati sweeps (control thread)

// Coefficients of one stage as the backward sweep consumes them.
struct StageCoef {
    double a13, a14, a23, a24, a51, a54, a56;
    double dx, dy, dth, dv, dc, de;
    double qv, qc, qe, qw, qa;
    double hxx, htt, htv, hee, hev;
    double rw, ra;
};
template <class SM>
MPC_HD void load_coef(const SM &sm, int k, int p, StageCoef &c)
{
    c.a13 = sm.at(k, A_13, p); c.a14 = sm.at(k, A_14, p); c.a23 = sm.at(k, A_23, p); c.a24 = sm.at(k, A_24, p);
    c.a51 = sm.at(k, A_51, p); c.a54 = sm.at(k, A_54, p); c.a56 = sm.at(k, A_56, p);
    c.dx = sm.at(k, D_X, p); c.dy = sm.at(k, D_Y, p); c.dth = sm.at(k, D_T, p);
    c.dv = sm.at(k, D_V, p); c.dc = sm.at(k, D_C, p); c.de = sm.at(k, D_E, p);
    c.qv = sm.at(k, W_0, p); c.qc = sm.at(k, W_1, p); c.qe = sm.at(k, W_2, p);
    c.qw = sm.at(k, W_3, p); c.qa = sm.at(k, W_4, p);
    c.hxx = sm.at(k, W_5, p); c.htt = sm.at(k, W_6, p); c.htv = sm.at(k, W_7, p);
    c.hee = sm.at(k, W_8, p); c.hev = sm.at(k, W_9, p);
    c.rw = sm.at(k, W_10, p); c.ra = sm.at(k, W_11, p);
}

// Backward sweep over stages N-1 .. 0.  5x5 value matrix over (x,y,theta,v,etheta); the cte
// row/column of A is zero, so cte only contributes a rank-one term.  Returns 0 if some
// R~_k is not positive definite (wrong KKT inertia), else 1.  Overwrites W_0..W_11 of each
// stage k <= N-2 with the gains K (2x5) and k_ff (2).  The sweep is one long dependency chain
// through P; everything that does not depend on P is kept off that chain.  (Prefetching the next
// stage's coefficients into registers was measured slower: it costs 50 live registers.)
// RATE: the rate penalties add the cross term  -du_k^T D du_{k-1}  (D = diag(hd.rw, hd.ra)) to the QP; the
// value function then also depends on the previous control step pi = du_{k-1}:
//   V_k = 1/2 ds'P ds + p'ds + ds'M pi + 1/2 pi'N pi + n'pi,   M_k = -K_k^T D,  N_k = -D R~_k^{-1} D,  n_k = -D kff_k,
// so stage k needs K, R~^{-1} and kff of stage k+1 (kept in registers) and contributes
//   R~ += B'M + M'B + N,   S~ += M'A,   r~_u += M'd + n;   forward: du_k += R~^{-1} D du_{k-1}.
template <bool RATE = false, class SM>
MPC_HD int riccati_backward5(const Params &prm, const SM &sm, int p, const HessDiag &hd)
{
    const int N = prm.N;
    const double dt = prm.dt, dt2 = dt * dt;
    // terminal stage
    double Pxx = hd.dx, Pxy = 0, Pxt = 0, Pxv = 0, Pxe = 0, Pyy = hd.dy, Pyt = 0, Pyv = 0, Pye = 0;
    double Ptt = hd.dt_, Ptv = 0, Pte = 0, Pvv = hd.dv, Pve = 0, Pee = hd.de;
    double px = 0, py = 0, pt = 0, pv = sm.at(N - 1, W_0, p), pe = sm.at(N - 1, W_2, p);
    double qc_next = sm.at(N - 1, W_1, p);
    const double gam = hd.dc;
    int ok = 1;
    StageCoef c;
    // RATE: M, N, n of stage k+1 (zero at the terminal stage)
    double Mxw = 0, Myw = 0, Mtw = 0, Mvw = 0, Mew = 0, Mxa = 0, Mya = 0, Mta = 0, Mva = 0, Mea = 0;
    double Nww = 0, Nwa = 0, Naa = 0, nw = 0, na = 0;
#pragma unroll 1
    for (int k = N - 2; k >= 0; k--) {
        load_coef(sm, k, p, c);

        // ---- R~ = R + B^T P B  (B = dt [e_theta + e_etheta | e_v]) and its inverse: the head of the
        //      critical chain, needs only P_{k+1}
        // (c.rw, c.ra, c.hxx, c.htt, c.hee include hess_diag.  Plain variant: the sweeps work with the control step
        //  scaled by dt, du~ = dt du, so that B has unit entries and R~, S~, r~_u need no multiplications by dt:
        //  c.rw, c.ra are R / dt^2 and c.qw, c.qa are q_u / dt; the gains are those of du~.)
        double Rww = RATE ? c.rw + dt2 * ((Ptt + Pee) + 2.0 * Pte) : c.rw + ((Ptt + Pee) + 2.0 * Pte);
        double Rwa = RATE ? dt2 * (Ptv + Pve) : Ptv + Pve;
        double Raa = RATE ? c.ra + dt2 * Pvv : c.ra + Pvv;
        if (RATE) {
            Rww += 2.0 * dt * (Mtw + Mew) + Nww;
            Rwa += dt * ((Mta + Mea) + Mvw) + Nwa;
            Raa += 2.0 * dt * Mva + Naa;
        }
        const double det = Rww * Raa - Rwa * Rwa;
        if (!(Rww > 0.0) || !(det > 0.0)) ok = 0;
        const double idet = fast_rcp(det);
        const double i11 = Raa * idet, i12 = -Rwa * idet, i22 = Rww * idet;

        // ---- W = P A5 (columns theta, v change), M = A5^T W
        const double Mxt = Pxt + c.a13 * Pxx + c.a23 * Pxy;
        const double Myt = Pyt + c.a13 * Pxy + c.a23 * Pyy;
        const double Met = Pte + c.a13 * Pxe + c.a23 * Pye;
        const double Mxv = Pxv + c.a14 * Pxx + c.a24 * Pxy;
        const double Myv = Pyv + c.a14 * Pxy + c.a24 * Pyy;
        const double Mev = Pve + c.a14 * Pxe + c.a24 * Pye;
        const double Wtt = Ptt + c.a13 * Pxt + c.a23 * Pyt;
        const double Wtv = Ptv + c.a14 * Pxt + c.a24 * Pyt;   // W[theta][v]
        const double Wvt = Ptv + c.a13 * Pxv + c.a23 * Pyv;   // W[v][theta]
        const double Wvv = Pvv + c.a14 * Pxv + c.a24 * Pyv;
        const double Mtt = Wtt + c.a13 * Mxt + c.a23 * Myt;
        const double Mtv = Wtv + c.a13 * Mxv + c.a23 * Myv;
        const double Mvv = Wvv + c.a14 * Mxv + c.a24 * Myv;

        // ---- S~ = B^T W
        const double sB = RATE ? dt : 1.0;      // (compile-time 1 in the plain variant: the products vanish)
        double Swx = sB * (Pxt + Pxe), Swy = sB * (Pyt + Pye), Swt = sB * (Wtt + Met),
               Swv = sB * (Wtv + Mev), Swe = sB * (Pte + Pee);
        double Sax = sB * Pxv, Say = sB * Pyv, Sat = sB * Wvt, Sav = sB * Wvv, Sae = sB * Pve;
        if (RATE) {   // S~ += M^T A5
            Swx += Mxw; Swy += Myw; Swe += Mew;
            Swt += Mtw + c.a13 * Mxw + c.a23 * Myw; Swv += Mvw + c.a14 * Mxw + c.a24 * Myw;
            Sax += Mxa; Say += Mya; Sae += Mea;
            Sat += Mta + c.a13 * Mxa + c.a23 * Mya; Sav += Mva + c.a14 * Mxa + c.a24 * Mya;
        }

        // ---- vector part (uses P_{k+1}):  p~ = P d + p,  pi_c = gam d_c + q_c,k+1
        // (five independent FMA chains: the sweep is bound by FP64 issue, not by the depth of these sums)
        const double tx = fma(Pxx, c.dx, fma(Pxy, c.dy, fma(Pxt, c.dth, fma(Pxv, c.dv, fma(Pxe, c.de, px)))));
        const double ty = fma(Pxy, c.dx, fma(Pyy, c.dy, fma(Pyt, c.dth, fma(Pyv, c.dv, fma(Pye, c.de, py)))));
        const double tt = fma(Pxt, c.dx, fma(Pyt, c.dy, fma(Ptt, c.dth, fma(Ptv, c.dv, fma(Pte, c.de, pt)))));
        const double tv = fma(Pxv, c.dx, fma(Pyv, c.dy, fma(Ptv, c.dth, fma(Pvv, c.dv, fma(Pve, c.de, pv)))));
        const double te = fma(Pxe, c.dx, fma(Pye, c.dy, fma(Pte, c.dth, fma(Pve, c.dv, fma(Pee, c.de, pe)))));
        const double pic = gam * c.dc + qc_next;

        // ---- Q~ = Q + M + gam a_c a_c^T   (a_c = [a51, -1, 0, a54, a56] over x,y,theta,v,etheta)
        const double g1 = gam * c.a51, g4 = gam * c.a54, g6 = gam * c.a56;
        const double Qxx = Pxx + (g1 * c.a51 + c.hxx);
        const double Qxy = Pxy - g1;
        const double Qxv = Mxv + g1 * c.a54;
        const double Qxe = Pxe + g1 * c.a56;
        const double Qyy = Pyy + (gam + hd.dy);
        const double Qyv = Myv - g4;
        const double Qye = Pye - g6;
        const double Qtt = Mtt + c.htt;
        const double Qtv = Mtv + c.htv;
        const double Qvv = Mvv + (g4 * c.a54 + hd.dv);
        const double Qve = Mev + (g4 * c.a56 + c.hev);
        const double Qee = Pee + (g6 * c.a56 + c.hee);

        // ---- gains  K = -R~^{-1} S~
        const double Kwx = -(i11 * Swx + i12 * Sax), Kax = -(i12 * Swx + i22 * Sax);
        const double Kwy = -(i11 * Swy + i12 * Say), Kay = -(i12 * Swy + i22 * Say);
        const double Kwt = -(i11 * Swt + i12 * Sat), Kat = -(i12 * Swt + i22 * Sat);
        const double Kwv = -(i11 * Swv + i12 * Sav), Kav = -(i12 * Swv + i22 * Sav);
        const double Kwe = -(i11 * Swe + i12 * Sae), Kae = -(i12 * Swe + i22 * Sae);
        // ---- feed-forward
        double ruw = c.qw + sB * (tt + te), rua = c.qa + sB * tv;
        if (RATE) {   // r~_u += M^T d + n
            ruw += (Mxw * c.dx + Myw * c.dy) + (Mtw * c.dth + Mvw * c.dv) + (Mew * c.de + nw);
            rua += (Mxa * c.dx + Mya * c.dy) + (Mta * c.dth + Mva * c.dv) + (Mea * c.de + na);
        }
        const double kfw = -(i11 * ruw + i12 * rua), kfa = -(i12 * ruw + i22 * rua);

        sm.at(k, W_0, p) = Kwx; sm.at(k, W_1, p) = Kwy; sm.at(k, W_2, p) = Kwt; sm.at(k, W_3, p) = Kwv;
        sm.at(k, W_4, p) = Kwe; sm.at(k, W_5, p) = Kax; sm.at(k, W_6, p) = Kay; sm.at(k, W_7, p) = Kat;
        sm.at(k, W_8, p) = Kav; sm.at(k, W_9, p) = Kae; sm.at(k, W_10, p) = kfw; sm.at(k, W_11, p) = kfa;
        if (RATE) {
            sm.at(k, RI_11, p) = i11; sm.at(k, RI_12, p) = i12; sm.at(k, RI_22, p) = i22;
            // M_k = -K^T D, N_k = -D R~^{-1} D, n_k = -D kff  (for stage k-1)
            Mxw = -Kwx * hd.rw; Myw = -Kwy * hd.rw; Mtw = -Kwt * hd.rw; Mvw = -Kwv * hd.rw; Mew = -Kwe * hd.rw;
            Mxa = -Kax * hd.ra; Mya = -Kay * hd.ra; Mta = -Kat * hd.ra; Mva = -Kav * hd.ra; Mea = -Kae * hd.ra;
            Nww = -hd.rw * hd.rw * i11; Nwa = -hd.rw * hd.ra * i12; Naa = -hd.ra * hd.ra * i22;
            nw = -hd.rw * kfw; na = -hd.ra * kfa;
        }

        // ---- P_k = Q~ + S~^T K   (two fused operations per entry)
        Pxx = fma(Swx, Kwx, fma(Sax, Kax, Qxx));
        Pxy = fma(Swx, Kwy, fma(Sax, Kay, Qxy));
        Pxt = fma(Swx, Kwt, fma(Sax, Kat, Mxt));
        Pxv = fma(Swx, Kwv, fma(Sax, Kav, Qxv));
        Pxe = fma(Swx, Kwe, fma(Sax, Kae, Qxe));
        Pyy = fma(Swy, Kwy, fma(Say, Kay, Qyy));
        Pyt = fma(Swy, Kwt, fma(Say, Kat, Myt));
        Pyv = fma(Swy, Kwv, fma(Say, Kav, Qyv));
        Pye = fma(Swy, Kwe, fma(Say, Kae, Qye));
        Ptt = fma(Swt, Kwt, fma(Sat, Kat, Qtt));
        Ptv = fma(Swt, Kwv, fma(Sat, Kav, Qtv));
        Pte = fma(Swt, Kwe, fma(Sat, Kae, Met));
        Pvv = fma(Swv, Kwv, fma(Sav, Kav, Qvv));
        Pve = fma(Swv, Kwe, fma(Sav, Kae, Qve));
        Pee = fma(Swe, Kwe, fma(Sae, Kae, Qee));
        // ---- p_k = q_s + A^T p~ + S~^T k_ff
        px = fma(Swx, kfw, fma(Sax, kfa, fma(c.a51, pic, tx)));
        py = fma(Swy, kfw, fma(Say, kfa, ty - pic));
        pt = fma(Swt, kfw, fma(Sat, kfa, fma(c.a23, ty, fma(c.a13, tx, tt))));
        pv = fma(Swv, kfw, fma(Sav, kfa, fma(c.a54, pic, fma(c.a24, ty, fma(c.a14, tx, c.qv + tv)))));
        pe = fma(Swe, kfw, fma(Sae, kfa, fma(c.a56, pic, c.qe + te)));
        qc_next = c.qc;
    }
    return ok;
}

// Forward sweep: ds_0 = 0 (the initial-condition rows stay satisfied).  Leaves du_k in
// W_10/W_11 of stage k and ds_{k+1} in the D slots of stage k.
template <bool RATE = false, class SM>
MPC_HD void riccati_forward5(const Params &prm, const SM &sm, int p, const HessDiag &hd)
{
    const int N = prm.N;
    const double dt = prm.dt, idt = prm.idt;
    (void)idt;
    double sx = 0, sy = 0, st = 0, sv = 0, sc = 0, se = 0;
    double pw = 0, pa = 0;      // RATE: previous control step
    (void)sc; (void)pw; (void)pa;
#pragma unroll 4
    for (int k = 0; k < N - 1; k++) {
        // du_k = K ds_k + k_ff as a depth-3 tree (this is the loop-carried chain)
        double duw = fma(sm.at(k, W_0, p), sx, sm.at(k, W_1, p) * sy) + fma(sm.at(k, W_2, p), st, sm.at(k, W_3, p) * sv) +
                     fma(sm.at(k, W_4, p), se, sm.at(k, W_10, p));
        double dua = fma(sm.at(k, W_5, p), sx, sm.at(k, W_6, p) * sy) + fma(sm.at(k, W_7, p), st, sm.at(k, W_8, p) * sv) +
                     fma(sm.at(k, W_9, p), se, sm.at(k, W_11, p));
        if (RATE && k >= 1) {   // + R~^{-1} D du_{k-1}
            const double i11 = sm.at(k, RI_11, p), i12 = sm.at(k, RI_12, p), i22 = sm.at(k, RI_22, p);
            duw += i11 * hd.rw * pw + i12 * hd.ra * pa;
            dua += i12 * hd.rw * pw + i22 * hd.ra * pa;
        }
        pw = duw; pa = dua;
        const double a13 = sm.at(k, A_13, p), a14 = sm.at(k, A_14, p), a23 = sm.at(k, A_23, p),
                     a24 = sm.at(k, A_24, p), a51 = sm.at(k, A_51, p), a54 = sm.at(k, A_54, p),
                     a56 = sm.at(k, A_56, p);
        const double nx = sx + a13 * st + a14 * sv + sm.at(k, D_X, p);
        const double ny = sy + a23 * st + a24 * sv + sm.at(k, D_Y, p);
        // (plain variant: duw, dua are the scaled steps dt du; the true step is stored for the stage threads)
        const double bw = RATE ? dt * duw : duw, ba = RATE ? dt * dua : dua;
        const double nt = st + bw + sm.at(k, D_T, p);
        const double nv = sv + ba + sm.at(k, D_V, p);
        const double nc = a51 * sx - sy + a54 * sv + a56 * se + sm.at(k, D_C, p);
        const double ne = se + bw + sm.at(k, D_E, p);
        sm.at(k, W_10, p) = RATE ? duw : duw * idt; sm.at(k, W_11, p) = RATE ? dua : dua * idt;
        sm.at(k, D_X, p) = nx; sm.at(k, D_Y, p) = ny; sm.at(k, D_T, p) = nt;
        sm.at(k, D_V, p) = nv; sm.at(k, D_C, p) = nc; sm.at(k, D_E, p) = ne;
        sx = nx; sy = ny; st = nt; sv = nv; sc = nc; se = ne;
    }
}


// ---------------------------------------------------------------- Riccati sweeps, plain variant: 4 x 4
// theta and etheta obey the same linearised dynamics (both advance by dt du_w), so with ds_0 = 0
//   ds_e,k = ds_theta,k + eps_k,    eps_0 = 0,  eps_{k+1} = eps_k + (d_e,k - d_theta,k)
// is known before the sweep: etheta is eliminated like cte.  The value matrix is 4 x 4 over (x, y, theta, v)
// (10 entries instead of 15, 8 gains instead of 10): the stage cost's etheta terms fold into the theta row / column
//   Q_tt += Q_ee, Q_tv += Q_ev, q_t += q_e + Q_ee eps_k, q_v += Q_ev eps_k,
// and the cte row reads  a_c = [a51, -1, a56, a54],  d_c += a56 eps_k.  About 140 FP64 instructions per stage
// instead of 170.  Gains: W_0..W_3 = K_w (x, y, theta, v), W_4..W_7 = K_a, W_10 / W_11 = k_ff (of the step scaled by dt).
template <class SM>
MPC_HD int riccati_backward4(const Params &prm, const SM &sm, int p, const HessDiag &hd)
{
    const int N = prm.N;
    // eps_{N-1}: the sum of all defect differences (a short serial pre-pass)
    double eps = 0.0;
#pragma unroll 4
    for (int k = 0; k < N - 1; k++) eps += sm.at(k, D_E, p) - sm.at(k, D_T, p);
    // terminal stage (cost diagonal; e = theta + eps)
    double Pxx = hd.dx, Pxy = 0, Pxt = 0, Pxv = 0, Pyy = hd.dy, Pyt = 0, Pyv = 0;
    double Ptt = hd.dt_ + hd.de, Ptv = 0, Pvv = hd.dv;
    double px = 0, py = 0, pt = fma(hd.de, eps, sm.at(N - 1, W_2, p)), pv = sm.at(N - 1, W_0, p);
    double qc_next = sm.at(N - 1, W_1, p);
    const double gam = hd.dc, gdy = gam + hd.dy;
    int ok = 1;
    StageCoef c;
#pragma unroll 1
    for (int k = N - 2; k >= 0; k--) {
        load_coef(sm, k, p, c);
        // ---- R~ = R + B^T P B and its inverse: the head of the critical chain (unit B: the step is scaled by dt)
        const double Rww = c.rw + Ptt, Rwa = Ptv, Raa = c.ra + Pvv;
        const double det = Rww * Raa - Rwa * Rwa;
        if (!(Rww > 0.0) || !(det > 0.0)) ok = 0;
        const double idet = fast_rcp(det);
        const double i11 = Raa * idet, i12 = -Rwa * idet, i22 = Rww * idet;
        // ---- etheta folded into theta
        const double ek = eps - (c.de - c.dth);                  // eps_k
        const double Qtt = c.htt + c.hee, Qtv = c.htv + c.hev;
        const double qt = fma(c.hee, ek, c.qe), qv = fma(c.hev, ek, c.qv);
        const double dc = fma(c.a56, ek, c.dc);
        // ---- W = P A4 (columns theta, v change), M = A4^T W
        const double Mxt = Pxt + c.a13 * Pxx + c.a23 * Pxy;
        const double Myt = Pyt + c.a13 * Pxy + c.a23 * Pyy;
        const double Mxv = Pxv + c.a14 * Pxx + c.a24 * Pxy;
        const double Myv = Pyv + c.a14 * Pxy + c.a24 * Pyy;
        const double Wtt = Ptt + c.a13 * Pxt + c.a23 * Pyt;
        const double Wtv = Ptv + c.a14 * Pxt + c.a24 * Pyt;   // W[theta][v]
        const double Wvt = Ptv + c.a13 * Pxv + c.a23 * Pyv;   // W[v][theta]
        const double Wvv = Pvv + c.a14 * Pxv + c.a24 * Pyv;
        const double Mtt = Wtt + c.a13 * Mxt + c.a23 * Myt;
        const double Mtv = Wtv + c.a13 * Mxv + c.a23 * Myv;
        const double Mvv = Wvv + c.a14 * Mxv + c.a24 * Myv;
        // ---- S~ = B^T W: rows theta and v of W
        const double Swx = Pxt, Swy = Pyt, Swt = Wtt, Swv = Wtv;
        const double Sax = Pxv, Say = Pyv, Sat = Wvt, Sav = Wvv;
        // ---- vector part:  p~ = P d + p,  pi_c = gam d_c + q_c,k+1
        const double tx = fma(Pxx, c.dx, fma(Pxy, c.dy, fma(Pxt, c.dth, fma(Pxv, c.dv, px))));
        const double ty = fma(Pxy, c.dx, fma(Pyy, c.dy, fma(Pyt, c.dth, fma(Pyv, c.dv, py))));
        const double tt = fma(Pxt, c.dx, fma(Pyt, c.dy, fma(Ptt, c.dth, fma(Ptv, c.dv, pt))));
        const double tv = fma(Pxv, c.dx, fma(Pyv, c.dy, fma(Ptv, c.dth, fma(Pvv, c.dv, pv))));
        const double pic = fma(gam, dc, qc_next);
        // ---- Q~ = Q + M + gam a_c a_c^T   (a_c = [a51, -1, a56, a54] over x, y, theta, v)
        const double g1 = gam * c.a51, g4 = gam * c.a54, g6 = gam * c.a56;
        const double Qxx = Pxx + fma(g1, c.a51, c.hxx);
        const double Qxy = Pxy - g1;
        const double Qxt = fma(g1, c.a56, Mxt);
        const double Qxv = fma(g1, c.a54, Mxv);
        const double Qyy = Pyy + gdy;
        const double Qyt = Myt - g6;
        const double Qyv = Myv - g4;
        const double Qtt_ = Mtt + fma(g6, c.a56, Qtt);
        const double Qtv_ = Mtv + fma(g6, c.a54, Qtv);
        const double Qvv = Mvv + fma(g4, c.a54, hd.dv);
        // ---- gains  K = -R~^{-1} S~,  feed-forward
        const double Kwx = -(i11 * Swx + i12 * Sax), Kax = -(i12 * Swx + i22 * Sax);
        const double Kwy = -(i11 * Swy + i12 * Say), Kay = -(i12 * Swy + i22 * Say);
        const double Kwt = -(i11 * Swt + i12 * Sat), Kat = -(i12 * Swt + i22 * Sat);
        const double Kwv = -(i11 * Swv + i12 * Sav), Kav = -(i12 * Swv + i22 * Sav);
        const double ruw = c.qw + tt, rua = c.qa + tv;
        const double kfw = -(i11 * ruw + i12 * rua), kfa = -(i12 * ruw + i22 * rua);
        sm.at(k, W_0, p) = Kwx; sm.at(k, W_1, p) = Kwy; sm.at(k, W_2, p) = Kwt; sm.at(k, W_3, p) = Kwv;
        sm.at(k, W_4, p) = Kax; sm.at(k, W_5, p) = Kay; sm.at(k, W_6, p) = Kat; sm.at(k, W_7, p) = Kav;
        sm.at(k, W_10, p) = kfw; sm.at(k, W_11, p) = kfa;
        // ---- P_k = Q~ + S~^T K
        Pxx = fma(Swx, Kwx, fma(Sax, Kax, Qxx));
        Pxy = fma(Swx, Kwy, fma(Sax, Kay, Qxy));
        Pxt = fma(Swx, Kwt, fma(Sax, Kat, Qxt));
        Pxv = fma(Swx, Kwv, fma(Sax, Kav, Qxv));
        Pyy = fma(Swy, Kwy, fma(Say, Kay, Qyy));
        Pyt = fma(Swy, Kwt, fma(Say, Kat, Qyt));
        Pyv = fma(Swy, Kwv, fma(Say, Kav, Qyv));
        Ptt = fma(Swt, Kwt, fma(Sat, Kat, Qtt_));
        Ptv = fma(Swt, Kwv, fma(Sat, Kav, Qtv_));
        Pvv = fma(Swv, Kwv, fma(Sav, Kav, Qvv));
        // ---- p_k = q_s + A^T p~ + a_c pi_c + S~^T k_ff
        px = fma(Swx, kfw, fma(Sax, kfa, fma(c.a51, pic, tx)));
        py = fma(Swy, kfw, fma(Say, kfa, ty - pic));
        pt = fma(Swt, kfw, fma(Sat, kfa, fma(c.a56, pic, fma(c.a23, ty, fma(c.a13, tx, qt + tt)))));
        pv = fma(Swv, kfw, fma(Sav, kfa, fma(c.a54, pic, fma(c.a24, ty, fma(c.a14, tx, qv + tv)))));
        qc_next = c.qc;
        eps = ek;
    }
    return ok;
}

// Forward sweep of the 4 x 4 form: ds_0 = 0; leaves du_k in W_10 / W_11 of stage k and ds_{k+1} (all six
// components) in the D slots of stage k.
template <class SM>
MPC_HD void riccati_forward4(const Params &prm, const SM &sm, int p)
{
    const int N = prm.N;
    const double idt = prm.idt;
    double sx = 0, sy = 0, st = 0, sv = 0, eps = 0;
#pragma unroll 4
    for (int k = 0; k < N - 1; k++) {
        // du_k = K ds_k + k_ff as a depth-3 tree (this is the loop-carried chain)
        const double duw = fma(sm.at(k, W_0, p), sx, sm.at(k, W_1, p) * sy) + fma(sm.at(k, W_2, p), st, fma(sm.at(k, W_3, p), sv, sm.at(k, W_10, p)));
        const double dua = fma(sm.at(k, W_4, p), sx, sm.at(k, W_5, p) * sy) + fma(sm.at(k, W_6, p), st, fma(sm.at(k, W_7, p), sv, sm.at(k, W_11, p)));
        const double a13 = sm.at(k, A_13, p), a14 = sm.at(k, A_14, p), a23 = sm.at(k, A_23, p),
                     a24 = sm.at(k, A_24, p), a51 = sm.at(k, A_51, p), a54 = sm.at(k, A_54, p),
                     a56 = sm.at(k, A_56, p);
        const double dth = sm.at(k, D_T, p), de = sm.at(k, D_E, p);
        const double nx = sx + a13 * st + a14 * sv + sm.at(k, D_X, p);
        const double ny = sy + a23 * st + a24 * sv + sm.at(k, D_Y, p);
        const double nt = st + duw + dth;
        const double nv = sv + dua + sm.at(k, D_V, p);
        const double nc = a51 * sx - sy + a54 * sv + a56 * (st + eps) + sm.at(k, D_C, p);
        eps += de - dth;
        const double ne = nt + eps;
        // (duw, dua are the scaled steps dt du; the true step is stored for the stage threads)
        sm.at(k, W_10, p) = duw * idt; sm.at(k, W_11, p) = dua * idt;
        sm.at(k, D_X, p) = nx; sm.at(k, D_Y, p) = ny; sm.at(k, D_T, p) = nt;
        sm.at(k, D_V, p) = nv; sm.at(k, D_C, p) = nc; sm.at(k, D_E, p) = ne;
        sx = nx; sy = ny; st = nt; sv = nv;
    }
}

// The sweeps of a variant: rate penalties keep the 5 x 5 + augmented form, the plain variant runs the 4 x 4 one.
template <bool RATE = false, class SM>
MPC_HD int riccati_backward(const Params &prm, const SM &sm, int p, const HessDiag &hd)
{
    if (RATE) return riccati_backward5<RATE>(prm, sm, p, hd);
    return riccati_backward4(prm, sm, p, hd);
}
template <bool RATE = false, class SM>
MPC_HD void riccati_forward(const Params &prm, const SM &sm, int p, const HessDiag &hd)
{
    if (RATE) riccati_forward5<RATE>(prm, sm, p, hd);
    else riccati_forward4(prm, sm, p);
}

// ---------------------------------------------------------------- P5: step-dependent stage work
// Reads ds_k, du_k; returns g_k = q_s + Q_k ds_k (to be stored into W_0..W_5) and accumulates the partials
// (primal fraction-to-boundary limit, dual limit, grad(phi_mu)^T d) into `acc`.
template <bool RATE = false, int NC = 4, class SM>
MPC_HD void stage_step(const Params &prm, const SM &sm, StageRegs &r, int k, int p, const HessDiag &hd, int lsq,
                       StepPart &acc, double *g6, const double *cf)
{
    const int N = prm.N;
    const double mu = sm.P(PS_MU, p), sf = sm.P(PS_SF, p), dt = prm.dt;
    const double v = sm.at(k, S_V, p);
    // objective gradient at the iterate (recomputed: cheaper than three live registers per stage)
    const double qv = 2.0 * sf * prm.w_vel * (v - sm.P(PS_REFV, p));
    const double qc = 2.0 * sf * prm.w_cte * (sm.at(k, S_C, p) - prm.ref_cte);
    const double qe = 2.0 * sf * prm.w_etheta * (sm.at(k, S_E, p) - prm.ref_etheta);
    double dsx = 0, dsy = 0, dst = 0, dsv = 0, dsc = 0, dse = 0;
    if (k > 0) {
        dsx = sm.at(k - 1, D_X, p); dsy = sm.at(k - 1, D_Y, p); dst = sm.at(k - 1, D_T, p);
        dsv = sm.at(k - 1, D_V, p); dsc = sm.at(k - 1, D_C, p); dse = sm.at(k - 1, D_E, p);
    }
    // fraction to the boundary (W&B eq. (15)) as the largest step / slack ratio: alpha_max = min(1, tau / ratio)
    double rmax = 0.0, rzmax = 0.0, gd = qv * dsv + qc * dsc + qe * dse;
    if (k < N - 1) {
        const double duw = sm.at(k, W_DU, p), dua = sm.at(k, W_DU + 1, p);
        if (RATE) { sm.at(k, DU_W, p) = duw; sm.at(k, DU_A, p) = dua; }
        // reciprocal slacks at the iterate, the same values stage_coeffs used; left in W_ISL.. for the trial
        // multipliers of P1 / P3a (the gains that occupied these slots were consumed by the forward sweep)
        const double Uw = relaxed(prm.max_angvel), Ua = relaxed(prm.max_throttle);
        const double ilw = fast_rcp(r.uw + Uw), iuw = fast_rcp(Uw - r.uw);
        const double ila = fast_rcp(r.ua + Ua), iua = fast_rcp(Ua - r.ua);
        sm.at(k, W_ISL, p) = ilw; sm.at(k, W_ISL + 1, p) = iuw; sm.at(k, W_ISL + 2, p) = ila; sm.at(k, W_ISL + 3, p) = iua;
        if (lsq != 1) rmax = fmax2(fmax2(-duw * ilw, duw * iuw), fmax2(-dua * ila, dua * iua));
        if (!lsq) {
            const double mlw = mu * ilw, muw = mu * iuw, mla = mu * ila, mua = mu * iua;
            const double dzlw = mlw - r.zlw - r.zlw * ilw * duw;
            const double dzuw = muw - r.zuw + r.zuw * iuw * duw;
            const double dzla = mla - r.zla - r.zla * ila * dua;
            const double dzua = mua - r.zua + r.zua * iua * dua;
            rzmax = fmax2(fmax2(-dzlw * fast_rcp(r.zlw), -dzuw * fast_rcp(r.zuw)),
                          fmax2(-dzla * fast_rcp(r.zla), -dzua * fast_rcp(r.zua)));
            double gw = 2.0 * sf * prm.w_angvel * r.uw - mlw + muw;
            double ga = 2.0 * sf * prm.w_accel * r.ua - mla + mua;
            if (RATE) {
                const bool hp = k >= 1, hn = k <= N - 3;
                const double upw = hp ? sm.at(k - 1, U_W, p) : 0.0, upa = hp ? sm.at(k - 1, U_A, p) : 0.0;
                const double unw = hn ? sm.at(k + 1, U_W, p) : 0.0, una = hn ? sm.at(k + 1, U_A, p) : 0.0;
                gw += rate_grad(hd.rw, r.uw, upw, unw, hp, hn);
                ga += rate_grad(hd.ra, r.ua, upa, una, hp, hn);
            }
            gd += gw * duw + ga * dua;
        }
    }
    // the five lambda-weighted Hessian entries, exactly as stage_coeffs formed them for the sweep (same
    // operands: the iterate has not moved since); recomputed here so that they do not occupy ten registers
    // per stage for the whole cycle
    double hxx = 0.0, htt = 0.0, htv = 0.0, hee = 0.0, hev = 0.0;
    if (k < N - 1 && !lsq) {
        const double mx = sm.at(k, L_X, p), my = sm.at(k, L_Y, p), mc = sm.at(k, L_C, p);
        double poly_unused, dpoly_unused, ddpoly;
        path_poly<NC>(cf, sm.at(k, S_X, p), poly_unused, dpoly_unused, ddpoly);
        (void)poly_unused; (void)dpoly_unused;
        hxx = -mc * ddpoly;
        htt = (mx * r.cs + my * r.sn) * v * dt;
        htv = (mx * r.sn - my * r.cs) * dt;
        hee = mc * v * r.se * dt;
        hev = -mc * r.ce * dt;
    }
    // g_k = q_s,k + Q_k ds_k  (Q_k = diag + the five lambda-weighted entries)
    // (returned in g6; the caller stores W_0..W_5 after all of its stages are computed)
    g6[0] = (hd.dx + hxx) * dsx;
    g6[1] = hd.dy * dsy;
    g6[2] = (hd.dt_ + htt) * dst + htv * dsv;
    g6[3] = qv + htv * dst + hd.dv * dsv + hev * dse;
    g6[4] = qc + hd.dc * dsc;
    g6[5] = qe + hev * dsv + (hd.de + hee) * dse;
    acc.rmax = fmax2(acc.rmax, rmax); acc.rzmax = fmax2(acc.rzmax, rzmax); acc.gd += gd;
}

// Adjoint sweep: lambda_k^+ = A_k^T lambda_{k+1}^+ - g_k, k = N-1 .. 0.
// lambda_{k+1}^+ replaces g_k in W_LAM..+5 of stage k (stage N-1 keeps g_{N-1}); lambda_0^+ goes to PS_N0*.
// Runs on the lane's stage thread of group 0 while the control thread sets the step sizes (it needs only the
// P5 results).  Returns 1 if some multiplier exceeds NMPC_LAM_MAX in magnitude (or is NaN): the test the
// least-squares start makes (W&B Sec. 3.6), folded into the sweep so that it costs no extra pass.
#define NMPC_LAM_MAX 1e3
template <class SM>
MPC_HD int adjoint_sweep(const Params &prm, const SM &sm, int p)
{
    const int N = prm.N;
    double lx = -sm.at(N - 1, W_0, p), ly = -sm.at(N - 1, W_1, p), lt = -sm.at(N - 1, W_2, p);
    double lv = -sm.at(N - 1, W_3, p), lc = -sm.at(N - 1, W_4, p), le = -sm.at(N - 1, W_5, p);
    int big = 0;
#define NMPC_BIG6() big |= !(fabs(lx) <= NMPC_LAM_MAX) | !(fabs(ly) <= NMPC_LAM_MAX) | !(fabs(lt) <= NMPC_LAM_MAX) | \
                           !(fabs(lv) <= NMPC_LAM_MAX) | !(fabs(lc) <= NMPC_LAM_MAX) | !(fabs(le) <= NMPC_LAM_MAX)
#pragma unroll 4
    for (int k = N - 2; k >= 0; k--) {
        const double g0 = sm.at(k, W_0, p), g1 = sm.at(k, W_1, p), g2 = sm.at(k, W_2, p);
        const double g3 = sm.at(k, W_3, p), g4 = sm.at(k, W_4, p), g5 = sm.at(k, W_5, p);
        sm.at(k, W_LAM, p) = lx; sm.at(k, W_LAM + 1, p) = ly; sm.at(k, W_LAM + 2, p) = lt;
        sm.at(k, W_LAM + 3, p) = lv; sm.at(k, W_LAM + 4, p) = lc; sm.at(k, W_LAM + 5, p) = le;
        NMPC_BIG6();
        const double a13 = sm.at(k, A_13, p), a14 = sm.at(k, A_14, p), a23 = sm.at(k, A_23, p),
                     a24 = sm.at(k, A_24, p), a51 = sm.at(k, A_51, p), a54 = sm.at(k, A_54, p),
                     a56 = sm.at(k, A_56, p);
        const double nx = lx + a51 * lc - g0;
        const double ny = ly - lc - g1;
        const double nt = a13 * lx + a23 * ly + lt - g2;
        const double nv = a14 * lx + a24 * ly + lv + a54 * lc - g3;
        const double nc = -g4;
        const double ne = a56 * lc + le - g5;
        lx = nx; ly = ny; lt = nt; lv = nv; lc = nc; le = ne;
    }
    NMPC_BIG6();
#undef NMPC_BIG6
    sm.P(PS_N0X, p) = lx; sm.P(PS_N0Y, p) = ly; sm.P(PS_N0T, p) = lt;
    sm.P(PS_N0V, p) = lv; sm.P(PS_N0C, p) = lc; sm.P(PS_N0E, p) = le;
    return big;
}

// ---------------------------------------------------------------- control thread state + logic
// Scalars only (lives in registers); the filter entries are in shared memory (sm.F).
struct Ctrl {
    int iter;
    int status;
    int n_accept;          // consecutive "acceptable" iterations
    int nfilt;
    int have_theta0;
    int age;               // global cycles spent on the current problem (watchdog)
    double dw_last;
    double theta_min, theta_max;
    double theta, phi, gd;          // at the current iterate, for the line search
    double alpha_min, sw_log, sw_alpha;
    double E0, obj;
};


// Gradient-based objective scaling at the start point (Ipopt nlp_scaling_max_gradient = 100).
MPC_HD double objective_scaling(const Params &prm, const double *state6, double refv)
{
    double g = fabs(2.0 * prm.w_cte * (state6[4] - prm.ref_cte));
    g = fmax2(g, fabs(2.0 * prm.w_etheta * (state6[5] - prm.ref_etheta)));
    g = fmax2(g, fabs(2.0 * prm.w_vel * (state6[3] - refv)));
    if (prm.N > 1) {
        g = fmax2(g, fabs(2.0 * prm.w_cte * prm.ref_cte));
        g = fmax2(g, fabs(2.0 * prm.w_etheta * prm.ref_etheta));
        g = fmax2(g, fabs(2.0 * prm.w_vel * refv));
    }
    return g > 100.0 ? 100.0 / g : 1.0;
}

// New problem in lane p: the first cycle solves the least-squares multiplier system.
template <class SM>
MPC_HD void ctrl_init(const Params &prm, const SM &sm, Ctrl &c, int p, const double *state6, double refv)
{
    c.iter = 0; c.status = 0; c.n_accept = 0; c.nfilt = 0; c.have_theta0 = 0; c.age = 0;
    c.dw_last = 0.0; c.theta_min = 0.0; c.theta_max = 0.0; c.theta = 0.0; c.phi = 0.0; c.gd = 0.0;
    c.alpha_min = 0.0; c.sw_log = 0.0; c.sw_alpha = 1.0; c.E0 = 1e300; c.obj = 0.0;
    sm.P(PS_MU, p) = NMPC_MU_INIT;
    sm.P(PS_MU_STEP, p) = NMPC_MU_INIT;
    sm.P(PS_TAU, p) = fmax2(NMPC_TAU_MIN, 1.0 - NMPC_MU_INIT);
    sm.P(PS_SF, p) = objective_scaling(prm, state6, refv);
    sm.P(PS_REFV, p) = refv;
    sm.P(PS_ALPHA, p) = 0.0; sm.P(PS_ALPHA_Z, p) = 0.0; sm.P(PS_DW, p) = 0.0;
    for (int i = 0; i < 6; i++) { sm.P(PS_L0X + i, p) = 0.0; sm.P(PS_N0X + i, p) = 0.0; }
}

template <class SM>
MPC_HD int filter_acceptable(const SM &sm, const Ctrl &c, int p, double theta, double phi)
{
    if (!(theta < c.theta_max)) return 0;
    for (int i = 0; i < c.nfilt; i++)
        if (theta >= sm.F(2 * i, p) && phi >= sm.F(2 * i + 1, p)) return 0;
    return 1;
}

template <class SM>
MPC_HD void filter_add(const SM &sm, Ctrl &c, int p, double theta, double phi)
{
    const double th = (1.0 - NMPC_GAMMA_THETA) * theta, ph = phi - NMPC_GAMMA_PHI * theta;
    int j = c.nfilt;
    if (j < NMPC_MAX_FILTER) c.nfilt++;
    else {
        // full: overwrite the entry that dominates least (largest theta)
        j = 0;
        for (int i = 1; i < NMPC_MAX_FILTER; i++) if (sm.F(2 * i, p) > sm.F(2 * j, p)) j = i;
    }
    sm.F(2 * j, p) = th; sm.F(2 * j + 1, p) = ph;
}

// ---- feasibility restoration (rare path).  Ipopt switches to its restoration phase when the backtracking line search
// runs below alpha_min.  As in the oracle (oracle/ipm.c: the stand-in for that phase) the violation theta = ||c||_1 is
// reduced by min-norm Gauss-Newton steps  [I J'; J 0] (dx, .) = (0, -c)  with a backtracking test on theta alone, until
// theta has dropped to 90 % of its value at entry (kappa_resto) and the point is acceptable to the filter; then the bound
// multipliers are reset and the regular iteration continues.  State: theta at entry in PS_ALPHA_LS, current theta_r in
// PS_SOC_THETA, 64 * steps + backtracks in PI_SOC (the second-order-correction slots, idle while restoring).
// Entry (line search failed at the iterate with violation th, barrier objective phi): returns 5 = solve a restoration
// step, or 2 = terminate (status set).
// (Both helpers are kept out of line and take / return plain values -- packed result: low byte = the return code, the
//  rest = the new filter size / iteration count -- so that the control thread's state stays in registers on the hot path.)
template <class SM>
MPC_HD_RARE int ctrl_enter_resto(const SM &sm, int p, double th, double phi, double theta_min, int nfilt)
{
    sm.P(PS_ALPHA, p) = 0.0; sm.P(PS_ALPHA_Z, p) = 0.0;           // (nothing to apply if this terminates)
    if (th <= 1e-13 * (1e4 * theta_min)) return 2 | (3 << 8);      // 1e4 theta_min = max(1, theta_0): tiny step, status 3
    Ctrl t; t.nfilt = nfilt;
    filter_add(sm, t, p, th, phi);                                  // W&B A-9
    sm.P(PS_ALPHA_LS, p) = th; sm.P(PS_SOC_THETA, p) = th; sm.I(PI_SOC, p) = 0;
    return 5 | (t.nfilt << 8);
}
// A restoration trial point (step length PS_ALPHA) has been evaluated: th_t = its violation, phi_t its barrier objective.
// Returns (low byte) 0 = shorter step, same direction; 6 = step taken, another restoration step; 7 = restoration finished,
// the trial point is the new iterate (the caller goes on as for an accepted line-search trial); 2 = terminate with the
// status in the upper bits.
template <class SM>
MPC_HD_RARE int ctrl_decide_resto(const SM &sm, int p, int ok, double th_t, double phi_t, double theta_max, int nfilt)
{
    const double a = sm.P(PS_ALPHA, p), thr = sm.P(PS_SOC_THETA, p);
    const int st = sm.I(PI_SOC, p), steps = st >> 6, bts = st & 63;
    if (ok && th_t < (1.0 - 1e-4 * a) * thr) {
        sm.P(PS_SOC_THETA, p) = th_t;
        Ctrl t; t.theta_max = theta_max; t.nfilt = nfilt;
        if (th_t <= 0.9 * sm.P(PS_ALPHA_LS, p) && filter_acceptable(sm, t, p, th_t, phi_t)) return 7;
        if (steps + 1 >= NMPC_RESTO_MAX_IT) return 2 | ((th_t > 1e-6 ? 5 : 9) << 8);
        sm.I(PI_SOC, p) = (steps + 1) << 6;
        return 6;
    }
    if (bts + 1 >= NMPC_RESTO_MAX_BT) {
        sm.P(PS_ALPHA, p) = 0.0; sm.P(PS_ALPHA_Z, p) = 0.0;
        return 2 | ((thr > 1e-6 ? 5 : 9) << 8);                      // local infeasibility / restoration failure
    }
    sm.I(PI_SOC, p) = (steps << 6) | (bts + 1);
    sm.P(PS_ALPHA, p) = 0.5 * a;
    return 0;
}

// P2: the point evaluated in P1.  Line-search trial (FL_LS): filter test (W&B A-5); a rejected trial
// halves alpha and is evaluated again next cycle.  An accepted point (or a plain evaluation) becomes the
// iterate: convergence test (W&B eq. (5), (6)) and monotone barrier update (eq. (7)).
// Returns: 0 = evaluate again (alpha halved), 1 = iterate accepted, continue with a Newton step,
//          2 = terminated (c.status set; the step, if any, still has to be applied before flushing),
//          3 = solve the same Newton system for a second-order correction (FL_SOC),
//          4 = the corrections failed: recompute the Newton step and resume the backtracking (FL_RESUME),
//          5 = the line search failed: solve a restoration step (FL_RESTO), 6 = restoration step taken, solve another.
#if defined(NMPC_PROFILE) && defined(__CUDACC__)
__device__ long long nmpc_dec_acc[8];
#endif
#if defined(NMPC_PROFILE) && defined(__CUDA_ARCH__)
#define DEC_MARK(i) do { if (threadIdx.x == 0) { long long t_ = clock64(); atomicAdd((unsigned long long *)&nmpc_dec_acc[i], (unsigned long long)(t_ - nmpc_dec_t)); nmpc_dec_t = t_; } } while (0)
#define DEC_START() long long nmpc_dec_t = clock64()
#elif defined(__CUDA_ARCH__)
#define DEC_MARK(i) asm volatile("" ::: "memory")     /* compiler-level fence between the blocks (see PROF_MARK) */
#define DEC_START()
#else
#define DEC_MARK(i)
#define DEC_START()
#endif
// Partial sums of the stage groups [g0, g1) of lane p, added up in group order.
template <class SM>
MPC_HD void ctrl_reduce(const SM &sm, int p, int g0, int g1, EvalPart &s)
{
    s.prinf = 0; s.pr1 = 0; s.duinf = 0; s.vmax = -1e300; s.vmin = 1e300; s.l1 = 0; s.z1 = 0; s.f = 0; s.lnsum = 0; s.inside = 1;
    for (int g = g0; g < g1; g++) {
        s.prinf = fmax2(s.prinf, sm.part(g, PT_0, p)); s.pr1 += sm.part(g, PT_1, p);
        s.duinf = fmax2(s.duinf, sm.part(g, PT_2, p));
        s.vmax = fmax2(s.vmax, sm.part(g, PT_3, p)); s.vmin = fmin2(s.vmin, sm.part(g, PT_4, p));
        s.l1 += sm.part(g, PT_5, p); s.z1 += sm.part(g, PT_6, p); s.f += sm.part(g, PT_7, p);
        const double l = sm.part(g, PT_8, p);
        if (l <= -1e299) s.inside = 0; else s.lnsum += l;
    }
}
// lower half of the groups (+) upper half: the order every build adds them in (the kernel reduces the halves on the two
// half-warps of a control warp, nmpc_kernel.cuh; the host emulator one after the other)
MPC_HD void eval_combine(EvalPart &lo, const EvalPart &hi)
{
    lo.prinf = fmax2(lo.prinf, hi.prinf); lo.pr1 += hi.pr1; lo.duinf = fmax2(lo.duinf, hi.duinf);
    lo.vmax = fmax2(lo.vmax, hi.vmax); lo.vmin = fmin2(lo.vmin, hi.vmin); lo.l1 += hi.l1; lo.z1 += hi.z1; lo.f += hi.f;
    lo.lnsum += hi.lnsum; lo.inside &= hi.inside;
}
MPC_HD int reduce_split(int NG) { return (NG + 1) / 2; }

template <class SM>
MPC_HD int ctrl_decide_sums(const Params &prm, const SM &sm, Ctrl &c, int p, int flags, const EvalPart &sums)
{
    DEC_START();
    const double prinf = sums.prinf, pr1 = sums.pr1, duinf = sums.duinf, vmax = sums.vmax, vmin = sums.vmin, l1 = sums.l1, z1 = sums.z1,
                 f = sums.f, lnsum = sums.lnsum;
    const int inside = sums.inside;
    double mu = sm.P(PS_MU, p);
    const double sf = sm.P(PS_SF, p);
    DEC_MARK(0);
    // The function is written without early returns (ret < 0 = still undecided) so that the lanes of the warp
    // reconverge after every block instead of running the common tail once per path.
    int ret = -1;
    if ((flags & (FL_LS | FL_RESTO)) == (FL_LS | FL_RESTO)) {
        const int ok = inside && (pr1 == pr1) && (f == f);
        const int rr = ctrl_decide_resto(sm, p, ok, pr1, f - mu * lnsum, c.theta_max, c.nfilt);
        ret = rr & 255;
        if (ret == 2) c.status = rr >> 8;
        if (ret == 7) { c.iter++; ret = -1; }
    } else if (flags & FL_LS) {
        const int soc = flags & FL_SOC;
        const double alpha = sm.P(PS_ALPHA, p);
        // a second-order correction is judged with the step length of the rejected first trial (Ipopt:
        // CheckAcceptabilityOfTrialPoint(alpha_primal) inside TrySecondOrderCorrection)
        const double alpha_t = soc ? sm.P(PS_ALPHA_LS, p) : alpha;
        const double phi_t = f - mu * lnsum;
        const double th = c.theta, phi = c.phi, gd = c.gd;
        const int ok = inside && (pr1 == pr1) && (phi_t == phi_t);
        int acc = 0, armijo = 0;
        if (ok && filter_acceptable(sm, c, p, pr1, phi_t)) {
            // switching condition (W&B eq. (19)): alpha (-gd)^s_phi > theta^s_theta, with the right-hand side
            // brought over in ctrl_step_late (c.sw_alpha)
            if (th <= c.theta_min && gd < 0.0 && alpha_t > c.sw_alpha) {
                if (phi_t - phi - 10.0 * NMPC_EPS_MACH * fabs(phi) <= NMPC_ETA_PHI * alpha_t * gd) { acc = 1; armijo = 1; }
            } else {
                if (pr1 <= (1.0 - NMPC_GAMMA_THETA) * th ||
                    phi_t - 10.0 * NMPC_EPS_MACH * fabs(phi) <= phi - NMPC_GAMMA_PHI * th) acc = 1;
            }
        }
        if (!acc) {
            // second-order correction (W&B A-5.5 .. A-5.9): only after the first trial of a step, and only if it did not
            // reduce the constraint violation; up to NMPC_MAX_SOC corrections while theta keeps shrinking by kappa_soc
            const int st = sm.I(PI_SOC, p);
            int again = 0;      // 1: solve for a(nother) correction, 2: corrections given up, resume the backtracking
            if (soc) {
                if (ok && st < NMPC_MAX_SOC && !(pr1 > NMPC_KAPPA_SOC * sm.P(PS_SOC_THETA, p))) {
                    again = 1; sm.I(PI_SOC, p) = st + 1; sm.P(PS_SOC_THETA, p) = pr1;
                } else again = 2;
            } else if (st == 0 && ok && pr1 >= th) {
                again = 1; sm.I(PI_SOC, p) = 1; sm.P(PS_SOC_THETA, p) = th; sm.P(PS_ALPHA_LS, p) = alpha;
            }
            if (again != 1) sm.I(PI_SOC, p) = -1;
            const double a2 = 0.5 * alpha_t;
            if (again == 1) ret = 3;
            // (alpha_min can be 0 or NaN in degenerate cases: the absolute floor bounds the number of halvings)
            else if (a2 < c.alpha_min || !(a2 > 1e-40)) {
                const int rr = ctrl_enter_resto(sm, p, th, phi, c.theta_min, c.nfilt);
                ret = rr & 255;
                if (ret == 2) c.status = rr >> 8; else c.nfilt = rr >> 8;
            }
            else if (again == 2) ret = 4;
            else { sm.P(PS_ALPHA, p) = a2; ret = 0; }
        } else {
            if (!armijo) filter_add(sm, c, p, th, phi);
            c.iter++;
        }
    }
    DEC_MARK(1);
    // ---- the evaluated point is now the iterate
    double base_err = 0.0, isc = 0.0;
    if (ret < 0) {
        // (s_d, s_c of W&B eq. (6); the means over the m + nb and nb multipliers as products with prm.i_mnb, prm.i_nb)
        const double s_d = fmax2(NMPC_S_MAX, (l1 + z1) * prm.i_mnb) * (1.0 / NMPC_S_MAX);
        const double s_c = fmax2(NMPC_S_MAX, z1 * prm.i_nb) * (1.0 / NMPC_S_MAX);
        const double isd = fast_rcp(s_d), isf = fast_rcp(sf);
        isc = fast_rcp(s_c);
        const double compl0 = fmax2(fabs(vmax), fabs(vmin));
        const double du_s = duinf * isd;
        const double E0 = fmax2(fmax2(du_s, prinf), compl0 * isc);
        base_err = fmax2(du_s, prinf);
        c.E0 = E0; c.obj = f * isf;
        if (E0 <= 1e-6 && prinf <= 1e-2 && compl0 * isf <= 1e-2) c.n_accept++; else c.n_accept = 0;
        if (!(E0 == E0) || !(f == f)) { c.status = 11; ret = 2; }
        else if (E0 <= prm.tol && duinf * isf <= 1.0 && prinf <= 1e-4 && compl0 * isf <= 1e-4) { c.status = 1; ret = 2; }
        else if (c.n_accept >= 15) { c.status = 4; ret = 2; }
        else if (c.iter >= prm.max_iter) { c.status = 2; ret = 2; }
    }
    DEC_MARK(2);
    if (ret < 0) {
        // monotone barrier update (W&B eq. (7)); repeated while the barrier problem is already solved
        int changed = 0;
        const double floor_ = fmin2(prm.tol, 1e-4) * (1.0 / (NMPC_KAPPA_EPS + 1.0));
        for (;;) {
            const double cmu = fmax2(fabs(vmax - mu), fabs(vmin - mu));
            const double Emu = fmax2(base_err, cmu * isc);
            if (!(Emu <= NMPC_KAPPA_EPS * mu)) break;
            const double mun = fmax2(floor_, fmin2(NMPC_KAPPA_MU * mu, mu * sqrt(mu)));   // theta_mu = 1.5
            if (!(mun < mu)) break;
            mu = mun; changed = 1;
        }
        if (changed) {
            c.nfilt = 0;
            sm.P(PS_MU, p) = mu;
            sm.P(PS_TAU, p) = fmax2(NMPC_TAU_MIN, 1.0 - mu);
        }
        c.theta = pr1;
        c.phi = f - mu * lnsum;
        if (!c.have_theta0) {
            c.have_theta0 = 1;
            c.theta_max = 1e4 * fmax2(1.0, pr1);
            c.theta_min = 1e-4 * fmax2(1.0, pr1);
        }
        ret = 1;
    }
    DEC_MARK(3);
    return ret;
}

template <class SM>
MPC_HD int ctrl_decide(const Params &prm, const SM &sm, Ctrl &c, int p, int flags, int NG)
{
    EvalPart lo, hi;
    ctrl_reduce(sm, p, 0, reduce_split(NG), lo);
    ctrl_reduce(sm, p, reduce_split(NG), NG, hi);
    eval_combine(lo, hi);
    return ctrl_decide_sums(prm, sm, c, p, flags, lo);
}

// Next regularisation value of the inertia-correction sequence (W&B Algorithm IC).
MPC_HD double next_dw(const Ctrl &c, double dw)
{
    if (dw == 0.0) return (c.dw_last == 0.0) ? NMPC_DW_0 : fmax2(NMPC_DW_MIN, NMPC_KW_MINUS * c.dw_last);
    return (c.dw_last == 0.0) ? NMPC_KW_PLUS_BAR * dw : NMPC_KW_PLUS * dw;
}

// P6: after the step is known and adjoint_sweep has run.  Reduces the step partials and leaves PS_ALPHA
// (first trial), PS_ALPHA_Z and PS_MU_STEP: all the evaluation in P1 needs.
template <class SM>
MPC_HD void ctrl_step(const Params &prm, const SM &sm, Ctrl &c, int p, int NG, int mode = 0)
{
    double rmax = 0.0, rzmax = 0.0, gd = 0.0;
    for (int g = 0; g < NG; g++) {
        rmax = fmax2(rmax, sm.part(g, PT_0, p)); rzmax = fmax2(rzmax, sm.part(g, PT_1, p)); gd += sm.part(g, PT_2, p);
    }
    const double tau = sm.P(PS_TAU, p);
    const double amax = (rmax > tau) ? tau / rmax : 1.0;      // fraction to the boundary, W&B eq. (15)
    const double az = (rzmax > tau) ? tau / rzmax : 1.0;
    // mode & FL_SOC: the step is a second-order correction -- tried at its own fraction-to-the-boundary length, judged with
    // the original step's directional derivative; FL_RESUME: the original step again, its first trial is already rejected
    if (mode & FL_RESTO) {
        // restoration step: the fraction-to-the-boundary length, bound multipliers untouched; line-search state kept
        sm.P(PS_ALPHA, p) = amax; sm.P(PS_ALPHA_Z, p) = 0.0;
        sm.P(PS_MU_STEP, p) = sm.P(PS_MU, p);
        return;
    }
    if (!(mode & FL_SOC)) c.gd = gd;
    if (mode & FL_RESUME) sm.P(PS_ALPHA, p) = 0.5 * sm.P(PS_ALPHA_LS, p);
    else sm.P(PS_ALPHA, p) = amax;
    if (!(mode & (FL_SOC | FL_RESUME))) sm.I(PI_SOC, p) = 0;
    sm.P(PS_ALPHA_Z, p) = az;
    sm.P(PS_MU_STEP, p) = sm.P(PS_MU, p);
}

// The rest of the line-search set-up (only the decision in P2 needs it, so the control thread computes it
// while the stage threads evaluate the first trial point): switching condition (W&B eq. (19)) in log form,
//   log alpha + s_phi log(-gd) > s_theta log theta,   and the minimal step size (eq. (23)).
MPC_HD void ctrl_step_late(Ctrl &c)
{
    const double gd = c.gd, th = c.theta;
    c.sw_log = 0.0; c.sw_alpha = 1.0;
    if (gd < 0.0 && th <= c.theta_min) {
        c.sw_log = NMPC_S_THETA * log(th) - NMPC_S_PHI * log(-gd);      // -inf when theta == 0
        c.sw_alpha = exp(c.sw_log);                                      // 0 .. inf
        c.alpha_min = NMPC_GAMMA_ALPHA * fmin2(fmin2(NMPC_GAMMA_THETA, NMPC_GAMMA_PHI * th / (-gd)), c.sw_alpha);
    } else if (gd < 0.0)
        c.alpha_min = NMPC_GAMMA_ALPHA * fmin2(NMPC_GAMMA_THETA, NMPC_GAMMA_PHI * th / (-gd));
    else
        c.alpha_min = NMPC_GAMMA_ALPHA * NMPC_GAMMA_THETA;
}

// P6 of the first cycle (after adjoint_sweep, `big` = its result): keep the least-squares multipliers unless
// they are huge (W&B Sec. 3.6).
// Returns the FL_KEEP flag (or 0).
template <class SM>
MPC_HD int ctrl_lsq_finish(const Params &prm, const SM &sm, int p, int big)
{
    const int keep = big ? 0 : 1;
    for (int i = 0; i < 6; i++) sm.P(PS_L0X + i, p) = keep ? sm.P(PS_N0X + i, p) : 0.0;
    return keep ? FL_KEEP : 0;
}

// Control-thread part of applying an accepted step: lambda_0.
template <class SM>
MPC_HD void ctrl_apply(const SM &sm, int p)
{
    const double alpha = sm.P(PS_ALPHA, p);
    for (int i = 0; i < 6; i++) {
        const double l = sm.P(PS_L0X + i, p);
        sm.P(PS_L0X + i, p) = l + alpha * (sm.P(PS_N0X + i, p) - l);
    }
}

// ---------------------------------------------------------------- lane transitions, start and write-out of a problem
// The helpers that read or write the batch's arrays take N = prm.N and batch = a.batch as the caller holds them: the kernels
// load both once, and reading them from the arguments again here would keep the compiler from hoisting the index arithmetic.
//
// Refill, control side: problem nidx (after the a.order mapping) takes over lane p.  Its inputs are staged in PS_NX* for
// the stage threads (stage_inputs, P3a); the first cycle rolls a warm start out, or solves the least-squares multiplier
// system of a cold start.
template <bool WARM, int NC, class SM>
MPC_HD void lane_start(const Params &prm, const SM &sm, Ctrl &c, int p, const SolveArgs &a, int nidx, const int N, const int batch)
{
    for (int i = 0; i < 6; i++) sm.P(PS_NX0 + i, p) = a.state[(size_t)i * batch + nidx];
    for (int i = 0; i < 4; i++) sm.P(PS_NX6 + i, p) = a.coeffs[(size_t)i * batch + nidx];
    if (NC > 4)
        for (int i = 4; i < NC; i++)
            sm.P(PS_NXC4 + (i - 4), p) = i < a.ncoef ? a.coeffs[(size_t)i * batch + nidx] : 0.0;
    sm.P(PS_NX10, p) = a.ref_vel ? a.ref_vel[nidx] : prm.ref_vel;
    double s6[6];
    for (int i = 0; i < 6; i++) s6[i] = sm.P(PS_NX0 + i, p);
    ctrl_init(prm, sm, c, p, s6, sm.P(PS_NX10, p));
    if (WARM) {
        sm.P(PS_MU, p) = prm.warm_mu; sm.P(PS_MU_STEP, p) = prm.warm_mu;
        sm.P(PS_TAU, p) = fmax2(NMPC_TAU_MIN, 1.0 - prm.warm_mu);
        const size_t offl = warm_lam(N);
        for (int i = 0; i < 6; i++)
            sm.P(PS_L0X + i, p) = sm.P(PS_SF, p) * a.warm_in[(offl + (size_t)i * N) * batch + nidx];
        sm.I(PI_MODE, p) = MODE_ROLLOUT;
        sm.I(PI_FLAGS, p) |= FL_WARM;
    } else {
        sm.I(PI_MODE, p) = MODE_NEWTON;
        sm.I(PI_FLAGS, p) |= FL_LSQ;
    }
}

// P3a, stage side: the state and path polynomial lane_start staged (cf[0..3] is the cubic part).
template <int NC, class SM>
MPC_HD void stage_inputs(const SM &sm, int p, double *s6, double *cf)
{
    for (int i = 0; i < 6; i++) s6[i] = sm.P(PS_NX0 + i, p);
    for (int i = 0; i < 4; i++) cf[i] = sm.P(PS_NX6 + i, p);
#pragma unroll
    for (int i = 4; i < NC; i++) cf[i] = sm.P(PS_NXC4 + (i - 4), p);
}

// P2, after the decision r = ctrl_decide (md == MODE_EVAL; fl: the flags it decided with): the lane's next mode and flags,
// and in PS_AP_* the step P3a0 applies.  Returns 1 when the lane's problem terminates (then ctrl_finish).
template <class SM>
MPC_HD int ctrl_transition(const Params &prm, const SM &sm, Ctrl &c, int p, int md, int fl, int r)
{
    int term = 0;
    if (md == MODE_EVAL) {
        if (r == 0) {
            sm.I(PI_FLAGS, p) = FL_LS | (fl & FL_RESTO);
        } else if (r == 3 || r == 4) {
            // second-order correction (3) / resume after failed corrections (4): the same Newton system again
            // (PS_DW kept), no step applied
            sm.I(PI_MODE, p) = MODE_NEWTON; sm.I(PI_FLAGS, p) = (r == 3) ? FL_SOC : FL_RESUME;
        } else if (r == 5) {
            // the line search failed: feasibility restoration from the iterate (nothing applied)
            sm.I(PI_MODE, p) = MODE_NEWTON; sm.I(PI_FLAGS, p) = FL_RESTO; sm.P(PS_DW, p) = 0.0;
        } else if (r == 6) {
            // restoration step taken (primal only), the next restoration system from the new point
            sm.P(PS_AP_ALPHA, p) = sm.P(PS_ALPHA, p); sm.P(PS_AP_AZ, p) = NMPC_AZ_RESTO; sm.P(PS_AP_MU, p) = sm.P(PS_MU_STEP, p);
            sm.I(PI_MODE, p) = MODE_NEWTON; sm.I(PI_FLAGS, p) = FL_APPLY | FL_RESTO; sm.P(PS_DW, p) = 0.0;
        } else {
            // the evaluated point becomes the iterate: P3a applies the step (a plain evaluation is
            // a step of length 0 -- it still adopts the sin/cos computed at the evaluated point)
            const int nf = FL_APPLY;
            if ((fl & (FL_LS | FL_RESTO)) == (FL_LS | FL_RESTO)) {
                // restoration ends here (or the problem does): primal step, multipliers kept, z reset
                sm.P(PS_AP_ALPHA, p) = sm.P(PS_ALPHA, p); sm.P(PS_AP_AZ, p) = NMPC_AZ_RESTO_END;
            } else if (fl & FL_LS) {
                sm.P(PS_AP_ALPHA, p) = sm.P(PS_ALPHA, p); sm.P(PS_AP_AZ, p) = sm.P(PS_ALPHA_Z, p);
                ctrl_apply(sm, p);
            } else {
                sm.P(PS_AP_ALPHA, p) = 0.0; sm.P(PS_AP_AZ, p) = 0.0;
            }
            sm.P(PS_AP_MU, p) = sm.P(PS_MU_STEP, p);
            if (r == 1) { sm.I(PI_MODE, p) = MODE_NEWTON; sm.P(PS_DW, p) = 0.0; sm.I(PI_FLAGS, p) = nf; }
            else { term = 1; sm.I(PI_FLAGS, p) = nf | FL_FLUSH; }
        }
    } else if (md == MODE_FAIL) {
        term = 1; sm.I(PI_FLAGS, p) = FL_FLUSH;
    }
    // watchdog: retries and backtracks are bounded, this only guards against the unforeseen
    if (!term && md != MODE_IDLE && ++c.age > 8 * prm.max_iter + 64) {
        if (c.status == 0) c.status = 2;
        term = 1; sm.I(PI_FLAGS, p) = FL_FLUSH;
    }
    return term;
}

// P2, the lane's problem has terminated: its scalar results and lambda_0 (unscaled) are written out, and the lane idles.
// The stage threads flush the last iterate in the next P3a0 (stage_flush), with the scaling kept in PS_AP_SF.
template <class SM>
MPC_HD void ctrl_finish(const Params &prm, const SM &sm, const Ctrl &c, int p, const SolveArgs &a, const int N, const int batch)
{
    const size_t i = (size_t)sm.I(PI_PROB, p);
    if (a.obj) a.obj[i] = c.obj;
    if (a.status) a.status[i] = c.status;
    if (a.iters) a.iters[i] = c.iter;
    if (a.kkt) a.kkt[i] = c.E0;
    sm.P(PS_AP_SF, p) = sm.P(PS_SF, p);
    if (a.warm_out) {
        const size_t offl = warm_lam(N);
        for (int cc = 0; cc < 6; cc++)
            a.warm_out[(offl + (size_t)cc * N) * batch + i] = sm.P(PS_L0X + cc, p) / sm.P(PS_SF, p);
    }
    sm.I(PI_MODE, p) = MODE_IDLE;
}

// P3a0, stage k of a finished problem: the last iterate whatever the status (mpc_planner.cpp:378-401).  Runs after
// ctrl_finish has written the status.
template <class SM>
MPC_HD void stage_flush(const Params &prm, const SM &sm, const StageRegs &r, int k, int p, const SolveArgs &a, const int N, const int batch)
{
    const size_t i = (size_t)sm.I(PI_PROB, p);
    a.pred[((size_t)0 * N + k) * batch + i] = sm.at(k, S_X, p);
    a.pred[((size_t)1 * N + k) * batch + i] = sm.at(k, S_Y, p);
    a.pred[((size_t)2 * N + k) * batch + i] = sm.at(k, S_T, p);
    if (a.status && stage_bound_hit(prm, sm, k, p)) {
        // (every stage that hits writes the same value)
        const int st = a.status[i];
        if (st == 1 || st == 4) a.status[i] = NMPC_STATUS_BOUND_ACTIVE;
    }
    if (k == 0) { a.u0[i] = r.uw; a.u0[(size_t)batch + i] = r.ua; }
    if (a.warm_out) {
        // the warm-start record (layout: stage_init_warm), multipliers unscaled
        double *wo = a.warm_out;
        const double isf = 1.0 / sm.P(PS_AP_SF, p);
        for (int cc = 0; cc < 6; cc++) wo[((size_t)cc * N + k) * batch + i] = sm.at(k, S_X + cc, p);
        const size_t offl = warm_lam(N);
        if (k < N - 1) {
            wo[(warm_uw(N) + k) * batch + i] = r.uw;
            wo[(warm_ua(N) + k) * batch + i] = r.ua;
            for (int cc = 0; cc < 6; cc++)
                wo[(offl + (size_t)cc * N + k + 1) * batch + i] = sm.at(k, L_X + cc, p) * isf;
            const size_t offz = warm_z(N);
            const int nu = N - 1;
            wo[(offz + k) * batch + i] = r.zlw * isf;
            wo[(offz + nu + k) * batch + i] = r.zla * isf;
            wo[(offz + 2 * nu + k) * batch + i] = r.zuw * isf;
            wo[(offz + 3 * nu + k) * batch + i] = r.zua * isf;
        }
    }
}

// ---------------------------------------------------------------- the phases of one lane
// What a lane does in each phase, written once for both kernels and the host emulator; the callers keep their own barriers
// and loops.  The stage side works on one thread's run of stages k0 .. k0+S-1 of lane p (stages >= N are skipped), with the
// run's registers in r[0 .. S-1] and the lane's path polynomial in cf.  The P5 and P1 helpers accumulate partial sums into
// the caller's `acc` and leave storing them to the caller: the dual-group kernel first combines them across the two halves
// of a warp.  As above, N, batch, k0 and p come from the caller.

// P3a, stage side: a lane taking over a new problem (PI_NEXT) initialises the run, from the warm-start record with FL_WARM;
// a lane about to solve a second-order correction computes its right-hand side from the rejected trial point, before the
// coefficients of any stage overwrite the step slots.
template <int S, bool WARM, bool RATE, int NC, class SM>
MPC_HD void stages_init(const Params &prm, const SM &sm, StageRegs *r, double *cf, int k0, int p, const SolveArgs &a,
                        const int N, const int batch)
{
    const int fl = sm.I(PI_FLAGS, p);
    const int idx = sm.I(PI_NEXT, p);
    if (idx >= 0) {
        // (the polynomial goes to cf last: stored through cf before the initialisation, it changes the register
        //  allocation of the kernels whose lane count is a run-time value)
        double s6[6], c[NC];
        stage_inputs<NC>(sm, p, s6, c);
        if (WARM && (fl & FL_WARM)) {
#pragma unroll
            for (int j = 0; j < S; j++)
                if (k0 + j < N) stage_init_warm<RATE>(prm, sm, r[j], k0 + j, p, s6, c, a.warm_in, (size_t)batch, (size_t)idx);
        } else {
#pragma unroll
            for (int j = 0; j < S; j++)
                if (k0 + j < N) stage_init<RATE>(prm, sm, r[j], k0 + j, p, s6, c);
        }
#pragma unroll
        for (int i = 0; i < NC; i++) cf[i] = c[i];
    } else if ((fl & (FL_SOC | FL_APPLY)) == FL_SOC && sm.I(PI_MODE, p) == MODE_NEWTON) {
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_soc_rhs<NC>(prm, sm, r[j], k0 + j, p, cf);
    }
}

// P3a, control side, after the stage side: the flags it consumed are cleared (FL_SOC next to FL_APPLY: the applied step
// was a correction), and the lane's next problem becomes its problem.
template <class SM>
MPC_HD void ctrl_handover(const SM &sm, int p)
{
    const int f0 = sm.I(PI_FLAGS, p);
    sm.I(PI_FLAGS, p) = f0 & ~(FL_APPLY | FL_FLUSH | FL_WARM | ((f0 & FL_APPLY) ? FL_SOC : 0));
    if (sm.I(PI_NEXT, p) >= 0) { sm.I(PI_PROB, p) = sm.I(PI_NEXT, p); sm.I(PI_NEXT, p) = -1; }
}

// P3b, stage side: the Newton-system coefficients of a lane in MODE_NEWTON.
template <int S, bool RATE, int NC, class SM>
MPC_HD void stages_coeffs(const Params &prm, const SM &sm, StageRegs *r, const double *cf, int k0, int p, const int N)
{
    if (sm.I(PI_MODE, p) == MODE_NEWTON) {
        const int lsq = sys_kind(sm.I(PI_FLAGS, p)), soc = sm.I(PI_FLAGS, p) & FL_SOC;
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_coeffs<RATE, NC>(prm, sm, r[j], k0 + j, p, lsq, cf, soc);
    }
}

// P4, control side, lane in MODE_NEWTON, in two parts (the kernels mark the profile between them).  The first samples the
// system to solve (lsq: its sys_kind; mode: its FL_SOC / FL_RESUME / FL_RESTO, kept for P6, where the adjoint sweep's
// thread may rewrite PI_FLAGS), forms the regularised Hessian diagonal and runs the backward sweep.
struct NewtonSys { int lsq, mode, ok; double dw; HessDiag hd; };
template <bool RATE, class SM>
MPC_HD NewtonSys ctrl_newton_backward(const Params &prm, const SM &sm, int p)
{
    NewtonSys s;
    s.lsq = sys_kind(sm.I(PI_FLAGS, p));
    s.mode = sm.I(PI_FLAGS, p) & (FL_SOC | FL_RESUME | FL_RESTO);
    s.dw = sm.P(PS_DW, p);
    s.hd = hess_diag(prm, sm.P(PS_SF, p), s.dw, s.lsq);
    s.ok = riccati_backward<RATE>(prm, sm, p, s.hd);
    return s;
}
// The second runs the forward sweep, after which the lane steps.  If the factorisation had the wrong inertia, the lane
// stays in MODE_NEWTON with the next regularisation (its coefficients are rewritten next cycle), or fails with status 10
// when that would exceed NMPC_DW_MAX; either way it returns 1 (an inertia-correction retry).
template <bool RATE, class SM>
MPC_HD int ctrl_newton_forward(const Params &prm, const SM &sm, Ctrl &c, int p, const NewtonSys &s)
{
    if (s.ok || s.lsq) {
        riccati_forward<RATE>(prm, sm, p, s.hd);
        if (s.dw > 0.0) c.dw_last = s.dw;
        sm.I(PI_MODE, p) = MODE_STEP;
        return 0;
    }
    const double nd = next_dw(c, s.dw);
    if (nd > NMPC_DW_MAX) { c.status = 10; sm.I(PI_MODE, p) = MODE_FAIL; }
    else sm.P(PS_DW, p) = nd;
    return 1;
}

// P5, stage side, lane in MODE_STEP: the step-dependent work of the run, then its g_k into W_0..W_5.  Returns the sys_kind
// of the system stepped, or -1 when the lane is not stepping.  The kernels sample it before B6 for P6, since the control
// thread rewrites the lane's mode and flags there.  (One return value chosen up front: with an early return the
// dual-group kernel keeps a different set of values live across B6.)
template <int S, bool RATE, int NC, class SM>
MPC_HD int stages_step(const Params &prm, const SM &sm, StageRegs *r, const double *cf, int k0, int p, const int N, StepPart &acc)
{
    const bool stepping = sm.I(PI_MODE, p) == MODE_STEP;
    const int kind = stepping ? sys_kind(sm.I(PI_FLAGS, p)) : -1;
    if (stepping) {
        const HessDiag hd = hess_diag(prm, sm.P(PS_SF, p), sm.P(PS_DW, p), kind);
        double gk[S][6];
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_step<RATE, NC>(prm, sm, r[j], k0 + j, p, hd, kind, acc, gk[j], cf);
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N)
                for (int q = 0; q < 6; q++) sm.at(k0 + j, W_0 + q, p) = gk[j][q];
    }
    return kind;
}

// P6, stage side, lane stepping a system of sys_kind `kind` (stages_step): the adjoint sweep; after the least-squares start
// it also sets the lane's flags for P1, which adopts or zeroes the multipliers.
template <class SM>
MPC_HD void stage_adjoint(const Params &prm, const SM &sm, int p, int kind)
{
    const int big = adjoint_sweep(prm, sm, p);
    if (kind == 1) sm.I(PI_FLAGS, p) = FL_ADOPT | ctrl_lsq_finish(prm, sm, p, big);
}

// P6, control side, lane in MODE_STEP (lsq: the system was the least-squares start; mode: as sampled in P4): the step sizes
// and the line-search flags, except after the least-squares start, whose flags stage_adjoint sets.  The lane evaluates in
// P1.  Returns 1 when ctrl_step ran: ctrl_step_late is then due before P2.
template <class SM>
MPC_HD int ctrl_step_sizes(const Params &prm, const SM &sm, Ctrl &c, int p, int NG, int lsq, int mode)
{
    int late = 0;
    if (!lsq) {
        ctrl_step(prm, sm, c, p, NG, mode);
        sm.I(PI_FLAGS, p) = FL_LS | (mode & (FL_SOC | FL_RESTO));
        late = 1;
    }
    sm.I(PI_MODE, p) = MODE_EVAL;
    return late;
}

// P1, stage side, lane in MODE_EVAL: adopts the least-squares multipliers first (FL_ADOPT), then evaluates the run into acc.
// Returns whether the lane evaluated.
template <int S, bool RATE, int NC, class SM>
MPC_HD bool stages_eval(const Params &prm, const SM &sm, StageRegs *r, const double *cf, int k0, int p, const int N, EvalPart &acc)
{
    if (sm.I(PI_MODE, p) != MODE_EVAL) return false;
    const int fl = sm.I(PI_FLAGS, p);
    if (fl & FL_ADOPT) {
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_adopt(prm, sm, k0 + j, p, fl);
    }
#pragma unroll
    for (int j = 0; j < S; j++)
        if (k0 + j < N) stage_eval<RATE, NC>(prm, sm, r[j], k0 + j, p, fl, acc, cf);
    return true;
}

// P3a0, stage side: applies the step P2 accepted (FL_APPLY) and writes a finished problem out (FL_FLUSH).
template <int S, bool RATE, class SM>
MPC_HD void stages_apply(const Params &prm, const SM &sm, StageRegs *r, int k0, int p, const SolveArgs &a, const int N,
                         const int batch)
{
    const int fl = sm.I(PI_FLAGS, p);
    if (fl & FL_APPLY) {
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_apply<RATE>(prm, sm, r[j], k0 + j, p);
    }
    if (fl & FL_FLUSH) {
#pragma unroll
        for (int j = 0; j < S; j++)
            if (k0 + j < N) stage_flush(prm, sm, r[j], k0 + j, p, a, N, batch);
    }
}

}  // namespace nmpc
