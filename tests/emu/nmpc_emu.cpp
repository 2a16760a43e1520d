// tests/emu/nmpc_emu.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// Runs the solver's phase functions (mpc_ros_b200/csrc/nmpc_phases.cuh, the code both CUDA kernels
// execute: the arithmetic, what each lane does in each phase, the per-lane state machine, the start of
// a problem in a lane and the write-out of its results) sequentially on the host, one emulated CTA of
// PB lanes at a time.  What is the emulator's own is the driver: the kernel's cycle (nmpc_kernel.cuh)
// as one loop per phase over the lanes and their stage groups of SPT stages, in the kernel's phase
// order and in ascending groups, in place of the barriers; the P2 loop; the warm start's roll-out in P4
// (control_loop's MODE_ROLLOUT branch); and the counters.  (The kernel's work queue is not emulated: lanes
// get their problems statically; results do not depend on the lane, which the tests check.)  With a
// warm-start record (warm_in) it runs the kernel's warm instantiation: lane_start<true> and
// stages_init<SPT, true, ...>.  It exists so that the solver
// LOGIC can be checked against the oracle in the CPU-only test tier (this container has no GPU).  It
// is built only by tests/ into tests/emu/libnmpc_emu.so, is never linked into libmpc_b200.so, and
// nothing in the product path can reach it.
#include "../../mpc_ros_b200/csrc/nmpc_phases.cuh"
#include <vector>
#include <cstring>

using namespace nmpc;

static long long g_lane_cycles = 0;
static std::vector<int> g_ages, g_kinds;   // g_kinds: 4 per problem: backtracks, corrections, resumes, inertia retries
static std::vector<int> g_kind_lane;
static std::vector<int> g_ages_unused;      // global cycles each problem of the last run took (tail studies)

static const int SPT = 2;   // same grouping of partial sums as the kernel's stage threads

// The kernel's arguments for one batch.  prm14: dt, ref_cte, ref_etheta, ref_vel, w_cte, w_etheta, w_vel, w_angvel,
// w_accel, max_angvel, max_throttle, w_angvel_d, w_accel_d, bound_value (0 = the 1e3 default).
static SolveArgs emu_args(int N, const double *prm14, double tol, int max_iter, int PB, int batch, int ncoef,
                          const double *state, const double *coeffs, const double *ref_vel, const double *warm_in, double warm_mu,
                          double *u0, double *pred, double *obj, int *status, int *iters, double *kkt, double *warm_out)
{
    SolveArgs a = {};
    Params &prm = a.prm;
    prm.N = N;
    prm.dt = prm14[0]; prm.ref_cte = prm14[1]; prm.ref_etheta = prm14[2]; prm.ref_vel = prm14[3];
    prm.w_cte = prm14[4]; prm.w_etheta = prm14[5]; prm.w_vel = prm14[6]; prm.w_angvel = prm14[7];
    prm.w_accel = prm14[8]; prm.max_angvel = prm14[9]; prm.max_throttle = prm14[10];
    prm.tol = tol; prm.max_iter = max_iter;
    prm.warm_mu = warm_mu;
    prm.w_angvel_d = prm14[11]; prm.w_accel_d = prm14[12];
    prm.grp = SPT;
    prm.idt = 1.0 / prm.dt;
    prm.i_mnb = 1.0 / (double)(6 * N + 4 * (N - 1)); prm.i_nb = 1.0 / (double)(4 * (N - 1));
    prm.bound_chk = (prm14[13] > 0.0 ? prm14[13] : 1e3) * (1.0 - 1e-3);
    a.PB = PB; a.batch = batch; a.ncoef = ncoef;
    a.state = state; a.coeffs = coeffs; a.ref_vel = ref_vel;
    a.u0 = u0; a.pred = pred; a.obj = obj; a.status = status; a.iters = iters; a.kkt = kkt; a.warm_out = warm_out;
    a.warm_in = warm_in;
    return a;
}

template <bool RATE, int NC = 4, bool WARM = false>
static int emu_run(const SolveArgs &a, int *n_reg)
{
    const Params &prm = a.prm;
    const int N = prm.N, PB = a.PB, batch = a.batch;
    const int NG = (N + SPT - 1) / SPT;
    g_ages.assign((size_t)batch, 0); g_kinds.assign((size_t)4 * batch, 0); g_kind_lane.assign((size_t)4 * PB, 0);

    const int NS = RATE ? NSLOTS_RATE : NSLOTS;
    std::vector<double> mem(smem_bytes(N, NG, PB, NS) / sizeof(double) + 8);
    SmemT<0, RATE ? NSLOTS_RATE : NSLOTS> sm; sm.PB = PB; sm.carve(mem.data(), N, NG);
    std::vector<StageRegs> regs((size_t)PB * N);   // [lane][stage]: the run of a stage group is contiguous
    std::vector<double> cfs((size_t)NC * PB);
    std::vector<Ctrl> ctrl(PB);
    std::vector<NewtonSys> sys(PB);                // P4 -> P6, as the control thread keeps it
    std::vector<int> nreg(PB), step_kind(PB);      // step_kind: P5 -> P6, as the stage threads keep it
    // the arguments of the stage helpers for group g of lane p: its run of registers, the path polynomial, k0 and p
#define RUN(p, g) &regs[(size_t)(p) * N + (g) * SPT], &cfs[(size_t)NC * (p)], (g) * SPT, (p)

    for (int base = 0; base < batch; base += PB) {
        const int np = (batch - base < PB) ? batch - base : PB;
        std::fill(mem.begin(), mem.end(), 0.0);
        for (int p = 0; p < PB; p++) { sm.I(PI_MODE, p) = MODE_IDLE; sm.I(PI_FLAGS, p) = 0; sm.I(PI_PROB, p) = -1; sm.I(PI_NEXT, p) = -1; }
        // ---- "refill": every lane starts its problem
        for (int p = 0; p < np; p++) {
            sm.I(PI_NEXT, p) = base + p;
            lane_start<WARM, NC>(prm, sm, ctrl[p], p, a, base + p, N, batch);
            nreg[p] = 0; for (int q = 0; q < 4; q++) g_kind_lane[4 * p + q] = 0;
        }
        for (;;) {
            int active = 0;
            for (int p = 0; p < np; p++) active |= (sm.I(PI_MODE, p) != MODE_IDLE) || (sm.I(PI_FLAGS, p) & FL_FLUSH);
            if (!active) break;
            for (int p = 0; p < np; p++) g_lane_cycles += (sm.I(PI_MODE, p) != MODE_IDLE);
            // ---- P3a
            for (int p = 0; p < np; p++)
                for (int g = 0; g < NG; g++) stages_init<SPT, WARM, RATE, NC>(prm, sm, RUN(p, g), a, N, batch);
            for (int p = 0; p < np; p++) ctrl_handover(sm, p);
            // ---- P3b
            for (int p = 0; p < np; p++)
                for (int g = 0; g < NG; g++) stages_coeffs<SPT, RATE, NC>(prm, sm, RUN(p, g), N);
            // ---- P4
            for (int p = 0; p < np; p++) {
                if (sm.I(PI_MODE, p) == MODE_NEWTON) {
                    sys[p] = ctrl_newton_backward<RATE>(prm, sm, p);
                    nreg[p] += ctrl_newton_forward<RATE>(prm, sm, ctrl[p], p, sys[p]);
                }
                if (WARM && sm.I(PI_MODE, p) == MODE_ROLLOUT) {
                    // as control_loop: the roll-out of the warm controls, then a plain evaluation of the start point
                    const size_t i = (size_t)sm.I(PI_PROB, p);
                    double c4[NC];
                    for (int q = 0; q < NC; q++) c4[q] = q < a.ncoef ? a.coeffs[(size_t)q * batch + i] : 0.0;
                    ctrl_rollout<NC>(prm, sm, p, c4);
                    sm.I(PI_MODE, p) = MODE_EVAL;
                    sm.I(PI_FLAGS, p) = 0;
                }
            }
            // ---- P5
            for (int p = 0; p < np; p++)
                for (int g = 0; g < NG; g++) {
                    StepPart acc; part_reset(acc);
                    step_kind[p] = stages_step<SPT, RATE, NC>(prm, sm, RUN(p, g), N, acc);
                    if (step_kind[p] >= 0) part_store(sm, g, p, acc);
                }
            // ---- P6
            for (int p = 0; p < np; p++) {
                if (step_kind[p] >= 0) stage_adjoint(prm, sm, p, step_kind[p]);
                if (sm.I(PI_MODE, p) == MODE_STEP && ctrl_step_sizes(prm, sm, ctrl[p], p, NG, sys[p].lsq == 1, sys[p].mode))
                    ctrl_step_late(ctrl[p]);
            }
            // ---- P1 (each group adopts before it evaluates, as in the kernels: after an adoption, an evaluation uses the
            //      L slots of its own stages only)
            for (int p = 0; p < np; p++)
                for (int g = 0; g < NG; g++) {
                    EvalPart acc; part_reset(acc);
                    if (stages_eval<SPT, RATE, NC>(prm, sm, RUN(p, g), N, acc)) part_store(sm, g, p, acc);
                }
            // ---- P2
            for (int p = 0; p < np; p++) {
                Ctrl &c = ctrl[p];
                const int md = sm.I(PI_MODE, p);
                int fl = 0, r = 0;
                if (md == MODE_EVAL) {
                    fl = sm.I(PI_FLAGS, p);
                    r = ctrl_decide(prm, sm, c, p, fl, NG);
                    if (r == 0) g_kind_lane[4 * p]++; else if (r == 3) g_kind_lane[4 * p + 1]++; else if (r == 4) g_kind_lane[4 * p + 2]++;
                    if (r == 5 || r == 6) g_kind_lane[4 * p + 1]++;      // (restoration steps are counted with the corrections)
                }
                if (ctrl_transition(prm, sm, c, p, md, fl, r)) {
                    const size_t i = (size_t)sm.I(PI_PROB, p);
                    if (n_reg) n_reg[i] = nreg[p];
                    g_ages[i] = c.age + 1; g_kind_lane[4 * p + 3] = nreg[p];
                    for (int q = 0; q < 4; q++) g_kinds[4 * i + q] = g_kind_lane[4 * p + q];
                    ctrl_finish(prm, sm, c, p, a, N, batch);
                }
            }
            // ---- P3a0
            for (int p = 0; p < np; p++)
                for (int g = 0; g < NG; g++) stages_apply<SPT, RATE>(prm, sm, &regs[(size_t)p * N + g * SPT], g * SPT, p, a, N, batch);
        }
    }
#undef RUN
    return 0;
}

extern "C" int nmpc_emu_last_ages(int *out, int n) { int m = (int)g_ages.size() < n ? (int)g_ages.size() : n; for (int i = 0; i < m; i++) out[i] = g_ages[i]; return m; }

extern "C" int nmpc_emu_last_kinds(int *out, int n) { int m = (int)g_kinds.size() < 4 * n ? (int)g_kinds.size() : 4 * n; for (int i = 0; i < m; i++) out[i] = g_kinds[i]; return m; }

// lane-cycles (one lane busy for one global cycle) spent since the last reset: utilisation studies
extern "C" long long nmpc_emu_lane_cycles(int reset) { const long long v = g_lane_cycles; if (reset) g_lane_cycles = 0; return v; }

extern "C" int nmpc_emu_solve(int N, const double *prm14, double tol, int max_iter, int PB, int batch,
                              const double *state, const double *coeffs, const double *ref_vel,
                              double *u0, double *pred, double *obj, int *status, int *iters, double *kkt,
                              double *warm_out /* warm_size x batch, optional */, int *n_reg /* batch, optional */,
                              const double *warm_in /* warm_size x batch, NULL = cold start */, double warm_mu)
{
    const SolveArgs a = emu_args(N, prm14, tol, max_iter, PB, batch, 4, state, coeffs, ref_vel, warm_in, warm_mu, u0, pred, obj,
                                 status, iters, kkt, warm_out);
    // prm14[11], prm14[12]: w_angvel_d, w_accel_d (rate penalties) select the augmented-Riccati variant
    const bool rate = prm14[11] != 0.0 || prm14[12] != 0.0;
    if (warm_in) return rate ? emu_run<true, 4, true>(a, n_reg) : emu_run<false, 4, true>(a, n_reg);
    if (rate) return emu_run<true>(a, n_reg);
    return emu_run<false>(a, n_reg);
}

// Path polynomial of order ncoef - 1 in 4 .. NMPC_MAX_COEFFS - 1 (coeffs: ncoef x batch): the instantiation the
// kernel uses for orders above 3.
extern "C" int nmpc_emu_solve_poly(int N, const double *prm14, double tol, int max_iter, int PB, int batch, int ncoef,
                                   const double *state, const double *coeffs, double *u0, double *pred, double *obj,
                                   int *status, int *iters, double *kkt, double *warm_out /* optional */,
                                   const double *warm_in /* NULL = cold start */, double warm_mu)
{
    if (ncoef < 4 || ncoef > NMPC_MAX_COEFFS) return -1;
    const SolveArgs a = emu_args(N, prm14, tol, max_iter, PB, batch, ncoef, state, coeffs, nullptr, warm_in, warm_mu, u0, pred, obj,
                                 status, iters, kkt, warm_out);
    const bool rate = prm14[11] != 0.0 || prm14[12] != 0.0;
    if (warm_in) return rate ? emu_run<true, NMPC_MAX_COEFFS, true>(a, nullptr) : emu_run<false, NMPC_MAX_COEFFS, true>(a, nullptr);
    if (rate) return emu_run<true, NMPC_MAX_COEFFS>(a, nullptr);
    return emu_run<false, NMPC_MAX_COEFFS>(a, nullptr);
}
