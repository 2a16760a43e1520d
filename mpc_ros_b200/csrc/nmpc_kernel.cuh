// nmpc_kernel.cuh -- the batched NMPC solve kernel for sm_100a.
//
// Persistent CTAs over a global work queue.  A CTA has PB <= 32 problem lanes.  Warps 0 and 1 are the control
// warps (16 lanes each): lane p runs the interior-point logic and the serial Riccati sweeps of the problem
// currently in lane p -- one thread per problem, a different problem in every lane of a warp instruction (no
// shuffles in the recursions).  The other warps are stage threads: thread (g, p) owns stages
// g*SPT .. g*SPT+SPT-1 of lane p's problem and does everything that is parallel over the horizon
// (sin/cos, model derivatives, residual norms, trial-point evaluation, step application).
// All exchange goes through shared memory [stage][slot][lane].  SPT = 2 at N = 20: 2 + 10 warps, 384 threads at
// 168 registers (the register file).
//
// One global cycle = the fixed phase sequence
//   P3a init | P3b coefficients | P4 sweeps | P5 step work | P6 step sizes + adjoint sweep | P1 evaluate |
//   P2 decide | P3a0 apply / flush + refill
// separated by CTA barriers; each lane is a state machine (nmpc::Mode) and takes part in the phases its
// state asks for.  A lane that needs another factorisation (inertia correction) or a shorter trial step
// simply repeats on the next cycle; it never stalls the other lanes.  When a lane's problem terminates,
// its results are written out and the lane pops the next problem from the queue, so lanes never wait
// for the slowest problem of a batch (iteration counts range from 5 to the cap).
// The control warp's serial chain bounds the cycle, so what need not be on it runs beside it: the adjoint
// sweep on the lane's stage thread of group 0 (P6), apply / flush on the stage threads during the refill.
// What a lane does in each phase (the stages_* / stage_adjoint helpers of the stage threads, the ctrl_* helpers of
// the control thread, the lane start and the write-out) is in nmpc_phases.cuh, shared with the dual-group kernel
// and the host emulator (tests/emu).  This file keeps the barriers, the work-queue pop, the vote, the P2 reduction,
// the warm roll-out and the profiling marks.
//
// Replaces, per problem: CppAD::ipopt::solve + Ipopt (mpc_ros/src/mpc_planner.cpp:373-375).
#pragma once
#include "nmpc_phases.cuh"

namespace nmpc {

#ifdef NMPC_PROFILE
#define PROF_DECL long long prof_t = clock64(), prof_acc[12] = {0,0,0,0,0,0,0,0,0,0,0,0}
#define PROF_MARK(i) do { long long t_ = clock64(); prof_acc[i] += t_ - prof_t; prof_t = t_; } while (0)
#define PROF_FLUSH() do { if (a.prof && tid == 0) for (int q_ = 0; q_ < 12; q_++) { if (blockIdx.x == 0) a.prof[q_] = prof_acc[q_]; atomicAdd((unsigned long long *)&a.prof[1008 + q_], (unsigned long long)prof_acc[q_]); } } while (0)
// raw timestamp trace of the first cycles: control thread 0 -> prof[16 + 16*cyc + i], stage thread 32 -> prof[512 + 16*cyc + i]
#define TRACE_C(i) do { if (a.prof && blockIdx.x == 0 && tid == 0 && trace_cyc < 24) a.prof[16 + 16 * trace_cyc + (i)] = clock64(); } while (0)
#define TRACE_S(i) do { if (a.prof && blockIdx.x == 0 && tid == NMPC_CTRL_THREADS && trace_cyc < 24) a.prof[512 + 16 * trace_cyc + (i)] = clock64(); } while (0)
#else
#define PROF_DECL
// (a compiler-level fence at the phase boundaries: the profile build, whose clock reads keep the scheduler from
// moving code across them, was measured 5 % faster than the build without)
#define PROF_MARK(i) asm volatile("" ::: "memory")
#define PROF_FLUSH()
#define TRACE_C(i) asm volatile("" ::: "memory")
#define TRACE_S(i) asm volatile("" ::: "memory")
#endif

// Two control warps of 16 lanes each (on different SM sub-partitions): a warp instruction costs the FP64 pipe the
// same whether 16 or 32 lanes are active, but a 64-bit shared-memory access of 16 lanes is one wavefront instead of
// two, and each warp's divergent P2 logic covers half as many different problems.
#define NMPC_CTRL_WARPS 2
#define NMPC_CTRL_LANES 16
#define NMPC_CTRL_THREADS (32 * NMPC_CTRL_WARPS)
// Barriers.  The single-group kernel synchronises the whole CTA; the dual-group kernel (nmpc_kernel_dual.cuh) runs two
// lane groups out of phase and synchronises each group's control warp with the stage warps on a named barrier of its own.
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ int named_vote(int pred, int id, int count)
{
    int r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
                 : "=r"(r) : "r"(pred), "r"(id), "r"(count) : "memory");
    return r;
}
template <bool DUAL> __device__ __forceinline__ void cta_sync(int id, int count) { if (DUAL) named_sync(id, count); else __syncthreads(); }
template <bool DUAL> __device__ __forceinline__ int cta_vote(int pred, int id, int count) { return DUAL ? named_vote(pred, id, count) : __syncthreads_or(pred); }

// The control warps' loop (one thread per problem lane, 16 lanes per warp): refill, Riccati sweeps, step sizes, decision.
// DUAL: the barriers are the named barrier `bar_id` over `bar_count` threads (this warp + the stage warps).
template <int CPB, bool WARM, bool RATE, int NC, bool DUAL, class SM>
__device__ __forceinline__ void control_loop(const SolveArgs &a, const SM &sm, const int N, const int PB, const int NG, const int batch,
                                             const int tid, const int bar_id, const int bar_count)
{
    const Params &prm = a.prm;
    (void)N; (void)bar_id; (void)bar_count;
    const int p = (tid & 31) % NMPC_CTRL_LANES + NMPC_CTRL_LANES * (tid >> 5);
    const int wl = tid & 31;      // lane within the warp (ballots, shuffles)
    const bool lane = wl < NMPC_CTRL_LANES && p < PB;
    Ctrl c;
    c.status = 0; c.iter = 0; c.E0 = 0.0; c.obj = 0.0;
    if (lane) { sm.I(PI_MODE, p) = MODE_IDLE; sm.I(PI_FLAGS, p) = 0; sm.I(PI_PROB, p) = -1; sm.I(PI_NEXT, p) = -1; }
    bool fin = lane;          // every lane starts by popping a problem
    PROF_DECL;
#ifdef NMPC_PROFILE
    const long long prof_t0 = clock64();
#endif
    int trace_cyc = -1; (void)trace_cyc;
    for (;;) {
        trace_cyc++;
        TRACE_C(0);
        // ---- refill the lanes that finished (fin): one warp-aggregated pop from the work queue; the new
        //      problem's inputs are staged in shared memory for the stage threads (P3a).
        //      (Prefetching the next problem during the sweeps was measured: no gain.)
        {
            const unsigned m = __ballot_sync(0xffffffffu, fin);
            int nb = 0;
            if (wl == 0 && m) nb = atomicAdd(a.queue, __popc(m));
            nb = __shfl_sync(0xffffffffu, nb, 0);
            if (fin) {
                int nidx = nb + __popc(m & ((1u << wl) - 1u));
                if (nidx >= batch) nidx = -1;
                else if (a.order) nidx = a.order[nidx];
                sm.I(PI_NEXT, p) = nidx;
                if (nidx >= 0) lane_start<WARM, NC>(prm, sm, c, p, a, nidx, N, batch);
                else sm.I(PI_MODE, p) = MODE_IDLE;
            }
            fin = false;
        }
        PROF_MARK(1);
        int active = 0;
        if (lane) active = (sm.I(PI_MODE, p) != MODE_IDLE) || (sm.I(PI_FLAGS, p) & FL_FLUSH);
#ifdef NMPC_PROFILE
        {   // busy lanes of this cycle
            const unsigned bz = __ballot_sync(0xffffffffu, lane && sm.I(PI_MODE, p) != MODE_IDLE);
            if (a.prof && wl == 0) atomicAdd((unsigned long long *)&a.prof[1002], (unsigned long long)__popc(bz));
        }
#endif
        if (!cta_vote<DUAL>(active, bar_id, bar_count)) break;   // B2 (vote)
        TRACE_C(1);
        // ---- P3a: stage threads apply / flush / init
        cta_sync<DUAL>(bar_id, bar_count);  // B3
        TRACE_C(2);
        if (lane) ctrl_handover(sm, p);
        // ---- P3b: stage threads write coefficients
        cta_sync<DUAL>(bar_id, bar_count);  // B4
        TRACE_C(3);
        PROF_MARK(2);
        // ---- P4: Riccati sweeps
        int step_lsq = 0;     // sampled here for P6: the lane's adjoint stage thread rewrites PI_FLAGS there
        int step_mode = 0;    // FL_SOC / FL_RESUME / FL_RESTO of the system being solved
        if (lane && sm.I(PI_MODE, p) == MODE_NEWTON) {
            const NewtonSys ns = ctrl_newton_backward<RATE>(prm, sm, p);
            PROF_MARK(3);
            ctrl_newton_forward<RATE>(prm, sm, c, p, ns);
            step_lsq = ns.lsq == 1;
            step_mode = ns.mode;
        }
        if (WARM && lane && sm.I(PI_MODE, p) == MODE_ROLLOUT) {
            const size_t i = (size_t)sm.I(PI_PROB, p);
            double c4[NC];
#pragma unroll
            for (int q = 0; q < NC; q++) c4[q] = q < a.ncoef ? a.coeffs[(size_t)q * batch + i] : 0.0;
            ctrl_rollout<NC>(prm, sm, p, c4);
            sm.I(PI_MODE, p) = MODE_EVAL;       // plain evaluation of the start point in P1
            sm.I(PI_FLAGS, p) = 0;
        }
        PROF_MARK(4);
        TRACE_C(4);
        cta_sync<DUAL>(bar_id, bar_count);  // B5
        TRACE_C(5);
        // ---- P5: stage threads, step-dependent work
        cta_sync<DUAL>(bar_id, bar_count);  // B6
        TRACE_C(6);
        PROF_MARK(5);
        // ---- P6: step sizes; meanwhile the lane's stage thread of group 0 runs the adjoint sweep (multipliers),
        //      which nothing here depends on.  A least-squares lane (FL_LSQ) gets its flags from that thread.
        bool late = false;
        if (lane && sm.I(PI_MODE, p) == MODE_STEP) late = ctrl_step_sizes(prm, sm, c, p, NG, step_lsq, step_mode);
        PROF_MARK(6);
        TRACE_C(7);
        cta_sync<DUAL>(bar_id, bar_count);  // B7
        TRACE_C(8);
        // ---- P1: stage threads evaluate; meanwhile the part of the line-search set-up only P2 needs
        if (late) ctrl_step_late(c);
        cta_sync<DUAL>(bar_id, bar_count);  // B1
        TRACE_C(9);
        PROF_MARK(7);
        // ---- P2: decide.  First the partial sums of the stage groups: the two half-warps take half of the groups each
        //      (lanes l and l + 16 work for the problem of lane l), one exchange, lower half (+) upper half.
        EvalPart sums;
        {
            const int hs = reduce_split(NG), up = wl >> 4;
            if (p < PB) ctrl_reduce(sm, p, up ? hs : 0, up ? NG : hs, sums);
            else ctrl_reduce(sm, 0, 0, 0, sums);
            EvalPart o;
            o.prinf = __shfl_xor_sync(0xffffffffu, sums.prinf, 16); o.pr1 = __shfl_xor_sync(0xffffffffu, sums.pr1, 16);
            o.duinf = __shfl_xor_sync(0xffffffffu, sums.duinf, 16); o.vmax = __shfl_xor_sync(0xffffffffu, sums.vmax, 16);
            o.vmin = __shfl_xor_sync(0xffffffffu, sums.vmin, 16); o.l1 = __shfl_xor_sync(0xffffffffu, sums.l1, 16);
            o.z1 = __shfl_xor_sync(0xffffffffu, sums.z1, 16); o.f = __shfl_xor_sync(0xffffffffu, sums.f, 16);
            o.lnsum = __shfl_xor_sync(0xffffffffu, sums.lnsum, 16); o.inside = __shfl_xor_sync(0xffffffffu, sums.inside, 16);
            eval_combine(sums, o);      // (meaningful in the lower half-warp, the lanes that decide)
        }
        if (lane) {
            const int md = sm.I(PI_MODE, p);
            int fl = 0, r = 0;
            if (md == MODE_EVAL) {
                fl = sm.I(PI_FLAGS, p);
                r = ctrl_decide_sums(prm, sm, c, p, fl, sums);
                PROF_MARK(10);
            }
            if (ctrl_transition(prm, sm, c, p, md, fl, r)) {
                ctrl_finish(prm, sm, c, p, a, N, batch);
                fin = true;
            }
        }
        PROF_MARK(8);
        TRACE_C(10);
        cta_sync<DUAL>(bar_id, bar_count);  // B1b: the stage threads apply / flush while the lanes are refilled
    }
    PROF_FLUSH();
#ifdef NMPC_PROFILE
    if (a.prof && tid == 0) {   // all CTAs: number of global cycles and their total duration
        atomicAdd((unsigned long long *)&a.prof[1000], (unsigned long long)(trace_cyc));
        atomicAdd((unsigned long long *)&a.prof[1001], (unsigned long long)(clock64() - prof_t0));
    }
#endif
}

// NC: coefficients of the path polynomial the instantiation carries (4 = the cubic of the reference's only caller;
// 8 serves orders 4..7, rows beyond a.ncoef read as zero).
// (one stage per thread is the latency mode of narrow CTAs at short horizons: 8 / 4 / 1 lanes need fewer threads, so the
//  compiler may use more registers -- no spills; the host checks the thread count against these bounds)
#define NMPC_MAX_THREADS(SPT, CPB) ((SPT) >= 3 ? 256 : (SPT) == 1 ? ((CPB) == 8 ? 256 : (CPB) == 4 ? 160 : (CPB) == 1 ? 128 : 384) : 384)
template <int SPT, int CPB, bool WARM, bool RATE, int NC = 4>
__global__ void __launch_bounds__(NMPC_MAX_THREADS(SPT, CPB), 1) nmpc_solve_kernel(const SolveArgs a)
{
    extern __shared__ double smem_raw[];
    const Params &prm = a.prm;
    const int N = prm.N, PB = (CPB > 0) ? CPB : a.PB, batch = a.batch;
    const int NG = (N + SPT - 1) / SPT;
    SmemT<CPB, RATE ? NSLOTS_RATE : NSLOTS> sm;
    sm.PB = PB;
    sm.carve(smem_raw, N, NG);

    const int tid = threadIdx.x;

    if (tid < NMPC_CTRL_THREADS) {
        control_loop<CPB, WARM, RATE, NC, false>(a, sm, N, PB, NG, batch, tid, 0, 0);
    } else {
        // ------------------------------------------------------------ stage threads
        const int t = tid - NMPC_CTRL_THREADS;
        const int p = t % PB;
        const int g = t / PB;
        const int k0 = g * SPT;
        const bool mine = k0 < N;
        StageRegs r[SPT];
        double cf[NC];                         // path polynomial of the lane's problem
#pragma unroll
        for (int i = 0; i < NC; i++) cf[i] = 0.0;
        int trace_cyc = -1; (void)trace_cyc;
        for (;;) {
            trace_cyc++;
            TRACE_S(0);
            if (!__syncthreads_or(0)) break;   // B2 (vote)
            TRACE_S(1);
            // ---- P3a: start the lane's next problem, or the right-hand side of a second-order correction (the accepted
            //      step was applied and a finished problem flushed before the vote, while the control thread fetched the
            //      next problems)
            if (mine) stages_init<SPT, WARM, RATE, NC>(prm, sm, r, cf, k0, p, a, N, batch);
            TRACE_S(2);
            __syncthreads();  // B3
            TRACE_S(3);
            // ---- P3b: Newton-system coefficients
            if (mine) stages_coeffs<SPT, RATE, NC>(prm, sm, r, cf, k0, p, N);
            TRACE_S(4);
            __syncthreads();  // B4
            // ---- P4: control
            __syncthreads();  // B5
            TRACE_S(5);
            // ---- P5: step-dependent work
            StepPart sp;
            part_reset(sp);
            const int step_kind = mine ? stages_step<SPT, RATE, NC>(prm, sm, r, cf, k0, p, N, sp) : -1;
            if (step_kind >= 0) part_store(sm, g, p, sp);
            TRACE_S(6);
            __syncthreads();  // B6
            // ---- P6: the control thread sets the step sizes; a stage thread of lane p runs its adjoint sweep
            // (lanes 0..15 on the thread of group 0, lanes 16..31 on that of group 1: a 64-bit shared-memory access of
            //  16 lanes is one wavefront, and the two half-warps sit on different sub-partitions)
            if (g == ((NG >= 2) ? (p >> 4) : 0) && step_kind >= 0) stage_adjoint(prm, sm, p, step_kind);
            __syncthreads();  // B7
            TRACE_S(7);
            // ---- P1: evaluate
            if (mine) {
                EvalPart ep;
                part_reset(ep);
                if (stages_eval<SPT, RATE, NC>(prm, sm, r, cf, k0, p, N, ep)) part_store(sm, g, p, ep);
            }
            TRACE_S(8);
            __syncthreads();  // B1
            TRACE_S(9);
            // ---- P2: control
            __syncthreads();  // B1b
            // ---- P3a0: apply the accepted step, flush a finished problem -- while the control thread refills the
            //      lanes (neither touches what the other reads: the step to apply was copied to PS_AP_* in P2)
            if (mine) stages_apply<SPT, RATE>(prm, sm, r, k0, p, a, N, batch);
        }
    }
}

}  // namespace nmpc
