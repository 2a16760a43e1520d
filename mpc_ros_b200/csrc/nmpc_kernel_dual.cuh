// nmpc_kernel_dual.cuh -- the solve kernel for full CTAs (32 lanes, or 28 in the rate-penalty variant; horizons up to 20
// stages): two lane groups run OUT OF PHASE on one set of stage threads.
//
// Why.  A global cycle of nmpc_solve_kernel alternates between the control warps (Riccati sweeps, decisions: ~20 k SM
// cycles during which the ten stage warps wait) and the stage warps (~16 k cycles during which the control warps wait),
// and neither side can be shortened by adding lanes: the SM's shared memory and register file hold 32 problems, and the
// phases are bound by the latency of one thread's chain, not by throughput (two 16-lane CTAs per SM take exactly as long
// per cycle as one 32-lane CTA).  Here the 32 lanes are split into group A (lanes 0..15, control warp 0) and group B
// (lanes 16..31, control warp 1).  A stage thread owns ONE stage of lane p of group A and the same stage of lane p of
// group B (instead of two consecutive stages of one lane): its chain per phase is half as long, and while it works for
// one group the other group's control warp runs its sweeps.  Same shared-memory footprint, same registers per thread
// (the stage registers of both groups; the idle group's set is parked by a register swap), same phase functions
// (nmpc_phases.cuh), same arithmetic: the pairs of stages whose partial sums the single-group kernel adds inside a
// thread sit in the two halves of a warp here and are combined by one shuffle in the same order, so results are
// bit-identical.
//
// Synchronisation.  Group g's control warp and the stage warps meet on named barrier 1 + g (bar.sync id, count) in the
// phase order of nmpc_kernel.cuh.  The stage warps serve the groups in a fixed rotation
//     X(A)  Y(B)  X(B)  Y(A)  ...      X = apply / flush, vote, init, coefficients      Y = step work, adjoint, evaluate
// so that X(A) is followed by A's sweeps (control warp 0) while the stage warps evaluate B, and so on.  A control warp
// only ever waits on its own group's barrier and the stage warps execute both groups' barriers in one fixed order, so
// the wait-for graph has no cycle.
#pragma once
#include "nmpc_kernel.cuh"

namespace nmpc {

#define NMPC_DUAL_MAX_N 20

// combine the partial sums of the two stages a warp holds for one lane (threads l and l + 16), lower stage first
__device__ __forceinline__ double shx16(double v) { return __shfl_xor_sync(0xffffffffu, v, 16); }
__device__ __forceinline__ void part_pair(EvalPart &a)
{
    const double prinf = shx16(a.prinf), pr1 = shx16(a.pr1), duinf = shx16(a.duinf), vmax = shx16(a.vmax), vmin = shx16(a.vmin);
    const double l1 = shx16(a.l1), z1 = shx16(a.z1), f = shx16(a.f), lnsum = shx16(a.lnsum);
    const int inside = __shfl_xor_sync(0xffffffffu, a.inside, 16);
    a.prinf = fmax2(a.prinf, prinf); a.pr1 += pr1; a.duinf = fmax2(a.duinf, duinf);
    a.vmax = fmax2(a.vmax, vmax); a.vmin = fmin2(a.vmin, vmin); a.l1 += l1; a.z1 += z1; a.f += f; a.lnsum += lnsum;
    a.inside &= inside;
}
__device__ __forceinline__ void part_pair(StepPart &a)
{
    const double rmax = shx16(a.rmax), rzmax = shx16(a.rzmax), gd = shx16(a.gd);
    a.rmax = fmax2(a.rmax, rmax); a.rzmax = fmax2(a.rzmax, rzmax); a.gd += gd;
}

// RATE: the rate-penalty variant (44 slots per stage: 28 lanes = group A with 16 lanes, group B with 12).
template <bool WARM, int NC = 4, bool RATE = false>
__global__ void __launch_bounds__(384, 1) nmpc_solve_kernel_dual(const SolveArgs a)
{
    extern __shared__ double smem_raw[];
    const Params &prm = a.prm;
    const int N = prm.N, batch = a.batch;
    constexpr int PB = RATE ? 28 : 32;
    const int NG = (N + 1) / 2;            // partial sums per pair of stages, as in the single-group kernel (SPT = 2)
    SmemT<PB, RATE ? NSLOTS_RATE : NSLOTS> sm;
    sm.PB = PB;
    sm.carve(smem_raw, N, NG);
    const int tid = threadIdx.x;
    const int bar_count = blockDim.x - 32;         // one control warp + the stage warps

    if (tid < NMPC_CTRL_THREADS) {
        control_loop<PB, WARM, RATE, NC, true>(a, sm, N, PB, NG, batch, tid, 1 + (tid >> 5), bar_count);
        return;
    }

    // ------------------------------------------------------------ stage threads
    const int t = tid - NMPC_CTRL_THREADS;
    const int k = t >> 4;                  // the thread's stage (both groups)
    const int p16 = t & 15;
    const bool mine_k = k < N;
    const bool lower = (tid & 16) == 0;    // holds the even stage of the warp's pair
    const int g = k >> 1;
    StageRegs r, ro;                       // current / other group
    double cf[NC], cfo[NC];
#pragma unroll
    for (int i = 0; i < NC; i++) { cf[i] = 0.0; cfo[i] = 0.0; }
    // (never read before stage_init; zeroed so that the swap moves defined values)
    r.uw = r.ua = r.zlw = r.zuw = r.zla = r.zua = r.sn = r.cs = r.se = r.ce = r.tsn = r.tcs = r.tse = r.tce = 0.0;
    ro = r;
    int G = 0;                             // current group
    int alive = 3, started = 0;            // bit g: group g still has work / has been through X once
#pragma unroll 1
    for (;;) {
        // rotation  X(A) Y(B) X(B) Y(A): while a group's control warp sweeps, the stage warps work for the other group.
        // (Measured: 27.7 M solves/s saturated against 27.3 for the single-group kernel and 26.2 for the rotation
        //  X(A) X(B) Y(A) Y(B); a one-shot batch of 8,192 takes 2.54 ms against 2.89.  The stage blocks do take half as long,
        //  but a sweep that shares its sub-partition with two busy stage warps runs ~45 % slower -- 17.7 k cycles instead of
        //  12.1 k -- which eats most of the gain: profiles/r2_dual_groups.txt.)
        // ================================================= X(G)
        if (alive & (1 << G)) {
            const int p = p16 + 16 * G, bid = 1 + G;
            const bool mine = mine_k && p < PB;
            if (started & (1 << G)) {
                named_sync(bid, bar_count);   // B1b
                // ---- P3a0: apply the accepted step, flush a finished problem (the control warp refills meanwhile)
                if (mine) stages_apply<1, RATE>(prm, sm, &r, k, p, a, N, batch);
            }
            asm volatile("" ::: "memory");
            if (!named_vote(0, bid, bar_count)) {      // B2 (vote): the group has run out of work
                alive &= ~(1 << G);
            } else {
                started |= 1 << G;
                // ---- P3a: start the lane's next problem / right-hand side of a second-order correction
                if (mine) stages_init<1, WARM, RATE, NC>(prm, sm, &r, cf, k, p, a, N, batch);
                named_sync(bid, bar_count);   // B3
                // ---- P3b: Newton-system coefficients
                if (mine) stages_coeffs<1, RATE, NC>(prm, sm, &r, cf, k, p, N);
                named_sync(bid, bar_count);   // B4: the group's control warp starts its sweeps
            }
        }
        if (!alive) break;
        // ================================================= the other group
        {
            const StageRegs tr = r; r = ro; ro = tr;
#pragma unroll
            for (int i = 0; i < NC; i++) { const double tc = cf[i]; cf[i] = cfo[i]; cfo[i] = tc; }
            G ^= 1;
        }
        // ================================================= Y(G)
        if ((alive & started) & (1 << G)) {
            const int p = p16 + 16 * G, bid = 1 + G;
            const bool mine = mine_k && p < PB;
            named_sync(bid, bar_count);       // B5: the sweeps are done
            // ---- P5: step-dependent work
            StepPart sp;
            part_reset(sp);
            const int step_kind = mine ? stages_step<1, RATE, NC>(prm, sm, &r, cf, k, p, N, sp) : -1;
            part_pair(sp);
            if (step_kind >= 0 && lower) part_store(sm, g, p, sp);
            named_sync(bid, bar_count);       // B6
            // ---- P6: the control thread sets the step sizes; the lane's stage-0 thread runs the adjoint sweep
            if (k == 0 && step_kind >= 0) stage_adjoint(prm, sm, p, step_kind);
            named_sync(bid, bar_count);       // B7
            // ---- P1: evaluate
            EvalPart ep;
            part_reset(ep);
            const bool ev = mine && stages_eval<1, RATE, NC>(prm, sm, &r, cf, k, p, N, ep);
            part_pair(ep);
            if (ev && lower) part_store(sm, g, p, ep);
            named_sync(bid, bar_count);       // B1: the control warp decides
        }
    }
}

}  // namespace nmpc
