// oracle/ref_bench.cpp -- TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE.
//
// CPU baseline of bench.py (SURVEY 8d "CPU baseline timed beside it"): the reference's UNMODIFIED MPC class
// (mpc_ros/src/mpc_planner.cpp + vendored CppAD, compiled from /root/reference, see oracle/Makefile) driven by an
// std::thread-per-core loop, one MPC object per thread, after CppAD::thread_alloc::parallel_setup +
// CppAD::parallel_ad<double>() (cppad/core/parallel_ad.hpp:26-45; MPC::Solve is not thread-safe without them: CppAD
// keeps one tape per AD<Base> and thread).  The NLP solver behind CppAD::ipopt::solve is oracle/ipm.c, NOT Ipopt 3.12.8.
//
//   ref_bench <threads (0 = hardware_concurrency)> <problems per thread> <seed> [offset]
// Problems: the config-2 generator (bench/problem_gen.cpp) followed by the reference pre-step as restated in
// oracle/mpc_oracle.c (driving_state.cpp restated).  Prints one JSON object.
#include "mpc_planner.h"
#include "mpc_oracle.h"
#include "shim/ip_standin.h"
#include <cppad/cppad.hpp>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

extern "C" {
int mpcgen_num_waypoints(double path_length);
void mpcgen_problems(uint64_t seed, int batch, double path_length, double *wx, double *wy, double *pose, double *vel,
                     int *kind_out);
}

namespace {
thread_local size_t t_thread_num = 0;
std::atomic<bool> g_parallel(false);
bool in_parallel() { return g_parallel.load(); }
size_t thread_num() { return t_thread_num; }
double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Out { long conv; long iters; double busy; };

void worker(MPC *mpc_ptr, size_t tn, int per, int B, int M, const double *wx, const double *wy, const double *pose, const double *vel, Out *out)
{
    t_thread_num = tn;
    MPC &mpc = *mpc_ptr;           // one MPC object per thread, built by main (MPC::MPC writes to std::cout)
    std::vector<double> x(M), y(M);
    const double t0 = now_s();
    long conv = 0, iters = 0;
    for (int j = 0; j < per; j++) {
        const size_t i = (tn - 1) * (size_t)per + j;     // thread numbers start at 1 (0 is main)
        for (int q = 0; q < M; q++) { x[q] = wx[(size_t)q * B + i]; y[q] = wy[(size_t)q * B + i]; }
        double c4[4], cte, eth;
        mpc_oracle_prestep(x.data(), y.data(), M, pose[i], pose[(size_t)B + i], pose[2 * (size_t)B + i], c4, &cte, &eth);
        Eigen::VectorXd st(6), co(4);
        st[0] = 0; st[1] = 0; st[2] = 0; st[3] = vel[i]; st[4] = cte; st[5] = eth;       // delay_mode off (configs 2-4)
        for (int q = 0; q < 4; q++) co[q] = c4[q];
        mpc.Solve(st, co);
        conv += standin_last().status == 1;
        iters += standin_last().iters;
    }
    out->conv = conv; out->iters = iters; out->busy = now_s() - t0;
}
}  // namespace

int main(int argc, char **argv)
{
    int T = argc > 1 ? atoi(argv[1]) : 0;
    const int per = argc > 2 ? atoi(argv[2]) : 64;
    const uint64_t seed = argc > 3 ? strtoull(argv[3], nullptr, 10) : 20261020ULL;
    if (T <= 0) T = (int)std::thread::hardware_concurrency();
    if (T <= 0) T = 1;
    if (T > 47) T = 47;          // CPPAD_MAX_NUM_THREADS 48 (cppad/configure.hpp:176), thread 0 is main
    const int B = T * per;
    const int M = mpcgen_num_waypoints(5.0);
    std::vector<double> wx((size_t)M * B), wy((size_t)M * B), pose(3 * (size_t)B), vel(3 * (size_t)B);
    mpcgen_problems(seed, B, 5.0, wx.data(), wy.data(), pose.data(), vel.data(), nullptr);

    // P8 of the survey: one tape per thread needs this before any thread records
    CppAD::thread_alloc::parallel_setup((size_t)T + 1, in_parallel, thread_num);
    CppAD::thread_alloc::hold_memory(true);
    CppAD::parallel_ad<double>();

    std::vector<Out> outs(T);
    std::vector<std::thread> ths;
    // one MPC per thread, constructed here: MPC::MPC prints "init mpc" (mpc_planner.cpp:225), kept off the JSON output
    std::vector<MPC *> mpcs;
    {
        std::streambuf *old = std::cout.rdbuf();
        std::ostringstream sink;
        std::cout.rdbuf(sink.rdbuf());
        std::map<std::string, double> p;   // mpc_params.yaml:9-25 through the LoadParams keys
        p["DT"] = 0.1; p["STEPS"] = 20; p["REF_CTE"] = 0; p["REF_ETHETA"] = 0; p["REF_V"] = 0.5; p["W_CTE"] = 100;
        p["W_EPSI"] = 0; p["W_V"] = 1000; p["W_ANGVEL"] = 100; p["W_A"] = 50; p["W_DANGVEL"] = 0; p["W_DA"] = 0;
        p["ANGVEL"] = 1.5; p["MAXTHR"] = 1.0; p["BOUND"] = 1e3;
        for (int t = 0; t < T; t++) { mpcs.push_back(new MPC()); mpcs.back()->LoadParams(p); }
        std::cout.rdbuf(old);
    }
    g_parallel.store(true);
    const double t0 = now_s();
    for (int t = 0; t < T; t++)
        ths.emplace_back(worker, mpcs[t], (size_t)t + 1, per, B, M, wx.data(), wy.data(), pose.data(), vel.data(), &outs[t]);
    for (auto &th : ths) th.join();
    const double wall = now_s() - t0;
    g_parallel.store(false);
    long conv = 0, iters = 0; double busy = 0;
    for (int t = 0; t < T; t++) { conv += outs[t].conv; iters += outs[t].iters; if (outs[t].busy > busy) busy = outs[t].busy; }
    printf("{\"threads\": %d, \"per_thread\": %d, \"problems\": %d, \"seed\": %llu, \"converged\": %ld, \"mean_iters\": %.3f, "
           "\"wall_s\": %.6f, \"busy_s\": %.6f, \"solves_per_s\": %.3f, \"threading\": \"std::thread per core, "
           "CppAD::thread_alloc::parallel_setup + parallel_ad<double>\"}\n",
           T, per, B, (unsigned long long)seed, conv, (double)iters / B, wall, busy, conv / wall);
    return 0;
}
