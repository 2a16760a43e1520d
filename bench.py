#!/usr/bin/env python
"""bench.py -- converged NMPC solves/sec (N = 20) of the hot path on N B200 GPUs of one node.

    python bench.py --gpus 1 --steps K --warmup W           # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W   # the reference's CPU MPC::Solve

A "step" is one pass of the hot path over 256 independent batches of BASELINE config 2 (4,096 N = 20
problems each: random poses along the infinity / epitrochoid / square tracks, mpc_params.yaml
weights), streamed: per batch the reference pre-step (waypoint transform + cubic polyfit + state
assembly, driving_state.cpp:196-256) followed by the batched MPC::Solve, i.e.
mpc_b200_prestep_batch + mpc_b200_solve_batch.  K steps are timed back to back (steady state; a
step is ~1 M solves, so the figure does not depend on K).  For N > 1 every rank streams its own
batches (weak scaling, no collective on the solve path); the timed region is bracketed by a
barrier + synchronize and the slowest rank's device time is used.

`value`   : inputs already resident in HBM, device-pointer C-ABI calls on 64 streams.
`e2e`     : the same K steps as control ticks through the C ABI with HOST buffers (one packed
            page-locked buffer per batch: one H2D + one D2H copy inside the timed region).
`latency` : config 1, p50 / p99 of one MPC::Solve through the C++ adapter (mpc_bench latency).
`config3` : BASELINE config 3, ONE batch of 65,536 problems split contiguously over the N GPUs,
            first submit to last host gather, through the C++ harness (mpc_bench multi).
`roofline`: FP64 pipe.  achieved = algorithmic flops of the solve kernel (SURVEY section 8d:
            27,879 flop per interior-point iteration at N = 20, times the iterations actually
            taken) / its CUDA-event duration on the launching stream; peak = DFMA-chain peak
            measured live (MEASURED_PEAKS.json has no FP64 entry).
`cpu_baseline`: oracle/_ref/ref_bench (the reference's unmodified mpc_planner.cpp + CppAD, std::thread
            per core; solver inside is the repo's Ipopt stand-in, Ipopt itself is not installed) on all
            host cores, bounded sample; `--impl reference` times the same thing.

`--dump-outputs DIR` writes what the `value` leg computed in its last timed step (rank 0) as float64
DIR/<name>.npy, one column per problem: the pre-step's coeffs (4) and state (6), the solve's u0 (2),
pred (3N), obj, status, iters and kkt, and problem = the column's index in the rank's generated input
sets.  Above DUMP_MAX_PROBLEMS problems a fixed, seeded sample of them is written.  The inputs depend
only on --batch and --sets, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# batches in flight on different streams must not alias onto the default 8 hardware queues
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np  # noqa: E402

METRIC = "converged_nmpc_solves_per_sec_N20"
UNIT = "solves/s"
BATCH = 4096                 # BASELINE config 2
SEED = 20261018 + 2          # SURVEY 8d: seed = 20261018 + config#
FLOP_PER_ITER_N20 = 27879.0  # SURVEY 8d algorithmic flops per interior-point iteration, N = 20
# dram__bytes_read.sum + dram__bytes_write.sum of ONE solve-kernel launch (4,096 problems) from the latest ncu --set full
# capture, profiles/r*_solve_kernel_ncu_raw.csv (read at start; the constant is the round-1 capture: 446,720 + 0 B).
# Algorithmic: 88 B in + ~520 B out per problem = 2.5 MB per launch; the 2.1 MB of results are still in the 126 MB
# L2 when the kernel ends, so DRAM sees less than the algorithmic bytes -- nothing is re-read.
NCU_DRAM_BYTES_PER_LAUNCH = 446720
DUMP_MAX_PROBLEMS = 65536    # 77 float64 values per problem: 40 MB


def _ncu_dram_bytes():
    import csv
    import glob
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        f = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r*_solve_kernel_ncu_raw.csv")))[-1]
        rr = list(csv.reader(open(f)))
        h, u, v = rr[0], rr[1], rr[2]
        tot = 0.0
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(v[h.index(k)].replace(",", "")) * unit[u[h.index(k)]]
        return int(round(tot))
    except Exception:
        return NCU_DRAM_BYTES_PER_LAUNCH


WORKLOAD = ("config2 streamed: batches of 4096 independent N=20 diff-drive NMPC problems, random poses on "
            "infinity/epitrochoid/square tracks, mpc_params.yaml weights, cold start; per batch prestep "
            "(transform+polyfit+state) + solve; a step = batches_per_step such batches per GPU")


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=50):
        self.index = index; self.rows = []; self.proc = None; self.thr = None; self.period_ms = int(period_ms)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def rd():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.thr = threading.Thread(target=rd, daemon=True); self.thr.start()

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = []; smax = None; reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons),
                    samples=len(sm))


# ------------------------------------------------------------------ reference arm (CPU)
REF_BENCH = os.path.join(ROOT, "oracle", "_ref", "ref_bench")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libmpc_ref.so")
_REF_LOADED = []


def _load_ref_in_parent():
    """The baseline binary (oracle/_ref/ref_bench) is a separate process; the same reference objects are also loaded
    into THIS process (oracle/_ref/libmpc_ref.so) and called once, so that what runs is visible from here."""
    if _REF_LOADED or not os.path.exists(REF_LIB):
        return
    from oracle.oracle_py import Reference, YAML_DEFAULT
    r = Reference(YAML_DEFAULT)
    r.solve(np.array([0.0, 0.0, 0.0, 0.3, 0.05, -0.1]), np.array([0.05, -0.1, 0.02, 0.003]))
    _REF_LOADED.append(r)


def _port_worker(args):
    seed, count, offset = args
    from oracle.oracle_py import Oracle, YAML_DEFAULT
    from bench import gen_py
    g = gen_py.problems(seed, offset + count)
    orc = Oracle()
    conv = 0; iters = 0
    t0 = time.perf_counter()
    for i in range(offset, offset + count):
        c, cte, eth = orc.prestep(g["wx"][:, i], g["wy"][:, i], *g["pose"][:, i])
        r = orc.solve(YAML_DEFAULT, np.array([0.0, 0.0, 0.0, g["vel"][0, i], cte, eth]), c)
        conv += int(r["status"] == 1); iters += r["iters"]
    return conv, iters, time.perf_counter() - t0


def cpu_reference_rate(per_core, cores=None):
    """The reference's MPC::Solve on the host cores.  kind "reference": oracle/_ref/ref_bench -- the reference's
    unmodified mpc_planner.cpp + CppAD, std::thread per core (CppAD::thread_alloc::parallel_setup), C++ harness
    oracle/ref_bench.cpp.  kind "port" (only where oracle/_ref was never built): the C restatement, fork per core."""
    cores = cores or os.cpu_count() or 1
    if os.path.exists(REF_BENCH):
        _load_ref_in_parent()
        T = min(cores, 47)      # CPPAD_MAX_NUM_THREADS
        r = subprocess.run([REF_BENCH, str(T), str(per_core), str(SEED)], capture_output=True, text=True, timeout=1200)
        if r.returncode != 0:
            raise RuntimeError("ref_bench failed: " + r.stderr[-2000:])
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        return dict(value=d["solves_per_s"], unit=UNIT, cores=d["threads"], kind="reference",
                    sample="%d problems (%d per thread x %d std::threads) of the config-2 generator, seed %d; %d converged; "
                           "mean %.1f iterations; reference mpc_planner.cpp + CppAD unmodified (oracle/_ref/ref_bench), solver "
                           "inside: oracle/ipm.c stand-in for Ipopt 3.12.8" % (d["problems"], d["per_thread"], d["threads"], SEED,
                                                                          d["converged"], d["mean_iters"]),
                    wall_s=d["wall_s"])
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    jobs = [(SEED, per_core, k * per_core) for k in range(cores)]
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_port_worker, jobs)
    wall = time.perf_counter() - t0
    conv = sum(r[0] for r in res); iters = sum(r[1] for r in res)
    return dict(value=conv / wall, unit=UNIT, cores=cores, kind="port",
                sample="%d problems (%d per core x %d processes) of the config-2 generator, seed %d; %d converged; mean %.1f "
                       "iterations; oracle/mpc_oracle.c + oracle/ipm.c" % (per_core * cores, per_core, cores, SEED, conv,
                                                                          iters / max(1, per_core * cores)),
                wall_s=wall)


def bench_config(a, world):
    """The `config` object both arms print (the reference arm runs the same workload definition)."""
    return dict(workload=WORKLOAD, batch_per_gpu=a.batch, batches_per_step=a.batches_per_step, mpc_steps=20,
                max_iter=a.max_iter, n_gpus=world)


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    per_core = a.ref_per_core          # the same bounded sample as the cpu_baseline leg of the CUDA arm
    for _ in range(min(a.warmup, 2)):
        cpu_reference_rate(max(8, per_core // 8))
    vals = []; last = None
    t0 = time.perf_counter()
    for _ in range(a.steps):
        last = cpu_reference_rate(per_core)
        vals.append(last["value"])
    ms = (time.perf_counter() - t0) * 1e3 / max(1, a.steps)
    v = float(np.mean(vals))
    last["value"] = v
    last["sample"] = "each step: " + last["sample"]
    print(json.dumps(dict(impl="reference", metric=METRIC, value=v, unit=UNIT, n_gpus=a.gpus, steps=a.steps,
                          warmup=a.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None,
                          dtype="f64", data="synthetic", config=bench_config(a, world),
                          cpu_baseline=last,
                          e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))


# ------------------------------------------------------------------ our arm (CUDA)
def _ncu_executed_flops():
    """FP64 flops one solve-kernel launch really executes (2 x DFMA + DMUL + DADD thread instructions) from the latest
    ncu --set full capture under profiles/, or None."""
    import csv
    import glob
    try:
        f = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_solve_kernel_ncu_raw.csv")))[-1]
        rr = list(csv.reader(open(f)))
        h, v = rr[0], rr[2]
        def g(k):
            return float(v[h.index(k)].replace(",", ""))
        cyc = g("smsp__cycles_elapsed.max") if "smsp__cycles_elapsed.max" in h else g("sm__cycles_elapsed.max")
        fl = 0.0
        for k, w in (("dfma", 2.0), ("dmul", 1.0), ("dadd", 1.0)):
            fl += w * g("smsp__sass_thread_inst_executed_op_%s_pred_on.sum.per_cycle_elapsed" % k) * cyc
        return fl, os.path.basename(f)
    except Exception:
        return None, None


def _pin_to_gpu_numa_node(torch, local):
    """Several ranks share one host: keep this rank's threads (and, by first touch, its page-locked buffers) on the NUMA
    node its GPU hangs off, so that the H2D / D2H traffic of the e2e leg does not cross sockets.  Returns what was done."""
    try:
        bdf = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        if bdf is None:
            import subprocess as sp
            bdf = sp.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
        if isinstance(bdf, int):
            return None
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]                      # nvidia-smi prints an 8-digit PCI domain, sysfs a 4-digit one
        base = "/sys/bus/pci/devices/" + bdf
        node = int(open(base + "/numa_node").read())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if node < 0 or not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return dict(numa_node=node, cpus=len(cpus))
    except Exception:
        return None


def dump_outputs(out_dir, sets, B, bufs):
    """Writes the result buffers of input sets `sets` (name -> per-set device tensors of shape (rows, B) or (B,)) as
    out_dir/<name>.npy, float64, the sets' problems side by side on the last axis, plus problem.npy."""
    cols = {"problem": np.concatenate([q * B + np.arange(B) for q in sets]).astype(np.float64)}
    for name, per_set in bufs.items():
        cols[name] = np.concatenate([per_set[q].cpu().numpy() for q in sets], axis=-1).astype(np.float64)
    n = cols["problem"].size
    if n > DUMP_MAX_PROBLEMS:
        keep = np.sort(np.random.default_rng(SEED).choice(n, DUMP_MAX_PROBLEMS, replace=False))
        cols = {k: v[..., keep] for k, v in cols.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, v in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v))


def run_ours(a):
    import torch
    import torch.distributed as dist
    from mpc_ros_b200 import capi
    from bench import gen_py

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if capi.lib().mpc_b200_device_count() < 1:
        raise RuntimeError("bench.py: no CUDA device; the solver has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = _pin_to_gpu_numa_node(torch, local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = a.batch; N = 20; NB = a.batches_per_step
    prm = capi.yaml_default_params()
    prm.delay_mode = 0                       # configs 2-4 use the plain state (SURVEY 8d)
    prm.max_iter = a.max_iter
    solver = capi.Solver(prm, B, local)
    L = capi.lib()

    # ---- synthetic inputs: R distinct batches, more than L2 in total with their outputs
    R = a.sets
    M = gen_py._lib().mpcgen_num_waypoints(5.0)
    g = gen_py.problems(SEED + 1000 * rank, B * R)
    def split(x):   # (C, B*R) -> R contiguous (C, B) device tensors
        return [torch.from_numpy(np.ascontiguousarray(x[:, j * B:(j + 1) * B])).to(dev) for j in range(R)]
    d_wx = split(g["wx"]); d_wy = split(g["wy"]); d_pose = split(g["pose"]); d_vel = split(g["vel"])
    f64 = dict(dtype=torch.float64, device=dev); i32 = dict(dtype=torch.int32, device=dev)
    d_coef = [torch.zeros((4, B), **f64) for _ in range(R)]; d_state = [torch.zeros((6, B), **f64) for _ in range(R)]
    d_u0 = [torch.zeros((2, B), **f64) for _ in range(R)]; d_pred = [torch.zeros((3 * N, B), **f64) for _ in range(R)]
    d_obj = [torch.zeros(B, **f64) for _ in range(R)]; d_kkt = [torch.zeros(B, **f64) for _ in range(R)]
    d_stat = [torch.zeros(B, **i32) for _ in range(R)]; d_it = [torch.zeros(B, **i32) for _ in range(R)]
    in_bytes = (2 * M + 6) * B * 8
    out_bytes = (2 + 3 * N + 2) * B * 8 + 2 * B * 4
    set_bytes = in_bytes + out_bytes + 10 * B * 8
    flush = torch.empty(256 * 1024 * 1024 // 8, **f64)
    # A step = NB independent batches, issued round-robin on S streams so that the tail of one batch (a few problems
    # need 10-25x the median iteration count) overlaps the next batches.  Every stream keeps at most DEPTH batches
    # in flight (the host waits on the batch DEPTH back), which bounds the launches a handle has in flight.
    S = max(1, min(a.streams, NB))
    DEPTH = max(1, a.depth)
    raw_streams = [capi.stream_create(local) for _ in range(S)]      # torch hands out only 32 distinct streams
    streams = [torch.cuda.ExternalStream(p, device=dev) for p in raw_streams]
    max_ctas = a.max_ctas if a.max_ctas > 0 else max(4, min(128, -(-512 // S)))
    solver.set_option("max_ctas", max_ctas)
    pre_f = L.mpc_b200_prestep_batch; sol_f = L.mpc_b200_solve_batch
    pre_args = [(B, M, d_wx[j].data_ptr(), d_wy[j].data_ptr(), d_pose[j].data_ptr(), d_vel[j].data_ptr(),
                 d_coef[j].data_ptr(), d_state[j].data_ptr()) for j in range(R)]
    sol_args = [(B, d_state[j].data_ptr(), d_coef[j].data_ptr(), None, None, d_u0[j].data_ptr(),
                 d_pred[j].data_ptr(), d_obj[j].data_ptr(), d_stat[j].data_ptr(), d_it[j].data_ptr(),
                 d_kkt[j].data_ptr(), None) for j in range(R)]
    hh = solver._h
    done_ev = [[torch.cuda.Event() for _ in range(DEPTH)] for _ in range(S)]
    issued = [0] * S
    launch_ev = []            # (start, end) CUDA events around sampled solve launches, on their own streams

    def batch_dev(j, sample=False):
        s_ = j % S
        sp = raw_streams[s_]; st = streams[s_]
        k = issued[s_]
        if k >= DEPTH:
            done_ev[s_][k % DEPTH].synchronize()
        q = j % R
        rc = pre_f(hh, *pre_args[q], sp)
        if sample:
            x = torch.cuda.Event(enable_timing=True); y = torch.cuda.Event(enable_timing=True)
            x.record(st)
        rc |= sol_f(hh, *sol_args[q], sp)
        if sample:
            y.record(st); launch_ev.append((x, y))
        done_ev[s_][k % DEPTH].record(st)
        issued[s_] = k + 1
        if rc != 0:
            raise RuntimeError("C ABI call failed: %d %s" % (rc, L.mpc_b200_last_cuda_error(hh).decode()))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The issue loop in C++ (bench/issue_loop.cpp: the same two C-ABI calls per batch, the same depth control): a Python
    # loop costs about as much per batch as the device needs for it.  --python-issue keeps the Python loop.
    import ctypes as C
    IL = None; ictx = None
    iss_path = os.path.join(ROOT, "bench", "libmpc_issue.so")
    if not a.python_issue and os.path.exists(iss_path):      # (not built: the Python loop issues the same calls)
        IL = C.CDLL(iss_path)
        IL.mpcb_issue_create.restype = C.c_void_p; IL.mpcb_issue_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        IL.mpcb_issue_run.restype = C.c_int
        IL.mpcb_issue_run.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
        IL.mpcb_issue_samples.restype = C.c_int; IL.mpcb_issue_samples.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        IL.mpcb_issue_destroy.argtypes = [C.c_void_p]
        ictx = IL.mpcb_issue_create(local, S, DEPTH, 4096)
        if not ictx:
            raise RuntimeError("mpcb_issue_create failed")
        stream_arr = (C.c_void_p * S)(*raw_streams)
        ptr_arr = (C.c_size_t * (12 * R))()
        for q in range(R):
            for i_, t_ in enumerate((d_wx[q], d_wy[q], d_pose[q], d_vel[q], d_coef[q], d_state[q], d_u0[q], d_pred[q], d_obj[q],
                                     d_stat[q], d_it[q], d_kkt[q])):
                ptr_arr[12 * q + i_] = t_.data_ptr()

    def issue(j0, n, sample_every=0):
        if IL is None:
            for j in range(j0, j0 + n):
                batch_dev(j, sample=(sample_every > 0 and (j - j0) % sample_every == 0))
            return
        rc = IL.mpcb_issue_run(ictx, hh, j0, n, stream_arr, R, ptr_arr, B, M, sample_every)
        if rc != 0:
            raise RuntimeError("issue loop failed: %d %s" % (rc, L.mpc_b200_last_cuda_error(hh).decode()))

    fp64_peak = L.mpc_b200_measure_fp64_peak(local, 100000)   # also brings the clocks up
    jb = 0
    issue(jb, a.warmup * NB); jb += a.warmup * NB
    torch.cuda.synchronize()
    flush.fill_(1.0)                        # one L2 flush; the timed steps then rotate over > L2 of data
    barrier()
    sampler = ClockSampler(local, a.clock_period_ms)
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    n0 = solver.launch_count
    main = torch.cuda.current_stream()
    e0.record(main)
    for st in streams:
        st.wait_event(e0)
    j_first = jb
    issue(jb, a.steps * NB, sample_every=16); jb += a.steps * NB
    for st in streams:
        main.wait_stream(st)
    e1.record(main)
    barrier()
    launches = solver.launch_count - n0
    clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    n_batches = a.steps * NB
    if a.dump_outputs and rank == 0:
        # every batch of a step reads one input set and writes that set's result buffers (the same values each time), so
        # the buffers of the sets the last step used hold what it computed -- until the isolated launches below
        dump_outputs(a.dump_outputs, sorted({j % R for j in range(jb - NB, jb)}), B,
                     dict(coeffs=d_coef, state=d_state, u0=d_u0, pred=d_pred, obj=d_obj, status=d_stat, iters=d_it,
                          kkt=d_kkt))

    # converged problems and iterations actually taken in the timed steps (results are deterministic per set)
    conv_steps = 0; iter_steps = 0.0; per_set = {}
    for j in range(j_first, j_first + n_batches):
        s = j % R
        if s not in per_set:
            st = d_stat[s].cpu().numpy(); kk = d_kkt[s].cpu().numpy(); it = d_it[s].cpu().numpy()
            ok = (st == 1) & (kk <= 1e-8)
            per_set[s] = (int(ok.sum()), float(it.sum()), float(it[ok].mean()) if ok.any() else 0.0, int(it.max()))
        conv_steps += per_set[s][0]; iter_steps += per_set[s][1]
    from mpc_ros_b200.sharding import reduce_over_ranks
    ms_total, (conv_total, _iters_all) = reduce_over_ranks(ms_total, [conv_steps, iter_steps], device=dev)
    value = conv_total / (ms_total * 1e-3)

    # ---- roofline of the dominant kernel (the solve kernel), this rank.
    # Launches overlap on the device (S streams, a slice of the SMs each), so the duration that relates one launch's
    # flops to the machine's peak is the device time per launch of the timed region: region / launches (the pre-step
    # and queue-order kernels are < 1 % of it).  The CUDA-event duration of single launches on their own streams is
    # reported beside it (launch_ms_event_avg: it includes the time a launch shares the SMs with its neighbours;
    # concurrency = launch_ms_event_avg / kernel_ms launches are in flight on average).
    flops_per_launch = FLOP_PER_ITER_N20 * iter_steps / n_batches
    eff_ms = ms_total / n_batches
    achieved = flops_per_launch / (eff_ms * 1e-3) / 1e12
    ev_ms = [x.elapsed_time(y) for x, y in launch_ev]
    if IL is not None:
        buf = (C.c_float * 4096)()
        ev_ms = list(buf[:IL.mpcb_issue_samples(ictx, buf, 4096)])
    iso = []
    for j in range(5):
        x = torch.cuda.Event(enable_timing=True); y = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        st0 = streams[0]
        pre_f(hh, *pre_args[j % R], raw_streams[0]); x.record(st0); sol_f(hh, *sol_args[j % R], raw_streams[0]); y.record(st0)
        torch.cuda.synchronize()
        iso.append(x.elapsed_time(y))
    iso_ms = float(np.median(iso))
    exe, exe_src = _ncu_executed_flops()
    roofline = dict(bound="fp64", achieved=achieved, peak=fp64_peak, unit="TFLOP/s", frac=achieved / fp64_peak,
                    traffic=_ncu_dram_bytes() if B == BATCH else None, kernel="nmpc_solve_kernel", kernel_ms=eff_ms,
                    launch_ms_event_avg=float(np.mean(ev_ms)) if ev_ms else None,
                    concurrency=(float(np.mean(ev_ms)) / eff_ms) if ev_ms else None,
                    kernel_ms_isolated=iso_ms, achieved_isolated=flops_per_launch / (iso_ms * 1e-3) / 1e12,
                    streams=S, flops_per_launch=flops_per_launch,
                    flops="algorithmic: SURVEY 8d count, 27,879 flop per interior-point iteration at N = 20 x iterations taken",
                    executed_flops_per_launch_ncu=exe, executed_source=exe_src,
                    frac_executed=(exe / (eff_ms * 1e-3) / 1e12 / fp64_peak) if exe else None,
                    peak_source="DFMA-chain peak measured live by mpc_b200_measure_fp64_peak (datasheet: 148 SM x 64 FMA/clk "
                                "x 2 x 1.965 GHz = 37.2); MEASURED_PEAKS.json has no FP64 entry")

    # ---- e2e: the same K steps of NB batches through the C ABI with HOST buffers, copies inside the timed region.
    # T host threads, each keeping several ticks in flight on as many handles (a handle owns a stream and its device
    # scratch) through the ONE-buffer tick mpc_b200_track_packed_submit / _wait: one H2D and one D2H copy per tick.
    T = max(1, a.e2e_threads)
    K = max(1, a.e2e_inflight // T)
    sub_f = L.mpc_b200_track_packed_submit; wait_f = L.mpc_b200_track_wait

    class Slot:
        def __init__(self, q):
            self.solver = capi.Solver(prm, B, local)
            self.solver.set_option("max_ctas", a.e2e_max_ctas if a.e2e_max_ctas > 0 else max(8, min(128, -(-512 // (T * K)))))
            total, self.off = self.solver.packed_layout(B, M)
            self.ptr = L.mpc_b200_host_alloc(total)
            if not self.ptr:
                raise RuntimeError("mpc_b200_host_alloc failed")
            self.buf = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(total,))
            self.v = self.solver.packed_views(self.buf, B, M)
            self.v["wx"][:] = d_wx[q].cpu().numpy(); self.v["wy"][:] = d_wy[q].cpu().numpy()
            self.v["pose"][:] = d_pose[q].cpu().numpy(); self.v["vel"][:] = d_vel[q].cpu().numpy()
            self.h2d = self.off["u0"]; self.d2h = total - self.off["vel"]
            self.args = (self.solver._h, B, M, 0, self.ptr)
            self.busy = False

        def submit(self):
            if sub_f(*self.args) != 0:
                raise RuntimeError("mpc_b200_track_packed_submit failed")
            self.busy = True

        def wait(self):
            if not self.busy:
                return 0
            if wait_f(self.solver._h) != 0:
                raise RuntimeError("mpc_b200_track_wait failed")
            self.busy = False
            return int(((self.v["status"] == 1) & (self.v["kkt"] <= 1e-8)).sum())

        def close(self):
            self.solver.close()
            L.mpc_b200_host_free(self.ptr)

    import ctypes as C

    class Worker:
        def __init__(self, t):
            self.slots = [Slot((t * K + k) % R) for k in range(K)]
            self.conv = 0

        def run(self, n):
            self.conv = 0
            for j in range(n):
                s = self.slots[j % K]
                self.conv += s.wait()
                s.submit()
            for s in self.slots:
                self.conv += s.wait()

    workers = [Worker(t) for t in range(T)]
    e2e_ticks = a.steps * NB
    per_thread = max(2, e2e_ticks // T)
    for w in workers:
        w.run(K)
    barrier()
    t0 = time.perf_counter()
    ths = [threading.Thread(target=w.run, args=(per_thread,)) for w in workers]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    conv_h = sum(w.conv for w in workers)
    te = torch.tensor([t_e2e], dtype=torch.float64, device=dev); ce = torch.tensor([float(conv_h)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX); dist.all_reduce(ce, op=dist.ReduceOp.SUM)
    s0 = workers[0].slots[0]
    e2e = dict(value=float(ce.item()) / float(te.item()), unit=UNIT, h2d_bytes_per_step=s0.h2d * NB, d2h_bytes_per_step=s0.d2h * NB,
               h2d_bytes_per_batch=s0.h2d, d2h_bytes_per_batch=s0.d2h,
               steps=a.steps, batches=per_thread * T, threads=T, in_flight=T * K, seconds=float(te.item()),
               note="the same %d steps x %d batches as control ticks (pre-step + solve + post-step) through "
                    "mpc_b200_track_packed_submit/_wait with page-locked host buffers: one H2D + one D2H copy per batch "
                    "inside the timed region; %d host thread(s) x %d handles in flight each; host wall clock, max over ranks"
                    % (a.steps, NB, T, K))
    # the same copies WITHOUT any solve (all ranks at once, 8 streams each, ~0.3 s): what the host's memory / PCIe fabric
    # can feed.  Where e2e sits at this ceiling the end-to-end rate is bound by the box, not by the solver or its host code.
    try:
        cs = 8; n_copy = max(256, min(4000, per_thread * T))
        hin = [torch.empty(s0.h2d, dtype=torch.uint8).pin_memory() for _ in range(cs)]
        hout = [torch.empty(s0.d2h, dtype=torch.uint8).pin_memory() for _ in range(cs)]
        din = [torch.empty(s0.h2d, dtype=torch.uint8, device=dev) for _ in range(cs)]
        dout = [torch.empty(s0.d2h, dtype=torch.uint8, device=dev) for _ in range(cs)]
        cst = [torch.cuda.Stream() for _ in range(cs)]

        def copies(n):
            for j in range(n):
                with torch.cuda.stream(cst[j % cs]):
                    din[j % cs].copy_(hin[j % cs], non_blocking=True)
                    hout[j % cs].copy_(dout[j % cs], non_blocking=True)
            torch.cuda.synchronize()
        copies(64)
        barrier()
        t0 = time.perf_counter(); copies(n_copy); tc = time.perf_counter() - t0
        tct = torch.tensor([tc], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tct, op=dist.ReduceOp.MAX)
        e2e["copies_alone"] = dict(value=world * n_copy * B / float(tct.item()), unit=UNIT,
                                   gbytes_per_s=world * n_copy * (s0.h2d + s0.d2h) / float(tct.item()) / 1e9,
                                   note="the e2e leg's H2D + D2H copies with no solve in between, all ranks at once")
        del hin, hout, din, dout
    except Exception as ex:      # (a probe: never fails the bench)
        e2e["copies_alone"] = dict(error=str(ex))
    for w in workers:
        for s in w.slots:
            s.close()

    # ---- the rest of the line (rank 0): config-1 latency through the C++ MPC adapter, config-3 one-shot through the
    # C++ multi-GPU harness (mpc_bench multi: std::thread per GPU, contiguous slices, host gather), CPU baseline
    latency = None; config3 = None; cpu = None
    bench_bin = os.path.join(ROOT, "mpc_ros_b200", "lib", "mpc_bench")
    # (the other ranks leave first: a rank waiting in an NCCL barrier keeps a kernel spinning on its GPU, which is one of
    #  the GPUs mpc_bench multi is about to time)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
        if rank != 0:
            solver.close()
            return
        time.sleep(1.0)
    if rank == 0 and os.path.exists(bench_bin) and not a.no_extras:
        def run_json(args, timeout=600):
            r = subprocess.run([bench_bin] + args, capture_output=True, text=True, timeout=timeout)
            if r.returncode != 0:
                return dict(error=r.stderr[-500:])
            return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        if world == 1:
            lt = run_json(["latency", "3000"])
            latency = dict(p50_us=lt.get("p50_us"), p99_us=lt.get("p99_us"), calls=lt.get("calls"),
                           what="config 1: one MPC::Solve through the C++ adapter (batch of one, host buffers, H2D/D2H inside)") \
                if "error" not in lt else lt
        config3 = run_json(["multi", str(world), "65536", "5"])
    if rank == 0:
        if world == 1 and not a.no_cpu_baseline:
            cpu = cpu_reference_rate(a.ref_per_core)
        it_mean = float(np.mean([v[2] for v in per_set.values()])); it_max = int(max(v[3] for v in per_set.values()))
        cfg = bench_config(a, world)
        cfg.update(streams=S, max_ctas=max_ctas, in_flight_per_stream=DEPTH, host_affinity=numa,
                   issue_loop="python" if IL is None else "C++ (bench/issue_loop.cpp) over the C ABI",
                   step="one step = %d independent config-2 batches of %d problems, streamed on %d streams "
                        "(prestep + solve each); %d steps are timed back to back" % (NB, B, S, a.steps),
                   l2="inputs+outputs rotate over %d distinct batches (%.0f MB > 126 MB L2) after one L2 flush"
                      % (R, R * set_bytes / 1e6),
                   converged_fraction=conv_total / (B * n_batches * world), mean_iters_converged=it_mean, max_iters=it_max)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup,
                    ms_per_step=ms_total / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f64", data="synthetic", config=cfg,
                    clocks=clocks, e2e=e2e, gpu_launches=int(launches), roofline=roofline, latency=latency,
                    config3=config3, cpu_baseline=cpu)
        print(json.dumps(line))
    solver.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches-per-step", type=int, default=256, help="independent 4,096-problem batches per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--sets", type=int, default=48)
    ap.add_argument("--max-iter", type=int, default=100)
    ap.add_argument("--streams", type=int, default=64,
                    help="streams the batches of a step are issued on (64 x 8-CTA launches: measured best, profiles/r2_harness_sweep.txt)")
    ap.add_argument("--max-ctas", type=int, default=0)
    ap.add_argument("--depth", type=int, default=2, help="batches in flight per stream")
    ap.add_argument("--clock-period-ms", type=int, default=50, help="nvidia-smi sampling period during the timed region")
    ap.add_argument("--python-issue", action="store_true", help="issue the device-resident leg from Python instead of bench/issue_loop.cpp")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-1 latency and config-3 one-shot legs")
    ap.add_argument("--e2e-threads", type=int, default=2)
    ap.add_argument("--e2e-max-ctas", type=int, default=0)
    ap.add_argument("--e2e-inflight", type=int, default=96, help="ticks in flight over all e2e threads")
    ap.add_argument("--ref-per-core", type=int, default=160)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.warmup < 3:
        a.warmup = 3
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
