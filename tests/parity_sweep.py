"""tests/parity_sweep.py -- large GPU-vs-oracle parity sweep (a script, not a pytest module: it needs a GPU
and minutes of host CPU).  For each weight set (mpc_params.yaml defaults; MPCPlanner.cfg defaults = rate
penalties) it solves the same seeded config-2 problems on the GPU through the C ABI and with the oracle
(the checker) on all host cores, and prints one JSON line of agreement statistics:
    python tests/parity_sweep.py [n_problems] > profiles/rN_parity_sweep.json
Tolerances are the north-star's: |du0| <= 1e-5, objective <= 1e-6 relative, scaled KKT error <= 1e-8."""
import json
import multiprocessing as mp
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

MAX_ITER = 100


def _oracle_chunk(args):
    """args: (pm, state, coeffs) or (pm, state, coeffs, warm records, warm_mu) for warm-started solves"""
    from oracle.oracle_py import Oracle
    pm, state, coeffs = args[:3]
    warm, warm_mu = args[3:] if len(args) > 3 else (None, 1e-3)
    orc = Oracle()
    opt = orc.default_options(); opt.max_iter = MAX_ITER
    B = state.shape[1]
    out = dict(u0=np.zeros((2, B)), obj=np.zeros(B), status=np.zeros(B, dtype=np.int32), iters=np.zeros(B, dtype=np.int32),
               kkt=np.zeros(B))
    for i in range(B):
        r = orc.solve(pm, state[:, i], coeffs[:, i], opt, warm=None if warm is None else warm[:, i], warm_mu=warm_mu)
        out["u0"][:, i] = r["u0"]; out["obj"][i] = r["obj"]; out["status"][i] = r["status"]
        out["iters"][i] = r["iters"]; out["kkt"][i] = r["kkt_error"]
    return out


def sweep(name, pm, n, seed):
    from mpc_ros_b200 import capi
    from bench import gen_py
    g = gen_py.problems(seed, n)
    prm = capi.params_from_map(pm, capi.yaml_default_params()); prm.delay_mode = 0; prm.max_iter = MAX_ITER
    sv = capi.Solver(prm, n, 0)
    coeffs, state = sv.prestep(g["wx"], g["wy"], g["pose"], g["vel"])
    gpu = sv.solve(state, coeffs)
    ms = sv.last_kernel_seconds * 1e3
    sv.close()
    P = os.cpu_count() or 1
    cuts = np.linspace(0, n, 4 * P + 1).astype(int)
    with mp.get_context("fork").Pool(P) as pool:
        parts = pool.map(_oracle_chunk, [(pm, state[:, a:b].copy(), coeffs[:, a:b].copy()) for a, b in zip(cuts[:-1], cuts[1:]) if b > a])
    orc = {k: np.concatenate([p[k] for p in parts], axis=-1) for k in parts[0]}
    okg = (gpu["status"] == 1) & (gpu["kkt"] <= 1e-8); oko = (orc["status"] == 1)
    both = okg & oko
    du = np.abs(gpu["u0"] - orc["u0"]).max(axis=0)
    dobj = np.abs(gpu["obj"] - orc["obj"]) / np.maximum(1.0, np.abs(orc["obj"]))
    res = dict(weights=name, problems=n, seed=seed, max_iter=MAX_ITER, gpu_kernel_ms=ms,
               gpu_converged=int(okg.sum()), oracle_converged=int(oko.sum()), both_converged=int(both.sum()),
               only_gpu=int((okg & ~oko).sum()), only_oracle=int((~okg & oko).sum()),
               status_equal=int((gpu["status"] == orc["status"]).sum()),
               iters_equal_among_both=int((gpu["iters"][both] == orc["iters"][both]).sum()),
               max_abs_du0=float(du[both].max()), p999_abs_du0=float(np.quantile(du[both], 0.999)),
               within_1e5_du0=int((du[both] <= 1e-5).sum()),
               max_rel_dobj=float(dobj[both].max()), within_1e6_dobj=int((dobj[both] <= 1e-6).sum()),
               max_gpu_kkt_converged=float(gpu["kkt"][okg].max()),
               gpu_status_hist={int(k): int(v) for k, v in zip(*np.unique(gpu["status"], return_counts=True))},
               oracle_status_hist={int(k): int(v) for k, v in zip(*np.unique(orc["status"], return_counts=True))},
               mean_iters_gpu=float(gpu["iters"][okg].mean()), mean_iters_oracle=float(orc["iters"][oko].mean()))
    return res


def main():
    from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
    # third sweep: the oracle without the (never active) +-1e3 state bounds, which the GPU path leaves out --
    # isolates their effect on the iterates
    out = [sweep("mpc_params.yaml", YAML_DEFAULT, n, 20261018 + 2), sweep("MPCPlanner.cfg", CFG_DEFAULT, n, 20261018 + 12),
           sweep("mpc_params.yaml, oracle BOUND=1e19", dict(YAML_DEFAULT, BOUND=1.0e19), n, 20261018 + 2)]
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
