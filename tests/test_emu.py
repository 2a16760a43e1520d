"""CPU tier: the solver's phase functions (the code the CUDA kernel runs, nmpc_phases.cuh) executed
by the test-only host emulator, against the oracle.  Checks the LOGIC of the structure-exploiting
interior-point method here where there is no GPU; the -m gpu tier checks the kernel itself."""
import ctypes as C
import os

import numpy as np

from mpc_ros_b200 import capi
from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
from tests.problems import mild, generated, restoration_cases

_EMU = None


def emu_solve(pm, state, coeffs, PB=4, tol=1e-8, max_iter=200, ref_vel=None, warm=None, warm_mu=1e-3):
    """warm: warm-start records (warm_size x B, the kernel's layout) or None for the cold start."""
    global _EMU
    if _EMU is None:
        _EMU = C.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu", "libnmpc_emu.so"))
    dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int)
    N = int(pm["STEPS"]); B = state.shape[1]
    prm = np.array([pm["DT"], pm["REF_CTE"], pm["REF_ETHETA"], pm["REF_V"], pm["W_CTE"], pm["W_EPSI"], pm["W_V"],
                    pm["W_ANGVEL"], pm["W_A"], pm["ANGVEL"], pm["MAXTHR"], pm.get("W_DANGVEL", 0.0), pm.get("W_DA", 0.0),
                    min(pm.get("BOUND", 1e3), 1e300)],
                   dtype=np.float64)
    state = np.ascontiguousarray(state, dtype=np.float64); coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    u0 = np.zeros((2, B)); pred = np.zeros((3 * N, B)); obj = np.zeros(B); kkt = np.zeros(B)
    rec = np.zeros((capi.lib().mpc_b200_warm_size(N), B))      # the kernel's warm-start record
    st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32); nreg = np.zeros(B, dtype=np.int32)
    rv = None if ref_vel is None else np.ascontiguousarray(ref_vel, dtype=np.float64).ctypes.data_as(dp)
    P = lambda a: a.ctypes.data_as(dp)  # noqa: E731
    if warm is not None:
        warm_in = np.ascontiguousarray(warm, dtype=np.float64)
        assert warm_in.shape == warm.shape == (capi.lib().mpc_b200_warm_size(N), B)
    _EMU.nmpc_emu_solve(C.c_int(N), P(prm), C.c_double(tol), C.c_int(max_iter), C.c_int(PB), C.c_int(B), P(state),
                        P(coeffs), rv, P(u0), P(pred), P(obj), st.ctypes.data_as(ip), it.ctypes.data_as(ip), P(kkt),
                        P(rec), nreg.ctypes.data_as(ip), None if warm is None else P(warm_in), C.c_double(warm_mu))
    n = 8 * N - 2       # equality multipliers: rows [n, n + 6N) of the record
    return dict(u0=u0, pred=pred, obj=obj, status=st, iters=it, kkt=kkt, lam=rec[n:n + 6 * N], warm=rec, nreg=nreg)


def test_emu_matches_oracle_mild(oracle):
    state, coeffs = mild(21, 24)
    r = emu_solve(YAML_DEFAULT, state, coeffs, PB=5)
    nobound = dict(YAML_DEFAULT, BOUND=1e19)
    for i in range(24):
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5            # north-star tolerance
        assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"])
        assert r["kkt"][i] <= 1e-8
        # same algorithm, same iterates: against the oracle without the (inactive) state bounds the
        # Riccati solver reproduces iteration count, controls and multipliers to rounding
        o2 = oracle.solve(nobound, state[:, i], coeffs[:, i])
        assert r["iters"][i] == o2["iters"]
        assert np.abs(r["u0"][:, i] - o2["u0"]).max() <= 1e-10
        assert np.abs(r["lam"][:, i] - o2["lam"]).max() <= 1e-8 * max(1.0, np.abs(o2["lam"]).max())
        assert np.abs(r["pred"][:, i].reshape(3, -1) - o["pred"]).max() <= 1e-6


def test_emu_warm_record_matches_oracle(oracle):
    """The whole warm-start record the kernel's write-out fills (primal, equality multipliers, control-bound multipliers,
    all unscaled) against the oracle's solution without the (inactive) state bounds: same iterates, so equal to rounding."""
    pm = dict(YAML_DEFAULT, BOUND=1e19)
    N = int(pm["STEPS"]); n = 8 * N - 2; m = 6 * N; nu = N - 1
    w, a = slice(6 * N, 7 * N - 1), slice(7 * N - 1, n)        # the controls in the reference's variable layout
    state, coeffs = mild(27, 12)
    r = emu_solve(pm, state, coeffs, PB=5)
    assert r["warm"].shape[0] == n + m + 4 * nu
    close = lambda x, ref: np.abs(x - ref).max() <= 1e-8 * max(1.0, np.abs(ref).max())  # noqa: E731
    for i in range(12):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        rec = r["warm"][:, i]
        assert close(rec[:n], o["sol"])
        assert close(rec[n:n + m], o["lam"])
        zlw, zla, zuw, zua = (rec[n + m + j * nu:n + m + (j + 1) * nu] for j in range(4))
        assert close(zlw, o["zl"][w]) and close(zla, o["zl"][a])
        assert close(zuw, o["zu"][w]) and close(zua, o["zu"][a])


def test_emu_matches_oracle_generated(oracle):
    g, state, coeffs = generated(20261020, 150, oracle)
    r = emu_solve(YAML_DEFAULT, state, coeffs, PB=32)
    both = 0; close = 0
    for i in range(150):
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        if o["status"] == 1 and r["status"][i] == 1:
            both += 1
            if np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5 and abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"]):
                close += 1
    assert both >= 147
    assert close >= both - 1       # a non-convex corner case may settle in another local minimum


def test_emu_cfg_weights(oracle):
    pm = dict(CFG_DEFAULT, W_DA=0.0)
    state, coeffs = mild(22, 8)
    r = emu_solve(pm, state, coeffs, PB=3)
    for i in range(8):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5
        assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"])


def test_emu_rate_penalties(oracle):
    """w_angvel_d / w_accel_d != 0 (the reference's cfg defaults, MPCPlanner.cfg:31-33): augmented Riccati."""
    for pm in (dict(CFG_DEFAULT), dict(YAML_DEFAULT, W_DANGVEL=30.0, W_DA=5.0), dict(YAML_DEFAULT, W_DANGVEL=200.0, W_DA=0.0)):
        state, coeffs = mild(26, 10)
        r = emu_solve(pm, state, coeffs, PB=3)
        nobound = dict(pm, BOUND=1e19)
        for i in range(10):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert r["status"][i] == 1 and o["status"] == 1
            assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5
            assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"])
            assert r["kkt"][i] <= 1e-8
            o2 = oracle.solve(nobound, state[:, i], coeffs[:, i])
            assert r["iters"][i] == o2["iters"]
            assert np.abs(r["u0"][:, i] - o2["u0"]).max() <= 1e-9


def test_emu_long_horizon(oracle):
    pm = dict(YAML_DEFAULT, STEPS=100)
    state, coeffs = mild(23, 2)
    coeffs[2:] *= 0.1      # keep a 10 s horizon on a sane path
    r = emu_solve(pm, state, coeffs, PB=2)
    for i in range(2):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5
        assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"])


def test_emu_lane_independence():
    """A problem's result must not depend on which CTA lane it lands in or on its neighbours."""
    state, coeffs = mild(24, 13)
    a = emu_solve(YAML_DEFAULT, state, coeffs, PB=1)
    b = emu_solve(YAML_DEFAULT, state, coeffs, PB=32)
    perm = np.random.default_rng(0).permutation(13)
    c = emu_solve(YAML_DEFAULT, state[:, perm], coeffs[:, perm], PB=4)
    np.testing.assert_array_equal(a["u0"], b["u0"])
    np.testing.assert_array_equal(a["u0"][:, perm], c["u0"])
    np.testing.assert_array_equal(a["iters"][perm], c["iters"])


def test_emu_ref_vel_override(oracle):
    state, coeffs = mild(25, 4)
    rv = np.array([0.2, 0.5, 0.8, 0.05])
    r = emu_solve(YAML_DEFAULT, state, coeffs, PB=4, ref_vel=rv)
    for i in range(4):
        o = oracle.solve(dict(YAML_DEFAULT, REF_V=rv[i]), state[:, i], coeffs[:, i])
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5


def test_emu_small_weights_keep_lsq_multipliers(oracle):
    """With small weights the least-squares multiplier start stays below 1e3 and is KEPT (W&B Sec. 3.6); with
    the YAML weights it is discarded (test_emu_matches_oracle_mild).  The size test is folded into the adjoint
    sweep: both outcomes must reproduce the oracle's iterates."""
    pm = dict(YAML_DEFAULT, W_CTE=2.0, W_V=5.0, W_ANGVEL=1.0, W_A=1.0, BOUND=1e19)
    state, coeffs = mild(23, 16)
    r = emu_solve(pm, state, coeffs, PB=7)
    big = dict(YAML_DEFAULT, BOUND=1e19)
    rb = emu_solve(big, state, coeffs, PB=7)
    kept = 0
    for i in range(16):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        assert r["iters"][i] == o["iters"]
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-9
        assert np.abs(r["lam"][:, i] - o["lam"]).max() <= 1e-8 * max(1.0, np.abs(o["lam"]).max())
        ob = oracle.solve(big, state[:, i], coeffs[:, i])
        assert rb["iters"][i] == ob["iters"]
        kept += int(np.abs(o["lam"]).max() < 1e3)
    assert kept == 16      # (the converged multipliers are small too: the start was not the discarded kind)


def emu_solve_poly(pm, state, coeffs, PB=4, tol=1e-8, max_iter=200, warm=None, warm_mu=1e-3):
    """Path polynomial of order coeffs.shape[0] - 1 in 4..7 (the kernel's higher-order instantiation)."""
    emu_solve(pm, state[:, :1], coeffs[:4, :1])      # (loads the library)
    dp = C.POINTER(C.c_double); ip = C.POINTER(C.c_int)
    N = int(pm["STEPS"]); B = state.shape[1]; nc = coeffs.shape[0]
    prm = np.array([pm["DT"], pm["REF_CTE"], pm["REF_ETHETA"], pm["REF_V"], pm["W_CTE"], pm["W_EPSI"], pm["W_V"],
                    pm["W_ANGVEL"], pm["W_A"], pm["ANGVEL"], pm["MAXTHR"], pm.get("W_DANGVEL", 0.0), pm.get("W_DA", 0.0),
                    min(pm.get("BOUND", 1e3), 1e300)],
                   dtype=np.float64)
    state = np.ascontiguousarray(state, dtype=np.float64); coeffs = np.ascontiguousarray(coeffs, dtype=np.float64)
    u0 = np.zeros((2, B)); pred = np.zeros((3 * N, B)); obj = np.zeros(B); kkt = np.zeros(B)
    st = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32)
    rec = np.zeros((capi.lib().mpc_b200_warm_size(N), B))
    P = lambda a: a.ctypes.data_as(dp)  # noqa: E731
    if warm is not None:
        warm_in = np.ascontiguousarray(warm, dtype=np.float64)
        assert warm_in.shape == rec.shape
    rc = _EMU.nmpc_emu_solve_poly(C.c_int(N), P(prm), C.c_double(tol), C.c_int(max_iter), C.c_int(PB), C.c_int(B), C.c_int(nc),
                                  P(state), P(coeffs), P(u0), P(pred), P(obj), st.ctypes.data_as(ip), it.ctypes.data_as(ip), P(kkt),
                                  P(rec), None if warm is None else P(warm_in), C.c_double(warm_mu))
    assert rc == 0
    return dict(u0=u0, pred=pred, obj=obj, status=st, iters=it, kkt=kkt, warm=rec)


def higher_order(seed, batch, ncoef):
    """Mild problems with a path polynomial of order ncoef - 1 (FG_eval takes any order, mpc_planner.cpp:186-190)."""
    state, c4 = mild(seed, batch)
    rng = np.random.default_rng(seed + 1000)
    coeffs = np.zeros((ncoef, batch)); coeffs[:4] = c4
    coeffs[4:] = rng.uniform(-0.05, 0.05, size=(ncoef - 4, batch))
    return state, coeffs


def test_emu_higher_order_path_polynomial(oracle):
    pm = dict(YAML_DEFAULT, BOUND=1e19)
    for ncoef in (5, 6, 8):
        state, coeffs = higher_order(70 + ncoef, 10, ncoef)
        r = emu_solve_poly(pm, state, coeffs, PB=3)
        for i in range(10):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert r["status"][i] == 1 and o["status"] == 1
            assert r["iters"][i] == o["iters"]
            assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-9
            assert abs(r["obj"][i] - o["obj"]) <= 1e-9 * abs(o["obj"])
            # the higher coefficients matter: the cubic part alone gives another answer
            o3 = oracle.solve(pm, state[:, i], coeffs[:4, i])
            assert abs(o3["obj"] - o["obj"]) > 1e-7 * abs(o["obj"])


def test_emu_higher_order_with_rate_penalties(oracle):
    pm = dict(CFG_DEFAULT, BOUND=1e19)
    state, coeffs = higher_order(77, 8, 6)
    r = emu_solve_poly(pm, state, coeffs, PB=3)
    for i in range(8):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert r["status"][i] == 1 and o["status"] == 1
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-7
        assert abs(r["obj"][i] - o["obj"]) <= 1e-8 * abs(o["obj"])


def test_emu_short_and_odd_horizons(oracle):
    """mpc_steps is a parameter (mpc_planner.cpp:247): horizons that do not fill the stage groups evenly, down to 3."""
    for N in (3, 5, 7, 21):
        pm = dict(YAML_DEFAULT, STEPS=N, BOUND=1e19)
        state, coeffs = mild(30 + N, 6)
        r = emu_solve(pm, state, coeffs, PB=4)
        for i in range(6):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert r["status"][i] == 1 and o["status"] == 1, (N, i)
            assert r["iters"][i] == o["iters"], (N, i)
            assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-9
            assert abs(r["obj"][i] - o["obj"]) <= 1e-9 * max(1e-12, abs(o["obj"]))


def test_emu_second_order_correction_matches_oracle_iterates(oracle):
    """The kernel's second-order correction (W&B A-5.5 .. A-5.9) against the oracle's: on the real config-4 generator at
    N = 100 (where the correction triggers in several per cent of the problems and decides which local minimum is
    reached) the emulated kernel and the oracle without the +-1e3 state bounds end in the same point with the same
    status, and take the same number of iterations in > 98 % of the problems."""
    from bench import gen_py
    n, N = 72, 100
    g = gen_py.problems(20261018 + 4, n)
    coeffs = np.zeros((4, n)); state = np.zeros((6, n))
    for i in range(n):
        c, cte, eth = oracle.prestep(g["wx"][:, i], g["wy"][:, i], *g["pose"][:, i])
        coeffs[:, i] = c; state[3, i] = g["vel"][0, i]; state[4, i] = cte; state[5, i] = eth
    pm = dict(YAML_DEFAULT, STEPS=N)
    r = emu_solve(pm, state, coeffs, PB=32, max_iter=100)
    opt = oracle.default_options(); opt.max_iter = 100
    nob = dict(pm, BOUND=1e19)
    same_iters = 0; both = 0; nsoc_matter = 0
    opt0 = oracle.default_options(); opt0.max_iter = 100; opt0.max_soc = 0
    for i in range(n):
        o = oracle.solve(nob, state[:, i], coeffs[:, i], opt)
        assert (r["status"][i] == 1) == (o["status"] == 1), (i, r["status"][i], o["status"])
        if o["status"] != 1:
            continue
        both += 1
        assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5, i
        assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"]), i
        same_iters += int(r["iters"][i] == o["iters"])
        if o["iters"] > 12:        # (the easy problems never reject a first trial)
            o0 = oracle.solve(nob, state[:, i], coeffs[:, i], opt0)
            nsoc_matter += int(o0["iters"] != o["iters"] or o0["status"] != o["status"])
    assert both >= n - 2
    assert same_iters >= 0.97 * both, (same_iters, both)
    assert nsoc_matter >= 2, nsoc_matter       # the correction does make a difference on this set


def test_emu_restoration_matches_oracle(oracle):
    """Line search below alpha_min: the kernel logic runs the same feasibility restoration as the oracle (min-norm steps on
    the constraint violation, kappa_resto = 0.9, filter test, bound multipliers reset) instead of giving up with status 9:
    problems the oracle rescues converge to the same point in the same number of iterations, the others end with the
    oracle's status (5 = locally infeasible)."""
    state, coeffs = restoration_cases(oracle)
    opt = oracle.default_options(); opt.max_iter = 100
    r = emu_solve(YAML_DEFAULT, state, coeffs, PB=3, max_iter=100)
    rescued = 0
    for i in range(state.shape[1]):
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i], opt)
        assert o["n_resto"] >= 1
        assert r["status"][i] == o["status"], (i, r["status"][i], o["status"])
        if o["status"] == 1:
            rescued += 1
            assert r["iters"][i] == o["iters"]
            assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-5
            assert abs(r["obj"][i] - o["obj"]) <= 1e-6 * abs(o["obj"])
            assert r["kkt"][i] <= 1e-8
    assert rescued == 3
