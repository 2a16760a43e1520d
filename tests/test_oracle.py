"""CPU tier: the oracle (oracle/*.c) against the reference's own outputs and known answers."""
import json
import os

import numpy as np
import pytest

from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
from tests.problems import mild, generated

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _dense(n, m, triplets, sym=False):
    M = np.zeros((n, m))
    for i, j, v in triplets:
        M[i, j] = v
        if sym:
            M[j, i] = v
    return M


def test_fg_eval_matches_reference_golden(oracle):
    """Analytic f, grad, g, J, Hessian vs the reference FG_eval + CppAD dump (mpc_planner.cpp:102-217)."""
    cases = json.load(open(os.path.join(GOLD, "fg_eval_golden.json")))
    assert cases[0]["nnz_jac"] == 424 and cases[0]["nnz_hess"] == 210      # SURVEY P4
    assert abs(cases[0]["f"] - 4796.9161862598567) < 1e-9                   # SURVEY 8c golden value
    for cs in cases:
        N = int(cs["params"]["STEPS"]); n = 8 * N - 2; m = 6 * N
        o = oracle.eval_all(cs["params"], cs["coeffs"], cs["x"], cs["lam"], 1.0)
        scale = max(1.0, abs(cs["f"]))
        assert abs(o["f"] - cs["f"]) <= 1e-13 * scale
        np.testing.assert_allclose(o["grad"], cs["grad"], rtol=0, atol=1e-12 * scale)
        np.testing.assert_allclose(o["g"], cs["g"], rtol=0, atol=1e-13)
        np.testing.assert_allclose(o["J"], _dense(m, n, cs["jac"]), rtol=0, atol=1e-13)
        np.testing.assert_allclose(o["H"], _dense(n, n, cs["hess_lower"], sym=True), rtol=0, atol=1e-11)


def test_hs071_known_answer():
    """The reference's shipped known answer (assets/document/example/CppAD_Ipopt.cpp:146-150)."""
    g = json.load(open(os.path.join(GOLD, "hs071_golden.json")))
    s = g["standin"]
    assert s["status"] == 1
    np.testing.assert_allclose(s["x"], g["known_x"], rtol=1e-6, atol=1e-6)
    assert abs(s["zl"][0] - g["known_zl0"]) <= 1e-6
    np.testing.assert_allclose(s["zl"][1:], 0.0, atol=1e-6)
    np.testing.assert_allclose(s["zu"], 0.0, atol=1e-6)
    assert abs(s["obj"] - 17.0140171) < 1e-6          # Ipopt manual value for HS071


def test_hs071_live_through_cppad_glue():
    """HS071 run through the reference's CppAD glue and the stand-in solver (Reference.hs071(1e-8), stored by
    make_golden.py as the "standin" record) reaches the answer the reference ships."""
    r = json.load(open(os.path.join(GOLD, "hs071_golden.json")))["standin"]
    assert r["status"] == 1
    np.testing.assert_allclose(r["x"], [1.0, 4.743, 3.82115, 1.379408], rtol=1e-6, atol=1e-6)
    assert abs(r["zl"][0] - 1.087871) <= 1e-6


def test_solve_matches_reference_golden(oracle):
    """oracle restatement vs MPC::Solve of the reference class (same stand-in solver, CppAD derivatives)."""
    sols = json.load(open(os.path.join(GOLD, "solve_golden.json")))
    for s in sols:
        o = oracle.solve(s["params"], s["state"], s["coeffs"])
        assert o["status"] == s["status"] == 1
        np.testing.assert_allclose(o["u0"], s["u0"], rtol=0, atol=1e-9)
        assert abs(o["obj"] - s["obj"]) <= 1e-9 * abs(s["obj"])
        np.testing.assert_allclose(o["pred"], np.array(s["pred"]), rtol=0, atol=1e-8)
        assert o["kkt_error"] <= 1e-8


def test_solve_matches_reference_live(oracle):
    """The oracle takes the reference's iterations: same iteration count and u0 to 1e-10 as MPC::Solve of the reference
    class (stored in solve_golden.json by make_golden.py with the CPU-time limit lifted)."""
    for s in json.load(open(os.path.join(GOLD, "solve_golden.json"))):
        o = oracle.solve(s["params"], s["state"], s["coeffs"])
        assert s["status"] == o["status"] == 1
        assert s["iters"] == o["iters"]
        np.testing.assert_allclose(s["u0"], o["u0"], rtol=0, atol=1e-10)


def test_oracle_against_scipy(oracle):
    """Independent solver (SciPy SLSQP on the same NLP) reaches the same KKT point."""
    scipy_opt = pytest.importorskip("scipy.optimize")
    pm = dict(YAML_DEFAULT, STEPS=8)
    N = 8; n = 8 * N - 2; m = 6 * N
    state, coeffs = mild(3, 3)
    for i in range(3):
        s6, c4 = state[:, i], coeffs[:, i]
        o = oracle.solve(pm, s6, c4)
        assert o["status"] == 1
        lam0 = np.zeros(m)
        gl = np.zeros(m)
        for k in range(6):
            gl[k * N] = s6[k]

        def f(x): return oracle.eval_all(pm, c4, x, lam0)["f"]
        def gf(x): return oracle.eval_all(pm, c4, x, lam0)["grad"]
        def g(x): return oracle.eval_all(pm, c4, x, lam0)["g"] - gl
        def gj(x): return oracle.eval_all(pm, c4, x, lam0)["J"]
        lb = np.full(n, -pm["BOUND"]); ub = np.full(n, pm["BOUND"])
        lb[6 * N:7 * N - 1] = -pm["ANGVEL"]; ub[6 * N:7 * N - 1] = pm["ANGVEL"]
        lb[7 * N - 1:] = -pm["MAXTHR"]; ub[7 * N - 1:] = pm["MAXTHR"]
        x0 = np.zeros(n)
        for k in range(6):
            x0[k * N] = s6[k]
        r = scipy_opt.minimize(f, x0, jac=gf, method="SLSQP", bounds=list(zip(lb, ub)),
                               constraints=[dict(type="eq", fun=g, jac=gj)], options=dict(maxiter=500, ftol=1e-13))
        # status 8 ("positive directional derivative") is SLSQP's way of stopping AT the optimum with a tight ftol
        assert r.status in (0, 8), r.message
        assert abs(r.fun - o["obj"]) <= 1e-7 * abs(o["obj"])
        np.testing.assert_allclose([r.x[6 * N], r.x[7 * N - 1]], o["u0"], atol=2e-5)


def test_state_bounds_inactive(oracle):
    """The +-bound_value state bounds (mpc_planner.cpp:308-312) never bind: dropping them moves the
    solution by O(mu/bound) only.  This is what licenses the GPU path to carry control bounds only."""
    state, coeffs = mild(11, 6)
    for i in range(6):
        a = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        b = oracle.solve(dict(YAML_DEFAULT, BOUND=1e19), state[:, i], coeffs[:, i])
        assert a["status"] == b["status"] == 1
        np.testing.assert_allclose(a["u0"], b["u0"], atol=1e-7)
        assert abs(a["obj"] - b["obj"]) <= 1e-8 * abs(a["obj"])


def test_cfg_weights_and_rate_terms(oracle):
    """cfg-default weights incl. the rate penalty (MPCPlanner.cfg:22-37) solve and satisfy KKT."""
    state, coeffs = mild(5, 4)
    for i in range(4):
        o = oracle.solve(CFG_DEFAULT, state[:, i], coeffs[:, i])
        assert o["status"] == 1 and o["kkt_error"] <= 1e-8
        assert abs(o["u0"][0]) <= CFG_DEFAULT["ANGVEL"] * (1 + 2e-8)


def test_polyfit_matches_numpy(oracle):
    rng = np.random.default_rng(0)
    for M in (4, 5, 11, 30):
        x = np.sort(rng.uniform(-1, 5, M)); y = rng.normal(size=M)
        c = oracle.polyfit(x, y, 3)
        ref = np.polynomial.polynomial.polyfit(x, y, 3)
        np.testing.assert_allclose(c, ref, rtol=1e-9, atol=1e-9)
    with pytest.raises(ValueError):
        oracle.polyfit([0.0, 1.0, 2.0], [0.0, 1.0, 2.0], 3)       # order > M-1: the reference asserts


def test_prestep_quirks(oracle):
    """etheta rule of driving_state.cpp:215-235: zero when gx or gy is exactly zero (axis-aligned path)."""
    wx = np.arange(11) * 0.5; wy = np.zeros(11)
    c, cte, eth = oracle.prestep(wx, wy, 0.0, 0.2, 0.3)
    assert eth == 0.0                                  # gy == 0 -> forced to 0
    assert abs(cte - (-0.2 / np.cos(0.3))) < 1e-9      # c[0] = where the path crosses the robot's y axis
    wy2 = 0.1 * wx
    c, cte, eth = oracle.prestep(wx, wy2, 0.0, 0.0, 0.3)
    assert abs(eth - (0.3 - np.arctan2(0.1, 1.0))) < 1e-12
    # wrap: theta <= -pi + traj_deg gets 2 pi added, then the < 1.8 pi guard
    c, cte, eth = oracle.prestep(wx, wy2, 0.0, 0.0, -3.1)
    assert abs(eth - (-3.1 + 2 * np.pi - np.arctan2(0.1, 1.0))) < 1e-12


def test_generated_set_statistics(oracle):
    """The benchmark generator (SURVEY 8d): deterministic, three tracks, M = 11 waypoints."""
    g, state, coeffs = generated(20261020, 96, oracle)
    g2, state2, coeffs2 = generated(20261020, 96, oracle)
    assert g["M"] == 11
    np.testing.assert_array_equal(state, state2)
    assert set(g["kind"].tolist()) == {0, 1, 2}
    assert np.all(state[3] >= 0) and np.all(state[3] <= 0.6)


def test_decel_known_answers(oracle):
    """Tracking::deceleration (driving_state.cpp:121-141) worked by hand."""
    thr, vmax, vmin = 1.0, 0.7, 0.05
    # outside the braking distance: REF_V untouched
    assert oracle.decel(0, 0, 1.0, 0, 0.5, thr, vmax, vmin, 0.5) == 0.5
    # inside, speed = thr * dist = 1.0 > REF_V -> max_speed (the reference's branch, as written)
    assert oracle.decel(0, 0, 1.0, 0, 1.2, thr, vmax, vmin, 0.5) == 0.7
    # inside, min_speed <= speed <= REF_V -> speed
    assert abs(oracle.decel(0, 0, 0.3, 0, 0.6, thr, vmax, vmin, 0.5) - 0.3) < 1e-16
    # inside, speed < min_speed -> min_speed
    assert oracle.decel(0, 0, 0.0, 0.02, 0.2, thr, vmax, vmin, 0.5) == 0.05
    # boundary: dist == v^2 / thr counts as inside
    assert oracle.decel(0, 0, 0.25, 0, 0.5, thr, vmax, vmin, 0.5) == 0.25


def test_oracle_solution_satisfies_the_reference_kkt_conditions(oracle):
    """grad f + J^T lambda - zL + zU = 0, g = g_target at the oracle's solutions, with f, g, J from the restatement
    of FG_eval that the golden vectors pin to the reference's CppAD output (the same check runs on the GPU results
    in tests/test_gpu_parity.py::test_kkt_conditions_in_the_reference_formulation)."""
    pm = YAML_DEFAULT
    N = int(pm["STEPS"]); m = 6 * N
    state, coeffs = mild(61, 8)
    for i in range(8):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert o["status"] == 1
        ev = oracle.eval_all(pm, coeffs[:, i], o["sol"], o["lam"], 1.0)
        target = np.zeros(m)
        for c in range(6):
            target[c * N] = state[c, i]
        assert np.abs(ev["g"] - target).max() <= 1e-8
        r = ev["grad"] + ev["J"].T @ o["lam"] - o["zl"] + o["zu"]
        assert np.abs(r).max() <= 1e-6          # unscaled; the scaled error is o["kkt_error"] <= 1e-8
        assert o["kkt_error"] <= 1e-8
