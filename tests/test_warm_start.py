"""Warm-started solves, iterate for iterate: the oracle's warm start (oracle/mpc_oracle.c, mpc_oracle_solve_warm, a
restatement of the record's rule from include/mpc_b200.h) against the emulated kernel phases (CPU tier) and the solve
kernels (GPU tier), from the same record bits.

The rule (record layout: nmpc_phases.cuh warm_uw / warm_ua / warm_lam / warm_z, multipliers unscaled; U = the relaxed
control bound, sf = the cold start's objective scaling, mu_w = warm_mu_init):
  controls from the record clipped into [-U + 1e-3 U, U - 1e-3 U]; states rolled out from the given state with those
  controls (the record's state rows are not read); lambda (lambda_0 included) times sf; z = max(sf z, mu_w / slack);
  mu = mu_w, tau = max(0.99, 1 - mu_w), no least-squares multipliers; then the cold iteration.
A wrong warm start still converges to the same KKT point, so these tests compare iteration counts and iterates."""

import numpy as np
import pytest

from mpc_ros_b200 import capi
from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
from tests.problems import mild
from tests.test_emu import emu_solve, emu_solve_poly, higher_order

CASES = ("a", "b", "c", "d", "e", "f")


def blocks(N):
    """lengths of the record's 18 blocks: 6 state components, 2 controls, 6 multiplier components, zL_w, zL_a, zU_w, zU_a"""
    return [N] * 6 + [N - 1] * 2 + [N] * 6 + [N - 1] * 4


def shift(rec, N):
    """numpy restatement of mpc_b200_warm_shift: every block moves one stage forward, its last entry is repeated"""
    out = np.empty_like(rec)
    off = 0
    for n in blocks(N):
        out[off:off + n - 1] = rec[off + 1:off + n]
        out[off + n - 1] = rec[off + n - 1]
        off += n
    assert off == rec.shape[0]
    return out


def record_from_oracle(o, N):
    """the record of an oracle solution, in the kernel's layout"""
    n = 8 * N - 2
    w, a = slice(6 * N, 7 * N - 1), slice(7 * N - 1, n)
    return np.concatenate([o["sol"], o["lam"], o["zl"][w], o["zl"][a], o["zu"][w], o["zu"][a]])


def relaxed(b):
    return b + 1e-8 * max(1.0, b)


def record_case(case, rec, state, pm):
    """(state, records) of record source `case` built from the converged records `rec` (warm_size x B) of `state`:
    (a) the problems' own records; (b) their shifted records, on the state one closed-loop tick moves to (the
    solution's stage 1 in the robot frame: v_1, cte_1, etheta_1); (c) the record of another problem (columns rolled by
    one); (d) controls at exactly +-U and +-2U (the push into the interior); (e) all multipliers zero (the mu / slack
    floor of z, lambda = 0); (f) (a) with the state rows set to 1e6 (they are not read)."""
    N = int(pm["STEPS"]); n = 8 * N - 2
    rec = np.array(rec, dtype=np.float64, copy=True); state = np.array(state, dtype=np.float64, copy=True)
    if case == "b":
        st = np.zeros_like(state)
        st[3], st[4], st[5] = rec[3 * N + 1], rec[4 * N + 1], rec[5 * N + 1]
        return st, shift(rec, N)
    if case == "c":
        return state, np.roll(rec, 1, axis=1)
    if case == "d":
        Uw, Ua = relaxed(pm["ANGVEL"]), relaxed(pm["MAXTHR"])
        pat = np.array([1.0, -1.0, 2.0, -2.0])
        k = np.arange(N - 1)[:, None] + np.arange(rec.shape[1])[None, :]
        rec[6 * N:7 * N - 1] = Uw * pat[k % 4]
        rec[7 * N - 1:n] = -Ua * pat[(k + 1) % 4]
        return state, rec
    if case == "e":
        rec[n:] = 0.0
        return state, rec
    if case == "f":
        rec[:6 * N] = 1e6
        return state, rec
    return state, rec


def kkt_ok(oracle, pm, state, coeffs, o):
    """the reference-NLP KKT conditions at an oracle result (as test_oracle_solution_satisfies_the_reference_kkt_conditions)"""
    N = int(pm["STEPS"])
    ev = oracle.eval_all(pm, coeffs, o["sol"], o["lam"], 1.0)
    target = np.zeros(6 * N)
    for c in range(6):
        target[c * N] = state[c]
    r = ev["grad"] + ev["J"].T @ o["lam"] - o["zl"] + o["zu"]
    return np.abs(ev["g"] - target).max() <= 1e-8 and np.abs(r).max() <= 1e-6 and o["kkt_error"] <= 1e-8


# ---------------------------------------------------------------- CPU tier: the oracle's warm start on its own

def test_oracle_warm_start(oracle):
    """The oracle's warm start is pinned to the NLP, not to the kernel: from its own converged record it ends at its cold
    solution in fewer iterations; from every record source it ends at a point that satisfies the reference NLP's KKT
    conditions; and it reaches SciPy's solution."""
    pm = dict(YAML_DEFAULT, BOUND=1e19)
    N = int(pm["STEPS"])
    state, coeffs = mild(81, 6)
    cold = [oracle.solve(pm, state[:, i], coeffs[:, i]) for i in range(6)]
    rec = np.stack([record_from_oracle(o, N) for o in cold], axis=1)
    assert rec.shape[0] == capi.lib().mpc_b200_warm_size(N)
    for i, o in enumerate(cold):
        assert o["status"] == 1
        w = oracle.solve(pm, state[:, i], coeffs[:, i], warm=rec[:, i])
        assert w["status"] == 1 and w["iters"] < o["iters"], (i, w["iters"], o["iters"])
        assert np.abs(w["u0"] - o["u0"]).max() <= 1e-9
        assert abs(w["obj"] - o["obj"]) <= 1e-10 * abs(o["obj"])
        assert np.abs(w["sol"] - o["sol"]).max() <= 1e-7 * max(1.0, np.abs(o["sol"]).max())   # (both stop at tol 1e-8)
    for case in CASES[:5]:
        st, rc = record_case(case, rec, state, pm)
        for i in range(6):
            w = oracle.solve(pm, st[:, i], coeffs[:, i], warm=rc[:, i])
            assert w["status"] == 1, (case, i)
            assert kkt_ok(oracle, pm, st[:, i], coeffs[:, i], w), (case, i)
    # the rule is refused where it does not apply: finite state bounds have no multipliers in the record
    with pytest.raises(ValueError):
        oracle.solve(YAML_DEFAULT, state[:, 0], coeffs[:, 0], warm=rec[:, 0])


def test_oracle_warm_start_against_scipy(oracle):
    """Independent solver (SciPy SLSQP, as test_oracle_against_scipy) on the same NLP: the warm-started oracle from a poor
    start (another problem's record) and from the shifted record reaches SciPy's minimum."""
    scipy_opt = pytest.importorskip("scipy.optimize")
    pm = dict(YAML_DEFAULT, STEPS=8, BOUND=1e19)
    N = 8; n = 8 * N - 2; m = 6 * N
    state, coeffs = mild(83, 3)
    rec = np.stack([record_from_oracle(oracle.solve(pm, state[:, i], coeffs[:, i]), N) for i in range(3)], axis=1)
    for case in ("b", "c"):
        st, rc = record_case(case, rec, state, pm)
        for i in range(3):
            s6, c4 = st[:, i], coeffs[:, i]
            o = oracle.solve(pm, s6, c4, warm=rc[:, i])
            assert o["status"] == 1
            lam0 = np.zeros(m); gl = np.zeros(m)
            for k in range(6):
                gl[k * N] = s6[k]

            def f(x): return oracle.eval_all(pm, c4, x, lam0)["f"]
            def gf(x): return oracle.eval_all(pm, c4, x, lam0)["grad"]
            def g(x): return oracle.eval_all(pm, c4, x, lam0)["g"] - gl
            def gj(x): return oracle.eval_all(pm, c4, x, lam0)["J"]
            lb = np.full(n, -1e19); ub = np.full(n, 1e19)
            lb[6 * N:7 * N - 1] = -pm["ANGVEL"]; ub[6 * N:7 * N - 1] = pm["ANGVEL"]
            lb[7 * N - 1:] = -pm["MAXTHR"]; ub[7 * N - 1:] = pm["MAXTHR"]
            x0 = np.zeros(n)
            for k in range(6):
                x0[k * N] = s6[k]
            r = scipy_opt.minimize(f, x0, jac=gf, method="SLSQP", bounds=list(zip(lb, ub)),
                                   constraints=[dict(type="eq", fun=g, jac=gj)], options=dict(maxiter=500, ftol=1e-13))
            assert r.status in (0, 8), r.message
            assert abs(r.fun - o["obj"]) <= 1e-7 * abs(o["obj"])
            np.testing.assert_allclose([r.x[6 * N], r.x[7 * N - 1]], o["u0"], atol=2e-5)


# ---------------------------------------------------------------- CPU tier: emulated kernel phases vs the oracle

def _set(pm, N, B, seed, PB=3, ncoef=4, ref_vel=False, mu=1e-3):
    return dict(pm=dict(pm, STEPS=N, BOUND=1e19), B=B, seed=seed, PB=PB, ncoef=ncoef, ref_vel=ref_vel, mu=mu)


SMALL_W = dict(YAML_DEFAULT, W_CTE=2.0, W_V=5.0, W_ANGVEL=1.0, W_A=1.0)
EMU_SETS = {
    "yaml": _set(YAML_DEFAULT, 20, 6, 91),
    "cfg-rate": _set(CFG_DEFAULT, 20, 6, 92),
    "yaml-rate": _set(dict(YAML_DEFAULT, W_DANGVEL=30.0, W_DA=5.0), 20, 5, 93),
    "small-weights": _set(SMALL_W, 20, 5, 94),
    "N3": _set(YAML_DEFAULT, 3, 5, 95),
    "N5": _set(YAML_DEFAULT, 5, 5, 96),
    "N21": _set(YAML_DEFAULT, 21, 5, 97, PB=2),
    "N100": _set(YAML_DEFAULT, 100, 2, 98, PB=2),
    "nc6": _set(YAML_DEFAULT, 20, 4, 99, ncoef=6),
    "nc8-rate": _set(CFG_DEFAULT, 20, 4, 100, ncoef=8),
    "ref-vel": _set(YAML_DEFAULT, 20, 4, 101, ref_vel=True),
    "mu1e-1": _set(YAML_DEFAULT, 20, 4, 102, mu=1e-1),
    "mu1e-6": _set(YAML_DEFAULT, 20, 4, 103, mu=1e-6),
}


def _emu_problems(s):
    if s["ncoef"] > 4:
        state, coeffs = higher_order(s["seed"], s["B"], s["ncoef"])
    else:
        state, coeffs = mild(s["seed"], s["B"])
    if s["pm"]["STEPS"] == 100:
        coeffs[2:] *= 0.1          # a sane path over a 10 s horizon (as test_emu_long_horizon)
    rv = np.linspace(0.2, 0.8, s["B"]) if s["ref_vel"] else None
    return state, coeffs, rv


def _emu(s, state, coeffs, rv, warm=None):
    if s["ncoef"] > 4:
        return emu_solve_poly(s["pm"], state, coeffs, PB=s["PB"], warm=warm, warm_mu=s["mu"])
    return emu_solve(s["pm"], state, coeffs, PB=s["PB"], ref_vel=rv, warm=warm, warm_mu=s["mu"])


@pytest.mark.parametrize("name", list(EMU_SETS))
def test_emu_warm_matches_oracle_warm(oracle, name):
    """The emulated warm kernel phases (lane_start<true>, stage_init_warm, ctrl_rollout, then the cold iteration) take the
    oracle's warm iterations from the same record bits, over every record source: same status and iteration count, u0
    to 1e-9, objective to 1e-10 relative, predicted states to 1e-8 and the whole output record to 1e-8 of its scale."""
    s = EMU_SETS[name]
    pm = s["pm"]; N = int(pm["STEPS"]); B = s["B"]
    state, coeffs, rv = _emu_problems(s)
    cold = _emu(s, state, coeffs, rv)
    assert np.all(cold["status"] == 1)
    close = lambda x, ref, tol: np.abs(x - ref).max() <= tol * max(1.0, np.abs(ref).max())  # noqa: E731
    res = {}
    for case in CASES:
        st, rec = record_case(case, cold["warm"], state, pm)
        r = res[case] = _emu(s, st, coeffs, rv, warm=rec)
        for i in range(B):
            pmi = dict(pm, REF_V=rv[i]) if rv is not None else pm
            o = oracle.solve(pmi, st[:, i], coeffs[:, i], warm=rec[:, i], warm_mu=s["mu"])
            tag = (name, case, i)
            assert r["status"][i] == o["status"], tag
            assert r["iters"][i] == o["iters"], tag + (r["iters"][i], o["iters"])
            assert np.abs(r["u0"][:, i] - o["u0"]).max() <= 1e-9, tag
            assert abs(r["obj"][i] - o["obj"]) <= 1e-10 * abs(o["obj"]), tag
            assert np.abs(r["pred"][:, i] - o["pred"].ravel()).max() <= 1e-8, tag
            out = r["warm"][:, i]
            assert close(out, record_from_oracle(o, N), 1e-8), tag
        if case in ("a", "b"):
            assert r["iters"].mean() < cold["iters"].mean(), (name, case)
    # the record's state rows are not read
    for k in ("u0", "pred", "obj", "status", "iters", "warm"):
        assert res["f"][k].tobytes() == res["a"][k].tobytes(), (name, k)


def test_emu_warm_start_lane_independence():
    """A warm-started problem's result does not depend on its lane or neighbours: a permuted batch with its records
    permuted alike gives the permuted results bit for bit (a record read by the wrong column would not)."""
    pm = dict(YAML_DEFAULT, BOUND=1e19)
    state, coeffs = mild(105, 11)
    rec = emu_solve(pm, state, coeffs, PB=4)["warm"]
    st, sh = record_case("b", rec, state, pm)
    a = emu_solve(pm, st, coeffs, PB=4, warm=sh)
    perm = np.random.default_rng(1).permutation(11)
    b = emu_solve(pm, st[:, perm], coeffs[:, perm], PB=3, warm=sh[:, perm])
    for k in ("u0", "pred", "warm"):
        assert np.array_equal(a[k][:, perm], b[k]), k
    for k in ("obj", "status", "iters"):
        assert np.array_equal(a[k][perm], b[k]), k


def _bad_rows(N):
    """(what, record row, value) of the non-finite-record cases (stage indices clipped to the horizon)"""
    n = 8 * N - 2
    lam = lambda c, k: n + c * N + min(k, N - 1)  # noqa: E731
    u, z = min(3, N - 2), min(2, N - 2)
    return [("control", 6 * N + u, np.nan), ("control", 7 * N - 1, np.inf), ("z", n + 6 * N + 2 * (N - 1) + z, np.nan),
            ("z-inf", n + 6 * N, np.inf), ("lam", lam(4, 5), np.nan), ("lam", lam(0, 0), np.nan), ("lam", lam(5, 0), np.inf),
            ("lam", lam(3, 1), np.nan), ("lam", lam(0, 1), np.nan), ("lam", lam(3, 7), np.nan), ("lam", lam(5, N - 1), np.nan)]


@pytest.mark.parametrize("N", [2, 3, 20])
def test_emu_warm_record_with_nan(oracle, N):
    """A NaN (or infinity) in one row of a record: the solve ends, and a success is a real one.  The clip of the controls
    and the floor of z absorb a NaN control or bound multiplier: the problem converges to the oracle's solution in the
    oracle's iterations.  A non-finite equality multiplier -- lambda_0, lambda_1 and the rows of the linear dynamics
    included, which enter no Newton system -- stops the first Newton step with status 10, as in the oracle; at N = 2, where
    no multiplier enters a Newton system, it ends the problem at its first evaluation with status 11 (invalid number),
    where the oracle reports 10, also at 0 iterations.  An infinite bound multiplier is reported as an invalid number (11)
    at once (the oracle's fmin / fmax drop the NaNs it makes)."""
    pm = dict(YAML_DEFAULT, STEPS=N, BOUND=1e19)
    state, coeffs = mild(107, 4)
    rec = emu_solve(pm, state, coeffs, PB=2)["warm"]
    clean = emu_solve(pm, state, coeffs, PB=2, warm=rec)
    for what, row, val in _bad_rows(N):
        bad = rec.copy(); bad[row, 1] = val
        r = emu_solve(pm, state, coeffs, PB=2, warm=bad)
        tag = (N, what, row, val, r["status"][1], r["iters"][1])
        for i in (0, 2, 3):     # the neighbours are untouched
            assert r["iters"][i] == clean["iters"][i] and np.array_equal(r["u0"][:, i], clean["u0"][:, i]), tag
        if what == "z-inf":
            assert r["status"][1] == 11 and r["iters"][1] == 0, tag
            continue
        o = oracle.solve(pm, state[:, 1], coeffs[:, 1], warm=bad[:, 1])
        if what == "lam" and N == 2:
            assert r["status"][1] == 11 and r["iters"][1] == 0 and o["status"] == 10 and o["iters"] == 0, tag
            continue
        assert r["status"][1] == o["status"] and r["iters"][1] == o["iters"], tag + (o["status"], o["iters"])
        if what in ("control", "z"):
            assert r["status"][1] == 1 and kkt_ok(oracle, pm, state[:, 1], coeffs[:, 1], o), tag
            assert np.abs(r["u0"][:, 1] - o["u0"]).max() <= 1e-9, tag
            assert np.all(np.isfinite(r["warm"][:, 1])), tag
        else:
            assert r["status"][1] == 10 and r["iters"][1] == 0, tag


# ---------------------------------------------------------------- GPU tier: the warm solve kernels vs the oracle

def _sms():
    torch = pytest.importorskip("torch")
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gpu_solver(pm, B, opts=()):
    sv = capi.Solver(capi.params_from_map(pm, capi.yaml_default_params()), B, 0)
    for k, v in dict(opts).items():
        sv.set_option(k, v)
    return sv


def _gpu_solve(sv, state, coeffs, warm_in=None):
    """one solve through the C ABI, host arrays; returns every output and the record written"""
    B = state.shape[1]; N = sv.N
    out = dict(u0=np.zeros((2, B)), pred=np.zeros((3 * N, B)), obj=np.zeros(B), status=np.zeros(B, dtype=np.int32),
               iters=np.zeros(B, dtype=np.int32), kkt=np.zeros(B), rec=np.zeros((capi.lib().mpc_b200_warm_size(N), B)))
    sv.solve_raw(B, np.ascontiguousarray(state), np.ascontiguousarray(coeffs), out["u0"], out["pred"],
                 warm_in=None if warm_in is None else np.ascontiguousarray(warm_in), obj=out["obj"], status=out["status"],
                 iters=out["iters"], kkt=out["kkt"], warm_out=out["rec"])
    return out


def _gpu_problems(seed, B, nc):
    state, c4 = mild(seed, B)
    coeffs = np.zeros((nc, B)); coeffs[:4] = c4
    if nc > 4:
        coeffs[4:] = np.random.default_rng(seed + 1000).uniform(-0.05, 0.05, size=(nc - 4, B))
    return state, coeffs


def _oracle_warm(pm, state, coeffs, rec, cols, warm_mu=1e-3):
    from tests.test_gpu_parity import _oracle_many
    return _oracle_many(dict(pm, BOUND=1e19), state[:, cols], coeffs[:, cols], warm=rec[:, cols], warm_mu=warm_mu)


def _check_against_oracle(tag, g, o, cols, bar=0.995):
    """status and iteration count equal for >= 99.5 % of the problems (98 % at N = 100, where more of the 798 relative
    step components sit at the tiny-step threshold; test_emu_second_order_correction_matches_oracle_iterates allows 97 %
    cold); on the both-converged problems with the same count,
    u0 to 1e-9 and the objective to 1e-10 relative.  The rest are knife edges of the tiny-step test: a warm start from a
    converged or shifted record takes steps of 1e-15 relative, where whether a step counts as tiny (10 machine epsilons)
    or the last iterate meets tol depends on rounding (the GPU contracts to FMA, the oracle does not).  There both must
    end at the solution (status 1, or 3 = stopped at a tiny step), with u0 to 1e-7.  Measured on a B200: 0 to 5 such
    problems per set of 148 to 5,920 at N = 20 (at most 0.17 %, narrow8-warm source (e)), 10 of 1,776 at N = 100
    (0.56 %); the printed line gives the count of each set."""
    st, it = g["status"][cols], g["iters"][cols]
    same = (st == o["status"]) & (it == o["iters"])
    print("warm vs oracle %s: %d of %d problems differ in status or iterations" % (tag, int((~same).sum()), len(cols)))
    assert same.mean() >= bar, (tag, np.flatnonzero(~same)[:8], st[~same][:8], o["status"][~same][:8], it[~same][:8],
                                  o["iters"][~same][:8])
    edge = ~same
    assert np.isin(st[edge], (1, 3)).all() and np.isin(o["status"][edge], (1, 3)).all(), tag
    np.testing.assert_allclose(g["u0"][:, cols][:, edge], o["u0"][:, edge], rtol=0, atol=1e-7, err_msg=tag + " knife edges")
    ok = same & (st == 1)
    assert ok.mean() >= 0.99, tag
    np.testing.assert_allclose(g["u0"][:, cols][:, ok], o["u0"][:, ok], rtol=0, atol=1e-9, err_msg=tag)
    np.testing.assert_allclose(g["obj"][cols][ok], o["obj"][ok], rtol=1e-10, atol=0, err_msg=tag)


def _warm_rows():
    from tests.test_kernel_choice import ROWS
    return [r for r in ROWS if r[5]]


@pytest.mark.gpu
@pytest.mark.parametrize("row", _warm_rows(), ids=[r[0] for r in _warm_rows()])
def test_warm_kernels_match_oracle_warm(row):
    """Every warm specialisation of the solve kernels (the warm rows of test_kernel_choice, same batch sizes and options,
    so the same kernel runs; max_iter at its default) takes the oracle's warm iterations: a cold solve writes the records,
    then the moved states of one closed-loop tick are solved from the shifted records (source (b)) and compared with the
    oracle's warm start from the same record bits, on every problem."""
    name, weights, N, per_sm, opts, _, _, _ = row
    B = per_sm * _sms()
    pm = dict(weights, STEPS=N)
    nc = int(opts.get("poly_coeffs", 4))
    sv = _gpu_solver(pm, B, opts)
    state, coeffs = _gpu_problems(11, B, nc)
    cold = _gpu_solve(sv, state, coeffs)
    assert (cold["status"] == 1).mean() >= 0.99
    st, rec = record_case("b", cold["rec"], state, pm)
    g = _gpu_solve(sv, st, coeffs, warm_in=rec)
    sv.close()
    assert g["iters"].mean() < cold["iters"].mean()
    cols = np.arange(B)
    _check_against_oracle(name, g, _oracle_warm(pm, st, coeffs, rec, cols), cols, bar=0.98 if N >= 100 else 0.995)


@pytest.mark.gpu
def test_warm_records_follow_hard_first_order():
    """With more problems than the grid has lanes, queue_order_kernel hands them out hardest first; each problem must
    still read its own record column.  Warm results with hard_first 1 and 0 are bit-identical, a permuted batch (states,
    coefficients and record columns permuted together) returns the permuted results bit for bit, and the iteration counts
    are the oracle's."""
    pm = dict(YAML_DEFAULT, STEPS=20)
    B = 3000
    opts = dict(max_ctas=4, problems_per_cta=32)          # 128 lanes: the queue is ordered
    state, coeffs = _gpu_problems(13, B, 4)
    sv = _gpu_solver(pm, B, dict(opts, hard_first=1))
    cold = _gpu_solve(sv, state, coeffs)
    st, rec = record_case("b", cold["rec"], state, pm)
    ordered = _gpu_solve(sv, st, coeffs, warm_in=rec)
    perm = np.random.default_rng(2).permutation(B)
    permuted = _gpu_solve(sv, st[:, perm], coeffs[:, perm], warm_in=rec[:, perm])
    sv.close()
    sv = _gpu_solver(pm, B, dict(opts, hard_first=0))
    plain = _gpu_solve(sv, st, coeffs, warm_in=rec)
    sv.close()
    for k in ("u0", "pred", "obj", "status", "iters", "kkt", "rec"):
        assert ordered[k].tobytes() == plain[k].tobytes(), k
        assert ordered[k][..., perm].tobytes() == permuted[k].tobytes(), k
    cols = np.arange(B)
    _check_against_oracle("hard-first", ordered, _oracle_warm(pm, st, coeffs, rec, cols), cols)


@pytest.mark.gpu
@pytest.mark.parametrize("row", ["yaml-full-warm", "narrow8-warm"])
def test_warm_record_sources_on_gpu(row):
    """Record sources (a) and (c)-(f) in the dual-group kernel and in a one-stage narrow kernel: the oracle's iterations
    from a poor start, from controls on and beyond the bounds and from zero multipliers; (f) is bit-identical to (a)."""
    from tests.test_kernel_choice import ROWS
    _, weights, N, per_sm, opts, _, _, _ = [r for r in ROWS if r[0] == row][0]
    B = per_sm * _sms()
    pm = dict(weights, STEPS=N)
    sv = _gpu_solver(pm, B, opts)
    state, coeffs = _gpu_problems(17, B, 4)
    cold = _gpu_solve(sv, state, coeffs)
    res = {}
    cols = np.arange(B)
    for case in ("a", "c", "d", "e", "f"):
        st, rec = record_case(case, cold["rec"], state, pm)
        res[case] = _gpu_solve(sv, st, coeffs, warm_in=rec)
        if case != "f":
            _check_against_oracle(row + " " + case, res[case], _oracle_warm(pm, st, coeffs, rec, cols), cols)
    sv.close()
    for k in ("u0", "pred", "obj", "status", "iters", "kkt", "rec"):
        assert res["f"][k].tobytes() == res["a"][k].tobytes(), k


@pytest.mark.gpu
def test_warm_shift_kernel_matches_numpy():
    """mpc_b200_warm_shift against the numpy restatement, bit for bit, at horizons 3 / 20 / 100 and batches around the
    kernel's block of 128; aliased buffers, host buffers and an empty batch are refused or do nothing."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(5)
    for N in (3, 20, 100):
        ws = capi.lib().mpc_b200_warm_size(N)
        assert sum(blocks(N)) == ws
        sv = _gpu_solver(dict(YAML_DEFAULT, STEPS=N), 5000)
        for B in (1, 127, 128, 129, 5000):
            prev = rng.normal(size=(ws, B))
            d_prev = torch.from_numpy(prev).to(dev)
            d_next = torch.full((ws, B), float("nan"), dtype=torch.float64, device=dev)
            sv.warm_shift(B, d_prev, d_next)
            torch.cuda.synchronize()
            assert d_next.cpu().numpy().tobytes() == shift(prev, N).tobytes(), (N, B)
            assert d_prev.cpu().numpy().tobytes() == prev.tobytes(), (N, B)
        with pytest.raises(capi.MpcError) as e:
            sv.warm_shift(B, d_prev, d_prev)
        assert e.value.code == -1
        with pytest.raises(capi.MpcError) as e:
            sv.warm_shift(B, prev, np.zeros_like(prev))
        assert e.value.code == -3
        before = d_next.cpu().numpy().copy()
        sv.warm_shift(0, d_prev, d_next)
        torch.cuda.synchronize()
        assert d_next.cpu().numpy().tobytes() == before.tobytes()
        sv.close()


@pytest.mark.gpu
def test_warm_record_with_nan_on_gpu(oracle):
    """The non-finite record rows of test_emu_warm_record_with_nan, one per problem of one one-stage narrow solve: the call
    returns, the other problems are unaffected, and each status and iteration count is the emulated kernel's (which
    test_emu_warm_record_with_nan checks against the oracle)."""
    pm = dict(YAML_DEFAULT, STEPS=20)
    N = 20; rows = _bad_rows(N); B = 16
    state, coeffs = _gpu_problems(107, B, 4)
    sv = _gpu_solver(pm, B)
    cold = _gpu_solve(sv, state, coeffs)
    clean = _gpu_solve(sv, state, coeffs, warm_in=cold["rec"])
    bad = cold["rec"].copy()
    for j, (_, row, val) in enumerate(rows):
        bad[row, j] = val
    g = _gpu_solve(sv, state, coeffs, warm_in=bad)
    sv.close()
    e = emu_solve(dict(pm, BOUND=1e19), state, coeffs, PB=4, max_iter=100, warm=bad)
    assert np.array_equal(g["status"], e["status"]) and np.array_equal(g["iters"], e["iters"])
    for j, (what, _, _) in enumerate(rows):
        assert g["status"][j] == {"control": 1, "z": 1, "z-inf": 11}.get(what, 10), (j, what)
    rest = np.arange(len(rows), B)
    assert np.array_equal(g["iters"][rest], clean["iters"][rest]) and np.all(g["status"][rest] == 1)
    assert np.abs(g["u0"][:, rest] - clean["u0"][:, rest]).max() <= 1e-9
