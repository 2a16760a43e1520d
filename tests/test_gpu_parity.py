"""GPU tier: the CUDA path, called through the C ABI (include/mpc_b200.h), against the oracle.

Tolerances are the north-star's: first-step controls within 1e-5 absolute, objective within 1e-6
relative, scaled KKT residual <= Ipopt's tol 1e-8."""
import json
import os

import numpy as np
import pytest

from mpc_ros_b200 import capi
from oracle.oracle_py import YAML_DEFAULT, CFG_DEFAULT
from tests.problems import mild, generated, restoration_cases

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

U_TOL = 1e-5      # north-star: first-step controls, absolute
F_TOL = 1e-6      # north-star: objective, relative
KKT_TOL = 1e-8    # Ipopt tol (scaled optimality error E_0)


def _solver(pm, max_batch):
    return capi.Solver(capi.params_from_map(pm, capi.yaml_default_params()), max_batch, 0)


def test_library_is_the_cuda_path():
    assert capi.lib().mpc_b200_device_count() >= 1
    s = _solver(YAML_DEFAULT, 4)
    state, coeffs = mild(1, 4)
    n0 = s.launch_count
    out = s.solve(state, coeffs)
    assert s.launch_count == n0 + 1 and s.last_kernel_seconds > 0.0
    assert np.all(out["status"] == 1)
    s.close()


def test_golden_solutions():
    """Committed reference MPC::Solve outputs (tests/golden/solve_golden.json)."""
    sols = json.load(open(os.path.join(GOLD, "solve_golden.json")))
    groups = {}
    for s in sols:
        groups.setdefault(json.dumps(s["params"], sort_keys=True), []).append(s)
    for key, grp in groups.items():
        pm = json.loads(key)
        B = len(grp)
        state = np.array([g["state"] for g in grp]).T.copy(); coeffs = np.array([g["coeffs"] for g in grp]).T.copy()
        sv = _solver(pm, B)
        out = sv.solve(state, coeffs)
        sv.close()
        N = int(pm["STEPS"])
        for i, g in enumerate(grp):
            assert out["status"][i] == 1 == g["status"]
            assert np.abs(out["u0"][:, i] - g["u0"]).max() <= U_TOL
            assert abs(out["obj"][i] - g["obj"]) <= F_TOL * abs(g["obj"])
            assert out["kkt"][i] <= KKT_TOL
            assert np.abs(out["pred"][:, i].reshape(3, N) - np.array(g["pred"])).max() <= 1e-5


def test_matches_oracle_mild(oracle):
    state, coeffs = mild(31, 96)
    sv = _solver(YAML_DEFAULT, 96)
    out = sv.solve(state, coeffs)
    sv.close()
    nobound = dict(YAML_DEFAULT, BOUND=1e19)
    for i in range(96):
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        assert out["status"][i] == 1 and o["status"] == 1
        assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
        assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
        assert out["kkt"][i] <= KKT_TOL
        if i < 24:
            o2 = oracle.solve(nobound, state[:, i], coeffs[:, i])
            assert out["iters"][i] == o2["iters"]          # same algorithm, same path
            assert np.abs(out["u0"][:, i] - o2["u0"]).max() <= 1e-9


def test_matches_oracle_generated(oracle):
    """BASELINE config 2's generator at a size the oracle finishes in seconds."""
    g, state, coeffs = generated(20261018 + 2, 384, oracle)
    sv = _solver(YAML_DEFAULT, 384)
    out = sv.solve(state, coeffs)
    sv.close()
    both = close = 0
    for i in range(384):
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        if o["status"] == 1 and out["status"][i] == 1:
            both += 1
            ok = np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL and abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
            close += bool(ok)
    assert both >= 380
    assert close >= both - 2       # non-convex corner windows may settle in another local minimum


def test_prestep_kernel_matches_oracle(oracle):
    """K1: transform + polyfit + (cte, etheta) vs driving_state.cpp:196-235 restated in the oracle."""
    from bench import gen_py
    B = 300
    g = gen_py.problems(77, B)
    sv = _solver(YAML_DEFAULT, B)
    coeffs, cte, eth = sv.polyfit(g["wx"], g["wy"], g["pose"])
    sv.close()
    for i in range(B):
        c, ct, e = oracle.prestep(g["wx"][:, i], g["wy"][:, i], *g["pose"][:, i])
        scale = max(1.0, np.abs(c).max())
        assert np.abs(coeffs[:, i] - c).max() <= 1e-9 * scale
        assert abs(cte[i] - ct) <= 1e-9 * scale
        assert abs(eth[i] - e) <= 1e-12


def test_prestep_axis_aligned_quirk(oracle):
    wx = np.tile((np.arange(11) * 0.5)[:, None], (1, 3)); wy = np.zeros((11, 3))
    pose = np.array([[0.0, 0.0, 0.0], [0.2, -0.1, 0.0], [0.3, 0.1, -0.2]]).T.copy()
    sv = _solver(YAML_DEFAULT, 3)
    coeffs, cte, eth = sv.polyfit(wx, wy, pose)
    sv.close()
    assert np.all(eth == 0.0)      # gy == 0 exactly -> etheta forced to 0 (driving_state.cpp:232)


def test_full_size_properties(oracle):
    """BASELINE config 2 at full size (4,096): size-independent properties."""
    B = 4096
    g, state, coeffs = generated(20261018 + 2, B, oracle)
    sv = _solver(YAML_DEFAULT, B)
    a = sv.solve(state, coeffs)
    b = sv.solve(state, coeffs)
    perm = np.random.default_rng(5).permutation(B)
    c = sv.solve(state[:, perm].copy(), coeffs[:, perm].copy())
    sv.close()
    conv = a["status"] == 1
    assert conv.mean() >= 0.995
    assert np.all(a["kkt"][conv] <= KKT_TOL)
    # determinism and independence from the lane / CTA a problem lands in
    for k in ("u0", "pred", "obj", "kkt"):
        np.testing.assert_array_equal(a[k], b[k])
    np.testing.assert_array_equal(a["u0"][:, perm], c["u0"])
    np.testing.assert_array_equal(a["iters"][perm], c["iters"])
    # bounds respected (relaxed by Ipopt's 1e-8 factor)
    assert np.all(np.abs(a["u0"][0, conv]) <= 1.5 * (1 + 2e-8))
    assert np.all(np.abs(a["u0"][1, conv]) <= 1.0 * (1 + 2e-8))
    # predicted trajectory satisfies the model: theta_{k+1} = theta_k + w_k dt can be checked on stage 0
    N = 20
    th = a["pred"][2 * N:3 * N]
    assert np.all(np.abs(th[1, conv] - (th[0, conv] + a["u0"][0, conv] * 0.1)) <= 1e-7)
    # a random sample against the oracle
    idx = np.random.default_rng(6).choice(B, 64, replace=False)
    ok = 0
    for i in idx:
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        if o["status"] == 1 and a["status"][i] == 1:
            ok += np.abs(a["u0"][:, i] - o["u0"]).max() <= U_TOL and abs(a["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
    assert ok >= 62


def test_device_pointers_and_ref_vel(oracle):
    torch = pytest.importorskip("torch")
    state, coeffs = mild(41, 40)
    rv = np.linspace(0.1, 0.9, 40)
    sv = _solver(YAML_DEFAULT, 40)
    host = sv.solve(state, coeffs, ref_vel=rv)
    dev = torch.device("cuda:0")
    ds = torch.from_numpy(state).to(dev); dc = torch.from_numpy(coeffs).to(dev); dr = torch.from_numpy(rv).to(dev)
    du0 = torch.zeros((2, 40), dtype=torch.float64, device=dev); dpred = torch.zeros((60, 40), dtype=torch.float64, device=dev)
    dst = torch.zeros(40, dtype=torch.int32, device=dev)
    sv.solve_raw(40, ds, dc, du0, dpred, ref_vel=dr, status=dst)
    torch.cuda.synchronize()
    sv.close()
    np.testing.assert_array_equal(du0.cpu().numpy(), host["u0"])
    np.testing.assert_array_equal(dpred.cpu().numpy(), host["pred"])
    for i in range(0, 40, 5):
        o = oracle.solve(dict(YAML_DEFAULT, REF_V=float(rv[i])), state[:, i], coeffs[:, i])
        assert np.abs(host["u0"][:, i] - o["u0"]).max() <= U_TOL


def test_cfg_weights(oracle):
    pm = dict(CFG_DEFAULT, W_DA=0.0)
    state, coeffs = mild(42, 32)
    sv = _solver(pm, 32)
    out = sv.solve(state, coeffs)
    sv.close()
    for i in range(32):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert out["status"][i] == 1 and o["status"] == 1
        assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
        assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])


def test_rate_penalties_cfg_defaults(oracle):
    """The reference's dynamic_reconfigure defaults (MPCPlanner.cfg:22-37) include w_accel_d = 10: the rate
    terms couple u_k and u_{k+1} (mpc_planner.cpp:144-147) and run through the augmented Riccati variant."""
    for pm, seed in ((dict(CFG_DEFAULT), 45), (dict(YAML_DEFAULT, W_DANGVEL=30.0, W_DA=5.0), 46)):
        state, coeffs = mild(seed, 48)
        sv = _solver(pm, 48)
        out = sv.solve(state, coeffs)
        sv.close()
        for i in range(48):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert out["status"][i] == 1 and o["status"] == 1
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
            assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
            assert out["kkt"][i] <= KKT_TOL


def test_long_horizon(oracle):
    """BASELINE config 4 (N = 100) on a small batch."""
    pm = dict(YAML_DEFAULT, STEPS=100)
    state, coeffs = mild(43, 12)
    coeffs[2:] *= 0.1
    sv = _solver(pm, 12)
    out = sv.solve(state, coeffs)
    sv.close()
    for i in range(12):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert out["status"][i] == 1 and o["status"] == 1
        assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
        assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])


def test_edge_cases():
    sv = _solver(YAML_DEFAULT, 8)
    # empty batch is a no-op
    z = np.zeros((6, 0)); c = np.zeros((4, 0))
    sv.solve_raw(0, z, c, np.zeros((2, 0)), np.zeros((60, 0)))
    # batch of one; batch above max_batch is refused
    state, coeffs = mild(44, 9)
    one = sv.solve(state[:, :1].copy(), coeffs[:, :1].copy())
    assert one["status"][0] == 1
    with pytest.raises(capi.MpcError):
        sv.solve(state, coeffs)
    # a problem already at the reference needs (almost) no control
    st = np.zeros((6, 1)); st[3] = 0.5
    out = sv.solve(st, np.zeros((4, 1)))
    assert out["status"][0] == 1 and np.abs(out["u0"]).max() <= 1e-6
    # NaN input: reported, not hung
    st[4] = np.nan
    out = sv.solve(st, np.zeros((4, 1)))
    assert out["status"][0] != 1
    sv.close()


def test_warm_start_reaches_the_same_solution(oracle):
    """Warm start (new capability): re-solving from a converged record gives the same KKT point in far
    fewer iterations; a shifted record of a neighbouring problem still converges to the oracle's answer."""
    torch = pytest.importorskip("torch")
    state, coeffs = mild(51, 64)
    B = 64; N = 20
    dev = torch.device("cuda:0")
    sv = _solver(YAML_DEFAULT, B)
    ws = capi.lib().mpc_b200_warm_size(N)
    f64 = dict(dtype=torch.float64, device=dev)
    ds = torch.from_numpy(state).to(dev); dc = torch.from_numpy(coeffs).to(dev)
    u_cold = torch.zeros((2, B), **f64); pred = torch.zeros((3 * N, B), **f64)
    it_cold = torch.zeros(B, dtype=torch.int32, device=dev); st = torch.zeros(B, dtype=torch.int32, device=dev)
    wo = torch.zeros((ws, B), **f64)
    sv.solve_raw(B, ds, dc, u_cold, pred, status=st, iters=it_cold, warm_out=wo)
    torch.cuda.synchronize()
    assert bool((st == 1).all())
    # the record's primal block is the solution in the reference's variable layout
    rec = wo.cpu().numpy()
    np.testing.assert_allclose(rec[6 * N], u_cold.cpu().numpy()[0], atol=0)         # w_0
    np.testing.assert_allclose(rec[7 * N - 1], u_cold.cpu().numpy()[1], atol=0)     # a_0
    np.testing.assert_allclose(rec[:N], pred.cpu().numpy()[:N], atol=0)             # x_k
    # (a) same problem, warm: same answer, fewer iterations
    u_w = torch.zeros((2, B), **f64); it_w = torch.zeros(B, dtype=torch.int32, device=dev)
    sv.solve_raw(B, ds, dc, u_w, pred, warm_in=wo, status=st, iters=it_w)
    torch.cuda.synchronize()
    assert bool((st == 1).all())
    assert float((u_w - u_cold).abs().max()) <= U_TOL
    assert float(it_w.double().mean()) <= 0.7 * float(it_cold.double().mean())
    # (b) perturbed problem warm-started from the shifted record: still the oracle's solution
    state2 = state.copy(); state2[3] += 0.03; state2[4] += 0.02; state2[5] -= 0.03
    ds2 = torch.from_numpy(state2).to(dev)
    wsft = torch.zeros((ws, B), **f64)
    sv.warm_shift(B, wo, wsft)
    sv.solve_raw(B, ds2, dc, u_w, pred, warm_in=wsft, status=st, iters=it_w)
    torch.cuda.synchronize()
    sv.close()
    uw = u_w.cpu().numpy()
    assert bool((st == 1).all())
    for i in range(0, B, 4):
        o = oracle.solve(YAML_DEFAULT, state2[:, i], coeffs[:, i])
        assert np.abs(uw[:, i] - o["u0"]).max() <= U_TOL


def test_closed_loop_tracks_like_the_reference_loop():
    """BASELINE config 5 in small: warm-started GPU loop vs the cold-started oracle loop (the reference
    cold-starts every tick), same robots, same plant."""
    from bench import closed_loop
    from tests.closed_loop_ref import run_oracle
    R, T = 12, 40
    g = closed_loop.run_gpu(R, T, warm=True)
    o = run_oracle(R, T)
    assert g["conv"].mean() >= 0.99
    # same commands tick by tick while the two loops see the same states (they do until round-off grows)
    assert np.abs(g["w"][:5] - o["w"][:5]).max() <= 1e-4
    assert np.abs(g["thr"][:5] - o["thr"][:5]).max() <= 1e-4
    # and the same tracking quality over the run
    assert abs(np.abs(g["cte"]).mean() - np.abs(o["cte"]).mean()) <= 0.01
    # (the reference's own trace, assets/mpc.csv, has mean |cte| 0.05 m on an unknown path with unknown parameters; with the
    #  mpc_params.yaml weights on these tracks the reference LOOP itself settles at 0.13 .. 0.15 m: DESIGN section "config 5")
    assert abs(np.abs(g["cte"][-10:]).mean() - np.abs(o["cte"][-10:]).mean()) <= 0.02
    assert np.abs(g["cte"][-10:]).mean() <= 0.2
    assert g["iters"][1:].mean() < o["iters"][1:].mean()  # warm start pays


def test_device_resident_loop_matches_host_loop():
    """SURVEY 8f-1 / 8f-2: windowing (mpc_planner_ros.cpp:266-291, :365-391) and post-step
    (driving_state.cpp:263-269) as kernels; the device-resident loop tracks like the host-driven one."""
    from bench import closed_loop
    R, T = 24, 30
    h = closed_loop.run_gpu(R, T, warm=True)
    d = closed_loop.run_gpu_device(R, T, groups=3)
    assert d["conv"].mean() >= 0.99
    # same robots, same rule for the cut, same solver: identical tracking errors while round-off has not diverged
    assert np.abs(d["cte"][:3] - h["cte"][:3]).max() <= 1e-6
    assert abs(np.median(np.abs(d["cte"])) - np.median(np.abs(h["cte"]))) <= 0.01


def test_all_kernel_specialisations_agree(oracle):
    """Every lanes-per-CTA specialisation (compile-time 1/4/8/16/32 and the run-time generic path), with and
    without queue refill and hard-first ordering, returns the same results: same status and iteration
    counts, values equal to rounding (the instantiations are separate compilations: FMA contraction may
    differ; a given configuration is bit-reproducible, see test_full_size_properties)."""
    g, state, coeffs = generated(20261018 + 3, 600, oracle)
    ref = None
    for pb, ctas, hard in ((32, 0, 1), (32, 2, 1), (32, 2, 0), (16, 0, 1), (8, 3, 1), (4, 0, 1), (1, 0, 1), (7, 5, 1), (28, 1, 0)):
        sv = _solver(YAML_DEFAULT, 600)
        sv.set_option("problems_per_cta", pb); sv.set_option("max_ctas", ctas); sv.set_option("hard_first", hard)
        out = sv.solve(state, coeffs)
        sv.close()
        if ref is None:
            ref = out
            assert (out["status"] == 1).mean() >= 0.99
        else:
            tag = "pb=%d ctas=%d hard=%d " % (pb, ctas, hard)
            same = (out["status"] == ref["status"]) & (out["iters"] == ref["iters"])
            assert same.mean() >= 0.995, tag          # a knife-edge line-search decision may flip on a hard problem
            ok = same & (ref["status"] == 1)
            np.testing.assert_allclose(out["u0"][:, ok], ref["u0"][:, ok], rtol=0, atol=1e-9, err_msg=tag + "u0")
            np.testing.assert_allclose(out["pred"][:, ok], ref["pred"][:, ok], rtol=0, atol=1e-8, err_msg=tag + "pred")
            np.testing.assert_allclose(out["obj"][ok], ref["obj"][ok], rtol=1e-10, err_msg=tag + "obj")


def test_dual_group_kernel_equals_single_group_kernel(oracle):
    """Full CTAs of the plain variant run as two groups of 16 lanes out of phase (nmpc_kernel_dual.cuh, one stage per
    stage thread and group; option dual_groups).  Same phase functions, partial sums added in the same order: status
    and iteration counts are identical to the single-group kernel's, controls and predicted states equal to rounding, cold and warm, for
    even and odd horizons (an odd horizon leaves the upper half of the last stage warp without a stage)."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    g, state, coeffs = generated(20261018 + 3, 4500, oracle)
    B = state.shape[1]
    for base, N, lanes in ((YAML_DEFAULT, 20, 32), (YAML_DEFAULT, 15, 32), (YAML_DEFAULT, 11, 32), (CFG_DEFAULT, 20, 28)):
        # (the last one: the rate-penalty variant, 28 lanes per CTA = a group of 16 and a group of 12)
        pm = dict(base, STEPS=N)
        res = {}
        for dual in (1, 0):
            sv = _solver(pm, B)
            sv.set_option("dual_groups", dual); sv.set_option("problems_per_cta", lanes); sv.set_option("max_ctas", 6)
            ws = capi.lib().mpc_b200_warm_size(N)
            f64 = dict(dtype=torch.float64, device=dev)
            ds = torch.from_numpy(state).to(dev); dc = torch.from_numpy(coeffs).to(dev)
            u = torch.zeros((2, B), **f64); pred = torch.zeros((3 * N, B), **f64); wo = torch.zeros((ws, B), **f64)
            st = torch.zeros(B, dtype=torch.int32, device=dev); it = torch.zeros(B, dtype=torch.int32, device=dev)
            sv.solve_raw(B, ds, dc, u, pred, status=st, iters=it, warm_out=wo)
            torch.cuda.synchronize()
            cold = (u.cpu().numpy().copy(), pred.cpu().numpy().copy(), st.cpu().numpy().copy(), it.cpu().numpy().copy(), wo.cpu().numpy().copy())
            # warm re-solve of a slightly moved problem from the cold record
            ds2 = ds.clone(); ds2[3] += 0.02; ds2[4] -= 0.01
            sv.solve_raw(B, ds2, dc, u, pred, warm_in=wo, status=st, iters=it)
            torch.cuda.synchronize()
            warm = (u.cpu().numpy().copy(), pred.cpu().numpy().copy(), st.cpu().numpy().copy(), it.cpu().numpy().copy())
            sv.close()
            res[dual] = (cold, warm)
        tag = "N=%d lanes=%d " % (N, lanes)
        assert (res[1][0][2] == 1).mean() >= 0.99, tag
        for which in (0, 1):
            a, b = res[1][which], res[0][which]
            assert np.array_equal(a[2], b[2]), tag + "status"
            assert np.array_equal(a[3], b[3]), tag + "iterations"
            # (values equal to rounding: the two kernels are separate compilations of the same phase functions, FMA
            #  contraction may differ -- as between the lanes-per-CTA specialisations)
            ok = a[2] == 1
            np.testing.assert_allclose(a[0][:, ok], b[0][:, ok], rtol=0, atol=1e-9, err_msg=tag + "u0")
            np.testing.assert_allclose(a[1][:, ok], b[1][:, ok], rtol=0, atol=1e-8, err_msg=tag + "pred")
        okc = res[1][0][2] == 1
        np.testing.assert_allclose(res[1][0][4][:, okc], res[0][0][4][:, okc], rtol=1e-7, atol=1e-8, err_msg=tag + "warm record")
        # and both are the oracle's answer
        for i in range(0, B, 450):
            if res[1][0][2][i] != 1:
                continue
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            if o["status"] == 1:
                assert np.abs(res[1][0][0][:, i] - o["u0"]).max() <= U_TOL, tag


def test_restoration_phase(oracle):
    """The same on the GPU, in a full CTA of the dual-group kernel (the cases are mixed into a batch of ordinary problems)
    and in the single-solve kernel."""
    rs, rc = restoration_cases(oracle)
    g, state, coeffs = generated(20261018 + 2, 40, oracle)
    nr = rs.shape[1]
    st = np.concatenate([state, rs], axis=1); co = np.concatenate([coeffs, rc], axis=1)
    opt = oracle.default_options(); opt.max_iter = 100
    for pb in (32, 1):
        sv = _solver(YAML_DEFAULT, st.shape[1])
        sv.set_option("problems_per_cta", pb)
        out = sv.solve(st, co)
        sv.close()
        for j in range(nr):
            i = 40 + j
            o = oracle.solve(YAML_DEFAULT, rs[:, j], rc[:, j], opt)
            assert out["status"][i] == o["status"], (pb, j, out["status"][i], o["status"])
            if o["status"] == 1:
                assert out["iters"][i] == o["iters"]
                assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
                assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
                assert out["kkt"][i] <= KKT_TOL


def test_kernel_choice_options():
    """The launch-shaping options are accepted by name, unknown names refused; the latency mode (one stage per stage thread in
    narrow CTAs) returns what the two-stage kernels return."""
    state, coeffs = mild(77, 96)
    res = {}
    for one in (1, 0):
        sv = _solver(YAML_DEFAULT, 96)
        for name in ("dual_groups", "narrow_one_stage", "hard_first", "max_ctas", "problems_per_cta"):
            sv.set_option(name, 1 if name != "max_ctas" else 0)
        sv.set_option("problems_per_cta", 0); sv.set_option("narrow_one_stage", one)
        with pytest.raises(capi.MpcError):
            sv.set_option("no_such_option", 1)
        res[one] = sv.solve(state, coeffs)
        sv.close()
    assert np.all(res[1]["status"] == 1) and np.array_equal(res[1]["status"], res[0]["status"])
    assert np.array_equal(res[1]["iters"], res[0]["iters"])
    np.testing.assert_allclose(res[1]["u0"], res[0]["u0"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(res[1]["pred"], res[0]["pred"], rtol=0, atol=1e-8)


def test_prestep_ragged_windows_and_delay_mode(oracle):
    """K1 at the edges: the shortest (M = 4: cubic through 4 points) and longest (M = 64) windows, refused
    sizes, and the delay-compensated state of driving_state.cpp:243-254."""
    rng = np.random.default_rng(3)
    for M in (4, 7, 64):
        B = 33
        wx = np.cumsum(rng.uniform(0.05, 0.6, (M, B)), axis=0); wy = 0.3 * np.sin(wx) + rng.normal(0, 0.01, (M, B))
        pose = np.stack([rng.uniform(-0.2, 0.2, B), rng.uniform(-0.2, 0.2, B), rng.uniform(-0.4, 0.4, B)])
        vel = np.stack([rng.uniform(0, 0.6, B), rng.uniform(-0.5, 0.5, B), rng.uniform(-0.5, 0.5, B)])
        for delay in (0, 1):
            prm = capi.yaml_default_params(); prm.delay_mode = delay
            sv = capi.Solver(prm, B, 0)
            coeffs, state = sv.prestep(wx, wy, pose, vel)
            sv.close()
            for i in range(B):
                c, cte, eth = oracle.prestep(wx[:, i], wy[:, i], *pose[:, i])
                scale = max(1.0, np.abs(c).max())
                assert np.abs(coeffs[:, i] - c).max() <= 1e-8 * scale
                v, w, thr = vel[:, i]
                dt = prm.dt
                exp = [v * dt, 0.0, w * dt, v + thr * dt, cte + v * np.sin(eth) * dt, eth - w * dt] if delay else [0, 0, 0, v, cte, eth]
                assert np.abs(state[:, i] - np.array(exp)).max() <= 1e-8 * scale
    sv = capi.Solver(capi.yaml_default_params(), 4, 0)
    for M in (3, 65):
        with pytest.raises(capi.MpcError):
            sv.polyfit(np.zeros((M, 4)), np.zeros((M, 4)), np.zeros((3, 4)))
    # degenerate window (all waypoints identical): NaN coefficients, reported, no hang
    coeffs, cte, eth = sv.polyfit(np.zeros((11, 4)), np.zeros((11, 4)), np.zeros((3, 4)))
    assert np.all(np.isnan(coeffs)) or np.all(np.isfinite(coeffs))
    sv.close()


def test_track_batch_equals_prestep_solve_poststep(oracle):
    """mpc_b200_track_batch (the whole findBestPath tick, driving_state.cpp:175-271) must give exactly what
    the three separate calls give, with and without delay compensation and per-robot reference speeds."""
    from bench import gen_py
    B = 777
    g = gen_py.problems(4242, B)
    rng = np.random.default_rng(9)
    for delay, per_robot in ((0, False), (1, True)):
        prm = capi.yaml_default_params(); prm.delay_mode = delay
        vel = g["vel"].copy()
        vel[1] = rng.uniform(-0.5, 0.5, B); vel[2] = rng.uniform(-0.5, 0.5, B)
        refv = rng.uniform(0.3, 1.0, B) if per_robot else None
        sv = capi.Solver(prm, B, 0)
        coeffs, state = sv.prestep(g["wx"], g["wy"], g["pose"], vel)
        a = sv.solve(state, coeffs, ref_vel=refv)
        v2 = vel.copy()
        b = sv.track(g["wx"], g["wy"], g["pose"], v2, ref_vel=refv)
        sv.close()
        for k in ("u0", "pred", "obj", "kkt", "status", "iters"):
            np.testing.assert_array_equal(a[k], b[k])
        # post-step (driving_state.cpp:263-269): speed clamped above at the reference speed only
        rv = refv if per_robot else np.full(B, prm.ref_vel)
        speed = np.minimum(vel[0] + a["u0"][1] * prm.dt, rv)
        np.testing.assert_allclose(b["cmd"][0], speed, rtol=0, atol=1e-15)   # v + thr*dt is one FMA on the device
        np.testing.assert_array_equal(b["cmd"][1], a["u0"][0])
        np.testing.assert_array_equal(v2[0], vel[0])
        np.testing.assert_array_equal(v2[1], a["u0"][0])
        np.testing.assert_array_equal(v2[2], a["u0"][1])
        # the oracle's own pre-step + solve on a few of them
        for i in range(0, B, 97):
            c, ct, e = oracle.prestep(g["wx"][:, i], g["wy"][:, i], *g["pose"][:, i])
            assert np.abs(coeffs[:, i] - c).max() <= 1e-9 * max(1.0, np.abs(c).max())


def test_track_submit_wait_pipelined():
    """Two handles with a tick in flight each give the results of the synchronous call; a second submit on a
    busy handle is refused."""
    from bench import gen_py
    B = 512
    N = 20
    g = [gen_py.problems(900 + k, B) for k in range(2)]
    prm = capi.yaml_default_params()
    ref = []
    sv = capi.Solver(prm, B, 0)
    for k in range(2):
        ref.append(sv.track(g[k]["wx"], g[k]["wy"], g[k]["pose"], g[k]["vel"].copy()))
    sv.close()
    hs = [capi.Solver(prm, B, 0) for _ in range(2)]
    outs = []
    for k in range(2):
        o = dict(u0=np.zeros((2, B)), pred=np.zeros((3 * N, B)), cmd=np.zeros((2, B)), status=np.zeros(B, dtype=np.int32),
                 vel=g[k]["vel"].copy())
        M = g[k]["wx"].shape[0]
        hs[k].track_submit_raw(B, M, g[k]["wx"], g[k]["wy"], g[k]["pose"], o["vel"], o["u0"], o["pred"], cmd=o["cmd"],
                               status=o["status"])
        outs.append(o)
    with pytest.raises(capi.MpcError):
        hs[0].track_submit_raw(B, M, g[0]["wx"], g[0]["wy"], g[0]["pose"], outs[0]["vel"], outs[0]["u0"], outs[0]["pred"])
    for k in (1, 0):
        hs[k].track_wait()
        hs[k].track_wait()          # idempotent
        for key in ("u0", "pred", "cmd", "status"):
            np.testing.assert_array_equal(outs[k][key], ref[k][key])
        hs[k].close()


def test_decel_and_plant_kernels(oracle):
    """8f-1: the REF_V schedule near the goal (driving_state.cpp:121-141) against the oracle, and the plant step."""
    import torch
    B = 5000
    rng = np.random.default_rng(31)
    prm = capi.yaml_default_params()
    pose = np.vstack([rng.uniform(-2, 2, B), rng.uniform(-2, 2, B), rng.uniform(-np.pi, np.pi, B)])
    goal = pose[:2] + rng.uniform(-0.6, 0.6, (2, B))
    vel = np.vstack([rng.uniform(0, 1.0, B), rng.uniform(-0.5, 0.5, B), rng.uniform(-0.5, 0.5, B)])
    refv = rng.uniform(0.2, 0.7, B)
    dev = torch.device("cuda:0")
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    sv = capi.Solver(prm, B, 0)
    d_pose, d_goal, d_vel, d_ref = d(pose), d(goal), d(vel), d(refv)
    sv.decel_raw(B, d_pose, d_goal, d_vel, 0.05, d_ref)
    got = d_ref.cpu().numpy()
    thr = max(prm.max_throttle, 0.1)
    want = np.array([oracle.decel(pose[0, i], pose[1, i], goal[0, i], goal[1, i], vel[0, i], thr, prm.max_speed, 0.05, refv[i])
                     for i in range(B)])
    assert (want != refv).sum() > B // 10          # the schedule is exercised
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-15)
    # plant: unicycle driven by the command
    cmd = np.vstack([rng.uniform(0, 0.7, B), rng.uniform(-1.5, 1.5, B)])
    d_cmd = d(cmd)
    sv.plant_step_raw(B, d_cmd, d_pose, d_vel)
    p2 = d_pose.cpu().numpy(); v2 = d_vel.cpu().numpy()
    sv.close()
    np.testing.assert_allclose(p2[0], pose[0] + cmd[0] * np.cos(pose[2]) * prm.dt, rtol=0, atol=1e-14)
    np.testing.assert_allclose(p2[1], pose[1] + cmd[0] * np.sin(pose[2]) * prm.dt, rtol=0, atol=1e-14)
    th = np.remainder(pose[2] + cmd[1] * prm.dt + np.pi, 2 * np.pi) - np.pi
    np.testing.assert_allclose(p2[2], th, rtol=0, atol=1e-14)
    np.testing.assert_array_equal(v2[0], cmd[0]); np.testing.assert_array_equal(v2[1:], vel[1:])


def test_small_weights_keep_lsq_multipliers(oracle):
    """Both outcomes of the least-squares multiplier size test (folded into the adjoint sweep, which runs on a
    stage thread) reproduce the oracle's iterates: small weights -> multipliers kept, YAML weights -> discarded."""
    state, coeffs = mild(23, 96)
    for pm in (dict(YAML_DEFAULT, W_CTE=2.0, W_V=5.0, W_ANGVEL=1.0, W_A=1.0, BOUND=1e19), dict(YAML_DEFAULT, BOUND=1e19)):
        sv = _solver(pm, 96)
        out = sv.solve(state, coeffs)
        sv.close()
        for i in range(0, 96, 3):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert out["status"][i] == 1 and o["status"] == 1
            assert out["iters"][i] == o["iters"]
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= 1e-9


def test_rate_penalties_full_width_ctas(oracle):
    """The rate-penalty variant with as many lanes per CTA as fit (28: both control warps, both half-warps of the
    adjoint sweep, queue refill) agrees with the narrow launch of the same problems and with the oracle."""
    pm = dict(CFG_DEFAULT)
    state, coeffs = mild(47, 224)
    outs = []
    for pb, ctas in ((28, 2), (4, 0)):
        sv = _solver(pm, 224)
        sv.set_option("problems_per_cta", pb); sv.set_option("max_ctas", ctas)
        outs.append(sv.solve(state, coeffs))
        sv.close()
    wide, narrow = outs
    assert (wide["status"] == 1).all() and (narrow["status"] == 1).all()
    assert (wide["iters"] == narrow["iters"]).all()
    np.testing.assert_allclose(wide["u0"], narrow["u0"], rtol=0, atol=1e-9)
    for i in range(0, 224, 7):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert o["status"] == 1
        assert np.abs(wide["u0"][:, i] - o["u0"]).max() <= U_TOL
        assert abs(wide["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])


def test_kkt_conditions_in_the_reference_formulation(oracle):
    """Independent of the kernel's own error computation: the returned point with its multipliers (the record of
    mpc_b200_warm_size doubles, laid out like the reference's variables mpc_planner.cpp:232-239 and constraint rows
    :153-158) satisfies the first-order conditions of the REFERENCE's NLP, evaluated by the oracle's restatement of
    FG_eval (pinned to the reference's CppAD output by tests/golden/fg_eval_golden.json), to Ipopt's tolerance
    (W&B eq. (5)-(6): 1e-8 on the scaled error)."""
    torch = pytest.importorskip("torch")
    B = 32; N = 20; n = 8 * N - 2; m = 6 * N; nu = N - 1
    pm = YAML_DEFAULT
    state, coeffs = mild(61, B)
    dev = torch.device("cuda:0")
    sv = _solver(pm, B)
    ws = capi.lib().mpc_b200_warm_size(N)
    assert ws == n + m + 4 * nu
    f64 = dict(dtype=torch.float64, device=dev)
    u0 = torch.zeros((2, B), **f64); pred = torch.zeros((3 * N, B), **f64); wo = torch.zeros((ws, B), **f64)
    st = torch.zeros(B, dtype=torch.int32, device=dev)
    sv.solve_raw(B, torch.from_numpy(state).to(dev), torch.from_numpy(coeffs).to(dev), u0, pred, status=st, warm_out=wo)
    torch.cuda.synchronize()
    sv.close()
    assert bool((st == 1).all())
    rec = wo.cpu().numpy()
    Uw = pm["ANGVEL"]; Ua = pm["MAXTHR"]
    for i in range(B):
        x = rec[:n, i].copy(); lam = rec[n:n + m, i].copy()
        zlw, zla, zuw, zua = (rec[n + m + j * nu: n + m + (j + 1) * nu, i] for j in range(4))
        ev = oracle.eval_all(pm, coeffs[:, i], x, lam, 1.0)
        # primal feasibility: initial-condition rows equal the state, dynamics rows vanish
        target = np.zeros(m)
        for c in range(6):
            target[c * N] = state[c, i]
        assert np.abs(ev["g"] - target).max() <= 1e-8
        # the objective scaling Ipopt applies (nlp_scaling_max_gradient = 100) and the multiplier scaling s_d, s_c
        g0 = max(abs(2 * pm["W_CTE"] * (state[4, i] - pm["REF_CTE"])), abs(2 * pm["W_EPSI"] * (state[5, i] - pm["REF_ETHETA"])),
                 abs(2 * pm["W_V"] * (state[3, i] - pm["REF_V"])), abs(2 * pm["W_V"] * pm["REF_V"]),
                 abs(2 * pm["W_CTE"] * pm["REF_CTE"]), abs(2 * pm["W_EPSI"] * pm["REF_ETHETA"]))
        sf = 100.0 / g0 if g0 > 100.0 else 1.0
        z1 = sf * (zlw.sum() + zla.sum() + zuw.sum() + zua.sum())
        s_d = max(100.0, (sf * np.abs(lam).sum() + z1) / (m + 4 * nu)) / 100.0
        s_c = max(100.0, z1 / (4 * nu)) / 100.0
        # stationarity: grad f + J^T lambda - zL + zU = 0 (only the controls carry bound multipliers on this path)
        r = ev["grad"] + ev["J"].T @ lam
        r[6 * N:7 * N - 1] += zuw - zlw
        r[7 * N - 1:] += zua - zla
        assert sf * np.abs(r).max() <= 1e-8 * s_d * 1.001
        # bounds, multiplier signs, complementarity
        w = x[6 * N:7 * N - 1]; a = x[7 * N - 1:]
        assert np.abs(w).max() <= Uw * (1 + 1e-8) and np.abs(a).max() <= Ua * (1 + 1e-8)
        assert min(zlw.min(), zla.min(), zuw.min(), zua.min()) > 0.0
        compl = max((zlw * (w + Uw)).max(), (zuw * (Uw - w)).max(), (zla * (a + Ua)).max(), (zua * (Ua - a)).max())
        assert sf * compl <= 1e-8 * s_c * 1.001 + 1e-8 * sf * max(zlw.max(), zla.max(), zuw.max(), zua.max())   # (+ the 1e-8 bound relaxation)


def test_higher_order_path_polynomial(oracle):
    """FG_eval takes a path polynomial of any order (mpc_planner.cpp:186-190: coeffs.size()); orders 4..7 run through
    the option "poly_coeffs" (every variant carries it; the tick entry points, whose pre-step fits a cubic, refuse)."""
    from tests.test_emu import higher_order
    pm = YAML_DEFAULT
    for ncoef in (5, 8):
        state, coeffs = higher_order(80 + ncoef, 40, ncoef)
        sv = _solver(pm, 40)
        sv.set_option("poly_coeffs", ncoef)
        out = sv.solve(state, coeffs)
        for i in range(0, 40, 2):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert out["status"][i] == 1 and o["status"] == 1
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
            assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
            assert out["kkt"][i] <= KKT_TOL
        # back to cubics on the same handle: the first four rows alone
        sv.set_option("poly_coeffs", 4)
        out3 = sv.solve(state, coeffs[:4])
        o3 = oracle.solve(pm, state[:, 0], coeffs[:4, 0])
        assert np.abs(out3["u0"][:, 0] - o3["u0"]).max() <= U_TOL
        with pytest.raises(capi.MpcError):
            sv.set_option("poly_coeffs", 9)
        sv.close()
    # rate penalties (the cfg defaults) + a quintic: the augmented variant carries the higher-order polynomial too
    pm = dict(CFG_DEFAULT)
    sv = _solver(pm, 24)
    sv.set_option("poly_coeffs", 6)
    state, coeffs = higher_order(90, 24, 6)
    out = sv.solve(state, coeffs)
    sv.close()
    for i in range(0, 24, 2):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        assert out["status"][i] == 1 and o["status"] == 1
        assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
        assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])


def test_higher_order_warm_start():
    """Warm start with a quintic path: the roll-out of the model uses the same polynomial; re-solving from the converged
    record reproduces the cold solution in fewer iterations."""
    torch = pytest.importorskip("torch")
    from tests.test_emu import higher_order
    B = 32; N = 20
    state, coeffs = higher_order(95, B, 6)
    dev = torch.device("cuda:0")
    sv = _solver(YAML_DEFAULT, B)
    sv.set_option("poly_coeffs", 6)
    ws = capi.lib().mpc_b200_warm_size(N)
    f64 = dict(dtype=torch.float64, device=dev)
    ds = torch.from_numpy(state).to(dev); dc = torch.from_numpy(coeffs).to(dev)
    u_cold = torch.zeros((2, B), **f64); u_w = torch.zeros((2, B), **f64); pred = torch.zeros((3 * N, B), **f64)
    it_cold = torch.zeros(B, dtype=torch.int32, device=dev); it_w = torch.zeros(B, dtype=torch.int32, device=dev)
    st = torch.zeros(B, dtype=torch.int32, device=dev)
    wo = torch.zeros((ws, B), **f64)
    sv.solve_raw(B, ds, dc, u_cold, pred, status=st, iters=it_cold, warm_out=wo)
    torch.cuda.synchronize()
    assert bool((st == 1).all())
    sv.solve_raw(B, ds, dc, u_w, pred, warm_in=wo, status=st, iters=it_w)
    torch.cuda.synchronize()
    sv.close()
    assert bool((st == 1).all())
    assert float((u_w - u_cold).abs().max()) <= U_TOL
    assert float(it_w.double().mean()) <= 0.7 * float(it_cold.double().mean())


def test_prestep_fits_higher_orders(oracle):
    """polyfit(x, y, order) takes any order (driving_state.cpp:283-300); with the option poly_coeffs the pre-step fits
    and writes that many coefficients, and the whole tick (pre-step -> solve) then runs on the higher-order path."""
    from bench import gen_py
    B = 48
    g = gen_py.problems(20261031, B)
    sv = _solver(YAML_DEFAULT, B)
    sv.set_option("poly_coeffs", 6)
    coeffs, cte, eth = sv.polyfit(g["wx"], g["wy"], g["pose"])
    assert coeffs.shape == (6, B)
    for i in range(B):
        px, py, th = g["pose"][:, i]
        dx = g["wx"][:, i] - px; dy = g["wy"][:, i] - py
        xs = dx * np.cos(th) + dy * np.sin(th); ys = dy * np.cos(th) - dx * np.sin(th)
        c_o = oracle.polyfit(xs, ys, 5)
        scale = max(1.0, np.abs(c_o).max())
        assert np.abs(c_o - coeffs[:, i]).max() <= 1e-7 * scale, (i, c_o, coeffs[:, i])
        assert cte[i] == coeffs[0, i]
    # pre-step + solve on the quintic fits = the oracle's solve on them (mild problems only: a quintic through a sharp
    # corner is as wild as the cubic)
    state = np.zeros((6, B)); state[3] = g["vel"][0]; state[4] = cte; state[5] = eth
    out = sv.solve(state, coeffs)
    sv.close()
    checked = 0
    for i in range(B):
        if np.abs(coeffs[1:, i]).sum() > 2.0:
            continue
        o = oracle.solve(YAML_DEFAULT, state[:, i], coeffs[:, i])
        if o["status"] == 1 and out["status"][i] == 1:
            checked += 1
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
            assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
    assert checked >= B // 3


def test_short_and_odd_horizons(oracle):
    """mpc_steps is a parameter (mpc_planner.cpp:247): horizons that do not fill the stage groups evenly, down to 3
    (one stage group, the adjoint sweep of all lanes on group 0), with narrow and full-width CTAs."""
    for N, pb in ((3, 0), (5, 32), (7, 0), (21, 32)):
        pm = dict(YAML_DEFAULT, STEPS=N)
        B = 64
        state, coeffs = mild(30 + N, B)
        sv = _solver(pm, B)
        if pb:
            sv.set_option("problems_per_cta", pb); sv.set_option("max_ctas", 1)
        out = sv.solve(state, coeffs)
        sv.close()
        assert out["pred"].shape == (3 * N, B)
        for i in range(0, B, 4):
            o = oracle.solve(pm, state[:, i], coeffs[:, i])
            assert out["status"][i] == 1 and o["status"] == 1, (N, i)
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL
            assert abs(out["obj"][i] - o["obj"]) <= F_TOL * max(1e-12, abs(o["obj"]))
            assert np.abs(out["pred"][:, i].reshape(3, N) - o["pred"]).max() <= 1e-6


# ---------------------------------------------------------------- round 2: windowing, state bounds, large sweeps
def test_window_kernel_matches_oracle(oracle):
    """SURVEY 8f-2: window_kernel against the oracle's restatement of MPCPlannerROS::getCutOffPlan (:266-291) and
    downSamplePlan (:365-391) (mpc_oracle_cutoff / _downsample), over several ticks so that the persistent plan index is exercised."""
    import torch
    from bench import gen_py
    from bench.closed_loop import Fleet
    R = 240
    fleet = Fleet(R, seed=99)
    prm = capi.yaml_default_params()
    sv = capi.Solver(prm, R, 0)
    M = capi.lib().mpc_b200_num_waypoints(prm)
    dev = torch.device("cuda:0")
    lens = [len(p[0]) for p in fleet.paths]
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32)
    d_px = torch.from_numpy(np.concatenate([p[0] for p in fleet.paths])).to(dev)
    d_py = torch.from_numpy(np.concatenate([p[1] for p in fleet.paths])).to(dev)
    d_off = torch.from_numpy(offs).to(dev); d_len = torch.tensor(lens, dtype=torch.int32, device=dev)
    d_tid = torch.from_numpy(fleet.kind.astype(np.int32)).to(dev)
    d_idx = torch.from_numpy(fleet.idx.astype(np.int32)).to(dev)
    d_wx = torch.zeros((M, R), dtype=torch.float64, device=dev); d_wy = torch.zeros_like(d_wx)
    rng = np.random.default_rng(4)
    idx = fleet.idx.copy()
    for tick in range(6):
        d_pose = torch.from_numpy(np.ascontiguousarray(fleet.pose)).to(dev)
        sv.window_raw(R, d_px, d_py, d_off, d_len, d_tid, d_idx, d_pose, d_wx, d_wy)
        torch.cuda.synchronize()
        wx = d_wx.cpu().numpy(); wy = d_wy.cpu().numpy(); gi = d_idx.cpu().numpy()
        for i in range(R):
            px, py = fleet.paths[fleet.kind[i]]
            e = oracle.cutoff(px, py, int(idx[i]), fleet.pose[0, i], fleet.pose[1, i], ring=True, max_erase=64)
            idx[i] = (int(idx[i]) + e) % len(px)
            ox, oy, m = oracle.downsample(px, py, int(idx[i]), fleet.win, fleet.step, ring=True)
            assert m == M and gi[i] == idx[i], (tick, i, gi[i], idx[i])
            assert np.array_equal(wx[:, i], ox) and np.array_equal(wy[:, i], oy)
        # move the robots along (and a little off) their tracks, up to ~2.5 m per tick: cuts of 0 .. 50 points
        for i in range(R):
            px, py = fleet.paths[fleet.kind[i]]
            j = (int(idx[i]) + int(rng.integers(0, 50))) % len(px)
            fleet.pose[0, i] = px[j] + rng.uniform(-0.2, 0.2); fleet.pose[1, i] = py[j] + rng.uniform(-0.2, 0.2)
    sv.close()


@pytest.mark.parametrize("bound", [0.5, 2.0, 1e3])
def test_state_bounds_honoured_or_refused(oracle, bound):
    """mpc_planner.cpp:303-312: every state variable is bounded by +-bound_value (cfg range 0.01 .. 1000).  The GPU path
    has no barrier for these bounds: where the returned point lies strictly inside them it must be the oracle's solution
    of the BOUNDED problem (within the north-star tolerances); everywhere else it must say MPC_B200_STATUS_BOUND_ACTIVE
    and never SUCCESS."""
    pm = dict(YAML_DEFAULT, BOUND=bound)
    state, coeffs = mild(41, 64)
    sv = _solver(pm, 64)
    out = sv.solve(state, coeffs)
    sv.close()
    n_inside = n_flag = 0
    for i in range(64):
        o = oracle.solve(pm, state[:, i], coeffs[:, i])
        smax_gpu = max(np.abs(out["pred"][:, i]).max(), np.abs(state[:, i]).max())
        if out["status"][i] == 1:
            n_inside += 1
            assert smax_gpu < bound
            assert o["status"] == 1
            assert np.abs(out["u0"][:, i] - o["u0"]).max() <= U_TOL, (i, out["u0"][:, i], o["u0"])
            assert abs(out["obj"][i] - o["obj"]) <= F_TOL * abs(o["obj"])
        else:
            assert out["status"][i] == 64, out["status"][i]
            n_flag += 1
            # the oracle's bounded solution does lean on a bound (or the unbounded one would leave the box)
            s_o = np.abs(o["sol"][:6 * 20]).max()
            assert s_o >= bound * (1.0 - 2e-3) or smax_gpu >= bound * (1.0 - 1e-3)
    if bound >= 1e3:
        assert n_flag == 0
    if bound <= 0.5:
        assert n_flag > 0          # x reaches ~1 m within the horizon: the bound would bind for most problems
    assert n_inside + n_flag == 64


def _oracle_many(pm, state, coeffs, max_iter=100, warm=None, warm_mu=1e-3):
    """the oracle on all host cores; warm: warm-start records (warm_size x B) or None for cold starts"""
    import multiprocessing as mp
    from tests.parity_sweep import _oracle_chunk
    import tests.parity_sweep as ps
    ps.MAX_ITER = max_iter
    n = state.shape[1]
    P = os.cpu_count() or 1
    cuts = np.linspace(0, n, 4 * P + 1).astype(int)
    w = (lambda a, b: ()) if warm is None else (lambda a, b: (warm[:, a:b].copy(), warm_mu))  # noqa: E731
    with mp.get_context("fork").Pool(P) as pool:
        parts = pool.map(_oracle_chunk, [(pm, state[:, a:b].copy(), coeffs[:, a:b].copy()) + w(a, b)
                                         for a, b in zip(cuts[:-1], cuts[1:]) if b > a])
    return {k: np.concatenate([p[k] for p in parts], axis=-1) for k in parts[0]}


def _sweep_check(name, pm, seed, n, max_both_miss, max_conv_gap):
    """GPU through the C ABI vs the oracle on all host cores, both capped at 100 iterations; returns the statistics."""
    from bench import gen_py
    g = gen_py.problems(seed, n)
    prm = capi.params_from_map(pm, capi.yaml_default_params()); prm.delay_mode = 0; prm.max_iter = 100
    sv = capi.Solver(prm, n, 0)
    coeffs, state = sv.prestep(g["wx"], g["wy"], g["pose"], g["vel"])
    gpu = sv.solve(state, coeffs)
    sv.close()
    orc = _oracle_many(pm, state, coeffs)
    okg = (gpu["status"] == 1) & (gpu["kkt"] <= KKT_TOL); oko = orc["status"] == 1
    both = okg & oko
    du = np.abs(gpu["u0"] - orc["u0"]).max(axis=0)
    dobj = np.abs(gpu["obj"] - orc["obj"]) / np.maximum(1.0, np.abs(orc["obj"]))
    miss = int((both & ((du > U_TOL) | (dobj > F_TOL))).sum())
    stats = dict(sweep=name, problems=n, gpu_converged=int(okg.sum()), oracle_converged=int(oko.sum()), both=int(both.sum()),
                 miss=miss, only_oracle=int((~okg & oko).sum()), only_gpu=int((okg & ~oko).sum()),
                 gpu_status={int(k): int(v) for k, v in zip(*np.unique(gpu["status"], return_counts=True))})
    print(json.dumps(stats))
    assert miss <= max_both_miss, stats
    assert abs(stats["gpu_converged"] - stats["oracle_converged"]) <= max_conv_gap, stats
    assert both.sum() >= 0.995 * n, stats
    return stats


def test_sweep_config2_yaml_weights():
    """4,096 problems of BASELINE config 2's generator (mpc_params.yaml weights) against the oracle, miss count asserted:
    a both-converged problem may differ only where the non-convex NLP has a second local minimum (<= 2 per 16k)."""
    _sweep_check("config2 yaml", YAML_DEFAULT, 20261018 + 2, 4096, max_both_miss=1, max_conv_gap=3)


def test_sweep_config2_cfg_weights():
    """The same with the MPCPlanner.cfg defaults (rate penalties: the augmented-Riccati variant)."""
    _sweep_check("config2 cfg", CFG_DEFAULT, 20261018 + 12, 4096, max_both_miss=1, max_conv_gap=3)


def test_sweep_config3_seed():
    """BASELINE config 3's problem set (seed 20261018 + 3), first 4,096 problems."""
    _sweep_check("config3 seed", YAML_DEFAULT, 20261018 + 3, 4096, max_both_miss=1, max_conv_gap=3)


def test_sweep_config4_real_generator_N100():
    """BASELINE config 4 as benchmarked: the REAL generator (seed 20261018 + 4) at N = 100, 1,024 problems.
    A 10 s horizon over a cubic fitted to 5 m of path is strongly non-convex: with the second-order correction in the kernel
    the iterates equal the oracle's when the oracle runs without the +-1e3 state bounds (0 misses, tests/test_emu.py); with
    them (the reference's NLP) the z / s terms of those bounds perturb the early iterates by 1e-3, which sends 2 of the
    1,024 problems to another local minimum (both KKT points, both converged)."""
    _sweep_check("config4 N=100", dict(YAML_DEFAULT, STEPS=100), 20261018 + 4, 1024, max_both_miss=3, max_conv_gap=4)


def test_packed_and_sliced_ticks_equal_the_plain_tick():
    """mpc_b200_track_packed_submit (one buffer, one copy each way) and mpc_b200_track_slice_submit (contiguous slices of
    the caller's SoA arrays, SURVEY 8e) return bit for bit what mpc_b200_track_batch returns."""
    import ctypes as C
    from bench import gen_py
    B = 500
    g = gen_py.problems(20261018 + 3, B)
    M = g["M"]
    prm = capi.yaml_default_params()
    sv = capi.Solver(prm, B, 0)
    vel = np.ascontiguousarray(g["vel"]).copy()
    ref = sv.track(g["wx"], g["wy"], g["pose"], vel)
    # ---- packed
    total, off = sv.packed_layout(B, M)
    L = capi.lib()
    ptr = L.mpc_b200_host_alloc(total)
    buf = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(total,))
    v = sv.packed_views(buf, B, M)
    v["wx"][:] = g["wx"]; v["wy"][:] = g["wy"]; v["pose"][:] = g["pose"]; v["vel"][:] = g["vel"]
    sv.track_packed_submit(B, M, ptr)
    sv.track_wait()
    for k in ("u0", "pred", "cmd", "obj", "kkt", "status", "iters"):
        assert np.array_equal(v[k], ref[k]), k
    assert np.array_equal(v["vel"], vel)
    L.mpc_b200_host_free(ptr)
    # ---- sliced: two handles on the same device share the batch 200 / 300
    import torch
    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    N = prm.mpc_steps
    t = dict(wx=pin(g["wx"]), wy=pin(g["wy"]), pose=pin(g["pose"]), vel=pin(g["vel"]), u0=pin(np.zeros((2, B))),
             pred=pin(np.zeros((3 * N, B))), cmd=pin(np.zeros((2, B))), obj=pin(np.zeros(B)), kkt=pin(np.zeros(B)),
             status=pin(np.zeros(B, dtype=np.int32)), iters=pin(np.zeros(B, dtype=np.int32)))
    hs = [capi.Solver(prm, 200, 0), capi.Solver(prm, 300, 0)]
    for s_, (lo, n) in zip(hs, ((0, 200), (200, 300))):
        rc = L.mpc_b200_track_slice_submit(s_._h, B, lo, n, M, t["wx"].data_ptr(), t["wy"].data_ptr(), t["pose"].data_ptr(),
                                           t["vel"].data_ptr(), None, t["u0"].data_ptr(), t["pred"].data_ptr(), t["cmd"].data_ptr(),
                                           t["obj"].data_ptr(), t["status"].data_ptr(), t["iters"].data_ptr(), t["kkt"].data_ptr())
        assert rc == 0
    for s_ in hs:
        s_.track_wait(); s_.close()
    for k in ("u0", "pred", "cmd", "obj", "kkt", "status", "iters"):
        assert np.array_equal(t[k].numpy(), ref[k]), k
    assert np.array_equal(t["vel"].numpy(), vel)
    # pageable arrays are refused, not silently staged
    rc = L.mpc_b200_track_slice_submit(sv._h, B, 0, B, M, g["wx"].ctypes.data, g["wy"].ctypes.data, g["pose"].ctypes.data,
                                       vel.ctypes.data, None, ref["u0"].ctypes.data, ref["pred"].ctypes.data, None, None, None, None, None)
    assert rc == -3
    sv.close()


def test_host_warm_records_are_staged(oracle):
    """SURVEY 8b ownership: warm-start records may live in host memory too.  Host and device records give the same solves
    bit for bit: u0, pred, iterations, status and the records written, cold and warm."""
    torch = pytest.importorskip("torch")
    dev = torch.device("cuda:0")
    state, coeffs = mild(7, 16)
    state2 = state.copy(); state2[3] += 0.02; state2[4] -= 0.01
    sv = _solver(YAML_DEFAULT, 16)
    N = 20; ws = capi.lib().mpc_b200_warm_size(N)

    def run(on_dev, st, warm_in):
        """one solve with the records in host (on_dev False) or device memory; inputs and other outputs on the host"""
        out = dict(u0=np.zeros((2, 16)), pred=np.zeros((3 * N, 16)), status=np.zeros(16, dtype=np.int32),
                   iters=np.zeros(16, dtype=np.int32))
        wo = torch.zeros((ws, 16), dtype=torch.float64, device=dev) if on_dev else np.zeros((ws, 16))
        wi = None if warm_in is None else (torch.from_numpy(warm_in).to(dev) if on_dev else warm_in.copy())
        sv.solve_raw(16, st, coeffs, out["u0"], out["pred"], status=out["status"], iters=out["iters"], warm_in=wi, warm_out=wo)
        out["rec"] = wo.cpu().numpy() if on_dev else wo
        return out

    res = {}
    for on_dev in (False, True):
        cold = run(on_dev, state, None)
        res[on_dev] = (cold, run(on_dev, state, cold["rec"]), run(on_dev, state2, cold["rec"]))
    sv.close()
    cold, same, moved = res[False]
    assert np.all(cold["status"] == 1) and np.abs(cold["rec"]).max() > 0
    assert np.all(same["status"] == 1) and np.all(moved["status"] == 1)
    assert np.abs(same["u0"] - cold["u0"]).max() <= U_TOL
    assert same["iters"].mean() < cold["iters"].mean()
    for h, d in zip(res[False], res[True]):
        for k in ("u0", "pred", "status", "iters", "rec"):
            assert h[k].tobytes() == d[k].tobytes(), k
