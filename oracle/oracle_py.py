"""oracle/oracle_py.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes bindings for the CPU oracle (oracle/liboracle.so, the plain-C
restatement of the reference's MPC::Solve path) and for oracle/_ref/libmpc_ref.so
(the reference's unmodified mpc_planner.cpp + vendored CppAD behind the stand-in
Ipopt interface).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

PARAM_KEYS = ["DT", "STEPS", "REF_CTE", "REF_ETHETA", "REF_V", "W_CTE", "W_EPSI", "W_V",
              "W_ANGVEL", "W_A", "W_DANGVEL", "W_DA", "ANGVEL", "MAXTHR", "BOUND"]

# mpc_ros/params/mpc_params.yaml:9-25 (dt = 1/controller_freq)
YAML_DEFAULT = dict(DT=0.1, STEPS=20, REF_CTE=0.0, REF_ETHETA=0.0, REF_V=0.5, W_CTE=100.0, W_EPSI=0.0,
                    W_V=1000.0, W_ANGVEL=100.0, W_A=50.0, W_DANGVEL=0.0, W_DA=0.0, ANGVEL=1.5, MAXTHR=1.0,
                    BOUND=1.0e3)
# mpc_ros/cfg/MPCPlanner.cfg:22-37 defaults (dt from controller_freq 10)
CFG_DEFAULT = dict(DT=0.1, STEPS=20, REF_CTE=0.0, REF_ETHETA=0.0, REF_V=1.0, W_CTE=1000.0, W_EPSI=1000.0,
                   W_V=100.0, W_ANGVEL=100.0, W_A=50.0, W_DANGVEL=0.0, W_DA=10.0, ANGVEL=1.0, MAXTHR=1.0,
                   BOUND=1.0e3)


def build(verbose=False):
    """make -C oracle (liboracle.so always; _ref only where /root/reference exists)."""
    r = subprocess.run(["make", "-C", _HERE], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout)


class OracleParams(C.Structure):
    _fields_ = [("mpc_steps", C.c_int)] + [(k, C.c_double) for k in (
        "dt", "ref_cte", "ref_etheta", "ref_vel", "w_cte", "w_etheta", "w_vel", "w_angvel", "w_accel",
        "w_angvel_d", "w_accel_d", "max_angvel", "max_throttle", "bound_value")]


class OracleResult(C.Structure):
    _fields_ = [("status", C.c_int), ("iters", C.c_int), ("obj", C.c_double), ("kkt_error", C.c_double),
                ("dual_inf", C.c_double), ("constr_viol", C.c_double), ("compl_inf", C.c_double),
                ("n_inertia_corrections", C.c_int), ("n_restorations", C.c_int)]


class IpmOptions(C.Structure):
    _fields_ = [("tol", C.c_double), ("max_iter", C.c_int), ("max_cpu_time", C.c_double),
                ("dual_inf_tol", C.c_double), ("constr_viol_tol", C.c_double), ("compl_inf_tol", C.c_double),
                ("acceptable_tol", C.c_double), ("acceptable_iter", C.c_int), ("mu_init", C.c_double),
                ("bound_push", C.c_double), ("bound_frac", C.c_double), ("bound_relax_factor", C.c_double),
                ("nlp_scaling_max_gradient", C.c_double), ("max_soc", C.c_int), ("print_level", C.c_int),
                ("use_dense_ldl", C.c_int)]


def params_from_map(pm):
    p = OracleParams()
    p.mpc_steps = int(pm["STEPS"])
    p.dt = pm["DT"]; p.ref_cte = pm["REF_CTE"]; p.ref_etheta = pm["REF_ETHETA"]; p.ref_vel = pm["REF_V"]
    p.w_cte = pm["W_CTE"]; p.w_etheta = pm["W_EPSI"]; p.w_vel = pm["W_V"]; p.w_angvel = pm["W_ANGVEL"]
    p.w_accel = pm["W_A"]; p.w_angvel_d = pm["W_DANGVEL"]; p.w_accel_d = pm["W_DA"]
    p.max_angvel = pm["ANGVEL"]; p.max_throttle = pm["MAXTHR"]; p.bound_value = pm["BOUND"]
    return p


def _arr(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp)


class Oracle:
    """The plain-C restatement (oracle/liboracle.so)."""

    def __init__(self):
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            build()
        self.lib = C.CDLL(path)
        L = self.lib
        L.mpc_oracle_solve.restype = C.c_int
        L.mpc_oracle_solve.argtypes = [C.POINTER(OracleParams), _dp, _dp, C.c_int, C.POINTER(IpmOptions),
                                       _dp, _dp, _dp, _dp, _dp, _dp, C.POINTER(OracleResult)]
        L.mpc_oracle_solve_warm.restype = C.c_int
        L.mpc_oracle_solve_warm.argtypes = [C.POINTER(OracleParams), _dp, _dp, C.c_int, C.POINTER(IpmOptions), _dp,
                                            C.c_double, _dp, _dp, _dp, _dp, _dp, _dp, C.POINTER(OracleResult)]
        L.mpc_oracle_eval_fg.argtypes = [C.POINTER(OracleParams), _dp, C.c_int, _dp, _dp, _dp]
        L.mpc_oracle_eval_grad.argtypes = [C.POINTER(OracleParams), _dp, C.c_int, _dp, _dp]
        L.mpc_oracle_eval_jac_dense.argtypes = [C.POINTER(OracleParams), _dp, C.c_int, _dp, _dp]
        L.mpc_oracle_eval_hess_dense.argtypes = [C.POINTER(OracleParams), _dp, C.c_int, _dp, C.c_double, _dp, _dp]
        L.mpc_oracle_polyfit.restype = C.c_int
        L.mpc_oracle_polyfit.argtypes = [_dp, _dp, C.c_int, C.c_int, _dp]
        L.mpc_oracle_decel.argtypes = [C.c_double] * 9
        L.mpc_oracle_decel.restype = C.c_double
        L.mpc_oracle_prestep.argtypes = [_dp, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _dp, _dp, _dp]
        L.ipm_default_options.argtypes = [C.POINTER(IpmOptions)]
        L.mpc_oracle_state.argtypes = [C.c_int] + [C.c_double] * 6 + [_dp]
        L.mpc_oracle_poststep_speed.argtypes = [C.c_double] * 4
        L.mpc_oracle_poststep_speed.restype = C.c_double
        L.mpc_oracle_cutoff.restype = C.c_int
        L.mpc_oracle_cutoff.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double]
        L.mpc_oracle_downsample_step.restype = C.c_int
        L.mpc_oracle_downsample_step.argtypes = [C.c_double, C.c_double]
        L.mpc_oracle_downsample.restype = C.c_int
        L.mpc_oracle_downsample.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp]

    def default_options(self):
        o = IpmOptions()
        self.lib.ipm_default_options(C.byref(o))
        return o

    def solve(self, pm, state, coeffs, opt=None, warm=None, warm_mu=1e-3):
        """warm: a warm-start record (mpc_b200_warm_size(N) doubles, the GPU path's layout) or None for the cold start.
        A warm solve needs BOUND >= 1e19 (no state bounds)."""
        p = params_from_map(pm)
        N = p.mpc_steps
        n, m = 8 * N - 2, 6 * N
        state = _arr(state); coeffs = _arr(coeffs)
        u0 = np.zeros(2); pred = np.zeros(3 * N); sol = np.zeros(n); lam = np.zeros(m)
        zl = np.zeros(n); zu = np.zeros(n)
        r = OracleResult()
        o = C.byref(opt) if opt is not None else None
        if warm is None:
            self.lib.mpc_oracle_solve(C.byref(p), _ptr(state), _ptr(coeffs), len(coeffs), o,
                                      _ptr(u0), _ptr(pred), _ptr(sol), _ptr(lam), _ptr(zl), _ptr(zu), C.byref(r))
        else:
            warm = _arr(warm)
            if warm.shape != (n + m + 4 * (N - 1),):
                raise ValueError("warm record of %s doubles, expected %d" % (warm.shape, n + m + 4 * (N - 1)))
            rc = self.lib.mpc_oracle_solve_warm(C.byref(p), _ptr(state), _ptr(coeffs), len(coeffs), o, _ptr(warm),
                                                float(warm_mu), _ptr(u0), _ptr(pred), _ptr(sol), _ptr(lam), _ptr(zl),
                                                _ptr(zu), C.byref(r))
            if rc == -1:
                raise ValueError("warm start refused: finite state bounds or a scaled constraint row")
        return dict(u0=u0, pred=pred.reshape(3, N), sol=sol, lam=lam, zl=zl, zu=zu, status=r.status,
                    iters=r.iters, obj=r.obj, kkt_error=r.kkt_error, dual_inf=r.dual_inf,
                    constr_viol=r.constr_viol, compl_inf=r.compl_inf,
                    n_inertia=r.n_inertia_corrections, n_resto=r.n_restorations)

    def eval_all(self, pm, coeffs, x, lam, sigma=1.0):
        p = params_from_map(pm)
        N = p.mpc_steps
        n, m = 8 * N - 2, 6 * N
        coeffs = _arr(coeffs); x = _arr(x); lam = _arr(lam)
        f = C.c_double(); g = np.zeros(m); grad = np.zeros(n); J = np.zeros((m, n)); H = np.zeros((n, n))
        self.lib.mpc_oracle_eval_fg(C.byref(p), _ptr(coeffs), len(coeffs), _ptr(x), C.byref(f), _ptr(g))
        self.lib.mpc_oracle_eval_grad(C.byref(p), _ptr(coeffs), len(coeffs), _ptr(x), _ptr(grad))
        self.lib.mpc_oracle_eval_jac_dense(C.byref(p), _ptr(coeffs), len(coeffs), _ptr(x), _ptr(J))
        self.lib.mpc_oracle_eval_hess_dense(C.byref(p), _ptr(coeffs), len(coeffs), _ptr(x), sigma, _ptr(lam), _ptr(H))
        return dict(f=f.value, g=g, grad=grad, J=J, H=H)

    def polyfit(self, xs, ys, order=3):
        xs = _arr(xs); ys = _arr(ys)
        c = np.zeros(order + 1)
        rc = self.lib.mpc_oracle_polyfit(_ptr(xs), _ptr(ys), len(xs), order, _ptr(c))
        if rc != 0:
            raise ValueError("polyfit failed rc=%d" % rc)
        return c

    def prestep(self, wx, wy, px, py, theta):
        wx = _arr(wx); wy = _arr(wy)
        c = np.zeros(4); cte = C.c_double(); eth = C.c_double()
        self.lib.mpc_oracle_prestep(_ptr(wx), _ptr(wy), len(wx), px, py, theta, _ptr(c), C.byref(cte), C.byref(eth))
        return c, cte.value, eth.value

    def decel(self, px, py, gx, gy, v, max_throttle, max_speed, min_speed, ref_v):
        return self.lib.mpc_oracle_decel(px, py, gx, gy, v, max_throttle, max_speed, min_speed, ref_v)

    def state(self, delay_mode, v, w_prev, thr_prev, dt, cte, etheta):
        s6 = np.zeros(6)
        self.lib.mpc_oracle_state(int(bool(delay_mode)), v, w_prev, thr_prev, dt, cte, etheta, _ptr(s6))
        return s6

    def poststep_speed(self, v, throttle, dt, ref_v):
        return self.lib.mpc_oracle_poststep_speed(v, throttle, dt, ref_v)

    def cutoff(self, px, py, first, rx, ry, ring=True, max_erase=None):
        px = _arr(px); py = _arr(py)
        return self.lib.mpc_oracle_cutoff(len(px), _ptr(px), _ptr(py), int(first), int(bool(ring)),
                                          len(px) if max_erase is None else int(max_erase), rx, ry)

    def downsample_step(self, path_length, waypoints_dist):
        return self.lib.mpc_oracle_downsample_step(path_length, waypoints_dist)

    def downsample(self, px, py, first, win, step, ring=True, cap=64):
        px = _arr(px); py = _arr(py)
        wx = np.zeros(cap); wy = np.zeros(cap)
        m = self.lib.mpc_oracle_downsample(len(px), _ptr(px), _ptr(py), int(first), int(bool(ring)), int(win), int(step),
                                           cap, _ptr(wx), _ptr(wy))
        return wx[:min(m, cap)], wy[:min(m, cap)], m


def ref_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libmpc_ref.so"))


class Reference:
    """The reference's own MPC class (oracle/_ref/libmpc_ref.so).  Solver inside: oracle/ipm.c, not Ipopt."""

    def __init__(self, pm):
        path = os.path.join(_HERE, "_ref", "libmpc_ref.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path + " (build with make -C oracle where /root/reference exists)")
        self.lib = C.CDLL(path)
        L = self.lib
        L.ref_mpc_create.restype = C.c_void_p
        L.ref_mpc_create.argtypes = [_dp]
        L.ref_mpc_destroy.argtypes = [C.c_void_p]
        L.ref_set_cpu_time_override.argtypes = [C.c_double]
        L.ref_set_dense_ldl.argtypes = [C.c_int]
        L.ref_mpc_solve.restype = C.c_int
        L.ref_mpc_solve.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]
        L.ref_fg_eval.restype = C.c_int
        L.ref_fg_eval.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.c_int, _dp, _dp, C.c_double,
                                  _dp, _dp, _dp, _dp, _dp, _ip]
        L.ref_hs071.restype = C.c_int
        L.ref_hs071.argtypes = [C.c_double, _dp, _dp, _dp, _dp, _ip]
        self.pm = dict(pm)
        self.N = int(pm["STEPS"])
        pv = _arr([pm[k] for k in PARAM_KEYS])
        self.h = L.ref_mpc_create(_ptr(pv))

    def __del__(self):
        try:
            self.lib.ref_mpc_destroy(self.h)
        except Exception:
            pass

    def set_cpu_time_override(self, s):
        self.lib.ref_set_cpu_time_override(float(s))

    def solve(self, state, coeffs):
        N = self.N
        n, m = 8 * N - 2, 6 * N
        state = _arr(state); coeffs = _arr(coeffs)
        u0 = np.zeros(2); pred = np.zeros(3 * N); info = np.zeros(10)
        sol = np.zeros(n); lam = np.zeros(m); zl = np.zeros(n); zu = np.zeros(n)
        self.lib.ref_mpc_solve(self.h, N, _ptr(state), _ptr(coeffs), len(coeffs), _ptr(u0), _ptr(pred), _ptr(info),
                               _ptr(sol), _ptr(lam), _ptr(zl), _ptr(zu))
        return dict(u0=u0, pred=pred.reshape(3, N), sol=sol, lam=lam, zl=zl, zu=zu, status=int(info[0]),
                    iters=int(info[1]), obj=info[2], kkt_error=info[3], dual_inf=info[4], constr_viol=info[5],
                    compl_inf=info[6], n_inertia=int(info[7]), n_resto=int(info[8]), n_fact=int(info[9]))

    def fg_eval(self, state, coeffs, x, lam, sigma=1.0):
        N = self.N
        n, m = 8 * N - 2, 6 * N
        state = _arr(state); coeffs = _arr(coeffs); x = _arr(x); lam = _arr(lam)
        f = C.c_double(); grad = np.zeros(n); g = np.zeros(m); J = np.zeros((m, n)); H = np.zeros((n, n))
        nnz = (C.c_int * 2)()
        rc = self.lib.ref_fg_eval(self.h, N, _ptr(state), _ptr(coeffs), len(coeffs), _ptr(x), _ptr(lam), sigma,
                                  C.byref(f), _ptr(grad), _ptr(g), _ptr(J), _ptr(H), nnz)
        if rc != 0:
            raise RuntimeError("ref_fg_eval rc=%d" % rc)
        return dict(f=f.value, grad=grad, g=g, J=J, H=H, nnz_jac=nnz[0], nnz_hess=nnz[1])

    def hs071(self, tol=1e-8):
        x = np.zeros(4); zl = np.zeros(4); zu = np.zeros(4); obj = C.c_double(); it = C.c_int()
        st = self.lib.ref_hs071(tol, _ptr(x), _ptr(zl), _ptr(zu), C.byref(obj), C.byref(it))
        return dict(status=st, x=x, zl=zl, zu=zu, obj=obj.value, iters=it.value)


def ros_ref_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libros_ref.so"))


class RosReference:
    """The reference's UNMODIFIED ROS-side sources (driving_state.cpp, mpc_planner_ros.cpp) behind the stand-in ROS
    headers of oracle/shim/ros_stubs, with the reference's own MPC (oracle/_ref/libros_ref.so, oracle/ros_ref_driver.cpp)."""

    def __init__(self):
        path = os.path.join(_HERE, "_ref", "libros_ref.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path + " (build with make -C oracle where /root/reference exists)")
        self.lib = C.CDLL(path)
        L = self.lib
        L.ros_ref_window.restype = C.c_int
        L.ros_ref_window.argtypes = [C.c_int, _dp, _dp, C.c_double, C.c_double, C.c_double, C.c_int, _dp, _dp, _ip, _ip]
        L.ros_ref_tick_new.restype = C.c_void_p
        L.ros_ref_tick_new.argtypes = [_dp, C.c_int, C.c_double]
        L.ros_ref_tick.restype = C.c_int
        L.ros_ref_tick.argtypes = [C.c_void_p] + [C.c_double] * 6 + [C.c_int, _dp, _dp, _dp, _dp, _dp, C.c_int]
        L.ros_ref_polyfit.argtypes = [C.c_int, _dp, _dp, C.c_int, _dp]
        L.ros_ref_polyeval.restype = C.c_double
        L.ros_ref_polyeval.argtypes = [C.c_int, _dp, C.c_double]

    def window(self, px, py, rx, ry, path_length, cap=256):
        px = _arr(px); py = _arr(py)
        wx = np.zeros(cap); wy = np.zeros(cap); ne = C.c_int(); ds = C.c_int()
        m = self.lib.ros_ref_window(len(px), _ptr(px), _ptr(py), rx, ry, path_length, cap, _ptr(wx), _ptr(wy),
                                    C.byref(ne), C.byref(ds))
        return dict(m=m, wx=wx[:max(0, min(m, cap))], wy=wy[:max(0, min(m, cap))], erased=ne.value, step=ds.value)

    def tracker(self, pm, delay_mode, max_speed):
        cfg = _arr([pm[k] for k in PARAM_KEYS])
        return self.lib.ros_ref_tick_new(_ptr(cfg), int(bool(delay_mode)), float(max_speed))

    def tick(self, h, pose, goal, v, wx, wy, state3, N=20):
        """state3 = [_w, _throttle, REF_V] in / out.  Returns dict(cmd=(linear.x, angular.z), w, throttle, ref_v, pred)."""
        wx = _arr(wx); wy = _arr(wy); st = _arr(state3).copy(); out = np.zeros(5); pred = np.zeros(3 * N)
        ok = self.lib.ros_ref_tick(h, pose[0], pose[1], pose[2], goal[0], goal[1], v, len(wx), _ptr(wx), _ptr(wy),
                                   _ptr(st), _ptr(out), _ptr(pred), N)
        return dict(ok=ok, cmd=out[:2].copy(), w=out[2], throttle=out[3], ref_v=out[4], state3=st, pred=pred.reshape(3, N))

    def polyfit(self, xs, ys, order=3):
        xs = _arr(xs); ys = _arr(ys); c = np.zeros(order + 1)
        self.lib.ros_ref_polyfit(len(xs), _ptr(xs), _ptr(ys), order, _ptr(c))
        return c

    def polyeval(self, coeffs, x):
        coeffs = _arr(coeffs)
        return self.lib.ros_ref_polyeval(len(coeffs), _ptr(coeffs), x)
