"""ctypes binding of the C ABI declared in include/mpcb200.h.

This module is plumbing only: it loads ``libmpcb200.so`` (hand-written sm_100a CUDA behind a C ABI) and exposes the
entry points with numpy arrays.  There is NO CPU fallback: if the shared library is missing or no CUDA device is
present, the calls raise.

Reference boundary: ``Controller::configure/step/reset`` (mpc_local_planner/include/mpc_local_planner/controller.h:61-104).
"""
import ctypes as C
import os

import numpy as np

MAX_POLY = 16
OBST_STRIDE = 7
INF = 1e30
KKT_WORDS = 42
STEP_WORDS = 8
SCAL_WORDS = 32

# enums (mirror include/mpcb200.h)
ROBOT_UNICYCLE, ROBOT_SIMPLE_CAR, ROBOT_SIMPLE_CAR_FRONT, ROBOT_KIN_BICYCLE = 0, 1, 2, 3
COLLOC_FORWARD, COLLOC_MIDPOINT, COLLOC_CRANK_NICOLSON = 0, 1, 2
COST_LEFT_SUM, COST_TRAPEZOIDAL = 0, 1
OBJ_MINIMUM_TIME, OBJ_QUADRATIC_FORM, OBJ_MINIMUM_TIME_VIA_POINTS = 0, 1, 2
FOOTPRINT_POINT, FOOTPRINT_CIRCULAR, FOOTPRINT_TWO_CIRCLES, FOOTPRINT_LINE, FOOTPRINT_POLYGON = 0, 1, 2, 3, 4
OBST_POINT, OBST_CIRCLE, OBST_LINE = 0, 1, 2
STATUS_CONVERGED, STATUS_MAX_ITER, STATUS_NUMERICAL_ERROR, STATUS_INVALID_INPUT = 0, 1, 2, 3
E_INVALID, E_UNSUPPORTED, E_CUDA, E_NOMEM, E_NODEVICE = -1, -2, -3, -4, -5
F_X, F_U, F_NU, F_S, F_LAM, F_KKT, F_STEP, F_SCAL, F_OBSIDX, F_OBSGIDX = range(10)
PHASE_INIT, PHASE_ASSOCIATE, PHASE_EVAL, PHASE_KKT, PHASE_LINESEARCH = range(5)
OPT_SOLVE_MODE = 3
OPT_CTAS_PER_SM = 4
OPT_SM_PHASE_SYNC = 5
OPT_ORDER_BY_HISTORY = 6
SOLVE_FUSED, SOLVE_PHASED = 0, 1
NUM_PHASES = 5
K_H, K_G, K_A, K_B, K_E, K_C, K_HB, K_D = 0, 15, 20, 23, 29, 32, 34, 39
(SC_DT, SC_MU, SC_RHO, SC_DELTA, SC_HTT, SC_GT, SC_DDT, SC_ERR0, SC_ERRMU, SC_ITER, SC_STATUS, SC_ALPHA, SC_OBJ,
 SC_INF, SC_DELTA_LAST, SC_NREG, SC_BLOG, SC_GLDT, SC_NBT, SC_COLD, SC_TINY, SC_DEFER, SC_VALID, SC_OBST_DROPPED) = range(24)


class Config(C.Structure):
    """``mpcb200_config`` -- field for field (include/mpcb200.h)."""
    _fields_ = [
        ("robot_type", C.c_int),
        ("wheelbase", C.c_double),
        ("length_rear", C.c_double),
        ("length_front", C.c_double),
        ("u_lb", C.c_double * 2),
        ("u_ub", C.c_double * 2),
        ("du_lb", C.c_double * 2),
        ("du_ub", C.c_double * 2),
        ("n", C.c_int),
        ("dt_ref", C.c_double),
        ("variable_dt", C.c_int),
        ("dt_lb", C.c_double),
        ("dt_ub", C.c_double),
        ("xf_fixed", C.c_int * 3),
        ("collocation", C.c_int),
        ("warm_start", C.c_int),
        ("objective", C.c_int),
        ("Q", C.c_double * 9),
        ("R", C.c_double * 4),
        ("terminal_cost", C.c_int),
        ("Qf", C.c_double * 9),
        ("vp_position_weight", C.c_double),
        ("vp_orientation_weight", C.c_double),
        ("vp_ordered", C.c_int),
        ("vp_attraction_with_quadratic", C.c_int),
        ("min_obstacle_dist", C.c_double),
        ("force_inclusion_dist", C.c_double),
        ("cutoff_dist", C.c_double),
        ("footprint_type", C.c_int),
        ("footprint_params", C.c_double * 4),
        ("n_poly", C.c_int),
        ("poly_xy", C.c_double * (2 * MAX_POLY)),
        ("k_max_obstacles_per_stage", C.c_int),
        ("max_iter", C.c_int),
        ("tol", C.c_double),
        ("mu_init", C.c_double),
        ("outer_iterations", C.c_int),
        ("quadratic_integral_form", C.c_int),
        ("initial_guess_bumps", C.c_int),
        ("enable_dynamic_obstacles", C.c_int),
        ("terminal_ball", C.c_int),
        ("terminal_ball_S", C.c_double * 9),
        ("terminal_ball_gamma", C.c_double),
        ("cost_integration", C.c_int),
        ("hybrid_cost_minimum_time", C.c_int),
        ("reference_initial_guess", C.c_int),
    ]

    def copy(self):
        c = Config()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(Config))
        return c


class Costmaps(C.Structure):
    _fields_ = [("size_x", C.c_int), ("size_y", C.c_int), ("resolution", C.c_double), ("origin", C.POINTER(C.c_double)),
                ("cost", C.POINTER(C.c_ubyte))]


class Obstacles(C.Structure):
    _fields_ = [("max_per_instance", C.c_int), ("count", C.POINTER(C.c_int)), ("type", C.POINTER(C.c_int)),
                ("params", C.POINTER(C.c_double))]


class ViaPoints(C.Structure):
    _fields_ = [("max_per_instance", C.c_int), ("count", C.POINTER(C.c_int)), ("poses", C.POINTER(C.c_double))]


class Stats(C.Structure):
    _fields_ = [("launches", C.c_longlong * NUM_PHASES), ("ms", C.c_double * NUM_PHASES),
                ("launches_total", C.c_longlong), ("h2d_bytes", C.c_longlong), ("d2h_bytes", C.c_longlong),
                ("kkt_instances", C.c_longlong), ("kkt_sweeps", C.c_longlong), ("gate_ms", C.c_double)]


def default_config():
    """In-code defaults of the reference (SURVEY App. D; src/controller.cpp:225-805). Pure Python twin of
    ``mpcb200_default_config`` so that oracle-only tests do not need the CUDA library."""
    c = Config()
    c.robot_type = ROBOT_UNICYCLE
    c.wheelbase, c.length_rear, c.length_front = 0.5, 1.0, 1.0
    c.u_lb[:] = [-0.2, -0.3]
    c.u_ub[:] = [0.4, 0.3]
    c.du_lb[:] = [-INF, -INF]
    c.du_ub[:] = [INF, INF]
    c.n, c.dt_ref = 20, 0.3
    c.variable_dt, c.dt_lb, c.dt_ub = 1, 0.0, 10.0
    c.xf_fixed[:] = [1, 1, 1]
    c.collocation = COLLOC_FORWARD
    c.warm_start = 1
    c.objective = OBJ_MINIMUM_TIME
    c.Q[:] = [0.0] * 9
    c.R[:] = [0.0] * 4
    c.terminal_cost = 0
    c.Qf[:] = [0.0] * 9
    c.vp_position_weight, c.vp_orientation_weight, c.vp_ordered = 1.0, 0.0, 0
    c.vp_attraction_with_quadratic = 0
    c.min_obstacle_dist, c.force_inclusion_dist, c.cutoff_dist = 0.5, 0.5, 2.0
    c.footprint_type = FOOTPRINT_POINT
    c.n_poly = 0
    c.k_max_obstacles_per_stage = 5
    c.max_iter, c.tol, c.mu_init = 100, 1e-6, 0.0
    c.outer_iterations = 1
    c.quadratic_integral_form = 0
    c.initial_guess_bumps = 4
    c.enable_dynamic_obstacles = 0
    c.terminal_ball = 0
    for i in range(9):
        c.terminal_ball_S[i] = 1.0 if i % 4 == 0 else 0.0
    c.terminal_ball_gamma = 5.0
    c.cost_integration = COST_LEFT_SUM
    c.hybrid_cost_minimum_time = 0
    return c


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int)) if a is not None else None


def pack_obstacles(count, types, params):
    """count [B] int32, types [B,M] int32, params [B,M,5] float64 -> (Obstacles struct, keep-alive tuple)."""
    count = np.ascontiguousarray(count, dtype=np.int32)
    types = np.ascontiguousarray(types, dtype=np.int32)
    params = np.ascontiguousarray(params, dtype=np.float64)
    o = Obstacles(int(types.shape[1]) if types.ndim == 2 else 0, _ip(count), _ip(types), _dp(params))
    return o, (count, types, params)


def pack_viapoints(count, poses):
    count = np.ascontiguousarray(count, dtype=np.int32)
    poses = np.ascontiguousarray(poses, dtype=np.float64)
    v = ViaPoints(int(poses.shape[1]) if poses.ndim == 3 else 0, _ip(count), _dp(poses))
    return v, (count, poses)


def pack_costmaps(cost, origin, resolution):
    """cost [B, size_y, size_x] uint8, origin [B, 2] -> (Costmaps struct, keep-alive tuple (cost, origin))."""
    cost = np.ascontiguousarray(cost, dtype=np.uint8)
    origin = np.ascontiguousarray(origin, dtype=np.float64)
    m = Costmaps(cost.shape[2], cost.shape[1], float(resolution), _dp(origin), cost.ctypes.data_as(C.POINTER(C.c_ubyte)))
    return m, (cost, origin)


def _results(B, N):
    """host arrays for the results of B instances"""
    return dict(u_seq=np.empty((B, N, 2)), x_seq=np.empty((B, N, 3)), dt=np.empty(B),
                status=np.empty(B, dtype=np.int32), kkt_err=np.empty(B), iters=np.empty(B, dtype=np.int32))


def _result_ptrs(out):
    """the output arguments u_seq, x_seq, dt, status, kkt_err, iters of the C calls"""
    return (_dp(out["u_seq"]), _dp(out["x_seq"]), _dp(out["dt"]), _ip(out["status"]), _dp(out["kkt_err"]), _ip(out["iters"]))


_LIB = None
_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libmpcb200.so")

EXPORTS = [
    "mpcb200_default_config", "mpcb200_create", "mpcb200_step_batch", "mpcb200_reset", "mpcb200_destroy",
    "mpcb200_last_error", "mpcb200_upload_inputs", "mpcb200_solve_resident", "mpcb200_fetch_results",
    "mpcb200_device_controls", "mpcb200_ws_count", "mpcb200_ws_read", "mpcb200_ws_write", "mpcb200_run_phase",
    "mpcb200_check_feasible", "mpcb200_time_phase", "mpcb200_set_timing", "mpcb200_set_stream", "mpcb200_set_option", "mpcb200_solve_stream", "mpcb200_stats_get", "mpcb200_stats_reset", "mpcb200_export_controls", "mpcb200_flush_l2",
    "mpcb200_resample", "mpcb200_get_horizon", "mpcb200_costmap_obstacles", "mpcb200_step_batch_costmap", "mpcb200_costmap_last_ms",
    "mpcb200_create_multi", "mpcb200_step_batch_multi", "mpcb200_multi_device_controls", "mpcb200_multi_fetch_controls", "mpcb200_multi_handle",
    "mpcb200_destroy_multi", "mpcb200_multi_last_error",
]


def load_library(path=None):
    """Load libmpcb200.so (built in-tree by __graft_entry__.build()). Raises if it is missing: no fallback."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback for the solver.")
    lib = C.CDLL(path)
    vp, dp, ip, cp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_char_p
    ucp = C.POINTER(C.c_ubyte)
    lib.mpcb200_default_config.argtypes = [C.POINTER(Config)]
    lib.mpcb200_default_config.restype = None
    lib.mpcb200_create.argtypes = [C.POINTER(Config), C.c_int, C.c_int, C.POINTER(vp)]
    lib.mpcb200_step_batch.argtypes = [vp, C.c_int, dp, dp, dp, C.c_double, C.POINTER(Obstacles), C.POINTER(ViaPoints),
                                       dp, ucp, dp, dp, dp, ip, dp, ip, dp]
    lib.mpcb200_solve_stream.argtypes = [vp, C.c_int, dp, dp, dp, C.c_double, C.POINTER(Obstacles), C.POINTER(ViaPoints),
                                         dp, dp, dp, ip, dp, ip, dp]
    lib.mpcb200_reset.argtypes = [vp, ucp, C.c_int]
    lib.mpcb200_resample.argtypes = [vp, C.c_int]
    lib.mpcb200_costmap_obstacles.argtypes = [vp, C.c_int, C.POINTER(Costmaps), dp, C.c_double, C.c_int, ip, ip, ip, dp]
    lib.mpcb200_step_batch_costmap.argtypes = [vp, C.c_int, dp, dp, dp, C.c_double, C.POINTER(Costmaps), C.c_double, C.c_int, C.POINTER(ViaPoints),
                                               dp, ucp, dp, dp, dp, ip, dp, ip, ip, dp]
    lib.mpcb200_costmap_last_ms.argtypes = [vp]
    lib.mpcb200_costmap_last_ms.restype = C.c_double
    lib.mpcb200_get_horizon.argtypes = [vp, ip, ip]
    lib.mpcb200_destroy.argtypes = [vp]
    lib.mpcb200_destroy.restype = None
    lib.mpcb200_last_error.argtypes = [vp]
    lib.mpcb200_last_error.restype = cp
    lib.mpcb200_upload_inputs.argtypes = [vp, C.c_int, dp, dp, dp, C.c_double, C.POINTER(Obstacles),
                                          C.POINTER(ViaPoints), dp]
    lib.mpcb200_solve_resident.argtypes = [vp, C.c_int, dp]
    lib.mpcb200_fetch_results.argtypes = [vp, dp, dp, dp, ip, dp, ip]
    lib.mpcb200_device_controls.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_longlong)]
    lib.mpcb200_export_controls.argtypes = [vp, vp]
    lib.mpcb200_flush_l2.argtypes = [vp]
    lib.mpcb200_ws_count.argtypes = [vp, C.c_int]
    lib.mpcb200_ws_read.argtypes = [vp, C.c_int, C.c_int, dp]
    lib.mpcb200_ws_write.argtypes = [vp, C.c_int, C.c_int, dp]
    lib.mpcb200_run_phase.argtypes = [vp, C.c_int, C.c_int]
    lib.mpcb200_create_multi.argtypes = [C.POINTER(Config), C.c_int, C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    lib.mpcb200_step_batch_multi.argtypes = lib.mpcb200_step_batch.argtypes
    lib.mpcb200_multi_device_controls.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_longlong)]
    lib.mpcb200_multi_fetch_controls.argtypes = [vp, C.c_int, dp]
    lib.mpcb200_multi_handle.argtypes = [vp, C.c_int]
    lib.mpcb200_multi_handle.restype = vp
    lib.mpcb200_destroy_multi.argtypes = [vp]
    lib.mpcb200_destroy_multi.restype = None
    lib.mpcb200_multi_last_error.argtypes = [vp]
    lib.mpcb200_multi_last_error.restype = C.c_char_p
    lib.mpcb200_check_feasible.argtypes = [vp, C.c_int, C.POINTER(Costmaps), dp, C.c_int, dp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.POINTER(C.c_ubyte)]
    lib.mpcb200_time_phase.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, dp]
    lib.mpcb200_set_timing.argtypes = [vp, C.c_uint]
    lib.mpcb200_set_stream.argtypes = [vp, vp]
    lib.mpcb200_set_option.argtypes = [vp, C.c_int, C.c_int]
    lib.mpcb200_stats_get.argtypes = [vp, C.POINTER(Stats)]
    lib.mpcb200_stats_reset.argtypes = [vp]
    if path == LIB_PATH:
        _LIB = lib
    return lib


class SolverError(RuntimeError):
    pass


class BatchSolver:
    """Thin owner of one ``mpcb200_handle`` (one CUDA device). Mirrors Controller::configure/step/reset for a batch."""

    def __init__(self, cfg, max_batch, device=0):
        self.lib = load_library()
        self.cfg = cfg.copy()
        self.max_batch = int(max_batch)
        self.N = int(cfg.n)
        self.K = int(cfg.k_max_obstacles_per_stage)
        h = C.c_void_p()
        rc = self.lib.mpcb200_create(C.byref(self.cfg), self.max_batch, int(device), C.byref(h))
        if rc != 0:
            msg = self.lib.mpcb200_last_error(None).decode()
            raise SolverError(f"mpcb200_create failed ({rc}): {msg}")
        self.h = h
        self.B = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.mpcb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise SolverError(f"{what} failed ({rc}): {self.lib.mpcb200_last_error(self.h).decode()}")

    @staticmethod
    def _prep_inputs(x0, xf, u_prev, obstacles, viapoints, x_init):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        xf = np.ascontiguousarray(xf, dtype=np.float64)
        B = x0.shape[0]
        u_prev = np.zeros((B, 2)) if u_prev is None else np.ascontiguousarray(u_prev, dtype=np.float64)
        keep = [x0, xf, u_prev]
        o = v = None
        if obstacles is not None:
            o, k = pack_obstacles(*obstacles)
            keep.append(k)
        if viapoints is not None:
            v, k = pack_viapoints(*viapoints)
            keep.append(k)
        xi = None
        if x_init is not None:
            xi = np.ascontiguousarray(x_init, dtype=np.float64)
            keep.append(xi)
        return B, x0, xf, u_prev, o, v, xi, keep

    def solve_stream(self, x0, xf, u_prev=None, u_prev_dt=0.0, obstacles=None, viapoints=None):
        """A queue of len(x0) instances (any number) through the pool of max_batch slots: continuous batching, cold starts."""
        T, x0, xf, u_prev, o, v, xi, keep = self._prep_inputs(x0, xf, u_prev, obstacles, viapoints, None)
        out = _results(T, self.N)
        t = C.c_double(0.0)
        rc = self.lib.mpcb200_solve_stream(
            self.h, T, _dp(x0), _dp(xf), _dp(u_prev), float(u_prev_dt), C.byref(o) if o else None, C.byref(v) if v else None,
            *_result_ptrs(out), C.byref(t))
        self._check(rc, "mpcb200_solve_stream")
        out["solve_time_s"] = t.value
        return out

    def alloc_outputs(self, B, pin=None):
        """Result buffers for step(..., out=...).  pin: optional callable array -> (pinned array, owner) (e.g. through
        torch.Tensor.pin_memory): page-locked buffers take the device-to-host copies without a staging copy."""
        out = _results(B, self.N)
        if pin is not None:
            owners = []
            for k in list(out):
                out[k], owner = pin(out[k])
                owners.append(owner)
            out["_owners"] = owners
        return out

    def step(self, x0, xf, u_prev=None, u_prev_dt=0.0, obstacles=None, viapoints=None, x_init=None, reinit=None, out=None):
        """Controller::step for a batch (host arrays in, host arrays out; copies inside the call).  out: buffers of
        alloc_outputs() to write the results into (default: fresh arrays)."""
        B, x0, xf, u_prev, o, v, xi, keep = self._prep_inputs(x0, xf, u_prev, obstacles, viapoints, x_init)
        if out is None:
            out = self.alloc_outputs(B)
        t = C.c_double(0.0)
        ri = None
        if reinit is not None:
            ri = np.ascontiguousarray(reinit, dtype=np.uint8)
        rc = self.lib.mpcb200_step_batch(
            self.h, B, _dp(x0), _dp(xf), _dp(u_prev), float(u_prev_dt), C.byref(o) if o else None,
            C.byref(v) if v else None, _dp(xi), ri.ctypes.data_as(C.POINTER(C.c_ubyte)) if ri is not None else None,
            *_result_ptrs(out), C.byref(t))
        self._check(rc, "mpcb200_step_batch")
        out["solve_time_s"] = t.value
        self.B = B
        return out

    def upload(self, x0, xf, u_prev=None, u_prev_dt=0.0, obstacles=None, viapoints=None, x_init=None):
        B, x0, xf, u_prev, o, v, xi, keep = self._prep_inputs(x0, xf, u_prev, obstacles, viapoints, x_init)
        rc = self.lib.mpcb200_upload_inputs(self.h, B, _dp(x0), _dp(xf), _dp(u_prev), float(u_prev_dt),
                                            C.byref(o) if o else None, C.byref(v) if v else None, _dp(xi))
        self._check(rc, "mpcb200_upload_inputs")
        self.B = B

    def solve_resident(self, cold=True):
        t = C.c_double(0.0)
        self._check(self.lib.mpcb200_solve_resident(self.h, 1 if cold else 0, C.byref(t)), "mpcb200_solve_resident")
        return t.value

    def fetch(self):
        out = _results(self.B, self.N)
        self._check(self.lib.mpcb200_fetch_results(self.h, *_result_ptrs(out)), "mpcb200_fetch_results")
        return out

    def reset(self, which=None):
        w = None
        if which is not None:
            w = np.ascontiguousarray(which, dtype=np.uint8)
        self._check(self.lib.mpcb200_reset(self.h, w.ctypes.data_as(C.POINTER(C.c_ubyte)) if w is not None else None,
                                           self.B), "mpcb200_reset")

    def costmap_obstacles(self, cost, origin, resolution, robot_pose, behind_robot_dist, max_per_instance):
        """updateObstacleContainerWithCostmap for B robots: cost [B, size_y, size_x] uint8, origin [B, 2], robot_pose [B, 3]
        -> (count [B], type [B, M], params [B, M, OBST_STRIDE]) in the layout step() takes as `obstacles`, and found [B]."""
        m, (cost, origin) = pack_costmaps(cost, origin, resolution)
        pose = np.ascontiguousarray(robot_pose, dtype=np.float64)
        B, M = cost.shape[0], int(max_per_instance)
        count = np.zeros(B, dtype=np.int32); found = np.zeros(B, dtype=np.int32)
        typ = np.zeros((B, M), dtype=np.int32); par = np.zeros((B, M, OBST_STRIDE))
        self._check(self.lib.mpcb200_costmap_obstacles(self.h, B, C.byref(m), _dp(pose), float(behind_robot_dist), M, _ip(count), _ip(found),
                                                       _ip(typ), _dp(par)), "mpcb200_costmap_obstacles")
        return (count, typ, par), found

    def step_from_costmaps(self, x0, xf, cost, origin, resolution, behind_robot_dist, max_per_instance, u_prev=None, u_prev_dt=0.0,
                           viapoints=None, x_init=None, reinit=None, out=None):
        """One planning cycle from the costmaps (updateObstacleContainerWithCostmap with robot pose = x0, then Controller::step): the
        obstacle lists stay on the device.  Returns step()'s dict plus obst_found [B]."""
        B, x0, xf, u_prev, _, v, xi, keep = self._prep_inputs(x0, xf, u_prev, None, viapoints, x_init)
        m, maps_keep = pack_costmaps(cost, origin, resolution)
        if out is None:
            out = self.alloc_outputs(B)
        found = np.zeros(B, dtype=np.int32)
        t = C.c_double(0.0)
        ri = np.ascontiguousarray(reinit, dtype=np.uint8) if reinit is not None else None
        rc = self.lib.mpcb200_step_batch_costmap(
            self.h, B, _dp(x0), _dp(xf), _dp(u_prev), float(u_prev_dt), C.byref(m), float(behind_robot_dist), int(max_per_instance),
            C.byref(v) if v else None, _dp(xi), ri.ctypes.data_as(C.POINTER(C.c_ubyte)) if ri is not None else None,
            *_result_ptrs(out), _ip(found), C.byref(t))
        self._check(rc, "mpcb200_step_batch_costmap")
        out["solve_time_s"] = t.value
        out["obst_found"] = found
        self.B = B
        return out

    def check_feasible(self, cost, origin, resolution, footprint, inscribed_radius, min_resolution_angular, look_ahead_idx=-1, x_seq=None,
                       circumscribed_radius=0.0):
        """isPoseTrajectoryFeasible for B robots: cost [B, size_y, size_x] uint8, origin [B, 2], footprint [n_fp, 2] (robot frame);
        x_seq [B, n, 3] or None = the trajectories of the last solve on the device.  -> bool [B]"""
        m, (cost, origin) = pack_costmaps(cost, origin, resolution)
        fp = np.ascontiguousarray(footprint, dtype=np.float64).reshape(-1, 2)
        B = cost.shape[0]
        xs = np.ascontiguousarray(x_seq, dtype=np.float64) if x_seq is not None else None
        ok = np.zeros(B, dtype=np.uint8)
        self._check(self.lib.mpcb200_check_feasible(self.h, B, C.byref(m), _dp(xs), xs.shape[1] if xs is not None else 0, _dp(fp), fp.shape[0],
                                                    float(inscribed_radius), float(circumscribed_radius), float(min_resolution_angular),
                                                    int(look_ahead_idx), ok.ctypes.data_as(C.POINTER(C.c_ubyte))), "mpcb200_check_feasible")
        return ok.astype(bool)

    def costmap_last_ms(self):
        return float(self.lib.mpcb200_costmap_last_ms(self.h))

    def resample(self, n_new):
        """resampleTrajectory(n_new) for every instance: the horizon of the batch becomes n_new (<= cfg.n at create)."""
        self._check(self.lib.mpcb200_resample(self.h, int(n_new)), "mpcb200_resample")
        self.N = self.horizon()[0]

    def horizon(self):
        n, cap = C.c_int(0), C.c_int(0)
        self._check(self.lib.mpcb200_get_horizon(self.h, C.byref(n), C.byref(cap)), "mpcb200_get_horizon")
        return n.value, cap.value

    # kernel-level access ------------------------------------------------------------------------------------
    def ws_count(self, field):
        return self.lib.mpcb200_ws_count(self.h, field)

    def ws_read(self, field, B=None):
        B = B or self.B
        cnt = self.ws_count(field)
        shape = (B, cnt) if field in (F_SCAL, F_OBSGIDX) else (B, cnt, self.N)
        a = np.empty(shape)
        self._check(self.lib.mpcb200_ws_read(self.h, field, B, _dp(a)), "mpcb200_ws_read")
        return a

    def ws_write(self, field, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        self._check(self.lib.mpcb200_ws_write(self.h, field, a.shape[0], _dp(a)), "mpcb200_ws_write")

    def run_phase(self, phase, B=None):
        self._check(self.lib.mpcb200_run_phase(self.h, phase, B or self.B), "mpcb200_run_phase")

    def set_stream(self, cuda_stream):
        """Run on the caller's CUDA stream (an integer cudaStream_t, e.g. torch.cuda.Stream().cuda_stream); 0 restores."""
        self._check(self.lib.mpcb200_set_stream(self.h, C.c_void_p(int(cuda_stream) if cuda_stream else None)), "mpcb200_set_stream")

    def set_option(self, option, value):
        self._check(self.lib.mpcb200_set_option(self.h, option, value), "mpcb200_set_option")

    def set_timing(self, phase_mask):
        """Phases bracketed by CUDA events inside a solve (bit p = phase p); default KKT only, 0x1f = all."""
        self._check(self.lib.mpcb200_set_timing(self.h, phase_mask), "mpcb200_set_timing")

    def time_phase(self, phase, reps=10, flush_l2=True, B=None):
        ms = C.c_double(0.0)
        self._check(self.lib.mpcb200_time_phase(self.h, phase, B or self.B, reps, 1 if flush_l2 else 0, C.byref(ms)),
                    "mpcb200_time_phase")
        return ms.value

    def stats(self):
        s = Stats()
        self._check(self.lib.mpcb200_stats_get(self.h, C.byref(s)), "mpcb200_stats_get")
        return dict(launches=list(s.launches), ms=list(s.ms), launches_total=s.launches_total,
                    h2d_bytes=s.h2d_bytes, d2h_bytes=s.d2h_bytes, kkt_instances=s.kkt_instances,
                    kkt_sweeps=s.kkt_sweeps, gate_ms=s.gate_ms)

    def stats_reset(self):
        self._check(self.lib.mpcb200_stats_reset(self.h), "mpcb200_stats_reset")

    def export_controls(self, dst_dev_ptr):
        self._check(self.lib.mpcb200_export_controls(self.h, C.c_void_p(int(dst_dev_ptr))), "mpcb200_export_controls")

    def flush_l2(self):
        self._check(self.lib.mpcb200_flush_l2(self.h), "mpcb200_flush_l2")

    def device_controls(self):
        p = C.c_void_p()
        n = C.c_longlong()
        self._check(self.lib.mpcb200_device_controls(self.h, C.byref(p), C.byref(n)), "mpcb200_device_controls")
        return p.value, n.value


class MultiSolver:
    """Several devices of one node behind one handle (mpcb200_create_multi): contiguous blocks of the batch per device, one NCCL
    all-gather of the packed optimal controls."""

    def __init__(self, cfg, max_batch_total, devices):
        self.lib = load_library()
        self.cfg = cfg.copy()
        self.N = int(cfg.n)
        self.devices = list(devices)
        devs = (C.c_int * len(self.devices))(*self.devices)
        h = C.c_void_p()
        rc = self.lib.mpcb200_create_multi(C.byref(self.cfg), int(max_batch_total), devs, len(self.devices), C.byref(h))
        if rc != 0:
            raise SolverError(f"mpcb200_create_multi failed ({rc}): {self.lib.mpcb200_multi_last_error(None).decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.mpcb200_destroy_multi(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, x0, xf, u_prev=None, u_prev_dt=0.0, obstacles=None, viapoints=None):
        B, x0, xf, u_prev, o, v, xi, keep = BatchSolver._prep_inputs(x0, xf, u_prev, obstacles, viapoints, None)
        out = _results(B, self.N)
        t = C.c_double(0.0)
        rc = self.lib.mpcb200_step_batch_multi(
            self.h, B, _dp(x0), _dp(xf), _dp(u_prev), float(u_prev_dt), C.byref(o) if o else None, C.byref(v) if v else None, None, None,
            *_result_ptrs(out), C.byref(t))
        if rc != 0:
            raise SolverError(f"mpcb200_step_batch_multi failed ({rc}): {self.lib.mpcb200_multi_last_error(self.h).decode()}")
        out["solve_time_s"] = t.value
        self.B = B
        return out

    def gathered_controls(self, rank):
        """the all-gathered packed controls on device `rank` as a host array [G, ceil(B/G), N-1, 2] (copied back for inspection)"""
        p = C.c_void_p(); n = C.c_longlong()
        rc = self.lib.mpcb200_multi_device_controls(self.h, rank, C.byref(p), C.byref(n))
        if rc != 0:
            raise SolverError("mpcb200_multi_device_controls failed")
        G = len(self.devices)
        per = n.value // (G * (self.N - 1) * 2)
        host = np.empty(n.value)
        if self.lib.mpcb200_multi_fetch_controls(self.h, rank, _dp(host)) != 0:
            raise SolverError("mpcb200_multi_fetch_controls failed")
        return host.reshape(G, per, self.N - 1, 2)
