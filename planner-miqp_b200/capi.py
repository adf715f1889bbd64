"""ctypes binding of the C ABI in include/miqp_b200.h.

A problem is any object with the attributes of the reference's ModelParameters in flat
form (N, R, C, O, L, E, scal, safety, safety_slack, car, x0, ref, lim, initial_region,
possible_region, obs_edges, obs_nedges, obs_soft, env_edges, env_off, frac, poly) -- the
same field names the OPL data files use (src/model_input_data_source.cpp:180-275).
"""
from __future__ import annotations

import ctypes as C
import os
import queue
import threading
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

DECLARED_SYMBOLS = [
    "miqp_b200_version", "miqp_b200_default_options", "miqp_b200_create", "miqp_b200_destroy",
    "miqp_b200_last_error", "miqp_b200_layout", "miqp_b200_sizes", "miqp_b200_assemble",
    "miqp_b200_evaluate", "miqp_b200_assemble_batch", "miqp_b200_solve_batch", "miqp_b200_batch_upload", "miqp_b200_batch_run",
    "miqp_b200_batch_fetch", "miqp_b200_run_stats", "miqp_b200_measure_fp64_peak",
    "miqp_b200_debug_profile", "miqp_b200_debug_traces",
    "miqp_b200_frontier_start", "miqp_b200_frontier_rounds", "miqp_b200_frontier_split", "miqp_b200_frontier_get_ub",
    "miqp_b200_frontier_tighten", "miqp_b200_frontier_finish", "miqp_b200_frontier_fingerprint", "miqp_b200_frontier_ub_device", "miqp_b200_batch_upload_replan", "miqp_b200_mark", "miqp_b200_elapsed", "miqp_b200_batch_fetch_compact", "miqp_b200_fetch_vector",
    "miqp_b200_solve_batch_compact",
    "miqp_b200_set_solution_pool", "miqp_b200_pool_sizes", "miqp_b200_pool_fetch",
    "miqp_b200_batch_run_streaming", "miqp_b200_pool_export", "miqp_b200_pool_merge",
]


class MiqpB200Error(RuntimeError):
    pass


class CProblem(C.Structure):
    _fields_ = (
        [(n, C.c_int) for n in ("N", "R", "C", "O", "L", "E")]
        + [(n, C.c_double) for n in (
            "ts", "min_vel", "max_vel", "total_min_acc", "total_max_acc", "total_min_jerk",
            "total_max_jerk", "maximum_slack", "w_slack", "w_slack_obs",
            "min_region_change_speed", "gap_tol", "time_limit")]
        + [("safety", _dp), ("safety_slack", _dp)]
        + [(n, _dp) for n in ("w_pos_x", "w_vel_x", "w_acc_x", "w_pos_y", "w_vel_y", "w_acc_y",
                              "w_jerk_x", "w_jerk_y", "wheelbase", "radius", "x0",
                              "x_ref", "vx_ref", "y_ref", "vy_ref",
                              "min_acc_x", "max_acc_x", "min_acc_y", "max_acc_y",
                              "min_jerk_x", "max_jerk_x", "min_jerk_y", "max_jerk_y")]
        + [("initial_region", _ip), ("possible_region", _ip), ("obs_edges", _dp),
           ("obs_nedges", _ip), ("obs_soft", _ip), ("env_edges", _dp), ("env_off", _ip),
           ("frac", _dp)]
        + [(n, _dp) for n in ("poly_sint_ub", "poly_sint_lb", "poly_coss_ub", "poly_coss_lb",
                              "poly_kappa_max", "poly_kappa_min")]
    )


class CLayout(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "C", "N", "R", "O", "L", "E", "K", "base_nwe", "base_ar", "base_rcna", "base_dcc",
        "base_dcf", "base_so", "base_sof", "base_c2c", "base_sv", "ncols")]


class CSizes(C.Structure):
    _fields_ = [("ncols", C.c_int), ("ncont", C.c_int), ("nbin", C.c_int),
                ("nrows", C.c_long), ("nnz_struct", C.c_long), ("nnz", C.c_long)]


class CSolveInfo(C.Structure):
    _fields_ = [("status", C.c_int), ("proven", C.c_int), ("objective", C.c_double),
                ("best_bound", C.c_double), ("gap", C.c_double), ("seconds", C.c_double),
                ("max_violation", C.c_double), ("nodes", C.c_long), ("qp_iters", C.c_long),
                ("rounds", C.c_long), ("uncertified", C.c_long), ("pool_exhausted", C.c_int)]


class COptions(C.Structure):
    _fields_ = [("device", C.c_int), ("nodes_per_round", C.c_int), ("pool_capacity", C.c_int),
                ("max_rounds", C.c_int), ("verbose", C.c_int)]


class CPoolEntry(C.Structure):
    _fields_ = [("objective", C.c_double), ("max_violation", C.c_double), ("search_value", C.c_double),
                ("converged", C.c_int), ("round", C.c_int), ("uid", C.c_ulonglong)]


# void (*MiqpB200PlanDone)(void *user, int k, const double *traj, const MiqpB200SolveInfo *info)
PLAN_DONE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, _dp, C.POINTER(CSolveInfo))


class CRunStats(C.Structure):
    _fields_ = [("launches", C.c_long), ("node_kernel_launches", C.c_long), ("nodes", C.c_long),
                ("qp_iters", C.c_long), ("rounds", C.c_long), ("node_kernel_ms", C.c_double),
                ("total_ms", C.c_double), ("h2d_bytes", C.c_long), ("d2h_bytes", C.c_long),
                ("rows_visited", C.c_long), ("pack_ms", C.c_double), ("upload_ms", C.c_double), ("fetch_ms", C.c_double)]


@dataclass
class SolveInfo:
    status: int
    proven: bool
    objective: float
    best_bound: float
    gap: float
    seconds: float
    max_violation: float
    nodes: int
    qp_iters: int
    rounds: int
    uncertified: int = 0
    pool_exhausted: int = 0


@dataclass
class PoolEntry:
    """One member of a plan's solution pool (miqp_b200_pool_fetch): objective and max violation of its full column
    vector `x` (device-evaluated), the value the search stored for the leaf, and its trajectory `traj` [C][N][8]."""
    objective: float
    max_violation: float
    search_value: float
    converged: bool
    round: int
    uid: int
    x: np.ndarray | None = None
    traj: np.ndarray | None = None


class _DevView:
    """device memory of the solver as a __cuda_array_interface__ object (torch.as_tensor wraps it without a copy)"""

    def __init__(self, ptr: int, n: int, typestr: str = "<f8"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3, "strides": None}


def library_path() -> str:
    return os.path.join(_HERE, "libmiqp_b200.so")


_lib = None


def load_library():
    """Loads libmiqp_b200.so; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise MiqpB200Error(f"{path} is missing: run __graft_entry__.build() / planner-miqp_b200/build.py")
    lib = C.CDLL(path)
    lib.miqp_b200_version.restype = C.c_char_p
    lib.miqp_b200_last_error.restype = C.c_char_p
    lib.miqp_b200_last_error.argtypes = [C.c_void_p]
    lib.miqp_b200_create.argtypes = [C.POINTER(COptions), C.POINTER(C.c_void_p)]
    lib.miqp_b200_destroy.argtypes = [C.c_void_p]
    lib.miqp_b200_layout.argtypes = [C.POINTER(CProblem), C.POINTER(CLayout)]
    lib.miqp_b200_sizes.argtypes = [C.c_void_p, C.POINTER(CProblem), C.POINTER(CSizes)]
    lib.miqp_b200_assemble.argtypes = [C.c_void_p, C.POINTER(CProblem), C.POINTER(C.c_long), _ip, _dp, _dp, _dp]
    lib.miqp_b200_evaluate.argtypes = [C.c_void_p, C.POINTER(CProblem), _dp, _dp, _dp]
    lib.miqp_b200_solve_batch.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int, C.POINTER(_dp),
                                          C.POINTER(_dp), C.POINTER(CSolveInfo)]
    lib.miqp_b200_batch_upload.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int, C.POINTER(_dp)]
    lib.miqp_b200_batch_run.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    lib.miqp_b200_batch_fetch.argtypes = [C.c_void_p, C.POINTER(_dp), C.POINTER(CSolveInfo)]
    lib.miqp_b200_run_stats.argtypes = [C.c_void_p, C.POINTER(CRunStats)]
    lib.miqp_b200_measure_fp64_peak.argtypes = [C.c_void_p, _dp]
    lib.miqp_b200_debug_profile.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong)]
    lib.miqp_b200_debug_traces.argtypes = [C.c_void_p, _dp]
    lib.miqp_b200_set_solution_pool.argtypes = [C.c_void_p, C.c_int]
    lib.miqp_b200_pool_sizes.argtypes = [C.c_void_p, _ip]
    lib.miqp_b200_pool_fetch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(CPoolEntry), _dp, _dp, _ip]
    lib.miqp_b200_batch_run_streaming.argtypes = [C.c_void_p, PLAN_DONE, C.c_void_p, C.POINTER(C.c_float)]
    lib.miqp_b200_pool_export.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    lib.miqp_b200_pool_merge.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    _lib = lib
    return lib


def exported_symbols() -> list[str]:
    lib = load_library()
    return [s for s in DECLARED_SYMBOLS if hasattr(lib, s)]


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


def _i(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(_ip)


def to_c(p, gap_tol=None, time_limit=None, keep=None) -> CProblem:
    """Flat problem -> C struct.  Arrays are kept alive in `keep`."""
    s = CProblem()
    keep = keep if keep is not None else []
    s.N, s.R, s.C, s.O, s.L, s.E = p.N, p.R, p.C, p.O, p.L, p.E
    sc = p.scal
    s.ts = sc["ts"]
    s.min_vel, s.max_vel = sc["min_vel_x_y"], sc["max_vel_x_y"]
    s.total_min_acc, s.total_max_acc = sc["total_min_acc"], sc["total_max_acc"]
    s.total_min_jerk, s.total_max_jerk = sc["total_min_jerk"], sc["total_max_jerk"]
    s.maximum_slack = sc["maximum_slack"]
    s.w_slack, s.w_slack_obs = sc["WEIGHTS_SLACK"], sc["WEIGHTS_SLACK_OBSTACLE"]
    s.min_region_change_speed = sc["minimum_region_change_speed"]
    s.gap_tol = sc["relative_mip_gap_tolerance"] if gap_tol is None else gap_tol
    s.time_limit = sc["max_solution_time"] if time_limit is None else time_limit

    def setd(name, arr):
        a, ptr = _d(arr)
        keep.append(a)
        setattr(s, name, ptr)

    def seti(name, arr):
        a, ptr = _i(arr)
        keep.append(a)
        setattr(s, name, ptr)

    setd("safety", p.safety)
    setd("safety_slack", p.safety_slack)
    for cn, key in (("w_pos_x", "WEIGHTS_POS_X"), ("w_vel_x", "WEIGHTS_VEL_X"), ("w_acc_x", "WEIGHTS_ACC_X"),
                    ("w_pos_y", "WEIGHTS_POS_Y"), ("w_vel_y", "WEIGHTS_VEL_Y"), ("w_acc_y", "WEIGHTS_ACC_Y"),
                    ("w_jerk_x", "WEIGHTS_JERK_X"), ("w_jerk_y", "WEIGHTS_JERK_Y"),
                    ("wheelbase", "WheelBase"), ("radius", "CollisionRadius")):
        setd(cn, p.car[key])
    setd("x0", p.x0)
    for k in ("x_ref", "vx_ref", "y_ref", "vy_ref"):
        setd(k, p.ref[k])
    for k in ("min_acc_x", "max_acc_x", "min_acc_y", "max_acc_y",
              "min_jerk_x", "max_jerk_x", "min_jerk_y", "max_jerk_y"):
        setd(k, p.lim[k])
    seti("initial_region", p.initial_region)
    seti("possible_region", p.possible_region)
    setd("obs_edges", p.obs_edges if np.size(p.obs_edges) else np.zeros(4))
    seti("obs_nedges", p.obs_nedges if np.size(p.obs_nedges) else np.zeros(1, dtype=np.int32))
    seti("obs_soft", p.obs_soft if np.size(p.obs_soft) else np.zeros(1, dtype=np.int32))
    setd("env_edges", p.env_edges if np.size(p.env_edges) else np.zeros(4))
    seti("env_off", p.env_off)
    setd("frac", p.frac)
    for cn, key in (("poly_sint_ub", "POLY_SINT_UB"), ("poly_sint_lb", "POLY_SINT_LB"),
                    ("poly_coss_ub", "POLY_COSS_UB"), ("poly_coss_lb", "POLY_COSS_LB"),
                    ("poly_kappa_max", "POLY_KAPPA_AX_MAX"), ("poly_kappa_min", "POLY_KAPPA_AX_MIN")):
        setd(cn, p.poly[key])
    return s


def ncols_of(p) -> int:
    """number of columns of the OPL model (decision_variables.mod), closed form of miqp_b200_layout"""
    C_, N, R, O, L, E = p.C, p.N, p.R, p.O, p.L, p.E
    K = C_ - 1
    return (12 * C_ * N + 5 * C_ * E * N + C_ * N * R + 5 * C_ * N + C_ * O * N * L + 4 * C_ * O * N * L
            + C_ * O * N + 4 * C_ * O * N + 16 * K * K * N + 4 * K * K * N)


def layout(p) -> CLayout:
    keep = []
    cp = to_c(p, keep=keep)
    out = CLayout()
    rc = load_library().miqp_b200_layout(C.byref(cp), C.byref(out))
    if rc != 0:
        raise MiqpB200Error(f"miqp_b200_layout failed ({rc})")
    return out


class Solver:
    """Owns one MiqpB200Solver handle (one CUDA device, one stream)."""

    def __init__(self, device: int = 0, nodes_per_round: int = 0, pool_capacity: int = 0,
                 max_rounds: int = 0, verbose: int = 0, solution_pool: int = 0):
        """pool_capacity: open-node slots per plan (0 = auto).  solution_pool: up to this many distinct feasible plans
        per problem are kept (0 = off, at most 64; see set_solution_pool)."""
        self._lib = load_library()
        opt = COptions(device, nodes_per_round, pool_capacity, max_rounds, verbose)
        h = C.c_void_p()
        rc = self._lib.miqp_b200_create(C.byref(opt), C.byref(h))
        if rc != 0 or not h:
            raise MiqpB200Error("miqp_b200_create failed: no usable CUDA device "
                                "(this backend has no CPU fallback)")
        self._h = h
        self._device = device
        self._batch = None
        if solution_pool:
            self.set_solution_pool(solution_pool)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.miqp_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self._lib.miqp_b200_last_error(self._h)
            raise MiqpB200Error(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    # ---- formulation ---------------------------------------------------------------
    def sizes(self, p) -> CSizes:
        keep = []
        cp = to_c(p, keep=keep)
        out = CSizes()
        self._check(self._lib.miqp_b200_sizes(self._h, C.byref(cp), C.byref(out)), "miqp_b200_sizes")
        return out

    def assemble(self, p):
        """Big-M model rows in OPL order: (rowptr, cols, vals, lo, hi), structural zeros kept."""
        sz = self.sizes(p)
        keep = []
        cp = to_c(p, keep=keep)
        rowptr = np.zeros(sz.nrows + 1, dtype=np.int64)
        cols = np.zeros(sz.nnz_struct, dtype=np.int32)
        vals = np.zeros(sz.nnz_struct)
        lo = np.zeros(sz.nrows)
        hi = np.zeros(sz.nrows)
        self._check(self._lib.miqp_b200_assemble(
            self._h, C.byref(cp), rowptr.ctypes.data_as(C.POINTER(C.c_long)), cols.ctypes.data_as(_ip),
            vals.ctypes.data_as(_dp), lo.ctypes.data_as(_dp), hi.ctypes.data_as(_dp)), "miqp_b200_assemble")
        return rowptr, cols, vals, lo, hi

    def assemble_batch(self, plans, repeats: int = 5):
        """Row instantiation of a batch on the device (buffers stay in HBM): (ms per pass, rows, structural nnz)."""
        keep = []
        arr = (CProblem * len(plans))(*[to_c(p, keep=keep) for p in plans])
        ms, rows, nnz = C.c_float(), C.c_long(), C.c_long()
        f = self._lib.miqp_b200_assemble_batch
        f.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_long), C.POINTER(C.c_long)]
        self._check(f(self._h, arr, len(plans), int(repeats), C.byref(ms), C.byref(rows), C.byref(nnz)), "miqp_b200_assemble_batch")
        return ms.value, rows.value, nnz.value

    def evaluate(self, p, x):
        keep = []
        cp = to_c(p, keep=keep)
        x = np.ascontiguousarray(x, dtype=np.float64)
        obj = C.c_double()
        viol = C.c_double()
        self._check(self._lib.miqp_b200_evaluate(self._h, C.byref(cp), x.ctypes.data_as(_dp),
                                                 C.byref(obj), C.byref(viol)), "miqp_b200_evaluate")
        return obj.value, viol.value

    # ---- solve ---------------------------------------------------------------------
    def _pack(self, problems, gap_tol, time_limit, warm):
        n = len(problems)
        keep = []
        arr = (CProblem * n)()
        for k, p in enumerate(problems):
            arr[k] = to_c(p, gap_tol, time_limit, keep)
        warm_arr = None
        if warm is not None:
            warm_arr = (_dp * n)()
            for k, w in enumerate(warm):
                if w is not None:
                    a, ptr = _d(w)
                    keep.append(a)
                    warm_arr[k] = ptr
        ncols = [ncols_of(p) for p in problems]
        return arr, warm_arr, ncols, keep

    def prepare(self, problems, gap_tol=None, time_limit=None, warm=None):
        """Builds the C structs and the output buffers of a batch once (host memory); the result can be
        passed to solve_prepared() repeatedly.  What a C/C++ caller of the ABI holds anyway."""
        n = len(problems)
        arr, warm_arr, ncols, keep = self._pack(problems, gap_tol, time_limit, warm)
        xs = [np.zeros(c) for c in ncols]
        xptr = (_dp * n)(*[x.ctypes.data_as(_dp) for x in xs])
        infos = (CSolveInfo * n)()
        return dict(n=n, arr=arr, warm=warm_arr, xs=xs, xptr=xptr, infos=infos, keep=keep, problems=list(problems))

    def solve_prepared(self, b):
        """One miqp_b200_solve_batch call on host buffers: pack + H2D + device solve + D2H."""
        self._check(self._lib.miqp_b200_solve_batch(self._h, b["arr"], b["n"], b["warm"], b["xptr"], b["infos"]),
                    "miqp_b200_solve_batch")
        self._batch = (b["n"], [len(x) for x in b["xs"]]); self._shapes = [(p.C, p.N) for p in b["problems"]]
        return b["xs"], b["infos"]

    def solve_batch(self, problems, gap_tol=None, time_limit=None, warm=None):
        """Host buffers in, host buffers out (H2D + solve + D2H).  Returns (xs, infos)."""
        n = len(problems)
        arr, warm_arr, ncols, keep = self._pack(problems, gap_tol, time_limit, warm)
        xs = [np.zeros(c) for c in ncols]
        xptr = (_dp * n)(*[x.ctypes.data_as(_dp) for x in xs])
        infos = (CSolveInfo * n)()
        self._check(self._lib.miqp_b200_solve_batch(self._h, arr, n, warm_arr, xptr, infos), "miqp_b200_solve_batch")
        self._batch = (n, ncols); self._shapes = [(p.C, p.N) for p in problems]
        return xs, [self._info(i) for i in infos]

    def solve(self, p, gap_tol=None, time_limit=None, warm=None):
        xs, infos = self.solve_batch([p], gap_tol, time_limit, None if warm is None else [warm])
        return xs[0], infos[0]

    def upload(self, problems, gap_tol=None, time_limit=None, warm=None):
        n = len(problems)
        arr, warm_arr, ncols, keep = self._pack(problems, gap_tol, time_limit, warm)
        self._check(self._lib.miqp_b200_batch_upload(self._h, arr, n, warm_arr), "miqp_b200_batch_upload")
        self._batch = (n, ncols); self._shapes = [(p.C, p.N) for p in problems]

    def fetch_compact(self):
        """trajectories [C][N][8] per plan + infos (miqp_b200_batch_fetch_compact); the full vectors stay on the device"""
        n, ncols = self._batch
        shapes = self._shapes if getattr(self, "_shapes", None) and len(self._shapes) == n else None
        if shapes is None:
            raise MiqpB200Error("fetch_compact needs upload() / upload_prepared() of this batch")
        tr = [np.zeros((c, nn, 8)) for c, nn in shapes]
        tptr = (_dp * n)(*[t.ctypes.data_as(_dp) for t in tr])
        infos = (CSolveInfo * n)()
        self._lib.miqp_b200_batch_fetch_compact.argtypes = [C.c_void_p, C.POINTER(_dp), C.POINTER(CSolveInfo)]
        self._check(self._lib.miqp_b200_batch_fetch_compact(self._h, tptr, infos), "miqp_b200_batch_fetch_compact")
        return tr, [self._info(i) for i in infos]

    def fetch_vector(self, k: int) -> np.ndarray:
        n, ncols = self._batch
        x = np.zeros(ncols[k])
        self._lib.miqp_b200_fetch_vector.argtypes = [C.c_void_p, C.c_int, _dp]
        self._check(self._lib.miqp_b200_fetch_vector(self._h, int(k), x.ctypes.data_as(_dp)), "miqp_b200_fetch_vector")
        return x

    # ---- solution pool ---------------------------------------------------------------
    def set_solution_pool(self, capacity: int):
        """keep up to `capacity` (1..64) best distinct integer-feasible plans per problem from the next upload on; 0 = off"""
        self._check(self._lib.miqp_b200_set_solution_pool(self._h, int(capacity)), "miqp_b200_set_solution_pool")

    def pool_sizes(self) -> np.ndarray:
        """number of pool entries of every plan of the last run"""
        out = np.zeros(self._batch[0], dtype=np.int32)
        self._check(self._lib.miqp_b200_pool_sizes(self._h, out.ctypes.data_as(_ip)), "miqp_b200_pool_sizes")
        return out

    def pool(self, k: int, vectors: bool = True, max_entries: int = 64) -> list[PoolEntry]:
        """pool of plan k, best first (entry 0 is the incumbent); vectors: also the full column vectors and trajectories"""
        n, ncols = self._batch
        if not 0 <= k < n:
            raise IndexError(k)
        m = int(max_entries)
        ents = (CPoolEntry * max(m, 1))()
        x = tr = None
        if vectors:
            c, nn = self._shapes[k]
            x = np.zeros((m, ncols[k]))
            tr = np.zeros((m, c, nn, 8))
        got = C.c_int()
        self._check(self._lib.miqp_b200_pool_fetch(self._h, int(k), m, ents, None if x is None else x.ctypes.data_as(_dp),
                                                   None if tr is None else tr.ctypes.data_as(_dp), C.byref(got)),
                    "miqp_b200_pool_fetch")
        return [PoolEntry(e.objective, e.max_violation, e.search_value, bool(e.converged), e.round, e.uid,
                          None if x is None else x[j].copy(), None if tr is None else tr[j].copy())
                for j, e in enumerate(ents[:got.value])]

    def pool_export(self):
        """this solver's pool packed for an all-gather (miqp_b200_pool_export): a torch.uint8 CUDA tensor that views the
        solver's export buffer without a copy; valid until the next pool_export, upload or close"""
        import torch
        ptr, n = C.c_void_p(), C.c_size_t()
        self._check(self._lib.miqp_b200_pool_export(self._h, C.byref(ptr), C.byref(n)), "miqp_b200_pool_export")
        return torch.as_tensor(_DevView(ptr.value, n.value, "|u1"), device=torch.device("cuda", self._device))

    def pool_merge(self, gathered, world: int):
        """replaces this solver's pool by the merge of `world` exports stored back to back in `gathered` (a CPU or CUDA
        tensor, miqp_b200_pool_merge): the pool of the union of the ranks' leaves"""
        import torch
        g = gathered.contiguous()
        if g.is_cuda:
            torch.cuda.synchronize(g.device)      # the C call reads it on the solver's own stream
        self._check(self._lib.miqp_b200_pool_merge(self._h, C.c_void_p(g.data_ptr()), int(world)), "miqp_b200_pool_merge")

    def solve_prepared_compact(self, b, on_plan=None):
        """One miqp_b200_solve_batch_compact call on host buffers: pack + H2D + device solve + D2H of trajectories and infos.
        on_plan(k, traj, info): a streaming run (run_streaming) instead, with the same results."""
        if on_plan is not None:
            self.upload_prepared(b)
            self.run_streaming(on_plan)
            if "traj" not in b:
                b["traj"] = [np.zeros((p.C, p.N, 8)) for p in b["problems"]]
                b["tptr"] = (_dp * b["n"])(*[t.ctypes.data_as(_dp) for t in b["traj"]])
            self._lib.miqp_b200_batch_fetch_compact.argtypes = [C.c_void_p, C.POINTER(_dp), C.POINTER(CSolveInfo)]
            self._check(self._lib.miqp_b200_batch_fetch_compact(self._h, b["tptr"], b["infos"]), "miqp_b200_batch_fetch_compact")
            return b["traj"], b["infos"]
        if "traj" not in b:
            b["traj"] = [np.zeros((p.C, p.N, 8)) for p in b["problems"]]
            b["tptr"] = (_dp * b["n"])(*[t.ctypes.data_as(_dp) for t in b["traj"]])
        self._lib.miqp_b200_solve_batch_compact.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int, C.POINTER(_dp), C.POINTER(_dp), C.POINTER(CSolveInfo)]
        self._check(self._lib.miqp_b200_solve_batch_compact(self._h, b["arr"], b["n"], b["warm"], b["tptr"], b["infos"]), "miqp_b200_solve_batch_compact")
        self._batch = (b["n"], [len(x) for x in b["xs"]]); self._shapes = [(p.C, p.N) for p in b["problems"]]
        return b["traj"], b["infos"]

    def upload_replan(self, problems, gap_tol=None, time_limit=None):
        """next planning cycle of the previous batch: MIP starts = previous incumbents shifted by one step on the device"""
        n = len(problems)
        arr, _, ncols, keep = self._pack(problems, gap_tol, time_limit, None)
        self._lib.miqp_b200_batch_upload_replan.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int]
        self._check(self._lib.miqp_b200_batch_upload_replan(self._h, arr, n), "miqp_b200_batch_upload_replan")
        self._batch = (n, ncols); self._shapes = [(p.C, p.N) for p in problems]

    def upload_replan_prepared(self, b):
        self._lib.miqp_b200_batch_upload_replan.argtypes = [C.c_void_p, C.POINTER(CProblem), C.c_int]
        self._check(self._lib.miqp_b200_batch_upload_replan(self._h, b["arr"], b["n"]), "miqp_b200_batch_upload_replan")
        self._batch = (b["n"], [len(x) for x in b["xs"]]); self._shapes = [(p.C, p.N) for p in b["problems"]]

    def upload_prepared(self, b):
        """miqp_b200_batch_upload of a batch built by prepare() (no Python-side packing)."""
        self._check(self._lib.miqp_b200_batch_upload(self._h, b["arr"], b["n"], b["warm"]), "miqp_b200_batch_upload")
        self._batch = (b["n"], [len(x) for x in b["xs"]]); self._shapes = [(p.C, p.N) for p in b["problems"]]

    def run(self) -> float:
        ms = C.c_float()
        self._check(self._lib.miqp_b200_batch_run(self._h, C.byref(ms)), "miqp_b200_batch_run")
        return ms.value

    def run_streaming(self, on_plan) -> float:
        """miqp_b200_batch_run_streaming: the same run as run(), with on_plan(k, traj, info) called for every plan as soon as its
        search ends (on this thread, between rounds, ascending k within a round; traj is a copy [C][N][8], info a SolveInfo whose
        `rounds` is the rounds run when the plan finished).  fetch() and the other results afterwards are those of run().  An
        exception raised by on_plan stops the calls to it; the run finishes and the exception is raised here.  Returns the
        device time in ms."""
        shapes = getattr(self, "_shapes", None)   # (None before an upload: the C call refuses the run)
        failed = []

        def cb(_user, k, traj, info):
            if failed:
                return
            try:
                c, nn = shapes[k]
                t = np.ctypeslib.as_array(traj, shape=(c * nn * 8,)).reshape(c, nn, 8).copy()
                on_plan(k, t, self._info(info.contents))
            except BaseException as ex:   # ctypes would print and drop it
                failed.append(ex)

        return self._run_streaming_raw(PLAN_DONE(cb), failed)

    def _run_streaming_raw(self, cfunc, failed):
        ms = C.c_float()
        rc = self._lib.miqp_b200_batch_run_streaming(self._h, cfunc, None, C.byref(ms))
        if failed:
            raise failed[0]
        self._check(rc, "miqp_b200_batch_run_streaming")
        return ms.value

    def solve_batch_streaming(self, problems, gap_tol=None, time_limit=None, warm=None):
        """Generator of (k, traj, info) in the order the plans finish: upload + run_streaming on a worker thread (the C call
        releases the GIL), results through a queue.  Closing the generator early waits for the run to end, so no thread is left
        behind; the solver is busy until the generator is exhausted or closed.  fetch() etc. afterwards give the whole batch."""
        self.upload(problems, gap_tol, time_limit, warm)
        return _stream_results(lambda on_plan: self.run_streaming(on_plan))

    def fetch(self):
        n, ncols = self._batch
        xs = [np.zeros(c) for c in ncols]
        xptr = (_dp * n)(*[x.ctypes.data_as(_dp) for x in xs])
        infos = (CSolveInfo * n)()
        self._check(self._lib.miqp_b200_batch_fetch(self._h, xptr, infos), "miqp_b200_batch_fetch")
        return xs, [self._info(i) for i in infos]

    # ---- the search in steps (frontier sharding, sharding.py:solve_frontier_sharded) -----------
    def frontier_start(self):
        self._lib.miqp_b200_frontier_start.argtypes = [C.c_void_p]
        self._check(self._lib.miqp_b200_frontier_start(self._h), "miqp_b200_frontier_start")

    def frontier_rounds(self, nrounds: int) -> int:
        left = C.c_int()
        self._lib.miqp_b200_frontier_rounds.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        self._check(self._lib.miqp_b200_frontier_rounds(self._h, int(nrounds), C.byref(left)), "miqp_b200_frontier_rounds")
        return left.value

    def frontier_split(self, rank: int, world: int):
        self._lib.miqp_b200_frontier_split.argtypes = [C.c_void_p, C.c_int, C.c_int]
        self._check(self._lib.miqp_b200_frontier_split(self._h, int(rank), int(world)), "miqp_b200_frontier_split")

    def frontier_get_ub(self) -> np.ndarray:
        ub = np.zeros(self._batch[0])
        self._lib.miqp_b200_frontier_get_ub.argtypes = [C.c_void_p, _dp]
        self._check(self._lib.miqp_b200_frontier_get_ub(self._h, ub.ctypes.data_as(_dp)), "miqp_b200_frontier_get_ub")
        return ub

    def frontier_fingerprint(self) -> np.ndarray:
        fp = np.zeros(self._batch[0], dtype=np.int64)
        self._lib.miqp_b200_frontier_fingerprint.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
        self._check(self._lib.miqp_b200_frontier_fingerprint(self._h, fp.ctypes.data_as(C.POINTER(C.c_longlong))), "miqp_b200_frontier_fingerprint")
        return fp

    def frontier_ub_device(self):
        """(device address, count) of the incumbent objectives, for an in-place NCCL min-allreduce"""
        ptr, n = C.c_void_p(), C.c_int()
        self._lib.miqp_b200_frontier_ub_device.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]
        self._check(self._lib.miqp_b200_frontier_ub_device(self._h, C.byref(ptr), C.byref(n)), "miqp_b200_frontier_ub_device")
        return ptr.value, n.value

    def frontier_tighten(self, ub):
        ub = np.ascontiguousarray(ub, dtype=np.float64)
        self._lib.miqp_b200_frontier_tighten.argtypes = [C.c_void_p, _dp]
        self._check(self._lib.miqp_b200_frontier_tighten(self._h, ub.ctypes.data_as(_dp)), "miqp_b200_frontier_tighten")

    def frontier_finish(self) -> float:
        ms = C.c_float()
        self._lib.miqp_b200_frontier_finish.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        self._check(self._lib.miqp_b200_frontier_finish(self._h, C.byref(ms)), "miqp_b200_frontier_finish")
        return ms.value

    def mark(self, which: int):
        self._lib.miqp_b200_mark.argtypes = [C.c_void_p, C.c_int]
        self._check(self._lib.miqp_b200_mark(self._h, int(which)), "miqp_b200_mark")

    def elapsed_to(self, other: "Solver") -> float:
        """device milliseconds from this solver's mark 0 to `other`'s mark 1"""
        ms = C.c_float()
        self._lib.miqp_b200_elapsed.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        self._check(self._lib.miqp_b200_elapsed(self._h, other._h, C.byref(ms)), "miqp_b200_elapsed")
        return ms.value

    def run_stats(self) -> dict:
        st = CRunStats()
        self._check(self._lib.miqp_b200_run_stats(self._h, C.byref(st)), "miqp_b200_run_stats")
        return {n: getattr(st, n) for n, _ in CRunStats._fields_}

    def debug_traces(self):
        import numpy as _np
        out = _np.zeros(4096)
        self._check(self._lib.miqp_b200_debug_traces(self._h, out.ctypes.data_as(_dp)), "miqp_b200_debug_traces")
        return out.reshape(8, 512)

    def debug_profile(self):
        out = (C.c_ulonglong * 256)()
        self._check(self._lib.miqp_b200_debug_profile(self._h, out), "miqp_b200_debug_profile")
        return list(out)

    def measure_fp64_peak(self) -> float:
        tf = C.c_double()
        self._check(self._lib.miqp_b200_measure_fp64_peak(self._h, C.byref(tf)), "miqp_b200_measure_fp64_peak")
        return tf.value

    @staticmethod
    def _info(i: CSolveInfo) -> SolveInfo:
        return SolveInfo(i.status, bool(i.proven), i.objective, i.best_bound, i.gap, i.seconds,
                         i.max_violation, i.nodes, i.qp_iters, i.rounds, i.uncertified, i.pool_exhausted)


class PipelinedSolver:
    """`depth` solver instances on ONE GPU (own stream, node pool and pinned staging buffers each), fed alternately by host
    threads, so that consecutive batches overlap:

    * the tail rounds of batch k (a few hard plans, a near-empty GPU, latency-bound) run next to the head rounds of batch
      k + 1 (every plan active, throughput-bound) -- the persistent node kernels of the two streams share the SMs as their
      CTAs come and go;
    * packing + H2D of batch k + 1 and D2H + scatter of batch k - 1 run on the host threads of the idle instance while the
      other one searches.

    The C calls release the GIL.  Results are identical to Solver.solve_batch (each batch is still one deterministic search).
    """

    def __init__(self, device: int = 0, depth: int = 2, **kw):
        self.solvers = [Solver(device=device, **kw) for _ in range(max(1, depth))]

    def close(self):
        for s in self.solvers:
            s.close()

    def prepare(self, problems, gap_tol=None, time_limit=None, warm=None):
        return self.solvers[0].prepare(problems, gap_tol, time_limit, warm)

    def _run_threads(self, jobs, fn, stagger_s):
        import threading
        import time as _t
        depth = len(self.solvers)
        out, err = [None] * len(jobs), []

        def worker(w):
            try:
                if stagger_s > 0 and w > 0:
                    _t.sleep(stagger_s * w / depth)
                for k in range(w, len(jobs), depth):
                    out[k] = fn(self.solvers[w], jobs[k])
            except Exception as ex:        # surfaced by the caller
                err.append(ex)
        ths = [threading.Thread(target=worker, args=(w,)) for w in range(depth)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if err:
            raise err[0]
        return out

    def solve_stream(self, prepared_batches, stagger_s: float = 0.0):
        """miqp_b200_solve_batch of every prepared batch (host buffers in and out), batch k on instance k mod depth.
        Two batches that are in flight together must not share their prepared buffers.  Returns [(xs, infos), ...]."""
        return self._run_threads(list(prepared_batches), lambda s, b: s.solve_prepared(b), stagger_s)

    def solve_stream_compact(self, prepared_batches, stagger_s: float = 0.0, on_plan=None):
        """solve_stream with compact results (trajectories + infos; the full vectors stay on the device).  on_plan(batch_index,
        k, traj, info): every plan as soon as its search ends (Solver.run_streaming), called from the instance's worker thread."""
        jobs = list(enumerate(prepared_batches))
        if on_plan is None:
            return self._run_threads(jobs, lambda s, j: s.solve_prepared_compact(j[1]), stagger_s)
        return self._run_threads(jobs, lambda s, j: s.solve_prepared_compact(
            j[1], on_plan=lambda k, t, i, bi=j[0]: on_plan(bi, k, t, i)), stagger_s)

    def upload_resident(self, prepared_batches):
        """one resident batch per instance (miqp_b200_batch_upload)"""
        for s, b in zip(self.solvers, prepared_batches):
            s.upload_prepared(b)

    def run_resident(self, runs: int, stagger_s: float = 0.0, on_plan=None):
        """`runs` searches over the resident batches (miqp_b200_batch_run), run k on instance k mod depth; returns the
        device time of every run (CUDA events on its own stream; the runs overlap, so their sum exceeds the wall time).
        on_plan(run_index, k, traj, info): streaming runs (Solver.run_streaming), called from the instance's worker thread."""
        if on_plan is None:
            return self._run_threads(list(range(runs)), lambda s, k: s.run(), stagger_s)
        return self._run_threads(list(range(runs)), lambda s, r: s.run_streaming(lambda k, t, i: on_plan(r, k, t, i)), stagger_s)

    def timed_resident(self, runs: int, stagger_s: float = 0.0):
        """run_resident, timed on the device: CUDA events on the solvers' own streams, from the start of the first run to the
        end of the last one on either stream.  Returns (total device ms, per-run device ms)."""
        self.solvers[0].mark(0)
        per_run = self.run_resident(runs, stagger_s)
        for s in self.solvers:
            s.mark(1)
        return max(self.solvers[0].elapsed_to(s) for s in self.solvers), per_run


_DONE = object()


def _stream_results(run):
    """Generator over the plans a streaming run delivers: run(on_plan) executes on a worker thread and feeds a queue; the
    run's exception, if any, is raised after the plans delivered before it.  Closing the generator joins the thread."""
    q = queue.Queue()
    stop = threading.Event()

    def on_plan(k, traj, info):
        if not stop.is_set():
            q.put((k, traj, info))

    def work():
        try:
            run(on_plan)
            q.put(_DONE)
        except BaseException as ex:
            q.put(ex)

    th = threading.Thread(target=work, name="miqp_b200-streaming", daemon=True)
    th.start()
    try:
        while True:
            item = q.get()
            if item is _DONE:
                return
            if isinstance(item, BaseException):
                raise item
            yield item
    finally:
        stop.set()
        th.join()
