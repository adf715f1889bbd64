"""ctypes binding of libmiqp_planner_c_api.so (include/miqp_planner_c_api.h): the planner-level C ABI
that Apollo links in the reference (src/miqp_planner_c_api.h:21-226), backed here by the C++ host
facade (planner-miqp_b200/host/) and the CUDA solver library."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
TRAJECTORY_SIZE = 9

C_API_SYMBOLS = [
    "NewCMiqpPlanner", "NewCMiqpPlannerSettings", "DelCMiqpPlanner", "AddCarCMiqpPlanner", "PlanCMiqpPlanner",
    "UpdateCarCMiqpPlanner", "ActivateDebugFileWriteCMiqpPlanner", "GetNCMiqpPlanner", "GetTsCMiqpPlanner",
    "GetCollisionRadius", "GetRawCMiqpTrajectoryCMiqpPlanner", "GetRawCLastReferenceTrajectoryCMiqpPlaner",
    "UpdateConvexifiedMapCMiqpPlaner", "UpdateDesiredVelocityCMiqpPlanner", "AddObstacleCMiqpPlanner",
    "UpdateObstacleCMiqpPlanner", "RemoveAllObstaclesCMiqpPlanner",
    # additions of this backend
    "PlanBatchCMiqpPlanner", "GetSolutionPropertiesCMiqpPlanner", "DeviceWarmstartBatchesCMiqpPlanner",
]
# include/miqp_planner_solution_pool.h
SOLUTION_POOL_SYMBOLS = [
    "SetSolutionPoolCapacityCMiqpPlanner", "GetSolutionPoolSizeCMiqpPlanner", "GetSolutionPoolTrajectoryCMiqpPlanner",
]


class MiqpPlannerSettings(C.Structure):
    """field-for-field include/miqp_planner_settings.h"""
    _fields_ = [
        ("nr_regions", C.c_int), ("nr_steps", C.c_int), ("nr_neighbouring_possible_regions", C.c_int),
        ("ts", C.c_float), ("precision", C.c_int),
        ("constant_agent_safety_distance_slack", C.c_float), ("minimum_region_change_speed", C.c_float),
        ("lambda_", C.c_float), ("wheelBase", C.c_float), ("collisionRadius", C.c_float),
        ("slackWeight", C.c_float), ("slackWeightObstacle", C.c_float), ("jerkWeight", C.c_float),
        ("positionWeight", C.c_float), ("velocityWeight", C.c_float), ("acclerationWeight", C.c_float),
        ("accLonMaxLimit", C.c_float), ("accLonMinLimit", C.c_float), ("jerkLonMaxLimit", C.c_float),
        ("accLatMinMaxLimit", C.c_float), ("jerkLatMinMaxLimit", C.c_float),
        ("simplificationDistanceMap", C.c_float), ("simplificationDistanceReferenceLine", C.c_float),
        ("bufferReference", C.c_float), ("buffer_for_merging_tolerance", C.c_float), ("refLineInterpInc", C.c_float),
        ("additionalStepsForReferenceLongerHorizon", C.c_int),
        ("max_solution_time", C.c_float), ("relative_mip_gap_tolerance", C.c_float),
        ("mipdisplay", C.c_int), ("mipemphasis", C.c_int), ("relobjdif", C.c_float),
        ("cutpass", C.c_int), ("probe", C.c_int), ("repairtries", C.c_int), ("rinsheur", C.c_int),
        ("varsel", C.c_int), ("mircuts", C.c_int),
        ("cplexModelpath", C.c_char * 1000),
        ("useSos", C.c_bool), ("useBranchingPriorities", C.c_bool),
        ("warmstartType", C.c_int), ("parallelMode", C.c_int),
        ("max_velocity_fitting", C.c_float), ("buffer_cplex_outputs", C.c_bool),
        ("obstacle_roi_filter", C.c_bool), ("obstacle_roi_behind_distance", C.c_float),
        ("obstacle_roi_front_distance", C.c_float), ("obstacle_roi_side_distance", C.c_float),
    ]


def default_settings() -> MiqpPlannerSettings:
    """DefaultSettings() of the reference (src/miqp_planner_data.hpp:190-242)."""
    s = MiqpPlannerSettings()
    s.nr_regions, s.nr_steps, s.nr_neighbouring_possible_regions = 16, 20, 1
    s.ts, s.precision = 0.25, 12
    s.constant_agent_safety_distance_slack, s.minimum_region_change_speed = 3, 2
    s.lambda_, s.wheelBase, s.collisionRadius = 0.5, 2.8, 1
    s.slackWeight, s.slackWeightObstacle, s.jerkWeight, s.positionWeight = 30, 2000, 1, 2
    s.velocityWeight, s.acclerationWeight = 0, 0
    s.accLonMaxLimit, s.accLonMinLimit, s.jerkLonMaxLimit, s.accLatMinMaxLimit, s.jerkLatMinMaxLimit = 2, -4, 3, 1.6, 1.4
    s.simplificationDistanceMap, s.simplificationDistanceReferenceLine = 0.2, 0.05
    s.bufferReference, s.buffer_for_merging_tolerance, s.refLineInterpInc = 1, 0.1, 0.2
    s.additionalStepsForReferenceLongerHorizon = 4
    s.max_solution_time, s.relative_mip_gap_tolerance, s.mipdisplay = 10, 0.1, 2
    s.cplexModelpath = b"cplexmodel/"
    s.warmstartType, s.parallelMode = 0, 1
    s.max_velocity_fitting = 20.0
    s.obstacle_roi_behind_distance, s.obstacle_roi_front_distance, s.obstacle_roi_side_distance = 5, 30, 15
    return s


_lib = None
_dp = C.POINTER(C.c_double)


def library_path() -> str:
    return os.path.join(_HERE, "libmiqp_planner_c_api.so")


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python __graft_entry__.py` (g++ + nvcc build)")
    lib = C.CDLL(path)
    vp, d, i, b = C.c_void_p, C.c_double, C.c_int, C.c_bool
    lib.NewCMiqpPlanner.restype = vp
    lib.NewCMiqpPlannerSettings.restype = vp
    lib.NewCMiqpPlannerSettings.argtypes = [MiqpPlannerSettings]
    lib.DelCMiqpPlanner.argtypes = [vp]
    lib.AddCarCMiqpPlanner.argtypes = [vp, _dp, _dp, i, d, d, d, b]
    lib.AddCarCMiqpPlanner.restype = i
    lib.PlanCMiqpPlanner.argtypes = [vp, d]
    lib.PlanCMiqpPlanner.restype = b
    lib.UpdateCarCMiqpPlanner.argtypes = [vp, i, _dp, _dp, i, d, b]
    lib.ActivateDebugFileWriteCMiqpPlanner.argtypes = [vp, C.c_char_p, C.c_char_p]
    lib.GetNCMiqpPlanner.argtypes = [vp]
    lib.GetNCMiqpPlanner.restype = i
    lib.GetTsCMiqpPlanner.argtypes = [vp]
    lib.GetTsCMiqpPlanner.restype = C.c_float
    lib.GetCollisionRadius.argtypes = [vp]
    lib.GetCollisionRadius.restype = C.c_float
    lib.GetRawCMiqpTrajectoryCMiqpPlanner.argtypes = [vp, i, d, _dp, C.POINTER(i)]
    lib.GetRawCLastReferenceTrajectoryCMiqpPlaner.argtypes = [vp, i, d, _dp, C.POINTER(i)]
    lib.UpdateConvexifiedMapCMiqpPlaner.argtypes = [vp, _dp, i]
    lib.UpdateConvexifiedMapCMiqpPlaner.restype = b
    lib.UpdateDesiredVelocityCMiqpPlanner.argtypes = [vp, i, d, d]
    lib.AddObstacleCMiqpPlanner.argtypes = [vp] + [_dp] * 8 + [i, b, b]
    lib.AddObstacleCMiqpPlanner.restype = i
    lib.UpdateObstacleCMiqpPlanner.argtypes = [vp, i] + [_dp] * 8 + [i, b]
    lib.RemoveAllObstaclesCMiqpPlanner.argtypes = [vp]
    lib.PlanBatchCMiqpPlanner.argtypes = [C.POINTER(vp), i, d, C.POINTER(b)]
    lib.PlanBatchCMiqpPlanner.restype = i
    lib.GetSolutionPropertiesCMiqpPlanner.argtypes = [vp, _dp]
    lib.DebugWriteParametersCMiqpPlanner.argtypes = [vp, C.c_char_p, i]
    lib.DebugWriteParametersCMiqpPlanner.restype = b
    lib.DebugSetSolutionCMiqpPlanner.argtypes = [vp, _dp, i]
    lib.DebugSetSolutionCMiqpPlanner.restype = b
    lib.DebugWarmstartCMiqpPlanner.argtypes = [vp, _dp, i, b]
    lib.DebugWarmstartCMiqpPlanner.restype = i
    lib.SetSolutionPoolCapacityCMiqpPlanner.argtypes = [vp, i]
    lib.SetSolutionPoolCapacityCMiqpPlanner.restype = b
    lib.GetSolutionPoolSizeCMiqpPlanner.argtypes = [vp]
    lib.GetSolutionPoolSizeCMiqpPlanner.restype = i
    lib.GetSolutionPoolTrajectoryCMiqpPlanner.argtypes = [vp, i, i, d, _dp, C.POINTER(i)]
    lib.GetSolutionPoolTrajectoryCMiqpPlanner.restype = d
    _lib = lib
    return lib


def exported_symbols() -> list[str]:
    lib = load_library()
    return [s for s in C_API_SYMBOLS if hasattr(lib, s)]


def _arr(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


class CMiqpPlanner:
    """Thin object wrapper over the C handle (what an Apollo-side caller does in C)."""

    def __init__(self, settings: MiqpPlannerSettings | None = None):
        self.lib = load_library()
        self.h = self.lib.NewCMiqpPlanner() if settings is None else self.lib.NewCMiqpPlannerSettings(settings)
        if not self.h:
            raise ValueError("Invalid number of regions or velocity!")

    def close(self):
        if getattr(self, "h", None):
            self.lib.DelCMiqpPlanner(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add_car(self, state6, ref_xy, v_des, delta_s_des, t=0.0, track=True) -> int:
        s, sp = _arr(state6)
        r, rp = _arr(np.asarray(ref_xy, dtype=np.float64).reshape(-1))
        return self.lib.AddCarCMiqpPlanner(self.h, sp, rp, r.size // 2, v_des, delta_s_des, t, track)

    def update_car(self, idx, state6, ref_xy, t=0.0, track=True):
        s, sp = _arr(state6)
        r, rp = _arr(np.asarray(ref_xy, dtype=np.float64).reshape(-1))
        self.lib.UpdateCarCMiqpPlanner(self.h, idx, sp, rp, r.size // 2, t, track)

    def plan(self, t=0.0) -> bool:
        return bool(self.lib.PlanCMiqpPlanner(self.h, t))

    @property
    def N(self) -> int:
        return self.lib.GetNCMiqpPlanner(self.h)

    @property
    def ts(self) -> float:
        return self.lib.GetTsCMiqpPlanner(self.h)

    def trajectory(self, car=0, t0=0.0) -> np.ndarray:
        out = np.zeros((self.N, TRAJECTORY_SIZE))
        n = C.c_int(0)
        self.lib.GetRawCMiqpTrajectoryCMiqpPlanner(self.h, car, t0, out.ctypes.data_as(_dp), C.byref(n))
        return out[:n.value]

    def last_reference(self, car=0, t0=0.0) -> np.ndarray:
        out = np.zeros((self.N, TRAJECTORY_SIZE))
        n = C.c_int(0)
        self.lib.GetRawCLastReferenceTrajectoryCMiqpPlaner(self.h, car, t0, out.ctypes.data_as(_dp), C.byref(n))
        return out[:n.value]

    def update_map(self, poly_xy) -> bool:
        p, pp = _arr(np.asarray(poly_xy, dtype=np.float64).reshape(-1))
        return bool(self.lib.UpdateConvexifiedMapCMiqpPlaner(self.h, pp, p.size // 2))

    def update_desired_velocity(self, car, v_des, delta_s_des):
        self.lib.UpdateDesiredVelocityCMiqpPlanner(self.h, car, v_des, delta_s_des)

    def _corners(self, corners):
        c = np.asarray(corners, dtype=np.float64).reshape(-1, 4, 2)   # [steps][4 corners][x, y]
        keep = [np.ascontiguousarray(c[:, k, a]) for k in range(4) for a in range(2)]
        return keep, [a.ctypes.data_as(_dp) for a in keep], c.shape[0]

    def add_obstacle(self, corners, is_static=False, is_soft=False) -> int:
        keep, ptrs, n = self._corners(corners)
        return self.lib.AddObstacleCMiqpPlanner(self.h, *ptrs, n, is_static, is_soft)

    def update_obstacle(self, oid, corners, is_static=False):
        keep, ptrs, n = self._corners(corners)
        self.lib.UpdateObstacleCMiqpPlanner(self.h, oid, *ptrs, n, is_static)

    def remove_all_obstacles(self):
        self.lib.RemoveAllObstaclesCMiqpPlanner(self.h)

    def activate_debug_file_write(self, path: str, name: str):
        self.lib.ActivateDebugFileWriteCMiqpPlanner(self.h, path.encode(), name.encode())

    def solution_properties(self) -> dict:
        out = np.zeros(8)
        self.lib.GetSolutionPropertiesCMiqpPlanner(self.h, out.ctypes.data_as(_dp))
        keys = ("objective", "gap", "time", "status", "nodes", "rows", "binaries", "continuous")
        return dict(zip(keys, out.tolist()))

    def set_solution(self, x) -> bool:
        a, ap = _arr(x)
        return bool(self.lib.DebugSetSolutionCMiqpPlanner(self.h, ap, a.size))

    def warmstart_vector(self, ncols: int, relax_last_step: bool = True) -> np.ndarray:
        out = np.zeros(ncols)
        n = self.lib.DebugWarmstartCMiqpPlanner(self.h, out.ctypes.data_as(_dp), ncols, relax_last_step)
        if n != ncols:
            raise ValueError("column count does not match the planner's model")
        return out

    # ---- solution pool (include/miqp_planner_solution_pool.h) ----
    def set_solution_pool(self, capacity: int) -> bool:
        return bool(self.lib.SetSolutionPoolCapacityCMiqpPlanner(self.h, int(capacity)))

    def solution_pool_size(self) -> int:
        return self.lib.GetSolutionPoolSizeCMiqpPlanner(self.h)

    def solution_pool_trajectory(self, j: int, car=0, t0=0.0):
        """(objective, rows like trajectory()) of pool entry j"""
        out = np.zeros((self.N, TRAJECTORY_SIZE))
        n = C.c_int(0)
        obj = self.lib.GetSolutionPoolTrajectoryCMiqpPlanner(self.h, int(j), car, t0, out.ctypes.data_as(_dp), C.byref(n))
        return obj, out[:n.value]

    def write_parameters(self, path: str) -> bool:
        return bool(self.lib.DebugWriteParametersCMiqpPlanner(self.h, path.encode(), 0))


def device_warmstart_batches() -> int:
    lib = load_library()
    lib.DeviceWarmstartBatchesCMiqpPlanner.restype = C.c_long
    return int(lib.DeviceWarmstartBatchesCMiqpPlanner())


def plan_batch(planners, t=0.0):
    lib = load_library()
    n = len(planners)
    hs = (C.c_void_p * n)(*[p.h for p in planners])
    ok = (C.c_bool * n)()
    rc = lib.PlanBatchCMiqpPlanner(hs, n, t, ok)
    if rc < 0:
        raise RuntimeError("PlanBatchCMiqpPlanner failed")
    return [bool(v) for v in ok]
