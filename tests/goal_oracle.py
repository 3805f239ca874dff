"""ctypes binding of oracle/goals/liboracle_goals.so: the oracle's planning query for every GoalConstraint type
(XYZ, XYZ_RPY, JOINT_STATE), on the scenes of oracle_api.OracleScene.  Goal records are smpl_b200.api.GOAL_DTYPE."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_api import _bp, _dp, _ip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(ROOT, "oracle", "goals", "liboracle_goals.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        L.oracle_plan_goal.restype = C.c_double
        dp, ip, bp, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_int, C.c_double
        L.oracle_plan_goal.argtypes = [C.c_void_p, dp, i, dp, dp, d, dp, dp, dp, dp, bp, dp, i, i, d, d, i, ip, ip, i, dp]
        L.oracle_rpy_goal_angles.argtypes = [dp, i, dp, dp]
        _LIB = L
    return _LIB


def plan(o, start, goal, params, max_path=4096):
    """o: oracle_api.OracleScene (kinematics and heuristic set up); goal: one GOAL_DTYPE record; params:
    smpl_b200.scenes.PlanParams.  Returns dict(success, expansions, cost, path_ids, num_states, path_states, seconds)
    like OracleScene.plan."""
    start = np.ascontiguousarray(start, dtype=np.float64)
    dof = len(start)
    rec = goal.reshape(()) if isinstance(goal, np.ndarray) else goal
    pose = np.ascontiguousarray(rec["pose"], dtype=np.float64)
    tol = np.ascontiguousarray(rec["xyz_tolerance"], dtype=np.float64)
    angles = np.ascontiguousarray(rec["angles"][:dof], dtype=np.float64)
    atol = np.ascontiguousarray(rec["angle_tolerances"][:dof], dtype=np.float64)
    res = np.ascontiguousarray(params.resolutions, dtype=np.float64)
    prims = np.ascontiguousarray(params.mprims, dtype=np.float64)
    flags = np.ascontiguousarray(params.short_flags, dtype=np.uint8)
    w = getattr(params, "weights", None)
    w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    summary = np.zeros(8, np.int32)
    path = np.zeros(max_path, np.int32)
    pstates = np.zeros((max_path, dof), np.float64)
    secs = lib().oracle_plan_goal(o.h, _dp(start), int(rec["type"]), _dp(pose), _dp(tol), float(rec["rpy_tolerance"]),
                                  _dp(angles), _dp(atol), _dp(res), _dp(prims), _bp(flags), None if w is None else _dp(w),
                                  len(prims), int(params.use_short_dist), float(params.short_dist_thresh),
                                  float(params.epsilon), int(params.max_expansions), _ip(summary), _ip(path), max_path,
                                  _dp(pstates))
    assert secs >= 0.0, "unknown goal type or scene without kinematics / heuristic"
    n = int(summary[3])
    assert int(summary[5]) == n, "extractPath failed"
    return dict(success=bool(summary[0]), expansions=int(summary[1]), cost=int(summary[2]),
                path_ids=path[:min(n, max_path)].copy(), num_states=int(summary[4]),
                path_states=pstates[:min(n, max_path)].copy(), seconds=float(secs))


def rpy_goal_angles(rpy, goal_rpy):
    """XYZ_RPY_GOAL's angle between state orientations rpy[n][3] and goal orientations goal_rpy[n][3].
    Returns (theta[n], q . qg[n] before the sign flip)."""
    pairs = np.ascontiguousarray(np.concatenate([np.asarray(rpy, np.float64).reshape(-1, 3),
                                                 np.asarray(goal_rpy, np.float64).reshape(-1, 3)], axis=1))
    theta = np.zeros(len(pairs))
    d = np.zeros(len(pairs))
    lib().oracle_rpy_goal_angles(_dp(pairs), len(pairs), _dp(theta), _dp(d))
    return theta, d
