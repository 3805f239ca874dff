"""ctypes binding of the oracle's goal-set planner (oracle_plan_goal_set in oracle/goal_sets/liboracle_goal_sets.so):
the goal-typed planning query with the snap action for a query that succeeds at any record of its goal set.  Goal
records are smpl_b200.api.GOAL_DTYPE, snap settings smpl_b200.api.SnapParams (None = no snap action)."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_api import _bp, _dp, _ip
from smpl_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(ROOT, "oracle", "goal_sets", "liboracle_goal_sets.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        dp, ip, bp, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_int, C.c_double
        L.oracle_plan_goal_set.restype = C.c_double
        L.oracle_plan_goal_set.argtypes = [C.c_void_p, dp, C.c_void_p, i, dp, dp, bp, dp, i, i, d, d, i, dp, i, d, d, i,
                                           d, ip, ip, i, dp, C.POINTER(C.c_int64), ip]
        L.oracle_goal_set_bfs.argtypes = [C.c_void_p, dp, i, ip]
        _LIB = L
    return _LIB


def plan_set(o, T_kin_to_planning, start, goals, params, snap=None, max_path=4096):
    """snap_oracle.plan_snap for a goal set: goals is a GOAL_DTYPE array of 1 to 64 records.  The result also has
    reached_goal (the record the path's goal action satisfies first; -1 when unsolved)."""
    start = np.ascontiguousarray(start, dtype=np.float64)
    dof = len(start)
    goals = np.ascontiguousarray(np.asarray(goals).reshape(-1))
    assert goals.dtype == api.GOAL_DTYPE
    T = np.ascontiguousarray(np.asarray(T_kin_to_planning, np.float64).reshape(3, 4))
    res = np.ascontiguousarray(params.resolutions, dtype=np.float64)
    prims = np.ascontiguousarray(params.mprims, dtype=np.float64)
    flags = np.ascontiguousarray(params.short_flags, dtype=np.uint8)
    w = getattr(params, "weights", None)
    w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
    en = snap is not None and bool(snap.enabled)
    summary = np.zeros(8, np.int32)
    path = np.zeros(max_path, np.int32)
    pstates = np.zeros((max_path, dof), np.float64)
    counters = np.zeros(2, np.int64)
    reached = np.zeros(1, np.int32)
    secs = lib().oracle_plan_goal_set(
        o.h, _dp(start), goals.ctypes.data, len(goals), _dp(res), _dp(prims), _bp(flags), None if w is None else _dp(w),
        len(prims), int(params.use_short_dist), float(params.short_dist_thresh), float(params.epsilon),
        int(params.max_expansions), _dp(T), int(en), float(snap.dist_thresh) if snap is not None else 0.0,
        float(snap.weight) if snap is not None else 0.5, int(snap.max_iterations) if snap is not None else 100,
        float(snap.tolerance) if snap is not None else 1e-6, _ip(summary), _ip(path), max_path, _dp(pstates),
        counters.ctypes.data_as(C.POINTER(C.c_int64)), _ip(reached))
    assert secs >= 0.0, "bad goal set or scene without kinematics / heuristic"
    n = int(summary[3])
    assert int(summary[5]) == n, "extractPath failed"
    return dict(success=bool(summary[0]), expansions=int(summary[1]), cost=int(summary[2]),
                path_ids=path[:min(n, max_path)].copy(), num_states=int(summary[4]),
                path_states=pstates[:min(n, max_path)].copy(), seconds=float(secs),
                ik_attempted=int(counters[0]), ik_converged=int(counters[1]), reached_goal=int(reached[0]))


def goal_set_bfs(o, xyz):
    """The scene heuristic's BFS after seeding it at every position of xyz (n, 3), as the goal-set planner does.
    Returns (seeds in bounds, padded distance grid as oracle_api.OracleScene.heur_grid gives it)."""
    xyz = np.ascontiguousarray(np.asarray(xyz, np.float64).reshape(-1, 3))
    out = np.zeros_like(o.heur_grid())
    k = lib().oracle_goal_set_bfs(o.h, _dp(xyz), len(xyz), _ip(out))
    assert k >= 0
    return k, out
