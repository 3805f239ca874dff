"""ctypes binding of oracle/snap_kinds/liboracle_snap_kinds.so: the oracle's goal-set planner with the three snap kinds
SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY (oracle_plan_goal_set_snaps) and its position-only planning-link IK
(oracle_planning_link_ik_position).  Goal records are smpl_b200.api.GOAL_DTYPE, snap settings smpl_b200.api.SnapParams
(None = no snap action)."""
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
        path = os.path.join(ROOT, "oracle", "snap_kinds", "liboracle_snap_kinds.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        dp, ip, bp, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_int, C.c_double
        L.oracle_plan_goal_set_snaps.restype = C.c_double
        L.oracle_plan_goal_set_snaps.argtypes = [C.c_void_p, dp, C.c_void_p, i, dp, dp, bp, dp, i, i, d, d, i, dp, ip,
                                                 dp, d, i, d, ip, ip, i, dp, C.POINTER(C.c_int64), ip]
        L.oracle_planning_link_ik_position.argtypes = [C.c_void_p, dp, dp, dp, i, i, d, dp, bp, ip]
        _LIB = L
    return _LIB


def plan_set_snaps(o, T_kin_to_planning, start, goals, params, snap=None, max_path=4096):
    """goal_set_oracle.plan_set with the snap kinds of snap (SnapParams: enabled / dist_thresh for SNAP_TO_XYZ_RPY,
    xyz_dist_thresh and rpy_dist_thresh for the other two).  The result also has ik_by_kind, (3, 2) int: per
    api.SNAP_* kind the IK solves the search ran and how many converged; ik_attempted / ik_converged are their sums."""
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
    en, th = snap.kinds() if snap is not None else ([False] * 3, [0.0] * 3)
    en = np.asarray(en, np.int32)
    th = np.asarray(th, np.float64)
    summary = np.zeros(8, np.int32)
    path = np.zeros(max_path, np.int32)
    pstates = np.zeros((max_path, dof), np.float64)
    counters = np.zeros(6, np.int64)
    reached = np.zeros(1, np.int32)
    secs = lib().oracle_plan_goal_set_snaps(
        o.h, _dp(start), goals.ctypes.data, len(goals), _dp(res), _dp(prims), _bp(flags), None if w is None else _dp(w),
        len(prims), int(params.use_short_dist), float(params.short_dist_thresh), float(params.epsilon),
        int(params.max_expansions), _dp(T), _ip(en), _dp(th), float(snap.weight) if snap is not None else 0.5,
        int(snap.max_iterations) if snap is not None else 100, float(snap.tolerance) if snap is not None else 1e-6,
        _ip(summary), _ip(path), max_path, _dp(pstates), counters.ctypes.data_as(C.POINTER(C.c_int64)), _ip(reached))
    assert secs >= 0.0, "bad goal set or scene without kinematics / heuristic"
    n = int(summary[3])
    assert int(summary[5]) == n, "extractPath failed"
    by_kind = counters.reshape(3, 2).copy()
    return dict(success=bool(summary[0]), expansions=int(summary[1]), cost=int(summary[2]),
                path_ids=path[:min(n, max_path)].copy(), num_states=int(summary[4]),
                path_states=pstates[:min(n, max_path)].copy(), seconds=float(secs),
                ik_attempted=int(by_kind[:, 0].sum()), ik_converged=int(by_kind[:, 1].sum()), ik_by_kind=by_kind,
                reached_goal=int(reached[0]))


def planning_link_ik_position(o, T_kin_to_planning, xyz, seeds, max_iterations=100, tolerance=1e-6):
    """The oracle's position-only planning-link IK: xyz (n, 3) target-offset positions, seeds (n, dof).
    Returns (q (n, dof), ok (n,) bool, iterations (n,))."""
    xyz = np.ascontiguousarray(np.asarray(xyz, np.float64).reshape(-1, 3))
    seeds = np.ascontiguousarray(np.asarray(seeds, np.float64).reshape(len(xyz), -1))
    T = np.ascontiguousarray(np.asarray(T_kin_to_planning, np.float64).reshape(3, 4))
    n, dof = seeds.shape
    q = np.zeros((n, dof))
    ok = np.zeros(n, np.uint8)
    it = np.zeros(n, np.int32)
    r = lib().oracle_planning_link_ik_position(o.h, _dp(T), _dp(xyz), _dp(seeds), n, int(max_iterations),
                                               float(tolerance), _dp(q), _bp(ok), _ip(it))
    assert r >= 0, "scene without kinematics"
    return q, ok.astype(bool), it
