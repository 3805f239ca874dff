"""ctypes binding of oracle/snap/liboracle_snap.so: the oracle's goal-typed planning query with the snap-to-goal action
(oracle_plan_goal_snap) and its planning-link IK (oracle_planning_link_ik), on the scenes of oracle_api.OracleScene.
Goal records are smpl_b200.api.GOAL_DTYPE, snap settings smpl_b200.api.SnapParams."""
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
        path = os.path.join(ROOT, "oracle", "snap", "liboracle_snap.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        dp, ip, bp, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_int, C.c_double
        L.oracle_plan_goal_snap.restype = C.c_double
        L.oracle_plan_goal_snap.argtypes = [C.c_void_p, dp, i, dp, dp, d, dp, dp, dp, dp, bp, dp, i, i, d, d, i, dp, i, d,
                                            d, i, d, ip, ip, i, dp, C.POINTER(C.c_int64)]
        L.oracle_planning_link_ik.argtypes = [C.c_void_p, dp, dp, dp, i, i, d, dp, bp, ip]
        _LIB = L
    return _LIB


def _goal_args(start, goal, params):
    start = np.ascontiguousarray(start, dtype=np.float64)
    dof = len(start)
    rec = goal.reshape(()) if isinstance(goal, np.ndarray) else goal
    w = getattr(params, "weights", None)
    return dict(start=start, dof=dof, type=int(rec["type"]),
                pose=np.ascontiguousarray(rec["pose"], dtype=np.float64),
                tol=np.ascontiguousarray(rec["xyz_tolerance"], dtype=np.float64), rpy_tol=float(rec["rpy_tolerance"]),
                angles=np.ascontiguousarray(rec["angles"][:dof], dtype=np.float64),
                atol=np.ascontiguousarray(rec["angle_tolerances"][:dof], dtype=np.float64),
                res=np.ascontiguousarray(params.resolutions, dtype=np.float64),
                prims=np.ascontiguousarray(params.mprims, dtype=np.float64),
                flags=np.ascontiguousarray(params.short_flags, dtype=np.uint8),
                w=None if w is None else np.ascontiguousarray(w, dtype=np.float64))


def plan_snap(o, T_kin_to_planning, start, goal, params, snap, max_path=4096):
    """goal_oracle.plan() with the snap action: snap = smpl_b200.api.SnapParams (None or disabled: plans as plan()).
    T_kin_to_planning: the scene's (3, 4) transform, as given to OracleScene.init_kdl.  The result also has
    ik_attempted / ik_converged (the IK solves the search ran)."""
    a = _goal_args(start, goal, params)
    dof = a["dof"]
    T = np.ascontiguousarray(np.asarray(T_kin_to_planning, np.float64).reshape(3, 4))
    en = snap is not None and bool(snap.enabled)
    thresh = float(snap.dist_thresh) if snap is not None else 0.0
    weight = float(snap.weight) if snap is not None else 0.5
    max_it = int(snap.max_iterations) if snap is not None else 100
    tol = float(snap.tolerance) if snap is not None else 1e-6
    summary = np.zeros(8, np.int32)
    path = np.zeros(max_path, np.int32)
    pstates = np.zeros((max_path, dof), np.float64)
    counters = np.zeros(2, np.int64)
    secs = lib().oracle_plan_goal_snap(o.h, _dp(a["start"]), a["type"], _dp(a["pose"]), _dp(a["tol"]), a["rpy_tol"],
                                       _dp(a["angles"]), _dp(a["atol"]), _dp(a["res"]), _dp(a["prims"]),
                                       _bp(a["flags"]), None if a["w"] is None else _dp(a["w"]), len(a["prims"]),
                                       int(params.use_short_dist), float(params.short_dist_thresh),
                                       float(params.epsilon), int(params.max_expansions), _dp(T), int(en), thresh,
                                       weight, max_it, tol, _ip(summary), _ip(path), max_path, _dp(pstates),
                                       counters.ctypes.data_as(C.POINTER(C.c_int64)))
    assert secs >= 0.0, "unknown goal type or scene without kinematics / heuristic"
    n = int(summary[3])
    assert int(summary[5]) == n, "extractPath failed"
    return dict(success=bool(summary[0]), expansions=int(summary[1]), cost=int(summary[2]),
                path_ids=path[:min(n, max_path)].copy(), num_states=int(summary[4]),
                path_states=pstates[:min(n, max_path)].copy(), seconds=float(secs),
                ik_attempted=int(counters[0]), ik_converged=int(counters[1]))


def planning_link_ik(o, T_kin_to_planning, poses, seeds, max_iterations=100, tolerance=1e-6):
    """The oracle's planning-link IK: poses (n, 6) target-offset x y z roll pitch yaw, seeds (n, dof).
    Returns (q (n, dof), ok (n,) bool, iterations (n,))."""
    poses = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 6))
    seeds = np.ascontiguousarray(np.asarray(seeds, np.float64).reshape(len(poses), -1))
    T = np.ascontiguousarray(np.asarray(T_kin_to_planning, np.float64).reshape(3, 4))
    n, dof = seeds.shape
    q = np.zeros((n, dof))
    ok = np.zeros(n, np.uint8)
    it = np.zeros(n, np.int32)
    r = lib().oracle_planning_link_ik(o.h, _dp(T), _dp(poses), _dp(seeds), n, int(max_iterations), float(tolerance),
                                      _dp(q), _bp(ok), _ip(it))
    assert r >= 0, "scene without kinematics"
    return q, ok.astype(bool), it
