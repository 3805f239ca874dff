"""ctypes binding of oracle/euclid_shortcut/liboracle_euclid_shortcut.so: the sequential EUCLID_SPACE shortcut of the
oracle -- its Euclidean-space motions (oracle_euclid_motions) and the greedy ShortcutPath over them
(oracle_shortcut_path_euclid).  Parameters are smpl_b200.api.EuclidParams (None = the defaults)."""
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
        path = os.path.join(ROOT, "oracle", "euclid_shortcut", "liboracle_euclid_shortcut.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        dp, ip, bp, i, d = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_int, C.c_double
        lp = C.POINTER(C.c_int64)
        L.oracle_euclid_motions.argtypes = [C.c_void_p, dp, dp, i, ip, ip, i, d, d, i, i, d, bp, dp, ip, lp, dp, lp]
        L.oracle_shortcut_path_euclid.argtypes = [C.c_void_p, dp, dp, i, d, d, i, i, d, dp, ip, i, lp]
        _LIB = L
    return _LIB


def _prm(params):
    p = params or api.EuclidParams()
    return (float(p.max_step_m), float(p.max_step_rad), int(p.max_steps), int(p.max_iterations), float(p.tolerance))


def _T(T_kin_to_planning):
    return np.ascontiguousarray(np.asarray(T_kin_to_planning, np.float64).reshape(3, 4))


def euclid_motions(o, T_kin_to_planning, points, idx_a, idx_b, params=None, want_states=False):
    """The oracle's answer to smplgpu_euclid_motions: dict(ok, cost, n_steps, ik_solves, ik_converged), with
    want_states also states as GpuContext.euclid_motions returns them (a second pass; NaN where the IK chain did not
    complete).  Raises ValueError for bad parameters or indices."""
    pts = np.ascontiguousarray(points, dtype=np.float64)
    a = np.ascontiguousarray(idx_a, dtype=np.int32)
    b = np.ascontiguousarray(idx_b, dtype=np.int32)
    n, dof = len(a), pts.shape[1]
    p = _prm(params)
    lp = C.POINTER(C.c_int64)

    def run(offs, st):
        ok, cost, steps = np.zeros(n, np.uint8), np.zeros(n), np.zeros(n, np.int32)
        ctr = np.zeros(2, np.int64)
        r = lib().oracle_euclid_motions(o.h, _dp(_T(T_kin_to_planning)), _dp(pts), len(pts), _ip(a), _ip(b), n, *p,
                                        _bp(ok), _dp(cost), _ip(steps),
                                        None if offs is None else offs.ctypes.data_as(lp),
                                        None if st is None else _dp(st), ctr.ctypes.data_as(lp))
        if r != 0:
            raise ValueError("oracle_euclid_motions: bad parameters, indices or scene")
        return dict(ok=ok.astype(bool), cost=cost, n_steps=steps, ik_solves=int(ctr[0]), ik_converged=int(ctr[1]))

    out = run(None, None)
    if want_states:
        steps = out["n_steps"]
        inner = np.where(steps <= p[2], np.maximum(steps - 1, 0), 0).astype(np.int64)
        offs = np.zeros(n + 1, np.int64)
        offs[1:] = np.cumsum(inner)
        st = np.full((max(1, int(offs[-1])), dof), np.nan)
        run(offs, st)
        out["states"] = [st[offs[e]:offs[e + 1]].copy() for e in range(n)]
    return out


def shortcut_path_euclid(o, T_kin_to_planning, path, params=None):
    """ShortcutPath with the EUCLID_SPACE type for one path: (points (m, dof), source (m,) -- input index or -1 --,
    (IK solves, converged))."""
    path = np.ascontiguousarray(path, dtype=np.float64)
    n, dof = path.shape
    p = _prm(params)
    room = max(1, n + (n - 1) * max(p[2] - 1, 0))
    out = np.zeros((room, dof))
    src = np.zeros(room, np.int32)
    ctr = np.zeros(2, np.int64)
    m = lib().oracle_shortcut_path_euclid(o.h, _dp(_T(T_kin_to_planning)), _dp(path), n, *p, _dp(out), _ip(src), room,
                                          ctr.ctypes.data_as(C.POINTER(C.c_int64)))
    if m < 0:
        raise ValueError("oracle_shortcut_path_euclid: bad parameters or scene")
    assert m <= room
    return out[:m].copy(), src[:m].copy(), (int(ctr[0]), int(ctr[1]))
