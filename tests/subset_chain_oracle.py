"""ctypes binding of oracle/subset_chain/liboracle_subset_chain.so: the oracle's planning model (KDLRobotModel) with a
planning chain over a subset of the planning variables (oracle_scene_init_kdl_subset), installed on an
oracle_api.OracleScene; the oracle planners then run on it unchanged."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_api import _dp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(ROOT, "oracle", "subset_chain", "liboracle_subset_chain.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-C", os.path.dirname(path)], check=True)
        L = C.CDLL(path)
        dp = C.POINTER(C.c_double)
        L.oracle_subset_chain_last_error.restype = C.c_char_p
        L.oracle_scene_init_kdl_subset.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, dp, dp]
        _LIB = L
    return _LIB


def init_kdl_subset(o, chain_root, chain_tip, planning_link, T_kin_to_planning=None, xyz_offset=None):
    """OracleScene.init_kdl for a chain that moves only some of the planning variables: every movable chain joint
    must be a planning variable (at any index), planning variables off the chain are allowed.  Raises RuntimeError
    with the oracle's error text when the model is refused."""
    T = np.eye(4)[:3] if T_kin_to_planning is None else np.asarray(T_kin_to_planning, np.float64).reshape(3, 4)
    T = np.ascontiguousarray(T, dtype=np.float64)
    off = np.ascontiguousarray(np.zeros(3) if xyz_offset is None else np.asarray(xyz_offset, np.float64))
    L = lib()
    if L.oracle_scene_init_kdl_subset(o.h, chain_root.encode(), chain_tip.encode(), planning_link.encode(), _dp(T),
                                      _dp(off)) != 0:
        raise RuntimeError("init_kdl_subset: " + L.oracle_subset_chain_last_error().decode())
