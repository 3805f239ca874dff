"""ctypes plumbing over the C ABI (include/smplgpu.h, include/smplhost.h).

The compute path is libsmplgpu.so (hand-written sm_100a kernels).  There is no
CPU fallback: a missing library or a missing GPU raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIBDIR = os.path.join(HERE, "lib")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_uint8_p = C.POINTER(C.c_uint8)
c_uint16_p = C.POINTER(C.c_uint16)

_gpu = None
_host = None


class SmplGpuError(RuntimeError):
    pass


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _ip(a):
    return a.ctypes.data_as(c_int32_p)


def _bp(a):
    return a.ctypes.data_as(c_uint8_p)


class SuccInfoC(C.Structure):
    """smplgpu_succ_info (include/smplgpu.h)."""
    _fields_ = [("state", C.c_double * 16), ("pose", C.c_double * 6), ("link_xyz", C.c_double * 3), ("h", C.c_int32),
                ("goal_dist_cells", C.c_int32), ("waypoints", C.c_int32), ("edge_valid", C.c_uint8),
                ("limits_ok", C.c_uint8), ("state_valid", C.c_uint8), ("is_parent", C.c_uint8)]


MAX_DOF = 16   # SMPLGPU_MAX_DOF
GOAL_XYZ, GOAL_XYZ_RPY, GOAL_JOINT_STATE = 0, 1, 2   # SMPLGPU_GOAL_*


class GoalC(C.Structure):
    """smplgpu_goal (include/smplgpu.h): GoalConstraint of one query."""
    _fields_ = [("type", C.c_int32), ("pose", C.c_double * 6), ("xyz_tolerance", C.c_double * 3),
                ("rpy_tolerance", C.c_double), ("angles", C.c_double * MAX_DOF),
                ("angle_tolerances", C.c_double * MAX_DOF)]


GOAL_DTYPE = np.dtype(GoalC)   # goal records as a numpy structured array: concatenate / index them like any array


def pose_goals(poses, xyz_tolerance=(0.015, 0.015, 0.015), rpy_tolerance=None):
    """Goal records for target-offset poses.  poses: (n, 3) positions or (n, 6) x y z roll pitch yaw.
    rpy_tolerance None: XYZ goals (orientation ignored); a number: XYZ_RPY goals, the state is a goal when its
    orientation is within that angle of the goal's (ManipLattice::isGoal)."""
    poses = np.asarray(poses, np.float64)
    poses = poses.reshape(-1, poses.shape[-1])
    if rpy_tolerance is not None and poses.shape[1] != 6:
        raise ValueError("pose goals with an orientation tolerance need x y z roll pitch yaw")
    out = np.zeros(len(poses), GOAL_DTYPE)
    out["type"] = GOAL_XYZ if rpy_tolerance is None else GOAL_XYZ_RPY
    out["pose"][:, :poses.shape[1]] = poses
    out["xyz_tolerance"] = np.broadcast_to(np.asarray(xyz_tolerance, np.float64), (len(poses), 3))
    out["rpy_tolerance"] = 0.0 if rpy_tolerance is None else float(rpy_tolerance)
    return out


MAX_GOAL_SET = 64   # SMPLGPU_MAX_GOAL_SET: records in one query's goal set


def goal_sets(sets):
    """A goal set per query, for plan_batch(goals=...): sets is a list of GOAL_DTYPE record arrays (1 to MAX_GOAL_SET
    records each, types may be mixed).  A query succeeds at a state that satisfies any record of its set.
    Returns (records, offsets): the records concatenated, and offsets (nq + 1,) int32 with query i's records at
    records[offsets[i]:offsets[i + 1]]."""
    sets = [np.asarray(g).reshape(-1) for g in sets]
    for i, g in enumerate(sets):
        if g.dtype != GOAL_DTYPE:
            raise ValueError("goal set %d: records must be GOAL_DTYPE" % i)
        if not 1 <= len(g) <= MAX_GOAL_SET:
            raise ValueError("goal set %d has %d records (1 to %d)" % (i, len(g), MAX_GOAL_SET))
    offsets = np.zeros(len(sets) + 1, np.int32)
    offsets[1:] = np.cumsum([len(g) for g in sets])
    records = np.concatenate(sets) if sets else np.zeros(0, GOAL_DTYPE)
    return np.ascontiguousarray(records), offsets


def joint_goals(angles, angle_tolerances):
    """Goal records for joint configurations: angles (n, dof); angle_tolerances (dof,) or (n, dof).  The state is a
    goal when every planning variable is within its tolerance (no angle wrapping)."""
    angles = np.asarray(angles, np.float64)
    angles = angles.reshape(-1, angles.shape[-1])
    n, dof = angles.shape
    if dof > MAX_DOF:
        raise ValueError("more than %d planning variables" % MAX_DOF)
    out = np.zeros(n, GOAL_DTYPE)
    out["type"] = GOAL_JOINT_STATE
    out["angles"][:, :dof] = angles
    out["angle_tolerances"][:, :dof] = np.broadcast_to(np.asarray(angle_tolerances, np.float64), (n, dof))
    return out


class PlanParamsC(C.Structure):
    """smplhost_plan_params (include/smplhost.h)."""
    _fields_ = [("dof", C.c_int), ("resolutions", c_double_p), ("mprims", c_double_p), ("short_flags", c_uint8_p),
                ("n_prims", C.c_int), ("use_short_dist", C.c_int), ("short_dist_thresh", C.c_double),
                ("epsilon", C.c_double), ("max_expansions", C.c_int), ("xyz_tolerance", C.c_double * 3),
                ("cost_per_cell", C.c_int), ("inflation_radius", C.c_double), ("var_min", c_double_p),
                ("var_max", c_double_p), ("var_continuous", c_uint8_p), ("origin", C.c_double * 3),
                ("res", C.c_double), ("dims", C.c_int * 3), ("n_threads", C.c_int), ("prim_weights", c_double_p)]


class IkParamsC(C.Structure):
    """smplgpu_ik_params (include/smplgpu.h)."""
    _fields_ = [("max_iterations", C.c_int32), ("tolerance", C.c_double)]


class SnapParamsC(C.Structure):
    """smplhost_snap_params (include/smplhost.h)."""
    _fields_ = [("enabled", C.c_int32), ("dist_thresh", C.c_double), ("weight", C.c_double), ("ik", IkParamsC)]


SNAP_RPY, SNAP_XYZ, SNAP_XYZ_RPY = 0, 1, 2   # SMPLGPU_SNAP_*: the snap kinds, in successor-word order
SNAP_KIND_NAMES = ("rpy", "xyz", "xyz_rpy")


class SnapKindsC(C.Structure):
    """smplgpu_snap_kinds (include/smplgpu.h)."""
    _fields_ = [("enabled", C.c_int32 * 3), ("dist_thresh", C.c_double * 3), ("ik", IkParamsC)]


class SnapsParamsC(C.Structure):
    """smplhost_snaps_params (include/smplhost.h)."""
    _fields_ = [("kinds", SnapKindsC), ("weight", C.c_double)]


class SnapParams:
    """The snap-to-goal actions of the batched planner.  enabled / dist_thresh: SNAP_TO_XYZ_RPY -- an expansion whose
    metric goal distance is within dist_thresh metres first tries to jump straight to the goal: to an IK solution for a
    pose goal's full pose, to the angles of a joint goal.  xyz_dist_thresh: SNAP_TO_XYZ (None = off), a position-only
    IK solution for a pose goal's position, the orientation free.  rpy_dist_thresh: SNAP_TO_RPY (None = off), for an
    XYZ_RPY goal an IK solution that keeps the expanded state's position and turns it to the goal's orientation.  Every
    snap costs int(1000 * weight).  dist_thresh = 0.0 is the reference demo's setting."""

    def __init__(self, enabled=True, dist_thresh=0.0, weight=0.5, max_iterations=100, tolerance=1e-6,
                 xyz_dist_thresh=None, rpy_dist_thresh=None):
        self.enabled = enabled
        self.dist_thresh = dist_thresh
        self.weight = weight
        self.max_iterations = max_iterations
        self.tolerance = tolerance
        self.xyz_dist_thresh = xyz_dist_thresh
        self.rpy_dist_thresh = rpy_dist_thresh

    def c(self):
        return SnapParamsC(int(bool(self.enabled)), float(self.dist_thresh), float(self.weight),
                           IkParamsC(int(self.max_iterations), float(self.tolerance)))

    def new_kinds(self):
        """whether SNAP_TO_XYZ or SNAP_TO_RPY is on"""
        return self.xyz_dist_thresh is not None or self.rpy_dist_thresh is not None

    def kinds(self):
        """(enabled (3,), dist_thresh (3,)) by SNAP_* kind"""
        en = [self.rpy_dist_thresh is not None, self.xyz_dist_thresh is not None, bool(self.enabled)]
        th = [0.0 if self.rpy_dist_thresh is None else float(self.rpy_dist_thresh),
              0.0 if self.xyz_dist_thresh is None else float(self.xyz_dist_thresh), float(self.dist_thresh)]
        return en, th

    def c_kinds(self):
        en, th = self.kinds()
        k = SnapKindsC()
        for i in range(3):
            k.enabled[i] = int(en[i])
            k.dist_thresh[i] = th[i]
        k.ik = IkParamsC(int(self.max_iterations), float(self.tolerance))
        return SnapsParamsC(k, float(self.weight))


def gpu_lib():
    """libsmplgpu.so; raises when it has not been built (no fallback)."""
    global _gpu
    if _gpu is None:
        path = os.path.join(LIBDIR, "libsmplgpu.so")
        if not os.path.exists(path):
            raise SmplGpuError("CUDA extension %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`" % path)
        L = C.CDLL(path, mode=C.RTLD_GLOBAL)
        L.smplgpu_create.restype = C.c_void_p
        L.smplgpu_create.argtypes = [C.c_int]
        L.smplgpu_last_error.restype = C.c_char_p
        L.smplgpu_last_error.argtypes = [C.c_void_p]
        L.smplgpu_launch_count.restype = C.c_int64
        L.smplgpu_launch_count.argtypes = [C.c_void_p]
        L.smplgpu_destroy.argtypes = [C.c_void_p]
        L.smplgpu_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.smplgpu_bind_thread.argtypes = [C.c_void_p]
        L.smplgpu_synchronize.argtypes = [C.c_void_p]
        vp, dp, ip, bp, i, d = C.c_void_p, c_double_p, c_int32_p, c_uint8_p, C.c_int, C.c_double
        L.smplgpu_set_distance_field.argtypes = [vp, c_uint16_p, i, i, i, dp, d, i, d]
        L.smplgpu_set_distance_field_dev.argtypes = [vp, vp, i, i, i, dp, d, i, d]
        L.smplgpu_build_distance_field.argtypes = [vp, ip, i, i, i, i, dp, d, d, d]
        L.smplgpu_download_distance_field.argtypes = [vp, c_uint16_p]
        L.smplgpu_distance_field_add_cells.argtypes = [vp, c_int32_p, C.c_int]
        L.smplgpu_distance_field_remove_cells.argtypes = [vp, c_int32_p, C.c_int]
        L.smplgpu_distance_field_dev_ptr.argtypes = [vp, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
        L.smplgpu_is_states_valid.argtypes = [vp, dp, i, bp]
        L.smplgpu_is_states_valid_dev.argtypes = [vp, vp, i, vp]
        L.smplgpu_is_edges_valid.argtypes = [vp, dp, dp, i, bp, ip]
        L.smplgpu_is_edges_valid_dev.argtypes = [vp, vp, vp, i, vp, vp]
        L.smplgpu_fk_sphere_centers.argtypes = [vp, dp, i, dp]
        L.smplgpu_check_joint_limits.argtypes = [vp, dp, i, bp]
        L.smplgpu_collision_distance.argtypes = [vp, dp, i, dp]
        L.smplgpu_last_validity_stats.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.smplgpu_bfs_set_walls_from_df.argtypes = [vp, d]
        L.smplgpu_bfs_set_walls.argtypes = [vp, i, i, i, bp]
        L.smplgpu_bfs_set_walls_dev.argtypes = [vp, i, i, i, vp]
        L.smplgpu_bfs_run.argtypes = [vp, ip, i]
        L.smplgpu_bfs_distances.argtypes = [vp, ip, i, ip]
        L.smplgpu_bfs_download.argtypes = [vp, ip]
        L.smplgpu_bfs_dims.argtypes = [vp, ip]
        L.smplgpu_bfs_last_levels.argtypes = [vp]
        L.smplgpu_goal_heuristics.argtypes = [vp, dp, i, i, ip]
        L.smplgpu_goal_heuristics_dev.argtypes = [vp, vp, i, i, vp]
        L.smplgpu_planning_frame_fk.argtypes = [vp, dp, i, dp]
        L.smplgpu_planning_link_ik.argtypes = [vp, dp, dp, i, C.POINTER(IkParamsC), dp, bp, ip]
        L.smplgpu_planning_link_ik_position.argtypes = [vp, dp, dp, i, C.POINTER(IkParamsC), dp, bp, ip]
        L.smplgpu_is_mprim_edges_valid.argtypes = [vp, dp, ip, i, dp, i, bp, ip]
        L.smplgpu_is_indexed_edges_valid.argtypes = [vp, dp, i, ip, ip, i, bp, ip]
        L.smplgpu_set_precision_mode.argtypes = [vp, i]
        L.smplgpu_bfs_set_mode.argtypes = [vp, i]
        L.smplgpu_certified_bounds.argtypes = [vp, dp, dp]
        L.smplgpu_last_f64_resolved.argtypes = [vp, C.POINTER(C.c_int64)]
        L.smplgpu_probe_df_lookup_rate.argtypes = [vp, C.POINTER(C.c_double)]
        L.smplgpu_fk_sphere_centers_f32.argtypes = [vp, dp, i, C.POINTER(C.c_float)]
        L.smplgpu_bfs_bank_create.argtypes = [vp, i, d]
        L.smplgpu_bfs_bank_max_slots.argtypes = [vp]
        L.smplgpu_voxelize_mesh.argtypes = [vp, dp, i, ip, i, d, dp, dp, i]
        L.smplgpu_build_distance_field_from_meshes.argtypes = [vp, dp, i, ip, i, ip, i, i, i, i, dp, d, d, d]
        L.smplgpu_bfs_bank_run.argtypes = [vp, ip]
        L.smplgpu_bfs_bank_run_slots.argtypes = [vp, ip, ip, i]
        L.smplgpu_bfs_bank_run_slots_async.argtypes = [vp, ip, ip, i]
        L.smplgpu_bfs_bank_run_slots_multi.argtypes = [vp, ip, ip, ip, i]
        L.smplgpu_bfs_bank_run_slots_multi_async.argtypes = [vp, ip, ip, ip, i]
        L.smplgpu_bfs_bank_run_done.argtypes = [vp]
        L.smplgpu_bfs_bank_run_wait.argtypes = [vp]
        L.smplgpu_bfs_bank_distances.argtypes = [vp, ip, ip, i, ip]
        L.smplgpu_expand_batch.argtypes = [vp, dp, dp, ip, i, i, bp, ip, ip, dp]
        L.smplgpu_set_motion_primitives.argtypes = [vp, dp, i]
        L.smplgpu_set_lattice.argtypes = [vp, dp, ip]
        L.smplgpu_reserve_distance_field.argtypes = [vp, i, i, i, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
        L.smplgpu_set_distance_field_l2_persistence.argtypes = [vp, i, dp]
        L.smplgpu_is_lattice_states_valid.argtypes = [vp, C.POINTER(C.c_int16), i, bp]
        L.smplgpu_is_lattice_edges_valid.argtypes = [vp, C.POINTER(C.c_int16), bp, i, dp, i, bp, ip]
        L.smplgpu_expand_state.argtypes = [vp, dp, i, C.POINTER(C.POINTER(SuccInfoC))]
        L.smplgpu_scene_epoch.restype = C.c_int64
        L.smplgpu_scene_epoch.argtypes = [vp]
        _gpu = L
    return _gpu


def host_lib():
    global _host
    if _host is None:
        gpu_lib()
        path = os.path.join(LIBDIR, "libsmplhost.so")
        if not os.path.exists(path):
            raise SmplGpuError("host library %s is missing: run __graft_entry__.build()" % path)
        H = C.CDLL(path)
        H.smplhost_last_error.restype = C.c_char_p
        H.smplhost_tables_load.restype = C.c_void_p
        H.smplhost_tables_load.argtypes = [C.c_char_p]
        vp = C.c_void_p
        H.smplhost_tables_destroy.argtypes = [vp]
        H.smplhost_tables_configure.argtypes = [vp, C.c_char_p, C.c_char_p]
        H.smplhost_tables_set_joint.argtypes = [vp, C.c_char_p, C.c_double]
        H.smplhost_tables_use_file_acm.argtypes = [vp]
        H.smplhost_tables_set_acm_entry.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int]
        H.smplhost_tables_attach_spheres.argtypes = [vp, C.c_char_p, C.c_char_p, c_double_p, C.c_int, C.c_double]
        H.smplhost_tables_detach.argtypes = [vp, C.c_char_p]
        H.smplhost_tables_set_planning_chain.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p, c_double_p, c_double_p]
        H.smplhost_tables_dof.argtypes = [vp]
        H.smplhost_tables_limits.argtypes = [vp, c_double_p, c_double_p, c_uint8_p]
        H.smplhost_tables_apply.argtypes = [vp, vp]
        H.smplhost_tables_outside_voxels.argtypes = [vp, C.POINTER(c_double_p)]
        H.smplhost_tables_node_table.argtypes = [vp, c_double_p, C.c_int]
        H.smplhost_tables_motion_weights.argtypes = [vp, c_double_p, c_int32_p]
        H.smplhost_tables_pairs.argtypes = [vp, c_int32_p, C.c_int]
        H.smplhost_plan_batch.argtypes = [vp, C.POINTER(PlanParamsC), c_double_p, c_double_p, C.c_int, C.c_int,
                                          c_int32_p, c_int32_p, C.c_int, c_double_p, c_double_p]
        H.smplhost_plan_batch_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(PlanParamsC), c_double_p, c_double_p,
                                                C.c_int, C.c_int, c_int32_p, c_int32_p, C.c_int, c_double_p, c_double_p]
        H.smplhost_plan_batch_goals.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(PlanParamsC), c_double_p,
                                                C.POINTER(GoalC), C.c_int, C.c_int, c_int32_p, c_int32_p, C.c_int,
                                                c_double_p, c_double_p]
        H.smplhost_plan_batch_snap.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(PlanParamsC), c_double_p,
                                               C.POINTER(GoalC), C.c_int, C.c_int, c_int32_p, c_int32_p, C.c_int,
                                               c_double_p, c_double_p, C.POINTER(SnapParamsC), C.POINTER(C.c_int64)]
        H.smplhost_plan_batch_goal_sets.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(PlanParamsC), c_double_p,
                                                    C.POINTER(GoalC), c_int32_p, C.c_int, C.c_int, c_int32_p, c_int32_p,
                                                    C.c_int, c_double_p, c_double_p, C.POINTER(SnapParamsC),
                                                    C.POINTER(C.c_int64), c_int32_p]
        H.smplhost_plan_batch_snaps.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(PlanParamsC), c_double_p,
                                                C.POINTER(GoalC), c_int32_p, C.c_int, C.c_int, c_int32_p, c_int32_p,
                                                C.c_int, c_double_p, c_double_p, C.POINTER(SnapsParamsC),
                                                C.POINTER(C.c_int64), c_int32_p]
        H.smplhost_shortcut_paths.argtypes = [vp, C.c_int, c_uint8_p, c_double_p, c_int32_p, C.c_int, C.c_int, c_int32_p,
                                              c_int32_p, c_double_p]
        H.smplhost_interpolate_paths.argtypes = [vp, vp, c_double_p, c_int32_p, C.c_int, c_double_p, C.c_int, c_int32_p,
                                                 c_double_p]
        H.smplhost_tables_attach_box.argtypes = [vp, vp, C.c_char_p, C.c_char_p, c_double_p, c_double_p]
        H.smplhost_box_meshes.argtypes = [c_double_p, C.c_int, c_double_p, c_int32_p]
        H.smplhost_shape_mesh_size.argtypes = [C.c_int, c_int32_p, c_int32_p]
        H.smplhost_shape_meshes.argtypes = [c_double_p, C.c_int, c_double_p, c_int32_p]
        H.smplhost_adapters_create.restype = C.c_void_p
        H.smplhost_adapters_create.argtypes = [vp, vp, C.c_char_p, c_double_p, C.c_double, c_int32_p, C.c_double, C.c_int]
        H.smplhost_adapters_destroy.argtypes = [vp]
        H.smplhost_cc_is_state_valid.argtypes = [vp, c_double_p]
        H.smplhost_cc_is_state_to_state_valid.argtypes = [vp, c_double_p, c_double_p]
        H.smplhost_cc_interpolate_path.argtypes = [vp, c_double_p, c_double_p, c_double_p, C.c_int]
        H.smplhost_cc_is_states_valid.argtypes = [vp, c_double_p, C.c_int, c_uint8_p]
        H.smplhost_cc_is_edges_valid.argtypes = [vp, c_double_p, c_double_p, C.c_int, c_uint8_p]
        H.smplhost_rm_check_joint_limits.argtypes = [vp, c_double_p]
        H.smplhost_rm_compute_planning_link_fk.argtypes = [vp, c_double_p, c_double_p]
        H.smplhost_heur_update_goal.argtypes = [vp, c_double_p]
        H.smplhost_heur_goal_heuristic.argtypes = [vp, c_double_p]
        H.smplhost_heur_metric_goal_distance.restype = C.c_double
        H.smplhost_heur_metric_goal_distance.argtypes = [vp, C.c_double, C.c_double, C.c_double]
        _host = H
    return _host


class RobotTables:
    """Host-side model builder (smpl_b200/host/robot_tables.cpp)."""

    def __init__(self, robot_path):
        self.H = host_lib()
        h = self.H.smplhost_tables_load(robot_path.encode())
        if not h:
            raise SmplGpuError("smplhost_tables_load: " + self.H.smplhost_last_error().decode())
        self.h = C.c_void_p(h)

    def close(self):
        if getattr(self, "h", None):
            self.H.smplhost_tables_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, r, what):
        if r != 0:
            raise SmplGpuError("%s: %s" % (what, self.H.smplhost_last_error().decode()))

    def configure(self, group, planning_joints):
        self._ck(self.H.smplhost_tables_configure(self.h, group.encode(), ",".join(planning_joints).encode()), "configure")

    def set_joint(self, name, value):
        self._ck(self.H.smplhost_tables_set_joint(self.h, name.encode(), float(value)), "set_joint")

    def use_file_acm(self):
        self.H.smplhost_tables_use_file_acm(self.h)

    def set_acm_entry(self, a, b, allowed):
        self.H.smplhost_tables_set_acm_entry(self.h, a.encode(), b.encode(), int(allowed))

    def attach_spheres(self, body_id, link, centers, radius):
        c = np.ascontiguousarray(centers, dtype=np.float64).reshape(-1, 3)
        self._ck(self.H.smplhost_tables_attach_spheres(self.h, body_id.encode(), link.encode(), _dp(c), len(c),
                                                       float(radius)), "attach_spheres")

    def attach_box(self, ctx, body_id, link, size, pose3x4):
        """attachBody for a box: sphere model generated from the shape's surface voxels (on the device)."""
        sz = np.ascontiguousarray(size, dtype=np.float64)
        p = np.ascontiguousarray(pose3x4, dtype=np.float64).reshape(3, 4)
        n = self.H.smplhost_tables_attach_box(self.h, ctx.h, body_id.encode(), link.encode(), _dp(sz), _dp(p))
        if n < 0:
            raise SmplGpuError("attach_box: " + self.H.smplhost_last_error().decode())
        return n

    def detach(self, body_id):
        return self.H.smplhost_tables_detach(self.h, body_id.encode()) == 0

    def set_planning_chain(self, root, tip, planning_link, T_kin_to_planning=None, xyz_offset=None):
        T = np.eye(4)[:3] if T_kin_to_planning is None else np.asarray(T_kin_to_planning, np.float64).reshape(3, 4)
        T = np.ascontiguousarray(T, dtype=np.float64)
        off = np.ascontiguousarray(np.zeros(3) if xyz_offset is None else np.asarray(xyz_offset, np.float64))
        self._ck(self.H.smplhost_tables_set_planning_chain(self.h, root.encode(), tip.encode(), planning_link.encode(),
                                                           _dp(T), _dp(off)), "set_planning_chain")

    @property
    def dof(self):
        return self.H.smplhost_tables_dof(self.h)

    def limits(self):
        n = self.dof
        lo, hi, c = np.zeros(n), np.zeros(n), np.zeros(n, np.uint8)
        self.H.smplhost_tables_limits(self.h, _dp(lo), _dp(hi), _bp(c))
        return lo, hi, c

    def apply(self, ctx):
        self._ck(self.H.smplhost_tables_apply(self.h, ctx.h), "apply")

    def outside_voxels(self):
        p = c_double_p()
        n = self.H.smplhost_tables_outside_voxels(self.h, C.byref(p))
        if n <= 0:
            return np.zeros((0, 3))
        return np.ctypeslib.as_array(p, shape=(n, 3)).copy()

    def node_table(self):
        out = np.zeros((4096, 8))
        n = self.H.smplhost_tables_node_table(self.h, _dp(out), 4096)
        return out[:n].copy()

    def motion_weights(self):
        n = self.dof
        w, t = np.zeros(n), np.zeros(n, np.int32)
        self.H.smplhost_tables_motion_weights(self.h, _dp(w), _ip(t))
        return w, t

    def pairs(self):
        out = np.zeros((4096, 2), np.int32)
        n = self.H.smplhost_tables_pairs(self.h, _ip(out), 4096)
        return out[:n].copy()


class GpuContext:
    """One smplgpu context (one GPU, one stream)."""

    def __init__(self, device=0):
        self.L = gpu_lib()
        h = self.L.smplgpu_create(int(device))
        if not h:
            raise SmplGpuError("smplgpu_create: " + self.L.smplgpu_last_error(None).decode())
        self.h = C.c_void_p(h)
        self.dof = None
        self.n_nodes = None

    def close(self):
        if getattr(self, "h", None):
            self.L.smplgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, r, what):
        if r < 0:
            raise SmplGpuError("%s: %s" % (what, self.L.smplgpu_last_error(self.h).decode()))
        return r

    def set_stream(self, cuda_stream):
        self._ck(self.L.smplgpu_set_stream(self.h, C.c_void_p(cuda_stream)), "set_stream")

    def synchronize(self):
        self._ck(self.L.smplgpu_synchronize(self.h), "synchronize")

    def launch_count(self):
        return int(self.L.smplgpu_launch_count(self.h))

    # ---- scene ----
    def set_robot(self, tables):
        tables.apply(self)
        self.dof = tables.dof
        self.n_nodes = len(tables.node_table())

    def set_distance_field(self, d2, origin, res, dmax_sq, padding=0.0):
        d2 = np.ascontiguousarray(d2, dtype=np.uint16)
        nx, ny, nz = d2.shape
        o = np.ascontiguousarray(origin, dtype=np.float64)
        self._ck(self.L.smplgpu_set_distance_field(self.h, d2.ctypes.data_as(c_uint16_p), nx, ny, nz, _dp(o),
                                                   float(res), int(dmax_sq), float(padding)), "set_distance_field")
        self.df_dims = (nx, ny, nz)

    def set_distance_field_dev(self, ptr, dims, origin, res, dmax_sq, padding=0.0):
        o = np.ascontiguousarray(origin, dtype=np.float64)
        self._ck(self.L.smplgpu_set_distance_field_dev(self.h, C.c_void_p(ptr), int(dims[0]), int(dims[1]), int(dims[2]),
                                                       _dp(o), float(res), int(dmax_sq), float(padding)),
                 "set_distance_field_dev")
        self.df_dims = tuple(int(d) for d in dims)

    def build_distance_field(self, cells, dims, origin, res, max_dist, padding=0.0):
        cells = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        o = np.ascontiguousarray(origin, dtype=np.float64)
        self._ck(self.L.smplgpu_build_distance_field(self.h, _ip(cells), len(cells), int(dims[0]), int(dims[1]),
                                                     int(dims[2]), _dp(o), float(res), float(max_dist), float(padding)),
                 "build_distance_field")
        self.df_dims = tuple(int(d) for d in dims)

    def build_distance_field_from_meshes(self, vertices, triangles, cells, dims, origin, res, max_dist, padding=0.0):
        """WorldCollisionModel::insertObject for a whole scene + the field: meshes voxelised on the device."""
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.int32).reshape(-1, 3)
        cells = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        o = np.ascontiguousarray(origin, dtype=np.float64)
        self._ck(self.L.smplgpu_build_distance_field_from_meshes(
            self.h, _dp(v), len(v), _ip(t), len(t), _ip(cells), len(cells), int(dims[0]), int(dims[1]), int(dims[2]),
            _dp(o), float(res), float(max_dist), float(padding)), "build_distance_field_from_meshes")
        self.df_dims = tuple(int(d) for d in dims)

    def voxelize_mesh(self, vertices, triangles, res, voxel_origin=None):
        """geometry::VoxelizeMesh (fill = false) on the device: voxel centres [n][3] in ExtractVoxels order."""
        v = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 3)
        t = np.ascontiguousarray(triangles, dtype=np.int32).reshape(-1, 3)
        o = None if voxel_origin is None else np.ascontiguousarray(voxel_origin, dtype=np.float64)
        cap = 1 << 16
        while True:
            out = np.zeros((cap, 3), np.float64)
            n = self._ck(self.L.smplgpu_voxelize_mesh(self.h, _dp(v), len(v), _ip(t), len(t), float(res),
                                                      None if o is None else _dp(o), _dp(out), cap), "voxelize_mesh")
            if n <= cap:
                return out[:n].copy()
            cap = n

    def distance_field_add_cells(self, cells):
        """OccupancyGrid::addPointsToField on the resident field (grid coordinates)."""
        cells = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        self._ck(self.L.smplgpu_distance_field_add_cells(self.h, _ip(cells), len(cells)), "distance_field_add_cells")

    def distance_field_remove_cells(self, cells):
        """OccupancyGrid::removePointsFromField on the resident field (grid coordinates)."""
        cells = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        self._ck(self.L.smplgpu_distance_field_remove_cells(self.h, _ip(cells), len(cells)), "distance_field_remove_cells")

    def download_distance_field(self):
        out = np.zeros(self.df_dims, np.uint16)
        self._ck(self.L.smplgpu_download_distance_field(self.h, out.ctypes.data_as(c_uint16_p)), "download_distance_field")
        return out

    def distance_field_dev_ptr(self):
        p = C.c_void_p()
        n = C.c_int64()
        self._ck(self.L.smplgpu_distance_field_dev_ptr(self.h, C.byref(p), C.byref(n)), "distance_field_dev_ptr")
        return p.value, n.value

    # ---- validity ----
    def reserve_distance_field(self, dims):
        """Device room for a field of `dims` (contents to be received from a peer); -> (pointer, bytes)."""
        ptr, nb = C.c_void_p(), C.c_int64()
        self._ck(self.L.smplgpu_reserve_distance_field(self.h, int(dims[0]), int(dims[1]), int(dims[2]), C.byref(ptr),
                                                       C.byref(nb)), "reserve_distance_field")
        return ptr.value, nb.value

    def set_distance_field_l2_persistence(self, on):
        mb = C.c_double()
        self._ck(self.L.smplgpu_set_distance_field_l2_persistence(self.h, int(bool(on)), C.byref(mb)), "l2_persistence")
        return mb.value

    def _q(self, q):
        return np.ascontiguousarray(q, dtype=np.float64).reshape(-1, self.dof)

    def is_states_valid(self, q):
        q = self._q(q)
        v = np.zeros(len(q), np.uint8)
        self._ck(self.L.smplgpu_is_states_valid(self.h, _dp(q), len(q), _bp(v)), "is_states_valid")
        return v

    def is_states_valid_dev(self, q_ptr, n, verdict_ptr):
        self._ck(self.L.smplgpu_is_states_valid_dev(self.h, C.c_void_p(q_ptr), int(n), C.c_void_p(verdict_ptr)),
                 "is_states_valid_dev")

    def is_edges_valid(self, q0, q1, want_counts=True):
        q0, q1 = self._q(q0), self._q(q1)
        v = np.zeros(len(q0), np.uint8)
        c = np.zeros(len(q0), np.int32) if want_counts else None
        self._ck(self.L.smplgpu_is_edges_valid(self.h, _dp(q0), _dp(q1), len(q0), _bp(v),
                                               _ip(c) if want_counts else None), "is_edges_valid")
        return (v, c) if want_counts else v

    def is_mprim_edges_valid(self, q0, prim_id, deltas, want_counts=True):
        """Edges q0[i] -> q0[i] + deltas[prim_id[i]] (the form GetSuccs produces them in)."""
        q0 = self._q(q0)
        pid = np.ascontiguousarray(prim_id, dtype=np.int32)
        d = np.ascontiguousarray(deltas, dtype=np.float64).reshape(-1, self.dof)
        v = np.zeros(len(q0), np.uint8)
        c = np.zeros(len(q0), np.int32) if want_counts else None
        self._ck(self.L.smplgpu_is_mprim_edges_valid(self.h, _dp(q0), _ip(pid), len(q0), _dp(d), len(d), _bp(v),
                                                     _ip(c) if want_counts else None), "is_mprim_edges_valid")
        return (v, c) if want_counts else v

    def is_indexed_edges_valid(self, points, idx_a, idx_b, want_counts=True):
        """Edges points[idx_a[e]] -> points[idx_b[e]] between rows of one point table."""
        pts = self._q(points)
        a = np.ascontiguousarray(idx_a, dtype=np.int32)
        b = np.ascontiguousarray(idx_b, dtype=np.int32)
        v = np.zeros(len(a), np.uint8)
        c = np.zeros(len(a), np.int32) if want_counts else None
        self._ck(self.L.smplgpu_is_indexed_edges_valid(self.h, _dp(pts), len(pts), _ip(a), _ip(b), len(a), _bp(v),
                                                       _ip(c) if want_counts else None), "is_indexed_edges_valid")
        return (v, c) if want_counts else v

    def is_edges_valid_dev(self, q0_ptr, q1_ptr, n, verdict_ptr, counts_ptr=None):
        self._ck(self.L.smplgpu_is_edges_valid_dev(self.h, C.c_void_p(q0_ptr), C.c_void_p(q1_ptr), int(n),
                                                   C.c_void_p(verdict_ptr), C.c_void_p(counts_ptr) if counts_ptr else None),
                 "is_edges_valid_dev")

    def fk_sphere_centers(self, q):
        q = self._q(q)
        out = np.zeros((len(q), self.n_nodes, 3))
        self._ck(self.L.smplgpu_fk_sphere_centers(self.h, _dp(q), len(q), _dp(out)), "fk_sphere_centers")
        return out

    def collision_distance(self, q):
        """CollisionSpace::collisionDistance per state (metres)."""
        q = self._q(q)
        out = np.zeros(len(q), np.float64)
        self._ck(self.L.smplgpu_collision_distance(self.h, _dp(q), len(q), _dp(out)), "collision_distance")
        return out

    def check_joint_limits(self, q):
        q = self._q(q)
        ok = np.zeros(len(q), np.uint8)
        self._ck(self.L.smplgpu_check_joint_limits(self.h, _dp(q), len(q), _bp(ok)), "check_joint_limits")
        return ok

    CERTIFIED_F32, EXACT_F64 = 0, 1

    def set_precision_mode(self, mode):
        self._ck(self.L.smplgpu_set_precision_mode(self.h, int(mode)), "set_precision_mode")

    def certified_bounds(self):
        """(in_use, e_pos metres, eps cells) of the certified single-precision model."""
        a, b = C.c_double(), C.c_double()
        r = self._ck(self.L.smplgpu_certified_bounds(self.h, C.byref(a), C.byref(b)), "certified_bounds")
        return bool(r), a.value, b.value

    def probe_df_lookup_rate(self):
        """independent random distance-field lookups per second (roofline of the validity kernels' lookups)"""
        r = C.c_double()
        self._ck(self.L.smplgpu_probe_df_lookup_rate(self.h, C.byref(r)), "probe_df_lookup_rate")
        return r.value

    def last_f64_resolved(self):
        n = C.c_int64()
        self._ck(self.L.smplgpu_last_f64_resolved(self.h, C.byref(n)), "last_f64_resolved")
        return n.value

    def fk_sphere_centers_f32(self, q):
        q = self._q(q)
        out = np.zeros((len(q), self.n_nodes, 3), np.float32)
        self._ck(self.L.smplgpu_fk_sphere_centers_f32(self.h, _dp(q), len(q), out.ctypes.data_as(C.POINTER(C.c_float))),
                 "fk_sphere_centers_f32")
        return out

    def last_validity_stats(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.L.smplgpu_last_validity_stats(self.h, C.byref(a), C.byref(b), C.byref(c)), "last_validity_stats")
        return dict(df_lookups=a.value, pair_tests=b.value, waypoints=c.value)

    # ---- BFS / heuristic ----
    BFS_TILES, BFS_LEVELS, BFS_AUTO = 0, 1, 2

    def bfs_set_mode(self, mode):
        self._ck(self.L.smplgpu_bfs_set_mode(self.h, int(mode)), "bfs_set_mode")

    def bfs_set_walls_from_df(self, inflation_radius):
        return self._ck(self.L.smplgpu_bfs_set_walls_from_df(self.h, float(inflation_radius)), "bfs_set_walls_from_df")

    def bfs_set_walls(self, walls_zyx):
        w = np.ascontiguousarray(walls_zyx, dtype=np.uint8)
        nz, ny, nx = w.shape
        self._ck(self.L.smplgpu_bfs_set_walls(self.h, nx, ny, nz, _bp(w)), "bfs_set_walls")

    def bfs_set_walls_dev(self, ptr, nx, ny, nz):
        self._ck(self.L.smplgpu_bfs_set_walls_dev(self.h, int(nx), int(ny), int(nz), C.c_void_p(ptr)), "bfs_set_walls_dev")

    def bfs_run(self, seeds):
        s = np.ascontiguousarray(seeds, dtype=np.int32).reshape(-1, 3)
        return self._ck(self.L.smplgpu_bfs_run(self.h, _ip(s), len(s)), "bfs_run")

    def bfs_dims(self):
        d = np.zeros(3, np.int32)
        self._ck(self.L.smplgpu_bfs_dims(self.h, _ip(d)), "bfs_dims")
        return tuple(int(v) for v in d)

    def bfs_download(self):
        nx, ny, nz = self.bfs_dims()
        out = np.zeros((nz + 2, ny + 2, nx + 2), np.int32)
        self._ck(self.L.smplgpu_bfs_download(self.h, _ip(out)), "bfs_download")
        return out

    def bfs_distances(self, cells):
        c = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        out = np.zeros(len(c), np.int32)
        self._ck(self.L.smplgpu_bfs_distances(self.h, _ip(c), len(c), _ip(out)), "bfs_distances")
        return out

    def bfs_last_levels(self):
        return self.L.smplgpu_bfs_last_levels(self.h)

    def goal_heuristics(self, q, cost_per_cell):
        q = self._q(q)
        h = np.zeros(len(q), np.int32)
        self._ck(self.L.smplgpu_goal_heuristics(self.h, _dp(q), len(q), int(cost_per_cell), _ip(h)), "goal_heuristics")
        return h

    def goal_heuristics_dev(self, q_ptr, n, cost_per_cell, h_ptr):
        self._ck(self.L.smplgpu_goal_heuristics_dev(self.h, C.c_void_p(q_ptr), int(n), int(cost_per_cell),
                                                    C.c_void_p(h_ptr)), "goal_heuristics_dev")

    def planning_frame_fk(self, q):
        q = self._q(q)
        out = np.zeros((len(q), 6))
        self._ck(self.L.smplgpu_planning_frame_fk(self.h, _dp(q), len(q), _dp(out)), "planning_frame_fk")
        return out

    def planning_link_ik(self, poses, seeds, max_iterations=100, tolerance=1e-6):
        """smplgpu_planning_link_ik: the planning link's IK for target-offset poses (n, 6) x y z roll pitch yaw,
        seeded at seeds (n, dof).  Targets of shape (n, 3) (positions) take the position-only IK,
        smplgpu_planning_link_ik_position, whose answers leave the orientation free.
        Returns (q (n, dof), ok (n,) bool, iterations (n,))."""
        poses = np.ascontiguousarray(poses, dtype=np.float64)
        width = 3 if poses.shape[-1] == 3 else 6
        poses = poses.reshape(-1, width)
        seeds = self._q(seeds)
        if len(seeds) != len(poses):
            raise ValueError("%d poses, %d seeds" % (len(poses), len(seeds)))
        n = len(poses)
        q = np.zeros_like(seeds)
        ok = np.zeros(n, np.uint8)
        it = np.zeros(n, np.int32)
        prm = IkParamsC(int(max_iterations), float(tolerance))
        f = self.L.smplgpu_planning_link_ik if width == 6 else self.L.smplgpu_planning_link_ik_position
        self._ck(f(self.h, _dp(poses), _dp(seeds), n, C.byref(prm), _dp(q), _bp(ok), _ip(it)), "planning_link_ik")
        return q, ok.astype(bool), it


    # ---- many queries at once ----
    def bfs_bank_create(self, n_slots, inflation_radius):
        return self._ck(self.L.smplgpu_bfs_bank_create(self.h, int(n_slots), float(inflation_radius)), "bfs_bank_create")

    def bfs_bank_max_slots(self):
        return self._ck(self.L.smplgpu_bfs_bank_max_slots(self.h), "bfs_bank_max_slots")

    def bfs_bank_run_slots(self, slots, seeds):
        sl = np.ascontiguousarray(slots, dtype=np.int32)
        s = np.ascontiguousarray(seeds, dtype=np.int32).reshape(-1, 3)
        return self._ck(self.L.smplgpu_bfs_bank_run_slots(self.h, _ip(sl), _ip(s), len(sl)), "bfs_bank_run_slots")

    def bfs_bank_run_slots_multi(self, slots, seed_sets, wait=True):
        """smplgpu_bfs_bank_run_slots_multi (_async when wait is False): slot slots[i] seeded at every cell of
        seed_sets[i] ((k, 3) ints, k >= 0).  Returns the seeds in bounds (synchronous) or the slot count."""
        sl = np.ascontiguousarray(slots, dtype=np.int32)
        cells = [np.asarray(c, np.int32).reshape(-1, 3) for c in seed_sets]
        off = np.zeros(len(cells) + 1, np.int32)
        off[1:] = np.cumsum([len(c) for c in cells])
        s = np.ascontiguousarray(np.concatenate(cells) if cells else np.zeros((0, 3), np.int32), dtype=np.int32)
        s = s if s.size else np.zeros(3, np.int32)
        f = self.L.smplgpu_bfs_bank_run_slots_multi if wait else self.L.smplgpu_bfs_bank_run_slots_multi_async
        return self._ck(f(self.h, _ip(sl), _ip(s), _ip(off), len(sl)), "bfs_bank_run_slots_multi")

    def bfs_bank_run_slots_async(self, slots, seeds):
        """Queues the BFS of the listed slots and returns; poll bfs_bank_run_done() or call bfs_bank_run_wait()."""
        sl = np.ascontiguousarray(slots, dtype=np.int32)
        s = np.ascontiguousarray(seeds, dtype=np.int32).reshape(-1, 3)
        return self._ck(self.L.smplgpu_bfs_bank_run_slots_async(self.h, _ip(sl), _ip(s), len(sl)), "bfs_bank_run_slots_async")

    def bfs_bank_run_done(self):
        return self._ck(self.L.smplgpu_bfs_bank_run_done(self.h), "bfs_bank_run_done") == 1

    def bfs_bank_run_wait(self):
        self._ck(self.L.smplgpu_bfs_bank_run_wait(self.h), "bfs_bank_run_wait")

    def bfs_bank_run(self, seeds):
        s = np.ascontiguousarray(seeds, dtype=np.int32).reshape(-1, 3)
        return self._ck(self.L.smplgpu_bfs_bank_run(self.h, _ip(s)), "bfs_bank_run")

    def bfs_bank_distances(self, slot, cells):
        c = np.ascontiguousarray(cells, dtype=np.int32).reshape(-1, 3)
        sl = np.ascontiguousarray(slot, dtype=np.int32)
        out = np.zeros(len(c), np.int32)
        self._ck(self.L.smplgpu_bfs_bank_distances(self.h, _ip(sl), _ip(c), len(c), _ip(out)), "bfs_bank_distances")
        return out

    def expand_batch(self, q0, q1, slot, cost_per_cell):
        q0, q1 = self._q(q0), self._q(q1)
        n = len(q0)
        sl = np.ascontiguousarray(slot, dtype=np.int32)
        v, h, g, off = np.zeros(n, np.uint8), np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros((n, 3))
        self._ck(self.L.smplgpu_expand_batch(self.h, _dp(q0), _dp(q1), _ip(sl), n, int(cost_per_cell), _bp(v), _ip(h),
                                             _ip(g), _dp(off)), "expand_batch")
        return v, h, g, off


    def set_lattice(self, resolutions):
        """ManipLattice::init discretisation; returns the number of lattice values per variable."""
        r = np.ascontiguousarray(resolutions, dtype=np.float64)
        vals = np.zeros(len(r), np.int32)
        self._ck(self.L.smplgpu_set_lattice(self.h, _dp(r), _ip(vals)), "set_lattice")
        return vals

    def is_lattice_states_valid(self, coords):
        c = np.ascontiguousarray(coords, dtype=np.int16)
        v = np.zeros(len(c), np.uint8)
        self._ck(self.L.smplgpu_is_lattice_states_valid(self.h, c.ctypes.data_as(C.POINTER(C.c_int16)), len(c), _bp(v)),
                 "is_lattice_states_valid")
        return v

    def is_lattice_edges_valid(self, coords, prim_id, deltas, want_counts=True):
        c = np.ascontiguousarray(coords, dtype=np.int16)
        p = np.ascontiguousarray(prim_id, dtype=np.uint8)
        d = np.ascontiguousarray(deltas, dtype=np.float64)
        v = np.zeros(len(c), np.uint8)
        cnt = np.zeros(len(c), np.int32) if want_counts else None
        self._ck(self.L.smplgpu_is_lattice_edges_valid(self.h, c.ctypes.data_as(C.POINTER(C.c_int16)), _bp(p), len(c), _dp(d),
                                                       len(d), _bp(v), _ip(cnt) if want_counts else None),
                 "is_lattice_edges_valid")
        return (v, cnt) if want_counts else v

    def set_motion_primitives(self, deltas):
        d = np.ascontiguousarray(deltas, dtype=np.float64)
        self._n_prims = len(d)
        self._ck(self.L.smplgpu_set_motion_primitives(self.h, _dp(d), len(d)), "set_motion_primitives")

    def expand_state(self, parent, cost_per_cell):
        """One launch: the records of `parent` (index 0) and of parent + every primitive, as a dict of arrays."""
        q = np.ascontiguousarray(parent, dtype=np.float64)
        info = C.POINTER(SuccInfoC)()
        self._ck(self.L.smplgpu_expand_state(self.h, _dp(q), int(cost_per_cell), C.byref(info)), "expand_state")
        n = self._n_prims + 1
        dof = len(q)
        return {
            "state": np.array([list(info[k].state)[:dof] for k in range(n)]),
            "pose": np.array([list(info[k].pose) for k in range(n)]),
            "link_xyz": np.array([list(info[k].link_xyz) for k in range(n)]),
            "h": np.array([info[k].h for k in range(n)], np.int32),
            "goal_dist_cells": np.array([info[k].goal_dist_cells for k in range(n)], np.int32),
            "waypoints": np.array([info[k].waypoints for k in range(n)], np.int32),
            "edge_valid": np.array([info[k].edge_valid for k in range(n)], np.uint8),
            "limits_ok": np.array([info[k].limits_ok for k in range(n)], np.uint8),
            "state_valid": np.array([info[k].state_valid for k in range(n)], np.uint8),
            "is_parent": np.array([info[k].is_parent for k in range(n)], np.uint8),
        }

    def scene_epoch(self):
        return int(self.L.smplgpu_scene_epoch(self.h))


class Adapters:
    """The C++ drop-in adapters (GpuCollisionSpace / GpuRobotModel / GpuBfsHeuristic) driven one virtual call
    at a time, as the reference's planner drives its plugins."""

    def __init__(self, ctx, scene, tables):
        self.H = host_lib()
        self.dof = tables.dof
        o = np.ascontiguousarray(scene.origin, dtype=np.float64)
        d = np.ascontiguousarray(scene.dims, dtype=np.int32)
        h = self.H.smplhost_adapters_create(ctx.h, tables.h, (scene.planning_link or "").encode(), _dp(o),
                                            float(scene.res), _ip(d), float(scene.inflation_radius),
                                            int(scene.cost_per_cell))
        if not h:
            raise SmplGpuError("adapters: " + self.H.smplhost_last_error().decode())
        self.h = C.c_void_p(h)

    def close(self):
        if getattr(self, "h", None):
            self.H.smplhost_adapters_destroy(self.h)
            self.h = None

    def _v(self, q):
        return np.ascontiguousarray(q, dtype=np.float64)

    def enable_expansion_cache(self, deltas):
        """ExpansionCache: one smplgpu_expand_state launch per expanded state answers the per-call virtuals."""
        d = np.ascontiguousarray(deltas, dtype=np.float64).reshape(-1, self.dof)
        self.H.smplhost_adapters_enable_expansion_cache.argtypes = [C.c_void_p, c_double_p, C.c_int, C.POINTER(C.c_int64)]
        if self.H.smplhost_adapters_enable_expansion_cache(self.h, _dp(d), len(d), None) != 0:
            raise SmplGpuError("expansion cache: " + self.H.smplhost_last_error().decode())

    def expansion_cache_counters(self):
        c = (C.c_int64 * 2)()
        self.H.smplhost_adapters_enable_expansion_cache.argtypes = [C.c_void_p, c_double_p, C.c_int, C.POINTER(C.c_int64)]
        self.H.smplhost_adapters_enable_expansion_cache(self.h, None, 0, c)
        return int(c[0]), int(c[1])

    def is_state_valid(self, q):
        return self.H.smplhost_cc_is_state_valid(self.h, _dp(self._v(q)))

    def is_state_to_state_valid(self, q0, q1):
        return self.H.smplhost_cc_is_state_to_state_valid(self.h, _dp(self._v(q0)), _dp(self._v(q1)))

    def interpolate_path(self, q0, q1, max_waypoints=512):
        out = np.zeros((max_waypoints, self.dof))
        n = self.H.smplhost_cc_interpolate_path(self.h, _dp(self._v(q0)), _dp(self._v(q1)), _dp(out), max_waypoints)
        return None if n < 0 else out[:n].copy()

    def is_states_valid(self, q):
        q = self._v(q).reshape(-1, self.dof)
        v = np.zeros(len(q), np.uint8)
        if self.H.smplhost_cc_is_states_valid(self.h, _dp(q), len(q), _bp(v)) != 0:
            raise SmplGpuError("isStatesValid failed")
        return v

    def is_edges_valid(self, q0, q1):
        q0, q1 = self._v(q0).reshape(-1, self.dof), self._v(q1).reshape(-1, self.dof)
        v = np.zeros(len(q0), np.uint8)
        if self.H.smplhost_cc_is_edges_valid(self.h, _dp(q0), _dp(q1), len(q0), _bp(v)) != 0:
            raise SmplGpuError("isEdgesValid failed")
        return v

    def distance_to_collision(self, q0, q1=None):
        self.H.smplhost_cc_distance_to_collision.restype = C.c_double
        self.H.smplhost_cc_distance_to_collision.argtypes = [C.c_void_p, c_double_p, c_double_p]
        return self.H.smplhost_cc_distance_to_collision(self.h, _dp(self._v(q0)), _dp(self._v(q1)) if q1 is not None else None)

    def check_joint_limits(self, q):
        return self.H.smplhost_rm_check_joint_limits(self.h, _dp(self._v(q)))

    def compute_planning_link_fk(self, q):
        out = np.zeros(6)
        if self.H.smplhost_rm_compute_planning_link_fk(self.h, _dp(self._v(q)), _dp(out)) != 0:
            return None
        return out

    def update_goal(self, xyz):
        return self.H.smplhost_heur_update_goal(self.h, _dp(self._v(xyz)))

    def goal_heuristic(self, q):
        return self.H.smplhost_heur_goal_heuristic(self.h, _dp(self._v(q)))

    def metric_goal_distance(self, x, y, z):
        return self.H.smplhost_heur_metric_goal_distance(self.h, float(x), float(y), float(z))


def clone_context(ctx, scene, tables, device=0):
    """Another context on the same GPU with the same robot tables and a device-to-device copy of the distance field
    (one context per planner thread)."""
    c = GpuContext(device)
    c.set_robot(tables)
    ptr, _ = ctx.distance_field_dev_ptr()
    dmax = int(np.ceil(scene.max_dist * (1.0 / scene.res)))
    c.set_distance_field_dev(ptr, scene.dims, scene.origin, scene.res, dmax * dmax, scene.padding)
    return c


def plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=64, max_path=512, n_threads=1,
               want_states=False, snap=None):
    """smplhost_plan_batch: many ARA* queries in lock step, one device call per round.
    params: smpl_b200.scenes.PlanParams.  Returns (list of dict per query, stats dict).
    goals: (nq, 3) positions (XYZ goals with params.xyz_tolerance), or goal records of GOAL_DTYPE (pose_goals,
    joint_goals; types may be mixed), which go through smplhost_plan_batch_goals, or a goal set per query, the
    (records, offsets) pair of goal_sets(), through smplhost_plan_batch_goal_sets: each result then also holds
    reached_goal, the index in the query's set of the record its path reaches (-1 when unsolved).
    `ctx` may be a list of contexts (same GPU, same scene): one planner thread per context
    (smplhost_plan_batch_multi), max_concurrent is then per context.
    snap: SnapParams -- the snap-to-goal actions, through smplhost_plan_batch_snap (position goals become XYZ goal
    records), or smplhost_plan_batch_snaps when SNAP_TO_XYZ or SNAP_TO_RPY is on; the stats then also hold
    ik_attempted / ik_converged (totals over the kinds) and, per kind name of SNAP_KIND_NAMES, ik_attempted_<kind> /
    ik_converged_<kind>."""
    H = host_lib()
    dof = tables.dof
    starts = np.ascontiguousarray(starts, dtype=np.float64).reshape(-1, dof)
    offsets = None
    if isinstance(goals, tuple):
        goals, offsets = goals
        offsets = np.ascontiguousarray(offsets, dtype=np.int32).reshape(-1)
        if len(offsets) != len(starts) + 1:
            raise ValueError("%d starts, %d goal sets" % (len(starts), len(offsets) - 1))
    records = isinstance(goals, np.ndarray) and goals.dtype == GOAL_DTYPE
    if snap is not None and not records:
        goals = pose_goals(np.asarray(goals, np.float64).reshape(-1, 3), params.xyz_tolerance)
        records = True
    if records:
        goals = np.ascontiguousarray(goals.reshape(-1))
    else:
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(-1, 3)
    if offsets is None and len(goals) != len(starts):
        raise ValueError("%d starts, %d goals" % (len(starts), len(goals)))
    nq = len(starts)
    lo, hi, cont = tables.limits()
    res = np.ascontiguousarray(params.resolutions, dtype=np.float64)
    prims = np.ascontiguousarray(params.mprims, dtype=np.float64)
    flags = np.ascontiguousarray(params.short_flags, dtype=np.uint8)
    P = PlanParamsC()
    P.dof = dof
    P.resolutions, P.mprims, P.short_flags, P.n_prims = _dp(res), _dp(prims), _bp(flags), len(prims)
    P.use_short_dist, P.short_dist_thresh = int(params.use_short_dist), float(params.short_dist_thresh)
    P.epsilon, P.max_expansions = float(params.epsilon), int(params.max_expansions)
    P.cost_per_cell, P.inflation_radius = int(scene.cost_per_cell), float(scene.inflation_radius)
    P.var_min, P.var_max, P.var_continuous = _dp(lo), _dp(hi), _bp(cont)
    P.res = float(scene.res)
    P.n_threads = int(n_threads)
    weights = getattr(params, "weights", None)
    if weights is not None:
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        assert len(weights) == len(prims)
        P.prim_weights = _dp(weights)
    for a in range(3):
        P.xyz_tolerance[a] = float(params.xyz_tolerance[a])
        P.origin[a] = float(scene.origin[a])
        P.dims[a] = int(scene.dims[a])
    summary = np.zeros((nq, 5), np.int32)
    paths = np.full((nq, max_path), -1, np.int32)
    stats = np.zeros(12)
    pstates = np.zeros((nq, max_path, dof), np.float64) if want_states else None
    ps_ptr = _dp(pstates) if want_states else None
    counters = np.zeros(6, np.int64)
    reached = np.full(nq, -1, np.int32)
    if snap is not None and snap.new_kinds():
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
        sp = snap.c_kinds()
        off = offsets if offsets is not None else np.arange(nq + 1, dtype=np.int32)
        r = H.smplhost_plan_batch_snaps(arr, len(ctxs), C.byref(P), _dp(starts), goals.ctypes.data_as(C.POINTER(GoalC)),
                                        _ip(off), nq, int(max_concurrent), _ip(summary), _ip(paths), int(max_path),
                                        _dp(stats), ps_ptr, C.byref(sp), counters.ctypes.data_as(C.POINTER(C.c_int64)),
                                        _ip(reached))
    elif offsets is not None:
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
        sp = snap.c() if snap is not None else None
        r = H.smplhost_plan_batch_goal_sets(arr, len(ctxs), C.byref(P), _dp(starts),
                                            goals.ctypes.data_as(C.POINTER(GoalC)), _ip(offsets), nq,
                                            int(max_concurrent), _ip(summary), _ip(paths), int(max_path), _dp(stats),
                                            ps_ptr, C.byref(sp) if sp is not None else None,
                                            counters.ctypes.data_as(C.POINTER(C.c_int64)), _ip(reached))
    elif snap is not None:
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
        sp = snap.c()
        r = H.smplhost_plan_batch_snap(arr, len(ctxs), C.byref(P), _dp(starts), goals.ctypes.data_as(C.POINTER(GoalC)), nq,
                                       int(max_concurrent), _ip(summary), _ip(paths), int(max_path), _dp(stats), ps_ptr,
                                       C.byref(sp), counters.ctypes.data_as(C.POINTER(C.c_int64)))
    elif records:
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
        r = H.smplhost_plan_batch_goals(arr, len(ctxs), C.byref(P), _dp(starts), goals.ctypes.data_as(C.POINTER(GoalC)), nq,
                                        int(max_concurrent), _ip(summary), _ip(paths), int(max_path), _dp(stats), ps_ptr)
    elif isinstance(ctx, (list, tuple)):
        arr = (C.c_void_p * len(ctx))(*[c.h for c in ctx])
        r = H.smplhost_plan_batch_multi(arr, len(ctx), C.byref(P), _dp(starts), _dp(goals), nq, int(max_concurrent),
                                        _ip(summary), _ip(paths), int(max_path), _dp(stats), ps_ptr)
    else:
        r = H.smplhost_plan_batch(ctx.h, C.byref(P), _dp(starts), _dp(goals), nq, int(max_concurrent), _ip(summary),
                                  _ip(paths), int(max_path), _dp(stats), ps_ptr)
    if r != 0:
        raise SmplGpuError("plan_batch: " + H.smplhost_last_error().decode())
    out = []
    for i in range(nq):
        n = int(summary[i, 3])
        out.append(dict(success=bool(summary[i, 0]), expansions=int(summary[i, 1]), cost=int(summary[i, 2]),
                        path_ids=paths[i, :min(n, max_path)].copy(), num_states=int(summary[i, 4])))
        if want_states:   # ManipLattice::extractPath: joint values of the path states
            out[-1]["path_states"] = pstates[i, :min(n, max_path)].copy()
        if offsets is not None:
            out[-1]["reached_goal"] = int(reached[i])
    st = dict(rounds=int(stats[0]), edges_submitted=int(stats[1]), device_calls=int(stats[2]),
              device_seconds=float(stats[3]), host_seconds=float(stats[4]), total_seconds=float(stats[5]),
              bfs_runs=int(stats[6]), edges_resolved_f64=int(stats[7]), setup_seconds=float(stats[8]),
              max_wait_seconds=float(stats[9]), n_threads=int(n_threads))
    if snap is not None:
        if not snap.new_kinds():   # the two-counter entry points: every solve is SNAP_TO_XYZ_RPY's
            counters[2 * SNAP_XYZ_RPY:2 * SNAP_XYZ_RPY + 2] = counters[:2]
            counters[:2] = 0
        st.update(ik_attempted=int(counters[0::2].sum()), ik_converged=int(counters[1::2].sum()))
        for k, name in enumerate(SNAP_KIND_NAMES):
            st.update({"ik_attempted_" + name: int(counters[2 * k]), "ik_converged_" + name: int(counters[2 * k + 1])})
    return out, st


def _concat_paths(paths, dof):
    pts = [np.ascontiguousarray(p, dtype=np.float64).reshape(-1, dof) for p in paths]
    offsets = np.zeros(len(pts) + 1, np.int32)
    offsets[1:] = np.cumsum([len(p) for p in pts])
    flat = np.ascontiguousarray(np.concatenate(pts) if pts else np.zeros((0, dof)), dtype=np.float64)
    return flat, offsets


def shortcut_paths(ctx, tables, paths, kind=0):
    """smplhost_shortcut_paths: ShortcutPath (post_processing.cpp:284-365) for a list of joint-space paths; every
    candidate motion is checked in one device call.  kind 0 = JOINT_SPACE, 1 = JOINT_POSITION_VELOCITY_SPACE.
    Returns (list of index arrays -- the points each shortcut path keeps, stats dict)."""
    H = host_lib()
    dof = tables.dof
    flat, offsets = _concat_paths(paths, dof)
    _, _, cont = tables.limits()
    cont = np.ascontiguousarray(cont, dtype=np.uint8)
    out_idx = np.zeros(max(1, int(offsets[-1])), np.int32)
    out_off = np.zeros(len(offsets), np.int32)
    stats = np.zeros(5)
    r = H.smplhost_shortcut_paths(ctx.h, dof, _bp(cont), _dp(flat), _ip(offsets), len(paths), int(kind), _ip(out_idx),
                                  _ip(out_off), _dp(stats))
    if r != 0:
        raise SmplGpuError("shortcut_paths: " + H.smplhost_last_error().decode())
    st = dict(edges_checked=int(stats[0]), states_checked=int(stats[1]), device_calls=int(stats[2]),
              device_seconds=float(stats[3]), host_seconds=float(stats[4]))
    return [out_idx[out_off[i]:out_off[i + 1]].copy() for i in range(len(paths))], st


def interpolate_paths(ctx, tables, paths):
    """smplhost_interpolate_paths: InterpolatePath (post_processing.cpp:476-540) for a list of joint-space paths; the
    waypoints of every segment are checked in one device call.  Returns (list of point arrays, stats dict)."""
    H = host_lib()
    dof = tables.dof
    flat, offsets = _concat_paths(paths, dof)
    out_off = np.zeros(len(offsets), np.int32)
    stats = np.zeros(5)
    total = H.smplhost_interpolate_paths(ctx.h, tables.h, _dp(flat), _ip(offsets), len(paths), None, 0, _ip(out_off), None)
    if total < 0:
        raise SmplGpuError("interpolate_paths: " + H.smplhost_last_error().decode())
    out = np.zeros((max(1, total), dof), np.float64)
    r = H.smplhost_interpolate_paths(ctx.h, tables.h, _dp(flat), _ip(offsets), len(paths), _dp(out), max(1, total),
                                     _ip(out_off), _dp(stats))
    if r < 0:
        raise SmplGpuError("interpolate_paths: " + H.smplhost_last_error().decode())
    st = dict(edges_checked=int(stats[0]), states_checked=int(stats[1]), device_calls=int(stats[2]),
              device_seconds=float(stats[3]), host_seconds=float(stats[4]))
    return [out[out_off[i]:out_off[i + 1]].copy() for i in range(len(paths))], st


def world_to_grid(points, origin, res):
    """DistanceMap::worldToGrid (distance_map.hpp:520-527) in IEEE double, C truncation."""
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    inv = 1.0 / res
    o = np.asarray(origin, dtype=np.float64) - res
    t = inv * (p - o) + 0.5
    return np.trunc(t).astype(np.int64).astype(np.int32) - 1


def build_tables(scene):
    """RobotTables configured for a smpl_b200.scenes.Scene."""
    t = RobotTables(scene.robot_path)
    t.configure(scene.group, scene.planning_joints)
    for k, v in scene.fixed_joints.items():
        t.set_joint(k, v)
    if scene.use_desc_acm:
        t.use_file_acm()
    for a, b, allowed in scene.acm_extra:
        t.set_acm_entry(a, b, allowed)
    if scene.attached is not None:
        body_id, link, centers, radius = scene.attached
        t.attach_spheres(body_id, link, centers, radius)
    if scene.chain_root is not None:
        t.set_planning_chain(scene.chain_root, scene.chain_tip, scene.planning_link, scene.T_kin_to_planning,
                             scene.xyz_offset)
    return t


def scene_cells(scene, tables):
    """Occupied cells of a scene: world obstacles + voxels of out-of-group robot links."""
    vox = tables.outside_voxels()
    cells = scene.cells
    if len(vox):
        g = world_to_grid(vox, scene.origin, scene.res)
        ok = np.all((g >= 0) & (g < np.asarray(scene.dims)), axis=1)
        cells = np.concatenate([cells, g[ok]], axis=0)
    return np.ascontiguousarray(cells, dtype=np.int32)


def box_meshes(boxes):
    """smplhost_box_meshes: boxes[n][15] (size, pose 3x4) -> (vertices[8n][3], triangles[12n][3])."""
    H = host_lib()
    b = np.ascontiguousarray(boxes, dtype=np.float64).reshape(-1, 15)
    v = np.zeros((8 * len(b), 3), np.float64)
    t = np.zeros((12 * len(b), 3), np.int32)
    if H.smplhost_box_meshes(_dp(b), len(b), _dp(v), _ip(t)) != 0:
        raise SmplGpuError("box_meshes: " + H.smplhost_last_error().decode())
    return v, t


SHAPE_BOX, SHAPE_SPHERE, SHAPE_CYLINDER, SHAPE_CONE = 0, 1, 2, 3


def shape_meshes(shapes):
    """smplhost_shape_meshes: shapes[n][16] = kind, 3 dimensions, pose 3x4 -> (vertices[.][3], triangles[.][3])."""
    H = host_lib()
    sh = np.ascontiguousarray(shapes, dtype=np.float64).reshape(-1, 16)
    nv = nt = 0
    for row in sh:
        a, b = np.zeros(1, np.int32), np.zeros(1, np.int32)
        if H.smplhost_shape_mesh_size(int(row[0]), _ip(a), _ip(b)) != 0:
            raise SmplGpuError("shape_meshes: unknown shape kind %d" % int(row[0]))
        nv += int(a[0])
        nt += int(b[0])
    v = np.zeros((max(nv, 1), 3), np.float64)
    t = np.zeros((max(nt, 1), 3), np.int32)
    if H.smplhost_shape_meshes(_dp(sh), len(sh), _dp(v), _ip(t)) != nt:
        raise SmplGpuError("shape_meshes: " + H.smplhost_last_error().decode())
    return v[:nv], t[:nt]


def setup_context(scene, device=0, ctx=None):
    """Create a context with robot tables and a device-built distance field for `scene`.  Box objects of the scene
    (scene.boxes) go through the device voxeliser, the way WorldCollisionModel::insertObject ingests them."""
    ctx = ctx or GpuContext(device)
    tables = build_tables(scene)
    ctx.set_robot(tables)
    cells = scene_cells(scene, tables)
    if len(getattr(scene, "boxes", [])):
        v, t = box_meshes(scene.boxes)
        ctx.build_distance_field_from_meshes(v, t, cells, scene.dims, scene.origin, scene.res, scene.max_dist,
                                             scene.padding)
    else:
        ctx.build_distance_field(cells, scene.dims, scene.origin, scene.res, scene.max_dist, scene.padding)
    return ctx, tables
