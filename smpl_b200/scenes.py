"""Synthetic scenes and query sets of the shapes BASELINE.json names (SURVEY.md section 8d).

Pure input generators (numpy): occupied-cell lists, random joint states,
motion-primitive edges, BFS wall grids.  Both the CUDA path and the CPU oracle
consume exactly these arrays, so no RNG has to agree across languages.
"""
import math
import os

import numpy as np

DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")

PR2_RIGHT_ARM_JOINTS = [
    "r_shoulder_pan_joint", "r_shoulder_lift_joint", "r_upper_arm_roll_joint", "r_elbow_flex_joint",
    "r_forearm_roll_joint", "r_wrist_flex_joint", "r_wrist_roll_joint",
]
PR2_LEFT_ARM_JOINTS = ["l" + j[1:] for j in PR2_RIGHT_ARM_JOINTS]
UBR1_ARM_JOINTS = [
    "shoulder_pan_joint", "shoulder_lift_joint", "upperarm_roll_joint", "elbow_flex_joint",
    "forearm_roll_joint", "wrist_flex_joint", "wrist_roll_joint",
]


def grid_dims(size, res):
    """Cell counts as DistanceMap's constructor computes them (distance_map.hpp:136-138)."""
    inv = 1.0 / res
    return tuple(int(s * inv + 0.5) for s in size)


def box_cells(origin, res, dims, center, size):
    """Effective grid cells whose centres (origin + i*res) lie inside an axis-aligned box."""
    lo = [int(math.ceil((center[a] - 0.5 * size[a] - origin[a]) / res - 1e-9)) for a in range(3)]
    hi = [int(math.floor((center[a] + 0.5 * size[a] - origin[a]) / res + 1e-9)) for a in range(3)]
    lo = [max(0, v) for v in lo]
    hi = [min(dims[a] - 1, hi[a]) for a in range(3)]
    if any(hi[a] < lo[a] for a in range(3)):
        return np.zeros((0, 3), np.int32)
    xs, ys, zs = np.meshgrid(np.arange(lo[0], hi[0] + 1), np.arange(lo[1], hi[1] + 1),
                             np.arange(lo[2], hi[2] + 1), indexing="ij")
    return np.stack([xs.ravel(), ys.ravel(), zs.ravel()], axis=1).astype(np.int32)


class Scene:
    """Grid parameters + occupied cells + robot setup of one benchmark configuration."""

    def __init__(self, robot, group, planning_joints, origin, size, res, max_dist):
        self.robot_path = os.path.join(DATA, robot + ".robot")
        self.group = group
        self.planning_joints = list(planning_joints)
        self.origin = tuple(float(v) for v in origin)
        self.size = tuple(float(v) for v in size)
        self.res = float(res)
        self.max_dist = float(max_dist)
        self.dims = grid_dims(size, res)
        self.cells = np.zeros((0, 3), np.int32)
        self.fixed_joints = {}
        self.use_desc_acm = False
        self.padding = 0.0
        # planning model (KDL chain) parameters
        self.chain_root = None
        self.chain_tip = None
        self.planning_link = None
        self.T_kin_to_planning = np.eye(4)[:3].copy()
        self.xyz_offset = (0.0, 0.0, 0.0)
        self.chain_subset = False      # True: the chain moves only some of the planning variables (set_planning_chain)
        self.inflation_radius = 0.02   # planning_link_sphere_radius, call_planner.cpp:1715
        self.cost_per_cell = 250       # planning_params.h:68 default... set by callers
        self.attached = None           # (id, link, centers[n,3], radius)
        self.acm_extra = []            # (a, b, allowed) entries applied on top of the ACM
        # box collision objects ingested the reference's way (VoxelizeBox, surface voxels): rows of 15 doubles =
        # length, width, height, pose 3x4 row-major in the grid frame
        self.boxes = np.zeros((0, 15), np.float64)

    def add_box(self, center, size):
        c = box_cells(self.origin, self.res, self.dims, center, size)
        self.cells = np.concatenate([self.cells, c], axis=0)

    def add_box_object(self, center, size, rpy=(0.0, 0.0, 0.0)):
        """A box collision object (call_planner.cpp GetCollisionCube: id x y z dx dy dz; rpy for rotated shelves)."""
        cr, sr = math.cos(rpy[0]), math.sin(rpy[0])
        cp, sp = math.cos(rpy[1]), math.sin(rpy[1])
        cy, sy = math.cos(rpy[2]), math.sin(rpy[2])
        R = np.array([[cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr],
                      [sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr],
                      [-sp, cp * sr, cp * cr]]) if any(rpy) else np.eye(3)
        pose = np.concatenate([R, np.asarray(center, dtype=np.float64).reshape(3, 1)], axis=1)
        row = np.concatenate([np.asarray(size, dtype=np.float64), pose.ravel()])
        self.boxes = np.concatenate([self.boxes, row[None, :]], axis=0)

    @property
    def dof(self):
        return len(self.planning_joints)


def _pr2_common(scene):
    scene.fixed_joints = {"torso_lift_joint": 0.16825}           # pr2_goal.yaml:3
    scene.use_desc_acm = True                                     # call_planner.cpp:1630-1632
    scene.chain_root = "torso_lift_link"                          # goal_pr2.launch kinematics_frame
    scene.chain_tip = "r_gripper_palm_link"
    scene.planning_link = "r_gripper_palm_link"
    T = np.eye(4)[:3].copy()
    T[:, 3] = (-0.05, 0.0, 0.959)                                 # pr2_goal.yaml:13-19
    scene.T_kin_to_planning = T
    scene.cost_per_cell = 100


def pr2_tabletop_scene():
    """Config 1: smpl_test PR2 right arm in the tabletop env (call_planner.cpp:1587-1594, tabletop.env)."""
    s = Scene("pr2", "right_arm", PR2_RIGHT_ARM_JOINTS, (-0.75, -1.5, 0.0), (3.0, 3.0, 3.0), 0.02, 1.8)
    _pr2_common(s)
    # tabletop.env declares 1 object: id x y z dx dy dz
    s.add_box((0.55, 0.0, 0.6), (0.4, 1.5, 0.02))
    return s


def pr2_tabletop_env_scene():
    """Config 1 with the table ingested the reference's way: the env box goes through VoxelizeBox (surface voxels,
    voxel origin = grid origin) and addPointsToField instead of our filled cell box."""
    s = Scene("pr2", "right_arm", PR2_RIGHT_ARM_JOINTS, (-0.75, -1.5, 0.0), (3.0, 3.0, 3.0), 0.02, 1.8)
    _pr2_common(s)
    s.add_box_object((0.55, 0.0, 0.6), (0.4, 1.5, 0.02))
    return s


def pr2_shelf_objects_scene(seed=23, n_boxes=30):
    """The clutter volume (2 m^3 at 2 cm) filled with box OBJECTS at arbitrary orientations: shelf boards, tilted
    panels and small items, some sticking out of the grid."""
    s = Scene("pr2", "right_arm", PR2_RIGHT_ARM_JOINTS, (-0.5, -1.0, 0.0), (2.0, 2.0, 2.0), 0.02, 0.4)
    _pr2_common(s)
    rng = np.random.Generator(np.random.PCG64(seed))
    for z in (0.4, 0.8, 1.2):
        s.add_box_object((0.95, 0.0, z), (0.5, 1.6, 0.02))
    s.add_box_object((1.45, 0.9, 1.0), (0.3, 0.5, 1.2), rpy=(0.0, 0.0, 0.3))          # half outside the grid
    placed = 0
    while placed < n_boxes:
        size = rng.uniform(0.03, 0.3, 3)
        center = np.array(s.origin) + rng.uniform(0.0, 1.0, 3) * np.array(s.size)
        if abs(center[0] + 0.1) < 0.5 + 0.5 * size.max() and abs(center[1]) < 0.6 + 0.5 * size.max():
            continue  # robot body column
        s.add_box_object(center, size, rpy=tuple(rng.uniform(-1.0, 1.0, 3)) if placed % 3 else (0.0, 0.0, 0.0))
        placed += 1
    return s


def pr2_clutter_scene(seed=7, n_boxes=40):
    """Config 2: 2x2x2 m scene at 2 cm, 40 random boxes (SURVEY.md section 8d)."""
    s = Scene("pr2", "right_arm", PR2_RIGHT_ARM_JOINTS, (-0.5, -1.0, 0.0), (2.0, 2.0, 2.0), 0.02, 0.4)
    _pr2_common(s)
    rng = np.random.Generator(np.random.PCG64(seed))
    shoulder = np.array([-0.05, -0.188, 0.959])
    placed = 0
    while placed < n_boxes:
        size = rng.uniform(0.04, 0.4, 3)
        center = np.array(s.origin) + rng.uniform(0.0, 1.0, 3) * np.array(s.size)
        # reject boxes overlapping the shoulder / torso column
        d = np.maximum(np.abs(center - shoulder) - 0.5 * size, 0.0)
        if np.linalg.norm(d) < 0.30:
            continue
        if abs(center[0] + 0.1) < 0.35 + 0.5 * size[0] and abs(center[1]) < 0.45 + 0.5 * size[1]:
            continue  # robot body column
        s.add_box(center, size)
        placed += 1
    return s


def ubr1_tabletop_scene(attach=True):
    """Config 4 shape: UBR1 arm (7-DOF) with an attached 0.05 x 0.05 x 0.20 m box, tabletop_ubr1.env."""
    s = Scene("ubr1", "arm", UBR1_ARM_JOINTS, (-0.75, -1.25, -0.05), (2.0, 2.0, 2.0), 0.02, 0.4)
    s.fixed_joints = {"torso_lift_joint": 0.0}
    s.chain_root = "torso_lift_link"           # ubr1_goal.yaml kinematics_frame
    s.chain_tip = "gripper_link"               # (the demo's chain tip is a finger link behind a prismatic
    s.planning_link = "gripper_link"           #  joint that is not a planning joint; we stop at gripper_link)
    T = np.eye(4)[:3].copy()
    T[:, 3] = (-0.086875, 0.0, 0.37743)        # base_link -> torso_lift_link at torso_lift_joint = 0
    s.T_kin_to_planning = T
    s.cost_per_cell = 100
    s.add_box((0.8, 0.0, 0.55), (0.3, 1.5, 0.02))   # tabletop_ubr1.env
    # OUR fixture (the reference would take these from the robot's SRDF): sphere models of links
    # separated only by a sphere-less link overlap by construction
    for a, b in (("shoulder_pan_link", "upperarm_roll_link"), ("upperarm_roll_link", "forearm_roll_link"),
                 ("forearm_roll_link", "wrist_roll_link"), ("wrist_roll_link", "left_gripper_finger_link"),
                 ("wrist_roll_link", "right_gripper_finger_link"),
                 ("left_gripper_finger_link", "right_gripper_finger_link")):
        s.acm_extra.append((a, b, True))
    if attach:
        centers = attached_box_spheres((0.05, 0.05, 0.20), offset=(0.26, 0.0, 0.0))
        s.attached = ("object", "wrist_roll_link", centers, 0.025)
        for link in ("wrist_roll_link", "gripper_link", "left_gripper_finger_link", "right_gripper_finger_link"):
            s.acm_extra.append(("object", link, True))   # gripper <-> grasped object ALWAYS (SURVEY.md 8d config 4)
    return s


def pr2_dual_arm_scene(seed=17):
    """Config 5 shape: PR2 torso + both arms (15-DOF), 3 x 3 x 2 m dense shelf scene at 1 cm."""
    joints = ["torso_lift_joint"] + PR2_RIGHT_ARM_JOINTS + PR2_LEFT_ARM_JOINTS
    s = Scene("pr2", "torso", joints, (-1.0, -1.5, 0.0), (3.0, 3.0, 2.0), 0.01, 0.2)
    s.use_desc_acm = True
    s.cost_per_cell = 100
    _dual_arm_shelf(s, seed)
    return s


def _dual_arm_shelf(s, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    # shelf unit in front of the robot: 5 shelves x 4 bays of 2-cell-thick planes
    x0, x1, y0, y1 = 0.75, 1.25, -1.0, 1.0
    for k in range(5):
        s.add_box((0.5 * (x0 + x1), 0.0, 0.3 + 0.35 * k), (x1 - x0, y1 - y0, 0.02))
    for b in range(5):
        y = y0 + b * (y1 - y0) / 4.0
        s.add_box((0.5 * (x0 + x1), y, 1.0), (x1 - x0, 0.02, 1.7))
    s.add_box((x1, 0.0, 1.0), (0.02, y1 - y0, 1.7))
    for _ in range(60):
        size = rng.uniform(0.04, 0.2, 3)
        c = np.array([rng.uniform(x0 + 0.1, x1 - 0.1), rng.uniform(y0 + 0.1, y1 - 0.1), rng.uniform(0.35, 1.7)])
        s.add_box(c, size)


def pr2_dual_arm_planning_scene(res=0.01, planning_link="r_gripper_palm_link", seed=17):
    """Config 5 as a planning problem: pr2_dual_arm_scene's robot, group and shelf at `res`, planned over all 15
    variables with the chain base_link -> planning_link (torso and one arm); the other arm moves collision geometry
    only (Scene.chain_subset).  Planning frame base_footprint, as in the 7-DOF fixtures."""
    joints = ["torso_lift_joint"] + PR2_RIGHT_ARM_JOINTS + PR2_LEFT_ARM_JOINTS
    s = Scene("pr2", "torso", joints, (-1.0, -1.5, 0.0), (3.0, 3.0, 2.0), res, 0.2)
    s.use_desc_acm = True
    s.cost_per_cell = 100
    _dual_arm_shelf(s, seed)
    s.chain_root = "base_link"
    s.chain_tip = planning_link
    s.planning_link = planning_link
    T = np.eye(4)[:3].copy()
    T[:, 3] = (0.0, 0.0, 0.051)                                   # base_footprint_joint
    s.T_kin_to_planning = T
    s.chain_subset = True
    return s


# OUR fixture: the right arm at PR2_DEMO_START and the left arm its mirror image (pan and roll joints negated); the torso
# at 0.25 m, mid-range (below about 0.18 m the torso link's spheres meet the base's voxels, so the 7-DOF scenes' fixed
# 0.16825 m is not collision-free in this group)
DUAL_ARM_START = (0.25,
                  -0.5, 0.3, 0.0, -1.0, 0.0, -0.5, 0.0,
                  0.5, 0.3, 0.0, -1.0, 0.0, -0.5, 0.0)


def random_states(n, lo, hi, continuous, seed):
    """Uniform joint states in [lo, hi] (continuous joints: [-pi, pi]); benchmark_cc.cpp:280-302 recipe."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lo = np.where(np.asarray(continuous, bool), -math.pi, np.asarray(lo, np.float64))
    hi = np.where(np.asarray(continuous, bool), math.pi, np.asarray(hi, np.float64))
    u = rng.random((n, len(lo)))
    return np.ascontiguousarray(lo + u * (hi - lo))


def pr2_mprim_deltas():
    """8 long (7 deg) + 14 short (4 deg) primitives with converses (pr2.mprim, SURVEY 8a defect 2)."""
    d = []
    for j in range(4):
        for sgn in (1.0, -1.0):
            v = np.zeros(7)
            v[j] = sgn * math.radians(7.0)
            d.append(v)
    for j in range(7):
        for sgn in (1.0, -1.0):
            v = np.zeros(7)
            v[j] = sgn * math.radians(4.0)
            d.append(v)
    return np.array(d)


class PlanParams:
    """Planner parameters of the smpl_test demo (pr2_right_arm.yaml, pr2.mprim, call_planner.cpp:93-96, 1715-1729)."""

    def __init__(self, dof=7):
        deg = math.pi / 180.0
        self.resolutions = [0.017453292519943295] * dof
        prims, flags = [], []
        for j in range(min(4, dof)):          # pr2.mprim rows 1-4: 7 degrees on the first four joints (long)
            v = [0.0] * dof
            v[j] = 7.0 * deg
            prims.append(v)
            flags.append(0)
        for j in range(dof):                  # rows 5-11: 4 degrees on every joint (short)
            v = [0.0] * dof
            v[j] = 4.0 * deg
            prims.append(v)
            flags.append(1)
        self.mprims = np.array(prims)
        self.short_flags = np.array(flags, np.uint8)
        self.weights = None                   # per-primitive action weights (None = 1): edge cost = int(1000 * weight)
        self.use_short_dist = True
        self.short_dist_thresh = 0.4
        self.epsilon = 100.0
        self.max_expansions = 200000
        self.xyz_tolerance = [0.015, 0.015, 0.015]


class DualArmPlanParams(PlanParams):
    """Lattice of the 15-DOF planning scene (torso, right arm, left arm): resolutions 0.01 m for the torso and 1 degree
    for the arm joints; long primitives torso +-0.02 m and joints 1-4 of each arm +-7 degrees (18 successor words),
    short primitives every arm joint +-4 degrees (28 words).  Stride 28: with the 3 snap words 31 successors, within the
    lattice kernels' 32."""

    def __init__(self):
        super().__init__(15)
        deg = math.pi / 180.0
        self.resolutions = [0.01] + [0.017453292519943295] * 14
        prims, flags = [], []
        for j, d in [(0, 0.02)] + [(a + j, 7.0 * deg) for a in (1, 8) for j in range(4)]:
            v = [0.0] * 15
            v[j] = d
            prims.append(v)
            flags.append(0)
        for j in range(1, 15):
            v = [0.0] * 15
            v[j] = 4.0 * deg
            prims.append(v)
            flags.append(1)
        self.mprims = np.array(prims)
        self.short_flags = np.array(flags, np.uint8)


def mprim_edges(q, deltas=None):
    """Edge i goes from q[i] to q[i] + delta[i mod K]."""
    if deltas is None:
        deltas = pr2_mprim_deltas()
    k = np.arange(len(q)) % len(deltas)
    return np.ascontiguousarray(q), np.ascontiguousarray(q + deltas[k])


def bfs_clutter_walls(n=400, seed=11, n_boxes=3000):
    """Config 3: n^3 occupancy (uint8 [z,y,x]): random boxes + shelf planes with door gaps."""
    rng = np.random.Generator(np.random.PCG64(seed))
    w = np.zeros((n, n, n), np.uint8)
    scale = n / 400.0
    nb = max(1, int(n_boxes * scale ** 3)) if n < 400 else n_boxes
    for _ in range(nb):
        e = rng.integers(2, max(3, int(40 * scale)) + 1, 3)
        c = rng.integers(0, n, 3)
        lo = np.maximum(c - e // 2, 0)
        hi = np.minimum(lo + e, n)
        w[lo[2]:hi[2], lo[1]:hi[1], lo[0]:hi[0]] = 1
    # six full planes ("shelves") with door gaps
    for k in range(6):
        axis = k % 3
        pos = int(n * (0.15 + 0.14 * k))
        sl = [slice(None)] * 3
        sl[2 - axis] = slice(pos, pos + 2)
        w[tuple(sl)] = 1
        # door gap
        g = max(2, int(12 * scale))
        a = rng.integers(0, n - g, 2)
        gap = [slice(None)] * 3
        gap[2 - axis] = slice(pos, pos + 2)
        others = [i for i in range(3) if i != 2 - axis]
        gap[others[0]] = slice(int(a[0]), int(a[0]) + g)
        gap[others[1]] = slice(int(a[1]), int(a[1]) + g)
        w[tuple(gap)] = 0
    return w


def first_free_cell(walls, start):
    """First free cell at or after `start` (x,y,z) scanning x fastest."""
    n_z, n_y, n_x = walls.shape
    flat = walls.reshape(-1)
    i0 = (start[2] * n_y + start[1]) * n_x + start[0]
    free = np.flatnonzero(flat[i0:] == 0)
    i = i0 + int(free[0])
    return (i % n_x, (i // n_x) % n_y, i // (n_x * n_y))


def attached_box_spheres(size, offset=(0.0, 0.0, 0.0), radius=0.025):
    """Sphere centres for an attached box: one r=0.025 sphere per voxel at pitch 0.025/sqrt(2)
    (attached_bodies_collision_model.cpp:281-309)."""
    pitch = radius / math.sqrt(2.0)
    axes = []
    for a in range(3):
        n = max(1, int(math.ceil(size[a] / pitch)))
        start = offset[a] - 0.5 * (n - 1) * pitch
        axes.append(start + pitch * np.arange(n))
    xs, ys, zs = np.meshgrid(*axes, indexing="ij")
    return np.stack([xs.ravel(), ys.ravel(), zs.ravel()], axis=1)


PR2_DEMO_START = (-0.5, 0.3, 0.0, -1.0, 0.0, -0.5, 0.0)   # OUR fixture: a collision-free right-arm pose


def tabletop_queries(n, seed=13, dof=7):
    """Config 4 recipe on the PR2 tabletop scene: start fixed, goal positions uniform over a
    0.6 x 1.0 x 0.5 m box above the table (SURVEY.md section 8d)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lo = np.array([0.35, -0.6, 0.70])
    goals = lo + rng.random((n, 3)) * np.array([0.45, 0.9, 0.5])
    starts = np.tile(np.array(PR2_DEMO_START[:dof], np.float64), (n, 1))
    return np.ascontiguousarray(starts), np.ascontiguousarray(goals)


UBR1_DEMO_START = (0.0, 0.3, 0.0, -1.2, 0.0, 0.9, 0.0)    # OUR fixture: arm over the table, object in hand


def ubr1_tabletop_queries(n, seed=13):
    """Config 4: UBR1 arm + attached object, start fixed, goals uniform over a 0.6 x 1.0 x 0.5 m box above the
    table (SURVEY.md section 8d)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lo = np.array([0.45, -0.5, 0.65])
    goals = lo + rng.random((n, 3)) * np.array([0.6, 1.0, 0.5])
    starts = np.tile(np.array(UBR1_DEMO_START, np.float64), (n, 1))
    return np.ascontiguousarray(starts), np.ascontiguousarray(goals)


def lattice_walks(starts, params, k, seed, valid):
    """Joint states a planner can reach: walker i starts at starts[i] and takes k random motion-primitive steps
    (converses included) that valid(q0, q1) -> bool[n] accepts (joint limits and edge validity of the checker in use);
    a walker that finds no valid step in 8 tries stays where it is for that step.  Goals built from these states
    (their pose, or their joint values) are reachable by construction."""
    rng = np.random.Generator(np.random.PCG64(seed))
    prims = np.asarray(params.mprims, np.float64)
    deltas = np.stack([prims, -prims], axis=1).reshape(-1, prims.shape[1])
    q = np.array(starts, np.float64).reshape(-1, prims.shape[1])
    for _ in range(k):
        moved = np.zeros(len(q), bool)
        for _ in range(8):
            q1 = q + deltas[rng.integers(len(deltas), size=len(q))]
            ok = ~moved & np.asarray(valid(q, q1), bool)
            q[ok] = q1[ok]
            moved |= ok
    return np.ascontiguousarray(q)


def lattice_discretisation(lo, hi, cont, resolutions):
    """ManipLattice::init (manip_lattice.cpp:125-139): (coord_vals, coord_deltas, base) per planning variable."""
    vals, deltas, base = [], [], []
    for a, b, c, r in zip(lo, hi, cont, resolutions):
        if c:
            v = int(round((2.0 * math.pi) / r))
            vals.append(v)
            deltas.append((2.0 * math.pi) / float(v))
            base.append(None)
        else:
            span = abs(b - a)
            v = max(1, int(round(span / r)))
            vals.append(v)
            deltas.append(span / float(v))
            base.append(a)
    return np.array(vals, np.int32), np.array(deltas), base


def random_lattice_coords(n, lo, hi, cont, resolutions, seed):
    """n uniformly random lattice states as ManipLattice holds them (RobotCoord, 16-bit here) and their joint values
    by ManipLattice::coordToState (manip_lattice.cpp:1245-1261): coord * delta (+ min limit for bounded variables)."""
    vals, deltas, base = lattice_discretisation(lo, hi, cont, resolutions)
    rng = np.random.Generator(np.random.PCG64(seed))
    coords = np.empty((n, len(vals)), np.int16)
    q = np.empty((n, len(vals)), np.float64)
    for v in range(len(vals)):
        # bounded variables: 0 .. vals inclusive (both limits are lattice states); continuous: 0 .. vals - 1
        c = rng.integers(0, vals[v] + (0 if base[v] is None else 1), n)
        coords[:, v] = c
        prod = c.astype(np.float64) * deltas[v]
        q[:, v] = prod if base[v] is None else base[v] + prod
    return coords, q
