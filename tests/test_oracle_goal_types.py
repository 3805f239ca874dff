"""GoalConstraint types in the oracle's planner (ManipLattice::isGoal, manip_lattice.cpp:1582-1696): XYZ_RPY_GOAL's
orientation test on constructed rotations, XYZ_RPY with a tolerance above pi equal to XYZ, and JOINT_STATE_GOAL and
pose goals on reachable lattice states.  The goal records are the ones smpl_b200.api hands to the device; the
goal-typed planner (oracle/goals) is pinned against the oracle's XYZ planner (oracle/lattice.cpp) on XYZ goals."""
import copy
import math

import numpy as np
import pytest

from helpers import make_oracle
import goal_oracle
from goal_oracle import rpy_goal_angles
from smpl_b200 import api, scenes


def _rot(axis, angle):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + math.sin(angle) * K + (1 - math.cos(angle)) * (K @ K)


def _rpy_matrix(r, p, y):
    return _rot((0, 0, 1), y) @ _rot((0, 1, 0), p) @ _rot((1, 0, 0), r)


def _matrix_rpy(M):
    """KDL Rotation::GetRPY (the planning_frame_fk convention)"""
    pitch = math.atan2(-M[2, 0], math.sqrt(M[0, 0] ** 2 + M[1, 0] ** 2))
    return math.atan2(M[2, 1], M[2, 2]), pitch, math.atan2(M[1, 0], M[0, 0])


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


def _plan(o, scene, params, start, goal):
    """goal: a position (the oracle's own XYZ planner, oracle/lattice.cpp) or a goal record (oracle/goals)"""
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
    if isinstance(goal, np.void):
        return goal_oracle.plan(o, start, goal, params)
    return o.plan(start, goal, params)


def _same(a, b):
    return (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
           (b["success"], b["expansions"], b["cost"], b["num_states"]) and np.array_equal(a["path_ids"], b["path_ids"])


def _short_only(params):
    p = copy.copy(params)
    p.mprims = params.mprims[params.short_flags == 1]
    return p


def _valid(o):
    return lambda q0, q1: o.check_joint_limits(q1).astype(bool) & o.is_edges_valid(q0, q1)[0].astype(bool)


def test_orientation_angle_of_constructed_rotations():
    rng = np.random.default_rng(4)
    rpy, goal_rpy, want = [], [], []
    for _ in range(300):
        g = rng.uniform(-1.4, 1.4, 3)                 # goal orientation, pitch away from the GetRPY singularity
        axis = rng.normal(size=3)
        angle = rng.uniform(0.05, 3.1)
        r = _matrix_rpy(_rpy_matrix(*g) @ _rot(axis, angle))
        rpy.append(r)
        goal_rpy.append(g)
        want.append(angle)
    theta, d = rpy_goal_angles(rpy, goal_rpy)
    assert np.abs(theta - np.array(want)).max() < 1e-12
    assert (d < 0).any() and (d > 0).any()            # both signs of q . qg occur
    # a goal yaw near +pi and a state yaw near -pi: q . qg < 0, the flip gives the short way round
    theta, d = rpy_goal_angles([[0.0, 0.0, -3.0]], [[0.0, 0.0, 3.0]])
    assert d[0] < 0 and abs(theta[0] - (2 * math.pi - 6.0)) < 1e-12
    # an identical orientation: angle 0 (or NaN when rounding puts |q . qg| above 1: then it is no goal at all)
    theta, _ = rpy_goal_angles([[0.3, -0.2, 1.1]], [[0.3, -0.2, 1.1]])
    assert theta[0] < 1e-7 or np.isnan(theta[0])


def test_rpy_tolerance_above_pi_plans_like_xyz(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 2000
    starts, goals = scenes.tabletop_queries(12, seed=19)
    rng = np.random.default_rng(8)
    poses = np.concatenate([goals, rng.uniform(-3.0, 3.0, (12, 3))], axis=1)
    rpy_goals = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=4.0)
    xyz_goals = api.pose_goals(goals, params.xyz_tolerance)
    n_ok = 0
    for i in range(12):
        ref = _plan(o, scene, params, starts[i], goals[i])
        by_record = _plan(o, scene, params, starts[i], xyz_goals[i])
        assert _same(ref, by_record) and np.array_equal(ref["path_states"], by_record["path_states"]), i
        assert _same(ref, _plan(o, scene, params, starts[i], rpy_goals[i])), i
        n_ok += ref["success"]
    assert n_ok >= 4


def test_joint_goal_on_a_reachable_lattice_state_is_solved(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 3000
    starts, _ = scenes.tabletop_queries(6)
    # steps of the short-distance primitives: the ones the planner applies within short_dist_thresh of the goal
    targets = scenes.lattice_walks(starts, _short_only(params), 8, seed=3, valid=_valid(o))
    tol = 0.5 * np.asarray(params.resolutions)
    goals = api.joint_goals(targets, tol)
    for i in range(6):
        r = _plan(o, scene, params, starts[i], goals[i])
        assert r["success"], i
        last = r["path_states"][-1]
        assert np.all(np.abs(last - targets[i]) <= tol), i


def test_joint_goal_with_huge_tolerances_ends_after_one_expansion(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    starts, _ = scenes.tabletop_queries(1)
    r = _plan(o, scene, params, starts[0], api.joint_goals(starts, np.full(scene.dof, 100.0))[0])
    assert r["success"] and r["expansions"] == 1 and list(r["path_ids"]) == [1, 0]


def test_pose_goals_with_orientation_tolerance_on_reachable_poses(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 3000
    starts, _ = scenes.tabletop_queries(8)
    targets = scenes.lattice_walks(starts, params, 20, seed=11, valid=_valid(o))
    goals = api.pose_goals(o.planning_frame_fk(targets), params.xyz_tolerance, rpy_tolerance=0.05)
    solved = 0
    for i in range(8):
        r = _plan(o, scene, params, starts[i], goals[i])
        if r["success"]:
            solved += 1
            pose = o.planning_frame_fk(r["path_states"][-1:])[0]
            assert np.all(np.abs(pose[:3] - goals[i]["pose"][:3]) <= params.xyz_tolerance)
            theta, _ = rpy_goal_angles(pose[None, 3:], goals[i]["pose"][None, 3:])
            assert theta[0] < 0.05
    assert solved >= 4
