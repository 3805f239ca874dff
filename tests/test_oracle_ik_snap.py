"""The snap-to-goal action (SNAP_TO_XYZ_RPY, manip_lattice_action_space.cpp:376-449, 507-573, 662-691) and its
planning-link IK in the oracle (oracle/snap/snap_lattice.cpp: planningLinkIk, oracle_plan_goal_snap).  The IK is the
project's own (the reference's solvers are third-party): it must converge on reachable targets, stay within the joint
limits and give up after max_iterations on unreachable ones.  With snaps off the snap planner must be the goal-typed
planner; with snaps on, joint goals end at the goal's angles and pose goals are solved more often."""
import numpy as np
import pytest

from helpers import make_oracle
import snap_oracle
from goal_oracle import rpy_goal_angles
from smpl_b200 import api, scenes

from test_oracle_goal_types import _plan, _short_only, _valid


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


def _valid_states(o, n, seed):
    lo, hi, cont = o.joint_limits()
    lo = np.where(cont, -np.pi, lo)
    hi = np.where(cont, np.pi, hi)
    q = np.random.default_rng(seed).uniform(lo, hi, (6 * n, len(lo)))
    return q[o.is_states_valid(q).astype(bool)][:n]


def ik_problems(o, n, seed):
    """IK targets: the target-offset poses of random valid states; seeds: those states moved by up to 0.1 rad (or
    metre) per joint"""
    q = _valid_states(o, n, seed)
    assert len(q) == n
    seeds = q + np.random.default_rng(seed + 1).uniform(-0.1, 0.1, q.shape)
    return o.planning_frame_fk(q), seeds


def _residual(o, q, poses):
    """max over position (metres) and orientation angle (radians) of the distance between FK(q) and poses"""
    got = o.planning_frame_fk(q)
    pos = np.abs(got[:, :3] - poses[:, :3]).max(axis=1)
    ang, _ = rpy_goal_angles(got[:, 3:], poses[:, 3:])
    return np.maximum(pos, np.nan_to_num(ang, nan=0.0))


def test_ik_converges_on_reachable_targets(tabletop):
    scene, o = tabletop
    poses, seeds = ik_problems(o, 2000, seed=7)
    q, ok, it = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, seeds)
    print("converged %.4f, mean iterations %.2f" % (ok.mean(), it[ok].mean()))
    assert ok.mean() >= 0.99
    assert (it[ok] <= 100).all() and (it[~ok] == 100).all()
    # residual: each error component is <= 1e-6, so the rotation angle is <= sqrt(3) 1e-6
    assert _residual(o, q[ok], poses[ok]).max() <= 2e-6
    # within the limits (KDLRobotModel::checkJointLimits itself may still refuse a value clamped to an upper limit: its
    # wrap into [min, min + 2 pi) rounds; the snap action checks it like any action)
    lo, hi, cont = o.joint_limits()
    bounded = ~cont.astype(bool)
    assert ((q[:, bounded] >= lo[bounded]) & (q[:, bounded] <= hi[bounded])).all()
    assert (np.abs(q[:, ~bounded]) <= np.pi).all()


def test_ik_at_the_target_takes_no_step_and_tolerance_bounds_the_work(tabletop):
    scene, o = tabletop
    q0 = _valid_states(o, 8, seed=9)
    poses = o.planning_frame_fk(q0)
    q, ok, it = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, q0)
    assert ok.all() and (it == 0).all() and np.array_equal(q, q0)
    _, seeds = ik_problems(o, 64, seed=13)
    poses, _ = ik_problems(o, 64, seed=13)
    _, ok_a, it_a = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, seeds, tolerance=1e-3)
    _, ok_b, it_b = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, seeds, tolerance=1e-9)
    both = ok_a & ok_b
    assert both.sum() >= 60 and (it_a[both] <= it_b[both]).all() and (it_a[both] < it_b[both]).any()


def test_ik_of_an_unreachable_target_fails_after_max_iterations(tabletop):
    scene, o = tabletop
    q0 = _valid_states(o, 4, seed=15)
    poses = o.planning_frame_fk(q0)
    poses[:, 0] += 5.0   # 5 m away: outside the grid and the arm's reach
    for max_it in (1, 37, 100):
        _, ok, it = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, q0, max_iterations=max_it)
        assert not ok.any() and (it == max_it).all()


# ---- the snap planner ----

def _plan_snap(o, scene, params, start, goal, snap):
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
    return snap_oracle.plan_snap(o, scene.T_kin_to_planning, start, goal, params, snap)


def _same(a, b):
    return (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
           (b["success"], b["expansions"], b["cost"], b["num_states"]) and \
        np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])


def _query_sets(o, scene):
    """the XYZ, XYZ_RPY and JOINT_STATE query sets of test_oracle_goal_types.py"""
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 2000
    starts, goals = scenes.tabletop_queries(12, seed=19)
    rng = np.random.default_rng(8)
    poses = np.concatenate([goals, rng.uniform(-3.0, 3.0, (12, 3))], axis=1)
    out = [(params, starts, api.pose_goals(goals, params.xyz_tolerance)),
           (params, starts, api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=4.0))]
    p3 = scenes.PlanParams(scene.dof)
    p3.max_expansions = 3000
    s3, _ = scenes.tabletop_queries(8)
    targets = scenes.lattice_walks(s3, p3, 20, seed=11, valid=_valid(o))
    out.append((p3, s3, api.pose_goals(o.planning_frame_fk(targets), p3.xyz_tolerance, rpy_tolerance=0.05)))
    s4, _ = scenes.tabletop_queries(6)
    targets = scenes.lattice_walks(s4, _short_only(p3), 8, seed=3, valid=_valid(o))
    out.append((p3, s4, api.joint_goals(targets, 0.5 * np.asarray(p3.resolutions))))
    return out


def test_snaps_off_plans_as_the_goal_planner(tabletop):
    scene, o = tabletop
    off = api.SnapParams(enabled=False, dist_thresh=0.2)
    for params, starts, goals in _query_sets(o, scene):
        for i in range(len(starts)):
            ref = _plan(o, scene, params, starts[i], goals[i])
            got = _plan_snap(o, scene, params, starts[i], goals[i], off)
            assert _same(ref, got), i
            assert got["ik_attempted"] == 0


def test_snapped_joint_goal_paths_end_at_the_goal_angles(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 2000
    starts, _ = scenes.tabletop_queries(10, seed=5)
    targets = scenes.lattice_walks(starts, params, 12, seed=17, valid=_valid(o))
    targets += np.random.default_rng(3).uniform(-0.02, 0.02, targets.shape)   # off the lattice
    goals = api.joint_goals(targets, 0.005)
    n_off = n_on = 0
    for i in range(len(starts)):
        off = _plan(o, scene, params, starts[i], goals[i])
        on = _plan_snap(o, scene, params, starts[i], goals[i], api.SnapParams(dist_thresh=0.2))
        n_off += off["success"]
        n_on += on["success"]
        assert on["ik_attempted"] == 0
        if on["success"]:
            assert np.array_equal(on["path_states"][-1], targets[i]), i
    print("joint goals solved: %d without snaps, %d with" % (n_off, n_on))
    assert n_on > n_off


def test_snapped_pose_goals_are_goals_and_solve_more(tabletop):
    scene, o = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 2000
    n = 12
    starts, _ = scenes.tabletop_queries(n, seed=29)
    poses = o.planning_frame_fk(_valid_states(o, n, seed=31))   # reachable pose goals
    goals = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)
    n_off = n_on = attempted = 0
    for i in range(n):
        off = _plan(o, scene, params, starts[i], goals[i])
        on = _plan_snap(o, scene, params, starts[i], goals[i], api.SnapParams(dist_thresh=0.2))
        n_off += off["success"]
        n_on += on["success"]
        attempted += on["ik_attempted"]
        if on["success"]:
            last = o.planning_frame_fk(on["path_states"][-1:])[0]
            assert np.all(np.abs(last[:3] - poses[i, :3]) <= params.xyz_tolerance), i
            theta, d = rpy_goal_angles(last[None, 3:], poses[i, None, 3:])
            # an orientation equal to the goal's up to rounding can give q . qg > 1 and a NaN angle, which isGoal's
            # unclamped acos takes for no goal; such a state still ends a path when a primitive reaches its cell
            assert theta[0] < 0.05 or (np.isnan(theta[0]) and abs(d[0]) > 1.0), i
    print("pose goals solved: %d without snaps, %d with (%d IK solves)" % (n_off, n_on, attempted))
    assert n_on > n_off and attempted > 0
