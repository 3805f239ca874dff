"""The snap kinds SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY in the oracle (oracle/snap_kinds/snap_kinds_lattice.cpp:
planningLinkIkPosition, oracle_plan_goal_set_snaps).  The position-only IK must converge on reachable positions and
give up after max_iterations on unreachable ones; SNAP_TO_XYZ_RPY alone must plan as the goal-set planner; SNAP_TO_XYZ
must land XYZ goals, SNAP_TO_RPY must turn in place, and kinds that never act must change nothing."""
import numpy as np
import pytest

from helpers import make_oracle
import goal_set_oracle
import snap_kinds_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_types import _joint_queries, _params, _pose_queries
from test_oracle_ik_snap import _valid_states, ik_problems


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


def _snaps(o, scene, params, start, goals, snap):
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
    return snap_kinds_oracle.plan_set_snaps(o, scene.T_kin_to_planning, start, goals, params, snap)


def _set(o, scene, params, start, goals, snap):
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)
    return goal_set_oracle.plan_set(o, scene.T_kin_to_planning, start, goals, params, snap)


def _assert_same(a, b):
    assert (a["success"], a["expansions"], a["cost"], a["num_states"], a["reached_goal"]) == \
           (b["success"], b["expansions"], b["cost"], b["num_states"], b["reached_goal"])
    assert np.array_equal(a["path_ids"], b["path_ids"])
    assert np.array_equal(a["path_states"], b["path_states"])


def test_position_ik_converges_on_reachable_positions(tabletop):
    scene, o = tabletop
    poses, seeds = ik_problems(o, 2000, seed=7)   # the full-pose IK's protocol (tests/test_oracle_ik_snap.py)
    q, ok, it = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning, poses[:, :3], seeds)
    print("position-only IK: converged %.4f, mean iterations %.2f" % (ok.mean(), it[ok].mean()))
    assert ok.mean() >= 0.99
    assert (it[ok] <= 100).all() and (it[~ok] == 100).all()
    got = o.planning_frame_fk(q[ok])
    assert np.abs(got[:, :3] - poses[ok, :3]).max() <= 1e-6   # every position row within the tolerance
    lo, hi, cont = o.joint_limits()
    bounded = ~cont.astype(bool)
    assert (q[:, bounded] >= lo[bounded]).all() and (q[:, bounded] <= hi[bounded]).all()
    # the orientation is free: with the position alone the answers do not keep the orientation of the targets
    assert np.abs(got[:, 3:] - poses[ok, 3:]).max() > 1e-3


def test_position_ik_of_an_unreachable_position_fails_after_max_iterations(tabletop):
    scene, o = tabletop
    poses, seeds = ik_problems(o, 32, seed=9)
    xyz = poses[:, :3] + np.array([5.0, 0.0, 0.0])
    _, ok, it = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning, xyz, seeds)
    assert not ok.any() and (it == 100).all()
    _, ok, it = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning, xyz, seeds, max_iterations=7)
    assert not ok.any() and (it == 7).all()


def _xyz_rpy_fixtures(scene, o, params):
    s_pose, g_pose = _pose_queries(scene, o, params, 4, seed=11)
    s_joint, g_joint = _joint_queries(scene, o, params, 3, seed=23)
    base, xyz = scenes.tabletop_queries(3, seed=25)
    starts = np.concatenate([s_pose, s_joint, base])
    goals = np.concatenate([g_pose, g_joint, api.pose_goals(xyz, params.xyz_tolerance)])
    return starts, goals


@pytest.mark.parametrize("thresh", [0.0, 0.2])
def test_xyz_rpy_alone_is_the_goal_set_planner(tabletop, thresh):
    scene, o = tabletop
    params = _params(scene, 1000)
    starts, goals = _xyz_rpy_fixtures(scene, o, params)
    snap = api.SnapParams(dist_thresh=thresh)
    n = len(starts)
    sets = [goals[i:i + 1] for i in range(n)] + [goals[[i, (i + 3) % n, (i + 5) % n]] for i in range(n)]
    solved = 0
    for s, g in zip(np.concatenate([starts, starts]), sets):
        a = _set(o, scene, params, s, g, snap)
        b = _snaps(o, scene, params, s, g, snap)
        _assert_same(a, b)
        assert (a["ik_attempted"], a["ik_converged"]) == (b["ik_attempted"], b["ik_converged"])
        assert b["ik_by_kind"][:2].sum() == 0
        solved += b["success"]
    assert solved >= 6


def _tight_xyz_queries(o, n, seed, tol=2e-4):
    """XYZ goals at the target-offset positions of valid states, with a box so small that the primitives almost never
    land in it"""
    q = _valid_states(o, n, seed)
    starts = scenes.tabletop_queries(n, seed=seed + 1)[0]
    return starts, api.pose_goals(o.planning_frame_fk(q)[:, :3], (tol, tol, tol))


def test_snapped_xyz_goals_end_inside_the_goal_box(tabletop):
    scene, o = tabletop
    params = _params(scene, 1000)
    starts, goals = _tight_xyz_queries(o, 8, seed=31)
    xyz = api.SnapParams(enabled=False, xyz_dist_thresh=0.2)
    solved_off = solved = 0
    for s, g in zip(starts, goals):
        off = _snaps(o, scene, params, s, g[None], None)
        r = _snaps(o, scene, params, s, g[None], xyz)
        solved_off += off["success"]
        solved += r["success"]
        assert r["ik_by_kind"][[0, 2]].sum() == 0
        if r["success"]:
            last = o.planning_frame_fk(r["path_states"][-1:])[0]
            assert (np.abs(last[:3] - g["pose"][:3]) <= g["xyz_tolerance"]).all()
    print("tight XYZ goals solved: %d with SNAP_TO_XYZ, %d without" % (solved, solved_off))
    assert solved >= 4 and solved > solved_off


def test_rpy_snaps_turn_in_place(tabletop):
    """XYZ_RPY goals with an orientation tolerance the primitives almost never meet: the solved paths end with the
    SNAP_TO_RPY action, whose answer keeps the parent's target-offset position to the IK tolerance"""
    scene, o = tabletop
    params = _params(scene, 1000)
    q = _valid_states(o, 8, seed=41)
    starts = scenes.tabletop_queries(8, seed=42)[0]
    goals = api.pose_goals(o.planning_frame_fk(q), (0.015, 0.015, 0.015), rpy_tolerance=1e-3)
    rpy = api.SnapParams(enabled=False, rpy_dist_thresh=0.2)
    solved = 0
    for s, g in zip(starts, goals):
        r = _snaps(o, scene, params, s, g[None], rpy)
        assert r["ik_by_kind"][1:].sum() == 0
        if not r["success"]:
            continue
        solved += 1
        pos = o.planning_frame_fk(r["path_states"][-2:])[:, :3]
        assert np.abs(pos[1] - pos[0]).max() <= 1e-6
    print("XYZ_RPY goals (1e-3 rad) solved with SNAP_TO_RPY: %d of %d" % (solved, len(goals)))
    assert solved >= 3


def test_xyz_and_rpy_kinds_leave_joint_records_alone(tabletop):
    scene, o = tabletop
    params = _params(scene, 1000)
    starts, goals = _joint_queries(scene, o, params, 6, seed=5)
    kinds = api.SnapParams(enabled=False, xyz_dist_thresh=0.5, rpy_dist_thresh=0.5)
    solved = 0
    for s, g in zip(starts, goals):
        a = _snaps(o, scene, params, s, g[None], None)
        b = _snaps(o, scene, params, s, g[None], kinds)
        _assert_same(a, b)
        assert b["ik_attempted"] == 0
        solved += a["success"]
    assert solved >= 3


def test_a_kind_whose_threshold_no_expansion_meets_changes_nothing(tabletop):
    """a tiny budget from starts far from the goal: no expanded state is within 1 mm, so the kind runs no IK"""
    scene, o = tabletop
    params = _params(scene, 40)
    starts, goals = _pose_queries(scene, o, params, 6, seed=13)
    for kinds in (api.SnapParams(enabled=False, xyz_dist_thresh=0.001),
                  api.SnapParams(enabled=False, rpy_dist_thresh=0.001),
                  api.SnapParams(dist_thresh=0.001)):
        for s, g in zip(starts, goals):
            a = _snaps(o, scene, params, s, g[None], None)
            b = _snaps(o, scene, params, s, g[None], kinds)
            _assert_same(a, b)
            assert b["ik_by_kind"].sum() == 0
