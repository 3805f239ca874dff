"""Planning chains over a subset of the planning variables (RobotTables.set_planning_chain(subset=True),
the oracle's oracle_scene_init_kdl_subset) on the CPU: the refusals of both modes, the 7-DOF chain inside a 15-variable
model against the strict 7-DOF model, the limits, and the oracle planners on the 15-DOF PR2 planning scene
(smpl_b200.scenes.pr2_dual_arm_planning_scene)."""
import numpy as np
import pytest

import goal_set_oracle
import snap_kinds_oracle
import snap_oracle
import subset_chain_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes
from test_oracle_ik_snap import ik_problems

DUAL = ["torso_lift_joint"] + scenes.PR2_RIGHT_ARM_JOINTS + scenes.PR2_LEFT_ARM_JOINTS
RIGHT = slice(1, 8)      # the right arm's columns in DUAL
T_TORSO = np.array([[1.0, 0.0, 0.0, -0.05], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.959]])


def dual_arm_oracle(scene):
    o = make_oracle(scene, with_kdl=False)
    subset_chain_oracle.init_kdl_subset(o, scene.chain_root, scene.chain_tip, scene.planning_link,
                                        scene.T_kin_to_planning, scene.xyz_offset)
    return o


def dual_arm_starts(n):
    return np.ascontiguousarray(np.tile(np.array(scenes.DUAL_ARM_START, np.float64), (n, 1)))


def dual_arm_walks(valid, n, params, k, seed):
    """n lattice states k random primitive steps from DUAL_ARM_START (scenes.lattice_walks)"""
    return scenes.lattice_walks(dual_arm_starts(n), params, k, seed=seed, valid=valid)


def oracle_valid(o):
    return lambda q0, q1: o.check_joint_limits(q1).astype(bool) & o.is_edges_valid(q0, q1)[0].astype(bool)


def snap_steps(path_states):
    """(parent, successor) row pairs of a path whose step moves more than one variable: every primitive moves one, so
    these are snap actions"""
    d = np.diff(path_states, axis=0)
    k = np.flatnonzero((d != 0.0).sum(axis=1) > 1)
    return path_states[k], path_states[k + 1]


def off_chain_unchanged(parent, succ, off, cont):
    """the off-chain columns `off` of snap successors equal the parent's; continuous ones modulo 2 pi (the IK wraps
    them into [-pi, pi])"""
    d = succ[:, off] - parent[:, off]
    c = cont[off].astype(bool)
    d[:, c] = np.angle(np.exp(1j * d[:, c]))
    return bool((np.abs(d[:, c]) <= 1e-12).all() and (d[:, ~c] == 0.0).all())


@pytest.fixture(scope="module")
def scene2():
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    return scene, dual_arm_oracle(scene)


def _tables(scene, joints):
    t = api.RobotTables(scene.robot_path)
    t.configure(scene.group, joints)
    return t


def test_strict_mode_still_refuses_the_15_variable_model():
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    o = make_oracle(scene, with_kdl=False)
    with pytest.raises(RuntimeError, match="planning joints do not match the movable joints of the chain"):
        o.init_kdl(scene.chain_root, scene.chain_tip, scene.planning_link, scene.T_kin_to_planning)
    t = _tables(scene, DUAL)
    with pytest.raises(api.SmplGpuError, match="a planning joint is not part of the kinematic chain"):
        t.set_planning_chain(scene.chain_root, scene.chain_tip, scene.planning_link, scene.T_kin_to_planning)
    t.close()


@pytest.mark.parametrize("case", ["torso_not_planned", "planning_link_off_chain"])
def test_subset_mode_refusals(case):
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    if case == "torso_not_planned":     # the chain from base_link moves the torso joint, which is not planned
        scene.planning_joints = list(scenes.PR2_RIGHT_ARM_JOINTS)
        args = ("base_link", "r_gripper_palm_link", "r_gripper_palm_link")
        text = "chain joint 'torso_lift_joint' is not a planning variable"
    else:
        args = ("base_link", "r_gripper_palm_link", "l_gripper_palm_link")
        text = "planning link"
    o = make_oracle(scene, with_kdl=False)
    with pytest.raises(RuntimeError, match=text):
        subset_chain_oracle.init_kdl_subset(o, *args, scene.T_kin_to_planning)
    t = _tables(scene, scene.planning_joints)
    with pytest.raises(api.SmplGpuError, match=text):
        t.set_planning_chain(*args, scene.T_kin_to_planning, subset=True)
    t.close()


def seven_dof_pair():
    """the strict 7-DOF right-arm model (the tabletop scene's chain) and a 15-variable subset model with the same
    chain (root torso_lift_link, planning frame base_footprint at the 7-DOF scenes' torso height)"""
    strict = make_oracle(scenes.pr2_tabletop_scene())
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    scene.chain_root = "torso_lift_link"
    scene.T_kin_to_planning = T_TORSO
    return strict, scene, dual_arm_oracle(scene)


def seven_dof_embedding(q7, lo, hi, cont, seed):
    """15-variable states whose right-arm columns are q7 and whose other columns are random within their limits"""
    q = scenes.random_states(len(q7), lo, hi, cont, seed)
    q[:, RIGHT] = q7
    return np.ascontiguousarray(q)


def test_seven_dof_chain_in_a_15_variable_model_is_the_strict_model_bit_for_bit():
    strict, scene, o = seven_dof_pair()
    lo, hi, cont = o.joint_limits()
    poses, seeds7 = ik_problems(strict, 512, seed=5)
    q7 = scenes.random_states(2000, *strict.joint_limits(), seed=3)
    q15 = seven_dof_embedding(q7, lo, hi, cont, seed=4)
    assert np.array_equal(o.planning_frame_fk(q15), strict.planning_frame_fk(q7))
    q15[:, [0] + list(range(8, 15))] = 1e3     # the other columns, whatever they hold, move nothing
    assert np.array_equal(o.planning_frame_fk(q15), strict.planning_frame_fk(q7))
    seeds15 = seven_dof_embedding(seeds7, lo, hi, cont, seed=6)
    off = [0] + list(range(8, 15))
    for kind in ("pose", "position"):
        if kind == "pose":
            want = snap_oracle.planning_link_ik(strict, T_TORSO, poses, seeds7)
            got = snap_oracle.planning_link_ik(o, T_TORSO, poses, seeds15)
        else:
            want = snap_kinds_oracle.planning_link_ik_position(strict, T_TORSO, poses[:, :3], seeds7)
            got = snap_kinds_oracle.planning_link_ik_position(o, T_TORSO, poses[:, :3], seeds15)
        assert np.array_equal(got[0][:, RIGHT], want[0]), kind
        assert np.array_equal(got[0][:, off], seeds15[:, off]), kind
        assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]), kind
        assert want[1].mean() >= 0.95, kind


def test_exact_chain_order_gives_the_strict_tables():
    """planning variables that are exactly the chain's joints in chain order: subset mode builds what strict mode
    builds (compared through the limits and the planning-frame FK of the oracle built from each mode)"""
    scene = scenes.pr2_tabletop_scene()
    strict = make_oracle(scene)
    o = make_oracle(scene, with_kdl=False)
    subset_chain_oracle.init_kdl_subset(o, scene.chain_root, scene.chain_tip, scene.planning_link,
                                        scene.T_kin_to_planning)
    q = scenes.random_states(500, *strict.joint_limits(), seed=8)
    assert np.array_equal(o.planning_frame_fk(q), strict.planning_frame_fk(q))
    for a, b in zip(o.joint_limits(), strict.joint_limits()):
        assert np.array_equal(a, b)
    t = api.build_tables(scene)
    scene.chain_subset = True
    t2 = api.build_tables(scene)
    for a, b in zip(t.limits(), t2.limits()):
        assert np.array_equal(a, b)
    t.close()
    t2.close()


def test_limits_of_all_15_variables_match_the_tables(scene2):
    scene, o = scene2
    t = api.build_tables(scene)
    assert t.dof == 15
    lo, hi, cont = t.limits()
    olo, ohi, ocont = o.joint_limits()
    assert np.array_equal(lo, olo) and np.array_equal(hi, ohi) and np.array_equal(cont, ocont)
    assert cont.tolist() == [0, 0, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 1, 0, 1]
    t.close()


def test_start_is_collision_free_at_2cm(scene2):
    scene, o = scene2
    q = dual_arm_starts(1)
    assert o.is_states_valid(q)[0] == 1 and o.check_joint_limits(q)[0] == 1


def test_oracle_planners_solve_reachable_queries(scene2):
    """8 XYZ_RPY queries at the poses of lattice states 12 primitive steps from the start: the goal-set planner
    without snaps and the snap-kinds planner with all three kinds each solve at least half; snap actions leave the
    left arm where it was"""
    scene, o = scene2
    params = scenes.DualArmPlanParams()
    params.max_expansions = 2500
    goals = api.pose_goals(o.planning_frame_fk(dual_arm_walks(oracle_valid(o), 8, params, 12, seed=9)),
                           params.xyz_tolerance, rpy_tolerance=0.05)
    starts = dual_arm_starts(8)
    snap = api.SnapParams(dist_thresh=0.2, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2)
    _, _, cont = o.joint_limits()
    for s in (None, snap):
        solved = snaps = 0
        for i in range(8):
            o.heur_init(scene.inflation_radius, scene.cost_per_cell)
            if s is None:
                r = goal_set_oracle.plan_set(o, scene.T_kin_to_planning, starts[i], goals[i:i + 1], params)
            else:
                r = snap_kinds_oracle.plan_set_snaps(o, scene.T_kin_to_planning, starts[i], goals[i:i + 1], params, s)
            if not r["success"]:
                continue
            solved += 1
            p = r["path_states"]
            assert np.array_equal(p[0], starts[i]) and o.check_joint_limits(p).all()
            end = o.planning_frame_fk(p[-1:])[0]
            assert (np.abs(end[:3] - goals[i]["pose"][:3]) <= 0.015).all()
            parent, succ = snap_steps(p)
            snaps += len(parent)
            assert off_chain_unchanged(parent, succ, slice(8, 15), cont)
        assert solved >= 4, s
        assert (snaps > 0) == (s is not None)
