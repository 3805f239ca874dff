"""The batched planner on the 15-DOF PR2 (torso and both arms; smpl_b200.scenes.pr2_dual_arm_planning_scene): a
planning chain that moves only some of the planning variables (RobotTables.set_planning_chain(subset=True)).  The
device's planning-frame FK, both IKs and plans against the oracle's subset model (oracle_scene_init_kdl_subset,
tests/subset_chain_oracle.py), query for query; one context against several; the left-gripper chain, whose variables
are not a prefix (torso -> 0, left arm -> 8..14); and config 5 itself at 1 cm, device against device."""
import numpy as np
import pytest

import goal_set_oracle
import snap_kinds_oracle
import snap_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_sets import _assert_sets_same
from test_gpu_planner_limits import _stride_in_use
from test_gpu_snap_kinds import _Snaps
from test_oracle_dual_arm import (RIGHT, T_TORSO, dual_arm_oracle, dual_arm_starts, dual_arm_walks, off_chain_unchanged,
                                  oracle_valid, seven_dof_embedding, snap_steps)
from test_oracle_ik_snap import ik_problems

SNAPS = {"off": None,
         "rpy": _Snaps(enabled=False, rpy_dist_thresh=0.2),
         "xyz": _Snaps(enabled=False, xyz_dist_thresh=0.2),
         "xyz_rpy": _Snaps(dist_thresh=0.2),
         "all": _Snaps(dist_thresh=0.2, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2)}
LEFT, RIGHT_COLS = slice(8, 15), slice(1, 8)


@pytest.fixture(scope="module")
def dual2():
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    o = dual_arm_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


def _params(max_expansions):
    p = scenes.DualArmPlanParams()
    p.max_expansions = max_expansions
    return p


def _oracle(o, scene, params, starts, records, offsets, snap):
    out = []
    for i, s in enumerate(starts):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        g = records[offsets[i]:offsets[i + 1]]
        if snap is None:
            out.append(goal_set_oracle.plan_set(o, scene.T_kin_to_planning, s, g, params))
        else:
            out.append(snap_kinds_oracle.plan_set_snaps(o, scene.T_kin_to_planning, s, g, params, snap))
    return out


def _pose_sets(o, params, n, seed, rpy_tolerance, k=12):
    poses = o.planning_frame_fk(dual_arm_walks(oracle_valid(o), n, params, k, seed))
    recs = api.pose_goals(poses if rpy_tolerance is not None else poses[:, :3], params.xyz_tolerance,
                          rpy_tolerance=rpy_tolerance)
    return [recs[i:i + 1] for i in range(n)]


def _joint_sets(o, params, n, seed):
    q = dual_arm_walks(oracle_valid(o), n, params, 8, seed)
    recs = api.joint_goals(q, 0.5 * np.asarray(params.resolutions))
    return [recs[i:i + 1] for i in range(n)]


def _off_chain_snaps(got, off, cont):
    """snap steps of the device's paths; asserts each leaves the off-chain columns at the parent's values"""
    n = 0
    for g in got:
        parent, succ = snap_steps(g["path_states"])
        assert off_chain_unchanged(parent, succ, off, cont)
        n += len(parent)
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("res", [0.01, 0.02])
def test_start_is_collision_free(res):
    scene = scenes.pr2_dual_arm_planning_scene(res)
    ctx, tables = api.setup_context(scene)
    try:
        q = dual_arm_starts(1)
        assert ctx.is_states_valid(q)[0] == 1 and ctx.check_joint_limits(q)[0] == 1
    finally:
        ctx.close()


@pytest.mark.gpu
def test_device_fk_and_ik_match_oracle(dual2):
    scene, o, ctx, tables = dual2
    lo, hi, cont = tables.limits()
    q = scenes.random_states(2000, lo, hi, cont, seed=21)
    assert np.abs(ctx.planning_frame_fk(q) - o.planning_frame_fk(q)).max() < 1e-12
    poses, seeds = ik_problems(o, 2000, seed=23)
    c = cont.astype(bool)
    for kind in ("pose", "position"):
        if kind == "pose":
            q_ref, ok_ref, it_ref = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, seeds)
            q_dev, ok, it = ctx.planning_link_ik(poses, seeds)
        else:
            q_ref, ok_ref, it_ref = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning,
                                                                                poses[:, :3], seeds)
            q_dev, ok, it = ctx.planning_link_ik(poses[:, :3], seeds)
        d = q_dev - q_ref
        d[:, c] = np.angle(np.exp(1j * d[:, c]))
        print("%s IK: %d problems, %d converged, largest |q difference| %.3g" % (kind, len(q_dev), ok.sum(),
                                                                                np.abs(d).max()))
        assert np.array_equal(ok, ok_ref) and np.array_equal(it, it_ref), kind
        assert np.abs(d).max() <= 1e-9, kind
        assert ok.mean() >= 0.95, kind
        # the left arm, off the chain, keeps its seed (clamped to the limits, continuous joints wrapped)
        d = q_dev[:, LEFT] - np.clip(seeds[:, LEFT], lo[LEFT], hi[LEFT])
        cl = c[LEFT]
        assert (d[:, ~cl] == 0.0).all(), kind
        assert (np.abs(np.angle(np.exp(1j * (q_dev[:, LEFT][:, cl] - seeds[:, LEFT][:, cl])))) <= 1e-12).all(), kind


@pytest.mark.gpu
def test_seven_dof_chain_in_a_15_variable_model_is_the_strict_model_on_the_device():
    strict_scene = scenes.pr2_tabletop_scene()
    strict = make_oracle(strict_scene)
    ctx7, t7 = api.setup_context(strict_scene)
    scene = scenes.pr2_dual_arm_planning_scene(0.02)
    scene.chain_root = "torso_lift_link"
    scene.T_kin_to_planning = T_TORSO
    t15 = api.build_tables(scene)
    ctx15 = api.GpuContext(0)
    try:
        ctx15.set_robot(t15)
        lo, hi, cont = t15.limits()
        q7 = scenes.random_states(2000, *t7.limits(), seed=31)
        q15 = seven_dof_embedding(q7, lo, hi, cont, seed=32)
        assert np.array_equal(ctx15.planning_frame_fk(q15), ctx7.planning_frame_fk(q7))
        poses, seeds7 = ik_problems(strict, 1024, seed=33)
        seeds15 = seven_dof_embedding(seeds7, lo, hi, cont, seed=34)
        off = [0] + list(range(8, 15))
        for targets in (poses, poses[:, :3]):
            want = ctx7.planning_link_ik(targets, seeds7)
            got = ctx15.planning_link_ik(targets, seeds15)
            assert np.array_equal(got[0][:, RIGHT], want[0])
            assert np.array_equal(got[0][:, off], seeds15[:, off])
            assert np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2])
            assert want[1].mean() >= 0.95
    finally:
        ctx15.close()
        ctx7.close()
        t15.close()


@pytest.mark.gpu
@pytest.mark.parametrize("snap", list(SNAPS))
def test_pose_queries_match_oracle(dual2, snap):
    """12 XYZ and 12 XYZ_RPY queries; every snap kind alone and all three; snap steps leave the left arm alone"""
    scene, o, ctx, tables = dual2
    params = _params(1500)
    sets = _pose_sets(o, params, 12, seed=41, rpy_tolerance=None) + _pose_sets(o, params, 12, seed=43,
                                                                              rpy_tolerance=0.05)
    records, offsets = api.goal_sets(sets)
    starts = dual_arm_starts(len(sets))
    ref = _oracle(o, scene, params, starts, records, offsets, SNAPS[snap])
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=8, n_threads=2,
                                want_states=True, snap=SNAPS[snap])
    # the documented rounding allowance of the snap tests (tests/test_gpu_ik_snap.py _assert_same)
    _assert_sets_same(ref, got, max_differing=0 if snap == "off" else 1)
    assert sum(a["success"] for a in ref) >= 12 and sum(a["success"] for a in got) >= 12
    n_snaps = _off_chain_snaps(got, LEFT, tables.limits()[2])
    assert (n_snaps > 0) == (snap != "off")
    if snap == "all":
        assert _stride_in_use(stats, got) == 31   # 28 primitive words + 3 snap words


@pytest.mark.gpu
def test_joint_queries_match_oracle(dual2):
    """12 joint goals at half a resolution (all 15 variables), with all three snap kinds: the lattice alone rarely
    lands within half a resolution of 15 values in 1500 expansions"""
    snap = "all"
    scene, o, ctx, tables = dual2
    params = _params(1500)
    records, offsets = api.goal_sets(_joint_sets(o, params, 12, seed=51))
    starts = dual_arm_starts(12)
    ref = _oracle(o, scene, params, starts, records, offsets, SNAPS[snap])
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=6, n_threads=2,
                            want_states=True, snap=SNAPS[snap])
    _assert_sets_same(ref, got, max_differing=1)
    assert sum(a["success"] for a in ref) >= 10 and sum(a["success"] for a in got) >= 10
    for g, r in zip(got, records):
        if g["success"]:
            assert (np.abs(g["path_states"][-1] - r["angles"][:15]) <= 0.5 * np.asarray(params.resolutions)).all()


@pytest.mark.gpu
def test_mixed_goal_sets_on_one_and_three_contexts(dual2):
    """12 sets of an XYZ_RPY, a joint and an XYZ record, all three snap kinds: the oracle against one context, one
    context against three bit for bit"""
    scene, o, ctx, tables = dual2
    params = _params(1500)
    rpy = _pose_sets(o, params, 12, seed=61, rpy_tolerance=0.05)
    joint = _joint_sets(o, params, 12, seed=63)
    xyz = _pose_sets(o, params, 12, seed=65, rpy_tolerance=None)
    records, offsets = api.goal_sets([np.concatenate([rpy[i], joint[i], xyz[i]]) for i in range(12)])
    starts = dual_arm_starts(12)
    snap = SNAPS["all"]
    ref = _oracle(o, scene, params, starts, records, offsets, snap)
    one, stats = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=5, n_threads=2,
                                want_states=True, snap=snap)
    _assert_sets_same(ref, one, max_differing=1)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, mstats = api.plan_batch(ctxs, scene, tables, params, starts, (records, offsets), max_concurrent=3,
                                       want_states=True, snap=snap)
    finally:
        for c in ctxs[1:]:
            c.close()
    for a, b in zip(one, multi):   # device against device: bit for bit
        assert (a["success"], a["expansions"], a["cost"], a["reached_goal"]) == \
               (b["success"], b["expansions"], b["cost"], b["reached_goal"])
        assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])
    assert stats["ik_attempted"] == mstats["ik_attempted"] > 0
    assert sum(a["success"] for a in ref) >= 8 and sum(a["success"] for a in one) >= 8


@pytest.mark.gpu
def test_left_gripper_chain_matches_oracle():
    """the chain base_link -> l_gripper_palm_link: torso -> variable 0, left arm -> variables 8..14 (not a prefix);
    the right arm moves collision geometry only"""
    scene = scenes.pr2_dual_arm_planning_scene(0.02, planning_link="l_gripper_palm_link")
    o = dual_arm_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        lo, hi, cont = tables.limits()
        q = scenes.random_states(1000, lo, hi, cont, seed=71)
        assert np.abs(ctx.planning_frame_fk(q) - o.planning_frame_fk(q)).max() < 1e-12
        q2 = q.copy()
        q2[:, RIGHT_COLS] = q[::-1, RIGHT_COLS]
        assert np.array_equal(ctx.planning_frame_fk(q2), ctx.planning_frame_fk(q))   # the right arm moves nothing
        params = _params(1500)
        for snap in ("off", "all"):
            sets = _pose_sets(o, params, 6, seed=73, rpy_tolerance=0.05) + _pose_sets(o, params, 6, seed=75,
                                                                                      rpy_tolerance=None)
            records, offsets = api.goal_sets(sets)
            starts = dual_arm_starts(len(sets))
            ref = _oracle(o, scene, params, starts, records, offsets, SNAPS[snap])
            got, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=6,
                                    n_threads=2, want_states=True, snap=SNAPS[snap])
            _assert_sets_same(ref, got, max_differing=0 if snap == "off" else 1)
            assert sum(a["success"] for a in ref) >= 6 and sum(a["success"] for a in got) >= 6
            assert (_off_chain_snaps(got, RIGHT_COLS, cont) > 0) == (snap != "off")
    finally:
        ctx.close()


@pytest.mark.gpu
def test_config5_at_1cm_one_context_against_several():
    """BASELINE configuration 5 at its 1 cm resolution: 24 reachable XYZ_RPY queries with all three snap kinds, one
    context against three, bit for bit (device against device: a 1 cm oracle field would take about a gigabyte)"""
    scene = scenes.pr2_dual_arm_planning_scene(0.01)
    ctx, tables = api.setup_context(scene)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        params = _params(3000)
        valid = lambda q0, q1: ctx.check_joint_limits(q1).astype(bool) & ctx.is_edges_valid(q0, q1)[0].astype(bool)
        poses = ctx.planning_frame_fk(dual_arm_walks(valid, 24, params, 16, seed=81))
        goals = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)
        starts = dual_arm_starts(24)
        snap = api.SnapParams(dist_thresh=0.2, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2)
        one, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=12, want_states=True,
                                    snap=snap)
        multi, _ = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=4, want_states=True,
                                  snap=snap)
        for a, b in zip(one, multi):
            assert (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
                   (b["success"], b["expansions"], b["cost"], b["num_states"])
            assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])
        lo, hi, cont = tables.limits()
        for a, g in zip(one, goals):
            if a["success"]:
                p = a["path_states"]
                assert ctx.check_joint_limits(p).all() and ctx.is_edges_valid(p[:-1], p[1:])[0].all()
                assert (np.abs(ctx.planning_frame_fk(p[-1:])[0, :3] - g["pose"][:3]) <= 0.015).all()
        assert _off_chain_snaps(one, LEFT, cont) > 0
        print("config 5 at 1 cm: %d of 24 solved, %d expansions, %.3f s" % (
            sum(a["success"] for a in one), sum(a["expansions"] for a in one), stats["total_seconds"]))
        assert sum(a["success"] for a in one) >= 16
    finally:
        for c in ctxs[1:]:
            c.close()
        ctx.close()


@pytest.mark.gpu
def test_a_smaller_robot_in_the_same_process_leaves_the_15_dof_context_working(dual2):
    """the kernels' shared-memory caps belong to the process: creating a 7-DOF context after the 15-DOF one must not
    lower them below what the 15-DOF context launches with"""
    scene, o, ctx, tables = dual2
    lo, hi, cont = tables.limits()
    q = scenes.random_states(4096, lo, hi, cont, seed=91)
    q0, q1 = q[:-1], q[1:]
    want_s = ctx.is_states_valid(q)
    want_e = ctx.is_edges_valid(q0, q1)
    small, _ = api.setup_context(scenes.pr2_tabletop_scene())
    try:
        assert np.array_equal(ctx.is_states_valid(q), want_s)
        got_e = ctx.is_edges_valid(q0, q1)
        assert np.array_equal(got_e[0], want_e[0]) and np.array_equal(got_e[1], want_e[1])
        params = _params(200)
        records, offsets = api.goal_sets(_pose_sets(o, params, 2, seed=93, rpy_tolerance=None, k=4))
        got, _ = api.plan_batch(ctx, scene, tables, params, dual_arm_starts(2), (records, offsets), snap=SNAPS["all"])
        assert all(g["success"] for g in got)
    finally:
        small.close()
