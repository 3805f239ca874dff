"""GoalConstraint types in the batched planner (smplhost_plan_batch_goals): pose goals with an orientation tolerance
and joint-configuration goals must give, query by query, the oracle's success, expansions, cost, lattice size, id
path and path states (ManipLattice::isGoal, manip_lattice.cpp:1582-1696; the device's goal test is
csrc/lattice.cuh:lattice_is_goal)."""
import copy
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
import goal_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes


def test_goal_record_layout_matches_the_header():
    """api.GoalC / GOAL_DTYPE against sizeof / offsetof of smplgpu_goal as a C compiler lays it out"""
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "smplgpu.h"
int main(void)
{
    printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(smplgpu_goal), offsetof(smplgpu_goal, type),
           offsetof(smplgpu_goal, pose), offsetof(smplgpu_goal, xyz_tolerance), offsetof(smplgpu_goal, rpy_tolerance),
           offsetof(smplgpu_goal, angles), offsetof(smplgpu_goal, angle_tolerances));
    return 0;
}
'''
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "layout.c"), "w") as f:
            f.write(src)
        exe = os.path.join(d, "layout")
        subprocess.run(["/usr/bin/g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), os.path.join(d, "layout.c"),
                        "-o", exe], check=True)
        got = list(map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()))
    names = ["type", "pose", "xyz_tolerance", "rpy_tolerance", "angles", "angle_tolerances"]
    assert got == [C.sizeof(api.GoalC)] + [getattr(api.GoalC, n).offset for n in names]
    assert api.GOAL_DTYPE.itemsize == C.sizeof(api.GoalC)


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


def _params(scene, max_expansions):
    p = scenes.PlanParams(scene.dof)
    p.max_expansions = max_expansions
    return p


def _short_only(params):
    p = copy.copy(params)
    p.mprims = params.mprims[params.short_flags == 1]
    return p


def _walks(o, starts, params, k, seed):
    valid = lambda q0, q1: o.check_joint_limits(q1).astype(bool) & o.is_edges_valid(q0, q1)[0].astype(bool)
    return scenes.lattice_walks(starts, params, k, seed=seed, valid=valid)


def _oracle(o, scene, params, starts, goals):
    out = []
    for s, g in zip(starts, goals):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        out.append(goal_oracle.plan(o, s, g, params))
    return out


def _assert_same(ref, got, states=True):
    for i, (a, b) in enumerate(zip(ref, got)):
        assert (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"]), (i, a["expansions"], b["expansions"])
        assert np.array_equal(a["path_ids"], b["path_ids"]), i
        if states:
            assert np.array_equal(a["path_states"], b["path_states"]), i


def _pose_queries(scene, o, params, n, seed):
    """n tabletop pose goals at 0.015 m / 0.05 rad: the demo goal (pr2_goal.yaml:38-44, call_planner.cpp:93-96), one
    outside the grid, the rest the poses of lattice states reached by random primitive steps"""
    starts, _ = scenes.tabletop_queries(n)
    poses = o.planning_frame_fk(_walks(o, starts, params, 20, seed))
    poses[0] = (0.4, -0.2, 0.36, 0.0, 0.0, 0.0)
    poses[1, :3] = (5.0, 0.0, 1.0)
    return starts, api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)


def _joint_queries(scene, o, params, n, seed):
    """n joint goals at half a lattice resolution: two thirds reached by short-distance primitive steps (the ones
    active near the goal), the rest by any primitives"""
    starts, _ = scenes.tabletop_queries(n)
    m = 2 * n // 3
    targets = np.concatenate([_walks(o, starts[:m], _short_only(params), 8, seed),
                              _walks(o, starts[m:], params, 8, seed + 1)])
    return starts, api.joint_goals(targets, 0.5 * np.asarray(params.resolutions))


@pytest.mark.gpu
def test_pose_goals_match_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 2500)
    starts, goals = _pose_queries(scene, o, params, 24, seed=11)
    ref = _oracle(o, scene, params, starts, goals)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=10, n_threads=3, want_states=True)
    _assert_same(ref, got)
    assert sum(a["success"] for a in ref) >= 8 and not ref[1]["success"]
    assert stats["rounds"] > 0


@pytest.mark.gpu
def test_joint_goals_match_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 2500)
    starts, goals = _joint_queries(scene, o, params, 24, seed=3)
    ref = _oracle(o, scene, params, starts, goals)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=10, n_threads=3, want_states=True)
    _assert_same(ref, got)
    assert sum(a["success"] for a in ref) >= 12


@pytest.mark.gpu
def test_mixed_goal_types_in_one_call_equal_single_type_calls(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    s_pose, g_pose = _pose_queries(scene, o, params, 8, seed=21)
    s_joint, g_joint = _joint_queries(scene, o, params, 8, seed=23)
    s_xyz, xyz = scenes.tabletop_queries(8, seed=25)
    g_xyz = api.pose_goals(xyz, params.xyz_tolerance)
    singles = [api.plan_batch(ctx, scene, tables, params, s, g, max_concurrent=5, want_states=True)[0]
               for s, g in ((s_pose, g_pose), (s_joint, g_joint), (s_xyz, g_xyz))]
    order = np.arange(24).reshape(3, 8).T.reshape(-1)   # pose, joint, xyz, pose, ...
    starts = np.concatenate([s_pose, s_joint, s_xyz])[order]
    goals = np.concatenate([g_pose, g_joint, g_xyz])[order]
    mixed, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=7, n_threads=2, want_states=True)
    _assert_same([sum(singles, [])[k] for k in order], mixed)


@pytest.mark.gpu
def test_rpy_tolerance_above_pi_equals_xyz_bit_for_bit(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 2000)
    starts, xyz = scenes.tabletop_queries(16, seed=27)
    rpy = np.random.default_rng(9).uniform(-3.0, 3.0, (16, 3))
    goals = api.pose_goals(np.concatenate([xyz, rpy], axis=1), params.xyz_tolerance, rpy_tolerance=4.0)
    want, _ = api.plan_batch(ctx, scene, tables, params, starts, xyz, max_concurrent=6, want_states=True)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, want_states=True)
    _assert_same(want, got)
    assert sum(a["success"] for a in want) >= 4


@pytest.mark.gpu
def test_one_planner_thread_per_context_gives_the_same_plans(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1200)
    s_pose, g_pose = _pose_queries(scene, o, params, 12, seed=31)
    s_joint, g_joint = _joint_queries(scene, o, params, 12, seed=33)
    starts, goals = np.concatenate([s_pose, s_joint]), np.concatenate([g_pose, g_joint])
    single, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=8, want_states=True)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, stats = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=4, want_states=True)
    finally:
        for c in ctxs[1:]:
            c.close()
    _assert_same(single, multi)
    assert stats["edges_submitted"] > 0


@pytest.mark.gpu
def test_ubr1_with_attached_object_pose_goals_match_oracle():
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        params = _params(scene, 1500)
        starts, _ = scenes.ubr1_tabletop_queries(16)
        poses = o.planning_frame_fk(_walks(o, starts, params, 16, seed=41))
        goals = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)
        ref = _oracle(o, scene, params, starts, goals)
        got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, n_threads=2, want_states=True)
        _assert_same(ref, got)
        assert sum(a["success"] for a in ref) >= 4
    finally:
        ctx.close()


SMPLGPU_ERR_INVALID = -1


def _raw_plan(ctxs, scene, tables, params, goals):
    """smplhost_plan_batch_goals on one start per goal; returns its code"""
    H = api.host_lib()
    dof = tables.dof
    lo, hi, cont = tables.limits()
    res = np.ascontiguousarray(params.resolutions, dtype=np.float64)
    prims = np.ascontiguousarray(params.mprims, dtype=np.float64)
    flags = np.ascontiguousarray(params.short_flags, dtype=np.uint8)
    P = api.PlanParamsC()
    P.dof = dof
    P.resolutions, P.mprims, P.short_flags, P.n_prims = api._dp(res), api._dp(prims), api._bp(flags), len(prims)
    P.epsilon, P.max_expansions, P.short_dist_thresh, P.use_short_dist = 100.0, 50, 0.4, 1
    P.cost_per_cell, P.inflation_radius = int(scene.cost_per_cell), float(scene.inflation_radius)
    P.var_min, P.var_max, P.var_continuous = api._dp(lo), api._dp(hi), api._bp(cont)
    P.res, P.n_threads = float(scene.res), 1
    for a in range(3):
        P.origin[a], P.dims[a] = float(scene.origin[a]), int(scene.dims[a])
    goals = np.ascontiguousarray(goals)
    nq = len(goals)
    starts = np.ascontiguousarray(scenes.tabletop_queries(nq)[0])
    summary = np.zeros((nq, 5), np.int32)
    arr = (C.c_void_p * len(ctxs))(*ctxs)
    return H.smplhost_plan_batch_goals(arr, len(ctxs), C.byref(P), api._dp(starts), goals.ctypes.data_as(C.POINTER(api.GoalC)),
                                       nq, 4, api._ip(summary), None, 0, None, None)


@pytest.mark.gpu
def test_bad_goal_records_are_refused(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 50)
    starts, xyz = scenes.tabletop_queries(2)
    good = api.pose_goals(np.concatenate([xyz, np.zeros((2, 3))], axis=1), params.xyz_tolerance, rpy_tolerance=0.05)
    assert _raw_plan([ctx.h], scene, tables, params, good) == 0
    assert _raw_plan([None], scene, tables, params, good) < 0
    bad = []
    g = good.copy(); g["type"][1] = 3; bad.append(g)
    g = good.copy(); g["type"][0] = -1; bad.append(g)
    g = good.copy(); g["xyz_tolerance"][0, 2] = -0.01; bad.append(g)
    g = good.copy(); g["rpy_tolerance"][1] = np.nan; bad.append(g)
    g = good.copy(); g["rpy_tolerance"][1] = -0.1; bad.append(g)
    j = api.joint_goals(starts, 0.01)
    g = j.copy(); g["angle_tolerances"][0, 6] = np.nan; bad.append(g)
    g = j.copy(); g["angle_tolerances"][1, 0] = -1.0; bad.append(g)
    for k, g in enumerate(bad):
        assert _raw_plan([ctx.h], scene, tables, params, g) == SMPLGPU_ERR_INVALID, k
    # the device entry point checks the same (the planner above left the context with lattices), and a null context
    L = api.gpu_lib()
    slots = np.zeros(2, np.int32)
    gd = np.zeros(2, np.int32)
    q = np.ascontiguousarray(starts[:2])
    begin = L.smplgpu_lattice_begin_goals
    begin.argtypes = [C.c_void_p, api.c_int32_p, api.c_double_p, api.c_int32_p, C.POINTER(api.GoalC), C.c_int]
    assert begin(None, api._ip(slots), api._dp(q), api._ip(gd), good.ctypes.data_as(C.POINTER(api.GoalC)), 2) < 0
    for k, g in enumerate(bad):
        g = np.ascontiguousarray(g)
        assert begin(ctx.h, api._ip(slots), api._dp(q), api._ip(gd), g.ctypes.data_as(C.POINTER(api.GoalC)), 2) == \
            SMPLGPU_ERR_INVALID, k
    # the context still plans afterwards
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, good, max_concurrent=2)
    assert len(got) == 2
