"""Goal sets in the oracle (oracle/goal_sets/goal_set_lattice.cpp: oracle_plan_goal_set): a query succeeds at any
record of its set.  A set of one is the single-goal planner (oracle_plan_goal, oracle_plan_goal_snap); repeated records
and records outside the grid change nothing but the reached index; the BFS is seeded at every record's position, as
BFS_3D::run(begin, end) seeds its range."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
import goal_oracle
import goal_set_oracle
import snap_oracle
from helpers import make_oracle
from oracle_api import OracleBfs
from smpl_b200 import api, scenes

from test_gpu_goal_types import _joint_queries, _params, _pose_queries
from test_gpu_ik_snap import _reachable_pose_queries

WALL = 0x7FFFFFFF
SNAP = api.SnapParams(dist_thresh=0.2)


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


def _set(o, scene, params, start, goals, snap=None):
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
    return goal_set_oracle.plan_set(o, scene.T_kin_to_planning, start, goals, params, snap)


def _single(o, scene, params, start, goal, snap=None):
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)
    if snap is None:
        return goal_oracle.plan(o, start, goal, params)
    return snap_oracle.plan_snap(o, scene.T_kin_to_planning, start, goal, params, snap)


def _assert_same(a, b):
    assert (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
           (b["success"], b["expansions"], b["cost"], b["num_states"])
    assert np.array_equal(a["path_ids"], b["path_ids"])
    assert np.array_equal(a["path_states"], b["path_states"])


def _fixtures(scene, o):
    """the PR2 pose, joint and mixed fixtures of the goal-type and snap tests"""
    params = _params(scene, 1500)
    s_pose, g_pose = _pose_queries(scene, o, params, 8, seed=11)
    s_reach, g_reach = _reachable_pose_queries(o, scenes.tabletop_queries(6, seed=41)[0], 6, seed=43)
    s_joint, g_joint = _joint_queries(scene, o, params, 6, seed=23)
    base, xyz = scenes.tabletop_queries(4, seed=25)
    starts = np.concatenate([s_pose, s_reach, s_joint, base])
    goals = np.concatenate([g_pose, g_reach, g_joint, api.pose_goals(xyz, params.xyz_tolerance)])
    return params, starts, goals


@pytest.mark.parametrize("snap", [None, SNAP], ids=["snaps_off", "snaps_on"])
def test_sets_of_one_are_the_single_goal_planner(tabletop, snap):
    scene, o = tabletop
    params, starts, goals = _fixtures(scene, o)
    solved = 0
    for s, g in zip(starts, goals):
        a = _single(o, scene, params, s, g, snap)
        b = _set(o, scene, params, s, g[None], snap)
        _assert_same(a, b)
        if snap is not None:
            assert (a["ik_attempted"], a["ik_converged"]) == (b["ik_attempted"], b["ik_converged"])
        assert b["reached_goal"] == (0 if b["success"] else -1)
        solved += b["success"]
    assert solved >= 6


def test_repeated_records_plan_as_the_record_alone(tabletop):
    scene, o = tabletop
    params, starts, goals = _fixtures(scene, o)
    for s, g in list(zip(starts, goals))[::3]:
        a = _set(o, scene, params, s, g[None], SNAP)
        b = _set(o, scene, params, s, np.repeat(g[None], 4), SNAP)
        _assert_same(a, b)
        assert b["reached_goal"] == a["reached_goal"]


def test_a_record_outside_the_grid_changes_nothing_but_the_index(tabletop):
    scene, o = tabletop
    params, starts, goals = _fixtures(scene, o)
    out = api.pose_goals([(5.0, 0.0, 1.0)], params.xyz_tolerance)
    solved = 0
    for s, g in zip(starts, goals):
        for snap in (None, SNAP):
            a = _set(o, scene, params, s, g[None], snap)
            b = _set(o, scene, params, s, np.concatenate([out, g[None]]), snap)
            _assert_same(a, b)
            assert b["reached_goal"] == (1 if a["success"] else -1)
            solved += a["success"]
    assert solved >= 10


def test_any_record_of_a_set_may_be_reached(tabletop):
    """sets of 4 joint goals: the planner stops at whichever it reaches first, never costs more than the best single
    record, and the reached record is one the path's last state satisfies"""
    scene, o = tabletop
    params = _params(scene, 1500)
    starts, goals = _joint_queries(scene, o, params, 12, seed=5)
    reached = set()
    for i in range(0, 12, 4):
        rec = goals[i:i + 4]
        for s in starts[i:i + 4]:
            b = _set(o, scene, params, s, rec)
            singles = [_set(o, scene, params, s, g[None]) for g in rec]
            if not any(x["success"] for x in singles):
                continue
            assert b["success"]
            k = b["reached_goal"]
            reached.add(k)
            last = b["path_states"][-1]
            g = rec[k]
            dof = len(last)
            assert (np.abs(last - g["angles"][:dof]) <= g["angle_tolerances"][:dof]).all()
            for j in range(k):   # records before the reached one are not satisfied
                assert not (np.abs(last - rec[j]["angles"][:dof]) <= rec[j]["angle_tolerances"][:dof]).all()
    assert len(reached) >= 2


def test_multi_seed_heuristic_is_bfs3d_run_over_the_range(tabletop):
    scene, o = tabletop
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)
    walls = o.heur_grid() == WALL                     # padded: the border cells are walls too
    nz, ny, nx = walls.shape
    rng = np.random.default_rng(3)
    xyz = np.concatenate([scenes.tabletop_queries(5, seed=9)[1], [(5.0, 0.0, 1.0)], rng.uniform(-0.5, 1.5, (6, 3))])
    xyz = np.concatenate([xyz, xyz[:2]])              # duplicates
    dims, origin, res, _ = o.grid_info()
    cells = [tuple(int(1.0 / res * (p[a] - (origin[a] - res)) + 0.5) - 1 for a in range(3)) for p in xyz]
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)
    k, got = goal_set_oracle.goal_set_bfs(o, xyz)
    b = OracleBfs(nx - 2, ny - 2, nz - 2)
    b.set_walls(walls[1:-1, 1:-1, 1:-1].astype(np.uint8))
    want_k = b.run_multi(cells + [(0, 0, 0)])         # the trailing triple commits the last real one
    assert k == want_k and 0 < k < len(xyz)
    assert np.array_equal(got, b.grid())


def test_goal_record_layout_matches_the_header():
    """api.GoalC (the records of goal sets) against sizeof / offsetof of smplgpu_goal, and the bound"""
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "smplgpu.h"
int main(void)
{
    printf("%zu %zu %zu %zu %zu %zu %zu %d\n", sizeof(smplgpu_goal), offsetof(smplgpu_goal, type),
           offsetof(smplgpu_goal, pose), offsetof(smplgpu_goal, xyz_tolerance), offsetof(smplgpu_goal, rpy_tolerance),
           offsetof(smplgpu_goal, angles), offsetof(smplgpu_goal, angle_tolerances), SMPLGPU_MAX_GOAL_SET);
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
    G = api.GoalC
    assert got == [C.sizeof(G), G.type.offset, G.pose.offset, G.xyz_tolerance.offset, G.rpy_tolerance.offset,
                   G.angles.offset, G.angle_tolerances.offset, api.MAX_GOAL_SET]
    assert api.GOAL_DTYPE.itemsize == C.sizeof(G)


def test_goal_sets_builds_records_and_offsets():
    a = api.pose_goals([(0.1, 0.2, 0.3)])
    b = api.joint_goals(np.zeros((3, 7)), 0.1)
    recs, off = api.goal_sets([a, b, np.concatenate([a, b[:1]])])
    assert off.tolist() == [0, 1, 4, 6] and off.dtype == np.int32 and len(recs) == 6
    assert recs["type"].tolist() == [0, 2, 2, 2, 0, 2]
    with pytest.raises(ValueError):
        api.goal_sets([a, a[:0]])
    with pytest.raises(ValueError):
        api.goal_sets([np.repeat(a, api.MAX_GOAL_SET + 1)])
