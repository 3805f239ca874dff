"""The planning-link IK (smplgpu_planning_link_ik) and the snap-to-goal action in the batched planner
(smplhost_plan_batch_snap) against the oracle (oracle/snap/snap_lattice.cpp: planningLinkIk, oracle_plan_goal_snap).
The IK is the project's own, defined once and restated on both sides, so ok flags and iteration counts must be equal
and the answers agree to 1e-9 (only CUDA's sin / cos / atan2 differ from glibc's, by <= 2 ulp)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
import snap_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_types import _joint_queries, _params, _walks
from test_oracle_ik_snap import _valid_states, ik_problems


def test_snap_records_layout_matches_the_headers():
    """api.IkParamsC / SnapParamsC against sizeof / offsetof of smplgpu_ik_params / smplhost_snap_params"""
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "smplhost.h"
int main(void)
{
    printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(smplgpu_ik_params), offsetof(smplgpu_ik_params, max_iterations),
           offsetof(smplgpu_ik_params, tolerance), sizeof(smplhost_snap_params), offsetof(smplhost_snap_params, enabled),
           offsetof(smplhost_snap_params, dist_thresh), offsetof(smplhost_snap_params, weight),
           offsetof(smplhost_snap_params, ik));
    printf("%zu %zu %zu %zu\n", sizeof(smplgpu_snap_params), offsetof(smplgpu_snap_params, enabled),
           offsetof(smplgpu_snap_params, dist_thresh), offsetof(smplgpu_snap_params, ik));
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
    I, S = api.IkParamsC, api.SnapParamsC
    assert got[:8] == [C.sizeof(I), I.max_iterations.offset, I.tolerance.offset, C.sizeof(S), S.enabled.offset,
                       S.dist_thresh.offset, S.weight.offset, S.ik.offset]
    # smplgpu_snap_params: enabled, dist_thresh, ik (the device record has no weight)
    assert got[8:] == [8 + 8 + C.sizeof(I), 0, 8, 16]


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


@pytest.mark.gpu
def test_device_ik_matches_oracle_ik(tabletop):
    scene, o, ctx, tables = tabletop
    poses, seeds = ik_problems(o, 4096, seed=7)
    far = seeds.copy()                                      # and unreachable targets: every step, no convergence
    far_poses = poses.copy()
    far_poses[:64, 0] += 5.0
    poses = np.concatenate([poses, far_poses[:64]])
    seeds = np.concatenate([seeds, far[:64]])
    q_ref, ok_ref, it_ref = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses, seeds)
    q, ok, it = ctx.planning_link_ik(poses, seeds)
    _, _, cont = tables.limits()
    d = q - q_ref
    d[:, cont.astype(bool)] = np.angle(np.exp(1j * d[:, cont.astype(bool)]))   # continuous joints: modulo 2 pi
    diff = np.abs(d[:4096]).max()
    print("device vs oracle IK: %d problems, %d converged, largest |q difference| %.3g (reachable targets)"
          % (len(q), ok.sum(), diff))
    assert np.array_equal(ok, ok_ref) and np.array_equal(it, it_ref)
    # 100 steps towards an unreachable target amplify the last-bit differences of sin / cos: only the verdicts match
    assert diff <= 1e-9
    assert ok[:4096].mean() >= 0.99 and not ok[4096:].any() and (it[4096:] == 100).all()
    # the parameters reach the kernel
    _, ok2, it2 = ctx.planning_link_ik(poses[:256], seeds[:256], max_iterations=2, tolerance=1e-3)
    _, ok2r, it2r = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, poses[:256], seeds[:256], 2, 1e-3)
    assert np.array_equal(ok2, ok2r) and np.array_equal(it2, it2r) and it2.max() == 2


def _oracle_snap(o, scene, params, starts, goals, snap):
    out = []
    for s, g in zip(starts, goals):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        out.append(snap_oracle.plan_snap(o, scene.T_kin_to_planning, s, g, params, snap))
    return out


def _assert_same(ref, got, max_differing=0):
    """success, expansions, cost, lattice size and id path equal; path states equal except the rows a snap produced
    (an IK answer), which agree to 1e-6 (two IK runs whose error sits at the tolerance after the same step can take one
    step more or less: ulps of sin / cos decide).  Up to max_differing queries may differ altogether: an IK answer that
    reaches the goal orientation to ~1e-8 rad puts isGoal's unclamped acos argument at 1 +- a few ulps, where the
    oracle's and the device's sin / cos can decide goal (0) against no goal (NaN) (DESIGN.md section 2).  Returns the
    largest path-state difference of the matching queries."""
    worst = 0.0
    differing = []
    for i, (a, b) in enumerate(zip(ref, got)):
        same = (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"]) and np.array_equal(a["path_ids"], b["path_ids"])
        if not same:
            differing.append((i, a["expansions"], b["expansions"], a["cost"], b["cost"]))
            continue
        d = np.abs(a["path_states"] - b["path_states"]).max(axis=1) if len(a["path_states"]) else np.zeros(0)
        assert (d <= 1e-6).all(), (i, d.max())
        worst = max(worst, float(d.max()) if len(d) else 0.0)
    print("largest path-state difference %.3g; queries that differ (index, expansions, cost): %s" % (worst, differing))
    assert len(differing) <= max_differing, differing
    return worst


def _reachable_pose_queries(o, starts, n, seed):
    poses = o.planning_frame_fk(_valid_states(o, n, seed=seed))
    return starts[:n], api.pose_goals(poses, (0.015, 0.015, 0.015), rpy_tolerance=0.05)


SNAP = api.SnapParams(dist_thresh=0.2)


@pytest.mark.gpu
def test_snap_pose_goals_match_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 2000)
    starts, goals = _reachable_pose_queries(o, scenes.tabletop_queries(16, seed=29)[0], 16, seed=31)
    ref = _oracle_snap(o, scene, params, starts, goals, SNAP)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=8, n_threads=2,
                                want_states=True, snap=SNAP)
    _assert_same(ref, got, max_differing=1)
    assert sum(a["success"] for a in ref) >= 8
    assert stats["ik_attempted"] > 0 and stats["ik_converged"] > 0


@pytest.mark.gpu
def test_snap_joint_goals_match_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 2000)
    starts, goals = _joint_queries(scene, o, params, 16, seed=3)
    ref = _oracle_snap(o, scene, params, starts, goals, SNAP)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=8, want_states=True, snap=SNAP)
    _assert_same(ref, got)
    assert stats["ik_attempted"] == 0 and sum(a["success"] for a in ref) >= 8


@pytest.mark.gpu
def test_snap_mixed_goal_types_and_contexts_match_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    base, xyz = scenes.tabletop_queries(8, seed=25)
    s_pose, g_pose = _reachable_pose_queries(o, scenes.tabletop_queries(8, seed=41)[0], 8, seed=43)
    s_joint, g_joint = _joint_queries(scene, o, params, 8, seed=23)
    g_xyz = api.pose_goals(xyz, params.xyz_tolerance)
    order = np.arange(24).reshape(3, 8).T.reshape(-1)   # pose, joint, xyz, pose, ...
    starts = np.concatenate([s_pose, s_joint, base])[order]
    goals = np.concatenate([g_pose, g_joint, g_xyz])[order]
    snap = api.SnapParams(dist_thresh=0.0)   # the demo's threshold
    ref = _oracle_snap(o, scene, params, starts, goals, snap)
    one, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=7, n_threads=2, want_states=True,
                            snap=snap)
    _assert_same(ref, one, max_differing=1)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, stats = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=4, want_states=True,
                                      snap=snap)
    finally:
        for c in ctxs[1:]:
            c.close()
    _assert_same(ref, multi, max_differing=1)
    for a, b in zip(one, multi):   # device against device: bit for bit
        assert a["expansions"] == b["expansions"] and np.array_equal(a["path_states"], b["path_states"])
    assert stats["ik_attempted"] > 0


@pytest.mark.gpu
def test_snap_ubr1_pose_goals_match_oracle():
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        params = _params(scene, 1500)
        starts, _ = scenes.ubr1_tabletop_queries(12)
        poses = o.planning_frame_fk(_walks(o, starts, params, 16, seed=41))
        goals = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)
        ref = _oracle_snap(o, scene, params, starts, goals, SNAP)
        got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, n_threads=2,
                                    want_states=True, snap=SNAP)
        _assert_same(ref, got, max_differing=2)
        assert sum(a["success"] for a in ref) >= 4 and stats["ik_attempted"] > 0
    finally:
        ctx.close()


@pytest.mark.gpu
def test_snaps_off_is_the_goal_entry_point_bit_for_bit(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    s_pose, g_pose = _reachable_pose_queries(o, scenes.tabletop_queries(8, seed=51)[0], 8, seed=53)
    s_joint, g_joint = _joint_queries(scene, o, params, 8, seed=55)
    starts, goals = np.concatenate([s_pose, s_joint]), np.concatenate([g_pose, g_joint])
    want, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, want_states=True)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, want_states=True,
                                snap=api.SnapParams(enabled=False, dist_thresh=0.2))
    for a, b in zip(want, got):
        assert (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"])
        assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])
    assert stats["ik_attempted"] == 0


SMPLGPU_ERR_INVALID = -1


@pytest.mark.gpu
def test_bad_snap_and_ik_parameters_are_refused(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 50)
    starts, xyz = scenes.tabletop_queries(2)
    goals = api.pose_goals(xyz, params.xyz_tolerance)
    bad = [dict(dist_thresh=-0.1), dict(dist_thresh=np.nan), dict(weight=-1.0), dict(weight=np.nan),
           dict(max_iterations=0), dict(tolerance=0.0), dict(tolerance=-1e-6), dict(tolerance=np.nan)]
    for k, kw in enumerate(bad):
        with pytest.raises(api.SmplGpuError):
            api.plan_batch(ctx, scene, tables, params, starts, goals, snap=api.SnapParams(**kw))
    # the device entry points check the same
    L = api.gpu_lib()
    L.smplgpu_lattice_set_snap.argtypes = [C.c_void_p, C.c_void_p]

    class DevSnap(C.Structure):
        _fields_ = [("enabled", C.c_int32), ("dist_thresh", C.c_double), ("ik", api.IkParamsC)]

    for kw in ({"dist_thresh": -1.0}, {"dist_thresh": np.nan}, {"max_iterations": 0}, {"tolerance": np.nan}):
        p = DevSnap(1, kw.get("dist_thresh", 0.1), api.IkParamsC(kw.get("max_iterations", 100), kw.get("tolerance", 1e-6)))
        assert L.smplgpu_lattice_set_snap(ctx.h, C.byref(p)) == SMPLGPU_ERR_INVALID, kw
    q = np.zeros((1, scene.dof))
    for kw in (dict(max_iterations=0), dict(tolerance=0.0), dict(tolerance=np.nan)):
        with pytest.raises(api.SmplGpuError):
            ctx.planning_link_ik(np.zeros((1, 6)), q, **kw)
    # the context still plans afterwards, with snaps
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=2, snap=SNAP)
    assert len(got) == 2
