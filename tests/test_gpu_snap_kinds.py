"""The snap kinds SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY in the batched planner (smplhost_plan_batch_snaps,
smplgpu_lattice_set_snaps) and the position-only planning-link IK (smplgpu_planning_link_ik_position), against the
oracle (oracle/snap_kinds/snap_kinds_lattice.cpp: planningLinkIkPosition, oracle_plan_goal_set_snaps) and against the
SNAP_TO_XYZ_RPY entry points."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT
import snap_kinds_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_sets import _assert_sets_same, _walk_pose_sets
from test_gpu_goal_types import _joint_queries, _params
from test_gpu_planner_limits import _stride_in_use, _wide_params
from test_oracle_ik_snap import ik_problems

SMPLGPU_ERR_INVALID = -1


class _Snaps(api.SnapParams):
    """SnapParams that always go through smplhost_plan_batch_snaps, also with SNAP_TO_XYZ_RPY alone"""

    def new_kinds(self):
        return True


KINDS = {"rpy": _Snaps(enabled=False, rpy_dist_thresh=0.2),
         "xyz": _Snaps(enabled=False, xyz_dist_thresh=0.2),
         "xyz_rpy": _Snaps(dist_thresh=0.2),
         "all": _Snaps(dist_thresh=0.0, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2)}


def test_snap_kinds_records_layout_matches_the_headers():
    """api.SnapKindsC / SnapsParamsC against sizeof / offsetof of smplgpu_snap_kinds / smplhost_snaps_params"""
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "smplhost.h"
int main(void)
{
    printf("%zu %zu %zu %zu %zu %zu %zu %d %d %d\n", sizeof(smplgpu_snap_kinds), offsetof(smplgpu_snap_kinds, enabled),
           offsetof(smplgpu_snap_kinds, dist_thresh), offsetof(smplgpu_snap_kinds, ik), sizeof(smplhost_snaps_params),
           offsetof(smplhost_snaps_params, kinds), offsetof(smplhost_snaps_params, weight), SMPLGPU_SNAP_RPY,
           SMPLGPU_SNAP_XYZ, SMPLGPU_SNAP_XYZ_RPY);
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
    K, S = api.SnapKindsC, api.SnapsParamsC
    assert got == [C.sizeof(K), K.enabled.offset, K.dist_thresh.offset, K.ik.offset, C.sizeof(S), S.kinds.offset,
                   S.weight.offset, api.SNAP_RPY, api.SNAP_XYZ, api.SNAP_XYZ_RPY]


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


@pytest.mark.gpu
def test_device_position_ik_matches_oracle(tabletop):
    scene, o, ctx, tables = tabletop
    poses, seeds = ik_problems(o, 4096, seed=7)
    xyz = np.concatenate([poses[:, :3], poses[:64, :3] + np.array([5.0, 0.0, 0.0])])   # and 64 unreachable targets
    seeds = np.concatenate([seeds, seeds[:64]])
    q_ref, ok_ref, it_ref = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning, xyz, seeds)
    q, ok, it = ctx.planning_link_ik(xyz, seeds)
    _, _, cont = tables.limits()
    d = q - q_ref
    d[:, cont.astype(bool)] = np.angle(np.exp(1j * d[:, cont.astype(bool)]))   # continuous joints: modulo 2 pi
    diff = np.abs(d[:4096]).max()
    print("device vs oracle position-only IK: %d problems, %d converged, largest |q difference| %.3g"
          % (len(q), ok.sum(), diff))
    assert np.array_equal(ok, ok_ref) and np.array_equal(it, it_ref)
    assert diff <= 1e-9
    assert ok[:4096].mean() >= 0.99 and not ok[4096:].any() and (it[4096:] == 100).all()
    _, ok2, it2 = ctx.planning_link_ik(xyz[:256], seeds[:256], max_iterations=2, tolerance=1e-3)
    _, ok2r, it2r = snap_kinds_oracle.planning_link_ik_position(o, scene.T_kin_to_planning, xyz[:256], seeds[:256], 2,
                                                                1e-3)
    assert np.array_equal(ok2, ok2r) and np.array_equal(it2, it2r) and it2.max() == 2


def _oracle(o, scene, params, starts, records, offsets, snap):
    out = []
    for i, s in enumerate(starts):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        out.append(snap_kinds_oracle.plan_set_snaps(o, scene.T_kin_to_planning, s, records[offsets[i]:offsets[i + 1]],
                                                    params, snap))
    return out


def _mixed_queries(scene, o, params):
    """16 PR2 queries: XYZ records, XYZ_RPY sets of two, joint records, and mixed sets (XYZ_RPY, joint, XYZ)"""
    starts, _ = scenes.tabletop_queries(8, seed=61)
    xyz_recs, xyz_off = _walk_pose_sets(o, starts, params, 2, seed=63, rpy_tolerance=None)
    rpy_recs, rpy_off = _walk_pose_sets(o, starts, params, 2, seed=65, rpy_tolerance=0.05)
    s_joint, g_joint = _joint_queries(scene, o, params, 8, seed=71)
    sets = []
    for i in range(4):
        sets.append(xyz_recs[xyz_off[i + 4]:xyz_off[i + 4] + 1])
    for i in range(4):
        sets.append(rpy_recs[rpy_off[i]:rpy_off[i + 1]])
    for i in range(4):
        sets.append(g_joint[i:i + 1])
    for i in range(4, 8):
        sets.append(np.concatenate([rpy_recs[rpy_off[i]:rpy_off[i] + 1], g_joint[i:i + 1],
                                    xyz_recs[xyz_off[i]:xyz_off[i] + 1]]))
    all_starts = np.concatenate([starts[4:8], starts[:4], s_joint[:4], s_joint[4:8]])
    return all_starts, api.goal_sets(sets)


def _check_counters(snap, stats):
    en, _ = snap.kinds()
    for k, name in enumerate(api.SNAP_KIND_NAMES):
        if not en[k]:
            assert stats["ik_attempted_" + name] == 0
    assert stats["ik_attempted"] == sum(stats["ik_attempted_" + n] for n in api.SNAP_KIND_NAMES)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_kinds_match_oracle_on_one_and_three_contexts(tabletop, kind):
    scene, o, ctx, tables = tabletop
    snap = KINDS[kind]
    params = _params(scene, 1500)
    starts, (records, offsets) = _mixed_queries(scene, o, params)
    ref = _oracle(o, scene, params, starts, records, offsets, snap)
    one, stats = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=5, n_threads=2,
                                want_states=True, snap=snap)
    # the documented rounding allowance of the snap tests (tests/test_gpu_ik_snap.py _assert_same): one query may
    # differ where an IK answer puts isGoal's acos argument within ulps of 1
    _assert_sets_same(ref, one, max_differing=1)
    _check_counters(snap, stats)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, mstats = api.plan_batch(ctxs, scene, tables, params, starts, (records, offsets), max_concurrent=3,
                                       want_states=True, snap=snap)
    finally:
        for c in ctxs[1:]:
            c.close()
    for a, b in zip(one, multi):   # device against device: bit for bit
        assert (a["expansions"], a["reached_goal"]) == (b["expansions"], b["reached_goal"])
        assert np.array_equal(a["path_states"], b["path_states"])
    for name in api.SNAP_KIND_NAMES:
        assert stats["ik_attempted_" + name] == mstats["ik_attempted_" + name]
    oracle_ik = np.sum([a["ik_by_kind"] for a in ref], axis=0)
    print("%s: oracle IK solves by kind (run, converged) %s; device %s" % (
        kind, oracle_ik.tolist(), [(stats["ik_attempted_" + n], stats["ik_converged_" + n]) for n in api.SNAP_KIND_NAMES]))
    assert sum(a["success"] for a in ref) >= 6 and stats["ik_attempted"] > 0


@pytest.mark.gpu
def test_ubr1_with_attached_box_all_kinds_match_oracle():
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        params = _params(scene, 1500)
        starts, _ = scenes.ubr1_tabletop_queries(8)
        rpy_recs, rpy_off = _walk_pose_sets(o, starts, params, 2, seed=81, rpy_tolerance=0.05)
        xyz_recs, xyz_off = _walk_pose_sets(o, starts, params, 1, seed=83, rpy_tolerance=None)
        sets = [np.concatenate([rpy_recs[rpy_off[i]:rpy_off[i + 1]], xyz_recs[xyz_off[i]:xyz_off[i + 1]]])
                if i % 2 else xyz_recs[xyz_off[i]:xyz_off[i + 1]] for i in range(8)]
        records, offsets = api.goal_sets(sets)
        snap = KINDS["all"]
        ref = _oracle(o, scene, params, starts, records, offsets, snap)
        got, stats = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=4,
                                    n_threads=2, want_states=True, snap=snap)
        _assert_sets_same(ref, got, max_differing=2)   # the UBR1 allowance of the snap tests
        _check_counters(snap, stats)
        assert sum(a["success"] for a in ref) >= 3 and stats["ik_attempted"] > 0
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("thresh", [0.0, 0.2])
def test_xyz_rpy_alone_through_snaps_equals_goal_sets(tabletop, thresh):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    starts, goals = _mixed_queries(scene, o, params)
    want, wst = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=5, n_threads=2,
                               want_states=True, snap=api.SnapParams(dist_thresh=thresh))
    got, gst = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=5, n_threads=2,
                              want_states=True, snap=_Snaps(dist_thresh=thresh))
    for a, b in zip(want, got):
        assert (a["success"], a["expansions"], a["cost"], a["num_states"], a["reached_goal"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"], b["reached_goal"])
        assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])
    # (the round count is not compared: when a refilled slot's bank BFS finishes depends on timing, so it differs
    # between runs of the same call; the edges submitted, one stride per expansion, do not)
    for key in ("edges_submitted", "ik_attempted", "ik_converged", "ik_attempted_xyz_rpy"):
        assert wst[key] == gst[key], key
    assert gst["ik_attempted"] > 0


@pytest.mark.gpu
def test_stride_limit_with_three_kinds(tabletop):
    scene, o, ctx, tables = tabletop
    snap = KINDS["all"]
    starts, (records, offsets) = _mixed_queries(scene, o, _params(scene, 1200))   # goals from the default primitives
    params = _wide_params(scene, 15, 1200)   # 14 of its primitives: 28 primitive words + 3 snap words = 31
    params.mprims, params.short_flags, params.weights = params.mprims[1:], params.short_flags[1:], params.weights[1:]
    ref = _oracle(o, scene, params, starts, records, offsets, snap)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=6, n_threads=2,
                                want_states=True, snap=snap)
    assert _stride_in_use(stats, got) == 31
    _assert_sets_same(ref, got, max_differing=1)
    assert sum(a["success"] for a in ref) >= 4
    with pytest.raises(api.SmplGpuError):   # 30 primitive words + 3 snap words = 33
        api.plan_batch(ctx, scene, tables, _wide_params(scene, 15, 50), starts, (records, offsets), snap=snap)
    with pytest.raises(api.SmplGpuError):   # 32 primitive words + one snap word = 33
        api.plan_batch(ctx, scene, tables, _wide_params(scene, 16, 50), starts, (records, offsets),
                       snap=_Snaps(enabled=False, xyz_dist_thresh=0.2))
    got, _ = api.plan_batch(ctx, scene, tables, _wide_params(scene, 15, 50), starts, (records, offsets),
                            snap=_Snaps(dist_thresh=0.0, xyz_dist_thresh=0.2))   # 30 + 2 = 32 words still plan
    assert len(got) == len(starts)


@pytest.mark.gpu
def test_bad_thresholds_and_ik_parameters_are_refused(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 50)
    starts, xyz = scenes.tabletop_queries(2)
    goals = api.goal_sets([api.pose_goals(xyz[i:i + 1], params.xyz_tolerance) for i in range(2)])
    bad = []
    for field in ("dist_thresh", "xyz_dist_thresh", "rpy_dist_thresh"):
        for v in (np.nan, -0.1):
            s = _Snaps(enabled=False, xyz_dist_thresh=0.2)
            setattr(s, field, v)
            bad.append(s)
    bad.append(_Snaps(dist_thresh=0.1, enabled=False, xyz_dist_thresh=0.1, max_iterations=0))
    bad.append(_Snaps(enabled=False, rpy_dist_thresh=0.1, tolerance=0.0))
    bad.append(_Snaps(enabled=False, rpy_dist_thresh=0.1, weight=np.nan))
    for s in bad:
        with pytest.raises(api.SmplGpuError):
            api.plan_batch(ctx, scene, tables, params, starts, goals, snap=s)
    # the device entry point checks the same, disabled kinds included
    L = api.gpu_lib()
    L.smplgpu_lattice_set_snaps.argtypes = [C.c_void_p, C.POINTER(api.SnapKindsC)]
    for s in bad[:-1]:
        k = s.c_kinds().kinds
        assert L.smplgpu_lattice_set_snaps(ctx.h, C.byref(k)) == SMPLGPU_ERR_INVALID
    # the context still plans afterwards, with every kind
    got, st = api.plan_batch(ctx, scene, tables, params, starts, goals, snap=KINDS["all"])
    assert len(got) == 2 and "ik_attempted_rpy" in st
