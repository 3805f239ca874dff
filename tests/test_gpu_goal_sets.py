"""Goal sets in the batched planner (smplhost_plan_batch_goal_sets, smplgpu_lattice_begin_goal_sets) and the
multi-seed BFS bank runs behind them (smplgpu_bfs_bank_run_slots_multi[_async]), against the oracle's goal-set planner
(oracle/goal_sets/goal_set_lattice.cpp: oracle_plan_goal_set) and against the single-goal entry points."""
import ctypes as C

import numpy as np
import pytest

import goal_set_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_types import _joint_queries, _params, _walks
from test_gpu_ik_snap import _assert_same, _reachable_pose_queries

SMPLGPU_ERR_INVALID = -1


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


def _oracle_sets(o, scene, params, starts, records, offsets, snap):
    out = []
    for i, s in enumerate(starts):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        out.append(goal_set_oracle.plan_set(o, scene.T_kin_to_planning, s, records[offsets[i]:offsets[i + 1]], params,
                                            snap))
    return out


def _assert_sets_same(ref, got, max_differing=0):
    _assert_same(ref, got, max_differing)
    differing = 0
    for a, b in zip(ref, got):
        if a["path_ids"].tolist() == b["path_ids"].tolist() and a["expansions"] == b["expansions"]:
            assert a["reached_goal"] == b["reached_goal"]
        else:
            differing += 1
    assert differing <= max_differing


@pytest.mark.gpu
def test_multi_seed_bank_runs_equal_single_grid_runs(tabletop):
    scene, o, ctx, tables = tabletop
    walls = ctx.bfs_set_walls_from_df(scene.inflation_radius)
    ctx.bfs_bank_create(6, scene.inflation_radius)
    nx, ny, nz = (int(d) for d in scene.dims)
    o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # the same walls (tests/test_gpu_planner.py)
    wall_cells = np.argwhere(o.heur_grid()[1:-1, 1:-1, 1:-1] == 0x7FFFFFFF)[:, ::-1]   # (x, y, z)
    assert walls > 0 and len(wall_cells) > 0
    rng = np.random.default_rng(17)
    free = lambda k: np.stack([rng.integers(0, d, k) for d in (nx, ny, nz)], axis=1)
    sets = [free(1),                                                        # one seed
            free(3),                                                        # three
            free(64),                                                       # a full goal set
            np.concatenate([free(2), free(2)[:1], [[-1, 0, 0], [nx, 2, 2]]]),  # duplicates and out-of-bounds seeds
            np.concatenate([wall_cells[rng.integers(0, len(wall_cells), 2)], free(1)]),   # seeds on walls
            np.zeros((0, 3), np.int64)]                                     # no seed at all
    sets[3] = np.concatenate([sets[3], sets[3][:1]])
    all_cells = np.stack(np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"), -1).reshape(-1, 3)
    all_cells = np.ascontiguousarray(all_cells, np.int32)
    for wait in (True, False):
        slots = [5, 0, 3, 1, 4, 2] if wait else [0, 1, 2, 3, 4, 5]
        n_in = ctx.bfs_bank_run_slots_multi(slots, sets, wait=wait)
        if wait:
            assert n_in == sum(int(((s >= 0) & (s < (nx, ny, nz))).all(axis=1).sum()) for s in sets)
        else:
            ctx.bfs_bank_run_wait()
        for k, s in enumerate(sets):
            ctx.bfs_set_walls_from_df(scene.inflation_radius)   # fresh walls: a seed on a wall un-walls it
            ctx.bfs_run(s.astype(np.int32))
            single = ctx.bfs_download()[1:-1, 1:-1, 1:-1]
            bank = ctx.bfs_bank_distances(np.full(len(all_cells), slots[k], np.int32), all_cells)
            want = single[all_cells[:, 2], all_cells[:, 1], all_cells[:, 0]]
            assert np.array_equal(bank, want), (wait, k)
            assert ((want == 0).sum() > 0) == (k != 5)


def _walk_pose_sets(o, starts, params, k, seed, rpy_tolerance):
    """k pose records per query at the poses of lattice states a few primitive steps from the start (often solved),
    the first query's set led by a record outside the grid"""
    poses = np.concatenate([o.planning_frame_fk(_walks(o, starts, params, 12 + 4 * j, seed + j)) for j in range(k)])
    poses = poses.reshape(k, len(starts), 6).transpose(1, 0, 2)
    poses[0, 0, :3] = (5.0, 0.0, 1.0)
    sets = [api.pose_goals(p if rpy_tolerance is not None else p[:, :3], (0.015, 0.015, 0.015),
                           rpy_tolerance=rpy_tolerance) for p in poses]
    return api.goal_sets(sets)


SNAPS = [None, api.SnapParams(dist_thresh=0.0), api.SnapParams(dist_thresh=0.2)]
SNAP_IDS = ["off", "0.0", "0.2"]


@pytest.mark.gpu
@pytest.mark.parametrize("snap", SNAPS, ids=SNAP_IDS)
@pytest.mark.parametrize("rpy", [None, 0.05], ids=["xyz", "xyz_rpy"])
def test_pose_sets_match_oracle(tabletop, snap, rpy):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    starts, _ = scenes.tabletop_queries(12, seed=61)
    records, offsets = _walk_pose_sets(o, starts, params, 3, seed=63, rpy_tolerance=rpy)
    ref = _oracle_sets(o, scene, params, starts, records, offsets, snap)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=5, n_threads=2,
                            want_states=True, snap=snap)
    _assert_sets_same(ref, got, max_differing=0 if snap is None else 1)
    assert sum(a["success"] for a in ref) >= 4
    assert all((a["reached_goal"] >= 0) == a["success"] for a in got)


@pytest.mark.gpu
@pytest.mark.parametrize("snap", SNAPS, ids=SNAP_IDS)
def test_joint_and_mixed_sets_match_oracle_on_one_and_several_contexts(tabletop, snap):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    starts, g_joint = _joint_queries(scene, o, params, 12, seed=71)
    _, g_joint2 = _joint_queries(scene, o, params, 12, seed=73)
    pose_recs, pose_off = _walk_pose_sets(o, starts, params, 2, seed=75, rpy_tolerance=0.05)
    sets = []
    for i in range(12):
        poses = pose_recs[pose_off[i]:pose_off[i + 1]]
        if i % 3 == 0:
            sets.append(np.concatenate([g_joint2[i:i + 1], g_joint[i:i + 1]]))          # joint sets
        else:
            sets.append(np.concatenate([poses[:1], g_joint[i:i + 1], poses[1:]]))    # mixed sets
    records, offsets = api.goal_sets(sets)
    ref = _oracle_sets(o, scene, params, starts, records, offsets, snap)
    one, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=5, n_threads=2,
                            want_states=True, snap=snap)
    _assert_sets_same(ref, one, max_differing=0 if snap is None else 1)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, _ = api.plan_batch(ctxs, scene, tables, params, starts, (records, offsets), max_concurrent=3,
                                  want_states=True, snap=snap)
    finally:
        for c in ctxs[1:]:
            c.close()
    for a, b in zip(one, multi):   # device against device: bit for bit
        assert (a["expansions"], a["reached_goal"]) == (b["expansions"], b["reached_goal"])
        assert np.array_equal(a["path_states"], b["path_states"])
    assert sum(a["success"] for a in ref) >= 6
    assert len({a["reached_goal"] for a in ref if a["success"]}) >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("snap", SNAPS, ids=SNAP_IDS)
def test_ubr1_pose_sets_match_oracle(snap):
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        params = _params(scene, 1500)
        starts, _ = scenes.ubr1_tabletop_queries(8)
        records, offsets = _walk_pose_sets(o, starts, params, 3, seed=81, rpy_tolerance=0.05)
        ref = _oracle_sets(o, scene, params, starts, records, offsets, snap)
        got, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=4,
                                n_threads=2, want_states=True, snap=snap)
        _assert_sets_same(ref, got, max_differing=0 if snap is None else 2)
        assert sum(a["success"] for a in ref) >= 3
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("snap", SNAPS, ids=SNAP_IDS)
def test_sets_of_one_equal_the_single_goal_entry_points(tabletop, snap):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    s_pose, g_pose = _reachable_pose_queries(o, scenes.tabletop_queries(8, seed=91)[0], 8, seed=93)
    s_joint, g_joint = _joint_queries(scene, o, params, 8, seed=95)
    starts, goals = np.concatenate([s_pose, s_joint]), np.concatenate([g_pose, g_joint])
    want, wst = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, want_states=True, snap=snap)
    got, gst = api.plan_batch(ctx, scene, tables, params, starts, api.goal_sets([g[None] for g in goals]),
                              max_concurrent=6, want_states=True, snap=snap)
    for a, b in zip(want, got):
        assert (a["success"], a["expansions"], a["cost"], a["num_states"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"])
        assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"])
        assert b["reached_goal"] == (0 if b["success"] else -1)
    if snap is not None:
        assert (wst["ik_attempted"], wst["ik_converged"]) == (gst["ik_attempted"], gst["ik_converged"])


@pytest.mark.gpu
def test_bad_sets_and_offsets_are_refused(tabletop):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 50)
    starts, xyz = scenes.tabletop_queries(2)
    recs = api.pose_goals(xyz, params.xyz_tolerance)
    bad_tol = recs.copy()
    bad_tol["xyz_tolerance"][1, 0] = np.nan
    bad_type = recs.copy()
    bad_type["type"][1] = 7
    big = np.repeat(recs[:1], api.MAX_GOAL_SET + 1)
    cases = [(recs, [0, 1, 1]),                     # an empty set
             (recs, [0, 2, 1]),                     # decreasing offsets
             (recs, [1, 1, 2]),                     # not from 0
             (np.concatenate([big, recs[1:]]), [0, len(big), len(big) + 1]),   # above the bound
             (bad_tol, [0, 1, 2]), (bad_type, [0, 1, 2])]
    for records, offsets in cases:
        with pytest.raises(api.SmplGpuError):
            api.plan_batch(ctx, scene, tables, params, starts, (records, np.asarray(offsets, np.int32)))
    # the device entry point checks the same
    L = api.gpu_lib()
    L.smplgpu_lattice_begin_goal_sets.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [C.c_int]
    sl = np.zeros(2, np.int32)
    q = np.ascontiguousarray(starts, np.float64)
    gd = np.zeros(2, np.int32)
    for records, offsets in cases:
        records = np.ascontiguousarray(records)
        off = np.asarray(offsets, np.int32)
        r = L.smplgpu_lattice_begin_goal_sets(ctx.h, sl.ctypes.data, q.ctypes.data, gd.ctypes.data,
                                              records.ctypes.data, off.ctypes.data, 2)
        assert r == SMPLGPU_ERR_INVALID, offsets
    # the contexts still plan afterwards
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, api.goal_sets([recs[:1], recs[1:]]), max_concurrent=2)
    assert len(got) == 2 and all("reached_goal" in g for g in got)
