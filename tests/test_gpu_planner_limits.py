"""The batched planner at the limits of its device code, against the oracle: expansions of 32 successor words (one full
warp in lattice_commit_warp, every thread of the fused lattice_round_kernel, every word of the host's absorbOne), goal
sets of 64 records, continuous joints whose stored values cross +-pi, and one step of the planning-link IK against a
float64 reference written here with numpy / scipy rather than restated from the oracle."""
import math

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import snap_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

from test_gpu_goal_sets import _assert_sets_same, _oracle_sets
from test_gpu_goal_types import _assert_same as _assert_exact
from test_gpu_goal_types import _params, _short_only, _walks
from test_gpu_ik_snap import _assert_same as _assert_snap
from test_gpu_ik_snap import SNAP, _oracle_snap, _reachable_pose_queries
from test_oracle_ik_snap import _valid_states

DEG = math.pi / 180.0
# The snap runs whose queries mostly end with a snap onto an XYZ_RPY record stop the IK at 1e-3 instead of 1e-6.  At
# 1e-6 the last step lands within ~1e-8 rad of the goal orientation, where isGoal's unclamped acos argument sits at
# 1 +- an ulp and CUDA's and glibc's sin / cos decide goal against no goal (DESIGN.md section 2): about one such snap in
# six differs, more than the allowance of these comparisons, which stays as in tests/test_gpu_ik_snap.py.  At 1e-3 the
# snapped orientations of these queries stay >= 38 ulps below 1 on the oracle.  SNAP (1e-6) is kept where few plans
# end in such a snap.
SNAP_STOP_EARLY = api.SnapParams(dist_thresh=0.2, tolerance=1e-3)


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


@pytest.fixture(scope="module")
def pr2_oracle():
    """the PR2 tabletop oracle alone, for the CPU tests"""
    scene = scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


# ---- 1. full-warp expansions ----

def _wide_params(scene, n_prims, max_expansions, with_short=False):
    """n_prims long primitives, each followed by its converse: 2 n_prims successor words.  The two-joint primitives
    come first and the single-joint ones, which are valid most often, last, so that with 16 primitives words 16-31
    carry most of the successors.  Every primitive has its own action weight (edge cost int(1000 w)), so a word read
    as the wrong primitive changes the cost.  with_short: the 7 short primitives of PlanParams as well, with the
    short-distance switch on."""
    dof = scene.dof
    multi = []
    for j in range(dof):
        v = np.zeros(dof)
        v[j], v[(j + 1) % dof] = 7.0 * DEG, (7.0 if j % 2 == 0 else -7.0) * DEG
        multi.append(v)
    v = np.zeros(dof)
    v[0], v[2] = 7.0 * DEG, 7.0 * DEG
    multi.append(v)
    single = [np.eye(dof)[j] * 7.0 * DEG for j in range(dof)] + [np.eye(dof)[1] * 3.0 * DEG]
    extra = [np.eye(dof)[3] * 3.0 * DEG]
    prims = multi[:min(8, n_prims - 8)] + single + extra[:max(0, n_prims - 16)]
    assert len(prims) == n_prims
    p = _params(scene, max_expansions)
    weights = [0.75 + 0.0625 * ((7 * k) % n_prims) for k in range(n_prims)]   # distinct, exact in binary
    flags = [0] * n_prims
    if with_short:
        short = scenes.PlanParams(dof)
        sp = short.mprims[short.short_flags == 1]
        prims += list(sp)
        flags += [1] * len(sp)
        weights += [0.5 + 0.03125 * k for k in range(len(sp))]   # below every long weight
    assert len({int(1000 * w) for w in weights}) == len(weights)
    p.mprims = np.array(prims)
    p.short_flags = np.array(flags, np.uint8)
    p.weights = weights
    p.use_short_dist = with_short
    return p


def _xyz_queries(n, seed):
    """tabletop queries: one goal under the table top (the demo's, hard: runs out of expansions) and one outside
    the grid"""
    starts, goals = scenes.tabletop_queries(n, seed=seed)
    goals[3] = (0.4, -0.2, 0.36)
    goals[7] = (5.0, 0.0, 1.0)
    return starts, goals


def _run_oracle_xyz(o, scene, params, starts, goals):
    out = []
    for s, g in zip(starts, goals):
        o.heur_init(scene.inflation_radius, scene.cost_per_cell)   # a fresh BfsHeuristic per query
        out.append(o.plan(s, g, params))
    return out


def _stride_in_use(stats, got):
    """successor words per expansion of the call: every expansion a query counts was submitted once"""
    n = sum(g["expansions"] for g in got)
    assert n > 0 and stats["edges_submitted"] % n == 0
    return stats["edges_submitted"] // n


@pytest.mark.gpu
@pytest.mark.parametrize("with_short", [False, True], ids=["long32", "long32_short14"])
def test_full_warp_expansions_match_oracle_on_one_and_three_contexts(tabletop, with_short):
    scene, o, ctx, tables = tabletop
    params = _wide_params(scene, 16, 1200, with_short)
    starts, goals = _xyz_queries(16, seed=37)
    ref = _run_oracle_xyz(o, scene, params, starts, goals)
    one, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, n_threads=2,
                                want_states=True)
    stride = _stride_in_use(stats, one)
    print("stride %d in use: %d queries, %d solved, %d expansions" % (stride, len(one), sum(a["success"] for a in ref),
                                                                      sum(a["expansions"] for a in ref)))
    assert stride == 32
    _assert_exact(ref, one)
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(2)]
    try:
        multi, _ = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=3, want_states=True)
    finally:
        for c in ctxs[1:]:
            c.close()
    _assert_exact(ref, multi)
    assert sum(a["success"] for a in ref) >= 4 and not ref[7]["success"]
    assert any(not a["success"] and a["expansions"] == params.max_expansions for a in ref)
    # the weights reach the costs: not multiples of 1000
    assert any(a["success"] and a["cost"] % 1000 != 0 for a in ref)
    # with the short set, expansions near the goal switch to its 14 words: 4-degree steps (no long primitive has one)
    short_steps = sum(int((np.abs(np.abs(np.diff(a["path_states"], axis=0)) - 4.0 * DEG) < 1e-9).any(axis=1).sum())
                      for a in ref if a["success"])
    print("4-degree (short primitive) steps on the solved paths: %d" % short_steps)
    assert (short_steps > 0) == with_short


@pytest.mark.gpu
def test_stride_limit_of_32_successor_words(tabletop):
    scene, o, ctx, tables = tabletop
    starts, goals = scenes.tabletop_queries(2, seed=39)
    with pytest.raises(api.SmplGpuError):   # 17 primitives: 34 words
        api.plan_batch(ctx, scene, tables, _wide_params(scene, 17, 50), starts, goals)
    with pytest.raises(api.SmplGpuError):   # 16 primitives and the snap: 33 words
        api.plan_batch(ctx, scene, tables, _wide_params(scene, 16, 50), starts, goals, snap=SNAP)
    got, _ = api.plan_batch(ctx, scene, tables, _wide_params(scene, 16, 50), starts, goals)   # 32 words still plan
    assert len(got) == 2


@pytest.mark.gpu
def test_fifteen_primitives_and_the_snap_match_oracle(tabletop):
    """31 words: the snap in word 0, 30 primitive words"""
    scene, o, ctx, tables = tabletop
    params = _wide_params(scene, 15, 1500)
    s_pose, g_pose = _reachable_pose_queries(o, scenes.tabletop_queries(10, seed=43)[0], 10, seed=45)
    s_joint, _ = scenes.tabletop_queries(6)
    g_joint = api.joint_goals(_walks(o, s_joint, params, 6, seed=47), 0.5 * np.asarray(params.resolutions))
    starts, goals = np.concatenate([s_pose, s_joint]), np.concatenate([g_pose, g_joint])
    ref = _oracle_snap(o, scene, params, starts, goals, SNAP)
    got, stats = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, n_threads=2,
                                want_states=True, snap=SNAP)
    stride = _stride_in_use(stats, got)
    print("stride %d in use (15 primitives + the snap)" % stride)
    assert stride == 31
    _assert_snap(ref, got, max_differing=1)
    assert sum(a["success"] for a in ref) >= 6 and stats["ik_attempted"] > 0


# ---- 2. full goal sets ----

REACHABLE = (31, 32, 63)


def _full_sets(o, params, starts, seed):
    """64 records per query, most of which fail: a position outside the grid, XYZ_RPY records whose 4 cm boxes hold
    reachable states but whose orientation is a quarter turn off (the state's quaternion is computed once and
    compared with many records), joint records half a lattice step off every joint (no lattice state within their
    0.2-step tolerance), and duplicates of these.  Query i holds reachable records at 31 (XYZ), 32 (XYZ_RPY) and 63
    (joint) by i % 4: only 31, only 32, only 63, all three; the others get a failing record."""
    n = len(starts)
    res = np.asarray(params.resolutions)
    walk = lambda k, s, p=params: _walks(o, starts, p, k, seed + s)
    wrong = []
    for k in range(31):
        pose = o.planning_frame_fk(walk(4 + k % 12, k))
        pose[:, 3] += 0.5 * math.pi
        wrong.append(api.pose_goals(pose, (0.04, 0.04, 0.04), rpy_tolerance=0.05))
    off = [api.joint_goals(walk(3 + k, 40 + k, _short_only(params)) + 0.5 * res, 0.2 * res) for k in range(16)]
    outside = api.pose_goals(np.tile([[5.0, 0.0, 1.0]], (n, 1)), params.xyz_tolerance)
    reach = [api.pose_goals(o.planning_frame_fk(walk(4, 60))[:, :3], params.xyz_tolerance),
             api.pose_goals(o.planning_frame_fk(walk(4, 61)), params.xyz_tolerance, rpy_tolerance=0.1),
             api.joint_goals(walk(3, 62, _short_only(params)), 0.5 * res)]
    sets = []
    for i in range(n):
        recs = ([outside[i]] + [w[i] for w in wrong[:16]] + [f[i] for f in off[:8]] +
                [outside[i], wrong[0][i], wrong[1][i], off[0][i], off[1][i], wrong[4][i]] +       # 25-30: duplicates
                [None, None] + [w[i] for w in wrong[16:]] + [f[i] for f in off[8:]] +
                [wrong[2][i], off[2][i], outside[i], wrong[7][i], off[5][i], wrong[9][i], wrong[3][i]] + [None])
        assert len(recs) == 64
        which = {0: (31,), 1: (32,), 2: (63,), 3: REACHABLE}[i % 4]
        for slot, r in zip(REACHABLE, reach):
            recs[slot] = r[i] if slot in which else wrong[5 + slot % 7][i]
        sets.append(np.array(recs, api.GOAL_DTYPE))
    return sets


@pytest.mark.gpu
@pytest.mark.parametrize("snap", [None, SNAP_STOP_EARLY], ids=["off", "0.2"])
def test_full_goal_sets_match_oracle(tabletop, snap):
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    starts, _ = scenes.tabletop_queries(12, seed=53)
    records, offsets = api.goal_sets(_full_sets(o, params, starts, seed=55))
    ref = _oracle_sets(o, scene, params, starts, records, offsets, snap)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=5, n_threads=2,
                            want_states=True, snap=snap)
    _assert_sets_same(ref, got, max_differing=0 if snap is None else 1)
    reached = sorted(a["reached_goal"] for a in got if a["success"])
    print("full goal sets, snap %s: reached indices %s" % ("off" if snap is None else snap.dist_thresh, reached))
    assert all((a["reached_goal"] >= 0) == a["success"] for a in got)
    if snap is None:
        assert set(REACHABLE) <= set(reached)


@pytest.mark.gpu
def test_refilled_slots_with_smaller_sets_equal_single_calls(tabletop):
    """sets of 64, 1, 17, 64, 2, ... through 3 slots: a slot that held 64 records takes a query with fewer"""
    scene, o, ctx, tables = tabletop
    params = _params(scene, 1500)
    starts, _ = scenes.tabletop_queries(10, seed=57)
    full = _full_sets(o, params, starts, seed=59)
    sizes = [64, 1, 17, 64, 2, 64, 5, 64, 1, 33]
    sets = []
    for i, k in enumerate(sizes):
        order = list(REACHABLE) + [r for r in range(64) if r not in REACHABLE]   # the reachable ones first
        sets.append(full[i] if k == 64 else full[i][order[:k]])
    records, offsets = api.goal_sets(sets)
    batch, _ = api.plan_batch(ctx, scene, tables, params, starts, (records, offsets), max_concurrent=3,
                              want_states=True)
    ref = _oracle_sets(o, scene, params, starts, records, offsets, None)
    _assert_sets_same(ref, batch)
    for i, g in enumerate(sets):
        one, _ = api.plan_batch(ctx, scene, tables, params, starts[i:i + 1], api.goal_sets([g]), max_concurrent=1,
                                want_states=True)
        a, b = one[0], batch[i]
        assert (a["success"], a["expansions"], a["cost"], a["num_states"], a["reached_goal"]) == \
               (b["success"], b["expansions"], b["cost"], b["num_states"], b["reached_goal"]), i
        assert np.array_equal(a["path_ids"], b["path_ids"]) and np.array_equal(a["path_states"], b["path_states"]), i
    print("refilled slots: set sizes %s, reached %s" % (sizes, [b["reached_goal"] for b in batch]))
    assert sum(b["success"] for b in batch) >= 4


# ---- 3. continuous joints across +-pi ----

WRAP_VALUES = (math.pi - 2.0 * DEG, -math.pi + 1.0 * DEG, math.pi, -math.pi, 3.0 * math.pi - 0.5 * DEG)


def _wrap_queries(o, scene, params, base, joints, seed):
    """starts with one continuous joint at each of WRAP_VALUES (3 pi - 0.5 deg lies outside [-pi, pi]; joint limits
    wrap it); for each a joint goal two short steps (8 deg) past the wrap on that joint, whose stored value is
    beyond +-pi (joint goals do not wrap), and a pose goal from a lattice walk started that far past the wrap"""
    starts, shifted = [], []
    for j in joints:
        for v in WRAP_VALUES:
            q = np.array(base, np.float64)
            q[j] = v
            starts.append(q)
            q2 = q.copy()
            q2[j] += math.copysign(8.0 * DEG, v)
            shifted.append((j, q2))
    starts = np.array(starts)
    res = np.asarray(params.resolutions)
    walk = _walks(o, starts, _short_only(params), 4, seed)
    angles = walk.copy()
    for k, (j, q2) in enumerate(shifted):
        angles[k, j] = q2[j] + (walk[k, j] - starts[k, j])
    g_joint = api.joint_goals(angles, 0.5 * res)
    poses = o.planning_frame_fk(_walks(o, np.array([q2 for _, q2 in shifted]), params, 10, seed + 1))
    g_pose = api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)
    return np.concatenate([starts, starts]), np.concatenate([g_joint, g_pose])


def _wrap_crossings(got, cont):
    """paths from a start inside [-pi, pi] that hold a continuous-joint value beyond +-pi, or change sign across pi
    between two states (a start at 3 pi - 0.5 deg is beyond pi without crossing anything)"""
    n = 0
    for a in got:
        p = a["path_states"][:, cont]
        if len(p) == 0 or (np.abs(p[0]) > math.pi).any():
            continue
        beyond = (np.abs(p) > math.pi).any()
        across = ((np.sign(p[1:]) != np.sign(p[:-1])) & (np.abs(p[1:]) > 0.5 * math.pi) &
                  (np.abs(p[:-1]) > 0.5 * math.pi)).any()
        n += bool(beyond or across)
    return n


def _check_wrap(scene, o, ctx, tables, base, joints, snap, max_differing, seed):
    params = _params(scene, 1200)
    starts, goals = _wrap_queries(o, scene, params, base, joints, seed)
    ref = _oracle_snap(o, scene, params, starts, goals, snap)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=6, n_threads=2,
                            want_states=True, snap=snap)
    if snap is None:
        _assert_exact(ref, got)
    else:
        _assert_snap(ref, got, max_differing=max_differing)
    _, _, cont = tables.limits()
    crossings = _wrap_crossings(got, cont.astype(bool))
    print("%s wrap, snap %s: %d queries, %d solved, %d paths cross +-pi" % (
        scene.group, "off" if snap is None else snap.dist_thresh, len(got), sum(a["success"] for a in got), crossings))
    assert sum(a["success"] for a in ref) >= len(ref) // 3
    assert crossings >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("snap", [None, SNAP_STOP_EARLY], ids=["off", "0.2"])
def test_pr2_paths_across_the_wrap_match_oracle(tabletop, snap):
    scene, o, ctx, tables = tabletop
    _check_wrap(scene, o, ctx, tables, scenes.PR2_DEMO_START, (4, 6), snap, 1, seed=63)


@pytest.mark.gpu
@pytest.mark.parametrize("snap", [None, SNAP_STOP_EARLY], ids=["off", "0.2"])
def test_ubr1_paths_across_the_wrap_match_oracle(snap):
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        _check_wrap(scene, o, ctx, tables, scenes.UBR1_DEMO_START, (4, 6), snap, 2, seed=65)
    finally:
        ctx.close()


# ---- 4. the IK step against an independent float64 reference ----

THETAS = (0.0, 1e-10, 1e-6, 0.5, 2.0, math.pi - 0.1, math.pi - 1e-3, math.pi - 1e-6)


def _rot(pose):
    return Rotation.from_euler("xyz", pose[:, 3:]).as_matrix()


def _step_problems(o, n, seed):
    """valid states with |pitch| < 1.4 (rpy -> matrix is well conditioned) and, per theta, targets at each state's
    own pose turned by theta about a random axis and moved by up to 5 cm"""
    q = _valid_states(o, 4 * n, seed)
    q = q[np.abs(o.planning_frame_fk(q)[:, 4]) < 1.4][:n]
    assert len(q) == n
    pose = o.planning_frame_fk(q)
    rng = np.random.default_rng(seed + 1)
    out = []
    for theta in THETAS:
        ax = rng.normal(size=(n, 3))
        ax /= np.linalg.norm(ax, axis=1)[:, None]
        Rt = Rotation.from_rotvec(ax * theta).as_matrix() @ _rot(pose)
        tgt = np.concatenate([pose[:, :3] + rng.uniform(-0.05, 0.05, (n, 3)), Rotation.from_matrix(Rt).as_euler("xyz")],
                             axis=1)
        out.append((theta, tgt))
    return q, out


def _reference_step(o, q, tgt):
    """one damped least-squares step, lambda = 1e-3, from FK (the oracle's planning_frame_fk), a central-difference
    Jacobian (h = 1e-6) and scipy's rotation vectors; bounded joints clamped, continuous ones wrapped.  Returns the
    new joint values for both signs of the orientation error (they differ only where its angle is pi)."""
    lo, hi, cont = o.joint_limits()
    cont = cont.astype(bool)
    h = 1e-6
    n, dof = q.shape
    J = np.zeros((n, 6, dof))
    for v in range(dof):
        a, b = q.copy(), q.copy()
        a[:, v] += h
        b[:, v] -= h
        pa, pb = o.planning_frame_fk(a), o.planning_frame_fk(b)
        J[:, :3, v] = (pa[:, :3] - pb[:, :3]) / (2 * h)
        J[:, 3:, v] = Rotation.from_matrix(_rot(pa) @ np.transpose(_rot(pb), (0, 2, 1))).as_rotvec() / (2 * h)
    pose = o.planning_frame_fk(q)
    w = Rotation.from_matrix(_rot(tgt) @ np.transpose(_rot(pose), (0, 2, 1))).as_rotvec()
    A = J @ np.transpose(J, (0, 2, 1)) + 1e-6 * np.eye(6)
    outs = []
    for sign in (1.0, -1.0):
        e = np.concatenate([tgt[:, :3] - pose[:, :3], sign * w], axis=1)
        dq = np.einsum("nrv,nr->nv", J, np.linalg.solve(A, e[:, :, None])[:, :, 0])
        q1 = q + dq
        q1[:, cont] = np.angle(np.exp(1j * q1[:, cont]))
        q1[:, ~cont] = np.clip(q1[:, ~cont], lo[~cont], hi[~cont])
        outs.append(q1)
    return outs, np.linalg.norm(w, axis=1), np.abs(outs[0] - q).max()


def _step_error(o, got, refs, angle):
    _, _, cont = o.joint_limits()
    cont = cont.astype(bool)
    errs = []
    for r in refs:
        d = got - r
        d[:, cont] = np.angle(np.exp(1j * d[:, cont]))   # continuous joints: modulo 2 pi
        errs.append(np.abs(d).max(axis=1))
    half_turn = np.abs(angle - math.pi) <= 1e-9         # either axis sign is a rotation vector of a half turn
    return np.where(half_turn, np.minimum(errs[0], errs[1]), errs[0])


def _check_ik_step(o, solve, n, seed):
    q, problems = _step_problems(o, n, seed)
    worst = 0.0
    for theta, tgt in problems:
        got = solve(tgt, q)
        refs, angle, big = _reference_step(o, q, tgt)
        err = _step_error(o, got, refs, angle)
        print("theta %.6g: largest |dq| %.3g, largest step error %.3g" % (theta, big, err.max()))
        assert err.max() <= 1e-6, (theta, err.max())
        worst = max(worst, float(err.max()))
    return worst


def test_oracle_ik_step_matches_an_independent_reference(pr2_oracle):
    scene, o = pr2_oracle
    T = scene.T_kin_to_planning
    solve = lambda tgt, q: snap_oracle.planning_link_ik(o, T, tgt, q, max_iterations=1)[0]
    print("oracle IK step: largest error %.3g" % _check_ik_step(o, solve, 200, seed=3))


@pytest.mark.gpu
def test_device_ik_step_matches_an_independent_reference(tabletop):
    scene, o, ctx, tables = tabletop
    T = scene.T_kin_to_planning

    def solve(tgt, q):
        got, ok, it = ctx.planning_link_ik(tgt, q, max_iterations=1)
        _, ok_ref, it_ref = snap_oracle.planning_link_ik(o, T, tgt, q, max_iterations=1)
        assert np.array_equal(ok, ok_ref) and np.array_equal(it, it_ref)
        return got

    print("device IK step: largest error %.3g" % _check_ik_step(o, solve, 200, seed=3))


@pytest.mark.gpu
def test_device_ik_from_far_seeds_reaches_its_targets(tabletop):
    """seeds at random valid states, not near an answer: a converged answer must be at its target by FK and scipy,
    every answer within the limits.  The ok flags are only reported: a hundred steps amplify last-bit differences
    of sin / cos between device and oracle."""
    scene, o, ctx, tables = tabletop
    n = 2048
    targets = o.planning_frame_fk(_valid_states(o, n, seed=71))
    seeds = _valid_states(o, n, seed=73)
    assert len(targets) == n and len(seeds) == n
    q, ok, it = ctx.planning_link_ik(targets, seeds)
    _, ok_ref, _ = snap_oracle.planning_link_ik(o, scene.T_kin_to_planning, targets, seeds)
    reached = o.planning_frame_fk(q[ok])
    pos = np.abs(reached[:, :3] - targets[ok, :3]).max(axis=1)
    ang = Rotation.from_matrix(_rot(targets[ok]) @ np.transpose(_rot(reached), (0, 2, 1))).magnitude()
    print("device IK from far seeds: %d problems, %d converged (oracle %d), ok flags agree on %.4f; largest position "
          "error %.3g m, angle %.3g rad" % (n, ok.sum(), ok_ref.sum(), (ok == ok_ref).mean(), pos.max(), ang.max()))
    assert ok.sum() >= n // 4
    assert pos.max() <= 1e-6 and ang.max() <= 2e-6
    lo, hi, cont = tables.limits()
    b = ~cont.astype(bool)
    assert ((q[:, b] >= lo[b]) & (q[:, b] <= hi[b])).all() and (np.abs(q[:, ~b]) <= math.pi).all()
