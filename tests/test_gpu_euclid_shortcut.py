"""The EUCLID_SPACE shortcut on the device (smplgpu_euclid_motions, smplhost_shortcut_paths_euclid) against the sequential
oracle (oracle/euclid_shortcut/euclid_shortcut.cpp) and against the JOINT_SPACE shortcut.  The motion is the project's
own definition (DESIGN.md section 2), pinned oracle <-> device: step counts and IK counters equal, costs to 1e-9
relative, IK states to 1e-6 (CUDA's sin / cos / atan2 are within 2 ulp of glibc's).  An ok flag that differs must be a
documented rounding boundary -- a motion whose device states, checked by the oracle, get the device's verdict -- and
is counted."""
import numpy as np
import pytest

import euclid_shortcut_oracle as eo
from helpers import make_oracle
from smpl_b200 import api, scenes

pytestmark = pytest.mark.gpu

ONE_STEP = api.EuclidParams(max_step_m=1e9, max_step_rad=1e9)


@pytest.fixture(scope="module")
def clutter():
    scene = scenes.pr2_clutter_scene()
    ctx, tables = api.setup_context(scene)
    o = make_oracle(scene)
    yield scene, o, ctx, tables
    ctx.close()


@pytest.fixture(scope="module")
def tabletop():
    scene = scenes.pr2_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    yield scene, o, ctx, tables
    ctx.close()


def wandering_paths(tables, ctx, n_paths, seed, max_len=40):
    """Joint-space paths of mixed quality: random walks of small steps, straight lines between random states cut into
    pieces with jitter, detours, and degenerate ones (test_gpu_postprocessing.py's generator)."""
    lo, hi, cont = tables.limits()
    rng = np.random.default_rng(seed)
    paths = []
    q = scenes.random_states(4 * n_paths, lo, hi, cont, seed=seed)
    valid = ctx.is_states_valid(q).astype(bool)
    anchors = q[valid]
    for p in range(n_paths):
        n = int(rng.integers(3, max_len))
        a, b = anchors[rng.integers(0, len(anchors), 2)]
        kind = p % 3
        if kind == 0:
            steps = rng.normal(0.0, 0.06, (n, tables.dof))
            steps[rng.random(n) < 0.15] = 0.0
            pts = a + np.cumsum(steps, axis=0)
        elif kind == 1:
            t = np.linspace(0.0, 1.0, n)[:, None]
            pts = a + t * (b - a) * 0.5 + rng.normal(0.0, 0.02, (n, tables.dof))
        else:
            t = np.concatenate([np.linspace(0, 1, n // 2 + 1), np.linspace(1, 0.2, n - n // 2 - 1)])[:, None]
            pts = a + t * (b - a) * 0.4
        paths.append(np.ascontiguousarray(pts[:n]))
    paths.append(anchors[:1].copy())
    paths.append(anchors[:2].copy())
    paths.append(np.zeros((0, tables.dof)))
    return paths


def _all_pairs(paths):
    pts = np.concatenate([p for p in paths if len(p)])
    a, b, base = [], [], 0
    for p in paths:
        for i in range(len(p)):
            for j in range(i + 1, len(p)):
                a.append(base + i)
                b.append(base + j)
        base += len(p)
    return pts, np.asarray(a, np.int32), np.asarray(b, np.int32)


def _chain_done(r, max_steps):
    """per motion: the IK chain completed (one-step motions have none)"""
    n = r["n_steps"]
    return np.array([n[e] <= max_steps and (n[e] == 1 or not np.isnan(r["states"][e]).any()) for e in range(len(n))])


def compare_motion_table(ctx, o, scene, pts, a, b, params):
    """device vs oracle on one motion table; returns (motions, ok disagreements)"""
    params = params or api.EuclidParams()
    got = ctx.euclid_motions(pts, a, b, params, want_states=True)
    ref = eo.euclid_motions(o, scene.T_kin_to_planning, pts, a, b, params, want_states=True)
    assert np.array_equal(got["n_steps"], ref["n_steps"])
    cg, cr = _chain_done(got, params.max_steps), _chain_done(ref, params.max_steps)
    chain_diff = np.flatnonzero(cg != cr)
    # an IK chain that ends differently is a convergence one step apart: the counters may then differ by its solves
    if len(chain_diff) == 0:
        assert got["ik_solves"] == ref["ik_solves"] and got["ik_converged"] == ref["ik_converged"]
    both = cg & cr
    c1, c2 = got["cost"][both], ref["cost"][both]
    assert np.all(np.abs(c1 - c2) <= 1e-9 * np.maximum(np.abs(c2), 1e-300) + 1e-15)
    for e in np.flatnonzero(both):
        if len(got["states"][e]):
            assert np.abs(got["states"][e] - ref["states"][e]).max() <= 1e-6, e
    assert (got["cost"][~cg] == 0.0).all()
    flips = np.flatnonzero(got["ok"] != ref["ok"])
    for e in flips:
        if cg[e] != cr[e]:
            continue                                   # the IK boundary: one chain converged, the other did not
        # the edge boundary: the oracle's verdict on the device's own states is the device's
        chain = np.concatenate([pts[a[e]][None], got["states"][e], pts[b[e]][None]])
        v, _ = o.is_edges_valid(chain[:-1], chain[1:])
        assert bool(v.all()) == bool(got["ok"][e]), "motion %d: unexplained ok flag" % e
    print("%d motions, %d ok, %d IK solves; ok flags differing: %d (IK chains differing: %d)" % (
        len(a), got["ok"].sum(), got["ik_solves"], len(flips), len(chain_diff)))
    assert len(flips) <= max(2, len(a) // 500)
    return len(a), len(flips)


def compare_shortcuts(ctx, o, scene, tables, paths, params=None):
    got_pts, got_src, stats = api.shortcut_paths_euclid(ctx, tables, paths, params)
    differing = 0
    for p, gp, gs in zip(paths, got_pts, got_src):
        if len(p) == 0:
            assert len(gp) == 0 and len(gs) == 0
            continue
        rp, rs, _ = eo.shortcut_path_euclid(o, scene.T_kin_to_planning, p, params)
        if not np.array_equal(gs, rs):
            differing += 1
            continue
        keep = gs >= 0
        assert np.array_equal(gp[keep], p[gs[keep]])           # input points bit for bit
        if (~keep).any():
            assert np.abs(gp[~keep] - rp[~keep]).max() <= 1e-6
        assert np.array_equal(gp[0], p[0]) and np.array_equal(gp[-1], p[-1])
        if len(gp) > 1:
            gen = (gs[:-1] < 0) | (gs[1:] < 0)
            v, _ = ctx.is_edges_valid(gp[:-1], gp[1:])
            assert v[gen].all()
    assert differing <= max(1, len(paths) // 50), differing
    return got_pts, got_src, stats


def test_motion_table_matches_oracle_clutter(clutter):
    scene, o, ctx, tables = clutter
    paths = wandering_paths(tables, ctx, 14, seed=41, max_len=16)
    pts, a, b = _all_pairs(paths)
    compare_motion_table(ctx, o, scene, pts, a, b, None)


def test_shortcut_paths_match_oracle_clutter(clutter):
    scene, o, ctx, tables = clutter
    paths = wandering_paths(tables, ctx, 24, seed=43, max_len=20)
    got_pts, got_src, stats = compare_shortcuts(ctx, o, scene, tables, paths)
    with_ik = sum(int((s < 0).any()) for s in got_src)
    print("clutter: %d paths, %d with IK states; stats %s" % (len(paths), with_ik, stats))
    assert with_ik >= 3
    assert stats["device_calls"] == 2
    assert stats["motions"] == sum(len(p) * (len(p) - 1) // 2 for p in paths)


def test_one_step_equals_joint_space_shortcut(clutter):
    scene, o, ctx, tables = clutter
    paths = wandering_paths(tables, ctx, 30, seed=47)
    want, _ = api.shortcut_paths(ctx, tables, paths, kind=0)
    got_pts, got_src, stats = api.shortcut_paths_euclid(ctx, tables, paths, ONE_STEP)
    for p, w, gp, gs in zip(paths, want, got_pts, got_src):
        assert np.array_equal(gs, w)
        assert np.array_equal(gp, p[w])
    assert stats["ik_solves"] == 0 and stats["device_calls"] == 1


def test_planned_tabletop_paths(tabletop):
    scene, o, ctx, tables = tabletop
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 3000
    starts, goals = scenes.tabletop_queries(16, seed=13)
    got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=8, want_states=True)
    paths = [r["path_states"] for r in got if r["success"]]
    assert len(paths) >= 6
    pts, a, b = _all_pairs(paths)
    compare_motion_table(ctx, o, scene, pts, a, b, None)
    short_pts, short_src, stats = compare_shortcuts(ctx, o, scene, tables, paths)
    _, _, cont = tables.limits()
    cost = lambda q: np.where(cont.astype(bool), np.abs((np.diff(q, axis=0) + np.pi) % (2 * np.pi) - np.pi),
                              np.abs(np.diff(q, axis=0))).sum()
    for p, sp in zip(paths, short_pts):
        assert cost(sp) <= cost(p) + 1e-9
    print("tabletop: %d planned paths, %d -> %d points; stats %s" % (
        len(paths), sum(map(len, paths)), sum(map(len, short_pts)), stats))


def test_ubr1_with_attached_box():
    scene = scenes.ubr1_tabletop_scene()
    o = make_oracle(scene)
    ctx, tables = api.setup_context(scene)
    try:
        paths = wandering_paths(tables, ctx, 12, seed=53, max_len=14)
        pts, a, b = _all_pairs(paths)
        compare_motion_table(ctx, o, scene, pts, a, b, None)
        compare_shortcuts(ctx, o, scene, tables, paths)
    finally:
        ctx.close()


def test_degenerate_paths(clutter):
    scene, o, ctx, tables = clutter
    lo, hi, cont = tables.limits()
    q = scenes.random_states(64, lo, hi, cont, seed=59)
    q = q[ctx.is_states_valid(q).astype(bool)]
    paths = [np.zeros((0, tables.dof)), q[:1].copy(), q[1:3].copy(), np.repeat(q[3:4], 4, axis=0),
             np.concatenate([q[4:5], q[4:5], q[5:6], q[5:6]]), np.zeros((0, tables.dof))]
    got_pts, got_src, stats = compare_shortcuts(ctx, o, scene, tables, paths)
    assert len(got_pts[0]) == 0 and len(got_pts[-1]) == 0
    assert np.array_equal(got_src[1], [0])
    assert got_src[2][0] == 0 and got_src[2][-1] == 1
    assert np.array_equal(got_src[3], [0, 3])                  # repeated points: one zero-cost motion
    assert np.array_equal(got_pts[3], q[[3, 3]])
    empty_pts, empty_src, st = api.shortcut_paths_euclid(ctx, tables, [])
    assert empty_pts == [] and st["device_calls"] == 0


def test_batch_spanning_chunks_is_chunk_independent(clutter):
    scene, o, ctx, tables = clutter
    lo, hi, cont = tables.limits()
    q = scenes.random_states(6000, lo, hi, cont, seed=61)
    q = q[ctx.is_states_valid(q).astype(bool)][:1200]
    rng = np.random.default_rng(3)
    n = 24000
    a = rng.integers(0, len(q), n).astype(np.int32)
    b = rng.integers(0, len(q), n).astype(np.int32)
    prm = api.EuclidParams()
    big = ctx.euclid_motions(q, a, b, prm)
    steps = big["n_steps"]
    edges = int(steps[steps <= prm.max_steps].sum())
    print("%d motions, %d waypoint edges, %d IK solves" % (n, edges, big["ik_solves"]))
    assert edges > 2 * (1 << 18)                              # SMPLGPU_EUCLID_CHUNK_EDGES: three chunks or more
    solves = 0
    for s in range(0, n, 3000):
        part = ctx.euclid_motions(q, a[s:s + 3000], b[s:s + 3000], prm)
        assert np.array_equal(part["ok"], big["ok"][s:s + 3000])
        assert np.array_equal(part["cost"], big["cost"][s:s + 3000])
        assert np.array_equal(part["n_steps"], steps[s:s + 3000])
        solves += part["ik_solves"]
    assert solves == big["ik_solves"]
    compare_motion_table(ctx, o, scene, q, a[:400], b[:400], prm)


def test_states_call_repeats_the_deciding_call(clutter):
    scene, o, ctx, tables = clutter
    paths = wandering_paths(tables, ctx, 6, seed=67, max_len=12)
    pts, a, b = _all_pairs(paths)
    r1 = ctx.euclid_motions(pts, a, b, want_states=True)
    r2 = ctx.euclid_motions(pts, a[::-1], b[::-1], want_states=True)
    for e in range(len(a)):
        s1, s2 = r1["states"][e], r2["states"][len(a) - 1 - e]
        assert np.array_equal(np.isnan(s1), np.isnan(s2)) and np.array_equal(s1[~np.isnan(s1)], s2[~np.isnan(s2)])
    assert np.array_equal(r1["ok"], r2["ok"][::-1]) and np.array_equal(r1["cost"], r2["cost"][::-1])


@pytest.mark.parametrize("bad", [dict(max_step_m=0.0), dict(max_step_m=float("nan")), dict(max_step_rad=-1.0),
                                 dict(max_steps=0), dict(max_steps=5000), dict(max_iterations=0),
                                 dict(tolerance=float("nan"))])
def test_bad_parameters_and_indices_are_refused(clutter, bad):
    scene, o, ctx, tables = clutter
    q = np.zeros((2, tables.dof))
    with pytest.raises(api.SmplGpuError):
        ctx.euclid_motions(q, [0], [1], api.EuclidParams(**bad))
    with pytest.raises(api.SmplGpuError):
        ctx.euclid_motions(q, [0], [2])
    with pytest.raises(api.SmplGpuError):
        api.shortcut_paths_euclid(ctx, tables, [q], api.EuclidParams(**bad))
