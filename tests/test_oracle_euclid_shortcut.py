"""The EUCLID_SPACE shortcut in the oracle (oracle/euclid_shortcut/euclid_shortcut.cpp): a straight, constant-rate-of-turn
motion of the planning link between two path states, followed through the planning-link IK (the project's own
definition, DESIGN.md section 2).  With one step per motion it must be the JOINT_SPACE shortcut; with the defaults its
paths keep their end points, cost no more than the input, are valid edge by edge, and its IK states lie on the
straight segment and the constant-rate turn."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import euclid_shortcut_oracle as eo
import snap_oracle
from helpers import make_oracle
from smpl_b200 import api, scenes

ONE_STEP = api.EuclidParams(max_step_m=1e9, max_step_rad=1e9)


@pytest.fixture(scope="module", params=["clutter", "tabletop"])
def scene_oracle(request):
    scene = scenes.pr2_clutter_scene() if request.param == "clutter" else scenes.pr2_tabletop_scene()
    return scene, make_oracle(scene)


def _valid(o, n, seed):
    lo, hi, cont = o.joint_limits()
    q = scenes.random_states(8 * n, lo, hi, cont, seed=seed)
    return q[o.is_states_valid(q).astype(bool)][:n]


def oracle_paths(o, n_paths, seed, max_len=14):
    """random walks of small steps around valid states, jittered straight lines between them, and detours"""
    rng = np.random.default_rng(seed)
    anchors = _valid(o, 2 * n_paths, seed)
    dof = anchors.shape[1]
    paths = []
    for p in range(n_paths):
        n = int(rng.integers(3, max_len))
        a, b = anchors[rng.integers(0, len(anchors), 2)]
        if p % 3 == 0:
            steps = rng.normal(0.0, 0.05, (n, dof))
            steps[rng.random(n) < 0.15] = 0.0
            pts = a + np.cumsum(steps, axis=0)
        elif p % 3 == 1:
            t = np.linspace(0.0, 1.0, n)[:, None]
            pts = a + t * (b - a) * 0.3 + rng.normal(0.0, 0.01, (n, dof))
        else:
            t = np.concatenate([np.linspace(0, 1, n // 2 + 1), np.linspace(1, 0.2, n - n // 2 - 1)])[:, None]
            pts = a + t * (b - a) * 0.3
        paths.append(np.ascontiguousarray(pts[:n]))
    return paths


def _joint_cost(path, cont):
    d = np.diff(path, axis=0)
    d = np.where(cont.astype(bool), np.abs((d + np.pi) % (2 * np.pi) - np.pi), np.abs(d))
    return d.sum()


def _rpy_matrix(rpy):
    return Rotation.from_euler("xyz", rpy).as_matrix()


def test_one_step_motions_are_the_joint_space_shortcut(scene_oracle):
    scene, o = scene_oracle
    _, _, cont = o.joint_limits()
    shortened = 0
    for p in oracle_paths(o, 24, seed=5):
        pts, src, (solves, _) = eo.shortcut_path_euclid(o, scene.T_kin_to_planning, p, ONE_STEP)
        ref, _ = o.shortcut_path(p, cont, kind=0)
        assert solves == 0 and np.array_equal(src, ref)
        assert np.array_equal(pts, p[ref])
        shortened += len(ref) < len(p)
    assert shortened >= 5


def test_default_shortcuts_keep_ends_cost_validity_and_geometry(scene_oracle):
    scene, o = scene_oracle
    _, _, cont = o.joint_limits()
    prm = api.EuclidParams()
    with_ik, checked = 0, 0
    for p in oracle_paths(o, 18, seed=9):
        valid_in = o.is_edges_valid(p[:-1], p[1:])[0].all()
        pts, src, _ = eo.shortcut_path_euclid(o, scene.T_kin_to_planning, p, prm)
        assert np.array_equal(pts[0], p[0]) and np.array_equal(pts[-1], p[-1])
        assert src[0] == 0 and src[-1] == len(p) - 1
        keep = src >= 0
        assert np.array_equal(pts[keep], p[src[keep]])          # input points copied bit for bit
        assert _joint_cost(pts, cont) <= _joint_cost(p, cont) + 1e-9
        # every generated edge is valid; an original step is kept as it was
        ok, _ = o.is_edges_valid(pts[:-1], pts[1:])
        gen = (src[:-1] < 0) | (src[1:] < 0)
        assert ok[gen].all()
        if valid_in:
            assert ok.all()
        # IK states: on the straight segment and the constant-rate turn between the input points around them
        inputs = np.flatnonzero(keep)
        for a, b in zip(inputs[:-1], inputs[1:]):
            if b - a < 2:
                continue
            with_ik += 1
            n = b - a
            fa, fb, fk = o.planning_frame_fk(pts[a]), o.planning_frame_fk(pts[b]), o.planning_frame_fk(pts[a + 1:b])
            Ra, Rb = _rpy_matrix(fa[0, 3:]), _rpy_matrix(fb[0, 3:])
            w = Rotation.from_matrix(Rb @ Ra.T).as_rotvec()
            for k in range(1, n):
                alpha = k / n
                tp = fa[0, :3] + alpha * (fb[0, :3] - fa[0, :3])
                assert np.abs(fk[k - 1, :3] - tp).max() <= 2e-6
                tR = Rotation.from_rotvec(alpha * w).as_matrix() @ Ra
                err = Rotation.from_matrix(_rpy_matrix(fk[k - 1, 3:]) @ tR.T).magnitude()
                assert err <= 1e-5
                checked += 1
    assert with_ik >= 3 and checked >= 10


def test_zero_length_and_pure_rotation_motions(scene_oracle):
    scene, o = scene_oracle
    q = _valid(o, 8, seed=13)
    T = scene.T_kin_to_planning
    r = eo.euclid_motions(o, T, q, np.arange(8), np.arange(8))
    assert (r["n_steps"] == 1).all() and (r["cost"] == 0.0).all() and r["ik_solves"] == 0
    # a pure rotation: the same position, the orientation turned by 0.35 rad about the planning frame's z axis
    pose = o.planning_frame_fk(q)
    turned = 0
    for i in range(len(q)):
        R = Rotation.from_rotvec([0.0, 0.0, 0.35]).as_matrix() @ _rpy_matrix(pose[i, 3:])
        target = np.concatenate([pose[i, :3], Rotation.from_matrix(R).as_euler("xyz")])[None]
        qb, ok, _ = snap_oracle.planning_link_ik(o, T, target, q[i:i + 1])
        if not ok[0]:
            continue
        r = eo.euclid_motions(o, T, np.concatenate([q[i:i + 1], qb]), [0], [1], want_states=True)
        assert r["n_steps"][0] == 4                            # ceil(0.35 / max_step_rad); the distance is ~1e-6 m
        if r["ik_solves"] == 3 and r["ik_converged"] == 3 and not np.isnan(r["states"][0]).any():
            fk = o.planning_frame_fk(r["states"][0])
            assert np.abs(fk[:, :3] - pose[i, :3]).max() <= 2e-6   # the position stays put
            turned += 1
    assert turned >= 1


def test_refusals_joint_limits_and_step_bound(scene_oracle):
    scene, o = scene_oracle
    T = scene.T_kin_to_planning
    q = _valid(o, 60, seed=17)
    a, b = np.arange(0, 60, 2), np.arange(1, 60, 2)
    # more than max_steps steps: refused before any IK solve
    few = api.EuclidParams(max_steps=3)
    r = eo.euclid_motions(o, T, q, a, b, few)
    long_ = r["n_steps"] == 4
    assert long_.sum() >= 10 and not r["ok"][long_].any() and (r["cost"][long_] == 0.0).all()
    assert eo.euclid_motions(o, T, q, a[long_], b[long_], few)["ik_solves"] == 0
    # a refusal with every solve converged is a joint-limit refusal
    limit_refused = 0
    for i, j in zip(a, b):
        m = eo.euclid_motions(o, T, q, [i], [j])
        if m["n_steps"][0] <= 256 and m["ik_solves"] > 0 and m["ik_solves"] == m["ik_converged"] and m["cost"][0] == 0.0:
            assert not m["ok"][0]
            limit_refused += 1
    print("joint-limit refusals: %d of %d" % (limit_refused, len(a)))
    assert limit_refused >= 1


@pytest.mark.parametrize("bad", [dict(max_step_m=0.0), dict(max_step_m=float("nan")), dict(max_step_rad=-0.1),
                                 dict(max_step_rad=float("inf")), dict(max_steps=0), dict(max_steps=5000),
                                 dict(max_iterations=0), dict(tolerance=0.0), dict(tolerance=float("nan"))])
def test_bad_parameters_are_rejected(scene_oracle, bad):
    scene, o = scene_oracle
    q = _valid(o, 2, seed=19)
    with pytest.raises(ValueError):
        eo.euclid_motions(o, scene.T_kin_to_planning, q, [0], [1], api.EuclidParams(**bad))
    with pytest.raises(ValueError):
        eo.shortcut_path_euclid(o, scene.T_kin_to_planning, q, api.EuclidParams(**bad))


def test_out_of_range_indices_are_rejected(scene_oracle):
    scene, o = scene_oracle
    q = _valid(o, 2, seed=19)
    with pytest.raises(ValueError):
        eo.euclid_motions(o, scene.T_kin_to_planning, q, [0], [2])
    with pytest.raises(ValueError):
        eo.euclid_motions(o, scene.T_kin_to_planning, q, [-1], [1])
