"""Pins oracle/collision_model.cpp + oracle/collision_space.cpp (SURVEY 8a rows a1-a11) against the REFERENCE's own
collision checker: sbpl_collision_checking + smpl's OccupancyGrid / EuclidDistanceMap / voxeliser compiled where they
lie under /root/reference into oracle/_ref/libref_collision.so (oracle/ref_collision_shim.cpp says what the stand-in
third-party headers do and do not pin).  Both sides are driven from the same robot description and scene:

* the distance field after the priming check (the reference has inserted the voxels of the out-of-group links by then),
* the sphere trees the reference builds (centre, radius, children, link) and the max-sphere-motion weights,
* the world position of every sphere-tree node for random states -- bit for bit,
* isStateValid / isStateToStateValid verdicts, waypoint counts and the interpolated waypoints themselves,

on the PR2 right arm (tabletop = config 1, clutter = config 2, box objects at arbitrary poses through
CollisionSpace::insertObject, padding), the UBR1 arm with a box attached through CollisionSpace::attachObject and
extra ACM entries (config 4 shape) and the 15-DOF torso + both arms group (config 5 shape, coarser grid).

tests/golden/collision_reference.npz holds outputs of that reference build with what regenerates its inputs
(tools/gen_golden_collision.py); the oracle is checked against it where oracle/_ref is absent.
"""
import os

import numpy as np
import pytest

from smpl_b200 import scenes
from helpers import make_oracle
from oracle_api import RefCollisionScene, ref_collision_lib

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "collision_reference.npz")

needs_ref = pytest.mark.skipif(ref_collision_lib() is None, reason="oracle/_ref/libref_collision.so not built")

UBR1_BOX = ((0.05, 0.05, 0.20), np.array([[1.0, 0.0, 0.0, 0.26], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0]]))


def dual_arm_coarse_scene():
    """Config 5's robot setup (torso + both arms, 15-DOF) in a 2 cm grid: the reference's 48-byte cells make the 1 cm
    grid a gigabyte."""
    full = scenes.pr2_dual_arm_scene()
    s = scenes.Scene("pr2", "torso", full.planning_joints, full.origin, full.size, 0.02, 0.2)
    s.use_desc_acm = True
    for k in range(5):
        s.add_box((1.0, 0.0, 0.3 + 0.35 * k), (0.5, 2.0, 0.02))
    s.add_box((0.55, -0.4, 0.9), (0.1, 0.1, 0.4))
    return s


def case_scene(name):
    """-> (scene, attach) for a named case; attach = (id, link, size, pose3x4) or None"""
    if name == "pr2_tabletop":
        return scenes.pr2_tabletop_scene(), None
    if name == "pr2_clutter":
        return scenes.pr2_clutter_scene(), None
    if name == "pr2_box_objects":
        return scenes.pr2_shelf_objects_scene(), None
    if name == "pr2_clutter_padded":
        s = scenes.pr2_clutter_scene()
        s.padding = 0.013
        return s, None
    if name == "ubr1_attached_box":
        s = scenes.ubr1_tabletop_scene(attach=False)
        for link in ("wrist_roll_link", "gripper_link", "left_gripper_finger_link", "right_gripper_finger_link"):
            s.acm_extra.append(("object", link, True))
        return s, ("object", "wrist_roll_link") + UBR1_BOX
    if name == "pr2_dual_arm_15dof":
        return dual_arm_coarse_scene(), None
    raise KeyError(name)


CASES = ["pr2_tabletop", "pr2_clutter", "pr2_box_objects", "pr2_clutter_padded", "ubr1_attached_box",
         "pr2_dual_arm_15dof"]


def make_reference(scene, attach):
    r = RefCollisionScene(scene.robot_path, scene.group, scene.planning_joints, scene.origin, scene.size, scene.res,
                          scene.max_dist)
    for k, v in scene.fixed_joints.items():
        assert r.set_joint(k, v) == 0
    if scene.use_desc_acm:
        r.use_desc_acm()
    for a, b, allowed in scene.acm_extra:
        r.acm_set(a, b, allowed)
    if scene.padding:
        r.set_padding(scene.padding)
    if attach is not None:
        r.attach_box(*attach)
    if len(scene.cells):
        r.add_cells(scene.cells)
    if len(scene.boxes):
        r.insert_boxes(scene.boxes)
    r.prime(np.zeros(scene.dof))
    return r


def make_restatement(scene, attach, with_kdl=False):
    o = make_oracle(scene, with_kdl=with_kdl)
    if attach is not None:
        assert o.attach_box(*attach) > 0
    return o


def case_inputs(scene, limits, n_states, n_edges, seed):
    """Random states inside `limits` (lo, hi, continuous: what the reference's model reports), lattice-sized edges plus
    long random edges (many waypoints)."""
    lo, hi, cont = limits
    q = scenes.random_states(n_states, lo, hi, cont, seed=seed)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    q0 = q[:n_edges].copy()
    q1 = q0.copy()
    half = n_edges // 2
    prim = rng.integers(-7, 8, size=(half, scene.dof)) * np.pi / 180.0        # lattice moves of up to 7 degrees
    q1[:half] += prim * (np.asarray(hi) - np.asarray(lo) > 0.5)                  # prismatic torso: stays put
    q1[half:] = q0[half:] + rng.uniform(-0.6, 0.6, size=(n_edges - half, scene.dof)) * np.minimum(1.0, (np.asarray(hi) - np.asarray(lo)))
    return q, q0, q1


def golden_inputs(g, name):
    """The states and edges the reference build checked for GOLDEN: case_inputs(seed=211) under the limits stored with
    them.  The file keeps every 50th row of q and q1 rather than all of them; those rows must come out the same."""
    scene, _ = case_scene(name)
    limits = g[name + "/limits_lo"], g[name + "/limits_hi"], g[name + "/limits_continuous"]
    q, q0, q1 = case_inputs(scene, limits, 1500, 600, seed=211)
    assert np.array_equal(q[::50], g[name + "/q_rows"]) and np.array_equal(q1[::50], g[name + "/q1_rows"]), \
        "regenerated inputs differ from the ones the reference build saw"
    return q, q0, q1


@needs_ref
@pytest.mark.parametrize("name", CASES)
def test_restatement_equals_reference_build(name):
    scene, attach = case_scene(name)
    o = make_restatement(scene, attach)
    r = make_reference(scene, attach)
    # the field both sides check against (after priming)
    assert np.array_equal(o.df_d2(), r.df_d2())
    # the trees and the interpolation weights
    nt_o, nt_r = o.node_table(), r.node_table()
    assert nt_o.shape == nt_r.shape and np.array_equal(nt_o, nt_r)
    assert np.array_equal(o.motion_weights()[0], r.motion_weights())
    q, q0, q1 = case_inputs(scene, r.limits(), 3000, 1200, seed=101)
    # FK of every sphere-tree node: bit for bit
    c_o = np.asarray(o.sphere_centers(q[:300])).reshape(300, len(nt_r), 3)
    c_r = r.sphere_centers(q[:300], len(nt_r))
    assert np.array_equal(c_o, c_r)
    # verdicts
    v_o, v_r = o.is_states_valid(q), r.is_states_valid(q)
    assert np.array_equal(v_o, v_r)
    assert 0.02 < v_o.mean() < 0.98          # the case exercises both outcomes
    e_o, n_o = o.is_edges_valid(q0, q1)
    e_r, n_r = r.is_edges_valid(q0, q1)
    assert np.array_equal(n_o, n_r)
    assert np.array_equal(e_o, e_r)
    assert n_o.max() > 5                      # the staggered check order (inc_cc = 5) is exercised
    # the waypoints themselves
    for i in (0, 1, len(q0) // 2, len(q0) - 1):
        assert np.array_equal(o.edge_waypoints(q0[i], q1[i]), r.edge_waypoints(q0[i], q1[i]))


@needs_ref
def test_detach_restores_verdicts():
    """Detaching: the reference build segfaults in the first large batch of checks after CollisionSpace::detachObject
    (stale pointers to the erased sphere model; it survives a few dozen checks), so the restatement's detach is checked
    against a reference scene that never had the body."""
    scene, attach = case_scene("ubr1_attached_box")
    o = make_restatement(scene, attach)
    r_with = make_reference(scene, attach)
    r_without = make_reference(scene, None)
    q, _, _ = case_inputs(scene, r_with.limits(), 1500, 10, seed=7)
    with_body = r_with.is_states_valid(q)
    assert np.array_equal(with_body, o.is_states_valid(q))
    assert o.detach("object") == 0
    without = r_without.is_states_valid(q)
    assert np.array_equal(without, o.is_states_valid(q))
    assert (without >= with_body).all() and (without != with_body).any()


def test_restatement_equals_golden_reference_outputs():
    """The same comparison against the committed outputs of the reference build (no oracle/_ref needed)."""
    g = np.load(GOLDEN)
    for name in CASES:
        scene, attach = case_scene(name)
        o = make_restatement(scene, attach)
        q, q0, q1 = golden_inputs(g, name)
        assert np.array_equal(o.node_table(), g[name + "/node_table"])
        n_nodes = len(g[name + "/node_table"])
        k = len(g[name + "/centers"])
        assert np.array_equal(np.asarray(o.sphere_centers(q[:k])).reshape(k, n_nodes, 3), g[name + "/centers"])
        assert np.array_equal(o.is_states_valid(q), g[name + "/states_valid"])
        e, n = o.is_edges_valid(q0, q1)
        assert np.array_equal(e, g[name + "/edges_valid"])
        assert np.array_equal(n, g[name + "/waypoint_counts"])
        assert int(o.df_d2().astype(np.int64).sum()) == int(g[name + "/df_d2_sum"])


@needs_ref
def test_shape_objects_occupy_the_cells_of_the_reference_insert_object():
    """SURVEY 8f row 3 for every primitive shape: boxes, spheres, cylinders and cones at arbitrary poses inserted through
    the reference's CollisionSpace::insertObject (VoxelizeObject -> VoxelizeShape -> geometry::Voxelize{Box,Sphere,
    Cylinder,Cone} -> addPointsToField) occupy exactly the cells that the product's host mesh builders
    (smplhost_shape_meshes = CreateIndexed*Mesh + TransformVertices) followed by the voxeliser give -- the meshes the
    device voxeliser is fed (tests/test_gpu_scene_ingest.py checks the device against the same oracle voxeliser)."""
    from smpl_b200 import api
    from oracle_api import voxelize_mesh
    from test_oracle_voxelize import random_pose
    scene = scenes.pr2_clutter_scene()
    rng = np.random.default_rng(3)
    rows = []
    for kind, dims in ((0, (0.3, 0.2, 0.1)), (1, (0.17, 0, 0)), (2, (0.09, 0.42, 0)), (3, (0.12, 0.3, 0)),
                       (1, (0.05, 0, 0)), (2, (0.2, 0.05, 0)), (3, (0.3, 0.1, 0)), (0, (0.02, 0.5, 0.5))):
        pose = random_pose(rng, 0.4)
        pose[:, 3] += (0.5, 0.0, 1.0)
        rows.append(np.concatenate([[kind], dims, pose.ravel()]))
    rows = np.array(rows)
    r = RefCollisionScene(scene.robot_path, scene.group, scene.planning_joints, scene.origin, scene.size, scene.res,
                          scene.max_dist)
    r.insert_shapes(rows)
    occupied_ref = r.df_d2() == 0
    occupied = np.zeros_like(occupied_ref)
    for row in rows:
        v, t = api.shape_meshes(row[None, :])
        g = api.world_to_grid(voxelize_mesh("oracle", v, t, scene.res, scene.origin, False), scene.origin, scene.res)
        inside = np.all((g >= 0) & (g < np.asarray(scene.dims)), axis=1)
        occupied[tuple(g[inside].T)] = True
    assert occupied_ref.sum() > 4000
    assert np.array_equal(occupied, occupied_ref)


DIST_CASES = ["pr2_tabletop", "pr2_clutter", "pr2_clutter_padded", "ubr1_attached_box", "pr2_dual_arm_15dof"]


@needs_ref
@pytest.mark.parametrize("name", DIST_CASES)
def test_collision_distance_equals_reference_build(name):
    """CollisionSpace::collisionDistance (collision_space.cpp:496-500; self_collision_model.cpp:503-531, 1386-1468): the
    order-dependent clearance descent, restated visit for visit -- equal to the reference build bit for bit, including
    its quirk (every checked sphere-tree pair contributes `return true` = 1.0, :1640-1642)."""
    scene, attach = case_scene(name)
    o = make_restatement(scene, attach)
    r = make_reference(scene, attach)
    q, _, _ = case_inputs(scene, r.limits(), 2000, 10, seed=5)
    d_o, d_r = o.collision_distance(q), r.collision_distance(q)
    assert np.array_equal(d_o, d_r)
    # a clearance of 0 is what an invalid state gets from the field term (a failing leaf has obs_dist < 0)
    v = o.is_states_valid(q)
    assert (d_o >= 0).all() and (d_o[v == 0] <= 1.0).all()


@pytest.mark.parametrize("name", DIST_CASES)
def test_collision_distance_golden_from_reference_build(name):
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "collision_distance_reference.npz"))
    scene, attach = case_scene(name)
    o = make_restatement(scene, attach)
    assert np.array_equal(o.collision_distance(g[name + "/q"]), g[name + "/distance"])
