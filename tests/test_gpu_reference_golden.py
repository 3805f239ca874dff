"""The CUDA path against the REFERENCE's own collision checker: tests/golden/collision_reference.npz holds verdicts and
waypoint counts for seeded states and edges (golden_inputs), produced by sbpl_collision_checking compiled from the
reference sources (oracle/_ref/libref_collision.so, tools/gen_golden_collision.py).  Everything goes through the C ABI
(smplgpu_is_states_valid / smplgpu_is_edges_valid) in both precision modes; verdicts and waypoint counts must be equal."""
import os

import numpy as np
import pytest

from smpl_b200 import api
from test_oracle_collision import CASES, GOLDEN, case_scene, golden_inputs

pytestmark = pytest.mark.gpu


def setup(scene, attach):
    ctx = api.GpuContext(0)
    tables = api.build_tables(scene)
    if attach is not None:
        body_id, link, size, pose = attach
        assert tables.attach_box(ctx, body_id, link, size, pose) > 0
        for a, b, allowed in scene.acm_extra:
            if body_id in (a, b):
                tables.set_acm_entry(a, b, allowed)
    ctx.set_robot(tables)
    cells = api.scene_cells(scene, tables)
    if len(scene.boxes):
        v, t = api.box_meshes(scene.boxes)
        ctx.build_distance_field_from_meshes(v, t, cells, scene.dims, scene.origin, scene.res, scene.max_dist,
                                             scene.padding)
    else:
        ctx.build_distance_field(cells, scene.dims, scene.origin, scene.res, scene.max_dist, scene.padding)
    return ctx


@pytest.mark.parametrize("name", CASES)
def test_cuda_verdicts_equal_reference_build(name):
    g = np.load(GOLDEN)
    scene, attach = case_scene(name)
    ctx = setup(scene, attach)
    try:
        q, q0, q1 = golden_inputs(g, name)
        for mode in (api.GpuContext.CERTIFIED_F32, api.GpuContext.EXACT_F64):
            ctx.set_precision_mode(mode)
            v = ctx.is_states_valid(q)
            # the device field is the exact transform; the reference's propagation over-estimates a few cells per
            # million on scenes with rotated objects (DESIGN.md section 2), which may flip a state whose sphere
            # centre falls into one of them
            budget = 1 if name == "pr2_box_objects" else 0
            assert int((v != g[name + "/states_valid"]).sum()) <= budget
            e, n = ctx.is_edges_valid(q0, q1)
            assert np.array_equal(n, g[name + "/waypoint_counts"])
            assert int((e != g[name + "/edges_valid"]).sum()) <= budget
    finally:
        ctx.close()


@pytest.mark.parametrize("name", ["pr2_tabletop", "ubr1_tabletop"])
def test_batch_planner_returns_the_reference_builds_plans(name):
    """smplhost_plan_batch (many ARA* searches in lock step over smplgpu_expand_batch) against
    tests/golden/plans_reference.json -- plans of the reference's own ManipLattice + BfsHeuristic + ARAStar +
    CollisionSpace + KDLRobotModel (oracle/ref_planner_shim.cpp): PR2 tabletop (config 1) and UBR1 with a box attached
    through attachObject and extra ACM entries (config 4 shape).  Same success flag, expansions, cost, lattice size
    and state-id path, whatever the concurrency."""
    import json
    from conftest import ROOT
    from test_oracle_planner_reference import plan_cases
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "plans_reference.json")))[name]
    scene, attach, params, starts, goals = plan_cases()[name]
    ctx = api.GpuContext(0)
    try:
        tables = api.build_tables(scene)
        if attach is not None:
            body_id, link, size, pose = attach
            assert tables.attach_box(ctx, body_id, link, size, pose) > 0
            for a, b, allowed in scene.acm_extra:
                if body_id in (a, b):
                    tables.set_acm_entry(a, b, allowed)
        ctx.set_robot(tables)
        ctx.build_distance_field(api.scene_cells(scene, tables), scene.dims, scene.origin, scene.res, scene.max_dist,
                                 scene.padding)
        for conc in (3, 64):
            got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=conc)
            for g, want in zip(got, gold):
                assert [int(g["success"]), g["expansions"], g["cost"], g["num_states"],
                        [int(i) for i in g["path_ids"]]] == want
    finally:
        ctx.close()


@pytest.mark.parametrize("name", ["pr2_tabletop", "pr2_clutter", "pr2_clutter_padded", "ubr1_attached_box", "pr2_dual_arm_15dof"])
def test_collision_distance_equals_the_reference_builds(name):
    """smplgpu_collision_distance = CollisionSpace::collisionDistance (collision_space.cpp:496-500): the clearance of
    1500 states per scene, bit for bit the values the reference build returned (tools/gen_golden_collision_distance.py);
    and through the adapter's CollisionDistanceExtension (collision_checker.h:132-144)."""
    g = np.load(os.path.join(os.path.dirname(GOLDEN), "collision_distance_reference.npz"))
    scene, attach = case_scene(name)
    ctx, tables = api.setup_context(scene)
    try:
        if attach is not None:
            tables.attach_box(ctx, *attach)
            tables.apply(ctx)
        q, want = g[name + "/q"], g[name + "/distance"]
        got = ctx.collision_distance(q)
        assert np.array_equal(got, want)
        ad = api.Adapters(ctx, scene, tables)
        for i in (0, 1, 2, len(q) // 2):
            assert ad.distance_to_collision(q[i]) == want[i]
        # motion form: the minimum over the waypoints of the motion
        a, b = q[3], q[3] + 0.2
        wp = ad.interpolate_path(a, b)
        assert ad.distance_to_collision(a, b) == ctx.collision_distance(wp).min()
        ad.close()
        assert len(ctx.collision_distance(np.zeros((0, scene.dof)))) == 0
    finally:
        ctx.close()
