"""Small end-to-end case for compute-sanitizer: every kernel family once, small sizes."""
import sys
sys.path.insert(0, '.'); sys.path.insert(0, 'tests')
import numpy as np
from smpl_b200 import api, scenes

scene = scenes.pr2_clutter_scene()
ctx, tables = api.setup_context(scene)
lo, hi, cont = tables.limits()
q = scenes.random_states(3000, lo, hi, cont, seed=3)
q0, q1 = scenes.mprim_edges(q)
v = ctx.is_states_valid(q)
e, c = ctx.is_edges_valid(q0, q1)
d = scenes.pr2_mprim_deltas()
e2, c2 = ctx.is_mprim_edges_valid(q, (np.arange(len(q)) % len(d)).astype(np.int32), d)
assert np.array_equal(e, e2) and np.array_equal(c, c2)
ctx.set_precision_mode(ctx.EXACT_F64)
assert np.array_equal(v, ctx.is_states_valid(q))
assert np.array_equal(e, ctx.is_edges_valid(q0, q1)[0])
ctx.set_precision_mode(ctx.CERTIFIED_F32)
ctx.fk_sphere_centers(q[:64]); ctx.fk_sphere_centers_f32(q[:64]); ctx.check_joint_limits(q); ctx.planning_frame_fk(q[:64])
ctx.bfs_set_walls_from_df(scene.inflation_radius)
ctx.bfs_run([api.world_to_grid([[0.4, -0.2, 0.8]], scene.origin, scene.res)[0]])
ctx.goal_heuristics(q[:256], 100)
# round-2 entry points: one-launch expansion records, lattice states as 16-bit coordinates, clearance
pr = scenes.PlanParams(scene.dof)
ctx.set_motion_primitives(np.concatenate([pr.mprims, -pr.mprims]))
for k in range(8):
    ctx.expand_state(q[k], 100)
ctx.set_lattice(pr.resolutions)
lc, lq = scenes.random_lattice_coords(3000, lo, hi, cont, pr.resolutions, seed=4)
assert np.array_equal(ctx.is_lattice_states_valid(lc), ctx.is_states_valid(lq))
ctx.is_lattice_edges_valid(lc, (np.arange(len(lc)) % len(d)).astype(np.uint8), d)
ctx.collision_distance(q[:256])
walls = scenes.bfs_clutter_walls(48, seed=5)
ctx.bfs_set_walls(walls); ctx.bfs_run([scenes.first_free_cell(walls, (24, 24, 24))]); ctx.bfs_download()
ctx.close()
ps = scenes.pr2_tabletop_scene()
pctx, pt = api.setup_context(ps)
pp = scenes.PlanParams(7); pp.max_expansions = 60
st, g = scenes.tabletop_queries(6, seed=13)
res, stats = api.plan_batch(pctx, ps, pt, pp, st, g, max_concurrent=4, n_threads=2)
pctx.probe_df_lookup_rate()
# the planning-link IK kernel and a round chain with the snap action
ik_seeds = st + 0.05
pctx.planning_link_ik(pctx.planning_frame_fk(st), ik_seeds)
api.plan_batch(pctx, ps, pt, pp, st, g, max_concurrent=4, snap=api.SnapParams(dist_thresh=0.2))
# the position-only IK kernel and a round chain with all three snap kinds
pctx.planning_link_ik(pctx.planning_frame_fk(st)[:, :3], ik_seeds)
rg = api.pose_goals(np.concatenate([g, np.zeros((len(g), 3))], axis=1), pp.xyz_tolerance, rpy_tolerance=0.05)
api.plan_batch(pctx, ps, pt, pp, st, rg, max_concurrent=4,
               snap=api.SnapParams(dist_thresh=0.2, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2))
# scene ingest (voxeliser + EDT) and the indexed-edge batch of path shortcutting
ictx, it = api.setup_context(scenes.pr2_shelf_objects_scene())
paths = [q[:12].copy(), q[20:40].copy()]
api.shortcut_paths(ictx, it, paths, kind=0)
ictx.close()
print("sanitize case ok:", int(v.sum()), int(e.sum()), [r["expansions"] for r in res])
