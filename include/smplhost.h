/*
 * smplhost.h -- flat C entry points of the host-side C++ library
 * (smpl_b200/host): the model builder that produces the tables of smplgpu.h
 * from a robot description, and the adapter objects that mirror the reference's
 * plugin interfaces.  Used by the Python plumbing (tests, bench.py) via ctypes;
 * a C++ caller would use the classes in smpl_b200/host/ directly.
 */
#ifndef SMPLHOST_H
#define SMPLHOST_H

#include <stdint.h>

#include "smplgpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smplhost_tables smplhost_tables;

const char* smplhost_last_error(void);

/* ---- model builder (RobotCollisionModel::init + CollisionSpace::init, collision_space.cpp:649-739) ---- */
smplhost_tables* smplhost_tables_load(const char* robot_path);
void smplhost_tables_destroy(smplhost_tables* h);
int smplhost_tables_configure(smplhost_tables* h, const char* group, const char* planning_joints_csv);
/* CollisionSpace::setJointPosition (collision_space.cpp:166-183) for non-planning variables */
int smplhost_tables_set_joint(smplhost_tables* h, const char* variable, double value);
/* CollisionSpace::setAllowedCollisionMatrix with the description's acm records (call_planner.cpp:441-1527, 1631) */
int smplhost_tables_use_file_acm(smplhost_tables* h);
int smplhost_tables_set_acm_entry(smplhost_tables* h, const char* a, const char* b, int allowed);
/* AttachedBodiesCollisionModel::attachBody with a ready spheres model (attached_bodies_collision_model.cpp:70-141) */
int smplhost_tables_attach_spheres(smplhost_tables* h, const char* id, const char* link,
                                   const double* centers, int n, double radius);
/* AttachedBodiesCollisionModel::attachBody for a box (attached_bodies_collision_model.cpp:94-160, 264-309): the
 * sphere model is generated as the reference does -- surface voxels of the shape at 0.025 / sqrt(2) with the voxel
 * origin at zero (voxelised on the device, smplgpu_voxelize_mesh), one sphere of radius 0.025 per voxel.  pose3x4:
 * the box in the frame of `link`.  Returns the number of spheres, negative on error. */
int smplhost_tables_attach_box(smplhost_tables* h, smplgpu_ctx* ctx, const char* id, const char* link,
                               const double size[3], const double* pose3x4);
int smplhost_tables_detach(smplhost_tables* h, const char* id);
/* KDLRobotModel::init + setPlanningLink + setKinematicsToPlanningTransform (kdl_robot_model.cpp:59-171) */
int smplhost_tables_set_planning_chain(smplhost_tables* h, const char* root, const char* tip,
                                       const char* planning_link, const double* T_kin_to_planning /*[12] or NULL*/,
                                       const double* xyz_offset /*[3] or NULL*/);
/* A planning chain over a subset of the planning variables (the project's own rule; KDLRobotModel, and so
 * smplhost_tables_set_planning_chain, refuses such models): every movable joint of the root -> tip chain must be a
 * planning variable, at any index and in any order; planning variables off the chain are allowed and move collision
 * geometry only (their limits are configure's).  The planning link must be a segment of the chain.  When the planning
 * variables are exactly the chain's movable joints in chain order, the tables equal those of
 * smplhost_tables_set_planning_chain.  Returns 0, or -1 with smplhost_last_error set. */
int smplhost_tables_set_planning_chain_subset(smplhost_tables* h, const char* root, const char* tip,
                                              const char* planning_link, const double* T_kin_to_planning /*[12] or NULL*/,
                                              const double* xyz_offset /*[3] or NULL*/);
int smplhost_tables_dof(smplhost_tables* h);
int smplhost_tables_limits(smplhost_tables* h, double* mins, double* maxs, uint8_t* continuous);
const smplgpu_robot_desc* smplhost_tables_desc(smplhost_tables* h);
/* smplgpu_set_robot(ctx, desc) */
int smplhost_tables_apply(smplhost_tables* h, smplgpu_ctx* ctx);
/* world-frame voxels of out-of-group links (SelfCollisionModelImpl::updateGroup, self_collision_model.cpp:616-760) */
int smplhost_tables_outside_voxels(smplhost_tables* h, const double** xyz);
/* inspection, for parity tests against the oracle's tables */
int smplhost_tables_node_table(smplhost_tables* h, double* out /*[n][8]*/, int max_nodes);
int smplhost_tables_motion_weights(smplhost_tables* h, double* weights, int32_t* types);
int smplhost_tables_pairs(smplhost_tables* h, int32_t* out /*[n][2]*/, int max_pairs);

/* ---- batched planner: many ARA* searches on the manipulation lattice in lock step, one device call per
 * round (smpl_b200/host/batch_planner.h; mirrors ManipLattice::GetSuccs + ARAStar::improvePath,
 * manip_lattice.cpp:219-313, arastar.cpp:486-568).  The OPEN lists and the lattice stay on the host. ---- */
typedef struct smplhost_plan_params
{
    int dof;
    const double* resolutions;      /* [dof] lattice discretisation (pr2_right_arm.yaml:1-8) */
    const double* mprims;           /* [n_prims][dof] deltas in radians, file order; converses are added */
    const uint8_t* short_flags;     /* [n_prims] 1 = short-distance primitive */
    int n_prims;
    int use_short_dist;
    double short_dist_thresh;       /* metres (pr2_right_arm.yaml:16) */
    double epsilon;                 /* ARA* initial epsilon (call_planner.cpp:1729) */
    int max_expansions;
    double xyz_tolerance[3];        /* XYZ_GOAL tolerance (call_planner.cpp:93-96) */
    int cost_per_cell;
    double inflation_radius;        /* planning_link_sphere_radius (call_planner.cpp:1715) */
    const double* var_min;          /* [dof] KDLRobotModel limits */
    const double* var_max;
    const uint8_t* var_continuous;
    double origin[3];               /* grid geometry (OccupancyGrid), for the goal cell */
    double res;
    int dims[3];
    int n_threads;                  /* host threads for the per-query work (>= 1); results do not depend on it */
    const double* prim_weights;     /* [n_prims] action weights (manip_lattice_action_space.cpp:182-190): an edge costs
                                     * (int)(1000 * weight), manip_lattice.cpp:1414-1437; NULL = 1 for every primitive */
} smplhost_plan_params;

/* Plans nq queries (starts[nq][dof], goals[nq][3]) with at most max_concurrent searches in flight.
 * summary[nq][5] = success, expansions, cost, path length, lattice states created;
 * path_ids[nq][max_path] = state ids of the path (goal state id = 0, start = 1), truncated to max_path;
 * stats[10] = rounds, edges submitted, device calls, seconds inside smplgpu_* calls, host seconds, total seconds,
 * BFS bank runs, edges resolved by the double-precision kernels, seconds of set-up device calls (bank, BFS,
 * setStart), longest single wait for a batch.
 * path_states (nullable) [nq][max_path][dof] = ManipLattice::extractPath (manip_lattice.cpp:2018-2160): the joint
 * values of every path state, the goal id replaced by the state of the first valid goal-reaching action.
 * Returns 0, or a negative smplgpu error code (smplhost_last_error() has the text). */
int smplhost_plan_batch(smplgpu_ctx* ctx, const smplhost_plan_params* params, const double* starts,
                        const double* goals, int nq, int max_concurrent, int32_t* summary, int32_t* path_ids,
                        int max_path, double* stats, double* path_states);

/* The same with one planner thread per context (the reference's threading model: one CollisionSpace per planner
 * thread): queries are dealt round-robin to n_ctx contexts, each driven by its own host thread (bound to its
 * context's device with smplgpu_bind_thread) with its own stream, BFS bank, device lattices and lock-step pipeline,
 * so the host-side OPEN-list work runs in parallel without a barrier per round.  The contexts may sit on the same
 * GPU or on DIFFERENT GPUs of the box: one process drives all eight B200s without torchrun (the field of one context
 * reaches the others with smplgpu_distance_field_dev_ptr + smplgpu_set_distance_field_dev; cudaMemcpy between peers).
 * Every context must hold the same robot and distance field.
 * stats: sums over the contexts, except the seconds entries (maximum). */
int smplhost_plan_batch_multi(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* params,
                              const double* starts, const double* goals, int nq, int max_concurrent_per_ctx,
                              int32_t* summary, int32_t* path_ids, int max_path, double* stats, double* path_states);

/* smplhost_plan_batch_multi with one GoalConstraint per query (smplgpu_goal; types may be mixed): pose goals with an
 * orientation tolerance and joint-configuration goals besides XYZ goals (params->xyz_tolerance is not read).  The
 * goal positions of all joint goals are computed in one smplgpu_planning_frame_fk call before the first query starts.
 * n_ctx = 1 is the single-context case.  An unknown goal type or a NaN or negative tolerance is SMPLGPU_ERR_INVALID
 * before anything is planned. */
int smplhost_plan_batch_goals(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* params,
                              const double* starts, const smplgpu_goal* goals, int nq, int max_concurrent_per_ctx,
                              int32_t* summary, int32_t* path_ids, int max_path, double* stats, double* path_states);

/* The snap-to-goal action (SNAP_TO_XYZ_RPY, smplgpu_lattice_set_snap) in the batched planner: an expansion within
 * dist_thresh metres of metric goal distance first tries to jump straight to the goal -- to an IK solution for a pose
 * goal, to the angles of a joint goal -- at a cost of (int)(1000 * weight) (the reference registers it with weight
 * 0.5).  enabled = 0 plans as without it. */
typedef struct smplhost_snap_params {
    int32_t enabled;
    double  dist_thresh;        /* metres, >= 0 */
    double  weight;             /* >= 0 */
    smplgpu_ik_params ik;       /* max_iterations >= 1, tolerance > 0 */
} smplhost_snap_params;
/* smplhost_plan_batch_goals with the snap action.  counters[2] (nullable): IK solves the snaps ran, and how many
 * converged (summed over the contexts).  Bad goal records or snap parameters are SMPLGPU_ERR_INVALID before anything
 * is planned. */
int smplhost_plan_batch_snap(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* params,
                             const double* starts, const smplgpu_goal* goals, int nq, int max_concurrent_per_ctx,
                             int32_t* summary, int32_t* path_ids, int max_path, double* stats, double* path_states,
                             const smplhost_snap_params* snap, int64_t* counters);
/* Goal sets: query i succeeds at a state that satisfies any record of goals[goal_offsets[i] .. goal_offsets[i + 1] - 1]
 * (1 to SMPLGPU_MAX_GOAL_SET records, types may be mixed; goal_offsets[nq + 1] non-decreasing from 0).  Its BFS
 * heuristic is seeded at the goal positions of all records; the snap action (snap nullable = off) targets the record
 * nearest to the expanded state (smplgpu_lattice_begin_goal_sets).  reached_goal[nq]: the index in the set of the
 * first record that the path's goal-reaching action satisfies, -1 when the query is unsolved.  The other outputs are
 * those of smplhost_plan_batch_snap; a set of one plans as smplhost_plan_batch_goals / _snap.  Bad sets, offsets,
 * records or snap parameters are SMPLGPU_ERR_INVALID before anything is planned. */
int smplhost_plan_batch_goal_sets(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* params,
                                  const double* starts, const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
                                  int max_concurrent_per_ctx, int32_t* summary, int32_t* path_ids, int max_path,
                                  double* stats, double* path_states, const smplhost_snap_params* snap,
                                  int64_t* counters, int32_t* reached_goal);
/* The snap actions SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY (smplgpu_lattice_set_snaps), each enabled on its own
 * with its own threshold, at one cost of (int)(1000 * weight) (weight >= 0) and with one set of IK parameters. */
typedef struct smplhost_snaps_params {
    smplgpu_snap_kinds kinds;
    double weight;
} smplhost_snaps_params;
/* smplhost_plan_batch_goal_sets with any set of snap kinds (snaps nullable = off).  counters[6] (nullable): by
 * SMPLGPU_SNAP_* kind k, counters[2 k] the IK solves that kind ran and counters[2 k + 1] how many converged (summed
 * over the contexts).  The goal action extractPath takes from an expansion is the first valid goal-reaching word (the
 * snaps in kind order, then the primitives).  smplhost_plan_batch_snap and smplhost_plan_batch_goal_sets are this call
 * with SMPLGPU_SNAP_XYZ_RPY alone.  Bad sets, offsets, records, thresholds (NaN or negative, of any kind) or IK
 * parameters are SMPLGPU_ERR_INVALID before anything is planned. */
int smplhost_plan_batch_snaps(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* params,
                              const double* starts, const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
                              int max_concurrent_per_ctx, int32_t* summary, int32_t* path_ids, int max_path,
                              double* stats, double* path_states, const smplhost_snaps_params* snaps,
                              int64_t* counters, int32_t* reached_goal);

/* ---- drop-in adapters (smpl_b200/host/gpu_adapters.h): the reference's CollisionChecker / RobotModel /
 * RobotHeuristic virtuals implemented over the C ABI.  These shims drive the C++ objects one virtual call at
 * a time, the way the reference's planner does (n = 1 per call); a C++ caller uses the classes directly. ---- */
typedef struct smplhost_adapters smplhost_adapters;
smplhost_adapters* smplhost_adapters_create(smplgpu_ctx* ctx, smplhost_tables* tables, const char* planning_link,
                                            const double origin[3], double res, const int32_t dims[3],
                                            double inflation_radius, int cost_per_cell);
void smplhost_adapters_destroy(smplhost_adapters* a);
/* smplhost::ExpansionCache behind the three adapters: given the action space's motion primitives
 * (deltas[n_prims][dof], converses included), the first virtual call about a state the adapters hold no record
 * for triggers ONE smplgpu_expand_state launch, and the ~65 calls the reference's GetSuccs + ARA* expand make about
 * that state and its successors (manip_lattice.cpp:219-313, 1511-1580; arastar.cpp:613-618) are answered from its
 * record.  n_prims = 0 switches back to one device call per virtual.  deltas = NULL only reads the counters
 * (counters[2], nullable: launches, hits). */
int smplhost_adapters_enable_expansion_cache(smplhost_adapters* a, const double* deltas, int n_prims, int64_t* counters);
/* CollisionChecker::isStateValid / isStateToStateValid (collision_checker.h:62-88): 1 valid, 0 invalid */
int smplhost_cc_is_state_valid(smplhost_adapters* a, const double* q);
int smplhost_cc_is_state_to_state_valid(smplhost_adapters* a, const double* q0, const double* q1);
/* CollisionChecker::interpolatePath: waypoints out[count][dof]; returns count, -1 on failure or overflow */
int smplhost_cc_interpolate_path(smplhost_adapters* a, const double* q0, const double* q1, double* out, int max_waypoints);
/* GpuCollisionSpace::isStatesValid / isEdgesValid (the batched entry points behind the same object) */
int smplhost_cc_is_states_valid(smplhost_adapters* a, const double* q, int n, uint8_t* valid);
int smplhost_cc_is_edges_valid(smplhost_adapters* a, const double* q0, const double* q1, int n, uint8_t* valid);
/* CollisionDistanceExtension::distanceToCollision (collision_checker.h:132-144) through getExtension: q1 = NULL is the
 * state form = CollisionSpace::collisionDistance (collision_space.cpp:496-500); with q1 the minimum over the
 * waypoints of the motion.  -1 on a missing extension. */
double smplhost_cc_distance_to_collision(smplhost_adapters* a, const double* q0, const double* q1);
/* RobotModel::checkJointLimits, ForwardKinematicsInterface::computePlanningLinkFK (robot_model.h:50-110) */
int smplhost_rm_check_joint_limits(smplhost_adapters* a, const double* q);
int smplhost_rm_compute_planning_link_fk(smplhost_adapters* a, const double* q, double* pose6);
/* RobotHeuristic::updateGoal / GetGoalHeuristic / getMetricGoalDistance (robot_heuristic.h:53-100); the state
 * is registered as a lattice state first and the heuristic is asked for by state id, as ARA* does */
int smplhost_heur_update_goal(smplhost_adapters* a, const double xyz[3]);
int smplhost_heur_goal_heuristic(smplhost_adapters* a, const double* q);
double smplhost_heur_metric_goal_distance(smplhost_adapters* a, double x, double y, double z);

/* ---- path post-processing over the batched validity path (smpl_b200/host/post_processing.h; SURVEY.md 8f row 4) ----
 * Paths are concatenated: path p = points[offsets[p] .. offsets[p+1]) rows of dof joint positions, offsets[0] = 0.
 * stats[5] (nullable) = motions checked, states checked, device calls, seconds inside smplgpu_* calls, host seconds. */
/* ShortcutPath(rm, cc, pin, pout, type) (smpl/src/post_processing.cpp:284-365) for n_paths paths at once: every
 * candidate motion (all point pairs of every path) is checked in ONE smplgpu_is_indexed_edges_valid call, then
 * shortcut::ShortcutPath (and, for type 1, DivideAndConquerShortcutPath; the cheaper result wins) runs per path.
 * type 0 = ShortcutType::JOINT_SPACE, 1 = JOINT_POSITION_VELOCITY_SPACE; continuous[dof] = !RobotModel::hasPosLimit.
 * out_idx (room for offsets[n_paths] ints) / out_offsets[n_paths+1]: the points each shortcut path keeps, as
 * indices into its input path. */
int smplhost_shortcut_paths(smplgpu_ctx* ctx, int dof, const uint8_t* continuous, const double* points,
                            const int32_t* offsets, int n_paths, int type, int32_t* out_idx, int32_t* out_offsets,
                            double* stats);
/* ShortcutPath(rm, cc, pin, pout, type) with type EUCLID_SPACE for n_paths paths at once, over the project's own
 * straight planning-link motion (smplgpu_euclid_motions; DESIGN.md section 2, parity unpinned): every motion (i, j),
 * i < j, of every path is decided in ONE smplgpu_euclid_motions call, shortcut::ShortcutPath's greedy walk (granularity
 * 1, the original segments costed by JointDistance) runs per path over the answers, and one more call returns the
 * interior IK states of the motions the walks emitted.  Output points are input points, copied bit for bit, or IK
 * states: out_points[max_points][dof], out_source[max_points] (the point's index in its input path, or -1 for an IK
 * state), out_offsets[n_paths+1], *n_out_points = the total.  SMPLGPU_ERR_LIMIT when max_points is too small (the
 * offsets and *n_out_points are written).  stats[7] (nullable) = motions decided, IK solves, IK solves converged,
 * waypoint edges checked, device calls, seconds inside smplgpu_* calls, host seconds. */
int smplhost_shortcut_paths_euclid(smplgpu_ctx* ctx, smplhost_tables* tables, const double* points, const int32_t* offsets,
                                   int n_paths, const smplgpu_euclid_params* params, double* out_points,
                                   int32_t* out_source, int max_points, int32_t* out_offsets, int32_t* n_out_points,
                                   double* stats);
/* InterpolatePath(cc, path) (post_processing.cpp:476-540) for n_paths paths at once: the waypoints of every
 * segment (CollisionChecker::interpolatePath) are checked in ONE smplgpu_is_states_valid call; a segment whose
 * waypoints are all valid is replaced by them, otherwise its end point is kept.  Returns the total number of
 * output points (written to out_points[max_points][dof], out_offsets[n_paths+1]); with out_points == NULL only
 * counts; SMPLGPU_ERR_LIMIT when max_points is too small. */
int smplhost_interpolate_paths(smplgpu_ctx* ctx, smplhost_tables* tables, const double* points, const int32_t* offsets,
                               int n_paths, double* out_points, int max_points, int32_t* out_offsets, double* stats);

/* ---- scene ingest (smpl_b200/host/scene_ingest.h; SURVEY.md 8f row 3) ----
 * Box primitives -> triangle meshes in the grid frame: geometry::CreateIndexedBoxMesh + TransformVertices
 * (smpl/src/geometry/mesh_utils.cpp:39-113, voxelize.cpp:608-615).  boxes[n_boxes][15] = length, width, height and
 * the pose as a 3x4 row-major rigid transform; vertices[8 n_boxes][3], triangles[12 n_boxes][3] (indices into the
 * concatenated vertex array).  Feed the result to smplgpu_voxelize_mesh or smplgpu_build_distance_field_from_meshes. */
int smplhost_box_meshes(const double* boxes, int n_boxes, double* vertices, int32_t* triangles);
/* The same for any primitive of voxel_operations.cpp:121-170: shapes[n_shapes][16] = kind (0 box, 1 sphere,
 * 2 cylinder, 3 cone), three dimensions (box l w h; sphere r; cylinder r length; cone r height), pose 3x4.
 * CreateIndexed{Sphere,Cylinder,Cone}Mesh (mesh_utils.cpp:116-300) with the counts VoxelizeSphere etc. use
 * (7 x 8 sphere, 16 rim points).  smplhost_shape_mesh_size gives the vertices / triangles one shape adds;
 * smplhost_shape_meshes returns the total triangle count. */
int smplhost_shape_mesh_size(int kind, int32_t* n_vertices, int32_t* n_triangles);
int smplhost_shape_meshes(const double* shapes, int n_shapes, double* vertices, int32_t* triangles);

#ifdef __cplusplus
}
#endif

#endif /* SMPLHOST_H */
