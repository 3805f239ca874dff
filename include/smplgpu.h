/*
 * smplgpu.h -- C ABI of the B200-native validity + heuristic hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 * Every entry point names the reference interface (file:line under the
 * dyouakim/smpl tree) it replaces.  The reference itself has no FFI -- its
 * boundary is three pure-virtual C++ plugin classes (smpl/collision_checker.h:48,
 * smpl/heuristic/robot_heuristic.h:53, smpl/robot_model.h:50-110); the adapter
 * classes in smpl_b200/host/ implement those virtuals by calling this ABI and
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - return 0 on success, a negative SMPLGPU_ERR_* code on failure;
 *     smplgpu_last_error() gives the message.  There is NO CPU fallback: with
 *     no CUDA device smplgpu_create() fails.
 *   - a context is single-threaded and non-reentrant, like the reference's
 *     CollisionSpace (collision_space.cpp:741-774); use one context per
 *     planner thread / per GPU.
 *   - "host" pointers are ordinary process memory; entry points ending in
 *     _dev take device pointers valid on the context's device and enqueue on
 *     the context's stream without synchronising.
 *   - joint states are row-major double[n][dof] in planning-variable order
 *     (RobotState = std::vector<double>, smpl/types.h:67).
 */
#ifndef SMPLGPU_H
#define SMPLGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMPLGPU_OK               0
#define SMPLGPU_ERR_INVALID     -1  /* bad argument */
#define SMPLGPU_ERR_CUDA        -2  /* CUDA runtime error */
#define SMPLGPU_ERR_STATE       -3  /* robot / distance field / BFS grid not set */
#define SMPLGPU_ERR_NO_DEVICE   -4  /* no usable CUDA device */
#define SMPLGPU_ERR_LIMIT       -5  /* table exceeds a compiled-in limit */

#define SMPLGPU_MAX_DOF 16          /* planning variables */

/* BFS_3D cell values (smpl/bfs3d/bfs3d.h:50-51) */
#define SMPLGPU_BFS_WALL          0x7FFFFFFF
#define SMPLGPU_BFS_UNDISCOVERED  (-1)
/* returned by smplgpu_bfs_distances for out-of-bounds cells (undefined
 * behaviour in the reference, bfs3d.cpp:373-378 indexes node -1) */
#define SMPLGPU_BFS_OUT_OF_BOUNDS (-2)
/* RobotHeuristic::Infinity (smpl/heuristic/robot_heuristic.h:62) */
#define SMPLGPU_HEURISTIC_INFINITY 32767

/* How the validity kernels compute (smplgpu_set_precision_mode).  Verdicts are identical in both modes:
 * CERTIFIED_F32 decides in single precision only what is provably unaffected by the single-precision
 * error and resolves the rest with the double-precision kernels; EXACT_F64 uses those alone. */
/* Which wavefront kernel runs BFS_3D (smplgpu_bfs_set_mode); distances are identical. */
#define SMPLGPU_BFS_TILES  0   /* 8 levels per grid barrier on shared-memory tiles (bfs_tiles.cuh): latency-bound grids */
#define SMPLGPU_BFS_LEVELS 1   /* one level per grid barrier, sparse (row, word) items (bfs.cuh): throughput-bound grids */
#define SMPLGPU_BFS_AUTO   2   /* default: the tile kernel (bank runs queued asynchronously: one launch per super-step) */

#define SMPLGPU_PRECISION_CERTIFIED_F32 0   /* default */
#define SMPLGPU_PRECISION_EXACT_F64     1

/* joint transform selector: which function the reference would pick
 * (robot_collision_model.cpp:331-359, 382-407; transform_functions.h:95-258) */
enum {
    SMPLGPU_JOINT_FIXED = 0,
    SMPLGPU_JOINT_REVOLUTE_X = 1,
    SMPLGPU_JOINT_REVOLUTE_Y = 2,
    SMPLGPU_JOINT_REVOLUTE_Z = 3,
    SMPLGPU_JOINT_REVOLUTE_AXIS = 4,   /* origin * AngleAxis(q, axis) */
    SMPLGPU_JOINT_PRISMATIC = 5        /* origin * Translate(0, 0, q) */
};

/* planning variable kind, for interpolation / motion bound
 * (robot_motion_collision_model.h:224-249, .cpp:371-407) */
enum {
    SMPLGPU_VAR_REVOLUTE = 0,
    SMPLGPU_VAR_CONTINUOUS = 1,
    SMPLGPU_VAR_PRISMATIC = 2
};

/* KDL-style chain segment joint kind (orocos_kdl Joint::None/RotAxis/TransAxis) */
enum {
    SMPLGPU_SEG_NONE = 0,
    SMPLGPU_SEG_ROT = 1,
    SMPLGPU_SEG_TRANS = 2
};

/*
 * Flat robot tables.  They restate, as arrays, what the reference keeps in
 * RobotCollisionModel / RobotCollisionState / RobotMotionCollisionModel /
 * SelfCollisionModelImpl for ONE collision group and ONE set of planning
 * variables.  All 3x4 transforms are row-major double[12] (rotation | translation).
 *
 * Links: only the links whose pose depends on a planning variable AND that
 * carry (or lead to) a sphere tree of the group, in topological order (parents
 * first).  A link whose parent is not in the table has link_parent = -1 and
 * link_base = the (constant) world pose of its parent link.
 *   T_link = T_parent * joint_fn(origin, axis, value)       robot_collision_state.h:385-431
 * value = q[link_var] when link_var >= 0, else link_const.
 *
 * Nodes: every node of every sphere tree of the group (robot links first, then
 * attached bodies), CollisionSphereModelTree order (base_collision_models.cpp:337-444).
 *   pos = T_link * center                                   robot_collision_state.h:560-581
 * A group link that no planning variable moves is listed as a link with
 * link_parent = -1, SMPLGPU_JOINT_FIXED, identity origin and link_base = its pose
 * (base * identity is exact in IEEE arithmetic).
 */
typedef struct smplgpu_robot_desc {
    int32_t dof;

    int32_t n_links;
    const int32_t* link_parent;      /* [n_links] */
    const int32_t* link_joint;       /* [n_links] SMPLGPU_JOINT_* */
    const double*  link_origin;      /* [n_links][12] */
    const double*  link_axis;        /* [n_links][3] */
    const int32_t* link_var;         /* [n_links] planning variable index or -1 */
    const double*  link_const;       /* [n_links] */
    const double*  link_base;        /* [n_links][12], used when link_parent < 0 */

    int32_t n_nodes;
    const int32_t* node_link;        /* [n_nodes] index into the link table */
    const double*  node_center;      /* [n_nodes][3] */
    const double*  node_radius;      /* [n_nodes] */
    const int32_t* node_left;        /* [n_nodes] node index or -1 */
    const int32_t* node_right;       /* [n_nodes] */

    int32_t n_trees;
    const int32_t* tree_root;        /* [n_trees] node index; checked against the distance field */

    /* sphere-tree pairs checked for self collision
     * (SelfCollisionModelImpl::m_checked_*_spheres_states, self_collision_model.cpp:1233-1345) */
    int32_t n_pairs;
    const int32_t* pair_a;           /* [n_pairs] tree index */
    const int32_t* pair_b;           /* [n_pairs] */

    /* leaf pairs whose *sphere names* have an ALWAYS entry in the ACM
     * (self_collision_model.cpp:1133-1149); normally empty */
    int32_t n_allowed_leaf_pairs;
    const int32_t* allowed_leaf_a;   /* node index */
    const int32_t* allowed_leaf_b;

    /* per planning variable */
    const int32_t* var_type;         /* [dof] SMPLGPU_VAR_* */
    const double*  var_motion_weight;/* [dof] ||MR_center|| + MR_radius of the variable's joint */
    const double*  var_min;          /* [dof] KDLRobotModel min_limits_ (kdl_robot_model.cpp:276-318) */
    const double*  var_max;          /* [dof] */

    /* planning-link forward kinematics chain (KDLRobotModel, kdl_robot_model.cpp:400-423):
     * pose = T_kin_to_planning * prod_{i < n_segments} ( joint_pose_i(q) * seg_f_tip_i ) */
    int32_t n_segments;              /* number of segments multiplied (= the planning link's segment index) */
    const int32_t* seg_kind;         /* [n_segments] SMPLGPU_SEG_* */
    const double*  seg_axis;         /* [n_segments][3] */
    const double*  seg_origin;       /* [n_segments][3] */
    const double*  seg_f_tip;        /* [n_segments][12] */
    const int32_t* seg_var;          /* [n_segments] planning variable or -1 */
    const double*  T_kin_to_planning;/* [12] */
    double xyz_offset[3];            /* GoalConstraint::xyz_offset (manip_lattice.cpp:2297-2312) */

    /* the first n_robot_trees trees belong to robot links, the rest to attached bodies (0 = all of them are robot
     * trees).  Only smplgpu_collision_distance tells them apart: the reference's clearance query covers the robot's
     * trees alone (self_collision_model.cpp:1497-1510). */
    int32_t n_robot_trees;
} smplgpu_robot_desc;

typedef struct smplgpu_ctx smplgpu_ctx;

/* ---- context -------------------------------------------------------------- */
smplgpu_ctx* smplgpu_create(int device);              /* NULL when no device; see smplgpu_last_error(NULL) */
void         smplgpu_destroy(smplgpu_ctx* ctx);
const char*  smplgpu_last_error(const smplgpu_ctx* ctx);
int          smplgpu_device(const smplgpu_ctx* ctx);
/* make the context's device current for the calling host thread (a new thread starts on device 0); call once
 * from every thread that will use the context.  One context per planner thread, as in the reference. */
int          smplgpu_bind_thread(smplgpu_ctx* ctx);
/* run on an externally owned cudaStream_t (e.g. torch's current stream); NULL = the context's own stream */
int          smplgpu_set_stream(smplgpu_ctx* ctx, void* cuda_stream);
int          smplgpu_synchronize(smplgpu_ctx* ctx);
/* number of kernels this context has launched since creation */
int64_t      smplgpu_launch_count(const smplgpu_ctx* ctx);

/* ---- scene state ---------------------------------------------------------- */
/* replaces CollisionSpace::init + RobotCollisionModel/State tables (collision_space.cpp:689-739) */
int smplgpu_set_robot(smplgpu_ctx* ctx, const smplgpu_robot_desc* desc);

/* OccupancyGrid::addPointsToField / removePointsFromField (smpl/src/occupancy_grid.cpp:357-410) ->
 * DistanceMap::addPointsToMap / removePointsFromMap (smpl/include/smpl/distance_map/detail/distance_map.hpp:305-367)
 * on the resident field: `n` cells (grid coordinates; cells outside the grid are ignored, as the reference ignores
 * points outside the map) enter / leave the obstacle set -- set semantics, like the reference: adding an obstacle cell
 * or removing a free one changes nothing.  The obstacle set is the field's own cells at distance 0, so this works on
 * a field uploaded with smplgpu_set_distance_field* as well as on one built here.  Where the reference propagates the
 * change through its bucket queues, the device recomputes the exact transform of the changed set (0.4 ms at 100^3,
 * 10 ms at 18 M cells): the result is the field smplgpu_build_distance_field would build for that set.  BFS walls
 * derived from the field have to be derived again (smplgpu_bfs_set_walls_from_df / smplgpu_bfs_bank_create), as after
 * any change of the field.  Returns 0. */
int smplgpu_distance_field_add_cells(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n);
int smplgpu_distance_field_remove_cells(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n);

/* replaces the read side of OccupancyGrid / DistanceMap (occupancy_grid.h:233-237,
 * distance_map.hpp:281-300, 520-536).  d2 = integer squared cell distance to the
 * nearest obstacle or border cell, capped at dmax_sq, unpadded nx*ny*nz,
 * x-major / z-fastest like Grid3 (detail/grid.hpp:361-366).  padding is
 * SelfCollisionModel's sphere padding (self_collision_model.cpp:394-397). */
int smplgpu_set_distance_field(smplgpu_ctx* ctx, const uint16_t* d2, int nx, int ny, int nz,
                               const double origin[3], double res, int dmax_sq, double padding);
int smplgpu_set_distance_field_dev(smplgpu_ctx* ctx, const uint16_t* d2_dev, int nx, int ny, int nz,
                                   const double origin[3], double res, int dmax_sq, double padding);
/* build the field on the device from occupied cells (x,y,z triples, effective grid
 * coordinates): exact Euclidean transform incl. border-as-obstacle, capped.
 * "next" row f1 (distance_map.hpp:305-328, 728-762) */
int smplgpu_build_distance_field(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n_cells,
                                 int nx, int ny, int nz, const double origin[3], double res,
                                 double max_dist, double padding);
/* ---- scene ingest on the device (SURVEY.md section 8f row 3) ---- */
/* geometry::VoxelizeMesh(vertices, triangles, res[, voxel_origin], voxels, fill = false)
 * (smpl/src/geometry/voxelize.cpp:962-1054; VoxelizeTriangle, geometry/detail/voxelize.hpp:45-181): the surface
 * voxels of a triangle mesh, vertices[n_vertices][3], triangles[n_triangles][3].  voxel_origin != NULL: cells centred
 * on voxel_origin + i res (PivotVoxelGrid, what the world / attached-body models use); NULL: on (i + 1/2) res
 * (HalfResVoxelGrid, robot link meshes).  voxels[max_voxels][3] receives the voxel centres in the reference's
 * ExtractVoxels order; returns the number of voxels found (which may exceed max_voxels).  Every collision-model
 * caller of the reference passes fill = false (voxel_operations.cpp:319-401), so ScanFill is not built. */
int smplgpu_voxelize_mesh(smplgpu_ctx* ctx, const double* vertices, int n_vertices, const int32_t* triangles,
                          int n_triangles, double res, const double* voxel_origin /*nullable*/, double* voxels,
                          int max_voxels);
/* WorldCollisionModel::insertObject for a whole scene (world_collision_model.cpp:193-234) + the distance field:
 * the meshes (all objects concatenated, already in the grid frame) are voxelised with the grid origin as voxel
 * origin, their voxel centres go through OccupancyGrid::addPointsToField (occupancy_grid.cpp:357-382), the extra
 * cells (e.g. the robot's out-of-group link voxels) are added, and the field is built as by
 * smplgpu_build_distance_field.  Nothing but the vertices and triangles crosses the bus. */
int smplgpu_build_distance_field_from_meshes(smplgpu_ctx* ctx, const double* vertices, int n_vertices,
                                             const int32_t* triangles, int n_triangles, const int32_t* cells_xyz,
                                             int n_cells, int nx, int ny, int nz, const double origin[3], double res,
                                             double max_dist, double padding);
int smplgpu_download_distance_field(smplgpu_ctx* ctx, uint16_t* d2_out);
/* device pointer + byte size of the resident field, for a torch.distributed broadcast */
int smplgpu_distance_field_dev_ptr(smplgpu_ctx* ctx, void** ptr, int64_t* bytes);

/* Room for an nx*ny*nz field on the device WITHOUT contents, so that a peer's field can be received straight into
 * it (one NCCL broadcast per scene update, SURVEY.md section 8e: no host hop, no staging copy); follow with
 * smplgpu_set_distance_field_dev(ctx, *ptr, ...), which then adopts the buffer in place. */
int smplgpu_reserve_distance_field(smplgpu_ctx* ctx, int nx, int ny, int nz, void** ptr, int64_t* bytes);
/* Pin the field in L2 with an access-policy window on the context's current stream (on = 1) or drop the window
 * (on = 0): for fields of tens of MB (the 36 MB 1 cm field of BASELINE config 4) while hundreds of MB of states
 * stream through the same cache.  set_aside_mb (nullable) receives the persisting carve-out. */
int smplgpu_set_distance_field_l2_persistence(smplgpu_ctx* ctx, int on, double* set_aside_mb);

/* ---- validity (CollisionChecker) ------------------------------------------ */
/* CollisionSpace::isStateValid batched (collision_space.cpp:532-536 -> 479-488);
 * verdict[i] = 1 valid / 0 invalid */
int smplgpu_is_states_valid(smplgpu_ctx* ctx, const double* q, int n, uint8_t* verdict);
int smplgpu_is_states_valid_dev(smplgpu_ctx* ctx, const double* q_dev, int n, uint8_t* verdict_dev);
/* CollisionSpace::isStateToStateValid batched (collision_space.cpp:538-581);
 * waypoint_counts may be NULL */
int smplgpu_is_edges_valid(smplgpu_ctx* ctx, const double* q0, const double* q1, int n,
                           uint8_t* verdict, int32_t* waypoint_counts);
int smplgpu_is_edges_valid_dev(smplgpu_ctx* ctx, const double* q0_dev, const double* q1_dev, int n,
                               uint8_t* verdict_dev, int32_t* waypoint_counts_dev);
/* CollisionSpace::collisionDistance batched (collision_space.cpp:496-500 -> SelfCollisionModelImpl::collisionDistance,
 * self_collision_model.cpp:503-531, 1386-1468): the reference's clearance estimate per state, in metres -- the
 * order-dependent branch-and-bound descent of the robot's sphere trees against the field (bound halves at every
 * sphere that undercuts it), restated visit for visit; out[i] equals the reference build's value bit for bit
 * (including its quirk: the sphere-pair term contributes the constant 1.0, DESIGN.md). */
int smplgpu_collision_distance(smplgpu_ctx* ctx, const double* q, int n, double* out);
/* kernel (1) alone: sphere centres of every tree node, double out[n][n_nodes][3]
 * (RobotCollisionState::updateSphereStates, robot_collision_state.h:546-581) */
int smplgpu_fk_sphere_centers(smplgpu_ctx* ctx, const double* q, int n, double* out);
/* KDLRobotModel::checkJointLimits batched (kdl_robot_model.cpp:210-235, 326-337) */
int smplgpu_check_joint_limits(smplgpu_ctx* ctx, const double* q, int n, uint8_t* ok);
/* counters of the last validity call: DF lookups performed, sphere pairs tested, waypoints checked */
int smplgpu_last_validity_stats(smplgpu_ctx* ctx, int64_t* df_lookups, int64_t* pair_tests, int64_t* waypoints);

/* ---- BFS heuristic (BFS_3D + BfsHeuristic) -------------------------------- */
/* BfsHeuristic::syncGridAndBfs (bfs_heuristic.cpp:331-353): wall iff getDistance(cell) <= radius.
 * Returns the wall count (>= 0) or a negative error. */
int smplgpu_bfs_set_walls_from_df(smplgpu_ctx* ctx, double inflation_radius);
/* BFS_3D(nx,ny,nz) + setWall (bfs3d.cpp:40-111, 132-141); walls: 1 byte per cell, x fastest */
int smplgpu_bfs_set_walls(smplgpu_ctx* ctx, int nx, int ny, int nz, const uint8_t* walls);
int smplgpu_bfs_set_walls_dev(smplgpu_ctx* ctx, int nx, int ny, int nz, const uint8_t* walls_dev);
/* BFS_3D::run (bfs3d.cpp:156-201; multi-seed bfs3d.h:157-211).  Synchronous on the
 * stream; returns the number of seeds that were in bounds, or a negative error. */
int smplgpu_bfs_run(smplgpu_ctx* ctx, const int32_t* seeds_xyz, int n_seeds);
/* BFS_3D::getDistance for a list of cells (bfs3d.cpp:373-378) */
int smplgpu_bfs_distances(smplgpu_ctx* ctx, const int32_t* cells_xyz, int n, int32_t* out);
/* the whole padded grid, int32[(nz+2)][(ny+2)][(nx+2)], x fastest (bfs3d.h:213-220) */
int smplgpu_bfs_download(smplgpu_ctx* ctx, int32_t* padded_grid);
int smplgpu_bfs_dims(smplgpu_ctx* ctx, int32_t dims[3]);
/* number of level-synchronous sweeps the last run needed */
int smplgpu_bfs_last_levels(smplgpu_ctx* ctx);
/* BfsHeuristic::GetGoalHeuristic batched (bfs_heuristic.cpp:148-163, 355-366):
 * planning-link FK + target offset + worldToGrid + cost_per_cell * distance */
int smplgpu_goal_heuristics(smplgpu_ctx* ctx, const double* q, int n, int cost_per_cell, int32_t* h);
int smplgpu_goal_heuristics_dev(smplgpu_ctx* ctx, const double* q_dev, int n, int cost_per_cell, int32_t* h_dev);
/* ForwardKinematicsInterface::computePlanningLinkFK + getTargetOffsetPose: double pose6[n][6] */
int smplgpu_planning_frame_fk(smplgpu_ctx* ctx, const double* q, int n, double* pose6);

/* The same for edges given the way ManipLattice::GetSuccs produces them -- a parent state and a motion primitive
 * (ManipLatticeActionSpace::applyMotionPrimitive, manip_lattice_action_space.cpp:575-610): edge i goes from q0[i]
 * to q0[i] + deltas[prim_id[i]] (deltas[n_prims][dof]; an id outside [0, n_prims) means a zero-length edge).  The
 * successor is formed on the device with the same single IEEE addition per joint the host would do, so only the
 * parents and one int per edge cross the bus. */
int smplgpu_is_mprim_edges_valid(smplgpu_ctx* ctx, const double* q0, const int32_t* prim_id, int n,
                                 const double* deltas, int n_prims, uint8_t* verdict, int32_t* waypoint_counts);
/* isStateToStateValid for n edges between rows of ONE point table: edge e runs from points[idx_a[e]] to
 * points[idx_b[e]] (points[n_points][dof]).  Path post-processing asks for many motions between the points of a
 * path (JointPositionShortcutPathGenerator, post_processing.cpp:99-121; shortcut.hpp:112-283): the points cross
 * the bus once and an edge costs 8 bytes. */
int smplgpu_is_indexed_edges_valid(smplgpu_ctx* ctx, const double* points, int n_points, const int32_t* idx_a,
                                   const int32_t* idx_b, int n, uint8_t* verdict, int32_t* waypoint_counts /*nullable*/);

int smplgpu_bfs_set_mode(smplgpu_ctx* ctx, int mode);

/* ---- precision control / certification (no counterpart in the reference) ---- */
int smplgpu_set_precision_mode(smplgpu_ctx* ctx, int mode);
/* bound on |sphere centre (float) - sphere centre (double)| in metres and on the grid-coordinate error in cells;
 * returns 1 when the single-precision model is in use for this scene, 0 when the scene falls back to double */
int smplgpu_certified_bounds(smplgpu_ctx* ctx, double* e_pos, double* eps_cells);
/* items (states / edges) of the last validity call that the double-precision kernels had to resolve */
int smplgpu_last_f64_resolved(smplgpu_ctx* ctx, int64_t* items);
/* Diagnostic (bench.py's roofline): independent random lookups per second this device sustains on the loaded distance
 * field (one 32-byte sector each, field cache resident) -- the ceiling of the validity kernels' dependent lookups.
 * New API, nothing in the reference corresponds to it. */
int smplgpu_probe_df_lookup_rate(smplgpu_ctx* ctx, double* lookups_per_s);
/* sphere centres as the single-precision path computes them, float out[n][n_nodes][3] (error-bound test) */
int smplgpu_fk_sphere_centers_f32(smplgpu_ctx* ctx, const double* q, int n, float* out);

/* ---- many queries at once (batched GetSuccs; SURVEY.md section 8f row 2) ---- */
/* A bank of n_slots BfsHeuristic instances over the current distance field: one BFS_3D per
 * planning query (each query has its own goal => its own BFS, bfs_heuristic.cpp:83-101).
 * The slots are stacked along z in ONE padded grid, so a single wavefront launch runs every
 * slot's search at once.  Returns the wall count of one slot. */
int smplgpu_bfs_bank_create(smplgpu_ctx* ctx, int n_slots, double inflation_radius);
/* Largest n_slots smplgpu_bfs_bank_create accepts for the current distance field: the stacked grid keeps the
 * reference's `int` node indices (bfs3d.h:213-220), so slots * padded cells must stay below 2^31, and the
 * bank must fit in the free device memory.  Callers clamp their concurrency to it. */
int smplgpu_bfs_bank_max_slots(smplgpu_ctx* ctx);
/* BFS_3D::run for every slot: seeds_xyz[n_slots][3]; a slot whose seed is out of bounds is left undiscovered */
int smplgpu_bfs_bank_run(smplgpu_ctx* ctx, const int32_t* seeds_xyz);
/* The same for n listed slots only (slots[n], seeds_xyz[n][3]); the other slots keep their distances, so a
 * finished query's slot can be handed to the next query while the rest keep searching */
int smplgpu_bfs_bank_run_slots(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, int n);
/* The same without waiting: the run is queued on a stream of its own and the call returns, so expansion batches of
 * the OTHER slots keep flowing while the newly admitted queries' BFS runs (BFS_3D runs in a background thread in the
 * reference too, bfs3d.cpp:156-201).  One run in flight per context; the listed slots must not be read
 * (smplgpu_expand_batch*, smplgpu_bfs_bank_distances) before smplgpu_bfs_bank_run_done returns 1 or
 * smplgpu_bfs_bank_run_wait returns.  smplgpu_bfs_bank_run_done: 1 finished / nothing in flight, 0 still running. */
int smplgpu_bfs_bank_run_slots_async(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz, int n);
/* The two above with any number of seeds per slot (BFS_3D::run(begin, end), bfs3d.h:157-211, every seed of the list
 * committed): slot slots[i] is seeded at seeds_xyz[seed_offsets[i] .. seed_offsets[i + 1] - 1][3].  seed_offsets[n + 1]
 * is non-decreasing from 0.  Seeds outside the grid are dropped; a slot with none has no goal cell.  Returns the
 * number of seeds inside the grid (the synchronous form) or n (the asynchronous one). */
int smplgpu_bfs_bank_run_slots_multi(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz,
                                     const int32_t* seed_offsets, int n);
int smplgpu_bfs_bank_run_slots_multi_async(smplgpu_ctx* ctx, const int32_t* slots, const int32_t* seeds_xyz,
                                           const int32_t* seed_offsets, int n);
int smplgpu_bfs_bank_run_done(smplgpu_ctx* ctx);
int smplgpu_bfs_bank_run_wait(smplgpu_ctx* ctx);
/* BFS_3D::getDistance(cell) of slot[i] */
int smplgpu_bfs_bank_distances(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* cells_xyz, int n, int32_t* out);
/* One ManipLattice::GetSuccs worth of device work for MANY expansions at once
 * (manip_lattice.cpp:219-313, 1511-1580; manip_lattice_action_space.cpp:385-396; arastar.cpp:613-618):
 * for edge i from q0[i] to q1[i] of the query that owns bank slot[i]:
 *   verdict[i]         CollisionSpace::isStateToStateValid(q0, q1)
 *   h[i]               BfsHeuristic::GetGoalHeuristic of q1 (cost_per_cell * BFS distance at the target-offset pose cell)
 *   goal_dist_cells[i] BFS_3D distance at the planning link cell of q1 (WALL when out of bounds), i.e.
 *                      getMetricGoalDistance / resolution (bfs_heuristic.cpp:127-138)
 *   offset_xyz[i][3]   computePlanningFrameFK(q1) position, for ManipLattice::isGoal */
int smplgpu_expand_batch(smplgpu_ctx* ctx, const double* q0, const double* q1, const int32_t* slot, int n,
                         int cost_per_cell, uint8_t* verdict, int32_t* h, int32_t* goal_dist_cells,
                         double* offset_xyz);

/* edges of all expansion batches so far that the double-precision kernels had to resolve */
int64_t smplgpu_expand_batch_resolved(const smplgpu_ctx* ctx);
/* Size the batch buffers for up to max_n edges once (device allocations synchronise the whole device, which
 * stalls every other context's stream: do it before the planners start, not while they run). */
int smplgpu_expand_batch_reserve(smplgpu_ctx* ctx, int max_n);
/* The same in two halves, so the host can prepare / absorb one batch while the device works on another:
 * submit copies the inputs and queues the work on the context's stream and returns at once; wait blocks until
 * that batch is done and copies the results out (returns n).  buffer = 0 .. SMPLGPU_EXPAND_BUFFERS - 1: that many
 * batches may be in flight (they run in submission order on the context's stream). */
#define SMPLGPU_EXPAND_BUFFERS 4
int smplgpu_expand_batch_submit(smplgpu_ctx* ctx, const double* q0, const double* q1, const int32_t* slot, int n,
                                int cost_per_cell, int buffer);
int smplgpu_expand_batch_wait(smplgpu_ctx* ctx, int buffer, uint8_t* verdict, int32_t* h, int32_t* goal_dist_cells,
                              double* offset_xyz);

/* ---- the lattice of many concurrent queries, resident on the device ---- */
/* What ManipLattice::GetSuccs does besides the edge check -- apply the active motion primitives, joint limits,
 * stateToCoord, getOrCreateState (the coordinate hash table), isGoal -- and the per-successor GetGoalHeuristic run on
 * the device for every query in flight (manip_lattice.cpp:219-313, 1263-1356, 1511-1580, 1673-1687;
 * manip_lattice_action_space.cpp:376-449, 662-691; arastar.cpp:613-618).  A round ships 8 bytes per expansion (bank
 * slot, state id) and returns one word pair per successor.  State ids are handed out in the reference's creation
 * order (id 0 = the goal state, 1 = the start state), so the host's ARA* -- OPEN list and search states indexed by
 * these ids -- returns the reference's paths, costs and expansion counts.  One lattice per BFS bank slot. */
typedef struct smplgpu_lattice_params {
    const double*  resolutions;      /* [dof] ManipLattice::init discretisation (manip_lattice.cpp:125-139) */
    const double*  deltas;           /* [n_prims][dof], converses included, table order */
    const uint8_t* prim_short;       /* [n_prims] 1 = short-distance primitive */
    int32_t n_prims;
    int32_t use_short_dist;
    double  short_dist_thresh;       /* metres (mprimActive, manip_lattice_action_space.cpp:674-687) */
    double  xyz_tolerance[3];        /* GoalConstraint::xyz_tolerance */
    int32_t cost_per_cell;
    int32_t max_states;              /* room per query; a query creates at most 2 + expansions * stride states */
} smplgpu_lattice_params;
#define SMPLGPU_LATTICE_GOAL_FLAG (1 << 30)   /* in a successor word: the action reaches the goal region */
#define SMPLGPU_LATTICE_SHORT_FLAG (1 << 29)  /* in a count word: the expansion applied the short-distance primitives */
/* largest n_slots smplgpu_lattice_create can hold in the free device memory */
int smplgpu_lattice_max_slots(smplgpu_ctx* ctx, int max_states);
/* returns the stride: successor words per expansion = max(#long, #short primitives) */
int smplgpu_lattice_create(smplgpu_ctx* ctx, const smplgpu_lattice_params* params, int n_slots);
/* setGoal + setStart bookkeeping for n queries: slot[i] gets an empty lattice, goal position goals_xyz[i] and start
 * state starts[i] (id 1) whose metric goal distance is start_goal_dist_cells[i] (smplgpu_expand_batch reports it).
 * The goal is an XYZ goal with the xyz_tolerance of smplgpu_lattice_params.
 * The slot's BFS (smplgpu_bfs_bank_run_slots*) must have run. */
int smplgpu_lattice_begin(smplgpu_ctx* ctx, const int32_t* slots, const double* starts,
                          const int32_t* start_goal_dist_cells, const double* goals_xyz, int n);

/* GoalConstraint (smpl/planning_params.h; smpl_b200/host/smpl/interfaces.h:49-62) and the three branches of
 * ManipLattice::isGoal (manip_lattice.cpp:1582-1696).  `pose` of a state is the target-offset planning-frame pose
 * x y z roll pitch yaw (smplgpu_planning_frame_fk).
 *   SMPLGPU_GOAL_XYZ          |pose[a] - goal.pose[a]| <= xyz_tolerance[a], a = 0, 1, 2
 *   SMPLGPU_GOAL_XYZ_RPY      the XYZ test, then theta < rpy_tolerance, where theta = normalize_angle(2 acos(q . qg)),
 *                             q and qg = AngleAxis(yaw, Z) * AngleAxis(pitch, Y) * AngleAxis(roll, X) of the state's
 *                             and of the goal's rpy, qg negated when q . qg < 0 (no clamp: |q . qg| > 1 is no goal)
 *   SMPLGPU_GOAL_JOINT_STATE  |state[i] - angles[i]| <= angle_tolerances[i] for every planning variable (no wrapping)
 * A type reads only its own fields.  The BFS heuristic is seeded at the goal position: pose[0..2], or for a joint goal
 * the target-offset position of `angles` (ManipLattice::setGoalConfiguration), which the caller computes. */
#define SMPLGPU_GOAL_XYZ          0
#define SMPLGPU_GOAL_XYZ_RPY      1
#define SMPLGPU_GOAL_JOINT_STATE  2
typedef struct smplgpu_goal {
    int32_t type;                              /* SMPLGPU_GOAL_* */
    double  pose[6];                           /* x y z roll pitch yaw (XYZ, XYZ_RPY) */
    double  xyz_tolerance[3];                  /* metres (XYZ, XYZ_RPY) */
    double  rpy_tolerance;                     /* radians (XYZ_RPY) */
    double  angles[SMPLGPU_MAX_DOF];           /* [dof] (JOINT_STATE) */
    double  angle_tolerances[SMPLGPU_MAX_DOF]; /* [dof] (JOINT_STATE) */
} smplgpu_goal;
/* smplgpu_lattice_begin with a goal record per query (types may be mixed).  The goal quaternion of an XYZ_RPY goal is
 * computed here, on the host.  An unknown type, or a NaN or negative tolerance the type reads, is SMPLGPU_ERR_INVALID. */
int smplgpu_lattice_begin_goals(smplgpu_ctx* ctx, const int32_t* slots, const double* starts,
                                const int32_t* start_goal_dist_cells, const smplgpu_goal* goals, int n);
/* Goal sets: query i accepts any record of goals[goal_offsets[i] .. goal_offsets[i + 1] - 1] (1 to
 * SMPLGPU_MAX_GOAL_SET records, types may be mixed; goal_offsets[n + 1] non-decreasing from 0).  A successor is tested
 * against the records in set order, and the first one it satisfies is its reached index: the h word of a successor
 * flagged SMPLGPU_LATTICE_GOAL_FLAG carries that index instead of a heuristic.  The slot's BFS must have been seeded at
 * the goal positions of all records (smplgpu_bfs_bank_run_slots_multi*).  The snap action (smplgpu_lattice_set_snap)
 * targets the record whose goal position is nearest to the expanded state's target-offset position (squared
 * Euclidean distance, the lower index on a tie).  smplgpu_lattice_begin_goals is this call with sets of one.  Each
 * record is checked as smplgpu_lattice_begin_goals checks it; a set that is empty or larger than the bound is
 * SMPLGPU_ERR_INVALID too. */
#define SMPLGPU_MAX_GOAL_SET 64
int smplgpu_lattice_begin_goal_sets(smplgpu_ctx* ctx, const int32_t* slots, const double* starts,
                                    const int32_t* start_goal_dist_cells, const smplgpu_goal* goals,
                                    const int32_t* goal_offsets, int n);
/* One round: expansion i expands state parent_id[i] of the query in slot[i] (at most one expansion per slot and
 * round).  submit queues the work and returns; wait blocks and hands out pointers into page-locked memory valid
 * until the next submit on `buffer` (0 .. SMPLGPU_EXPAND_BUFFERS - 1):
 *   succ[i * stride + j]  id of the j-th active primitive's successor | SMPLGPU_LATTICE_GOAL_FLAG, or -1 when the
 *                         primitive is inactive, leaves the joint limits or its edge is in collision
 *   h[i * stride + j]     BfsHeuristic::GetGoalHeuristic of that successor
 *   count[i]              lattice size of the query after this expansion | SMPLGPU_LATTICE_SHORT_FLAG when word j
 *                         stands for the j-th SHORT-distance primitive (mprimActive), else the j-th long one; -1 = full */
int smplgpu_lattice_expand_submit(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* parent_id, int n, int buffer);
int smplgpu_lattice_expand_wait(smplgpu_ctx* ctx, int buffer, const int32_t** succ, const int32_t** h,
                                const int32_t** count);
/* joint values of lattice states (ManipLattice::extractPath): q_out[i] = state id[i] of slot[i] */
int smplgpu_lattice_states(smplgpu_ctx* ctx, const int32_t* slot, const int32_t* id, int n, double* q_out);

/* ---- planning-link IK and the snap-to-goal action ---- */
/* The IK of the planning link: the batched counterpart of InverseKinematicsInterface::computeIK with
 * ik_option::UNRESTRICTED.  The reference's solvers are third-party, so this IK is the project's own (DESIGN.md
 * section 2): damped least squares from the seed, q += J^T (J J^T + 1e-6 I)^-1 e, where e is the target-offset position
 * error and the rotation vector of R_goal R^T, J the planning link's geometric Jacobian at the target point (of
 * smplgpu_planning_frame_fk's chain); bounded variables are clamped to their limits, continuous ones wrapped.  A
 * problem converges when every |e_i| <= tolerance (metres / radians), within max_iterations steps. */
typedef struct smplgpu_ik_params {
    int32_t max_iterations;   /* >= 1; 100 by default */
    double  tolerance;        /* > 0; 1e-6 by default */
} smplgpu_ik_params;
/* n problems: pose6[n][6] goal poses (x y z roll pitch yaw of the target-offset frame, as smplgpu_planning_frame_fk
 * reports them), seeds[n][dof]; q_out[n][dof], ok[n] (1 = converged), iterations[n] (steps taken).  Returns the number
 * that converged; bad parameters are SMPLGPU_ERR_INVALID. */
int smplgpu_planning_link_ik(smplgpu_ctx* ctx, const double* pose6, const double* seeds, int n,
                             const smplgpu_ik_params* params, double* q_out, uint8_t* ok, int32_t* iterations);
/* The SNAP_TO_XYZ_RPY action of ManipLatticeActionSpace (manip_lattice_action_space.cpp:376-449, 507-573, 662-691):
 * when the expanded state's metric goal distance (BFS cells * resolution, the quantity of the short-distance switch)
 * is <= dist_thresh, its first successor is an IK solution for the goal pose (XYZ and XYZ_RPY goals; the full pose of
 * the record, seeded at the expanded state) or the goal's angles (JOINT_STATE goals), checked like any action.  Call
 * after smplgpu_lattice_create (which turns snaps off) and before the queries begin.  With snaps enabled, successor
 * word 0 of every expansion is the snap's (-1 when inactive, failed or invalid) and words 1 .. are the primitives'
 * (SMPLGPU_LATTICE_SHORT_FLAG keeps its meaning for them); the rounds run as a chain of kernels (SMPLGPU_LATTICE_FUSED
 * has no snap form).  Returns the stride, 1 + the primitives' (the primitives' alone when disabled);
 * SMPLGPU_ERR_LIMIT above the stride limit, SMPLGPU_ERR_INVALID for a NaN or negative threshold or bad IK parameters. */
typedef struct smplgpu_snap_params {
    int32_t enabled;
    double  dist_thresh;      /* metres */
    smplgpu_ik_params ik;
} smplgpu_snap_params;
int smplgpu_lattice_set_snap(smplgpu_ctx* ctx, const smplgpu_snap_params* params);
/* IK solves the snap actions of this context's rounds ran so far, and how many converged (running totals over the
 * snap kinds) */
int smplgpu_lattice_snap_counters(smplgpu_ctx* ctx, int64_t counters[2]);

/* The three adaptive actions of ManipLatticeActionSpace, each enabled on its own and with its own threshold (metres
 * of metric goal distance, as for smplgpu_snap_params).  Enabled kinds take successor words 0 .. k-1 in the order of
 * their indices below, before the primitives'.  Every kind of an expansion aims at the same record, the one
 * smplgpu_lattice_begin_goal_sets names, seeds its IK at the expanded state and produces nothing for a record type it
 * does not apply to:
 *   SMPLGPU_SNAP_RPY      XYZ_RPY records: the full-pose IK for the expanded state's own target-offset position (as
 *                         smplgpu_planning_frame_fk reports it) and the record's orientation -- a turn in place
 *   SMPLGPU_SNAP_XYZ      XYZ and XYZ_RPY records: the position-only IK (smplgpu_planning_link_ik_position) for the
 *                         record's position, the orientation free
 *   SMPLGPU_SNAP_XYZ_RPY  every record: smplgpu_lattice_set_snap's action (the full pose, or a joint record's angles)
 * The IK parameters are shared. */
#define SMPLGPU_SNAP_RPY      0
#define SMPLGPU_SNAP_XYZ      1
#define SMPLGPU_SNAP_XYZ_RPY  2
typedef struct smplgpu_snap_kinds {
    int32_t enabled[3];       /* by SMPLGPU_SNAP_* */
    double  dist_thresh[3];   /* metres, >= 0 (checked for disabled kinds too) */
    smplgpu_ik_params ik;
} smplgpu_snap_kinds;
/* smplgpu_lattice_set_snap for any set of kinds; smplgpu_lattice_set_snap is this call with SMPLGPU_SNAP_XYZ_RPY alone.
 * Returns the stride, the number of enabled kinds + the primitives'; SMPLGPU_ERR_LIMIT above the stride limit,
 * SMPLGPU_ERR_INVALID for a NaN or negative threshold of any kind or bad IK parameters. */
int smplgpu_lattice_set_snaps(smplgpu_ctx* ctx, const smplgpu_snap_kinds* kinds);
/* counters[2 k] / [2 k + 1]: IK solves the snap kind k (SMPLGPU_SNAP_*) ran so far, and how many converged */
int smplgpu_lattice_snap_counters_by_kind(smplgpu_ctx* ctx, int64_t counters[6]);
/* The position-only IK of the planning link: smplgpu_planning_link_ik with only the position rows -- e = the target
 * position - the target-offset position, J its 3 x dof block, q += J^T (J J^T + 1e-6 I)^-1 e by a 3 x 3 Cholesky,
 * converged when the three |e_i| <= tolerance; the orientation is free.  xyz[n][3] target positions, seeds[n][dof];
 * outputs and return value as smplgpu_planning_link_ik. */
int smplgpu_planning_link_ik_position(smplgpu_ctx* ctx, const double* xyz, const double* seeds, int n,
                                      const smplgpu_ik_params* params, double* q_out, uint8_t* ok,
                                      int32_t* iterations);

/* ---- lattice states on the wire as 16-bit coordinates ---- */
/* The real caller of the validity path, ManipLattice, holds a state as dof small integers (RobotCoord) and forms the
 * joint values with coordToState (manip_lattice.cpp:1245-1261).  These entry points take the coordinates and do
 * that on the device with the reference's expression (coord * delta, + min limit for bounded variables), so a state
 * costs 2 dof bytes on the bus instead of 8 dof, an edge one more byte (its motion primitive).  Verdicts equal
 * smplgpu_is_states_valid / smplgpu_is_mprim_edges_valid on coordToState(coords); arbitrary (off-lattice) states keep
 * using those. */
/* ManipLattice::init discretisation (manip_lattice.cpp:125-139) from resolutions[dof] and the robot's limits;
 * coord_vals[dof] (nullable) receives the number of lattice values per variable */
int smplgpu_set_lattice(smplgpu_ctx* ctx, const double* resolutions, int32_t* coord_vals);
int smplgpu_is_lattice_states_valid(smplgpu_ctx* ctx, const int16_t* coords, int n, uint8_t* verdict);
/* edge i: coordToState(parent_coords[i]) -> that + deltas[prim_id[i]] (prim_id >= n_prims: zero-length edge) */
int smplgpu_is_lattice_edges_valid(smplgpu_ctx* ctx, const int16_t* parent_coords, const uint8_t* prim_id, int n,
                                   const double* deltas, int n_prims, uint8_t* verdict, int32_t* waypoint_counts);

/* ---- one expansion at a time, for UNCHANGED callers (ManipLattice::GetSuccs + ARAStar::expand) ---- */
/* The reference's search asks its plug-ins ~65 questions per expansion, one virtual call each
 * (manip_lattice_action_space.cpp:385-396; manip_lattice.cpp:1520, 1549, 1582-1640; arastar.cpp:613-618).
 * smplgpu_expand_state answers all of them for one parent state in ONE launch: for the parent (info[0]) and for
 * every successor parent + deltas[k] (info[1 + k]) of the table given to smplgpu_set_motion_primitives.  The
 * adapters of smpl_b200/host/gpu_adapters.cpp call it on a cache miss and serve the following virtual calls
 * from the record. */
typedef struct smplgpu_succ_info {
    double  state[SMPLGPU_MAX_DOF]; /* info[0]: the parent; info[1+k]: deltas[k][j] + parent[j] (one IEEE addition) */
    double  pose[6];                /* computePlanningLinkFK + getTargetOffsetPose of `state`: x y z roll pitch yaw */
    double  link_xyz[3];            /* position of the planning link itself (what getMetricGoalDistance is given) */
    int32_t h;                      /* BfsHeuristic::GetGoalHeuristic(state); 0 when no BFS has been set up */
    int32_t goal_dist_cells;        /* BFS_3D::getDistance at link_xyz's cell; SMPLGPU_BFS_OUT_OF_BOUNDS outside */
    int32_t waypoints;              /* waypoint count of the edge parent -> state (0 for info[0]) */
    uint8_t edge_valid;             /* isStateToStateValid(parent, state); info[0]: isStateValid(parent) */
    uint8_t limits_ok;              /* KDLRobotModel::checkJointLimits(state) */
    uint8_t state_valid;            /* info[0] only: isStateValid(parent) */
    uint8_t is_parent;              /* 1 for info[0] */
} smplgpu_succ_info;
/* the motion-primitive table, deltas[n_prims][dof] (converses included, as ManipLatticeActionSpace::addMotionPrim
 * stores them, manip_lattice_action_space.cpp:201-228); resident until replaced */
int smplgpu_set_motion_primitives(smplgpu_ctx* ctx, const double* deltas, int n_prims);
/* *info points at n_prims + 1 records in page-locked memory owned by the context, valid until the next call.
 * Uses the single BFS grid of smplgpu_bfs_run (h = 0, goal_dist_cells = WALL when none is set). */
int smplgpu_expand_state(smplgpu_ctx* ctx, const double* parent, int cost_per_cell, const smplgpu_succ_info** info);
/* changes whenever an earlier answer may no longer hold (robot tables, distance field, BFS walls or run):
 * host-side caches of smplgpu_expand_state records compare it */
int64_t smplgpu_scene_epoch(const smplgpu_ctx* ctx);

#ifdef __cplusplus
}
#endif

#endif /* SMPLGPU_H */
