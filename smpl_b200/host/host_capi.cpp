// Flat C entry points over the host-side C++ (model builder + adapters) so the
// Python plumbing (tests, bench.py) can drive it with ctypes.  Declared in
// include/smplhost.h.
#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstring>
#include <memory>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../include/smplgpu.h"
#include "../../include/smplhost.h"
#include "batch_planner.h"
#include "gpu_adapters.h"
#include "post_processing.h"
#include "scene_ingest.h"
#include "robot_tables.h"

using smplhost::RobotTables;

static thread_local std::string g_err;

struct smplhost_tables
{
    RobotTables t;
    std::vector<double> voxels;
};

static std::vector<std::string> split_csv(const char* s)
{
    std::vector<std::string> out;
    std::stringstream ss(s ? s : "");
    std::string item;
    while (std::getline(ss, item, ',')) {
        if (!item.empty()) out.push_back(item);
    }
    return out;
}

extern "C" {

const char* smplhost_last_error(void) { return g_err.c_str(); }

smplhost_tables* smplhost_tables_load(const char* robot_path)
{
    std::unique_ptr<smplhost_tables> h(new smplhost_tables);
    if (!robot_path || !h->t.load(robot_path, &g_err)) {
        return nullptr;
    }
    return h.release();
}

void smplhost_tables_destroy(smplhost_tables* h) { delete h; }

int smplhost_tables_configure(smplhost_tables* h, const char* group, const char* planning_joints_csv)
{
    if (!h || !group) return -1;
    return h->t.configure(group, split_csv(planning_joints_csv), &g_err) ? 0 : -1;
}

int smplhost_tables_set_joint(smplhost_tables* h, const char* variable, double value)
{
    if (!h || !variable) return -1;
    if (!h->t.setJointPosition(variable, value)) {
        g_err = std::string("joint variable '") + variable + "' not found";
        return -1;
    }
    return 0;
}

int smplhost_tables_use_file_acm(smplhost_tables* h)
{
    if (!h) return -1;
    h->t.useFileAcm();
    return 0;
}

int smplhost_tables_set_acm_entry(smplhost_tables* h, const char* a, const char* b, int allowed)
{
    if (!h || !a || !b) return -1;
    h->t.setAcmEntry(a, b, allowed != 0);
    return 0;
}

int smplhost_tables_attach_spheres(smplhost_tables* h, const char* id, const char* link,
                                   const double* centers, int n, double radius)
{
    if (!h || !id || !link || !centers) return -1;
    if (!h->t.attachSpheres(id, link, centers, n, radius)) {
        g_err = "attach failed (unknown link, duplicate id or empty body)";
        return -1;
    }
    return 0;
}

// AttachedBodiesCollisionModel::attachBody for a box shape (attached_bodies_collision_model.cpp:94-160, 264-309):
// generateSpheresModel voxelises the shape at 0.025 / sqrt(2) with the voxel origin at zero (surface voxels) and
// puts a sphere of radius 0.025 on every voxel; the voxelisation runs on the device
int smplhost_tables_attach_box(smplhost_tables* h, smplgpu_ctx* ctx, const char* id, const char* link,
                               const double size[3], const double* pose3x4)
{
    if (!h || !ctx || !id || !link || !size || !pose3x4) return -1;
    const double object_enclosing_sphere_radius = 0.025;
    std::vector<double> vertices;
    std::vector<int32_t> triangles;
    smplhost::AppendBoxMesh(size[0], size[1], size[2], pose3x4, vertices, triangles);
    const double zero[3] = { 0.0, 0.0, 0.0 };
    const double res = object_enclosing_sphere_radius / std::sqrt(2);
    int n = smplgpu_voxelize_mesh(ctx, vertices.data(), 8, triangles.data(), 12, res, zero, nullptr, 0);
    if (n < 0) {
        g_err = smplgpu_last_error(ctx);
        return n;
    }
    std::vector<double> centers((size_t)std::max(n, 1) * 3);
    n = smplgpu_voxelize_mesh(ctx, vertices.data(), 8, triangles.data(), 12, res, zero, centers.data(), n);
    if (n < 0) {
        g_err = smplgpu_last_error(ctx);
        return n;
    }
    if (!h->t.attachSpheres(id, link, centers.data(), n, object_enclosing_sphere_radius)) {
        g_err = "attach failed (unknown link, duplicate id or empty body)";
        return -1;
    }
    return n;
}

int smplhost_tables_detach(smplhost_tables* h, const char* id)
{
    if (!h || !id) return -1;
    return h->t.detach(id) ? 0 : -1;
}

int smplhost_tables_set_planning_chain(smplhost_tables* h, const char* root, const char* tip,
                                       const char* planning_link, const double* T_kin_to_planning,
                                       const double* xyz_offset)
{
    if (!h || !root || !tip || !planning_link) return -1;
    return h->t.setPlanningChain(root, tip, planning_link, T_kin_to_planning, xyz_offset, &g_err) ? 0 : -1;
}

int smplhost_tables_dof(smplhost_tables* h) { return h ? h->t.dof() : -1; }

int smplhost_tables_limits(smplhost_tables* h, double* mins, double* maxs, uint8_t* continuous)
{
    if (!h) return -1;
    for (int i = 0; i < h->t.dof(); ++i) {
        mins[i] = h->t.varMin()[i];
        maxs[i] = h->t.varMax()[i];
        continuous[i] = (uint8_t)h->t.varContinuous()[i];
    }
    return 0;
}

const smplgpu_robot_desc* smplhost_tables_desc(smplhost_tables* h) { return h ? h->t.desc() : nullptr; }

int smplhost_tables_apply(smplhost_tables* h, smplgpu_ctx* ctx)
{
    if (!h || !ctx) return -1;
    int r = smplgpu_set_robot(ctx, h->t.desc());
    if (r != 0) {
        g_err = smplgpu_last_error(ctx);
    }
    return r;
}

int smplhost_tables_outside_voxels(smplhost_tables* h, const double** xyz)
{
    if (!h) return -1;
    h->voxels = h->t.outsideGroupVoxels();
    if (xyz) *xyz = h->voxels.data();
    return (int)(h->voxels.size() / 3);
}

/* per node: cx cy cz radius left right tree link (8 doubles), for comparison with the oracle */
int smplhost_tables_node_table(smplhost_tables* h, double* out, int max_nodes)
{
    if (!h) return -1;
    const smplgpu_robot_desc* d = h->t.desc();
    if (d->n_nodes > max_nodes) return -1;
    std::vector<int> tree_of(d->n_nodes, -1);
    for (int t = 0; t < d->n_trees; ++t) {
        std::vector<int> st(1, d->tree_root[t]);
        while (!st.empty()) {
            int n = st.back();
            st.pop_back();
            tree_of[n] = t;
            if (d->node_left[n] >= 0) {
                st.push_back(d->node_left[n]);
                st.push_back(d->node_right[n]);
            }
        }
    }
    // first node of each tree, to report children tree-relative like the oracle
    std::vector<int> first(d->n_trees, d->n_nodes);
    for (int n = 0; n < d->n_nodes; ++n) {
        if (tree_of[n] >= 0) first[tree_of[n]] = std::min(first[tree_of[n]], n);
    }
    for (int n = 0; n < d->n_nodes; ++n) {
        double* o = out + 8 * n;
        o[0] = d->node_center[3 * n]; o[1] = d->node_center[3 * n + 1]; o[2] = d->node_center[3 * n + 2];
        o[3] = d->node_radius[n];
        const int f = first[tree_of[n]];
        o[4] = d->node_left[n] < 0 ? -1 : d->node_left[n] - f;
        o[5] = d->node_right[n] < 0 ? -1 : d->node_right[n] - f;
        o[6] = tree_of[n];
        o[7] = d->node_link[n];
    }
    return d->n_nodes;
}

int smplhost_tables_motion_weights(smplhost_tables* h, double* weights, int32_t* types)
{
    if (!h) return -1;
    const smplgpu_robot_desc* d = h->t.desc();
    for (int i = 0; i < d->dof; ++i) {
        weights[i] = d->var_motion_weight[i];
        types[i] = d->var_type[i];
    }
    return 0;
}

int smplhost_tables_pairs(smplhost_tables* h, int32_t* out, int max_pairs)
{
    if (!h) return -1;
    const smplgpu_robot_desc* d = h->t.desc();
    for (int p = 0; p < d->n_pairs && p < max_pairs; ++p) {
        out[2 * p] = d->pair_a[p];
        out[2 * p + 1] = d->pair_b[p];
    }
    return d->n_pairs;
}

// goal_offsets (nullable: one goal record per query) gives each query's goal set; reached (nullable) gets each query's
// reached_goal
static int plan_batch_one(smplgpu_ctx* ctx, const smplhost_plan_params* p, const double* starts,
                          const smplgpu_goal* goals, int nq, int max_concurrent, int32_t* summary, int32_t* path_ids,
                          int max_path, double* stats, double* path_states, const smplhost_snaps_params* snaps = nullptr,
                          int64_t* counters = nullptr, const int32_t* goal_offsets = nullptr, int32_t* reached = nullptr)
{
    if (!ctx || !p || nq < 0 || (nq > 0 && (!starts || !goals || !summary))) {
        g_err = "smplhost_plan_batch: null argument";
        return SMPLGPU_ERR_INVALID;
    }
    if (p->dof <= 0 || p->n_prims < 0 || !p->resolutions || !p->var_min || !p->var_max || !p->var_continuous ||
        (p->n_prims > 0 && (!p->mprims || !p->short_flags))) {
        g_err = "smplhost_plan_batch: incomplete parameters";
        return SMPLGPU_ERR_INVALID;
    }
    smplhost::PlannerConfig cfg;
    cfg.dof = p->dof;
    cfg.resolutions.assign(p->resolutions, p->resolutions + p->dof);
    cfg.mprims.assign(p->mprims, p->mprims + (size_t)p->n_prims * p->dof);
    cfg.short_flags.assign(p->short_flags, p->short_flags + p->n_prims);
    if (p->prim_weights) cfg.prim_weights.assign(p->prim_weights, p->prim_weights + p->n_prims);
    cfg.use_short_dist = p->use_short_dist != 0;
    cfg.short_dist_thresh = p->short_dist_thresh;
    cfg.epsilon = p->epsilon;
    cfg.max_expansions = p->max_expansions;
    cfg.cost_per_cell = p->cost_per_cell;
    cfg.inflation_radius = p->inflation_radius;
    cfg.var_min.assign(p->var_min, p->var_min + p->dof);
    cfg.var_max.assign(p->var_max, p->var_max + p->dof);
    cfg.var_continuous.assign(p->var_continuous, p->var_continuous + p->dof);
    cfg.res = p->res;
    cfg.n_threads = p->n_threads > 0 ? p->n_threads : 1;
    cfg.want_path_states = path_states != nullptr;
    for (int a = 0; a < 3; ++a) {
        cfg.xyz_tolerance[a] = p->xyz_tolerance[a];
        cfg.origin[a] = p->origin[a];
        cfg.dims[a] = p->dims[a];
    }
    if (snaps) {
        for (int k = 0; k < 3; ++k) {
            cfg.snap[k] = snaps->kinds.enabled[k] != 0;
            cfg.snap_dist_thresh[k] = snaps->kinds.dist_thresh[k];
        }
        cfg.snap_weight = snaps->weight;
        cfg.ik = snaps->kinds.ik;
    }
    smplhost::BatchPlanner planner(ctx, cfg, max_concurrent);
    std::vector<smplhost::QueryResult> out;
    std::string err;
    const auto t0 = std::chrono::steady_clock::now();
    if (!planner.plan(starts, goals, goal_offsets, nq, out, &err)) {
        g_err = err;
        return SMPLGPU_ERR_CUDA;
    }
    const double total = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    for (int i = 0; i < nq; ++i) {
        const smplhost::QueryResult& r = out[i];
        summary[5 * i] = r.success ? 1 : 0;
        summary[5 * i + 1] = r.expansions;
        summary[5 * i + 2] = r.cost;
        summary[5 * i + 3] = (int)r.path_ids.size();
        summary[5 * i + 4] = r.num_states;
        if (reached) {
            reached[i] = r.reached_goal;
        }
        if (path_ids) {
            for (int k = 0; k < max_path; ++k) {
                path_ids[(size_t)i * max_path + k] = k < (int)r.path_ids.size() ? r.path_ids[k] : -1;
            }
        }
        if (path_states) {
            const size_t m = std::min(r.path_states.size(), (size_t)max_path * p->dof);
            std::copy(r.path_states.begin(), r.path_states.begin() + m, path_states + (size_t)i * max_path * p->dof);
        }
    }
    if (stats) {
        const smplhost::BatchStats& s = planner.stats();
        stats[0] = s.rounds;
        stats[1] = (double)s.edges_submitted;
        stats[2] = (double)s.device_calls;
        stats[3] = s.device_seconds;
        stats[4] = s.host_seconds;
        stats[5] = total;
        stats[6] = s.bfs_runs;
        stats[7] = (double)s.edges_resolved_f64;
        stats[8] = s.setup_seconds;
        stats[9] = s.max_wait_seconds;
    }
    if (counters) {
        for (int k = 0; k < 3; ++k) {
            counters[2 * k] = planner.stats().ik_attempted[k];
            counters[2 * k + 1] = planner.stats().ik_converged[k];
        }
    }
    return 0;
}

// one planner thread per context, queries dealt round-robin
static int plan_batch_contexts(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p, const double* starts,
                               const smplgpu_goal* goals, int nq, int max_concurrent_per_ctx, int32_t* summary,
                               int32_t* path_ids, int max_path, double* stats, double* path_states,
                               const smplhost_snaps_params* snaps = nullptr, int64_t* counters = nullptr,
                               const int32_t* goal_offsets = nullptr, int32_t* reached = nullptr)
{
    if (counters) {
        std::fill(counters, counters + 6, 0);
    }
    if (n_ctx == 1) {
        return plan_batch_one(ctxs[0], p, starts, goals, nq, max_concurrent_per_ctx, summary, path_ids, max_path, stats,
                              path_states, snaps, counters, goal_offsets, reached);
    }
    auto set_begin = [&](int i) { return goal_offsets ? goal_offsets[i] : i; };
    std::vector<std::array<int64_t, 6>> ik(n_ctx, std::array<int64_t, 6>{ { 0, 0, 0, 0, 0, 0 } });
    const int dof = p->dof;
    std::vector<int> rc(n_ctx, 0);
    std::vector<std::string> errs(n_ctx);
    std::vector<std::vector<double>> st(n_ctx, std::vector<double>(10, 0.0));
    std::vector<std::thread> threads;
    for (int t = 0; t < n_ctx; ++t) {
        threads.emplace_back([&, t]() {
            // this thread's share: queries t, t + n_ctx, ...
            std::vector<int> mine;
            for (int i = t; i < nq; i += n_ctx) mine.push_back(i);
            const int m = (int)mine.size();
            if (m == 0) {
                return;
            }
            if (smplgpu_bind_thread(ctxs[t]) != 0) {
                rc[t] = SMPLGPU_ERR_CUDA;
                errs[t] = smplgpu_last_error(ctxs[t]);
                return;
            }
            std::vector<double> s((size_t)m * dof);
            std::vector<smplgpu_goal> g;
            std::vector<int32_t> off(1, 0), got(m, -1);
            for (int k = 0; k < m; ++k) {
                std::copy(starts + (size_t)mine[k] * dof, starts + (size_t)(mine[k] + 1) * dof, s.begin() + (size_t)k * dof);
                g.insert(g.end(), goals + set_begin(mine[k]), goals + set_begin(mine[k] + 1));
                off.push_back((int32_t)g.size());
            }
            std::vector<int32_t> sum((size_t)m * 5), paths(path_ids ? (size_t)m * max_path : 0);
            const size_t ps = (size_t)max_path * dof;
            std::vector<double> pstates(path_states ? (size_t)m * ps : 0);
            smplhost_plan_params pt = *p;
            pt.n_threads = 1;
            rc[t] = plan_batch_one(ctxs[t], &pt, s.data(), g.data(), m, max_concurrent_per_ctx, sum.data(),
                                   path_ids ? paths.data() : nullptr, max_path, st[t].data(),
                                   path_states ? pstates.data() : nullptr, snaps, ik[t].data(), off.data(), got.data());
            if (rc[t] != 0) {
                errs[t] = g_err;   // thread-local: copy it out
                return;
            }
            for (int k = 0; k < m; ++k) {
                std::copy(sum.begin() + (size_t)k * 5, sum.begin() + (size_t)(k + 1) * 5, summary + (size_t)mine[k] * 5);
                if (reached) {
                    reached[mine[k]] = got[k];
                }
                if (path_ids) {
                    std::copy(paths.begin() + (size_t)k * max_path, paths.begin() + (size_t)(k + 1) * max_path,
                              path_ids + (size_t)mine[k] * max_path);
                }
                if (path_states) {
                    std::copy(pstates.begin() + (size_t)k * ps, pstates.begin() + (size_t)(k + 1) * ps,
                              path_states + (size_t)mine[k] * ps);
                }
            }
        });
    }
    for (std::thread& th : threads) {
        th.join();
    }
    for (int t = 0; t < n_ctx; ++t) {
        if (rc[t] != 0) {
            g_err = errs[t];
            return rc[t];
        }
    }
    if (counters) {
        for (int t = 0; t < n_ctx; ++t) {
            for (int k = 0; k < 6; ++k) counters[k] += ik[t][k];
        }
    }
    if (stats) {
        for (int k = 0; k < 10; ++k) stats[k] = 0.0;
        for (int t = 0; t < n_ctx; ++t) {
            for (int k : { 0, 1, 2, 6, 7 }) stats[k] += st[t][k];
            for (int k : { 3, 4, 5, 8, 9 }) stats[k] = std::max(stats[k], st[t][k]);
        }
    }
    return 0;
}

// XYZ goals with the parameters' tolerance
static std::vector<smplgpu_goal> xyz_goals(const smplhost_plan_params* p, const double* goals_xyz, int nq)
{
    std::vector<smplgpu_goal> recs(nq > 0 && goals_xyz ? nq : 0);   // zero-filled
    for (size_t i = 0; i < recs.size(); ++i) {
        recs[i].type = SMPLGPU_GOAL_XYZ;
        for (int a = 0; a < 3; ++a) {
            recs[i].pose[a] = goals_xyz[3 * i + a];
            recs[i].xyz_tolerance[a] = p->xyz_tolerance[a];
        }
    }
    return recs;
}

int smplhost_plan_batch(smplgpu_ctx* ctx, const smplhost_plan_params* p, const double* starts,
                        const double* goals, int nq, int max_concurrent, int32_t* summary, int32_t* path_ids,
                        int max_path, double* stats, double* path_states)
{
    if (!ctx || !p || nq < 0 || (nq > 0 && (!starts || !goals || !summary))) {
        g_err = "smplhost_plan_batch: null argument";
        return SMPLGPU_ERR_INVALID;
    }
    const std::vector<smplgpu_goal> recs = xyz_goals(p, goals, nq);
    return plan_batch_one(ctx, p, starts, recs.data(), nq, max_concurrent, summary, path_ids, max_path, stats, path_states);
}

int smplhost_plan_batch_multi(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p,
                              const double* starts, const double* goals, int nq, int max_concurrent_per_ctx,
                              int32_t* summary, int32_t* path_ids, int max_path, double* stats, double* path_states)
{
    if (!ctxs || n_ctx <= 0 || !p || nq < 0) {
        g_err = "smplhost_plan_batch_multi: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    if (nq > 0 && !goals) {
        g_err = "smplhost_plan_batch: null argument";
        return SMPLGPU_ERR_INVALID;
    }
    const std::vector<smplgpu_goal> recs = xyz_goals(p, goals, nq);
    return plan_batch_contexts(ctxs, n_ctx, p, starts, recs.data(), nq, max_concurrent_per_ctx, summary, path_ids,
                               max_path, stats, path_states);
}

static bool bad_tolerance(double t)
{
    return std::isnan(t) || t < 0.0;
}

// the argument and goal-record checks of smplhost_plan_batch_goals (those of smplgpu_lattice_begin_goals) of nq goal
// records, before any query starts
static int check_goal_args(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p, const smplgpu_goal* goals,
                           int nq)
{
    if (!ctxs || n_ctx <= 0 || !p || nq < 0 || (nq > 0 && !goals)) {
        g_err = "smplhost_plan_batch_goals: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    for (int t = 0; t < n_ctx; ++t) {
        if (!ctxs[t]) {
            g_err = "smplhost_plan_batch_goals: null context";
            return SMPLGPU_ERR_INVALID;
        }
    }
    if (p->dof <= 0 || p->dof > SMPLGPU_MAX_DOF) {
        g_err = "smplhost_plan_batch_goals: dof out of range";
        return SMPLGPU_ERR_INVALID;
    }
    // the checks of smplgpu_lattice_begin_goals, before any query starts
    for (int i = 0; i < nq; ++i) {
        const smplgpu_goal& g = goals[i];
        bool ok = true;
        if (g.type == SMPLGPU_GOAL_XYZ || g.type == SMPLGPU_GOAL_XYZ_RPY) {
            for (int a = 0; a < 3; ++a) ok = ok && !bad_tolerance(g.xyz_tolerance[a]);
            ok = ok && (g.type == SMPLGPU_GOAL_XYZ || !bad_tolerance(g.rpy_tolerance));
        } else if (g.type == SMPLGPU_GOAL_JOINT_STATE) {
            for (int v = 0; v < p->dof; ++v) ok = ok && !bad_tolerance(g.angle_tolerances[v]);
        } else {
            g_err = "smplhost_plan_batch_goals: goal " + std::to_string(i) + " has unknown type " + std::to_string(g.type);
            return SMPLGPU_ERR_INVALID;
        }
        if (!ok) {
            g_err = "smplhost_plan_batch_goals: goal " + std::to_string(i) + " has a NaN or negative tolerance";
            return SMPLGPU_ERR_INVALID;
        }
    }
    return 0;
}

int smplhost_plan_batch_goals(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p, const double* starts,
                              const smplgpu_goal* goals, int nq, int max_concurrent_per_ctx, int32_t* summary,
                              int32_t* path_ids, int max_path, double* stats, double* path_states)
{
    const int r = check_goal_args(ctxs, n_ctx, p, goals, nq);
    if (r) return r;
    return plan_batch_contexts(ctxs, n_ctx, p, starts, goals, nq, max_concurrent_per_ctx, summary, path_ids, max_path,
                               stats, path_states);
}

// the checks of smplgpu_lattice_set_snaps and the snaps' cost weight, before any query starts
static int check_snaps_args(const smplhost_snaps_params* snaps)
{
    if (std::isnan(snaps->weight) || snaps->weight < 0.0 || snaps->weight > 1e6) {
        g_err = "smplhost_plan_batch_snaps: snap weight is NaN, negative or too large";
        return SMPLGPU_ERR_INVALID;
    }
    for (int k = 0; k < 3; ++k) {
        if (std::isnan(snaps->kinds.dist_thresh[k]) || snaps->kinds.dist_thresh[k] < 0.0) {
            g_err = "smplhost_plan_batch_snaps: the threshold of snap kind " + std::to_string(k) + " is NaN or negative";
            return SMPLGPU_ERR_INVALID;
        }
    }
    if (snaps->kinds.ik.max_iterations < 1 || !(snaps->kinds.ik.tolerance > 0.0)) {
        g_err = "smplhost_plan_batch_snaps: IK max_iterations < 1, or a tolerance that is not positive";
        return SMPLGPU_ERR_INVALID;
    }
    return 0;
}

// smplhost_snap_params as the SNAP_TO_XYZ_RPY kind alone
static smplhost_snaps_params xyz_rpy_alone(const smplhost_snap_params* snap)
{
    smplhost_snaps_params s = {};
    s.kinds.enabled[SMPLGPU_SNAP_XYZ_RPY] = snap->enabled;
    s.kinds.dist_thresh[SMPLGPU_SNAP_XYZ_RPY] = snap->dist_thresh;
    s.kinds.ik = snap->ik;
    s.weight = snap->weight;
    return s;
}

// counters[6] by kind -> counters[2] summed over the kinds
static void counter_totals(const int64_t* by_kind, int64_t* counters)
{
    if (counters) {
        counters[0] = by_kind[0] + by_kind[2] + by_kind[4];
        counters[1] = by_kind[1] + by_kind[3] + by_kind[5];
    }
}

int smplhost_plan_batch_snap(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p, const double* starts,
                             const smplgpu_goal* goals, int nq, int max_concurrent_per_ctx, int32_t* summary,
                             int32_t* path_ids, int max_path, double* stats, double* path_states,
                             const smplhost_snap_params* snap, int64_t* counters)
{
    int r = check_goal_args(ctxs, n_ctx, p, goals, nq);
    if (r) return r;
    if (!snap) {
        g_err = "smplhost_plan_batch_snap: null snap parameters";
        return SMPLGPU_ERR_INVALID;
    }
    const smplhost_snaps_params snaps = xyz_rpy_alone(snap);
    r = check_snaps_args(&snaps);
    if (r) return r;
    int64_t by_kind[6] = { 0, 0, 0, 0, 0, 0 };
    r = plan_batch_contexts(ctxs, n_ctx, p, starts, goals, nq, max_concurrent_per_ctx, summary, path_ids, max_path,
                            stats, path_states, &snaps, by_kind);
    counter_totals(by_kind, counters);
    return r;
}

int smplhost_plan_batch_goal_sets(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p,
                                  const double* starts, const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
                                  int max_concurrent_per_ctx, int32_t* summary, int32_t* path_ids, int max_path,
                                  double* stats, double* path_states, const smplhost_snap_params* snap,
                                  int64_t* counters, int32_t* reached_goal)
{
    smplhost_snaps_params snaps;
    if (snap) {
        snaps = xyz_rpy_alone(snap);
    }
    int64_t by_kind[6] = { 0, 0, 0, 0, 0, 0 };
    const int r = smplhost_plan_batch_snaps(ctxs, n_ctx, p, starts, goals, goal_offsets, nq, max_concurrent_per_ctx,
                                            summary, path_ids, max_path, stats, path_states, snap ? &snaps : nullptr,
                                            by_kind, reached_goal);
    counter_totals(by_kind, counters);
    return r;
}

int smplhost_plan_batch_snaps(smplgpu_ctx* const* ctxs, int n_ctx, const smplhost_plan_params* p, const double* starts,
                              const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
                              int max_concurrent_per_ctx, int32_t* summary, int32_t* path_ids, int max_path,
                              double* stats, double* path_states, const smplhost_snaps_params* snaps,
                              int64_t* counters, int32_t* reached_goal)
{
    if (nq < 0 || (nq > 0 && (!goal_offsets || !reached_goal))) {
        g_err = "smplhost_plan_batch_goal_sets: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    // the set checks of smplgpu_lattice_begin_goal_sets, before any query starts
    if (nq > 0 && goal_offsets[0] != 0) {
        g_err = "smplhost_plan_batch_goal_sets: goal_offsets[0] is not 0";
        return SMPLGPU_ERR_INVALID;
    }
    for (int i = 0; i < nq; ++i) {
        const long long m = (long long)goal_offsets[i + 1] - goal_offsets[i];
        if (m < 1 || m > SMPLGPU_MAX_GOAL_SET) {
            g_err = "smplhost_plan_batch_goal_sets: query " + std::to_string(i) + " has a goal set of " + std::to_string(m) +
                    " records (1 to " + std::to_string(SMPLGPU_MAX_GOAL_SET) + ")";
            return SMPLGPU_ERR_INVALID;
        }
    }
    int r = check_goal_args(ctxs, n_ctx, p, goals, nq > 0 ? goal_offsets[nq] : 0);
    if (r) return r;
    if (snaps) {
        r = check_snaps_args(snaps);
        if (r) return r;
    }
    if (counters) {
        std::fill(counters, counters + 6, 0);
    }
    return plan_batch_contexts(ctxs, n_ctx, p, starts, goals, nq, max_concurrent_per_ctx, summary, path_ids, max_path,
                               stats, path_states, snaps, counters, goal_offsets, reached_goal);
}

struct smplhost_adapters
{
    std::unique_ptr<smplhost::GpuCollisionSpace> cc;
    std::unique_ptr<smplhost::GpuRobotModel> rm;
    std::unique_ptr<smplhost::GpuBfsHeuristic> heur;
    std::vector<sbpl::motion::RobotState> states; // the "lattice": state id -> joint state; id 0 = goal state
    int dof = 0;
    smplgpu_ctx* ctx = nullptr;
    int cost_per_cell = 1;
    std::unique_ptr<smplhost::ExpansionCache> cache;
};

smplhost_adapters* smplhost_adapters_create(smplgpu_ctx* ctx, smplhost_tables* tables, const char* planning_link,
                                            const double origin[3], double res, const int32_t dims[3],
                                            double inflation_radius, int cost_per_cell)
{
    if (!ctx || !tables || !planning_link || !origin || !dims) {
        g_err = "smplhost_adapters_create: null argument";
        return nullptr;
    }
    std::unique_ptr<smplhost_adapters> a(new smplhost_adapters);
    const smplgpu_robot_desc* d = tables->t.desc();
    a->dof = d->dof;
    a->ctx = ctx;
    a->cost_per_cell = cost_per_cell;
    a->cc.reset(new smplhost::GpuCollisionSpace(ctx, d->dof));
    std::vector<int> types(d->var_type, d->var_type + d->dof);
    std::vector<double> weights(d->var_motion_weight, d->var_motion_weight + d->dof);
    a->cc->setVariableInfo(tables->t.varContinuous(), weights, types);
    a->rm.reset(new smplhost::GpuRobotModel(ctx, &tables->t, planning_link));
    const int idims[3] = { dims[0], dims[1], dims[2] };
    a->heur.reset(new smplhost::GpuBfsHeuristic(ctx, origin, res, idims));
    a->heur->setInflationRadius(inflation_radius);
    a->heur->setCostPerCell(cost_per_cell);
    a->states.push_back(sbpl::motion::RobotState()); // goal state placeholder
    smplhost_adapters* raw = a.get();
    auto lookup = [raw](int id, sbpl::motion::RobotState& q) {
        if (id <= 0 || id >= (int)raw->states.size()) return false;
        q = raw->states[id];
        return true;
    };
    if (!a->heur->init(lookup, 0)) {
        g_err = smplgpu_last_error(ctx);
        return nullptr;
    }
    return a.release();
}

void smplhost_adapters_destroy(smplhost_adapters* a) { delete a; }

int smplhost_adapters_enable_expansion_cache(smplhost_adapters* a, const double* deltas, int n_prims, int64_t* counters)
{
    if (!a) return -1;
    if (counters && a->cache) {
        counters[0] = a->cache->launches();
        counters[1] = a->cache->hits();
    }
    if (!deltas) {
        return a->cache ? 0 : -1;   // counters only
    }
    a->cc->setExpansionCache(nullptr);
    a->rm->setExpansionCache(nullptr);
    a->heur->setExpansionCache(nullptr);
    a->cache.reset();
    if (n_prims <= 0) {
        return 0;
    }
    a->cache.reset(new smplhost::ExpansionCache(a->ctx, a->dof, deltas, n_prims, a->cost_per_cell));
    if (!a->cache->ok()) {
        g_err = smplgpu_last_error(a->ctx);
        a->cache.reset();
        return -1;
    }
    a->cc->setExpansionCache(a->cache.get());
    a->rm->setExpansionCache(a->cache.get());
    a->heur->setExpansionCache(a->cache.get());
    return 0;
}

static sbpl::motion::RobotState to_state(const smplhost_adapters* a, const double* q)
{
    return sbpl::motion::RobotState(q, q + a->dof);
}

int smplhost_cc_is_state_valid(smplhost_adapters* a, const double* q)
{
    if (!a || !q) return -1;
    sbpl::motion::CollisionChecker* cc = a->cc.get(); // through the interface, as the planner holds it
    return cc->isStateValid(to_state(a, q)) ? 1 : 0;
}

int smplhost_cc_is_state_to_state_valid(smplhost_adapters* a, const double* q0, const double* q1)
{
    if (!a || !q0 || !q1) return -1;
    sbpl::motion::CollisionChecker* cc = a->cc.get();
    return cc->isStateToStateValid(to_state(a, q0), to_state(a, q1)) ? 1 : 0;
}

int smplhost_cc_interpolate_path(smplhost_adapters* a, const double* q0, const double* q1, double* out, int max_waypoints)
{
    if (!a || !q0 || !q1 || !out) return -1;
    std::vector<sbpl::motion::RobotState> path;
    if (!a->cc->interpolatePath(to_state(a, q0), to_state(a, q1), path) || (int)path.size() > max_waypoints) {
        return -1;
    }
    for (size_t i = 0; i < path.size(); ++i) {
        std::copy(path[i].begin(), path[i].end(), out + i * a->dof);
    }
    return (int)path.size();
}

int smplhost_cc_is_states_valid(smplhost_adapters* a, const double* q, int n, uint8_t* valid)
{
    if (!a || n < 0 || (n > 0 && (!q || !valid))) return -1;
    std::vector<sbpl::motion::RobotState> states(n);
    for (int i = 0; i < n; ++i) states[i].assign(q + (size_t)i * a->dof, q + (size_t)(i + 1) * a->dof);
    std::vector<uint8_t> v;
    if (!a->cc->isStatesValid(states, v)) return -1;
    std::copy(v.begin(), v.end(), valid);
    return 0;
}

int smplhost_cc_is_edges_valid(smplhost_adapters* a, const double* q0, const double* q1, int n, uint8_t* valid)
{
    if (!a || n < 0 || (n > 0 && (!q0 || !q1 || !valid))) return -1;
    std::vector<sbpl::motion::RobotState> s0(n), s1(n);
    for (int i = 0; i < n; ++i) {
        s0[i].assign(q0 + (size_t)i * a->dof, q0 + (size_t)(i + 1) * a->dof);
        s1[i].assign(q1 + (size_t)i * a->dof, q1 + (size_t)(i + 1) * a->dof);
    }
    std::vector<uint8_t> v;
    if (!a->cc->isEdgesValid(s0, s1, v)) return -1;
    std::copy(v.begin(), v.end(), valid);
    return 0;
}

double smplhost_cc_distance_to_collision(smplhost_adapters* a, const double* q0, const double* q1)
{
    if (!a || !q0) return -1.0;
    auto* ext = a->cc->getExtension(sbpl::motion::GetClassCode<sbpl::motion::CollisionDistanceExtension>());
    auto* cd = dynamic_cast<sbpl::motion::CollisionDistanceExtension*>(ext);
    if (!cd) return -1.0;
    return q1 ? cd->distanceToCollision(to_state(a, q0), to_state(a, q1)) : cd->distanceToCollision(to_state(a, q0));
}

int smplhost_rm_check_joint_limits(smplhost_adapters* a, const double* q)
{
    if (!a || !q) return -1;
    sbpl::motion::RobotModel* rm = a->rm.get();
    return rm->checkJointLimits(to_state(a, q)) ? 1 : 0;
}

int smplhost_rm_compute_planning_link_fk(smplhost_adapters* a, const double* q, double* pose6)
{
    if (!a || !q || !pose6) return -1;
    sbpl::motion::Extension* ext = a->rm.get(); // looked up the way the planner does (extension.h:40-60)
    sbpl::motion::ForwardKinematicsInterface* fk = ext->getExtension<sbpl::motion::ForwardKinematicsInterface>();
    std::vector<double> pose;
    if (!fk || !fk->computePlanningLinkFK(to_state(a, q), pose)) return -1;
    std::copy(pose.begin(), pose.end(), pose6);
    return 0;
}

int smplhost_heur_update_goal(smplhost_adapters* a, const double xyz[3])
{
    if (!a || !xyz) return -1;
    sbpl::motion::GoalConstraint goal;
    goal.type = sbpl::motion::XYZ_GOAL;
    goal.tgt_off_pose = { xyz[0], xyz[1], xyz[2], 0.0, 0.0, 0.0 };
    sbpl::motion::RobotHeuristic* h = a->heur.get();
    h->updateGoal(goal);
    return 0;
}

int smplhost_heur_goal_heuristic(smplhost_adapters* a, const double* q)
{
    if (!a || !q) return -1;
    a->states.push_back(to_state(a, q));
    sbpl::motion::RobotHeuristic* h = a->heur.get();
    return h->GetGoalHeuristic((int)a->states.size() - 1);
}

double smplhost_heur_metric_goal_distance(smplhost_adapters* a, double x, double y, double z)
{
    if (!a) return -1.0;
    return a->heur->getMetricGoalDistance(x, y, z);
}

///////////////////////////////////////////////////////////////////////////////
// path post-processing (post_processing.h)
///////////////////////////////////////////////////////////////////////////////

static void copy_post_stats(const smplhost::PostProcessingStats& st, double* stats)
{
    if (stats) {
        stats[0] = (double)st.edges_checked;
        stats[1] = (double)st.states_checked;
        stats[2] = (double)st.device_calls;
        stats[3] = st.device_seconds;
        stats[4] = st.host_seconds;
    }
}

int smplhost_shortcut_paths(smplgpu_ctx* ctx, int dof, const uint8_t* continuous, const double* points,
                            const int32_t* offsets, int n_paths, int type, int32_t* out_idx, int32_t* out_offsets,
                            double* stats)
{
    if (!ctx || dof <= 0 || n_paths < 0 || (n_paths > 0 && (!continuous || !points || !offsets || !out_idx || !out_offsets))) {
        g_err = "smplhost_shortcut_paths: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    if (type != smplhost::SHORTCUT_JOINT_SPACE && type != smplhost::SHORTCUT_JOINT_POSITION_VELOCITY_SPACE) {
        g_err = "smplhost_shortcut_paths: only the joint-space shortcut types run here (EUCLID_SPACE needs the IK plugin)";
        return SMPLGPU_ERR_INVALID;
    }
    for (int p = 0; p < n_paths; ++p) {
        if (offsets[p + 1] < offsets[p] || offsets[0] != 0) {
            g_err = "smplhost_shortcut_paths: offsets must start at 0 and not decrease";
            return SMPLGPU_ERR_INVALID;
        }
    }
    std::vector<int32_t> idx, off;
    smplhost::PostProcessingStats st;
    std::string err;
    if (!smplhost::ShortcutPaths(ctx, dof, continuous, points, offsets, n_paths, type, idx, off, &st, &err)) {
        g_err = err;
        return SMPLGPU_ERR_CUDA;
    }
    std::copy(idx.begin(), idx.end(), out_idx);
    std::copy(off.begin(), off.end(), out_offsets);
    copy_post_stats(st, stats);
    return 0;
}

int smplhost_interpolate_paths(smplgpu_ctx* ctx, smplhost_tables* tables, const double* points, const int32_t* offsets,
                               int n_paths, double* out_points, int max_points, int32_t* out_offsets, double* stats)
{
    if (!ctx || !tables || n_paths < 0 || (n_paths > 0 && (!points || !offsets || !out_offsets))) {
        g_err = "smplhost_interpolate_paths: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    const smplgpu_robot_desc* d = tables->t.desc();
    std::vector<double> pts;
    std::vector<int32_t> off;
    smplhost::PostProcessingStats st;
    std::string err;
    if (!smplhost::InterpolatePaths(ctx, d->dof, d->var_type, d->var_motion_weight, points, offsets, n_paths, pts, off, &st, &err)) {
        g_err = err;
        return SMPLGPU_ERR_CUDA;
    }
    std::copy(off.begin(), off.end(), out_offsets);
    copy_post_stats(st, stats);
    const int total = (int)(pts.size() / d->dof);
    if (total > max_points || !out_points) {
        return total > 0 && out_points ? SMPLGPU_ERR_LIMIT : total;   // call again with room for out_offsets[n_paths] points
    }
    std::copy(pts.begin(), pts.end(), out_points);
    return total;
}

///////////////////////////////////////////////////////////////////////////////
// scene ingest (scene_ingest.h)
///////////////////////////////////////////////////////////////////////////////

int smplhost_shape_mesh_size(int kind, int32_t* n_vertices, int32_t* n_triangles)
{
    if (!n_vertices || !n_triangles) return SMPLGPU_ERR_INVALID;
    int nv = 0, nt = 0;
    smplhost::ShapeMeshSize(kind, &nv, &nt);
    *n_vertices = nv;
    *n_triangles = nt;
    return nv > 0 ? 0 : SMPLGPU_ERR_INVALID;
}

int smplhost_shape_meshes(const double* shapes, int n_shapes, double* vertices, int32_t* triangles)
{
    if (n_shapes < 0 || (n_shapes > 0 && (!shapes || !vertices || !triangles))) {
        g_err = "smplhost_shape_meshes: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    std::vector<double> v;
    std::vector<int32_t> t;
    for (int i = 0; i < n_shapes; ++i) {
        const double* s = shapes + 16 * (size_t)i;
        if (!smplhost::AppendShapeMesh((int)s[0], s + 1, s + 4, v, t)) {
            g_err = "smplhost_shape_meshes: unknown shape kind";
            return SMPLGPU_ERR_INVALID;
        }
    }
    std::copy(v.begin(), v.end(), vertices);
    std::copy(t.begin(), t.end(), triangles);
    return (int)(t.size() / 3);
}

int smplhost_box_meshes(const double* boxes, int n_boxes, double* vertices, int32_t* triangles)
{
    if (n_boxes < 0 || (n_boxes > 0 && (!boxes || !vertices || !triangles))) {
        g_err = "smplhost_box_meshes: bad argument";
        return SMPLGPU_ERR_INVALID;
    }
    std::vector<double> v;
    std::vector<int32_t> t;
    for (int i = 0; i < n_boxes; ++i) {
        const double* b = boxes + 15 * (size_t)i;
        smplhost::AppendBoxMesh(b[0], b[1], b[2], b + 3, v, t);
    }
    std::copy(v.begin(), v.end(), vertices);
    std::copy(t.begin(), t.end(), triangles);
    return 0;
}

} // extern "C"
