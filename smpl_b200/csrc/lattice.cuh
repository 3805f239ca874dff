// The manipulation lattice of MANY concurrent queries, resident on the device: successor generation, joint limits,
// stateToCoord, the coordinate hash table (getOrCreateState), the goal test and the heuristic of one expansion round
// run here, so that a round ships 8 bytes per expansion (bank slot, state id) and gets back one int pair per
// successor (state id | goal flag, heuristic).  The host keeps what north_star says it keeps: ARA*'s OPEN list and
// search states, indexed by the ids this table hands out.
//
// Reference semantics restated (file:line under dyouakim/smpl):
//   ManipLattice::GetSuccs                          smpl/src/graph/manip_lattice.cpp:219-313
//   ManipLatticeActionSpace::apply / mprimActive    smpl/src/graph/manip_lattice_action_space.cpp:376-449, 662-691
//   ManipLattice::checkAction (joint limits first)  manip_lattice.cpp:1511-1580
//   ManipLattice::stateToCoord                      manip_lattice.cpp:1263-1289
//   ManipLattice::getOrCreateState / createHashEntry  manip_lattice.cpp:1291-1356  (ids in creation order)
//   ManipLattice::isGoal (XYZ, XYZ_RPY, JOINT_STATE) manip_lattice.cpp:1582-1696
//   BfsHeuristic::GetGoalHeuristic                  smpl/src/heuristic/bfs_heuristic.cpp:148-163
// State ids must come out in the reference's creation order (they are what plans are compared by): an expansion's
// successors are entered one after the other in primitive order by ONE warp, and a query has at most one
// expansion per round, so no two warps ever touch the same query's table.
#pragma once

#include "heuristic.cuh"
#include "model.cuh"
#include "validity.cuh"
#include "validity32.cuh"

namespace smplgpu {

constexpr int LATTICE_MAX_STRIDE = 32;        // successors per expansion: one lane each
constexpr int LATTICE_GOAL_FLAG = 1 << 30;    // in a successor word: the action reaches the goal region
constexpr int LATTICE_SHORT_FLAG = 1 << 29;   // in a count word: the expansion used the short-distance primitives

// One goal record of a query's goal set (smplgpu_goal, as the device reads it).  qg is the goal orientation's quaternion
// x y z w and R its rotation matrix (the snap action's IK target), both computed on the host
// (smplgpu_lattice_begin_goal_sets) so that only the state's quaternion rounds the device's way.  pos is the record's
// goal position: xyz, or for a joint record the target-offset position of its angles (lattice_begin_kernel).
struct LatticeGoal
{
    int type;                 // SMPLGPU_GOAL_*
    double xyz[3], xyz_tol[3];
    double pos[3];
    double qg[4];
    double R[9];
    double rpy_tol;
    double angles[MAX_DOF], angle_tol[MAX_DOF];
};

struct LatticeBank
{
    int n_slots, cap, table_size;             // states per slot, hash slots per slot (power of two)
    int stride;                               // successor words per expansion = snap + max(#long, #short primitives)
    int n_long, n_short;
    int use_short_dist;
    double short_dist_thresh, res;
    int cost_per_cell;
    double* q;        // [n_slots][cap][dof]
    int* coord;       // [n_slots][cap][dof]
    int* gdist;       // [n_slots][cap]   BFS cells at the planning link (getMetricGoalDistance / res)
    int* table;       // [n_slots][table_size] state id, -1 = empty
    int* count;       // [n_slots] lattice size (ids 0 .. count-1; 0 = the goal state, 1 = the start state)
    LatticeGoal* goal;        // [n_slots][SMPLGPU_MAX_GOAL_SET]: the slot's goal set
    int* n_goals;             // [n_slots] records in the set
    const double* deltas;     // [n_prims][dof]
    const int* long_list;     // primitive indices in table order
    const int* short_list;
    // the snap actions (smplgpu_lattice_set_snaps): snap = the number of enabled kinds, which take words 0 .. snap-1
    // of every expansion (word k is kind snap_kind[k]), the primitives the words after them; 0 = no snap word
    int snap;
    int snap_kind[3];          // SMPLGPU_SNAP_* of word k, in the order RPY, XYZ, XYZ_RPY
    double snap_thresh[3];     // by SMPLGPU_SNAP_* kind
    int ik_max_iterations;
    double ik_tolerance;
};

// ManipLattice::stateToCoord (manip_lattice.cpp:1263-1289; every KDL planning variable is continuous or bounded)
__device__ __forceinline__ int state_to_coord(const DevModel* __restrict__ M, const LatticeParams& L, const int* vals,
                                              int v, double q)
{
    const double PI = 3.14159265358979323846;
    if (M->var_type[v] == 1) {
        double pos = normalize_angle(q);
        if (pos < 0.0) {
            pos += 2.0 * PI;
        }
        int c = __double2int_rz((pos + L.delta[v] * 0.5) / L.delta[v]);
        if (c == vals[v]) {
            c = 0;
        }
        return c;
    }
    return __double2int_rz(((q - M->var_min[v]) / L.delta[v]) + 0.5);
}

struct LatticeVals { int v[MAX_DOF]; };

__device__ __forceinline__ unsigned int coord_hash(const int* c, int dof)
{
    unsigned long long x = 0x9E3779B97F4A7C15ull;
    for (int i = 0; i < dof; ++i) {
        x ^= (unsigned long long)(unsigned int)c[i] + 0x9E3779B97F4A7C15ull + (x << 6) + (x >> 2);
    }
    return (unsigned int)(x ^ (x >> 32));
}

// tables of the listed slots -> empty
__global__ void lattice_clear_kernel(LatticeBank B, const int* __restrict__ slots, int n)
{
    const size_t total = (size_t)n * B.table_size;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(i / B.table_size);
        B.table[(size_t)slots[k] * B.table_size + (i - (size_t)k * B.table_size)] = -1;
    }
}

// ManipLattice::setGoal + setStart bookkeeping: id 0 = the goal state (no coordinates), id 1 = the start state.
// Thread k < n sets up query k; thread r < n_rec copies record r (of query goal_set[r], whose set starts at
// goal_offsets[goal_set[r]]) into the query's slot, with its goal position.
__global__ void lattice_begin_kernel(const DevModel* __restrict__ M, LatticeBank B, LatticeParams L, LatticeVals V,
                                     const int* __restrict__ slots, const double* __restrict__ starts,
                                     const int* __restrict__ start_gd, const LatticeGoal* __restrict__ goals,
                                     const int* __restrict__ goal_set, const int* __restrict__ goal_offsets, int n,
                                     int n_rec)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int dof = M->dof;
    if (k < n_rec) {
        const int qk = goal_set[k];
        LatticeGoal* g = B.goal + (size_t)slots[qk] * SMPLGPU_MAX_GOAL_SET + (k - goal_offsets[qk]);
        *g = goals[k];
        if (g->type == SMPLGPU_GOAL_JOINT_STATE) {
            double pose[6];
            planning_frame_fk(M, goals[k].angles, pose);
            g->pos[0] = pose[0]; g->pos[1] = pose[1]; g->pos[2] = pose[2];
        } else {
            g->pos[0] = g->xyz[0]; g->pos[1] = g->xyz[1]; g->pos[2] = g->xyz[2];
        }
    }
    if (k >= n) {
        return;
    }
    const int s = slots[k];
    int c[MAX_DOF];
    double* q1 = B.q + ((size_t)s * B.cap + 1) * dof;
    int* c1 = B.coord + ((size_t)s * B.cap + 1) * dof;
    for (int v = 0; v < dof; ++v) {
        const double a = starts[(size_t)k * dof + v];
        q1[v] = a;
        c[v] = state_to_coord(M, L, V.v, v, a);
        c1[v] = c[v];
        B.q[((size_t)s * B.cap) * dof + v] = 0.0;
    }
    B.gdist[(size_t)s * B.cap] = 0;
    B.gdist[(size_t)s * B.cap + 1] = start_gd[k];
    B.table[(size_t)s * B.table_size + (coord_hash(c, dof) & (unsigned int)(B.table_size - 1))] = 1;
    B.count[s] = 2;
    B.n_goals[s] = goal_offsets[k + 1] - goal_offsets[k];
}

// Eigen's generic quat_product (x y z w), the operation order of the oracle's Eigen stand-in
__device__ __forceinline__ void quat_mul(const double* a, const double* b, double* r)
{
    r[3] = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
    r[0] = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
    r[1] = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
    r[2] = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
}

// q = AngleAxisd(yaw, Z) * AngleAxisd(pitch, Y) * AngleAxisd(roll, X) of a target-offset pose (Quaterniond(AngleAxisd):
// w = cos(a/2), xyz = sin(a/2) axis)
__device__ __forceinline__ void pose_quat(const double* pose, double* qs)
{
    double sy, cy, sp, cp, sr, cr;
    sincos(0.5 * pose[5], &sy, &cy);
    sincos(0.5 * pose[4], &sp, &cp);
    sincos(0.5 * pose[3], &sr, &cr);
    const double qz[4] = { sy * 0.0, sy * 0.0, sy * 1.0, cy };
    const double qy[4] = { sp * 0.0, sp * 1.0, sp * 0.0, cp };
    const double qx[4] = { sr * 1.0, sr * 0.0, sr * 0.0, cr };
    double qzy[4];
    quat_mul(qz, qy, qzy);
    quat_mul(qzy, qx, qs);
}

// ManipLattice::isGoal (manip_lattice.cpp:1582-1696) of a state q whose target-offset pose is `pose`, against one
// record; the record is the same for every lane of the warp (one warp serves one query).  qs is the state's quaternion
// (pose_quat), computed by the caller the first time an XYZ_RPY record's box test passes (*have_qs).
__device__ __forceinline__ bool lattice_is_goal(int dof, const LatticeGoal* __restrict__ g, const double* q,
                                                const double* pose, double* qs, bool* have_qs)
{
    const int type = g->type;
    if (type == SMPLGPU_GOAL_JOINT_STATE) {
        bool in = true;
        for (int v = 0; v < dof; ++v) {
            in = in && fabs(q[v] - g->angles[v]) <= g->angle_tol[v];
        }
        return in;
    }
    const bool in_box = fabs(pose[0] - g->xyz[0]) <= g->xyz_tol[0] && fabs(pose[1] - g->xyz[1]) <= g->xyz_tol[1] &&
                        fabs(pose[2] - g->xyz[2]) <= g->xyz_tol[2];
    if (type != SMPLGPU_GOAL_XYZ_RPY || !in_box) {
        return in_box;
    }
    if (!*have_qs) {
        pose_quat(pose, qs);
        *have_qs = true;
    }
    double d = ((qs[0] * g->qg[0] + qs[1] * g->qg[1]) + qs[2] * g->qg[2]) + qs[3] * g->qg[3];
    if (d < 0.0) {
        d = -d;   // the dot product with the negated qg: every term changes sign exactly
    }
    return normalize_angle(2.0 * acos(d)) < g->rpy_tol;
}

// Round, step 1: the edges of every expansion.  Thread (i, j): j-th active primitive of the state expansion i pops
// (with k snap kinds enabled words 0 .. k-1 are the snaps', which lattice_snap_kernel fills in, and word j the
// (j-k)-th primitive).
// Inactive positions and successors beyond a joint limit become zero-length edges (no waypoint, no work in the
// edge kernels) and are flagged.
__global__ void lattice_gen_kernel(const DevModel* __restrict__ M, LatticeBank B, const int* __restrict__ slot,
                                   const int* __restrict__ parent, int n, double* __restrict__ q0,
                                   double* __restrict__ q1, uint8_t* __restrict__ active, unsigned long long* stats)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < 4) {
        stats[t] = 0;   // counters of the edge kernels that follow (saves a memset call per round)
    }
    if (t >= n * B.stride) {
        return;
    }
    const int i = t / B.stride, j = t - i * B.stride;
    const int s = slot[i], p = parent[i];
    const int dof = M->dof;
    const double* a = B.q + ((size_t)s * B.cap + p) * dof;
    // mprimActive: short-distance primitives once the planning link is within the threshold of the goal
    const double goal_dist = (double)B.gdist[(size_t)s * B.cap + p] * B.res;
    const bool near_goal = B.use_short_dist && goal_dist <= B.short_dist_thresh;
    const int cnt = near_goal ? B.n_short : B.n_long;
    double succ[MAX_DOF];
    const int w = j - B.snap;
    bool on = w >= 0 && w < cnt;
    if (on) {
        const int prim = near_goal ? B.short_list[w] : B.long_list[w];
        for (int v = 0; v < dof; ++v) {
            succ[v] = B.deltas[(size_t)prim * dof + v] + a[v];
        }
        on = joint_limits_ok(M, succ);
    }
    for (int v = 0; v < dof; ++v) {
        const double av = a[v];
        q0[(size_t)t * dof + v] = av;
        q1[(size_t)t * dof + v] = on ? succ[v] : av;
    }
    active[t] = on ? 1 : 0;
}

// The commit step of one expansion, by ONE warp, lane j = successor j.  Valid successors get their planning-frame pose
// (goal test, heuristic, metric goal distance), their coordinates and hash in parallel; then they are looked up /
// entered ONE AFTER THE OTHER in primitive order, so ids come out in the reference's creation order.
// succ_out[j] = id | LATTICE_GOAL_FLAG, or -1; h_out[j] = GetGoalHeuristic(successor), or for a goal-flagged successor
// the index of the first record of the slot's goal set it satisfies; *count_out = lattice size of the query afterwards
// (-1: out of room).
__device__ __forceinline__ void lattice_commit_warp(const DevModel* __restrict__ M, const GridParams& G, const LatticeBank& B,
                                                    const LatticeParams& L, const LatticeVals& V, const int* __restrict__ bfs,
                                                    int dimx, int dimy, int slot_dimz, int s, int lane, bool valid,
                                                    const double* q, int* succ_out, int* h_out, int* count_out,
                                                    bool near_goal)
{
    const int dof = M->dof;
    int c[MAX_DOF];
    unsigned int hv = 0;
    int h = 0, gd = 0;
    bool is_goal = false;
    if (valid) {
        double pose[6], link[3];
        planning_frame_fk(M, q, pose, link);
        bool inb;
        const int d_off = bank_lookup(bfs, dimx, dimy, slot_dimz, s, G, pose[0], pose[1], pose[2], inb);
        h = (!inb || d_off == 0x7FFFFFFF) ? 32767 : B.cost_per_cell * d_off;
        gd = bank_lookup(bfs, dimx, dimy, slot_dimz, s, G, link[0], link[1], link[2], inb);
        // the goal set in order: the first record satisfied is the reached index (the host never reads the heuristic
        // of a goal-flagged successor: it stands for the goal state, whose heuristic the host knows)
        const LatticeGoal* set = B.goal + (size_t)s * SMPLGPU_MAX_GOAL_SET;
        const int n_goals = B.n_goals[s];
        double qs[4];
        bool have_qs = false;
        for (int r = 0; r < n_goals; ++r) {
            if (lattice_is_goal(dof, set + r, q, pose, qs, &have_qs)) {
                is_goal = true;
                h = r;
                break;
            }
        }
        for (int v = 0; v < dof; ++v) {
            c[v] = state_to_coord(M, L, V.v, v, q[v]);
        }
        hv = coord_hash(c, dof);
    }
    int id = -1;
    bool full = false;
    unsigned int todo = __ballot_sync(0xffffffffu, valid);
    int* table = B.table + (size_t)s * B.table_size;
    const unsigned int mask = (unsigned int)(B.table_size - 1);
    while (todo) {
        const int j = __ffs(todo) - 1;
        todo &= todo - 1;
        if (lane == j) {
            unsigned int slot_i = hv & mask;
            for (;;) {
                const int cand = table[slot_i];
                if (cand < 0) {
                    break;
                }
                const int* cc = B.coord + ((size_t)s * B.cap + cand) * dof;
                bool same = true;
                for (int v = 0; v < dof; ++v) {
                    same = same && cc[v] == c[v];
                }
                if (same) {
                    id = cand;
                    break;
                }
                slot_i = (slot_i + 1) & mask;
            }
            if (id < 0) {
                const int fresh = B.count[s];
                if (fresh >= B.cap) {
                    full = true;
                } else {
                    B.count[s] = fresh + 1;
                    double* qq = B.q + ((size_t)s * B.cap + fresh) * dof;
                    int* cc = B.coord + ((size_t)s * B.cap + fresh) * dof;
                    for (int v = 0; v < dof; ++v) {
                        qq[v] = q[v];
                        cc[v] = c[v];
                    }
                    B.gdist[(size_t)s * B.cap + fresh] = gd;
                    table[slot_i] = fresh;
                    id = fresh;
                }
            }
        }
        __syncwarp();
    }
    if (lane < B.stride) {
        succ_out[lane] = id < 0 ? -1 : (id | (is_goal ? LATTICE_GOAL_FLAG : 0));
        h_out[lane] = h;
    }
    full = __any_sync(0xffffffffu, full);
    if (lane == 0) {
        // which primitive set the successor words belong to travels with the count (the host needs it for the
        // per-primitive action weights)
        *count_out = full ? -1 : (B.count[s] | (near_goal ? LATTICE_SHORT_FLAG : 0));
    }
}

// Round, step 3 of the three-kernel form (after the edge kernels): one warp per expansion.
__global__ void __launch_bounds__(128)
lattice_commit_kernel(const DevModel* __restrict__ M, GridParams G, LatticeBank B, LatticeParams L, LatticeVals V,
                      const int* __restrict__ bfs, int dimx, int dimy, int slot_dimz,
                      const int* __restrict__ slot, const int* __restrict__ parent, int n, const double* __restrict__ q1,
                      const uint8_t* __restrict__ active, const uint8_t* __restrict__ verdict,
                      int* __restrict__ out_succ, int* __restrict__ out_h, int* __restrict__ out_count,
                      const unsigned long long* __restrict__ stats, unsigned long long* resolved_total)
{
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) {
        return;
    }
    const int t = i * B.stride + lane;
    const bool valid = lane < B.stride && active[t] != 0 && verdict[t] != 0;
    // mprimActive, as lattice_gen_kernel decided it for this expansion
    const double goal_dist = (double)B.gdist[(size_t)slot[i] * B.cap + parent[i]] * B.res;
    const bool near_goal = B.use_short_dist && goal_dist <= B.short_dist_thresh;
    lattice_commit_warp(M, G, B, L, V, bfs, dimx, dimy, slot_dimz, slot[i], lane, valid, q1 + (size_t)t * M->dof,
                        out_succ + (size_t)i * B.stride, out_h + (size_t)i * B.stride, out_count + i, near_goal);
    if (i == 0 && lane == 0 && stats[3] != 0) {
        atomicAdd(resolved_total, stats[3]);   // edges of this round that the double-precision pass resolved
    }
}

// ONE KERNEL PER ROUND (SMPLGPU_LATTICE_FUSED=1; off by default): a block per expansion does everything the
// three-kernel form does -- successor generation and joint limits (threads 0 .. stride-1), the edges' waypoints in
// certified single precision spread over the block, the undecided edges again in double by warp 0 (rare: ~0.4 % of
// edges), then the commit step by warp 0 -- so a round is one launch, not a chain of five.
// Measured on one B200 (2048 PR2 tabletop queries; DESIGN.md): it wins only when many contexts share the GPU and the
// chain is launch bound (12 planner threads: 2240 vs 1470 queries/s); with the 4-6 contexts that are the optimum of the
// three-kernel form it LOSES (1540-1600 vs 1810-2000 queries/s, UBR1 3050 vs 4540): a block per expansion keeps
// ~56 of its 128 threads busy for one waypoint each and then waits for one warp's commit, where the chain packs all
// rounds' waypoints densely; and its longer-lived blocks delay the cooperative BFS launches of newly admitted queries.
// dynamic shared memory: blob | per-thread f32 slots + root centres | f64 slots of ONE warp (32 columns)
constexpr int LROUND_THREADS = 128;

__global__ void __launch_bounds__(LROUND_THREADS)
lattice_round_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                     const uint16_t* __restrict__ df, Grid32 G32, GridParams G, LatticeBank B, LatticeParams L, LatticeVals V,
                     const int* __restrict__ bfs, int dimx, int dimy, int slot_dimz,
                     const int* __restrict__ slot, const int* __restrict__ parent, int n,
                     int* __restrict__ out_succ, int* __restrict__ out_h, int* __restrict__ out_count,
                     unsigned long long* resolved_total)
{
    extern __shared__ float4 smem4[];
    __shared__ double s_q0[MAX_DOF];
    __shared__ double s_q1[LATTICE_MAX_STRIDE][MAX_DOF];
    __shared__ int s_cnt[LATTICE_MAX_STRIDE], s_off[LATTICE_MAX_STRIDE + 1], s_ok[LATTICE_MAX_STRIDE], s_unc[LATTICE_MAX_STRIDE];
    __shared__ int s_active[LATTICE_MAX_STRIDE];
    const int i = blockIdx.x;
    if (i >= n) {
        return;
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = slot[i], p = parent[i];
    const int dof = M->dof;
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    if (tid < dof) {
        s_q0[tid] = B.q[((size_t)s * B.cap + p) * dof + tid];
    }
    __syncthreads();
    const S32 S = view32(blob);
    float* slots32 = blob + blob_words;
    double* slots64 = reinterpret_cast<double*>(slots32 + ((size_t)S.h->n_slots * 12 + (size_t)S.h->n_ptrees * 3) * blockDim.x);

    // ---- successors (ManipLatticeActionSpace::apply + the joint-limit half of checkAction) and waypoint counts ----
    if (tid < B.stride) {
        const int j = tid;
        const double goal_dist = (double)B.gdist[(size_t)s * B.cap + p] * B.res;
        const bool near_goal = B.use_short_dist && goal_dist <= B.short_dist_thresh;
        const int cnt = near_goal ? B.n_short : B.n_long;
        bool on = j < cnt;
        if (on) {
            const int prim = near_goal ? B.short_list[j] : B.long_list[j];
            for (int v = 0; v < dof; ++v) {
                s_q1[j][v] = B.deltas[(size_t)prim * dof + v] + s_q0[v];
            }
            on = joint_limits_ok(M, s_q1[j]);
        }
        int count = 0;
        if (on) {
            double motion = 0.0;
            for (int v = 0; v < dof; ++v) {
                const int ty = M->var_type[v];
                if (ty == 1) {
                    motion += M->var_weight[v] * fabs(normalize_angle(s_q1[j][v] - s_q0[v]));
                } else if (ty == 0) {
                    motion += M->var_weight[v] * fabs(s_q1[j][v] - s_q0[v]);
                } else {
                    motion += fabs(s_q1[j][v] - s_q0[v]);
                }
            }
            if (motion != 0.0) {
                count = max(2, (int)ceil(motion / 0.05) + 1);
            }
        }
        s_active[j] = on ? 1 : 0;
        s_cnt[j] = count;
        s_ok[j] = on ? 1 : 0;     // an edge without waypoints is valid without a check
        s_unc[j] = 0;
    }
    __syncthreads();
    if (tid == 0) {
        int acc = 0;
        for (int j = 0; j < B.stride; ++j) {
            s_off[j] = acc;
            acc += s_cnt[j];
        }
        s_off[B.stride] = acc;
    }
    __syncthreads();
    const int total = s_off[B.stride];
    auto edge_of = [&](int item) {
        int e = 0;
        while (e + 1 < B.stride && s_off[e + 1] <= item) {
            ++e;
        }
        return e;
    };

    // ---- CollisionSpace::isStateToStateValid of every successor: waypoints over the block, certified f32 ----
    Counters cnt = { 0u, 0u, 0u };
    for (int item = tid; item < total; item += blockDim.x) {
        const int e = edge_of(item);
        if (*((volatile int*)&s_ok[e]) == 0) {
            continue;
        }
        const int w = item - s_off[e];
        const double alpha = (double)w * (1.0 / (double)(s_cnt[e] - 1));
        const int r = check_state32(S, M->var_type, df, G32, s_q0, s_q1[e], alpha, slots32, cnt);
        if (r == 0) {
            atomicAnd(&s_ok[e], 0);
        } else if (r == 2) {
            atomicOr(&s_unc[e], 1);
        }
    }
    __syncthreads();

    // ---- the undecided edges, exactly, by warp 0 (every waypoint, as the double-precision kernel does) ----
    if (warp == 0) {
        int n_res = 0;
        for (int e = 0; e < B.stride; ++e) {
            if (!(s_ok[e] != 0 && s_unc[e] != 0)) {   // warp-uniform
                continue;
            }
            ++n_res;
            bool ok = true;
            const double inv = 1.0 / (double)(s_cnt[e] - 1);
            for (int w0 = 0; w0 < s_cnt[e] && ok; w0 += 32) {
                const int w = w0 + lane;
                bool mine = true;
                if (w < s_cnt[e]) {
                    mine = check_state(M, df, G, s_q0, s_q1[e], (double)w * inv, slots64, cnt, 32, lane);
                }
                ok = __all_sync(0xffffffffu, mine);
            }
            if (lane == 0 && !ok) {
                s_ok[e] = 0;
            }
            __syncwarp();
        }
        if (lane == 0 && n_res > 0) {
            atomicAdd(resolved_total, (unsigned long long)n_res);
        }
        // ---- commit ----
        const bool valid = lane < B.stride && s_active[lane] != 0 && s_ok[lane] != 0;
        const bool near_goal = B.use_short_dist && (double)B.gdist[(size_t)s * B.cap + p] * B.res <= B.short_dist_thresh;
        lattice_commit_warp(M, G, B, L, V, bfs, dimx, dimy, slot_dimz, s, lane, valid, s_q1[lane < B.stride ? lane : 0],
                            out_succ + (size_t)i * B.stride, out_h + (size_t)i * B.stride, out_count + i, near_goal);
    }
}

// joint values of listed states (path extraction): out[k] = q[slot[k]][id[k]]
__global__ void lattice_gather_kernel(LatticeBank B, int dof, const int* __restrict__ slot, const int* __restrict__ id,
                                      int n, double* __restrict__ out)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * dof) {
        return;
    }
    const int k = t / dof, v = t - k * dof;
    out[t] = B.q[((size_t)slot[k] * B.cap + id[k]) * dof + v];
}

} // namespace smplgpu
