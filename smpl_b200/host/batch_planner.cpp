#include "batch_planner.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cmath>
#include <limits>

namespace smplhost {

static const int INFINITECOST = 1000000000;
static const int BFS_WALL = 0x7FFFFFFF;

namespace {
struct Timer
{
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double lap()
    {
        auto t1 = std::chrono::steady_clock::now();
        double s = std::chrono::duration<double>(t1 - t0).count();
        t0 = t1;
        return s;
    }
};

// smpl/angles.h:45-62
double normalizeAngle(double angle)
{
    if (std::fabs(angle) > 2.0 * M_PI) {
        angle = std::fmod(angle, 2.0 * M_PI);
    }
    if (angle < -M_PI) {
        angle += 2.0 * M_PI;
    }
    if (angle > M_PI) {
        angle -= 2.0 * M_PI;
    }
    return angle;
}
} // namespace

BatchPlanner::BatchPlanner(smplgpu_ctx* ctx, const PlannerConfig& cfg, int max_concurrent) :
    m_ctx(ctx), m_cfg(cfg), m_max_concurrent(std::max(1, max_concurrent))
{
    const int dof = cfg.dof;
    const int n_prims = (int)cfg.short_flags.size();
    // ManipLatticeActionSpace::addMotionPrim(..., add_converse = true): the converse follows each primitive
    int n_long = 0, n_short = 0;
    for (int p = 0; p < n_prims; ++p) {
        for (int sign = 0; sign < 2; ++sign) {
            for (int j = 0; j < dof; ++j) {
                const double d = cfg.mprims[(size_t)p * dof + j];
                m_prim_deltas.push_back(sign == 0 ? d : d * -1.0);
            }
            m_prim_short.push_back(cfg.short_flags[p] != 0 ? 1 : 0);
            (cfg.short_flags[p] != 0 ? n_short : n_long) += 1;
            // cost(parent, succ, actionWeight, goal) = DefaultCostMultiplier * actionWeight, truncated (manip_lattice.cpp:1436)
            const double w = cfg.prim_weights.empty() ? 1.0 : cfg.prim_weights[p];
            (cfg.short_flags[p] != 0 ? m_cost_short : m_cost_long).push_back((int)(1000 * w));
        }
    }
    m_snap_words = (cfg.snap[0] ? 1 : 0) + (cfg.snap[1] ? 1 : 0) + (cfg.snap[2] ? 1 : 0);
    m_snap_cost = (int)(1000 * cfg.snap_weight);
    m_stride = m_snap_words + std::max(n_long, cfg.use_short_dist ? n_short : 0);
}

// KDLRobotModel::checkJointLimits -> normalizeAnglesIntoRange (kdl_robot_model.cpp:173-235, 326-337)
bool BatchPlanner::checkJointLimits(const double* q) const
{
    for (int i = 0; i < m_cfg.dof; ++i) {
        if (m_cfg.var_min[i] > m_cfg.var_max[i]) {
            return false;
        }
    }
    for (int i = 0; i < m_cfg.dof; ++i) {
        const double a_min = m_cfg.var_min[i];
        const double a_max = normalizeAngle(m_cfg.var_min[i]); // sic: the reference passes normalize(min) as the upper wrap bound
        double a = q[i];
        if (std::fabs(a) > 2.0 * M_PI) {
            a = std::fmod(a, 2.0 * M_PI);
        }
        while (a > a_max) {
            a -= 2.0 * M_PI;
        }
        while (a < a_min) {
            a += 2.0 * M_PI;
        }
        if (a < m_cfg.var_min[i] || a > m_cfg.var_max[i]) {
            return false;
        }
    }
    return true;
}

// DistanceMap::worldToGrid (distance_map.hpp:520-527)
void BatchPlanner::worldToGrid(const double* p, int* cell) const
{
    const double inv = 1.0 / m_cfg.res;
    for (int a = 0; a < 3; ++a) {
        cell[a] = (int)(inv * (p[a] - (m_cfg.origin[a] - m_cfg.res)) + 0.5) - 1;
    }
}

int BatchPlanner::computeKey(const SState& s) const
{
    return s.g + (unsigned int)(m_cfg.epsilon * s.h);
}

BatchPlanner::SState& BatchPlanner::sstate(Query& Q, int id)
{
    if ((int)Q.search.size() <= id) {
        SState blank;
        blank.g = blank.h = blank.f = blank.eg = 0;
        blank.iteration_closed = 0;
        blank.bp = -1;
        blank.heap_index = 0;
        blank.touched = false;
        Q.search.resize(id + 1, blank);
    }
    return Q.search[id];
}

// ARAStar::reinitSearchState (arastar.cpp:613-627); one search call per query, so "reinit" == first touch
void BatchPlanner::touch(Query& Q, int id, int h)
{
    SState& s = sstate(Q, id);
    if (!s.touched) {
        s.g = INFINITECOST;
        s.h = (id == 0) ? Q.goal_h : h;   // GetGoalHeuristic(id), computed on the device when the state was created
        s.f = INFINITECOST;
        s.eg = INFINITECOST;
        s.iteration_closed = 0;
        s.bp = -1;
        s.touched = true;
    }
}

void BatchPlanner::percolateUp(Query& Q, size_t pivot)
{
    const Query::HeapEntry tmp = Q.open[pivot];
    while (pivot != 1) {
        const size_t p = pivot >> 1;
        if (Q.open[p].f < tmp.f) {
            break;
        }
        Q.open[pivot] = Q.open[p];
        Q.search[Q.open[pivot].id].heap_index = (int)pivot;
        pivot = p;
    }
    Q.open[pivot] = tmp;
    Q.search[tmp.id].heap_index = (int)pivot;
}

void BatchPlanner::percolateDown(Query& Q, size_t pivot)
{
    if (pivot >= Q.open.size()) {
        return;
    }
    size_t left = pivot << 1, right = left + 1;
    const Query::HeapEntry tmp = Q.open[pivot];
    while (left < Q.open.size()) {
        size_t s = right;
        if (right >= Q.open.size() || Q.open[left].f < Q.open[right].f) {
            s = left;
        }
        if (Q.open[s].f < tmp.f) {
            Q.open[pivot] = Q.open[s];
            Q.search[Q.open[pivot].id].heap_index = (int)pivot;
            pivot = s;
        } else {
            break;
        }
        left = pivot << 1;
        right = left + 1;
    }
    Q.open[pivot] = tmp;
    Q.search[tmp.id].heap_index = (int)pivot;
}

void BatchPlanner::heapPush(Query& Q, int id)
{
    Q.search[id].heap_index = (int)Q.open.size();
    Q.open.push_back(Query::HeapEntry{ Q.search[id].f, id });
    percolateUp(Q, Q.open.size() - 1);
}

void BatchPlanner::heapPop(Query& Q)
{
    Q.search[Q.open[1].id].heap_index = 0;
    Q.open[1] = Q.open.back();
    Q.open.pop_back();
    percolateDown(Q, 1);
}

void BatchPlanner::finish(Query& Q, bool found)
{
    Q.done = true;
    Q.result.num_states = Q.num_states;
    if (!found || Q.search.empty() || Q.search[0].g >= (unsigned int)INFINITECOST) {
        return;
    }
    for (int s = 0; s >= 0; s = Q.search[s].bp) {
        Q.result.path_ids.push_back(s);
    }
    std::reverse(Q.result.path_ids.begin(), Q.result.path_ids.end());
    Q.result.cost = Q.search[0].g;
    Q.result.success = true;
    const std::vector<int>& ids = Q.result.path_ids;
    const Query::GoalAction* a = ids.size() > 1 ? goalAction(Q, ids[ids.size() - 2]) : nullptr;
    Q.result.reached_goal = a ? a->reached : -1;
}

// the goal-reaching action extractPath selects after `expanded`: the first valid one of its expansion
const BatchPlanner::Query::GoalAction* BatchPlanner::goalAction(const Query& Q, int expanded)
{
    for (const Query::GoalAction& a : Q.goal_succ) {
        if (a.expanded == expanded) {
            return &a;
        }
    }
    return nullptr;
}

// ManipLattice::extractPath (manip_lattice.cpp:2018-2160): the joint values of the path's states, read from the
// device lattice while the query still owns its slot; the goal id stands for "any state satisfying the goal" and
// is replaced by the first valid goal-reaching successor of its predecessor
bool BatchPlanner::fetchPathStates(Query& Q, std::string* err)
{
    const int dof = m_cfg.dof;
    const std::vector<int>& ids = Q.result.path_ids;
    std::vector<int32_t> real(ids.size()), slots(ids.size(), Q.slot);
    size_t n = 0;
    for (size_t i = 0; i < ids.size(); ++i, ++n) {
        int id = ids[i];
        if (id == 0) {
            const Query::GoalAction* a = i > 0 ? goalAction(Q, ids[i - 1]) : nullptr;
            id = a ? a->succ : -1;
            if (id < 0) {
                break;   // cannot happen for a found path; keep what is known
            }
        }
        real[i] = id;
    }
    Q.result.path_states.assign(n * (size_t)dof, 0.0);
    if (n > 0 && smplgpu_lattice_states(m_ctx, slots.data(), real.data(), (int)n, Q.result.path_states.data()) < 0) {
        if (err) *err = smplgpu_last_error(m_ctx);
        return false;
    }
    return true;
}

///////////////////////////////////////////////////////////////////////////////
// fork-join pool
///////////////////////////////////////////////////////////////////////////////

BatchPlanner::Pool::Pool(int n) : m_n(std::max(1, n))
{
    for (int t = 1; t < m_n; ++t) {
        m_threads.emplace_back(&Pool::worker, this, t);
    }
}

BatchPlanner::Pool::~Pool()
{
    {
        std::lock_guard<std::mutex> lk(m_mutex);
        m_stop.store(true);
        m_generation.fetch_add(1);
    }
    m_cv.notify_all();
    for (std::thread& t : m_threads) {
        t.join();
    }
}

// workers spin briefly for the next job (jobs arrive every few tens of microseconds while the planner is
// busy) and block on the condition variable when nothing comes, so idle workers do not eat the cores the
// other ranks' planners need
void BatchPlanner::Pool::worker(int tid)
{
    int seen = 0;
    for (;;) {
        int spins = 0;
        while (m_generation.load(std::memory_order_acquire) == seen) {
            if (++spins < 4000) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
            } else {
                std::unique_lock<std::mutex> lk(m_mutex);
                m_sleepers.fetch_add(1);
                m_cv.wait(lk, [&] { return m_generation.load(std::memory_order_acquire) != seen; });
                m_sleepers.fetch_sub(1);
            }
        }
        seen = m_generation.load(std::memory_order_acquire);
        if (m_stop.load()) {
            return;
        }
        (*m_job)(tid);
        m_done.fetch_add(1, std::memory_order_release);
    }
}

void BatchPlanner::Pool::run(const std::function<void(int)>& f)
{
    if (m_n == 1) {
        f(0);
        return;
    }
    m_job = &f;
    m_done.store(0, std::memory_order_relaxed);
    {
        std::lock_guard<std::mutex> lk(m_mutex);   // a worker between its predicate check and its wait cannot miss this
        m_generation.fetch_add(1, std::memory_order_release);
    }
    if (m_sleepers.load() > 0) {
        m_cv.notify_all();
    }
    f(0);
    int spins = 0;
    while (m_done.load(std::memory_order_acquire) != m_n - 1) {
        if (++spins > 256) {
            std::this_thread::yield();
        }
    }
}

///////////////////////////////////////////////////////////////////////////////
// per-query steps
///////////////////////////////////////////////////////////////////////////////

void BatchPlanner::initQuery(Query& Q, int index, int slot, const smplgpu_goal* goals, int n_goals, const double* goal_xyz)
{
    // keep the slot's allocations from the query it served before (growing a multi-megabyte vector means mmap +
    // copy + munmap, and every munmap interrupts all planner threads); a fresh slot reserves room up front
    Query fresh = Query();
    std::swap(fresh.search, Q.search);
    std::swap(fresh.open, Q.open);
    fresh.search.clear();
    fresh.open.clear();
    Q = std::move(fresh);
    {
        const size_t n = std::min<size_t>(2 + (size_t)std::max(0, m_cfg.max_expansions) * (size_t)std::max(1, m_stride), (size_t)1 << 15);
        Q.search.reserve(n);
    }
    Q.index = index;
    Q.slot = slot;
    Q.done = false;
    Q.expanding = -1;
    Q.edge_begin = 0;
    Q.num_states = 1;   // id 0 = the goal state (manip_lattice.cpp:122)
    Q.goals = goals;
    Q.n_goals = n_goals;
    Q.goal_xyz = goal_xyz;
    // the goal state projects onto a seed cell, which holds distance 0 even if it was a wall (bfs3d.cpp:181-187); with
    // no seed in bounds it is out of reach
    bool inb = false;
    for (int r = 0; r < n_goals && !inb; ++r) {
        int cell[3];
        worldToGrid(goal_xyz + 3 * (size_t)r, cell);
        inb = cell[0] >= 0 && cell[1] >= 0 && cell[2] >= 0 &&
              cell[0] < m_cfg.dims[0] && cell[1] < m_cfg.dims[1] && cell[2] < m_cfg.dims[2];
    }
    Q.goal_h = inb ? 0 : SMPLGPU_HEURISTIC_INFINITY;
    Q.open.assign(1, Query::HeapEntry{ 0u, -1 });
}

// ARAStar::improvePath loop head (arastar.cpp:486-527): the state this query expands this round
void BatchPlanner::expandOne(Query& Q)
{
    Q.expanding = -1;
    if (Q.open.size() <= 1) {
        finish(Q, false);
        return;
    }
    const int min_id = Q.open[1].id;
    if (Q.search[min_id].f >= Q.search[0].f || min_id == 0) {
        finish(Q, true);
        return;
    }
    if (Q.result.expansions >= m_cfg.max_expansions) {
        finish(Q, false);
        return;
    }
    heapPop(Q);
    Q.search[min_id].iteration_closed = 1;
    Q.search[min_id].eg = Q.search[min_id].g;
    Q.expanding = min_id;
    ++Q.result.expansions;
}

// ARAStar::expand relaxations (arastar.cpp:531-568) over the successors the device returned for this query's
// expansion, in primitive order (the snaps first, when enabled): succ[j] = lattice id | goal flag, or -1 (inactive
// action, joint limit, collision)
void BatchPlanner::absorbOne(Query& Q, const int32_t* succ, const int32_t* h, int count)
{
    // word e stands for the e-th active primitive: of the short-distance set when the device flagged the expansion
    const std::vector<int>& edge_costs = (count >= 0 && (count & SMPLGPU_LATTICE_SHORT_FLAG)) ? m_cost_short : m_cost_long;
    if (count >= 0) {
        count &= ~SMPLGPU_LATTICE_SHORT_FLAG;
    }
    Q.num_states = count;
    // the search states of the successors are scattered over a megabyte-sized array: start the loads first
    for (int e = 0; e < m_stride; ++e) {
        if (succ[e] >= 0) {
            const int id = succ[e] & ~SMPLGPU_LATTICE_GOAL_FLAG;
            if ((size_t)id < Q.search.size()) {
                __builtin_prefetch(&Q.search[id]);
            }
        }
    }
    for (int e = 0; e < m_stride; ++e) {
        if (succ[e] < 0) {
            continue;
        }
        const bool is_goal = (succ[e] & SMPLGPU_LATTICE_GOAL_FLAG) != 0;   // ManipLattice::isGoal, on the device
        const int succ_id = succ[e] & ~SMPLGPU_LATTICE_GOAL_FLAG;
        if (is_goal && (Q.goal_succ.empty() || Q.goal_succ.back().expanded != Q.expanding)) {
            // first valid goal action of this expansion; a goal-flagged h word is the reached record's index
            Q.goal_succ.push_back(Query::GoalAction{ Q.expanding, succ_id, h[e] });
        }
        const int target = is_goal ? 0 : succ_id;
        sstate(Q, target);
        touch(Q, target, h[e]);
        SState& ss = Q.search[target];
        const int k = e - m_snap_words;   // primitive index; negative = a snap
        const int edge_cost = k < 0 ? m_snap_cost : ((size_t)k < edge_costs.size() ? edge_costs[k] : 1000);
        const int new_cost = Q.search[Q.expanding].eg + edge_cost;
        if ((unsigned int)new_cost < ss.g) {   // int vs unsigned, compared as unsigned (arastar.cpp:545-548)
            ss.g = new_cost;
            ss.bp = Q.expanding;
            if (ss.iteration_closed != 1) {
                ss.f = computeKey(ss);
                if (ss.heap_index != 0) {
                    Q.open[ss.heap_index].f = ss.f;
                    percolateUp(Q, (size_t)ss.heap_index);
                } else {
                    heapPush(Q, target);
                }
            }
        }
    }
    // the state this query expands next round (unless a better one arrives)
    if (Q.open.size() > 1) {
        __builtin_prefetch(&Q.search[Q.open[1].id]);
    }
}

///////////////////////////////////////////////////////////////////////////////
// the lock-step driver
///////////////////////////////////////////////////////////////////////////////

bool BatchPlanner::plan(const double* starts, const double* goals, int nq, std::vector<QueryResult>& out, std::string* err)
{
    std::vector<smplgpu_goal> recs(nq);
    for (int i = 0; i < nq; ++i) {
        smplgpu_goal& g = recs[i];   // zero-filled
        g.type = SMPLGPU_GOAL_XYZ;
        for (int a = 0; a < 3; ++a) {
            g.pose[a] = goals[3 * (size_t)i + a];
            g.xyz_tolerance[a] = m_cfg.xyz_tolerance[a];
        }
    }
    return plan(starts, recs.data(), nq, out, err);
}

bool BatchPlanner::plan(const double* starts, const smplgpu_goal* goals, int nq, std::vector<QueryResult>& out, std::string* err)
{
    return plan(starts, goals, nullptr, nq, out, err);
}

bool BatchPlanner::plan(const double* starts, const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
                        std::vector<QueryResult>& out, std::string* err)
{
    out.assign(nq, QueryResult());
    m_stats = BatchStats();
    if (nq == 0) {
        return true;
    }
    const int dof = m_cfg.dof;
    Timer t;
    auto fail_dev = [&]() {
        if (err) *err = smplgpu_last_error(m_ctx);
        return false;
    };
    // query i's goal set: records set_begin(i) .. set_begin(i + 1) - 1
    auto set_begin = [&](int i) { return goal_offsets ? goal_offsets[i] : i; };
    const int n_rec = set_begin(nq);
    // where each query's BFS is seeded: the goal position of every record of its set, for a joint goal the
    // target-offset position of its angles (ManipLattice::setGoalConfiguration), all joint goals in one device call
    std::vector<double> goal_xyz((size_t)n_rec * 3);
    {
        std::vector<int> joint;
        std::vector<double> angles;
        for (int i = 0; i < n_rec; ++i) {
            if (goals[i].type == SMPLGPU_GOAL_JOINT_STATE) {
                joint.push_back(i);
                angles.insert(angles.end(), goals[i].angles, goals[i].angles + dof);
            } else {
                std::copy(goals[i].pose, goals[i].pose + 3, goal_xyz.begin() + 3 * (size_t)i);
            }
        }
        if (!joint.empty()) {
            std::vector<double> pose6(joint.size() * 6);
            if (smplgpu_planning_frame_fk(m_ctx, angles.data(), (int)joint.size(), pose6.data()) < 0) return fail_dev();
            ++m_stats.device_calls;
            for (size_t k = 0; k < joint.size(); ++k) {
                std::copy(pose6.begin() + 6 * k, pose6.begin() + 6 * k + 3, goal_xyz.begin() + 3 * (size_t)joint[k]);
            }
        }
    }
    const long long resolved0 = smplgpu_expand_batch_resolved(m_ctx);
    int64_t ik0[6] = { 0, 0, 0, 0, 0, 0 };
    if (m_snap_words && smplgpu_lattice_snap_counters_by_kind(m_ctx, ik0) < 0) return fail_dev();
    // a query creates at most (its expansions) x (successors per expansion) states besides the goal and the start
    const long long want_states = 2 + (long long)std::max(0, m_cfg.max_expansions) * std::max(1, m_stride);
    const int max_states = (int)std::min<long long>(want_states, 1LL << 26);
    // the BFS bank keeps the reference's int node indices, and bank and lattices have to fit in device memory
    const int max_slots = smplgpu_bfs_bank_max_slots(m_ctx);
    if (max_slots < 0) return fail_dev();
    const int max_lat = smplgpu_lattice_max_slots(m_ctx, max_states);
    if (max_lat < 0) return fail_dev();
    const int n_slots = std::min(std::min(std::min(m_max_concurrent, nq), max_slots), max_lat);
    if (smplgpu_bfs_bank_create(m_ctx, n_slots, m_cfg.inflation_radius) < 0) return fail_dev();
    // every device / pinned allocation happens here: allocating while other planner threads run would stall
    // their streams (allocation synchronises the device)
    {
        smplgpu_lattice_params lp;
        lp.resolutions = m_cfg.resolutions.data();
        lp.deltas = m_prim_deltas.data();
        lp.prim_short = m_prim_short.data();
        lp.n_prims = (int)m_prim_short.size();
        lp.use_short_dist = m_cfg.use_short_dist ? 1 : 0;
        lp.short_dist_thresh = m_cfg.short_dist_thresh;
        for (int a = 0; a < 3; ++a) lp.xyz_tolerance[a] = m_cfg.xyz_tolerance[a];
        lp.cost_per_cell = m_cfg.cost_per_cell;
        lp.max_states = max_states;
        int stride = smplgpu_lattice_create(m_ctx, &lp, n_slots);
        if (stride < 0) return fail_dev();
        if (m_snap_words) {
            smplgpu_snap_kinds sk;
            for (int k = 0; k < 3; ++k) {
                sk.enabled[k] = m_cfg.snap[k] ? 1 : 0;
                sk.dist_thresh[k] = m_cfg.snap_dist_thresh[k];
            }
            sk.ik = m_cfg.ik;
            stride = smplgpu_lattice_set_snaps(m_ctx, &sk);
            if (stride < 0) return fail_dev();
        }
        if (stride != m_stride) {
            if (err) *err = "lattice stride mismatch";
            return false;
        }
    }
    if (smplgpu_expand_batch_reserve(m_ctx, n_slots + 1) < 0) return fail_dev();   // setStart's batch
    ++m_stats.device_calls;
    {
        const double dt = t.lap();
        m_stats.device_seconds += dt;
        m_stats.setup_seconds += dt;
    }

    Pool pool(m_cfg.n_threads);
    std::vector<Query> S(n_slots);          // slot -> query occupying it
    std::vector<char> occupied(n_slots, 0);
    int next_query = 0, finished = 0;
    // refill in groups so that one bank run (one wavefront launch sequence) serves several new queries
    const int refill_min = std::max(1, n_slots / 4);

    // The active queries work in NG groups (slot modulo NG).  While the device expands one group's round the host
    // absorbs the other groups' results and pops their next states, so host and device overlap.
    struct Group
    {
        std::vector<int> active;            // occupied slots of this group with a search in progress
        std::vector<int32_t> slot, parent;  // this round's expansions
        std::vector<int> owner;             // expansion -> index into `active`
        const int32_t* succ = nullptr;      // results of the round in flight (page-locked memory of the context)
        const int32_t* h = nullptr;
        const int32_t* count = nullptr;
        bool in_flight = false;
        int ne = 0;
    };
    static const int NG = [] {
        const char* e = getenv("SMPLHOST_PLAN_GROUPS");
        const int v = e ? atoi(e) : 2;
        return std::min(std::max(v, 2), (int)SMPLGPU_EXPAND_BUFFERS);
    }();
    std::vector<Group> G(NG);
    auto all_idle = [&]() {
        for (const Group& g : G) {
            if (!g.active.empty()) return false;
        }
        return true;
    };
    // SMPLHOST_PLAN_PROFILE=1: where the host time of this planner thread goes (printed to stderr at the end)
    static const bool profile = getenv("SMPLHOST_PLAN_PROFILE") != nullptr;
    double prof[6] = { 0, 0, 0, 0, 0, 0 };  // absorb, retire, expand, pack, submit, refill
    Timer pt;
    std::vector<double> sq;                 // setStart scratch
    std::vector<int32_t> sh, sgd;
    std::vector<uint8_t> sv;
    std::vector<double> soff;

    // wait for a group's round, relax its queries, retire the finished ones
    auto absorb = [&](int gi) -> bool {
        Group& g = G[gi];
        if (g.in_flight) {
            m_stats.host_seconds += t.lap();
            if (smplgpu_lattice_expand_wait(m_ctx, gi, &g.succ, &g.h, &g.count) < 0) return false;
            {
                const double dt = t.lap();
                m_stats.device_seconds += dt;
                m_stats.max_wait_seconds = std::max(m_stats.max_wait_seconds, dt);
            }
            g.in_flight = false;
            const int ne = g.ne;
            pt.lap();
            pool.run([&](int tid) {
                for (int k = tid; k < ne; k += pool.size()) {
                    Query& Q = S[g.active[g.owner[k]]];
                    absorbOne(Q, g.succ + (size_t)k * m_stride, g.h + (size_t)k * m_stride, g.count[k]);
                }
            });
            prof[0] += pt.lap();
        }
        pt.lap();
        size_t keep = 0;
        for (size_t k = 0; k < g.active.size(); ++k) {
            const int s = g.active[k];
            if (S[s].done) {
                if (S[s].result.success && m_cfg.want_path_states) {
                    m_stats.host_seconds += t.lap();
                    if (!fetchPathStates(S[s], err)) return false;   // while the query still owns its slot
                    m_stats.device_seconds += t.lap();
                    ++m_stats.device_calls;
                }
                out[S[s].index] = S[s].result;
                occupied[s] = 0;
                ++finished;
            } else {
                g.active[keep++] = s;
            }
        }
        g.active.resize(keep);
        prof[1] += pt.lap();
        return true;
    };

    // every active query of the group pops one state; one device round expands them all
    auto expand = [&](int gi) -> bool {
        Group& g = G[gi];
        const int na = (int)g.active.size();
        if (na == 0) {
            return true;
        }
        pt.lap();
        pool.run([&](int tid) {
            for (int k = tid; k < na; k += pool.size()) {
                Query& Q = S[g.active[k]];
                if (!Q.done) {
                    expandOne(Q);
                }
            }
        });
        prof[2] += pt.lap();
        g.slot.clear();
        g.parent.clear();
        g.owner.clear();
        for (int k = 0; k < na; ++k) {
            Query& Q = S[g.active[k]];
            if (Q.done) {
                continue;   // retired by the next absorb
            }
            Q.edge_begin = (int)g.slot.size();
            g.slot.push_back(Q.slot);
            g.parent.push_back(Q.expanding);
            g.owner.push_back(k);
        }
        g.ne = (int)g.slot.size();
        prof[3] += pt.lap();
        if (g.ne == 0) {
            return true;
        }
        if (smplgpu_lattice_expand_submit(m_ctx, g.slot.data(), g.parent.data(), g.ne, gi) < 0) return false;
        prof[4] += pt.lap();
        g.in_flight = true;
        ++m_stats.device_calls;
        ++m_stats.rounds;
        m_stats.edges_submitted += (long long)g.ne * m_stride;
        return true;
    };

    // Admission in two steps: (1) setGoal -- a free slot gets the query's goal and its BFS is queued on the device
    // WITHOUT waiting (the reference's BFS_3D also searches in a background thread, bfs3d.cpp:156-201), the running
    // searches keep expanding; (2) when that BFS is done, setStart (limits, validity, heuristic of the start state,
    // a fresh device lattice holding it) and the queries join the rounds.  One group of pending slots at a time.
    std::vector<int32_t> pending;           // slots whose BFS is in flight
    std::vector<int32_t> seeds, seed_offsets;
    bool first_fill = true;

    auto activate = [&]() -> bool {
        // setStart uses the synchronous entry points: nothing of ours may be in flight
        for (int gi = 0; gi < NG; ++gi) {
            if (!absorb(gi)) return false;
        }
        m_stats.host_seconds += t.lap();
        if (smplgpu_bfs_bank_run_wait(m_ctx) < 0) return false;
        const int nn = (int)pending.size();
        sq.resize((size_t)nn * dof);
        for (int k = 0; k < nn; ++k) {
            const int qi = S[pending[k]].index;
            std::copy(starts + (size_t)qi * dof, starts + (size_t)(qi + 1) * dof, sq.begin() + (size_t)k * dof);
        }
        sv.resize(nn);
        sh.resize(nn);
        sgd.resize(nn);
        soff.resize((size_t)nn * 3);
        std::vector<uint8_t> dummy(nn);
        if (smplgpu_is_states_valid(m_ctx, sq.data(), nn, sv.data()) < 0) return false;
        if (smplgpu_expand_batch(m_ctx, sq.data(), sq.data(), pending.data(), nn, m_cfg.cost_per_cell,
                                 dummy.data(), sh.data(), sgd.data(), soff.data()) < 0) return false;
        m_stats.device_calls += 2;
        // the valid starts become state 1 of a fresh lattice in their slot
        std::vector<int32_t> bslot, bgd, boff(1, 0);
        std::vector<double> bq;
        std::vector<smplgpu_goal> bgoal;
        for (int k = 0; k < nn; ++k) {
            Query& Q = S[pending[k]];
            const double* qs = &sq[(size_t)k * dof];
            G[pending[k] % NG].active.push_back(pending[k]);
            if (!checkJointLimits(qs) || !sv[k]) {
                finish(Q, false);   // retired by the group's next absorb
                continue;
            }
            bslot.push_back(pending[k]);
            bgd.push_back(sgd[k]);
            bq.insert(bq.end(), qs, qs + dof);
            bgoal.insert(bgoal.end(), Q.goals, Q.goals + Q.n_goals);
            boff.push_back((int32_t)bgoal.size());
            Q.num_states = 2;
            sstate(Q, 1);
            touch(Q, 1, sh[k]);
            touch(Q, 0, 0);
            Q.search[1].g = 0;
            Q.search[1].f = computeKey(Q.search[1]);
            heapPush(Q, 1);
        }
        if (!bslot.empty()) {
            if (smplgpu_lattice_begin_goal_sets(m_ctx, bslot.data(), bq.data(), bgd.data(), bgoal.data(), boff.data(),
                                                (int)bslot.size()) < 0) return false;
            ++m_stats.device_calls;
        }
        {
            const double dt = t.lap();
            m_stats.device_seconds += dt;
            m_stats.setup_seconds += dt;
        }
        pending.clear();
        return true;
    };

    while (finished < nq) {
        const bool idle = all_idle();
        // ---- (2) the pending queries' BFS is done (or there is nothing else to do): setStart, join the rounds ----
        if (!pending.empty() && (idle || smplgpu_bfs_bank_run_done(m_ctx) != 0)) {
            if (!activate()) return fail_dev();
            continue;
        }
        // ---- (1) hand free slots to waiting queries: setGoal (one BFS per query, queued) ----
        int n_free = 0;
        for (int s = 0; s < n_slots; ++s) n_free += occupied[s] ? 0 : 1;
        if (pending.empty() && next_query < nq && (n_free >= refill_min || idle)) {
            // the first group is kept small so that the searches start while the other slots' BFS still runs
            // (SMPLHOST_ADMIT_CHUNKS overrides)
            static const int chunks = getenv("SMPLHOST_ADMIT_CHUNKS") ? std::max(1, atoi(getenv("SMPLHOST_ADMIT_CHUNKS"))) : 2;
            const int take = (first_fill || chunks > 4) ? std::max(1, n_slots / chunks) : n_slots;
            first_fill = false;
            seeds.clear();
            seed_offsets.assign(1, 0);
            for (int s = 0; s < n_slots && next_query < nq && (int)pending.size() < take; ++s) {
                if (occupied[s]) {
                    continue;
                }
                const int r0 = set_begin(next_query), r1 = set_begin(next_query + 1);
                initQuery(S[s], next_query, s, goals + r0, r1 - r0, &goal_xyz[3 * (size_t)r0]);
                ++next_query;
                occupied[s] = 1;
                pending.push_back(s);
                // BfsHeuristic::updateGoal over all the set's positions: BFS_3D::run(begin, end)
                for (int r = r0; r < r1; ++r) {
                    int cell[3];
                    worldToGrid(&goal_xyz[3 * (size_t)r], cell);
                    seeds.insert(seeds.end(), cell, cell + 3);
                }
                seed_offsets.push_back((int32_t)(seeds.size() / 3));
            }
            m_stats.host_seconds += t.lap();
            if (smplgpu_bfs_bank_run_slots_multi_async(m_ctx, pending.data(), seeds.data(), seed_offsets.data(),
                                                       (int)pending.size()) < 0) return fail_dev();
            ++m_stats.bfs_runs;
            ++m_stats.device_calls;
            {
                const double dt = t.lap();
                m_stats.device_seconds += dt;
                m_stats.setup_seconds += dt;
            }
            if (all_idle()) {
                continue;   // nothing to expand meanwhile: go and wait for it
            }
        }

        // ---- one pipelined round: each group absorbs its previous round and submits the next ----
        for (int gi = 0; gi < NG; ++gi) {
            if (!absorb(gi)) return fail_dev();
            if (!expand(gi)) return fail_dev();
        }
        m_stats.host_seconds += t.lap();
    }
    if (profile) {
        fprintf(stderr, "[plan profile] rounds %d successor slots %lld: absorb %.3f retire %.3f pop %.3f pack %.3f submit %.3f | "
                        "device wait %.3f setup %.3f host %.3f s\n", m_stats.rounds, m_stats.edges_submitted, prof[0], prof[1],
                prof[2], prof[3], prof[4], m_stats.device_seconds - m_stats.setup_seconds, m_stats.setup_seconds,
                m_stats.host_seconds);
    }
    m_stats.edges_resolved_f64 = smplgpu_expand_batch_resolved(m_ctx) - resolved0;
    if (m_snap_words) {
        int64_t ik1[6];
        if (smplgpu_lattice_snap_counters_by_kind(m_ctx, ik1) < 0) return fail_dev();
        for (int k = 0; k < 3; ++k) {
            m_stats.ik_attempted[k] = ik1[2 * k] - ik0[2 * k];
            m_stats.ik_converged[k] = ik1[2 * k + 1] - ik0[2 * k + 1];
        }
    }
    // nothing can be in flight here: a group's queries finish in absorb or expand, and a round is only submitted for
    // queries that are not done; drain defensively anyway
    for (int gi = 0; gi < NG; ++gi) {
        if (G[gi].in_flight) {
            if (smplgpu_lattice_expand_wait(m_ctx, gi, &G[gi].succ, &G[gi].h, &G[gi].count) < 0) return fail_dev();
        }
    }
    return true;
}

} // namespace smplhost
