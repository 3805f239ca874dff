// Host side of the caller of the hot path, B200-first: MANY independent ARA* searches on the
// manipulation lattice advance in lock step, and every round submits ONE expansion per active
// query to the device (smplgpu_lattice_expand_*): 8 bytes go out per expansion (bank slot, state
// id), one word pair per successor comes back (state id | goal flag, heuristic).  Successor
// generation, joint limits, edge validity, stateToCoord, the coordinate hash table
// (getOrCreateState), the goal test and the heuristic run on the device (csrc/lattice.cuh); the
// host keeps ARA* -- the OPEN lists and the search states -- indexed by the device's state ids.
//
// It mirrors, per query, the reference's
//   ManipLattice::GetSuccs / checkAction / isGoal / stateToCoord   smpl/src/graph/manip_lattice.cpp:219-313, 1263-1289, 1511-1580, 1673-1687
//   ManipLatticeActionSpace::apply / mprimActive                   smpl/src/graph/manip_lattice_action_space.cpp:376-449, 662-691
//   ARAStar::replan / improvePath / expand / computeKey            smpl/src/search/arastar.cpp:107-215, 486-568, 579-582
//   intrusive_heap                                                 smpl/include/smpl/detail/intrusive_heap.hpp
// so that each query returns the same path, cost and expansion count as the reference-shaped
// sequential planner (first solution at the initial epsilon; see SURVEY.md section 8 defect 2 for
// the motion-primitive format and goal type decisions).  Round 1 kept the hash tables and the lattice states on
// the host as well; with hundreds of megabyte-sized lattices taking turns on a core, their cache misses bounded
// plan queries/s by the host cores (DESIGN.md section 5), so they moved next to the kernels that fill them.
#ifndef SMPLHOST_BATCH_PLANNER_H
#define SMPLHOST_BATCH_PLANNER_H

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <cstdint>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../include/smplgpu.h"

namespace smplhost {

struct PlannerConfig
{
    int dof = 0;
    std::vector<double> resolutions;
    std::vector<double> mprims;         // n_prims x dof deltas, file order (converses are added here)
    std::vector<uint8_t> short_flags;   // n_prims
    // per-primitive action weight (the `weight` column of this fork's primitive files, manip_lattice_action_space.cpp:
    // 182-190): an edge costs (int)(1000 * weight) (manip_lattice.cpp:1414-1437); empty = 1 for every primitive
    std::vector<double> prim_weights;   // n_prims, or empty
    bool use_short_dist = true;
    double short_dist_thresh = 0.4;
    double epsilon = 100.0;
    int max_expansions = 200000;
    double xyz_tolerance[3] = { 0.015, 0.015, 0.015 };
    int cost_per_cell = 100;
    double inflation_radius = 0.02;
    // joint limits as KDLRobotModel reports them (min/max/continuous per planning variable)
    std::vector<double> var_min, var_max;
    std::vector<int> var_continuous;
    // grid geometry for host-side worldToGrid of the goal
    double origin[3] = { 0, 0, 0 };
    double res = 0.02;
    int dims[3] = { 0, 0, 0 };
    // host threads for the per-query work (OPEN list updates); queries are independent, so the result does not
    // depend on this
    int n_threads = 1;
    // fetch the joint values along every found path from the device (ManipLattice::extractPath)
    bool want_path_states = true;
    // the snap actions SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY (smplgpu_lattice_set_snaps), by SMPLGPU_SNAP_*
    // kind: each active within its own snap_dist_thresh metres of metric goal distance; every kind costs
    // (int)(1000 * snap_weight) (the fork registers them with weight 0.5) and solves with the same IK parameters
    bool snap[3] = { false, false, false };
    double snap_dist_thresh[3] = { 0.0, 0.0, 0.0 };
    double snap_weight = 0.5;
    smplgpu_ik_params ik = { 100, 1e-6 };
};

struct QueryResult
{
    bool success = false;
    int expansions = 0;
    int cost = 0;
    int num_states = 0;
    std::vector<int> path_ids;
    // ManipLattice::extractPath (manip_lattice.cpp:2018-2160): the joint-space state of every path id; the goal id
    // is replaced by the lattice state of the first valid goal-reaching action of its predecessor
    std::vector<double> path_states;   // path_ids.size() x dof
    // the index, in the query's goal set, of the first record that the goal-reaching action of the path satisfies
    // (the action extractPath selects); -1 when the query is unsolved
    int reached_goal = -1;
};

struct BatchStats
{
    int rounds = 0;
    int bfs_runs = 0;              // bank runs (each covers every slot that was refilled at that point)
    long long edges_submitted = 0;
    long long edges_resolved_f64 = 0;   // of those, decided by the double-precision kernels
    long long device_calls = 0;
    double device_seconds = 0.0;   // time inside smplgpu_* calls
    double host_seconds = 0.0;     // everything else
    double setup_seconds = 0.0;    // of device_seconds: bank creation, BFS bank runs, setStart (per refill)
    double max_wait_seconds = 0.0; // longest single wait for an expansion batch
    long long ik_attempted[3] = { 0, 0, 0 };   // IK solves of the snap actions by SMPLGPU_SNAP_* kind, and how many
    long long ik_converged[3] = { 0, 0, 0 };   // converged
};

class BatchPlanner
{
public:
    BatchPlanner(smplgpu_ctx* ctx, const PlannerConfig& cfg, int max_concurrent);

    /// starts: nq x dof, goals: nq x 3 (target-offset position in the planning frame); XYZ goals with
    /// PlannerConfig::xyz_tolerance
    bool plan(const double* starts, const double* goals, int nq, std::vector<QueryResult>& out, std::string* err);
    /// the same with one GoalConstraint per query (types may be mixed)
    bool plan(const double* starts, const smplgpu_goal* goals, int nq, std::vector<QueryResult>& out, std::string* err);
    /// the same with a goal set per query: query i succeeds at any of goals[goal_offsets[i] .. goal_offsets[i + 1] - 1]
    /// (1 to SMPLGPU_MAX_GOAL_SET records, checked by the caller; goal_offsets null = one record per query)
    bool plan(const double* starts, const smplgpu_goal* goals, const int32_t* goal_offsets, int nq,
              std::vector<QueryResult>& out, std::string* err);

    const BatchStats& stats() const { return m_stats; }

private:
    // g, h, f, eg are unsigned as in the reference's ARAStar::SearchState (arastar.h:176-187): a negative heuristic
    // (unreachable BFS cell: cost_per_cell * -1) sorts last in OPEN
    struct SState { unsigned int g, h, f, eg; int iteration_closed, bp, heap_index; bool touched; };
    struct Query
    {
        int index;
        int slot;
        const smplgpu_goal* goals;   // the goal set
        int n_goals;
        const double* goal_xyz;      // [n_goals][3] where the BFS is seeded: each record's goal position, for a joint
                                     // record that of its angles
        int goal_h;
        int num_states;        // lattice size on the device (ids handed out so far, goal and start included)
        std::vector<SState> search;
        // 1-based binary heap of (f, state id): the key travels with the entry so that sifting reads one
        // contiguous array instead of one search state per comparison (same comparisons as intrusive_heap.h)
        struct HeapEntry { unsigned int f; int id; };
        std::vector<HeapEntry> open;
        int expanding;         // state popped this round
        bool done;
        QueryResult result;
        // (expanded state, lattice id of its first valid successor that satisfied the goal, the index of the record
        // it satisfied first): what extractPath's "cheapest valid goal action" search finds, every action costing the
        // same (manip_lattice.cpp:2098-2124)
        struct GoalAction { int expanded, succ, reached; };
        std::vector<GoalAction> goal_succ;
        int edge_begin;        // index of this query's expansion in its group's round
    };

    // minimal fork-join pool: run(f) calls f(tid) on every thread (the caller is tid 0)
    class Pool
    {
    public:
        explicit Pool(int n);
        ~Pool();
        void run(const std::function<void(int)>& f);
        int size() const { return m_n; }
    private:
        int m_n;
        std::vector<std::thread> m_threads;
        std::atomic<int> m_generation{ 0 };
        std::atomic<int> m_done{ 0 };
        std::atomic<bool> m_stop{ false };
        std::atomic<int> m_sleepers{ 0 };
        std::mutex m_mutex;
        std::condition_variable m_cv;
        const std::function<void(int)>* m_job = nullptr;
        void worker(int tid);
    };

    smplgpu_ctx* m_ctx;
    PlannerConfig m_cfg;
    int m_max_concurrent;
    std::vector<double> m_prim_deltas;     // [n_prims][dof], converses included
    std::vector<uint8_t> m_prim_short;
    std::vector<int> m_cost_long, m_cost_short;   // edge cost of the j-th active long / short primitive (converses included)
    int m_stride = 0;                      // successor words per expansion (the snaps' first when enabled)
    int m_snap_words = 0;                  // the number of enabled snap kinds
    int m_snap_cost = 0;
    BatchStats m_stats;

    bool checkJointLimits(const double* q) const;
    void worldToGrid(const double* p, int* cell) const;
    int computeKey(const SState& s) const;
    SState& sstate(Query& Q, int id);
    void touch(Query& Q, int id, int h);
    void heapPush(Query& Q, int id);
    void heapPop(Query& Q);
    void percolateUp(Query& Q, size_t pivot);
    void percolateDown(Query& Q, size_t pivot);
    void finish(Query& Q, bool found);
    void initQuery(Query& Q, int index, int slot, const smplgpu_goal* goals, int n_goals, const double* goal_xyz);
    static const Query::GoalAction* goalAction(const Query& Q, int expanded);
    void expandOne(Query& Q);   // pop the next state (no device work)
    void absorbOne(Query& Q, const int32_t* succ, const int32_t* h, int count);
    bool fetchPathStates(Query& Q, std::string* err);
};

} // namespace smplhost

#endif
