// ORACLE (test infrastructure only -- never linked into the product path).
//
// The three adaptive actions of ManipLatticeActionSpace -- SNAP_TO_RPY, SNAP_TO_XYZ and SNAP_TO_XYZ_RPY, each enabled
// on its own with its own distance threshold -- in the goal-set planner (the project's own definition; DESIGN.md
// section 2: parity unpinned, pinned oracle <-> device).  SnapKindsLatticePlanner is
// oracle/goal_sets/goal_set_lattice.cpp's GoalSetLatticePlanner with these rules, and nothing else changed:
//   getSuccs       the enabled kinds come first, in the order SNAP_RPY, SNAP_XYZ, SNAP_XYZ_RPY, each active when the
//                  parent's metric goal distance is within its threshold; all aim at the record nearest to the parent
//                  (nearestRecord); a kind that does not apply to that record's type produces nothing
//                    SNAP_XYZ_RPY  (XYZ, XYZ_RPY, JOINT_STATE) the goal-set planner's snap, unchanged
//                    SNAP_XYZ      (XYZ, XYZ_RPY) the position-only IK (planningLinkIkPosition) for the record's
//                                  position, seeded at the parent, the orientation free
//                    SNAP_RPY      (XYZ_RPY) planningLinkIk for the parent's own target-offset position and the
//                                  record's rotation, seeded at the parent: the orientation turned in place
//                  every snap answer is checked like any action (joint limits, then isStateToStateValid) and costs
//                  (int)(1000 snap_weight); the IK parameters are shared
//   extractPath    the snaps are re-run in kind order and the first valid goal-reaching one is taken, before any
//                  primitive
// With SNAP_XYZ_RPY alone it plans as oracle_plan_goal_set (tests/test_oracle_snap_kinds.py pins the two against each
// other).  smpl_b200/csrc/ik.cuh restates planningLinkIkPosition (ik_warp<3>) and the snap kinds
// (lattice_snap_kernel).
//
// Built as oracle/snap_kinds/liboracle_snap_kinds.so over oracle/liboracle.so; it takes the scene handles of the
// oracle's C API.  The goal-set planner's source is included unchanged for the goal records, the goal-set rules, the
// IK and the snap settings; the library therefore also exports that source's entry points.
#include "../goal_sets/goal_set_lattice.cpp"

namespace {

enum { SNAP_RPY = 0, SNAP_XYZ = 1, SNAP_XYZ_RPY = 2 };   // SMPLGPU_SNAP_*: the successor word order

// planningLinkIk with the position rows alone: e = target_p - pt, the 3 x dof position block Jp of the Jacobian,
// step = Jp^T (Jp Jp^T + IK_LAMBDA^2 I)^-1 e by a 3 x 3 Cholesky, converged when |e_i| <= tolerance for the three
// rows; the chain, the target point, the columns, the clamping and the wrapping are planningLinkIk's.  The orientation
// is free.  Returns converged; *iterations = steps taken.
bool planningLinkIkPosition(const KDLRobotModel& m, const KdlFrame& Tk, const double offset[3], const double target_p[3],
                            const IkParams& prm, std::vector<double>& q, int* iterations)
{
    const int dof = (int)q.size();
    const int nseg = m.planning_segment_nr;
    std::vector<KdlFrame> prefix(nseg + 1);
    std::vector<double> J(3 * (size_t)dof, 0.0);   // row-major 3 x dof; variables beyond the chain keep 0 columns
    for (int it = 0;; ++it) {
        KdlFrame f1 = KdlFrame::Identity();
        for (int s = 0; s < nseg; ++s) {
            prefix[s] = f1;
            f1 = f1 * segmentPose(m, s, q);
        }
        const KdlFrame f = Tk * f1;
        double pt[3], e[3];
        for (int i = 0; i < 3; ++i) {
            pt[i] = (f.M[3 * i] * offset[0] + f.M[3 * i + 1] * offset[1] + f.M[3 * i + 2] * offset[2]) + f.p[i];
            e[i] = target_p[i] - pt[i];
        }
        bool conv = true;
        for (int i = 0; i < 3; ++i) {
            conv = conv && std::fabs(e[i]) <= prm.tolerance;   // false for NaN
        }
        if (conv || it == prm.max_iterations) {
            *iterations = it;
            return conv;
        }
        for (int s = 0; s < nseg; ++s) {
            const KDLRobotModel::Segment& seg = m.segments[s];
            if (seg.q_index < 0 || seg.joint_kind == 0) {
                continue;
            }
            const KdlFrame W = Tk * prefix[s];
            double a[3], o[3];
            for (int i = 0; i < 3; ++i) {
                a[i] = (W.M[3 * i] * seg.axis[0] + W.M[3 * i + 1] * seg.axis[1]) + W.M[3 * i + 2] * seg.axis[2];
                o[i] = ((W.M[3 * i] * seg.origin[0] + W.M[3 * i + 1] * seg.origin[1]) + W.M[3 * i + 2] * seg.origin[2]) + W.p[i];
            }
            double col[3];
            if (seg.joint_kind == 1) {
                const double d0 = pt[0] - o[0], d1 = pt[1] - o[1], d2 = pt[2] - o[2];
                col[0] = a[1] * d2 - a[2] * d1;
                col[1] = a[2] * d0 - a[0] * d2;
                col[2] = a[0] * d1 - a[1] * d0;
            } else {
                col[0] = a[0]; col[1] = a[1]; col[2] = a[2];
            }
            for (int r = 0; r < 3; ++r) {
                J[(size_t)r * dof + seg.q_index] = col[r];
            }
        }
        double A[3][3], L[3][3], x[3], y[3];
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c <= r; ++c) {
                double acc = 0.0;
                for (int v = 0; v < dof; ++v) {
                    acc = acc + J[(size_t)r * dof + v] * J[(size_t)c * dof + v];
                }
                A[r][c] = r == c ? acc + IK_LAMBDA * IK_LAMBDA : acc;
            }
        }
        for (int j = 0; j < 3; ++j) {
            double d = A[j][j];
            for (int k = 0; k < j; ++k) {
                d = d - L[j][k] * L[j][k];
            }
            L[j][j] = std::sqrt(d);
            for (int i = j + 1; i < 3; ++i) {
                double t = A[i][j];
                for (int k = 0; k < j; ++k) {
                    t = t - L[i][k] * L[j][k];
                }
                L[i][j] = t / L[j][j];
            }
        }
        for (int i = 0; i < 3; ++i) {
            double t = e[i];
            for (int k = 0; k < i; ++k) {
                t = t - L[i][k] * y[k];
            }
            y[i] = t / L[i][i];
        }
        for (int i = 2; i >= 0; --i) {
            double t = y[i];
            for (int k = i + 1; k < 3; ++k) {
                t = t - L[k][i] * x[k];
            }
            x[i] = t / L[i][i];
        }
        for (int v = 0; v < dof; ++v) {
            double dq = 0.0;
            for (int r = 0; r < 3; ++r) {
                dq = dq + J[(size_t)r * dof + v] * x[r];
            }
            double nq = q[v] + dq;
            if (m.continuous[v]) {
                nq = normalize_angle(nq);
            } else {
                nq = nq < m.min_limits[v] ? m.min_limits[v] : (nq > m.max_limits[v] ? m.max_limits[v] : nq);
            }
            q[v] = nq;
        }
    }
}

// the settings and counters of the three kinds, by SNAP_* index (cost, IK parameters and Tk the same in all three)
struct SnapKinds
{
    Snap kind[3];
};

class SnapKindsLatticePlanner
{
public:
    SnapKindsLatticePlanner(oracle_scene* s, const std::vector<double>& resolutions, const std::vector<Prim>& prims,
                       bool use_short_dist, double short_dist_thresh, double epsilon, int max_expansions,
                       SnapKinds* snaps) :
        m_cc(s->cc.get()), m_robot(s->kdl.get()), m_heur(s->heur.get()), m_prims(), m_use_short_dist(use_short_dist),
        m_short_dist_thresh(short_dist_thresh), m_epsilon(epsilon), m_max_expansions(max_expansions), m_snaps(snaps),
        m_df(s->df.get())
    {
        for (int i = 0; i < 3; ++i) m_xyz_offset[i] = s->xyz_offset[i];
        // addMotionPrim(..., add_converse = true): each primitive is followed by its negation
        for (const Prim& p : prims) {
            m_prims.push_back(p);
            Prim neg = p;
            for (double& v : neg.delta) v *= -1.0;
            m_prims.push_back(neg);
        }
        // ManipLattice::init (manip_lattice.cpp:105-146)
        const size_t n = m_robot->min_limits.size();
        m_min_limits = m_robot->min_limits;
        m_continuous.resize(n);
        m_bounded.resize(n);
        m_coord_vals.resize(n);
        m_coord_deltas.resize(n);
        for (size_t v = 0; v < n; ++v) {
            m_continuous[v] = m_robot->continuous[v];
            m_bounded[v] = !m_robot->continuous[v];
            const double res = resolutions[v];
            if (m_continuous[v]) {
                m_coord_vals[v] = (int)std::round((2.0 * M_PI) / res);
                m_coord_deltas[v] = (2.0 * M_PI) / (double)m_coord_vals[v];
            } else if (m_bounded[v]) {
                const double span = std::fabs(m_robot->max_limits[v] - m_min_limits[v]);
                m_coord_vals[v] = std::max(1, (int)std::round(span / res));
                m_coord_deltas[v] = span / (double)m_coord_vals[v];
            } else {
                m_coord_vals[v] = std::numeric_limits<int>::max();
                m_coord_deltas[v] = res;
            }
        }
    }

    // *reached: the index of the first record that the path's goal-reaching action satisfies, -1 when unsolved
    Result plan(const std::vector<double>& start, const std::vector<Goal>& goals, int* reached)
    {
        Result res;
        m_states.clear();
        m_coord_to_id.clear();
        m_goals = goals;
        m_reached = -1;
        *reached = -1;
        m_goal_xyz.assign(3 * goals.size(), 0.0);
        m_goal_in_grid = false;
        std::vector<int> cells;
        for (size_t r = 0; r < goals.size(); ++r) {
            if (goals[r].type == JOINT_STATE_GOAL) {
                std::vector<double> pose;   // ManipLattice::setGoalConfiguration: the target offset pose of the angles
                m_robot->computePlanningLinkFK(goals[r].angles, pose);
                pose = GetTargetOffsetPose(pose, m_xyz_offset);
                for (int i = 0; i < 3; ++i) m_goal_xyz[3 * r + i] = pose[i];
            } else {
                for (int i = 0; i < 3; ++i) m_goal_xyz[3 * r + i] = goals[r].pose[i];
            }
            int c[3];
            m_df->worldToGrid(m_goal_xyz[3 * r], m_goal_xyz[3 * r + 1], m_goal_xyz[3 * r + 2], c[0], c[1], c[2]);
            cells.insert(cells.end(), c, c + 3);
            m_goal_in_grid = m_goal_in_grid || m_heur->bfs()->inBounds(c[0], c[1], c[2]);
        }
        m_goal_id = 0;                            // reserveHashEntry for the goal state (manip_lattice.cpp:122)
        m_states.push_back(State());
        // setGoal -> BfsHeuristic::updateGoal over every record's position: BFS_3D::run(begin, end), whose iterator walk
        // commits a triple only when another element follows it (bfs3d.h:157-211), hence the trailing triple
        cells.insert(cells.end(), { 0, 0, 0 });
        m_heur->bfs()->run(cells.data(), (int)goals.size() + 1);
        if (!m_robot->checkJointLimits(start) || !m_cc->isStateValid(start)) {   // setStart (manip_lattice.cpp:1944-1980)
            res.num_states = (int)m_states.size();
            return res;
        }
        std::vector<int> coord;
        stateToCoord(start, coord);
        m_start_id = getOrCreateState(coord, start);
        AraStar search(
            [this](int id, std::vector<int>& succs, std::vector<int>& costs) { getSuccs(id, succs, costs); },
            [this](int id) { return goalHeuristic(id); });
        const AraStar::Result r = search.search(m_start_id, m_goal_id, m_epsilon, m_max_expansions);
        res.expansions = r.expansions;
        res.num_states = (int)m_states.size();
        if (!r.found || r.cost >= AraStar::INFINITE_COST) {
            return res;
        }
        res.path_ids = r.path;
        res.cost = r.cost;
        res.success = true;
        extractPath(res.path_ids, res.path_states);
        *reached = m_reached;
        return res;
    }

private:
    struct State { std::vector<int> coord; std::vector<double> state; };
    CollisionSpace* m_cc;
    KDLRobotModel* m_robot;
    BfsHeuristic* m_heur;
    double m_xyz_offset[3];
    std::vector<Prim> m_prims;
    bool m_use_short_dist;
    double m_short_dist_thresh, m_epsilon;
    int m_max_expansions;
    SnapKinds* m_snaps;   // by kind; disabled kinds produce nothing
    EuclidDistanceMap* m_df;   // the heuristic's grid (worldToGrid of the goal positions)
    std::vector<double> m_min_limits, m_coord_deltas;
    std::vector<bool> m_continuous, m_bounded;
    std::vector<int> m_coord_vals;
    std::vector<State> m_states;
    std::map<std::vector<int>, int> m_coord_to_id;
    int m_goal_id = 0, m_start_id = 1;
    std::vector<Goal> m_goals;       // the goal set
    std::vector<double> m_goal_xyz;  // [n][3] each record's goal position
    bool m_goal_in_grid = false;     // some record's position lies in the grid
    int m_reached = -1;              // extractPath: the record the path's goal action satisfies first

    // manip_lattice.cpp:1263-1289
    void stateToCoord(const std::vector<double>& state, std::vector<int>& coord) const
    {
        coord.resize(state.size());
        for (size_t i = 0; i < state.size(); ++i) {
            if (m_continuous[i]) {
                double pos_angle = normalize_angle(state[i]);
                if (pos_angle < 0.0) {
                    pos_angle += 2.0 * M_PI;
                }
                coord[i] = (int)((pos_angle + m_coord_deltas[i] * 0.5) / m_coord_deltas[i]);
                if (coord[i] == m_coord_vals[i]) {
                    coord[i] = 0;
                }
            } else if (!m_bounded[i]) {
                coord[i] = state[i] >= 0.0 ? (int)(state[i] / m_coord_deltas[i] + 0.5) : (int)(state[i] / m_coord_deltas[i] - 0.5);
            } else {
                coord[i] = (int)(((state[i] - m_min_limits[i]) / m_coord_deltas[i]) + 0.5);
            }
        }
    }

    int getOrCreateState(const std::vector<int>& coord, const std::vector<double>& state)
    {
        auto it = m_coord_to_id.find(coord);
        if (it != m_coord_to_id.end()) {
            return it->second;
        }
        const int id = (int)m_states.size();
        m_states.push_back(State{ coord, state });
        m_coord_to_id[coord] = id;
        return id;
    }

    // ManipLattice::isGoal (manip_lattice.cpp:1582-1696) over the goal set in order: the index of the first record
    // the state satisfies, or -1
    int isGoal(const std::vector<double>& state) const
    {
        std::vector<double> pose;
        for (size_t r = 0; r < m_goals.size(); ++r) {
            const Goal& g = m_goals[r];
            if (g.type == JOINT_STATE_GOAL) {
                bool in = true;
                for (size_t i = 0; i < state.size() && in; ++i) {
                    in = std::fabs(state[i] - g.angles[i]) <= g.angle_tolerances[i];
                }
                if (in) {
                    return (int)r;
                }
                continue;
            }
            if (pose.empty()) {
                m_robot->computePlanningLinkFK(state, pose);
                pose = GetTargetOffsetPose(pose, m_xyz_offset);
            }
            if (!(std::fabs(pose[0] - g.pose[0]) <= g.xyz_tolerance[0] &&
                  std::fabs(pose[1] - g.pose[1]) <= g.xyz_tolerance[1] &&
                  std::fabs(pose[2] - g.pose[2]) <= g.xyz_tolerance[2])) {
                continue;
            }
            if (g.type == XYZ_GOAL || rpyGoalAngle(&pose[3], &g.pose[3]) < g.rpy_tolerance) {
                return (int)r;
            }
        }
        return -1;
    }

    // the snap's target: the record whose goal position is nearest to p (squared Euclidean distance, the lower index
    // on a tie; smpl_b200/csrc/ik.cuh nearest_goal_record uses the same expression)
    int nearestRecord(const double* p) const
    {
        int best = 0;
        double best_d = 0.0;
        for (size_t r = 0; r < m_goals.size(); ++r) {
            const double dx = m_goal_xyz[3 * r] - p[0], dy = m_goal_xyz[3 * r + 1] - p[1], dz = m_goal_xyz[3 * r + 2] - p[2];
            const double d = (dx * dx + dy * dy) + dz * dz;
            if (r == 0 || d < best_d) {
                best = (int)r;
                best_d = d;
            }
        }
        return best;
    }

    // BfsHeuristic::GetGoalHeuristic over ManipLattice::projectToPose: the goal state projects to the goal position
    int goalHeuristic(int id) const
    {
        if (id == m_goal_id) {
            // the goal state projects onto a seed cell (distance 0, even on a wall), or nowhere in the grid
            return m_goal_in_grid ? 0 : BfsHeuristic::Infinity;
        }
        std::vector<double> pose;
        m_robot->computePlanningLinkFK(m_states[id].state, pose);
        pose = GetTargetOffsetPose(pose, m_xyz_offset);
        return m_heur->getGoalHeuristicAt(pose[0], pose[1], pose[2]);
    }

    // mprimActive (manip_lattice_action_space.cpp:662-691)
    bool primActive(size_t p, bool near_goal) const
    {
        if (!m_prims[p].short_dist) {
            return !(m_use_short_dist && near_goal);
        }
        return m_use_short_dist && near_goal;
    }

    bool nearGoal(const std::vector<double>& parent) const
    {
        std::vector<double> pose;
        m_robot->computePlanningLinkFK(parent, pose);
        return m_heur->getMetricGoalDistance(pose[0], pose[1], pose[2]) <= m_short_dist_thresh;
    }

    // The snap action of `kind` (SNAP_RPY, SNAP_XYZ, SNAP_XYZ_RPY): active when the parent's metric goal distance is
    // within the kind's threshold, whatever mprimActive decides.  Every kind aims at the record nearest to the parent
    // (nearestRecord) and seeds its IK at the parent:
    //   SNAP_XYZ_RPY  an IK solution for the record's full pose (XYZ, XYZ_RPY records), or a joint record's angles
    //   SNAP_XYZ      a position-only IK solution (planningLinkIkPosition) for the record's position (XYZ, XYZ_RPY)
    //   SNAP_RPY      an IK solution for the parent's own target-offset position and the record's rotation (XYZ_RPY)
    // Returns false when the kind is disabled or inactive, does not apply to the record's type, or its IK does not
    // converge.
    bool snapAction(int kind, const std::vector<double>& parent, std::vector<double>& succ) const
    {
        Snap& snap = m_snaps->kind[kind];
        if (!snap.enabled) {
            return false;
        }
        std::vector<double> pose;
        m_robot->computePlanningLinkFK(parent, pose);
        if (!(m_heur->getMetricGoalDistance(pose[0], pose[1], pose[2]) <= snap.dist_thresh)) {
            return false;
        }
        const std::vector<double> tgt = GetTargetOffsetPose(pose, m_xyz_offset);
        int target = 0;
        if (m_goals.size() > 1) {
            target = nearestRecord(tgt.data());
        }
        const Goal& goal = m_goals[target];
        if ((kind == SNAP_XYZ && goal.type == JOINT_STATE_GOAL) || (kind == SNAP_RPY && goal.type != XYZ_RPY_GOAL)) {
            return false;
        }
        if (goal.type == JOINT_STATE_GOAL) {
            succ = goal.angles;
            return true;
        }
        succ = parent;
        int iterations = 0;
        bool ok;
        if (kind == SNAP_XYZ) {
            ok = planningLinkIkPosition(*m_robot, snap.Tk, m_xyz_offset, goal.pose, snap.ik, succ, &iterations);
        } else {
            double R[9];
            rpyMatrix(goal.pose[3], goal.pose[4], goal.pose[5], R);
            ok = planningLinkIk(*m_robot, snap.Tk, m_xyz_offset, kind == SNAP_RPY ? tgt.data() : goal.pose, R, snap.ik,
                                succ, &iterations);
        }
        ++snap.attempted;
        snap.converged += ok ? 1 : 0;
        return ok;
    }

    // ManipLattice::GetSuccs + ManipLatticeActionSpace::apply + ManipLattice::checkAction
    void getSuccs(int id, std::vector<int>& succs, std::vector<int>& costs)
    {
        if (id == m_goal_id) {
            return;
        }
        const std::vector<double> parent = m_states[id].state;
        const bool near_goal = nearGoal(parent);
        std::vector<double> succ(parent.size());
        std::vector<int> coord;
        // the snap actions come first, in kind order: their successors are created before the primitives'
        for (int kind = 0; kind < 3; ++kind) {
            if (snapAction(kind, parent, succ) && m_robot->checkJointLimits(succ) && m_cc->isStateToStateValid(parent, succ)) {
                stateToCoord(succ, coord);
                const int succ_id = getOrCreateState(coord, succ);
                succs.push_back(isGoal(succ) >= 0 ? m_goal_id : succ_id);
                costs.push_back(m_snaps->kind[kind].cost);
            }
            succ.resize(parent.size());
        }
        for (size_t p = 0; p < m_prims.size(); ++p) {
            if (!primActive(p, near_goal)) {
                continue;
            }
            for (size_t j = 0; j < parent.size(); ++j) {
                succ[j] = m_prims[p].delta[j] + parent[j];
            }
            if (!m_robot->checkJointLimits(succ) || !m_cc->isStateToStateValid(parent, succ)) {
                continue;
            }
            stateToCoord(succ, coord);
            const int succ_id = getOrCreateState(coord, succ);
            succs.push_back(isGoal(succ) >= 0 ? m_goal_id : succ_id);
            costs.push_back(m_prims[p].cost);
        }
    }

    // ManipLattice::extractPath (manip_lattice.cpp:2018-2160): the goal id is replaced by the lattice state of the
    // cheapest valid goal-reaching action of its predecessor (strict <: the first of equal cost); the snaps come first,
    // in kind order, and no primitive costs less (the snap actions are re-run: they are deterministic)
    bool extractPath(const std::vector<int>& ids, std::vector<std::vector<double>>& path)
    {
        path.clear();
        if (ids.empty()) {
            return true;
        }
        if (ids.size() == 1) {
            path.push_back(m_states[ids[0] == m_goal_id ? m_start_id : ids[0]].state);
            return true;
        }
        if (ids[0] == m_goal_id) {
            return false;
        }
        path.push_back(m_states[ids[0]].state);
        for (size_t i = 1; i < ids.size(); ++i) {
            const int prev_id = ids[i - 1], curr_id = ids[i];
            if (prev_id == m_goal_id) {
                return false;
            }
            if (curr_id != m_goal_id) {
                path.push_back(m_states[curr_id].state);
                continue;
            }
            const std::vector<double>& parent = m_states[prev_id].state;
            const bool near_goal = nearGoal(parent);
            std::vector<double> succ(parent.size());
            std::vector<int> coord;
            int best_cost = std::numeric_limits<int>::max();
            int best = -1, best_reached = -1;
            for (int kind = 0; kind < 3 && best_cost != std::numeric_limits<int>::min(); ++kind) {
                Snap& snap = m_snaps->kind[kind];
                const long long attempted = snap.attempted, converged = snap.converged;   // count the search's IK only
                int reached = -1;
                if (snapAction(kind, parent, succ) && (reached = isGoal(succ)) >= 0 && m_robot->checkJointLimits(succ) &&
                    m_cc->isStateToStateValid(parent, succ)) {
                    stateToCoord(succ, coord);
                    auto it = m_coord_to_id.find(coord);
                    if (it != m_coord_to_id.end()) {
                        best_cost = std::numeric_limits<int>::min();
                        best = it->second;
                        best_reached = reached;
                    }
                }
                snap.attempted = attempted;
                snap.converged = converged;
                succ.resize(parent.size());
            }
            for (size_t p = 0; p < m_prims.size() && best_cost != std::numeric_limits<int>::min(); ++p) {
                if (!primActive(p, near_goal)) {
                    continue;
                }
                for (size_t j = 0; j < parent.size(); ++j) {
                    succ[j] = m_prims[p].delta[j] + parent[j];
                }
                const int reached = isGoal(succ);
                if (reached < 0) {
                    continue;
                }
                if (!m_robot->checkJointLimits(succ) || !m_cc->isStateToStateValid(parent, succ)) {
                    continue;
                }
                stateToCoord(succ, coord);
                auto it = m_coord_to_id.find(coord);
                if (it == m_coord_to_id.end()) {
                    continue;
                }
                const int edge_cost = (int)(1000 * 1.0);   // as oracle/lattice.cpp: every goal action compared at unit weight
                if (edge_cost < best_cost) {
                    best_cost = edge_cost;
                    best = it->second;
                    best_reached = reached;
                }
            }
            if (best < 0) {
                return false;
            }
            path.push_back(m_states[best].state);
            m_reached = best_reached;
        }
        return true;
    }
};

// the planning query of a goal set with the three snap kinds; the other parameters as oracle_plan_goal_set's
double planSnapKinds(oracle_scene* s, const double* start, const std::vector<Goal>& goals, const double* resolutions,
                     const double* mprims, const uint8_t* short_flags, const double* prim_weights, int n_prims,
                     int use_short_dist, double short_dist_thresh, double epsilon, int max_expansions,
                     const double* T_kin_to_planning, const int32_t* snap_enabled, const double* snap_dist_thresh,
                     double snap_weight, int ik_max_iterations, double ik_tolerance, int32_t* out_summary,
                     int32_t* path_ids, int max_path, double* path_states, int64_t* counters, int32_t* reached_goal)
{
    const int dof = s->dof;
    std::vector<Prim> prims(n_prims);
    for (int p = 0; p < n_prims; ++p) {
        prims[p].delta.assign(mprims + (size_t)p * dof, mprims + (size_t)(p + 1) * dof);
        prims[p].short_dist = short_flags[p] != 0;
        prims[p].cost = (int)(1000 * (prim_weights ? prim_weights[p] : 1.0));
    }
    SnapKinds snaps;
    for (int k = 0; k < 3; ++k) {
        Snap& snap = snaps.kind[k];
        snap.enabled = snap_enabled[k] != 0;
        snap.dist_thresh = snap_dist_thresh[k];
        snap.cost = (int)(1000 * snap_weight);
        snap.ik.max_iterations = ik_max_iterations;
        snap.ik.tolerance = ik_tolerance;
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) snap.Tk.M[3 * r + c] = T_kin_to_planning[4 * r + c];
            snap.Tk.p[r] = T_kin_to_planning[4 * r + 3];
        }
    }
    SnapKindsLatticePlanner planner(s, std::vector<double>(resolutions, resolutions + dof), prims, use_short_dist != 0,
                                    short_dist_thresh, epsilon, max_expansions, &snaps);
    const std::vector<double> st(start, start + dof);
    int reached = -1;
    const auto t0 = std::chrono::steady_clock::now();
    const Result r = planner.plan(st, goals, &reached);
    const auto t1 = std::chrono::steady_clock::now();
    out_summary[0] = r.success ? 1 : 0;
    out_summary[1] = r.expansions;
    out_summary[2] = r.cost;
    out_summary[3] = (int)r.path_ids.size();
    out_summary[4] = r.num_states;
    out_summary[5] = (int)r.path_states.size();
    for (size_t i = 0; i < r.path_ids.size() && (int)i < max_path; ++i) {
        path_ids[i] = r.path_ids[i];
        if (path_states && i < r.path_states.size()) {
            std::copy(r.path_states[i].begin(), r.path_states[i].end(), path_states + i * (size_t)dof);
        }
    }
    if (counters) {
        for (int k = 0; k < 3; ++k) {
            counters[2 * k] = snaps.kind[k].attempted;
            counters[2 * k + 1] = snaps.kind[k].converged;
        }
    }
    if (reached_goal) {
        *reached_goal = reached;
    }
    return std::chrono::duration<double>(t1 - t0).count();
}

} // namespace

extern "C" {

/// oracle_plan_goal_set with the three snap kinds of SnapKindsLatticePlanner: snap_enabled[3] and snap_dist_thresh[3]
/// by SNAP_* kind (RPY, XYZ, XYZ_RPY), one snap_weight and one set of IK parameters.  counters[6] (nullable): by kind
/// k, counters[2 k] the IK solves the search ran and counters[2 k + 1] how many converged.  Returns -1 for a bad set or
/// scene.
double oracle_plan_goal_set_snaps(oracle_scene* s, const double* start, const oracle_goal_record* goals, int n_goals,
                                  const double* resolutions, const double* mprims, const uint8_t* short_flags,
                                  const double* prim_weights, int n_prims, int use_short_dist, double short_dist_thresh,
                                  double epsilon, int max_expansions, const double* T_kin_to_planning,
                                  const int32_t* snap_enabled, const double* snap_dist_thresh, double snap_weight,
                                  int ik_max_iterations, double ik_tolerance, int32_t* out_summary, int32_t* path_ids,
                                  int max_path, double* path_states, int64_t* counters, int32_t* reached_goal)
{
    if (!(s && s->kdl && s->heur && s->dof == oracle_scene_dof(s) && T_kin_to_planning) || !goals || n_goals < 1 ||
        n_goals > 64 || s->dof > 16 || !snap_enabled || !snap_dist_thresh) {
        return -1.0;
    }
    const int dof = s->dof;
    std::vector<Goal> set(n_goals);
    for (int r = 0; r < n_goals; ++r) {
        const oracle_goal_record& in = goals[r];
        if (in.type < XYZ_GOAL || in.type > JOINT_STATE_GOAL) {
            return -1.0;
        }
        Goal& g = set[r];
        g.type = in.type;
        std::copy(in.pose, in.pose + 6, g.pose);
        std::copy(in.xyz_tolerance, in.xyz_tolerance + 3, g.xyz_tolerance);
        g.rpy_tolerance = in.rpy_tolerance;
        g.angles.assign(in.angles, in.angles + dof);
        g.angle_tolerances.assign(in.angle_tolerances, in.angle_tolerances + dof);
    }
    return planSnapKinds(s, start, set, resolutions, mprims, short_flags, prim_weights, n_prims, use_short_dist,
                         short_dist_thresh, epsilon, max_expansions, T_kin_to_planning, snap_enabled, snap_dist_thresh,
                         snap_weight, ik_max_iterations, ik_tolerance, out_summary, path_ids, max_path, path_states,
                         counters, reached_goal);
}

/// The position-only IK (planningLinkIkPosition) of n problems: xyz[n][3] target-offset positions, seeds[n][dof];
/// q_out[n][dof], ok[n], iterations[n].  T_kin_to_planning as for oracle_planning_link_ik.  Returns the number that
/// converged, or -1 for a scene without kinematics.
int oracle_planning_link_ik_position(oracle_scene* s, const double* T_kin_to_planning, const double* xyz,
                                     const double* seeds, int n, int max_iterations, double tolerance, double* q_out,
                                     uint8_t* ok, int32_t* iterations)
{
    if (!s || !s->kdl || !T_kin_to_planning) {
        return -1;
    }
    const int dof = s->dof;
    KdlFrame Tk;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) Tk.M[3 * r + c] = T_kin_to_planning[4 * r + c];
        Tk.p[r] = T_kin_to_planning[4 * r + 3];
    }
    const IkParams prm{ max_iterations, tolerance };
    int n_ok = 0;
    std::vector<double> q(dof);
    for (int i = 0; i < n; ++i) {
        q.assign(seeds + (size_t)i * dof, seeds + (size_t)(i + 1) * dof);
        int it = 0;
        const bool conv = planningLinkIkPosition(*s->kdl, Tk, s->xyz_offset, xyz + 3 * (size_t)i, prm, q, &it);
        std::copy(q.begin(), q.end(), q_out + (size_t)i * dof);
        ok[i] = conv ? 1 : 0;
        iterations[i] = it;
        n_ok += conv ? 1 : 0;
    }
    return n_ok;
}

} // extern "C"
