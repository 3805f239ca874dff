// ORACLE (test infrastructure only -- never linked into the product path).
//
// The planning query of oracle/lattice.cpp (ManipLattice + ARA*, first solution at the initial epsilon) for a
// GoalConstraint of any of the three types ManipLattice::isGoal tests (manip_lattice.cpp:1582-1696):
//   XYZ_GOAL          |pose[a] - goal[a]| <= xyz_tolerance[a], a = 0, 1, 2                      (:1673-1687)
//   XYZ_RPY_GOAL      the XYZ test, then normalize_angle(2 acos(q . qg)) < rpy_tolerance[0], q and qg =
//                     AngleAxisd(yaw, Z) * AngleAxisd(pitch, Y) * AngleAxisd(roll, X) of the state's and the goal's
//                     roll pitch yaw, qg negated when q . qg < 0, no clamp of the acos argument
//   JOINT_STATE_GOAL  |state[i] - angles[i]| <= angle_tolerances[i] for every planning variable, no angle wrapping
// A joint goal's position (BFS seed, heuristic of the goal state, short-distance switch) is the target offset position
// of its angles (ManipLattice::setGoalConfiguration).  Everything else -- successors, limits, edge checks, stateToCoord,
// getOrCreateState, heuristic, extractPath -- restates oracle/lattice.cpp line for line over the same oracle classes,
// so an XYZ goal gives that planner's plans (tests/test_oracle_goal_types.py pins the two against each other).  The
// quaternion arithmetic follows Eigen's (oracle/ref_stubs/eigen_arith/Eigen/Dense: Quaterniond(AngleAxisd), the
// generic quat_product, dot).  The reference build's planner is driven with XYZ goals only, so the XYZ_RPY and
// JOINT_STATE branches are parity unpinned (DESIGN.md section 2).
//
// Built as oracle/goals/liboracle_goals.so over oracle/liboracle.so; it takes the scene handles of the oracle's C API.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <limits>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../arastar.h"
#include "../bfs3d.h"
#include "../collision_space.h"
#include "../distance_map.h"
#include "../kdl_model.h"
#include "../robot_desc.h"

using namespace oracle;

// The scene handle of oracle/oracle_capi.cpp, restated token for token (one definition across the two libraries)
struct oracle_scene
{
    RobotDesc desc;
    std::string group;
    std::vector<std::string> planning_joints;
    std::unique_ptr<EuclidDistanceMap> df;
    std::unique_ptr<OccupancyGrid> grid;
    std::unique_ptr<CollisionSpace> cc;
    std::unique_ptr<KDLRobotModel> kdl;
    std::unique_ptr<BfsHeuristic> heur;
    double xyz_offset[3];
    int dof;
    oracle_scene() : dof(0) { xyz_offset[0] = xyz_offset[1] = xyz_offset[2] = 0.0; }
};

extern "C" int oracle_scene_dof(oracle_scene* s);

namespace {

enum GoalType { XYZ_GOAL = 0, XYZ_RPY_GOAL = 1, JOINT_STATE_GOAL = 2 };   // smpl/planning_params.h order

struct Goal
{
    int type;
    double pose[6];
    double xyz_tolerance[3];
    double rpy_tolerance;
    std::vector<double> angles, angle_tolerances;
};

struct Quat
{
    double q[4];   // x y z w, Eigen's coefficient order
};

// Eigen's generic quat_product
Quat operator*(const Quat& a, const Quat& b)
{
    Quat r;
    r.q[3] = a.q[3] * b.q[3] - a.q[0] * b.q[0] - a.q[1] * b.q[1] - a.q[2] * b.q[2];
    r.q[0] = a.q[3] * b.q[0] + a.q[0] * b.q[3] + a.q[1] * b.q[2] - a.q[2] * b.q[1];
    r.q[1] = a.q[3] * b.q[1] + a.q[1] * b.q[3] + a.q[2] * b.q[0] - a.q[0] * b.q[2];
    r.q[2] = a.q[3] * b.q[2] + a.q[2] * b.q[3] + a.q[0] * b.q[1] - a.q[1] * b.q[0];
    return r;
}

double dot(const Quat& a, const Quat& b)
{
    return ((a.q[0] * b.q[0] + a.q[1] * b.q[1]) + a.q[2] * b.q[2]) + a.q[3] * b.q[3];
}

// Quaterniond(AngleAxisd(angle, axis)): w = cos(angle / 2), xyz = sin(angle / 2) axis
Quat angleAxis(double angle, double x, double y, double z)
{
    const double ha = 0.5 * angle;
    const double sh = std::sin(ha);
    Quat r;
    r.q[0] = sh * x;
    r.q[1] = sh * y;
    r.q[2] = sh * z;
    r.q[3] = std::cos(ha);
    return r;
}

Quat quatFromRpy(double roll, double pitch, double yaw)
{
    return (angleAxis(yaw, 0.0, 0.0, 1.0) * angleAxis(pitch, 0.0, 1.0, 0.0)) * angleAxis(roll, 1.0, 0.0, 0.0);
}

// the angle XYZ_RPY_GOAL compares with rpy_tolerance (|q . qg| > 1 after rounding gives NaN: no goal)
double rpyGoalAngle(const double* rpy, const double* goal_rpy)
{
    Quat qg = quatFromRpy(goal_rpy[0], goal_rpy[1], goal_rpy[2]);
    const Quat q = quatFromRpy(rpy[0], rpy[1], rpy[2]);
    if (dot(q, qg) < 0.0) {
        for (double& c : qg.q) c = -c;
    }
    return normalize_angle(2.0 * std::acos(dot(q, qg)));
}

struct Prim
{
    std::vector<double> delta;
    bool short_dist;
    int cost;
};

struct Result
{
    bool success = false;
    int expansions = 0, cost = 0, num_states = 0;
    std::vector<int> path_ids;
    std::vector<std::vector<double>> path_states;
};

class GoalLatticePlanner
{
public:
    GoalLatticePlanner(oracle_scene* s, const std::vector<double>& resolutions, const std::vector<Prim>& prims,
                       bool use_short_dist, double short_dist_thresh, double epsilon, int max_expansions) :
        m_cc(s->cc.get()), m_robot(s->kdl.get()), m_heur(s->heur.get()), m_prims(), m_use_short_dist(use_short_dist),
        m_short_dist_thresh(short_dist_thresh), m_epsilon(epsilon), m_max_expansions(max_expansions)
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

    Result plan(const std::vector<double>& start, const Goal& goal)
    {
        Result res;
        m_states.clear();
        m_coord_to_id.clear();
        m_goal = goal;
        if (goal.type == JOINT_STATE_GOAL) {
            std::vector<double> pose;   // ManipLattice::setGoalConfiguration: the target offset pose of the angles
            m_robot->computePlanningLinkFK(goal.angles, pose);
            pose = GetTargetOffsetPose(pose, m_xyz_offset);
            for (int i = 0; i < 3; ++i) m_goal_xyz[i] = pose[i];
        } else {
            for (int i = 0; i < 3; ++i) m_goal_xyz[i] = goal.pose[i];
        }
        m_goal_id = 0;                            // reserveHashEntry for the goal state (manip_lattice.cpp:122)
        m_states.push_back(State());
        m_heur->updateGoal(m_goal_xyz[0], m_goal_xyz[1], m_goal_xyz[2]);   // setGoal -> BfsHeuristic::updateGoal
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
    std::vector<double> m_min_limits, m_coord_deltas;
    std::vector<bool> m_continuous, m_bounded;
    std::vector<int> m_coord_vals;
    std::vector<State> m_states;
    std::map<std::vector<int>, int> m_coord_to_id;
    int m_goal_id = 0, m_start_id = 1;
    Goal m_goal;
    double m_goal_xyz[3] = { 0.0, 0.0, 0.0 };

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

    // ManipLattice::isGoal (manip_lattice.cpp:1582-1696)
    bool isGoal(const std::vector<double>& state) const
    {
        if (m_goal.type == JOINT_STATE_GOAL) {
            for (size_t i = 0; i < state.size(); ++i) {
                if (!(std::fabs(state[i] - m_goal.angles[i]) <= m_goal.angle_tolerances[i])) {
                    return false;
                }
            }
            return true;
        }
        std::vector<double> pose;
        m_robot->computePlanningLinkFK(state, pose);
        pose = GetTargetOffsetPose(pose, m_xyz_offset);
        if (!(std::fabs(pose[0] - m_goal.pose[0]) <= m_goal.xyz_tolerance[0] &&
              std::fabs(pose[1] - m_goal.pose[1]) <= m_goal.xyz_tolerance[1] &&
              std::fabs(pose[2] - m_goal.pose[2]) <= m_goal.xyz_tolerance[2])) {
            return false;
        }
        if (m_goal.type == XYZ_GOAL) {
            return true;
        }
        return rpyGoalAngle(&pose[3], &m_goal.pose[3]) < m_goal.rpy_tolerance;
    }

    // BfsHeuristic::GetGoalHeuristic over ManipLattice::projectToPose: the goal state projects to the goal position
    int goalHeuristic(int id) const
    {
        if (id == m_goal_id) {
            return m_heur->getGoalHeuristicAt(m_goal_xyz[0], m_goal_xyz[1], m_goal_xyz[2]);
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
            succs.push_back(isGoal(succ) ? m_goal_id : succ_id);
            costs.push_back(m_prims[p].cost);
        }
    }

    // ManipLattice::extractPath (manip_lattice.cpp:2018-2160): the goal id is replaced by the lattice state of the
    // cheapest valid goal-reaching action of its predecessor (strict <: the first of equal cost)
    bool extractPath(const std::vector<int>& ids, std::vector<std::vector<double>>& path) const
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
            int best = -1;
            for (size_t p = 0; p < m_prims.size(); ++p) {
                if (!primActive(p, near_goal)) {
                    continue;
                }
                for (size_t j = 0; j < parent.size(); ++j) {
                    succ[j] = m_prims[p].delta[j] + parent[j];
                }
                if (!isGoal(succ)) {
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
                }
            }
            if (best < 0) {
                return false;
            }
            path.push_back(m_states[best].state);
        }
        return true;
    }
};

} // namespace

extern "C" {

/// The oracle_plan query (oracle/oracle_capi.cpp) for a GoalConstraint: type 0 XYZ_GOAL, 1 XYZ_RPY_GOAL,
/// 2 JOINT_STATE_GOAL; pose6 = x y z roll pitch yaw, xyz_tolerance[3], rpy_tolerance, angles / angle_tolerances [dof];
/// prim_weights [n_prims] (nullable: 1 each).  out_summary: success, expansions, cost, path length, num_states, path
/// states written.  Returns the seconds spent planning, or -1 for an unknown type or a scene without kinematics /
/// heuristic.
double oracle_plan_goal(oracle_scene* s, const double* start, int type, const double* pose6, const double* xyz_tolerance,
                        double rpy_tolerance, const double* angles, const double* angle_tolerances,
                        const double* resolutions, const double* mprims, const uint8_t* short_flags,
                        const double* prim_weights, int n_prims, int use_short_dist, double short_dist_thresh,
                        double epsilon, int max_expansions, int32_t* out_summary, int32_t* path_ids, int max_path,
                        double* path_states)
{
    if (!s || type < XYZ_GOAL || type > JOINT_STATE_GOAL || !s->kdl || !s->heur || s->dof != oracle_scene_dof(s)) {
        return -1.0;
    }
    const int dof = s->dof;
    Goal g;
    g.type = type;
    std::copy(pose6, pose6 + 6, g.pose);
    std::copy(xyz_tolerance, xyz_tolerance + 3, g.xyz_tolerance);
    g.rpy_tolerance = rpy_tolerance;
    g.angles.assign(angles, angles + dof);
    g.angle_tolerances.assign(angle_tolerances, angle_tolerances + dof);
    std::vector<Prim> prims(n_prims);
    for (int p = 0; p < n_prims; ++p) {
        prims[p].delta.assign(mprims + (size_t)p * dof, mprims + (size_t)(p + 1) * dof);
        prims[p].short_dist = short_flags[p] != 0;
        prims[p].cost = (int)(1000 * (prim_weights ? prim_weights[p] : 1.0));   // DefaultCostMultiplier * actionWeight
    }
    GoalLatticePlanner planner(s, std::vector<double>(resolutions, resolutions + dof), prims, use_short_dist != 0,
                               short_dist_thresh, epsilon, max_expansions);
    const std::vector<double> st(start, start + dof);
    const auto t0 = std::chrono::steady_clock::now();
    const Result r = planner.plan(st, g);
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
    return std::chrono::duration<double>(t1 - t0).count();
}

/// The XYZ_RPY_GOAL angle of n (state rpy, goal rpy) pairs, rpy[n][2][3]; qg_dot[i] (nullable) = q . qg before the
/// sign flip
int oracle_rpy_goal_angles(const double* rpy, int n, double* theta, double* qg_dot)
{
    for (int i = 0; i < n; ++i) {
        const double* a = rpy + 6 * (size_t)i;
        theta[i] = rpyGoalAngle(a, a + 3);
        if (qg_dot) qg_dot[i] = dot(quatFromRpy(a[0], a[1], a[2]), quatFromRpy(a[3], a[4], a[5]));
    }
    return 0;
}

} // extern "C"
