// ORACLE (test infrastructure only -- never linked into the product path).
//
// The goal-typed planning query of oracle/goals/goal_lattice.cpp with the SNAP_TO_XYZ_RPY action of
// ManipLatticeActionSpace (manip_lattice_action_space.cpp:376-449, 507-573, 662-691): when the parent's metric goal
// distance is within the snap threshold, whatever mprimActive decides, the first successor is an IK solution for the goal
// pose seeded at the parent (XYZ and XYZ_RPY goals: the full pose of the record), or the angles of a JOINT_STATE goal,
// checked like any action (joint limits, then isStateToStateValid) and costing (int)(1000 snap_weight); extractPath
// re-runs it (it is deterministic) and takes it first.  With snaps disabled SnapLatticePlanner is GoalLatticePlanner
// (tests/test_oracle_ik_snap.py pins the two against each other).
//
// The reference's IK solvers (pr2_arm_kinematics, KDL's ChainIkSolverPos_NR_JL) are third-party and absent, so the IK
// is the project's own (planningLinkIk below; DESIGN.md section 2: parity unpinned, pinned oracle <-> device);
// smpl_b200/csrc/ik.cuh restates it expression for expression.
//
// Built as oracle/snap/liboracle_snap.so over oracle/liboracle.so; it takes the scene handles of the oracle's C API.
// The goal-typed planner's definitions (scene handle, goal records, the quaternion goal test, Prim, Result) come from
// its source, included here unchanged so that both planners share one copy of them (the library therefore also
// exports that file's oracle_plan_goal and oracle_rpy_goal_angles; tests call those from liboracle_goals.so).
#include "../goals/goal_lattice.cpp"

namespace {

// ---- planning-link IK (the device's restatement: smpl_b200/csrc/ik.cuh) ----

// damping of the least-squares step, in the units of the error (metres / radians)
const double IK_LAMBDA = 1e-3;

struct IkParams
{
    int max_iterations;
    double tolerance;
};

// KDL Rotation::Rot2 (restated from oracle/kdl_model.cpp, where it is file-local)
void rot2(const double v[3], double angle, double M[9])
{
    double ct = std::cos(angle);
    double st = std::sin(angle);
    double vt = 1 - ct;
    double m_vt_0 = vt * v[0];
    double m_vt_1 = vt * v[1];
    double m_vt_2 = vt * v[2];
    double m_st_0 = v[0] * st;
    double m_st_1 = v[1] * st;
    double m_st_2 = v[2] * st;
    double m_vt_0_1 = m_vt_0 * v[1];
    double m_vt_0_2 = m_vt_0 * v[2];
    double m_vt_1_2 = m_vt_1 * v[2];
    M[0] = ct + m_vt_0 * v[0];   M[1] = -m_st_2 + m_vt_0_1;   M[2] = m_st_1 + m_vt_0_2;
    M[3] = m_st_2 + m_vt_0_1;    M[4] = ct + m_vt_1 * v[1];   M[5] = -m_st_0 + m_vt_1_2;
    M[6] = -m_st_1 + m_vt_0_2;   M[7] = m_st_0 + m_vt_1_2;    M[8] = ct + m_vt_2 * v[2];
}

// Segment::pose(q) = joint.pose(q) * f_tip (oracle/kdl_model.cpp JointPose; the continuous-joint normalisation of
// computePlanningLinkFK)
KdlFrame segmentPose(const KDLRobotModel& m, int s, const std::vector<double>& q)
{
    const KDLRobotModel::Segment& seg = m.segments[s];
    double qq = 0.0;
    if (seg.q_index >= 0) {
        qq = q[seg.q_index];
        if (m.continuous[seg.q_index]) {
            qq = normalize_angle(qq);
        }
    }
    KdlFrame jp = KdlFrame::Identity();
    if (seg.joint_kind == 1) {
        rot2(seg.axis, qq, jp.M);
        jp.p[0] = seg.origin[0]; jp.p[1] = seg.origin[1]; jp.p[2] = seg.origin[2];
    } else if (seg.joint_kind == 2) {
        jp.p[0] = seg.origin[0] + seg.axis[0] * qq;
        jp.p[1] = seg.origin[1] + seg.axis[1] * qq;
        jp.p[2] = seg.origin[2] + seg.axis[2] * qq;
    }
    return jp * seg.f_tip;
}

// KDL Rotation::RPY(roll, pitch, yaw) = Rz(yaw) Ry(pitch) Rx(roll), row-major; the host computes a goal's rotation
// with this expression (smplgpu.cu rpy_matrix)
void rpyMatrix(double roll, double pitch, double yaw, double R[9])
{
    const double ca1 = std::cos(yaw), sa1 = std::sin(yaw);
    const double cb1 = std::cos(pitch), sb1 = std::sin(pitch);
    const double cc1 = std::cos(roll), sc1 = std::sin(roll);
    R[0] = ca1 * cb1;  R[1] = ca1 * sb1 * sc1 - sa1 * cc1;  R[2] = ca1 * sb1 * cc1 + sa1 * sc1;
    R[3] = sa1 * cb1;  R[4] = sa1 * sb1 * sc1 + ca1 * cc1;  R[5] = sa1 * sb1 * cc1 - ca1 * sc1;
    R[6] = -sb1;       R[7] = cb1 * sc1;                    R[8] = cb1 * cc1;
}

// The rotation vector (axis * angle, angle in [0, pi]) of the rotation matrix E.  v = (E21 - E12, E02 - E20,
// E10 - E01) = 2 sin(angle) axis and cos(angle) = (trace - 1) / 2 give angle = atan2(|v| / 2, cos); then
//   near 0 (|v| / 2 < 1e-9):  the rotation vector is v / 2 (angle / (2 sin angle) = 1/2 + O(angle^2));
//   near pi (cos < -0.99):     v is too short to carry the axis, which comes from the symmetric part instead,
//                              (E + E^T) / 2 = cos I + (1 - cos) a a^T, largest diagonal first, its sign from v;
//   otherwise:                 v * angle / (2 sin angle).
void rotationVector(const double E[9], double w[3])
{
    const double v0 = E[7] - E[5], v1 = E[2] - E[6], v2 = E[3] - E[1];
    const double c = (((E[0] + E[4]) + E[8]) - 1.0) * 0.5;
    const double s = 0.5 * std::sqrt((v0 * v0 + v1 * v1) + v2 * v2);
    const double angle = std::atan2(s, c);
    if (s < 1e-9 && c > 0.0) {
        w[0] = 0.5 * v0; w[1] = 0.5 * v1; w[2] = 0.5 * v2;
        return;
    }
    if (c < -0.99) {
        int k = 0;
        if (E[4] > E[0]) k = 1;
        if (E[8] > E[4 * k]) k = 2;
        const double omc = 1.0 - c;
        double a[3];
        const double t = (E[4 * k] - c) / omc;
        a[k] = std::sqrt(0.0 < t ? t : 0.0);
        for (int j = 0; j < 3; ++j) {
            if (j != k) {
                a[j] = ((E[3 * j + k] + E[3 * k + j]) * 0.5) / (omc * a[k]);
            }
        }
        if ((a[0] * v0 + a[1] * v1) + a[2] * v2 < 0.0) {
            a[0] = -a[0]; a[1] = -a[1]; a[2] = -a[2];
        }
        w[0] = angle * a[0]; w[1] = angle * a[1]; w[2] = angle * a[2];
        return;
    }
    const double f = angle / (2.0 * s);
    w[0] = v0 * f; w[1] = v1 * f; w[2] = v2 * f;
}

// The IK of the planning link (inverse of smplgpu_planning_frame_fk, including its segment-index quirk) for the
// target-offset pose (target_p, target_R), seeded at q (overwritten with the answer):
//   f(q)  = T_kin_to_planning * segments 0 .. planning_segment_nr - 1: rotation R, position p; the target point is
//           pt = R offset + p
//   e     = (target_p - pt, rotationVector(target_R R^T)); converged when |e_i| <= tolerance for all six
//   step  = J^T (J J^T + IK_LAMBDA^2 I)^-1 e, J the geometric 6 x dof Jacobian at pt, the 6 x 6 system by Cholesky;
//           q += step, bounded variables clamped to their limits, continuous ones wrapped by normalize_angle
// at most max_iterations steps.  Returns converged; *iterations = steps taken.
bool planningLinkIk(const KDLRobotModel& m, const KdlFrame& Tk, const double offset[3], const double target_p[3],
                    const double target_R[9], const IkParams& prm, std::vector<double>& q, int* iterations)
{
    const int dof = (int)q.size();
    const int nseg = m.planning_segment_nr;
    std::vector<KdlFrame> prefix(nseg + 1);
    std::vector<double> J(6 * (size_t)dof, 0.0);   // row-major 6 x dof; variables beyond the chain keep 0 columns
    for (int it = 0;; ++it) {
        // chain: prefix[s] = segments 0 .. s-1
        KdlFrame f1 = KdlFrame::Identity();
        for (int s = 0; s < nseg; ++s) {
            prefix[s] = f1;
            f1 = f1 * segmentPose(m, s, q);
        }
        const KdlFrame f = Tk * f1;
        double pt[3], e[6], E[9];
        for (int i = 0; i < 3; ++i) {
            pt[i] = (f.M[3 * i] * offset[0] + f.M[3 * i + 1] * offset[1] + f.M[3 * i + 2] * offset[2]) + f.p[i];
            e[i] = target_p[i] - pt[i];
        }
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) {
                E[3 * i + j] = (target_R[3 * i] * f.M[3 * j] + target_R[3 * i + 1] * f.M[3 * j + 1]) +
                               target_R[3 * i + 2] * f.M[3 * j + 2];
            }
        }
        rotationVector(E, e + 3);
        bool conv = true;
        for (int i = 0; i < 6; ++i) {
            conv = conv && std::fabs(e[i]) <= prm.tolerance;   // false for NaN
        }
        if (conv || it == prm.max_iterations) {
            *iterations = it;
            return conv;
        }
        // Jacobian columns: the joint axis and origin in the planning frame
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
            double col[6];
            if (seg.joint_kind == 1) {
                const double d0 = pt[0] - o[0], d1 = pt[1] - o[1], d2 = pt[2] - o[2];
                col[0] = a[1] * d2 - a[2] * d1;
                col[1] = a[2] * d0 - a[0] * d2;
                col[2] = a[0] * d1 - a[1] * d0;
                col[3] = a[0]; col[4] = a[1]; col[5] = a[2];
            } else {
                col[0] = a[0]; col[1] = a[1]; col[2] = a[2];
                col[3] = 0.0; col[4] = 0.0; col[5] = 0.0;
            }
            for (int r = 0; r < 6; ++r) {
                J[(size_t)r * dof + seg.q_index] = col[r];
            }
        }
        // A = J J^T + lambda^2 I (lower triangle), Cholesky A = L L^T, A x = e
        double A[6][6], L[6][6], x[6], y[6];
        for (int r = 0; r < 6; ++r) {
            for (int c = 0; c <= r; ++c) {
                double acc = 0.0;
                for (int v = 0; v < dof; ++v) {
                    acc = acc + J[(size_t)r * dof + v] * J[(size_t)c * dof + v];
                }
                A[r][c] = r == c ? acc + IK_LAMBDA * IK_LAMBDA : acc;
            }
        }
        for (int j = 0; j < 6; ++j) {
            double d = A[j][j];
            for (int k = 0; k < j; ++k) {
                d = d - L[j][k] * L[j][k];
            }
            L[j][j] = std::sqrt(d);
            for (int i = j + 1; i < 6; ++i) {
                double t = A[i][j];
                for (int k = 0; k < j; ++k) {
                    t = t - L[i][k] * L[j][k];
                }
                L[i][j] = t / L[j][j];
            }
        }
        for (int i = 0; i < 6; ++i) {
            double t = e[i];
            for (int k = 0; k < i; ++k) {
                t = t - L[i][k] * y[k];
            }
            y[i] = t / L[i][i];
        }
        for (int i = 5; i >= 0; --i) {
            double t = y[i];
            for (int k = i + 1; k < 6; ++k) {
                t = t - L[k][i] * x[k];
            }
            x[i] = t / L[i][i];
        }
        for (int v = 0; v < dof; ++v) {
            double dq = 0.0;
            for (int r = 0; r < 6; ++r) {
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

struct Snap
{
    bool enabled = false;
    double dist_thresh = 0.0;
    int cost = 500;
    IkParams ik{ 100, 1e-6 };
    KdlFrame Tk = KdlFrame::Identity();   // T_kin_to_planning of the scene
    long long attempted = 0, converged = 0;
};

class SnapLatticePlanner
{
public:
    SnapLatticePlanner(oracle_scene* s, const std::vector<double>& resolutions, const std::vector<Prim>& prims,
                       bool use_short_dist, double short_dist_thresh, double epsilon, int max_expansions,
                       Snap* snap) :
        m_cc(s->cc.get()), m_robot(s->kdl.get()), m_heur(s->heur.get()), m_prims(), m_use_short_dist(use_short_dist),
        m_short_dist_thresh(short_dist_thresh), m_epsilon(epsilon), m_max_expansions(max_expansions), m_snap(snap)
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
    Snap* m_snap;   // disabled: no snap action
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

    // SNAP_TO_XYZ_RPY (manip_lattice_action_space.cpp:376-449, 507-573, 662-691): active when the parent's metric goal
    // distance is within the snap threshold, whatever mprimActive decides; the action is an IK solution for the goal
    // pose seeded at the parent (XYZ and XYZ_RPY goals: the full pose of the record), or the angles of a joint goal.
    // Returns false when the action is inactive or the IK does not converge.
    bool snapAction(const std::vector<double>& parent, std::vector<double>& succ) const
    {
        if (!m_snap || !m_snap->enabled) {
            return false;
        }
        std::vector<double> pose;
        m_robot->computePlanningLinkFK(parent, pose);
        if (!(m_heur->getMetricGoalDistance(pose[0], pose[1], pose[2]) <= m_snap->dist_thresh)) {
            return false;
        }
        if (m_goal.type == JOINT_STATE_GOAL) {
            succ = m_goal.angles;
            return true;
        }
        double R[9];
        rpyMatrix(m_goal.pose[3], m_goal.pose[4], m_goal.pose[5], R);
        succ = parent;
        int iterations = 0;
        const bool ok = planningLinkIk(*m_robot, m_snap->Tk, m_xyz_offset, m_goal.pose, R, m_snap->ik, succ, &iterations);
        ++m_snap->attempted;
        m_snap->converged += ok ? 1 : 0;
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
        // the snap action comes first: its successor is created before the primitives'
        if (snapAction(parent, succ) && m_robot->checkJointLimits(succ) && m_cc->isStateToStateValid(parent, succ)) {
            stateToCoord(succ, coord);
            const int succ_id = getOrCreateState(coord, succ);
            succs.push_back(isGoal(succ) ? m_goal_id : succ_id);
            costs.push_back(m_snap->cost);
        }
        succ.resize(parent.size());
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
    // cheapest valid goal-reaching action of its predecessor (strict <: the first of equal cost); a snap that reaches
    // the goal is the first action, and no primitive costs less (the snap action is re-run: it is deterministic)
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
            Snap* snap = m_snap;
            if (snap) {
                const long long attempted = snap->attempted, converged = snap->converged;   // count the search's IK only
                if (snapAction(parent, succ) && isGoal(succ) && m_robot->checkJointLimits(succ) &&
                    m_cc->isStateToStateValid(parent, succ)) {
                    stateToCoord(succ, coord);
                    auto it = m_coord_to_id.find(coord);
                    if (it != m_coord_to_id.end()) {
                        best_cost = std::numeric_limits<int>::min();
                        best = it->second;
                    }
                }
                snap->attempted = attempted;
                snap->converged = converged;
                succ.resize(parent.size());
            }
            for (size_t p = 0; p < m_prims.size() && best_cost != std::numeric_limits<int>::min(); ++p) {
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

/// oracle_plan_goal with the SNAP_TO_XYZ_RPY action (SnapLatticePlanner::snapAction): snap_enabled, snap_dist_thresh
/// (metres of metric goal distance), snap_weight (the action costs (int)(1000 snap_weight)), the IK's max_iterations
/// and tolerance, and the scene's T_kin_to_planning (3x4 row-major: the oracle scene keeps it private).  counters[2]
/// (nullable): IK solves the search ran, and how many converged.  With snap_enabled = 0 it plans as oracle_plan_goal.
double oracle_plan_goal_snap(oracle_scene* s, const double* start, int type, const double* pose6,
                             const double* xyz_tolerance, double rpy_tolerance, const double* angles,
                             const double* angle_tolerances, const double* resolutions, const double* mprims,
                             const uint8_t* short_flags, const double* prim_weights, int n_prims, int use_short_dist,
                             double short_dist_thresh, double epsilon, int max_expansions, const double* T_kin_to_planning,
                             int snap_enabled, double snap_dist_thresh, double snap_weight, int ik_max_iterations,
                             double ik_tolerance, int32_t* out_summary, int32_t* path_ids, int max_path,
                             double* path_states, int64_t* counters)
{
    if (!s || type < XYZ_GOAL || type > JOINT_STATE_GOAL || !s->kdl || !s->heur || s->dof != oracle_scene_dof(s) ||
        !T_kin_to_planning) {
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
        prims[p].cost = (int)(1000 * (prim_weights ? prim_weights[p] : 1.0));
    }
    Snap snap;
    snap.enabled = snap_enabled != 0;
    snap.dist_thresh = snap_dist_thresh;
    snap.cost = (int)(1000 * snap_weight);
    snap.ik.max_iterations = ik_max_iterations;
    snap.ik.tolerance = ik_tolerance;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) snap.Tk.M[3 * r + c] = T_kin_to_planning[4 * r + c];
        snap.Tk.p[r] = T_kin_to_planning[4 * r + 3];
    }
    SnapLatticePlanner planner(s, std::vector<double>(resolutions, resolutions + dof), prims, use_short_dist != 0,
                               short_dist_thresh, epsilon, max_expansions, &snap);
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
    if (counters) {
        counters[0] = snap.attempted;
        counters[1] = snap.converged;
    }
    return std::chrono::duration<double>(t1 - t0).count();
}

/// The planning-link IK (planningLinkIk) of n problems: pose6[n][6] target-offset goal poses x y z roll pitch yaw,
/// seeds[n][dof]; q_out[n][dof], ok[n], iterations[n].  T_kin_to_planning as for oracle_plan_goal_snap.  Returns the
/// number that converged, or -1 for a scene without kinematics.
int oracle_planning_link_ik(oracle_scene* s, const double* T_kin_to_planning, const double* pose6, const double* seeds,
                            int n, int max_iterations, double tolerance, double* q_out, uint8_t* ok, int32_t* iterations)
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
        const double* P = pose6 + 6 * (size_t)i;
        double R[9];
        rpyMatrix(P[3], P[4], P[5], R);
        q.assign(seeds + (size_t)i * dof, seeds + (size_t)(i + 1) * dof);
        int it = 0;
        const bool conv = planningLinkIk(*s->kdl, Tk, s->xyz_offset, P, R, prm, q, &it);
        std::copy(q.begin(), q.end(), q_out + (size_t)i * dof);
        ok[i] = conv ? 1 : 0;
        iterations[i] = it;
        n_ok += conv ? 1 : 0;
    }
    return n_ok;
}

} // extern "C"
