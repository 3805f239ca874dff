// ORACLE (test infrastructure only -- never linked into the product path).
//
// A planning chain over a subset of the planning variables: the project's own extension of KDLRobotModel, which
// refuses planning joints outside its single chain (kdl_robot_model.cpp:96-108).  The rules, shared with the host's
// RobotTables::setPlanningChain(..., subset = true) (DESIGN.md section 2, parity unpinned):
//   - every movable joint of the root -> tip chain must be a planning variable; it may sit at any index, and its
//     segment reads the variable of its joint's name (Segment::q_index);
//   - a movable chain joint that is not a planning variable is refused, and so is a planning link off the chain;
//   - planning variables off the chain are allowed: they move no segment, and their limits follow getJointLimits'
//     rule (kdl_robot_model.cpp:276-318: soft limits under a safety controller, continuous joints [-pi, pi]).
// The model is oracle/kdl_model.cpp's, unchanged: KDLRobotModel::init builds the chain's segments for the chain's own
// movable joints in chain order (which it accepts), then the segments are pointed at the full planning-variable list
// and the limits are taken for every planning variable.  When the planning variables are exactly the chain's joints
// in chain order, the result is what oracle_scene_init_kdl builds.
//
// Built as oracle/subset_chain/liboracle_subset_chain.so over oracle/liboracle.so; it takes the scene handles of the
// oracle's C API, and the planners of oracle/goals, oracle/goal_sets, oracle/snap and oracle/snap_kinds run on the
// model it installs unchanged (they index through q_index and the model's limits).
#include <algorithm>
#include <cmath>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../bfs3d.h"
#include "../collision_space.h"
#include "../distance_map.h"
#include "../kdl_model.h"
#include "../robot_desc.h"

using namespace oracle;

// The scene handle of oracle/oracle_capi.cpp, restated token for token (one definition across the libraries)
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

namespace {

thread_local std::string g_err;

bool initSubset(KDLRobotModel& m, const RobotDesc& desc, const std::vector<std::string>& planning_joints,
                const std::string& root, const std::string& tip, std::string* err)
{
    // the chain's joints root -> tip (KDL::Tree::getChain, as KDLRobotModel::init walks it)
    std::map<std::string, const JointDesc*> parent_joint;
    for (const JointDesc& j : desc.joints) {
        parent_joint[j.child] = &j;
    }
    std::vector<const JointDesc*> chain;
    for (std::string link = tip; link != root;) {
        auto it = parent_joint.find(link);
        if (it == parent_joint.end()) {
            *err = "Failed to fetch the KDL chain (root: " + root + ", tip: " + tip + ")";
            return false;
        }
        chain.insert(chain.begin(), it->second);
        link = it->second->parent;
    }
    std::vector<std::string> chain_vars;
    for (const JointDesc* j : chain) {
        if (j->type != "fixed") {
            chain_vars.push_back(j->name);
        }
    }
    if (!m.init(desc, chain_vars, root, tip, err)) {
        return false;
    }
    // segment s is chain[s] (init pushes one segment per chain joint, in chain order)
    for (size_t s = 0; s < m.segments.size(); ++s) {
        if (m.segments[s].joint_kind == 0) {
            continue;
        }
        auto it = std::find(planning_joints.begin(), planning_joints.end(), chain[s]->name);
        if (it == planning_joints.end()) {
            *err = "chain joint '" + chain[s]->name + "' is not a planning variable";
            return false;
        }
        m.segments[s].q_index = (int)(it - planning_joints.begin());
    }
    // joint limits of every planning variable: kdl_robot_model.cpp:276-318
    const size_t n = planning_joints.size();
    m.min_limits.assign(n, 0.0);
    m.max_limits.assign(n, 0.0);
    m.continuous.assign(n, false);
    for (size_t i = 0; i < n; ++i) {
        const JointDesc* jd = nullptr;
        for (const JointDesc& j : desc.joints) {
            if (j.name == planning_joints[i] && j.type != "fixed") jd = &j;
        }
        if (!jd) {
            *err = "Joint limits were not found for " + planning_joints[i];
            return false;
        }
        if (jd->type != "continuous") {
            m.min_limits[i] = jd->has_safety ? jd->soft_lower : jd->lower;
            m.max_limits[i] = jd->has_safety ? jd->soft_upper : jd->upper;
        } else {
            m.min_limits[i] = -M_PI;
            m.max_limits[i] = M_PI;
            m.continuous[i] = true;
        }
    }
    return true;
}

} // namespace

extern "C" {

const char* oracle_subset_chain_last_error(void) { return g_err.c_str(); }

/// oracle_scene_init_kdl with the subset rules above; returns 0, or -1 with oracle_subset_chain_last_error set (the
/// scene then has no planning model)
int oracle_scene_init_kdl_subset(oracle_scene* s, const char* chain_root, const char* chain_tip,
                                 const char* planning_link, const double* T_kin_to_planning_3x4,
                                 const double* xyz_offset)
{
    std::unique_ptr<KDLRobotModel> m(new KDLRobotModel);
    s->kdl.reset();
    if (!initSubset(*m, s->desc, s->planning_joints, chain_root, chain_tip, &g_err)) {
        return -1;
    }
    if (!m->setPlanningLink(planning_link)) {
        g_err = "planning link not in chain";
        return -1;
    }
    KdlFrame f;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) f.M[3 * r + c] = T_kin_to_planning_3x4[4 * r + c];
        f.p[r] = T_kin_to_planning_3x4[4 * r + 3];
    }
    m->setKinematicsToPlanningTransform(f);
    s->kdl = std::move(m);
    for (int i = 0; i < 3; ++i) s->xyz_offset[i] = xyz_offset ? xyz_offset[i] : 0.0;
    return 0;
}

} // extern "C"
