// Host-side model builder: turns a robot description + collision group +
// planning variables into the flat tables of include/smplgpu.h.
//
// It plays the role of the reference's host-side precompute, which stays on the
// CPU by design (SURVEY.md section 8a rows a3/a8/a9/a11):
//   RobotCollisionModel::init            sbpl_collision_checking/src/robot_collision_model.cpp:103-623
//   CollisionSphereModelTree::buildFrom  src/base_collision_models.cpp:184-222, 337-444, 569-641
//   RobotMotionCollisionModel ctor       src/robot_motion_collision_model.cpp:41-275
//   SelfCollisionModelImpl ACM + pairs   src/self_collision_model.cpp:280-312, 1233-1345
//   AttachedBodiesCollisionModel         src/attached_bodies_collision_model.cpp:70-141, 264-313
//   KDLRobotModel::init (chain, limits)  sbpl_kdl_robot_model/src/kdl_robot_model.cpp:59-158, 236-320
// Everything here is table-oriented (indices into flat vectors) because its
// only consumer is the device.
#ifndef SMPLHOST_ROBOT_TABLES_H
#define SMPLHOST_ROBOT_TABLES_H

#include <array>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/smplgpu.h"

namespace smplhost {

typedef std::array<double, 12> Mat34; // row-major rotation | translation

enum JointKind { J_FIXED = 0, J_REVOLUTE, J_PRISMATIC, J_CONTINUOUS, J_PLANAR, J_FLOATING };

struct JointRec
{
    std::string name, parent, child;
    JointKind kind;
    double xyz[3], rpy[3], axis[3];
    bool has_limits, has_safety;
    double lower, upper, soft_lower, soft_upper;
};

struct SphereRec { std::string name; double c[3]; double r; int priority; };
struct SpheresRec { std::string link; std::vector<SphereRec> spheres; };
struct VoxelsRec { std::string link; double res; double center[3], size[3]; };
struct GroupRec { std::string name; std::vector<std::string> links, subgroups; std::vector<std::pair<std::string, std::string>> chains; };

/// One bounding-sphere tree in CollisionSphereModelTree node order.
struct SphereTree
{
    std::vector<std::string> name;
    std::vector<double> cx, cy, cz, radius;
    std::vector<int> left, right;
    int root() const { return (int)radius.size() - 1; }
    int size() const { return (int)radius.size(); }
    void build(const std::vector<SphereRec>& spheres);
};

class RobotTables
{
public:
    bool load(const std::string& path, std::string* err);
    bool configure(const std::string& group, const std::vector<std::string>& planning_joints, std::string* err);

    bool setJointPosition(const std::string& variable, double value);
    void useFileAcm();                                       // CollisionSpace::setAllowedCollisionMatrix(file entries)
    void setAcmEntry(const std::string& a, const std::string& b, bool allowed);
    bool attachSpheres(const std::string& id, const std::string& link, const double* centers, int n, double radius);
    bool detach(const std::string& id);
    /// subset = false: KDLRobotModel's rule, the planning variables are exactly the chain's movable joints in chain
    /// order.  subset = true: every movable chain joint is a planning variable at any index; planning variables off
    /// the chain are allowed (they move collision geometry only).
    bool setPlanningChain(const std::string& root, const std::string& tip, const std::string& planning_link,
                          const double T_kin_to_planning[12], const double xyz_offset[3], std::string* err,
                          bool subset = false);

    /// flat tables for smplgpu_set_robot (valid until the next mutating call)
    const smplgpu_robot_desc* desc();

    /// voxels of out-of-group links in the world frame at the current
    /// non-planning joint values (what SelfCollisionModelImpl::updateGroup /
    /// updateVoxelsStates insert into the grid), x y z triples
    std::vector<double> outsideGroupVoxels() const;

    int dof() const { return (int)m_planning_vars.size(); }
    const std::vector<double>& varMin() const { return m_var_min; }
    const std::vector<double>& varMax() const { return m_var_max; }
    const std::vector<int>& varContinuous() const { return m_var_continuous; }
    const std::string& robotName() const { return m_name; }
    int nodeCount();

private:
    // file records
    std::string m_name, m_root, m_world_joint_name, m_world_joint_type;
    std::vector<JointRec> m_joint_recs;
    std::vector<SpheresRec> m_spheres_recs;
    std::vector<VoxelsRec> m_voxels_recs;
    std::vector<GroupRec> m_group_recs;
    std::vector<std::array<std::string, 3>> m_acm_recs; // a, b, "0"/"1"

    // kinematic tree, links in the reference's DFS order
    std::vector<std::string> m_links;
    std::map<std::string, int> m_link_index;
    std::vector<int> m_link_parent;        // parent link index, -1 for the root
    std::vector<int> m_link_joint;         // index into m_joint_recs, -1 for the root (world joint)
    std::vector<std::vector<int>> m_link_children;
    std::vector<double> m_joint_value;     // per joint rec (single-dof joints)
    std::map<std::string, int> m_var_to_joint;

    // collision model
    std::vector<SphereTree> m_trees;       // one per spheres record with >= 1 sphere
    std::vector<int> m_tree_link;
    std::vector<int> m_link_tree;          // link -> tree or -1
    std::vector<std::vector<double>> m_link_voxels; // link-frame voxel centres (xyz triples), per link
    std::vector<int> m_group_links;        // expanded group, sorted by link name
    std::vector<int> m_group_trees;        // trees of the group in spheres-record order

    // planning variables
    std::vector<std::string> m_planning_vars;
    std::vector<int> m_planning_joint;     // joint rec per planning variable
    std::vector<double> m_var_min, m_var_max;
    std::vector<int> m_var_continuous;
    std::vector<double> m_mr_weight;       // per joint rec: ||MR_center|| + MR_radius

    // ACM: symmetric entries, true = ALWAYS
    std::map<std::pair<std::string, std::string>, bool> m_acm;

    struct Attached { std::string id; int link; SphereTree tree; };
    std::vector<Attached> m_attached;

    // planning chain
    bool m_has_chain = false;
    std::vector<int> m_seg_kind, m_seg_var;
    std::vector<double> m_seg_axis, m_seg_origin, m_seg_f_tip;
    int m_n_segments = 0;
    Mat34 m_T_kin;
    double m_xyz_offset[3] = { 0, 0, 0 };

    // flat output
    bool m_dirty = true;
    smplgpu_robot_desc m_desc;
    std::vector<int32_t> o_link_parent, o_link_joint, o_link_var, o_node_link, o_node_left, o_node_right,
        o_tree_root, o_pair_a, o_pair_b, o_allowed_a, o_allowed_b, o_var_type, o_seg_kind, o_seg_var;
    std::vector<double> o_link_origin, o_link_axis, o_link_const, o_link_base, o_node_center, o_node_radius,
        o_var_weight, o_var_min, o_var_max, o_seg_axis, o_seg_origin, o_seg_f_tip, o_T_kin;

    bool expandGroup(const std::string& name, std::vector<std::string>& links, std::vector<std::string>& stack, std::string* err) const;
    void defaultAcm();
    bool acmAlways(const std::string& a, const std::string& b) const;
    void computeMotionWeights();
    std::vector<Mat34> worldPoses() const; // FK of every link at the current joint values
    Mat34 jointTransform(int joint_rec, double value) const;
    void rebuild();
};

} // namespace smplhost

#endif
