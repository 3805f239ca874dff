#include "robot_tables.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <fstream>
#include <functional>
#include <limits>
#include <numeric>
#include <set>
#include <sstream>

namespace smplhost {

///////////////////////////////////////////////////////////////////////////////
// small 3x4 algebra; operation order = Eigen fixed-size products (no FMA: the
// library is built with -ffp-contract=off)
///////////////////////////////////////////////////////////////////////////////

static Mat34 identity()
{
    return Mat34{ { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0 } };
}

static Mat34 mul(const Mat34& a, const Mat34& b)
{
    Mat34 r;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            r[4 * i + j] = (a[4 * i] * b[j] + a[4 * i + 1] * b[4 + j]) + a[4 * i + 2] * b[8 + j];
        }
        r[4 * i + 3] = ((a[4 * i] * b[3] + a[4 * i + 1] * b[7]) + a[4 * i + 2] * b[11]) + a[4 * i + 3];
    }
    return r;
}

static void apply(const Mat34& a, const double v[3], double out[3])
{
    for (int i = 0; i < 3; ++i) {
        out[i] = ((a[4 * i] * v[0] + a[4 * i + 1] * v[1]) + a[4 * i + 2] * v[2]) + a[4 * i + 3];
    }
}

// Eigen::AngleAxisd::toRotationMatrix
static Mat34 angleAxis(double angle, const double ax[3])
{
    Mat34 r = identity();
    const double s = std::sin(angle), c = std::cos(angle);
    const double sx = s * ax[0], sy = s * ax[1], sz = s * ax[2];
    const double k = 1.0 - c;
    const double cx = k * ax[0], cy = k * ax[1], cz = k * ax[2];
    double tmp;
    tmp = cx * ax[1]; r[1] = tmp - sz; r[4] = tmp + sz;
    tmp = cx * ax[2]; r[2] = tmp + sy; r[8] = tmp - sy;
    tmp = cy * ax[2]; r[6] = tmp - sx; r[9] = tmp + sx;
    r[0] = cx * ax[0] + c;
    r[5] = cy * ax[1] + c;
    r[10] = cz * ax[2] + c;
    return r;
}

// urdf rpy -> normalised quaternion; returns x y z w
static void rpyQuaternion(const double rpy[3], double q[4])
{
    const double phi = rpy[0] / 2.0, the = rpy[1] / 2.0, psi = rpy[2] / 2.0;
    q[0] = std::sin(phi) * std::cos(the) * std::cos(psi) - std::cos(phi) * std::sin(the) * std::sin(psi);
    q[1] = std::cos(phi) * std::sin(the) * std::cos(psi) + std::sin(phi) * std::cos(the) * std::sin(psi);
    q[2] = std::cos(phi) * std::cos(the) * std::sin(psi) - std::sin(phi) * std::sin(the) * std::cos(psi);
    q[3] = std::cos(phi) * std::cos(the) * std::cos(psi) + std::sin(phi) * std::sin(the) * std::sin(psi);
    const double s = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    if (std::fabs(s) < 1e-5) {
        q[0] = q[1] = q[2] = 0.0;
        q[3] = 1.0;
    } else {
        for (int i = 0; i < 4; ++i) q[i] /= s;
    }
}

// joint origin as poseUrdfToEigen builds it (Eigen::Quaterniond::toRotationMatrix)
static Mat34 originTransform(const JointRec& j)
{
    double q[4];
    rpyQuaternion(j.rpy, q);
    const double x = q[0], y = q[1], z = q[2], w = q[3];
    const double tx = 2.0 * x, ty = 2.0 * y, tz = 2.0 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    Mat34 r;
    r[0] = 1.0 - (tyy + tzz); r[1] = txy - twz;         r[2] = txz + twy;          r[3] = j.xyz[0];
    r[4] = txy + twz;         r[5] = 1.0 - (txx + tzz); r[6] = tyz - twx;          r[7] = j.xyz[1];
    r[8] = txz - twy;         r[9] = tyz + twx;         r[10] = 1.0 - (txx + tyy); r[11] = j.xyz[2];
    return r;
}

static int jointFn(const JointRec& j)
{
    switch (j.kind) {
    case J_FIXED:
        return SMPLGPU_JOINT_FIXED;
    case J_PRISMATIC:
        return SMPLGPU_JOINT_PRISMATIC;
    case J_REVOLUTE:
    case J_CONTINUOUS:
        if (j.axis[0] == 1.0 && j.axis[1] == 0.0 && j.axis[2] == 0.0) return SMPLGPU_JOINT_REVOLUTE_X;
        if (j.axis[0] == 0.0 && j.axis[1] == 1.0 && j.axis[2] == 0.0) return SMPLGPU_JOINT_REVOLUTE_Y;
        if (j.axis[0] == 0.0 && j.axis[1] == 0.0 && j.axis[2] == 1.0) return SMPLGPU_JOINT_REVOLUTE_Z;
        return SMPLGPU_JOINT_REVOLUTE_AXIS;
    default:
        return SMPLGPU_JOINT_FIXED;
    }
}

// transform_functions.h:95-258
Mat34 RobotTables::jointTransform(int jr, double val) const
{
    const JointRec& j = m_joint_recs[jr];
    const Mat34 o = originTransform(j);
    const int fn = jointFn(j);
    Mat34 t;
    if (fn == SMPLGPU_JOINT_FIXED) {
        return o;
    }
    if (fn == SMPLGPU_JOINT_REVOLUTE_X || fn == SMPLGPU_JOINT_REVOLUTE_Y || fn == SMPLGPU_JOINT_REVOLUTE_Z) {
        const double cth = std::cos(val), sth = std::sin(val);
        for (int r = 0; r < 3; ++r) {
            const double o0 = o[4 * r], o1 = o[4 * r + 1], o2 = o[4 * r + 2];
            if (fn == SMPLGPU_JOINT_REVOLUTE_X) {
                t[4 * r] = o0;
                t[4 * r + 1] = cth * o1 + sth * o2;
                t[4 * r + 2] = cth * o2 - sth * o1;
            } else if (fn == SMPLGPU_JOINT_REVOLUTE_Y) {
                t[4 * r] = cth * o0 - sth * o2;
                t[4 * r + 1] = o1;
                t[4 * r + 2] = sth * o0 + cth * o2;
            } else {
                t[4 * r] = o0 * cth + o1 * sth;
                t[4 * r + 1] = o1 * cth - o0 * sth;
                t[4 * r + 2] = o2;
            }
            t[4 * r + 3] = o[4 * r + 3];
        }
        return t;
    }
    if (fn == SMPLGPU_JOINT_REVOLUTE_AXIS) {
        return mul(o, angleAxis(val, j.axis));
    }
    Mat34 tr = identity();
    tr[11] = val; // prismatic: translation along the local z axis regardless of `axis`
    return mul(o, tr);
}

///////////////////////////////////////////////////////////////////////////////
// description file
///////////////////////////////////////////////////////////////////////////////

static bool parseKind(const std::string& s, JointKind& k)
{
    if (s == "fixed") k = J_FIXED;
    else if (s == "revolute") k = J_REVOLUTE;
    else if (s == "prismatic") k = J_PRISMATIC;
    else if (s == "continuous") k = J_CONTINUOUS;
    else if (s == "planar") k = J_PLANAR;
    else if (s == "floating") k = J_FLOATING;
    else return false;
    return true;
}

bool RobotTables::load(const std::string& path, std::string* err)
{
    std::ifstream f(path.c_str());
    if (!f) {
        if (err) *err = "cannot open " + path;
        return false;
    }
    *this = RobotTables();
    std::string line;
    int lineno = 0;
    while (std::getline(f, line)) {
        ++lineno;
        std::istringstream ss(line);
        std::string key;
        if (!(ss >> key) || key[0] == '#') continue;
        bool ok = true;
        if (key == "robot") ok = !!(ss >> m_name);
        else if (key == "root") ok = !!(ss >> m_root);
        else if (key == "world_joint") ok = !!(ss >> m_world_joint_name >> m_world_joint_type);
        else if (key == "joint") {
            JointRec j;
            std::string kind;
            int hl = 0, hs = 0;
            ok = !!(ss >> j.name >> kind >> j.parent >> j.child >> j.xyz[0] >> j.xyz[1] >> j.xyz[2]
                       >> j.rpy[0] >> j.rpy[1] >> j.rpy[2] >> j.axis[0] >> j.axis[1] >> j.axis[2]
                       >> hl >> j.lower >> j.upper >> hs >> j.soft_lower >> j.soft_upper)
                 && parseKind(kind, j.kind);
            j.has_limits = hl != 0;
            j.has_safety = hs != 0;
            m_joint_recs.push_back(j);
        } else if (key == "spheres_model") {
            SpheresRec s;
            ok = !!(ss >> s.link);
            m_spheres_recs.push_back(s);
        } else if (key == "sphere") {
            SphereRec s;
            ok = !m_spheres_recs.empty() && !!(ss >> s.name >> s.c[0] >> s.c[1] >> s.c[2] >> s.r >> s.priority);
            if (ok) m_spheres_recs.back().spheres.push_back(s);
        } else if (key == "voxels_model") {
            VoxelsRec v;
            ok = !!(ss >> v.link >> v.res >> v.center[0] >> v.center[1] >> v.center[2] >> v.size[0] >> v.size[1] >> v.size[2]);
            m_voxels_recs.push_back(v);
        } else if (key == "group") {
            GroupRec g;
            ok = !!(ss >> g.name);
            m_group_recs.push_back(g);
        } else if (key == "group_link") {
            std::string n;
            ok = !m_group_recs.empty() && !!(ss >> n);
            if (ok) m_group_recs.back().links.push_back(n);
        } else if (key == "group_chain") {
            std::string b, t;
            ok = !m_group_recs.empty() && !!(ss >> b >> t);
            if (ok) m_group_recs.back().chains.emplace_back(b, t);
        } else if (key == "group_sub") {
            std::string n;
            ok = !m_group_recs.empty() && !!(ss >> n);
            if (ok) m_group_recs.back().subgroups.push_back(n);
        } else if (key == "acm") {
            std::array<std::string, 3> e;
            ok = !!(ss >> e[0] >> e[1] >> e[2]);
            m_acm_recs.push_back(e);
        } else {
            ok = false;
        }
        if (!ok) {
            if (err) *err = path + ":" + std::to_string(lineno) + ": malformed '" + key + "' record";
            return false;
        }
    }
    if (m_name.empty() || m_root.empty()) {
        if (err) *err = path + ": missing robot/root record";
        return false;
    }

    // kinematic tree in the reference's link order: depth-first, children in
    // joint-name order (robot_collision_model.cpp:160-197 over urdfdom's map)
    std::map<std::string, std::vector<int>> children; // parent link -> joint recs
    {
        std::vector<int> by_name(m_joint_recs.size());
        std::iota(by_name.begin(), by_name.end(), 0);
        std::sort(by_name.begin(), by_name.end(), [&](int a, int b) { return m_joint_recs[a].name < m_joint_recs[b].name; });
        for (int jr : by_name) {
            children[m_joint_recs[jr].parent].push_back(jr);
        }
    }
    struct Item { std::string link; int parent; int joint; };
    std::vector<Item> stack;
    stack.push_back({ m_root, -1, -1 });
    while (!stack.empty()) {
        Item it = stack.back();
        stack.pop_back();
        const int lidx = (int)m_links.size();
        m_links.push_back(it.link);
        m_link_index[it.link] = lidx;
        m_link_parent.push_back(it.parent);
        m_link_joint.push_back(it.joint);
        auto c = children.find(it.link);
        if (c != children.end()) {
            for (auto jt = c->second.rbegin(); jt != c->second.rend(); ++jt) {
                stack.push_back({ m_joint_recs[*jt].child, lidx, *jt });
            }
        }
    }
    m_link_children.assign(m_links.size(), std::vector<int>());
    for (size_t l = 1; l < m_links.size(); ++l) {
        m_link_children[m_link_parent[l]].push_back((int)l);
    }

    // default joint values: RobotCollisionState::initRobotState (robot_collision_state.cpp:207-222)
    m_joint_value.assign(m_joint_recs.size(), 0.0);
    for (size_t jr = 0; jr < m_joint_recs.size(); ++jr) {
        const JointRec& j = m_joint_recs[jr];
        if (j.kind == J_REVOLUTE || j.kind == J_PRISMATIC) {
            const double lo = j.has_safety ? j.soft_lower : j.lower;
            const double hi = j.has_safety ? j.soft_upper : j.upper;
            if (j.has_limits && (lo > 0.0 || hi < 0.0)) {
                m_joint_value[jr] = 0.5 * (lo + hi);
            }
        }
        if (j.kind != J_FIXED) {
            m_var_to_joint[j.name] = (int)jr;
        }
    }

    // sphere trees and voxel lattices
    m_link_tree.assign(m_links.size(), -1);
    for (const SpheresRec& s : m_spheres_recs) {
        if (s.spheres.empty()) continue;
        auto it = m_link_index.find(s.link);
        if (it == m_link_index.end()) {
            if (err) *err = "spheres model for unknown link '" + s.link + "'";
            return false;
        }
        m_trees.emplace_back();
        m_trees.back().build(s.spheres);
        m_tree_link.push_back(it->second);
        m_link_tree[it->second] = (int)m_trees.size() - 1;
    }
    m_link_voxels.assign(m_links.size(), std::vector<double>());
    for (const VoxelsRec& v : m_voxels_recs) {
        auto it = m_link_index.find(v.link);
        if (it == m_link_index.end()) {
            if (err) *err = "voxels model for unknown link '" + v.link + "'";
            return false;
        }
        int n[3];
        for (int a = 0; a < 3; ++a) n[a] = (int)std::floor(v.size[a] / v.res + 0.5);
        std::vector<double>& out = m_link_voxels[it->second];
        if (n[0] > 0 && n[1] > 0 && n[2] > 0) {
            for (int ix = 0; ix < n[0]; ++ix)
            for (int iy = 0; iy < n[1]; ++iy)
            for (int iz = 0; iz < n[2]; ++iz) {
                out.push_back(v.center[0] - 0.5 * v.size[0] + (ix + 0.5) * v.res);
                out.push_back(v.center[1] - 0.5 * v.size[1] + (iy + 0.5) * v.res);
                out.push_back(v.center[2] - 0.5 * v.size[2] + (iz + 0.5) * v.res);
            }
        }
    }
    defaultAcm();
    computeMotionWeights();
    m_T_kin = identity();
    m_dirty = true;
    return true;
}

///////////////////////////////////////////////////////////////////////////////
// sphere tree: base_collision_models.cpp:337-444 (buildRecursive),
// :569-592 (optimal two-sphere bound), :594-641 (largest bounding-box axis)
///////////////////////////////////////////////////////////////////////////////

void SphereTree::build(const std::vector<SphereRec>& spheres)
{
    name.clear(); cx.clear(); cy.clear(); cz.clear(); radius.clear(); left.clear(); right.clear();
    std::vector<int> order(spheres.size());
    std::iota(order.begin(), order.end(), 0);

    std::function<int(std::vector<int>::iterator, std::vector<int>::iterator)> rec =
        [&](std::vector<int>::iterator first, std::vector<int>::iterator last) -> int {
        const long count = last - first;
        if (count == 0) {
            return -1;
        }
        if (count == 1) {
            const SphereRec& s = spheres[*first];
            name.push_back(s.name);
            cx.push_back(s.c[0]); cy.push_back(s.c[1]); cz.push_back(s.c[2]);
            radius.push_back(s.r);
            left.push_back(-1); right.push_back(-1);
            return size() - 1;
        }
        // split axis: largest extent of the centre bounding box
        double mn[3] = { spheres[*first].c[0], spheres[*first].c[1], spheres[*first].c[2] };
        double mx[3] = { mn[0], mn[1], mn[2] };
        for (auto it = first; it != last; ++it) {
            for (int a = 0; a < 3; ++a) {
                const double v = spheres[*it].c[a];
                if (v < mn[a]) mn[a] = v;
                if (v > mx[a]) mx[a] = v;
            }
        }
        const double sx = mx[0] - mn[0], sy = mx[1] - mn[1], sz = mx[2] - mn[2];
        const int axis = (sx > sy && sx > sz) ? 0 : (sy > sz ? 1 : 2);

        // centroid bound
        double cen[3] = { 0.0, 0.0, 0.0 };
        for (auto it = first; it != last; ++it) {
            for (int a = 0; a < 3; ++a) cen[a] = cen[a] + spheres[*it].c[a];
        }
        for (int a = 0; a < 3; ++a) cen[a] = cen[a] / (double)count;
        double cen_r = 0.0;
        for (auto it = first; it != last; ++it) {
            const SphereRec& s = spheres[*it];
            const double dx = s.c[0] - cen[0], dy = s.c[1] - cen[1], dz = s.c[2] - cen[2];
            const double r = std::sqrt((dx * dx + dy * dy) + dz * dz) + s.r;
            if (r > cen_r) cen_r = r;
        }

        const double pivot = cen[axis];
        auto mid = std::partition(first, last, [&](int i) { return spheres[i].c[axis] < pivot; });
        if (mid == first || mid == last) {
            mid = first + (count >> 1);
        }
        const int li = rec(first, mid);
        const int ri = rec(mid, last);

        // optimal sphere around the two children
        const double p[3] = { cx[li], cy[li], cz[li] }, q[3] = { cx[ri], cy[ri], cz[ri] };
        const double r1 = radius[li], r2 = radius[ri];
        const double v[3] = { q[0] - p[0], q[1] - p[1], q[2] - p[2] };
        const double dist = std::sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]);
        double gc[3], gr;
        if (r1 > dist + r2) {
            gc[0] = p[0]; gc[1] = p[1]; gc[2] = p[2]; gr = r1;
        } else if (r2 > dist + r1) {
            gc[0] = q[0]; gc[1] = q[1]; gc[2] = q[2]; gr = r2;
        } else {
            double vn[3] = { v[0], v[1], v[2] };
            if (dist > 0.0) {
                for (int a = 0; a < 3; ++a) vn[a] = v[a] / dist;
            }
            double a3[3], b3[3], d3[3];
            for (int a = 0; a < 3; ++a) {
                a3[a] = q[a] + vn[a] * r2;
                b3[a] = p[a] - vn[a] * r1;
                gc[a] = 0.5 * (a3[a] + b3[a]);
                d3[a] = a3[a] - b3[a];
            }
            gr = 0.5 * std::sqrt((d3[0] * d3[0] + d3[1] * d3[1]) + d3[2] * d3[2]);
        }
        name.push_back(std::string());
        if (gr < cen_r) {
            cx.push_back(gc[0]); cy.push_back(gc[1]); cz.push_back(gc[2]); radius.push_back(gr);
        } else {
            cx.push_back(cen[0]); cy.push_back(cen[1]); cz.push_back(cen[2]); radius.push_back(cen_r);
        }
        left.push_back(li);
        right.push_back(ri);
        return size() - 1;
    };
    rec(order.begin(), order.end());
}

///////////////////////////////////////////////////////////////////////////////
// groups, ACM, motion weights
///////////////////////////////////////////////////////////////////////////////

// robot_collision_model.cpp:625-756: own links + chain links + sub-group links
bool RobotTables::expandGroup(const std::string& name, std::vector<std::string>& links,
                              std::vector<std::string>& stack, std::string* err) const
{
    const GroupRec* g = nullptr;
    for (const GroupRec& r : m_group_recs) {
        if (r.name == name) g = &r;
    }
    if (!g) {
        if (err) *err = "group '" + name + "' not found";
        return false;
    }
    if (std::find(stack.begin(), stack.end(), name) != stack.end()) {
        if (err) *err = "cycle in group config";
        return false;
    }
    stack.push_back(name);
    links.insert(links.end(), g->links.begin(), g->links.end());
    for (const auto& ch : g->chains) {
        std::string link = ch.second;
        links.push_back(link);
        while (link != ch.first) {
            auto it = m_link_index.find(link);
            if (it == m_link_index.end() || m_link_parent[it->second] < 0) {
                if (err) *err = "(" + ch.first + ", " + ch.second + ") is not a chain in the robot model";
                return false;
            }
            link = m_links[m_link_parent[it->second]];
            links.push_back(link);
        }
    }
    for (const std::string& sub : g->subgroups) {
        if (!expandGroup(sub, links, stack, err)) return false;
    }
    stack.pop_back();
    return true;
}

// self_collision_model.cpp:280-312: adjacent links may touch
void RobotTables::defaultAcm()
{
    m_acm.clear();
    for (size_t l = 1; l < m_links.size(); ++l) {
        const int p = m_link_parent[l];
        // the reference skips the pair whose connecting joint is joint 0 (the world joint);
        // every other parent/child pair is allowed
        m_acm[std::make_pair(m_links[l], m_links[p])] = true;
        m_acm[std::make_pair(m_links[p], m_links[l])] = true;
    }
}

void RobotTables::useFileAcm()
{
    m_acm.clear();
    for (const auto& e : m_acm_recs) {
        const bool allowed = e[2] != "0";
        m_acm[std::make_pair(e[0], e[1])] = allowed;
        m_acm[std::make_pair(e[1], e[0])] = allowed;
    }
    m_dirty = true;
}

void RobotTables::setAcmEntry(const std::string& a, const std::string& b, bool allowed)
{
    m_acm[std::make_pair(a, b)] = allowed;
    m_acm[std::make_pair(b, a)] = allowed;
    m_dirty = true;
}

bool RobotTables::acmAlways(const std::string& a, const std::string& b) const
{
    auto it = m_acm.find(std::make_pair(a, b));
    return it != m_acm.end() && it->second;
}

// robot_motion_collision_model.cpp:41-275, bottom-up over the kinematic tree.
// Joint index j here is "the parent joint of link j" (link 0 = world joint).
void RobotTables::computeMotionWeights()
{
    const int nl = (int)m_links.size();
    std::vector<std::vector<double>> samples(nl); // xyz triples of MR(j) samples, in joint j's parent frame
    std::vector<double> sample_r(nl, 0.0);
    std::vector<double> weight(nl, 0.0);
    std::vector<int> pending(nl, 0), queue;
    for (int l = 0; l < nl; ++l) {
        pending[l] = (int)m_link_children[l].size();
        if (pending[l] == 0) queue.push_back(l);
    }
    const double PI = M_PI;
    for (size_t qi = 0; qi < queue.size(); ++qi) {
        const int l = queue[qi];
        std::vector<double> cen; // xyz triples
        std::vector<double> rad;
        if (m_link_tree[l] >= 0) {
            const SphereTree& t = m_trees[m_link_tree[l]];
            const int r = t.root();
            cen.push_back(t.cx[r]); cen.push_back(t.cy[r]); cen.push_back(t.cz[r]);
            rad.push_back(t.radius[r]);
        }
        for (int c : m_link_children[l]) {
            if (sample_r[c] != 0.0) {
                const Mat34 o = originTransform(m_joint_recs[m_link_joint[c]]);
                for (size_t k = 0; k + 2 < samples[c].size(); k += 3) {
                    double out[3];
                    apply(o, &samples[c][k], out);
                    cen.push_back(out[0]); cen.push_back(out[1]); cen.push_back(out[2]);
                    rad.push_back(sample_r[c]);
                }
            }
        }
        double mc[3] = { 0.0, 0.0, 0.0 };
        double mr = 0.0;
        const size_t n = rad.size();
        if (n > 0) {
            for (size_t k = 0; k < n; ++k) {
                for (int a = 0; a < 3; ++a) mc[a] = mc[a] + cen[3 * k + a];
            }
            for (int a = 0; a < 3; ++a) mc[a] = mc[a] / (double)n;
            for (size_t k = 0; k < n; ++k) {
                const double dx = cen[3 * k] - mc[0], dy = cen[3 * k + 1] - mc[1], dz = cen[3 * k + 2] - mc[2];
                mr = std::max(mr, std::sqrt((dx * dx + dy * dy) + dz * dz) + rad[k]);
            }
        }
        weight[l] = std::sqrt((mc[0] * mc[0] + mc[1] * mc[1]) + mc[2] * mc[2]) + mr;

        // samples of MR under this joint's motion
        std::vector<double>& out = samples[l];
        if (mr != 0.0 && m_link_joint[l] >= 0) {
            const JointRec& j = m_joint_recs[m_link_joint[l]];
            double res = 2.0 * PI / 180.0;
            auto push = [&](const Mat34& T) {
                double p[3];
                apply(T, mc, p);
                out.push_back(p[0]); out.push_back(p[1]); out.push_back(p[2]);
            };
            if (j.kind == J_REVOLUTE || j.kind == J_PRISMATIC) {
                const double lo = j.has_safety ? j.soft_lower : j.lower;
                const double hi = j.has_safety ? j.soft_upper : j.upper;
                const double span = hi - lo;
                const int count = (int)std::round(span / res) + 1;
                for (int i = 0; i < count; ++i) {
                    const double alpha = (double)i / (double)(count - 1);
                    const double val = (1.0 - alpha) * lo + alpha * hi;
                    if (j.kind == J_REVOLUTE) {
                        push(angleAxis(val, j.axis));
                    } else {
                        Mat34 T = identity();
                        T[3] = val * j.axis[0]; T[7] = val * j.axis[1]; T[11] = val * j.axis[2];
                        push(T);
                    }
                }
            } else if (j.kind == J_CONTINUOUS) {
                const int count = (int)std::round(2.0 * PI / res);
                res = 2.0 * PI / count;
                for (int i = 0; i < count; ++i) {
                    push(angleAxis(i * res, j.axis));
                }
            } else if (j.kind == J_FIXED) {
                push(originTransform(j));
            }
        }
        sample_r[l] = mr;

        const int p = m_link_parent[l];
        if (p >= 0 && --pending[p] == 0) {
            queue.push_back(p);
        }
    }
    m_mr_weight.assign(m_joint_recs.size(), 0.0);
    for (int l = 0; l < nl; ++l) {
        if (m_link_joint[l] >= 0) {
            m_mr_weight[m_link_joint[l]] = weight[l];
        }
    }
}

///////////////////////////////////////////////////////////////////////////////
// configuration
///////////////////////////////////////////////////////////////////////////////

bool RobotTables::configure(const std::string& group, const std::vector<std::string>& planning_joints, std::string* err)
{
    std::vector<std::string> names, stack;
    if (!expandGroup(group, names, stack, err)) {
        return false;
    }
    std::sort(names.begin(), names.end());
    names.erase(std::unique(names.begin(), names.end()), names.end());
    m_group_links.clear();
    for (const std::string& n : names) {
        auto it = m_link_index.find(n);
        if (it == m_link_index.end()) {
            if (err) *err = "group '" + group + "' references unknown link '" + n + "'";
            return false;
        }
        m_group_links.push_back(it->second);
    }
    m_group_trees.clear();
    for (size_t t = 0; t < m_trees.size(); ++t) {
        if (std::find(m_group_links.begin(), m_group_links.end(), m_tree_link[t]) != m_group_links.end()) {
            m_group_trees.push_back((int)t);
        }
    }
    m_planning_vars = planning_joints;
    m_planning_joint.clear();
    m_var_min.clear(); m_var_max.clear(); m_var_continuous.clear();
    for (const std::string& v : planning_joints) {
        auto it = m_var_to_joint.find(v);
        if (it == m_var_to_joint.end()) {
            if (err) *err = "Joint variable '" + v + "' not found in Robot Collision Model";
            return false;
        }
        const JointRec& j = m_joint_recs[it->second];
        if (j.kind == J_PLANAR || j.kind == J_FLOATING) {
            if (err) *err = "multi-dof planning joints are not supported";
            return false;
        }
        m_planning_joint.push_back(it->second);
        // KDLRobotModel::getJointLimits (kdl_robot_model.cpp:276-318)
        if (j.kind == J_CONTINUOUS) {
            m_var_min.push_back(-M_PI);
            m_var_max.push_back(M_PI);
            m_var_continuous.push_back(1);
        } else {
            m_var_min.push_back(j.has_safety ? j.soft_lower : j.lower);
            m_var_max.push_back(j.has_safety ? j.soft_upper : j.upper);
            m_var_continuous.push_back(0);
        }
    }
    m_dirty = true;
    return true;
}

bool RobotTables::setJointPosition(const std::string& variable, double value)
{
    auto it = m_var_to_joint.find(variable);
    if (it == m_var_to_joint.end()) {
        return false;
    }
    m_joint_value[it->second] = value;
    m_dirty = true;
    return true;
}

bool RobotTables::attachSpheres(const std::string& id, const std::string& link, const double* centers, int n, double radius)
{
    auto it = m_link_index.find(link);
    if (it == m_link_index.end() || n <= 0) {
        return false;
    }
    for (const Attached& a : m_attached) {
        if (a.id == id) return false;
    }
    std::vector<SphereRec> recs(n);
    for (int i = 0; i < n; ++i) {
        recs[i].name = id + "/" + std::to_string(i);
        recs[i].c[0] = centers[3 * i]; recs[i].c[1] = centers[3 * i + 1]; recs[i].c[2] = centers[3 * i + 2];
        recs[i].r = radius;
        recs[i].priority = 0;
    }
    m_attached.emplace_back();
    m_attached.back().id = id;
    m_attached.back().link = it->second;
    m_attached.back().tree.build(recs);
    m_dirty = true;
    return true;
}

bool RobotTables::detach(const std::string& id)
{
    for (size_t i = 0; i < m_attached.size(); ++i) {
        if (m_attached[i].id == id) {
            m_attached.erase(m_attached.begin() + i);
            m_dirty = true;
            return true;
        }
    }
    return false;
}

std::vector<Mat34> RobotTables::worldPoses() const
{
    std::vector<Mat34> T(m_links.size(), identity());
    for (size_t l = 1; l < m_links.size(); ++l) {
        const int jr = m_link_joint[l];
        T[l] = mul(T[m_link_parent[l]], jointTransform(jr, m_joint_value[jr]));
    }
    return T;
}

std::vector<double> RobotTables::outsideGroupVoxels() const
{
    const std::vector<Mat34> T = worldPoses();
    std::vector<double> out;
    for (size_t l = 0; l < m_links.size(); ++l) {
        if (m_link_voxels[l].empty()) continue;
        if (std::find(m_group_links.begin(), m_group_links.end(), (int)l) != m_group_links.end()) continue;
        for (size_t k = 0; k + 2 < m_link_voxels[l].size(); k += 3) {
            double p[3];
            apply(T[l], &m_link_voxels[l][k], p);
            out.push_back(p[0]); out.push_back(p[1]); out.push_back(p[2]);
        }
    }
    return out;
}

///////////////////////////////////////////////////////////////////////////////
// planning chain (KDLRobotModel + kdl_parser + orocos_kdl semantics)
///////////////////////////////////////////////////////////////////////////////

bool RobotTables::setPlanningChain(const std::string& root, const std::string& tip, const std::string& planning_link,
                                   const double T_kin[12], const double xyz_offset[3], std::string* err, bool subset)
{
    std::vector<int> chain; // joint recs root -> tip
    std::string link = tip;
    while (link != root) {
        auto it = m_link_index.find(link);
        if (it == m_link_index.end() || m_link_joint[it->second] < 0) {
            if (err) *err = "Failed to fetch the KDL chain for the robot. (root: " + root + ", tip: " + tip + ")";
            return false;
        }
        chain.insert(chain.begin(), m_link_joint[it->second]);
        link = m_links[m_link_parent[it->second]];
    }
    // every movable chain joint must be a planning variable, in chain order (subset mode: at any index)
    std::vector<int> seg_var;
    int k = 0;
    for (int jr : chain) {
        if (m_joint_recs[jr].kind == J_FIXED) {
            seg_var.push_back(-1);
        } else if (subset) {
            auto it = std::find(m_planning_joint.begin(), m_planning_joint.end(), jr);
            if (it == m_planning_joint.end()) {
                if (err) *err = "chain joint '" + m_joint_recs[jr].name + "' is not a planning variable";
                return false;
            }
            seg_var.push_back((int)(it - m_planning_joint.begin()));
        } else {
            if (k >= (int)m_planning_joint.size() || m_planning_joint[k] != jr) {
                if (err) *err = "planning joints do not match the movable joints of the chain at '" + m_joint_recs[jr].name + "'";
                return false;
            }
            seg_var.push_back(k++);
        }
    }
    if (!subset && k != (int)m_planning_joint.size()) {
        if (err) *err = "a planning joint is not part of the kinematic chain";
        return false;
    }
    int planning_seg = -1;
    for (size_t s = 0; s < chain.size(); ++s) {
        if (m_joint_recs[chain[s]].child == planning_link) planning_seg = (int)s;
    }
    if (planning_seg < 0) {
        if (err) *err = "planning link '" + planning_link + "' is not a segment of the chain";
        return false;
    }
    // JntToCart(q, out, segmentNr = planning_seg) multiplies segments [0, planning_seg)
    m_n_segments = planning_seg;
    m_seg_kind.clear(); m_seg_var.clear(); m_seg_axis.clear(); m_seg_origin.clear(); m_seg_f_tip.clear();
    for (int s = 0; s < planning_seg; ++s) {
        const JointRec& j = m_joint_recs[chain[s]];
        // F_parent_jnt: KDL Rotation::Quaternion(x,y,z,w) of the urdf origin
        double q[4];
        rpyQuaternion(j.rpy, q);
        const double x = q[0], y = q[1], z = q[2], w = q[3];
        const double x2 = x * x, y2 = y * y, z2 = z * z, w2 = w * w;
        const double M[9] = {
            w2 + x2 - y2 - z2, 2 * x * y - 2 * w * z, 2 * x * z + 2 * w * y,
            2 * x * y + 2 * w * z, w2 - x2 + y2 - z2, 2 * y * z - 2 * w * x,
            2 * x * z - 2 * w * y, 2 * y * z + 2 * w * x, w2 - x2 - y2 + z2 };
        double axis[3] = { 0, 0, 0 }, origin[3] = { 0, 0, 0 };
        int kind = SMPLGPU_SEG_NONE;
        // f_tip = joint.pose(0).Inverse() * F_parent_jnt
        double ftip[12];
        if (j.kind == J_FIXED) {
            // pose(0) = identity
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) ftip[4 * r + c] = M[3 * r + c];
                ftip[4 * r + 3] = j.xyz[r];
            }
        } else {
            kind = (j.kind == J_PRISMATIC) ? SMPLGPU_SEG_TRANS : SMPLGPU_SEG_ROT;
            double a[3];
            for (int r = 0; r < 3; ++r) {
                a[r] = M[3 * r] * j.axis[0] + M[3 * r + 1] * j.axis[1] + M[3 * r + 2] * j.axis[2];
            }
            const double n = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
            for (int r = 0; r < 3; ++r) {
                axis[r] = a[r] / n;
                origin[r] = j.xyz[r];
            }
            // joint.pose(0) = Frame(Identity, origin); inverse = Frame(Identity, -(I * origin));
            // Frame*Frame = (M1*M2, M1*p2 + p1) with M1 = I evaluated term by term
            const double ip[3] = { -((1.0 * origin[0] + 0.0 * origin[1]) + 0.0 * origin[2]),
                                   -((0.0 * origin[0] + 1.0 * origin[1]) + 0.0 * origin[2]),
                                   -((0.0 * origin[0] + 0.0 * origin[1]) + 1.0 * origin[2]) };
            const double I[9] = { 1, 0, 0, 0, 1, 0, 0, 0, 1 };
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) {
                    ftip[4 * r + c] = I[3 * r] * M[c] + I[3 * r + 1] * M[3 + c] + I[3 * r + 2] * M[6 + c];
                }
                ftip[4 * r + 3] = (I[3 * r] * j.xyz[0] + I[3 * r + 1] * j.xyz[1] + I[3 * r + 2] * j.xyz[2]) + ip[r];
            }
        }
        m_seg_kind.push_back(kind);
        m_seg_var.push_back(seg_var[s]);
        m_seg_axis.insert(m_seg_axis.end(), axis, axis + 3);
        m_seg_origin.insert(m_seg_origin.end(), origin, origin + 3);
        m_seg_f_tip.insert(m_seg_f_tip.end(), ftip, ftip + 12);
    }
    for (int i = 0; i < 12; ++i) m_T_kin[i] = T_kin ? T_kin[i] : identity()[i];
    for (int i = 0; i < 3; ++i) m_xyz_offset[i] = xyz_offset ? xyz_offset[i] : 0.0;
    m_has_chain = true;
    m_dirty = true;
    return true;
}

///////////////////////////////////////////////////////////////////////////////
// flat tables
///////////////////////////////////////////////////////////////////////////////

int RobotTables::nodeCount()
{
    return desc()->n_nodes;
}

const smplgpu_robot_desc* RobotTables::desc()
{
    if (m_dirty) {
        rebuild();
        m_dirty = false;
    }
    return &m_desc;
}

void RobotTables::rebuild()
{
    const int nl = (int)m_links.size();
    const std::vector<Mat34> T = worldPoses();

    // links moved by a planning variable
    std::vector<bool> moved(nl, false);
    for (int l = 1; l < nl; ++l) {
        const int jr = m_link_joint[l];
        const bool planning = std::find(m_planning_joint.begin(), m_planning_joint.end(), jr) != m_planning_joint.end();
        moved[l] = moved[m_link_parent[l]] || planning;
    }
    // links that carry group geometry: sphere trees of the group + attached bodies on group links
    std::vector<bool> needed(nl, false);
    for (int t : m_group_trees) needed[m_tree_link[t]] = true;
    std::vector<int> group_attached;
    for (size_t b = 0; b < m_attached.size(); ++b) {
        if (std::find(m_group_links.begin(), m_group_links.end(), m_attached[b].link) != m_group_links.end()) {
            group_attached.push_back((int)b);
            needed[m_attached[b].link] = true;
        }
    }
    // device links: needed links and their moved ancestors
    std::vector<bool> on_dev(nl, false);
    for (int l = 0; l < nl; ++l) {
        if (!needed[l]) continue;
        if (!moved[l]) {
            on_dev[l] = true; // static: listed as FIXED with base = pose
            continue;
        }
        for (int a = l; a >= 0 && moved[a]; a = m_link_parent[a]) {
            on_dev[a] = true;
        }
    }
    std::vector<int> dev_index(nl, -1);
    o_link_parent.clear(); o_link_joint.clear(); o_link_var.clear();
    o_link_origin.clear(); o_link_axis.clear(); o_link_const.clear(); o_link_base.clear();
    const Mat34 I = identity();
    for (int l = 0; l < nl; ++l) {
        if (!on_dev[l]) continue;
        dev_index[l] = (int)o_link_parent.size();
        if (!moved[l]) {
            o_link_parent.push_back(-1);
            o_link_joint.push_back(SMPLGPU_JOINT_FIXED);
            o_link_var.push_back(-1);
            o_link_const.push_back(0.0);
            o_link_origin.insert(o_link_origin.end(), I.begin(), I.end());
            const double z3[3] = { 0, 0, 0 };
            o_link_axis.insert(o_link_axis.end(), z3, z3 + 3);
            o_link_base.insert(o_link_base.end(), T[l].begin(), T[l].end());
            continue;
        }
        const int jr = m_link_joint[l];
        const JointRec& j = m_joint_recs[jr];
        const int p = m_link_parent[l];
        const Mat34 o = originTransform(j);
        o_link_parent.push_back(moved[p] ? dev_index[p] : -1);
        o_link_joint.push_back(jointFn(j));
        auto pv = std::find(m_planning_joint.begin(), m_planning_joint.end(), jr);
        o_link_var.push_back(pv == m_planning_joint.end() ? -1 : (int)(pv - m_planning_joint.begin()));
        o_link_const.push_back(m_joint_value[jr]);
        o_link_origin.insert(o_link_origin.end(), o.begin(), o.end());
        o_link_axis.insert(o_link_axis.end(), j.axis, j.axis + 3);
        o_link_base.insert(o_link_base.end(), T[p].begin(), T[p].end());
    }

    // nodes and trees: robot trees of the group in spheres-record order, then attached bodies
    o_node_link.clear(); o_node_left.clear(); o_node_right.clear(); o_node_center.clear(); o_node_radius.clear();
    o_tree_root.clear();
    std::vector<int> tree_first; // first node of every emitted tree
    std::vector<const SphereTree*> emitted;
    std::vector<std::string> tree_owner; // link name / body id for the ACM
    auto emit = [&](const SphereTree& t, int link, const std::string& owner) {
        const int base = (int)o_node_link.size();
        tree_first.push_back(base);
        emitted.push_back(&t);
        tree_owner.push_back(owner);
        for (int i = 0; i < t.size(); ++i) {
            o_node_link.push_back(dev_index[link]);
            o_node_left.push_back(t.left[i] < 0 ? -1 : base + t.left[i]);
            o_node_right.push_back(t.right[i] < 0 ? -1 : base + t.right[i]);
            o_node_center.push_back(t.cx[i]); o_node_center.push_back(t.cy[i]); o_node_center.push_back(t.cz[i]);
            o_node_radius.push_back(t.radius[i]);
        }
        o_tree_root.push_back(base + t.root());
    };
    for (int t : m_group_trees) emit(m_trees[t], m_tree_link[t], m_links[m_tree_link[t]]);
    const int n_robot_trees = (int)o_tree_root.size();
    for (int b : group_attached) emit(m_attached[b].tree, m_attached[b].link, m_attached[b].id);

    // checked pairs: robot x robot (self_collision_model.cpp:1233-1268), group links in sorted-name order
    o_pair_a.clear(); o_pair_b.clear();
    auto group_tree_of_link = [&](int link) {
        for (int k = 0; k < n_robot_trees; ++k) {
            if (m_tree_link[m_group_trees[k]] == link) return k;
        }
        return -1;
    };
    for (size_t a = 0; a < m_group_links.size(); ++a) {
        const int la = m_group_links[a];
        if (m_link_tree[la] < 0) continue;
        for (size_t b = a + 1; b < m_group_links.size(); ++b) {
            const int lb = m_group_links[b];
            if (m_link_tree[lb] < 0) continue;
            if (acmAlways(m_links[la], m_links[lb])) continue;
            o_pair_a.push_back(group_tree_of_link(la));
            o_pair_b.push_back(group_tree_of_link(lb));
        }
    }
    // attached x attached (:1309-1345), then attached x robot (:1270-1307)
    for (size_t a = 0; a < group_attached.size(); ++a) {
        for (size_t b = a + 1; b < group_attached.size(); ++b) {
            if (acmAlways(m_attached[group_attached[a]].id, m_attached[group_attached[b]].id)) continue;
            o_pair_a.push_back(n_robot_trees + (int)a);
            o_pair_b.push_back(n_robot_trees + (int)b);
        }
    }
    for (size_t a = 0; a < group_attached.size(); ++a) {
        for (size_t g = 0; g < m_group_links.size(); ++g) {
            const int lg = m_group_links[g];
            if (m_link_tree[lg] < 0) continue;
            if (acmAlways(m_attached[group_attached[a]].id, m_links[lg])) continue;
            o_pair_a.push_back(n_robot_trees + (int)a);
            o_pair_b.push_back(group_tree_of_link(lg));
        }
    }
    // leaf pairs allowed by sphere NAME (self_collision_model.cpp:1133-1149)
    o_allowed_a.clear(); o_allowed_b.clear();
    if (!m_acm.empty()) {
        std::set<std::string> acm_names;
        for (const auto& e : m_acm) acm_names.insert(e.first.first);
        for (size_t p = 0; p < o_pair_a.size(); ++p) {
            const SphereTree& ta = *emitted[o_pair_a[p]];
            const SphereTree& tb = *emitted[o_pair_b[p]];
            for (int i = 0; i < ta.size(); ++i) {
                if (ta.left[i] >= 0 || !acm_names.count(ta.name[i])) continue;
                for (int k = 0; k < tb.size(); ++k) {
                    if (tb.left[k] >= 0) continue;
                    if (acmAlways(ta.name[i], tb.name[k])) {
                        o_allowed_a.push_back(tree_first[o_pair_a[p]] + i);
                        o_allowed_b.push_back(tree_first[o_pair_b[p]] + k);
                    }
                }
            }
        }
    }

    // planning variables
    o_var_type.clear(); o_var_weight.clear();
    for (int jr : m_planning_joint) {
        const JointRec& j = m_joint_recs[jr];
        o_var_type.push_back(j.kind == J_CONTINUOUS ? SMPLGPU_VAR_CONTINUOUS
                             : (j.kind == J_PRISMATIC ? SMPLGPU_VAR_PRISMATIC : SMPLGPU_VAR_REVOLUTE));
        o_var_weight.push_back(m_mr_weight[jr]);
    }
    o_var_min = m_var_min;
    o_var_max = m_var_max;

    o_seg_kind.assign(m_seg_kind.begin(), m_seg_kind.end());
    o_seg_var.assign(m_seg_var.begin(), m_seg_var.end());
    o_seg_axis = m_seg_axis;
    o_seg_origin = m_seg_origin;
    o_seg_f_tip = m_seg_f_tip;
    o_T_kin.assign(m_T_kin.begin(), m_T_kin.end());

    memset(&m_desc, 0, sizeof(m_desc));
    m_desc.dof = (int)m_planning_joint.size();
    m_desc.n_links = (int)o_link_parent.size();
    m_desc.link_parent = o_link_parent.data();
    m_desc.link_joint = o_link_joint.data();
    m_desc.link_origin = o_link_origin.data();
    m_desc.link_axis = o_link_axis.data();
    m_desc.link_var = o_link_var.data();
    m_desc.link_const = o_link_const.data();
    m_desc.link_base = o_link_base.data();
    m_desc.n_nodes = (int)o_node_link.size();
    m_desc.node_link = o_node_link.data();
    m_desc.node_center = o_node_center.data();
    m_desc.node_radius = o_node_radius.data();
    m_desc.node_left = o_node_left.data();
    m_desc.node_right = o_node_right.data();
    m_desc.n_trees = (int)o_tree_root.size();
    m_desc.n_robot_trees = n_robot_trees;
    m_desc.tree_root = o_tree_root.data();
    m_desc.n_pairs = (int)o_pair_a.size();
    m_desc.pair_a = o_pair_a.data();
    m_desc.pair_b = o_pair_b.data();
    m_desc.n_allowed_leaf_pairs = (int)o_allowed_a.size();
    m_desc.allowed_leaf_a = o_allowed_a.data();
    m_desc.allowed_leaf_b = o_allowed_b.data();
    m_desc.var_type = o_var_type.data();
    m_desc.var_motion_weight = o_var_weight.data();
    m_desc.var_min = o_var_min.data();
    m_desc.var_max = o_var_max.data();
    m_desc.n_segments = m_has_chain ? m_n_segments : 0;
    m_desc.seg_kind = o_seg_kind.data();
    m_desc.seg_axis = o_seg_axis.data();
    m_desc.seg_origin = o_seg_origin.data();
    m_desc.seg_f_tip = o_seg_f_tip.data();
    m_desc.seg_var = o_seg_var.data();
    m_desc.T_kin_to_planning = o_T_kin.data();
    for (int i = 0; i < 3; ++i) m_desc.xyz_offset[i] = m_xyz_offset[i];
}

} // namespace smplhost
