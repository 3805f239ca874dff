// Batched BfsHeuristic::GetGoalHeuristic: planning-link forward kinematics
// (KDL chain semantics), target offset, worldToGrid and BFS grid gather.
//
// Reference (file:line under dyouakim/smpl):
//   sbpl_kdl_robot_model/src/kdl_robot_model.cpp:191-198, 400-423   normalizeAngles, computePlanningLinkFK
//   smpl/src/graph/manip_lattice.cpp:1358-1373, 2297-2312          computePlanningFrameFK, getTargetOffsetPose
//   smpl/src/heuristic/bfs_heuristic.cpp:148-163, 355-366          GetGoalHeuristic, getBfsCostToGoal
// The chain arithmetic is orocos_kdl's (third-party, un-vendored): Frame*Frame =
// (M1*M2, M1*p2 + p1) with left-to-right sums, Rotation::Rot2, Rotation::GetRPY.
#pragma once

#include "model.cuh"
#include "validity.cuh"

namespace smplgpu {

struct KFrame { double M[9]; double p[3]; };

__device__ __forceinline__ void kframe_mul(const KFrame& a, const KFrame& b, KFrame& r)
{
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            r.M[3 * i + j] = a.M[3 * i] * b.M[j] + a.M[3 * i + 1] * b.M[3 + j] + a.M[3 * i + 2] * b.M[6 + j];
        }
        r.p[i] = (a.M[3 * i] * b.p[0] + a.M[3 * i + 1] * b.p[1] + a.M[3 * i + 2] * b.p[2]) + a.p[i];
    }
}

__device__ __forceinline__ void kframe_from12(const double* t, KFrame& f)
{
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        f.M[3 * r] = t[4 * r];
        f.M[3 * r + 1] = t[4 * r + 1];
        f.M[3 * r + 2] = t[4 * r + 2];
        f.p[r] = t[4 * r + 3];
    }
}

// KDL Rotation::Rot2
__device__ __forceinline__ void rot2(const double* v, double angle, double* M)
{
    double st, ct;
    sincos(angle, &st, &ct);
    const double vt = 1 - ct;
    const double m_vt_0 = vt * v[0], m_vt_1 = vt * v[1], m_vt_2 = vt * v[2];
    const double m_st_0 = v[0] * st, m_st_1 = v[1] * st, m_st_2 = v[2] * st;
    const double m_vt_0_1 = m_vt_0 * v[1], m_vt_0_2 = m_vt_0 * v[2], m_vt_1_2 = m_vt_1 * v[2];
    M[0] = ct + m_vt_0 * v[0];  M[1] = -m_st_2 + m_vt_0_1;  M[2] = m_st_1 + m_vt_0_2;
    M[3] = m_st_2 + m_vt_0_1;   M[4] = ct + m_vt_1 * v[1];  M[5] = -m_st_0 + m_vt_1_2;
    M[6] = -m_st_1 + m_vt_0_2;  M[7] = m_st_0 + m_vt_1_2;   M[8] = ct + m_vt_2 * v[2];
}

// Segment::pose(q) = joint.pose(q) * f_tip of chain segment s: one factor of the planning-link chain (also the
// per-lane part of the IK's chain, ik.cuh)
__device__ __forceinline__ void segment_pose(const DevModel* __restrict__ M, int s, const double* __restrict__ q, KFrame& seg)
{
    const int v = M->seg_var[s];
    double qq = 0.0;
    if (v >= 0) {
        qq = q[v];
        if (M->var_type[v] == 1) {
            qq = normalize_angle(qq); // KDLRobotModel::normalizeAngles (continuous joints only)
        }
    }
    KFrame jp;
    const int kind = M->seg_kind[s];
    if (kind == 1) {
        rot2(M->seg_axis[s], qq, jp.M);
        jp.p[0] = M->seg_origin[s][0]; jp.p[1] = M->seg_origin[s][1]; jp.p[2] = M->seg_origin[s][2];
    } else {
#pragma unroll
        for (int i = 0; i < 9; ++i) jp.M[i] = (i % 4 == 0) ? 1.0 : 0.0;
        if (kind == 2) {
            jp.p[0] = M->seg_origin[s][0] + M->seg_axis[s][0] * qq;
            jp.p[1] = M->seg_origin[s][1] + M->seg_axis[s][1] * qq;
            jp.p[2] = M->seg_origin[s][2] + M->seg_axis[s][2] * qq;
        } else {
            jp.p[0] = jp.p[1] = jp.p[2] = 0.0;
        }
    }
    KFrame tip;
    kframe_from12(M->seg_f_tip[s], tip);
    kframe_mul(jp, tip, seg);
}

// computePlanningLinkFK + getTargetOffsetPose: pose6 = x y z roll pitch yaw of the target-offset
// frame; link_xyz (optional) = position of the planning link itself (before the offset)
__device__ void planning_frame_fk(const DevModel* __restrict__ M, const double* __restrict__ q, double* pose,
                                  double* link_xyz = nullptr)
{
    KFrame f1;
#pragma unroll
    for (int i = 0; i < 9; ++i) f1.M[i] = (i % 4 == 0) ? 1.0 : 0.0;
    f1.p[0] = f1.p[1] = f1.p[2] = 0.0;

    for (int s = 0; s < M->n_segments; ++s) {
        KFrame seg, nf;
        segment_pose(M, s, q, seg);
        kframe_mul(f1, seg, nf);
        f1 = nf;
    }
    KFrame Tk, f;
    kframe_from12(M->T_kin_to_planning, Tk);
    kframe_mul(Tk, f1, f);
    if (link_xyz != nullptr) {
        link_xyz[0] = f.p[0]; link_xyz[1] = f.p[1]; link_xyz[2] = f.p[2];
    }

    // KDL Rotation::GetRPY
    double roll, pitch, yaw;
    const double PI = 3.14159265358979323846;
    pitch = atan2(-f.M[6], sqrt(f.M[0] * f.M[0] + f.M[3] * f.M[3]));
    if (fabs(pitch) > (PI / 2.0 - 1E-12)) {
        yaw = atan2(-f.M[1], f.M[4]);
        roll = 0.0;
    } else {
        roll = atan2(f.M[7], f.M[8]);
        yaw = atan2(f.M[3], f.M[0]);
    }

    // getTargetOffsetPose: Translation(p) * Rz(yaw) * Ry(pitch) * Rx(roll) * Translation(offset)
    Xf T, A, R;
#pragma unroll
    for (int i = 0; i < 12; ++i) T.m[i] = 0.0;
    T.m[0] = 1.0; T.m[5] = 1.0; T.m[10] = 1.0;
    T.m[3] = f.p[0]; T.m[7] = f.p[1]; T.m[11] = f.p[2];
    angle_axis(yaw, 0.0, 0.0, 1.0, A);
    xf_mul(T, A, R); T = R;
    angle_axis(pitch, 0.0, 1.0, 0.0, A);
    xf_mul(T, A, R); T = R;
    angle_axis(roll, 1.0, 0.0, 0.0, A);
    xf_mul(T, A, R); T = R;
#pragma unroll
    for (int i = 0; i < 12; ++i) A.m[i] = 0.0;
    A.m[0] = 1.0; A.m[5] = 1.0; A.m[10] = 1.0;
    A.m[3] = M->xyz_offset[0]; A.m[7] = M->xyz_offset[1]; A.m[11] = M->xyz_offset[2];
    xf_mul(T, A, R);
    pose[0] = R.m[3]; pose[1] = R.m[7]; pose[2] = R.m[11];
    pose[3] = roll; pose[4] = pitch; pose[5] = yaw;
}

__global__ void planning_fk_kernel(const DevModel* __restrict__ M, const double* __restrict__ q, int n,
                                   double* __restrict__ pose6)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) {
        return;
    }
    double pose[6];
    planning_frame_fk(M, q + (size_t)i * M->dof, pose);
#pragma unroll
    for (int k = 0; k < 6; ++k) pose6[(size_t)i * 6 + k] = pose[k];
}

// GetGoalHeuristic: h = Infinity when out of bounds or WALL, else cost_per_cell * distance
// (unreachable cells hold -1: the reference returns cost_per_cell * -1; preserved)
__global__ void goal_heuristic_kernel(const DevModel* __restrict__ M, GridParams G,
                                      const int* __restrict__ bfs, int dimx, int dimy, int dimz,
                                      const double* __restrict__ q, int n, int cost_per_cell, int* __restrict__ h)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) {
        return;
    }
    double pose[6];
    planning_frame_fk(M, q + (size_t)i * M->dof, pose);
    const int gx = __double2int_rz(G.inv_res * (pose[0] - G.ox) + 0.5) - 1;
    const int gy = __double2int_rz(G.inv_res * (pose[1] - G.oy) + 0.5) - 1;
    const int gz = __double2int_rz(G.inv_res * (pose[2] - G.oz) + 0.5) - 1;
    int out;
    if (gx < 0 || gy < 0 || gz < 0 || gx >= dimx - 2 || gy >= dimy - 2 || gz >= dimz - 2) {
        out = 32767;
    } else {
        const int d = bfs[((size_t)(gz + 1) * dimy + (gy + 1)) * dimx + (gx + 1)];
        out = (d == 0x7FFFFFFF) ? 32767 : cost_per_cell * d;
    }
    h[i] = out;
}

// BFS cell value at a world point in bank slot `slot` (slots stacked along z, each with its own
// padded shell); returns 0x7FFFFFFF (WALL) when the point is outside the grid
__device__ __forceinline__ int bank_lookup(const int* __restrict__ bfs, int dimx, int dimy, int slot_dimz, int slot,
                                           const GridParams& G, double x, double y, double z, bool& in_bounds)
{
    const int gx = __double2int_rz(G.inv_res * (x - G.ox) + 0.5) - 1;
    const int gy = __double2int_rz(G.inv_res * (y - G.oy) + 0.5) - 1;
    const int gz = __double2int_rz(G.inv_res * (z - G.oz) + 0.5) - 1;
    in_bounds = !(gx < 0 || gy < 0 || gz < 0 || gx >= dimx - 2 || gy >= dimy - 2 || gz >= slot_dimz - 2);
    if (!in_bounds) {
        return 0x7FFFFFFF;
    }
    return bfs[((size_t)(slot * slot_dimz + gz + 1) * dimy + (gy + 1)) * dimx + (gx + 1)];
}

// per successor: heuristic, metric goal distance (in cells) and target-offset position
__global__ void expand_info_kernel(const DevModel* __restrict__ M, GridParams G, const int* __restrict__ bfs,
                                   int dimx, int dimy, int slot_dimz, const double* __restrict__ q,
                                   const int* __restrict__ slot, int n, int cost_per_cell,
                                   int* __restrict__ h, int* __restrict__ gdist, double* __restrict__ off_xyz)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) {
        return;
    }
    double pose[6], link[3];
    planning_frame_fk(M, q + (size_t)i * M->dof, pose, link);
    const int s = slot[i];
    bool inb;
    const int d_off = bank_lookup(bfs, dimx, dimy, slot_dimz, s, G, pose[0], pose[1], pose[2], inb);
    h[i] = (!inb || d_off == 0x7FFFFFFF) ? 32767 : cost_per_cell * d_off;
    gdist[i] = bank_lookup(bfs, dimx, dimy, slot_dimz, s, G, link[0], link[1], link[2], inb);
    off_xyz[3 * i] = pose[0];
    off_xyz[3 * i + 1] = pose[1];
    off_xyz[3 * i + 2] = pose[2];
}

__global__ void bank_gather_kernel(const int* __restrict__ bfs, int nx, int ny, int nz, const int* __restrict__ slot,
                                   const int* __restrict__ cells, int n, int* __restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) {
        return;
    }
    const int x = cells[3 * i], y = cells[3 * i + 1], z = cells[3 * i + 2];
    if (x < 0 || y < 0 || z < 0 || x >= nx || y >= ny || z >= nz) {
        out[i] = -2;
        return;
    }
    out[i] = bfs[((size_t)(slot[i] * (nz + 2) + z + 1) * (ny + 2) + (y + 1)) * (nx + 2) + (x + 1)];
}

} // namespace smplgpu
