// Planning-link IK on the device: the batched counterpart of InverseKinematicsInterface::computeIK
// (ik_option::UNRESTRICTED), and the SNAP_TO_XYZ_RPY action of the lattice rounds
// (ManipLatticeActionSpace::apply / getAction / mprimActive, manip_lattice_action_space.cpp:376-449, 507-573, 662-691).
// The reference's IK solvers (pr2_arm_kinematics, KDL's ChainIkSolverPos_NR_JL) are third-party and absent, so the
// IK is the project's own, defined once and restated expression for expression here and in the oracle
// (oracle/snap/snap_lattice.cpp planningLinkIk; DESIGN.md section 2, parity unpinned):
//   f(q)  = T_kin_to_planning * segments 0 .. n_segments - 1 (planning_frame_fk's chain): rotation R, position p;
//           target point pt = R offset + p
//   e     = (target_p - pt, rotation_vector(target_R R^T)); converged when |e_i| <= tolerance for all six
//   step  = J^T (J J^T + IK_LAMBDA^2 I)^-1 e with J the geometric 6 x dof Jacobian at pt, the 6 x 6 system by
//           Cholesky; q += step, bounded variables clamped to their limits, continuous ones wrapped (normalize_angle)
// One WARP per problem: lane l forms segment l's transform (the sin/cos), lane 0 chains them, lane l forms the
// Jacobian column of segment l, lanes 0-20 the entries of J J^T, lane 0 the Cholesky solve, lane v the update of
// variable v.  Every number comes from the oracle's expression in the oracle's order (the build uses --fmad=false), so
// only CUDA's sin / cos / atan2 differ from glibc's (<= 2 ulp).
#pragma once

#include "heuristic.cuh"
#include "lattice.cuh"
#include "model.cuh"
#include "validity.cuh"

namespace smplgpu {

// damping of the least-squares step (metres / radians); chosen on the oracle: 99.4 % of PR2 targets (FK poses of valid
// states, seeded 0.1 rad per joint away) converge to 1e-6 in 3.4 steps on average, the rest stop at a joint limit
constexpr double IK_LAMBDA = 1e-3;
constexpr int IK_WARPS = 4;   // problems (warps) per block

// a goal pose as the IK reads it: position and KDL Rotation::RPY of roll pitch yaw (row-major), computed on the host
struct IkTarget { double p[3]; double R[9]; };

// shared memory of one warp
struct IkScratch
{
    KFrame seg[MAX_SEGMENTS];        // segment s at the current q
    KFrame pre[MAX_SEGMENTS + 1];    // product of segments 0 .. s-1
    double J[6][MAX_DOF];
    double A[21];                    // lower triangle of J J^T + lambda^2 I, row by row
    double x[6];
    double q[MAX_DOF];
    double tp[3];                    // lattice_snap_kernel's SNAP_TO_RPY target position
};

// The rotation vector (axis * angle, angle in [0, pi]) of the rotation matrix E.  v = (E21 - E12, E02 - E20,
// E10 - E01) = 2 sin(angle) axis and cos(angle) = (trace - 1) / 2 give angle = atan2(|v| / 2, cos); then
//   near 0 (|v| / 2 < 1e-9):  the rotation vector is v / 2 (angle / (2 sin angle) = 1/2 + O(angle^2));
//   near pi (cos < -0.99):     v is too short to carry the axis, which comes from the symmetric part instead,
//                              (E + E^T) / 2 = cos I + (1 - cos) a a^T, largest diagonal first, its sign from v;
//   otherwise:                 v * angle / (2 sin angle).
__device__ __forceinline__ void rotation_vector(const double* E, double* w)
{
    const double v0 = E[7] - E[5], v1 = E[2] - E[6], v2 = E[3] - E[1];
    const double c = (((E[0] + E[4]) + E[8]) - 1.0) * 0.5;
    const double s = 0.5 * sqrt((v0 * v0 + v1 * v1) + v2 * v2);
    const double angle = atan2(s, c);
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
        a[k] = sqrt(0.0 < t ? t : 0.0);
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

// The IK of one problem by one warp, seeded at S.q (set and __syncwarp'ed by the caller); the answer is left in S.q.
// ROWS = 6: the full pose (tp, tR).  ROWS = 3: the position alone (SNAP_TO_XYZ; oracle/snap_kinds/snap_kinds_lattice.cpp
// planningLinkIkPosition): e = tp - pt, the 3 x dof position block of J, a 3 x 3 Cholesky, converged when the three
// position rows are within the tolerance; tR is not read and the orientation is free.
// Returns converged (warp-uniform); *iterations = steps taken.
template <int ROWS>
__device__ bool ik_warp(const DevModel* __restrict__ M, const double* tp, const double* tR, int max_iterations,
                        double tolerance, IkScratch& S, int lane, int* iterations)
{
    static_assert(ROWS == 6 || ROWS == 3, "full pose or position only");
    constexpr int NA = ROWS * (ROWS + 1) / 2;   // entries of the lower triangle of J J^T
    const int dof = M->dof, nseg = M->n_segments;
    for (int k = lane; k < 6 * MAX_DOF; k += 32) {
        (&S.J[0][0])[k] = 0.0;   // variables beyond the chain keep zero columns
    }
    KFrame Tk;
    kframe_from12(M->T_kin_to_planning, Tk);
    for (int it = 0;; ++it) {
        // chain
        if (lane < nseg) {
            segment_pose(M, lane, S.q, S.seg[lane]);
        }
        __syncwarp();
        if (lane == 0) {
            KFrame f1, nf;
#pragma unroll
            for (int i = 0; i < 9; ++i) f1.M[i] = (i % 4 == 0) ? 1.0 : 0.0;
            f1.p[0] = f1.p[1] = f1.p[2] = 0.0;
            for (int s = 0; s < nseg; ++s) {
                S.pre[s] = f1;
                kframe_mul(f1, S.seg[s], nf);
                f1 = nf;
            }
            S.pre[nseg] = f1;
        }
        __syncwarp();
        // error (every lane, the same values)
        KFrame f;
        kframe_mul(Tk, S.pre[nseg], f);
        double pt[3], e[6];
        for (int i = 0; i < 3; ++i) {
            pt[i] = (f.M[3 * i] * M->xyz_offset[0] + f.M[3 * i + 1] * M->xyz_offset[1] + f.M[3 * i + 2] * M->xyz_offset[2]) + f.p[i];
            e[i] = tp[i] - pt[i];
        }
        if (ROWS == 6) {
            double E[9];
            for (int i = 0; i < 3; ++i) {
                for (int j = 0; j < 3; ++j) {
                    E[3 * i + j] = (tR[3 * i] * f.M[3 * j] + tR[3 * i + 1] * f.M[3 * j + 1]) + tR[3 * i + 2] * f.M[3 * j + 2];
                }
            }
            rotation_vector(E, e + 3);
        }
        bool conv = true;
        for (int i = 0; i < ROWS; ++i) {
            conv = conv && fabs(e[i]) <= tolerance;
        }
        if (conv || it == max_iterations) {
            *iterations = it;
            return conv;
        }
        // Jacobian column of segment `lane`: its joint axis and origin in the planning frame
        if (lane < nseg) {
            const int v = M->seg_var[lane], kind = M->seg_kind[lane];
            if (v >= 0 && kind != 0) {
                KFrame W;
                kframe_mul(Tk, S.pre[lane], W);
                const double* ax = M->seg_axis[lane];
                const double* og = M->seg_origin[lane];
                double a[3], o[3];
                for (int i = 0; i < 3; ++i) {
                    a[i] = (W.M[3 * i] * ax[0] + W.M[3 * i + 1] * ax[1]) + W.M[3 * i + 2] * ax[2];
                    o[i] = ((W.M[3 * i] * og[0] + W.M[3 * i + 1] * og[1]) + W.M[3 * i + 2] * og[2]) + W.p[i];
                }
                if (kind == 1) {
                    const double d0 = pt[0] - o[0], d1 = pt[1] - o[1], d2 = pt[2] - o[2];
                    S.J[0][v] = a[1] * d2 - a[2] * d1;
                    S.J[1][v] = a[2] * d0 - a[0] * d2;
                    S.J[2][v] = a[0] * d1 - a[1] * d0;
                    S.J[3][v] = a[0]; S.J[4][v] = a[1]; S.J[5][v] = a[2];
                } else {
                    S.J[0][v] = a[0]; S.J[1][v] = a[1]; S.J[2][v] = a[2];
                    S.J[3][v] = 0.0; S.J[4][v] = 0.0; S.J[5][v] = 0.0;
                }
            }
        }
        __syncwarp();
        // J J^T + lambda^2 I: entry (r, c), c <= r, by lane r (r + 1) / 2 + c
        if (lane < NA) {
            int r = 0;
            while ((r + 1) * (r + 2) / 2 <= lane) ++r;
            const int c = lane - r * (r + 1) / 2;
            double acc = 0.0;
            for (int v = 0; v < dof; ++v) {
                acc = acc + S.J[r][v] * S.J[c][v];
            }
            S.A[lane] = r == c ? acc + IK_LAMBDA * IK_LAMBDA : acc;
        }
        __syncwarp();
        // Cholesky and the two triangular solves
        if (lane == 0) {
            double L[ROWS][ROWS], y[ROWS];
            for (int j = 0; j < ROWS; ++j) {
                double d = S.A[j * (j + 1) / 2 + j];
                for (int k = 0; k < j; ++k) {
                    d = d - L[j][k] * L[j][k];
                }
                L[j][j] = sqrt(d);
                for (int i = j + 1; i < ROWS; ++i) {
                    double t = S.A[i * (i + 1) / 2 + j];
                    for (int k = 0; k < j; ++k) {
                        t = t - L[i][k] * L[j][k];
                    }
                    L[i][j] = t / L[j][j];
                }
            }
            for (int i = 0; i < ROWS; ++i) {
                double t = e[i];
                for (int k = 0; k < i; ++k) {
                    t = t - L[i][k] * y[k];
                }
                y[i] = t / L[i][i];
            }
            for (int i = ROWS - 1; i >= 0; --i) {
                double t = y[i];
                for (int k = i + 1; k < ROWS; ++k) {
                    t = t - L[k][i] * S.x[k];
                }
                S.x[i] = t / L[i][i];
            }
        }
        __syncwarp();
        // the step, variable `lane`
        if (lane < dof) {
            double dq = 0.0;
            for (int r = 0; r < ROWS; ++r) {
                dq = dq + S.J[r][lane] * S.x[r];
            }
            double nq = S.q[lane] + dq;
            if (M->var_type[lane] == 1) {
                nq = normalize_angle(nq);
            } else {
                nq = nq < M->var_min[lane] ? M->var_min[lane] : (nq > M->var_max[lane] ? M->var_max[lane] : nq);
            }
            S.q[lane] = nq;
        }
        __syncwarp();
    }
}

// smplgpu_planning_link_ik (ROWS = 6) and smplgpu_planning_link_ik_position (ROWS = 3): problem k = warp k
template <int ROWS>
__global__ void __launch_bounds__(32 * IK_WARPS)
planning_link_ik_kernel(const DevModel* __restrict__ M, const IkTarget* __restrict__ targets,
                        const double* __restrict__ seeds, int n, int max_iterations, double tolerance,
                        double* __restrict__ q_out, uint8_t* __restrict__ ok, int* __restrict__ iterations)
{
    __shared__ IkScratch sS[IK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = (int)blockIdx.x * IK_WARPS + warp;
    if (k >= n) {
        return;
    }
    IkScratch& S = sS[warp];
    const int dof = M->dof;
    if (lane < dof) {
        S.q[lane] = seeds[(size_t)k * dof + lane];
    }
    __syncwarp();
    int it = 0;
    const bool conv = ik_warp<ROWS>(M, targets[k].p, targets[k].R, max_iterations, tolerance, S, lane, &it);
    if (lane < dof) {
        q_out[(size_t)k * dof + lane] = S.q[lane];
    }
    if (lane == 0) {
        ok[k] = conv ? 1 : 0;
        iterations[k] = it;
    }
}

// The snap's target in a goal set: the record whose goal position is nearest to p (squared Euclidean distance, the
// lower index on a tie).  The oracle (oracle/goal_sets/goal_set_lattice.cpp nearestRecord) uses the same expression.
__device__ __forceinline__ int nearest_goal_record(const LatticeGoal* __restrict__ set, int n, const double* p)
{
    int best = 0;
    double best_d = 0.0;
    for (int r = 0; r < n; ++r) {
        const double dx = set[r].pos[0] - p[0], dy = set[r].pos[1] - p[1], dz = set[r].pos[2] - p[2];
        const double d = (dx * dx + dy * dy) + dz * dz;
        if (r == 0 || d < best_d) {
            best = r;
            best_d = d;
        }
    }
    return best;
}

// Round, step 1b with snaps enabled (between lattice_gen_kernel and the edge kernels): a warp per (expansion, enabled
// snap kind); kind index k fills successor word k (B.snap_kind[k]: SMPLGPU_SNAP_RPY, _XYZ, _XYZ_RPY in that order).  A
// kind is active when the parent's metric goal distance (the quantity of the short-distance switch) is within its
// threshold.  Every kind of an expansion aims at the same record: the one of the slot's goal set nearest to the
// parent's target-offset position (nearest_goal_record).  Its action, seeded at the parent:
//   SNAP_TO_XYZ_RPY  (XYZ, XYZ_RPY, JOINT_STATE records) an IK solution for the record's full pose, or a joint
//                    record's angles
//   SNAP_TO_XYZ      (XYZ, XYZ_RPY records) a position-only IK solution for the record's goal position
//   SNAP_TO_RPY      (XYZ_RPY records) an IK solution for the parent's own target-offset position and the record's
//                    rotation: the orientation turned in place
// A kind that does not apply to the record's type produces nothing.  The action becomes the word's edge when it exists
// and is within the joint limits.  lattice_gen_kernel left the snap words inactive zero-length edges.
// counters[2 kind] / [2 kind + 1]: IK solves of that kind run / converged.
// With both IK forms inlined the kernel spills under ptxas's default cap of 128 registers; a minimum of one block per
// SM lifts the cap (152 registers, no spills; DESIGN.md section 4).
__global__ void __launch_bounds__(32 * IK_WARPS, 1)
lattice_snap_kernel(const DevModel* __restrict__ M, LatticeBank B, const int* __restrict__ slot,
                    const int* __restrict__ parent, int n, double* __restrict__ q1, uint8_t* __restrict__ active,
                    unsigned long long* counters)
{
    __shared__ IkScratch sS[IK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = (int)blockIdx.x * IK_WARPS + warp;
    const int i = w / B.snap, word = w - i * B.snap;
    if (i >= n) {
        return;
    }
    const int kind = B.snap_kind[word];
    const int s = slot[i], p = parent[i];
    const double goal_dist = (double)B.gdist[(size_t)s * B.cap + p] * B.res;
    if (!(goal_dist <= B.snap_thresh[kind])) {
        return;
    }
    IkScratch& S = sS[warp];
    const int dof = M->dof;
    const double* a = B.q + ((size_t)s * B.cap + p) * dof;
    const LatticeGoal* set = B.goal + (size_t)s * SMPLGPU_MAX_GOAL_SET;
    const int n_goals = B.n_goals[s];
    int target = 0;
    if (n_goals > 1 || kind == SMPLGPU_SNAP_RPY) {
        double pose[6];
        planning_frame_fk(M, a, pose);   // the same in every lane
        if (n_goals > 1) {
            target = nearest_goal_record(set, n_goals, pose);
        }
        if (lane < 3) {
            S.tp[lane] = pose[lane];
        }
    }
    const LatticeGoal* g = set + target;
    if ((kind == SMPLGPU_SNAP_XYZ && g->type == SMPLGPU_GOAL_JOINT_STATE) ||
        (kind == SMPLGPU_SNAP_RPY && g->type != SMPLGPU_GOAL_XYZ_RPY)) {
        return;
    }
    bool found = true;
    if (g->type == SMPLGPU_GOAL_JOINT_STATE) {
        if (lane < dof) {
            S.q[lane] = g->angles[lane];
        }
        __syncwarp();
    } else {
        if (lane < dof) {
            S.q[lane] = a[lane];
        }
        __syncwarp();
        int it = 0;
        if (kind == SMPLGPU_SNAP_XYZ) {
            found = ik_warp<3>(M, g->xyz, g->R, B.ik_max_iterations, B.ik_tolerance, S, lane, &it);
        } else {
            found = ik_warp<6>(M, kind == SMPLGPU_SNAP_RPY ? S.tp : g->xyz, g->R, B.ik_max_iterations, B.ik_tolerance,
                               S, lane, &it);
        }
        if (lane == 0) {
            atomicAdd(&counters[2 * kind], 1ull);
            if (found) {
                atomicAdd(&counters[2 * kind + 1], 1ull);
            }
        }
    }
    // checkAction: joint limits first (the edge kernels that follow check the motion)
    const bool on = found && joint_limits_ok(M, S.q);
    const size_t t = (size_t)i * B.stride + word;
    if (on && lane < dof) {
        q1[t * dof + lane] = S.q[lane];
    }
    if (lane == 0) {
        active[t] = on ? 1 : 0;
    }
}

} // namespace smplgpu
