// Euclidean-space motions of the path shortcut (ShortcutPath's EUCLID_SPACE type, post_processing.cpp:284-365): a
// straight, constant-orientation-rate motion of the planning link between two joint states of a path, followed
// through the planning-link IK of ik.cuh.  The fork's EuclidShortcutPathGenerator rests on a third-party IK, so the
// definition is the project's own (DESIGN.md section 2, parity unpinned), written once in the oracle
// (oracle/euclid_shortcut/euclid_shortcut.cpp euclidMotion) and restated here expression for expression:
//   ends    f(qa) = (pa, Ra), f(qb) = (pb, Rb): ik_warp's forward map (T_kin_to_planning * the planning chain, the
//           target point R offset + p)
//   turn    w = rotation_vector(Rb Ra^T), theta = sqrt((w0^2 + w1^2) + w2^2); d = sqrt((dx^2 + dy^2) + dz^2) of pb - pa
//   steps   n = max(1, ceil(max(d / max_step_m, theta / max_step_rad))); refused when n > max_steps
//   states  qa, q1 .. q(n-1), qb: q_k the IK solution (ik_warp<6>, seeded at q(k-1)) for the position
//           pa + (k / n)(pb - pa) and the rotation Rot2(w / theta, (k / n) theta) Ra (Ra when theta = 0); the first
//           solve that does not converge or leaves the joint limits refuses the motion
//   valid   every consecutive pair passes isStateToStateValid (launch_edges: the verdicts of smplgpu_is_edges_valid)
//   cost    the JointDistance (post_processing.cpp:48-67) of the consecutive pairs, summed in order
#pragma once

#include "ik.cuh"

namespace smplgpu {

// smplgpu_euclid_params as the kernels read it
struct EuclidParams
{
    double max_step_m, max_step_rad;
    int max_steps, ik_max_iterations;
    double ik_tolerance;
};

// a motion's two end poses and its step count
struct EuclidEnds
{
    double pa[3], pb[3], Ra[9], u[3];   // u = w / theta, the turn's axis
    double theta;
    int n;                              // max_steps + 1 when the motion takes more than max_steps steps
};

// ik_warp's forward map in one thread: the same products in the same order as its chain
__device__ __forceinline__ void euclid_pose(const DevModel* __restrict__ M, const double* __restrict__ q, double* p,
                                            double* R)
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
    for (int i = 0; i < 3; ++i) {
        p[i] = (f.M[3 * i] * M->xyz_offset[0] + f.M[3 * i + 1] * M->xyz_offset[1] + f.M[3 * i + 2] * M->xyz_offset[2]) + f.p[i];
    }
    for (int i = 0; i < 9; ++i) R[i] = f.M[i];
}

__device__ __forceinline__ void euclid_ends(const DevModel* __restrict__ M, const double* __restrict__ qa,
                                            const double* __restrict__ qb, const EuclidParams& P, EuclidEnds& E)
{
    double Rb[9], Em[9], w[3];
    euclid_pose(M, qa, E.pa, E.Ra);
    euclid_pose(M, qb, E.pb, Rb);
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) {
            Em[3 * i + j] = (Rb[3 * i] * E.Ra[3 * j] + Rb[3 * i + 1] * E.Ra[3 * j + 1]) + Rb[3 * i + 2] * E.Ra[3 * j + 2];
        }
    }
    rotation_vector(Em, w);
    E.theta = sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
    for (int i = 0; i < 3; ++i) E.u[i] = E.theta > 0.0 ? w[i] / E.theta : 0.0;
    const double dx = E.pb[0] - E.pa[0], dy = E.pb[1] - E.pa[1], dz = E.pb[2] - E.pa[2];
    const double d = sqrt((dx * dx + dy * dy) + dz * dz);
    const double s = fmax(d / P.max_step_m, E.theta / P.max_step_rad);
    // s <= max_steps  <=>  ceil(s) <= max_steps; a NaN is refused too
    E.n = s <= (double)P.max_steps ? max(1, (int)ceil(s)) : P.max_steps + 1;
}

// JointDistance (post_processing.cpp:48-67): continuous variables by their wrapped difference
__device__ __forceinline__ double joint_distance(const DevModel* __restrict__ M, const double* a, const double* b)
{
    double d = 0.0;
    for (int v = 0; v < M->dof; ++v) {
        const double delta = b[v] - a[v];
        d += M->var_type[v] == 1 ? fabs(normalize_angle(delta)) : fabs(delta);
    }
    return d;
}

// The step count of motion e: a thread per motion (the host sizes the edge chunks from it)
__global__ void euclid_steps_kernel(const DevModel* __restrict__ M, const double* __restrict__ points,
                                    const int* __restrict__ idx_a, const int* __restrict__ idx_b, int n, EuclidParams P,
                                    int* __restrict__ n_steps)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) {
        return;
    }
    const int dof = M->dof;
    EuclidEnds E;
    euclid_ends(M, points + (size_t)idx_a[e] * dof, points + (size_t)idx_b[e] * dof, P, E);
    n_steps[e] = E.n;
}

// per warp, beside its IkScratch
struct EuclidScratch
{
    EuclidEnds ends;
    double tR[9];
    double prev[MAX_DOF];   // the state before the one being solved
};

// The IK chain of motions first .. first + count - 1, a warp each.  A motion of n <= max_steps steps owns the edge
// slots edge_off[e] .. edge_off[e] + n - 1 of q0 / q1 (offsets within the chunk): edge k is state k -> state k + 1.
// A chain that fails fills its slots with the zero-length edge qa -> qa.  chain_ok[e] = the chain completed;
// cost[e] = its JointDistance sum (0 when it did not complete).  counters[0] / [1]: IK solves run / converged.
__global__ void __launch_bounds__(32 * IK_WARPS, 1)
euclid_chain_kernel(const DevModel* __restrict__ M, const double* __restrict__ points, const int* __restrict__ idx_a,
                    const int* __restrict__ idx_b, int first, int count, EuclidParams P,
                    const int* __restrict__ edge_off, double* __restrict__ q0, double* __restrict__ q1,
                    uint8_t* __restrict__ chain_ok, double* __restrict__ cost, unsigned long long* counters)
{
    __shared__ IkScratch sS[IK_WARPS];
    __shared__ EuclidScratch sE[IK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w = (int)blockIdx.x * IK_WARPS + warp;
    if (w >= count) {
        return;
    }
    const int e = first + w;
    IkScratch& S = sS[warp];
    EuclidScratch& X = sE[warp];
    const int dof = M->dof;
    const double* qa = points + (size_t)idx_a[e] * dof;
    const double* qb = points + (size_t)idx_b[e] * dof;
    if (lane == 0) {
        euclid_ends(M, qa, qb, P, X.ends);
    }
    if (lane < dof) {
        S.q[lane] = qa[lane];
        X.prev[lane] = qa[lane];
    }
    __syncwarp();
    const int n = X.ends.n;
    if (n > P.max_steps) {
        if (lane == 0) {
            chain_ok[e] = 0;
            cost[e] = 0.0;
        }
        return;
    }
    const size_t base = (size_t)edge_off[e];
    double c = 0.0;   // lane 0's running sum
    bool good = true;
    int k = 1;
    for (; k < n; ++k) {
        const double alpha = (double)k / (double)n;
        double tp[3];
        for (int i = 0; i < 3; ++i) {
            tp[i] = X.ends.pa[i] + alpha * (X.ends.pb[i] - X.ends.pa[i]);
        }
        if (lane == 0) {
            if (X.ends.theta > 0.0) {
                double Rk[9];
                rot2(X.ends.u, alpha * X.ends.theta, Rk);
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 3; ++j) {
                        X.tR[3 * i + j] = (Rk[3 * i] * X.ends.Ra[j] + Rk[3 * i + 1] * X.ends.Ra[3 + j]) + Rk[3 * i + 2] * X.ends.Ra[6 + j];
                    }
                }
            } else {
                for (int i = 0; i < 9; ++i) X.tR[i] = X.ends.Ra[i];
            }
        }
        __syncwarp();
        int it = 0;
        const bool conv = ik_warp<6>(M, tp, X.tR, P.ik_max_iterations, P.ik_tolerance, S, lane, &it);
        const bool on = conv && joint_limits_ok(M, S.q);
        if (lane == 0) {
            atomicAdd(&counters[0], 1ull);
            if (conv) {
                atomicAdd(&counters[1], 1ull);
            }
        }
        if (!on) {
            good = false;
            break;
        }
        if (lane < dof) {
            q0[(base + k - 1) * dof + lane] = X.prev[lane];
            q1[(base + k - 1) * dof + lane] = S.q[lane];
        }
        if (lane == 0) {
            c = c + joint_distance(M, X.prev, S.q);
        }
        __syncwarp();
        if (lane < dof) {
            X.prev[lane] = S.q[lane];
        }
        __syncwarp();
    }
    if (good) {
        if (lane < dof) {
            q0[(base + n - 1) * dof + lane] = X.prev[lane];
            q1[(base + n - 1) * dof + lane] = qb[lane];
        }
        if (lane == 0) {
            c = c + joint_distance(M, X.prev, qb);
        }
    } else {
        for (int j = k - 1; j < n; ++j) {
            if (lane < dof) {
                q0[(base + j) * dof + lane] = qa[lane];
                q1[(base + j) * dof + lane] = qa[lane];
            }
        }
    }
    if (lane == 0) {
        chain_ok[e] = good ? 1 : 0;
        cost[e] = good ? c : 0.0;
    }
}

// ok[e] = the chain of motion e completed and every one of its edges is valid: a thread per motion
__global__ void euclid_reduce_kernel(int first, int count, int max_steps, const int* __restrict__ n_steps,
                                     const int* __restrict__ edge_off, const uint8_t* __restrict__ chain_ok,
                                     const uint8_t* __restrict__ verdict, uint8_t* __restrict__ ok)
{
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= count) {
        return;
    }
    const int e = first + w;
    const int n = n_steps[e];
    bool good = n <= max_steps && chain_ok[e] != 0;
    for (int j = 0; j < n && good; ++j) {
        good = verdict[edge_off[e] + j] != 0;
    }
    ok[e] = good ? 1 : 0;
}

} // namespace smplgpu
