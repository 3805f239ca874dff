// Path post-processing over the CUDA validity path (SURVEY.md section 8f row 4): the reference shortcuts and
// interpolates ONE path with one CollisionChecker call per candidate motion (smpl/src/post_processing.cpp);
// here every candidate motion of MANY paths goes to the device in one batch and the (sequential, cheap)
// decision logic of the reference then runs on the host over the verdict table.
//
//   ShortcutPath(rm, cc, pin, pout, type)    post_processing.cpp:284-365
//     JOINT_SPACE / JOINT_POSITION_VELOCITY_SPACE: ShortcutPaths; EUCLID_SPACE: ShortcutPathsEuclid, over the
//     project's own straight planning-link motion and planning-link IK (DESIGN.md section 2, parity unpinned)
//   shortcut::ShortcutPath / DivideAndConquerShortcutPath   smpl/include/smpl/geometry/detail/shortcut.hpp:112-438
//   InterpolatePath(cc, path)                post_processing.cpp:476-540
#ifndef SMPLHOST_POST_PROCESSING_H
#define SMPLHOST_POST_PROCESSING_H

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/smplgpu.h"

namespace smplhost {

/// post_processing.h ShortcutType (the two joint-space members)
enum ShortcutType { SHORTCUT_JOINT_SPACE = 0, SHORTCUT_JOINT_POSITION_VELOCITY_SPACE = 1 };

struct PostProcessingStats
{
    long long edges_checked = 0;    // isStateToStateValid motions submitted
    long long states_checked = 0;   // isStateValid states submitted
    long long device_calls = 0;
    double device_seconds = 0.0;
    double host_seconds = 0.0;
};

/// Paths are concatenated: path p = points[offsets[p] .. offsets[p + 1]) (rows of dof joint positions).
/// continuous[dof] = !RobotModel::hasPosLimit.  out_idx / out_offsets: the shortcut paths as indices into each
/// input path (both joint-space generators answer with the two end points, so a shortcut path is a subsequence).
bool ShortcutPaths(smplgpu_ctx* ctx, int dof, const uint8_t* continuous, const double* points,
                   const int32_t* offsets, int n_paths, int type, std::vector<int32_t>& out_idx,
                   std::vector<int32_t>& out_offsets, PostProcessingStats* stats, std::string* err);

struct EuclidShortcutStats
{
    long long motions = 0;          // Euclidean-space motions decided (all point pairs of every path)
    long long ik_solves = 0;        // planning-link IK solves of the deciding call, and how many converged
    long long ik_converged = 0;
    long long edges_checked = 0;    // waypoint edges (isStateToStateValid) of the deciding call
    long long device_calls = 0;
    double device_seconds = 0.0;
    double host_seconds = 0.0;
};

/// ShortcutPath with the EUCLID_SPACE type for many paths: every motion (i, j), i < j, of every path is decided in
/// one smplgpu_euclid_motions call, shortcut::ShortcutPath's greedy walk (greedyShortcut, granularity 1, original
/// costs by JointDistance) runs per path over the answers, and one more call returns the interior IK states of the
/// motions the walks emitted.  var_types[dof] SMPLGPU_VAR_* (continuous variables: wrapped JointDistance).
/// out_points: rows of dof; out_source: per output point its index in the input path, or -1 for an IK state;
/// out_offsets[n_paths + 1].
bool ShortcutPathsEuclid(smplgpu_ctx* ctx, int dof, const int32_t* var_types, const smplgpu_euclid_params& params,
                         const double* points, const int32_t* offsets, int n_paths, std::vector<double>& out_points,
                         std::vector<int32_t>& out_source, std::vector<int32_t>& out_offsets, EuclidShortcutStats* stats,
                         std::string* err);

/// The waypoints CollisionSpace::isStateToStateValid checks / CollisionSpace::interpolatePath returns
/// (robot_motion_collision_model.h:173-181, 224-249, 297-321; .cpp:371-407): var_types[dof] SMPLGPU_VAR_*,
/// weights[dof] = ||MR centre|| + MR radius of the variable's joint.  Appends count x dof values to `out`.
int InterpolateMotion(int dof, const int32_t* var_types, const double* weights, const double* start,
                      const double* finish, std::vector<double>& out);

/// InterpolatePath for many paths: every segment whose interpolated waypoints are all valid is replaced by them.
bool InterpolatePaths(smplgpu_ctx* ctx, int dof, const int32_t* var_types, const double* weights,
                      const double* points, const int32_t* offsets, int n_paths, std::vector<double>& out_points,
                      std::vector<int32_t>& out_offsets, PostProcessingStats* stats, std::string* err);

} // namespace smplhost

#endif
