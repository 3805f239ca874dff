#include "post_processing.h"

#include <algorithm>
#include <chrono>
#include <cmath>

namespace smplhost {

namespace {

struct Clock
{
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    double lap()
    {
        const auto n = std::chrono::steady_clock::now();
        const double d = std::chrono::duration<double>(n - t).count();
        t = n;
        return d;
    }
};

// angles::normalize_angle (smpl/include/smpl/angles.h:45-62)
double wrapAngle(double a)
{
    if (std::fabs(a) > 2.0 * M_PI) {
        a = std::fmod(a, 2.0 * M_PI);
    }
    if (a < -M_PI) {
        a += 2.0 * M_PI;
    }
    if (a > M_PI) {
        a -= 2.0 * M_PI;
    }
    return a;
}

// One path and its verdict table: verdict of the motion i -> j (i < j) sits at tri(i, j) of `ok`
struct PathView
{
    int dof;
    const uint8_t* continuous;
    const double* pts;       // n x dof
    int n;
    const uint8_t* ok;       // n (n - 1) / 2 verdicts, row i = pairs (i, i + 1 .. n - 1)
    std::vector<double> vel; // n x dof, position-velocity variant only

    const double* pt(int i) const { return pts + (size_t)i * dof; }
    size_t tri(int i, int j) const { return (size_t)i * (2 * (size_t)n - i - 1) / 2 + (size_t)(j - i - 1); }
    bool valid(int i, int j) const { return ok[tri(i, j)] != 0; }

    // distance() (post_processing.cpp:48-67)
    double posDistance(int a, int b) const
    {
        double d = 0.0;
        for (int v = 0; v < dof; ++v) {
            const double delta = pt(b)[v] - pt(a)[v];
            d += continuous[v] ? std::fabs(wrapAngle(delta)) : std::fabs(delta);
        }
        return d;
    }
    // pv_distance() (post_processing.cpp:69-97), both weights 1
    double pvDistance(int a, int b) const
    {
        const double d = posDistance(a, b);
        double vd = 0.0;
        for (int v = 0; v < dof; ++v) {
            vd += std::fabs(vel[(size_t)b * dof + v] - vel[(size_t)a * dof + v]);
        }
        return 1.0 * d + 1.0 * vd;
    }
};

typedef double (PathView::*CostFn)(int, int) const;

// The one generator of either joint-space variant: the straight motion a -> b when it is valid
// (JointPositionShortcutPathGenerator / JointPositionVelocityShortcutPathGenerator, post_processing.cpp:99-161)
inline bool straightMotion(const PathView& P, CostFn cost, int a, int b, double& c)
{
    if (!P.valid(a, b)) {
        return false;
    }
    c = (P.*cost)(a, b);
    return true;
}

std::vector<double> prefixCosts(const PathView& P, CostFn cost)
{
    std::vector<double> accum(P.n);
    accum[0] = 0.0;
    for (int i = 1; i < P.n; ++i) {
        accum[i] = accum[i - 1] + (P.*cost)(i - 1, i);
    }
    return accum;
}

// shortcut::ShortcutPath (shortcut.hpp:112-283) with granularity 1 and one generator: grow the segment
// [s, e] one point at a time for as long as the generator's motion s -> e+1 exists and costs no more than the
// best path over [s, e] plus the original step e -> e+1; otherwise emit the best path and open a new segment
// at e.  The best path over a segment is either its original points or the generator's motion between its end
// points.  motion(a, b, c) answers the generator: true and the motion's cost c when it has one.  via_motion
// (nullable) gets, per output point, 1 when the walk reaches it by a generator's motion, 0 by an original step.
template <class Motion>
void greedyShortcut(const PathView& P, CostFn cost, Motion motion, std::vector<int32_t>& out,
                    std::vector<uint8_t>* via_motion = nullptr)
{
    const int n = P.n;
    const std::vector<double> accum = prefixCosts(P, cost);
    int s = 0, e = 1;
    bool direct = false;      // best path over [s, e] is the generator's motion
    double best = 0.0;
    auto open = [&]() {
        direct = false;
        best = accum[e] - accum[s];
        double c;
        if (motion(s, e, c) && c <= best) {
            direct = true;
            best = c;
        }
    };
    auto emit = [&]() {       // the best path over [s, e] without its first point
        if (direct) {
            out.push_back(e);
            if (via_motion) via_motion->push_back(1);
        } else {
            for (int i = s + 1; i <= e; ++i) {
                out.push_back(i);
                if (via_motion) via_motion->push_back(0);
            }
        }
    };
    open();
    out.push_back(0);
    if (via_motion) via_motion->push_back(0);
    while (e != n - 1) {
        // the reference's last iteration (look-ahead 0 at the final point) only terminates the loop
        double extended = best + (accum[e + 1] - accum[e]);
        double c;
        if (motion(s, e + 1, c) && c <= extended) {
            direct = true;
            best = c;
            ++e;
        } else {
            emit();
            s = e;
            ++e;
            open();
        }
    }
    emit();
}

// shortcut::DivideAndConquerShortcutPath (shortcut.hpp:285-438)
void divideShortcut(const PathView& P, CostFn cost, const std::vector<double>& accum, int first, int last,
                    std::vector<int32_t>& out)
{
    if (last - first == 1) {
        out.push_back(last);
        return;
    }
    double c;
    if (straightMotion(P, cost, first, last, c) && c <= accum[last] - accum[first]) {
        out.push_back(last);
        return;
    }
    const int mid = first + ((last - first) >> 1);
    divideShortcut(P, cost, accum, first, mid, out);
    divideShortcut(P, cost, accum, mid, last, out);
}

// All motions (i, j), i < j, of every path as point indices; those of path p start at pair_begin[p], row i first
bool allPairs(const int32_t* offsets, int n_paths, std::vector<size_t>& pair_begin, std::vector<int32_t>& ia,
              std::vector<int32_t>& ib, const char* who, std::string* err)
{
    pair_begin.assign(n_paths + 1, 0);
    for (int p = 0; p < n_paths; ++p) {
        const size_t n = (size_t)(offsets[p + 1] - offsets[p]);
        pair_begin[p + 1] = pair_begin[p] + (n >= 2 ? n * (n - 1) / 2 : 0);
    }
    const size_t n_pairs = pair_begin[n_paths];
    if (n_pairs > 0x7FFFFFFFull) {
        if (err) *err = std::string(who) + ": more than 2^31 candidate motions";
        return false;
    }
    ia.resize(n_pairs);
    ib.resize(n_pairs);
    for (int p = 0; p < n_paths; ++p) {
        const int base = offsets[p], n = offsets[p + 1] - offsets[p];
        size_t k = pair_begin[p];
        for (int i = 0; i < n; ++i) {
            for (int j = i + 1; j < n; ++j, ++k) {
                ia[k] = base + i;
                ib[k] = base + j;
            }
        }
    }
    return true;
}

} // namespace

bool ShortcutPaths(smplgpu_ctx* ctx, int dof, const uint8_t* continuous, const double* points,
                   const int32_t* offsets, int n_paths, int type, std::vector<int32_t>& out_idx,
                   std::vector<int32_t>& out_offsets, PostProcessingStats* stats, std::string* err)
{
    out_idx.clear();
    out_offsets.assign(1, 0);
    PostProcessingStats st;
    Clock clk;
    if (n_paths <= 0) {
        if (stats) *stats = st;
        return true;
    }
    // every motion the generators can be asked for: all (i, j), i < j, of every path -- ONE device batch
    const int n_points = offsets[n_paths];
    std::vector<size_t> pair_begin;
    std::vector<int32_t> ia, ib;
    if (!allPairs(offsets, n_paths, pair_begin, ia, ib, "ShortcutPaths", err)) {
        return false;
    }
    const size_t n_pairs = pair_begin[n_paths];
    std::vector<uint8_t> ok(n_pairs);
    st.host_seconds += clk.lap();
    if (n_pairs > 0) {
        if (smplgpu_is_indexed_edges_valid(ctx, points, n_points, ia.data(), ib.data(), (int)n_pairs, ok.data(), nullptr) != 0) {
            if (err) *err = smplgpu_last_error(ctx);
            return false;
        }
        ++st.device_calls;
        st.edges_checked += (long long)n_pairs;
    }
    st.device_seconds += clk.lap();

    for (int p = 0; p < n_paths; ++p) {
        PathView P;
        P.dof = dof;
        P.continuous = continuous;
        P.pts = points + (size_t)offsets[p] * dof;
        P.n = offsets[p + 1] - offsets[p];
        P.ok = ok.data() + pair_begin[p];
        const size_t first_out = out_idx.size();
        if (P.n < 2) {   // "pout = pin" (post_processing.cpp:291-294)
            for (int i = 0; i < P.n; ++i) out_idx.push_back(i);
        } else if (type == SHORTCUT_JOINT_SPACE) {
            greedyShortcut(P, &PathView::posDistance, [&](int a, int b, double& c) {
                return straightMotion(P, &PathView::posDistance, a, b, c);
            }, out_idx);
        } else {
            // CreatePositionVelocityPath (post_processing.cpp:367-401): the sign of the motion into each point
            P.vel.assign((size_t)P.n * dof, 0.0);
            for (int i = 1; i < P.n; ++i) {
                for (int v = 0; v < dof; ++v) {
                    const double delta = P.pt(i)[v] - P.pt(i - 1)[v];
                    P.vel[(size_t)i * dof + v] = std::copysign(1.0, continuous[v] ? wrapAngle(delta) : delta);
                }
            }
            std::vector<int32_t> greedy, dnc;
            greedyShortcut(P, &PathView::pvDistance, [&](int a, int b, double& c) {
                return straightMotion(P, &PathView::pvDistance, a, b, c);
            }, greedy);
            dnc.push_back(0);
            divideShortcut(P, &PathView::pvDistance, prefixCosts(P, &PathView::pvDistance), 0, P.n - 1, dnc);
            auto total = [&](const std::vector<int32_t>& idx) {
                double c = 0.0;
                for (size_t i = 1; i < idx.size(); ++i) c = c + P.pvDistance(idx[i - 1], idx[i]);
                return c;
            };
            const std::vector<int32_t>& pick = total(dnc) < total(greedy) ? dnc : greedy;   // "Divide and Conquer Wins!"
            out_idx.insert(out_idx.end(), pick.begin(), pick.end());
        }
        (void)first_out;
        out_offsets.push_back((int32_t)out_idx.size());
    }
    st.host_seconds += clk.lap();
    if (stats) *stats = st;
    return true;
}

bool ShortcutPathsEuclid(smplgpu_ctx* ctx, int dof, const int32_t* var_types, const smplgpu_euclid_params& params,
                         const double* points, const int32_t* offsets, int n_paths, std::vector<double>& out_points,
                         std::vector<int32_t>& out_source, std::vector<int32_t>& out_offsets, EuclidShortcutStats* stats,
                         std::string* err)
{
    out_points.clear();
    out_source.clear();
    out_offsets.assign(1, 0);
    EuclidShortcutStats st;
    Clock clk;
    if (n_paths <= 0) {
        if (stats) *stats = st;
        return true;
    }
    std::vector<uint8_t> continuous(dof);
    for (int v = 0; v < dof; ++v) continuous[v] = var_types[v] == SMPLGPU_VAR_CONTINUOUS ? 1 : 0;
    // 1. every motion (i, j), i < j, of every path decided in ONE device call
    const int n_points = offsets[n_paths];
    std::vector<size_t> pair_begin;
    std::vector<int32_t> ia, ib;
    if (!allPairs(offsets, n_paths, pair_begin, ia, ib, "ShortcutPathsEuclid", err)) {
        return false;
    }
    const size_t n_pairs = pair_begin[n_paths];
    std::vector<uint8_t> ok(n_pairs);
    std::vector<double> cost(n_pairs);
    std::vector<int32_t> steps(n_pairs);
    int64_t ctr[2] = { 0, 0 };
    st.host_seconds += clk.lap();
    if (n_pairs > 0) {
        if (smplgpu_euclid_motions(ctx, points, n_points, ia.data(), ib.data(), (int)n_pairs, &params, ok.data(),
                                   cost.data(), steps.data(), nullptr, nullptr, ctr) != 0) {
            if (err) *err = smplgpu_last_error(ctx);
            return false;
        }
        ++st.device_calls;
        st.motions += (long long)n_pairs;
        st.ik_solves += ctr[0];
        st.ik_converged += ctr[1];
        for (size_t k = 0; k < n_pairs; ++k) {
            st.edges_checked += steps[k] <= params.max_steps ? steps[k] : 0;
        }
    }
    st.device_seconds += clk.lap();

    // 2. the greedy walk of each path over the answers
    std::vector<std::vector<int32_t>> idx(n_paths);
    std::vector<std::vector<uint8_t>> via(n_paths);
    std::vector<std::vector<int>> emitted(n_paths);   // per output point: the emitted motion into it, or -1
    std::vector<int32_t> sa, sb, sn;  // the emitted motions that have interior states, and their step counts
    std::vector<int64_t> soff;        // where their states go
    int64_t n_states = 0;
    for (int p = 0; p < n_paths; ++p) {
        PathView P;
        P.dof = dof;
        P.continuous = continuous.data();
        P.pts = points + (size_t)offsets[p] * dof;
        P.n = offsets[p + 1] - offsets[p];
        P.ok = ok.data() + pair_begin[p];
        if (P.n < 2) {   // "pout = pin"
            for (int i = 0; i < P.n; ++i) {
                idx[p].push_back(i);
                via[p].push_back(0);
            }
            continue;
        }
        const double* pc = cost.data() + pair_begin[p];
        greedyShortcut(P, &PathView::posDistance, [&](int a, int b, double& c) {
            if (!P.valid(a, b)) return false;
            c = pc[P.tri(a, b)];
            return true;
        }, idx[p], &via[p]);
        emitted[p].assign(idx[p].size(), -1);
        for (size_t i = 1; i < idx[p].size(); ++i) {
            const size_t k = pair_begin[p] + P.tri(idx[p][i - 1], idx[p][i]);
            if (via[p][i] && steps[k] > 1) {
                emitted[p][i] = (int)sa.size();
                sa.push_back(ia[k]);
                sb.push_back(ib[k]);
                sn.push_back(steps[k]);
                soff.push_back(n_states);
                n_states += steps[k] - 1;
            }
        }
    }
    st.host_seconds += clk.lap();

    // 3. the interior states of the emitted motions: the same motions again, deterministic
    std::vector<double> states((size_t)n_states * dof);
    if (!sa.empty()) {
        const int m = (int)sa.size();
        std::vector<uint8_t> ok2(m);
        std::vector<double> cost2(m);
        std::vector<int32_t> steps2(m);
        if (smplgpu_euclid_motions(ctx, points, n_points, sa.data(), sb.data(), m, &params, ok2.data(), cost2.data(),
                                   steps2.data(), soff.data(), states.data(), ctr) != 0) {
            if (err) *err = smplgpu_last_error(ctx);
            return false;
        }
        ++st.device_calls;
        for (int k = 0; k < m; ++k) {
            if (!ok2[k] || steps2[k] != sn[k]) {
                if (err) *err = "ShortcutPathsEuclid: a motion changed between the two device calls";
                return false;
            }
        }
    }
    st.device_seconds += clk.lap();

    // 4. the output: input points copied, IK states where a motion was emitted
    for (int p = 0; p < n_paths; ++p) {
        const int base = offsets[p];
        for (size_t i = 0; i < idx[p].size(); ++i) {
            const int m = emitted[p].empty() ? -1 : emitted[p][i];
            if (m >= 0) {
                out_points.insert(out_points.end(), states.begin() + soff[m] * dof, states.begin() + (soff[m] + sn[m] - 1) * dof);
                out_source.insert(out_source.end(), (size_t)(sn[m] - 1), -1);
            }
            const int j = base + idx[p][i];
            out_points.insert(out_points.end(), points + (size_t)j * dof, points + (size_t)(j + 1) * dof);
            out_source.push_back(idx[p][i]);
        }
        out_offsets.push_back((int32_t)out_source.size());
    }
    st.host_seconds += clk.lap();
    if (stats) *stats = st;
    return true;
}

int InterpolateMotion(int dof, const int32_t* var_types, const double* weights, const double* start,
                      const double* finish, std::vector<double>& out)
{
    double motion = 0.0;
    std::vector<double> diffs(dof);
    for (int v = 0; v < dof; ++v) {
        if (var_types[v] == SMPLGPU_VAR_CONTINUOUS) {
            diffs[v] = wrapAngle(finish[v] - start[v]);
            motion += weights[v] * std::fabs(diffs[v]);
        } else if (var_types[v] == SMPLGPU_VAR_REVOLUTE) {
            diffs[v] = finish[v] - start[v];
            motion += weights[v] * std::fabs(diffs[v]);
        } else {
            diffs[v] = finish[v] - start[v];
            motion += std::fabs(diffs[v]);
        }
    }
    int count = 0;
    if (motion != 0.0) {
        count = std::max(2, (int)std::ceil(motion / 0.05) + 1);
    }
    const double inv = count > 1 ? 1.0 / (double)(count - 1) : 0.0;
    for (int i = 0; i < count; ++i) {
        const double alpha = (double)i * inv;
        for (int v = 0; v < dof; ++v) {
            out.push_back(start[v] + alpha * diffs[v]);
        }
    }
    return count;
}

bool InterpolatePaths(smplgpu_ctx* ctx, int dof, const int32_t* var_types, const double* weights,
                      const double* points, const int32_t* offsets, int n_paths, std::vector<double>& out_points,
                      std::vector<int32_t>& out_offsets, PostProcessingStats* stats, std::string* err)
{
    out_points.clear();
    out_offsets.assign(1, 0);
    PostProcessingStats st;
    Clock clk;
    // the waypoints of every segment of every path, then ONE isStatesValid batch over all of them
    std::vector<double> wps;
    std::vector<size_t> seg_begin(1, 0);   // in waypoints
    for (int p = 0; p < n_paths; ++p) {
        for (int i = offsets[p]; i + 1 < offsets[p + 1]; ++i) {
            InterpolateMotion(dof, var_types, weights, points + (size_t)i * dof, points + (size_t)(i + 1) * dof, wps);
            seg_begin.push_back(wps.size() / dof);
        }
    }
    const size_t n_wp = wps.size() / dof;
    if (n_wp > 0x7FFFFFFFull) {
        if (err) *err = "InterpolatePaths: more than 2^31 waypoints";
        return false;
    }
    std::vector<uint8_t> ok(n_wp);
    st.host_seconds += clk.lap();
    if (n_wp > 0) {
        if (smplgpu_is_states_valid(ctx, wps.data(), (int)n_wp, ok.data()) != 0) {
            if (err) *err = smplgpu_last_error(ctx);
            return false;
        }
        ++st.device_calls;
        st.states_checked += (long long)n_wp;
    }
    st.device_seconds += clk.lap();
    size_t seg = 0;
    for (int p = 0; p < n_paths; ++p) {
        const int first = offsets[p], last = offsets[p + 1];
        if (last > first) {
            out_points.insert(out_points.end(), points + (size_t)first * dof, points + (size_t)(first + 1) * dof);
        }
        for (int i = first; i + 1 < last; ++i, ++seg) {
            const size_t b = seg_begin[seg], e = seg_begin[seg + 1];
            bool collision = false;
            for (size_t k = b; k < e; ++k) {
                if (!ok[k]) {
                    collision = true;
                    break;
                }
            }
            if (collision) {   // "Interpolated path collides. Resorting to original waypoints"
                out_points.insert(out_points.end(), points + (size_t)(i + 1) * dof, points + (size_t)(i + 2) * dof);
            } else if (e > b) {
                out_points.insert(out_points.end(), wps.begin() + (b + 1) * dof, wps.begin() + e * dof);
            }
        }
        out_offsets.push_back((int32_t)(out_points.size() / dof));
    }
    st.host_seconds += clk.lap();
    if (stats) *stats = st;
    return true;
}

} // namespace smplhost
