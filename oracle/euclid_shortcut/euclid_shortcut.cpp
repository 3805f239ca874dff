// ORACLE (test infrastructure only -- never linked into the product path).
//
// ShortcutPath(rm, cc, pin, pout, type) with type EUCLID_SPACE (post_processing.cpp:284-365), sequentially.  The
// reference's generator (EuclidShortcutPathGenerator) rests on a third-party IK, so the motion it generates is the
// project's own definition (DESIGN.md section 2, parity unpinned), written here once and restated on the device
// (smpl_b200/csrc/euclid.cuh), pinned oracle <-> device only:
//   ends    f(qa) = (pa, Ra), f(qb) = (pb, Rb): planningLinkIk's forward map (T_kin_to_planning * the planning chain,
//           the target point R offset + p)
//   turn    w = rotationVector(Rb Ra^T), theta = sqrt((w0^2 + w1^2) + w2^2); d = sqrt((dx^2 + dy^2) + dz^2) of pb - pa
//   steps   n = max(1, ceil(max(d / max_step_m, theta / max_step_rad))); refused when n > max_steps
//   states  qa, q1 .. q(n-1), qb: q_k = planningLinkIk (seeded at q(k-1)) for the position pa + (k / n)(pb - pa) and
//           the rotation Rot2(w / theta, (k / n) theta) Ra (Ra when theta = 0); the first solve that does not converge
//           or fails checkJointLimits refuses the motion, and no later one is run
//   valid   isStateToStateValid of every consecutive pair
//   cost    JointDistance (post_processing.cpp:48-67) of the consecutive pairs, summed in order
// The walk is shortcut.hpp's greedy ShortcutPath (granularity 1, one generator), restated from oracle/shortcut.h so that
// its best path carries the generated states.
//
// Built as oracle/euclid_shortcut/liboracle_euclid_shortcut.so over oracle/liboracle.so; it takes the scene handles of
// the oracle's C API.  planningLinkIk, rotationVector and rot2 come from the snap oracle's source, included unchanged.
#include "../snap/snap_lattice.cpp"
#include "../shortcut.h"

namespace {

struct EuclidParams
{
    double max_step_m, max_step_rad;
    int max_steps;
    IkParams ik;
};

bool badParams(const EuclidParams& p)
{
    return !(p.max_step_m > 0.0) || !std::isfinite(p.max_step_m) || !(p.max_step_rad > 0.0) ||
           !std::isfinite(p.max_step_rad) || p.max_steps < 1 || p.max_steps > 4096 || p.ik.max_iterations < 1 ||
           !(p.ik.tolerance > 0.0) || !std::isfinite(p.ik.tolerance);
}

// planningLinkIk's forward map: the chain in its order, then the target point
void planningPose(const KDLRobotModel& m, const KdlFrame& Tk, const double offset[3], const std::vector<double>& q,
                  double p[3], double R[9])
{
    KdlFrame f1 = KdlFrame::Identity();
    for (int s = 0; s < m.planning_segment_nr; ++s) {
        f1 = f1 * segmentPose(m, s, q);
    }
    const KdlFrame f = Tk * f1;
    for (int i = 0; i < 3; ++i) {
        p[i] = (f.M[3 * i] * offset[0] + f.M[3 * i + 1] * offset[1] + f.M[3 * i + 2] * offset[2]) + f.p[i];
    }
    for (int i = 0; i < 9; ++i) R[i] = f.M[i];
}

struct Motion
{
    int n = 0;                                    // max_steps + 1 when refused for its length
    bool chain = false;                           // every IK solve converged within the limits
    bool ok = false;                              // ... and every edge is valid
    double cost = 0.0;                            // 0 unless the chain completed
    std::vector<std::vector<double>> interior;    // q1 .. q(n-1)
    long long solves = 0, converged = 0;
};

class Euclid
{
public:
    Euclid(oracle_scene* s, const double* T, const EuclidParams& p) : m_s(s), m_p(p)
    {
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) m_Tk.M[3 * r + c] = T[4 * r + c];
            m_Tk.p[r] = T[4 * r + 3];
        }
        m_cont = s->kdl->continuous;
    }

    double jointDistance(const std::vector<double>& a, const std::vector<double>& b) const
    {
        return oracle::JointDistance(m_cont, a.data(), b.data());
    }

    Motion motion(const std::vector<double>& qa, const std::vector<double>& qb) const
    {
        const KDLRobotModel& m = *m_s->kdl;
        Motion r;
        double pa[3], Ra[9], pb[3], Rb[9], E[9], w[3];
        planningPose(m, m_Tk, m_s->xyz_offset, qa, pa, Ra);
        planningPose(m, m_Tk, m_s->xyz_offset, qb, pb, Rb);
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) {
                E[3 * i + j] = (Rb[3 * i] * Ra[3 * j] + Rb[3 * i + 1] * Ra[3 * j + 1]) + Rb[3 * i + 2] * Ra[3 * j + 2];
            }
        }
        rotationVector(E, w);
        const double theta = std::sqrt((w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]);
        double u[3];
        for (int i = 0; i < 3; ++i) u[i] = theta > 0.0 ? w[i] / theta : 0.0;
        const double dx = pb[0] - pa[0], dy = pb[1] - pa[1], dz = pb[2] - pa[2];
        const double d = std::sqrt((dx * dx + dy * dy) + dz * dz);
        const double steps = std::max(d / m_p.max_step_m, theta / m_p.max_step_rad);
        if (!(steps <= (double)m_p.max_steps)) {
            r.n = m_p.max_steps + 1;
            return r;
        }
        const int n = std::max(1, (int)std::ceil(steps));
        r.n = n;
        std::vector<double> q = qa;
        for (int k = 1; k < n; ++k) {
            const double alpha = (double)k / (double)n;
            double tp[3], tR[9];
            for (int i = 0; i < 3; ++i) tp[i] = pa[i] + alpha * (pb[i] - pa[i]);
            if (theta > 0.0) {
                double Rk[9];
                rot2(u, alpha * theta, Rk);
                for (int i = 0; i < 3; ++i) {
                    for (int j = 0; j < 3; ++j) {
                        tR[3 * i + j] = (Rk[3 * i] * Ra[j] + Rk[3 * i + 1] * Ra[3 + j]) + Rk[3 * i + 2] * Ra[6 + j];
                    }
                }
            } else {
                std::copy(Ra, Ra + 9, tR);
            }
            int it = 0;
            const bool conv = planningLinkIk(m, m_Tk, m_s->xyz_offset, tp, tR, m_p.ik, q, &it);
            ++r.solves;
            r.converged += conv ? 1 : 0;
            if (!conv || !m.checkJointLimits(q)) {
                r.interior.clear();
                return r;
            }
            r.interior.push_back(q);
        }
        r.chain = true;
        const std::vector<double>* prev = &qa;
        double c = 0.0;
        for (const std::vector<double>& s : r.interior) {
            c = c + jointDistance(*prev, s);
            prev = &s;
        }
        c = c + jointDistance(*prev, qb);
        r.cost = c;
        r.ok = true;
        prev = &qa;
        for (size_t k = 0; k <= r.interior.size() && r.ok; ++k) {
            const std::vector<double>& next = k < r.interior.size() ? r.interior[k] : qb;
            r.ok = m_s->cc->isStateToStateValid(*prev, next, nullptr);
            prev = &next;
        }
        return r;
    }

private:
    oracle_scene* m_s;
    EuclidParams m_p;
    KdlFrame m_Tk;
    std::vector<bool> m_cont;
};

// a path over a segment: its points, and per point the input index (-1 for an IK state)
struct SegPath
{
    std::vector<std::vector<double>> q;
    std::vector<int> src;
};

// shortcut.hpp:112-283 (oracle/shortcut.h ShortcutPath) with granularity 1 and the Euclidean generator, carrying the
// generated states: the best path over [seg_start, seg_end] is its original points or the generator's path
void shortcutPathEuclid(const Euclid& g, const std::vector<std::vector<double>>& pts, SegPath& out, long long* solves,
                        long long* converged)
{
    const size_t psize = pts.size();
    if (psize == 0) {
        return;
    }
    if (psize < 2) {
        out.q.push_back(pts[0]);
        out.src.push_back(0);
        return;
    }
    std::vector<double> costs(psize - 1);
    for (size_t i = 1; i < psize; ++i) costs[i - 1] = g.jointDistance(pts[i - 1], pts[i]);
    const std::vector<double> accum = oracle::shortcut_detail::Accumulate(costs);
    auto generate = [&](size_t a, size_t b, double& cost, SegPath& path) {
        const Motion mo = g.motion(pts[a], pts[b]);
        *solves += mo.solves;
        *converged += mo.converged;
        if (!mo.ok) return false;
        cost = mo.cost;
        path.q.assign(1, pts[a]);
        path.src.assign(1, (int)a);
        for (const std::vector<double>& s : mo.interior) {
            path.q.push_back(s);
            path.src.push_back(-1);
        }
        path.q.push_back(pts[b]);
        path.src.push_back((int)b);
        return true;
    };
    size_t seg_start = 0, seg_end = 1;
    SegPath best;
    double best_cost = 0.0;
    auto open_segment = [&]() {
        best.q.assign(pts.begin() + seg_start, pts.begin() + seg_end + 1);
        best.src.clear();
        for (size_t i = seg_start; i <= seg_end; ++i) best.src.push_back((int)i);
        best_cost = accum[seg_end] - accum[seg_start];
        double cost;
        SegPath p;
        if (generate(seg_start, seg_end, cost, p) && cost <= best_cost) {
            best = p;
            best_cost = cost;
        }
    };
    auto emit = [&]() {
        out.q.insert(out.q.end(), best.q.begin() + 1, best.q.end());
        out.src.insert(out.src.end(), best.src.begin() + 1, best.src.end());
    };
    open_segment();
    out.q.push_back(pts[0]);
    out.src.push_back(0);
    while (seg_end != psize) {
        bool improved = false;
        const size_t look = std::min((size_t)1, psize - seg_end - 1);
        if (look != 0) {
            double new_cost = best_cost + (accum[seg_end + look] - accum[seg_end]);
            double cost;
            SegPath p;
            if (generate(seg_start, seg_end + look, cost, p) && cost <= new_cost) {
                improved = true;
                best = p;
                new_cost = cost;
            }
            best_cost = new_cost;
        }
        if (improved) {
            seg_end += look;
        } else if (look == 0) {
            seg_end = psize;
        } else {
            emit();
            seg_start = seg_end;
            seg_end += look;
            open_segment();
        }
    }
    emit();
}

bool readParams(double max_step_m, double max_step_rad, int max_steps, int ik_max_iterations, double ik_tolerance,
                EuclidParams& p)
{
    p.max_step_m = max_step_m;
    p.max_step_rad = max_step_rad;
    p.max_steps = max_steps;
    p.ik.max_iterations = ik_max_iterations;
    p.ik.tolerance = ik_tolerance;
    return !badParams(p);
}

} // namespace

extern "C" {

/// The Euclidean-space motions points[idx_a[e]] -> points[idx_b[e]], one after the other: ok[e], cost[e] (0 unless
/// the IK chain completed), n_steps[e] (max_steps + 1 when refused for its length); with states (nullable) the n - 1
/// interior states of every completed chain at states[state_offsets[e] ..][dof].  counters[2] (nullable): IK solves
/// run, converged.  T_kin_to_planning 3x4 row-major.  Returns 0, or -1 for bad parameters, indices or scene.
int oracle_euclid_motions(oracle_scene* s, const double* T_kin_to_planning, const double* points, int n_points,
                          const int32_t* idx_a, const int32_t* idx_b, int n, double max_step_m, double max_step_rad,
                          int max_steps, int ik_max_iterations, double ik_tolerance, uint8_t* ok, double* cost,
                          int32_t* n_steps, const int64_t* state_offsets, double* states, int64_t* counters)
{
    EuclidParams p;
    if (!s || !s->kdl || !s->cc || !T_kin_to_planning || n < 0 ||
        !readParams(max_step_m, max_step_rad, max_steps, ik_max_iterations, ik_tolerance, p)) {
        return -1;
    }
    for (int e = 0; e < n; ++e) {
        if (idx_a[e] < 0 || idx_a[e] >= n_points || idx_b[e] < 0 || idx_b[e] >= n_points) return -1;
    }
    const int dof = s->dof;
    const Euclid g(s, T_kin_to_planning, p);
    long long solves = 0, conv = 0;
    for (int e = 0; e < n; ++e) {
        const std::vector<double> qa(points + (size_t)idx_a[e] * dof, points + (size_t)(idx_a[e] + 1) * dof);
        const std::vector<double> qb(points + (size_t)idx_b[e] * dof, points + (size_t)(idx_b[e] + 1) * dof);
        const Motion mo = g.motion(qa, qb);
        ok[e] = mo.ok ? 1 : 0;
        cost[e] = mo.cost;
        n_steps[e] = mo.n;
        solves += mo.solves;
        conv += mo.converged;
        if (states && mo.chain) {
            for (size_t k = 0; k < mo.interior.size(); ++k) {
                std::copy(mo.interior[k].begin(), mo.interior[k].end(), states + ((size_t)state_offsets[e] + k) * dof);
            }
        }
    }
    if (counters) {
        counters[0] = solves;
        counters[1] = conv;
    }
    return 0;
}

/// ShortcutPath with the EUCLID_SPACE type for one path (n x dof): out_points[max_out][dof] and out_source[max_out]
/// (the input index of each output point, -1 for an IK state).  counters[2] (nullable): IK solves run, converged.
/// Returns the number of output points (written only when it is <= max_out), or -1 for bad parameters or scene.
int oracle_shortcut_path_euclid(oracle_scene* s, const double* T_kin_to_planning, const double* path, int n,
                                double max_step_m, double max_step_rad, int max_steps, int ik_max_iterations,
                                double ik_tolerance, double* out_points, int32_t* out_source, int max_out,
                                int64_t* counters)
{
    EuclidParams p;
    if (!s || !s->kdl || !s->cc || !T_kin_to_planning || n < 0 ||
        !readParams(max_step_m, max_step_rad, max_steps, ik_max_iterations, ik_tolerance, p)) {
        return -1;
    }
    const int dof = s->dof;
    const Euclid g(s, T_kin_to_planning, p);
    std::vector<std::vector<double>> pts(n);
    for (int i = 0; i < n; ++i) pts[i].assign(path + (size_t)i * dof, path + (size_t)(i + 1) * dof);
    SegPath out;
    long long solves = 0, conv = 0;
    shortcutPathEuclid(g, pts, out, &solves, &conv);
    if (counters) {
        counters[0] = solves;
        counters[1] = conv;
    }
    const int total = (int)out.src.size();
    if (total <= max_out) {
        for (int i = 0; i < total; ++i) {
            std::copy(out.q[i].begin(), out.q[i].end(), out_points + (size_t)i * dof);
            out_source[i] = out.src[i];
        }
    }
    return total;
}

} // extern "C"
