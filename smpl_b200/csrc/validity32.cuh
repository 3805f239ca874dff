// Kernels (1)+(2)+(3), certified single-precision form.
//
// The reference decides validity with IEEE-double arithmetic, but every decision
// is a comparison of a *cell index* (worldToGrid of a sphere centre) or of a
// squared centre distance against a threshold.  Those decisions can be made in
// single precision whenever the double-precision value is provably not within
// the single-precision error bound of a decision boundary:
//
//   * forward kinematics runs in float with FMA (joint angle split hi + lo so the
//     sin/cos argument keeps double accuracy), in GRID UNITS: the host folds the
//     world -> grid map into the model (translations, centres and radii in cells, the
//     base transforms map to grid coordinates c = inv_res (x - o) - 1, whose
//     round-to-nearest is the cell), and derives a rigorous bound E on
//     |c_f32 - c_f64| from the chain (smplgpu.cu: build_model32);
//   * a sphere/field test whose grid coordinate lies within eps_cells of a cell
//     boundary evaluates EVERY cell the double value could fall in; if all of them
//     give the same outcome the decision is certain, otherwise it is ambiguous;
//   * a sphere-pair test with |d - (r1+r2)| within 2.5 E is ambiguous.
//
// A state with a certain collision is invalid; a state with no collision and no
// ambiguous decision is valid; anything else is appended to a list that the
// double-precision kernels (validity.cuh) then resolve exactly.  The verdicts
// are therefore bit-identical to the all-double path; the number of items that
// needed double precision is reported (smplgpu_last_validity_stats).
//
// Work decomposition: one thread per state (edges: the block's waypoints are
// spread over its threads as in validity.cuh); the robot tables live in shared
// memory (a compact float copy, pre-order sphere trees with skip links so the
// descent needs no stack); per thread, shared memory keeps the transforms of
// branching parents and the root-sphere centres of the trees that take part in
// pair tests (12 bytes per tree instead of a 48-byte transform per link, which
// doubles the resident warps).
//
// Reference semantics restated: see validity.cuh.
#pragma once

#include "model.cuh"
#include "validity.cuh"

namespace smplgpu {

constexpr int V32_THREADS = 128;
// -DV32_MIN_BLOCKS=n asks ptxas for n resident blocks per SM (tuning experiments).  By default the state and edge
// kernels ask for 9 and 8 (56 and 64 registers): left to itself ptxas picks the same counts but keeps the shared-memory
// addresses of the model's tables in local memory and reloads them on every link; with the target given, the edge kernel
// has no local memory and the state kernel 16 bytes (DESIGN.md section 5).
#ifdef V32_MIN_BLOCKS
#define V32_BOUNDS __launch_bounds__(V32_THREADS, V32_MIN_BLOCKS)
#define V32_STATES_BOUNDS V32_BOUNDS
#define V32_EDGES_BOUNDS V32_BOUNDS
#else
#define V32_BOUNDS __launch_bounds__(V32_THREADS)
#define V32_STATES_BOUNDS __launch_bounds__(V32_THREADS, 9)
#define V32_EDGES_BOUNDS __launch_bounds__(V32_THREADS, 8)
#endif
constexpr float V32_MAX_ANGLE = 64.0f;   // beyond this the hi/lo split no longer keeps the sin/cos argument exact enough

// Compact single-precision model: a blob of 4-byte words copied into shared memory by every block.
// Offsets are in words from the start of the blob.
struct Model32Header
{
    int words;            // total size of the blob
    int n_links, n_nodes, n_pairs, n_allowed, n_slots, dof;   // n_slots: transforms kept for branching parents
    int off_link_i;       // int4 per link: parent, fn, var, slot
    int off_link_n;       // int2 per link: first node, end node (pre-order ids of the trees riding on the link)
    int off_origin;       // float[12] per link, Xf32 word order (joint origin; constant joints pre-multiplied; translation in cells)
    int off_axis;         // float4 per link: joint axis (general revolute); prismatic: inv_res * third origin column
    int off_base;         // float[12] per link, Xf32 word order (used when parent < 0): world -> grid coordinates less K (Grid32)
    int off_node_c;       // float4 per node: centre xyz, radius (cells)
    int off_node_i;       // int4 per node: skip, threshold, z, rank of the (double) radius; z = pair-tree index of a
                          // paired tree's root (else -1) in roots-only mode, slot of the node's link in full mode
    int off_node_orig;    // int per node: index in the caller's node table
    int off_pair;         // int4 per pair: pair-tree index a, b; root node a, b (pre-order ids)
    int off_allowed;      // int2 per allowed leaf pair (pre-order ids)
    float e_cells;        // bound on |centre_f32 - centre_f64| (cells)
    float eps_cells;      // e_cells + the rounding of the decision itself (cells)
    float pair_k;         // 2.5 * e_cells
    float q_lin_max;      // largest |q| of a prismatic variable the bound covers (joint units)
    int n_ptrees;         // roots-only pair mode: trees in pair tests (one saved root centre each); 0 = full descent mode
    int pad[2];
};
static_assert(sizeof(Model32Header) % 16 == 0, "header must keep 16-byte alignment of the arrays");

// The world -> grid map itself is folded into the model's base transforms, less a whole number of cells K per axis
// (the robot base's cell) that keeps the chain's magnitudes, and so its rounding, small: the model yields c - K and
// the cell index is round(c - K) + K.  kx, ky, kz = bits(ROUND_MAGIC) - K, the integer round_cell subtracts.
struct Grid32
{
    int nx, ny, nz;
    int kx, ky, kz;
};

// A link transform [R | t] (3x4, grid units).  Rows 0 and 1 are kept as float2 pairs column by column,
// c[j] = (m[0][j], m[1][j]), row 2 as scalars, r2[j] = m[2][j]: a product or a point transform then does rows 0 and 1 in
// one packed FP32 instruction (FFMA2 / FMUL2, two IEEE single-precision operations) with the other operand a broadcast
// scalar, and row 2 in scalar instructions.  Each element is the same IEEE operation on the same operands, in the same
// nesting order, as in the scalar form, so centres are bit for bit those the error bound of build_model32 covers.
// Blob and slot words of a transform: c[0].x c[0].y c[1].x c[1].y c[2].x c[2].y c[3].x c[3].y r2[0..3].
struct Xf32
{
    float2 c[4];
    float r2[4];
};

__device__ __forceinline__ float2 bcast2(float s) { return make_float2(s, s); }
// s * a + b and s * a, in one rounding each, on a scalar or (packed) on a pair
__device__ __forceinline__ float vfma(float s, float a, float b) { return fmaf(s, a, b); }
__device__ __forceinline__ float2 vfma(float s, float2 a, float2 b) { return __ffma2_rn(bcast2(s), a, b); }
__device__ __forceinline__ float vmul(float s, float a) { return __fmul_rn(s, a); }
__device__ __forceinline__ float2 vmul(float s, float2 a) { return __fmul2_rn(bcast2(s), a); }

__device__ __forceinline__ void xf32_mul(const Xf32& a, const Xf32& b, Xf32& r)
{
    // r[i][j] = a[i][0] b[0][j] + a[i][1] b[1][j] + a[i][2] b[2][j] (+ a[i][3] for j = 3), innermost product first
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float b0 = b.c[j].x, b1 = b.c[j].y, b2 = b.r2[j];
        r.c[j] = vfma(b0, a.c[0], vfma(b1, a.c[1], vmul(b2, a.c[2])));
        r.r2[j] = vfma(b0, a.r2[0], vfma(b1, a.r2[1], vmul(b2, a.r2[2])));
    }
    const float b0 = b.c[3].x, b1 = b.c[3].y, b2 = b.r2[3];
    r.c[3] = vfma(b0, a.c[0], vfma(b1, a.c[1], vfma(b2, a.c[2], a.c[3])));
    r.r2[3] = vfma(b0, a.r2[0], vfma(b1, a.r2[1], vfma(b2, a.r2[2], a.r2[3])));
}

// p = T (x, y, z): (p.x, p.y) packed, p.z scalar
__device__ __forceinline__ void xf32_point(const Xf32& a, float x, float y, float z, float2& pxy, float& pz)
{
    pxy = vfma(x, a.c[0], vfma(y, a.c[1], vfma(z, a.c[2], a.c[3])));
    pz = vfma(x, a.r2[0], vfma(y, a.r2[1], vfma(z, a.r2[2], a.r2[3])));
}

__device__ __forceinline__ void load12(const float* __restrict__ p, Xf32& t)
{
    const float4 a = *reinterpret_cast<const float4*>(p);
    const float4 b = *reinterpret_cast<const float4*>(p + 4);
    const float4 c = *reinterpret_cast<const float4*>(p + 8);
    t.c[0] = make_float2(a.x, a.y); t.c[1] = make_float2(a.z, a.w);
    t.c[2] = make_float2(b.x, b.y); t.c[3] = make_float2(b.z, b.w);
    t.r2[0] = c.x; t.r2[1] = c.y; t.r2[2] = c.z; t.r2[3] = c.w;
}

__device__ __forceinline__ void slot32_store(float* slots, int slot, const Xf32& t)
{
    float* p = slots + (size_t)slot * 12 * blockDim.x + threadIdx.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        p[(2 * j) * blockDim.x] = t.c[j].x;
        p[(2 * j + 1) * blockDim.x] = t.c[j].y;
        p[(8 + j) * blockDim.x] = t.r2[j];
    }
}

__device__ __forceinline__ void slot32_load(const float* slots, int slot, Xf32& t)
{
    const float* p = slots + (size_t)slot * 12 * blockDim.x + threadIdx.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        t.c[j] = make_float2(p[(2 * j) * blockDim.x], p[(2 * j + 1) * blockDim.x]);
        t.r2[j] = p[(8 + j) * blockDim.x];
    }
}

// Cell and remainder of a grid coordinate c, on the FMA pipe.  For |c| < 2^22, c + 1.5 * 2^23 lies in (2^23, 2^24),
// where floats are spaced 1 apart, so this one add rounds c to the nearest integer (ties to even) and leaves it in
// the low mantissa bits: the integer difference of the two bit patterns is round(c).  (c + M) - M is round(c)
// exactly (Sterbenz), and so is rem = c - round(c) in [-1/2, 1/2] (both are multiples of ulp(c), or round(c) = 0).
// k = bits(M) - K adds the model's whole-cell offset K in the same integer subtract.
constexpr float ROUND_MAGIC = 12582912.0f;   // 1.5 * 2^23
__device__ __forceinline__ int round_cell(float c, int k, float& rem)
{
    const float t = __fadd_rn(c, ROUND_MAGIC);
    rem = __fsub_rn(c, __fsub_rn(t, ROUND_MAGIC));
    return __float_as_int(t) - k;
}

// round_cell of x and y at once, packed; c - s is formed as fma(s, -1, c), the same single rounding of the same exact
// difference
__device__ __forceinline__ void round_cell2(float2 c, int kx, int ky, int& ix, int& iy, float2& rem)
{
    const float2 t = __fadd2_rn(c, bcast2(ROUND_MAGIC));
    rem = __ffma2_rn(__fadd2_rn(t, bcast2(-ROUND_MAGIC)), bcast2(-1.0f), c);
    ix = __float_as_int(t.x) - kx;
    iy = __float_as_int(t.y) - ky;
}

// Sphere vs field with certification.  Returns 1 = passes, 0 = fails, 2 = ambiguous.
//   (xy, z): the centre in grid coordinates c = inv_res (p - o) - 1, less K, so the reference's cell
//   (int)(inv_res (p - o) + 0.5) - 1 is round(c) and the cell boundaries are the half-integers (for c < -1/2 both
//   are outside the grid); K is whole, so rem and the boundaries are the same for c - K.  c is within eps of a
//   boundary iff |rem| > lim = 1/2 - eps; an exact tie (|rem| = 1/2, rounded to either side) is one of those, and the
//   near branch then evaluates the cells on both sides of it.  build_model32 admits a model only if |K| < 2^21 and
//   every centre the kernels evaluate has |c - K| < 2^21, so round_cell is exact for all of them, the index does not
//   overflow, and an out-of-grid centre keeps its out-of-grid index and reads d2 = 0 as in the reference.
__device__ __forceinline__ int lookup32(const uint16_t* __restrict__ df, const Grid32& G, float lim,
                                        float2 xy, float z, int thresh)
{
    int ix, iy;
    float2 rxy;
    float rz;
    round_cell2(xy, G.kx, G.ky, ix, iy, rxy);
    const int iz = round_cell(z, G.kz, rz);
    const float rx = rxy.x, ry = rxy.y;
    const bool near = (fabsf(rx) > lim) | (fabsf(ry) > lim) | (fabsf(rz) > lim);
    if (!near) {
        int d2 = 0;
        if ((unsigned)ix < (unsigned)G.nx && (unsigned)iy < (unsigned)G.ny && (unsigned)iz < (unsigned)G.nz) {
            d2 = (int)__ldg(&df[(ix * G.ny + iy) * G.nz + iz]);   // fields have fewer than 2^31 cells
        }
        return d2 >= thresh ? 1 : 0;
    }
    // every cell the double-precision coordinate could fall in
    const int x0 = ix - (rx < -lim ? 1 : 0), x1 = ix + (rx > lim ? 1 : 0);
    const int y0 = iy - (ry < -lim ? 1 : 0), y1 = iy + (ry > lim ? 1 : 0);
    const int z0 = iz - (rz < -lim ? 1 : 0), z1 = iz + (rz > lim ? 1 : 0);
    bool any_pass = false, any_fail = false;
    for (int cx = x0; cx <= x1; ++cx) {
        for (int cy = y0; cy <= y1; ++cy) {
            for (int cz = z0; cz <= z1; ++cz) {
                int d2 = 0;
                if ((unsigned)cx < (unsigned)G.nx && (unsigned)cy < (unsigned)G.ny && (unsigned)cz < (unsigned)G.nz) {
                    d2 = (int)__ldg(&df[(cx * G.ny + cy) * G.nz + cz]);
                }
                if (d2 >= thresh) any_pass = true; else any_fail = true;
            }
        }
    }
    return (any_pass && any_fail) ? 2 : (any_pass ? 1 : 0);
}

// val with its low 29 mantissa bits cleared: 24 significant bits, so exact in float (below 2^-126 float drops less than
// 2^-149 of it), and val minus it is exact in double, so hi = (float)hi_part(val), lo = (float)(val - hi_part(val))
// keep the angle to ~2^-47 with one DADD and two conversions (|lo| < 2^-23 |val|; a prismatic joint drops lo)
__device__ __forceinline__ double hi_part(double val)
{
    return __hiloint2double(__double2hiint(val), __double2loint(val) & (int)0xE0000000u);
}

// shared-memory view of the blob
struct S32
{
    const Model32Header* h;
    const int4* link_i;
    const int2* link_n;
    const float* origin;
    const float4* axis;
    const float* base;
    const float4* node_c;
    const int4* node_i;
    const int4* pair;
    const int2* allowed;
    const int* node_orig;
};

__device__ __forceinline__ S32 view32(const float* blob)
{
    S32 s;
    const Model32Header* h = reinterpret_cast<const Model32Header*>(blob);
    s.h = h;
    s.link_i = reinterpret_cast<const int4*>(blob + h->off_link_i);
    s.link_n = reinterpret_cast<const int2*>(blob + h->off_link_n);
    s.origin = blob + h->off_origin;
    s.axis = reinterpret_cast<const float4*>(blob + h->off_axis);
    s.base = blob + h->off_base;
    s.node_c = reinterpret_cast<const float4*>(blob + h->off_node_c);
    s.node_i = reinterpret_cast<const int4*>(blob + h->off_node_i);
    s.pair = reinterpret_cast<const int4*>(blob + h->off_pair);
    s.allowed = reinterpret_cast<const int2*>(blob + h->off_allowed);
    s.node_orig = reinterpret_cast<const int*>(blob + h->off_node_orig);
    return s;
}

__device__ __forceinline__ void copy_blob(float* dst, const float* __restrict__ src, int words)
{
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (int i = threadIdx.x; i < words / 4; i += blockDim.x) {
        d4[i] = __ldg(&s4[i]);
    }
}

// How a kernel tests sphere-tree pairs (build_model32 picks the mode per robot: Model32Header::n_ptrees > 0 is
// roots-only).  The two hot kernels are compiled for the mode they run in, so the roots-only form carries neither the
// descent nor its stack; the other callers read the mode at run time.
enum PairMode { PAIRS_RUNTIME, PAIRS_ROOTS, PAIRS_DESCENT };

// Forward kinematics of link l in single precision: joint transform J(q), T = T_parent J, kept in the link's slot when
// a later link branches from it.  `T` holds the previous link's transform on entry and this link's on exit.
// Returns false, with T unchanged, when the joint value is beyond what the error bound covers (|angle| > V32_MAX_ANGLE,
// |q| > q_lin_max of a prismatic joint, NaN): the double-precision path decides those.
//   INTERP: the joint value is qa + alpha (qb - qa), continuous variables along the shortest arc (qb = nullptr: qa);
//   else qa.  var_type: SMPLGPU_VAR_* per planning variable
template <bool INTERP>
__device__ __forceinline__ bool link_fk32(const S32& S, const int* __restrict__ var_type, const double* __restrict__ qa,
                                          const double* __restrict__ qb, double alpha, float* slots, int l, Xf32& T)
{
    const Model32Header* H = S.h;
    const int4 li = S.link_i[l];   // parent, fn, var, slot
    const int fn = li.y;
    float sn = 0.0f, cs = 1.0f, lin = 0.0f;
    if (li.z >= 0) {
        double val = qa[li.z];
        if (INTERP && qb != nullptr) {
            const double a = val, b = qb[li.z];
            const double diff = (var_type[li.z] == 1) ? normalize_angle(b - a) : (b - a);
            val = a + alpha * diff;
        }
        const double h = hi_part(val);
        const float hi = (float)h;
        if (fn == 5) {
            if (!(fabsf(hi) <= H->q_lin_max)) {
                return false;
            }
            lin = hi;
        } else {
            if (!(fabsf(hi) <= V32_MAX_ANGLE)) {
                return false;   // also catches NaN / inf
            }
            const float lo = (float)(val - h);
            float s0, c0;
            sincosf(hi, &s0, &c0);
            sn = fmaf(lo, c0, s0);
            cs = fmaf(-lo, s0, c0);
        }
    }
    Xf32 O, J;
    load12(S.origin + 12 * l, O);
    if (fn == 0) {
        J = O;
    } else if (fn <= 3) {
        // rotation about x (1), y (2), z (3): two columns of the origin's rotation mix; rows 0 and 1 packed, row 2
        // scalar, (-sn) o = -(sn o) exactly
        const float nsn = -sn;
        J = O;
        if (fn == 1) {
            J.c[1] = vfma(cs, O.c[1], vmul(sn, O.c[2]));
            J.c[2] = vfma(cs, O.c[2], vmul(nsn, O.c[1]));
            J.r2[1] = vfma(cs, O.r2[1], vmul(sn, O.r2[2]));
            J.r2[2] = vfma(cs, O.r2[2], vmul(nsn, O.r2[1]));
        } else if (fn == 2) {
            J.c[0] = vfma(cs, O.c[0], vmul(nsn, O.c[2]));
            J.c[2] = vfma(sn, O.c[0], vmul(cs, O.c[2]));
            J.r2[0] = vfma(cs, O.r2[0], vmul(nsn, O.r2[2]));
            J.r2[2] = vfma(sn, O.r2[0], vmul(cs, O.r2[2]));
        } else {
            J.c[0] = vfma(cs, O.c[0], vmul(sn, O.c[1]));
            J.c[1] = vfma(cs, O.c[1], vmul(nsn, O.c[0]));
            J.r2[0] = vfma(cs, O.r2[0], vmul(sn, O.r2[1]));
            J.r2[1] = vfma(cs, O.r2[1], vmul(nsn, O.r2[0]));
        }
    } else if (fn == 4) {
        const float4 ax = S.axis[l];
        const float k = 1.0f - cs;
        const float cx = k * ax.x, cy = k * ax.y, cz = k * ax.z;
        Xf32 A;
        A.c[0] = make_float2(fmaf(cx, ax.x, cs), fmaf(cx, ax.y, sn * ax.z));
        A.c[1] = make_float2(fmaf(cx, ax.y, -sn * ax.z), fmaf(cy, ax.y, cs));
        A.c[2] = make_float2(fmaf(cx, ax.z, sn * ax.y), fmaf(cy, ax.z, -sn * ax.x));
        A.c[3] = make_float2(0.0f, 0.0f);
        A.r2[0] = fmaf(cx, ax.z, -sn * ax.y); A.r2[1] = fmaf(cy, ax.z, sn * ax.x); A.r2[2] = fmaf(cz, ax.z, cs); A.r2[3] = 0.0f;
        xf32_mul(O, A, J);
    } else {
        const float4 ax = S.axis[l];   // inv_res * third column of the origin
        J = O;   // origin * Translate(0, 0, q): translation += third column * q, in cells
        J.c[3] = vfma(lin, make_float2(ax.x, ax.y), O.c[3]);
        J.r2[3] = vfma(lin, ax.z, O.r2[3]);
    }
    Xf32 P;
    if (li.x < 0) {
        load12(S.base + 12 * l, P);
    } else if (li.x == l - 1) {
        P = T;
    } else {
        slot32_load(slots, S.link_i[li.x].w, P);
    }
    xf32_mul(P, J, T);
    if (li.w >= 0) {
        slot32_store(slots, li.w, T);
    }
    return true;
}

// One link of one state in single precision: link_fk32, then the sphere trees riding on the link.
// Returns 1 = go on with the next link, 0 = certainly invalid, 2 = needs double precision right away; `amb` collects
// undecidable tests.
template <bool INTERP, int PM>
__device__ __forceinline__ int link_step32(const S32& S, const int* __restrict__ var_type, const uint16_t* __restrict__ df,
                                           const Grid32& G, const double* __restrict__ qa, const double* __restrict__ qb,
                                           double alpha, float* slots, int l, Xf32& T, bool& amb, Counters& cnt)
{
    const Model32Header* H = S.h;
    if (!link_fk32<INTERP>(S, var_type, qa, qb, alpha, slots, l, T)) {
        return 2;
    }
    const float lim = 0.5f - H->eps_cells;
    const bool save_roots = PM == PAIRS_ROOTS || (PM == PAIRS_RUNTIME && H->n_ptrees > 0);
    // sphere trees riding on this link: stackless pre-order descent
    const int2 nr = S.link_n[l];
    int node = nr.x;
    while (node < nr.y) {
        const float4 c = S.node_c[node];
        const int4 ni = S.node_i[node];   // skip, thresh, pair-tree index, -
        float2 xy;
        float z;
        xf32_point(T, c.x, c.y, c.z, xy, z);
        if (save_roots && ni.z >= 0) {
            // root of a tree that takes part in pair tests: keep its centre
            float* o = slots + ((size_t)H->n_slots * 12 + (size_t)ni.z * 3) * blockDim.x + threadIdx.x;
            o[0] = xy.x; o[blockDim.x] = xy.y; o[2 * blockDim.x] = z;
        }
        ++cnt.lookups;
        const int r = lookup32(df, G, lim, xy, z, ni.y);
        if (r == 1) {
            node = ni.x;
        } else if (r == 2) {
            amb = true;       // undecidable here: do not descend, let double precision decide unless a
            node = ni.x;      // certain collision shows up elsewhere
        } else if (ni.x == node + 1) {
            return 0;         // failing leaf below certainly failing ancestors
        } else {
            ++node;
        }
    }
    return 1;
}

// The sphere-tree pairs of one state whose link chain is done (transforms / root centres in `slots`).
// Returns 1 = certainly valid, 0 = certainly invalid, 2 = needs double precision.
__device__ __forceinline__ int pairs32_roots(const S32& S, float* slots, bool amb, Counters& cnt)
{
    const Model32Header* H = S.h;
    const int np = H->n_pairs;
    // Sphere-tree pairs: only the root spheres are tested here, from the root centres saved above.  Roots that
    // are certainly apart prune the pair, which is what happens in all but a handful of states; a pair of
    // overlapping single-sphere trees is a certain collision; anything else (overlapping roots that need the
    // descent, or an undecidable distance) goes to the double-precision kernel, which keeps the link
    // transforms the descent needs.
    const float* rp = slots + (size_t)H->n_slots * 12 * blockDim.x + threadIdx.x;
    for (int pi = 0; pi < np; ++pi) {
        const int4 pr = S.pair[pi];   // pair-tree index a, b; root node a, b
        const float* pa = rp + (size_t)pr.x * 3 * blockDim.x;
        const float* pb = rp + (size_t)pr.y * 3 * blockDim.x;
        const float dx = pb[0] - pa[0], dy = pb[blockDim.x] - pa[blockDim.x], dz = pb[2 * blockDim.x] - pa[2 * blockDim.x];
        ++cnt.pairs;
        const float cd2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
        const float rr = S.node_c[pr.z].w + S.node_c[pr.w].w;
        const float rr2 = rr * rr;
        const float tol = fmaf(H->pair_k, sqrtf(cd2) + rr, 2e-6f * (cd2 + rr2));
        const float d = cd2 - rr2;
        if (d > tol) {
            continue;
        }
        const int4 i1 = S.node_i[pr.z], i2 = S.node_i[pr.w];
        if (d < -tol && i1.x == pr.z + 1 && i2.x == pr.w + 1) {
            bool allowed = false;
            for (int k = 0; k < H->n_allowed; ++k) {
                const int2 al = S.allowed[k];
                allowed |= (al.x == pr.z && al.y == pr.w) || (al.x == pr.w && al.y == pr.z);
            }
            if (!allowed) {
                return 0;
            }
            continue;
        }
        amb = true;
    }
    return amb ? 2 : 1;
}

__device__ __forceinline__ int pairs32_descent(const S32& S, float* slots, bool amb, Counters& cnt)
{
    const Model32Header* H = S.h;
    const int np = H->n_pairs;
    // Sphere-tree pairs, full descent (robots whose pair roots overlap often, e.g. two arms + torso): the
    // transforms of all links with paired trees are in the slots.
    int stack[MAX_TREE_DEPTH];
    for (int pi = 0; pi < np; ++pi) {
        int sp = 0;
        const int4 proots = S.pair[pi];
        stack[sp++] = (proots.z << 16) | proots.w;
        while (sp > 0) {
            const int packed = stack[--sp];
            const int n1 = packed >> 16, n2 = packed & 0xFFFF;
            const float4 c1 = S.node_c[n1], c2 = S.node_c[n2];
            const int4 i1 = S.node_i[n1], i2 = S.node_i[n2];
            Xf32 A;
            float2 xy1, xy2;
            float z1, z2;
            slot32_load(slots, i1.z, A);
            xf32_point(A, c1.x, c1.y, c1.z, xy1, z1);
            slot32_load(slots, i2.z, A);
            xf32_point(A, c2.x, c2.y, c2.z, xy2, z2);
            ++cnt.pairs;
            const float dx = xy2.x - xy1.x, dy = xy2.y - xy1.y, dz = z2 - z1;
            const float cd2 = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            const float rr = c1.w + c2.w;
            const float rr2 = rr * rr;
            const float tol = fmaf(H->pair_k, sqrtf(cd2) + rr, 2e-6f * (cd2 + rr2));
            const float d = cd2 - rr2;
            if (fabsf(d) <= tol) {
                amb = true;
                continue;
            }
            if (d > 0.0f) {
                continue;
            }
            const bool leaf1 = i1.x == n1 + 1, leaf2 = i2.x == n2 + 1;
            if (leaf1 && leaf2) {
                bool allowed = false;
                for (int k = 0; k < H->n_allowed; ++k) {
                    const int2 al = S.allowed[k];
                    allowed |= (al.x == n1 && al.y == n2) || (al.x == n2 && al.y == n1);
                }
                if (!allowed) {
                    return 0;
                }
                continue;
            }
            bool split1;
            if (leaf1) {
                split1 = false;
            } else if (leaf2) {
                split1 = true;
            } else {
                // the reference splits the larger sphere (r1 > r2 in double): compare the ranks of the
                // double radii, which the host computed, not the rounded radii
                split1 = i1.w > i2.w;
            }
            // children in pre-order: left = node + 1, right = skip(left)
            if (split1) {
                const int left = n1 + 1, right = S.node_i[left].x;
                stack[sp++] = (left << 16) | n2;
                stack[sp++] = (right << 16) | n2;
            } else {
                const int left = n2 + 1, right = S.node_i[left].x;
                stack[sp++] = (n1 << 16) | left;
                stack[sp++] = (n1 << 16) | right;
            }
        }
    }
    return amb ? 2 : 1;
}

template <int PM>
__device__ __forceinline__ int pairs32(const S32& S, float* slots, bool amb, Counters& cnt)
{
    if constexpr (PM == PAIRS_ROOTS) {
        return pairs32_roots(S, slots, amb, cnt);
    } else if constexpr (PM == PAIRS_DESCENT) {
        return pairs32_descent(S, slots, amb, cnt);
    } else {
        return S.h->n_ptrees > 0 ? pairs32_roots(S, slots, amb, cnt) : pairs32_descent(S, slots, amb, cnt);
    }
}

// One state in single precision.  Returns 1 = certainly valid, 0 = certainly invalid, 2 = needs double precision.
template <bool INTERP, int PM>
__device__ __forceinline__ int check_state32_t(const S32& S, const int* __restrict__ var_type,
                                               const uint16_t* __restrict__ df, const Grid32& G,
                                               const double* __restrict__ qa, const double* __restrict__ qb,
                                               double alpha, float* slots, Counters& cnt)
{
    Xf32 T;
    bool amb = false;
    const int nl = S.h->n_links;
    for (int l = 0; l < nl; ++l) {
        const int r = link_step32<INTERP, PM>(S, var_type, df, G, qa, qb, alpha, slots, l, T, amb, cnt);
        if (r != 1) {
            return r;
        }
    }
    return pairs32<PM>(S, slots, amb, cnt);
}

// the general form (the planner's kernels): a waypoint qa + alpha (qb - qa) (qb = nullptr: the state qa), either pair mode
__device__ int check_state32(const S32& S, const int* __restrict__ var_type, const uint16_t* __restrict__ df,
                             const Grid32& G, const double* __restrict__ qa, const double* __restrict__ qb,
                             double alpha, float* slots, Counters& cnt)
{
    return check_state32_t<true, PAIRS_RUNTIME>(S, var_type, df, G, qa, qb, alpha, slots, cnt);
}

// warp-aggregated append of item ids to the list of items that need double precision
__device__ __forceinline__ void append_uncertain(bool push, int item, int* __restrict__ list, int* __restrict__ count,
                                                 unsigned long long* stats)
{
    const unsigned m = __ballot_sync(0xffffffffu, push);
    if (m == 0) {
        return;
    }
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == (__ffs(m) - 1)) {
        base = atomicAdd(count, __popc(m));
        if (stats != nullptr) {
            atomicAdd(&stats[3], (unsigned long long)__popc(m));
        }
    }
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (push) {
        list[base + __popc(m & ((1u << lane) - 1u))] = item;
    }
}

// dynamic shared memory: blob | slots (n_slots * 12 * blockDim floats) | root centres (n_ptrees * 3 * blockDim floats)
//                        | edges: (blockDim + 1) offsets, blockDim ok, blockDim unc, blockDim counts
template <int PM>
__global__ void V32_STATES_BOUNDS
states_valid32_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                      const uint16_t* __restrict__ df, Grid32 G, const double* __restrict__ q, int n,
                      uint8_t* __restrict__ verdict, int* __restrict__ unc_list, int* __restrict__ unc_count,
                      unsigned long long* stats)
{
    extern __shared__ float4 smem4[];
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    __syncthreads();
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    Counters cnt = { 0u, 0u, 0u };
    // Persistent warps: the grid is one wave of resident blocks and every warp pulls 32 consecutive states at a time
    // from a global cursor (unc_count[1], zeroed with the count by the host).  A state check costs anything from one
    // sphere test to the whole chain; with one state per thread a block keeps its registers and shared memory until
    // its slowest warp is done, here a warp that finishes early simply takes the next 32 states.
    const int lane = threadIdx.x & 31;
    for (;;) {
        int base = 0;
        if (lane == 0) {
            base = atomicAdd(unc_count + 1, 32);
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n) {
            break;
        }
        const int i = base + lane;
        int r = 0;
        if (i < n) {
            ++cnt.waypoints;
            r = check_state32_t<false, PM>(S, M->var_type, df, G, q + (size_t)i * S.h->dof, nullptr, 0.0, slots, cnt);
            verdict[i] = r == 1 ? 1 : 0;
        }
        append_uncertain(i < n && r == 2, i, unc_list, unc_count, stats);
    }
    flush_counters(cnt, stats);
}

template <int PM>
__global__ void V32_EDGES_BOUNDS
edges_valid32_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                     const uint16_t* __restrict__ df, Grid32 G, const double* __restrict__ q0,
                     const double* __restrict__ q1, int n, uint8_t* __restrict__ verdict, int* __restrict__ counts,
                     int* __restrict__ unc_list, int* __restrict__ unc_count, unsigned long long* stats,
                     int* __restrict__ unc_mask)
{
    extern __shared__ float4 smem4[];
    __shared__ int s_cursor;   // next unclaimed (edge, waypoint) item of round B
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    const int tid = threadIdx.x;
    const int first = blockIdx.x * blockDim.x;
    const int i = first + tid;
    const int dof = M->dof;
    Counters cnt = { 0u, 0u, 0u };

    // waypoint count of this thread's edge, in double exactly as the reference computes it
    int count = 0;
    if (i < n) {
        const double* a = q0 + (size_t)i * dof;
        const double* b = q1 + (size_t)i * dof;
        double motion = 0.0;
        for (int v = 0; v < dof; ++v) {
            const int ty = M->var_type[v];
            double dist;
            if (ty == 1) {
                dist = fabs(normalize_angle(b[v] - a[v]));
                motion += M->var_weight[v] * dist;
            } else if (ty == 0) {
                dist = fabs(b[v] - a[v]);
                motion += M->var_weight[v] * dist;
            } else {
                dist = fabs(b[v] - a[v]);
                motion += dist;
            }
        }
        if (motion != 0.0) {
            count = max(2, (int)ceil(motion / 0.05) + 1);
        }
        if (counts != nullptr) {
            counts[i] = count;
        }
    }
    __syncthreads();   // blob copied
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    int* s_off = reinterpret_cast<int*>(slots + ((size_t)S.h->n_slots * 12 + (size_t)S.h->n_ptrees * 3) * blockDim.x);
    int* s_ok = s_off + blockDim.x + 1;
    int* s_unc = s_ok + blockDim.x;
    // Round A: every thread checks the first waypoint of its own edge (alpha = 0 is exactly q0), the one the
    // reference checks first too (collision_space.cpp:561-577), so an edge that starts in collision costs one
    // state check, not `count`.
    int ok = 1, unc = 0;
    if (count > 0) {
        ++cnt.waypoints;
        const int r = check_state32_t<true, PM>(S, M->var_type, df, G, q0 + (size_t)i * dof, q1 + (size_t)i * dof, 0.0,
                                                slots, cnt);
        ok = r != 0;
        unc = r == 2;
    }
    // Round B: the remaining waypoints of the surviving edges, flattened over the block
    const int rest = ok ? max(count - 1, 0) : 0;
    s_off[tid + 1] = rest;
    s_ok[tid] = ok;
    s_unc[tid] = unc;
    if (tid == 0) {
        s_off[0] = 0;
        s_cursor = 0;
    }
    __syncthreads();
    for (int d = 1; d < (int)blockDim.x; d <<= 1) {
        int add = 0;
        if (tid + 1 > d) {
            add = s_off[tid + 1 - d];
        }
        __syncthreads();
        s_off[tid + 1] += add;
        __syncthreads();
    }
    const int total = s_off[blockDim.x];
    int* s_cnt = s_unc + blockDim.x;     // waypoint count per edge of the block
    s_cnt[tid] = count;
    __syncthreads();

    // warps pull 32 consecutive items at a time from a block-wide cursor: a state check costs anything from one
    // sphere test to the whole chain, so a fixed stride leaves warps waiting at the final barrier
    const int lane = tid & 31;
    for (;;) {
        int base = 0;
        if (lane == 0) {
            base = atomicAdd(&s_cursor, 32);
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= total) {
            break;
        }
        const int item = base + lane;
        if (item < total) {
            int lo = 0, hi = blockDim.x;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_off[mid] <= item) {
                    lo = mid;
                } else {
                    hi = mid;
                }
            }
            const int e = lo;
            // early-out read; a stale 1 (another lane is just clearing it) only costs one redundant waypoint check
            if (*((volatile int*)&s_ok[e]) != 0) {
                const int w = item - s_off[e] + 1;               // waypoint 0 was round A
                const double inv = 1.0 / (double)(s_cnt[e] - 1); // m_waypoint_count_inv
                const double alpha = (double)w * inv;
                ++cnt.waypoints;
                const int r = check_state32_t<true, PM>(S, M->var_type, df, G, q0 + (size_t)(first + e) * dof,
                                                        q1 + (size_t)(first + e) * dof, alpha, slots, cnt);
                // several lanes may hold waypoints of one edge: atomics make the concurrent same-value writes a
                // defined (racecheck-clean) update; they only run on a failing / undecided waypoint
                if (r == 0) {
                    atomicAnd(&s_ok[e], 0);
                } else if (r == 2) {
                    atomicOr(&s_unc[e], 1 << min(w, 31));   // WHICH waypoints the double pass has to look at (31: "31 and up")
                }
            }
        }
    }
    __syncthreads();
    bool push = false;
    if (i < n) {
        verdict[i] = s_ok[tid] ? 1 : 0;
        push = s_ok[tid] && s_unc[tid];
        if (push && unc_mask != nullptr) {
            unc_mask[i] = s_unc[tid];
        }
    }
    append_uncertain(push, i, unc_list, unc_count, stats);
    flush_counters(cnt, stats);
}

// ---- batched persistent form of the edge kernel ----------------------------------------------------------------
// edges_valid32_kernel gives a block blockDim edges: ~300 round-B items for four warps, so every warp ends its block
// waiting up to one state check (a third of its round B) for the last puller, and the verdicts leave only after that
// barrier -- ncu (profiles/r02d_metrics.csv) counts 20 % of the stall samples at block barriers.  Here the grid is one
// wave of resident blocks that pull BATCHES of V32_EDGE_EPT * blockDim edges from a global cursor (unc_count[1]):
// round A is pulled 32 edges at a time too, the pool of round B is V32_EDGE_EPT times deeper (the wait for the last
// puller is the same one state check, now against V32_EDGE_EPT times the work), and there is no tail of half-empty
// blocks at the end of the grid.  Same verdicts, counts and undecided list (in a different order) as the form above.
#ifndef V32_EDGE_EPT_N
#define V32_EDGE_EPT_N 4
#endif
constexpr int V32_EDGE_EPT = V32_EDGE_EPT_N;
constexpr int EDGE_OK = 1 << 30, EDGE_UNC = 1 << 29, EDGE_COUNT = EDGE_UNC - 1;

__global__ void V32_BOUNDS
edges_valid32b_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                      const uint16_t* __restrict__ df, Grid32 G, const double* __restrict__ q0,
                      const double* __restrict__ q1, int n, uint8_t* __restrict__ verdict, int* __restrict__ counts,
                      int* __restrict__ unc_list, int* __restrict__ unc_count, unsigned long long* stats)
{
    extern __shared__ float4 smem4[];
    __shared__ int s_first;      // first edge of the batch
    __shared__ int s_cursor_a;   // next unclaimed edge of round A
    __shared__ int s_cursor;     // next unclaimed (edge, waypoint) item of round B
    __shared__ int s_wsum[32];
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int dof = M->dof;
    const int E = V32_EDGE_EPT * (int)blockDim.x;
    Counters cnt = { 0u, 0u, 0u };
    __syncthreads();   // blob copied
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    int* s_off = reinterpret_cast<int*>(slots + ((size_t)S.h->n_slots * 12 + (size_t)S.h->n_ptrees * 3) * blockDim.x);
    // per edge ONE word: waypoint count | EDGE_OK | EDGE_UNC (shared memory per block decides how many blocks an SM holds,
    // and these kernels live on resident warps)
    int* s_edge = s_off + E + 1;

    for (;;) {
        if (tid == 0) {
            s_first = atomicAdd(unc_count + 1, E);
            s_cursor_a = 0;
            s_cursor = 0;
            s_off[0] = 0;
        }
        __syncthreads();   // also: everyone is done with the previous batch's arrays
        const int first = s_first;
        if (first >= n) {
            break;
        }
        const int nb = min(E, n - first);

        // waypoint counts, in double exactly as the reference computes them
        for (int e = tid; e < E; e += blockDim.x) {
            int count = 0;
            if (e < nb) {
                const double* a = q0 + (size_t)(first + e) * dof;
                const double* b = q1 + (size_t)(first + e) * dof;
                double motion = 0.0;
                for (int v = 0; v < dof; ++v) {
                    const int ty = M->var_type[v];
                    double dist;
                    if (ty == 1) {
                        dist = fabs(normalize_angle(b[v] - a[v]));
                        motion += M->var_weight[v] * dist;
                    } else if (ty == 0) {
                        dist = fabs(b[v] - a[v]);
                        motion += M->var_weight[v] * dist;
                    } else {
                        dist = fabs(b[v] - a[v]);
                        motion += dist;
                    }
                }
                if (motion != 0.0) {
                    count = max(2, (int)ceil(motion / 0.05) + 1);
                }
                if (counts != nullptr) {
                    counts[first + e] = count;
                }
            }
            s_edge[e] = count | EDGE_OK;
            s_off[e + 1] = 0;
        }
        __syncthreads();

        // Round A: the first waypoint of every edge (alpha = 0 is exactly q0), the one the reference checks first too
        // (collision_space.cpp:561-577), so an edge that starts in collision costs one state check, not `count`
        for (;;) {
            int base = 0;
            if (lane == 0) {
                base = atomicAdd(&s_cursor_a, 32);
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= nb) {
                break;
            }
            const int e = base + lane;
            const int count = e < nb ? (s_edge[e] & EDGE_COUNT) : 0;
            if (count > 0) {
                ++cnt.waypoints;
                const int r = check_state32(S, M->var_type, df, G, q0 + (size_t)(first + e) * dof,
                                            q1 + (size_t)(first + e) * dof, 0.0, slots, cnt);
                s_edge[e] = count | (r != 0 ? EDGE_OK : 0) | (r == 2 ? EDGE_UNC : 0);
                s_off[e + 1] = r != 0 ? count - 1 : 0;
            }
        }
        __syncthreads();

        // inclusive scan of the survivors' remaining waypoints: V32_EDGE_EPT consecutive entries per thread
        {
            int v[V32_EDGE_EPT];
            int sum = 0;
#pragma unroll
            for (int k = 0; k < V32_EDGE_EPT; ++k) {
                sum += s_off[1 + tid * V32_EDGE_EPT + k];
                v[k] = sum;
            }
            int x = sum;
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) {
                    x += y;
                }
            }
            if (lane == 31) {
                s_wsum[warp] = x;
            }
            __syncthreads();
            int woff = 0;
            for (int w = 0; w < warp; ++w) {
                woff += s_wsum[w];
            }
            const int excl = woff + x - sum;
#pragma unroll
            for (int k = 0; k < V32_EDGE_EPT; ++k) {
                s_off[1 + tid * V32_EDGE_EPT + k] = excl + v[k];
            }
        }
        __syncthreads();
        const int total = s_off[E];

        // Round B: the remaining waypoints of the surviving edges, flattened over the batch, 32 consecutive items per pull
        for (;;) {
            int base = 0;
            if (lane == 0) {
                base = atomicAdd(&s_cursor, 32);
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= total) {
                break;
            }
            const int item = base + lane;
            if (item < total) {
                int lo = 0, hi = E;
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (s_off[mid] <= item) {
                        lo = mid;
                    } else {
                        hi = mid;
                    }
                }
                const int e = lo;
                // early-out read; a stale 1 (another lane is just clearing it) only costs one redundant waypoint check
                const int word = *((volatile int*)&s_edge[e]);
                if (word & EDGE_OK) {
                    const int w = item - s_off[e] + 1;               // waypoint 0 was round A
                    const double inv = 1.0 / (double)((word & EDGE_COUNT) - 1); // m_waypoint_count_inv
                    const double alpha = (double)w * inv;
                    ++cnt.waypoints;
                    const int r = check_state32(S, M->var_type, df, G, q0 + (size_t)(first + e) * dof,
                                                q1 + (size_t)(first + e) * dof, alpha, slots, cnt);
                    if (r == 0) {
                        atomicAnd(&s_edge[e], ~EDGE_OK);
                    } else if (r == 2) {
                        atomicOr(&s_edge[e], EDGE_UNC);
                    }
                }
            }
        }
        __syncthreads();
        for (int e = tid; e < E; e += blockDim.x) {
            bool push = false;
            if (e < nb) {
                const int word = s_edge[e];
                verdict[first + e] = (word & EDGE_OK) ? 1 : 0;
                push = (word & EDGE_OK) && (word & EDGE_UNC);
            }
            append_uncertain(push, first + e, unc_list, unc_count, stats);
        }
    }
    flush_counters(cnt, stats);
}

// ---- lane-persistent form -------------------------------------------------------------------------------------
// In the kernels above a lane whose state dies at link 3 idles until the slowest lane of its warp has walked the
// whole chain: ncu counted 14 (states) / 19 (edges) active lanes per issued instruction.  Here the link index is
// DATA, not control flow: every lane runs one loop whose body is "process link l of my item", and a lane whose item
// is decided takes the next item from the cursor at the top of the same loop, while its neighbours are in the middle
// of theirs.  All lanes stay on one instruction stream (the loop body); what still diverges is the per-link joint
// kind, the length of a link's tree descent and the pair phase of the survivors.
//
//   cursor, n_items   the pool (global for the state kernel, the block's for the edge kernel)
//   item_fn(i, qa, qb, alpha) -> false to skip item i (its edge is already known to be invalid)
//   live_fn(i)        polled once per link: false abandons the item (another lane just invalidated its edge)
//   done_fn(fin, i, r)  called by ALL lanes once per loop iteration: fin = this lane's item i was decided now with
//                     result r (1 valid, 0 invalid, 2 undecided)
template <class ItemFn, class LiveFn, class DoneFn>
__device__ __forceinline__ void persistent_items32(const S32& S, const int* __restrict__ var_type,
                                                   const uint16_t* __restrict__ df, const Grid32& G, float* slots,
                                                   int* cursor, int n_items, ItemFn item_fn, LiveFn live_fn, DoneFn done_fn,
                                                   Counters& cnt)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int nl = S.h->n_links;
    int item = -1, l = 0;
    bool amb = false, exhausted = false;
    const double* qa = nullptr;
    const double* qb = nullptr;
    double alpha = 0.0;
    Xf32 T;
    for (;;) {
        const unsigned need = __ballot_sync(FULL, item < 0 && !exhausted);
        if (need != 0u) {
            const int leader = __ffs(need) - 1;
            int base = 0;
            if (lane == leader) {
                base = atomicAdd(cursor, __popc(need));
            }
            base = __shfl_sync(FULL, base, leader);
            if (item < 0 && !exhausted) {
                const int mine = base + __popc(need & ((1u << lane) - 1u));
                if (mine < n_items) {
                    if (item_fn(mine, qa, qb, alpha)) {
                        item = mine;
                        l = 0;
                        amb = false;
                        ++cnt.waypoints;
                    }
                } else {
                    exhausted = true;
                }
            }
        }
        if (__all_sync(FULL, item < 0)) {
            if (__all_sync(FULL, exhausted)) {
                break;
            }
            done_fn(false, 0, 0);
            continue;
        }
        bool fin = false;
        int res = 0;
        const int cur = item;
        if (item >= 0) {
            if (!live_fn(item)) {
                item = -1;                       // abandoned: its edge is invalid anyway, nothing to report
            } else {
                int r = link_step32<true, PAIRS_RUNTIME>(S, var_type, df, G, qa, qb, alpha, slots, l, T, amb, cnt);
                if (r == 1 && ++l == nl) {
                    r = pairs32<PAIRS_RUNTIME>(S, slots, amb, cnt);
                    fin = true;
                    res = r;
                } else if (r != 1) {
                    fin = true;
                    res = r;
                }
                if (fin) {
                    item = -1;
                }
            }
        }
        done_fn(fin, cur, res);
    }
}

__global__ void __launch_bounds__(V32_THREADS)
states_valid32p_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                       const uint16_t* __restrict__ df, Grid32 G, const double* __restrict__ q, int n,
                       uint8_t* __restrict__ verdict, int* __restrict__ unc_list, int* __restrict__ unc_count,
                       unsigned long long* stats)
{
    extern __shared__ float4 smem4[];
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    __syncthreads();
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    Counters cnt = { 0u, 0u, 0u };
    const int dof = S.h->dof;
    persistent_items32(
        S, M->var_type, df, G, slots, unc_count + 1, n,
        [&](int i, const double*& qa, const double*& qb, double& alpha) {
            qa = q + (size_t)i * dof;
            qb = nullptr;
            alpha = 0.0;
            return true;
        },
        [](int) { return true; },
        [&](bool fin, int i, int r) {
            if (fin) {
                verdict[i] = r == 1 ? 1 : 0;
            }
            append_uncertain(fin && r == 2, i, unc_list, unc_count, stats);
        },
        cnt);
    flush_counters(cnt, stats);
}

// Edges, lane-persistent: a block takes EPB = V32P_EDGES_PER_THREAD * blockDim edges.  Round A checks the first
// waypoint of every edge (the reference's first check: an edge that starts in collision costs one state check),
// round B the remaining waypoints of the survivors; both rounds hand their items to the lanes one at a time.
constexpr int V32P_EDGES_PER_THREAD = 4;

__global__ void __launch_bounds__(V32_THREADS)
edges_valid32p_kernel(const float* __restrict__ blob_g, int blob_words, const DevModel* __restrict__ M,
                      const uint16_t* __restrict__ df, Grid32 G, const double* __restrict__ q0,
                      const double* __restrict__ q1, int n, uint8_t* __restrict__ verdict, int* __restrict__ counts,
                      int* __restrict__ unc_list, int* __restrict__ unc_count, unsigned long long* stats)
{
    extern __shared__ float4 smem4[];
    __shared__ int s_cursor[2];
    __shared__ int s_warp_tot[V32_THREADS / 32];
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    const int tid = threadIdx.x;
    const int epb = V32P_EDGES_PER_THREAD * (int)blockDim.x;
    const int first = blockIdx.x * epb;
    const int dof = M->dof;
    Counters cnt = { 0u, 0u, 0u };
    __syncthreads();   // blob copied
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    // per-edge block state behind the per-thread slots: offsets (epb + 1), ok, unc, waypoint counts
    int* s_off = reinterpret_cast<int*>(slots + ((size_t)S.h->n_slots * 12 + (size_t)S.h->n_ptrees * 3) * blockDim.x);
    int* s_ok = s_off + epb + 1;
    int* s_unc = s_ok + epb;
    int* s_cnt = s_unc + epb;

    // waypoint counts, in double exactly as the reference computes them
    for (int e = tid; e < epb; e += blockDim.x) {
        const int i = first + e;
        int count = 0;
        if (i < n) {
            const double* a = q0 + (size_t)i * dof;
            const double* b = q1 + (size_t)i * dof;
            double motion = 0.0;
            for (int v = 0; v < dof; ++v) {
                const int ty = M->var_type[v];
                double dist;
                if (ty == 1) {
                    dist = fabs(normalize_angle(b[v] - a[v]));
                    motion += M->var_weight[v] * dist;
                } else if (ty == 0) {
                    dist = fabs(b[v] - a[v]);
                    motion += M->var_weight[v] * dist;
                } else {
                    dist = fabs(b[v] - a[v]);
                    motion += dist;
                }
            }
            if (motion != 0.0) {
                count = max(2, (int)ceil(motion / 0.05) + 1);
            }
            if (counts != nullptr) {
                counts[i] = count;
            }
        }
        s_cnt[e] = count;
        s_ok[e] = 1;
        s_unc[e] = 0;
    }
    if (tid == 0) {
        s_cursor[0] = 0;
        s_cursor[1] = 0;
    }
    __syncthreads();

    // Round A: waypoint 0 (alpha = 0 is exactly q0) of every edge that has waypoints
    persistent_items32(
        S, M->var_type, df, G, slots, &s_cursor[0], epb,
        [&](int e, const double*& qa, const double*& qb, double& alpha) {
            if (s_cnt[e] == 0) {
                return false;
            }
            qa = q0 + (size_t)(first + e) * dof;
            qb = q1 + (size_t)(first + e) * dof;
            alpha = 0.0;
            return true;
        },
        [](int) { return true; },
        [&](bool fin, int e, int r) {
            if (fin) {
                s_ok[e] = r != 0;       // one item per edge in this round: no other writer
                s_unc[e] = r == 2;
            }
        },
        cnt);
    __syncthreads();

    // Round B: the remaining waypoints of the surviving edges, flattened (exclusive scan of the per-edge rests)
    {
        int rest[V32P_EDGES_PER_THREAD];
        int mine = 0;
#pragma unroll
        for (int k = 0; k < V32P_EDGES_PER_THREAD; ++k) {
            const int e = tid * V32P_EDGES_PER_THREAD + k;
            rest[k] = s_ok[e] ? max(s_cnt[e] - 1, 0) : 0;
            mine += rest[k];
        }
        const int lane = tid & 31, warp = tid >> 5;
        int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) {
            s_warp_tot[warp] = incl;
        }
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; ++w) base += s_warp_tot[w];
        int off = base + incl - mine;
#pragma unroll
        for (int k = 0; k < V32P_EDGES_PER_THREAD; ++k) {
            s_off[tid * V32P_EDGES_PER_THREAD + k] = off;
            off += rest[k];
        }
        if (tid == (int)blockDim.x - 1) {
            s_off[epb] = off;
        }
        __syncthreads();
    }
    const int total = s_off[epb];
    auto edge_of = [&](int item) {
        int lo = 0, hi = epb;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (s_off[mid] <= item) {
                lo = mid;
            } else {
                hi = mid;
            }
        }
        return lo;
    };
    // the edge of a lane's current item (items are handed out once, so the lookup is done at pull time)
    int my_edge = 0;
    persistent_items32(
        S, M->var_type, df, G, slots, &s_cursor[1], total,
        [&](int item, const double*& qa, const double*& qb, double& alpha) {
            const int e = edge_of(item);
            if (*((volatile int*)&s_ok[e]) == 0) {
                return false;             // its edge died meanwhile
            }
            my_edge = e;
            const int w = item - s_off[e] + 1;                      // waypoint 0 was round A
            const double inv = 1.0 / (double)(s_cnt[e] - 1);       // m_waypoint_count_inv
            alpha = (double)w * inv;
            qa = q0 + (size_t)(first + e) * dof;
            qb = q1 + (size_t)(first + e) * dof;
            return true;
        },
        [&](int) { return *((volatile int*)&s_ok[my_edge]) != 0; },
        [&](bool fin, int, int r) {
            if (fin) {
                if (r == 0) {
                    atomicAnd(&s_ok[my_edge], 0);
                } else if (r == 2) {
                    atomicOr(&s_unc[my_edge], 1);
                }
            }
        },
        cnt);
    __syncthreads();
    for (int e = tid; e < epb; e += blockDim.x) {
        const int i = first + e;
        bool push = false;
        if (i < n) {
            verdict[i] = s_ok[e] ? 1 : 0;
            push = s_ok[e] && s_unc[e];
        }
        append_uncertain(push, i, unc_list, unc_count, stats);
    }
    flush_counters(cnt, stats);
}

// sphere centres as the single-precision path computes them (original node order), for the error-bound test; the
// model's coordinates c - K are mapped back to metres in double (x = (c - K) res + o', o' = o + (K + 1) res), so the
// error is the model's, times res
__global__ void __launch_bounds__(V32_THREADS)
fk_centers32_kernel(const float* __restrict__ blob_g, int blob_words, const double* __restrict__ q, int n,
                    double res, double ox, double oy, double oz, float* __restrict__ out)
{
    extern __shared__ float4 smem4[];
    float* blob = reinterpret_cast<float*>(smem4);
    copy_blob(blob, blob_g, blob_words);
    __syncthreads();
    const S32 S = view32(blob);
    float* slots = blob + blob_words;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) {
        return;
    }
    const Model32Header* H = S.h;
    const double* qa = q + (size_t)i * H->dof;
    Xf32 T;
    for (int l = 0; l < H->n_links; ++l) {
        if (!link_fk32<false>(S, nullptr, qa, nullptr, 0.0, slots, l, T)) {
            // a joint value the bound does not cover: the kernels leave this state to double precision
            for (int k = 0; k < 3 * H->n_nodes; ++k) {
                out[(size_t)i * H->n_nodes * 3 + k] = __int_as_float(0x7fffffff);
            }
            return;
        }
        const int2 nr = S.link_n[l];
        for (int node = nr.x; node < nr.y; ++node) {
            const float4 c = S.node_c[node];
            float2 xy;
            float z;
            xf32_point(T, c.x, c.y, c.z, xy, z);
            float* o = out + ((size_t)i * H->n_nodes + S.node_orig[node]) * 3;
            o[0] = (float)((double)xy.x * res + ox);
            o[1] = (float)((double)xy.y * res + oy);
            o[2] = (float)((double)z * res + oz);
        }
    }
}

} // namespace smplgpu
