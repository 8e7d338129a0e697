// Ray / scene intersection on the device: primitive roots, point membership, CSG programs and the
// brute-force closest-hit loop of Universe::trace_closest (src/universe/mod.rs:85-147).
//
// The reference evaluates CSG with lazily pulled iterator objects (shape.rs:204-497).  Here each
// CSG program (post-order node list) is evaluated EAGERLY by a small stack machine: every node
// produces its hit list "up to the first None", which is exactly the prefix a parent can ever
// observe because a cached None is never stepped over (util.rs:395-419).  Hits are kept compact
// -- (t, primitive, flags) -- and locations / normals are recomputed from the primitive when
// needed, with the same expressions the reference uses, so results are bit-identical.
#pragma once
#include "scene_dev.cuh"
#include "vecmath.cuh"

namespace EUCL_NS {
using namespace eucl;

#ifndef EUCL_CSG_ARENA
#define EUCL_CSG_ARENA 256
#endif
constexpr int CSG_ARENA = EUCL_CSG_ARENA;     // compact hits per thread (scene_create validates programs against it)
constexpr int CSG_LIST_STACK = 16; // nesting depth of pending child lists
constexpr int CHAIN_ROOT_CAP = 32; // hits of a chain that is an entity's whole shape (<= 16 leaves)

struct CHit {
    real t;
    int prim;
    int flags; // bit 0: second root of the primitive; bit 1: normal negated (Complement / SymDiff)
};

// Roots of a*t^2 + b*t + c with the reference's selection of non-negative roots
// (shape.rs:672-694 sphere, :969-991 cylinder).  Returns the number of hits.
__device__ __forceinline__ int quadratic_hits(real a, real b, real c, real& t_first, real& t_second) {
    real disc = b * b - R(4.0) * a * c;
    if (disc < R(0.0)) return 0;
    real d_sqrt = sqrt(disc);
    real t1 = (-b - d_sqrt) / (R(2.0) * a);
    real t2 = (-b + d_sqrt) / (R(2.0) * a);
    if (t1 >= R(0.0)) {
        t_first = t1;
        if (t2 >= R(0.0)) {
            t_second = t2;
            return 2;
        }
        return 1;
    }
    if (t2 >= R(0.0)) {
        t_first = t2;
        return 1;
    }
    return 0;
}

// Parametric distances at which the ray meets primitive `prim` (sorted, t >= 0 only).
template <int D>
__device__ __forceinline__ int prim_roots(const SceneView& sv, int prim, const Vec<D>& o, const Vec<D>& d, real& t0,
                                          real& t1) {
    const int n = sv.n_prims;
    const int kind = sv.prim_kind()[prim];
    const double* __restrict__ rec = sv.planes() + (size_t)prim * kPlaneStride; // AoS: [v0[0..3], s0, s1]
    if (kind == EUCL_PRIM_SPHERE) { // shape.rs:662-670
        Vec<D> center = load_vec<D>(rec, 1);
        real radius = R(rec[4]);
        Vec<D> rel = o - center;
        real a = norm_squared(d);
        real b = R(2.0) * dot(d, rel);
        real c = norm_squared(rel) - radius * radius;
        return quadratic_hits(a, b, c, t0, t1);
    }
    if (kind == EUCL_PRIM_HYPERPLANE || kind == EUCL_PRIM_HALFSPACE) { // shape.rs:788-793
        Vec<D> nrm = load_vec<D>(rec, 1);
        real t = -(dot(nrm, o) + R(rec[4])) / dot(nrm, d);
        if (t < R(0.0)) return 0; // NaN and +inf pass, exactly like the reference
        t0 = t;
        return 1;
    }
    if (kind == EUCL_PRIM_CYLINDER) { // shape.rs:946-953
        Vec<D> center = load_vec<D>(rec, 1);
        Vec<D> axis = load_vec<D>(sv.prim_v1() + prim, n);
        real radius = R(rec[4]);
        Vec<D> a_vec = d - axis * dot(d, axis);
        Vec<D> delta = o - center;
        Vec<D> c_vec = delta - axis * dot(delta, axis);
        real a = norm_squared(a_vec);
        real b = (R(1.0) + R(1.0)) * dot(a_vec, c_vec);
        real c = norm_squared(c_vec) - radius * radius;
        return quadratic_hits(a, b, c, t0, t1);
    }
    return 0; // VoidShape: shape.rs:622-631
}

// Shape::is_point_inside of one primitive (shape.rs:614-619,734-738,812-817,873-881,1030-1038)
template <int D>
__device__ __forceinline__ bool prim_inside(const SceneView& sv, int prim, const Vec<D>& p) {
    const int n = sv.n_prims;
    const int kind = sv.prim_kind()[prim];
    const double* __restrict__ rec = sv.planes() + (size_t)prim * kPlaneStride;
    if (kind == EUCL_PRIM_HALFSPACE) {
        real r = dot(load_vec<D>(rec, 1), p) + R(rec[4]);
        return R(rec[5]) == rust_signum(r);
    }
    if (kind == EUCL_PRIM_SPHERE) {
        real radius = R(rec[4]);
        return norm_squared(load_vec<D>(rec, 1) - p) <= radius * radius;
    }
    if (kind == EUCL_PRIM_CYLINDER) {
        Vec<D> center = load_vec<D>(rec, 1);
        Vec<D> axis = load_vec<D>(sv.prim_v1() + prim, n);
        real radius = R(rec[4]);
        Vec<D> on_axis = axis * dot(axis, p - center) + center;
        return norm_squared(p - on_axis) <= radius * radius;
    }
    return kind == EUCL_PRIM_VOID; // hyperplane: never inside
}

// ---------------------------------------------------------------------------------------------
// Macro CSG programs.  The host (api_device.cu: build_macro_program) rewrites each entity's
// post-order node list into macro nodes:
//   M_PRIM  : one primitive
//   M_CHAIN : a maximal left fold  ((l0 op l1) op l2) ... op l(n-1)  of n LEAF primitives with
//             op = Intersection or Union and consecutive primitive indices (cuboid, hypercuboid,
//             capped cylinder, wall sets ...), evaluated by one tight loop
//   M_OP    : any other binary node, merging the lists of its two children
// Evaluation order and every comparison are those of the nested binary iterators, so results are
// identical; only the bookkeeping differs.
enum : int { M_PRIM = 0, M_CHAIN = 1, M_OP = 2 };
struct MNode {
    int32_t kind;
    int32_t a;     // PRIM: primitive; CHAIN: first primitive; OP: EuclCsgOp
    int32_t b;     // CHAIN: count | 0x4000 if every leaf is a half-space with signum +-1 | (EuclCsgOp << 16)
    int32_t first; // first macro node of this subtree (post-order; children of OP n: b = n-1, a = mnodes[n-1].first-1)
};

// is_point_inside of a chain prefix: nested `&&` / `||` over pure operands = all / any
template <int D>
__device__ __forceinline__ bool chain_inside(const SceneView& sv, int op, int p0, int count, const Vec<D>& p) {
    for (int k = 0; k < count; ++k) {
        const bool in = prim_inside<D>(sv, p0 + k, p);
        if (op == EUCL_CSG_INTERSECTION) {
            if (!in) return false;
        } else if (in) {
            return true;
        }
    }
    return op == EUCL_CSG_INTERSECTION;
}

// ComposableShape::is_point_inside (shape.rs:587-601) of macro node `n`: a bit stack over the
// macro post-order range (all operands are pure, so no short-circuit is needed between siblings).
template <int D>
__device__ __noinline__ bool node_inside(const SceneView& sv, int n, EUCL_VARG(Vec<D>) p) {
    const MNode* mn = reinterpret_cast<const MNode*>(sv.nodes());
    const MNode root = mn[n];
    if (root.kind == M_PRIM) return prim_inside<D>(sv, root.a, p);
    if (root.kind == M_CHAIN) return chain_inside<D>(sv, root.b >> 16, root.a, root.b & 0x3fff, p);
    unsigned long long bits = 0ull;
    int sp = 0;
    for (int m = root.first; m <= n; ++m) {
        const MNode nd = mn[m];
        if (nd.kind != M_OP) {
            const bool in = nd.kind == M_PRIM ? prim_inside<D>(sv, nd.a, p)
                                              : chain_inside<D>(sv, nd.b >> 16, nd.a, nd.b & 0x3fff, p);
            bits |= (unsigned long long)(in ? 1 : 0) << sp;
            ++sp;
        } else {
            const bool b = (bits >> (sp - 1)) & 1ull, a = (bits >> (sp - 2)) & 1ull;
            const bool r = nd.a == EUCL_CSG_UNION ? (a || b)
                           : nd.a == EUCL_CSG_INTERSECTION ? (a && b)
                           : nd.a == EUCL_CSG_COMPLEMENT ? (a && !b)
                                                         : (a != b);
            sp -= 2;
            bits &= ~(3ull << sp);
            bits |= (unsigned long long)(r ? 1 : 0) << sp;
            ++sp;
        }
    }
    return bits & 1ull;
}

// Universe::material_at (mod.rs:229-251): first entity in list order containing the point
template <int D>
__device__ __noinline__ int material_at(const SceneView& sv, EUCL_VARG(Vec<D>) p) {
    for (int e = 0; e < sv.n_entities; ++e) {
        const int root = sv.entities()[e].node_root;
        if (sv.ent_flags()[e] & ENT_NEGATED) { // Complement(VoidShape, X): true && !X (shape.rs:596); X's bound says nothing here
            if (!node_inside<D>(sv, root, p)) return e;
            continue;
        }
        // a point outside the (inflated) bounding sphere of the shape cannot be inside it; NaN -> not skipped
        const Bound& bnd = sv.bounds()[root];
        if (R(bnd.r2) >= R(0.0)) {
            real dist2 = R(0.0);
#pragma unroll
            for (int k = 0; k < D; ++k) dist2 += (p[k] - R(bnd.c[k])) * (p[k] - R(bnd.c[k]));
            if (dist2 > R(bnd.r2)) continue;
        }
        if (node_inside<D>(sv, root, p)) return e;
    }
    return -1;
}

// Ray / bounding-sphere rejection.  A macro node's Bound (built on the host, inflated by 1e-6)
// contains every point its shape can contain, hence every hit its stream can emit: an emitted hit
// is a boundary point of the shape -- it was tested inside all sibling leaves -- up to rounding of
// ~1e-13, far inside the inflation.  If the half-line o + t d, t >= 0, stays outside the sphere,
// the node's hit list is empty and the whole evaluation is skipped.  NaN anywhere makes every
// comparison false: such rays are never culled and take the exact path.
template <int D>
__device__ __forceinline__ bool ray_misses(const Bound& bnd, const Vec<D>& o, const Vec<D>& d, real dd) {
    if (!(R(bnd.r2) >= R(0.0))) return false;
    Vec<D> rel;
#pragma unroll
    for (int k = 0; k < D; ++k) rel[k] = o[k] - R(bnd.c[k]);
    const real b = dot(d, rel);
    const real c = dot(rel, rel) - R(bnd.r2);
    return (b * b - dd * c < R(0.0)) || (c > R(0.0) && b > R(0.0));
}

// Reach key of a ray: which of the scene's bounded, non-trivial entities its half-line can reach.
// Rays with equal keys take the same branches in closest_hit, so the rays of a level are walked
// grouped by this key (kernels.cu).  Purely an ordering hint: results do not depend on it.
template <int D>
__device__ __forceinline__ int reach_key(const SceneView& sv, const Vec<D>& o, const Vec<D>& d) {
    const real dd = dot(d, d);
    int key = 0;
    for (int k = 0; k < sv.n_cull; ++k)
        if (!ray_misses<D>(sv.bounds()[sv.cull_root[k]], o, d, dd)) key |= 1 << k;
    return key;
}

// Hit list of a chain macro node, "up to the first None", written to L (capacity cap; T is scratch
// of the same size).  Step k merges the list so far (stream A) with the hits of leaf k (stream B)
// exactly like IntersectionIterator / UnionIterator (shape.rs:212-340):
//   both streams non-empty : take the closer one (ties and NaN -> b); a rejected hit is skipped
//   one stream exhausted   : take from the other; a rejected hit ends the list (None)
// A hit of A is tested against leaf k, a hit of B against the prefix l0..l(k-1).
template <int D>
__device__ __forceinline__ int chain_eval(const SceneView& sv, int op, int p0, int count, const Vec<D>& o, const Vec<D>& d,
                                          CHit* L, CHit* T, int cap, bool first_only) {
    real t0 = R(0.0), t1 = R(0.0);
    int n = prim_roots<D>(sv, p0, o, d, t0, t1);
    if (n > 0) L[0] = CHit{t0, p0, 0};
    if (n > 1) L[1] = CHit{t1, p0, 1};
    for (int k = 1; k < count; ++k) {
        const int prim = p0 + k;
        const int nb = prim_roots<D>(sv, prim, o, d, t0, t1);
        const int limit = (first_only && k == count - 1) ? 1 : cap;
        int ia = 0, ib = 0, m = 0;
        while (m < limit) {
            const bool has_a = ia < n, has_b = ib < nb;
            if (!has_a && !has_b) break;
            const real tb = ib == 0 ? t0 : t1;
            CHit h;
            bool in;
            if (has_a && (!has_b || L[ia].t < tb)) {
                h = L[ia++];
                in = prim_inside<D>(sv, prim, o + d * h.t);
            } else {
                h = CHit{tb, prim, ib};
                ++ib;
                in = chain_inside<D>(sv, op, p0, k, o + d * h.t);
            }
            if (op == EUCL_CSG_INTERSECTION ? in : !in) T[m++] = h;
            else if (!(has_a && has_b)) break;
        }
        for (int i = 0; i < m; ++i) L[i] = T[i];
        n = m;
    }
    return n;
}

// Membership rows of G consecutive hit points of a plane chain against all N planes.
template <int D, int G>
__device__ __forceinline__ void plane_rows(const double* __restrict__ rec, int N, const Vec<D>& o, const Vec<D>& d,
                                           const real* ts, int ts_stride, int i0, unsigned long long& inside) {
    Vec<D> p[G];
    unsigned rows[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const int i = min(i0 + g, N - 1); // padding lanes of the last group repeat a valid point
        p[g] = d * ts[i * ts_stride] + o;
        rows[g] = 0u;
    }
#pragma unroll 1
    for (int j = 0; j < N; ++j) {
        const double* r = rec + j * kPlaneStride;
        Vec<D> nrm;
#pragma unroll
        for (int k = 0; k < D; ++k) nrm[k] = R(r[k]);
        const real c = R(r[4]);
        const bool s_neg = r[5] < R(0.0);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const real v = dot(nrm, p[g]) + c;
            const bool in = !isnan(v) && (sign_negative(v) == s_neg);
            rows[g] |= (in ? 1u : 0u) << j;
        }
    }
    const unsigned all = (1u << N) - 1u;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const int i = i0 + g;
        if (i < N) inside |= (unsigned long long)(rows[g] & all & ~(1u << i)) << (i * N); // never against itself
    }
}

// Chain of N <= 8 half-space leaves (one hit each, signum = +-1) -- cuboids (6), hypercuboids and
// 8-plane rooms (8), wall sets (4).  Same merge as chain_eval, organised for the GPU:
//   * all floating-point work (N roots, N*(N-1) membership tests) runs in ROLLED loops with tiny
//     bodies: the first version of this kernel executed ~80 KB of distinct SASS per ray and was
//     instruction-fetch bound (profiles/: stall_no_instruction); loop trip counts are identical
//     for every lane, so nothing diverges;
//   * the data-dependent list bookkeeping then runs on integer bit masks; root parameters live in
//     a per-thread shared-memory scratch column (ts[i * ts_stride]) because the loops index them
//     dynamically.
// The list is a packed array of 4-bit leaf indices.  Returns the list length.
constexpr int kPlaneChainMax = 8;
template <int D>
__device__ __forceinline__ int plane_chain(const SceneView& sv, int op, int p0, int N, const Vec<D>& o, const Vec<D>& d,
                                           bool first_only, real* ts, int ts_stride, unsigned long long& list_out) {
    const double* __restrict__ rec = sv.planes() + (size_t)p0 * kPlaneStride;
    unsigned exists = 0u;
#pragma unroll 1
    for (int i = 0; i < N; ++i) { // Hyperplane::intersect_linear, shape.rs:788-793
        const double* r = rec + i * kPlaneStride;
        Vec<D> nrm;
#pragma unroll
        for (int k = 0; k < D; ++k) nrm[k] = R(r[k]);
        const real t = -(dot(nrm, o) + R(r[4])) / dot(nrm, d);
        ts[i * ts_stride] = t;
        if (!(t < R(0.0))) exists |= 1u << i; // NaN and +inf pass
    }
    const bool want_in = op == EUCL_CSG_INTERSECTION;
    // (whole lists only in 4-D, where a hypercuboid's table is 8 x 7 tests.  For 3-D boxes (6 x 5) both ways of adding it were
    // measured and lost on 3d_room's heavy intersect kernel: inlined 6.75 -> 6.94 ms of code shape, out of line 6.84 -> 7.12 ms
    // of call overhead; profiles/README.md)
    if (first_only || D >= 4) {
        // Shortcut.  Let m be the existing hit whose distance is STRICTLY smaller than every other existing one (no NaN
        // anywhere), and let it pass the membership test against every other leaf (outside all of them for a Union, inside
        // all for an Intersection).  Then m is the FIRST item of the folded list: it enters the fold as `b` at its own step,
        // where it is closer than every item of the list so far and is tested against the fold of the earlier leaves; at
        // every later step it is the head of `a`, closer than the new `b`, and is tested against that one leaf.  Each of
        // these tests is one of the N - 1 evaluated here, so m is emitted first every time.  An entity's whole shape only
        // ever yields its first item (mod.rs:110-112): done.  Inside a CSG program the whole list is needed; every item
        // of the folded list has passed the test against ALL other leaves, so if every OTHER existing hit fails the test
        // against leaf m alone, the list is exactly [m].  That is the case of a ray that starts inside a box (or outside
        // every member of a union): one row and one column of the membership table instead of all of it, no replay.
        // Anything else -- ties, NaN, a rejected m, another surviving candidate -- takes the general evaluation below.
        int m = -1;
        real tm = R(0.0);
        bool clean = true;
#pragma unroll 1
        for (int i = 0; i < N; ++i) {
            if (!((exists >> i) & 1u)) continue;
            const real t = ts[i * ts_stride];
            if (isnan(t)) clean = false;
            if (m < 0 || t < tm) {
                m = i;
                tm = t;
            }
        }
        if (m < 0) { // no leaf is hit at all
            list_out = 0ull;
            return 0;
        }
        if (clean) {
            const Vec<D> pm = d * tm + o;
            bool ok = true;
#pragma unroll 1
            for (int j = 0; j < N; ++j) { // no early exit: the loop stays branch-free (the hot callers pass all N - 1 tests)
                const double* r = rec + j * kPlaneStride;
                Vec<D> nrm;
#pragma unroll
                for (int k = 0; k < D; ++k) nrm[k] = R(r[k]);
                const real v = dot(nrm, pm) + R(r[4]);
                const bool in = !isnan(v) && (sign_negative(v) == (r[5] < 0.0));
                const bool tie = j != m && ((exists >> j) & 1u) && !(tm < ts[j * ts_stride]);
                if (j != m && (in != want_in || tie)) ok = false;
            }
            if (ok && !first_only) { // column m: every other existing hit against leaf m
                const double* r = rec + m * kPlaneStride;
                Vec<D> nrm;
#pragma unroll
                for (int k = 0; k < D; ++k) nrm[k] = R(r[k]);
                const real c = R(r[4]);
                const bool s_neg = r[5] < 0.0;
#pragma unroll 1
                for (int i = 0; i < N && ok; ++i) {
                    if (i == m || !((exists >> i) & 1u)) continue;
                    const Vec<D> pi = d * ts[i * ts_stride] + o;
                    const real v = dot(nrm, pi) + c;
                    const bool in = !isnan(v) && (sign_negative(v) == s_neg);
                    ok = in != want_in; // rejected by leaf m: cannot be in the folded list
                }
            }
            if (ok) {
                list_out = (unsigned long long)m;
                return 1;
            }
        }
    }
    // inside bit (i, j): half-space j contains the hit point of leaf i (shape.rs:873-881):
    // signum == (n.p + c).signum(); Rust signum is +-1 by sign bit and NaN for NaN.
    // Hit points are processed in groups of G kept in registers while a rolled loop walks the
    // planes, so each plane record is loaded once per group and the loop body stays small.
    unsigned long long inside = 0ull;
    const unsigned all = (1u << N) - 1u;
    if (N % 3 == 0) {
        for (int i0 = 0; i0 < N; i0 += 3) plane_rows<D, 3>(rec, N, o, d, ts, ts_stride, i0, inside);
    } else {
        for (int i0 = 0; i0 < N; i0 += 4) plane_rows<D, 4>(rec, N, o, d, ts, ts_stride, i0, inside);
    }
    bool any = false;
#pragma unroll 1
    for (int i = 0; i < N; ++i) {
        const unsigned others = all & ~(1u << i);
        const unsigned row = (unsigned)(inside >> (i * N)) & others;
        any = any || (((exists >> i) & 1u) && (want_in ? row == others : row == 0u));
    }
    // Every item of the final list was tested against ALL other leaves on its way (as `b` against
    // the prefix, then as `a` against each later leaf) and kept only when inside (Intersection) /
    // outside (Union) each time.  If no existing hit has such a row the list is empty: most rays
    // miss most boxes and skip the replay.
    if (!any) {
        list_out = 0ull;
        return 0;
    }
    // integer replay of the N-1 merges (IntersectionIterator / UnionIterator, shape.rs:212-340)
    unsigned long long L = 0ull;
    int n = exists & 1u;
#pragma unroll 1
    for (int k = 1; k < N; ++k) {
        const unsigned prefix = (1u << k) - 1u;
        const unsigned mask_k = (unsigned)(inside >> (k * N)) & prefix;
        const bool b_in = want_in ? mask_k == prefix : mask_k != 0u; // inside the fold of leaves 0..k-1
        bool b_pending = (exists >> k) & 1u;
        const real tk = ts[k * ts_stride];
        const int limit = (first_only && k == N - 1) ? 1 : N;
        unsigned long long T = 0ull;
        int ia = 0, m = 0;
        while (m < limit && (ia < n || b_pending)) {
            const bool has_a = ia < n, both = has_a && b_pending;
            const unsigned a = (unsigned)(L >> (4 * ia)) & 15u;
            // `a.distance < b.distance`: ties and NaN take b
            const bool take_a = has_a && (!b_pending || ts[a * ts_stride] < tk);
            bool in;
            unsigned item;
            if (take_a) {
                item = a;
                in = (inside >> (a * N + k)) & 1ull;
                ++ia;
            } else {
                item = (unsigned)k;
                in = b_in;
                b_pending = false;
            }
            if (want_in ? in : !in) {
                T |= (unsigned long long)item << (4 * m);
                ++m;
            } else if (!both) {
                break; // None
            }
        }
        L = T;
        n = m;
    }
    list_out = L;
    return n;
}

// First item of the intersection stream of the macro program [first, root]
// (ComposableShape::intersect_linear + the four merge iterators, shape.rs:204-584).
template <int D>
__device__ __forceinline__ bool csg_first(const SceneView& sv, int first, int root, const Vec<D>& o, const Vec<D>& d,
                                          real* ts, int ts_stride, CHit& out) {
    const MNode* mn = reinterpret_cast<const MNode*>(sv.nodes());
    const real dd = dot(d, d);
    CHit arena[CSG_ARENA];
    int lstart[CSG_LIST_STACK], llen[CSG_LIST_STACK];
    int sp = 0, top = 0;
    for (int n = first; n <= root; ++n) {
        const MNode nd = mn[n];
        if (nd.kind == M_PRIM) {
            real t0 = R(0.0), t1 = R(0.0);
            const int c = prim_roots<D>(sv, nd.a, o, d, t0, t1);
            lstart[sp] = top;
            llen[sp] = c;
            ++sp;
            if (c > 0) arena[top++] = CHit{t0, nd.a, 0};
            if (c > 1) arena[top++] = CHit{t1, nd.a, 1};
            continue;
        }
        if (nd.kind == M_CHAIN) {
            const int count = nd.b & 0x3fff, cap = 2 * count;
            int c = 0;
            if (ray_misses<D>(sv.bounds()[n], o, d, dd)) {
                c = 0; // the chain's region is out of the ray's reach: empty list
            } else if ((nd.b & 0x4000) && count <= kPlaneChainMax) {
                unsigned long long L = 0ull;
                c = plane_chain<D>(sv, nd.b >> 16, nd.a, count, o, d, n == root, ts, ts_stride, L);
                if (first == root) { // the chain is the entity's whole shape: its first item is the answer
                    if (c == 0) return false;
                    const int idx = (int)(L & 15ull);
                    out = CHit{ts[idx * ts_stride], nd.a + idx, 0};
                    return true;
                }
                for (int i = 0; i < c; ++i) {
                    const int idx = (int)((L >> (4 * i)) & 15ull);
                    arena[top + i] = CHit{ts[idx * ts_stride], nd.a + idx, 0};
                }
            } else {
                c = chain_eval<D>(sv, nd.b >> 16, nd.a, count, o, d, arena + top, arena + top + cap, cap, n == root);
            }
            lstart[sp] = top;
            llen[sp] = c;
            ++sp;
            top += c;
            continue;
        }
        const int b0 = lstart[sp - 1], bl = llen[sp - 1], a0 = lstart[sp - 2], al = llen[sp - 2];
        sp -= 2;
        const int nb = n - 1, na = mn[n - 1].first - 1;
        const int op = nd.a;
        const int out0 = top;
        // The entity root only ever yields its first item (mod.rs:110-112); inner nodes are
        // bounded because a Complement with an exhausted `b` repeats `a` forever (shape.rs:392).
        const int limit = n == root ? 1 : min(al + bl + 2, CSG_ARENA - out0);
        int outn = 0, ia = 0, ib = 0;
        while (outn < limit) {
            const bool has_a = ia < al, has_b = ib < bl;
            if (!has_a && !has_b) break;
            CHit ha = arena[a0 + (has_a ? ia : 0)], hb = arena[b0 + (has_b ? ib : 0)];
            if (has_a && has_b) {
                const bool a_closer = ha.t < hb.t; // ties (and NaN) pick b
                if (op == EUCL_CSG_COMPLEMENT) {
                    if (a_closer) {
                        ++ia;
                        if (!node_inside<D>(sv, nb, o + d * ha.t)) arena[out0 + outn++] = ha;
                    } else {
                        ++ib;
                        if (node_inside<D>(sv, na, o + d * hb.t)) {
                            hb.flags ^= 2;
                            arena[out0 + outn++] = hb;
                        }
                    }
                } else {
                    CHit closer = a_closer ? ha : hb;
                    const int further = a_closer ? nb : na;
                    if (a_closer) ++ia;
                    else ++ib;
                    const bool in = node_inside<D>(sv, further, o + d * closer.t);
                    if (op == EUCL_CSG_UNION) {
                        if (!in) arena[out0 + outn++] = closer;
                    } else if (op == EUCL_CSG_INTERSECTION) {
                        if (in) arena[out0 + outn++] = closer;
                    } else { // SymmetricDifference: always yields, flipped when inside the other
                        if (in) closer.flags ^= 2;
                        arena[out0 + outn++] = closer;
                    }
                }
            } else if (has_a) {
                if (op == EUCL_CSG_COMPLEMENT) {
                    arena[out0 + outn++] = ha; // not advanced (reference quirk)
                    continue;
                }
                ++ia;
                const bool in = node_inside<D>(sv, nb, o + d * ha.t);
                if (op == EUCL_CSG_UNION) {
                    if (in) break; // None
                } else if (op == EUCL_CSG_INTERSECTION) {
                    if (!in) break;
                } else if (in) {
                    ha.flags ^= 2;
                }
                arena[out0 + outn++] = ha;
            } else {
                ++ib;
                const bool in = node_inside<D>(sv, na, o + d * hb.t);
                if (op == EUCL_CSG_UNION) {
                    if (in) break;
                } else if (op == EUCL_CSG_INTERSECTION) {
                    if (!in) break;
                } else if (op == EUCL_CSG_COMPLEMENT) {
                    if (!in) break;
                    hb.flags ^= 2;
                } else if (in) {
                    hb.flags ^= 2;
                }
                arena[out0 + outn++] = hb;
            }
        }
        for (int k = 0; k < outn; ++k) arena[a0 + k] = arena[out0 + k];
        top = a0 + outn;
        lstart[sp] = a0;
        llen[sp] = outn;
        ++sp;
    }
    if (llen[0] > 0) {
        out = arena[lstart[0]];
        return true;
    }
    return false;
}

// csg_first of a two-leaf program (ENT_CSG2): three macro nodes [A, B, M_OP(op)] at first .. first + 2, A a primitive or a
// chain of <= kPlaneChainMax half-spaces, B a primitive (3d_room's glass: Complement(cuboid, sphere)).  An exact
// restatement: A's list is what csg_first stores in its arena -- the same bound check and plane_chain call (whole list,
// distances in the scratch column `ts`, items as packed 4-bit leaf indices) or the same prim_roots -- and B's is prim_roots'
// two values; the merge is csg_first's M_OP branch at limit 1 step for step (ties and NaN pick b, the has_a-only quirk of
// Complement, the flag negations, the early ends), and node_inside of a leaf operand IS prim_inside / chain_inside, called
// here directly.  Same IEEE operations on the same operands in the same order; only the bookkeeping moves from the
// local-memory arena and the bit stack into registers, so a kernel built on this has no stack.
template <int D>
__device__ __forceinline__ bool csg2_first(const SceneView& sv, int first, const Vec<D>& o, const Vec<D>& d, real* ts,
                                           int ts_stride, CHit& out) {
    const MNode* mn = reinterpret_cast<const MNode*>(sv.nodes());
    const MNode na = mn[first], nb = mn[first + 1];
    const int op = mn[first + 2].a;
    const bool a_chain = na.kind == M_CHAIN;
    const int a_op = na.b >> 16, a_count = na.b & 0x3fff;
    int al = 0;
    real a0 = R(0.0), a1 = R(0.0);
    unsigned long long a_list = 0ull;
    if (!a_chain) {
        al = prim_roots<D>(sv, na.a, o, d, a0, a1);
    } else if (!ray_misses<D>(sv.bounds()[first], o, d, dot(d, d))) {
        al = plane_chain<D>(sv, a_op, na.a, a_count, o, d, false, ts, ts_stride, a_list);
    }
    real b0 = R(0.0), b1 = R(0.0);
    const int bl = prim_roots<D>(sv, nb.a, o, d, b0, b1);
    const auto a_hit = [&](int i) -> CHit {
        if (!a_chain) return CHit{i == 0 ? a0 : a1, na.a, i};
        const int idx = (int)((a_list >> (4 * i)) & 15ull);
        return CHit{ts[idx * ts_stride], na.a + idx, 0};
    };
    const auto inside_a = [&](const Vec<D>& p) {
        return a_chain ? chain_inside<D>(sv, a_op, na.a, a_count, p) : prim_inside<D>(sv, na.a, p);
    };
    int ia = 0, ib = 0;
    while (true) {
        const bool has_a = ia < al, has_b = ib < bl;
        if (!has_a && !has_b) return false;
        CHit ha = a_hit(has_a ? ia : 0);
        CHit hb{ib == 0 ? b0 : b1, nb.a, ib};
        if (has_a && has_b) {
            const bool a_closer = ha.t < hb.t; // ties (and NaN) pick b
            if (op == EUCL_CSG_COMPLEMENT) {
                if (a_closer) {
                    ++ia;
                    if (!prim_inside<D>(sv, nb.a, o + d * ha.t)) {
                        out = ha;
                        return true;
                    }
                } else {
                    ++ib;
                    if (inside_a(o + d * hb.t)) {
                        hb.flags ^= 2;
                        out = hb;
                        return true;
                    }
                }
            } else {
                CHit closer = a_closer ? ha : hb;
                if (a_closer) ++ia;
                else ++ib;
                const Vec<D> p = o + d * closer.t;
                const bool in = a_closer ? prim_inside<D>(sv, nb.a, p) : inside_a(p);
                if (op == EUCL_CSG_UNION) {
                    if (!in) {
                        out = closer;
                        return true;
                    }
                } else if (op == EUCL_CSG_INTERSECTION) {
                    if (in) {
                        out = closer;
                        return true;
                    }
                } else { // SymmetricDifference: always yields, flipped when inside the other
                    if (in) closer.flags ^= 2;
                    out = closer;
                    return true;
                }
            }
        } else if (has_a) {
            if (op == EUCL_CSG_COMPLEMENT) { // emitted without advancing (reference quirk): it is the first item
                out = ha;
                return true;
            }
            const bool in = prim_inside<D>(sv, nb.a, o + d * ha.t);
            if (op == EUCL_CSG_UNION) {
                if (in) return false; // None
            } else if (op == EUCL_CSG_INTERSECTION) {
                if (!in) return false;
            } else if (in) {
                ha.flags ^= 2;
            }
            out = ha;
            return true;
        } else {
            const bool in = inside_a(o + d * hb.t);
            if (op == EUCL_CSG_UNION) {
                if (in) return false; // None
            } else if (op == EUCL_CSG_INTERSECTION) {
                if (!in) return false;
            } else if (op == EUCL_CSG_COMPLEMENT) {
                if (!in) return false;
                hb.flags ^= 2;
            } else if (in) {
                hb.flags ^= 2;
            }
            out = hb;
            return true;
        }
    }
}

struct ClosestHit {
    int entity; // -1: no hit
    int prim;
    int flags;
    real t;
};

// trace_closest, distance part: every surfaced entity (including the one the ray is inside) is
// asked for the FIRST item of its stream; a candidate replaces the current one only if it is
// strictly closer (mod.rs:127-128), so a NaN distance wins only as the very first candidate.
template <int D>
__device__ __forceinline__ ClosestHit closest_hit(const SceneView& sv, const Vec<D>& o, const Vec<D>& d, real* ts,
                                                  int ts_stride) {
    ClosestHit best{-1, 0, 0, R(0.0)};
    const real dd = dot(d, d);
    for (int e = 0; e < sv.n_entities; ++e) {
        const EuclEntity ent = sv.entities()[e];
        if (ent.surface < 0) continue;
        CHit h;
        bool found;
        const MNode root = reinterpret_cast<const MNode*>(sv.nodes())[ent.node_root];
        if (root.kind != M_PRIM && ray_misses<D>(sv.bounds()[ent.node_root], o, d, dd)) continue; // no hit can come from this entity
        if (root.kind == M_PRIM) {
            real t0 = R(0.0), t1 = R(0.0);
            found = prim_roots<D>(sv, root.a, o, d, t0, t1) > 0;
            h = CHit{t0, root.a, 0};
        } else { // one call site: the evaluator (and the chain code inside it) exists once in the kernel
            found = csg_first<D>(sv, ent.node_first, ent.node_root, o, d, ts, ts_stride, h);
        }
        if (sv.ent_flags()[e] & ENT_NEGATED) h.flags ^= 2; // the `b`-only branch of ComplementIterator negates the normal
        if (found && (best.entity < 0 || best.t > h.t)) best = ClosestHit{e, h.prim, h.flags, h.t};
    }
    return best;
}

// trace_closest for rays whose reach key is 0 in a "light-capable" scene (SceneHeader::light_capable): every
// surfaced entity is one primitive, one root chain of half-spaces, or a cull root -- and a ray with key 0 stays
// outside the bound of every cull root, so those yield no hit (same argument as ray_misses) and are skipped
// without a test.  No general CSG evaluator, no hit arena: the kernel built on this keeps more warps resident.
template <int D>
__device__ __forceinline__ ClosestHit closest_hit_light(const SceneView& sv, const Vec<D>& o, const Vec<D>& d, real* ts,
                                                        int ts_stride) {
    ClosestHit best{-1, 0, 0, R(0.0)};
    for (int e = 0; e < sv.n_entities; ++e) {
        const int flags = sv.ent_flags()[e];
        if (!(flags & ENT_SURFACED) || (flags & ENT_CULL_ROOT)) continue;
        const MNode root = reinterpret_cast<const MNode*>(sv.nodes())[sv.entities()[e].node_root];
        real t0 = R(0.0), t1 = R(0.0);
        int prim = root.a;
        bool found;
        if (flags & ENT_PRIM) {
            found = prim_roots<D>(sv, root.a, o, d, t0, t1) > 0;
        } else { // ENT_ROOT_PLANES
            unsigned long long L = 0ull;
            found = plane_chain<D>(sv, root.b >> 16, root.a, root.b & 0x3fff, o, d, true, ts, ts_stride, L) > 0;
            const int idx = (int)(L & 15ull);
            t0 = ts[idx * ts_stride];
            prim = root.a + idx;
        }
        if (found && (best.entity < 0 || best.t > t0)) best = ClosestHit{e, prim, (flags & ENT_NEGATED) ? 2 : 0, t0};
    }
    return best;
}

// trace_closest in a "csg2-capable" scene (SceneHeader::csg2_capable): every surfaced entity is one primitive, one root
// chain of half-spaces or a two-leaf program, so closest_hit's loop runs with the light loop's root-chain shortcut and
// csg2_first in place of the general evaluator: no hit arena, no stack.  Everything closest_hit does around an entity
// stays: the bound check of every non-primitive root (a ray with some key bit set may still miss the other bounds), the
// ENT_NEGATED flip and the strictly-closer rule.
template <int D>
__device__ __forceinline__ ClosestHit closest_hit_csg2(const SceneView& sv, const Vec<D>& o, const Vec<D>& d, real* ts,
                                                       int ts_stride) {
    ClosestHit best{-1, 0, 0, R(0.0)};
    const real dd = dot(d, d);
    for (int e = 0; e < sv.n_entities; ++e) {
        const int flags = sv.ent_flags()[e];
        if (!(flags & ENT_SURFACED)) continue;
        const EuclEntity ent = sv.entities()[e];
        if (!(flags & ENT_PRIM) && ray_misses<D>(sv.bounds()[ent.node_root], o, d, dd)) continue;
        const MNode root = reinterpret_cast<const MNode*>(sv.nodes())[ent.node_root];
        CHit h{R(0.0), root.a, 0};
        bool found;
        if (flags & ENT_PRIM) {
            real t1 = R(0.0);
            found = prim_roots<D>(sv, root.a, o, d, h.t, t1) > 0;
        } else if (flags & ENT_ROOT_PLANES) {
            unsigned long long L = 0ull;
            found = plane_chain<D>(sv, root.b >> 16, root.a, root.b & 0x3fff, o, d, true, ts, ts_stride, L) > 0;
            const int idx = (int)(L & 15ull);
            h = CHit{ts[idx * ts_stride], root.a + idx, 0};
        } else { // ENT_CSG2
            found = csg2_first<D>(sv, ent.node_first, o, d, ts, ts_stride, h);
        }
        if (flags & ENT_NEGATED) h.flags ^= 2; // the `b`-only branch of ComplementIterator negates the normal
        if (found && (best.entity < 0 || best.t > h.t)) best = ClosestHit{e, h.prim, h.flags, h.t};
    }
    return best;
}

// Location and (raw) normal of a compact hit, as the primitive's intersector reports them
// (shape.rs:700-728 sphere, :795-806 plane, :858-861 half-space, :993-1024 cylinder).
template <int D>
__device__ __forceinline__ void hit_geometry(const SceneView& sv, int prim, int flags, const Vec<D>& o, const Vec<D>& d,
                                             real t, Vec<D>& p, Vec<D>& nrm) {
    const int n = sv.n_prims;
    const int kind = sv.prim_kind()[prim];
    if (kind == EUCL_PRIM_SPHERE) {
        p = o + d * t;
        nrm = normalize(p - load_vec<D>(sv.prim_v0() + prim, n));
    } else if (kind == EUCL_PRIM_CYLINDER) {
        Vec<D> center = load_vec<D>(sv.prim_v0() + prim, n);
        Vec<D> axis = load_vec<D>(sv.prim_v1() + prim, n);
        real t_first = t;
        if (flags & 1) { // the second hit reuses the axis point of the FIRST hit (shape.rs:999,1017)
            real r0 = R(0.0), r1 = R(0.0);
            prim_roots<D>(sv, prim, o, d, r0, r1);
            t_first = r0;
        }
        Vec<D> p1 = o + d * t_first;
        Vec<D> on_axis = axis * dot(axis, p1 - center) + center;
        p = o + d * t;
        nrm = normalize(p - on_axis);
    } else {
        p = d * t + o;
        nrm = load_vec<D>(sv.prim_v0() + prim, n);
        if (kind == EUCL_PRIM_HALFSPACE) nrm = nrm * -R(sv.prim_s1()[prim]);
    }
    if (flags & 2) nrm = -nrm;
}

} // namespace EUCL_NS
