// Device half of the C ABI (include/euclider_b200.h): scene upload, frame orchestration, IPC.
//
// eucl_render* is the drop-in for Environment::render (src/universe/mod.rs:300-357): it fans the
// pixels out to the GPU instead of a scoped thread pool and returns the same RGB8 buffer
// (row 0 = bottom).  There is no CPU rendering path here: without a usable CUDA device every
// entry point fails with EUCL_ERR_NO_DEVICE / EUCL_ERR_CUDA.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "error.h"
#include "euclider_b200.h"
#include "intersect.cuh"
#include "pipeline.cuh"
#include "scene_dev.cuh"

namespace {

using namespace eucl;

#define EUCL_CUDA(expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess)                                                                            \
            return fail(_e == cudaErrorMemoryAllocation ? EUCL_ERR_OUT_OF_MEMORY : EUCL_ERR_CUDA,         \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                              \
    } while (0)

// the launcher of the scene's precision: namespace eucl holds the f64 build of kernels.cu, eucl_f32 the f32 build
#define EUCL_PREC(fn) (s->real_bytes == 4 ? eucl_f32::fn : eucl::fn)

// pipelines a rank's share of a frame is rendered as (render_split); EUCL_SPLIT overrides
#ifndef EUCL_SPLIT_DEFAULT
#define EUCL_SPLIT_DEFAULT 2
#endif

int env_int(const char* name, int fallback) {
    const char* v = std::getenv(name);
    return v && *v ? std::atoi(v) : fallback;
}

struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    cudaError_t ensure(size_t want) {
        if (want <= bytes) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};

// One helper thread per split scene: runs the second pipeline's host side (enqueue, stream synchronise, retry loop)
// next to the caller's thread.  Kept alive between frames: waking it costs microseconds, creating it tens.
struct Worker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, done = false, quit = false;
    void start() {
        th = std::thread([this] {
            std::unique_lock<std::mutex> lk(m);
            for (;;) {
                cv.wait(lk, [this] { return has_job || quit; });
                if (quit) return;
                lk.unlock();
                job();
                lk.lock();
                has_job = false;
                done = true;
                cv.notify_all();
            }
        });
    }
    void run(std::function<void()> f) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(f);
        has_job = true;
        done = false;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [this] { return done; });
    }
    void stop() {
        if (!th.joinable()) return;
        {
            std::lock_guard<std::mutex> lk(m);
            quit = true;
            cv.notify_all();
        }
        th.join();
    }
};

} // namespace

struct EuclScene {
    int device = 0;
    int dim = 3;
    int sm_count = 148;
    int blob_bytes = 0;
    size_t smem_bytes = 0;  // staged scene + plane_chain scratch
    size_t smem_scene = 0;  // staged scene only
    unsigned long long shade_light_mask = 1ull, shade_heavy_mask = 0ull;
    uint8_t* d_blob = nullptr;
    std::vector<cudaArray_t> arrays;
    std::vector<cudaTextureObject_t> tex_objects;
    cudaStream_t stream = nullptr;     // the stream kernels run on (own_stream unless the caller set one)
    cudaStream_t own_stream = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    cudaStream_t side_stream = nullptr;                  // light builds of a level's kernels run here, next to the heavy ones
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::vector<cudaEvent_t> prof_events; // per-launch events, profile mode only
    // workspace (grow-only)
    DeviceBuffer nodes;    // the node arena
    DeviceBuffer small;    // counters
    DeviceBuffer frame;    // device frame buffer for eucl_render (host output)
    DeviceBuffer hit_ids;  // device hit-id map for eucl_render
    DeviceBuffer order;    // per-bin node lists of the level being shaded
    DeviceBuffer path_io;  // eucl_trace_path staging
    DeviceBuffer rorder;   // per-reach-key node lists of the next level
    // a batch of frames (eucl_render_frames*): the per-frame constants (leader only; its twins read them), their pinned
    // host staging, and per pipeline the frames' camera entities and the frame tag of every node
    DeviceBuffer frame_table;
    FrameParams* h_frame_table = nullptr;
    uint32_t h_frame_table_cap = 0;
    DeviceBuffer frame_entity;
    DeviceBuffer node_frame;
    DeviceBuffer node_cost; // (segments, levels) per node of this pipeline's arena: AOV renders that want either plane
    DeviceBuffer aov_stage; // device copies of the AOV planes for eucl_render_aovs (host output)
    DeviceBuffer ray_stage; // device copy of the rays of eucl_trace_rays (host input), refilled by every call
    int n_cull = 0;
    int light_capable = 0;
    // Grouping rays by reach key pays on scenes whose deep levels bounce around a few bounded objects
    // (3d_room: -13 % frame time) and costs a little elsewhere, so it is auto-tuned per scene: the
    // first two retry-free frames run with and without it, the faster setting is kept.  The picture
    // does not depend on it.  EUCL_BIN_RAYS=0/1 forces a setting.
    int ray_bins_mode = -1;      // -1 undecided, 0 off, 1 on
    bool ray_bins_now = true;    // setting of the frame being rendered
    float tune_ms[2] = {0.f, 0.f}; // fastest frame seen without / with grouping
    int tune_count[2] = {0, 0};    // frames measured without / with grouping
    uint64_t tune_pixels = 0;    // frame size the two timings belong to
    int warm_frames = 0;         // frames rendered so far
    int n_entities = 0;
    int real_bytes = 8;        // 8: f64 kernels (the reference's default `type F = f64`); 4: f32 kernels (`low_precision`)
    int arena_capacity = 0;
    double arena_factor = 0.0; // nodes per pixel the arena is sized for (learned from earlier frames)
    cudaGraphExec_t graph_exec = nullptr; // the last repeated chunk as a CUDA graph (render_impl)
    uint64_t graph_key = 0, seen_key = 0; // parameter hash of graph_exec / of the previous direct launch sequence
    uint32_t graph_launches = 0;
    int list_capacity = 0;     // entries per index list (bins, reach keys): the largest LEVEL a chunk may have
    double list_factor = 1.0;  // ... in nodes per pixel (level 0 has exactly one; deeper levels are smaller in every shipped scene)
    int32_t* h_small = nullptr; // pinned mirror of the counters
    // Further pipelines of a split frame (render_split): scenes of their own -- streams, arena, counters, graph --
    // over the same uploaded blob and textures, each rendering every k-th band next to this one.
    std::vector<EuclScene*> twins;
    std::vector<Worker*> workers; // one host thread per twin
    bool is_twin = false;
    cudaEvent_t ev_split[3] = {nullptr, nullptr, nullptr}; // start (timed), fork, end (timed)
    cudaEvent_t ev_done = nullptr;                         // twin: its part of the frame is on its stream
};

namespace {

constexpr int kSmallInts = 4 * (EUCL_MAX_LEVELS + 1) + 16 + (EUCL_MAX_LEVELS + 1) * (kMaxBins + kRayBins); // count, level_off, flags, bins
struct SmallLayout {                                        // one per chunk, in ints
    static constexpr int count = 0;
    static constexpr int level_off = EUCL_MAX_LEVELS + 1;
    static constexpr int overflow = 2 * (EUCL_MAX_LEVELS + 1);
    static constexpr int cam_entity = overflow + 1;
    static constexpr int undefined64 = overflow + 2;                  // 8-byte aligned (even index)
    static constexpr int mega64 = undefined64 + 2;                    // (EUCL_MAX_LEVELS + 1) x u64
    static constexpr int bins = mega64 + 2 * (EUCL_MAX_LEVELS + 1);       // [level][kMaxBins]
    static constexpr int rbins = bins + (EUCL_MAX_LEVELS + 1) * kMaxBins; // [level][kRayBins]
    static constexpr int untraced = rbins + (EUCL_MAX_LEVELS + 1) * kRayBins; // Workspace::untraced
    static constexpr int total = untraced + 1;
};
static_assert(SmallLayout::undefined64 % 2 == 0, "u64 counters must be 8-byte aligned");
static_assert(SmallLayout::total <= kSmallInts, "small buffer layout");

size_t align16(size_t v) { return (v + 15) & ~size_t(15); }

// Validation of a caller-built flat scene: every cross-table index, opcode and program that the
// device code dereferences without checks.  EUCL_ERR_INVALID_ARGUMENT for malformed tables,
// EUCL_ERR_SCENE_LIMIT for well-formed programs that exceed a fixed device stack (shade.cuh:
// kExprStackMax, kColorStackMax).
int validate_scene(const EuclFlatScene& f, std::string* why) {
    auto bad = [&](const std::string& msg) {
        *why = msg;
        return (int)EUCL_ERR_INVALID_ARGUMENT;
    };
    const int counts[] = {f.n_prims, f.n_nodes, f.n_entities, f.n_materials, f.n_transforms, f.n_expr_ops,
                          f.n_surfaces, f.n_color_ops, f.n_mapped_textures, f.n_textures};
    for (int c : counts)
        if (c < 0) return bad("negative table size");
    if ((f.n_prims && !f.prims) || (f.n_nodes && !f.nodes) || (f.n_entities && !f.entities) || (f.n_materials && !f.materials) ||
        (f.n_transforms && !f.transforms) || (f.n_expr_ops && !f.expr_ops) || (f.n_surfaces && !f.surfaces) ||
        (f.n_color_ops && !f.color_ops) || (f.n_mapped_textures && !f.mapped_textures) || (f.n_textures && !f.textures))
        return bad("null table with a non-zero size");
    for (int i = 0; i < f.n_prims; ++i)
        if (f.prims[i].kind < EUCL_PRIM_VOID || f.prims[i].kind > EUCL_PRIM_CYLINDER)
            return bad("primitive " + std::to_string(i) + ": unknown kind");
    for (int e = 0; e < f.n_entities; ++e) {
        const EuclEntity& ent = f.entities[e];
        if (ent.node_first < 0 || ent.node_root >= f.n_nodes || ent.node_first > ent.node_root)
            return bad("entity " + std::to_string(e) + ": node range out of bounds");
        if (ent.material < 0 || ent.material >= f.n_materials) return bad("entity " + std::to_string(e) + ": material index out of bounds");
        if (ent.surface < -1 || ent.surface >= f.n_surfaces) return bad("entity " + std::to_string(e) + ": surface index out of bounds");
        int depth = 0;
        for (int n = ent.node_first; n <= ent.node_root; ++n) {
            const EuclNode& nd = f.nodes[n];
            if (nd.op == EUCL_CSG_LEAF) {
                if (nd.prim < 0 || nd.prim >= f.n_prims) return bad("node " + std::to_string(n) + ": primitive index out of bounds");
                ++depth;
            } else {
                if (nd.op < EUCL_CSG_UNION || nd.op > EUCL_CSG_SYMDIFF || depth < 2 || nd.first < ent.node_first || nd.first >= n)
                    return bad("node " + std::to_string(n) + ": malformed post-order program");
                --depth;
            }
        }
        if (depth != 1) return bad("entity " + std::to_string(e) + ": CSG program does not reduce to one shape");
    }
    // expression programs: operand counts and the peak depth of the device's evaluation stack
    auto check_expr = [&](int first, int len, const std::string& what, int* status) {
        if (first < 0 || len < 0 || (long long)first + len > f.n_expr_ops) {
            *status = bad(what + ": expression range out of bounds");
            return;
        }
        int sp = 0, peak = 0;
        for (int i = first; i < first + len; ++i) {
            const EuclExprOp& o = f.expr_ops[i];
            int pops = 0;
            switch (o.op) {
            case EUCL_EX_CONST: break;
            case EUCL_EX_VAR:
                if (o.arg < 0 || o.arg >= f.dim) {
                    *status = bad(what + ": variable index out of range");
                    return;
                }
                break;
            case EUCL_EX_NEG: pops = 1; break;
            case EUCL_EX_FUNC1:
                if (o.arg < EUCL_FN_SQRT || o.arg > EUCL_FN_SIGNUM) {
                    *status = bad(what + ": unknown unary function");
                    return;
                }
                pops = 1;
                break;
            case EUCL_EX_FUNC2:
                if (o.arg < EUCL_FN_ATAN2 || o.arg > EUCL_FN_MIN) {
                    *status = bad(what + ": unknown binary function");
                    return;
                }
                pops = 2;
                break;
            case EUCL_EX_ADD: case EUCL_EX_SUB: case EUCL_EX_MUL: case EUCL_EX_DIV: case EUCL_EX_REM: case EUCL_EX_POW:
                pops = 2;
                break;
            default: *status = bad(what + ": unknown expression opcode"); return;
            }
            if (sp < pops) {
                *status = bad(what + ": expression stack underflow");
                return;
            }
            sp = sp - pops + 1;
            peak = std::max(peak, sp);
        }
        if (len > 0 && sp != 1) {
            *status = bad(what + ": expression does not reduce to one value");
            return;
        }
        if (peak > kExprStackMax) {
            *why = what + ": expression needs " + std::to_string(peak) + " stack slots, the device evaluator has " +
                   std::to_string(kExprStackMax);
            *status = EUCL_ERR_SCENE_LIMIT;
        }
    };
    for (int m = 0; m < f.n_materials; ++m) {
        const EuclMaterial& mat = f.materials[m];
        if (mat.kind != EUCL_MAT_VACUUM && mat.kind != EUCL_MAT_LINEAR_SPACE) return bad("material " + std::to_string(m) + ": unknown kind");
        if (mat.kind == EUCL_MAT_LINEAR_SPACE &&
            (mat.transform_first < 0 || mat.n_transforms < 0 || (long long)mat.transform_first + mat.n_transforms > f.n_transforms))
            return bad("material " + std::to_string(m) + ": transformation range out of bounds");
    }
    for (int t = 0; t < f.n_transforms; ++t)
        for (int k = 0; k < f.dim; ++k) {
            int status = EUCL_OK;
            check_expr(f.transforms[t].fwd_first[k], f.transforms[t].fwd_len[k], "transformation " + std::to_string(t), &status);
            if (status == EUCL_OK)
                check_expr(f.transforms[t].inv_first[k], f.transforms[t].inv_len[k], "transformation " + std::to_string(t) + " (inverse)", &status);
            if (status != EUCL_OK) return status;
        }
    auto mapped_ok = [&](int mt) {
        return mt >= 0 && mt < f.n_mapped_textures;
    };
    for (int m = 0; m < f.n_mapped_textures; ++m) {
        const EuclMappedTexture& mt = f.mapped_textures[m];
        if (mt.texture < 0 || mt.texture >= f.n_textures) return bad("mapped texture " + std::to_string(m) + ": texture index out of bounds");
        if (mt.filter != EUCL_TEX_NEAREST && mt.filter != EUCL_TEX_LINEAR) return bad("mapped texture " + std::to_string(m) + ": unknown filter");
        if (mt.uv_kind != EUCL_UV_SPHERE3) return bad("mapped texture " + std::to_string(m) + ": unknown uv mapping");
    }
    if (f.background < -1 || f.background >= f.n_mapped_textures) return bad("background: mapped texture index out of bounds");
    for (int sidx = 0; sidx < f.n_surfaces; ++sidx) {
        const EuclSurface& sf = f.surfaces[sidx];
        const std::string what = "surface " + std::to_string(sidx);
        if (sf.ratio_op != EUCL_RATIO_UNIFORM && sf.ratio_op != EUCL_RATIO_FRESNEL) return bad(what + ": unknown reflection ratio provider");
        if (sf.refl_op != EUCL_REFL_SPECULAR) return bad(what + ": unknown reflection direction provider");
        if (sf.thr_op != EUCL_THR_IDENTITY && sf.thr_op != EUCL_THR_SNELL) return bad(what + ": unknown threshold direction provider");
        if (sf.color_first < 0 || sf.color_len < 0 || (long long)sf.color_first + sf.color_len > f.n_color_ops)
            return bad(what + ": colour program out of bounds");
        int sp = 0, peak = 0;
        for (int i = sf.color_first; i < sf.color_first + sf.color_len; ++i) {
            const EuclColorOp& op = f.color_ops[i];
            if (op.op < EUCL_COL_UNIFORM || op.op > EUCL_COL_BLEND) return bad(what + ": unknown colour opcode");
            if (op.op == EUCL_COL_TEXTURE && op.i0 != -1 && !mapped_ok(op.i0)) return bad(what + ": mapped texture index out of bounds");
            if (op.op == EUCL_COL_PERLIN_HUE && f.dim != 3) return bad(what + ": perlin_hue is a 3-D provider");
            if (op.op == EUCL_COL_BLEND) {
                if (op.i0 < EUCL_BLEND_RATIO || op.i0 > EUCL_BLEND_EXCLUSION) return bad(what + ": unknown blend function");
                if (sp < 2) return bad(what + ": colour stack underflow");
                sp -= 1;
            } else {
                sp += 1;
            }
            peak = std::max(peak, sp);
        }
        if (sf.color_len > 0 && sp != 1) return bad(what + ": colour program does not reduce to one colour");
        if (peak > kColorStackMax) {
            *why = what + ": colour program nests " + std::to_string(peak) + " deep, the device evaluator has " +
                   std::to_string(kColorStackMax) + " slots";
            return EUCL_ERR_SCENE_LIMIT;
        }
    }
    return EUCL_OK;
}

// Rewrites the binary post-order programs into macro programs (intersect.cuh): maximal left folds
// of leaves under Union / Intersection become one M_CHAIN node.
struct MacroBuilder {
    const EuclFlatScene& f;
    std::vector<MNode> out;
    static constexpr int kMaxChain = CHAIN_ROOT_CAP / 2;

    int hits_of_prim(int prim) const {
        const int k = f.prims[prim].kind;
        return (k == EUCL_PRIM_SPHERE || k == EUCL_PRIM_CYLINDER) ? 2 : (k == EUCL_PRIM_VOID ? 0 : 1);
    }
    int child_b(int n) const { return n - 1; }
    int child_a(int n) const { return f.nodes[n - 1].first - 1; }

    void emit(int n) {
        const EuclNode& nd = f.nodes[n];
        if (nd.op == EUCL_CSG_LEAF) {
            out.push_back(MNode{M_PRIM, nd.prim, 0, (int)out.size()});
            return;
        }
        if (nd.op == EUCL_CSG_UNION || nd.op == EUCL_CSG_INTERSECTION) {
            // walk down the left spine while the right child is a leaf
            std::vector<int> prims;
            int m = n;
            while (f.nodes[m].op == nd.op && f.nodes[child_b(m)].op == EUCL_CSG_LEAF) {
                prims.push_back(f.nodes[child_b(m)].prim);
                m = child_a(m);
            }
            if (f.nodes[m].op == EUCL_CSG_LEAF && !prims.empty()) {
                prims.push_back(f.nodes[m].prim);
                std::reverse(prims.begin(), prims.end());
                bool consecutive = true;
                for (size_t i = 1; i < prims.size(); ++i) consecutive = consecutive && prims[i] == prims[0] + (int)i;
                if (consecutive) {
                    const int count = (int)prims.size(), head = std::min(count, kMaxChain);
                    const int first = (int)out.size();
                    bool planes = true; // every leaf a half-space with signum +-1: enables the plane_chain fast path
                    for (int i = 0; i < head; ++i) {
                        const EuclPrim& pr = f.prims[prims[(size_t)i]];
                        planes = planes && pr.kind == EUCL_PRIM_HALFSPACE && (pr.s1 == 1.0 || pr.s1 == -1.0);
                    }
                    out.push_back(MNode{M_CHAIN, prims[0], head | (planes ? 0x4000 : 0) | (nd.op << 16), first});
                    for (int i = head; i < count; ++i) { // very long folds: the tail stays binary (same fold order)
                        out.push_back(MNode{M_PRIM, prims[(size_t)i], 0, (int)out.size()});
                        out.push_back(MNode{M_OP, nd.op, 0, first});
                    }
                    return;
                }
            }
        }
        const int first = (int)out.size();
        emit(child_a(n));
        emit(child_b(n));
        out.push_back(MNode{M_OP, nd.op, 0, first});
    }

    // Conservative bounding spheres (intersect.cuh: Bound) of macro range [first, root]: for each
    // node a sphere containing every point the node's shape can contain and hence every hit its
    // stream can emit (rules in DESIGN.md, "ray/bound culling").  r2 < 0: unbounded.
    void compute_bounds(int first, int root, double inflate, std::vector<Bound>* bounds) const {
        const int D = f.dim;
        auto none = [] {
            Bound b{};
            b.r2 = -1.0;
            return b;
        };
        auto radius = [](const Bound& b) { return std::sqrt(b.r2); };
        auto enclose = [&](const Bound& x, const Bound& y) { // sphere around two spheres
            if (x.r2 < 0 || y.r2 < 0) return none();
            double dist2 = 0;
            for (int k = 0; k < D; ++k) dist2 += (x.c[k] - y.c[k]) * (x.c[k] - y.c[k]);
            Bound b{};
            for (int k = 0; k < D; ++k) b.c[k] = 0.5 * (x.c[k] + y.c[k]);
            const double r = 0.5 * std::sqrt(dist2) + std::max(radius(x), radius(y));
            b.r2 = r * r;
            return b;
        };
        auto smaller = [&](const Bound& x, const Bound& y) {
            if (x.r2 < 0) return y;
            if (y.r2 < 0) return x;
            return x.r2 <= y.r2 ? x : y;
        };
        auto prim_bound = [&](int prim) {
            const EuclPrim& p = f.prims[prim];
            Bound b = none();
            if (p.kind == EUCL_PRIM_SPHERE && std::isfinite(p.s0)) {
                for (int k = 0; k < D; ++k) b.c[k] = p.v0[k];
                b.r2 = p.s0 * p.s0;
            }
            return b;
        };
        auto chain_bound = [&](const MNode& nd) {
            const int count = nd.b & 0x3fff, op = nd.b >> 16;
            if (op == EUCL_CSG_UNION) {
                Bound acc = prim_bound(nd.a);
                for (int i = 1; i < count; ++i) acc = enclose(acc, prim_bound(nd.a + i));
                return acc;
            }
            // Intersection: the axis-aligned half-spaces of the chain may box the region in
            double lo[EUCL_MAX_DIM], hi[EUCL_MAX_DIM];
            for (int k = 0; k < D; ++k) {
                lo[k] = -INFINITY;
                hi[k] = INFINITY;
            }
            Bound best = none();
            for (int i = 0; i < count; ++i) {
                const EuclPrim& p = f.prims[nd.a + i];
                best = smaller(best, prim_bound(nd.a + i));
                if (p.kind != EUCL_PRIM_HALFSPACE || !(p.s1 == 1.0 || p.s1 == -1.0)) continue;
                int axis = -1, nonzero = 0;
                for (int k = 0; k < D; ++k)
                    if (p.v0[k] != 0.0) {
                        axis = k;
                        ++nonzero;
                    }
                if (nonzero != 1 || !std::isfinite(p.v0[axis]) || !std::isfinite(p.s0)) continue;
                const double edge = -p.s0 / p.v0[axis]; // region: signum * (n_k x_k + c) >= 0
                if (p.s1 * p.v0[axis] > 0) lo[axis] = std::max(lo[axis], edge);
                else hi[axis] = std::min(hi[axis], edge);
            }
            // a cylinder capped by two half-spaces whose normals are parallel to its axis
            // (Cylinder::new_with_height, shape.rs:906-927): sphere around the finite cylinder
            for (int i = 0; i < count; ++i) {
                const EuclPrim& cy = f.prims[nd.a + i];
                if (cy.kind != EUCL_PRIM_CYLINDER || !std::isfinite(cy.s0)) continue;
                double s_lo = -INFINITY, s_hi = INFINITY;
                for (int j = 0; j < count; ++j) {
                    const EuclPrim& hs = f.prims[nd.a + j];
                    if (hs.kind != EUCL_PRIM_HALFSPACE || !(hs.s1 == 1.0 || hs.s1 == -1.0)) continue;
                    double nu = 0, nn = 0, uu = 0, nc = 0;
                    for (int k = 0; k < D; ++k) {
                        nu += hs.v0[k] * cy.v1[k];
                        nn += hs.v0[k] * hs.v0[k];
                        uu += cy.v1[k] * cy.v1[k];
                        nc += hs.v0[k] * cy.v0[k];
                    }
                    if (!(nu * nu >= (1.0 - 1e-12) * nn * uu) || nu == 0.0) continue; // not parallel to the axis
                    const double s = -(nc + hs.s0) / nu; // axis coordinate of the cap plane
                    if (hs.s1 * nu > 0) s_lo = std::max(s_lo, s);
                    else s_hi = std::min(s_hi, s);
                }
                if (std::isfinite(s_lo) && std::isfinite(s_hi) && s_lo <= s_hi) {
                    Bound b{};
                    const double mid = 0.5 * (s_lo + s_hi), half = 0.5 * (s_hi - s_lo);
                    for (int k = 0; k < D; ++k) b.c[k] = cy.v0[k] + cy.v1[k] * mid;
                    b.r2 = cy.s0 * cy.s0 + half * half;
                    best = smaller(best, b);
                }
            }
            bool boxed = true;
            for (int k = 0; k < D; ++k) boxed = boxed && std::isfinite(lo[k]) && std::isfinite(hi[k]) && lo[k] <= hi[k];
            if (boxed) {
                Bound b{};
                double r2 = 0;
                for (int k = 0; k < D; ++k) {
                    b.c[k] = 0.5 * (lo[k] + hi[k]);
                    r2 += 0.25 * (hi[k] - lo[k]) * (hi[k] - lo[k]);
                }
                b.r2 = r2;
                best = smaller(best, b);
            }
            return best;
        };
        std::vector<Bound> stack;
        for (int n = first; n <= root; ++n) {
            const MNode& nd = out[(size_t)n];
            Bound b;
            if (nd.kind == M_PRIM) {
                b = prim_bound(nd.a);
            } else if (nd.kind == M_CHAIN) {
                b = chain_bound(nd);
            } else {
                const Bound y = stack.back();
                stack.pop_back();
                const Bound x = stack.back();
                stack.pop_back();
                b = nd.a == EUCL_CSG_INTERSECTION ? smaller(x, y) : nd.a == EUCL_CSG_COMPLEMENT ? x : enclose(x, y);
            }
            stack.push_back(b);
            // inflate: the culling test must stay conservative under rounding (errors ~1e-13 relative)
            Bound stored = b;
            if (stored.r2 >= 0) {
                double cmax = 1.0;
                for (int k = 0; k < D; ++k) cmax = std::max(cmax, std::fabs(stored.c[k]));
                // f64 kernels: hit points sit on their surfaces to ~1e-13 relative; f32 kernels: to ~1e-6
                const double r = std::sqrt(stored.r2) * (1.0 + inflate) + 0.1 * inflate * cmax;
                stored.r2 = r * r;
                if (!std::isfinite(stored.r2)) stored.r2 = -1.0;
            }
            (*bounds)[(size_t)n] = stored;
        }
    }

    // Worst-case arena use of the device evaluator (csg_first) for macro range [first, root]
    bool fits(int first, int root, int* peak_out, int* depth_out) const {
        std::vector<int> lens;
        int top = 0, peak = 0, depth = 0;
        for (int n = first; n <= root; ++n) {
            const MNode& nd = out[(size_t)n];
            if (nd.kind == M_PRIM) {
                const int c = hits_of_prim(nd.a);
                lens.push_back(c);
                top += c;
                peak = std::max(peak, top);
            } else if (nd.kind == M_CHAIN) {
                const int count = nd.b & 0x3fff;
                peak = std::max(peak, top + 4 * count); // list + scratch, 2 * count each
                int c = 0;
                for (int i = 0; i < count; ++i) c += hits_of_prim(nd.a + i);
                lens.push_back(c);
                top += c;
            } else {
                const int bl = lens.back();
                lens.pop_back();
                const int al = lens.back();
                lens.pop_back();
                const int outn = al + bl + 2;
                peak = std::max(peak, top + outn);
                top = top - al - bl + outn;
                lens.push_back(outn);
            }
            depth = std::max(depth, (int)lens.size());
        }
        *peak_out = peak;
        *depth_out = depth;
        return peak <= CSG_ARENA && depth <= CSG_LIST_STACK;
    }
};

// LinearSpace expressions in table form (scene_dev.cuh: LinRow): recognises RPN programs of the shape
//   term (term (+|-))*   with   term := VAR | VAR CONST (*|/) | CONST VAR (*|/)
// which is how the host compiler (csrc/host/expr.cc) lays out `x * 4`, `4 * x`, `x / 4`, `y`, `x * 2 + y - z / 3`.
// `in[var]` reads a component of the transformation's input, exactly like EUCL_EX_VAR.
LinRow lower_lin_row(const EuclExprOp* ops, int len, int dim) {
    LinRow row{};
    if (!env_int("EUCL_LIN_TABLE", 1)) return row;
    int i = 0, n = 0;
    auto parse_term = [&](LinTerm* out) -> bool {
        if (i >= len) return false;
        const EuclExprOp& a = ops[i];
        if (a.op == EUCL_EX_VAR) {
            if (a.arg < 0 || a.arg >= dim) return false;
            if (i + 2 < len && ops[i + 1].op == EUCL_EX_CONST && (ops[i + 2].op == EUCL_EX_MUL || ops[i + 2].op == EUCL_EX_DIV)) {
                *out = LinTerm{a.arg, ops[i + 2].op == EUCL_EX_MUL ? 1 : 2, ops[i + 1].value};
                i += 3;
            } else {
                *out = LinTerm{a.arg, 0, 0.0};
                i += 1;
            }
            return true;
        }
        if (a.op == EUCL_EX_CONST && i + 2 < len && ops[i + 1].op == EUCL_EX_VAR &&
            (ops[i + 2].op == EUCL_EX_MUL || ops[i + 2].op == EUCL_EX_DIV)) {
            if (ops[i + 1].arg < 0 || ops[i + 1].arg >= dim) return false;
            *out = LinTerm{ops[i + 1].arg, ops[i + 2].op == EUCL_EX_MUL ? 1 : 3, a.value}; // c * v == v * c in IEEE arithmetic
            i += 3;
            return true;
        }
        return false;
    };
    LinTerm t{};
    if (!parse_term(&t)) return LinRow{};
    row.t[n++] = t;
    while (i < len) {
        if (n >= kLinTermsMax || !parse_term(&t)) return LinRow{};
        if (i >= len || (ops[i].op != EUCL_EX_ADD && ops[i].op != EUCL_EX_SUB)) return LinRow{};
        if (ops[i].op == EUCL_EX_SUB) t.kind |= 16;
        ++i;
        row.t[n++] = t;
    }
    row.n_terms = n;
    return row;
}

struct BlobWriter {
    std::vector<uint8_t> bytes;
    int reserve(size_t n) {
        size_t off = align16(bytes.size());
        bytes.resize(off + align16(n), 0);
        return (int)off;
    }
    template <typename T>
    int put(const T* src, size_t count) {
        int off = reserve(sizeof(T) * std::max<size_t>(count, 1));
        if (count) std::memcpy(bytes.data() + off, src, sizeof(T) * count);
        return off;
    }
};

} // namespace

extern "C" {

int eucl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void eucl_scene_destroy(EuclScene* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    for (Worker* w : s->workers) {
        w->stop();
        delete w;
    }
    for (EuclScene* t : s->twins) eucl_scene_destroy(t);
    if (s->ev_done) cudaEventDestroy(s->ev_done);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (auto& e : s->ev_split)
        if (e) cudaEventDestroy(e);
    for (auto t : s->tex_objects) cudaDestroyTextureObject(t);
    for (auto a : s->arrays) cudaFreeArray(a);
    if (s->d_blob && !s->is_twin) cudaFree(s->d_blob);
    s->nodes.release();
    s->small.release();
    s->frame.release();
    s->hit_ids.release();
    s->order.release();
    s->path_io.release();
    s->rorder.release();
    s->frame_table.release();
    s->frame_entity.release();
    s->node_frame.release();
    s->node_cost.release();
    s->aov_stage.release();
    s->ray_stage.release();
    if (s->h_frame_table) cudaFreeHost(s->h_frame_table);
    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
    if (s->h_small) cudaFreeHost(s->h_small);
    for (auto& e : s->ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : s->prof_events) cudaEventDestroy(e);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    if (s->side_stream) cudaStreamDestroy(s->side_stream);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    delete s;
}

int eucl_scene_create(const EuclFlatScene* flat, int device, EuclScene** out) {
    return eucl_scene_create_precision(flat, device, EUCL_PRECISION_F64, out);
}

int eucl_scene_create_precision(const EuclFlatScene* flat, int device, int precision, EuclScene** out) {
    if (!flat || !out) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_create: null argument");
    *out = nullptr;
    if (precision != EUCL_PRECISION_F64 && precision != EUCL_PRECISION_F32)
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_create_precision: unknown precision");
    if (flat->dim != 3 && flat->dim != 4) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_create: dim must be 3 or 4");
    // the scene is validated before any device is touched (also without one: tests/test_scene_limits.py)
    std::string why;
    int status = validate_scene(*flat, &why);
    if (status != EUCL_OK) return fail(status, why);
    for (int t = 0; t < flat->n_textures; ++t)
        if (flat->textures[t].width == 0 || flat->textures[t].height == 0 || !flat->texels)
            return fail(EUCL_ERR_TEXTURE_MISSING, "texture slot " + std::to_string(t) + " was never filled");
    const int n_dev = eucl_device_count();
    if (n_dev <= 0) return fail(EUCL_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    if (device < 0 || device >= n_dev) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_create: device index out of range");

    EUCL_CUDA(cudaSetDevice(device));
    EuclScene* s = new EuclScene();
    s->device = device;
    s->real_bytes = precision == EUCL_PRECISION_F32 ? 4 : 8;
    s->dim = flat->dim;
    s->n_entities = flat->n_entities;
    cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device);
    auto bail = [&](int st, const std::string& msg) {
        eucl_scene_destroy(s);
        return fail(st, msg);
    };
#define EUCL_CUDA_S(expr)                                                                                   \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess)                                                                              \
            return bail(_e == cudaErrorMemoryAllocation ? EUCL_ERR_OUT_OF_MEMORY : EUCL_ERR_CUDA,           \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                                \
    } while (0)

    EUCL_CUDA_S(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
    s->stream = s->own_stream;
    EUCL_CUDA_S(cudaEventCreate(&s->ev[0]));
    EUCL_CUDA_S(cudaEventCreate(&s->ev[1]));
    EUCL_CUDA_S(cudaStreamCreateWithFlags(&s->side_stream, cudaStreamNonBlocking));
    EUCL_CUDA_S(cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
    EUCL_CUDA_S(cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));

    // textures -> CUDA arrays + point-sampled texture objects
    for (int t = 0; t < flat->n_textures; ++t) {
        const EuclTexture& tx = flat->textures[t];
        cudaChannelFormatDesc desc = cudaCreateChannelDesc<uchar4>();
        cudaArray_t arr = nullptr;
        EUCL_CUDA_S(cudaMallocArray(&arr, &desc, tx.width, tx.height));
        s->arrays.push_back(arr);
        EUCL_CUDA_S(cudaMemcpy2DToArray(arr, 0, 0, flat->texels + tx.texel_offset, (size_t)tx.width * 4,
                                        (size_t)tx.width * 4, tx.height, cudaMemcpyHostToDevice));
        cudaResourceDesc rd{};
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td{};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint; // bilinear is done in f64 in the kernel
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        cudaTextureObject_t obj = 0;
        EUCL_CUDA_S(cudaCreateTextureObject(&obj, &rd, &td, nullptr));
        s->tex_objects.push_back(obj);
    }

    // pack the blob
    BlobWriter w;
    w.reserve(sizeof(SceneHeader));
    SceneHeader h{};
    h.dim = flat->dim;
    h.n_prims = flat->n_prims;
    h.n_nodes = flat->n_nodes;
    h.n_entities = flat->n_entities;
    h.n_materials = flat->n_materials;
    h.n_transforms = flat->n_transforms;
    h.n_expr_ops = flat->n_expr_ops;
    h.n_surfaces = flat->n_surfaces;
    h.n_color_ops = flat->n_color_ops;
    h.n_mapped_textures = flat->n_mapped_textures;
    h.n_textures = flat->n_textures;
    h.background = flat->background;
    const int np = std::max(flat->n_prims, 1);
    std::vector<int32_t> kind((size_t)np, 0);
    std::vector<double> v0((size_t)np * EUCL_MAX_DIM, 0.0), v1((size_t)np * EUCL_MAX_DIM, 0.0), s0((size_t)np, 0.0),
        s1((size_t)np, 0.0);
    for (int i = 0; i < flat->n_prims; ++i) {
        const EuclPrim& p = flat->prims[i];
        kind[(size_t)i] = p.kind;
        for (int k = 0; k < EUCL_MAX_DIM; ++k) {
            v0[(size_t)k * flat->n_prims + i] = p.v0[k];
            v1[(size_t)k * flat->n_prims + i] = p.v1[k];
        }
        s0[(size_t)i] = p.s0;
        s1[(size_t)i] = p.s1;
    }
    h.off_prim_kind = w.put(kind.data(), kind.size());
    h.off_prim_v0 = w.put(v0.data(), v0.size());
    h.off_prim_v1 = w.put(v1.data(), v1.size());
    h.off_prim_s0 = w.put(s0.data(), s0.size());
    h.off_prim_s1 = w.put(s1.data(), s1.size());
    std::vector<double> planes((size_t)np * kPlaneStride, 0.0); // AoS copy: [v0[0..3], s0, s1] per primitive
    for (int i = 0; i < flat->n_prims; ++i) {
        for (int k = 0; k < EUCL_MAX_DIM; ++k) planes[(size_t)i * kPlaneStride + k] = flat->prims[i].v0[k];
        planes[(size_t)i * kPlaneStride + 4] = flat->prims[i].s0;
        planes[(size_t)i * kPlaneStride + 5] = flat->prims[i].s1;
    }
    h.off_planes = w.put(planes.data(), planes.size());
    // macro CSG programs replace the binary node list on the device
    MacroBuilder mb{*flat, {}};
    std::vector<EuclEntity> dev_entities((size_t)flat->n_entities);
    // Complement(VoidShape, X) -- "everything but X": a room described by its interior (4d_room's walls).  VoidShape has no
    // hits, so ComplementIterator only ever takes its `b`-only branch: every hit of X in order, normal negated, kept because
    // VoidShape contains every point (shape.rs:394-408); is_point_inside is `true && !X` (shape.rs:596).  The device program of
    // such an entity is X's program and the entity carries ENT_NEGATED: hits flip their normal flag, membership is inverted,
    // and X's bound still bounds the hits (not the points the entity contains).  With X a chain of half-spaces the entity
    // becomes a root plane chain: first-item shortcut, light intersect kernel.
    std::vector<char> negated((size_t)std::max(flat->n_entities, 1), 0);
    for (int e = 0; e < flat->n_entities; ++e) {
        EuclEntity de = flat->entities[e];
        de.node_first = (int)mb.out.size();
        const int root = flat->entities[e].node_root;
        const EuclNode& rn = flat->nodes[root];
        if (rn.op == EUCL_CSG_COMPLEMENT && flat->nodes[mb.child_a(root)].op == EUCL_CSG_LEAF &&
            flat->prims[flat->nodes[mb.child_a(root)].prim].kind == EUCL_PRIM_VOID && env_int("EUCL_NEGATED_ROOMS", 1)) {
            negated[(size_t)e] = 1;
            mb.emit(mb.child_b(root));
        } else {
            mb.emit(root);
        }
        de.node_root = (int)mb.out.size() - 1;
        int peak = 0, depth = 0;
        if (!mb.fits(de.node_first, de.node_root, &peak, &depth))
            return bail(EUCL_ERR_SCENE_LIMIT, "entity " + std::to_string(e) + ": CSG program too large for the device evaluator (" +
                                                  std::to_string(peak) + " arena slots of " + std::to_string(CSG_ARENA) + ", nesting " +
                                                  std::to_string(depth) + ")");
        dev_entities[(size_t)e] = de;
    }
    std::vector<Bound> bounds(mb.out.size());
    for (int e = 0; e < flat->n_entities; ++e)
        mb.compute_bounds(dev_entities[(size_t)e].node_first, dev_entities[(size_t)e].node_root, s->real_bytes == 4 ? 1e-3 : 1e-6, &bounds);
    if (!env_int("EUCL_BOUND_CULL", 1))
        for (auto& b : bounds) b.r2 = -1.0;
    h.n_nodes = (int)mb.out.size();
    h.off_nodes = w.put(mb.out.data(), mb.out.size());
    h.off_bounds = w.put(bounds.data(), bounds.size());
    for (int e = 0; e < flat->n_entities && h.n_cull < 4; ++e) { // entities worth a reach-key bit
        const EuclEntity& de = dev_entities[(size_t)e];
        // (not the negated ones: a room is reached by every ray inside it)
        if (de.surface >= 0 && !negated[(size_t)e] && mb.out[(size_t)de.node_root].kind != M_PRIM && bounds[(size_t)de.node_root].r2 >= 0.0)
            h.cull_root[h.n_cull++] = de.node_root;
    }
    s->n_cull = h.n_cull;
    // per-entity classification for the closest-hit loops; a scene is "light-capable" when a ray with reach key 0
    // can only meet primitives and root plane chains (k_intersect<LIGHT>)
    std::vector<int32_t> ent_flags((size_t)std::max(flat->n_entities, 1), 0);
    bool light_capable = true;
    for (int e = 0; e < flat->n_entities; ++e) {
        const EuclEntity& de = dev_entities[(size_t)e];
        if (negated[(size_t)e]) ent_flags[(size_t)e] = ENT_NEGATED; // material_at needs it for entities without a surface too
        if (de.surface < 0) continue;
        const MNode& root = mb.out[(size_t)de.node_root];
        int fl = ENT_SURFACED | ent_flags[(size_t)e];
        if (root.kind == M_PRIM) fl |= ENT_PRIM;
        else if (root.kind == M_CHAIN && de.node_first == de.node_root && (root.b & 0x4000) && (root.b & 0x3fff) <= kPlaneChainMax) fl |= ENT_ROOT_PLANES;
        for (int k = 0; k < h.n_cull; ++k)
            if (h.cull_root[k] == de.node_root) fl |= ENT_CULL_ROOT;
        if (!(fl & (ENT_PRIM | ENT_ROOT_PLANES | ENT_CULL_ROOT))) light_capable = false;
        ent_flags[(size_t)e] = fl;
    }
    if (!env_int("EUCL_INTERSECT_SPLIT", 1)) light_capable = false; // diagnostics: one build intersects every ray
    h.light_capable = light_capable ? 1 : 0;
    s->light_capable = h.light_capable;
    h.off_ent_flags = w.put(ent_flags.data(), ent_flags.size());
    h.off_entities = w.put(dev_entities.data(), dev_entities.size());
    h.off_materials = w.put(flat->materials, (size_t)flat->n_materials);
    h.off_transforms = w.put(flat->transforms, (size_t)flat->n_transforms);
    h.off_expr_ops = w.put(flat->expr_ops, (size_t)flat->n_expr_ops);
    std::vector<LinRow> lin_rows((size_t)std::max(flat->n_transforms, 1) * 2 * EUCL_MAX_DIM);
    for (int t = 0; t < flat->n_transforms; ++t)
        for (int k = 0; k < flat->dim; ++k) {
            const EuclTransform& tr = flat->transforms[t];
            lin_rows[(size_t)t * 2 * EUCL_MAX_DIM + k] = lower_lin_row(flat->expr_ops + tr.fwd_first[k], tr.fwd_len[k], flat->dim);
            lin_rows[(size_t)t * 2 * EUCL_MAX_DIM + EUCL_MAX_DIM + k] = lower_lin_row(flat->expr_ops + tr.inv_first[k], tr.inv_len[k], flat->dim);
        }
    h.off_lin_rows = w.put(lin_rows.data(), lin_rows.size());
    h.off_surfaces = w.put(flat->surfaces, (size_t)flat->n_surfaces);
    h.off_color_ops = w.put(flat->color_ops, (size_t)flat->n_color_ops);
    h.off_mapped = w.put(flat->mapped_textures, (size_t)flat->n_mapped_textures);
    h.off_textures = w.put(flat->textures, (size_t)flat->n_textures);
    h.off_tex_objects = w.put(s->tex_objects.data(), s->tex_objects.size());
    h.off_perlin = w.put(flat->perlin_perm, 256);
    int max_nodes = 1;
    for (int e = 0; e < flat->n_entities; ++e)
        max_nodes = std::max(max_nodes, flat->entities[e].node_root - flat->entities[e].node_first + 1);
    h.max_entity_nodes = max_nodes;
    h.blob_bytes = (int)w.bytes.size();
    std::memcpy(w.bytes.data(), &h, sizeof h);
    s->blob_bytes = h.blob_bytes;
    // staged scene + the per-thread plane_chain scratch columns (kernels.cu: plane_scratch)
    s->smem_scene = scene_smem_bytes(h.blob_bytes);
    s->smem_bytes = s->smem_scene + sizeof(double) * kPlaneChainMax * kBlock;
    // shade bins of the light build of k_shade: the miss bin and the bins of every entity whose surface has a uniform
    // reflection ratio and the identity threshold direction; the heavy build (Fresnel, Snell) shades the others
    s->shade_light_mask = 1ull;
    s->shade_heavy_mask = 0ull;
    if (kBinsPerEntity * flat->n_entities + 1 <= kMaxBins)
        for (int e = 0; e < flat->n_entities; ++e) {
            const int sf = flat->entities[e].surface;
            if (sf < 0) continue;
            const bool simple = flat->surfaces[sf].ratio_op == EUCL_RATIO_UNIFORM && flat->surfaces[sf].thr_op == EUCL_THR_IDENTITY;
            const unsigned long long bits = ((1ull << kBinsPerEntity) - 1ull) << (1 + kBinsPerEntity * e);
            (simple ? s->shade_light_mask : s->shade_heavy_mask) |= bits;
        }
    if (env_int("EUCL_SHADE_SPLIT", 1) == 0) { // one build shades every bin (diagnostics)
        s->shade_heavy_mask |= s->shade_light_mask;
        s->shade_light_mask = 0ull;
    }
    int smem_optin = 0;
    cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (s->smem_bytes > (size_t)smem_optin)
        return bail(EUCL_ERR_SCENE_LIMIT, "scene tables (" + std::to_string(s->smem_bytes) +
                                              " B) exceed the shared memory of one CTA (" + std::to_string(smem_optin) + " B)");
    EUCL_CUDA_S(cudaMalloc((void**)&s->d_blob, w.bytes.size()));
    EUCL_CUDA_S(cudaMemcpy(s->d_blob, w.bytes.data(), w.bytes.size(), cudaMemcpyHostToDevice));
    EUCL_CUDA_S(EUCL_PREC(configure_kernels)(s->smem_bytes, s->smem_scene));
    EUCL_CUDA_S(cudaMallocHost((void**)&s->h_small, sizeof(int32_t) * kSmallInts));
#undef EUCL_CUDA_S
    *out = s;
    return EUCL_OK;
}

} // extern "C"

namespace {

// Camera constants in the reference's order (d3/entity/camera.rs:61-67,174-182; d4: 167-173)
// T = the scalar the camera arithmetic runs in: double, or float for the reference's `low_precision` feature (the
// results are stored as doubles either way; the f32 kernels narrow them back without loss)
template <typename T>
void frame_params_t(const EuclCamera& cam, const EuclRenderOpts& o, FrameParams* fp) {
    const int D = cam.dim;
    std::memset(fp, 0, sizeof *fp);
    const T w = (T)o.width, h = (T)o.height;
    const T pi = (T)3.14159265358979323846264338327950288;
    const T fov_rad = pi * (T)cam.fov_deg / (T)180.0;
    volatile T diag = std::sqrt(w * w + h * h);
    volatile T denom = (T)2.0 * std::tan(fov_rad / (T)2.0);
    const T distance = diag / denom;
    T right[EUCL_MAX_DIM] = {0, 0, 0, 0};
    if (D == 3) {
        const T f0 = (T)cam.forward[0], f1 = (T)cam.forward[1], f2 = (T)cam.forward[2];
        const T u0 = (T)cam.up[0], u1 = (T)cam.up[1], u2 = (T)cam.up[2];
        volatile T p0 = f1 * u2, p1 = f2 * u1, p2 = f2 * u0, p3 = f0 * u2, p4 = f0 * u1, p5 = f1 * u0;
        volatile T cx = p0 - p1;
        volatile T cy = p2 - p3;
        volatile T cz = p4 - p5;
        volatile T n2 = cx * cx;
        volatile T t1 = cy * cy, t2 = cz * cz;
        n2 = n2 + t1;
        n2 = n2 + t2;
        const T n = std::sqrt(n2);
        right[0] = cx / n;
        right[1] = cy / n;
        right[2] = cz / n;
    } else {
        for (int k = 0; k < 4; ++k) right[k] = -(T)cam.left[k];
    }
    for (int k = 0; k < D; ++k) {
        fp->location[k] = (T)cam.location[k];
        volatile T step = (T)cam.forward[k] * distance;
        fp->center[k] = (T)((T)cam.location[k] + step);
        fp->up[k] = (T)cam.up[k];
        fp->right[k] = right[k];
    }
    // Duration * 1000 -> whole seconds -> / 1000 (d3/entity/surface.rs:32); `as F` narrows the f64 quotient
    fp->time_millis = (T)(std::floor(o.time_seconds * 1000.0) / 1000.0);
    fp->width = (int)o.width;
    fp->height = (int)o.height;
    fp->max_depth = (int)cam.max_depth;
}
void frame_params(const EuclCamera& cam, const EuclRenderOpts& o, int real_bytes, FrameParams* fp) {
    if (real_bytes == 4) frame_params_t<float>(cam, o, fp);
    else frame_params_t<double>(cam, o, fp);
}

size_t arena_bytes(int dim, int real_bytes, size_t cap) {
    size_t per = (size_t)(ray_reals(dim, real_bytes) + kHitReals + 4) * real_bytes + 4 + sizeof(NodeMeta);
    return per * cap + 16 * 16;
}

// The frames of one call.  A single frame (eucl_render*) is a batch of one and renders exactly as it always did;
// K > 1 frames (eucl_render_frames*) are ONE virtual frame of K * rows rows -- chunks, bands and pipelines split it
// like any other frame -- whose per-pixel constants the kernels look up in a device table by virtual row.
struct FrameBatch {
    const EuclFrame* frames;
    uint32_t n;                      // K
    uint32_t rows;                   // rows per frame
    const FrameParams* d_table;      // K > 1: [K] frame constants on the device, uploaded before the first launch
    uint64_t table_key;              // K > 1: hash of the table contents, part of the graph key
    // eucl_trace_rays*: the rays on the device ([n][dim] each) in place of a camera (K = 1; frames[0] carries only
    // max_depth and the time), null for camera frames.  The virtual frame has n / width rows of width rays.
    const double* ray_origins = nullptr;
    const double* ray_directions = nullptr;
};

Workspace carve(EuclScene* s, int dim, int cap, int list_cap, const FrameBatch& fb) {
    Workspace ws{};
    ws.capacity = cap;
    ws.list_cap = list_cap;
    ws.n_frames = (int32_t)fb.n;
    ws.frame_rows = (int32_t)fb.rows;
    if (fb.n > 1) {
        ws.frames = fb.d_table;
        ws.frame_entity = (int32_t*)s->frame_entity.ptr;
        ws.node_frame = (int32_t*)s->node_frame.ptr;
    }
    if (fb.n > 1 || fb.ray_origins) ws.untraced = (int32_t*)s->small.ptr + SmallLayout::untraced;
    uint8_t* p = (uint8_t*)s->nodes.ptr;
    auto take = [&](size_t bytes) {
        uint8_t* r = p;
        p += align16(bytes);
        return r;
    };
    const size_t rb = (size_t)s->real_bytes;
    ws.ray = take((size_t)ray_reals(dim, s->real_bytes) * rb * cap);
    ws.hit = take((size_t)kHitReals * rb * cap);
    ws.res = take((size_t)4 * rb * cap);
    ws.meta = (NodeMeta*)take(sizeof(NodeMeta) * (size_t)cap);
    ws.ray_cur = (int32_t*)take((size_t)4 * cap);
    int32_t* small = (int32_t*)s->small.ptr;
    ws.count = small + SmallLayout::count;
    ws.level_off = small + SmallLayout::level_off;
    ws.overflow = small + SmallLayout::overflow;
    ws.cam_entity = small + SmallLayout::cam_entity;
    ws.undefined_count = (unsigned long long*)(small + SmallLayout::undefined64);
    ws.mega_level_counts = (unsigned long long*)(small + SmallLayout::mega64);
    ws.bin_count = small + SmallLayout::bins;
    ws.order = (int32_t*)s->order.ptr;
    const bool bin = s->order.ptr != nullptr;
    ws.n_bins = bin ? kBinsPerEntity * s->n_entities + 1 : 1;
    ws.rbin_count = small + SmallLayout::rbins;
    ws.rorder = (int32_t*)s->rorder.ptr;
    ws.ray_bins = s->rorder.ptr != nullptr && s->ray_bins_now ? 1 : 0;
    return ws;
}

// ray grouping of the frame about to be rendered (see EuclScene::ray_bins_mode)
void choose_grouping(EuclScene* s) {
    const int forced = env_int("EUCL_BIN_RAYS", -1);
    if (forced >= 0) s->ray_bins_mode = forced ? 1 : 0;
    if (s->ray_bins_mode >= 0) s->ray_bins_now = s->ray_bins_mode == 1;
    else s->ray_bins_now = s->tune_count[1] <= s->tune_count[0]; // undecided: alternate, "on" first
}

// Auto-tuning of the ray grouping (EuclScene::ray_bins_mode) from whole retry-free frames.
void tune_grouping(EuclScene* s, const EuclStats& st, int pipeline) {
    if (s->ray_bins_mode >= 0 || st.retries != 0 || st.pixels == 0 || pipeline != EUCL_PIPELINE_WAVEFRONT) return;
    if (s->n_cull == 0) {
        s->ray_bins_mode = 0;
    } else if (s->warm_frames >= 1) { // never the scene's very first frame (allocations, cold caches)
        if (s->tune_pixels != st.pixels) { // only frames of one size are comparable
            s->tune_pixels = st.pixels;
            s->tune_ms[0] = s->tune_ms[1] = 0.f;
            s->tune_count[0] = s->tune_count[1] = 0;
        }
        // two frames per setting, alternating, the faster one of each counts: one slow frame (another process on
        // the GPU, a clock ramp) must not decide; EuclStats.ray_grouping reports what a frame used
        const int m = s->ray_bins_now ? 1 : 0;
        s->tune_ms[m] = s->tune_count[m] == 0 ? st.ms_total : std::min(s->tune_ms[m], st.ms_total);
        s->tune_count[m] += 1;
        if (s->tune_count[0] >= 2 && s->tune_count[1] >= 2) s->ray_bins_mode = s->tune_ms[1] < s->tune_ms[0] ? 1 : 0;
    }
}

// Renders this rank's rows of `o` (all of them, or -- sub_stride > 1 -- the bands that `o` names, which are every
// sub_stride-th band of the caller's rank starting at sub_offset: render_split).
// `o` describes the (virtual) frame: o->height = fb.n * fb.rows.
int render_impl(EuclScene* s, const FrameBatch& fb, const EuclRenderOpts* o, uint8_t* d_rgb, int32_t* d_hit,
                const AovPlanes& aov_out, EuclStats* stats, int sub_stride = 1, int sub_offset = 0) {
    const int dim = s->dim;
    const EuclCamera* cam = &fb.frames[0].camera; // (every frame of a batch has this max_depth)
    const bool rays = fb.ray_origins != nullptr;
    FrameParams fp;
    if (rays) { // no camera: the grid, the depth and the time (truncated as for a frame, then `as F`)
        std::memset(&fp, 0, sizeof fp);
        const double millis = std::floor(fb.frames[0].time_seconds * 1000.0) / 1000.0;
        fp.time_millis = s->real_bytes == 4 ? (double)(float)millis : millis;
        fp.width = (int)o->width;
        fp.height = (int)o->height;
        fp.max_depth = (int)cam->max_depth;
    } else {
        EuclRenderOpts first = *o;
        first.height = fb.rows;
        first.time_seconds = fb.frames[0].time_seconds;
        frame_params(*cam, first, s->real_bytes, &fp);
    }
    const int width = (int)o->width;
    const uint32_t my_rows = eucl_band_rows_for_rank(o);
    EuclStats st{};
    st.levels = cam->max_depth + 1;
    if (!s->is_twin) choose_grouping(s); // a twin renders with its leader's setting
    if (fb.n > 1) EUCL_CUDA(s->frame_entity.ensure(sizeof(int32_t) * fb.n));
    EUCL_CUDA(cudaEventRecord(s->ev[0], s->stream));
    if (my_rows > 0) {
        // chunking: whole local rows, about EUCL_CHUNK_PIXELS primaries per chunk.  Large chunks are faster (longer
        // levels, fewer host round trips: 4d_room 7680x4320 renders 10 % faster as one chunk than as eight), so the
        // default covers an 8K frame; the chunk shrinks by itself when its arena would not fit (2^31 nodes, the
        // memory budget, or an allocation failure).
        const long long chunk_pixels_target = std::max(1, env_int("EUCL_CHUNK_PIXELS", 1 << 25));
        int rows_per_chunk = (int)std::max<long long>(1, chunk_pixels_target / width);
        rows_per_chunk = std::min<int>(rows_per_chunk, (int)my_rows);
        if ((long long)width > (1ll << 30)) return fail(EUCL_ERR_INVALID_ARGUMENT, "frame rows too wide");
        EUCL_CUDA(s->small.ensure(sizeof(int32_t) * kSmallInts));
        if (s->arena_factor <= 0.0) s->arena_factor = std::max(1.0, (double)env_int("EUCL_ARENA_FACTOR_X10", 45) / 10.0);
        // queue kernels run as ONE wave of resident CTAs (512 threads per SM at 128 registers) walking their level with a grid
        // stride: measured faster than 2-8 waves on glass scenes (3d_room 20.7 -> 20.0 ms), equal elsewhere
        Launch l{s->stream, s->d_blob, s->smem_bytes, s->smem_scene,
                 s->sm_count * std::max(1, env_int("EUCL_BLOCKS_PER_SM", kResidentThreads / kBlock)),
                 s->sm_count * std::max(1, env_int("EUCL_LIGHT_BLOCKS_PER_SM", kLightResidentBlocks)),
                 s->sm_count * std::max(1, env_int("EUCL_SHADE_BLOCKS_PER_SM", kShadeResidentBlocks)),
                 s->sm_count * std::max(1, env_int("EUCL_MEM_BLOCKS_PER_SM", 8)),
                 s->shade_light_mask, s->shade_heavy_mask,
                 s->sm_count * std::max(1, env_int("EUCL_LIGHT_K2_BLOCKS_PER_SM", kLightK2ResidentBlocks)), s->light_capable, s->n_cull,
                 // per-launch profiling and the debugging modes keep everything on one stream
                 (o->profile || env_int("EUCL_DEBUG_SYNC", 0) || !env_int("EUCL_CONCURRENT", 1)) ? nullptr : s->side_stream, s->ev_fork,
                 s->ev_join, s->sm_count * std::max(1, env_int("EUCL_BACKGROUND_BLOCKS_PER_SM", EUCL_BACKGROUND_MIN_BLOCKS))};
        const bool want_rorder = o->pipeline == EUCL_PIPELINE_WAVEFRONT && s->n_cull > 0 && env_int("EUCL_BIN_RAYS", 1);
        // shade-coherence bins: one node list per hit entity (+ miss), each able to hold a whole level
        const bool want_order = o->pipeline == EUCL_PIPELINE_WAVEFRONT && kBinsPerEntity * s->n_entities + 1 <= kMaxBins && env_int("EUCL_BIN_SHADE", 1);
        const size_t n_lists = (want_rorder ? (size_t)kRayBins : 0) + (want_order ? (size_t)(kBinsPerEntity * s->n_entities + 1) : 0);
        // the COST builds keep a (segments, levels) pair per node next to the arena
        const bool want_cost = o->pipeline == EUCL_PIPELINE_WAVEFRONT && (aov_out.segments || aov_out.levels);
        auto workspace_bytes = [&](size_t cap, size_t list_cap) {
            return arena_bytes(dim, s->real_bytes, cap) + sizeof(int32_t) * n_lists * list_cap + (want_cost ? sizeof(uint2) * cap : 0);
        };

        for (int row0 = 0; row0 < (int)my_rows;) {
            ChunkParams cp{};
            cp.local_row0 = row0;
            cp.band_rows = o->band_rows ? (int)o->band_rows : (int)o->height;
            cp.band_rank = (int)o->band_rank;
            cp.band_world = o->band_world ? (int)o->band_world : 1;
            cp.compact_rows = o->compact_rows;
            cp.sub_stride = sub_stride;
            cp.sub_offset = sub_offset;
            for (;;) { // retry with a larger arena when a level overflowed, with a smaller chunk when the arena cannot grow
                cp.n_rows = std::min<int>(rows_per_chunk, (int)my_rows - row0);
                cp.n_pixels = cp.n_rows * width;
                long long want = (long long)std::ceil((double)rows_per_chunk * (double)width * s->arena_factor) + 1024;
                if (o->pipeline == EUCL_PIPELINE_MEGAKERNEL) want = 16;
                long long want_list = (long long)std::ceil((double)rows_per_chunk * (double)width * s->list_factor) + 1024;
                if (o->pipeline == EUCL_PIPELINE_MEGAKERNEL) want_list = 16;
                bool too_big = want > 0x7fff0000ll || want_list > 0x7fff0000ll;
                if (!too_big && ((int)want > s->arena_capacity || (int)want_list > s->list_capacity)) {
                    EUCL_CUDA(cudaStreamSynchronize(s->stream));
                    want = std::max<long long>(want, s->arena_capacity);
                    want_list = std::max<long long>(want_list, s->list_capacity);
                    size_t free_b = 0, total_b = 0;
                    EUCL_CUDA(cudaMemGetInfo(&free_b, &total_b));
                    const size_t held = s->nodes.bytes + s->order.bytes + s->rorder.bytes + s->node_cost.bytes;
                    size_t budget = (size_t)((double)(free_b + held) * 0.85);
                    const int cap_mb = env_int("EUCL_ARENA_MAX_MB", 0);
                    if (cap_mb > 0) budget = std::min(budget, (size_t)cap_mb << 20);
                    too_big = workspace_bytes((size_t)want, (size_t)want_list) > budget;
                    if (!too_big) {
                        cudaError_t e = s->nodes.ensure(arena_bytes(dim, s->real_bytes, (size_t)want));
                        if (e == cudaSuccess && want_rorder) e = s->rorder.ensure(sizeof(int32_t) * (size_t)kRayBins * (size_t)want_list);
                        if (e == cudaSuccess && want_order) e = s->order.ensure(sizeof(int32_t) * (size_t)(kBinsPerEntity * s->n_entities + 1) * (size_t)want_list);
                        if (e == cudaSuccess) {
                            s->arena_capacity = (int)want;
                            s->list_capacity = (int)want_list;
                        } else { // leave a consistent (empty) workspace behind and try a smaller chunk
                            cudaGetLastError();
                            s->nodes.release();
                            s->rorder.release();
                            s->order.release();
                            s->node_cost.release();
                            s->arena_capacity = 0;
                            s->list_capacity = 0;
                            if (e != cudaErrorMemoryAllocation) return fail(EUCL_ERR_CUDA, std::string("workspace allocation: ") + cudaGetErrorString(e));
                            too_big = true;
                        }
                    }
                }
                if (too_big) {
                    if (rows_per_chunk <= 1)
                        return fail(EUCL_ERR_OUT_OF_MEMORY, "the node arena of a single row of pixels does not fit in device memory");
                    rows_per_chunk = (rows_per_chunk + 1) / 2;
                    continue;
                }
                if (fb.n > 1) EUCL_CUDA(s->node_frame.ensure(sizeof(int32_t) * (size_t)s->arena_capacity));
                if (want_cost) EUCL_CUDA(s->node_cost.ensure(sizeof(uint2) * (size_t)s->arena_capacity));
                Workspace ws = carve(s, dim, s->arena_capacity, s->list_capacity, fb);
                AovPlanes aov = aov_out;
                aov.cost = want_cost ? (uint2*)s->node_cost.ptr : nullptr;
                // profile mode: one event after every launch; family = 0 raygen, 1 intersect, 2 shade, 3 resolve
                std::vector<int> prof_family;
                auto mark = [&](int family) {
                    if (!o->profile) return;
                    if (s->prof_events.size() <= prof_family.size()) {
                        cudaEvent_t e = nullptr;
                        cudaEventCreate(&e);
                        s->prof_events.push_back(e);
                    }
                    cudaEventRecord(s->prof_events[prof_family.size()], s->stream);
                    prof_family.push_back(family);
                };
                // EUCL_DEBUG_SYNC=1: synchronise after every launch and name the one that faulted;
                // EUCL_POISON=1: fill the work buffers with 0x7F bytes (huge positive indices) first, so that a read of anything this
                // frame did not write turns into a deterministic fault instead of depending on stale data
                const bool debug_sync = env_int("EUCL_DEBUG_SYNC", 0) != 0;
                const bool poison = env_int("EUCL_POISON", 0) != 0;
                std::string fault;
                auto dbg = [&](const char* what, int level) {
                    if (!debug_sync || !fault.empty()) return;
                    cudaError_t e = cudaStreamSynchronize(s->stream);
                    if (e == cudaSuccess) e = cudaGetLastError();
                    if (e != cudaSuccess) fault = std::string(what) + " level " + std::to_string(level) + ": " + cudaGetErrorString(e);
                };
                if (o->pipeline == EUCL_PIPELINE_MEGAKERNEL && cam->max_depth > 24)
                    return fail(EUCL_ERR_SCENE_LIMIT, "megakernel pipeline supports max_depth <= 24");
                // everything one chunk puts on the stream: counters reset, kernels, counters back to the pinned mirror
                auto enqueue = [&]() -> uint32_t {
                    uint32_t launches = 0;
                    cudaMemsetAsync(s->small.ptr, 0, sizeof(int32_t) * kSmallInts, s->stream);
                    if (poison) {
                        cudaMemsetAsync(s->nodes.ptr, 0x7F, s->nodes.bytes, s->stream);
                        if (s->order.ptr) cudaMemsetAsync(s->order.ptr, 0x7F, s->order.bytes, s->stream);
                        if (s->rorder.ptr) cudaMemsetAsync(s->rorder.ptr, 0x7F, s->rorder.bytes, s->stream);
                    }
                    mark(-1);
                    if (o->pipeline == EUCL_PIPELINE_MEGAKERNEL) {
                        if (!rays) {
                            EUCL_PREC(launch_camera_entity)(dim, l, fp, ws);
                            dbg("k_camera_entity", 0);
                            launches += 1;
                        }
                        EUCL_PREC(launch_megakernel)(dim, l, fp, cp, ws, d_rgb, d_hit, aov, fb.ray_origins, fb.ray_directions);
                        mark(1);
                        launches += 1;
                    } else {
                        if (ws.frames) {
                            EUCL_PREC(launch_camera_entity)(dim, l, fp, ws);
                            dbg("k_camera_entity", 0);
                            launches += 1;
                        }
                        if (rays) EUCL_PREC(launch_raygen_rays)(dim, l, fp, cp, ws, d_hit, fb.ray_origins, fb.ray_directions);
                        else EUCL_PREC(launch_raygen)(dim, l, fp, cp, ws, d_hit);
                        dbg("k_raygen", 0);
                        mark(0);
                        for (int level = 0; level < (int)cam->max_depth; ++level) {
                            launches += EUCL_PREC(launch_intersect)(dim, l, ws, level);
                            dbg("k_intersect", level);
                            mark(1);
                            launches += EUCL_PREC(launch_shade)(dim, l, fp, cp, ws, level, d_hit);
                            dbg("k_shade", level);
                            mark(2);
                        }
                        // the nodes of the last level are background lookups (depth 0: mod.rs:157,183).  Measured and not kept:
                        // finishing them inside k_shade of the level above, from the child direction in registers (one launch
                        // and one ray record per node less, but the lookups then run at the heavy kernel's occupancy:
                        // 3d_room shade 7.14 + 0.47 -> 7.34 + 0.67 ms)
                        launches += EUCL_PREC(launch_shade)(dim, l, fp, cp, ws, (int)cam->max_depth, d_hit);
                        dbg("k_shade", (int)cam->max_depth);
                        mark(2);
                        launches += EUCL_PREC(launch_resolve_and_final)(dim, l, fp, cp, ws, d_rgb, aov);
                        dbg("k_resolve / k_final", 0);
                        mark(3);
                        launches += 1; // raygen
                    }
                    cudaMemcpyAsync(s->h_small, s->small.ptr, sizeof(int32_t) * kSmallInts, cudaMemcpyDeviceToHost, s->stream);
                    return launches;
                };
                // A chunk whose launch parameters repeat (a fixed pose rendered again: benchmarks, a paused camera, every rank
                // of a band-split frame) is replayed as ONE CUDA graph launch: the ~50 kernels of a frame then cost one
                // driver call on the host and run back to back on the device.  The first sighting of a parameter set
                // launches directly, the second captures, later ones replay.  EUCL_GRAPH=0 disables.
                uint64_t key = 1469598103934665603ull;
                auto mix = [&](const void* data, size_t bytes) {
                    const unsigned char* b = (const unsigned char*)data;
                    for (size_t k = 0; k < bytes; ++k) key = (key ^ b[k]) * 1099511628211ull;
                };
                mix(&fp, sizeof fp);
                mix(&cp, sizeof cp);
                mix(&ws, sizeof ws);
                {   // the members of Launch one by one (the struct has padding bytes)
                    const void* ptrs[] = {l.stream, l.blob, l.side};
                    const unsigned long long nums[] = {l.smem_bytes, l.smem_scene, (unsigned long long)l.grid_max, (unsigned long long)l.grid_light,
                                                       (unsigned long long)l.grid_shade, (unsigned long long)l.grid_mem, l.shade_light_mask,
                                                       l.shade_heavy_mask, (unsigned long long)l.grid_light_k2,
                                                       (unsigned long long)l.light_capable, (unsigned long long)l.n_cull,
                                                       (unsigned long long)l.grid_background};
                    mix(ptrs, sizeof ptrs);
                    mix(nums, sizeof nums);
                }
                mix(&d_rgb, sizeof d_rgb);
                mix(&d_hit, sizeof d_hit);
                // the AOV planes a chunk writes (null = not wanted) and the cost buffer: a graph captured with or without
                // them never stands in for the other
                mix(&aov, sizeof aov);
                const int pipeline_id = o->pipeline;
                mix(&pipeline_id, sizeof pipeline_id);
                const uint32_t depth_id = cam->max_depth;
                mix(&depth_id, sizeof depth_id);
                // a batch: the graph reads the table the caller's poses were uploaded to, and it is keyed by its contents
                // too, so that a changed pose or time is never taken for a repeated batch
                if (fb.n > 1) mix(&fb.table_key, sizeof fb.table_key);
                // a ray call: tagged, so that a ray call and a render whose other parameters coincide never stand in for
                // each other, and keyed by the arrays it reads (their contents are read at replay time)
                if (rays) {
                    const uint64_t ray_id[] = {0x52415953ull /* "RAYS" */, (uint64_t)(uintptr_t)fb.ray_origins,
                                               (uint64_t)(uintptr_t)fb.ray_directions, (uint64_t)o->height * o->width, o->width};
                    mix(ray_id, sizeof ray_id);
                }
                // (not while the scene is still choosing its ray-grouping mode: capture time would distort the comparison;
                // ray calls take no part in that choice)
                const bool graph_ok = env_int("EUCL_GRAPH", 1) && !o->profile && !debug_sync && !poison &&
                                      (s->ray_bins_mode >= 0 || o->pipeline != EUCL_PIPELINE_WAVEFRONT || rays);
                if (graph_ok && s->graph_exec && s->graph_key == key) {
                    EUCL_CUDA(cudaGraphLaunch(s->graph_exec, s->stream));
                    st.launches += s->graph_launches;
                    st.graph_replays += 1;
                } else if (graph_ok && s->seen_key == key) {
                    if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
                    s->graph_exec = nullptr;
                    cudaGraph_t graph = nullptr;
                    // one capture at a time in the process (the pipelines of a split frame capture in the same frame)
                    static std::mutex capture_mutex;
                    std::unique_lock<std::mutex> capture_lock(capture_mutex);
                    EUCL_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
                    const uint32_t launches = enqueue();
                    cudaError_t ce = cudaStreamEndCapture(s->stream, &graph);
                    if (ce == cudaSuccess) ce = cudaGraphInstantiate(&s->graph_exec, graph, 0);
                    capture_lock.unlock();
                    if (graph) cudaGraphDestroy(graph);
                    if (ce != cudaSuccess) { // not capturable here (e.g. a caller's stream in a state that forbids it): launch directly
                        cudaGetLastError();
                        s->graph_exec = nullptr;
                        s->seen_key = 0;
                        st.launches += enqueue();
                    } else {
                        s->graph_key = key;
                        s->graph_launches = launches;
                        EUCL_CUDA(cudaGraphLaunch(s->graph_exec, s->stream));
                        st.launches += launches;
                        st.graph_replays += 1;
                    }
                } else {
                    s->seen_key = key;
                    st.launches += enqueue();
                }
                if (!fault.empty()) return fail(EUCL_ERR_CUDA, "EUCL_DEBUG_SYNC: " + fault);
                EUCL_CUDA(cudaStreamSynchronize(s->stream));
                EUCL_CUDA(cudaGetLastError());
                for (size_t k = 1; k < prof_family.size(); ++k) {
                    float ms = 0.f;
                    cudaEventElapsedTime(&ms, s->prof_events[k - 1], s->prof_events[k]);
                    float* slot = prof_family[k] == 0 ? &st.ms_raygen : prof_family[k] == 1 ? &st.ms_intersect
                                  : prof_family[k] == 2 ? &st.ms_shade : &st.ms_resolve;
                    *slot += ms;
                }
                if (env_int("EUCL_DUMP_LEVELS", 0) && !s->h_small[SmallLayout::overflow]) { // diagnostics: per-level counts, bins, launch times
                    for (uint32_t lv = 0; lv <= cam->max_depth; ++lv) {
                        fprintf(stderr, "level %2u count %9d | bins", lv, s->h_small[SmallLayout::count + lv]);
                        for (int b = 0; b < ws.n_bins && ws.n_bins > 1; ++b) fprintf(stderr, " %d", s->h_small[SmallLayout::bins + lv * kMaxBins + b]);
                        fprintf(stderr, " | rbins");
                        for (int b = 0; b < kRayBins; ++b) fprintf(stderr, " %d", s->h_small[SmallLayout::rbins + lv * kRayBins + b]);
                        fprintf(stderr, "\n");
                    }
                    for (size_t k = 1; k < prof_family.size(); ++k) {
                        float ms = 0.f;
                        cudaEventElapsedTime(&ms, s->prof_events[k - 1], s->prof_events[k]);
                        fprintf(stderr, "launch %2zu family %d %.3f ms\n", k, prof_family[k], ms);
                    }
                }
                if (s->h_small[SmallLayout::overflow] == 2)
                    return fail(EUCL_ERR_CUDA, "internal error: a queue index list and its level count disagree");
                if (s->h_small[SmallLayout::overflow]) {
                    // levels after the overflowing one were skipped, so the counts are a lower bound only
                    long long need = 0;
                    for (uint32_t lv = 0; lv <= cam->max_depth; ++lv) need += s->h_small[SmallLayout::count + lv];
                    if (s->h_small[SmallLayout::overflow] == 3) { // a level outgrew the index lists (they hold one level each)
                        s->list_factor = std::max(s->list_factor * 1.5, 1.0);
                    } else {
                        double factor = (double)need / (double)cp.n_pixels * 1.05 + 0.05;
                        s->arena_factor = std::max(s->arena_factor * 1.5, factor);
                    }
                    st.retries += 1;
                    if (st.retries > 32) return fail(EUCL_ERR_OUT_OF_MEMORY, "node arena keeps overflowing");
                    continue;
                }
                break;
            }
            row0 += cp.n_rows;
            st.pixels += (uint64_t)cp.n_pixels;
            // camera in no entity: checkerboard pixels, Universe::trace is never called (mod.rs:385-396).  In a batch with
            // some frames traced, level 0 holds the checkerboard pixels of the others: they are not counted either.
            const bool traced = s->h_small[SmallLayout::cam_entity] >= 0;
            for (uint32_t lv = 0; traced && lv <= cam->max_depth; ++lv) {
                uint64_t c = o->pipeline == EUCL_PIPELINE_MEGAKERNEL
                                 ? ((const unsigned long long*)(s->h_small + SmallLayout::mega64))[lv]
                                 : (uint64_t)s->h_small[SmallLayout::count + lv];
                if (lv == 0) c -= (uint64_t)s->h_small[SmallLayout::untraced];
                st.level_counts[lv] += c;
                st.nodes += c;
                if (lv < cam->max_depth) st.segments += c;
            }
        }
    }
    EUCL_CUDA(cudaEventRecord(s->ev[1], s->stream));
    EUCL_CUDA(cudaEventSynchronize(s->ev[1]));
    EUCL_CUDA(cudaEventElapsedTime(&st.ms_total, s->ev[0], s->ev[1]));
    // A frame that had to grow its arena over-shot (capacity grows by half each retry).  Now that the frame's real node
    // count is known, the scene keeps that plus a few per cent and gives the rest back: the next frame of this size
    // allocates once more, exactly, and nothing afterwards.
    if (st.retries > 0 && st.pixels > 0 && st.nodes > 0 && o->pipeline == EUCL_PIPELINE_WAVEFRONT && st.pixels == (uint64_t)my_rows * width) {
        uint64_t max_level = 0;
        for (uint32_t lv = 0; lv <= cam->max_depth; ++lv) max_level = std::max<uint64_t>(max_level, st.level_counts[lv]);
        const double tight = (double)st.nodes / (double)st.pixels * 1.03 + 0.02;
        const double tight_list = std::max(1.0, (double)max_level / (double)st.pixels * 1.03);
        if ((double)s->arena_capacity > ((double)st.pixels * tight + 1024) * 1.08) {
            s->arena_factor = tight;
            s->list_factor = tight_list;
            s->nodes.release();
            s->order.release();
            s->rorder.release();
            s->node_cost.release();
            s->arena_capacity = 0;
            s->list_capacity = 0;
            if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
            s->graph_exec = nullptr;
            s->graph_key = s->seen_key = 0;
        }
    }
    // (a split frame is judged as a whole: render_split).  A ray batch is not a frame of its size: it never tunes.
    if (!rays) {
        if (sub_stride <= 1) tune_grouping(s, st, o->pipeline);
        s->warm_frames++;
    }
    st.ray_grouping = s->ray_bins_now && s->rorder.ptr != nullptr && o->pipeline == EUCL_PIPELINE_WAVEFRONT ? 1u : 0u;
    if (stats) *stats = st;
    return EUCL_OK;
}

// One more scene over the leader's uploaded blob and textures, with streams, events, counters and (later) an arena of its own.
int add_twin(EuclScene* s) {
    EuclScene* t = new EuclScene();
    t->is_twin = true;
    t->device = s->device;
    t->dim = s->dim;
    t->sm_count = s->sm_count;
    t->blob_bytes = s->blob_bytes;
    t->smem_bytes = s->smem_bytes;
    t->smem_scene = s->smem_scene;
    t->shade_light_mask = s->shade_light_mask;
    t->shade_heavy_mask = s->shade_heavy_mask;
    t->d_blob = s->d_blob;
    t->n_cull = s->n_cull;
    t->light_capable = s->light_capable;
    t->n_entities = s->n_entities;
    t->real_bytes = s->real_bytes;
    cudaError_t e = cudaStreamCreateWithFlags(&t->own_stream, cudaStreamNonBlocking);
    t->stream = t->own_stream;
    if (e == cudaSuccess) e = cudaEventCreate(&t->ev[0]);
    if (e == cudaSuccess) e = cudaEventCreate(&t->ev[1]);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&t->side_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->ev_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&t->h_small, sizeof(int32_t) * kSmallInts);
    for (int k = 0; k < 3 && e == cudaSuccess; ++k)
        if (!s->ev_split[k]) e = cudaEventCreateWithFlags(&s->ev_split[k], k == 1 ? cudaEventDisableTiming : cudaEventDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        eucl_scene_destroy(t);
        return fail(e == cudaErrorMemoryAllocation ? EUCL_ERR_OUT_OF_MEMORY : EUCL_ERR_CUDA, std::string("split pipeline: ") + cudaGetErrorString(e));
    }
    s->twins.push_back(t);
    s->workers.push_back(new Worker());
    s->workers.back()->start();
    return EUCL_OK;
}

constexpr int kMaxSplit = 8;

// Environment::render for this rank's rows, as ONE pipeline or as k side by side.
//
// A frame is ~50 dependent launches (raygen, then per level intersect and shade, then the resolves), and every one
// of them ends with a tail in which the slowest rays of the level finish on a mostly idle GPU: about 0.55 ms per
// 3d_room frame whatever its size (profiles/r2_band_scaling.txt) -- 3 % of a 4K frame on one GPU, 20 % of an
// eighth of it.  Independent pipelines, each on every k-th 16-row band and on streams of its own, fill each other's
// tails.  The picture cannot depend on it: pixels are independent (mod.rs:316-348).
int render_split(EuclScene* s, const FrameBatch& fb, const EuclRenderOpts* o, uint8_t* d_rgb, int32_t* d_hit, const AovPlanes& aov,
                 EuclStats* stats) {
    const uint32_t my_rows = eucl_band_rows_for_rank(o);
    uint32_t world = o->band_world > 1 ? o->band_world : 1, rank = world > 1 ? o->band_rank : 0, band = o->band_rows;
    if (band == 0) { // one band: the frame belongs to rank 0
        world = 1;
        rank = 0;
        band = (uint32_t)std::max(1, env_int("EUCL_SPLIT_BAND_ROWS", 16));
    }
    int k = std::min(kMaxSplit, env_int("EUCL_SPLIT", EUCL_SPLIT_DEFAULT));
    k = (int)std::min<uint32_t>((uint32_t)std::max(k, 1), my_rows / band); // a band or more for every pipeline
    if (o->pipeline != EUCL_PIPELINE_WAVEFRONT || (long long)my_rows * o->width < (long long)env_int("EUCL_SPLIT_MIN_PIXELS", 1 << 16)) k = 1;
    if (k <= 1) return render_impl(s, fb, o, d_rgb, d_hit, aov, stats);
    while ((int)s->twins.size() < k - 1) {
        int rc = add_twin(s);
        if (rc != EUCL_OK) return rc;
    }
    choose_grouping(s);
    EuclRenderOpts opts[kMaxSplit];
    EuclStats part[kMaxSplit];
    int rc[kMaxSplit];
    std::string err[kMaxSplit];
    for (int p = 0; p < k; ++p) {
        opts[p] = *o;
        opts[p].band_rows = band;
        opts[p].band_world = (uint32_t)k * world;
        opts[p].band_rank = rank + (uint32_t)p * world;
        part[p] = EuclStats{};
        rc[p] = EUCL_OK;
    }
    EUCL_CUDA(cudaEventRecord(s->ev_split[0], s->stream));
    EUCL_CUDA(cudaEventRecord(s->ev_split[1], s->stream)); // the other pipelines start after whatever the caller's stream holds
    // per-launch profiling and the debugging modes run the pipelines one after the other on the caller's thread
    const bool serial = o->profile || env_int("EUCL_DEBUG_SYNC", 0) || env_int("EUCL_POISON", 0);
    auto pipeline = [&](int p) {
        EuclScene* t = s->twins[p - 1];
        cudaSetDevice(t->device);
        rc[p] = render_impl(t, fb, &opts[p], d_rgb, d_hit, aov, &part[p], k, p);
        if (rc[p] != EUCL_OK) err[p] = eucl_last_error();
    };
    for (int p = 1; p < k; ++p) {
        EuclScene* t = s->twins[p - 1];
        t->ray_bins_mode = s->ray_bins_mode;
        t->ray_bins_now = s->ray_bins_now;
        EUCL_CUDA(cudaStreamWaitEvent(t->stream, s->ev_split[1], 0));
    }
    // (no early return between here and the last wait(): the helper threads work on this frame's locals)
    for (int p = 1; p < k && !serial; ++p) s->workers[p - 1]->run([&pipeline, p] { pipeline(p); });
    rc[0] = render_impl(s, fb, &opts[0], d_rgb, d_hit, aov, &part[0], k, 0);
    for (int p = 1; p < k; ++p) {
        if (serial) pipeline(p);
        else s->workers[p - 1]->wait();
    }
    if (rc[0] != EUCL_OK) return rc[0];
    for (int p = 1; p < k; ++p)
        if (rc[p] != EUCL_OK) return fail(rc[p], err[p]);
    for (int p = 1; p < k; ++p) { // the caller's stream continues after every pipeline
        EuclScene* t = s->twins[p - 1];
        EUCL_CUDA(cudaEventRecord(t->ev_done, t->stream));
        EUCL_CUDA(cudaStreamWaitEvent(s->stream, t->ev_done, 0));
    }
    EUCL_CUDA(cudaEventRecord(s->ev_split[2], s->stream));
    EUCL_CUDA(cudaEventSynchronize(s->ev_split[2]));
    EuclStats st = part[0];
    EUCL_CUDA(cudaEventElapsedTime(&st.ms_total, s->ev_split[0], s->ev_split[2]));
    for (int p = 1; p < k; ++p) {
        const EuclStats& b = part[p];
        st.pixels += b.pixels;
        st.segments += b.segments;
        st.nodes += b.nodes;
        for (uint32_t lv = 0; lv < EUCL_MAX_LEVELS; ++lv) st.level_counts[lv] += b.level_counts[lv];
        st.launches += b.launches;
        st.retries += b.retries;
        st.graph_replays = std::min(st.graph_replays, b.graph_replays);
        st.ms_raygen += b.ms_raygen;
        st.ms_intersect += b.ms_intersect;
        st.ms_shade += b.ms_shade;
        st.ms_resolve += b.ms_resolve;
    }
    if (!fb.ray_origins) tune_grouping(s, st, o->pipeline);
    if (stats) *stats = st;
    return EUCL_OK;
}

int check_args(EuclScene* s, const EuclCamera* cam, const EuclRenderOpts* o) {
    if (!s || !cam || !o) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: null argument");
    if (cam->dim != s->dim) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: camera dimension does not match the scene");
    if (o->width == 0 || o->height == 0 || o->width > (1u << 20) || o->height > (1u << 20))
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: bad frame size");
    if (cam->max_depth >= EUCL_MAX_LEVELS) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: max_depth too large");
    if (o->band_world > 1 && o->band_rank >= o->band_world) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: band_rank >= band_world");
    if (o->pipeline != EUCL_PIPELINE_WAVEFRONT && o->pipeline != EUCL_PIPELINE_MEGAKERNEL)
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: unknown pipeline");
    return EUCL_OK;
}

// eucl_render_frames*: every frame as eucl_render would take it, one max_depth, no band split, and a virtual frame whose
// pixels the chunks can index with 32-bit integers.  Checked before any device is touched.
int check_frames(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o) {
    if (!s || !frames || !o) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: null argument");
    if (n_frames == 0) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: no frames");
    for (uint32_t k = 0; k < n_frames; ++k) {
        const int st = check_args(s, &frames[k].camera, o);
        if (st != EUCL_OK) return st;
        if (frames[k].camera.max_depth != frames[0].camera.max_depth)
            return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: the frames of a batch must share max_depth");
    }
    if (o->band_world > 1) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: band-split batches are not supported");
    if (o->compact_rows) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: compact_rows is not supported");
    if ((uint64_t)n_frames * o->height * o->width > 0x7fffffffull)
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: more than 2^31 - 1 pixels in one batch");
    return EUCL_OK;
}

// The batch of `n` frames and the virtual frame they form.  K > 1: the frame constants are computed on the host like
// a single frame's and uploaded, stream-ordered before the first launch (and outside any graph capture).
int prepare_batch(EuclScene* s, const EuclFrame* frames, uint32_t n, const EuclRenderOpts* o, FrameBatch* fb,
                  EuclRenderOpts* virt) {
    *fb = FrameBatch{frames, n, o->height, nullptr, 0};
    *virt = *o;
    virt->height = n * o->height;
    if (n == 1) return EUCL_OK;
    if (s->h_frame_table_cap < n) {
        if (s->h_frame_table) cudaFreeHost(s->h_frame_table);
        s->h_frame_table = nullptr;
        s->h_frame_table_cap = 0;
        EUCL_CUDA(cudaMallocHost((void**)&s->h_frame_table, sizeof(FrameParams) * n));
        s->h_frame_table_cap = n;
    }
    uint64_t key = 1469598103934665603ull;
    for (uint32_t k = 0; k < n; ++k) {
        EuclRenderOpts one = *o;
        one.time_seconds = frames[k].time_seconds;
        frame_params(frames[k].camera, one, s->real_bytes, &s->h_frame_table[k]);
        const unsigned char* b = (const unsigned char*)&s->h_frame_table[k];
        for (size_t i = 0; i < sizeof(FrameParams); ++i) key = (key ^ b[i]) * 1099511628211ull;
    }
    EUCL_CUDA(s->frame_table.ensure(sizeof(FrameParams) * n));
    EUCL_CUDA(cudaMemcpyAsync(s->frame_table.ptr, s->h_frame_table, sizeof(FrameParams) * n, cudaMemcpyHostToDevice, s->stream));
    fb->d_table = (const FrameParams*)s->frame_table.ptr;
    fb->table_key = key;
    return EUCL_OK;
}

// Device-output render of `n` frames (eucl_render_device: n = 1), or -- `rays` -- of a ray call's virtual frame (`o` then
// is that frame and `frames` is rays->frames).
int render_frames_to_device(EuclScene* s, const EuclFrame* frames, uint32_t n, const EuclRenderOpts* o, uint8_t* d_rgb,
                            int32_t* d_hit, const AovPlanes& aov, EuclStats* stats, const FrameBatch* rays = nullptr) {
    if (rays) return render_split(s, *rays, o, d_rgb, d_hit, aov, stats);
    FrameBatch fb;
    EuclRenderOpts virt;
    const int st = prepare_batch(s, frames, n, o, &fb, &virt);
    if (st != EUCL_OK) return st;
    return render_split(s, fb, &virt, d_rgb, d_hit, aov, stats);
}

// eucl_render_aovs*: at least one plane.  Checked before any device is touched.
int check_aovs(const EuclAovs* a, const char* fn) {
    if (!a || !(a->depth || a->position || a->normal || a->segments || a->levels))
        return fail(EUCL_ERR_INVALID_ARGUMENT, std::string(fn) + ": no AOV plane requested (use the plain entry point)");
    return EUCL_OK;
}
AovPlanes aov_planes(const EuclAovs* a) {
    if (!a) return AovPlanes{};
    return AovPlanes{a->depth, a->position, a->normal, a->segments, a->levels, nullptr};
}

// Host-output render of `n` frames (arguments already checked): rendered into the scene's device buffers, then copied out.
// A rank of a band-split render (band_world > 1, a single frame) renders its rows compactly on the device and then copies
// each band to its place in the caller's frame: rows of other ranks are never read or written, so N ranks can fill ONE
// host frame (shared pinned memory) over their own PCIe links at the same time.  The AOV planes go the same way.
int render_to_host(EuclScene* s, const EuclFrame* frames, uint32_t n, const EuclRenderOpts* o, uint8_t* out_rgb8,
                   int32_t* out_hit_ids, const EuclAovs* aovs, EuclStats* stats, const FrameBatch* rays = nullptr) {
    EUCL_CUDA(cudaSetDevice(s->device));
    const bool scatter = !o->compact_rows && o->band_world > 1;
    const size_t my_rows = eucl_band_rows_for_rank(o);
    const size_t rows = (o->compact_rows || scatter) ? my_rows : (size_t)n * o->height;
    const size_t pixels = rows * (size_t)o->width;
    const bool want_hit = o->want_hit_ids && out_hit_ids;
    EUCL_CUDA(s->frame.ensure(std::max<size_t>(pixels, 1) * 3));
    if (want_hit) EUCL_CUDA(s->hit_ids.ensure(std::max<size_t>(pixels, 1) * 4));
    // AOV planes: host pointer, bytes per pixel, device copy carved from one staging buffer
    const AovPlanes want = aov_planes(aovs);
    void* host[5] = {want.depth, want.position, want.normal, want.segments, want.levels};
    const size_t px_bytes[5] = {4, 4 * (size_t)s->dim, 4 * (size_t)s->dim, 4, 4};
    void* dev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t stage_bytes = 0;
    for (int k = 0; k < 5; ++k)
        if (host[k]) stage_bytes += align16(std::max<size_t>(pixels, 1) * px_bytes[k]);
    if (stage_bytes) {
        EUCL_CUDA(s->aov_stage.ensure(stage_bytes));
        uint8_t* p = (uint8_t*)s->aov_stage.ptr;
        for (int k = 0; k < 5; ++k)
            if (host[k]) {
                dev[k] = p;
                p += align16(std::max<size_t>(pixels, 1) * px_bytes[k]);
            }
    }
    const AovPlanes d_aov{(float*)dev[0], (float*)dev[1], (float*)dev[2], (uint32_t*)dev[3], (uint32_t*)dev[4], nullptr};
    EuclRenderOpts opts = *o;
    opts.want_hit_ids = want_hit ? 1 : 0;
    if (scatter) opts.compact_rows = 1;
    const int st = render_frames_to_device(s, frames, n, &opts, (uint8_t*)s->frame.ptr, want_hit ? (int32_t*)s->hit_ids.ptr : nullptr,
                                           d_aov, stats, rays);
    if (st != EUCL_OK) return st;
    if (!scatter) {
        EUCL_CUDA(cudaMemcpyAsync(out_rgb8, s->frame.ptr, pixels * 3, cudaMemcpyDeviceToHost, s->stream));
        if (want_hit) EUCL_CUDA(cudaMemcpyAsync(out_hit_ids, s->hit_ids.ptr, pixels * 4, cudaMemcpyDeviceToHost, s->stream));
        for (int k = 0; k < 5; ++k)
            if (host[k]) EUCL_CUDA(cudaMemcpyAsync(host[k], dev[k], pixels * px_bytes[k], cudaMemcpyDeviceToHost, s->stream));
    } else if (my_rows > 0) {
        // band k of this rank: compact rows [k * band, ...) -> frame rows [(k * world + rank) * band, ...)
        const size_t band = o->band_rows ? o->band_rows : o->height, world = o->band_world;
        const size_t full = my_rows / band, tail = my_rows % band; // whole bands, rows of a last partial band
        auto copy_bands = [&](void* dst, const void* src, size_t px_bytes) -> cudaError_t {
            const size_t band_bytes = band * o->width * px_bytes;
            uint8_t* d = (uint8_t*)dst + (size_t)o->band_rank * band_bytes;
            cudaError_t e = cudaSuccess;
            if (full) e = cudaMemcpy2DAsync(d, world * band_bytes, src, band_bytes, band_bytes, full, cudaMemcpyDeviceToHost, s->stream);
            if (e == cudaSuccess && tail)
                e = cudaMemcpyAsync(d + full * world * band_bytes, (const uint8_t*)src + full * band_bytes, tail * o->width * px_bytes,
                                    cudaMemcpyDeviceToHost, s->stream);
            return e;
        };
        EUCL_CUDA(copy_bands(out_rgb8, s->frame.ptr, 3));
        if (want_hit) EUCL_CUDA(copy_bands(out_hit_ids, s->hit_ids.ptr, 4));
        for (int k = 0; k < 5; ++k)
            if (host[k]) EUCL_CUDA(copy_bands(host[k], dev[k], px_bytes[k]));
    }
    EUCL_CUDA(cudaStreamSynchronize(s->stream));
    return EUCL_OK;
}

} // namespace

extern "C" {

int eucl_render_device(EuclScene* s, const EuclCamera* cam, const EuclRenderOpts* o, void* d_out_rgb8, void* d_out_hit_ids,
                       EuclStats* stats) {
    int st = check_args(s, cam, o);
    if (st != EUCL_OK) return st;
    if (!d_out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_device: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    const EuclFrame frame{*cam, o->time_seconds};
    return render_frames_to_device(s, &frame, 1, o, (uint8_t*)d_out_rgb8, o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr,
                                   AovPlanes{}, stats);
}

int eucl_render_frames_device(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o,
                              void* d_out_rgb8, void* d_out_hit_ids, EuclStats* stats) {
    int st = check_frames(s, frames, n_frames, o);
    if (st != EUCL_OK) return st;
    if (!d_out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames_device: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    return render_frames_to_device(s, frames, n_frames, o, (uint8_t*)d_out_rgb8,
                                   o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr, AovPlanes{}, stats);
}

int eucl_render_frames(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, uint8_t* out_rgb8,
                       int32_t* out_hit_ids, EuclStats* stats) {
    int st = check_frames(s, frames, n_frames, o);
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: null output");
    return render_to_host(s, frames, n_frames, o, out_rgb8, out_hit_ids, nullptr, stats);
}

int eucl_render(EuclScene* s, const EuclCamera* cam, const EuclRenderOpts* o, uint8_t* out_rgb8, int32_t* out_hit_ids,
                EuclStats* stats) {
    int st = check_args(s, cam, o);
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: null output");
    const EuclFrame frame{*cam, o->time_seconds};
    return render_to_host(s, &frame, 1, o, out_rgb8, out_hit_ids, nullptr, stats);
}

// One frame: what eucl_render accepts; K > 1 frames: what eucl_render_frames accepts.
static int check_aov_call(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, const EuclAovs* aovs,
                          const char* fn) {
    int st = n_frames == 1 ? check_args(s, frames ? &frames[0].camera : nullptr, o) : check_frames(s, frames, n_frames, o);
    if (st == EUCL_OK) st = check_aovs(aovs, fn);
    return st;
}

int eucl_render_aovs(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, uint8_t* out_rgb8,
                     int32_t* out_hit_ids, const EuclAovs* aovs, EuclStats* stats) {
    const int st = check_aov_call(s, frames, n_frames, o, aovs, "eucl_render_aovs");
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_aovs: null output");
    return render_to_host(s, frames, n_frames, o, out_rgb8, out_hit_ids, aovs, stats);
}

int eucl_render_aovs_device(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, void* d_out_rgb8,
                            void* d_out_hit_ids, const EuclAovs* d_aovs, EuclStats* stats) {
    const int st = check_aov_call(s, frames, n_frames, o, d_aovs, "eucl_render_aovs_device");
    if (st != EUCL_OK) return st;
    if (!d_out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_aovs_device: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    return render_frames_to_device(s, frames, n_frames, o, (uint8_t*)d_out_rgb8,
                                   o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr, aov_planes(d_aovs), stats);
}

} // extern "C"

namespace {

static_assert(sizeof(EuclRays) == 48, "EuclRays is part of the C ABI");

// eucl_trace_rays*: checked before any device is touched.
int check_rays(EuclScene* s, const EuclRays* r, const void* out, const char* fn) {
    const std::string f(fn);
    if (!s || !r) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": null argument");
    if (r->n == 0 || r->n > 0x7fffffffu) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": n must be 1 .. 2^31 - 1");
    if (!r->origins || !r->directions) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": null ray array");
    if (!out) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": null output");
    if (r->width > 1 && r->n % r->width != 0) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": width does not divide n");
    if (r->max_depth + 1ull > EUCL_MAX_LEVELS) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": max_depth too large");
    if (r->pipeline != EUCL_PIPELINE_WAVEFRONT && r->pipeline != EUCL_PIPELINE_MEGAKERNEL)
        return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": unknown pipeline");
    return EUCL_OK;
}

// The virtual frame of a ray call (n / width rows of width) and its batch: one "frame" that carries the depth and the
// time, and the device rays.
struct RayCall {
    EuclFrame frame;
    EuclRenderOpts opts;
    FrameBatch fb;
    RayCall(const EuclScene* s, const EuclRays* r, const double* d_origins, const double* d_directions, bool want_hit) {
        std::memset(&frame, 0, sizeof frame);
        frame.camera.dim = s->dim;
        frame.camera.max_depth = r->max_depth;
        frame.time_seconds = r->time_seconds;
        const uint32_t w = r->width > 1 ? r->width : 1;
        opts = EuclRenderOpts{};
        opts.width = w;
        opts.height = r->n / w;
        opts.time_seconds = r->time_seconds;
        opts.pipeline = r->pipeline;
        opts.want_hit_ids = want_hit ? 1 : 0;
        opts.profile = r->profile;
        fb = FrameBatch{&frame, 1, opts.height, nullptr, 0};
        fb.ray_origins = d_origins;
        fb.ray_directions = d_directions;
    }
};

const EuclAovs* any_plane(const EuclAovs* a) {
    return a && (a->depth || a->position || a->normal || a->segments || a->levels) ? a : nullptr;
}

} // namespace

extern "C" {

int eucl_trace_rays(EuclScene* s, const EuclRays* r, uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclAovs* aovs,
                    EuclStats* stats) {
    const int st = check_rays(s, r, out_rgb8, "eucl_trace_rays");
    if (st != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    // staged before the first launch, on the scene's stream and outside any graph capture: a replayed graph reads them
    const size_t bytes = sizeof(double) * (size_t)s->dim * r->n;
    EUCL_CUDA(s->ray_stage.ensure(2 * bytes));
    double* d_o = (double*)s->ray_stage.ptr;
    double* d_d = (double*)((uint8_t*)s->ray_stage.ptr + bytes);
    EUCL_CUDA(cudaMemcpyAsync(d_o, r->origins, bytes, cudaMemcpyHostToDevice, s->stream));
    EUCL_CUDA(cudaMemcpyAsync(d_d, r->directions, bytes, cudaMemcpyHostToDevice, s->stream));
    RayCall call(s, r, d_o, d_d, out_hit_ids != nullptr);
    return render_to_host(s, &call.frame, 1, &call.opts, out_rgb8, out_hit_ids, any_plane(aovs), stats, &call.fb);
}

int eucl_trace_rays_device(EuclScene* s, const EuclRays* r, void* d_out_rgb8, void* d_out_hit_ids, const EuclAovs* d_aovs,
                           EuclStats* stats) {
    const int st = check_rays(s, r, d_out_rgb8, "eucl_trace_rays_device");
    if (st != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    RayCall call(s, r, r->origins, r->directions, d_out_hit_ids != nullptr);
    return render_frames_to_device(s, &call.frame, 1, &call.opts, (uint8_t*)d_out_rgb8, (int32_t*)d_out_hit_ids,
                                   aov_planes(any_plane(d_aovs)), stats, &call.fb);
}

int eucl_scene_memory(const EuclScene* s, uint64_t* arena_bytes, uint64_t* list_bytes, uint64_t* node_capacity) {
    if (!s) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_memory: null scene");
    uint64_t arena = s->nodes.bytes, lists = s->order.bytes + s->rorder.bytes, cap = (uint64_t)s->arena_capacity;
    for (const EuclScene* t : s->twins) { // a split scene holds one arena per pipeline
        arena += t->nodes.bytes;
        lists += t->order.bytes + t->rorder.bytes;
        cap += (uint64_t)t->arena_capacity;
    }
    if (arena_bytes) *arena_bytes = arena;
    if (list_bytes) *list_bytes = lists;
    if (node_capacity) *node_capacity = cap;
    return EUCL_OK;
}

int eucl_scene_set_stream(EuclScene* s, void* cuda_stream) {
    if (!s) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_set_stream: null scene");
    EUCL_CUDA(cudaSetDevice(s->device));
    EUCL_CUDA(cudaStreamSynchronize(s->stream));
    s->stream = cuda_stream ? (cudaStream_t)cuda_stream : s->own_stream;
    return EUCL_OK;
}

int eucl_trace_path(EuclScene* s, const double* location, const double* direction, double distance, double* out_location,
                    double* out_direction) {
    if (!s || !location || !direction || !out_location || !out_direction)
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_trace_path: null argument");
    EUCL_CUDA(cudaSetDevice(s->device));
    const int D = s->dim;
    EUCL_CUDA(s->path_io.ensure(sizeof(double) * 4 * EUCL_MAX_DIM + 16));
    double* d_in = (double*)s->path_io.ptr;
    double* d_out = d_in + 2 * EUCL_MAX_DIM;
    int* d_found = (int*)(d_out + 2 * EUCL_MAX_DIM);
    double h_in[2 * EUCL_MAX_DIM] = {0};
    for (int k = 0; k < D; ++k) {
        h_in[k] = location[k];
        h_in[D + k] = direction[k];
    }
    EUCL_CUDA(cudaMemcpyAsync(d_in, h_in, sizeof h_in, cudaMemcpyHostToDevice, s->stream));
    Launch l{s->stream, s->d_blob, s->smem_bytes, s->smem_scene, 1, 1, 1, 1, 1ull, 0ull, 1, 0, 0, nullptr, nullptr, nullptr};
    EUCL_PREC(launch_trace_path)(D, l, d_in, distance, d_out, d_found);
    double h_out[2 * EUCL_MAX_DIM];
    int h_found = 0;
    EUCL_CUDA(cudaMemcpyAsync(h_out, d_out, sizeof h_out, cudaMemcpyDeviceToHost, s->stream));
    EUCL_CUDA(cudaMemcpyAsync(&h_found, d_found, sizeof h_found, cudaMemcpyDeviceToHost, s->stream));
    EUCL_CUDA(cudaStreamSynchronize(s->stream));
    EUCL_CUDA(cudaGetLastError());
    if (h_found < 0) return fail(EUCL_ERR_SCENE_LIMIT, "eucl_trace_path: more than 100000 surface crossings");
    if (h_found == 0) return 1; /* the start point lies in no entity: Option::None in the reference */
    for (int k = 0; k < D; ++k) {
        out_location[k] = h_out[k];
        out_direction[k] = h_out[D + k];
    }
    return EUCL_OK;
}

int eucl_device_malloc(int device, uint64_t bytes, void** d_ptr) {
    if (!d_ptr || bytes == 0) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_device_malloc: bad argument");
    if (eucl_device_count() <= 0) return fail(EUCL_ERR_NO_DEVICE, "no CUDA device available");
    EUCL_CUDA(cudaSetDevice(device));
    EUCL_CUDA(cudaMalloc(d_ptr, (size_t)bytes));
    return EUCL_OK;
}

int eucl_device_free(int device, void* d_ptr) {
    if (!d_ptr) return EUCL_OK;
    EUCL_CUDA(cudaSetDevice(device));
    EUCL_CUDA(cudaFree(d_ptr));
    return EUCL_OK;
}

int eucl_host_register(void* ptr, uint64_t bytes) {
    if (!ptr || bytes == 0) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_host_register: bad argument");
    if (eucl_device_count() <= 0) return fail(EUCL_ERR_NO_DEVICE, "no CUDA device available");
    EUCL_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
    return EUCL_OK;
}

int eucl_host_unregister(void* ptr) {
    if (!ptr) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_host_unregister: null argument");
    EUCL_CUDA(cudaHostUnregister(ptr));
    return EUCL_OK;
}

int eucl_ipc_export(void* d_ptr, uint8_t handle[EUCL_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) <= EUCL_IPC_HANDLE_BYTES, "IPC handle size");
    if (!d_ptr || !handle) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_ipc_export: null argument");
    cudaIpcMemHandle_t h;
    EUCL_CUDA(cudaIpcGetMemHandle(&h, d_ptr));
    std::memset(handle, 0, EUCL_IPC_HANDLE_BYTES);
    std::memcpy(handle, &h, sizeof h);
    return EUCL_OK;
}

int eucl_ipc_open(const uint8_t handle[EUCL_IPC_HANDLE_BYTES], int device, void** d_ptr) {
    if (!handle || !d_ptr) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_ipc_open: null argument");
    EUCL_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof h);
    EUCL_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return EUCL_OK;
}

int eucl_ipc_close(void* d_ptr) {
    if (!d_ptr) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_ipc_close: null argument");
    EUCL_CUDA(cudaIpcCloseMemHandle(d_ptr));
    return EUCL_OK;
}

int eucl_fp64_peak(int device, double* dadd_tops, double* dmul_tops, double* dfma_tops) {
    if (!dadd_tops || !dmul_tops || !dfma_tops) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_fp64_peak: null argument");
    if (eucl_device_count() <= 0) return fail(EUCL_ERR_NO_DEVICE, "no CUDA device available");
    EUCL_CUDA(cudaSetDevice(device));
    if (fp64_peak(dadd_tops, dmul_tops, dfma_tops) != 0) return fail(EUCL_ERR_CUDA, "fp64 microbenchmark failed");
    return EUCL_OK;
}

} // extern "C"
