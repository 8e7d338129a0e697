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
#include <memory>
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

// Grow-only device memory, or pinned host memory (kPinned), freed with its owner.
template <bool kPinned>
struct Buffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    Buffer() = default;
    Buffer(const Buffer&) = delete;
    Buffer& operator=(const Buffer&) = delete;
    ~Buffer() { release(); }
    cudaError_t ensure(size_t want) {
        if (want <= bytes) return cudaSuccess;
        release();
        cudaError_t e = kPinned ? cudaMallocHost(&ptr, want) : cudaMalloc(&ptr, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() {
        if (ptr) {
            if (kPinned) cudaFreeHost(ptr);
            else cudaFree(ptr);
        }
        ptr = nullptr;
        bytes = 0;
    }
};
using DeviceBuffer = Buffer<false>;
using PinnedBuffer = Buffer<true>;

// One helper thread per further pipeline of a split frame: runs that pipeline's host side (enqueue, stream synchronise,
// retry loop) next to the caller's thread.  Kept alive between frames: waking it costs microseconds, creating it tens.
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
    ~Worker() {
        if (!th.joinable()) return;
        {
            std::lock_guard<std::mutex> lk(m);
            quit = true;
            cv.notify_all();
        }
        th.join();
    }
};

// One pipeline of a frame: the streams a launch sequence runs on, its workspace and its CUDA graph.  Pipeline 0 renders
// every call; a split frame (render_split) adds more, each rendering every k-th band next to it over the scene's blob.
struct Pipeline {
    cudaStream_t stream = nullptr;      // the stream kernels run on (own_stream unless the caller set one for pipeline 0)
    cudaStream_t own_stream = nullptr;
    cudaStream_t side_stream = nullptr; // light builds of a level's kernels run here, next to the heavy ones
    cudaEvent_t ev[2] = {nullptr, nullptr}; // start and end of this pipeline's part of a call (timed)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::vector<cudaEvent_t> prof_events;   // per-launch events, profile mode only
    // workspace (grow-only)
    DeviceBuffer nodes;        // the node arena
    DeviceBuffer small;        // counters
    DeviceBuffer order;        // per-bin node lists of the level being shaded
    DeviceBuffer rorder;       // per-reach-key node lists of the next level
    DeviceBuffer frame_entity; // a batch of frames: the frames' camera entities ...
    DeviceBuffer node_frame;   // ... and the frame tag of every node
    DeviceBuffer node_cost;    // (segments, levels) per node of the arena: AOV renders that want either plane
    PinnedBuffer h_small;      // pinned mirror of the counters
    int arena_capacity = 0;
    double arena_factor = 0.0; // nodes per pixel the arena is sized for (learned from earlier frames)
    int list_capacity = 0;     // entries per index list (bins, reach keys): the largest LEVEL a chunk may have
    double list_factor = 1.0;  // ... in nodes per pixel (level 0 has exactly one; deeper levels are smaller in every shipped scene)
    cudaGraphExec_t graph_exec = nullptr; // the last repeated chunk as a CUDA graph (render_impl)
    uint64_t graph_key = 0, seen_key = 0; // parameter hash of graph_exec / of the previous direct launch sequence
    uint32_t graph_launches = 0;

    ~Pipeline() {
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        for (cudaEvent_t e : {ev[0], ev[1], ev_fork, ev_join})
            if (e) cudaEventDestroy(e);
        for (cudaEvent_t e : prof_events) cudaEventDestroy(e);
        if (side_stream) cudaStreamDestroy(side_stream);
        if (own_stream) cudaStreamDestroy(own_stream);
    }
};

} // namespace

struct EuclScene {
    int device = 0;
    int dim = 3;
    int sm_count = 148;
    size_t smem_bytes = 0;  // staged scene + plane_chain scratch
    size_t smem_scene = 0;  // staged scene only
    unsigned long long shade_light_mask = 1ull, shade_heavy_mask = 0ull;
    DeviceBuffer blob;
    std::vector<cudaArray_t> arrays;
    std::vector<cudaTextureObject_t> tex_objects;
    // host-output staging (grow-only)
    DeviceBuffer frame;     // device frame buffer for eucl_render (host output)
    DeviceBuffer hit_ids;   // device hit-id map for eucl_render
    DeviceBuffer aov_stage; // device copies of the AOV planes for eucl_render_aovs (host output)
    DeviceBuffer ray_stage; // device copy of the rays of eucl_trace_rays (host input), refilled by every call
    DeviceBuffer tree_stage; // a tree call: its query and the nodes and counts every pipeline exports into (host output)
    DeviceBuffer path_io;   // eucl_trace_path staging
    // a batch of frames (eucl_render_frames*): the per-frame constants, read by every pipeline, and their pinned host staging
    DeviceBuffer frame_table;
    PinnedBuffer h_frame_table;
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
    std::vector<std::unique_ptr<Pipeline>> pipes; // [0] always exists; render_split adds the others
    std::vector<std::unique_ptr<Worker>> workers; // one host thread per pipeline after the first
    cudaEvent_t ev_split[3] = {nullptr, nullptr, nullptr}; // a split frame: start (timed), fork, end (timed)

    cudaStream_t stream() const { return pipes[0]->stream; } // where calls stage their inputs and read back their outputs
    ~EuclScene() {
        for (cudaEvent_t e : ev_split)
            if (e) cudaEventDestroy(e);
        for (auto t : tex_objects) cudaDestroyTextureObject(t);
        for (auto a : arrays) cudaFreeArray(a);
    }
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

// One more pipeline: its streams, events and pinned counters; its workspace grows with the frames it renders.
int add_pipeline(EuclScene* s) {
    auto p = std::make_unique<Pipeline>();
    EUCL_CUDA(cudaStreamCreateWithFlags(&p->own_stream, cudaStreamNonBlocking));
    p->stream = p->own_stream;
    EUCL_CUDA(cudaEventCreate(&p->ev[0]));
    EUCL_CUDA(cudaEventCreate(&p->ev[1]));
    EUCL_CUDA(cudaStreamCreateWithFlags(&p->side_stream, cudaStreamNonBlocking));
    EUCL_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
    EUCL_CUDA(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
    EUCL_CUDA(p->h_small.ensure(sizeof(int32_t) * kSmallInts));
    s->pipes.push_back(std::move(p));
    return EUCL_OK;
}

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
    s->workers.clear();
    for (const auto& p : s->pipes) cudaStreamSynchronize(p->stream);
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
    auto s = std::make_unique<EuclScene>(); // freed with everything it holds on any early return
    s->device = device;
    s->real_bytes = precision == EUCL_PRECISION_F32 ? 4 : 8;
    s->dim = flat->dim;
    s->n_entities = flat->n_entities;
    cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device);
    status = add_pipeline(s.get());
    if (status != EUCL_OK) return status;
    for (int k = 0; k < 3; ++k)
        EUCL_CUDA(cudaEventCreateWithFlags(&s->ev_split[k], k == 1 ? cudaEventDisableTiming : cudaEventDefault));

    // textures -> CUDA arrays + point-sampled texture objects
    for (int t = 0; t < flat->n_textures; ++t) {
        const EuclTexture& tx = flat->textures[t];
        cudaChannelFormatDesc desc = cudaCreateChannelDesc<uchar4>();
        cudaArray_t arr = nullptr;
        EUCL_CUDA(cudaMallocArray(&arr, &desc, tx.width, tx.height));
        s->arrays.push_back(arr);
        EUCL_CUDA(cudaMemcpy2DToArray(arr, 0, 0, flat->texels + tx.texel_offset, (size_t)tx.width * 4,
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
        EUCL_CUDA(cudaCreateTextureObject(&obj, &rd, &td, nullptr));
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
            return fail(EUCL_ERR_SCENE_LIMIT, "entity " + std::to_string(e) + ": CSG program too large for the device evaluator (" +
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
        return fail(EUCL_ERR_SCENE_LIMIT, "scene tables (" + std::to_string(s->smem_bytes) +
                                              " B) exceed the shared memory of one CTA (" + std::to_string(smem_optin) + " B)");
    EUCL_CUDA(s->blob.ensure(w.bytes.size()));
    EUCL_CUDA(cudaMemcpy(s->blob.ptr, w.bytes.data(), w.bytes.size(), cudaMemcpyHostToDevice));
    EUCL_CUDA(EUCL_PREC(configure_kernels)(s->smem_bytes, s->smem_scene));
    *out = s.release();
    return EUCL_OK;
}

} // extern "C"

namespace {

// Camera constants in the reference's order (d3/entity/camera.rs:61-67,174-182; d4: 167-173)
// T = the scalar the camera arithmetic runs in: double, or float for the reference's `low_precision` feature (the
// results are stored as doubles either way; the f32 kernels narrow them back without loss)
template <typename T>
void frame_params_t(const EuclFrame& f, uint32_t width, uint32_t height, FrameParams* fp) {
    const EuclCamera& cam = f.camera;
    const int D = cam.dim;
    std::memset(fp, 0, sizeof *fp);
    const T w = (T)width, h = (T)height;
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
    fp->time_millis = (T)(std::floor(f.time_seconds * 1000.0) / 1000.0);
    fp->width = (int)width;
    fp->height = (int)height;
    fp->max_depth = (int)cam.max_depth;
}
void frame_params(const EuclFrame& f, uint32_t width, uint32_t height, int real_bytes, FrameParams* fp) {
    if (real_bytes == 4) frame_params_t<float>(f, width, height, fp);
    else frame_params_t<double>(f, width, height, fp);
}

size_t arena_bytes(int dim, int real_bytes, size_t cap) {
    size_t per = (size_t)(ray_reals(dim, real_bytes) + kHitReals + 4) * real_bytes + 4 + sizeof(NodeMeta);
    return per * cap + 16 * 16;
}

// FNV-1a over `bytes` bytes, continuing from `h`
uint64_t fnv1a(const void* data, size_t bytes, uint64_t h = 1469598103934665603ull) {
    const unsigned char* b = (const unsigned char*)data;
    for (size_t k = 0; k < bytes; ++k) h = (h ^ b[k]) * 1099511628211ull;
    return h;
}

// What one call renders.  Camera frames: K frames (eucl_render*: K = 1) are ONE virtual frame of K * rows rows -- chunks,
// bands and pipelines split it like any other frame -- whose per-pixel constants the kernels look up in a device table by
// virtual row; a single frame has no table and renders exactly as it always did.  Rays (eucl_trace_rays*): the rays on
// the device in place of a camera, as a virtual frame of n / width rows of width.
struct FrameBatch {
    uint32_t n;                    // K (rays: 1)
    uint32_t rows;                 // rows per frame
    uint32_t max_depth;            // (every frame of a batch has this one)
    FrameParams fp;                // frame 0's constants; rays: only the grid, the depth and the time
    const FrameParams* d_table;    // K > 1: [K] frame constants on the device, uploaded before the first launch
    uint64_t table_key;            // K > 1: hash of the table contents, part of the graph key
    const double* ray_origins;     // rays: [n][dim] each; null for camera frames
    const double* ray_directions;
    TreeQuery tree;                // a tree call: the items whose trees the chunks export (n_items 0: none)
};

// The batch of `n` camera frames (arguments checked) and `virt`, the virtual frame they form.  K > 1: the frame constants
// are computed on the host like a single frame's and uploaded on pipeline 0's stream, before the first launch and outside
// any graph capture.
int camera_batch(EuclScene* s, const EuclFrame* frames, uint32_t n, const EuclRenderOpts* o, FrameBatch* fb, EuclRenderOpts* virt) {
    *fb = FrameBatch{};
    fb->n = n;
    fb->rows = o->height;
    fb->max_depth = frames[0].camera.max_depth;
    frame_params(frames[0], o->width, o->height, s->real_bytes, &fb->fp);
    *virt = *o;
    virt->height = n * o->height;
    if (n == 1) return EUCL_OK;
    const size_t bytes = sizeof(FrameParams) * n;
    EUCL_CUDA(s->h_frame_table.ensure(bytes));
    FrameParams* table = (FrameParams*)s->h_frame_table.ptr;
    for (uint32_t k = 0; k < n; ++k) frame_params(frames[k], o->width, o->height, s->real_bytes, &table[k]);
    EUCL_CUDA(s->frame_table.ensure(bytes));
    EUCL_CUDA(cudaMemcpyAsync(s->frame_table.ptr, table, bytes, cudaMemcpyHostToDevice, s->stream()));
    fb->d_table = (const FrameParams*)s->frame_table.ptr;
    fb->table_key = fnv1a(table, bytes);
    return EUCL_OK;
}

// The batch of a ray call (arguments checked, rays on the device) and `o`, its virtual frame.  There is no camera: `fp`
// carries the grid, the depth and the time (truncated as for a frame, then `as F`).
FrameBatch ray_batch(const EuclScene* s, const EuclRays* r, const double* d_origins, const double* d_directions, bool want_hit,
                     EuclRenderOpts* o) {
    *o = EuclRenderOpts{};
    o->width = r->width > 1 ? r->width : 1;
    o->height = r->n / o->width;
    o->time_seconds = r->time_seconds;
    o->pipeline = r->pipeline;
    o->want_hit_ids = want_hit ? 1 : 0;
    o->profile = r->profile;
    FrameBatch fb{};
    fb.n = 1;
    fb.rows = o->height;
    fb.max_depth = r->max_depth;
    const double millis = std::floor(r->time_seconds * 1000.0) / 1000.0;
    fb.fp.time_millis = s->real_bytes == 4 ? (double)(float)millis : millis;
    fb.fp.width = (int)o->width;
    fb.fp.height = (int)o->height;
    fb.fp.max_depth = (int)r->max_depth;
    fb.ray_origins = d_origins;
    fb.ray_directions = d_directions;
    return fb;
}

// The launch configuration of `pipe`.  Queue kernels run as ONE wave of resident CTAs (512 threads per SM at 128
// registers) walking their level with a grid stride: measured faster than 2-8 waves on glass scenes (3d_room 20.7 ->
// 20.0 ms), equal elsewhere.
Launch make_launch(const EuclScene* s, const Pipeline& pipe, const EuclRenderOpts& o) {
    const int sms = s->sm_count;
    Launch l{};
    l.stream = pipe.stream;
    l.blob = (const uint8_t*)s->blob.ptr;
    l.smem_bytes = s->smem_bytes;
    l.smem_scene = s->smem_scene;
    l.grid_max = sms * std::max(1, env_int("EUCL_BLOCKS_PER_SM", kResidentThreads / kBlock));
    l.grid_light = sms * std::max(1, env_int("EUCL_LIGHT_BLOCKS_PER_SM", kLightResidentBlocks));
    l.grid_shade = sms * std::max(1, env_int("EUCL_SHADE_BLOCKS_PER_SM", kShadeResidentBlocks));
    l.grid_mem = sms * std::max(1, env_int("EUCL_MEM_BLOCKS_PER_SM", 8));
    l.shade_light_mask = s->shade_light_mask;
    l.shade_heavy_mask = s->shade_heavy_mask;
    l.grid_light_k2 = sms * std::max(1, env_int("EUCL_LIGHT_K2_BLOCKS_PER_SM", kLightK2ResidentBlocks));
    l.light_capable = s->light_capable;
    l.n_cull = s->n_cull;
    // per-launch profiling and the debugging modes keep everything on one stream
    l.side = (o.profile || env_int("EUCL_DEBUG_SYNC", 0) || !env_int("EUCL_CONCURRENT", 1)) ? nullptr : pipe.side_stream;
    l.ev_fork = pipe.ev_fork;
    l.ev_join = pipe.ev_join;
    l.grid_background = sms * std::max(1, env_int("EUCL_BACKGROUND_BLOCKS_PER_SM", EUCL_BACKGROUND_MIN_BLOCKS));
    return l;
}

Workspace carve(const EuclScene* s, const Pipeline& pipe, const FrameBatch& fb) {
    const int cap = pipe.arena_capacity;
    Workspace ws{};
    ws.capacity = cap;
    ws.list_cap = pipe.list_capacity;
    ws.n_frames = (int32_t)fb.n;
    ws.frame_rows = (int32_t)fb.rows;
    if (fb.n > 1) {
        ws.frames = fb.d_table;
        ws.frame_entity = (int32_t*)pipe.frame_entity.ptr;
        ws.node_frame = (int32_t*)pipe.node_frame.ptr;
    }
    if (fb.n > 1 || fb.ray_origins) ws.untraced = (int32_t*)pipe.small.ptr + SmallLayout::untraced;
    uint8_t* p = (uint8_t*)pipe.nodes.ptr;
    auto take = [&](size_t bytes) {
        uint8_t* r = p;
        p += align16(bytes);
        return r;
    };
    const size_t rb = (size_t)s->real_bytes;
    ws.ray = take((size_t)ray_reals(s->dim, s->real_bytes) * rb * cap);
    ws.hit = take((size_t)kHitReals * rb * cap);
    ws.res = take((size_t)4 * rb * cap);
    ws.meta = (NodeMeta*)take(sizeof(NodeMeta) * (size_t)cap);
    ws.ray_cur = (int32_t*)take((size_t)4 * cap);
    int32_t* small = (int32_t*)pipe.small.ptr;
    ws.count = small + SmallLayout::count;
    ws.level_off = small + SmallLayout::level_off;
    ws.overflow = small + SmallLayout::overflow;
    ws.cam_entity = small + SmallLayout::cam_entity;
    ws.undefined_count = (unsigned long long*)(small + SmallLayout::undefined64);
    ws.mega_level_counts = (unsigned long long*)(small + SmallLayout::mega64);
    ws.bin_count = small + SmallLayout::bins;
    ws.order = (int32_t*)pipe.order.ptr;
    const bool bin = pipe.order.ptr != nullptr;
    ws.n_bins = bin ? kBinsPerEntity * s->n_entities + 1 : 1;
    ws.rbin_count = small + SmallLayout::rbins;
    ws.rorder = (int32_t*)pipe.rorder.ptr;
    ws.ray_bins = pipe.rorder.ptr != nullptr && s->ray_bins_now ? 1 : 0;
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

// The index lists and per-node buffers a call's workspace holds next to the node arena.
struct WorkspaceNeeds {
    bool rorder; // reach-key lists of the next level
    bool order;  // shade-coherence bins: one node list per hit entity (+ miss), each able to hold a whole level
    bool cost;   // the COST builds' (segments, levels) pair per node
    bool frames; // a batch: the frame tag of every node
};

// Leaves a consistent, empty workspace: the next chunk allocates it again.
void release_workspace(Pipeline& pipe) {
    pipe.nodes.release();
    pipe.order.release();
    pipe.rorder.release();
    pipe.node_cost.release();
    pipe.arena_capacity = 0;
    pipe.list_capacity = 0;
}

// Grows `pipe`'s workspace for chunks of *rows rows of `width` pixels at its learned factors.  The chunk shrinks by half
// while its workspace does not fit: more than 2^31 nodes, over the memory budget, or an allocation failure.
int reserve_workspace(const EuclScene* s, Pipeline& pipe, const WorkspaceNeeds& need, int pipeline, int width, int* rows) {
    const size_t n_bins = (size_t)(kBinsPerEntity * s->n_entities + 1);
    const size_t n_lists = (need.rorder ? (size_t)kRayBins : 0) + (need.order ? n_bins : 0);
    for (;;) {
        long long want = (long long)std::ceil((double)*rows * (double)width * pipe.arena_factor) + 1024;
        long long want_list = (long long)std::ceil((double)*rows * (double)width * pipe.list_factor) + 1024;
        if (pipeline == EUCL_PIPELINE_MEGAKERNEL) want = want_list = 16;
        bool too_big = want > 0x7fff0000ll || want_list > 0x7fff0000ll;
        if (!too_big && ((int)want > pipe.arena_capacity || (int)want_list > pipe.list_capacity)) {
            EUCL_CUDA(cudaStreamSynchronize(pipe.stream));
            want = std::max<long long>(want, pipe.arena_capacity);
            want_list = std::max<long long>(want_list, pipe.list_capacity);
            size_t free_b = 0, total_b = 0;
            EUCL_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const size_t held = pipe.nodes.bytes + pipe.order.bytes + pipe.rorder.bytes + pipe.node_cost.bytes;
            size_t budget = (size_t)((double)(free_b + held) * 0.85);
            const int cap_mb = env_int("EUCL_ARENA_MAX_MB", 0);
            if (cap_mb > 0) budget = std::min(budget, (size_t)cap_mb << 20);
            const size_t bytes = arena_bytes(s->dim, s->real_bytes, (size_t)want) + sizeof(int32_t) * n_lists * (size_t)want_list +
                                 (need.cost ? sizeof(uint2) * (size_t)want : 0);
            too_big = bytes > budget;
            if (!too_big) {
                cudaError_t e = pipe.nodes.ensure(arena_bytes(s->dim, s->real_bytes, (size_t)want));
                if (e == cudaSuccess && need.rorder) e = pipe.rorder.ensure(sizeof(int32_t) * (size_t)kRayBins * (size_t)want_list);
                if (e == cudaSuccess && need.order) e = pipe.order.ensure(sizeof(int32_t) * n_bins * (size_t)want_list);
                if (e == cudaSuccess) {
                    pipe.arena_capacity = (int)want;
                    pipe.list_capacity = (int)want_list;
                } else { // try a smaller chunk
                    cudaGetLastError();
                    release_workspace(pipe);
                    if (e != cudaErrorMemoryAllocation) return fail(EUCL_ERR_CUDA, std::string("workspace allocation: ") + cudaGetErrorString(e));
                    too_big = true;
                }
            }
        }
        if (!too_big) break;
        if (*rows <= 1) return fail(EUCL_ERR_OUT_OF_MEMORY, "the node arena of a single row of pixels does not fit in device memory");
        *rows = (*rows + 1) / 2;
    }
    if (need.frames) EUCL_CUDA(pipe.node_frame.ensure(sizeof(int32_t) * (size_t)pipe.arena_capacity));
    if (need.cost) EUCL_CUDA(pipe.node_cost.ensure(sizeof(uint2) * (size_t)pipe.arena_capacity));
    return EUCL_OK;
}

// A frame that had to grow its arena over-shot (capacity grows by half each retry).  Now that the frame's real node count
// is known, the pipeline keeps that plus a few per cent and gives the rest back, and with it the graph that points into
// the old workspace: the next frame of this size allocates once more, exactly, and nothing afterwards.
void trim_workspace(Pipeline& pipe, const EuclStats& st) {
    if (st.retries == 0 || st.pixels == 0 || st.nodes == 0) return;
    uint64_t max_level = 0;
    for (uint32_t lv = 0; lv < st.levels; ++lv) max_level = std::max<uint64_t>(max_level, st.level_counts[lv]);
    const double tight = (double)st.nodes / (double)st.pixels * 1.03 + 0.02;
    const double tight_list = std::max(1.0, (double)max_level / (double)st.pixels * 1.03);
    if ((double)pipe.arena_capacity > ((double)st.pixels * tight + 1024) * 1.08) {
        pipe.arena_factor = tight;
        pipe.list_factor = tight_list;
        release_workspace(pipe);
        if (pipe.graph_exec) cudaGraphExecDestroy(pipe.graph_exec);
        pipe.graph_exec = nullptr;
        pipe.graph_key = pipe.seen_key = 0;
    }
}

// Everything the launch sequence of one chunk reads.
struct ChunkLaunch {
    const FrameBatch& fb;
    int pipeline; // EuclPipeline
    Launch l;
    ChunkParams cp;
    Workspace ws;
    AovPlanes aov; // the planes a chunk writes (null = not wanted) and the cost buffer
    uint8_t* d_rgb;
    int32_t* d_hit;
};

// The diagnostic modes of one chunk.  Profile mode records an event after every launch (family -1 start, 0 raygen,
// 1 intersect, 2 shade, 3 resolve).  EUCL_DEBUG_SYNC=1 synchronises after every launch and names the one that faulted.
// EUCL_POISON=1 fills the work buffers with 0x7F bytes (huge positive indices) first, so that a read of anything this
// frame did not write turns into a deterministic fault instead of depending on stale data.
struct ChunkDebug {
    bool profile, sync, poison;
    std::vector<int> prof_family;
    std::string fault;
};

// Everything one chunk puts on the stream: counters reset, kernels, counters back to the pinned mirror.  Returns the
// number of kernels.
uint32_t enqueue_chunk(const EuclScene* s, Pipeline& pipe, const ChunkLaunch& c, ChunkDebug& dbg) {
    const int dim = s->dim;
    const FrameBatch& fb = c.fb;
    const Launch& l = c.l;
    auto mark = [&](int family) {
        if (!dbg.profile) return;
        if (pipe.prof_events.size() <= dbg.prof_family.size()) {
            cudaEvent_t e = nullptr;
            cudaEventCreate(&e);
            pipe.prof_events.push_back(e);
        }
        cudaEventRecord(pipe.prof_events[dbg.prof_family.size()], pipe.stream);
        dbg.prof_family.push_back(family);
    };
    auto check = [&](const char* what, int level) {
        if (!dbg.sync || !dbg.fault.empty()) return;
        cudaError_t e = cudaStreamSynchronize(pipe.stream);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) dbg.fault = std::string(what) + " level " + std::to_string(level) + ": " + cudaGetErrorString(e);
    };
    uint32_t launches = 0;
    cudaMemsetAsync(pipe.small.ptr, 0, sizeof(int32_t) * kSmallInts, pipe.stream);
    if (dbg.poison) {
        cudaMemsetAsync(pipe.nodes.ptr, 0x7F, pipe.nodes.bytes, pipe.stream);
        if (pipe.order.ptr) cudaMemsetAsync(pipe.order.ptr, 0x7F, pipe.order.bytes, pipe.stream);
        if (pipe.rorder.ptr) cudaMemsetAsync(pipe.rorder.ptr, 0x7F, pipe.rorder.bytes, pipe.stream);
    }
    mark(-1);
    if (c.pipeline == EUCL_PIPELINE_MEGAKERNEL) {
        if (!fb.ray_origins) {
            EUCL_PREC(launch_camera_entity)(dim, l, fb.fp, c.ws);
            check("k_camera_entity", 0);
            launches += 1;
        }
        EUCL_PREC(launch_megakernel)(dim, l, fb.fp, c.cp, c.ws, c.d_rgb, c.d_hit, c.aov, fb.ray_origins, fb.ray_directions, fb.tree);
        mark(1);
        launches += 1;
    } else {
        if (c.ws.frames) {
            EUCL_PREC(launch_camera_entity)(dim, l, fb.fp, c.ws);
            check("k_camera_entity", 0);
            launches += 1;
        }
        if (fb.ray_origins) EUCL_PREC(launch_raygen_rays)(dim, l, fb.fp, c.cp, c.ws, c.d_hit, fb.ray_origins, fb.ray_directions);
        else EUCL_PREC(launch_raygen)(dim, l, fb.fp, c.cp, c.ws, c.d_hit);
        check("k_raygen", 0);
        mark(0);
        for (int level = 0; level < (int)fb.max_depth; ++level) {
            launches += EUCL_PREC(launch_intersect)(dim, l, c.ws, level);
            check("k_intersect", level);
            mark(1);
            launches += EUCL_PREC(launch_shade)(dim, l, fb.fp, c.cp, c.ws, level, c.d_hit);
            check("k_shade", level);
            mark(2);
        }
        // the nodes of the last level are background lookups (depth 0: mod.rs:157,183).  Measured and not kept:
        // finishing them inside k_shade of the level above, from the child direction in registers (one launch
        // and one ray record per node less, but the lookups then run at the heavy kernel's occupancy:
        // 3d_room shade 7.14 + 0.47 -> 7.34 + 0.67 ms)
        launches += EUCL_PREC(launch_shade)(dim, l, fb.fp, c.cp, c.ws, (int)fb.max_depth, c.d_hit);
        check("k_shade", (int)fb.max_depth);
        mark(2);
        launches += EUCL_PREC(launch_resolve_and_final)(dim, l, fb.fp, c.cp, c.ws, c.d_rgb, c.aov);
        check("k_resolve / k_final", 0);
        if (fb.tree.n_items) {
            launches += EUCL_PREC(launch_tree_export)(dim, l, fb.fp, c.cp, c.ws, fb.tree);
            check("k_tree_export", 0);
        }
        mark(3);
        launches += 1; // raygen
    }
    cudaMemcpyAsync(pipe.h_small.ptr, pipe.small.ptr, sizeof(int32_t) * kSmallInts, cudaMemcpyDeviceToHost, pipe.stream);
    return launches;
}

// The CUDA-graph key of a chunk: a hash of everything its launches read
uint64_t graph_key(const ChunkLaunch& c) {
    const FrameBatch& fb = c.fb;
    uint64_t key = fnv1a(&fb.fp, sizeof fb.fp);
    auto mix = [&](const void* data, size_t bytes) { key = fnv1a(data, bytes, key); };
    mix(&c.cp, sizeof c.cp);
    mix(&c.ws, sizeof c.ws);
    {   // the members of Launch one by one (the struct has padding bytes)
        const Launch& l = c.l;
        const void* ptrs[] = {l.stream, l.blob, l.side};
        const unsigned long long nums[] = {l.smem_bytes, l.smem_scene, (unsigned long long)l.grid_max, (unsigned long long)l.grid_light,
                                           (unsigned long long)l.grid_shade, (unsigned long long)l.grid_mem, l.shade_light_mask,
                                           l.shade_heavy_mask, (unsigned long long)l.grid_light_k2,
                                           (unsigned long long)l.light_capable, (unsigned long long)l.n_cull,
                                           (unsigned long long)l.grid_background};
        mix(ptrs, sizeof ptrs);
        mix(nums, sizeof nums);
    }
    mix(&c.d_rgb, sizeof c.d_rgb);
    mix(&c.d_hit, sizeof c.d_hit);
    // the AOV planes and the cost buffer: a graph captured with or without them never stands in for the other
    mix(&c.aov, sizeof c.aov);
    mix(&c.pipeline, sizeof c.pipeline);
    mix(&fb.max_depth, sizeof fb.max_depth);
    // a batch: the graph reads the table the caller's poses were uploaded to, and it is keyed by its contents too, so
    // that a changed pose or time is never taken for a repeated batch
    if (fb.n > 1) mix(&fb.table_key, sizeof fb.table_key);
    // a ray call: tagged, so that a ray call and a render whose other parameters coincide never stand in for each
    // other, and keyed by the arrays it reads (their contents are read at replay time)
    if (fb.ray_origins) {
        const uint64_t ray_id[] = {0x52415953ull /* "RAYS" */, (uint64_t)(uintptr_t)fb.ray_origins, (uint64_t)(uintptr_t)fb.ray_directions,
                                   (uint64_t)fb.fp.height * (uint64_t)fb.fp.width, (uint64_t)fb.fp.width};
        mix(ray_id, sizeof ray_id);
    }
    return key;
}

// A chunk whose launch parameters repeat (a fixed pose rendered again: benchmarks, a paused camera, every rank of a
// band-split frame) is replayed as ONE CUDA graph launch: the ~50 kernels of a frame then cost one driver call on the
// host and run back to back on the device.  The first sighting of a parameter set launches directly, the second
// captures, later ones replay.  Without `use_graph` every chunk launches directly.
int launch_chunk(const EuclScene* s, Pipeline& pipe, const ChunkLaunch& c, ChunkDebug& dbg, bool use_graph, EuclStats* st) {
    if (c.fb.tree.n_items) { // a tree call launches directly and leaves the plain calls' graph and keys as they were
        st->launches += enqueue_chunk(s, pipe, c, dbg);
        return EUCL_OK;
    }
    const uint64_t key = graph_key(c);
    if (use_graph && pipe.graph_exec && pipe.graph_key == key) {
        EUCL_CUDA(cudaGraphLaunch(pipe.graph_exec, pipe.stream));
        st->launches += pipe.graph_launches;
        st->graph_replays += 1;
    } else if (use_graph && pipe.seen_key == key) {
        if (pipe.graph_exec) cudaGraphExecDestroy(pipe.graph_exec);
        pipe.graph_exec = nullptr;
        cudaGraph_t graph = nullptr;
        // one capture at a time in the process (the pipelines of a split frame capture in the same frame)
        static std::mutex capture_mutex;
        std::unique_lock<std::mutex> capture_lock(capture_mutex);
        EUCL_CUDA(cudaStreamBeginCapture(pipe.stream, cudaStreamCaptureModeThreadLocal));
        const uint32_t launches = enqueue_chunk(s, pipe, c, dbg);
        cudaError_t ce = cudaStreamEndCapture(pipe.stream, &graph);
        if (ce == cudaSuccess) ce = cudaGraphInstantiate(&pipe.graph_exec, graph, 0);
        capture_lock.unlock();
        if (graph) cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { // not capturable here (e.g. a caller's stream in a state that forbids it): launch directly
            cudaGetLastError();
            pipe.graph_exec = nullptr;
            pipe.seen_key = 0;
            st->launches += enqueue_chunk(s, pipe, c, dbg);
        } else {
            pipe.graph_key = key;
            pipe.graph_launches = launches;
            EUCL_CUDA(cudaGraphLaunch(pipe.graph_exec, pipe.stream));
            st->launches += launches;
            st->graph_replays += 1;
        }
    } else {
        pipe.seen_key = key;
        st->launches += enqueue_chunk(s, pipe, c, dbg);
    }
    return EUCL_OK;
}

// Waits for a launched chunk and reads its counters back.  A level that overflowed the arena or the index lists grows
// the learned factor and sets `*retry`; a chunk that fit adds its pixels and level counts to `st`.
int read_back_chunk(Pipeline& pipe, const ChunkLaunch& c, const ChunkDebug& dbg, EuclStats* st, bool* retry) {
    if (!dbg.fault.empty()) return fail(EUCL_ERR_CUDA, "EUCL_DEBUG_SYNC: " + dbg.fault);
    EUCL_CUDA(cudaStreamSynchronize(pipe.stream));
    EUCL_CUDA(cudaGetLastError());
    const int32_t* h = (const int32_t*)pipe.h_small.ptr;
    const uint32_t depth = c.fb.max_depth;
    for (size_t k = 1; k < dbg.prof_family.size(); ++k) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, pipe.prof_events[k - 1], pipe.prof_events[k]);
        float* slot = dbg.prof_family[k] == 0 ? &st->ms_raygen : dbg.prof_family[k] == 1 ? &st->ms_intersect
                      : dbg.prof_family[k] == 2 ? &st->ms_shade : &st->ms_resolve;
        *slot += ms;
    }
    if (env_int("EUCL_DUMP_LEVELS", 0) && !h[SmallLayout::overflow]) { // diagnostics: per-level counts, bins, launch times
        for (uint32_t lv = 0; lv <= depth; ++lv) {
            fprintf(stderr, "level %2u count %9d | bins", lv, h[SmallLayout::count + lv]);
            for (int b = 0; b < c.ws.n_bins && c.ws.n_bins > 1; ++b) fprintf(stderr, " %d", h[SmallLayout::bins + lv * kMaxBins + b]);
            fprintf(stderr, " | rbins");
            for (int b = 0; b < kRayBins; ++b) fprintf(stderr, " %d", h[SmallLayout::rbins + lv * kRayBins + b]);
            fprintf(stderr, "\n");
        }
        for (size_t k = 1; k < dbg.prof_family.size(); ++k) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, pipe.prof_events[k - 1], pipe.prof_events[k]);
            fprintf(stderr, "launch %2zu family %d %.3f ms\n", k, dbg.prof_family[k], ms);
        }
    }
    if (h[SmallLayout::overflow] == 2) return fail(EUCL_ERR_CUDA, "internal error: a queue index list and its level count disagree");
    *retry = h[SmallLayout::overflow] != 0;
    if (*retry) {
        // levels after the overflowing one were skipped, so the counts are a lower bound only
        long long need = 0;
        for (uint32_t lv = 0; lv <= depth; ++lv) need += h[SmallLayout::count + lv];
        if (h[SmallLayout::overflow] == 3) { // a level outgrew the index lists (they hold one level each)
            pipe.list_factor = std::max(pipe.list_factor * 1.5, 1.0);
        } else {
            double factor = (double)need / (double)c.cp.n_pixels * 1.05 + 0.05;
            pipe.arena_factor = std::max(pipe.arena_factor * 1.5, factor);
        }
        st->retries += 1;
        if (st->retries > 32) return fail(EUCL_ERR_OUT_OF_MEMORY, "node arena keeps overflowing");
        return EUCL_OK;
    }
    st->pixels += (uint64_t)c.cp.n_pixels;
    // camera in no entity: checkerboard pixels, Universe::trace is never called (mod.rs:385-396).  In a batch with
    // some frames traced, level 0 holds the checkerboard pixels of the others: they are not counted either.
    const bool traced = h[SmallLayout::cam_entity] >= 0;
    for (uint32_t lv = 0; traced && lv <= depth; ++lv) {
        uint64_t n = c.pipeline == EUCL_PIPELINE_MEGAKERNEL ? ((const unsigned long long*)(h + SmallLayout::mega64))[lv]
                                                            : (uint64_t)h[SmallLayout::count + lv];
        if (lv == 0) n -= (uint64_t)h[SmallLayout::untraced];
        st->level_counts[lv] += n;
        st->nodes += n;
        if (lv < depth) st->segments += n;
    }
    return EUCL_OK;
}

// Renders this rank's rows of `o` on `pipe`: all of them, or -- sub_stride > 1 -- the bands that `o` names, which are
// every sub_stride-th band of the caller's rank starting at sub_offset (render_split).  `o` describes the (virtual)
// frame: o->height = fb.n * fb.rows.
int render_impl(EuclScene* s, Pipeline& pipe, const FrameBatch& fb, const EuclRenderOpts* o, uint8_t* d_rgb, int32_t* d_hit,
                const AovPlanes& aov_out, EuclStats* stats, int sub_stride = 1, int sub_offset = 0) {
    const int width = (int)o->width;
    const uint32_t my_rows = eucl_band_rows_for_rank(o);
    const bool wavefront = o->pipeline == EUCL_PIPELINE_WAVEFRONT;
    EuclStats st{};
    st.levels = fb.max_depth + 1;
    if (sub_stride <= 1) choose_grouping(s); // (render_split chooses for a split frame)
    if (fb.n > 1) EUCL_CUDA(pipe.frame_entity.ensure(sizeof(int32_t) * fb.n));
    EUCL_CUDA(cudaEventRecord(pipe.ev[0], pipe.stream));
    if (my_rows > 0) {
        if ((long long)width > (1ll << 30)) return fail(EUCL_ERR_INVALID_ARGUMENT, "frame rows too wide");
        if (!wavefront && fb.max_depth > 24) return fail(EUCL_ERR_SCENE_LIMIT, "megakernel pipeline supports max_depth <= 24");
        EUCL_CUDA(pipe.small.ensure(sizeof(int32_t) * kSmallInts));
        if (pipe.arena_factor <= 0.0) pipe.arena_factor = std::max(1.0, (double)env_int("EUCL_ARENA_FACTOR_X10", 45) / 10.0);
        const WorkspaceNeeds need{wavefront && s->n_cull > 0 && env_int("EUCL_BIN_RAYS", 1),
                                  wavefront && kBinsPerEntity * s->n_entities + 1 <= kMaxBins && env_int("EUCL_BIN_SHADE", 1),
                                  wavefront && (aov_out.segments || aov_out.levels), fb.n > 1};
        // chunking: whole local rows, about EUCL_CHUNK_PIXELS primaries per chunk.  Large chunks are faster (longer
        // levels, fewer host round trips: 4d_room 7680x4320 renders 10 % faster as one chunk than as eight), so the
        // default covers an 8K frame; the chunk shrinks by itself when its workspace does not fit (reserve_workspace).
        const long long chunk_pixels_target = std::max(1, env_int("EUCL_CHUNK_PIXELS", 1 << 25));
        int rows_per_chunk = (int)std::max<long long>(1, chunk_pixels_target / width);
        rows_per_chunk = std::min<int>(rows_per_chunk, (int)my_rows);
        const bool debug_sync = env_int("EUCL_DEBUG_SYNC", 0) != 0;
        const bool poison = env_int("EUCL_POISON", 0) != 0;
        // (no graph while the scene is still choosing its ray grouping: capture time would distort the comparison; ray
        // calls take no part in that choice)
        const bool use_graph = env_int("EUCL_GRAPH", 1) && !o->profile && !debug_sync && !poison &&
                               (s->ray_bins_mode >= 0 || !wavefront || fb.ray_origins);
        ChunkLaunch c{fb, o->pipeline, make_launch(s, pipe, *o), ChunkParams{}, Workspace{}, aov_out, d_rgb, d_hit};
        c.cp.band_rows = o->band_rows ? (int)o->band_rows : (int)o->height;
        c.cp.band_rank = (int)o->band_rank;
        c.cp.band_world = o->band_world ? (int)o->band_world : 1;
        c.cp.compact_rows = o->compact_rows;
        c.cp.sub_stride = sub_stride;
        c.cp.sub_offset = sub_offset;
        for (int row0 = 0; row0 < (int)my_rows; row0 += c.cp.n_rows) {
            c.cp.local_row0 = row0;
            for (bool retry = true; retry;) { // a larger arena when a level overflowed
                int rc = reserve_workspace(s, pipe, need, o->pipeline, width, &rows_per_chunk);
                if (rc != EUCL_OK) return rc;
                c.cp.n_rows = std::min<int>(rows_per_chunk, (int)my_rows - row0);
                c.cp.n_pixels = c.cp.n_rows * width;
                c.ws = carve(s, pipe, fb);
                c.aov.cost = need.cost ? (uint2*)pipe.node_cost.ptr : nullptr;
                ChunkDebug dbg{o->profile != 0, debug_sync, poison, {}, {}};
                rc = launch_chunk(s, pipe, c, dbg, use_graph, &st);
                if (rc == EUCL_OK) rc = read_back_chunk(pipe, c, dbg, &st, &retry);
                if (rc != EUCL_OK) return rc;
            }
        }
    }
    EUCL_CUDA(cudaEventRecord(pipe.ev[1], pipe.stream));
    EUCL_CUDA(cudaEventSynchronize(pipe.ev[1]));
    EUCL_CUDA(cudaEventElapsedTime(&st.ms_total, pipe.ev[0], pipe.ev[1]));
    if (wavefront && st.pixels == (uint64_t)my_rows * width) trim_workspace(pipe, st);
    // (a split frame is judged as a whole: render_split).  A ray batch is not a frame of its size, and a tree call pays
    // for its export: neither tunes.
    if (sub_stride <= 1 && !fb.ray_origins && !fb.tree.n_items) {
        tune_grouping(s, st, o->pipeline);
        s->warm_frames++;
    }
    st.ray_grouping = s->ray_bins_now && pipe.rorder.ptr != nullptr && wavefront ? 1u : 0u;
    if (stats) *stats = st;
    return EUCL_OK;
}

// `part`, rendered next to `st` as another part of the same frame, added to it: counts and times add up, and a chunk
// counts as replayed where every part replayed.
void add_stats(EuclStats* st, const EuclStats& part) {
    st->pixels += part.pixels;
    st->segments += part.segments;
    st->nodes += part.nodes;
    for (uint32_t lv = 0; lv < EUCL_MAX_LEVELS; ++lv) st->level_counts[lv] += part.level_counts[lv];
    st->launches += part.launches;
    st->retries += part.retries;
    st->graph_replays = std::min(st->graph_replays, part.graph_replays);
    st->ms_raygen += part.ms_raygen;
    st->ms_intersect += part.ms_intersect;
    st->ms_shade += part.ms_shade;
    st->ms_resolve += part.ms_resolve;
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
    if (k <= 1) return render_impl(s, *s->pipes[0], fb, o, d_rgb, d_hit, aov, stats);
    while ((int)s->pipes.size() < k) {
        const int rc = add_pipeline(s);
        if (rc != EUCL_OK) {
            cudaGetLastError(); // (a failed allocation must not fail the scene's next call)
            return rc;
        }
        s->workers.push_back(std::make_unique<Worker>());
        s->workers.back()->start();
    }
    choose_grouping(s);
    EuclRenderOpts opts[kMaxSplit];
    EuclStats part[kMaxSplit] = {};
    int rc[kMaxSplit] = {}; // EUCL_OK
    std::string err[kMaxSplit];
    for (int p = 0; p < k; ++p) {
        opts[p] = *o;
        opts[p].band_rows = band;
        opts[p].band_world = (uint32_t)k * world;
        opts[p].band_rank = rank + (uint32_t)p * world;
    }
    const cudaStream_t lead = s->stream();
    EUCL_CUDA(cudaEventRecord(s->ev_split[0], lead));
    EUCL_CUDA(cudaEventRecord(s->ev_split[1], lead)); // the other pipelines start after whatever the caller's stream holds
    for (int p = 1; p < k; ++p) EUCL_CUDA(cudaStreamWaitEvent(s->pipes[p]->stream, s->ev_split[1], 0));
    // per-launch profiling and the debugging modes run the pipelines one after the other on the caller's thread
    const bool serial = o->profile || env_int("EUCL_DEBUG_SYNC", 0) || env_int("EUCL_POISON", 0);
    auto run = [&](int p) {
        cudaSetDevice(s->device);
        rc[p] = render_impl(s, *s->pipes[p], fb, &opts[p], d_rgb, d_hit, aov, &part[p], k, p);
        if (rc[p] != EUCL_OK) err[p] = eucl_last_error();
    };
    // (no early return between here and the last wait(): the helper threads work on this frame's locals)
    for (int p = 1; p < k && !serial; ++p) s->workers[p - 1]->run([&run, p] { run(p); });
    run(0);
    for (int p = 1; p < k; ++p) {
        if (serial) run(p);
        else s->workers[p - 1]->wait();
    }
    for (int p = 0; p < k; ++p)
        if (rc[p] != EUCL_OK) return fail(rc[p], err[p]);
    for (int p = 1; p < k; ++p) // the caller's stream continues after every pipeline (ev[1]: the end of its part)
        EUCL_CUDA(cudaStreamWaitEvent(lead, s->pipes[p]->ev[1], 0));
    EUCL_CUDA(cudaEventRecord(s->ev_split[2], lead));
    EUCL_CUDA(cudaEventSynchronize(s->ev_split[2]));
    EuclStats st = part[0];
    EUCL_CUDA(cudaEventElapsedTime(&st.ms_total, s->ev_split[0], s->ev_split[2]));
    for (int p = 1; p < k; ++p) add_stats(&st, part[p]);
    if (!fb.ray_origins && !fb.tree.n_items) {
        tune_grouping(s, st, o->pipeline);
        s->warm_frames++;
    }
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

// One frame: what eucl_render accepts; K > 1 frames: what eucl_render_frames accepts.
int check_aov_call(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, const EuclAovs* aovs,
                   const char* fn) {
    int st = n_frames == 1 ? check_args(s, frames ? &frames[0].camera : nullptr, o) : check_frames(s, frames, n_frames, o);
    if (st == EUCL_OK) st = check_aovs(aovs, fn);
    return st;
}

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

// The host rays of a ray call, copied to the scene's device buffer before the first launch, on pipeline 0's stream and
// outside any graph capture: a replayed graph reads them.
int stage_rays(EuclScene* s, const EuclRays* r, double** d_origins, double** d_directions) {
    const size_t bytes = sizeof(double) * (size_t)s->dim * r->n;
    EUCL_CUDA(s->ray_stage.ensure(2 * bytes));
    *d_origins = (double*)s->ray_stage.ptr;
    *d_directions = (double*)((uint8_t*)s->ray_stage.ptr + bytes);
    EUCL_CUDA(cudaMemcpyAsync(*d_origins, r->origins, bytes, cudaMemcpyHostToDevice, s->stream()));
    EUCL_CUDA(cudaMemcpyAsync(*d_directions, r->directions, bytes, cudaMemcpyHostToDevice, s->stream()));
    return EUCL_OK;
}

static_assert(sizeof(EuclTreeNode) == 176, "EuclTreeNode is part of the C ABI");
static_assert(sizeof(EuclTreeQuery) == 32, "EuclTreeQuery is part of the C ABI");

// eucl_render_trees / eucl_trace_ray_trees: the query against a virtual frame of `cells` cells.  Checked before any device
// is touched.
int check_tree_query(const EuclTreeQuery* q, uint64_t cells, const char* fn) {
    const std::string f(fn);
    if (!q || q->n_items == 0) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": no tree query (use the plain entry point)");
    if (q->n_items > EUCL_TREE_MAX_ITEMS) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": more than EUCL_TREE_MAX_ITEMS items");
    if (!q->items || !q->nodes || !q->counts) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": null items, nodes or counts");
    if (q->capacity == 0) return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": capacity must be at least 1");
    if ((uint64_t)q->n_items * q->capacity > EUCL_TREE_MAX_NODES)
        return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": n_items * capacity above EUCL_TREE_MAX_NODES");
    for (uint32_t i = 0; i < q->n_items; ++i)
        if (q->items[i] >= cells)
            return fail(EUCL_ERR_INVALID_ARGUMENT, f + ": item " + std::to_string(i) + " (" + std::to_string(q->items[i]) +
                                                       ") is outside the virtual frame of " + std::to_string(cells) + " cells");
    return EUCL_OK;
}

// The device side of a checked query, staged on pipeline 0's stream before the first launch: the distinct items, sorted,
// each with its first request slot, and the slots' nodes (zeroed) and counts that the pipelines export into -- every item
// by exactly one chunk of one pipeline.
int stage_tree_query(EuclScene* s, const EuclTreeQuery* q, std::vector<uint32_t>* order, TreeQuery* out) {
    order->resize(q->n_items);
    for (uint32_t i = 0; i < q->n_items; ++i) (*order)[i] = i;
    std::stable_sort(order->begin(), order->end(), [q](uint32_t a, uint32_t b) { return q->items[a] < q->items[b]; });
    std::vector<uint32_t> items, slots;
    for (uint32_t i : *order)
        if (items.empty() || items.back() != q->items[i]) {
            items.push_back(q->items[i]);
            slots.push_back(i);
        }
    const size_t node_bytes = align16(sizeof(EuclTreeNode) * q->n_items * (size_t)q->capacity);
    const size_t list_bytes = align16(sizeof(uint32_t) * q->n_items);
    EUCL_CUDA(s->tree_stage.ensure(node_bytes + 3 * list_bytes));
    uint8_t* p = (uint8_t*)s->tree_stage.ptr;
    *out = TreeQuery{(const uint32_t*)(p + node_bytes + list_bytes), (const uint32_t*)(p + node_bytes + 2 * list_bytes),
                     (int32_t)items.size(), (int32_t)q->capacity, (EuclTreeNode*)p, (uint32_t*)(p + node_bytes)};
    const cudaStream_t stream = s->stream();
    EUCL_CUDA(cudaMemsetAsync(p, 0, node_bytes + list_bytes, stream));
    EUCL_CUDA(cudaMemcpyAsync((void*)out->items, items.data(), sizeof(uint32_t) * items.size(), cudaMemcpyHostToDevice, stream));
    EUCL_CUDA(cudaMemcpyAsync((void*)out->slots, slots.data(), sizeof(uint32_t) * slots.size(), cudaMemcpyHostToDevice, stream));
    return EUCL_OK;
}

// After a tree call has rendered (its pipelines joined): the staged nodes and counts to the caller's arrays, then every
// duplicate slot from the first slot of its item (`order`: the slots sorted by item, stable).
int read_back_trees(EuclScene* s, const EuclTreeQuery* q, const std::vector<uint32_t>& order, const TreeQuery& tq) {
    const size_t per_slot = sizeof(EuclTreeNode) * (size_t)q->capacity;
    EUCL_CUDA(cudaMemcpyAsync(q->nodes, tq.nodes, per_slot * q->n_items, cudaMemcpyDeviceToHost, s->stream()));
    EUCL_CUDA(cudaMemcpyAsync(q->counts, tq.counts, sizeof(uint32_t) * q->n_items, cudaMemcpyDeviceToHost, s->stream()));
    EUCL_CUDA(cudaStreamSynchronize(s->stream()));
    for (size_t k = 1; k < order.size(); ++k) { // a duplicate follows its item's first slot (or an earlier duplicate)
        const uint32_t prev = order[k - 1], slot = order[k];
        if (q->items[slot] != q->items[prev]) continue;
        std::memcpy(q->nodes + (size_t)slot * q->capacity, q->nodes + (size_t)prev * q->capacity, per_slot);
        q->counts[slot] = q->counts[prev];
    }
    return EUCL_OK;
}

const EuclAovs* any_plane(const EuclAovs* a) {
    return a && (a->depth || a->position || a->normal || a->segments || a->levels) ? a : nullptr;
}

// Host-output render of a batch whose virtual frame is `o`: rendered into the scene's device buffers, then copied out.
// A rank of a band-split render (band_world > 1, a single frame) renders its rows compactly on the device and then copies
// each band to its place in the caller's frame: rows of other ranks are never read or written, so N ranks can fill ONE
// host frame (shared pinned memory) over their own PCIe links at the same time.  The AOV planes go the same way.
int render_to_host(EuclScene* s, const FrameBatch& fb, const EuclRenderOpts* o, uint8_t* out_rgb8, int32_t* out_hit_ids,
                   const EuclAovs* aovs, EuclStats* stats) {
    const bool scatter = !o->compact_rows && o->band_world > 1;
    const size_t my_rows = eucl_band_rows_for_rank(o);
    const size_t rows = (o->compact_rows || scatter) ? my_rows : (size_t)o->height;
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
    const int st = render_split(s, fb, &opts, (uint8_t*)s->frame.ptr, want_hit ? (int32_t*)s->hit_ids.ptr : nullptr, d_aov, stats);
    if (st != EUCL_OK) return st;
    const cudaStream_t stream = s->stream();
    if (!scatter) {
        EUCL_CUDA(cudaMemcpyAsync(out_rgb8, s->frame.ptr, pixels * 3, cudaMemcpyDeviceToHost, stream));
        if (want_hit) EUCL_CUDA(cudaMemcpyAsync(out_hit_ids, s->hit_ids.ptr, pixels * 4, cudaMemcpyDeviceToHost, stream));
        for (int k = 0; k < 5; ++k)
            if (host[k]) EUCL_CUDA(cudaMemcpyAsync(host[k], dev[k], pixels * px_bytes[k], cudaMemcpyDeviceToHost, stream));
    } else if (my_rows > 0) {
        // band k of this rank: compact rows [k * band, ...) -> frame rows [(k * world + rank) * band, ...)
        const size_t band = o->band_rows ? o->band_rows : o->height, world = o->band_world;
        const size_t full = my_rows / band, tail = my_rows % band; // whole bands, rows of a last partial band
        auto copy_bands = [&](void* dst, const void* src, size_t px_bytes) -> cudaError_t {
            const size_t band_bytes = band * o->width * px_bytes;
            uint8_t* d = (uint8_t*)dst + (size_t)o->band_rank * band_bytes;
            cudaError_t e = cudaSuccess;
            if (full) e = cudaMemcpy2DAsync(d, world * band_bytes, src, band_bytes, band_bytes, full, cudaMemcpyDeviceToHost, stream);
            if (e == cudaSuccess && tail)
                e = cudaMemcpyAsync(d + full * world * band_bytes, (const uint8_t*)src + full * band_bytes, tail * o->width * px_bytes,
                                    cudaMemcpyDeviceToHost, stream);
            return e;
        };
        EUCL_CUDA(copy_bands(out_rgb8, s->frame.ptr, 3));
        if (want_hit) EUCL_CUDA(copy_bands(out_hit_ids, s->hit_ids.ptr, 4));
        for (int k = 0; k < 5; ++k)
            if (host[k]) EUCL_CUDA(copy_bands(host[k], dev[k], px_bytes[k]));
    }
    EUCL_CUDA(cudaStreamSynchronize(stream));
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
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, &frame, 1, o, &fb, &virt)) != EUCL_OK) return st;
    return render_split(s, fb, &virt, (uint8_t*)d_out_rgb8, o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr, AovPlanes{}, stats);
}

int eucl_render_frames_device(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o,
                              void* d_out_rgb8, void* d_out_hit_ids, EuclStats* stats) {
    int st = check_frames(s, frames, n_frames, o);
    if (st != EUCL_OK) return st;
    if (!d_out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames_device: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, frames, n_frames, o, &fb, &virt)) != EUCL_OK) return st;
    return render_split(s, fb, &virt, (uint8_t*)d_out_rgb8, o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr, AovPlanes{}, stats);
}

int eucl_render_frames(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, uint8_t* out_rgb8,
                       int32_t* out_hit_ids, EuclStats* stats) {
    int st = check_frames(s, frames, n_frames, o);
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_frames: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, frames, n_frames, o, &fb, &virt)) != EUCL_OK) return st;
    return render_to_host(s, fb, &virt, out_rgb8, out_hit_ids, nullptr, stats);
}

int eucl_render(EuclScene* s, const EuclCamera* cam, const EuclRenderOpts* o, uint8_t* out_rgb8, int32_t* out_hit_ids,
                EuclStats* stats) {
    int st = check_args(s, cam, o);
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    const EuclFrame frame{*cam, o->time_seconds};
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, &frame, 1, o, &fb, &virt)) != EUCL_OK) return st;
    return render_to_host(s, fb, &virt, out_rgb8, out_hit_ids, nullptr, stats);
}

int eucl_render_aovs(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, uint8_t* out_rgb8,
                     int32_t* out_hit_ids, const EuclAovs* aovs, EuclStats* stats) {
    int st = check_aov_call(s, frames, n_frames, o, aovs, "eucl_render_aovs");
    if (st != EUCL_OK) return st;
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_aovs: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, frames, n_frames, o, &fb, &virt)) != EUCL_OK) return st;
    return render_to_host(s, fb, &virt, out_rgb8, out_hit_ids, aovs, stats);
}

int eucl_render_aovs_device(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, void* d_out_rgb8,
                            void* d_out_hit_ids, const EuclAovs* d_aovs, EuclStats* stats) {
    int st = check_aov_call(s, frames, n_frames, o, d_aovs, "eucl_render_aovs_device");
    if (st != EUCL_OK) return st;
    if (!d_out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_render_aovs_device: null output");
    EUCL_CUDA(cudaSetDevice(s->device));
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, frames, n_frames, o, &fb, &virt)) != EUCL_OK) return st;
    return render_split(s, fb, &virt, (uint8_t*)d_out_rgb8, o->want_hit_ids ? (int32_t*)d_out_hit_ids : nullptr, aov_planes(d_aovs),
                        stats);
}

int eucl_trace_rays(EuclScene* s, const EuclRays* r, uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclAovs* aovs,
                    EuclStats* stats) {
    int st = check_rays(s, r, out_rgb8, "eucl_trace_rays");
    if (st != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    double *d_o, *d_d;
    if ((st = stage_rays(s, r, &d_o, &d_d)) != EUCL_OK) return st;
    EuclRenderOpts o;
    const FrameBatch fb = ray_batch(s, r, d_o, d_d, out_hit_ids != nullptr, &o);
    return render_to_host(s, fb, &o, out_rgb8, out_hit_ids, any_plane(aovs), stats);
}

int eucl_render_trees(EuclScene* s, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* o, uint8_t* out_rgb8,
                      int32_t* out_hit_ids, const EuclTreeQuery* query, EuclStats* stats) {
    const char* fn = "eucl_render_trees";
    int st = n_frames == 1 ? check_args(s, frames ? &frames[0].camera : nullptr, o) : check_frames(s, frames, n_frames, o);
    if (st != EUCL_OK) return st;
    if (o->band_world > 1 || o->compact_rows)
        return fail(EUCL_ERR_INVALID_ARGUMENT, std::string(fn) + ": band-split and compact-row tree calls are not supported");
    if (!out_rgb8) return fail(EUCL_ERR_INVALID_ARGUMENT, std::string(fn) + ": null output");
    if ((st = check_tree_query(query, (uint64_t)n_frames * o->height * o->width, fn)) != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    FrameBatch fb;
    EuclRenderOpts virt;
    if ((st = camera_batch(s, frames, n_frames, o, &fb, &virt)) != EUCL_OK) return st;
    std::vector<uint32_t> order;
    if ((st = stage_tree_query(s, query, &order, &fb.tree)) != EUCL_OK) return st;
    if ((st = render_to_host(s, fb, &virt, out_rgb8, out_hit_ids, nullptr, stats)) != EUCL_OK) return st;
    return read_back_trees(s, query, order, fb.tree);
}

int eucl_trace_ray_trees(EuclScene* s, const EuclRays* r, uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclTreeQuery* query,
                         EuclStats* stats) {
    const char* fn = "eucl_trace_ray_trees";
    int st = check_rays(s, r, out_rgb8, fn);
    if (st != EUCL_OK) return st;
    if ((st = check_tree_query(query, r->n, fn)) != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    double *d_o, *d_d;
    if ((st = stage_rays(s, r, &d_o, &d_d)) != EUCL_OK) return st;
    EuclRenderOpts o;
    FrameBatch fb = ray_batch(s, r, d_o, d_d, out_hit_ids != nullptr, &o);
    std::vector<uint32_t> order;
    if ((st = stage_tree_query(s, query, &order, &fb.tree)) != EUCL_OK) return st;
    if ((st = render_to_host(s, fb, &o, out_rgb8, out_hit_ids, nullptr, stats)) != EUCL_OK) return st;
    return read_back_trees(s, query, order, fb.tree);
}

int eucl_trace_rays_device(EuclScene* s, const EuclRays* r, void* d_out_rgb8, void* d_out_hit_ids, const EuclAovs* d_aovs,
                           EuclStats* stats) {
    const int st = check_rays(s, r, d_out_rgb8, "eucl_trace_rays_device");
    if (st != EUCL_OK) return st;
    EUCL_CUDA(cudaSetDevice(s->device));
    EuclRenderOpts o;
    const FrameBatch fb = ray_batch(s, r, r->origins, r->directions, d_out_hit_ids != nullptr, &o);
    return render_split(s, fb, &o, (uint8_t*)d_out_rgb8, (int32_t*)d_out_hit_ids, aov_planes(any_plane(d_aovs)), stats);
}

int eucl_scene_memory(const EuclScene* s, uint64_t* arena_bytes, uint64_t* list_bytes, uint64_t* node_capacity) {
    if (!s) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_memory: null scene");
    uint64_t arena = 0, lists = 0, cap = 0;
    for (const auto& p : s->pipes) { // a split scene holds one arena per pipeline
        arena += p->nodes.bytes;
        lists += p->order.bytes + p->rorder.bytes;
        cap += (uint64_t)p->arena_capacity;
    }
    if (arena_bytes) *arena_bytes = arena;
    if (list_bytes) *list_bytes = lists;
    if (node_capacity) *node_capacity = cap;
    return EUCL_OK;
}

int eucl_scene_set_stream(EuclScene* s, void* cuda_stream) {
    if (!s) return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_scene_set_stream: null scene");
    EUCL_CUDA(cudaSetDevice(s->device));
    Pipeline& p = *s->pipes[0];
    EUCL_CUDA(cudaStreamSynchronize(p.stream));
    p.stream = cuda_stream ? (cudaStream_t)cuda_stream : p.own_stream;
    return EUCL_OK;
}

int eucl_trace_path(EuclScene* s, const double* location, const double* direction, double distance, double* out_location,
                    double* out_direction) {
    if (!s || !location || !direction || !out_location || !out_direction)
        return fail(EUCL_ERR_INVALID_ARGUMENT, "eucl_trace_path: null argument");
    EUCL_CUDA(cudaSetDevice(s->device));
    const int D = s->dim;
    const cudaStream_t stream = s->stream();
    EUCL_CUDA(s->path_io.ensure(sizeof(double) * 4 * EUCL_MAX_DIM + 16));
    double* d_in = (double*)s->path_io.ptr;
    double* d_out = d_in + 2 * EUCL_MAX_DIM;
    int* d_found = (int*)(d_out + 2 * EUCL_MAX_DIM);
    double h_in[2 * EUCL_MAX_DIM] = {0};
    for (int k = 0; k < D; ++k) {
        h_in[k] = location[k];
        h_in[D + k] = direction[k];
    }
    EUCL_CUDA(cudaMemcpyAsync(d_in, h_in, sizeof h_in, cudaMemcpyHostToDevice, stream));
    EUCL_PREC(launch_trace_path)(D, make_launch(s, *s->pipes[0], EuclRenderOpts{}), d_in, distance, d_out, d_found);
    double h_out[2 * EUCL_MAX_DIM];
    int h_found = 0;
    EUCL_CUDA(cudaMemcpyAsync(h_out, d_out, sizeof h_out, cudaMemcpyDeviceToHost, stream));
    EUCL_CUDA(cudaMemcpyAsync(&h_found, d_found, sizeof h_found, cudaMemcpyDeviceToHost, stream));
    EUCL_CUDA(cudaStreamSynchronize(stream));
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
