// CUDA kernels of the trace loop for sm_100a.
//
// Wavefront pipeline (default): ray generation -> per level { intersect, shade + emit } ->
// bottom-up resolve of the ray tree -> composite + RGB8 pack.  A one-thread-per-pixel megakernel
// over the same device functions exists as a cross-check (EUCL_PIPELINE_MEGAKERNEL).
//
// Reference semantics: Environment::render / trace_screen_point / Universe::trace*
// (src/universe/mod.rs:85-184,229-271,300-397) and ComposableSurface::get_color
// (src/universe/entity/surface.rs:62-162).  Compiled with -fmad=false.
#include "pipeline.cuh"
#include "shade.cuh"
#include <cstdio>
#include <cstdlib>

namespace EUCL_NS {
using namespace eucl;

namespace {

// resident CTAs per SM the register allocator must allow (occupancy hides the long FP64
// div/sqrt dependency chains and the instruction-fetch bubbles of this branchy code)
#ifndef EUCL_INTERSECT_MIN_BLOCKS
#define EUCL_INTERSECT_MIN_BLOCKS (kResidentThreads / kBlock)
#endif

// ---------------------------------------------------------------------------------------------
// node arena access (array-of-structures records made of 128-bit words)

// One 128-bit word of `real`s: two doubles or four floats.  Every record of the arena is a whole number of them.
constexpr int kWordReals = 16 / (int)sizeof(real);
struct __align__(16) Word {
    real v[kWordReals];
};
template <int N> // N reals, N % kWordReals == 0
__device__ __forceinline__ void store_words(void* base, size_t record, const real (&v)[N]) {
    Word* rec = reinterpret_cast<Word*>(base) + record * (N / kWordReals);
#pragma unroll
    for (int k = 0; k < N / kWordReals; ++k) {
        Word w;
#pragma unroll
        for (int j = 0; j < kWordReals; ++j) w.v[j] = v[k * kWordReals + j];
        rec[k] = w;
    }
}
template <int N, int NLOAD = N> // reads the first NLOAD reals (rounded up to whole words) of a record of N
__device__ __forceinline__ void load_words(const void* base, size_t record, real (&v)[N]) {
    const Word* rec = reinterpret_cast<const Word*>(base) + record * (N / kWordReals);
#pragma unroll
    for (int k = 0; k < (NLOAD + kWordReals - 1) / kWordReals; ++k) {
        const Word w = rec[k];
#pragma unroll
        for (int j = 0; j < kWordReals; ++j) v[k * kWordReals + j] = w.v[j];
    }
}

template <int D>
__device__ __forceinline__ void store_ray(const Workspace& ws, int node, const Vec<D>& o, const Vec<D>& d, int cur) {
    constexpr int K = ray_reals(D, (int)sizeof(real));
    real v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = k < D ? o[k < D ? k : 0] : (k < 2 * D ? d[k < 2 * D ? k - D : 0] : R(0.0));
    store_words<K>(ws.ray, (size_t)node, v);
    ws.ray_cur[node] = cur;
}
template <int D>
__device__ __forceinline__ void load_ray(const Workspace& ws, int node, Vec<D>& o, Vec<D>& d) {
    constexpr int K = ray_reals(D, (int)sizeof(real));
    real v[K];
    load_words<K, 2 * D>(ws.ray, (size_t)node, v);
#pragma unroll
    for (int k = 0; k < D; ++k) {
        o[k] = v[k];
        d[k] = v[D + k];
    }
}
// (entity, exiting) in one 32-bit pattern: entity + 1 in the low 31 bits (entity >= -1), exiting in the top bit
struct HitHead {
    real t, cos_raw, angle_raw;
    int32_t entity, exiting;
};
__device__ __forceinline__ real pack_hit_ids(int entity, int exiting) {
    const unsigned bits = (unsigned)(entity + 1) | (exiting ? 0x80000000u : 0u);
    if (kRealIsDouble) return (real)__hiloint2double(0, (int)bits);
    return (real)__int_as_float((int)bits);
}
__device__ __forceinline__ unsigned unpack_hit_ids(real v) {
    if (kRealIsDouble) return (unsigned)__double2loint((double)v);
    return (unsigned)__float_as_int((float)v);
}
template <int D>
__device__ __forceinline__ void store_hit(const Workspace& ws, int node, const HitHead& h, const Vec<D>& n) {
    constexpr int K = kHitReals;
    real v[K];
    v[0] = h.t;
    v[1] = h.cos_raw;
    v[2] = pack_hit_ids(h.entity, h.exiting);
    v[3] = h.angle_raw;
#pragma unroll
    for (int k = 4; k < K; ++k) v[k] = k - 4 < D ? n[k - 4 < D ? k - 4 : 0] : R(0.0);
    store_words<K>(ws.hit, (size_t)node, v);
}
template <int D>
__device__ __forceinline__ HitHead load_hit(const Workspace& ws, int node, Vec<D>& n) {
    constexpr int K = kHitReals;
    real v[K];
    load_words<K, 4 + D>(ws.hit, (size_t)node, v);
#pragma unroll
    for (int k = 0; k < D; ++k) n[k] = v[4 + k];
    const unsigned ids = unpack_hit_ids(v[2]);
    return HitHead{v[0], v[1], v[3], (int)(ids & 0x7fffffffu) - 1, (int)(ids >> 31)};
}
__device__ __forceinline__ void store_res(const Workspace& ws, int node, const Rgba& c) {
    const real v[4] = {c.r, c.g, c.b, c.a};
    store_words<4>(ws.res, (size_t)node, v);
}
__device__ __forceinline__ Rgba load_res(const Workspace& ws, int node) {
    real v[4];
    load_words<4>(ws.res, (size_t)node, v);
    return Rgba{v[0], v[1], v[2], v[3]};
}

// First queue position of this warp in the grid-stride walk of the queue kernels (CTA-contiguous).  Measured and not kept:
// handing consecutive 32-entry chunks to different SMs so that the last, partly filled wave of a launch spreads over the
// whole GPU -- no gain on a full 3d_room frame (15.79 vs 15.59 ms) nor on a 1/8-frame band (2.54 vs 2.50 ms).
// Also measured and not kept: letting only ceil(total / (blockDim * m)) CTAs of a launch walk the level (m items or more per
// thread, the rest of the grid exits at once) so that small levels leave SM slots to the kernels running beside them:
// m = 2 / 4 / 8 -> an eighth of a 3d_room frame 2.26 / 2.53 / 3.60 ms against 2.29, full frames equal or slower.
__device__ __forceinline__ int warp_first_position() { return (int)(blockIdx.x * blockDim.x + (threadIdx.x & ~31u)); }

// Per-thread scratch column for plane_chain (kPlaneChainMax doubles per thread, element i of thread
// t at [i * blockDim.x + t]): lives in dynamic shared memory right after the staged scene.
__device__ __forceinline__ real* plane_scratch(const uint8_t* __restrict__ blob) {
    const int blob_bytes = reinterpret_cast<const SceneHeader*>(blob)->blob_bytes;
    return reinterpret_cast<real*>(g_smem + scene_smem_bytes(blob_bytes)) + threadIdx.x;
}

// ---------------------------------------------------------------------------------------------
// shared device logic (used by the wavefront kernels and the megakernel)

// trace_closest: closest first-hit over all surfaced entities, then the geometry of the winner
// and its orientation relative to the ray (mod.rs:114-125).
template <int D>
__device__ __forceinline__ int intersect_ray(const SceneView& sv, const Vec<D>& o, const Vec<D>& d, bool& exiting, Vec<D>& p,
                                             Vec<D>& n_raw, real& cos_raw, real& angle_raw, real& t, real* ts, int ts_stride) {
    const ClosestHit h = closest_hit<D>(sv, o, d, ts, ts_stride);
    if (h.entity < 0) return -1;
    t = h.t;
    hit_geometry<D>(sv, h.prim, h.flags, o, d, h.t, p, n_raw);
    cos_raw = angle_cos(d, n_raw);
    angle_raw = angle_from_cos(cos_raw);
    exiting = angle_raw < kFracPi2;
    return h.entity;
}

template <int D>
struct ChildRay {
    Vec<D> o, d;
    int cur;
};
template <int D>
struct ShadeOut {
    real ratio;
    unsigned q;
    unsigned flags;
    Rgba sc; // valid when flags & NODE_HAS_SC
    bool t_emit, r_emit;
    ChildRay<D> t, r;
};

// ComposableSurface::get_color up to (not including) the recursive trace calls (surface.rs:62-162), in two steps so
// that the wavefront kernel can reserve the children's slots between them and build each child ray only when it is
// about to store it (the two rays are 4 * D doubles that would otherwise stay live across the whole shading code).
//
// Step 1, shade_decide: reflection ratio, surface colour and its u8 quantisation, and WHICH children exist.
// GLASS = false compiles the Fresnel / Snell providers out: the light shade kernel only ever sees surfaces
// with a uniform reflection ratio and the identity threshold direction (the host routes the bins).
// UNIFORM_SC: the surface's colour program is one EUCL_COL_UNIFORM op (the host routes the bins, k_shade_glass); its colour
// is read from the op, the value surface_color would push and pop, without the program interpreter and its stack.
template <int D>
struct ShadeDecision {
    real ratio;
    unsigned q;
    unsigned flags;
    bool t_emit, r_emit;
    int dest;          // entity the transmitted ray continues in (valid when t_emit)
    real from_theta; // angle_between(direction, -normal_closer); Fresnel / Snell surfaces only
    RefractionCache rc;
};
template <int D, bool GLASS, bool UNIFORM_SC = false>
__device__ __forceinline__ void shade_decide(const SceneView& sv, real time_millis, int ent, bool exiting, real cos_raw,
                                             real angle_raw, const Vec<D>& p, const Vec<D>& n_raw, ShadeDecision<D>& out,
                                             Rgba& sc_out) {
    const EuclSurface& sf = sv.surfaces()[sv.entities()[ent].surface];
    const real cos_closer = exiting ? -cos_raw : cos_raw;
    const bool needs_theta = GLASS && (sf.ratio_op == EUCL_RATIO_FRESNEL || sf.thr_op == EUCL_THR_SNELL);
    // angle_between(direction, -normal_closer): when exiting, -normal_closer IS the raw normal and the angle is the stored one
#if EUCL_ANGLE_REUSE
    out.from_theta = needs_theta ? (exiting ? angle_raw : angle_from_cos(-cos_closer)) : R(0.0);
#else
    out.from_theta = needs_theta ? angle_from_cos(-cos_closer) : R(0.0);
#endif
    out.rc = RefractionCache{needs_theta ? dm_sin(out.from_theta) : R(0.0), R(0.0), R(0.0), false};
    // `.min(1).max(0)`: Rust min/max drop a NaN operand, so NaN -> 1
    const real ratio = fmax(fmin(reflection_ratio<D, GLASS>(sf, out.from_theta, exiting, out.rc), R(1.0)), R(0.0));
    out.ratio = ratio;
    out.q = 0u;
    out.flags = 0u;
    out.t_emit = false;
    out.dest = -1;
    bool have_t = false;
    if (!(ratio >= R(1.0))) { // get_intersection_color
        const Rgba sc = UNIFORM_SC ? uniform_surface_color(sv, sf)
                                   : surface_color<D>(sv, sf, p, n_raw, cos_raw, angle_raw, exiting, time_millis);
        const unsigned q = to_pixel4(sc);
        out.q = q;
        if ((q >> 24) == 255u) {
            sc_out = sc;
            out.flags |= NODE_HAS_SC;
            have_t = true;
        } else {
            int dest = ent;
            if (exiting) {
                const Vec<D> n_closer = -n_raw;
                dest = material_at<D>(sv, p + (-n_closer) * kApproxEpsilon * R(128.0));
            }
            if (dest >= 0) {
                out.t_emit = true;
                out.dest = dest;
                have_t = true;
            }
        }
    }
    out.r_emit = !(ratio <= R(0.0)); // get_reflection_color
    if (!have_t && !out.r_emit) out.flags |= NODE_UNDEFINED | NODE_LEAF;
}
// Step 2: the child rays (surface.rs:84-100 transmitted, :119-139 reflected).
template <int D, bool GLASS>
__device__ __forceinline__ void transmit_child(const SceneView& sv, const Vec<D>& dir, int cur, int ent, bool exiting, const Vec<D>& p,
                                               const Vec<D>& n_raw, ShadeDecision<D>& dec, ChildRay<D>& out) {
    const EuclSurface& sf = sv.surfaces()[sv.entities()[ent].surface];
    const Vec<D> n_closer = exiting ? -n_raw : n_raw;
    Vec<D> td = threshold_direction<D, GLASS>(sf, dir, n_closer, exiting, dec.from_theta, dec.rc);
    out.o = p + (-n_closer) * kApproxEpsilon * R(128.0);
    material_exit<D>(sv, cur, td);
    material_enter<D>(sv, dec.dest, td);
    out.d = td;
    out.cur = dec.dest;
}
template <int D>
__device__ __forceinline__ void reflect_child(const Vec<D>& dir, int cur, bool exiting, const Vec<D>& p, const Vec<D>& n_raw,
                                              ChildRay<D>& out) {
    const Vec<D> n_closer = exiting ? -n_raw : n_raw;
    out.o = p + n_closer * kApproxEpsilon * R(128.0);
    out.d = reflection_direction<D>(dir, n_closer);
    out.cur = cur;
}

// Both steps at once (megakernel, which keeps the children on its own stack).
template <int D, bool GLASS>
__device__ __forceinline__ void shade_hit(const SceneView& sv, real time_millis, const Vec<D>& dir, int cur, int ent,
                                          bool exiting, real cos_raw, real angle_raw, const Vec<D>& p, const Vec<D>& n_raw,
                                          ShadeOut<D>& out) {
    ShadeDecision<D> dec;
    shade_decide<D, GLASS>(sv, time_millis, ent, exiting, cos_raw, angle_raw, p, n_raw, dec, out.sc);
    out.ratio = dec.ratio;
    out.q = dec.q;
    out.flags = dec.flags;
    out.t_emit = dec.t_emit;
    out.r_emit = dec.r_emit;
    if (dec.t_emit) transmit_child<D, GLASS>(sv, dir, cur, ent, exiting, p, n_raw, dec, out.t);
    if (dec.r_emit) reflect_child<D>(dir, cur, exiting, p, n_raw, out.r);
}

// Colour of an inner node from its children (surface.rs:104-114,150-161)
__device__ __forceinline__ Rgba transmit_over(unsigned q, const Rgba& child) {
    return from_premultiplied(over_pre(into_premultiplied(new_u8(q)), into_premultiplied(new_u8(to_pixel4(child)))));
}
// The same with Rgba::new_u8's eight divisions by 255 read from a table of the 256 quotients (`unit[v] = v / 255`, filled by
// fill_unit_table with that very division, so the values are the same bits): the resolve kernels are issue-bound, not
// memory-bound, and an f64 division is ~30 instructions (profiles/README.md, resolve capture).
__device__ __forceinline__ Rgba new_u8(unsigned q, const real* __restrict__ unit) {
    return Rgba{unit[q & 255u], unit[(q >> 8) & 255u], unit[(q >> 16) & 255u], unit[q >> 24]};
}
__device__ __forceinline__ Rgba transmit_over(unsigned q, const Rgba& child, const real* __restrict__ unit) {
    return from_premultiplied(over_pre(into_premultiplied(new_u8(q, unit)), into_premultiplied(new_u8(to_pixel4(child), unit))));
}
// 256-thread CTAs: one quotient per thread
__device__ __forceinline__ void fill_unit_table(real* unit) {
    for (unsigned v = threadIdx.x; v < 256u; v += blockDim.x) unit[v] = (real)v / R(255.0);
    __syncthreads();
}

// trace_unknown tail (mod.rs:260-270) + to_pixel (mod.rs:342): composite over opaque white
__device__ __forceinline__ void final_rgb8(const Rgba& fg, bool composite, uint8_t* out) {
    Rgba c = fg;
    if (composite) c = from_premultiplied(over_pre(into_premultiplied(fg), Pre{R(1.0), R(1.0), R(1.0), R(1.0)}));
    out[0] = (uint8_t)channel_to_u8(c.r);
    out[1] = (uint8_t)channel_to_u8(c.g);
    out[2] = (uint8_t)channel_to_u8(c.b);
}

// Camera::get_ray_vector (d3/entity/camera.rs:164-185, d4/entity/camera.rs:155-176)
template <int D>
__device__ __forceinline__ Vec<D> camera_ray(const FrameParams& fp, int x, int y) {
    const real rel_x = (real)(x - fp.width / 2) + (real)(1 - fp.width % 2) / R(2.0);
    const real rel_y = (real)(y - fp.height / 2) + (real)(1 - fp.height % 2) / R(2.0);
    Vec<D> loc, center, up, right;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        loc[k] = R(fp.location[k]);
        center[k] = R(fp.center[k]);
        up[k] = R(fp.up[k]);
        right[k] = R(fp.right[k]);
    }
    const Vec<D> screen_point = center + (up * rel_y) + (right * rel_x);
    return normalize(screen_point - loc);
}

__device__ __forceinline__ Rgba checkerboard(int x, int y) { // mod.rs:387-395
    if ((x / 8 + y / 8) % 2 == 0) return Rgba{R(0.0), R(0.0), R(0.0), R(1.0)};
    return Rgba{R(1.0), R(0.0), R(1.0), R(1.0)};
}

// ---------------------------------------------------------------------------------------------
// kernels

// material_at(camera location) is the same for every pixel of a frame: computed once (a batch: once per frame, and
// cam_entity says whether any frame is traced at all).
template <int D>
__global__ void __launch_bounds__(32) k_camera_entity(const uint8_t* __restrict__ blob, FrameParams fp, Workspace ws) {
    const SceneView& sv = stage_scene(blob);
    if (!ws.frames) {
        if (threadIdx.x == 0) {
            Vec<D> loc;
#pragma unroll
            for (int k = 0; k < D; ++k) loc[k] = R(fp.location[k]);
            *ws.cam_entity = material_at<D>(sv, loc);
        }
        return;
    }
    bool traced = false;
    for (int f = threadIdx.x; f < ws.n_frames; f += blockDim.x) {
        Vec<D> loc;
#pragma unroll
        for (int k = 0; k < D; ++k) loc[k] = R(ws.frames[f].location[k]);
        const int e = material_at<D>(sv, loc);
        ws.frame_entity[f] = e;
        traced = traced || e >= 0;
    }
    traced = __any_sync(0xffffffffu, traced);
    if (threadIdx.x == 0) *ws.cam_entity = traced ? 0 : -1;
}

// Frame of virtual row `y` of a batch; `y` becomes the row within that frame.
__device__ __forceinline__ int frame_of_row(const Workspace& ws, int& y) {
    const int f = y / ws.frame_rows;
    y -= f * ws.frame_rows;
    return f;
}

// K1 (k_raygen, k_raygen_rays) with ws.ray_bins: primary ray i joins the reach-key list of its key when it is traced (one
// atomicAdd per warp and key).  Every lane of the warp calls it.
template <int D>
__device__ __forceinline__ void bin_primary(const SceneView& sv, const Workspace& ws, int i, unsigned lane, bool traced,
                                            const Vec<D>& o, const Vec<D>& dir) {
    const unsigned active = __ballot_sync(0xffffffffu, traced);
    if (traced) {
        const int key = reach_key<D>(sv, o, dir);
        const unsigned peers = __match_any_sync(active, key);
        const int leader = __ffs(peers) - 1;
        int s2 = 0;
        if ((int)lane == leader) s2 = atomicAdd(&ws.rbin_count[key], __popc(peers));
        s2 = __shfl_sync(peers, s2, leader);
        ws.rorder[(size_t)key * ws.list_cap + s2 + __popc(peers & ((1u << lane) - 1u))] = i;
    }
}

// K1: one primary ray per pixel of the chunk; level 0 of the node arena is the pixel order.
template <int D>
__global__ void __launch_bounds__(kBlock) k_raygen(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                   Workspace ws, int32_t* __restrict__ hit_ids_out) {
    const SceneView& sv = stage_scene(blob);
    const bool batch = ws.frames != nullptr;
    Vec<D> loc;
#pragma unroll
    for (int k = 0; k < D; ++k) loc[k] = R(fp.location[k]);
    // material_at(camera location) is the same for every pixel of a frame: one thread per CTA evaluates it (a few hundred
    // instructions) instead of a kernel of its own in front of this one.  A batch reads its frames' entities from the
    // table k_camera_entity filled (a CTA's pixels may belong to several frames).
    __shared__ int s_cam_entity;
    if (threadIdx.x == 0) {
        if (!batch) s_cam_entity = material_at<D>(sv, loc);
        if (blockIdx.x == 0) {
            if (!batch) *ws.cam_entity = s_cam_entity;
            ws.count[0] = cp.n_pixels;
            ws.level_off[0] = 0;
        }
    }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < cp.n_pixels; base += gridDim.x * blockDim.x) {
        const int i = base + (int)lane;
        const bool valid = i < cp.n_pixels;
        const int local_row = cp.local_row0 + (valid ? i : 0) / fp.width;
        const int x = (valid ? i : 0) % fp.width;
        int y = frame_row_of_local(cp, local_row);
        int belongs_to = s_cam_entity, f = 0;
        if (batch) {
            f = frame_of_row(ws, y);
            belongs_to = ws.frame_entity[f];
#pragma unroll
            for (int k = 0; k < D; ++k) loc[k] = R(ws.frames[f].location[k]);
            if (valid) ws.node_frame[i] = f;
            const unsigned untraced = __ballot_sync(0xffffffffu, valid && belongs_to < 0);
            if (lane == 0 && untraced) atomicAdd(ws.untraced, __popc(untraced));
        }
        if (belongs_to < 0) { // a single frame: the same for every pixel
            if (valid) {
                store_res(ws, i, checkerboard(x, y));
                ws.meta[i] = NodeMeta{R(0.0), -1, -1, 0u, NODE_LEAF | NODE_FINAL_RGB};
                ws.ray_cur[i] = -1;
                if (hit_ids_out) hit_ids_out[(size_t)out_row_of_local(cp, local_row) * fp.width + x] = -2;
            }
            // a batch goes on: the node gets a well-defined ray (k_intersect may walk it when the level is not grouped by
            // reach key); ray_cur -1 keeps k_shade off it
            if (!batch) continue;
        }
        const bool traced = belongs_to >= 0;
        Vec<D> dir = batch ? camera_ray<D>(ws.frames[f], x, y) : camera_ray<D>(fp, x, y);
        if (traced) material_enter<D>(sv, belongs_to, dir);
        if (valid) store_ray<D>(ws, i, loc, dir, traced ? belongs_to : -1);
        if (ws.ray_bins) bin_primary<D>(sv, ws, i, lane, valid && traced, loc, dir); // like k_shade groups the children
    }
}

// K1 of eucl_trace_rays*: the caller's rays instead of a camera.  Node i of the chunk is cell (x, y) of the call's virtual
// frame of n / width rows, i.e. ray y * width + x of the [n][dim] f64 arrays, narrowed once to `real`.  Every ray has an
// origin of its own, so every thread evaluates material_at (k_raygen does it once per CTA).  A ray whose origin lies in no
// entity is a checkerboard leaf of its cell, like a pixel of an untraced frame of a batch, and is counted in ws.untraced;
// *ws.cam_entity keeps the 0 of the counter reset, so the level is intersected whenever any of its rays is traced.
template <int D>
__global__ void __launch_bounds__(kBlock) k_raygen_rays(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                        Workspace ws, int32_t* __restrict__ hit_ids_out,
                                                        const double* __restrict__ origins, const double* __restrict__ directions) {
    const SceneView& sv = stage_scene(blob);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        ws.count[0] = cp.n_pixels;
        ws.level_off[0] = 0;
    }
    const unsigned lane = threadIdx.x & 31u;
    for (int base = blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < cp.n_pixels; base += gridDim.x * blockDim.x) {
        const int i = base + (int)lane;
        const bool valid = i < cp.n_pixels;
        const int local_row = cp.local_row0 + (valid ? i : 0) / fp.width;
        const int x = (valid ? i : 0) % fp.width;
        const int y = frame_row_of_local(cp, local_row);
        const size_t ray = ((size_t)y * fp.width + x) * D;
        Vec<D> o, dir;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            o[k] = R(origins[ray + k]);
            dir[k] = R(directions[ray + k]);
        }
        const int belongs_to = valid ? material_at<D>(sv, o) : -1;
        const bool traced = belongs_to >= 0;
        const unsigned untraced = __ballot_sync(0xffffffffu, valid && !traced);
        if (lane == 0 && untraced) atomicAdd(ws.untraced, __popc(untraced));
        if (valid && !traced) {
            store_res(ws, i, checkerboard(x, y));
            ws.meta[i] = NodeMeta{R(0.0), -1, -1, 0u, NODE_LEAF | NODE_FINAL_RGB};
            if (hit_ids_out) hit_ids_out[(size_t)out_row_of_local(cp, local_row) * fp.width + x] = -2;
        }
        // an untraced node keeps its ray as given (k_intersect may walk it when the level is not grouped by reach key);
        // ray_cur -1 keeps k_shade off it
        if (traced) material_enter<D>(sv, belongs_to, dir);
        if (valid) store_ray<D>(ws, i, o, dir, traced ? belongs_to : -1);
        if (ws.ray_bins) bin_primary<D>(sv, ws, i, lane, valid && traced, o, dir);
    }
}

// K2: closest hit of every ray of one level.
//
// Two builds share a level when its rays are grouped by reach key and the scene allows it (SceneHeader::light_capable):
// the LIGHT one walks the rays with key 0 -- they can only hit primitives and root plane chains -- without the CSG
// evaluator and its per-thread hit arena, at a fraction of the registers; the HEAVY one walks the other keys (or every
// ray when the level is not grouped).  `key_mask` selects the reach-key lists of a launch.  In a csg2-capable scene
// (SceneHeader::csg2_capable) k_intersect_csg2 takes the HEAVY one's place: closest_hit_csg2 instead of closest_hit, so
// no hit arena and no stack.
enum : int { K2_HEAVY = 0, K2_LIGHT = 1, K2_CSG2 = 2 };
template <int D, int BUILD>
__device__ __forceinline__ void intersect_level(const uint8_t* __restrict__ blob, const Workspace& ws, int level, unsigned key_mask) {
    // an earlier level did not fit: the host grows the arena and retries.  One decision per block (see k_shade).
    __shared__ int s_skip, s_total;
    __shared__ int s_rprefix[kRayBins + 1];
    const int off = ws.level_off[level], cnt = ws.count[level];
    const bool grouped = ws.ray_bins != 0;
    // list sizes: one global load per thread, all in flight at once (a serial loop of dependent loads in front of every
    // CTA's work was most of the fixed cost of a launch: ~10 us), then a prefix sum over shared memory
    __shared__ int s_rcount[kRayBins];
    if (threadIdx.x < kRayBins)
        s_rcount[threadIdx.x] = (grouped && ((key_mask >> threadIdx.x) & 1u)) ? ws.rbin_count[level * kRayBins + threadIdx.x] : 0;
    if (threadIdx.x == 32) // no ray at all when the camera is in no entity (checkerboard frame, mod.rs:385-396)
        s_skip = *ws.overflow != 0 || *ws.cam_entity < 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = cnt;
        if (grouped) {
            acc = 0;
            for (int b = 0; b < kRayBins; ++b) {
                s_rprefix[b] = acc;
                acc += s_rcount[b];
            }
            s_rprefix[kRayBins] = acc;
        }
        s_total = acc;
        if (blockIdx.x == 0) ws.level_off[level + 1] = off + cnt;
    }
    __syncthreads();
    const int total = s_total;
    if (s_skip || (int)(blockIdx.x * blockDim.x) >= total) return;
    const SceneView& sv = stage_scene(blob);
    real* ts = plane_scratch(blob);
    const unsigned lane = threadIdx.x & 31u;
    const int stride = gridDim.x * blockDim.x;
    const int first = warp_first_position();
    int bin = 0; // the lists of a launch are walked front to back: the cursor only moves forward
    auto node_at = [&](int i) -> int {
        if (i >= total) return -1;
        if (!grouped) return off + i;
        while (i >= s_rprefix[bin + 1]) ++bin;
        return ws.rorder[(size_t)bin * ws.list_cap + (i - s_rprefix[bin])];
    };
    int node_next = node_at(first + (int)lane);
    for (int base = first; base < total; base += stride) {
        int node = node_next;
        node_next = node_at(base + stride + (int)lane);
        bool valid = node >= 0;
        if (grouped && valid && (node < off || node >= off + cnt)) { // must not happen: reported, never dereferenced
            *ws.overflow = 2;
            valid = false;
        }
        int ent = -1;
        bool exiting_flag = false;
        real cos_hint = R(0.0);
        if (valid) {
            Vec<D> o, d;
            load_ray<D>(ws, node, o, d);
            const ClosestHit h = BUILD == K2_LIGHT  ? closest_hit_light<D>(sv, o, d, ts, (int)blockDim.x)
                                 : BUILD == K2_CSG2 ? closest_hit_csg2<D>(sv, o, d, ts, (int)blockDim.x)
                                                    : closest_hit<D>(sv, o, d, ts, (int)blockDim.x);
            HitHead rec{R(0.0), R(0.0), R(0.0), -1, 0};
            Vec<D> n;
#pragma unroll
            for (int k = 0; k < D; ++k) n[k] = R(0.0);
            if (h.entity >= 0) { // orientation of the winner relative to the ray (mod.rs:114-125)
                Vec<D> p;
                hit_geometry<D>(sv, h.prim, h.flags, o, d, h.t, p, n);
                const real cos_raw = angle_cos(d, n);
                const real angle_raw = angle_from_cos(cos_raw);
                const bool exiting = angle_raw < kFracPi2;
                rec = HitHead{h.t, cos_raw, angle_raw, h.entity, exiting ? 1 : 0};
                exiting_flag = exiting;
                cos_hint = cos_raw;
            }
            ent = h.entity;
            store_hit<D>(ws, node, rec, n);
        }
        if (ws.n_bins > 1) {
            // group the level's nodes by hit entity so that a shading warp runs ONE surface program:
            // one atomicAdd per (warp, distinct key), ranks from the match mask
            const unsigned active = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                // key: miss = 0, else 1 + 3 * entity + class.  Classes: 0 entering, 1 exiting (these run material_at),
                // 2 exiting a Fresnel surface beyond the critical angle (they only reflect: no Snell rotation, no
                // material_at).  The class is an ordering hint estimated from cos_raw; shading decides for real.
                int cls = exiting_flag ? 1 : 0;
                if (exiting_flag && ent >= 0) {
                    const EuclSurface& sf = sv.surfaces()[sv.entities()[ent].surface];
                    if (sf.ratio_op == EUCL_RATIO_FRESNEL) {
                        // (from_index / to_index)^2 sin^2 > 1 with from = ratio_a, to = ratio_b when exiting; no division
                        if (R(sf.ratio_a) * R(sf.ratio_a) * (R(1.0) - cos_hint * cos_hint) > R(sf.ratio_b) * R(sf.ratio_b)) cls = 2;
                    }
                }
                const int key = ent < 0 ? 0 : 1 + kBinsPerEntity * ent + cls;
                const unsigned peers = __match_any_sync(active, key);
                const int leader = __ffs(peers) - 1;
                int slot = 0;
                if ((int)lane == leader) slot = atomicAdd(&ws.bin_count[level * kMaxBins + key], __popc(peers));
                slot = __shfl_sync(peers, slot, leader);
                ws.order[(size_t)key * ws.list_cap + slot + __popc(peers & ((1u << lane) - 1u))] = node;
            }
        }
    }
}

template <int D, bool LIGHT>
__global__ void __launch_bounds__(LIGHT ? kLightK2Block : kBlock, LIGHT ? EUCL_INTERSECT_LIGHT_MIN_BLOCKS : EUCL_INTERSECT_MIN_BLOCKS)
    k_intersect(const uint8_t* __restrict__ blob, Workspace ws, int level, unsigned key_mask) {
    intersect_level<D, LIGHT ? K2_LIGHT : K2_HEAVY>(blob, ws, level, key_mask);
}

template <int D>
__global__ void __launch_bounds__(kCsg2Block, csg2_resident_blocks(D, (int)sizeof(real)))
    k_intersect_csg2(const uint8_t* __restrict__ blob, Workspace ws, int level, unsigned key_mask) {
    intersect_level<D, K2_CSG2>(blob, ws, level, key_mask);
}

// K3: shade every node of one level and append its children to the next level.  Children are
// appended with one atomicAdd per warp (ballot + popc ranks).
//
// Two builds of the kernel share a level: the LIGHT one (GLASS = false) shades the bins whose surfaces have a
// uniform reflection ratio and the identity threshold direction -- walls, mirrors, tinted and opaque objects --
// plus the rays that hit nothing; without the Fresnel / Snell / general_rotation code it needs far fewer registers
// and keeps more warps resident.  The HEAVY one (GLASS = true) shades the remaining bins (and everything when the
// level is not binned).  `bin_mask` selects the bins of a launch.
//
// FRAMES: a batch of frames (Workspace::node_frame): Perlin time from the node's frame, children tagged with it.  A build of
// its own so that the single-frame builds carry none of it.
//
// k_shade_glass is the heavy build for the bins of Fresnel / Snell surfaces whose colour program is one constant
// (UNIFORM_SC): the same code without the colour-program interpreter, so that it needs fewer registers and no colour stack.
template <int D, bool RAY_BINS, bool GLASS, bool FRAMES, bool UNIFORM_SC>
__device__ __forceinline__ void shade_level(const uint8_t* __restrict__ blob, const FrameParams& fp, const ChunkParams& cp,
                                            const Workspace& ws, int level, unsigned long long bin_mask, int32_t* __restrict__ hit_ids_out) {
    const int off = ws.level_off[level], cnt = ws.count[level];
    const bool last_level = level >= fp.max_depth; // depth 0: background without intersecting (mod.rs:157,183)
    // binned levels: position g of the concatenated bins of this launch -> (bin, index) through the bin prefix sums
    __shared__ int s_prefix[kMaxBins + 1];
    // An overflow flagged by an EARLIER kernel means this level's queue is incomplete: skip it (the host
    // retries with a larger arena).  Blocks of THIS launch set the flag too, so the decision must be taken
    // once per block: threads reading the flag on their own could disagree, and the ones that left would
    // be missing from the cooperative scene staging below (a partially staged scene = wild table offsets).
    __shared__ int s_skip, s_total;
    const bool binned = ws.n_bins > 1 && !last_level;
    // bin sizes: one global load per thread, all in flight at once, then a prefix sum over shared memory (see k_intersect)
    __shared__ int s_bcount[kMaxBins];
    if (threadIdx.x < kMaxBins)
        s_bcount[threadIdx.x] = (binned && (int)threadIdx.x < ws.n_bins && ((bin_mask >> threadIdx.x) & 1ull))
                                    ? ws.bin_count[level * kMaxBins + threadIdx.x] : 0;
    if (threadIdx.x == 64) s_skip = level > 0 && *ws.overflow != 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        int acc = cnt;
        if (binned) {
            acc = 0;
            for (int b = 0; b < ws.n_bins; ++b) {
                s_prefix[b] = acc;
                acc += s_bcount[b];
            }
            s_prefix[ws.n_bins] = acc;
        }
        s_total = acc;
    }
    __syncthreads();
    const int total = s_total;
    if (s_skip || (int)(blockIdx.x * blockDim.x) >= total) return;
    const SceneView& sv = stage_scene(blob);
    const int first = warp_first_position();
    const int next_off = last_level ? 0 : ws.level_off[level + 1];
    const unsigned lane = threadIdx.x & 31u;
    const int stride = gridDim.x * blockDim.x;
    // node of position g; the bins of a launch are walked front to back, so the bin cursor only moves forward
    int bin = 0;
    auto node_at = [&](int g) -> int {
        if (g >= total) return -1;
        if (!binned) return off + g;
        while (g >= s_prefix[bin + 1]) ++bin;
        return ws.order[(size_t)bin * ws.list_cap + (g - s_prefix[bin])];
    };
    int node_next = node_at(first + (int)lane);
    for (int base = first; base < total; base += stride) {
        int node = node_next;
        node_next = node_at(base + stride + (int)lane); // the index of the next iteration travels while this one computes
        bool valid = node >= 0;
        if (binned && valid && (node < off || node >= off + cnt)) { // must not happen: reported, never dereferenced
            *ws.overflow = 2;
            valid = false;
        }
        if (!valid) node = off;
        int cur = -1;
        if (valid) {
            cur = ws.ray_cur[node];
            valid = cur >= 0; // checkerboard pixels carry no ray
        }
        const int i = node - off;
        ShadeDecision<D> dec;
        dec.t_emit = false;
        dec.r_emit = false;
        bool shaded = false;
        if (valid) {
            Vec<D> o, d, n;
            load_ray<D>(ws, node, o, d);
            HitHead ei{R(0.0), R(0.0), R(0.0), -1, 0};
            if (!last_level) ei = load_hit<D>(ws, node, n);
            if (level == 0 && hit_ids_out) {
                const int local_row = cp.local_row0 + i / fp.width;
                const int orow = out_row_of_local(cp, local_row);
                hit_ids_out[(size_t)orow * fp.width + i % fp.width] = ei.entity;
            }
            if (ei.entity < 0) {
                store_res(ws, node, mapped_color<D>(sv, sv.background, d)); // background.get_color(direction.to_point())
                ws.meta[node] = NodeMeta{R(0.0), -1, -1, 0u, NODE_LEAF};
            } else {
                const Vec<D> p = o + d * ei.t; // the intersectors' expression for the hit location (shape.rs:700,795,993)
                Rgba sc;
                const real time_millis = R(FRAMES ? ws.frames[ws.node_frame[node]].time_millis : fp.time_millis);
                shade_decide<D, GLASS, UNIFORM_SC>(sv, time_millis, ei.entity, ei.exiting != 0, ei.cos_raw, ei.angle_raw, p, n, dec, sc);
                if (dec.flags & NODE_HAS_SC) {
                    store_res(ws, node, sc);
                    if (!dec.r_emit) dec.flags |= NODE_LEAF; // opaque without a mirror term: the colour is final
                }
                if (dec.flags & NODE_UNDEFINED) {
                    store_res(ws, node, Rgba{R(0.0), R(0.0), R(0.0), R(0.0)});
                    atomicAdd(ws.undefined_count, 1ull);
                }
                shaded = true;
            }
        }
        // warp-aggregated append of the children to level + 1: one atomicAdd per warp.  (Measured and not kept: adjacent
        // slots for the two children of a node, so that the resolve reads them as one 64-byte piece: resolve 1.77 -> 1.77 ms,
        // shade 7.60 -> 8.01.)
        const unsigned tmask = __ballot_sync(0xffffffffu, dec.t_emit), rmask = __ballot_sync(0xffffffffu, dec.r_emit);
        const int nt = __popc(tmask), n_children = nt + __popc(rmask);
        int slot = 0;
        if (n_children > 0) {
            if (lane == 0) slot = atomicAdd(&ws.count[level + 1], n_children);
            slot = __shfl_sync(0xffffffffu, slot, 0);
        }
        const bool fits_arena = (long long)next_off + slot + n_children <= (long long)ws.capacity;
        const bool fits = n_children > 0 && fits_arena && slot + n_children <= ws.list_cap; // the index lists hold one level each
        if (n_children > 0 && !fits && lane == 0) *ws.overflow = fits_arena ? 3 : 1;
        int tchild = -1, rchild = -1, tkey = 0, rkey = 0;
        if (shaded) {
            if (fits && (dec.t_emit || dec.r_emit)) {
                // The child rays need the ray and the hit again.  They are re-read from the node arena (L2-hot: this thread
                // loaded them a few microseconds ago) instead of being kept in ~40 registers across the whole shading code;
                // the loads are issued while the slot reservation above is still in flight.
                Vec<D> o, d, n;
                load_ray<D>(ws, node, o, d);
                const HitHead ei = load_hit<D>(ws, node, n);
                const Vec<D> p = o + d * ei.t;
                const bool exiting = ei.exiting != 0;
                const unsigned lt = (1u << lane) - 1u;
                ChildRay<D> child; // one child at a time: built, stored, forgotten
                if (dec.t_emit) {
                    tchild = next_off + slot + __popc(tmask & lt);
                    transmit_child<D, GLASS>(sv, d, cur, ei.entity, exiting, p, n, dec, child);
                    store_ray<D>(ws, tchild, child.o, child.d, child.cur);
                    if (FRAMES) ws.node_frame[tchild] = ws.node_frame[node]; // a batch: the children belong to their parent's frame
                    if (RAY_BINS) tkey = reach_key<D>(sv, child.o, child.d);
                }
                if (dec.r_emit) {
                    rchild = next_off + slot + nt + __popc(rmask & lt);
                    reflect_child<D>(d, cur, exiting, p, n, child);
                    store_ray<D>(ws, rchild, child.o, child.d, child.cur);
                    if (FRAMES) ws.node_frame[rchild] = ws.node_frame[node];
                    if (RAY_BINS) rkey = reach_key<D>(sv, child.o, child.d);
                }
            }
            ws.meta[node] = NodeMeta{dec.ratio, tchild, rchild, dec.q, dec.flags};
        }
        if (RAY_BINS) {
            // group the NEXT level's rays by reach key: one atomicAdd per warp and distinct key, for the transmitted
            // children and then for the reflected ones
            auto bin_child = [&](int child, int key) {
                const unsigned active = __ballot_sync(0xffffffffu, child >= 0);
                if (child >= 0) {
                    const unsigned peers = __match_any_sync(active, key);
                    const int leader = __ffs(peers) - 1;
                    int s2 = 0;
                    if ((int)lane == leader) s2 = atomicAdd(&ws.rbin_count[(level + 1) * kRayBins + key], __popc(peers));
                    s2 = __shfl_sync(peers, s2, leader);
                    ws.rorder[(size_t)key * ws.list_cap + s2 + __popc(peers & ((1u << lane) - 1u))] = child;
                }
            };
            bin_child(tchild, tkey);
            bin_child(rchild, rkey);
        }
    }
}
template <int D, bool RAY_BINS, bool GLASS, bool FRAMES>
__global__ void __launch_bounds__(GLASS ? kShadeBlock : kLightBlock, GLASS ? EUCL_SHADE_MIN_BLOCKS : EUCL_SHADE_LIGHT_MIN_BLOCKS)
    k_shade(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp, Workspace ws, int level, unsigned long long bin_mask,
            int32_t* __restrict__ hit_ids_out) {
    shade_level<D, RAY_BINS, GLASS, FRAMES, false>(blob, fp, cp, ws, level, bin_mask, hit_ids_out);
}
template <int D, bool RAY_BINS, bool FRAMES>
__global__ void __launch_bounds__(kShadeGlassBlock, shade_glass_resident_blocks(RAY_BINS, (int)sizeof(real)))
    k_shade_glass(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp, Workspace ws, int level,
                  unsigned long long bin_mask, int32_t* __restrict__ hit_ids_out) {
    shade_level<D, RAY_BINS, true, FRAMES, true>(blob, fp, cp, ws, level, bin_mask, hit_ids_out);
}

// K3 of the LAST level: depth 0, `background.get_color(direction)` without intersecting (mod.rs:157,183).  A kernel of its
// own because k_shade's register budget (128: the surface programs) would keep only 16 warps per SM resident for what is
// a direction -> texture lookup per node (profiles/README.md: last-level capture).
template <int D>
__global__ void __launch_bounds__(256, EUCL_BACKGROUND_MIN_BLOCKS)
    k_background(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp, Workspace ws, int level, int32_t* __restrict__ hit_ids_out) {
    const int off = ws.level_off[level], cnt = ws.count[level];
    __shared__ int s_skip; // decided once per block (see k_shade)
    if (threadIdx.x == 0) s_skip = level > 0 && *ws.overflow != 0;
    __syncthreads();
    if (s_skip || (int)(blockIdx.x * blockDim.x) >= cnt) return;
    const SceneView& sv = stage_scene(blob);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) {
        const int node = off + i;
        if (ws.ray_cur[node] < 0) continue; // checkerboard pixels carry no ray
        Vec<D> o, d;
        load_ray<D>(ws, node, o, d);
        if (level == 0 && hit_ids_out) { // max_depth 0: every primary ray goes to the background
            const int local_row = cp.local_row0 + i / fp.width;
            hit_ids_out[(size_t)out_row_of_local(cp, local_row) * fp.width + i % fp.width] = -1;
        }
        store_res(ws, node, mapped_color<D>(sv, sv.background, d));
        ws.meta[node] = NodeMeta{R(0.0), -1, -1, 0u, NODE_LEAF};
    }
}

// Colour of a node from the (already final) colours of its children (surface.rs:104-114 transmitted, :150-161 combine).
// Measured and not kept: resolving two levels per launch with the middle level's colours in registers (5 launches instead of
// 10, a quarter less traffic, but a dependent chain of two gathers per thread): 3d_room 1.68 -> 2.03 ms, 4d_room 0.95 -> 1.06;
// two nodes per thread and iteration with both nodes' gathers issued before either is composed: 0.98 -> 1.04 ms.
__device__ __forceinline__ Rgba node_color(const Workspace& ws, const NodeMeta& m, int node, const real* __restrict__ unit) {
    if (m.flags & NODE_LEAF) return load_res(ws, node);
    bool have_t = false;
    Rgba t{R(0.0), R(0.0), R(0.0), R(0.0)};
    if (m.flags & NODE_HAS_SC) {
        t = load_res(ws, node);
        have_t = true;
    } else if (m.tchild >= 0) {
        t = transmit_over(m.q, load_res(ws, m.tchild), unit);
        have_t = true;
    }
    Rgba out = t;
    if (m.rchild >= 0) {
        const Rgba r = load_res(ws, m.rchild);
        out = have_t ? combine_palette_color(r, t, (real)m.ratio) : r;
    }
    return out;
}

// Tree cost (segments, levels) of a node at `level` (AovPlanes::segments / levels): the node itself is one Universe::trace
// call with depth > 0 when level < max_depth, and reaches level + 1 levels; an inner node adds its children's segments and
// takes the maximum of their levels.  Every node of levels 1 .. max_depth - 1 gets its cost from k_resolve_cost of its own
// level -- leaves included, although their colour needs no resolving.  The nodes of level max_depth (background lookups,
// leaves all) are never resolved: their parents derive the cost from the level.
__device__ __forceinline__ uint2 leaf_cost(int level, int max_depth) {
    return make_uint2(level < max_depth ? 1u : 0u, (unsigned)level + 1u);
}
__device__ __forceinline__ uint2 tree_cost(const NodeMeta& m, int level, int max_depth, const uint2* __restrict__ cost) {
    uint2 c = leaf_cost(level, max_depth);
    if (m.flags & NODE_LEAF) return c;
    const int child[2] = {m.tchild, m.rchild};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        if (child[k] < 0) continue;
        const uint2 cc = level + 1 >= max_depth ? leaf_cost(level + 1, max_depth) : cost[child[k]];
        c.x += cc.x;
        c.y = max(c.y, cc.y);
    }
    return c;
}

// K4: colour of the inner nodes of one level from the colours of level + 1.  COST (k_resolve_cost): also the tree cost of
// every node of the level.  Two kernels over one body so that the plain one keeps its symbol and its code.
template <bool COST>
__device__ __forceinline__ void resolve_level(const Workspace& ws, int level, int max_depth, const AovPlanes& aov) {
    __shared__ real s_unit[256];
    if (*ws.overflow) return;
    fill_unit_table(s_unit);
    const int off = ws.level_off[level], cnt = ws.count[level];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += gridDim.x * blockDim.x) {
        const int node = off + i;
        const NodeMeta m = ws.meta[node];
        if (COST) aov.cost[node] = tree_cost(m, level, max_depth, aov.cost);
        if (m.flags & NODE_LEAF) continue;
        store_res(ws, node, node_color(ws, m, node, s_unit));
    }
}
__global__ void __launch_bounds__(256) k_resolve(Workspace ws, int level) { resolve_level<false>(ws, level, 0, AovPlanes{}); }
__global__ void __launch_bounds__(256) k_resolve_cost(Workspace ws, int level, int max_depth, AovPlanes aov) {
    resolve_level<true>(ws, level, max_depth, aov);
}

// K5: resolve level 0, composite over white, quantise and pack RGB8 rows (row 0 = bottom).  COST (k_final_cost): also the
// segments / levels planes from the tree cost of level 0 (0 / 0 for checkerboard pixels).
template <bool COST>
__device__ __forceinline__ void final_pixels(const FrameParams& fp, const ChunkParams& cp, const Workspace& ws,
                                             uint8_t* __restrict__ out_rgb8, const AovPlanes& aov) {
    __shared__ real s_unit[256];
    if (*ws.overflow) return;
    fill_unit_table(s_unit);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cp.n_pixels; i += gridDim.x * blockDim.x) {
        const NodeMeta m = ws.meta[i];
        const Rgba c = node_color(ws, m, i, s_unit);
        const int local_row = cp.local_row0 + i / fp.width;
        const int orow = out_row_of_local(cp, local_row);
        const size_t opix = (size_t)orow * fp.width + i % fp.width;
        final_rgb8(c, !(m.flags & NODE_FINAL_RGB), out_rgb8 + opix * 3);
        if (COST) {
            const uint2 cost = (m.flags & NODE_FINAL_RGB) ? make_uint2(0u, 0u) : tree_cost(m, 0, fp.max_depth, aov.cost);
            if (aov.segments) aov.segments[opix] = cost.x;
            if (aov.levels) aov.levels[opix] = cost.y;
        }
    }
}
__global__ void __launch_bounds__(256) k_final(FrameParams fp, ChunkParams cp, Workspace ws, uint8_t* __restrict__ out_rgb8) {
    final_pixels<false>(fp, cp, ws, out_rgb8, AovPlanes{});
}
__global__ void __launch_bounds__(256) k_final_cost(FrameParams fp, ChunkParams cp, Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                    AovPlanes aov) {
    final_pixels<true>(fp, cp, ws, out_rgb8, aov);
}

// The primary-hit planes of one level-0 node (AovPlanes::depth / position / normal), narrowed once to float:
// t, o + d * t (the intersectors' expression) and normal_closer.  hit = false: the primary ray hit nothing or max_depth
// is 0 (depth +inf); traced = false: checkerboard pixel (everything NaN).
template <int D>
__device__ __forceinline__ void write_primary(const AovPlanes& aov, size_t opix, bool traced, bool hit, real t, const Vec<D>& p,
                                              const Vec<D>& n_closer) {
    const float nan = __int_as_float(0x7fc00000);
    const float depth = !traced ? nan : (hit ? (float)t : __int_as_float(0x7f800000));
    const bool finite = isfinite(depth);
    if (aov.depth) aov.depth[opix] = depth;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        if (aov.position) aov.position[opix * D + k] = finite ? (float)p[k] : nan;
        if (aov.normal) aov.normal[opix * D + k] = hit ? (float)n_closer[k] : nan;
    }
}

// K6 (AOVs only): the primary-hit planes from level 0 of the arena -- the ray record, ray_cur and the hit record, all still
// there when the chunk ends.  No hit record exists for max_depth 0, nor for checkerboard nodes (ray_cur -1: a camera in
// no entity, or an untraced frame of a batch).
template <int D>
__global__ void __launch_bounds__(256) k_aov_primary(FrameParams fp, ChunkParams cp, Workspace ws, AovPlanes aov) {
    if (*ws.overflow) return;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cp.n_pixels; i += gridDim.x * blockDim.x) {
        const bool traced = ws.ray_cur[i] >= 0;
        bool hit = false;
        real t = R(0.0);
        Vec<D> p, n;
#pragma unroll
        for (int k = 0; k < D; ++k) p[k] = n[k] = R(0.0);
        if (traced && fp.max_depth > 0) {
            const HitHead h = load_hit<D>(ws, i, n);
            if (h.entity >= 0) {
                Vec<D> o, d;
                load_ray<D>(ws, i, o, d);
                hit = true;
                t = h.t;
                p = o + d * h.t;
                if (h.exiting) n = -n;
            }
        }
        const int local_row = cp.local_row0 + i / fp.width;
        write_primary<D>(aov, (size_t)out_row_of_local(cp, local_row) * fp.width + i % fp.width, traced, hit, t, p, n);
    }
}

// ---------------------------------------------------------------------------------------------
// ray-tree export (eucl_render_trees, eucl_trace_ray_trees; DESIGN.md §5.3)

// Request slot of virtual-frame cell `item`, or -1 when the query does not name it: binary search of the sorted items.
__device__ __forceinline__ int tree_slot(const TreeQuery& tq, uint32_t item) {
    int lo = 0, hi = tq.n_items;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tq.items[mid] < item) lo = mid + 1;
        else hi = mid;
    }
    return lo < tq.n_items && tq.items[lo] == item ? (int)tq.slots[lo] : -1;
}

// One Universe::trace call of an item's tree as the wavefront arena and the megakernel walk both know it.
template <int D>
struct TreeRecord {
    int parent, level, kind, medium, hit;
    bool exiting, checkerboard;
    unsigned flags, q;
    real ratio, t;
    Vec<D> o, d, n_raw; // n_raw: the intersector's normal (normal_closer = exiting ? -n_raw : n_raw)
};

// EUCL_TREE_* flags of a node from its shading outcome: `last` = level max_depth, `hit` entity or -1, NODE_* flags,
// `has_t` = a transmitted child exists.
__device__ __forceinline__ unsigned tree_flags(bool last, int hit, real ratio, unsigned node_flags, bool has_t) {
    if (last || hit < 0) return EUCL_TREE_BACKGROUND;
    unsigned f = 0u;
    if (!(ratio >= R(1.0))) {
        f |= EUCL_TREE_SURFACE;
        if (node_flags & NODE_HAS_SC) f |= EUCL_TREE_OPAQUE;
        else if (!has_t) f |= EUCL_TREE_NO_DESTINATION;
    }
    if (node_flags & NODE_UNDEFINED) f |= EUCL_TREE_UNDEFINED;
    return f;
}

// Everything of a node but its colour, widened to double; components beyond D are 0.
template <int D>
__device__ __forceinline__ void tree_store(EuclTreeNode* out, const TreeRecord<D>& r) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll), inf = __longlong_as_double(0x7ff0000000000000ll);
    const bool hit = r.hit >= 0 && !r.checkerboard;
    out->parent = r.parent;
    out->level = r.level;
    out->kind = r.kind;
    out->medium = r.checkerboard ? -1 : r.medium;
    out->hit_entity = hit ? r.hit : -1;
    out->exiting = hit && r.exiting ? 1 : 0;
    out->flags = r.checkerboard ? EUCL_TREE_CHECKERBOARD : r.flags;
    out->surface_rgba8 = r.checkerboard ? 0u : r.q;
    out->ratio = r.checkerboard ? 0.0 : (double)r.ratio;
    out->t = r.checkerboard ? nan : (hit ? (double)r.t : inf);
#pragma unroll
    for (int k = 0; k < EUCL_MAX_DIM; ++k) {
        const int j = k < D ? k : 0;
        const real n = r.exiting ? -r.n_raw[j] : r.n_raw[j];
        out->origin[k] = k >= D ? 0.0 : (r.checkerboard ? nan : (double)r.o[j]);
        out->direction[k] = k >= D ? 0.0 : (r.checkerboard ? nan : (double)r.d[j]);
        out->normal[k] = k >= D ? 0.0 : (hit ? (double)n : nan);
    }
}
__device__ __forceinline__ void tree_store_color(EuclTreeNode* out, const Rgba& c) {
    out->color[0] = (double)c.r;
    out->color[1] = (double)c.g;
    out->color[2] = (double)c.b;
    out->color[3] = (double)c.a;
}

// K7 (tree calls only, after the resolve): the trees of the query's items that lie in this chunk, read from the arena, which
// still holds every level of the chunk.  One thread per item walks its tree depth-first over tchild / rchild with an
// explicit stack of at most max_depth + 1 entries (the reflected child is pushed first, so the transmitted subtree comes out
// first: pre-order).  Resolved colours are in `res` for every level but 0, whose colour k_final composes without storing it.
// Items of other chunks or of another pipeline's bands are skipped: their chunk writes them.
template <int D>
__global__ void __launch_bounds__(128) k_tree_export(FrameParams fp, ChunkParams cp, Workspace ws, TreeQuery tq) {
    __shared__ real s_unit[256];
    if (*ws.overflow) return; // the chunk is retried with a larger arena and exports then
    fill_unit_table(s_unit);
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= tq.n_items) return;
    const uint32_t item = tq.items[u];
    const int row = (int)(item / (uint32_t)fp.width), x = (int)(item % (uint32_t)fp.width);
    int local = row; // frame_row_of_local inverted: this pipeline's bands, then the chunk's local rows
    if (cp.band_world > 1) {
        const int band = row / cp.band_rows;
        if (band % cp.band_world != cp.band_rank) return;
        local = (band / cp.band_world) * cp.band_rows + row % cp.band_rows;
    }
    if (local < cp.local_row0 || local >= cp.local_row0 + cp.n_rows) return;
    EuclTreeNode* out = tq.nodes + (size_t)tq.slots[u] * tq.capacity;
    int st_node[EUCL_MAX_LEVELS], st_parent[EUCL_MAX_LEVELS], st_level_kind[EUCL_MAX_LEVELS];
    st_node[0] = (local - cp.local_row0) * fp.width + x;
    st_parent[0] = -1;
    st_level_kind[0] = EUCL_TREE_ROOT;
    int sp = 1;
    uint32_t count = 0;
    while (sp > 0) {
        --sp;
        const int node = st_node[sp], level = st_level_kind[sp] >> 2;
        const int idx = (int)count++;
        const NodeMeta m = ws.meta[node];
        if (idx < tq.capacity) {
            TreeRecord<D> r{};
            r.parent = st_parent[sp];
            r.level = level;
            r.kind = st_level_kind[sp] & 3;
            r.medium = ws.ray_cur[node];
            r.checkerboard = (m.flags & NODE_FINAL_RGB) != 0;
            r.hit = -1;
            r.ratio = m.ratio;
            r.q = m.q;
            if (!r.checkerboard) {
                load_ray<D>(ws, node, r.o, r.d);
                if (level < fp.max_depth) { // level max_depth: a background lookup, never intersected
                    const HitHead h = load_hit<D>(ws, node, r.n_raw);
                    r.hit = h.entity;
                    r.exiting = h.exiting != 0;
                    r.t = h.t;
                }
                r.flags = tree_flags(level >= fp.max_depth, r.hit, m.ratio, m.flags, m.tchild >= 0);
            }
            tree_store<D>(out + idx, r);
            tree_store_color(out + idx, level == 0 ? node_color(ws, m, node, s_unit) : load_res(ws, node));
        }
        const int children[2] = {m.rchild, m.tchild};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if (children[k] < 0 || sp >= EUCL_MAX_LEVELS) continue;
            st_node[sp] = children[k];
            st_parent[sp] = idx;
            st_level_kind[sp] = ((level + 1) << 2) | (k == 0 ? EUCL_TREE_REFLECTED : EUCL_TREE_TRANSMITTED);
            ++sp;
        }
    }
    tq.counts[tq.slots[u]] = count;
}

// Cross-check pipeline: one thread walks the whole ray tree of its pixel depth-first with an
// explicit stack (transmitted subtree first, then the reflected one, as the reference recurses).
constexpr int kMegaMaxDepth = 24;
template <int D>
struct MegaFrame {
    real ratio;
    unsigned q;
    unsigned state; // bit 0: waiting for the reflected child (else the transmitted one); bit 1: have T; bit 2: reflect pending
    Rgba t;
    ChildRay<D> r;
};

// AOV (k_megakernel_aov): also the AOV planes -- the level-0 geometry, and the segments and levels counted along the walk.
// The cross-check of k_aov_primary and the COST builds of the wavefront.
// RAYS (k_megakernel_rays*): the caller's rays of eucl_trace_rays* instead of a camera, addressed as in k_raygen_rays.
// TREE (k_megakernel_tree, k_megakernel_rays_tree): also records the walk of the query's items, node by node as it descends
// (pre-order) and each node's colour once it is known -- the cross-check of k_tree_export.
template <int D, bool AOV, bool RAYS, bool TREE = false>
__device__ __forceinline__ void megakernel_pixels(const uint8_t* __restrict__ blob, const FrameParams& fp, const ChunkParams& cp,
                                                  const Workspace& ws, uint8_t* __restrict__ out_rgb8,
                                                  int32_t* __restrict__ hit_ids_out, const AovPlanes& aov,
                                                  const double* __restrict__ origins, const double* __restrict__ directions,
                                                  const TreeQuery& tq = TreeQuery{}) {
    const SceneView& sv = stage_scene(blob);
    real* ts = plane_scratch(blob);
    const int cam_entity = *ws.cam_entity;
    unsigned long long local_counts[kMegaMaxDepth + 1];
    for (int l = 0; l <= kMegaMaxDepth; ++l) local_counts[l] = 0ull;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cp.n_pixels; i += gridDim.x * blockDim.x) {
        const int local_row = cp.local_row0 + i / fp.width;
        const int x = i % fp.width;
        int y = frame_row_of_local(cp, local_row);
        const size_t opix = (size_t)out_row_of_local(cp, local_row) * fp.width + x;
        const int slot = TREE ? tree_slot(tq, (uint32_t)y * (uint32_t)fp.width + (uint32_t)x) : -1;
        EuclTreeNode* const tree_out = TREE && slot >= 0 ? tq.nodes + (size_t)slot * tq.capacity : nullptr;
        int belongs_to = cam_entity, f = 0;
        Vec<D> ray_o, ray_d;
        if (RAYS) {
            const size_t ray = ((size_t)y * fp.width + x) * D;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                ray_o[k] = R(origins[ray + k]);
                ray_d[k] = R(directions[ray + k]);
            }
            belongs_to = material_at<D>(sv, ray_o);
        } else if (ws.frames) {
            f = frame_of_row(ws, y);
            belongs_to = ws.frame_entity[f];
        }
        if (belongs_to < 0) {
            if (TREE && tree_out) {
                TreeRecord<D> r{};
                r.parent = -1;
                r.checkerboard = true;
                tree_store<D>(tree_out, r);
                tree_store_color(tree_out, checkerboard(x, y));
                tq.counts[slot] = 1u;
            }
            final_rgb8(checkerboard(x, y), false, out_rgb8 + opix * 3);
            if (hit_ids_out) hit_ids_out[opix] = -2;
            local_counts[0]++;
            if (RAYS || ws.frames) atomicAdd(ws.untraced, 1);
            if (AOV) {
                const Vec<D> zero{};
                write_primary<D>(aov, opix, false, false, R(0.0), zero, zero);
                if (aov.segments) aov.segments[opix] = 0u;
                if (aov.levels) aov.levels[opix] = 0u;
            }
            continue;
        }
        unsigned aov_segments = 0u, aov_levels = 0u;
        MegaFrame<D> stack[kMegaMaxDepth];
        Vec<D> o, d;
        if (RAYS) {
            o = ray_o;
            d = ray_d;
        } else {
#pragma unroll
            for (int k = 0; k < D; ++k) o[k] = R(ws.frames ? ws.frames[f].location[k] : fp.location[k]);
            d = ws.frames ? camera_ray<D>(ws.frames[f], x, y) : camera_ray<D>(fp, x, y);
        }
        const real time_millis = R(!RAYS && ws.frames ? ws.frames[f].time_millis : fp.time_millis);
        material_enter<D>(sv, belongs_to, d);
        int cur = belongs_to, level = 0;
        Rgba val{R(0.0), R(0.0), R(0.0), R(0.0)};
        // TREE: pre-order index of the node open at each level, the kind of the node about to be evaluated, nodes so far
        int tree_idx[TREE ? kMegaMaxDepth + 1 : 1];
        int tree_kind = EUCL_TREE_ROOT;
        uint32_t tree_count = 0u;
        for (;;) {
            // ---- descend: evaluate the node for ray (o, d, cur) at `level`
            bool leaf = true;
            local_counts[level]++;
            int ent = -1;
            bool exiting = false;
            Vec<D> p, n;
            real cos_raw = R(0.0), angle_raw = R(0.0), t_hit = R(0.0);
            if (level < fp.max_depth) ent = intersect_ray<D>(sv, o, d, exiting, p, n, cos_raw, angle_raw, t_hit, ts, (int)blockDim.x);
            if (level == 0 && hit_ids_out) hit_ids_out[opix] = ent;
            if (AOV) {
                aov_segments += level < fp.max_depth ? 1u : 0u;
                aov_levels = max(aov_levels, (unsigned)level + 1u);
                if (level == 0) write_primary<D>(aov, opix, true, ent >= 0, t_hit, p, exiting ? -n : n);
            }
            // TREE: the node, but its colour, from what this step evaluated
            auto record = [&](real ratio, unsigned q, unsigned node_flags, bool has_t) {
                const int idx = (int)tree_count++;
                tree_idx[TREE ? level : 0] = idx;
                if (idx >= tq.capacity) return;
                TreeRecord<D> r{};
                r.parent = level > 0 ? tree_idx[TREE ? level - 1 : 0] : -1;
                r.level = level;
                r.kind = tree_kind;
                r.medium = cur;
                r.hit = ent;
                r.exiting = ent >= 0 && exiting;
                r.flags = tree_flags(level >= fp.max_depth, ent, ratio, node_flags, has_t);
                r.q = q;
                r.ratio = ratio;
                r.t = t_hit;
                r.o = o;
                r.d = d;
                if (ent >= 0) r.n_raw = n;
                tree_store<D>(tree_out + idx, r);
            };
            if (ent < 0) {
                if (TREE && tree_out) record(R(0.0), 0u, NODE_LEAF, false);
                val = mapped_color<D>(sv, sv.background, d);
            } else {
                ShadeOut<D> so;
                shade_hit<D, true>(sv, time_millis, d, cur, ent, exiting, cos_raw, angle_raw, p, n, so);
                if (TREE && tree_out) record(so.ratio, so.q, so.flags, so.t_emit);
                if (so.flags & NODE_UNDEFINED) {
                    val = Rgba{R(0.0), R(0.0), R(0.0), R(0.0)};
                    atomicAdd(ws.undefined_count, 1ull);
                } else if (!so.t_emit && !so.r_emit) {
                    val = so.sc; // opaque, no mirror
                } else {
                    MegaFrame<D>& f = stack[level];
                    f.ratio = so.ratio;
                    f.q = so.q;
                    f.state = 0u;
                    if (so.flags & NODE_HAS_SC) {
                        f.t = so.sc;
                        f.state |= 2u;
                    }
                    if (so.r_emit) {
                        f.r = so.r;
                        f.state |= 4u;
                    }
                    tree_kind = so.t_emit ? EUCL_TREE_TRANSMITTED : EUCL_TREE_REFLECTED;
                    if (so.t_emit) {
                        o = so.t.o;
                        d = so.t.d;
                        cur = so.t.cur;
                    } else {
                        f.state |= 1u;
                        o = so.r.o;
                        d = so.r.d;
                        cur = so.r.cur;
                    }
                    ++level;
                    leaf = false;
                }
            }
            if (!leaf) continue;
            // ---- ascend with `val` until a pending reflected child is found
            bool done = false;
            for (;;) {
                // `val` is the colour of the node open at `level`
                if (TREE && tree_out && tree_idx[TREE ? level : 0] < tq.capacity) tree_store_color(tree_out + tree_idx[TREE ? level : 0], val);
                if (level == 0) {
                    done = true;
                    break;
                }
                --level;
                MegaFrame<D>& f = stack[level];
                if (!(f.state & 1u)) { // the transmitted child returned
                    f.t = transmit_over(f.q, val);
                    f.state |= 2u;
                    if (f.state & 4u) {
                        f.state |= 1u;
                        tree_kind = EUCL_TREE_REFLECTED;
                        o = f.r.o;
                        d = f.r.d;
                        cur = f.r.cur;
                        ++level;
                        break;
                    }
                    val = f.t;
                } else { // the reflected child returned
                    val = (f.state & 2u) ? combine_palette_color(val, f.t, f.ratio) : val;
                }
            }
            if (done) break;
        }
        final_rgb8(val, true, out_rgb8 + opix * 3);
        if (AOV) {
            if (aov.segments) aov.segments[opix] = aov_segments;
            if (aov.levels) aov.levels[opix] = aov_levels;
        }
        if (TREE && tree_out) tq.counts[slot] = tree_count;
    }
    for (int l = 0; l <= fp.max_depth && l <= kMegaMaxDepth; ++l) {
        // per-level node counts, warp-reduced
        unsigned long long v = local_counts[l];
        for (int s = 16; s > 0; s >>= 1) v += __shfl_down_sync(0xffffffffu, v, s);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(ws.mega_level_counts + l, v);
    }
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                       Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                       int32_t* __restrict__ hit_ids_out) {
    megakernel_pixels<D, false, false>(blob, fp, cp, ws, out_rgb8, hit_ids_out, AovPlanes{}, nullptr, nullptr);
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel_aov(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                           Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                           int32_t* __restrict__ hit_ids_out, AovPlanes aov) {
    megakernel_pixels<D, true, false>(blob, fp, cp, ws, out_rgb8, hit_ids_out, aov, nullptr, nullptr);
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel_rays(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                            Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                            int32_t* __restrict__ hit_ids_out, const double* __restrict__ origins,
                                                            const double* __restrict__ directions) {
    megakernel_pixels<D, false, true>(blob, fp, cp, ws, out_rgb8, hit_ids_out, AovPlanes{}, origins, directions);
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel_rays_aov(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                                Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                                int32_t* __restrict__ hit_ids_out, AovPlanes aov,
                                                                const double* __restrict__ origins,
                                                                const double* __restrict__ directions) {
    megakernel_pixels<D, true, true>(blob, fp, cp, ws, out_rgb8, hit_ids_out, aov, origins, directions);
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel_tree(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                            Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                            int32_t* __restrict__ hit_ids_out, TreeQuery tq) {
    megakernel_pixels<D, false, false, true>(blob, fp, cp, ws, out_rgb8, hit_ids_out, AovPlanes{}, nullptr, nullptr, tq);
}
template <int D>
__global__ void __launch_bounds__(kBlock) k_megakernel_rays_tree(const uint8_t* __restrict__ blob, FrameParams fp, ChunkParams cp,
                                                                 Workspace ws, uint8_t* __restrict__ out_rgb8,
                                                                 int32_t* __restrict__ hit_ids_out, const double* __restrict__ origins,
                                                                 const double* __restrict__ directions, TreeQuery tq) {
    megakernel_pixels<D, false, true, true>(blob, fp, cp, ws, out_rgb8, hit_ids_out, AovPlanes{}, origins, directions, tq);
}

// Universe::trace_path_unknown / trace_path (mod.rs:186-227,273-286) with Surface::get_path
// (surface.rs:164-197): moves a point `distance` along a direction through the universe, crossing
// surfaces and applying the material transitions (a LinearSpace void stretches the step).  This is
// what the reference's cameras call before every frame; one thread, the recursion unrolled into a
// loop (the reference recurses once per crossed surface).
// out: [0..D) location, [D..2D) direction, out_found: 1 ok, 0 start point in no entity, -1 step limit
template <int D>
__global__ void __launch_bounds__(32) k_trace_path(const uint8_t* __restrict__ blob, const double* __restrict__ in,
                                                   double distance_in, double* __restrict__ out, int* __restrict__ out_found) {
    const SceneView& sv = stage_scene(blob);
    real* ts = plane_scratch(blob);
    if (threadIdx.x != 0) return;
    real distance = R(distance_in);
    Vec<D> loc, dir;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        loc[k] = R(in[k]);
        dir[k] = R(in[D + k]);
    }
    int belongs_to = material_at<D>(sv, loc);
    if (belongs_to < 0) {
        *out_found = 0;
        return;
    }
    material_enter<D>(sv, belongs_to, dir);
    int found = -1;
    for (int step = 0; step < 100000; ++step) {
        const ClosestHit h = closest_hit<D>(sv, loc, dir, ts, (int)blockDim.x);
        bool moved = false;
        if (h.entity >= 0 && !(distance - h.t <= R(0.0))) { // get_path: Some
            Vec<D> p, n_raw;
            hit_geometry<D>(sv, h.prim, h.flags, loc, dir, h.t, p, n_raw);
            const bool exiting = angle_from_cos(angle_cos(dir, n_raw)) < kFracPi2;
            const Vec<D> n_closer = exiting ? -n_raw : n_raw;
            const Vec<D> new_origin = p + (-n_closer) * kApproxEpsilon * R(128.0);
            const int dest = exiting ? material_at<D>(sv, new_origin) : h.entity;
            if (dest >= 0) {
                Vec<D> nd = dir;
                material_exit<D>(sv, belongs_to, nd);
                material_enter<D>(sv, dest, nd);
                distance = distance - h.t;
                belongs_to = dest;
                loc = new_origin;
                dir = nd;
                moved = true;
            }
        }
        if (!moved) { // Material::trace_path (material.rs:54-56,144-146), then exit
            loc = loc + dir * distance;
            material_exit<D>(sv, belongs_to, dir);
            found = 1;
            break;
        }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        out[k] = loc[k];
        out[D + k] = dir[k];
    }
    *out_found = found;
}

// The walk of k_trace_path above for one thread of a larger CTA (k_trace_paths): `ts` / `ts_stride` are the thread's
// plane_chain scratch column.  Returns 1 moved (loc, dir: the end point and the direction there), 0 the start lies in no
// entity (loc and dir untouched), -1 more than 100000 surface crossings (loc and dir: where the walk stopped).
// k_trace_path keeps a copy of its own, and this one is not inlined: k_trace_path's resources are pinned
// (tests/golden/kernel_resources.json), and with an inlined copy in k_trace_path, or in k_trace_paths, its 3-D f64 build
// grows from 4512 to 4528 bytes of stack (CUDA 12.9).
template <int D>
__device__ __noinline__ int walk_path(const SceneView& sv, Vec<D>& loc, Vec<D>& dir, real distance, real* ts, int ts_stride) {
    int belongs_to = material_at<D>(sv, loc);
    if (belongs_to < 0) return 0;
    material_enter<D>(sv, belongs_to, dir);
    for (int step = 0; step < 100000; ++step) {
        const ClosestHit h = closest_hit<D>(sv, loc, dir, ts, ts_stride);
        bool moved = false;
        if (h.entity >= 0 && !(distance - h.t <= R(0.0))) { // get_path: Some
            Vec<D> p, n_raw;
            hit_geometry<D>(sv, h.prim, h.flags, loc, dir, h.t, p, n_raw);
            const bool exiting = angle_from_cos(angle_cos(dir, n_raw)) < kFracPi2;
            const Vec<D> n_closer = exiting ? -n_raw : n_raw;
            const Vec<D> new_origin = p + (-n_closer) * kApproxEpsilon * R(128.0);
            const int dest = exiting ? material_at<D>(sv, new_origin) : h.entity;
            if (dest >= 0) {
                Vec<D> nd = dir;
                material_exit<D>(sv, belongs_to, nd);
                material_enter<D>(sv, dest, nd);
                distance = distance - h.t;
                belongs_to = dest;
                loc = new_origin;
                dir = nd;
                moved = true;
            }
        }
        if (!moved) { // Material::trace_path (material.rs:54-56,144-146), then exit
            loc = loc + dir * distance;
            material_exit<D>(sv, belongs_to, dir);
            return 1;
        }
    }
    return -1;
}

// eucl_trace_paths*: one walker per thread, `steps` walks each.  Step j starts where step j-1 ended (step 0 at the
// walker's location) and walks the walker's own distance along its own direction (the move_camera rule).  Outputs
// [n][steps]: status 1 the end point and direction; 0 the start (the walker stays: step 0 gives the location as given,
// not narrowed) and NaN, repeated by every later step; -1 NaN and NaN, and the walker stops (every later step is -1
// too).  out_dir may be null.
template <int D>
__global__ void __launch_bounds__(kBlock) k_trace_paths(const uint8_t* __restrict__ blob, const double* __restrict__ locations,
                                                        const double* __restrict__ directions,
                                                        const double* __restrict__ distances, uint32_t n, uint32_t steps,
                                                        double* __restrict__ out_loc, double* __restrict__ out_dir,
                                                        int32_t* __restrict__ out_status) {
    const SceneView& sv = stage_scene(blob);
    real* ts = plane_scratch(blob);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Vec<D> loc, dir0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        loc[k] = R(locations[(size_t)i * D + k]);
        dir0[k] = R(directions[(size_t)i * D + k]);
    }
    const real distance = R(distances[i]);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    int status = 1;
    bool moved = false;
    for (uint32_t j = 0; j < steps; ++j) {
        Vec<D> dir = dir0;
        if (status == 1) status = walk_path<D>(sv, loc, dir, distance, ts, (int)blockDim.x);
        moved = moved || status == 1;
        const size_t o = ((size_t)i * steps + j) * D;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            out_loc[o + k] = status < 0 ? nan : moved ? (double)loc[k] : locations[(size_t)i * D + k];
            if (out_dir) out_dir[o + k] = status == 1 ? (double)dir[k] : nan;
        }
        out_status[(size_t)i * steps + j] = status;
    }
}

// eucl_locate_points*: Universe::material_at of each point (narrowed once), -1 in no entity.  Grid-stride over the points.
template <int D>
__global__ void __launch_bounds__(kBlock) k_locate(const uint8_t* __restrict__ blob, const double* __restrict__ points, uint32_t n,
                                                   int32_t* __restrict__ out) {
    const SceneView& sv = stage_scene(blob);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        Vec<D> p;
#pragma unroll
        for (int k = 0; k < D; ++k) p[k] = R(points[(size_t)i * D + k]);
        out[i] = material_at<D>(sv, p);
    }
}

#if EUCL_REAL_IS_DOUBLE
// BEGIN_KEEP64
// FP64 issue-rate microbenchmark: 8 independent dependency chains per thread
template <int OP>
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0, a6 = a0 + 6.0,
           a7 = a0 + 7.0;
    const double m = 1.0000000001, c = 1.0e-9;
    for (int i = 0; i < iters; ++i) {
        if (OP == 0) {
            a0 = __dadd_rn(a0, c); a1 = __dadd_rn(a1, c); a2 = __dadd_rn(a2, c); a3 = __dadd_rn(a3, c);
            a4 = __dadd_rn(a4, c); a5 = __dadd_rn(a5, c); a6 = __dadd_rn(a6, c); a7 = __dadd_rn(a7, c);
        } else if (OP == 1) {
            a0 = __dmul_rn(a0, m); a1 = __dmul_rn(a1, m); a2 = __dmul_rn(a2, m); a3 = __dmul_rn(a3, m);
            a4 = __dmul_rn(a4, m); a5 = __dmul_rn(a5, m); a6 = __dmul_rn(a6, m); a7 = __dmul_rn(a7, m);
        } else {
            a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
            a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

// END_KEEP64
#endif
inline int grid_for(int n, int block, int grid_max) {
    long long g = ((long long)n + block - 1) / block;
    if (g < 1) g = 1;
    if (g > grid_max) g = grid_max;
    return (int)g;
}

// The light and the heavy build of a level's kernel, each when wanted; returns the number launched.  When both run and
// there is a side stream, the light one runs there: it waits for everything enqueued on the main stream so far (fork), and
// the main stream waits for it (join).
template <typename LaunchLight, typename LaunchHeavy>
int launch_light_and_heavy(const Launch& l, bool light, bool heavy, LaunchLight launch_light, LaunchHeavy launch_heavy) {
    const bool fork = light && heavy && l.side != nullptr;
    if (fork) {
        cudaEventRecord(l.ev_fork, l.stream);
        cudaStreamWaitEvent(l.side, l.ev_fork, 0);
    }
    if (light) launch_light(fork ? l.side : l.stream);
    if (heavy) launch_heavy();
    if (fork) {
        cudaEventRecord(l.ev_join, l.side);
        cudaStreamWaitEvent(l.stream, l.ev_join, 0);
    }
    return (int)light + (int)heavy;
}

// The builds of k_shade by [GLASS][RAY_BINS][FRAMES]
template <int D>
auto shade_build(bool glass, bool ray_bins, bool frames) {
    static const decltype(&k_shade<D, false, false, false>) builds[2][2][2] = {
        {{k_shade<D, false, false, false>, k_shade<D, false, false, true>}, {k_shade<D, true, false, false>, k_shade<D, true, false, true>}},
        {{k_shade<D, false, true, false>, k_shade<D, false, true, true>}, {k_shade<D, true, true, false>, k_shade<D, true, true, true>}}};
    return builds[glass][ray_bins][frames];
}
// ... and of k_shade_glass by [RAY_BINS][FRAMES]
template <int D>
auto shade_glass_build(bool ray_bins, bool frames) {
    static const decltype(&k_shade_glass<D, false, false>) builds[2][2] = {
        {k_shade_glass<D, false, false>, k_shade_glass<D, false, true>}, {k_shade_glass<D, true, false>, k_shade_glass<D, true, true>}};
    return builds[ray_bins][frames];
}

template <int D>
void launch_camera_entity(const Launch& l, const FrameParams& fp, const Workspace& ws) {
    k_camera_entity<D><<<1, 32, l.smem_scene, l.stream>>>(l.blob, fp, ws);
}
template <int D>
void launch_raygen(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, int32_t* hit_ids_out,
                   const double* origins, const double* directions) {
    const int grid = grid_for(cp.n_pixels, kBlock, l.grid_mem);
    if (origins) k_raygen_rays<D><<<grid, kBlock, l.smem_scene, l.stream>>>(l.blob, fp, cp, ws, hit_ids_out, origins, directions);
    else k_raygen<D><<<grid, kBlock, l.smem_scene, l.stream>>>(l.blob, fp, cp, ws, hit_ids_out);
}

template <int D>
int launch_intersect(const Launch& l, const Workspace& ws, int level) {
    // grouped level of a light-capable scene: key 0 -> light build, the other keys -> heavy build;
    // a light-capable scene without cull roots (every ray has key 0) runs the light build in node order
    const bool light_all = l.light_capable && l.n_cull == 0;
    const bool split = l.light_capable && ws.ray_bins != 0;
    // a csg2-capable scene walks the heavy build's rays, grouped or not, with k_intersect_csg2
    const size_t smem_light = l.smem_scene + sizeof(real) * kPlaneChainMax * kLightK2Block;
    const size_t smem_csg2 = l.smem_scene + sizeof(real) * kPlaneChainMax * kCsg2Block;
    const unsigned heavy_mask = split ? 0xfffeu : 0xffffu;
    return launch_light_and_heavy(
        l, light_all || split, !light_all,
        [&](cudaStream_t stream) { k_intersect<D, true><<<l.grid_light_k2, kLightK2Block, smem_light, stream>>>(l.blob, ws, level, 1u); },
        [&] {
            if (l.csg2_capable) k_intersect_csg2<D><<<l.grid_csg2, kCsg2Block, smem_csg2, l.stream>>>(l.blob, ws, level, heavy_mask);
            else k_intersect<D, false><<<l.grid_max, kBlock, l.smem_bytes, l.stream>>>(l.blob, ws, level, heavy_mask);
        });
}

template <int D>
int launch_shade(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, int level,
                 int32_t* hit_ids_out) {
    if (level >= fp.max_depth) { // last level: background lookups only
        k_background<D><<<l.grid_background, 256, l.smem_scene, l.stream>>>(l.blob, fp, cp, ws, level, hit_ids_out);
        return 1;
    }
    unsigned long long light = l.shade_light_mask, glass = l.shade_glass_mask, heavy = l.shade_heavy_mask;
    if (ws.n_bins <= 1) { // not binned: one kernel that can shade everything
        light = 0ull;
        glass = 0ull;
        heavy = ~0ull;
    }
    const bool ray_bins = ws.ray_bins && level + 1 < fp.max_depth; // the next level will be intersected: group its rays
    const bool frames = ws.node_frame != nullptr;
    // k_shade_glass and the heavy build both run on the main stream, one after the other, when a level needs both
    return (glass != 0ull && heavy != 0ull) + launch_light_and_heavy(
        l, light != 0ull, (glass | heavy) != 0ull,
        [&](cudaStream_t stream) {
            shade_build<D>(false, ray_bins, frames)<<<l.grid_light, kLightBlock, l.smem_scene, stream>>>(l.blob, fp, cp, ws, level,
                                                                                                       light, hit_ids_out);
        },
        [&] {
            if (glass)
                shade_glass_build<D>(ray_bins, frames)<<<l.grid_shade_glass[ray_bins], kShadeGlassBlock, l.smem_scene, l.stream>>>(
                    l.blob, fp, cp, ws, level, glass, hit_ids_out);
            if (heavy)
                shade_build<D>(true, ray_bins, frames)<<<l.grid_shade, kShadeBlock, l.smem_scene, l.stream>>>(l.blob, fp, cp, ws, level,
                                                                                                           heavy, hit_ids_out);
        });
}

// Bottom-up resolve of the ray tree (level max_depth holds leaves only) and the RGB8 pack of level 0.
// With AOVs: the COST builds when segments or levels are wanted, and k_aov_primary for the primary-hit planes.
template <int D>
int launch_resolve_and_final(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, uint8_t* out_rgb8,
                             const AovPlanes& aov) {
    const bool cost = aov.segments || aov.levels;
    int launches = 0;
    for (int level = fp.max_depth - 1; level >= 1; --level) {
        if (cost) k_resolve_cost<<<l.grid_mem, 256, 0, l.stream>>>(ws, level, fp.max_depth, aov);
        else k_resolve<<<l.grid_mem, 256, 0, l.stream>>>(ws, level);
        ++launches;
    }
    const int grid = grid_for(cp.n_pixels, 256, l.grid_mem);
    if (cost) k_final_cost<<<grid, 256, 0, l.stream>>>(fp, cp, ws, out_rgb8, aov);
    else k_final<<<grid, 256, 0, l.stream>>>(fp, cp, ws, out_rgb8);
    ++launches;
    if (aov.depth || aov.position || aov.normal) {
        k_aov_primary<D><<<grid, 256, 0, l.stream>>>(fp, cp, ws, aov);
        ++launches;
    }
    return launches;
}

// The build of the megakernel: a tree call records the walk (and writes no AOV plane), else AOVs if any plane is wanted;
// each with or without the caller's rays.
template <int D>
void launch_megakernel(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, uint8_t* out_rgb8,
                       int32_t* hit_ids_out, const AovPlanes& aov, const double* origins, const double* directions,
                       const TreeQuery& tree) {
    const int grid = grid_for(cp.n_pixels, kBlock, 1 << 30);
    const auto launch = [&](auto kernel, auto... extra) {
        kernel<<<grid, kBlock, l.smem_bytes, l.stream>>>(l.blob, fp, cp, ws, out_rgb8, hit_ids_out, extra...);
    };
    const bool want_aov = aov.depth || aov.position || aov.normal || aov.segments || aov.levels;
    if (tree.n_items && origins) launch(k_megakernel_rays_tree<D>, origins, directions, tree);
    else if (tree.n_items) launch(k_megakernel_tree<D>, tree);
    else if (origins && want_aov) launch(k_megakernel_rays_aov<D>, aov, origins, directions);
    else if (origins) launch(k_megakernel_rays<D>, origins, directions);
    else if (want_aov) launch(k_megakernel_aov<D>, aov);
    else launch(k_megakernel<D>);
}

// The trees of the query's items in this chunk (after launch_resolve_and_final, while the arena is intact).
template <int D>
int launch_tree_export(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, const TreeQuery& tree) {
    k_tree_export<D><<<grid_for(tree.n_items, 128, 1 << 30), 128, 0, l.stream>>>(fp, cp, ws, tree);
    return 1;
}

template <int D>
void launch_trace_path(const Launch& l, const double* d_in, double distance, double* d_out, int* d_found) {
    k_trace_path<D><<<1, 32, l.smem_bytes, l.stream>>>(l.blob, d_in, distance, d_out, d_found);
}

template <int D>
void launch_trace_paths(const Launch& l, const double* d_locations, const double* d_directions, const double* d_distances,
                        uint32_t n, uint32_t steps, double* d_out_locations, double* d_out_directions, int32_t* d_out_status) {
    k_trace_paths<D><<<grid_for((int)n, kBlock, 1 << 30), kBlock, l.smem_bytes, l.stream>>>(
        l.blob, d_locations, d_directions, d_distances, n, steps, d_out_locations, d_out_directions, d_out_status);
}

template <int D>
void launch_locate(const Launch& l, const double* d_points, uint32_t n, int32_t* d_out) {
    k_locate<D><<<grid_for((int)n, kBlock, l.grid_mem), kBlock, l.smem_scene, l.stream>>>(l.blob, d_points, n, d_out);
}

template <int D>
const Kernels kKernels{launch_camera_entity<D>, launch_raygen<D>,      launch_intersect<D>,   launch_shade<D>,
                       launch_resolve_and_final<D>, launch_megakernel<D>, launch_tree_export<D>, launch_trace_path<D>,
                       launch_trace_paths<D>,   launch_locate<D>};

template <typename K>
cudaError_t configure_one(K kernel, size_t smem, int resident_ctas) {
    // Shared-memory carveout: just what the kernel's resident CTAs need, the rest of the 256 KB stays L1 for
    // local memory (CSG hit lists, spills).  Measured on 3d_room: 19.6 ms with the driver's default split,
    // 19.3 ms at 25 %, 21.3 ms at 100 %.  A hint only; EUCL_CARVEOUT (percent) overrides.
    int dev = 0, max_smem_sm = 228 * 1024;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    const size_t need = (size_t)resident_ctas * (smem + 2048);
    int pct = (int)((need * 100 + (size_t)max_smem_sm - 1) / (size_t)max_smem_sm);
    if (const char* c = getenv("EUCL_CARVEOUT")) pct = atoi(c);
    pct = pct < 0 ? 0 : (pct > 100 ? 100 : pct);
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    if (smem <= 48 * 1024) return cudaSuccess;
    // The limit belongs to the kernel, not to the scene, and is shared by every scene of the process: it only ever
    // grows, so that a scene created later with smaller tables cannot fail the launches of a larger one.
    cudaFuncAttributes attr{};
    cudaError_t e = cudaFuncGetAttributes(&attr, kernel);
    if (e != cudaSuccess || (size_t)attr.maxDynamicSharedSizeBytes >= smem) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

template <int D>
cudaError_t configure_dim(size_t smem_bytes, size_t smem_scene) {
    cudaError_t e = cudaSuccess;
    const auto conf = [&](auto kernel, size_t smem, int resident_ctas) {
        if (e == cudaSuccess) e = configure_one(kernel, smem, resident_ctas);
    };
    const int heavy = kResidentThreads / kBlock;
    conf(k_camera_entity<D>, smem_scene, 1);
    conf(k_raygen<D>, smem_scene, 2);
    conf(k_raygen_rays<D>, smem_scene, 2);
    conf(k_intersect<D, false>, smem_bytes, heavy);
    conf(k_intersect<D, true>, smem_scene + sizeof(real) * kPlaneChainMax * kLightK2Block, EUCL_INTERSECT_LIGHT_MIN_BLOCKS);
    conf(k_intersect_csg2<D>, smem_scene + sizeof(real) * kPlaneChainMax * kCsg2Block, csg2_resident_blocks(D, (int)sizeof(real)));
    for (int b = 0; b < 8; ++b) // [GLASS][RAY_BINS][FRAMES]
        conf(shade_build<D>(b & 4, b & 2, b & 1), smem_scene, (b & 4) ? kShadeResidentBlocks : kLightResidentBlocks);
    for (int b = 0; b < 4; ++b) // [RAY_BINS][FRAMES]
        conf(shade_glass_build<D>(b & 2, b & 1), smem_scene, shade_glass_resident_blocks(b & 2, (int)sizeof(real)));
    conf(k_background<D>, smem_scene, EUCL_BACKGROUND_MIN_BLOCKS);
    conf(k_megakernel<D>, smem_bytes, heavy);
    conf(k_megakernel_aov<D>, smem_bytes, heavy);
    conf(k_megakernel_rays<D>, smem_bytes, heavy);
    conf(k_megakernel_rays_aov<D>, smem_bytes, heavy);
    conf(k_megakernel_tree<D>, smem_bytes, heavy);
    conf(k_megakernel_rays_tree<D>, smem_bytes, heavy);
    conf(k_trace_path<D>, smem_bytes, 1);
    conf(k_trace_paths<D>, smem_bytes, heavy);
    conf(k_locate<D>, smem_scene, 2);
    return e;
}

} // namespace

const Kernels& kernels(int dim) { return dim == 3 ? kKernels<3> : kKernels<4>; }

cudaError_t configure_kernels(size_t smem_bytes, size_t smem_scene) {
    const cudaError_t e = configure_dim<3>(smem_bytes, smem_scene);
    return e != cudaSuccess ? e : configure_dim<4>(smem_bytes, smem_scene);
}

#if EUCL_REAL_IS_DOUBLE
// BEGIN_KEEP64
int fp64_peak(double* dadd, double* dmul, double* dfma) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 8, threads = 256, iters = 1 << 16;
    double* buf = nullptr;
    if (cudaMalloc(&buf, sizeof(double) * blocks * threads) != cudaSuccess) return -1;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double* outs[3] = {dadd, dmul, dfma};
    for (int op = 0; op < 3; ++op) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            cudaEventRecord(e0);
            if (op == 0) k_fp64_peak<0><<<blocks, threads>>>(buf, iters, 1.0);
            else if (op == 1) k_fp64_peak<1><<<blocks, threads>>>(buf, iters, 1.0);
            else k_fp64_peak<2><<<blocks, threads>>>(buf, iters, 1.0);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0 && ms < best) best = ms;
        }
        const double ops = (double)blocks * threads * (double)iters * 8.0;
        *outs[op] = ops / (best * 1e-3) / 1e12;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(buf);
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// END_KEEP64
#endif

} // namespace EUCL_NS
