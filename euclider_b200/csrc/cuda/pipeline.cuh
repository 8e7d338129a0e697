// Shared declarations of the wavefront pipeline: frame constants, the node arena and the launch
// interface between api_device.cu (host orchestration) and kernels.cu (device code).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "euclider_b200.h"

namespace eucl {

// Per-frame constants.  The camera terms that need libm (tan, sqrt) are computed once on the
// host in the reference's order (d3/entity/camera.rs:164-185, d4/entity/camera.rs:155-176);
// the per-pixel part uses only IEEE add/mul/div/sqrt and is bit-reproducible on the device.
struct FrameParams {
    double location[EUCL_MAX_DIM];
    double center[EUCL_MAX_DIM]; // location + forward * distance_from_screen_center
    double up[EUCL_MAX_DIM];
    double right[EUCL_MAX_DIM];
    double time_millis; // (time * 1000).as_secs() / 1000.0
    int32_t width, height;
    int32_t max_depth;
    int32_t _pad;
};

// Which rows of the frame one launch sequence covers.  A rank owns the bands b with
// b % band_world == band_rank (band = band_rows consecutive rows); its rows are numbered
// consecutively ("local rows") and processed in chunks of whole local rows.
struct ChunkParams {
    int32_t local_row0;  // first local row of this chunk
    int32_t n_rows;      // rows in this chunk
    int32_t band_rows, band_rank, band_world;
    int32_t compact_rows; // 1: output row index = local row; 0: output row index = frame row
    int32_t n_pixels;     // n_rows * width
    // one of `sub_stride` pipelines sharing a rank's bands (api_device.cu: render_split): band_rank / band_world above
    // already name this pipeline's bands in the frame; in the rank's COMPACT buffer its band i is band i * stride + offset
    int32_t sub_stride, sub_offset;
    int32_t _pad;
};

__host__ __device__ inline int frame_row_of_local(const ChunkParams& c, int local_row) {
    if (c.band_world <= 1) return local_row;
    int k = local_row / c.band_rows;
    return (k * c.band_world + c.band_rank) * c.band_rows + local_row % c.band_rows;
}

// row of the output buffer a local row is written to
__host__ __device__ inline int out_row_of_local(const ChunkParams& c, int local_row) {
    if (!c.compact_rows) return frame_row_of_local(c, local_row);
    if (c.sub_stride <= 1) return local_row;
    return ((local_row / c.band_rows) * c.sub_stride + c.sub_offset) * c.band_rows + local_row % c.band_rows;
}

// What the intersect kernel reports about a ray, one array-of-structures record of kHitDoubles doubles per node:
//   [0] t          parametric distance of the winning hit (the ray direction is not necessarily unit)
//   [1] cos_raw    dot(d, n) / (|d| |n|) for the intersector's normal: shading derives its angles from it
//   [2] (entity, exiting) as two int32: hit entity or -1; angle_between(direction, normal) < pi/2 (mod.rs:117)
//   [3] angle_raw  angle_between(direction, normal) = acos(cos_raw), NaN -> 0: evaluated here for `exiting`, reused by the
//                  illumination / Fresnel / Snell providers whenever they ask for the angle of this same cosine
//   [4 .. 4 + D)   the intersector's normal
// The hit location is not stored: o + d * t from the ray record is the intersectors' own expression for it.
// 64 bytes (3-D: one pad double): four 128-bit words, two whole DRAM sectors per gathered node.
constexpr int kHitReals = 8;
// reals per ray record: [origin, direction], padded to whole 16-byte words (f32, 3-D: 6 -> 8)
__host__ __device__ constexpr int ray_reals(int dim, int real_bytes) { return real_bytes == 8 ? 2 * dim : 8; }

// Ray-tree node record written by the shade kernel and consumed by the bottom-up resolve.
struct NodeMeta {
    double ratio;    // clamped reflection ratio
    int32_t tchild;  // node id of the transmitted child, -1 if none
    int32_t rchild;  // node id of the reflected child, -1 if none
    uint32_t q;      // surface colour quantised to u8x4 (surface.rs:72), r | g<<8 | b<<16 | a<<24
    uint32_t flags;
};
enum : uint32_t {
    NODE_LEAF = 1u,      // `res` already holds the final colour of the node
    NODE_HAS_SC = 2u,    // `res` holds the opaque surface colour (alpha quantises to 255): no transmitted child
    NODE_FINAL_RGB = 4u, // level-0 checkerboard pixel: `res` is written out without compositing
    NODE_UNDEFINED = 8u  // both branches None (the reference would panic): transparent black
};

// Node arena shared by all levels of one chunk: level l occupies node ids
// [level_off[l], level_off[l] + count[l]).  Rays, hits, metadata and resolved colours are all
// indexed by node id.  Every record is an array-of-structures entry made of whole 16-byte words
// (128-bit accesses) that starts on a 16-byte boundary: the kernels reach most records through index
// lists (bins), and a gathered node then costs 2 + 1 + 1 DRAM sectors (ray, hit, current entity)
// where per-component planes cost one half-used sector per plane.
struct Workspace {
    int32_t capacity;   // nodes
    int32_t list_cap;   // entries per index list = the largest level the lists can hold
    void* ray;          // [capacity][ray_reals] reals (f64 or f32 build): origin, direction
    int32_t* ray_cur;   // entity the ray travels in; -1 = no ray (checkerboard pixel)
    void* hit;          // [capacity][kHitReals] reals
    NodeMeta* meta;
    void* res;          // [capacity][4] reals: resolved colour r, g, b, a
    int32_t* count;     // [EUCL_MAX_LEVELS + 1] nodes per level
    int32_t* level_off; // [EUCL_MAX_LEVELS + 1] first node id of each level
    int32_t* overflow;  // 1: a child could not be appended (arena); 3: a level outgrew the index lists; 2: internal error
    int32_t* cam_entity; // material_at(camera location), -1 if none; a batch: -1 when no frame's camera is in an entity
    int32_t n_bins;      // 1: shade in node order; else kBinsPerEntity * n_entities + 1 bins keyed by (hit entity, class), 0 = miss
    int32_t frame_rows;  // a batch of frames (frames != nullptr): rows per frame of the virtual frame
    int32_t* bin_count;  // [EUCL_MAX_LEVELS + 1][kMaxBins] nodes per (level, hit-entity bin)
    int32_t* order;      // [n_bins][list_cap] node ids of the current level grouped by bin (reused per level)
    int32_t ray_bins;    // 1: the rays of a level are walked grouped by reach key (see SceneHeader::cull_root)
    int32_t n_frames;    // frames of a batch (1: a single frame)
    int32_t* rbin_count; // [EUCL_MAX_LEVELS + 1][kRayBins]
    int32_t* rorder;     // [kRayBins][list_cap] node ids of the NEXT level grouped by reach key
    unsigned long long* undefined_count;   // nodes that touched a corner the reference leaves undefined
    unsigned long long* mega_level_counts; // [EUCL_MAX_LEVELS + 1] nodes per level, megakernel pipeline only
    // A batch of frames rendered as ONE virtual frame of n_frames * frame_rows rows: virtual row r is row r % frame_rows
    // of frame r / frame_rows.  All four are null for a single frame, which reads FrameParams / cam_entity instead.
    const FrameParams* frames; // [n_frames] per-frame constants (pose, time)
    int32_t* frame_entity;     // [n_frames] material_at(camera location of the frame), -1 if none
    int32_t* node_frame;       // [capacity] frame of every node (Perlin time): level 0 by k_raygen, children by k_shade
    int32_t* untraced;         // level-0 nodes of this chunk whose frame's camera (eucl_trace_rays*: whose ray's origin) is in
                               // no entity (checkerboard pixels); also carved for ray calls, which have no frame table
};

// Per-pixel auxiliary outputs of the primary ray and its tree (eucl_render_aovs*, definitions in DESIGN.md §6): device planes
// addressed like the hit ids (out_row_of_local), each null when not wanted.  The kernels that write them are builds of
// their own (k_aov_primary, k_resolve_cost, k_final_cost, k_megakernel_aov): a render without AOVs runs none of this code.
struct AovPlanes {
    float* depth;       // [pixels] parametric distance t of the primary hit
    float* position;    // [pixels][dim] o + d * t
    float* normal;      // [pixels][dim] normal_closer of the primary hit
    uint32_t* segments; // [pixels] Universe::trace calls with depth > 0 in the pixel's ray tree
    uint32_t* levels;   // [pixels] deepest level of the tree + 1
    // [capacity] (segments, levels) of every node of the chunk, filled bottom-up by k_resolve_cost; the pipeline's own
    // buffer, set (wavefront only) when segments or levels are wanted
    uint2* cost;
};

// Ray-tree export of a tree call (eucl_render_trees, eucl_trace_ray_trees; DESIGN.md §5.3): the device view of the query.
// The distinct items, sorted, each with the first request slot that names it; the host copies that slot's tree to the
// slots of its duplicates.  n_items == 0: no tree call (k_tree_export and the TREE megakernels are builds of their own).
struct TreeQuery {
    const uint32_t* items; // [n_items] distinct virtual-frame cells, ascending
    const uint32_t* slots; // [n_items] request slot of each
    int32_t n_items;
    int32_t capacity;      // nodes kept per slot
    EuclTreeNode* nodes;   // [request slots][capacity]
    uint32_t* counts;      // [request slots] nodes of the whole tree
};

struct Launch {
    cudaStream_t stream;
    const uint8_t* blob;
    size_t smem_bytes; // staged scene + the per-thread plane_chain scratch of a kBlock-thread CTA (k_intersect, k_megakernel, k_trace_path*)
    size_t smem_scene; // staged scene only (the other kernels)
    int grid_max;   // blocks of the heavy queue kernels (k_intersect, k_shade<GLASS>): resident CTAs per SM x SMs, one wave
    int grid_light; // blocks of the light shade kernel (kLightBlock threads each), one wave
    int grid_shade; // blocks of the heavy shade kernel (kShadeBlock threads each), one wave
    int grid_mem;   // blocks of the memory-bound kernels (k_raygen, k_resolve, k_final, 256 threads each)
    unsigned long long shade_light_mask, shade_heavy_mask; // shade bins of the light / heavy build of k_shade
    int grid_light_k2;  // blocks of the light intersect kernel, one wave
    int light_capable;  // SceneHeader::light_capable
    int n_cull;         // SceneHeader::n_cull
    // The light and the heavy build of a level's kernel do not depend on each other: with a side stream they run
    // concurrently (fork / join through the two events), so the tail of one overlaps the body of the other.
    cudaStream_t side;  // nullptr: launch one after the other on `stream`
    cudaEvent_t ev_fork, ev_join;
    int grid_background; // blocks of the last level's kernel (256 threads each), one wave
    int grid_csg2;       // blocks of k_intersect_csg2 (kCsg2Block threads each), one wave
    int csg2_capable;    // SceneHeader::csg2_capable: k_intersect_csg2 replaces the heavy intersect build
    unsigned long long shade_glass_mask; // shade bins of k_shade_glass (Fresnel / Snell surfaces of one constant colour)
    int grid_shade_glass[2];             // blocks of k_shade_glass by RAY_BINS (kShadeGlassBlock threads each), one wave
};

#ifndef EUCL_BLOCK
#define EUCL_BLOCK 512 /* measured on 3d_room 4K: 64 -> 20.1 ms, 128 -> 20.0, 256 -> 19.5, 512 -> 19.1 (one wave each) */
#endif
constexpr int kBlock = EUCL_BLOCK;          // threads per CTA of the scene-walking kernels
constexpr int kResidentThreads = 512;       // per SM at 128 registers per thread (k_intersect, k_shade)
#ifndef EUCL_LIGHT_BLOCK
#define EUCL_LIGHT_BLOCK 256
#endif
#ifndef EUCL_BACKGROUND_MIN_BLOCKS
#define EUCL_BACKGROUND_MIN_BLOCKS 3 /* resident 256-thread CTAs per SM of k_background */
#endif
#ifndef EUCL_SHADE_LIGHT_MIN_BLOCKS
#define EUCL_SHADE_LIGHT_MIN_BLOCKS 2 /* 3d_room 4K, shade ms per frame: 3 CTAs of 256 (80 registers, 370 B of spills) 8.50; 5 of 128 (96) 8.03; 4 of 128 / 2 of 256 (128 registers, no spills) 7.29 / 7.16 */
#endif
#ifndef EUCL_SHADE_BLOCK
#define EUCL_SHADE_BLOCK EUCL_BLOCK
#endif
#ifndef EUCL_SHADE_MIN_BLOCKS
#define EUCL_SHADE_MIN_BLOCKS (512 / EUCL_SHADE_BLOCK > 0 ? 512 / EUCL_SHADE_BLOCK : 1)
#endif
constexpr int kShadeBlock = EUCL_SHADE_BLOCK; // threads per CTA of the heavy shade kernel
constexpr int kShadeResidentBlocks = EUCL_SHADE_MIN_BLOCKS;
constexpr int kLightBlock = EUCL_LIGHT_BLOCK; // threads per CTA of the light shade kernel
constexpr int kLightResidentBlocks = EUCL_SHADE_LIGHT_MIN_BLOCKS; // ... and CTAs per SM its register budget allows
#ifndef EUCL_SHADE_GLASS_BLOCK
#define EUCL_SHADE_GLASS_BLOCK 128
#endif
constexpr int kShadeGlassBlock = EUCL_SHADE_GLASS_BLOCK; // threads per CTA of k_shade_glass
// ... and CTAs per SM, by build.  Every setting below 128 registers spills.  The RAY_BINS builds (levels walked grouped by
// reach key) wait on reach_key's bound tests and the key-list atomics, and more resident warps pay for the spills: f64 6
// CTAs (80 registers), f32 5 (96).  The other builds spend their time in the shading arithmetic and keep 128 registers:
// 4 CTAs.  One B200 at 1000 W, ms per frame: 3d_room 4K (grouped) f64 at 4 / 5 / 6 / 7 CTAs 13.31 - 13.33 / 13.21 - 13.26
// / 13.12 - 13.13 / 13.17 - 13.19, f32 at 4 / 5 / 6 11.34 - 11.35 / 11.28 - 11.29 / 11.35 - 11.37; 3d_fresnel 1080p
// (ungrouped) f64 at 4 / 5 1.65 / 1.74 (parent 1.73).
constexpr int shade_glass_resident_blocks(bool ray_bins, int real_bytes) { return !ray_bins ? 4 : real_bytes == 8 ? 6 : 5; }
#ifndef EUCL_LIGHT_K2_BLOCK
#define EUCL_LIGHT_K2_BLOCK 128
#endif
#ifndef EUCL_INTERSECT_LIGHT_MIN_BLOCKS
#define EUCL_INTERSECT_LIGHT_MIN_BLOCKS 5 /* 640 threads per SM at 95 registers, no spills */
#endif
constexpr int kLightK2Block = EUCL_LIGHT_K2_BLOCK; // threads per CTA of the light intersect kernel
constexpr int kLightK2ResidentBlocks = EUCL_INTERSECT_LIGHT_MIN_BLOCKS;
#ifndef EUCL_CSG2_BLOCK
#define EUCL_CSG2_BLOCK 128
#endif
constexpr int kCsg2Block = EUCL_CSG2_BLOCK; // threads per CTA of k_intersect_csg2
// ... and CTAs per SM its register budget allows: 5 (<= 96 registers, no spills) except 4-D f64, which spills 140 B at
// 96 registers and runs at 4 (128).  3d_room 4K, one B200 at 1000 W, one call: 13.62 ms per frame at 5 CTAs, 13.81 at 4.
constexpr int csg2_resident_blocks(int dim, int real_bytes) { return dim == 4 && real_bytes == 8 ? 4 : 5; }
constexpr int kRayBins = 16; // 2^4 reach keys
constexpr int kBinsPerEntity = 3; // entering, exiting, exiting with total internal reflection predicted
constexpr int kMaxBins = 64; // shade-coherence bins (miss, then kBinsPerEntity per entity); larger scenes shade unbinned

// The launchers of one build of kernels.cu for one dimension.  `origins` / `directions`: the rays of eucl_trace_rays*,
// null for camera frames.  The int-returning launchers return the number of kernels they launched.
struct Kernels {
    void (*camera_entity)(const Launch& l, const FrameParams& fp, const Workspace& ws); // (a batch: in front of raygen too)
    void (*raygen)(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, int32_t* hit_ids_out,
                   const double* origins, const double* directions);
    int (*intersect)(const Launch& l, const Workspace& ws, int level);
    int (*shade)(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, int level,
                 int32_t* hit_ids_out);
    int (*resolve_and_final)(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws,
                             uint8_t* out_rgb8, const AovPlanes& aov);
    void (*megakernel)(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, uint8_t* out_rgb8,
                       int32_t* hit_ids_out, const AovPlanes& aov, const double* origins, const double* directions,
                       const TreeQuery& tree);
    int (*tree_export)(const Launch& l, const FrameParams& fp, const ChunkParams& cp, const Workspace& ws, const TreeQuery& tree);
    void (*trace_path)(const Launch& l, const double* d_in, double distance, double* d_out, int* d_found);
    // the universe queries (eucl_trace_paths*, eucl_locate_points*), every array on the device
    void (*trace_paths)(const Launch& l, const double* d_locations, const double* d_directions, const double* d_distances,
                        uint32_t n, uint32_t steps, double* d_out_locations, double* d_out_directions, int32_t* d_out_status);
    void (*locate)(const Launch& l, const double* d_points, uint32_t n, int32_t* d_out);
};

} // namespace eucl

// kernels.cu, compiled twice: namespace eucl (real = double) and namespace eucl_f32 (real = float, the reference's
// `low_precision` feature).  The structs above are shared; a scene picks its table once (EuclScene::k), so no launch
// can reach the other precision's build.  configure_kernels sets up every kernel of the build, both dimensions.
namespace eucl {
const Kernels& kernels(int dim);
cudaError_t configure_kernels(size_t smem_bytes, size_t smem_scene);
int fp64_peak(double* dadd, double* dmul, double* dfma); // T op/s on the current device (f64 build only)
} // namespace eucl
namespace eucl_f32 {
const eucl::Kernels& kernels(int dim);
cudaError_t configure_kernels(size_t smem_bytes, size_t smem_scene);
} // namespace eucl_f32
