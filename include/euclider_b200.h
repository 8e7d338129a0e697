/*
 * euclider_b200.h -- C ABI of the B200-native replacement for euclider's per-pixel trace loop.
 *
 * Drop-in boundary: the reference's `Environment::render(dimensions, time, threads, context)`
 * (src/universe/mod.rs:300-357), reached from `Simulation::render` (src/simulation.rs:86), and
 * the constructor `scene::Parser::default().parse::<Box<Environment>>(json)`
 * (src/scene.rs:1466-1478, src/main.rs:81-83).  Everything here is plain C: POD structs,
 * pointers and sizes; no C++/torch types cross this boundary.
 *
 * Two stages, mirroring the reference:
 *   1. eucl_scene_parse()   : scene JSON (the reference's constructor vocabulary,
 *                             src/scene.rs:618-1408) -> EuclFlatScene (host only, no GPU needed)
 *   2. eucl_scene_create()  : EuclFlatScene -> device-resident scene
 *      eucl_render*()       : one frame = the reference's Environment::render
 *
 * All arithmetic is f64 (the reference's default `type F = f64`, src/main.rs:46-49).
 * All functions return 0 on success or a negative EuclStatus; eucl_last_error() gives the
 * thread-local message.  Nothing in this library falls back to a CPU renderer.
 */
#ifndef EUCLIDER_B200_H
#define EUCLIDER_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EUCL_MAX_DIM 4
#define EUCL_MAX_LEVELS 64 /* max_depth + 1 must not exceed this */

/* ----------------------------------------------------------------------------------------- */
/* status codes; the PARSE_* values mirror `enum ParserError` (src/scene.rs:524-552)         */
typedef enum EuclStatus {
    EUCL_OK = 0,
    EUCL_ERR_INVALID_ARGUMENT = -1,
    EUCL_ERR_PARSE_NO_DESERIALIZER = -10,   /* ParserError::NoDeserializer     */
    EUCL_ERR_PARSE_SYNTAX = -11,            /* ParserError::SyntaxError        */
    EUCL_ERR_PARSE_MISSING_TYPE = -12,      /* ParserError::MissingType        */
    EUCL_ERR_PARSE_INVALID_CONSTRUCTOR = -13, /* ParserError::InvalidConstructor */
    EUCL_ERR_PARSE_MISSING_FIELD = -14,     /* ParserError::MissingField       */
    EUCL_ERR_PARSE_TYPE_MISMATCH = -15,     /* ParserError::TypeMismatch       */
    EUCL_ERR_PARSE_CUSTOM = -16,            /* ParserError::CustomError (+ reference panics at
                                               construction: zero normal, radius <= 0, ...) */
    EUCL_ERR_TEXTURE_MISSING = -20,         /* a texture slot was never filled */
    EUCL_ERR_SCENE_LIMIT = -21,             /* scene exceeds a device limit (smem, CSG list) */
    EUCL_ERR_CUDA = -30,
    EUCL_ERR_OUT_OF_MEMORY = -31,
    EUCL_ERR_NO_DEVICE = -32
} EuclStatus;

/* ----------------------------------------------------------------------------------------- */
/* Flat scene tables (SoA-of-small-PODs; shared verbatim by the library and the test oracle) */

typedef enum EuclPrimKind {
    EUCL_PRIM_VOID = 0,       /* VoidShape          shape.rs:603-631  */
    EUCL_PRIM_SPHERE = 1,     /* Sphere             shape.rs:633-738  */
    EUCL_PRIM_HYPERPLANE = 2, /* Hyperplane         shape.rs:740-817  */
    EUCL_PRIM_HALFSPACE = 3,  /* HalfSpace          shape.rs:819-881  */
    EUCL_PRIM_CYLINDER = 4    /* Cylinder           shape.rs:883-1038 */
} EuclPrimKind;

typedef struct EuclPrim {
    int32_t kind;
    int32_t _pad;
    double v0[EUCL_MAX_DIM]; /* sphere centre | plane normal (as given, NOT normalised) | cylinder centre */
    double v1[EUCL_MAX_DIM]; /* cylinder axis (normalised at construction, shape.rs:901) */
    double s0;               /* sphere/cylinder radius | plane constant */
    double s1;               /* half-space signum (+-1, shape.rs:829) */
} EuclPrim;

typedef enum EuclCsgOp {
    EUCL_CSG_LEAF = 0,
    EUCL_CSG_UNION = 1,        /* SetOperation::Union               shape.rs:204-265 */
    EUCL_CSG_INTERSECTION = 2, /* SetOperation::Intersection        shape.rs:283-341 */
    EUCL_CSG_COMPLEMENT = 3,   /* SetOperation::Complement          shape.rs:359-410 */
    EUCL_CSG_SYMDIFF = 4       /* SetOperation::SymmetricDifference shape.rs:428-497 */
} EuclCsgOp;

/* CSG nodes are stored per entity in POST-ORDER.  For a non-leaf node at index n: its `b`
 * child is the node n-1, its `a` child is the node (node[n-1].first - 1); the subtree of n
 * is the contiguous range [node[n].first, n].  (`ComposableShape::of` left fold,
 * shape.rs:523-545.) */
typedef struct EuclNode {
    int32_t op;    /* EuclCsgOp */
    int32_t prim;  /* leaf: index into prims; else -1 */
    int32_t first; /* index of the first node of this subtree */
    int32_t _pad;
} EuclNode;

typedef struct EuclEntity {
    int32_t node_first; /* first node of the entity's shape program */
    int32_t node_root;  /* last node (= root) */
    int32_t material;   /* index into materials */
    int32_t surface;    /* index into surfaces, or -1 (Void, new_without_surface) */
} EuclEntity;

/* Materials (material.rs).  LinearSpace keeps the scene's expressions as RPN programs that
 * the device evaluates per transition exactly like meval would (no matrix approximation). */
typedef enum EuclMaterialKind { EUCL_MAT_VACUUM = 0, EUCL_MAT_LINEAR_SPACE = 1 } EuclMaterialKind;

typedef struct EuclMaterial {
    int32_t kind;
    int32_t transform_first; /* index into transforms */
    int32_t n_transforms;    /* applied in order on enter, inverse in reverse order on exit */
    int32_t _pad;
} EuclMaterial;

typedef struct EuclTransform { /* one ComponentTransformation: D forward + D inverse programs */
    int32_t fwd_first[EUCL_MAX_DIM];
    int32_t fwd_len[EUCL_MAX_DIM];
    int32_t inv_first[EUCL_MAX_DIM];
    int32_t inv_len[EUCL_MAX_DIM];
} EuclTransform;

typedef enum EuclExprOpcode {
    EUCL_EX_CONST = 0, /* push value */
    EUCL_EX_VAR = 1,   /* push component `arg` of the INPUT vector */
    EUCL_EX_ADD = 2, EUCL_EX_SUB = 3, EUCL_EX_MUL = 4, EUCL_EX_DIV = 5, EUCL_EX_REM = 6,
    EUCL_EX_POW = 7, EUCL_EX_NEG = 8,
    EUCL_EX_FUNC1 = 9, /* arg = EuclExprFunc, one operand */
    EUCL_EX_FUNC2 = 10 /* arg = EuclExprFunc, two operands */
} EuclExprOpcode;

typedef enum EuclExprFunc {
    EUCL_FN_SQRT = 0, EUCL_FN_ABS, EUCL_FN_EXP, EUCL_FN_LN, EUCL_FN_SIN, EUCL_FN_COS,
    EUCL_FN_TAN, EUCL_FN_ASIN, EUCL_FN_ACOS, EUCL_FN_ATAN, EUCL_FN_SINH, EUCL_FN_COSH,
    EUCL_FN_TANH, EUCL_FN_FLOOR, EUCL_FN_CEIL, EUCL_FN_ROUND, EUCL_FN_SIGNUM,
    EUCL_FN_ATAN2, EUCL_FN_MAX, EUCL_FN_MIN
} EuclExprFunc;

typedef struct EuclExprOp {
    int32_t op;
    int32_t arg;
    double value;
} EuclExprOp;

/* Surfaces (surface.rs:39-162): four provider slots of ComposableSurface. */
typedef enum EuclRatioOp { EUCL_RATIO_UNIFORM = 0, EUCL_RATIO_FRESNEL = 1 } EuclRatioOp;
typedef enum EuclReflOp { EUCL_REFL_SPECULAR = 0 } EuclReflOp;
typedef enum EuclThresholdOp { EUCL_THR_IDENTITY = 0, EUCL_THR_SNELL = 1 } EuclThresholdOp;

typedef struct EuclSurface {
    int32_t ratio_op;
    int32_t refl_op;
    int32_t thr_op;
    int32_t color_first; /* first op of the colour program (postfix) */
    int32_t color_len;
    int32_t _pad;
    double ratio_a; /* uniform: ratio | fresnel: refractive_index_inside  */
    double ratio_b; /*                  fresnel: refractive_index_outside */
    double thr_a;   /* snell: refractive_index */
} EuclSurface;

typedef enum EuclColorOpcode {
    EUCL_COL_UNIFORM = 0,      /* push f[0..3]                                  surface.rs:425 */
    EUCL_COL_ILLUM_GLOBAL = 1, /* light f[0..3], dark f[4..7]                   surface.rs:410 */
    EUCL_COL_ILLUM_DIR = 2,    /* light f[0..3], dark f[4..7], direction f[8..] surface.rs:392 */
    EUCL_COL_PERLIN_HUE = 3,   /* size f[0], speed f[1] (3-D only)        d3/entity/surface.rs:22 */
    EUCL_COL_TEXTURE = 4,      /* i0 = mapped texture                           surface.rs:536 */
    EUCL_COL_BLEND = 5         /* pop destination, pop source; i0 = EuclBlendFn; f[0] = ratio */
} EuclColorOpcode;

typedef enum EuclBlendFn { /* surface.rs:309-390 */
    EUCL_BLEND_RATIO = 0, EUCL_BLEND_OVER, EUCL_BLEND_INSIDE, EUCL_BLEND_OUTSIDE, EUCL_BLEND_ATOP,
    EUCL_BLEND_XOR, EUCL_BLEND_PLUS, EUCL_BLEND_MULTIPLY, EUCL_BLEND_SCREEN, EUCL_BLEND_OVERLAY,
    EUCL_BLEND_DARKEN, EUCL_BLEND_LIGHTEN, EUCL_BLEND_DODGE, EUCL_BLEND_BURN,
    EUCL_BLEND_HARD_LIGHT, EUCL_BLEND_SOFT_LIGHT, EUCL_BLEND_DIFFERENCE, EUCL_BLEND_EXCLUSION
} EuclBlendFn;

typedef struct EuclColorOp {
    int32_t op;
    int32_t i0;
    double f[12];
} EuclColorOp;

typedef enum EuclUvKind { EUCL_UV_SPHERE3 = 0 /* uv_sphere, also under uv_derank_4 */ } EuclUvKind;
typedef enum EuclTexFilter { EUCL_TEX_NEAREST = 0, EUCL_TEX_LINEAR = 1 } EuclTexFilter;

typedef struct EuclMappedTexture {
    int32_t uv_kind;
    int32_t filter;
    int32_t texture; /* index into textures */
    int32_t _pad;
    double center[EUCL_MAX_DIM];
} EuclMappedTexture;

typedef struct EuclTexture {
    uint32_t width, height;
    uint64_t texel_offset; /* byte offset into texels (RGBA8, row-major, row 0 = top) */
} EuclTexture;

/* Camera: the reference only reads `location` from JSON; the rest are literals
 * (d3/entity/camera.rs:42-52, d4/entity/camera.rs:47-59).  They are explicit here so fixed
 * poses other than the default can be rendered. */
typedef struct EuclCamera {
    int32_t dim;        /* 3 or 4 */
    uint32_t max_depth; /* reference literal: 10 */
    uint32_t fov_deg;   /* reference literal: 90 (u8, of the screen diagonal) */
    uint32_t _pad;
    double location[EUCL_MAX_DIM];
    double forward[EUCL_MAX_DIM];
    double up[EUCL_MAX_DIM];
    double left[EUCL_MAX_DIM]; /* 4-D only (right = -left); 3-D uses normalize(forward x up) */
} EuclCamera;

typedef struct EuclFlatScene {
    int32_t dim;
    int32_t n_prims, n_nodes, n_entities, n_materials, n_transforms, n_expr_ops;
    int32_t n_surfaces, n_color_ops, n_mapped_textures, n_textures;
    int32_t background; /* mapped texture index, or -1 = MappedTextureTransparent */
    const EuclPrim* prims;
    const EuclNode* nodes;
    const EuclEntity* entities; /* reference list order (ties, material_at, NaN capture) */
    const EuclMaterial* materials;
    const EuclTransform* transforms;
    const EuclExprOp* expr_ops;
    const EuclSurface* surfaces;
    const EuclColorOp* color_ops;
    const EuclMappedTexture* mapped_textures;
    const EuclTexture* textures;
    const uint8_t* texels;
    uint64_t texel_bytes;
    uint8_t perlin_perm[256]; /* noise 0.4.1 PermutationTable for the default seed 0 */
    EuclCamera camera;        /* the camera the scene JSON constructs */
} EuclFlatScene;

/* ----------------------------------------------------------------------------------------- */
/* Stage 1: scene front end (host only).                                                     */

typedef struct EuclParsedScene EuclParsedScene;

/* Mirrors Parser::default().parse::<Box<Environment>>(json) (src/scene.rs:1466). Textures
 * named by texture_image_* constructors are NOT decoded here (the reference uses the `image`
 * crate at this point, src/scene.rs:1053,1065): the caller supplies decoded RGBA8 pixels per
 * slot with eucl_parsed_set_texture before the flat scene is used. */
int eucl_scene_parse(const char* json_text, EuclParsedScene** out);
int eucl_parsed_texture_count(const EuclParsedScene* p);
const char* eucl_parsed_texture_path(const EuclParsedScene* p, int slot);
int eucl_parsed_set_texture(EuclParsedScene* p, int slot, uint32_t width, uint32_t height,
                            const uint8_t* rgba8);
/* Borrowed view; valid until the parsed scene is destroyed or a texture is (re)set. */
const EuclFlatScene* eucl_parsed_flat(EuclParsedScene* p);
void eucl_parsed_destroy(EuclParsedScene* p);

/* ----------------------------------------------------------------------------------------- */
/* Stage 2: device scene + render.                                                           */

typedef struct EuclScene EuclScene;

typedef enum EuclPipeline {
    EUCL_PIPELINE_WAVEFRONT = 0, /* ray-gen -> per level {intersect, shade+emit} -> resolve */
    EUCL_PIPELINE_MEGAKERNEL = 1 /* one thread per pixel, explicit DFS stack (cross-check) */
} EuclPipeline;

typedef struct EuclRenderOpts {
    uint32_t width, height; /* full frame, already divided by the reference's `resolution` */
    double time_seconds;    /* only feeds Perlin, truncated to whole ms like the reference */
    uint32_t band_rows;     /* rows per band; 0 = the whole frame is one band */
    uint32_t band_rank;     /* this call renders bands b with b % band_world == band_rank */
    uint32_t band_world;    /* 0 or 1 = all bands */
    int32_t pipeline;       /* EuclPipeline */
    int32_t compact_rows;   /* 0: rows land at their frame position (buffer = full frame)
                               1: this rank's rows are packed contiguously in band order */
    int32_t want_hit_ids;   /* also write the primary-ray hit-entity id map */
    int32_t profile;        /* 1: record per-kernel-family device times into EuclStats (adds events) */
    int32_t _pad;
} EuclRenderOpts;

typedef struct EuclStats {
    uint64_t pixels;                        /* pixels rendered by this call */
    uint64_t segments;                      /* Universe::trace calls with depth > 0 */
    uint64_t nodes;                         /* all ray-tree nodes incl. depth-0 background rays */
    uint64_t level_counts[EUCL_MAX_LEVELS]; /* nodes per level */
    uint32_t levels;
    uint32_t retries;  /* queue-capacity retries taken inside this call */
    uint32_t launches; /* kernels launched by this call */
    uint32_t ray_grouping; /* 1: this frame walked its rays grouped by reach key (auto-tuned per scene, EUCL_BIN_RAYS forces) */
    float ms_total;     /* device time of the whole call (CUDA events on the render stream) */
    float ms_raygen, ms_intersect, ms_shade, ms_resolve; /* per kernel family */
    uint32_t graph_replays; /* chunks of this call that ran as one CUDA graph launch (repeated launch parameters) */
} EuclStats;

int eucl_device_count(void);
const char* eucl_last_error(void);
const char* eucl_version(void);

/* The flat scene is borrowed for the duration of the call only. */
int eucl_scene_create(const EuclFlatScene* flat, int device, EuclScene** out);

/* The reference's scalar type `F` (src/main.rs:46-49): f64 by default, f32 with its cargo feature `low_precision`
 * (Cargo.toml:19-21).  An f32 scene runs the same kernels compiled for float: geometry, colours and the node arena
 * are f32, LinearSpace expressions stay f64 (meval), scene tables are narrowed where they are read.  Its pictures are
 * compared with the f32 build of the test oracle, not with the f64 ones. */
typedef enum EuclPrecision { EUCL_PRECISION_F64 = 0, EUCL_PRECISION_F32 = 1 } EuclPrecision;
int eucl_scene_create_precision(const EuclFlatScene* flat, int device, int precision, EuclScene** out);
void eucl_scene_destroy(EuclScene* scene);

/* Device memory the scene holds for its frames right now: the node arena (rays, hits, node records, colours of every
 * ray-tree node of a chunk), the index lists (shade bins and reach-key groups, one level each) and the node capacity. */
int eucl_scene_memory(const EuclScene* scene, uint64_t* arena_bytes, uint64_t* list_bytes, uint64_t* node_capacity);

/* Run this scene's kernels on the caller's CUDA stream (a cudaStream_t, e.g. torch's current
 * stream) instead of the scene's own; NULL restores the private stream. */
int eucl_scene_set_stream(EuclScene* scene, void* cuda_stream);

/* Number of rows / bytes this rank's share of a frame occupies (compact layout). */
uint32_t eucl_band_rows_for_rank(const EuclRenderOpts* opts);

/* Environment::render with HOST output buffers (row 0 = bottom, RGB8, 3*w*rows bytes;
 * hit ids int32 per pixel: entity index of the primary hit, -1 background, -2 checkerboard).
 * Synchronous.  out_hit_ids and stats may be NULL.
 * Band-split renders (band_world > 1) with compact_rows == 0 write ONLY this rank's rows of the full-frame
 * buffer and touch nothing else: N processes, one per GPU, may pass the same shared (ideally pinned) host
 * frame and fill it over their own PCIe links at the same time.
 * Frames of 65536 pixels or more are rendered as two pipelines side by side (every other 16-row band each; EUCL_SPLIT=1
 * turns that off): the scene then owns a helper host thread and a second set of CUDA streams; both are created at the
 * first such frame, ordered after / joined into the scene's stream around every call, and released by eucl_scene_destroy.
 * EuclStats of such a frame are the sums over the pipelines (ms_total: first launch to last completion). */
int eucl_render(EuclScene* scene, const EuclCamera* camera, const EuclRenderOpts* opts,
                uint8_t* out_rgb8, int32_t* out_hit_ids, EuclStats* stats);

/* Same, with DEVICE output buffers on the scene's device (e.g. a torch tensor, or a
 * peer-mapped frame buffer of GPU 0 when opts->compact_rows == 0).  Synchronous. */
int eucl_render_device(EuclScene* scene, const EuclCamera* camera, const EuclRenderOpts* opts,
                       void* d_out_rgb8, void* d_out_hit_ids, EuclStats* stats);

/* One frame of a batch: the pose (fov, max_depth) as for eucl_render, and the time that EuclRenderOpts.time_seconds
 * would carry (Perlin only, truncated to whole ms). */
typedef struct EuclFrame {
    EuclCamera camera;
    double time_seconds;
} EuclFrame;

/* K = n_frames frames of opts->width x opts->height -- a camera path, a turntable, an animation -- rendered as ONE
 * wavefront: the fixed cost of a frame (its ~30 dependent kernel launches) is paid once per batch, not per frame.
 * Output frame k occupies rows [k*height, (k+1)*height) of a K*height-row RGB8 buffer (each frame bottom-up, as
 * eucl_render); hit ids likewise K*height*width int32.  Frame k is bit-identical to eucl_render(scene,
 * &frames[k].camera, opts with time_seconds = frames[k].time_seconds).  EuclStats are the sums over the frames
 * (ms_total: the whole batch).  Synchronous.
 * Frames may differ in location, axes, fov and time; every frame must have the scene's dim and the same max_depth.
 * opts->time_seconds is ignored.  EUCL_ERR_INVALID_ARGUMENT, before any device work, for n_frames == 0, a null
 * `frames`, differing max_depth, band_world > 1 or compact_rows = 1 (band-split batches are not supported), and
 * batches of more than 2^31 - 1 pixels.  A batch of identical frames replays its CUDA graph like a repeated
 * eucl_render; a batch with any pose or time changed is launched anew. */
int eucl_render_frames(EuclScene* scene, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* opts,
                       uint8_t* out_rgb8, int32_t* out_hit_ids, EuclStats* stats);

/* Same, with DEVICE output buffers on the scene's device (K*height*width*3 bytes, and K*height*width int32 hit ids
 * when opts->want_hit_ids).  Synchronous. */
int eucl_render_frames_device(EuclScene* scene, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* opts,
                              void* d_out_rgb8, void* d_out_hit_ids, EuclStats* stats);

/* Per-pixel auxiliary outputs (AOVs) of a render: what the primary ray hit and what the pixel's ray tree cost.  Every
 * plane has the layout of the hit ids -- row 0 at the bottom, frame k of a batch in rows [k*height, (k+1)*height),
 * band-split and compact rows exactly as the hit ids -- and is optional.  `dim` is the scene's dimension (3 or 4).
 *   depth     float32          the primary hit's parametric distance t (Intersection::distance, mod.rs:127-142);
 *                              +inf when the primary ray hits nothing or max_depth == 0; NaN for checkerboard pixels
 *                              (camera in no entity)
 *   position  float32 x dim    o + d * t in the scene's precision (the intersectors' expression), narrowed once;
 *                              NaN where depth is not finite
 *   normal    float32 x dim    the primary hit's normal_closer (exiting ? -n : n, mod.rs:117-125), not renormalised;
 *                              NaN where there is no hit
 *   segments  uint32           Universe::trace calls with depth > 0 in the pixel's ray tree (the pixel's share of
 *                              EuclStats.segments); 0 for checkerboard pixels
 *   levels    uint32           deepest level of the pixel's tree + 1 (1: the primary ray ended there); 0 for
 *                              checkerboard pixels
 * Float planes are float32 for both precisions: an f64 scene narrows once.  Asking for AOVs never changes the RGB8
 * frame, the hit ids or EuclStats. */
typedef struct EuclAovs {      /* each pointer NULL = plane not wanted */
    float* depth;              /* [pixels]       */
    float* position;           /* [pixels][dim]  */
    float* normal;             /* [pixels][dim]  */
    uint32_t* segments;        /* [pixels]       */
    uint32_t* levels;          /* [pixels]       */
} EuclAovs;

/* eucl_render / eucl_render_frames with AOVs, HOST buffers.  n_frames == 1 renders frames[0] (its time replaces
 * opts->time_seconds) and accepts everything eucl_render accepts: bands, compact_rows (the planes then hold this
 * rank's rows only), a band-split rank with compact_rows == 0 writing only its own rows of every full-frame plane,
 * both pipelines.  n_frames > 1 follows the rules of eucl_render_frames.  EUCL_ERR_INVALID_ARGUMENT, before any device
 * work, for a null `aovs` or one without any plane (the plain entry points cover that case).  Synchronous. */
int eucl_render_aovs(EuclScene* scene, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* opts,
                     uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclAovs* aovs, EuclStats* stats);

/* Same, with DEVICE buffers on the scene's device: the output, the hit ids and every plane of `d_aovs` (the struct
 * itself is read on the host). */
int eucl_render_aovs_device(EuclScene* scene, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* opts,
                            void* d_out_rgb8, void* d_out_hit_ids, const EuclAovs* d_aovs, EuclStats* stats);

/* Caller-supplied rays instead of a camera: custom projections (panoramas, fisheyes, stereo pairs), jittered or
 * supersampled primaries, picking and probes.  Ray i has origin o = origins[i] and direction d = directions[i] (`dim`
 * doubles each; an f32 scene narrows them once).  d is used AS GIVEN, not normalised, like the vector of
 * Universe::trace_unknown (mod.rs:253-271).  The outputs of ray i are those of a pixel whose camera ray is (o, d):
 *   e = material_at(o) >= 0: the colour of trace(max_depth, e, o, material_enter(e, d)) composited over opaque white,
 *       the primary hit entity (-1: a miss), and the AOV planes of the primary ray (o, d') with d' = material_enter(e, d)
 *       (depth in units of |d'|);
 *   e < 0: the reference's checkerboard (mod.rs:387-395) at grid cell (x, y) = (i % W, i / W) with W = `width`, hit id
 *       -2, depth / position / normal NaN, segments / levels 0; counted in EuclStats.pixels and in no level count.
 * Tracing the w x h camera rays of a pose (W = w, every origin the camera location) gives eucl_render's frame, hit
 * ids, AOVs and counted EuclStats bit for bit.  One time (Perlin only) and one max_depth per call.
 * The rays form a virtual frame of n / W rows of W and are chunked, split across pipelines and graph-replayed like a
 * frame; a row is never split across chunks, so keep W moderate (a flat list: W = 1).  There is no band split and no
 * compact layout: a ray list is split by the caller. */
typedef struct EuclRays {
    const double* origins;    /* [n][dim] */
    const double* directions; /* [n][dim], used as given (not normalised) */
    uint32_t n;               /* 1 .. 2^31 - 1 */
    uint32_t width;           /* rays per grid row; 0 or 1 = a flat list; must divide n */
    uint32_t max_depth;       /* as EuclCamera.max_depth */
    int32_t pipeline;         /* EuclPipeline */
    double time_seconds;      /* Perlin only, truncated to whole ms as for a frame */
    int32_t profile;          /* as EuclRenderOpts.profile */
    int32_t _pad;
} EuclRays;                   /* 48 bytes */

/* Traces `rays` (host arrays) into HOST outputs in ray order: n * 3 bytes of RGB8, and -- each optional -- n int32 hit
 * ids (entity of the primary hit, -1 a miss, -2 an origin in no entity) and the planes of `aovs` (n entries each, as
 * EuclAovs; an `aovs` without any plane counts as NULL).  The rays are copied to a scene-owned device buffer, stream-ordered
 * before the first launch.  Synchronous.  EUCL_ERR_INVALID_ARGUMENT, before any device work, for n == 0 or n > 2^31 - 1,
 * null origins, directions or output, a width that does not divide n, max_depth + 1 > EUCL_MAX_LEVELS and an unknown
 * pipeline; the megakernel pipeline with max_depth > 24 fails with EUCL_ERR_SCENE_LIMIT. */
int eucl_trace_rays(EuclScene* scene, const EuclRays* rays, uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclAovs* aovs,
                    EuclStats* stats);

/* Same, with DEVICE arrays on the scene's device: the rays' origins and directions, the output, the hit ids and every plane
 * of `d_aovs` (the two structs themselves are read on the host).  A repeated call replays its CUDA graph and reads the
 * arrays' current contents. */
int eucl_trace_rays_device(EuclScene* scene, const EuclRays* rays, void* d_out_rgb8, void* d_out_hit_ids,
                           const EuclAovs* d_aovs, EuclStats* stats);

/* Ray-tree inspection: the whole ray tree behind chosen pixels or rays, node by node.  An ITEM is one cell of a call's
 * virtual frame: row * width + x for a camera call (row 0 at the bottom; frame k of a batch uses rows k*height + y), the
 * ray index for a ray call.  The item's TREE lists the Universe::trace calls made for it (mod.rs:149-184), one node per
 * call, in PRE-ORDER: a node, then its transmitted subtree, then its reflected subtree -- the order in which the reference
 * evaluates them (get_intersection_color before get_reflection_color, surface.rs:144-162).  Float fields hold the scene's
 * real widened to double (an f32 scene gives f32 values).  Two rules tie a tree to the other outputs: the root colour
 * composited over opaque white and quantised is the pixel, and the nodes with level < max_depth are the pixel's
 * `segments` AOV (largest level + 1: its `levels`). */
#define EUCL_TREE_ROOT 0
#define EUCL_TREE_TRANSMITTED 1
#define EUCL_TREE_REFLECTED 2

#define EUCL_TREE_BACKGROUND 1u     /* colour = background.get_color(direction): a miss, or level == max_depth */
#define EUCL_TREE_SURFACE 2u        /* the surface colour was evaluated (a hit with ratio < 1) */
#define EUCL_TREE_OPAQUE 4u         /* the surface colour's alpha quantises to 255: it is the transmitted term, no transmitted ray */
#define EUCL_TREE_NO_DESTINATION 8u /* no transmitted ray: its origin lies in no entity */
#define EUCL_TREE_UNDEFINED 16u     /* neither term exists (the reference would panic): transparent black */
#define EUCL_TREE_CHECKERBOARD 32u  /* root of an item whose origin lies in no entity: origin, direction, normal and t are NaN */

typedef struct EuclTreeNode {
    int32_t parent;         /* index in this item's list; -1 for the root */
    int32_t level;          /* 0 = primary ray; a node at level max_depth is a background lookup, never intersected */
    int32_t kind;           /* EUCL_TREE_ROOT, EUCL_TREE_TRANSMITTED, EUCL_TREE_REFLECTED */
    int32_t medium;         /* entity the ray travels in (trace's belongs_to); -1 for a checkerboard root */
    int32_t hit_entity;     /* entity of the closest hit, -1 none */
    int32_t exiting;        /* 1: normal_closer = -normal */
    uint32_t flags;         /* EUCL_TREE_* flags */
    uint32_t surface_rgba8; /* to_pixel4(surface colour), r | g<<8 | b<<16 | a<<24; valid with EUCL_TREE_SURFACE, else 0 */
    double ratio;           /* clamped reflection ratio; 0 without a hit */
    double t;               /* hit distance; +inf without a hit; NaN for a checkerboard root */
    double origin[EUCL_MAX_DIM], direction[EUCL_MAX_DIM]; /* the ray as traced (after material transitions) */
    double normal[EUCL_MAX_DIM]; /* normal_closer; NaN without a hit */
    double color[4];        /* what Universe::trace returns for this node (RGBA); root: before compositing over white */
} EuclTreeNode;             /* 176 bytes */

#define EUCL_TREE_MAX_ITEMS 65536u
#define EUCL_TREE_MAX_NODES (1u << 24) /* n_items * capacity: 2816 MiB of nodes (4096 items of a full depth-10 tree fit) */

typedef struct EuclTreeQuery {
    const uint32_t* items; /* [n_items]; duplicates allowed */
    uint32_t n_items;      /* 1 .. EUCL_TREE_MAX_ITEMS */
    uint32_t capacity;     /* nodes kept per item, >= 1 */
    EuclTreeNode* nodes;   /* [n_items][capacity], host */
    uint32_t* counts;      /* [n_items]: nodes in the whole tree; > capacity = truncated to the first `capacity` in pre-order */
} EuclTreeQuery;           /* 32 bytes */

/* eucl_render_frames (n_frames == 1: eucl_render of frames[0]) and eucl_trace_rays that also export the trees of
 * query->items.  HOST buffers, synchronous.  The RGB8 output, the hit ids and the counted EuclStats equal the plain call's;
 * `launches` includes the export kernels.  A tree call is never captured or replayed as a CUDA graph and leaves the plain
 * calls' graphs alone, and it never feeds the ray-grouping tuner.  EUCL_ERR_INVALID_ARGUMENT, before any device work, for
 * a null or empty query, null items, nodes or counts, capacity 0, an item outside the virtual frame, n_items * capacity
 * above EUCL_TREE_MAX_NODES, band_world > 1 or compact_rows, and everything the plain entry point rejects. */
int eucl_render_trees(EuclScene* scene, const EuclFrame* frames, uint32_t n_frames, const EuclRenderOpts* opts,
                      uint8_t* out_rgb8, int32_t* out_hit_ids, const EuclTreeQuery* query, EuclStats* stats);
int eucl_trace_ray_trees(EuclScene* scene, const EuclRays* rays, uint8_t* out_rgb8, int32_t* out_hit_ids,
                         const EuclTreeQuery* query, EuclStats* stats);

/* Universe::trace_path_unknown (src/universe/mod.rs:273-286): moves `location` by `distance` along
 * `direction` THROUGH the universe -- surfaces are crossed with the material transitions of the
 * entities on either side, so a step through a LinearSpace void is stretched or shrunk.  The
 * reference's cameras call this before every frame to translate themselves
 * (d3/entity/camera.rs:223-243); here it lets a headless caller drive a camera path the same way.
 * Returns 0 and the new location / direction, 1 if `location` lies in no entity (the reference's
 * `None`), or a negative EuclStatus.  Arrays hold `dim` doubles. */
int eucl_trace_path(EuclScene* scene, const double* location, const double* direction, double distance,
                    double* out_location, double* out_direction);

/* Universe queries in bulk: the scene's geometry without a render, one launch and one thread per item.  They run on the
 * scene's stream (eucl_scene_set_stream), read nothing but the scene, and leave the render calls' CUDA graphs alone.  The
 * host variants stage their arrays through a scene-owned device buffer in chunks of a bounded number of items, so device
 * memory does not grow with n.  EUCL_ERR_INVALID_ARGUMENT, before any device work, for a null required pointer, n == 0,
 * steps == 0 and n * steps > 2^31 - 1.
 *
 * Universe::material_at (mod.rs:229-251) for n points: out_entity[i] = the first entity in list order whose shape
 * contains points[i] (dim doubles each; an f32 scene narrows them once), -1 when none does.  Synchronous. */
int eucl_locate_points(EuclScene* scene, const double* points, uint32_t n, int32_t* out_entity);
/* Same, with DEVICE arrays on the scene's device. */
int eucl_locate_points_device(EuclScene* scene, const double* d_points, uint32_t n, int32_t* d_out_entity);

/* Universe::trace_path_unknown for n walkers, `steps` steps each.  Step j of walker i starts where step j-1 ended
 * (step 0 at locations[i]) and moves distances[i] along directions[i] (used as given, not normalised), exactly as
 * eucl_trace_path(scene, start, directions[i], distances[i], ...) would.  This is the camera rule of
 * Environment.move_camera: every step uses the walker's own direction, not the direction returned by the previous step.
 * Outputs [n][steps]: the location and direction eucl_trace_path returns, and a status:
 *   1  moved;
 *   0  the step's start lies in no entity: the location is the start (the walker stays), the direction is NaN, and the
 *      later steps repeat the same result;
 *  -1  more than 100000 surface crossings: the location and direction are NaN, and the walker stops (the later steps are -1 too).
 * out_directions may be NULL.  One walker's status never fails the call.  Synchronous. */
int eucl_trace_paths(EuclScene* scene, const double* locations, const double* directions, const double* distances,
                     uint32_t n, uint32_t steps, double* out_locations, double* out_directions, int32_t* out_status);
/* Same, with DEVICE arrays on the scene's device (d_out_directions may be NULL). */
int eucl_trace_paths_device(EuclScene* scene, const double* d_locations, const double* d_directions, const double* d_distances,
                            uint32_t n, uint32_t steps, double* d_out_locations, double* d_out_directions,
                            int32_t* d_out_status);

/* Camera rotations: the view-turning part of the reference's per-frame Camera::update, on an EuclCamera pose
 * (host arithmetic; the translation part is eucl_trace_path).  Angles in radians.  Replaces
 * PitchYawCamera3::rotate_yaw_static / rotate_pitch_static (src/universe/d3/entity/camera.rs:110-136),
 * FreeCamera3::rotate_yaw_static / rotate_roll_static (:329-337) and the matrix part of
 * FreeCamera4::update_rotation (src/universe/d4/entity/camera.rs:68-130).
 *   rotate_yaw:    about_up = 0: forward and up turn about +z (PitchYawCamera3); 1: forward turns about up (FreeCamera3)
 *   rotate_pitch:  about forward x up; snap = 1 stops at straight up / down (PitchYawCamera3), 0 = FreeCamera3
 *   rotate_roll:   up turns about forward (FreeCamera3)
 *   rotate_plane4: rotation in the plane of two of the camera's own axes (0 forward, 1 left, 2 up, 3 ana), then
 *                  reorthonormalize_4 (src/util.rs:309-322) */
int eucl_camera_rotate_yaw(EuclCamera* camera, double angle, int about_up);
int eucl_camera_rotate_pitch(EuclCamera* camera, double angle, int snap);
int eucl_camera_rotate_roll(EuclCamera* camera, double angle);
int eucl_camera_rotate_plane4(EuclCamera* camera, int axis_a, int axis_b, double angle);

/* Plain device allocations (cudaMalloc / cudaFree) for buffers that are shared through eucl_ipc_*:
 * an IPC handle must name the base of its own allocation, which framework allocators that carve
 * tensors out of large pools cannot guarantee. */
int eucl_device_malloc(int device, uint64_t bytes, void** d_ptr);
int eucl_device_free(int device, void* d_ptr);

/* Page-locks / unlocks caller-owned host memory (cudaHostRegister, portable) so that eucl_render's copies into it
 * run at full PCIe speed; meant for frame buffers the caller cannot allocate pinned itself, e.g. one frame in shared
 * memory that the ranks of a band-split render fill together. */
int eucl_host_register(void* ptr, uint64_t bytes);
int eucl_host_unregister(void* ptr);

/* Cross-process frame buffer sharing for the multi-GPU gather (one process per GPU):
 * rank 0 exports its device frame buffer, the other ranks map it and render straight into it. */
#define EUCL_IPC_HANDLE_BYTES 64
int eucl_ipc_export(void* d_ptr, uint8_t handle[EUCL_IPC_HANDLE_BYTES]);
int eucl_ipc_open(const uint8_t handle[EUCL_IPC_HANDLE_BYTES], int device, void** d_ptr);
int eucl_ipc_close(void* d_ptr);

/* Presentation helper (the step AFTER the hot path; the reference uploads the buffer as a GL texture
 * and blits it, src/simulation.rs:88-96): writes a binary PPM (P6), flipping the bottom-up rows of
 * Environment::render to the top-down order image files use. */
int eucl_write_ppm(const char* path, uint32_t width, uint32_t height, const uint8_t* rgb8_bottom_up);

/* FP64 issue-rate microbenchmark (DADD/DMUL/DFMA), the roofline denominator of this path.
 * Returns measured T op/s (one op = one double instruction per lane). */
int eucl_fp64_peak(int device, double* dadd_tops, double* dmul_tops, double* dfma_tops);

#ifdef __cplusplus
}
#endif
#endif /* EUCLIDER_B200_H */
