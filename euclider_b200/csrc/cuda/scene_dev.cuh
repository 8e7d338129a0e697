// Device-resident flat scene.
//
// The host packs EuclFlatScene into ONE 16-byte-aligned blob (header + tables); every kernel
// stages the blob from global/L2 into shared memory with 128-bit loads and then walks the tables
// there.  Primitives are SoA (component k of v0 for primitive i lives at v0[k * n_prims + i]) so
// that lanes which diverge onto different primitives of a CSG program still hit distinct banks;
// in the brute-force entity loop all lanes read the same primitive and the load is a broadcast.
// Texels stay in HBM behind CUDA texture objects (point sampling; the bilinear filter is done in
// f64 to match the reference, surface.rs:453-489).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "euclider_b200.h"

namespace eucl {

struct SceneHeader {
    int32_t dim;
    int32_t n_prims, n_nodes, n_entities, n_materials, n_transforms, n_expr_ops;
    int32_t n_surfaces, n_color_ops, n_mapped_textures, n_textures;
    int32_t background;
    int32_t max_entity_nodes; // largest CSG program (nodes) of any entity
    int32_t blob_bytes;       // total size, multiple of 16
    // byte offsets from the start of the blob, all multiples of 16
    int32_t off_prim_kind, off_prim_v0, off_prim_v1, off_prim_s0, off_prim_s1;
    int32_t off_nodes, off_entities, off_materials, off_transforms, off_expr_ops;
    int32_t off_surfaces, off_color_ops, off_mapped, off_textures, off_tex_objects, off_perlin;
    int32_t off_planes, off_bounds;
    // "reach" key of a ray: bit k set when the ray can reach cull_root[k] (macro root nodes of up to 4 entities
    // that own a bounding sphere and are not a bare primitive); used to group the rays of a level
    int32_t n_cull;
    int32_t cull_root[4];
    int32_t off_ent_flags; // per entity: EntFlags
    int32_t light_capable; // 1: every surfaced entity is a primitive, a root plane chain or a cull root (see k_intersect<LIGHT>)
    int32_t off_lin_rows;  // LinRow table, 2 * EUCL_MAX_DIM rows per transform
    int32_t csg2_capable;  // 1: every surfaced entity is a primitive, a root plane chain or a two-leaf program (k_intersect_csg2)
    int32_t _pad[3];
};

// LinearSpace in table form.  eucl_scene_create recognises component expressions that are sums of terms
//   v | v * c | c * v | v / c      (v a legend variable, c a literal; terms joined by + or -, left to right)
// -- the hallway stretch `x * 4`, its inverse `x / 4`, pass-through `y` -- and lowers each to a row of at most
// kLinTermsMax terms.  A row performs exactly the IEEE operations meval's evaluation of the expression performs, in
// the same order, so results are bit-identical to the RPN interpreter, which stays as the fallback (n_terms == 0).
constexpr int kLinTermsMax = 4;
struct LinTerm {
    int32_t var;  // component of the INPUT vector
    int32_t kind; // 0: v, 1: v * c, 2: v / c, 3: c / v; bit 4 set: the term is subtracted from the running sum
    double c;
};
struct LinRow {
    int32_t n_terms; // 0: not a recognised row, evaluate the RPN program
    int32_t _pad;
    LinTerm t[kLinTermsMax];
};
static_assert(sizeof(LinRow) % 8 == 0, "LinRow alignment");
// rows of transform t: [t * 2 * EUCL_MAX_DIM + (inverse ? EUCL_MAX_DIM : 0) + component]

// Per-entity classification for the closest-hit loops (built by eucl_scene_create)
enum EntFlags : int32_t {
    ENT_SURFACED = 1,   // takes part in trace_closest
    ENT_PRIM = 2,       // the shape is one primitive
    ENT_ROOT_PLANES = 4, // the shape is one chain of <= kPlaneChainMax half-spaces
    ENT_CULL_ROOT = 8,  // owns a reach-key bit: rays with key 0 cannot hit it
    ENT_NEGATED = 16,   // Complement(VoidShape, X) lowered to X: hits flip their normal, membership is inverted
    ENT_CSG2 = 32       // the shape is M_OP(A, B): A a primitive or a chain of <= kPlaneChainMax half-spaces, B a primitive
};
static_assert(sizeof(SceneHeader) % 16 == 0, "header must keep 16-byte alignment");

// Conservative bounding sphere of a macro CSG node (r2 < 0: unbounded); see intersect.cuh: ray_misses.
struct Bound {
    double c[EUCL_MAX_DIM];
    double r2;
    double _pad;
};

#if defined(__CUDACC__)
// The one dynamic shared-memory array of every kernel: [SceneView][blob].  Declared here so that the
// table accessors below are expressed relative to a __shared__ symbol and compile to LDS (going
// through generic pointers stored in the view made them generic LD instructions).
extern __shared__ __align__(16) unsigned char g_smem[];
#endif

// Byte offsets (from g_smem) of the staged tables; lives at the start of shared memory.
struct SceneView {
    int dim, n_prims, n_nodes, n_entities, n_surfaces, background;
    int n_cull, cull_root[4];
    uint32_t o_prim_kind, o_prim_v0, o_prim_v1, o_prim_s0, o_prim_s1, o_planes, o_nodes, o_entities, o_materials,
        o_transforms, o_expr_ops, o_surfaces, o_color_ops, o_mapped, o_textures, o_tex_objects, o_perlin, o_bounds, o_ent_flags, o_lin_rows;
#if defined(__CUDACC__)
#define EUCL_TABLE(type, name) \
    __device__ __forceinline__ const type* name() const { return reinterpret_cast<const type*>(g_smem + o_##name); }
    EUCL_TABLE(int32_t, prim_kind)
    EUCL_TABLE(double, prim_v0)
    EUCL_TABLE(double, prim_v1)
    EUCL_TABLE(double, prim_s0)
    EUCL_TABLE(double, prim_s1)
    EUCL_TABLE(double, planes) // AoS copy of the primitives: kPlaneStride doubles each, [v0[0..3], s0, s1]
    EUCL_TABLE(EuclNode, nodes)
    EUCL_TABLE(EuclEntity, entities)
    EUCL_TABLE(EuclMaterial, materials)
    EUCL_TABLE(EuclTransform, transforms)
    EUCL_TABLE(EuclExprOp, expr_ops)
    EUCL_TABLE(EuclSurface, surfaces)
    EUCL_TABLE(EuclColorOp, color_ops)
    EUCL_TABLE(EuclMappedTexture, mapped)
    EUCL_TABLE(EuclTexture, textures)
    EUCL_TABLE(cudaTextureObject_t, tex_objects)
    EUCL_TABLE(uint8_t, perlin)
    EUCL_TABLE(Bound, bounds) // one per macro CSG node
    EUCL_TABLE(int32_t, ent_flags)
    EUCL_TABLE(LinRow, lin_rows)
#undef EUCL_TABLE
#endif
};
// fixed device evaluation stacks; eucl_scene_create rejects programs that need more (EUCL_ERR_SCENE_LIMIT)
constexpr int kExprStackMax = 16;  // shade.cuh: eval_expr
constexpr int kColorStackMax = 8;  // shade.cuh: surface_color
constexpr int kPlaneStride = 6; // doubles per record of the AoS primitive table (48 B, 16-byte aligned)

#if defined(__CUDACC__)
// Cooperative copy of the blob into shared memory + view construction.  g_smem must hold
// scene_smem_bytes(blob_bytes).
__device__ __forceinline__ const SceneView& stage_scene(const uint8_t* __restrict__ blob) {
    SceneView* view = reinterpret_cast<SceneView*>(g_smem);
    const uint32_t base = (uint32_t)((sizeof(SceneView) + 15) & ~size_t(15));
    unsigned char* dst = g_smem + base;
    const SceneHeader* gh = reinterpret_cast<const SceneHeader*>(blob);
    const int n16 = gh->blob_bytes >> 4;
    const uint4* src4 = reinterpret_cast<const uint4*>(blob);
    uint4* dst4 = reinterpret_cast<uint4*>(dst);
    for (int i = threadIdx.x; i < n16; i += blockDim.x) dst4[i] = __ldg(src4 + i);
    __syncthreads();
    if (threadIdx.x == 0) {
        const SceneHeader* h = reinterpret_cast<const SceneHeader*>(dst);
        view->dim = h->dim;
        view->n_prims = h->n_prims;
        view->n_nodes = h->n_nodes;
        view->n_entities = h->n_entities;
        view->n_surfaces = h->n_surfaces;
        view->background = h->background;
        view->n_cull = h->n_cull;
        for (int k = 0; k < 4; ++k) view->cull_root[k] = h->cull_root[k];
        view->o_prim_kind = base + h->off_prim_kind;
        view->o_prim_v0 = base + h->off_prim_v0;
        view->o_prim_v1 = base + h->off_prim_v1;
        view->o_prim_s0 = base + h->off_prim_s0;
        view->o_prim_s1 = base + h->off_prim_s1;
        view->o_planes = base + h->off_planes;
        view->o_nodes = base + h->off_nodes;
        view->o_entities = base + h->off_entities;
        view->o_materials = base + h->off_materials;
        view->o_transforms = base + h->off_transforms;
        view->o_expr_ops = base + h->off_expr_ops;
        view->o_surfaces = base + h->off_surfaces;
        view->o_color_ops = base + h->off_color_ops;
        view->o_mapped = base + h->off_mapped;
        view->o_textures = base + h->off_textures;
        view->o_tex_objects = base + h->off_tex_objects;
        view->o_perlin = base + h->off_perlin;
        view->o_bounds = base + h->off_bounds;
        view->o_ent_flags = base + h->off_ent_flags;
        view->o_lin_rows = base + h->off_lin_rows;
    }
    __syncthreads();
    return *view;
}
#endif

__host__ __device__ inline size_t scene_smem_bytes(int blob_bytes) {
    return ((sizeof(SceneView) + 15) & ~size_t(15)) + (size_t)blob_bytes;
}

} // namespace eucl
