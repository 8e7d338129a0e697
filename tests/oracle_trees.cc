// oracle_trees.cc -- the CPU oracle's statement of the ray trees of eucl_render_trees / eucl_trace_ray_trees
// (include/euclider_b200.h: EuclTreeNode, EuclTreeQuery).
//
// TEST INFRASTRUCTURE ONLY, like oracle/oracle.cc, which this file includes unchanged.  TreeRecorder::trace restates
// Tracer::trace (oracle.cc) with recording: the same member calls of the same Tracer in the same order, so the colours it
// returns and the level counts it bumps are those of oracle_render, and each call writes one node in pre-order (the node,
// its transmitted subtree, its reflected subtree -- the order of the recursion).  oracle_ray_tree restates the steps of
// Tracer::pixel / trace_unknown around it: material_at of the origin, material_enter, or the checkerboard of the item's
// cell.  A camera pixel is the ray oracle_camera_rays (tests/oracle_rays.cc) gives for it, so one function covers both
// kinds of call.
// Built by tests/oracle_trees_api.py (the f64 `det` build and the f32 build, the flags of oracle/Makefile).
#include <limits>

#include "../oracle/oracle.cc"

namespace {

template <int D>
struct TreeRecorder {
    Tracer<D>& tr;
    EuclTreeNode* out;
    uint32_t capacity;
    uint32_t count = 0;

    EuclTreeNode* node(int idx) { return (uint32_t)idx < capacity ? out + idx : nullptr; }

    // a new node in pre-order: everything the caller knows before the trace call looks at the scene
    int open(int parent, int level, int kind, int medium, const Vec<D>& o, const Vec<D>& d) {
        const int idx = (int)count++;
        EuclTreeNode* n = node(idx);
        if (!n) return idx;
        const double nan = std::numeric_limits<double>::quiet_NaN();
        std::memset(n, 0, sizeof *n);
        n->parent = parent;
        n->level = level;
        n->kind = kind;
        n->medium = medium;
        n->hit_entity = -1;
        n->t = std::numeric_limits<double>::infinity();
        for (int k = 0; k < D; ++k) {
            n->origin[k] = (double)o[k];
            n->direction[k] = (double)d[k];
            n->normal[k] = nan;
        }
        return idx;
    }
    static void set_color(EuclTreeNode* n, const Rgba& c) {
        n->color[0] = (double)c.r;
        n->color[1] = (double)c.g;
        n->color[2] = (double)c.b;
        n->color[3] = (double)c.a;
    }

    // Tracer::trace with recording (mod.rs:149-184, surface.rs:62-162)
    Rgba trace(uint32_t depth, int belongs_to, const Vec<D>& location, const Vec<D>& direction, int parent, int kind) {
        tr.level_counts[tr.max_depth - depth]++;
        const int idx = open(parent, (int)(tr.max_depth - depth), kind, belongs_to, location, direction);
        uint32_t flags = 0;
        Rgba result;
        typename Tracer<D>::Context c;
        c.origin_entity = belongs_to;
        if (depth > 0 && tr.trace_closest(location, direction, &c)) {
            const EuclSurface& sf = tr.s.surfaces[tr.s.entities[c.hit_entity].surface];
            real ratio = rust_max(rust_min(tr.reflection_ratio(sf, c), R(1.0)), R(0.0));
            if (EuclTreeNode* n = node(idx)) {
                n->hit_entity = c.hit_entity;
                n->exiting = c.exiting ? 1 : 0;
                n->t = (double)c.hit.distance;
                n->ratio = (double)ratio;
                for (int k = 0; k < D; ++k) n->normal[k] = (double)c.normal_closer[k];
            }
            const Vec<D> offset = c.normal_closer;
            // get_intersection_color
            bool have_intersection = false;
            Rgba intersection_color{0, 0, 0, 0};
            if (!(ratio >= R(1.0))) {
                flags |= EUCL_TREE_SURFACE;
                Rgba sc = tr.surface_color(sf, c);
                uint8_t data[4];
                to_pixel4(sc, data, &tr.counters);
                if (EuclTreeNode* n = node(idx))
                    n->surface_rgba8 = (uint32_t)data[0] | (uint32_t)data[1] << 8 | (uint32_t)data[2] << 16 | (uint32_t)data[3] << 24;
                if (data[3] == 255) {
                    flags |= EUCL_TREE_OPAQUE;
                    intersection_color = sc;
                    have_intersection = true;
                } else {
                    Vec<D> transitioned = tr.threshold_direction(sf, c);
                    Vec<D> new_origin = c.hit.location + (-offset) * APPROX_EPSILON * R(128.0);
                    int destination = c.exiting ? tr.material_at(new_origin) : c.hit_entity;
                    if (destination >= 0) {
                        tr.material_exit(belongs_to, transitioned);
                        tr.material_enter(destination, transitioned);
                        Rgba transition = trace(depth - 1, destination, new_origin, transitioned, idx, EUCL_TREE_TRANSMITTED);
                        uint8_t tdata[4];
                        to_pixel4(transition, tdata, &tr.counters);
                        intersection_color = from_premultiplied(
                            blend_pre(EUCL_BLEND_OVER, into_premultiplied(new_u8(data)), into_premultiplied(new_u8(tdata))));
                        have_intersection = true;
                    } else {
                        flags |= EUCL_TREE_NO_DESTINATION;
                    }
                }
            }
            // get_reflection_color
            bool have_reflection = false;
            Rgba reflection_color{0, 0, 0, 0};
            if (!(ratio <= R(0.0))) {
                Vec<D> rd = tr.reflection_direction(c);
                Vec<D> new_origin = c.hit.location + offset * APPROX_EPSILON * R(128.0);
                reflection_color = trace(depth - 1, belongs_to, new_origin, rd, idx, EUCL_TREE_REFLECTED);
                have_reflection = true;
            }
            if (!have_intersection) {
                if (!have_reflection) {
                    tr.counters.no_material++;
                    flags |= EUCL_TREE_UNDEFINED;
                    result = Rgba{0, 0, 0, 0};
                } else {
                    result = reflection_color;
                }
            } else if (!have_reflection) {
                result = intersection_color;
            } else {
                result = combine_palette_color(reflection_color, intersection_color, ratio);
            }
        } else {
            flags |= EUCL_TREE_BACKGROUND;
            result = tr.mapped_color(tr.s.background, direction);
        }
        if (EuclTreeNode* n = node(idx)) {
            n->flags = flags;
            set_color(n, result);
        }
        return result;
    }
};

template <int D>
uint32_t ray_tree_impl(const EuclFlatScene* scene, const double* origin, const double* direction, int cell_x, int cell_y,
                       uint32_t max_depth, double time, uint32_t capacity, EuclTreeNode* out, uint64_t* level_counts) {
    EuclCamera cam{};
    cam.dim = D;
    cam.max_depth = max_depth;
    Tracer<D> tr(*scene, cam, time);
    TreeRecorder<D> rec{tr, out, capacity};
    const Vec<D> point = load<D>(origin), vector = load<D>(direction);
    const int belongs_to = tr.material_at(point);
    if (belongs_to >= 0) {
        Vec<D> transitioned = vector;
        tr.material_enter(belongs_to, transitioned);
        rec.trace(max_depth, belongs_to, point, transitioned, -1, EUCL_TREE_ROOT);
    } else if (capacity > 0) { // the checkerboard of the item's cell (mod.rs:387-395); trace is never called
        const double nan = std::numeric_limits<double>::quiet_NaN();
        EuclTreeNode* n = out;
        std::memset(n, 0, sizeof *n);
        n->parent = -1;
        n->medium = -1;
        n->hit_entity = -1;
        n->flags = EUCL_TREE_CHECKERBOARD;
        n->t = nan;
        for (int k = 0; k < D; ++k) n->origin[k] = n->direction[k] = n->normal[k] = nan;
        const bool black = (cell_x / 8 + cell_y / 8) % 2 == 0;
        TreeRecorder<D>::set_color(n, black ? Rgba{R(0.0), R(0.0), R(0.0), R(1.0)} : Rgba{R(1.0), R(0.0), R(1.0), R(1.0)});
        rec.count = 1;
    } else {
        rec.count = 1;
    }
    if (level_counts)
        for (uint32_t l = 0; l <= max_depth; ++l) level_counts[l] = tr.level_counts[l];
    return rec.count;
}

} // namespace

extern "C" {

// The tree of one item: the ray (origin, direction) (`dim` doubles each, loaded `as F`, the direction used as given) of an
// item whose cell is (cell_x, cell_y).  Writes the first `capacity` nodes in pre-order and the whole tree's node count.
// level_counts (may be NULL): the Tracer's per-level trace calls, [max_depth + 1].
int oracle_ray_tree(const EuclFlatScene* scene, const double* origin, const double* direction, int cell_x, int cell_y,
                    uint32_t max_depth, double time, uint32_t capacity, EuclTreeNode* out_nodes, uint32_t* out_count,
                    uint64_t* level_counts) {
    if (!scene || !origin || !direction || !out_count || (capacity && !out_nodes) || max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    if (scene->dim == 3)
        *out_count = ray_tree_impl<3>(scene, origin, direction, cell_x, cell_y, max_depth, time, capacity, out_nodes, level_counts);
    else if (scene->dim == 4)
        *out_count = ray_tree_impl<4>(scene, origin, direction, cell_x, cell_y, max_depth, time, capacity, out_nodes, level_counts);
    else
        return -1;
    return 0;
}

// The pixel a tree's root gives: its colour (narrowed to the scene's real) composited over opaque white and quantised, as
// Tracer::pixel does; a checkerboard root's colour is quantised as it is.
void oracle_tree_pixel(const EuclTreeNode* root, uint8_t rgb[3]) {
    Rgba c{(real)root->color[0], (real)root->color[1], (real)root->color[2], (real)root->color[3]};
    if (!(root->flags & EUCL_TREE_CHECKERBOARD))
        c = from_premultiplied(blend_pre(EUCL_BLEND_OVER, into_premultiplied(c), into_premultiplied(Rgba{R(1.0), R(1.0), R(1.0), R(1.0)})));
    rgb[0] = channel_to_u8(c.r, nullptr);
    rgb[1] = channel_to_u8(c.g, nullptr);
    rgb[2] = channel_to_u8(c.b, nullptr);
}

} // extern "C"
