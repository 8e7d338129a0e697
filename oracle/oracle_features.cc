// oracle_features.cc -- the CPU oracle's statements of the library's features beyond the frame: the per-pixel auxiliary
// outputs (AOVs, include/euclider_b200.h: EuclAovs), eucl_trace_rays (EuclRays), the ray trees of eucl_render_trees /
// eucl_trace_ray_trees (EuclTreeNode, EuclTreeQuery) and eucl_locate_points.
//
// TEST INFRASTRUCTURE ONLY, like oracle.cc, which this file includes unchanged: the renderer, its Tracer and its counters
// stay exactly what every other test pins, and each feature is defined on top of them.  Built by the Makefile
// (liboracle_features_det.so, liboracle_features_f32.so), in libraries of their own so that the code of liboracle_det.so
// and liboracle_f32.so, which the golden frames pin, does not depend on this file.
//
// AOV planes (oracle_render_aovs), per pixel:
//   segments / levels  the per-pixel difference of the Tracer's level_counts across Tracer::pixel: Universe::trace calls
//                      with depth > 0, and the deepest level reached + 1 (0 / 0 when trace is never called: checkerboard)
//   depth / position / normal   the context of the pixel's first trace_closest -- the primary ray of
//                      trace_screen_point (mod.rs:371-397) -- hit.distance, hit.location and normal_closer, narrowed
//                      once to float; +inf / NaN / NaN when it finds nothing or max_depth is 0; NaN everywhere for a
//                      camera in no entity.  It is evaluated by a second Tracer, so the first one's counters see exactly
//                      the calls oracle_render makes.
//
// Caller rays (oracle_trace_rays): ray i is Tracer::pixel with the camera replaced by (origin i, direction i), both loaded
// `as F` once and the direction used as given, not normalised.
//   e = material_at(o) >= 0  colour of trace(max_depth, e, o, material_enter(e, d)) over opaque white, the primary hit, and
//                            the AOV planes of the primary ray (o, d') exactly as stated above for a pixel
//   e < 0                    the checkerboard of cell (i % width, i / width), hit -2, NaN / NaN / NaN, 0 / 0; the ray is in
//                            no level count (trace is never called)
// oracle_camera_rays exports the camera's own rays (Tracer::ray_vector) in both builds, so that a test can trace a frame's
// rays.
//
// Ray trees (oracle_ray_tree): TreeRecorder::trace restates Tracer::trace (oracle.cc) with recording: the same member calls
// of the same Tracer in the same order, so the colours it returns and the level counts it bumps are those of
// oracle_render, and each call writes one node in pre-order (the node, its transmitted subtree, its reflected subtree --
// the order of the recursion).  oracle_ray_tree restates the steps of Tracer::pixel / trace_unknown around it: material_at
// of the origin, material_enter, or the checkerboard of the item's cell.  A camera pixel is the ray oracle_camera_rays
// gives for it, so one function covers both kinds of call.
//
// Universe queries (oracle_locate): point i is loaded `as F` once and out[i] = Tracer::material_at(point),
// Universe::material_at (mod.rs:229-251).  oracle.cc exports material_at from its f64 builds only; this file exports it
// from the f32 build too.
#include <limits>
#include <type_traits>

#include "oracle.cc"

namespace {

const float NAN_F = std::numeric_limits<float>::quiet_NaN(), INF_F = std::numeric_limits<float>::infinity();

// f(std::integral_constant<int, D>()) for the scene's dimension D; -1 for a dimension other than 3 and 4
template <class F>
int by_dim(int dim, F&& f) {
    if (dim == 3) return f(std::integral_constant<int, 3>());
    if (dim == 4) return f(std::integral_constant<int, 4>());
    return -1;
}

// item(t, i) for every i in [0, n) on threads t = 0 .. threads - 1 (0 is the caller's), handed out in tiles of 128 items
// as oracle_render hands out pixels
template <class F>
void tile_pool(int threads, uint64_t n, F&& item) {
    const uint64_t tile = 128;
    std::atomic<uint64_t> next_tile{0};
    auto work = [&](int t) {
        for (;;) {
            const uint64_t begin = next_tile.fetch_add(tile);
            if (begin >= n) break;
            const uint64_t end = begin + tile < n ? begin + tile : n;
            for (uint64_t i = begin; i < end; ++i) item(t, i);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
}

// the level counts of all tracers in the layout of oracle_render's stats: [0] segments, [1] nodes, [8 + l] level l
template <int D>
void fold_stats(const std::vector<Tracer<D>>& tracers, uint32_t max_depth, uint64_t* stats) {
    if (!stats) return;
    std::memset(stats, 0, sizeof(uint64_t) * (8 + EUCL_MAX_LEVELS));
    for (const auto& tr : tracers)
        for (uint32_t l = 0; l <= max_depth; ++l) {
            stats[8 + l] += tr.level_counts[l];
            stats[1] += tr.level_counts[l];
            if (l < max_depth) stats[0] += tr.level_counts[l];
        }
}

// the checkerboard colour of cell (x, y), drawn where a ray starts in no entity (mod.rs:387-395)
Rgba checkerboard(int64_t x, int64_t y) {
    return (x / 8 + y / 8) % 2 == 0 ? Rgba{R(0.0), R(0.0), R(0.0), R(1.0)} : Rgba{R(1.0), R(0.0), R(1.0), R(1.0)};
}

// a traced colour composited over opaque white, as Tracer::pixel does
Rgba over_white(const Rgba& c) {
    return from_premultiplied(blend_pre(EUCL_BLEND_OVER, into_premultiplied(c), into_premultiplied(Rgba{R(1.0), R(1.0), R(1.0), R(1.0)})));
}

// the AOV planes of one item; NaN / NaN / NaN, 0 / 0 until set
template <int D>
struct Aovs {
    float depth = NAN_F, position[D], normal[D];
    uint32_t segments = 0, levels = 0;
    Aovs() {
        for (int k = 0; k < D; ++k) position[k] = normal[k] = NAN_F;
    }

    // the primary-hit planes of the ray (point, transitioned) in entity belongs_to >= 0, by a context of its own
    // (trace_closest leaves the counters alone)
    void primary_hit(Tracer<D>& tr, int belongs_to, const Vec<D>& point, const Vec<D>& transitioned) {
        depth = INF_F;
        typename Tracer<D>::Context c;
        c.origin_entity = belongs_to;
        if (tr.max_depth > 0 && tr.trace_closest(point, transitioned, &c)) {
            depth = (float)c.hit.distance;
            for (int k = 0; k < D; ++k) {
                normal[k] = (float)c.normal_closer[k];
                position[k] = std::isfinite(depth) ? (float)c.hit.location[k] : NAN_F;
            }
        }
    }

    // segments and levels from the tracer's level counts before and after the item's trace calls
    void cost(const Tracer<D>& tr, const uint64_t* before) {
        for (uint32_t l = 0; l <= tr.max_depth; ++l) {
            const uint64_t n = tr.level_counts[l] - before[l];
            if (l < tr.max_depth) segments += (uint32_t)n;
            if (n) levels = l + 1;
        }
    }
};

// the AOV planes of oracle_render_aovs and oracle_trace_rays, each may be NULL
struct AovPlanes {
    float *depth, *position, *normal;
    uint32_t *segments, *levels;

    template <int D>
    void store(uint64_t i, const Aovs<D>& a) const {
        if (depth) depth[i] = a.depth;
        for (int k = 0; k < D; ++k) {
            if (position) position[i * D + k] = a.position[k];
            if (normal) normal[i * D + k] = a.normal[k];
        }
        if (segments) segments[i] = a.segments;
        if (levels) levels[i] = a.levels;
    }
};

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

} // namespace

extern "C" {

// oracle_render of rows [row_begin, row_end) plus the AOV planes of those rows (each may be NULL), packed from row_begin.
int oracle_render_aovs(const EuclFlatScene* scene, const EuclCamera* camera, uint32_t width, uint32_t height, double time,
                       uint32_t row_begin, uint32_t row_end, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                       float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (!scene || !camera || !out_rgb || camera->max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    if (threads < 1) threads = 1;
    const AovPlanes planes{out_depth, out_position, out_normal, out_segments, out_levels};
    return by_dim(scene->dim, [&](auto dim) {
        constexpr int D = decltype(dim)::value;
        std::vector<Tracer<D>> tracers, probes;
        tracers.reserve((size_t)threads);
        probes.reserve((size_t)threads);
        for (int t = 0; t < threads; ++t) {
            tracers.emplace_back(*scene, *camera, time);
            probes.emplace_back(*scene, *camera, time);
        }
        tile_pool(threads, (uint64_t)(row_end - row_begin) * width, [&](int t, uint64_t idx) {
            Tracer<D>& tr = tracers[(size_t)t];
            Tracer<D>& probe = probes[(size_t)t];
            const int y = (int)(row_begin + (uint32_t)(idx / width)), x = (int)(idx % width);
            Aovs<D> a;
            const Vec<D> point = load<D>(probe.cam.location);
            const int belongs_to = probe.material_at(point);
            if (belongs_to >= 0) {
                Vec<D> transitioned = probe.ray_vector(x, y, (int)width, (int)height);
                probe.material_enter(belongs_to, transitioned);
                a.primary_hit(probe, belongs_to, point, transitioned);
            }
            // the pixel itself, and its ray tree's cost
            uint64_t before[EUCL_MAX_LEVELS];
            std::memcpy(before, tr.level_counts, sizeof before);
            tr.pixel(x, y, (int)width, (int)height, out_rgb + 3 * idx, out_hit ? out_hit + idx : nullptr);
            a.cost(tr, before);
            planes.store(idx, a);
        });
        fold_stats(tracers, camera->max_depth, stats);
        return 0;
    });
}

// n rays ([n][dim] doubles each) traced to RGB8, hit ids and the AOV planes (each but out_rgb may be NULL), in ray order.
int oracle_trace_rays(const EuclFlatScene* scene, const double* origins, const double* directions, uint32_t n, uint32_t width,
                      uint32_t max_depth, double time, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                      float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (!scene || !origins || !directions || !out_rgb || max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    if (width > 1 && n % width) return -1;
    if (threads < 1) threads = 1;
    const AovPlanes planes{out_depth, out_position, out_normal, out_segments, out_levels};
    return by_dim(scene->dim, [&](auto dim) {
        constexpr int D = decltype(dim)::value;
        EuclCamera cam{};
        cam.dim = D;
        cam.max_depth = max_depth;
        std::vector<Tracer<D>> tracers;
        tracers.reserve((size_t)threads);
        for (int t = 0; t < threads; ++t) tracers.emplace_back(*scene, cam, time);
        tile_pool(threads, n, [&](int t, uint64_t i) {
            Tracer<D>& tr = tracers[(size_t)t];
            const Vec<D> point = load<D>(origins + i * D), vector = load<D>(directions + i * D);
            uint64_t before[EUCL_MAX_LEVELS];
            std::memcpy(before, tr.level_counts, sizeof before);
            Aovs<D> a;
            const int belongs_to = tr.material_at(point);
            Rgba color;
            int32_t hit = -2;
            if (belongs_to >= 0) {
                Vec<D> transitioned = vector;
                tr.material_enter(belongs_to, transitioned);
                a.primary_hit(tr, belongs_to, point, transitioned);
                int primary = -1;
                color = over_white(tr.trace(max_depth, belongs_to, point, transitioned, &primary));
                hit = primary;
            } else {
                color = width > 1 ? checkerboard((int64_t)(i % width), (int64_t)(i / width)) : checkerboard(0, (int64_t)i);
            }
            out_rgb[3 * i + 0] = channel_to_u8(color.r, &tr.counters);
            out_rgb[3 * i + 1] = channel_to_u8(color.g, &tr.counters);
            out_rgb[3 * i + 2] = channel_to_u8(color.b, &tr.counters);
            if (out_hit) out_hit[i] = hit;
            a.cost(tr, before);
            planes.store(i, a);
        });
        fold_stats(tracers, max_depth, stats);
        return 0;
    });
}

// The w x h rays of a camera pose in row order (row 0 = bottom): the camera location (as F) and Tracer::ray_vector, the
// vectors Tracer::pixel traces, widened to double.
int oracle_camera_rays(const EuclFlatScene* scene, const EuclCamera* camera, int w, int h, double* origins, double* directions) {
    if (!scene || !camera || !origins || !directions || w < 1 || h < 1) return -1;
    return by_dim(scene->dim, [&](auto dim) {
        constexpr int D = decltype(dim)::value;
        const Tracer<D> tr(*scene, *camera, 0.0);
        const Vec<D> location = load<D>(camera->location);
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) {
                const Vec<D> v = tr.ray_vector(x, y, w, h);
                const size_t i = ((size_t)y * w + x) * D;
                for (int k = 0; k < D; ++k) {
                    origins[i + k] = location[k];
                    directions[i + k] = v[k];
                }
            }
        return 0;
    });
}

// The tree of one item: the ray (origin, direction) (`dim` doubles each, loaded `as F`, the direction used as given) of an
// item whose cell is (cell_x, cell_y).  Writes the first `capacity` nodes in pre-order and the whole tree's node count.
// level_counts (may be NULL): the Tracer's per-level trace calls, [max_depth + 1].
int oracle_ray_tree(const EuclFlatScene* scene, const double* origin, const double* direction, int cell_x, int cell_y,
                    uint32_t max_depth, double time, uint32_t capacity, EuclTreeNode* out_nodes, uint32_t* out_count,
                    uint64_t* level_counts) {
    if (!scene || !origin || !direction || !out_count || (capacity && !out_nodes) || max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    return by_dim(scene->dim, [&](auto dim) {
        constexpr int D = decltype(dim)::value;
        EuclCamera cam{};
        cam.dim = D;
        cam.max_depth = max_depth;
        Tracer<D> tr(*scene, cam, time);
        TreeRecorder<D> rec{tr, out_nodes, capacity};
        const Vec<D> point = load<D>(origin), vector = load<D>(direction);
        const int belongs_to = tr.material_at(point);
        if (belongs_to >= 0) {
            Vec<D> transitioned = vector;
            tr.material_enter(belongs_to, transitioned);
            rec.trace(max_depth, belongs_to, point, transitioned, -1, EUCL_TREE_ROOT);
        } else { // one checkerboard node (mod.rs:387-395); trace is never called
            if (capacity > 0) {
                const double nan = std::numeric_limits<double>::quiet_NaN();
                EuclTreeNode* n = out_nodes;
                std::memset(n, 0, sizeof *n);
                n->parent = -1;
                n->medium = -1;
                n->hit_entity = -1;
                n->flags = EUCL_TREE_CHECKERBOARD;
                n->t = nan;
                for (int k = 0; k < D; ++k) n->origin[k] = n->direction[k] = n->normal[k] = nan;
                TreeRecorder<D>::set_color(n, checkerboard(cell_x, cell_y));
            }
            rec.count = 1;
        }
        if (level_counts)
            for (uint32_t l = 0; l <= max_depth; ++l) level_counts[l] = tr.level_counts[l];
        *out_count = rec.count;
        return 0;
    });
}

// The pixel a tree's root gives: its colour (narrowed to the scene's real) composited over opaque white and quantised, as
// Tracer::pixel does; a checkerboard root's colour is quantised as it is.
void oracle_tree_pixel(const EuclTreeNode* root, uint8_t rgb[3]) {
    Rgba c{(real)root->color[0], (real)root->color[1], (real)root->color[2], (real)root->color[3]};
    if (!(root->flags & EUCL_TREE_CHECKERBOARD)) c = over_white(c);
    rgb[0] = channel_to_u8(c.r, nullptr);
    rgb[1] = channel_to_u8(c.g, nullptr);
    rgb[2] = channel_to_u8(c.b, nullptr);
}

// Universe::material_at of n points ([n][dim] doubles each), in point order.
int oracle_locate(const EuclFlatScene* scene, const double* points, uint32_t n, int32_t* out) {
    if (!scene || !points || !out) return -1;
    return by_dim(scene->dim, [&](auto dim) {
        constexpr int D = decltype(dim)::value;
        EuclCamera cam{};
        cam.dim = D;
        Tracer<D> tr(*scene, cam, 0.0);
        for (uint32_t i = 0; i < n; ++i) out[i] = tr.material_at(load<D>(points + (size_t)i * D));
        return 0;
    });
}

} // extern "C"
