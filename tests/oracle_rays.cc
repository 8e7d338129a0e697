// oracle_rays.cc -- the CPU oracle's statement of eucl_trace_rays (include/euclider_b200.h: EuclRays).
//
// TEST INFRASTRUCTURE ONLY, like oracle/oracle.cc, which this file includes unchanged: ray i is Tracer::pixel with the
// camera replaced by (origin i, direction i), both loaded `as F` once and the direction used as given, not normalised.
//   e = material_at(o) >= 0  colour of trace(max_depth, e, o, material_enter(e, d)) over opaque white, the primary hit, and
//                            the AOV planes of the primary ray (o, d') exactly as tests/oracle_aovs.cc states them for a pixel
//   e < 0                    the checkerboard of cell (i % width, i / width), hit -2, NaN / NaN / NaN, 0 / 0; the ray is in
//                            no level count (trace is never called)
// It also exports the camera's own rays (Tracer::ray_vector) in both builds, so that a test can trace a frame's rays.
// Built by tests/oracle_rays_api.py (the f64 `det` build and the f32 build, the flags of oracle/Makefile).
#include <limits>

#include "../oracle/oracle.cc"

namespace {

template <int D>
int trace_rays_impl(const EuclFlatScene* scene, const double* origins, const double* directions, uint32_t n, uint32_t width,
                    uint32_t max_depth, double time, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                    float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (threads < 1) threads = 1;
    const uint64_t tile = 128;
    std::atomic<uint64_t> next_tile{0};
    EuclCamera cam{};
    cam.dim = D;
    cam.max_depth = max_depth;
    std::vector<Tracer<D>> tracers;
    tracers.reserve((size_t)threads);
    for (int t = 0; t < threads; ++t) tracers.emplace_back(*scene, cam, time);
    const float nan = std::numeric_limits<float>::quiet_NaN(), inf = std::numeric_limits<float>::infinity();
    auto work = [&](int t) {
        Tracer<D>& tr = tracers[(size_t)t];
        for (;;) {
            const uint64_t begin = next_tile.fetch_add(tile);
            if (begin >= n) break;
            const uint64_t end = begin + tile < n ? begin + tile : n;
            for (uint64_t i = begin; i < end; ++i) {
                const Vec<D> point = load<D>(origins + i * D), vector = load<D>(directions + i * D);
                uint64_t before[EUCL_MAX_LEVELS];
                std::memcpy(before, tr.level_counts, sizeof before);
                float depth = nan, pos[D], nrm[D];
                for (int k = 0; k < D; ++k) pos[k] = nrm[k] = nan;
                const int belongs_to = tr.material_at(point);
                real r, g, b;
                int32_t hit = -2;
                if (belongs_to >= 0) {
                    Vec<D> transitioned = vector;
                    tr.material_enter(belongs_to, transitioned);
                    // the primary hit, by a context of its own (trace_closest leaves the counters alone)
                    depth = inf;
                    typename Tracer<D>::Context c;
                    c.origin_entity = belongs_to;
                    if (max_depth > 0 && tr.trace_closest(point, transitioned, &c)) {
                        depth = (float)c.hit.distance;
                        for (int k = 0; k < D; ++k) {
                            nrm[k] = (float)c.normal_closer[k];
                            pos[k] = std::isfinite(depth) ? (float)c.hit.location[k] : nan;
                        }
                    }
                    int primary = -1;
                    Rgba fg = tr.trace(max_depth, belongs_to, point, transitioned, &primary);
                    hit = primary;
                    Rgba over = from_premultiplied(
                        blend_pre(EUCL_BLEND_OVER, into_premultiplied(fg), into_premultiplied(Rgba{R(1.0), R(1.0), R(1.0), R(1.0)})));
                    r = over.r;
                    g = over.g;
                    b = over.b;
                } else {
                    const uint64_t x = width > 1 ? i % width : 0, y = width > 1 ? i / width : i;
                    if ((x / 8 + y / 8) % 2 == 0) {
                        r = g = b = R(0.0);
                    } else {
                        r = R(1.0);
                        g = R(0.0);
                        b = R(1.0);
                    }
                }
                out_rgb[3 * i + 0] = channel_to_u8(r, &tr.counters);
                out_rgb[3 * i + 1] = channel_to_u8(g, &tr.counters);
                out_rgb[3 * i + 2] = channel_to_u8(b, &tr.counters);
                if (out_hit) out_hit[i] = hit;
                uint32_t segments = 0, levels = 0;
                for (uint32_t l = 0; l <= max_depth; ++l) {
                    const uint64_t k = tr.level_counts[l] - before[l];
                    if (l < max_depth) segments += (uint32_t)k;
                    if (k) levels = l + 1;
                }
                if (out_depth) out_depth[i] = depth;
                for (int k = 0; k < D; ++k) {
                    if (out_position) out_position[i * D + k] = pos[k];
                    if (out_normal) out_normal[i * D + k] = nrm[k];
                }
                if (out_segments) out_segments[i] = segments;
                if (out_levels) out_levels[i] = levels;
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t) pool.emplace_back(work, t);
    work(0);
    for (auto& th : pool) th.join();
    if (stats) { // the layout of oracle_render's stats: [0] segments, [1] nodes, [8 + l] level l
        std::memset(stats, 0, sizeof(uint64_t) * (8 + EUCL_MAX_LEVELS));
        for (auto& tr : tracers)
            for (uint32_t l = 0; l <= max_depth; ++l) {
                stats[8 + l] += tr.level_counts[l];
                stats[1] += tr.level_counts[l];
                if (l < max_depth) stats[0] += tr.level_counts[l];
            }
    }
    return 0;
}

template <int D>
void camera_rays_impl(const EuclFlatScene* scene, const EuclCamera* camera, int w, int h, double* origins, double* directions) {
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
}

} // namespace

extern "C" {

// n rays ([n][dim] doubles each) traced to RGB8, hit ids and the AOV planes (each but out_rgb may be NULL), in ray order.
int oracle_trace_rays(const EuclFlatScene* scene, const double* origins, const double* directions, uint32_t n, uint32_t width,
                      uint32_t max_depth, double time, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                      float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (!scene || !origins || !directions || !out_rgb || max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    if (width > 1 && n % width) return -1;
    if (scene->dim == 3)
        return trace_rays_impl<3>(scene, origins, directions, n, width, max_depth, time, threads, out_rgb, out_hit, out_depth,
                                  out_position, out_normal, out_segments, out_levels, stats);
    if (scene->dim == 4)
        return trace_rays_impl<4>(scene, origins, directions, n, width, max_depth, time, threads, out_rgb, out_hit, out_depth,
                                  out_position, out_normal, out_segments, out_levels, stats);
    return -1;
}

// The w x h rays of a camera pose in row order (row 0 = bottom): the camera location (as F) and Tracer::ray_vector, the
// vectors Tracer::pixel traces, widened to double.
int oracle_camera_rays(const EuclFlatScene* scene, const EuclCamera* camera, int w, int h, double* origins, double* directions) {
    if (!scene || !camera || !origins || !directions || w < 1 || h < 1) return -1;
    if (scene->dim == 3) camera_rays_impl<3>(scene, camera, w, h, origins, directions);
    else if (scene->dim == 4) camera_rays_impl<4>(scene, camera, w, h, origins, directions);
    else return -1;
    return 0;
}

} // extern "C"
