// oracle_aovs.cc -- the CPU oracle's statement of the per-pixel auxiliary outputs (AOVs, include/euclider_b200.h: EuclAovs).
//
// TEST INFRASTRUCTURE ONLY, like oracle/oracle.cc, which this file includes unchanged: the renderer, its Tracer and its
// counters stay exactly what every other test pins, and the AOV planes are defined on top of them.
//   segments / levels  the per-pixel difference of the Tracer's level_counts across Tracer::pixel: Universe::trace calls
//                      with depth > 0, and the deepest level reached + 1 (0 / 0 when trace is never called: checkerboard)
//   depth / position / normal   the context of the pixel's first trace_closest -- the primary ray of
//                      trace_screen_point (mod.rs:371-397) -- hit.distance, hit.location and normal_closer, narrowed
//                      once to float; +inf / NaN / NaN when it finds nothing or max_depth is 0; NaN everywhere for a
//                      camera in no entity.  It is evaluated by a second Tracer, so the first one's counters see exactly
//                      the calls oracle_render makes.
// Built by tests/oracle_aovs_api.py (the f64 `det` build and the f32 build, the flags of oracle/Makefile).
#include <limits>

#include "../oracle/oracle.cc"

namespace {

template <int D>
int render_aovs_impl(const EuclFlatScene* scene, const EuclCamera* camera, uint32_t width, uint32_t height, double time,
                     uint32_t row_begin, uint32_t row_end, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                     float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (threads < 1) threads = 1;
    const uint64_t total = (uint64_t)(row_end - row_begin) * width;
    const uint64_t tile = 128;
    const uint32_t max_depth = camera->max_depth;
    std::atomic<uint64_t> next_tile{0};
    std::vector<Tracer<D>> tracers, probes;
    tracers.reserve((size_t)threads);
    probes.reserve((size_t)threads);
    for (int t = 0; t < threads; ++t) {
        tracers.emplace_back(*scene, *camera, time);
        probes.emplace_back(*scene, *camera, time);
    }
    const float nan = std::numeric_limits<float>::quiet_NaN(), inf = std::numeric_limits<float>::infinity();
    auto work = [&](int t) {
        Tracer<D>& tr = tracers[(size_t)t];
        Tracer<D>& probe = probes[(size_t)t];
        for (;;) {
            const uint64_t begin = next_tile.fetch_add(tile);
            if (begin >= total) break;
            const uint64_t end = begin + tile < total ? begin + tile : total;
            for (uint64_t idx = begin; idx < end; ++idx) {
                const int y = (int)(row_begin + (uint32_t)(idx / width)), x = (int)(idx % width);
                // primary hit
                float depth = nan, pos[D], nrm[D];
                for (int k = 0; k < D; ++k) pos[k] = nrm[k] = nan;
                const Vec<D> point = load<D>(probe.cam.location);
                const int belongs_to = probe.material_at(point);
                if (belongs_to >= 0) {
                    depth = inf;
                    Vec<D> transitioned = probe.ray_vector(x, y, (int)width, (int)height);
                    probe.material_enter(belongs_to, transitioned);
                    typename Tracer<D>::Context c;
                    c.origin_entity = belongs_to;
                    if (max_depth > 0 && probe.trace_closest(point, transitioned, &c)) {
                        depth = (float)c.hit.distance;
                        for (int k = 0; k < D; ++k) {
                            nrm[k] = (float)c.normal_closer[k];
                            pos[k] = std::isfinite(depth) ? (float)c.hit.location[k] : nan;
                        }
                    }
                }
                // the pixel itself, and its ray tree's cost
                uint64_t before[EUCL_MAX_LEVELS];
                std::memcpy(before, tr.level_counts, sizeof before);
                tr.pixel(x, y, (int)width, (int)height, out_rgb + 3 * idx, out_hit ? out_hit + idx : nullptr);
                uint32_t segments = 0, levels = 0;
                for (uint32_t l = 0; l <= max_depth; ++l) {
                    const uint64_t n = tr.level_counts[l] - before[l];
                    if (l < max_depth) segments += (uint32_t)n;
                    if (n) levels = l + 1;
                }
                if (out_depth) out_depth[idx] = depth;
                for (int k = 0; k < D; ++k) {
                    if (out_position) out_position[idx * D + k] = pos[k];
                    if (out_normal) out_normal[idx * D + k] = nrm[k];
                }
                if (out_segments) out_segments[idx] = segments;
                if (out_levels) out_levels[idx] = levels;
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

} // namespace

extern "C" {

// oracle_render of rows [row_begin, row_end) plus the AOV planes of those rows (each may be NULL), packed from row_begin.
int oracle_render_aovs(const EuclFlatScene* scene, const EuclCamera* camera, uint32_t width, uint32_t height, double time,
                       uint32_t row_begin, uint32_t row_end, int threads, uint8_t* out_rgb, int32_t* out_hit, float* out_depth,
                       float* out_position, float* out_normal, uint32_t* out_segments, uint32_t* out_levels, uint64_t* stats) {
    if (!scene || !camera || !out_rgb || camera->max_depth + 1 > EUCL_MAX_LEVELS) return -1;
    if (scene->dim == 3)
        return render_aovs_impl<3>(scene, camera, width, height, time, row_begin, row_end, threads, out_rgb, out_hit, out_depth,
                                   out_position, out_normal, out_segments, out_levels, stats);
    if (scene->dim == 4)
        return render_aovs_impl<4>(scene, camera, width, height, time, row_begin, row_end, threads, out_rgb, out_hit, out_depth,
                                   out_position, out_normal, out_segments, out_levels, stats);
    return -1;
}

} // extern "C"
