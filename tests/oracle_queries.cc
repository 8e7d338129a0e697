// oracle_queries.cc -- the CPU oracle's statement of eucl_locate_points (include/euclider_b200.h).
//
// TEST INFRASTRUCTURE ONLY, like oracle/oracle.cc, which this file includes unchanged: point i is loaded `as F` once and
// out[i] = Tracer::material_at(point), Universe::material_at (mod.rs:229-251).  oracle/oracle.cc exports material_at from
// its f64 builds only; this file exports it from the f32 build too.  Built by tests/oracle_queries_api.py (the f64 `det`
// build and the f32 build, the flags of oracle/Makefile).
#include "../oracle/oracle.cc"

namespace {

template <int D>
void locate_impl(const EuclFlatScene* scene, const double* points, uint32_t n, int32_t* out) {
    EuclCamera cam{};
    cam.dim = D;
    Tracer<D> tr(*scene, cam, 0.0);
    for (uint32_t i = 0; i < n; ++i) out[i] = tr.material_at(load<D>(points + (size_t)i * D));
}

} // namespace

extern "C" int oracle_locate(const EuclFlatScene* scene, const double* points, uint32_t n, int32_t* out) {
    if (!scene || !points || !out) return -1;
    if (scene->dim == 3) locate_impl<3>(scene, points, n, out);
    else if (scene->dim == 4) locate_impl<4>(scene, points, n, out);
    else return -1;
    return 0;
}
