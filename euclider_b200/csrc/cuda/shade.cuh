// Shading on the device: ComposableSurface providers (surface.rs:201-542), palette colour
// arithmetic, Perlin hue (d3/entity/surface.rs:22-40), mapped textures and LinearSpace material
// transitions (material.rs:70-163).  Everything is f64 in the reference's operation order.
#pragma once
#include "intersect.cuh"

namespace EUCL_NS {
using namespace eucl;

constexpr real kPi = R(3.14159265358979323846264338327950288);
constexpr real kFracPi2 = R(1.57079632679489661923132169163975144);
constexpr real kApproxEpsilon = R(1.0e-6); // nalgebra 0.8.2 approx_epsilon; the self-hit offset is (n * eps) * 128

struct Rgba {
    real r, g, b, a;
};
struct Pre { // palette PreAlpha<Rgb>
    real r, g, b, a;
};

__device__ __forceinline__ real clamp01(real v) { return v < R(0.0) ? R(0.0) : (v > R(1.0) ? R(1.0) : v); }

// palette to_pixel: clamp to [0,1], * 255, truncate.  A NaN channel (the reference would panic in
// to_u8().unwrap()) is defined as 0, the same definition the oracle uses.
__device__ __forceinline__ unsigned channel_to_u8(real c) {
    if (isnan(c)) return 0u;
    return (unsigned)(int)(clamp01(c) * R(255.0));
}
__device__ __forceinline__ unsigned to_pixel4(const Rgba& c) {
    return channel_to_u8(c.r) | (channel_to_u8(c.g) << 8) | (channel_to_u8(c.b) << 16) | (channel_to_u8(c.a) << 24);
}
__device__ __forceinline__ Rgba new_u8(unsigned q) {
    return Rgba{(real)(q & 255u) / R(255.0), (real)((q >> 8) & 255u) / R(255.0), (real)((q >> 16) & 255u) / R(255.0),
                (real)(q >> 24) / R(255.0)};
}
__device__ __forceinline__ Pre into_premultiplied(const Rgba& c) {
    real a = clamp01(c.a);
    return Pre{c.r * a, c.g * a, c.b * a, a};
}
__device__ __forceinline__ bool is_normal(real a) { return isfinite(a) && fabs(a) >= kMinNormal; }
__device__ __forceinline__ Rgba from_premultiplied(const Pre& p) {
    real a = clamp01(p.a);
    // x / 1 is x: the three divisions (~30 instructions each in f64) are skipped for an opaque colour, the usual case.
    // A NaN channel stays a NaN, which is all that is ever asked of it (channel_to_u8, comparisons).
    if (a == R(1.0)) return Rgba{p.r, p.g, p.b, a};
    if (is_normal(a)) return Rgba{p.r / a, p.g / a, p.b / a, a};
    return Rgba{R(0.0), R(0.0), R(0.0), a};
}

__device__ __forceinline__ real blend_channel(int fn, real a, real b, real sa, real da) {
    switch (fn) {
    case EUCL_BLEND_OVER: return a + b * (R(1.0) - sa);
    case EUCL_BLEND_INSIDE: return a * da;
    case EUCL_BLEND_OUTSIDE: return a * (R(1.0) - da);
    case EUCL_BLEND_ATOP: return a * da + b * (R(1.0) - sa);
    case EUCL_BLEND_XOR: return a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_PLUS: return a + b;
    case EUCL_BLEND_MULTIPLY: return a * b + a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_SCREEN: return a + b - a * b;
    case EUCL_BLEND_OVERLAY:
        if (b * R(2.0) <= da) return R(2.0) * a * b + a * (R(1.0) - da) + b * (R(1.0) - sa);
        return a * (R(1.0) + da) + b * (R(1.0) + sa) - R(2.0) * a * b - da * sa;
    case EUCL_BLEND_DARKEN: return fmin(a * da, b * sa) + a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_LIGHTEN: return fmax(a * da, b * sa) + a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_DODGE:
        if (a == sa && !is_normal(b)) return a * (R(1.0) - da);
        if (a == sa) return sa * da + a * (R(1.0) - da) + b * (R(1.0) - sa);
        return sa * da * fmin(R(1.0), (b / da) * sa / (sa - a)) + a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_BURN:
        if (!is_normal(a) && b == da) return sa * da + b * (R(1.0) - sa);
        if (!is_normal(a)) return b * (R(1.0) - sa);
        return sa * da * (R(1.0) - fmin(R(1.0), (R(1.0) - b / da) * sa / a)) + a * (R(1.0) - da) + b * (R(1.0) - sa);
    case EUCL_BLEND_HARD_LIGHT:
        if (a * R(2.0) <= sa) return R(2.0) * a * b + a * (R(1.0) - da) + b * (R(1.0) - sa);
        return a * (R(1.0) + da) + b * (R(1.0) + sa) - R(2.0) * a * b - da * sa;
    case EUCL_BLEND_SOFT_LIGHT: {
        real m = is_normal(da) ? b / da : R(0.0);
        if (a * R(2.0) <= sa) return b * (sa + (R(2.0) * a - sa) * (R(1.0) - m)) + a * (R(1.0) - da) + b * (R(1.0) - sa);
        if (b * R(4.0) <= da) {
            real m2 = m * m, m3 = m2 * m;
            return da * (R(2.0) * a - sa) * (m3 * R(16.0) - m2 * R(12.0) - m * R(3.0)) + a - a * da + b;
        }
        return da * (R(2.0) * a - sa) * (sqrt(m) - m) + a - a * da + b;
    }
    case EUCL_BLEND_DIFFERENCE: return a + b - R(2.0) * fmin(a * da, b * sa);
    case EUCL_BLEND_EXCLUSION: return a + b - R(2.0) * a * b;
    }
    return a;
}

// palette Blend on premultiplied colours: `s` = self (source), `d` = argument (destination)
__device__ __noinline__ Pre blend_pre(int fn, EUCL_VARG(Pre) s, EUCL_VARG(Pre) d) {
    const real sa = s.a, da = d.a;
    real alpha;
    switch (fn) {
    case EUCL_BLEND_INSIDE: alpha = clamp01(sa * da); break;
    case EUCL_BLEND_OUTSIDE: alpha = clamp01(sa * (R(1.0) - da)); break;
    case EUCL_BLEND_ATOP: alpha = clamp01(da); break;
    case EUCL_BLEND_XOR: alpha = clamp01(sa + da - R(2.0) * sa * da); break;
    case EUCL_BLEND_PLUS: alpha = clamp01(sa + da); break;
    default: alpha = clamp01(sa + da - sa * da); break;
    }
    // one rolled loop over the colour channels: a single copy of the 17-way switch in the kernel's code
    const real sc[3] = {s.r, s.g, s.b}, dc[3] = {d.r, d.g, d.b};
    real out[3];
#pragma unroll 1
    for (int k = 0; k < 3; ++k) out[k] = blend_channel(fn, sc[k], dc[k], sa, da);
    return Pre{out[0], out[1], out[2], alpha};
}
__device__ __forceinline__ Pre over_pre(const Pre& s, const Pre& d) {
    return Pre{s.r + d.r * (R(1.0) - s.a), s.g + d.g * (R(1.0) - s.a), s.b + d.b * (R(1.0) - s.a),
               clamp01(s.a + d.a - s.a * d.a)};
}

// util.rs:265-285
__device__ __forceinline__ Rgba combine_palette_color(const Rgba& a, const Rgba& b, real a_ratio) {
    if (a_ratio <= R(0.0)) return b;
    if (a_ratio >= R(1.0)) return a;
    return Rgba{a.r * a_ratio + b.r * (R(1.0) - a_ratio), a.g * a_ratio + b.g * (R(1.0) - a_ratio),
                a.b * a_ratio + b.b * (R(1.0) - a_ratio), a.a * a_ratio + b.a * (R(1.0) - a_ratio)};
}

// palette Hsv -> Rgb (hue in degrees), saturation = value = 1 at the only call site
__device__ __forceinline__ Rgba hue_to_rgba(real hue_degrees) {
    real deg = hue_degrees;
    if (isfinite(deg)) {
        while (deg >= R(360.0)) deg = deg - R(360.0);
        while (deg < R(0.0)) deg = deg + R(360.0);
    }
    const real c = R(1.0) * R(1.0);
    real h = deg / R(60.0);
    real x = c * (R(1.0) - fabs(fmod(h, R(2.0)) - R(1.0)));
    real m = R(1.0) - c;
    real r, g, b;
    if (h >= R(0.0) && h < R(1.0)) { r = c; g = x; b = R(0.0); }
    else if (h >= R(1.0) && h < R(2.0)) { r = x; g = c; b = R(0.0); }
    else if (h >= R(2.0) && h < R(3.0)) { r = R(0.0); g = c; b = x; }
    else if (h >= R(3.0) && h < R(4.0)) { r = R(0.0); g = x; b = c; }
    else if (h >= R(4.0) && h < R(5.0)) { r = x; g = R(0.0); b = c; }
    else { r = c; g = R(0.0); b = x; }
    return Rgba{r + m, g + m, b + m, R(1.0)};
}

// noise 0.4.1 Perlin::get([f64; 4]) with the seed-0 permutation table staged in shared memory
__device__ __noinline__ real perlin4(const uint8_t* perm, real px, real py, real pz, real pw) {
    const real point[4] = {px, py, pz, pw};
    const real diag = R(0.577350269189625764077083524672081875);
    real near_d[4], far_d[4];
    long long near_c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        real f = floor(point[k]);
        near_c[k] = (long long)f;
        near_d[k] = point[k] - f;
        far_d[k] = near_d[k] - R(1.0);
    }
    real total = R(0.0);
#pragma unroll 1
    for (int corner = 0; corner < 16; ++corner) {
        real dd[4];
        unsigned cc[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool far = (corner >> k) & 1;
            cc[k] = (unsigned)((far ? near_c[k] + 1 : near_c[k]) & 0xff);
            dd[k] = far ? far_d[k] : near_d[k];
        }
        real attn = R(1.0) - (((dd[0] * dd[0] + dd[1] * dd[1]) + dd[2] * dd[2]) + dd[3] * dd[3]);
        real v = R(0.0);
        if (attn > R(0.0)) {
            unsigned h = perm[cc[0]];
            h = perm[h ^ cc[1]];
            h = perm[h ^ cc[2]];
            h = perm[h ^ cc[3]];
            h &= 31u;
            const unsigned zero_at = h >> 3, signs = h & 7u;
            real g[4];
            int bit = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if ((unsigned)k == zero_at) {
                    g[k] = R(0.0);
                } else {
                    g[k] = ((signs >> bit) & 1u) ? -diag : diag;
                    ++bit;
                }
            }
            real a2 = attn * attn;
            v = (a2 * a2) * (((dd[0] * g[0] + dd[1] * g[1]) + dd[2] * g[2]) + dd[3] * g[3]);
        }
        total = corner == 0 ? v : total + v;
    }
    return total * R(4.424369240215691);
}

// util.rs:287-299 on floats
__device__ __forceinline__ real remainder_f(real a, real b) {
    real rem = fmod(a, b);
    if (rem == R(0.0)) return R(0.0);
    if (a < R(0.0)) return b + rem;
    return rem;
}
__device__ __forceinline__ long long remainder_i(long long a, long long b) {
    long long rem = a % b;
    if (rem == 0) return 0;
    if (a < 0) return b + rem;
    return rem;
}

// One texel as 4 doubles in 0..255.  Out-of-domain coordinates (the reference would panic in
// NumCast / get_pixel) fetch texel (0,0), the same definition the oracle uses.
__device__ __forceinline__ Rgba fetch_texel(cudaTextureObject_t tex, const EuclTexture& t, real xf, real yf) {
    long long x = 0, y = 0;
    if ((xf > -R(1.0) && xf < R(4294967296.0)) && (yf > -R(1.0) && yf < R(4294967296.0))) {
        x = (long long)xf;
        y = (long long)yf;
    }
    if (x >= (long long)t.width || y >= (long long)t.height) {
        x = 0;
        y = 0;
    }
    uchar4 px = tex2D<uchar4>(tex, (float)x + 0.5f, (float)y + 0.5f);
    return Rgba{(real)px.x, (real)px.y, (real)px.z, (real)px.w};
}

// MappedTextureImpl::get_color with uv_sphere (+ uv_derank in 4-D) and the two image filters
template <int D>
__device__ __noinline__ Rgba mapped_color(const SceneView& sv, int mapped, EUCL_VARG(Vec<D>) point) {
    if (mapped < 0) return Rgba{R(0.0), R(0.0), R(0.0), R(0.0)}; // MappedTextureTransparent
    const EuclMappedTexture mt = sv.mapped()[mapped];
    Vec<3> p;
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = point[k] - R(mt.center[k]);
    p = normalize(p);
    const real u = R(0.5) + dm_atan2(p[1], p[0]) / (R(2.0) * kPi);
    const real v = R(0.5) - dm_asin(p[2]) / kPi;
    const EuclTexture t = sv.textures()[mt.texture];
    const cudaTextureObject_t tex = sv.tex_objects()[mt.texture];
    const real width = (real)t.width, height = (real)t.height;
    if (mt.filter == EUCL_TEX_NEAREST) {
        real x = floor(u * width), y = floor(v * height);
        if (!((x > -R(1.0) && x < R(4294967296.0)) && (y > -R(1.0) && y < R(4294967296.0)))) {
            x = R(0.0);
            y = R(0.0);
        }
        long long xi = remainder_i((long long)x, (long long)t.width), yi = remainder_i((long long)y, (long long)t.height);
        Rgba px = fetch_texel(tex, t, (real)xi, (real)yi);
        return Rgba{px.r / R(255.0), px.g / R(255.0), px.b / R(255.0), px.a / R(255.0)};
    }
    const real x = u * width - R(0.5), y = v * height - R(0.5);
    const real fx = x - floor(x), fy = y - floor(y);
    const real x0 = remainder_f(x + R(0.0), width), x1 = remainder_f(x + R(1.0), width);
    const real y0 = remainder_f(y + R(0.0), height), y1 = remainder_f(y + R(1.0), height);
    const Rgba p0 = fetch_texel(tex, t, x0, y0), p1 = fetch_texel(tex, t, x1, y0);
    const Rgba p2 = fetch_texel(tex, t, x0, y1), p3 = fetch_texel(tex, t, x1, y1);
    const real gx = R(1.0) - fx, gy = R(1.0) - fy;
    return Rgba{((p0.r * gx + p1.r * fx) * gy + (p2.r * gx + p3.r * fx) * fy) / R(255.0),
                ((p0.g * gx + p1.g * fx) * gy + (p2.g * gx + p3.g * fx) * fy) / R(255.0),
                ((p0.b * gx + p1.b * fx) * gy + (p2.b * gx + p3.b * fx) * fy) / R(255.0),
                ((p0.a * gx + p1.a * fx) * gy + (p2.a * gx + p3.a * fx) * fy) / R(255.0)};
}

// --- materials ---------------------------------------------------------------------------------

// BEGIN_KEEP64
// meval-style RPN program (compiled on the host from the scene's expression strings); f64 in both precisions:
// the reference's LinearSpace evaluates meval expressions in f64 and narrows the result (material.rs:99-110)
__device__ __noinline__ double eval_expr(const SceneView& sv, int first, int len, const double* vars) {
    double st[kExprStackMax];
    int sp = 0;
    for (int i = first; i < first + len; ++i) {
        const EuclExprOp o = sv.expr_ops()[i];
        if (o.op == EUCL_EX_CONST) {
            st[sp++] = o.value;
        } else if (o.op == EUCL_EX_VAR) {
            st[sp++] = vars[o.arg];
        } else if (o.op == EUCL_EX_NEG) {
            st[sp - 1] = -st[sp - 1];
        } else if (o.op == EUCL_EX_FUNC1) {
            double x = st[sp - 1], r = x;
            switch (o.arg) {
            case EUCL_FN_SQRT: r = sqrt(x); break;
            case EUCL_FN_ABS: r = fabs(x); break;
            case EUCL_FN_EXP: r = exp(x); break;
            case EUCL_FN_LN: r = log(x); break;
            case EUCL_FN_SIN: r = dm_sin(x); break;
            case EUCL_FN_COS: r = dm_cos(x); break;
            case EUCL_FN_TAN: r = tan(x); break;
            case EUCL_FN_ASIN: r = dm_asin(x); break;
            case EUCL_FN_ACOS: r = dm_acos(x); break;
            case EUCL_FN_ATAN: r = dm_atan(x); break;
            case EUCL_FN_SINH: r = sinh(x); break;
            case EUCL_FN_COSH: r = cosh(x); break;
            case EUCL_FN_TANH: r = tanh(x); break;
            case EUCL_FN_FLOOR: r = floor(x); break;
            case EUCL_FN_CEIL: r = ceil(x); break;
            case EUCL_FN_ROUND: r = round(x); break;
            case EUCL_FN_SIGNUM: r = rust_signum(x); break;
            }
            st[sp - 1] = r;
        } else {
            double b = st[--sp], a = st[sp - 1], r = 0.0;
            switch (o.op) {
            case EUCL_EX_ADD: r = a + b; break;
            case EUCL_EX_SUB: r = a - b; break;
            case EUCL_EX_MUL: r = a * b; break;
            case EUCL_EX_DIV: r = a / b; break;
            case EUCL_EX_REM: r = fmod(a, b); break;
            case EUCL_EX_POW: r = pow(a, b); break;
            case EUCL_EX_FUNC2:
                if (o.arg == EUCL_FN_ATAN2) r = dm_atan2(a, b);
                else if (o.arg == EUCL_FN_MAX) r = fmax(a, b);
                else r = fmin(a, b);
                break;
            }
            st[sp - 1] = r;
        }
    }
    return sp > 0 ? st[sp - 1] : 0.0;
}

// ComponentTransformation::transform_with (material.rs:91-112): all component expressions see the
// same input vector.  Components lowered to table rows (scene_dev.cuh: LinRow) run as a few multiplications /
// divisions / additions; anything else goes through the RPN interpreter.
template <int D>
__device__ __noinline__ void apply_transform(const SceneView& sv, int t_index, bool inverse, Vec<D>& v) {
    const EuclTransform& t = sv.transforms()[t_index];
    const LinRow* rows = sv.lin_rows() + (size_t)t_index * 2 * EUCL_MAX_DIM + (inverse ? EUCL_MAX_DIM : 0);
    double in[D];
#pragma unroll
    for (int k = 0; k < D; ++k) in[k] = v[k];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const LinRow& row = rows[k];
        if (row.n_terms == 0) {
            v[k] = inverse ? eval_expr(sv, t.inv_first[k], t.inv_len[k], in) : eval_expr(sv, t.fwd_first[k], t.fwd_len[k], in);
            continue;
        }
        double acc = 0.0;
        for (int j = 0; j < row.n_terms; ++j) {
            const LinTerm term = row.t[j];
            const double x = in[term.var];
            const int kind = term.kind & 15;
            const double val = kind == 0 ? x : kind == 1 ? x * term.c : kind == 2 ? x / term.c : term.c / x;
            acc = j == 0 ? val : ((term.kind & 16) ? acc - val : acc + val);
        }
        v[k] = acc;
    }
}
// END_KEEP64
// Material::enter (Vacuum: no-op, material.rs:43-49; LinearSpace: forward transforms in order, :133-137)
template <int D>
__device__ __forceinline__ void material_enter(const SceneView& sv, int entity, Vec<D>& dir) {
    const EuclMaterial m = sv.materials()[sv.entities()[entity].material];
    if (m.kind != EUCL_MAT_LINEAR_SPACE) return;
    for (int k = 0; k < m.n_transforms; ++k) apply_transform<D>(sv, m.transform_first + k, false, dir);
}
// Material::exit (LinearSpace: inverse transforms in reverse order, material.rs:139-142,156-162)
template <int D>
__device__ __forceinline__ void material_exit(const SceneView& sv, int entity, Vec<D>& dir) {
    const EuclMaterial m = sv.materials()[sv.entities()[entity].material];
    if (m.kind != EUCL_MAT_LINEAR_SPACE) return;
    for (int k = m.n_transforms - 1; k >= 0; --k) apply_transform<D>(sv, m.transform_first + k, true, dir);
}

// --- surface providers -------------------------------------------------------------------------

// util.rs:631-666: rotate `v` in the plane spanned by (self_, other) by `angle`
template <int D>
__device__ __noinline__ Vec<D> general_rotation(EUCL_VARG(Vec<D>) self_, EUCL_VARG(Vec<D>) other, real angle, EUCL_VARG(Vec<D>) v) {
    real original[D][D], result[D][D]; // [row][col]
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = 0; c < D; ++c) original[r][c] = r == c ? R(1.0) : R(0.0);
#pragma unroll
    for (int r = 0; r < D; ++r) {
        original[r][0] = self_[r];
        original[r][1] = other[r];
    }
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = 0; c < D; ++c) result[r][c] = original[r][c];
#pragma unroll
    for (int i = 1; i < D; ++i) {
#pragma unroll
        for (int j = 0; j < i; ++j) {
            Vec<D> oc, rc;
#pragma unroll
            for (int r = 0; r < D; ++r) {
                oc[r] = original[r][i];
                rc[r] = result[r][j];
            }
            Vec<D> upd = oc - rc * dot(rc, oc);
#pragma unroll
            for (int r = 0; r < D; ++r) original[r][i] = upd[r];
        }
        Vec<D> col;
#pragma unroll
        for (int r = 0; r < D; ++r) col[r] = original[r][i];
        col = normalize(col);
#pragma unroll
        for (int r = 0; r < D; ++r) result[r][i] = col[r];
    }
    real rot[D][D];
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
        for (int c = 0; c < D; ++c) rot[r][c] = r == c ? R(1.0) : R(0.0);
    const real ca = dm_cos(angle), sa = dm_sin(angle);
    rot[0][0] = ca;
    rot[0][1] = -sa;
    rot[1][0] = sa;
    rot[1][1] = ca;
    // result * (rotation_matrix * result.transpose()); nalgebra accumulates from zero, so the
    // multiplications by the identity part of `rot` are kept (0 * NaN must stay NaN)
    real tmp[D][D], q[D][D];
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) {
            real acc = R(0.0);
#pragma unroll
            for (int k = 0; k < D; ++k) acc = acc + rot[i][k] * result[j][k];
            tmp[i][j] = acc;
        }
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) {
            real acc = R(0.0);
#pragma unroll
            for (int k = 0; k < D; ++k) acc = acc + result[i][k] * tmp[k][j];
            q[i][j] = acc;
        }
    Vec<D> out;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        real acc = R(0.0);
#pragma unroll
        for (int j = 0; j < D; ++j) acc = acc + v[j] * q[i][j];
        out[i] = acc;
    }
    return out;
}

// The angles every provider derives from the same two vectors.  The intersect kernel already
// evaluated c = dot(d, n) / (|d| |n|) for the raw normal; negating a vector negates the dot product
// and the quotient exactly, so cos(d, -n) = -c bit for bit and nothing is recomputed here.
//   cos_raw    : direction vs the intersector's normal          (illumination_directional)
//   cos_closer : direction vs normal_closer                     (illumination_global)
//   from_theta : angle_between(direction, -normal_closer)       (Fresnel, Snell)

// reflection_ratio_uniform / reflection_ratio_fresnel (surface.rs:201-244), before clamping
// Values Fresnel and Snell both derive from from_theta; computed at most once per hit.  The two
// providers take asin of (from_index / to_index) * sin and of modifier * sin: for a consistent glass
// description these arguments are the SAME double (e.g. 1.458 / 1 and 1.458), detected by comparing
// the bits of the arguments, never assumed.
struct RefractionCache {
    real sin_from;   // sin(from_theta)
    real asin_arg;   // argument of the cached asin
    real asin_value; // asin(asin_arg)
    bool have_asin;
};
__device__ __forceinline__ real cached_asin(RefractionCache& rc, real arg) {
    if (rc.have_asin && __double_as_longlong(arg) == __double_as_longlong(rc.asin_arg)) return rc.asin_value;
    rc.asin_arg = arg;
    rc.asin_value = dm_asin(arg);
    rc.have_asin = true;
    return rc.asin_value;
}

template <int D, bool GLASS = true>
__device__ __forceinline__ real reflection_ratio(const EuclSurface& sf, real from_theta, bool exiting,
                                                   RefractionCache& rc) {
    // from_theta = angle_between(direction, -normal_closer), computed once per hit
    if (!GLASS || sf.ratio_op == EUCL_RATIO_UNIFORM) return exiting ? R(0.0) : R(sf.ratio_a);
    const real from_index = exiting ? R(sf.ratio_a) : R(sf.ratio_b);
    const real to_index = exiting ? R(sf.ratio_b) : R(sf.ratio_a);
    const real to_theta = cached_asin(rc, (from_index / to_index) * rc.sin_from);
    if (isnan(to_theta)) return R(1.0);
    const real cf = dm_cos(from_theta), ct = dm_cos(to_theta);
    const real p1s = from_index * cf, p2s = to_index * ct;
    const real p1p = from_index * ct, p2p = to_index * cf;
    const real rs = (p1s - p2s) / (p1s + p2s);
    const real rp = (p1p - p2p) / (p1p + p2p);
    return (rs * rs + rp * rp) / (R(1.0) + R(1.0));
}

// reflection_direction_specular (surface.rs:246-256)
template <int D>
__device__ __forceinline__ Vec<D> reflection_direction(const Vec<D>& dir, const Vec<D>& normal_closer) {
    return normal_closer * -R(2.0) * dot(dir, normal_closer) + dir;
}

// threshold_direction_identity / threshold_direction_snell (surface.rs:259-288)
template <int D, bool GLASS = true>
__device__ __forceinline__ Vec<D> threshold_direction(const EuclSurface& sf, const Vec<D>& dir, const Vec<D>& normal_closer,
                                                      bool exiting, real from_theta, RefractionCache& rc) {
    if (!GLASS || sf.thr_op == EUCL_THR_IDENTITY) return dir;
    const Vec<D> normal = -normal_closer;
    const real modifier = exiting ? R(sf.thr_a) : R(1.0) / R(sf.thr_a);
    const real to_theta = cached_asin(rc, modifier * rc.sin_from);
    const real angle_delta = to_theta - from_theta;
    return general_rotation<D>(normal, dir, angle_delta, dir);
}

// The surface colour program (postfix) of surface `sf` at a hit.
template <int D>
#ifndef EUCL_INLINE_SURFACE_COLOR
#define EUCL_INLINE_SURFACE_COLOR 1 /* one call site per kernel; inlined: 3d_room shade R(7.45) -> R(7.14) ms, 4d_room R(4.48) -> R(4.26) */
#endif
#ifndef EUCL_ANGLE_REUSE
#define EUCL_ANGLE_REUSE 1
#endif
#if EUCL_INLINE_SURFACE_COLOR
#define EUCL_SC_INLINE __forceinline__
#else
#define EUCL_SC_INLINE __noinline__
#endif
__device__ EUCL_SC_INLINE Rgba surface_color(const SceneView& sv, const EuclSurface& sf, const Vec<D>& location,
                                     const Vec<D>& normal_raw, real cos_raw, real angle_raw_in, bool exiting, real time_millis) {
    // angle_raw = angle_between(direction, raw normal), evaluated by the intersect kernel; the angle to normal_closer is the
    // same number when entering and acos of the negated cosine when exiting (computed at most once per program)
#if EUCL_ANGLE_REUSE
    const real angle_raw = angle_raw_in;
    real angle_closer = angle_raw;
    bool have_closer = !exiting;
#else
    const real angle_raw = angle_from_cos(cos_raw);
    real angle_closer = R(0.0);
    bool have_closer = false;
    (void)angle_raw_in;
#endif
    Rgba stack[kColorStackMax];
    int sp = 0;
    for (int i = sf.color_first; i < sf.color_first + sf.color_len; ++i) {
        const EuclColorOp& op = sv.color_ops()[i];
        const int code = op.op;
        if (code == EUCL_COL_UNIFORM) { // surface.rs:425-429
            stack[sp++] = Rgba{R(op.f[0]), R(op.f[1]), R(op.f[2]), R(op.f[3])};
        } else if (code == EUCL_COL_ILLUM_GLOBAL) { // surface.rs:410-422
            const Rgba light{R(op.f[0]), R(op.f[1]), R(op.f[2]), R(op.f[3])}, dark{R(op.f[4]), R(op.f[5]), R(op.f[6]), R(op.f[7])};
            // angle_between(normal_closer, direction): same products and norms as (direction, normal_closer)
            if (!have_closer) {
                angle_closer = angle_from_cos(exiting ? -cos_raw : cos_raw);
                have_closer = true;
            }
            const real original_angle = angle_closer;
            const real angle = kPi - original_angle;
            const real ratio = angle / kFracPi2;
            stack[sp++] = combine_palette_color(dark, light, ratio);
        } else if (code == EUCL_COL_ILLUM_DIR) { // surface.rs:392-408
            const Rgba light{R(op.f[0]), R(op.f[1]), R(op.f[2]), R(op.f[3])}, dark{R(op.f[4]), R(op.f[5]), R(op.f[6]), R(op.f[7])};
            Vec<D> light_direction;
#pragma unroll
            for (int k = 0; k < D; ++k) light_direction[k] = R(op.f[8 + k]);
            Vec<D> normal = normal_raw;
            if (angle_raw > kFracPi2) normal = -normal; // angle_between(direction, raw normal)
            const real angle = angle_between(normal, -light_direction);
            const real ratio = R(1.0) - angle / kPi;
            stack[sp++] = combine_palette_color(dark, light, ratio);
        } else if (code == EUCL_COL_PERLIN_HUE) { // d3/entity/surface.rs:22-40
            const real size = R(op.f[0]), speed = R(op.f[1]);
            stack[sp++] = hue_to_rgba(perlin4(sv.perlin(), location[0] / size, location[1] / size, location[2] / size, time_millis * speed) * R(360.0));
        } else if (code == EUCL_COL_TEXTURE) { // surface.rs:536-542
            stack[sp++] = mapped_color<D>(sv, op.i0, location);
        } else { // EUCL_COL_BLEND, surface.rs:295-307
            const Rgba destination = stack[--sp];
            const Rgba source = stack[--sp];
            if (op.i0 == EUCL_BLEND_RATIO) stack[sp++] = combine_palette_color(source, destination, R(op.f[0]));
            else stack[sp++] = from_premultiplied(blend_pre(op.i0, into_premultiplied(source), into_premultiplied(destination)));
        }
    }
    return sp > 0 ? stack[sp - 1] : Rgba{R(0.0), R(0.0), R(0.0), R(0.0)};
}

// surface_color of a program that is one EUCL_COL_UNIFORM op (surface.rs:425-429): the op's constant
__device__ __forceinline__ Rgba uniform_surface_color(const SceneView& sv, const EuclSurface& sf) {
    const EuclColorOp& op = sv.color_ops()[sf.color_first];
    return Rgba{R(op.f[0]), R(op.f[1]), R(op.f[2]), R(op.f[3])};
}

} // namespace EUCL_NS
