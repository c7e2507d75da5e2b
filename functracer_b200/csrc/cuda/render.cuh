// render.cuh — the per-pixel render loop of FuncTracer (Shading.shade and everything below it,
// FuncTracer/Shading.fs:131-147) as ONE persistent CUDA kernel for sm_100a.
//
// Execution model (DESIGN.md "kernel"):
//   * persistent grid (a multiple of the SM count), every warp autonomous, no block barrier;
//   * work = 8x4-pixel blocks handed out by a per-GPU atomic queue; the pixels of a block are
//     dealt to lanes with ballot + popc (a warp-level scan), and a lane whose path ended is
//     re-armed at once with its next sample / pixel ("compaction by regeneration");
//   * every lane is a small state machine whose only expensive step is "trace my current ray":
//     the ray may be a primary / reflection ray (nearest hit) or a shadow ray (any hit).  One
//     loop iteration = one traced ray per lane, so the scene-intersection code exists ONCE in
//     the kernel (instruction-cache footprint) and lanes that missed do not wait for lanes that
//     shade.  F#'s recursion (getColourForRay, Shading.fs:131-139) becomes this iterative,
//     depth-bounded loop; the bounce "queue" is the lane's registers: zero HBM traffic;
//   * a lane owns a pixel for all of its samples: the blend happens in sample order exactly
//     like Array.average (Image.fs:112-116), no atomics;
//   * items (top-level objects) are visited in the reference's enumeration order (Ray.fs:34) so
//     ties break as Scene.closest does; a conservative bounding-sphere test per item skips
//     objects the ray's line cannot touch (the reference has no such index; it cannot change a
//     result because a culled item has no crossing at all on the line);
//   * the kernel is compiled in several feature-specialised variants (FEAT mask) so that a scene
//     only pays instruction-cache space for the primitive classes and shading terms it uses.
//
// Templated on R: float = product, double = FP64 verification build (compiled --fmad=false).
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../../include/ftb_rng.h"
#include "../../../include/functracer_b200.h"
#include "device_scene.h"
#include "lower.h"

namespace ftb {

#define FTB_DEV __device__ __forceinline__

// ---- scalar helpers -------------------------------------------------------------------------------
FTB_DEV float min_(float a, float b) { return fminf(a, b); }
FTB_DEV double min_(double a, double b) { return fmin(a, b); }
FTB_DEV float max_(float a, float b) { return fmaxf(a, b); }
FTB_DEV double max_(double a, double b) { return fmax(a, b); }
FTB_DEV float sqrt_(float x) { return sqrtf(x); }
FTB_DEV double sqrt_(double x) { return sqrt(x); }
FTB_DEV float abs_(float x) { return fabsf(x); }
FTB_DEV double abs_(double x) { return fabs(x); }
FTB_DEV float floor_(float x) { return floorf(x); }
FTB_DEV double floor_(double x) { return floor(x); }
// The next representable number above a finite x >= +0.
FTB_DEV float nextUp(float x) { return __int_as_float(__float_as_int(x) + 1); }
FTB_DEV double nextUp(double x) { return __longlong_as_double(__double_as_longlong(x) + 1); }
// System.Math.Pow semantics that matter to specularShader (Shading.fs:85-87): a negative base with an integral exponent
// gives +-|x|^y (sign by parity), with a non-integral exponent NaN.  Written out so that the product build can use the
// hardware exp2/log2 path (-use_fast_math) without losing that quirk.
FTB_DEV float pow_(float x, float y)
{
#ifdef FTB_FAST_MATH
    if (x >= 0.0f) return __powf(x, y);
    const float yi = truncf(y);
    if (yi != y) return CUDART_NAN_F;
    const float r = __powf(-x, y);
    return (((int)yi) & 1) ? -r : r;
#else
    return powf(x, y);
#endif
}
FTB_DEV double pow_(double x, double y) { return pow(x, y); }
FTB_DEV float acos_(float x) { return acosf(x); }
FTB_DEV double acos_(double x) { return acos(x); }
FTB_DEV float asin_(float x) { return asinf(x); }
FTB_DEV double asin_(double x) { return asin(x); }
FTB_DEV float atan2_(float y, float x) { return atan2f(y, x); }
FTB_DEV double atan2_(double y, double x) { return atan2(y, x); }
FTB_DEV float sin_(float x) { return sinf(x); }
FTB_DEV double sin_(double x) { return sin(x); }
FTB_DEV float cos_(float x) { return cosf(x); }
FTB_DEV double cos_(double x) { return cos(x); }
FTB_DEV float tan_(float x) { return tanf(x); }
FTB_DEV double tan_(double x) { return tan(x); }
template <typename R>
FTB_DEV R inf_();
template <>
FTB_DEV float inf_<float>() { return CUDART_INF_F; }
template <>
FTB_DEV double inf_<double>() { return CUDART_INF; }
template <typename R>
FTB_DEV R nan_();
template <>
FTB_DEV float nan_<float>() { return CUDART_NAN_F; }
template <>
FTB_DEV double nan_<double>() { return CUDART_NAN; }
template <typename R>
FTB_DEV R realmax_();  // System.Double.MaxValue of Shading.fs:25,36 in the working precision
template <>
FTB_DEV float realmax_<float>() { return 3.402823466e+38f; }
template <>
FTB_DEV double realmax_<double>() { return 1.7976931348623157e+308; }
// F# max/min on floats propagate NaN (SURVEY.md A.4)
template <typename R>
FTB_DEV R fsmax(R a, R b) { return (a != a || b != b) ? nan_<R>() : (a < b ? b : a); }
template <typename R>
FTB_DEV R fsmin(R a, R b) { return (a != a || b != b) ? nan_<R>() : (a < b ? a : b); }

// ---- CommonTypes.fs ---------------------------------------------------------------------------------
template <typename R>
struct Vec {
    R x, y, z;
};
template <typename R>
FTB_DEV Vec<R> mk(R x, R y, R z) { Vec<R> v; v.x = x; v.y = y; v.z = z; return v; }
template <typename R>
FTB_DEV Vec<R> operator+(Vec<R> a, Vec<R> b) { return mk<R>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename R>
FTB_DEV Vec<R> operator-(Vec<R> a, Vec<R> b) { return mk<R>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename R>
FTB_DEV Vec<R> operator-(Vec<R> a) { return mk<R>(-a.x, -a.y, -a.z); }
template <typename R>
FTB_DEV Vec<R> operator*(R s, Vec<R> v) { return mk<R>(s * v.x, s * v.y, s * v.z); }
template <typename R>
FTB_DEV R dot(Vec<R> a, Vec<R> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename R>
FTB_DEV Vec<R> cross(Vec<R> a, Vec<R> b) { return mk<R>(a.y * b.z - a.z * b.y, b.x * a.z - b.z * a.x, a.x * b.y - a.y * b.x); }  // CommonTypes.fs:17-18
template <typename R>
FTB_DEV R length(Vec<R> v) { return sqrt_(dot(v, v)); }
template <typename R>
FTB_DEV Vec<R> normalise(Vec<R> v)  // CommonTypes.fs:63-67
{
    R l = length(v);
    if (l < R(0.0000001)) return v;
    return (R(1) / l) * v;
}
template <typename R>
FTB_DEV Vec<R> reflect(Vec<R> n, Vec<R> v) { return v - (R(2) * dot(v, n)) * n; }  // :72
// CommonTypes.fs:74-75.  In FP32 the dot product of two normalised vectors exceeds 1 by an ulp whenever the angle is
// below ~3e-4 rad and acos would poison the pixel with NaN; in the reference's doubles that needs an angle below
// ~1e-8 rad, i.e. it does not happen.  The product build clamps, the verification build stays literal.
template <typename R>
FTB_DEV R angleBetween(Vec<R> a, Vec<R> b)
{
    R c = dot(normalise(a), normalise(b));
    if constexpr (sizeof(R) == 4) c = min_(R(1), max_(R(-1), c));
    return acos_(c);
}
template <typename R>
FTB_DEV Vec<R> perpendicularComponent(Vec<R> a, Vec<R> b) { Vec<R> na = normalise(a); return b - dot(b, na) * na; }  // :77-79

// ---- packed FP32 (sm_100: FADD2 / FMUL2 / FFMA2) -------------------------------------------------------------------
// Blackwell's FMA pipe takes two FP32 operations in one instruction when the operands sit in aligned register pairs
// (PTX add / mul / fma .f32x2); a pair built from twice the same scalar costs nothing, SASS has a broadcast operand form.
// Each half is rounded exactly like the scalar instruction.  The kernel is bounded by issue slots and dependent-issue
// latency, not by the pipe, so the two halves of a pair are work that would otherwise be two instructions of one chain
// after the other: the bound tests of two neighbouring items, origin and direction of a ray under the same matrix row.
// FP32 product build only; the FP64 verification build keeps the literal scalar forms.
typedef unsigned long long F2;  // two floats in one aligned register pair: lo = first, hi = second
FTB_DEV F2 pk2(float lo, float hi) { return ((F2)__float_as_uint(hi) << 32) | (F2)__float_as_uint(lo); }
FTB_DEV float lo2(F2 v) { return __uint_as_float((unsigned)v); }
FTB_DEV float hi2(F2 v) { return __uint_as_float((unsigned)(v >> 32)); }
FTB_DEV F2 add2(F2 a, F2 b) { F2 r; asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
FTB_DEV F2 sub2(F2 a, F2 b) { F2 r; asm("sub.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
FTB_DEV F2 mul2(F2 a, F2 b) { F2 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
FTB_DEV F2 fma2(F2 a, F2 b, F2 c) { F2 r; asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
FTB_DEV F2 dup2(float x) { return pk2(x, x); }

// Where the packed forms are used, per variant (measured, profiles/r2aa_packed_fp32_ab.txt):
//   the common-origin table two items per step: every FP32 variant (repeat -4.3 %, house -2.0 %, night-house -3.7 %, hollow-sphere -1.9 %,
//   frames identical);
//   the general bound loop two items per step: the house-family variants (on top of the table: repeat -0.7 %, house -1.1 %, night-house
//   -1.5 %); hollow-sphere +2.8 %, moon +2.3 %, the 960-triangle mesh +3.4 % with it (their unrolled compare loops already overlap the items);
//   origin and direction through a matrix row as one pair: the variants of the simple scenes (moon -1.3 %); it costs the CSG variants
//   72 bytes of spills for nothing (repeat +0.7 %, house -0.3 %, hollow-sphere +0.5 %).
template <typename R, unsigned FEAT> struct PackedBounds { static constexpr bool value = sizeof(R) == 4 && (FEAT & (FT_PAIRG | FT_CSGN)) != 0; };
// Per-tile item masks (DevFrame::tile_items) for primary rays: only in the variants compiled with FT_TMASK (the Makefile's
// F32_TMASK_FEATS).  The extra path costs the house-family kernel 5.5-7.3 % whether or not a frame has masks
// (profiles/r7a_tile_items_ab.txt), so it lives in a second instance of that variant, which api.cu launches only for frames whose
// masks drop enough of phase A's candidates (repeat -6.0 %); every other frame runs the plain instance, which has no such path.
template <typename R, unsigned FEAT> struct TileMasks { static constexpr bool value = sizeof(R) == 4 && (FEAT & FT_TMASK) != 0; };
template <typename R, unsigned FEAT> struct PackedXform { static constexpr bool value = sizeof(R) == 4 && (FEAT & (FT_CUBE | FT_ROUND | FT_MESH | FT_CSG | FT_CSGN)) == 0; };

template <typename R>
struct Ray {
    Vec<R> o, d;
};

template <typename R>
FTB_DEV typename V4<R>::type ldg4(const typename V4<R>::type* p) { return __ldg(p); }
template <>
FTB_DEV double4 ldg4<double>(const double4* p)
{
    const double2* q = reinterpret_cast<const double2*>(p);
    double2 a = __ldg(q), b = __ldg(q + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}

// world -> model with the leaf's composed matrix (Transform.fs:85, matrices pre-multiplied on the host)
template <bool PACK, typename R>
FTB_DEV Ray<R> toModel(const DevScene<R>& S, int leaf, bool identity, const Ray<R>& r)
{
    if (identity) return r;
    typedef typename V4<R>::type R4;
    R4 r0 = ldg4<R>(S.leaf_w2m + 3 * leaf), r1 = ldg4<R>(S.leaf_w2m + 3 * leaf + 1), r2 = ldg4<R>(S.leaf_w2m + 3 * leaf + 2);
    Ray<R> m;
    if constexpr (PACK) {
        // origin and direction go through a matrix row together: (o.c, d.c) pairs against the row's broadcast elements, the
        // translation as the origin half's first addend: 9 FFMA2 instead of 21 scalar operations (sum order w + x + y + z)
        const F2 px = pk2(r.o.x, r.d.x), py = pk2(r.o.y, r.d.y), pz = pk2(r.o.z, r.d.z);
        const F2 m0 = fma2(dup2(r0.z), pz, fma2(dup2(r0.y), py, fma2(dup2(r0.x), px, pk2(r0.w, 0.0f))));
        const F2 m1 = fma2(dup2(r1.z), pz, fma2(dup2(r1.y), py, fma2(dup2(r1.x), px, pk2(r1.w, 0.0f))));
        const F2 m2 = fma2(dup2(r2.z), pz, fma2(dup2(r2.y), py, fma2(dup2(r2.x), px, pk2(r2.w, 0.0f))));
        m.o = mk<R>(lo2(m0), lo2(m1), lo2(m2));
        m.d = mk<R>(hi2(m0), hi2(m1), hi2(m2));
    } else {
        m.o = mk<R>(r0.x * r.o.x + r0.y * r.o.y + r0.z * r.o.z + r0.w, r1.x * r.o.x + r1.y * r.o.y + r1.z * r.o.z + r1.w,
                    r2.x * r.o.x + r2.y * r.o.y + r2.z * r.o.z + r2.w);
        m.d = mk<R>(r0.x * r.d.x + r0.y * r.d.y + r0.z * r.d.z, r1.x * r.d.x + r1.y * r.d.y + r1.z * r.d.z,
                    r2.x * r.d.x + r2.y * r.d.y + r2.z * r.d.z);
    }
    return m;
}

// ---- per-lane work counters (stats kernels only) -----------------------------------------------------
template <bool STATS>
struct Counters {
    FTB_DEV void add(int, unsigned = 1) {}
    FTB_DEV unsigned get(int) const { return 0; }
};
template <>
struct Counters<true> {
    unsigned int c[ST_COUNT];
    FTB_DEV Counters()
    {
#pragma unroll
        for (int i = 0; i < ST_COUNT; ++i) c[i] = 0;
    }
    FTB_DEV void add(int slot, unsigned n = 1) { c[slot] += n; }
    FTB_DEV unsigned get(int slot) const { return c[slot]; }
};

// ---- Math.quadratic (Math.fs:4-10): far ("+") root first ----------------------------------------------
template <typename R>
FTB_DEV bool quadratic(R a, R b, R c, R& t0, R& t1)
{
    R discriminant = b * b - R(4) * a * c;
    if (discriminant < R(0)) return false;
    R sq = sqrt_(discriminant);
    R twoa = R(2) * a;
    t0 = (-b + sq) / twoa;
    t1 = (-b - sq) / twoa;
    return true;
}

// Roots of the canonical quadrics  x^2 + wy y^2 + z^2 = k  along o + t d  (sphere wy = 1, k = 1, Sphere.fs:11-15;
// cylinder wy = 0, k = 1, Cylinder.fs:9-13; cone about its apex wy = -1, k = 0, Cone.fs:9-15), far root first
// like Math.quadratic.
//   double (verification build): the reference's literal a, b, c and Math.quadratic, operation for operation.
//   float (product build): the same roots from a re-centred origin.  With o far from the surface (the moon
//   scene's camera is 50 model units from a unit sphere) b^2 and 4ac agree in their leading digits and FP32
//   loses the discriminant (error ~ 1e-4 in t: more than the 1e-4 shadow-ray offset of Shading.fs:111, i.e.
//   shadow acne).  Sliding the origin to the point of closest approach to the model origin, o' = o + ts d,
//   makes |o'| ~ the object's size and b ~ 0; t = t' + ts.  Same real-arithmetic roots, FP32-safe rounding.
template <int KIND, typename R>  // KIND: 0 sphere, 1 cylinder, 2 cone (o already relative to the apex)
FTB_DEV bool quadricRoots(Vec<R> o, Vec<R> d, R& t0, R& t1)
{
    if constexpr (sizeof(R) == 8) {
        R a, b, c;
        if (KIND == 0) { a = dot(d, d); b = R(2) * dot(o, d); c = dot(o, o) - R(1); }
        else if (KIND == 1) { a = d.x * d.x + d.z * d.z; b = R(2) * (o.x * d.x + o.z * d.z); c = o.x * o.x + o.z * o.z - R(1); }
        else { a = d.x * d.x + d.z * d.z - d.y * d.y; b = R(2) * (o.x * d.x + o.z * d.z - o.y * d.y); c = o.x * o.x + o.z * o.z - o.y * o.y; }
        return quadratic(a, b, c, t0, t1);
    } else {
        const R wy = KIND == 0 ? R(1) : (KIND == 1 ? R(0) : R(-1));
        const R k = KIND == 2 ? R(0) : R(1);
        const R dd = dot(d, d);
        const R ts = dd > R(0) ? -dot(o, d) / dd : R(0);
        const Vec<R> oc = mk<R>(fmaf(ts, d.x, o.x), fmaf(ts, d.y, o.y), fmaf(ts, d.z, o.z));
        const R a = d.x * d.x + d.z * d.z + wy * d.y * d.y;
        const R b = R(2) * (oc.x * d.x + oc.z * d.z + wy * oc.y * d.y);
        const R c = (oc.x * oc.x + oc.z * oc.z + wy * oc.y * oc.y) - k;
        if (!quadratic(a, b, c, t0, t1)) return false;
        t0 += ts; t1 += ts;
        return true;
    }
}

// Plane.intersect for Plane(Zero, unitY) in the leaf's frame (Plane.fs:9-20).  Returns false if no hit.
template <typename R>
FTB_DEV bool planeT(const Ray<R>& r, R& t, Vec<R>& p)
{
    const R eps = R(0.0000001);
    R num = -r.o.y;
    R denom = r.d.y;
    t = num / denom;
    if (abs_(denom) < eps) {  // parallel: the reference answers t = 0, p = o when the origin is on or below the plane (Plane.fs:13-16)
        if (!(num < eps)) return false;
        t = R(0);  // p below = o + 0 d = o for every finite d
    }
    p = mk<R>(r.o.x + t * r.d.x, r.o.y + t * r.d.y, r.o.z + t * r.d.z);
    return true;
}

// Triangle.fs:43-66 with e1, e2 precomputed; returns t or false.  rows = {v0, e1, e2}.
template <typename R>
FTB_DEV bool triangleT(const typename V4<R>::type* rows, const Ray<R>& ray, R& t, typename V4<R>::type& a0, typename V4<R>::type& a1)
{
    typedef typename V4<R>::type R4;
    const R epsilon = R(0.0000001);
    a0 = ldg4<R>(rows); a1 = ldg4<R>(rows + 1);
    const R4 a2 = ldg4<R>(rows + 2);
    Vec<R> v0 = mk<R>(a0.x, a0.y, a0.z), edge1 = mk<R>(a1.x, a1.y, a1.z), edge2 = mk<R>(a2.x, a2.y, a2.z);
    Vec<R> h = cross(ray.d, edge2);
    R a = dot(edge1, h);
    if (a > -epsilon && a < epsilon) return false;
    R f = R(1) / a;
    Vec<R> s = ray.o - v0;
    R u = f * dot(s, h);
    if (u < R(0) || u > R(1)) return false;
    Vec<R> q = cross(s, edge1);
    R v = dot(f * ray.d, q);
    if (v < R(0) || u + v > R(1)) return false;
    t = dot(f * edge2, q);
    return t > epsilon;
}


// Ray vs. one child box of a BVH node: entry distance, or +inf when the box cannot hold a hit with
// 0 <= t <= tmax.  fmin / fmax drop the NaNs that 0 * inf produces for rays parallel to a slab; the exit
// distance is widened by 4 ulp so that rounding can never reject a box that really holds the hit.
template <typename R>
FTB_DEV R boxEntry(R lx, R ly, R lz, R hx, R hy, R hz, const Vec<R>& o, const Vec<R>& inv, R tmax)
{
    const R x0 = (lx - o.x) * inv.x, x1 = (hx - o.x) * inv.x;
    const R y0 = (ly - o.y) * inv.y, y1 = (hy - o.y) * inv.y;
    const R z0 = (lz - o.z) * inv.z, z1 = (hz - o.z) * inv.z;
    const R tn = max_(max_(min_(x0, x1), min_(y0, y1)), max_(min_(z0, z1), R(0)));
    R tf = min_(min_(max_(x0, x1), max_(y0, y1)), min_(max_(z0, z1), tmax));
    tf = tf * (sizeof(R) == 4 ? R(1.0000005) : R(1.0000000000000009)) + (sizeof(R) == 4 ? R(1e-30) : R(0));
    return tn <= tf ? tn : inf_<R>();
}

// A node record = 4 rows (64 bytes, one piece of one cache line): three rows of boxes (below) and the two child links in the
// first two lanes of the fourth (FP32: the ints' bits; FP64: their values): a node visit reads one aligned 64-byte piece instead of 48 bytes
// of boxes here and 8 bytes of links in another array (measured with boxEntry2, profiles/r2ac_mesh_nodes_ab.txt: 960 triangles -2.4 %,
// 9.6 k -2.8 %, 355 k -7.7 %; prefetching both children's records from the packet walk: +12 % on the 355 k mesh, dropped).
template <typename R>
FTB_DEV int2 nodeLinks(const typename V4<R>::type& row)
{
    if constexpr (sizeof(R) == 4) return make_int2(__float_as_int(row.x), __float_as_int(row.y));
    else return make_int2((int)row.x, (int)row.y);
}
// Both child boxes of a node at once.  Node layout: b0 = (L.lo.x, R.lo.x, L.hi.x, R.hi.x), b1 and b2 the same for y and z, so that
// the left and the right box's slab distances along an axis are the two halves of one packed subtract and one packed multiply
// (12 FADD2 / FMUL2 instead of 24 scalar operations per node; each half rounds exactly like boxEntry's scalar form).
template <typename R>
FTB_DEV void boxEntry2(const typename V4<R>::type& b0, const typename V4<R>::type& b1, const typename V4<R>::type& b2, const Vec<R>& o, const Vec<R>& inv, R tmax, R& tl, R& tr)
{
    if constexpr (sizeof(R) == 4) {
        const F2 ox = dup2(o.x), oy = dup2(o.y), oz = dup2(o.z), ix = dup2(inv.x), iy = dup2(inv.y), iz = dup2(inv.z);
        const F2 x0 = mul2(sub2(pk2(b0.x, b0.y), ox), ix), x1 = mul2(sub2(pk2(b0.z, b0.w), ox), ix);
        const F2 y0 = mul2(sub2(pk2(b1.x, b1.y), oy), iy), y1 = mul2(sub2(pk2(b1.z, b1.w), oy), iy);
        const F2 z0 = mul2(sub2(pk2(b2.x, b2.y), oz), iz), z1 = mul2(sub2(pk2(b2.z, b2.w), oz), iz);
        const R tnl = max_(max_(min_(lo2(x0), lo2(x1)), min_(lo2(y0), lo2(y1))), max_(min_(lo2(z0), lo2(z1)), R(0)));
        const R tnr = max_(max_(min_(hi2(x0), hi2(x1)), min_(hi2(y0), hi2(y1))), max_(min_(hi2(z0), hi2(z1)), R(0)));
        const R tfl = min_(min_(max_(lo2(x0), lo2(x1)), max_(lo2(y0), lo2(y1))), min_(max_(lo2(z0), lo2(z1)), tmax));
        const R tfr = min_(min_(max_(hi2(x0), hi2(x1)), max_(hi2(y0), hi2(y1))), min_(max_(hi2(z0), hi2(z1)), tmax));
        const F2 tf = fma2(pk2(tfl, tfr), dup2(1.0000005f), dup2(1e-30f));
        tl = tnl <= lo2(tf) ? tnl : inf_<R>();
        tr = tnr <= hi2(tf) ? tnr : inf_<R>();
    } else {
        tl = boxEntry<R>(b0.x, b1.x, b2.x, b0.z, b1.z, b2.z, o, inv, tmax);
        tr = boxEntry<R>(b0.y, b1.y, b2.y, b0.w, b1.w, b2.w, o, inv, tmax);
    }
}

// Nearest / any hit of a mesh (Scene.fs:9 BspMesh), one private walk per lane: the device's BVH over the mesh's triangles, front to back,
// culled against the best t so far.  Result = BspMesh.intersect (BspMesh.fs:67-76) followed by Scene.closest
// (Scene.fs:112-116): smallest t, and among equal t the triangle that comes first in the reference's
// right-before-left enumeration (`seq`).  limit: only hits with t < limit count (ties with earlier items lose).
// Used for small meshes (DevScene::mesh_packet == 0), whose walks are short and hardly diverge; see packetMesh for the large ones.
template <typename R, bool STATS>
FTB_DEV bool intersectMesh(const DevScene<R>& S, int root, const Ray<R>& r, R limit, bool any, R& bt, int& btri, bool& overflow, Counters<STATS>& cn)
{
    typedef typename V4<R>::type R4;
    int stack[kBspStack];
    R stackT[kBspStack];
    int sp = 0;
    int link = root;
    bt = limit;
    btri = -1;
    int bseq = 0x7fffffff;
    const Vec<R> inv = mk<R>(R(1) / r.d.x, R(1) / r.d.y, R(1) / r.d.z);
    for (;;) {
        // ---- descend: inner nodes until a leaf is reached (every lane of the warp is doing box tests here) ----
        while (link >= 0) {
            cn.add(ST_BSP_NODES);
            const R4 b0 = ldg4<R>(S.bvh_node + 4 * link), b1 = ldg4<R>(S.bvh_node + 4 * link + 1), b2 = ldg4<R>(S.bvh_node + 4 * link + 2);
            const int2 ch = nodeLinks<R>(ldg4<R>(S.bvh_node + 4 * link + 3));
            R tl, tr;
            boxEntry2<R>(b0, b1, b2, r.o, inv, bt, tl, tr);
            const bool hl = tl < inf_<R>(), hr = tr < inf_<R>();
            if (hl && hr) {
                const bool leftFirst = tl <= tr;
                if (sp < kBspStack) { stack[sp] = leftFirst ? ch.y : ch.x; stackT[sp] = leftFirst ? tr : tl; ++sp; } else overflow = true;
                link = leftFirst ? ch.x : ch.y;
            } else if (hl || hr) {
                link = hl ? ch.x : ch.y;
            } else {
                link = 0x7fffffff;  // nothing below: pop
                break;
            }
        }
        // ---- leaf: a run of <= 7 triangles ---------------------------------------------------------------------------
        if (link < 0) {
            const int code = ~link, first = code >> 3, count = code & 7;
            for (int i = 0; i < count; ++i) {
                R t; R4 a0, a1;
                cn.add(ST_TRI_TESTS_IN_MESH);
                if (triangleT<R>(S.bvh_tris + 3 * (first + i), r, t, a0, a1)) {
                    const int seq = (int)a0.w;
                    if (t < bt || (t == bt && btri >= 0 && seq < bseq)) { bt = t; bseq = seq; btri = (int)a1.w; }
                }
            }
            if (any && btri >= 0) return true;
        }
        // ---- pop the nearest postponed subtree that can still hold a closer (or tying) hit -------------------------
        link = 0x7fffffff;
        while (sp > 0) {
            --sp;
            if (stackT[sp] <= bt) { link = stack[sp]; break; }
        }
        if (link == 0x7fffffff) break;
    }
    return btri >= 0;
}

// Nearest / any hit of a mesh (Scene.fs:9 BspMesh) for ALL rays of a warp at once: the device's BVH over the mesh's
// triangles, culled against each lane's best t so far.  Result per lane = BspMesh.intersect (BspMesh.fs:67-76) followed by
// Scene.closest (Scene.fs:112-116): smallest t, and among equal t the triangle that comes first in the reference's
// right-before-left enumeration (`seq`).  limit: only hits with t < limit count.
//   The rays a warp traces together come from a run of <= 8 neighbouring pixels of one block (primary rays through the
//   same few pixels, shadow rays from neighbouring surface points towards the same light), so they walk nearly the same
//   nodes.  The walk is therefore the WARP's: one link, one stack (in shared memory, 256 bytes per warp) and one node /
//   triangle fetch (the same address in every lane: a broadcast) per step; a node is entered when ANY lane's ray can still
//   find a closer hit in it (a ballot), the child that more lanes meet first is walked first, and every lane tests its own
//   ray against the boxes and triangles on the way.  Against 32 private walks (previous kernel: 11 of 32 lanes active in
//   the box tests, 5 in the triangle tests, a 64-entry stack per lane in local memory) there is no divergence in the
//   control flow and no per-lane stack traffic; the price is that a lane also sits through the nodes only its neighbours
//   need.  Which triangle wins does not depend on the order of the walk (min t, then min seq), so the picture cannot change.
//   want: this lane's ray takes part; mask: the lanes that execute this call (all of them must).
template <typename R, bool STATS>
FTB_DEV void packetMesh(const DevScene<R>& S, int root, const Ray<R>& r, R limit, bool any, bool want, unsigned mask, int* wstack, R& bt, int& btri, Counters<STATS>& cn)
{
    typedef typename V4<R>::type R4;
    bt = limit;
    btri = -1;
    bool live = want;
    if (!__any_sync(mask, live)) return;
    int bseq = 0x7fffffff;
    int sp = 0;
    int link = root;  // warp-uniform from here on (the item, hence the mesh, is the same in every lane)
    const Vec<R> inv = mk<R>(R(1) / r.d.x, R(1) / r.d.y, R(1) / r.d.z);
    const int lane = threadIdx.x & 31;
    for (;;) {
        // ---- descend: inner nodes until a leaf is reached ---------------------------------------------------------------
        while (link >= 0 && link != 0x7fffffff) {
            const R4 b0 = ldg4<R>(S.bvh_node + 4 * link), b1 = ldg4<R>(S.bvh_node + 4 * link + 1), b2 = ldg4<R>(S.bvh_node + 4 * link + 2);
            const int2 ch = nodeLinks<R>(ldg4<R>(S.bvh_node + 4 * link + 3));
            R tl = inf_<R>(), tr = inf_<R>();
            if (live) {
                cn.add(ST_BSP_NODES);
                boxEntry2<R>(b0, b1, b2, r.o, inv, bt, tl, tr);
            }
            const bool hl = tl < inf_<R>(), hr = tr < inf_<R>();
            const unsigned ml = __ballot_sync(mask, hl), mr = __ballot_sync(mask, hr);
            if (ml && mr) {
                // the child that more lanes reach first goes first
                const unsigned leftFirst = __ballot_sync(mask, hl && (!hr || tl <= tr));
                const bool lf = 2 * __popc(leftFirst) >= __popc(ml | mr);
                if (lane == (__ffs(mask) - 1)) wstack[sp] = lf ? ch.y : ch.x;
                ++sp;
                link = lf ? ch.x : ch.y;
            } else if (ml | mr) {
                link = ml ? ch.x : ch.y;
            } else {
                link = 0x7fffffff;  // nothing below for anybody: pop
            }
        }
        // ---- leaf: a run of <= 7 triangles, every live lane tests its own ray against each ----------------------------------
        if (link < 0) {
            const int code = ~link, first = code >> 3, count = code & 7;
            for (int i = 0; i < count; ++i) {
                R t; R4 a0, a1;
                if (live) {
                    cn.add(ST_TRI_TESTS_IN_MESH);
                    if (triangleT<R>(S.bvh_tris + 3 * (first + i), r, t, a0, a1)) {
                        const int seq = (int)a0.w;
                        if (t < bt || (t == bt && btri >= 0 && seq < bseq)) { bt = t; bseq = seq; btri = (int)a1.w; }
                    }
                }
            }
            if (any) live = live && btri < 0;  // Scene.lightIsBocked: one hit is enough
            if (!__any_sync(mask, live)) return;
        }
        // ---- pop.  A postponed subtree that no lane can use any more is dropped at its first node (both boxes miss for everybody);
        // remembering per entry which lanes wanted it and from what distance, to drop it here, measured 7 % SLOWER on the 355 k mesh.
        if (sp == 0) break;
        --sp;
        __syncwarp(mask);
        link = wstack[sp];
        __syncwarp(mask);
    }
}

// ---- leaf intersection: calls sink.hit(t, sub) for every crossing, in the reference's order ---------
// sub: cube face 0..5 (Cube.fs:24), triangle index for meshes, else the leaf's payload.
// Which mesh walks a variant contains: the per-lane one (small meshes) unless the variant is specialised for large meshes, the
// warp-packet one if it asks for it; FT_ALL has both and DevScene::mesh_packet chooses.
template <unsigned FEAT> struct MeshWalks {
    static constexpr bool kPacket = (FEAT & FT_MESH) != 0 && (FEAT & FT_MESHPK) != 0;
    static constexpr bool kPerLane = (FEAT & FT_MESH) != 0 && ((FEAT & FT_MESHPK) == 0 || FEAT == (unsigned)FT_ALL);
};

// kw = the leaf's kind | identity << 8 (the low bits of leaf_meta.x).  Top-level items and single-leaf pair operands carry it in
// their item record (DevScene::items), so that the walk does not wait for the leaf's own record before it can branch on the
// kind: the chain of dependent loads per candidate is item -> matrix instead of item -> leaf record -> branch (measured: moon -4.5 %, sample -4 %, the house family -0.5 %, the 960-triangle mesh -1 %; hollow-sphere +2 %).
// Only triangles and meshes read their payload from the leaf record; the sub-id of the other kinds is not used downstream.
template <typename R>
FTB_DEV int leafKw(const DevScene<R>& S, int leaf) { return __ldg(&S.leaf_meta[leaf].x) & 0x1ff; }

template <typename R, unsigned FEAT, bool STATS, class Sink>
FTB_DEV void intersectLeaf(const DevScene<R>& S, int leaf, int kw, const Ray<R>& wr, Sink& sink, Counters<STATS>& cn)
{
    const int kind = kw & 0xff;
    const bool identity = (kw >> 8) & 1;
    const Ray<R> r = toModel<PackedXform<R, FEAT>::value, R>(S, leaf, identity, wr);
    cn.add(ST_LEAF0 + kind);
    if (!identity) cn.add(ST_XFORM);
    if (kind == LEAF_SPHERE) {  // Sphere.fs:11-21
        R t0, t1;
        if (quadricRoots<0>(r.o, r.d, t0, t1)) { sink.hit(t0, 0); sink.hit(t1, 0); }
        return;
    }
    if (kind == LEAF_PLANE) {  // Plane.fs:32-33
        R t; Vec<R> p;
        if (planeT(r, t, p)) sink.hit(t, 0);
        return;
    }
    if constexpr ((FEAT & FT_CUBE) != 0) {
        if (kind == LEAF_CUBE) {  // Cube.fs:17-25, the six squares in the cube's centred frame shifted by +.5
            const R eps = R(0.0000001);
            const R ox = r.o.x + R(0.5), oy = r.o.y + R(0.5), oz = r.o.z + R(0.5);
            // face f: plane coordinate w (origin wo, direction wd), offset k in {0,1}, in-face coords (a, b)
            // bottom/top: w = y, (a,b) = (x,z); left/right: w = x, (a,b) = (y,z); front/back: w = z, (a,b) = (x,y).
            // num/denom signs follow each square's own frame (DESIGN.md "cube"): bottom/top: num = k - w, denom = +wd;
            // left/right/front/back (rotated frames): num = w - k, denom = -wd.
#define FTB_CUBE_FACE(face, wo, wd, ao, ad, bo, bd, k, rotated)                                   \
            {                                                                                         \
                R num = (rotated) ? ((wo) - R(k)) : (R(k) - (wo));                                    \
                R denom = (rotated) ? -(wd) : (wd);                                                   \
                R t; bool ok = true;                                                                  \
                if (abs_(denom) < eps) { if (num < eps) t = R(0); else ok = false; }                  \
                else t = num / denom;                                                                 \
                if (ok) {                                                                             \
                    R pa = (ao) + t * (ad), pb = (bo) + t * (bd);                                     \
                    if ((pa >= R(0)) && (pa <= R(1)) && (pb >= R(0)) && (pb <= R(1))) sink.hit(t, face); \
                }                                                                                     \
            }
            FTB_CUBE_FACE(0, oy, r.d.y, ox, r.d.x, oz, r.d.z, 0, false)
            FTB_CUBE_FACE(1, oy, r.d.y, ox, r.d.x, oz, r.d.z, 1, false)
            FTB_CUBE_FACE(2, ox, r.d.x, oy, r.d.y, oz, r.d.z, 0, true)
            FTB_CUBE_FACE(3, ox, r.d.x, oy, r.d.y, oz, r.d.z, 1, true)
            FTB_CUBE_FACE(4, oz, r.d.z, ox, r.d.x, oy, r.d.y, 0, true)
            FTB_CUBE_FACE(5, oz, r.d.z, ox, r.d.x, oy, r.d.y, 1, true)
#undef FTB_CUBE_FACE
            return;
        }
    }
    if constexpr ((FEAT & FT_ROUND) != 0) {
        if (kind == LEAF_SQUARE) {  // Cube.fs:9-15
            R t; Vec<R> p;
            if (planeT(r, t, p) && (p.x >= R(0)) && (p.x <= R(1)) && (p.z >= R(0)) && (p.z <= R(1))) sink.hit(t, 0);
            return;
        }
        if (kind == LEAF_CIRCLE) {  // Cylinder.fs:22
            R t; Vec<R> p;
            if (planeT(r, t, p) && length(p) < R(1)) sink.hit(t, 0);
            return;
        }
        if (kind == LEAF_CYLINDER) {  // Cylinder.fs:8-20
            R t0, t1;
            if (quadricRoots<1>(r.o, r.d, t0, t1)) {
                R py = r.o.y + t0 * r.d.y;
                if (py >= R(0) && py <= R(1)) sink.hit(t0, 0);
                py = r.o.y + t1 * r.d.y;
                if (py >= R(0) && py <= R(1)) sink.hit(t1, 0);
            }
            return;
        }
        if (kind == LEAF_SOLIDCYL) {
            // Cylinder.solidCylinder (Cylinder.fs:25-29) = group [top; bottom; sides] as ONE leaf in the cylinder's frame: the
            // parts' own transforms are applied here exactly as Transform.transform would (Transform.fs:15-22, 85: row . v,
            // products summed left to right), so a solidCylinder costs one matrix and one leaf visit instead of three.
            {  // top = translate (0,1,0) circle: o' = (x, y - 1, z), d' = d
                Ray<R> q = r;
                q.o.y = r.o.y + R(-1);
                R t; Vec<R> p;
                if (planeT(q, t, p) && length(p) < R(1)) sink.hit(t, 0);
            }
            {  // bottom = rotate unitZ 180 circle: rows (c, -s, 0) (s, c, 0) (0, 0, 1) with the host's c = cos(-pi), s = sin(-pi)
                const R c = S.cyl_c, sn = S.cyl_s;
                Ray<R> q;
                q.o = mk<R>(c * r.o.x + (-sn) * r.o.y, sn * r.o.x + c * r.o.y, r.o.z);
                q.d = mk<R>(c * r.d.x + (-sn) * r.d.y, sn * r.d.x + c * r.d.y, r.d.z);
                R t; Vec<R> p;
                if (planeT(q, t, p) && length(p) < R(1)) sink.hit(t, 1);
            }
            R t0, t1;  // sides = cylinder (Cylinder.fs:8-20)
            if (quadricRoots<1>(r.o, r.d, t0, t1)) {
                R py = r.o.y + t0 * r.d.y;
                if (py >= R(0) && py <= R(1)) sink.hit(t0, 2);
                py = r.o.y + t1 * r.d.y;
                if (py >= R(0) && py <= R(1)) sink.hit(t1, 2);
            }
            return;
        }
        if (kind == LEAF_CONE) {  // Cone.fs:7-28
            R oy = r.o.y - R(1);
            R t0, t1;
            if (quadricRoots<2>(mk<R>(r.o.x, oy, r.o.z), r.d, t0, t1)) {
                R py = (oy + t0 * r.d.y) + R(1);
                if (py >= R(0) && py <= R(1)) sink.hit(t0, 0);
                py = (oy + t1 * r.d.y) + R(1);
                if (py >= R(0) && py <= R(1)) sink.hit(t1, 0);
            }
            return;
        }
    }
    if constexpr ((FEAT & FT_MESH) != 0) {
        if (kind == LEAF_TRIANGLE) {
            R t; typename V4<R>::type a0, a1;
            if (triangleT<R>(S.tris + 3 * __ldg(&S.leaf_meta[leaf].w), r, t, a0, a1)) sink.hit(t, 0);
            return;
        }
        if constexpr (Sink::kIsRay && MeshWalks<FEAT>::kPerLane) {
            if (kind == LEAF_MESH) {  // small meshes only (mesh_packet == 0): large ones are walked by the whole warp in traceScene
                R bt; int btri;
                if (intersectMesh<R, STATS>(S, __ldg(S.mesh_root + __ldg(&S.leaf_meta[leaf].w)), r, sink.limit, sink.any, bt, btri, sink.overflow, cn)) sink.hit(bt, btri);
                return;
            }
        }
    }
}

// ---- sinks ----------------------------------------------------------------------------------------------
constexpr int kIdSubShiftI = 22, kIdFlipI = 1 << 30, kIdLeafMaskI = (1 << 22) - 1;  // = kIdSubShift, kIdFlip, kIdLeafMask below
// Scene.closest (Scene.fs:112-116): smallest t >= 0, first in enumeration order on ties — and, with
// `limit` preset to maxDistance and `any` set, Scene.lightIsBocked (Scene.fs:119-121) for leaves whose
// surface has applyLighting = true: any hit with 0 <= t < maxDistance.
// The winner lives in one register: id = leaf | sub << 22 | flip << 30 (-1: none).  Variants with meshes (WIDE) keep the
// sub-id - a triangle index there - in a register of its own.  A hit site of the leaf intersectors is then two compares
// and two selects.
template <typename R, bool WIDE>
struct RaySink {
    static constexpr bool kIsRay = true;
    R limit;
    int id, sub;  // sub: WIDE only (dead otherwise)
    int cur;  // leaf being intersected
    bool any;
    bool overflow;
    FTB_DEV void hit(R ht, int hsub)
    {
        if (ht >= R(0) && ht < limit) take(ht, cur, hsub, false);
    }
    FTB_DEV void take(R ht, int leaf, int hsub, bool flip)
    {
        limit = ht;
        id = leaf | (WIDE ? 0 : ((hsub & 7) << kIdSubShiftI)) | (flip ? (int)kIdFlipI : 0);
        if (WIDE) sub = hsub;
    }
    FTB_DEV void block(int leaf) { id = leaf; }  // Scene.lightIsBocked: which leaf does not matter
    FTB_DEV bool found() const { return id >= 0; }
    FTB_DEV int leaf() const { return id < 0 ? -1 : (id & (WIDE ? 0x3fffffff : (int)kIdLeafMaskI)); }
    FTB_DEV int subId() const { return WIDE ? sub : ((id >> kIdSubShiftI) & 7); }
    FTB_DEV int flipped() const { return (id >> 30) & 1; }
    FTB_DEV bool done() const { return any && found(); }
};
// A mesh item's answer, found after the other items of its batch (traceScene): it also wins a tie in t against a winner
// that comes LATER in the enumeration, as Scene.closest's stable sort would have it.
template <typename R, bool WIDE>
FTB_DEV void meshHit(RaySink<R, WIDE>& best, int& bestItem, int item, int leaf, R ht, int tri)
{
    if (ht >= R(0) && (ht < best.limit || (ht == best.limit && best.found() && item < bestItem))) {
        best.take(ht, leaf, tri, false); bestItem = item;
    }
}
// CSG operand: append to the per-ray hit stack.
template <typename R>
struct HitRec {
    R t;
    unsigned int id;  // leaf (0..21) | sub (22..24) | flip (30) | side B (31)
};
constexpr unsigned kIdFlip = 1u << 30, kIdSideB = 1u << 31, kIdSubShift = 22, kIdLeafMask = (1u << 22) - 1;
template <typename R>
struct ListSink {
    static constexpr bool kIsRay = false;
    HitRec<R>* stack;
    int top;
    int cur;
    bool overflow;
    FTB_DEV void hit(R ht, int hsub)
    {
        if (top < kHitCap) { stack[top].t = ht; stack[top].id = (unsigned)cur | ((unsigned)(hsub & 7) << kIdSubShift); ++top; }
        else overflow = true;
    }
    FTB_DEV bool done() const { return false; }
};

// Csg.fs:19-72 as a lookup: key = hitB * 4 + inA * 2 + inB -> 0 Take, 1 Discard, 2 Flip (2 bits each).
FTB_DEV unsigned csgRuleTable(int op)
{
    // keys: A-hit (inA,inB): 0 (F,F) OutsideIntoA, 1 (F,T) BIntoAB, 2 (T,F) AIntoOutside, 3 (T,T) ABleaveA
    //       B-hit:           4 (F,F) OutsideIntoB, 5 (F,T) BIntoOutside, 6 (T,F) AIntoAB, 7 (T,T) ABleaveB
#define FTB_RULES(k0, k1, k2, k3, k4, k5, k6, k7) ((k0) | ((k1) << 2) | ((k2) << 4) | ((k3) << 6) | ((k4) << 8) | ((k5) << 10) | ((k6) << 12) | ((k7) << 14))
    switch (op) {
    case OP_UNION: return FTB_RULES(0u, 1u, 0u, 1u, 0u, 0u, 1u, 1u);      // Csg.fs:19-25
    case OP_SUBTRACT: return FTB_RULES(0u, 1u, 0u, 1u, 1u, 1u, 2u, 2u);   // :27-33
    case OP_INTERSECT: return FTB_RULES(1u, 0u, 1u, 0u, 1u, 1u, 0u, 0u);  // :35-44
    default: return FTB_RULES(0u, 2u, 0u, 2u, 0u, 0u, 2u, 2u);            // exclude :46-55
    }
#undef FTB_RULES
}

// Evaluates one CSG program (Csg.constructedSolid, Csg.fs:74-94) on the per-ray hit stack.
// On return stack[0..n) holds the root's crossings sorted by t.
template <typename R, unsigned FEAT, bool STATS>
FTB_DEV int evalCsg(const DevScene<R>& S, int opFirst, int opCount, const Ray<R>& wr, HitRec<R>* stack, bool& overflow, Counters<STATS>& cn)
{
    int counts[kMaxLists];
    int nlists = 0;
    ListSink<R> sink;
    sink.stack = stack; sink.top = 0; sink.overflow = false;
    for (int i = 0; i < opCount; ++i) {
        const int2 op = __ldg(S.ops + opFirst + i);
        if (op.x == OP_LEAF) {
            int start = sink.top;
            sink.cur = op.y;
            intersectLeaf<R, FEAT & ~FT_MESH, STATS>(S, op.y, leafKw(S, op.y), wr, sink, cn);  // meshes are rejected as CSG operands at lowering
            if (nlists < kMaxLists) counts[nlists++] = sink.top - start; else sink.overflow = true;
        } else if (op.x == OP_GROUP) {
            int c = 0;
            for (int k = 0; k < op.y; ++k) c += counts[nlists - 1 - k];
            nlists -= op.y - 1;
            counts[nlists - 1] = c;
        } else if (op.x == OP_EMPTY) {
            if (nlists < kMaxLists) counts[nlists++] = 0; else sink.overflow = true;
        } else {
            cn.add(ST_CSG_OPS);
            const int nb = counts[nlists - 1], na = counts[nlists - 2];
            const int start = sink.top - na - nb, end = sink.top;
            for (int k = start + na; k < end; ++k) stack[k].id |= kIdSideB;
            // Seq.sortBy (stable): insertion sort, strict '<' so equal keys keep A-before-B order
            for (int k = start + 1; k < end; ++k) {
                HitRec<R> x = stack[k];
                int j = k;
                while (j > start && x.t < stack[j - 1].t) { stack[j] = stack[j - 1]; --j; }
                stack[j] = x;
            }
            const unsigned rules = csgRuleTable(op.x);
            bool inA = false, inB = false;
            int out = start;
            for (int k = start; k < end; ++k) {
                HitRec<R> x = stack[k];
                const bool hitB = (x.id & kIdSideB) != 0;
                const unsigned rule = (rules >> (2 * ((hitB ? 4 : 0) + (inA ? 2 : 0) + (inB ? 1 : 0)))) & 3u;
                if (hitB) inB = !inB; else inA = !inA;
                x.id &= ~kIdSideB;
                if (rule == 2u) x.id ^= kIdFlip;
                if (rule != 1u) stack[out++] = x;
            }
            sink.top = out;
            --nlists;
            counts[nlists - 1] = out - start;
        }
    }
    overflow = overflow || sink.overflow;
    return sink.top;
}

// A nearest/any query against one CSG item through the general program.  Out of line: it is the rare path for
// two-leaf items and keeps the per-ray hit stack (local memory) out of the hot loop's code.  Everything crosses the
// call by value so that the caller's sink and ray stay in registers.
template <typename R>
struct CsgAnswer {
    R t;
    int leaf, sub, flip;  // leaf < 0: the item offers nothing that beats `limit`
    bool overflow;
};
template <typename R, unsigned FEAT, bool STATS>
__device__ __noinline__ CsgAnswer<R> csgGeneral(const DevScene<R>* S, int opFirst, int opCount, Ray<R> wr, R limit, bool any, Counters<STATS>* cnp)
{
    Counters<STATS> scratch;
    Counters<STATS>& cn = cnp ? *cnp : scratch;
    CsgAnswer<R> ans;
    ans.t = limit; ans.leaf = -1; ans.sub = 0; ans.flip = 0; ans.overflow = false;
    HitRec<R> stack[kHitCap];
    const int nh = evalCsg<R, FEAT, STATS>(*S, opFirst, opCount, wr, stack, ans.overflow, cn);
    for (int k = 0; k < nh; ++k) {  // sorted by t
        const R ht = stack[k].t;
        if (!(ht >= R(0))) continue;
        if (!any) {  // the first t >= 0 is this item's candidate; it wins if it beats the best so far
            if (ht < limit) {
                ans.t = ht; ans.leaf = (int)(stack[k].id & kIdLeafMask); ans.sub = (int)((stack[k].id >> kIdSubShift) & 7u);
                ans.flip = (stack[k].id & kIdFlip) ? 1 : 0;
            }
            break;
        }
        if (!(ht < limit)) break;
        const int leaf = (int)(stack[k].id & kIdLeafMask);
        if (__ldg(S->surf_i + __ldg(S->leaf_meta + leaf).y).z) { ans.leaf = leaf; break; }
    }
    return ans;
}

// <= 2 crossings of one CSG operand, in registers.  RUNS: the operand may be a run of consecutive leaves (a Group such as
// solidCylinder = [top; bottom; sides], Cylinder.fs:25-29), so every crossing remembers the leaf it belongs to.
template <typename R, bool RUNS>
struct PairSink {
    static constexpr bool kIsRay = false;
    // The last two crossings, newest first (a push is four moves and no compare at every hit site of the leaf intersectors;
    // which one was first is sorted out once, in csgPair): n == 1: (t0, i0); n == 2: (t1, i1) then (t0, i0).
    R t0, t1;
    unsigned i0, i1;  // leaf | sub << kIdSubShift
    int n, cur;
    FTB_DEV void clear(int first) { n = 0; t0 = t1 = R(0); i0 = i1 = 0u; cur = first; }
    FTB_DEV void hit(R ht, int hsub)
    {
        t1 = t0; i1 = i0;
        t0 = ht; i0 = (unsigned)cur | ((unsigned)(hsub & 7) << kIdSubShiftI);
        ++n;
    }
    FTB_DEV R firstT() const { return n > 1 ? t1 : t0; }
    FTB_DEV unsigned firstId() const { return n > 1 ? i1 : i0; }
    FTB_DEV R secondT() const { return t0; }
    FTB_DEV unsigned secondId() const { return i0; }
    FTB_DEV bool done() const { return false; }
};

// Csg.constructedSolid (Csg.fs:74-94) for two operands with at most two crossings each (the common case: convex
// solids), entirely in registers: the same stable sort over A's hits then B's, the same toggling walk and rule tables
// as evalCsg, fused with the nearest / any selection.  Returns false (nothing consumed) when an operand reports more
// than two crossings; the caller then runs the general program.
//   leafA / leafB = first leaf | (leaves - 1) << 24 (lower.cpp).  Variants without FT_PAIRG only meet single-leaf operands
//   and inline one copy of the leaf intersectors per operand (the two copies overlap their loads: measured 13 % faster on
//   the hollow-sphere scene than one shared copy); variants with FT_PAIRG (the house family: `subtract (solidCylinder)
//   (sphere)` is the only CSG item of house / night-house / repeat) walk both operands' runs through ONE copy, which
//   keeps those scenes off the general evaluator and its local-memory hit stack (measured -6 % house, -8 % repeat).
template <typename R, unsigned FEAT, bool STATS>
FTB_DEV bool csgPair(const DevScene<R>& S, int leafA, int leafB, int op, int kwA, int kwB, const Ray<R>& wr, RaySink<R, (FEAT & FT_MESH) != 0>& best, Counters<STATS>& cn)
{
    constexpr bool RUNS = (FEAT & FT_PAIRG) != 0;
    PairSink<R, RUNS> a, b;
    if constexpr (RUNS) {
        const int firstA = leafA & 0xffffff, endA = firstA + (leafA >> 24) + 1, firstB = leafB & 0xffffff, endB = firstB + (leafB >> 24) + 1;
        a.clear(firstA); b.clear(firstB);
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
            PairSink<R, RUNS> h;
            const int first = side ? firstB : firstA, end = side ? endB : endA;
            h.clear(first);
#pragma unroll 1
            for (int l = first; l < end; ++l) {  // a single-leaf operand's kind word came with the item
                h.cur = l;
                intersectLeaf<R, FEAT & ~FT_MESH, STATS>(S, l, end - first == 1 ? (side ? kwB : kwA) : leafKw(S, l), wr, h, cn);
            }
            if (h.n > 2) return false;
            if (side) b = h; else a = h;
            if (side == 0 && h.n == 0 && (op == OP_SUBTRACT || op == OP_INTERSECT)) return true;  // see below
        }
    } else {
        a.clear(leafA); b.clear(leafB);
        intersectLeaf<R, FEAT & ~FT_MESH, STATS>(S, leafA, kwA, wr, a, cn);
        if (a.n > 2) return false;
        // A ray that never crosses A is never inside A: `subtract A B` and `intersect A B` then discard every crossing of B
        // (OutsideIntoB / BIntoOutside -> Discard in both rule tables, Csg.fs:27-44), so B need not be intersected at all.  The
        // bounding sphere of a cube lets many such rays through.
        if (a.n == 0 && (op == OP_SUBTRACT || op == OP_INTERSECT)) return true;
        intersectLeaf<R, FEAT & ~FT_MESH, STATS>(S, leafB, kwB, wr, b, cn);
        if (b.n > 2) return false;
    }
    cn.add(ST_CSG_OPS);
    // Seq.sortBy (stable) as a fixed network: the four slots (A's hits, then B's; absent ones at +inf and marked invalid)
    // go through an odd-even transposition network of six compare-exchanges that swap neighbours only when the later one
    // is strictly smaller, which keeps equal keys in emission order (tests/test_pair_merge_equivalence.py replays it
    // against the insertion sort of evalCsg).  Measured -6.5 % on the hollow-sphere scene against four insertions.
    constexpr unsigned kInvalid = 0xffffffffu;
    R mt[4];
    unsigned mid[4];
    mt[0] = a.n > 0 ? a.firstT() : inf_<R>(); mid[0] = a.n > 0 ? a.firstId() : kInvalid;
    mt[1] = a.n > 1 ? a.secondT() : inf_<R>(); mid[1] = a.n > 1 ? a.secondId() : kInvalid;
    mt[2] = b.n > 0 ? b.firstT() : inf_<R>(); mid[2] = b.n > 0 ? (b.firstId() | kIdSideB) : kInvalid;
    mt[3] = b.n > 1 ? b.secondT() : inf_<R>(); mid[3] = b.n > 1 ? (b.secondId() | kIdSideB) : kInvalid;
    auto cx = [&](int i, int j) {
        const bool sw = mt[j] < mt[i];
        const R ti = mt[i], tj = mt[j];
        const unsigned ii = mid[i], ij = mid[j];
        mt[i] = sw ? tj : ti; mt[j] = sw ? ti : tj;
        mid[i] = sw ? ij : ii; mid[j] = sw ? ii : ij;
    };
    cx(0, 1); cx(2, 3); cx(1, 2); cx(0, 1); cx(2, 3); cx(1, 2);
    const unsigned rules = csgRuleTable(op);
    bool inA = false, inB = false, decided = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (mid[k] != kInvalid && !decided) {
            const unsigned id = mid[k];
            const R ht = mt[k];
            const bool hitB = (id & kIdSideB) != 0;
            const unsigned rule = (rules >> (2 * ((hitB ? 4 : 0) + (inA ? 2 : 0) + (inB ? 1 : 0)))) & 3u;
            if (hitB) inB = !inB; else inA = !inA;
            if (rule != 1u && ht >= R(0)) {
                const int leaf = (int)(id & kIdLeafMask);
                if (!best.any) {  // the item's first crossing with t >= 0 is its candidate (Scene.closest)
                    if (ht < best.limit) best.take(ht, leaf, (int)((id >> kIdSubShift) & 7u), rule == 2u);
                    decided = true;
                } else if (!(ht < best.limit)) {
                    decided = true;
                } else if (__ldg(S.surf_i + __ldg(S.leaf_meta + leaf).y).z) {  // Scene.lightIsBocked: applyLighting surfaces only
                    best.block(leaf);
                    decided = true;
                }
            }
        }
    }
    return true;
}

// bit 31 = "x < 0".  FP32: the sign bit itself (a - b < 0 <=> a < b: the sign of a rounded difference is the sign of the exact one,
// flush-to-zero keeps it; -0 cannot come out of a subtraction or an FMA with a non-zero sum; a NaN result is the canonical,
// positive one: "not less", like the comparison).  The FP64 verification build compares.
FTB_DEV unsigned signWord(float x) { return __float_as_uint(x); }
FTB_DEV unsigned signWord(double x) { return x < 0.0 ? 0x80000000u : 0u; }
// Unrolling of the two bound loops, per variant (measured, profiles/r2t_*): 4 for the small kernels (hollow-sphere -1 % against 1,
// moon -1 %: the loads and arithmetic of neighbouring items overlap), 1 for the large ones (house -2.3 %, night-house -2.4 %,
// repeat -0.5 %, the 960-triangle mesh -1.9 %: 240 SASS instructions fewer in kernels whose limiter is instruction fetch).
// The general loop builds its mask from sign bits like the table loop in the variants with the heavy leaf classes (house -2.4 %,
// night-house -2.8 %, repeat -1.9 %, hollow-sphere -1.2 %); the simple scenes and the mesh-only variants keep the compares (moon +3 %,
// the 960-triangle mesh +0.7 % with the signs).
template <unsigned FEAT> struct BoundSigns { static constexpr bool value = (FEAT & (FT_CUBE | FT_ROUND | FT_CSG | FT_CSGN)) != 0; };
#ifdef FTB_BOUND_UNROLL
template <unsigned FEAT> struct BoundUnroll { static constexpr int value = FTB_BOUND_UNROLL; };
#else
template <unsigned FEAT> struct BoundUnroll { static constexpr int value = (FEAT & (FT_PAIRG | FT_CSGN | FT_MESH)) != 0 ? 1 : 4; };
#endif

// ---- the common-origin bound table (see the derivation in render_kernel's prologue) --------------------------------------
// Layout.  FP64: one row (v.xyz, threshold) per item.  FP32: the rows of two neighbouring items interleaved,
// (x0 x1 y0 y1) (z0 z1 -w0 -w1), so that the test of both is one chain of packed operations; an odd item count is padded
// with a row that the candidate mask drops.  Either way an origin's rows take tabStride(n_items) R4 slots.
template <typename R> struct TabPairs { static constexpr bool value = sizeof(R) == 4; };
FTB_DEV int tabStride(int n_items) { return (n_items + 1) & ~1; }
template <typename R>
FTB_DEV bool originTableFits(const DevScene<R>& S) { return S.n_items >= kOriginMinItems && (1 + S.n_lights) * tabStride(S.n_items) <= kOriginCap; }  // = wantsOriginTable
template <typename R>
FTB_DEV void buildOriginTable(const DevScene<R>& S, const DevFrame<R>& F, typename V4<R>::type* origin_tab)
{
    typedef typename V4<R>::type R4;
    const int n_origins = 1 + S.n_lights;
    const int stride = tabStride(S.n_items);
    for (int o = 0; o < n_origins; ++o) {
        R4 org;
        R sign = R(1);
        if (o == 0) { org.x = F.cam_o[0]; org.y = F.cam_o[1]; org.z = F.cam_o[2]; org.w = R(0); }
        else { org = ldg4<R>(S.light_a + (o - 1)); sign = R(-1); }
        for (int j = threadIdx.x; j < stride; j += blockDim.x) {
            R4 row;
            if (j < S.n_items) {
                const R4 bound = ldg4<R>(S.item_bound + j);
                const Vec<R> v = mk<R>(sign * (bound.x - org.x), sign * (bound.y - org.y), sign * (bound.z - org.z));
                const R k = dot(v, v) * R(1.0 - 8e-6) - bound.w;
                row.x = v.x; row.y = v.y; row.z = v.z;
                row.w = !(k > R(0)) ? -inf_<R>() : sqrt_(k);  // unbounded items (w = +inf) and origins inside the bound: always candidates
            } else {
                row.x = row.y = row.z = R(0); row.w = -inf_<R>();  // padding: outside the candidate mask, not counted
            }
            if constexpr (TabPairs<R>::value) {
                R* t = reinterpret_cast<R*>(origin_tab + o * stride + (j & ~1)) + (j & 1);
                t[0] = row.x; t[2] = row.y; t[4] = row.z; t[6] = -row.w;
            } else {
                origin_tab[o * stride + j] = row;
            }
        }
    }
    __syncthreads();
}

template <typename R>
struct HitInfo {
    R t;
    int leaf, sub, flip;
};

// One ray against the whole scene.
//   any = false: Scene.intersectScene = geometry >> closest (Scene.fs:112-118); limit = +inf.
//   any = true : Scene.lightIsBocked (Scene.fs:119-121); limit = maxDistance; leaf >= 0 means blocked.
//   tab != nullptr (warp-uniform): every lane of this call traces a ray whose bound tests can be answered from its row
//   of the common-origin table (primary rays from the camera, shadow rays towards a point light; built in the kernel's
//   prologue); tabSlack = how far the ray's actual line can pass from that common point, as a distance along the ray.
//   allow: the items of the first batch this ray may trace at all (a primary ray: its tile's mask, DevFrame::tile_items, which
//   exists for scenes of one batch only); ~0u: every item.
template <typename R, unsigned FEAT, bool STATS>
FTB_DEV HitInfo<R> traceScene(const DevScene<R>& S, const Ray<R>& wr, R limit, bool any, int skipLeaf, unsigned allow, const typename V4<R>::type* tab, R tabSlack, bool& overflow,
                              Counters<STATS>& cn, unsigned tracing, int* wstack)
{
    typedef typename V4<R>::type R4;
    constexpr int kUnroll = BoundUnroll<FEAT>::value;  // (#pragma unroll takes constants, not macros)
    constexpr int kPairUnroll = kUnroll > 1 ? kUnroll / 2 : 1;
    RaySink<R, (FEAT & FT_MESH) != 0> best;
    best.limit = limit; best.id = -1; best.sub = 0; best.any = any; best.cur = 0; best.overflow = false;
    int bestItem = -1;  // mesh variants: the item of the current winner (tie rule of meshHit)
    // unit direction for the bound tests (their slack covers its rounding)
    const R inv_len = R(1) / sqrt_(dot(wr.d, wr.d));
    const Vec<R> du = mk<R>(wr.d.x * inv_len, wr.d.y * inv_len, wr.d.z * inv_len);
    for (int base = 0; base < S.n_items; base += 32) {
        // ---- phase A: which of the next 32 items can this ray's line touch at all?  Branch-free and unrolled:
        // the loads and the arithmetic of neighbouring items overlap (the serial per-item version spent a third
        // of its stall samples waiting on these two loads).
        const int n = min(32, S.n_items - base);
        unsigned cand = 0;
        if (tab) {  // rays from a common origin: |oc|, the miss and the behind test fold into one threshold per (origin, item)
            // candidate <=> !(b < w) <=> the sign bit of b - w is clear (a NaN is the canonical, positive one; w = -inf gives +inf):
            // the items are walked from the last to the first and each sign is shifted into the mask by one funnel shift.
            unsigned out = 0;
            if constexpr (TabPairs<R>::value) {  // two items per step: (x0 x1 y0 y1) (z0 z1 -w0 -w1), one chain of packed operations
                const F2 dx2 = dup2(du.x), dy2 = dup2(du.y), dz2 = dup2(du.z), sl2 = dup2(tabSlack);
#pragma unroll kPairUnroll
                for (int j = ((n + 1) & ~1) - 2; j >= 0; j -= 2) {
                    const R4 e0 = tab[base + j], e1 = tab[base + j + 1];
                    const F2 bw = fma2(pk2(e0.x, e0.y), dx2, fma2(pk2(e0.z, e0.w), dy2, fma2(pk2(e1.x, e1.y), dz2, add2(sl2, pk2(e1.z, e1.w)))));
                    cn.add(ST_BOUND_FAST, (e1.z < inf_<R>() ? 1u : 0u) + (e1.w < inf_<R>() ? 1u : 0u));
                    out = __funnelshift_l(signWord(hi2(bw)), out, 1);
                    out = __funnelshift_l(signWord(lo2(bw)), out, 1);
                }
            } else {
#pragma unroll kUnroll
                for (int j = n - 1; j >= 0; --j) {
                    const R4 e = tab[base + j];  // xyz = centre - origin (origin - centre for a light: the ray points AT it), w = threshold
                    const R bw = e.x * du.x + (e.y * du.y + (e.z * du.z + (tabSlack - e.w)));
                    cn.add(ST_BOUND_FAST, e.w > -inf_<R>() ? 1u : 0u);
                    out = __funnelshift_l(signWord(bw), out, 1);
                }
            }
            cand = ~out & (n >= 32 ? 0xffffffffu : ((1u << n) - 1u));
        } else {
            if constexpr (PackedBounds<R, FEAT>::value) {  // two items per step, the same test in packed operations
                const F2 nox = dup2(-wr.o.x), noy = dup2(-wr.o.y), noz = dup2(-wr.o.z);
                const F2 dx2 = dup2(du.x), dy2 = dup2(du.y), dz2 = dup2(du.z);
                unsigned out = 0;
#pragma unroll kPairUnroll
                for (int j = ((n + 1) & ~1) - 2; j >= 0; j -= 2) {
                    const R4 e0 = ldg4<R>(S.item_bound2 + base + j), e1 = ldg4<R>(S.item_bound2 + base + j + 1);  // (x0 x1 y0 y1) (z0 z1 w0 w1)
                    const F2 ocx = add2(pk2(e0.x, e0.y), nox), ocy = add2(pk2(e0.z, e0.w), noy), ocz = add2(pk2(e1.x, e1.y), noz);
                    const F2 w = pk2(e1.z, e1.w);
                    const F2 b = fma2(ocz, dz2, fma2(ocy, dy2, mul2(ocx, dx2)));
                    const F2 oc2 = fma2(ocz, ocz, fma2(ocy, ocy, mul2(ocx, ocx)));
                    const F2 miss = fma2(b, b, sub2(fma2(dup2(1e-6f), oc2, w), oc2));  // (w + 1e-6 oc2) - oc2 + b^2 < 0: the line misses the bound
                    const F2 outside = sub2(w, oc2);                                       // < 0 and b < 0: entirely behind the origin
                    cn.add(ST_BOUND_TESTS, (e1.z < inf_<R>() ? 1u : 0u) + (e1.w < inf_<R>() ? 1u : 0u));
                    out = __funnelshift_l(signWord(hi2(miss)) | (signWord(hi2(b)) & signWord(hi2(outside))), out, 1);
                    out = __funnelshift_l(signWord(lo2(miss)) | (signWord(lo2(b)) & signWord(lo2(outside))), out, 1);
                }
                cand = ~out & (n >= 32 ? 0xffffffffu : ((1u << n) - 1u));
            } else if constexpr (BoundSigns<FEAT>::value) {
                unsigned out = 0;
#pragma unroll kUnroll
                for (int j = n - 1; j >= 0; --j) {
                    const R4 bound = ldg4<R>(S.item_bound + base + j);  // xyz = centre, w = inflated radius^2 (+inf: unbounded)
                    const Vec<R> oc = mk<R>(bound.x - wr.o.x, bound.y - wr.o.y, bound.z - wr.o.z);
                    const R b = dot(oc, du);                                 // distance along the ray to the point nearest the centre
                    const R oc2 = dot(oc, oc);
                    // |centre - line|^2 = oc2 - b^2; the 1e-6 oc2 slack covers the cancellation (and the radius is inflated)
                    const R miss = (bound.w + R(1e-6) * oc2) - (oc2 - b * b);  // < 0: the ray's line misses the bound: no crossing at all
                    const R outside = bound.w - oc2;                           // < 0 and b < 0: bound entirely behind the origin, every crossing has t < 0
                    cn.add(ST_BOUND_TESTS, bound.w < inf_<R>() ? 1u : 0u);
                    out = __funnelshift_l(signWord(miss) | (signWord(b) & signWord(outside)), out, 1);  // w = +inf: neither can be negative
                }
                cand = ~out & (n >= 32 ? 0xffffffffu : ((1u << n) - 1u));
            } else {
#pragma unroll kUnroll
                for (int j = 0; j < n; ++j) {
                    const R4 bound = ldg4<R>(S.item_bound + base + j);  // xyz = centre, w = inflated radius^2 (+inf: unbounded)
                    const Vec<R> oc = mk<R>(bound.x - wr.o.x, bound.y - wr.o.y, bound.z - wr.o.z);
                    const R b = dot(oc, du);                                 // distance along the ray to the point nearest the centre
                    const R oc2 = dot(oc, oc);
                    // |centre - line|^2 = oc2 - b^2; the 1e-6 oc2 slack covers the cancellation (and the radius is inflated)
                    const bool miss = oc2 - b * b > bound.w + R(1e-6) * oc2;  // the ray's line misses the bound: no crossing at all
                    const bool behind = b < R(0) && oc2 > bound.w;            // bound entirely behind the origin: every crossing has t < 0
                    cn.add(ST_BOUND_TESTS, bound.w < inf_<R>() ? 1u : 0u);
                    cand |= !(miss || behind) ? (1u << j) : 0u;                // w = +inf: neither
                }
            }
        }
        cand &= allow;
        if (any) cand &= __ldg(S.item_casts + (base >> 5));  // items with nothing that has applyLighting cannot block (Scene.fs:121)
        unsigned meshCand = 0;  // mesh items are walked by the whole warp after this lane's other candidates
        constexpr bool kPacket = MeshWalks<FEAT>::kPacket;
        const bool packet = kPacket && (!MeshWalks<FEAT>::kPerLane || S.mesh_packet != 0);  // warp-uniform
        if constexpr (kPacket) { if (packet) { meshCand = cand & __ldg(S.item_mesh + (base >> 5)); cand &= ~meshCand; } }
        // ---- phase B: this lane's candidates, in enumeration order (lanes walk their own lists) -----------------
        while (cand) {
            const int it = base + __ffs(cand) - 1;
            cand &= cand - 1;
            const int4 item = __ldg(S.items + it);
            const R before = best.limit;
            if ((item.x & 0xff) == ITEM_LEAF) {
                if (item.y != skipLeaf) {  // skipLeaf: the planar leaf this ray leaves and cannot meet again (FP32 build, see the kernel)
                    best.cur = item.y;
                    intersectLeaf<R, FEAT, STATS>(S, item.y, (item.x >> 12) & 0x1ff, wr, best, cn);
                }
            } else if constexpr ((FEAT & (FT_CSG | FT_CSGN)) != 0) {
                bool done = false;
                if constexpr ((FEAT & FT_CSG) != 0) {
                    if ((item.x & 0xff) == ITEM_CSG2) done = csgPair<R, FEAT, STATS>(S, item.y, item.z, (item.x >> 8) & 0xf, (item.x >> 12) & 0x1ff, (item.x >> 21) & 0x1ff, wr, best, cn);
                }
                if (!done) {  // general program, or a leaf with more than two crossings
                    const int2 prog = __ldg(S.item_prog + it);
                    if constexpr ((FEAT & FT_CSGN) != 0) {  // scenes with general CSG items: inline (no call, no spills around it)
                        HitRec<R> stack[kHitCap];
                        const int nh = evalCsg<R, FEAT, STATS>(S, prog.x, prog.y, wr, stack, best.overflow, cn);
                        for (int k = 0; k < nh; ++k) {  // sorted by t
                            const R ht = stack[k].t;
                            if (!(ht >= R(0))) continue;
                            if (!any) {  // the first t >= 0 is this item's candidate; it wins if it beats best
                                if (ht < best.limit) best.take(ht, (int)(stack[k].id & kIdLeafMask), (int)((stack[k].id >> kIdSubShift) & 7u), (stack[k].id & kIdFlip) != 0);
                                break;
                            }
                            if (!(ht < best.limit)) break;
                            const int leaf = (int)(stack[k].id & kIdLeafMask);
                            if (__ldg(S.surf_i + __ldg(S.leaf_meta + leaf).y).z) { best.block(leaf); break; }
                        }
                    } else {  // pair-only scenes: the rare fallback stays out of line, off the hot loop's instruction footprint
                        const CsgAnswer<R> ans = csgGeneral<R, FEAT, STATS>(&S, prog.x, prog.y, wr, best.limit, any, STATS ? &cn : nullptr);
                        if (ans.leaf >= 0) {
                            if (any) best.block(ans.leaf); else best.take(ans.t, ans.leaf, ans.sub, ans.flip != 0);
                        }
                        best.overflow = best.overflow || ans.overflow;
                    }
                }
            }
            if constexpr (MeshWalks<FEAT>::kPacket) { if (best.limit < before) bestItem = it; }
            if (any && best.found()) cand = 0;
        }
        if (kPacket && packet) {
            // every lane of the call is here (the batch loop is warp-uniform in this mode): the meshes any lane still wants
            unsigned todo = __reduce_or_sync(tracing, (any && best.found()) ? 0u : meshCand);
            while (todo) {
                const int j = __ffs(todo) - 1;
                todo &= todo - 1;
                const int it = base + j;
                const int leaf = __ldg(S.items + it).y;
                const int4 meta = __ldg(S.leaf_meta + leaf);
                const bool want = ((meshCand >> j) & 1u) && !(any && best.found());
                const Ray<R> r = toModel<PackedXform<R, FEAT>::value, R>(S, leaf, (meta.x >> 8) & 1, wr);
                if (want) { cn.add(ST_LEAF0 + LEAF_MESH); if (!((meta.x >> 8) & 1)) cn.add(ST_XFORM); }
                // The walk keeps hits with t < limit only.  When the winner so far comes later in the enumeration than this mesh,
                // a triangle at exactly its t must still reach meshHit, which gives the tie to the mesh: the walk then runs with
                // the next number above best.limit (finite and >= 0: a winner was found).
                const R lim = (!any && best.found() && bestItem > it) ? nextUp(best.limit) : best.limit;
                R bt; int btri;
                packetMesh<R, STATS>(S, __ldg(S.mesh_root + meta.w), r, lim, any, want, tracing, wstack, bt, btri, cn);
                if (want && btri >= 0) {
                    if (any) best.block(leaf);  // t < limit held inside the walk
                    else meshHit(best, bestItem, it, leaf, bt, btri);
                }
            }
            if (__all_sync(tracing, any && best.found())) break;
        } else {
            if (any && best.found()) break;
        }
    }
    overflow = overflow || best.overflow;
    HitInfo<R> h;
    h.t = best.limit; h.leaf = best.leaf(); h.sub = best.subId(); h.flip = best.flipped();
    return h;
}

// ---- textures (Textures/Texture.fs, Textures/Image.fs:27-36) ---------------------------------------------
template <typename R>
FTB_DEV R repeatOne(R x)
{
    R a = abs_(x - floor_(x));
    return (a < R(0)) ? R(1) - a : a;
}
template <typename R>
FTB_DEV Vec<R> evalTexture(const DevScene<R>& S, int tex, R u, R v)
{
    typedef typename V4<R>::type R4;
    const int4 ti = __ldg(S.tex_i + tex);
    for (int k = 0; k < ti.y; ++k) {
        const int kind = __ldg(S.texop_kind + ti.x + k);
        const R a = __ldg(S.texop_ab + 2 * (ti.x + k)), b = __ldg(S.texop_ab + 2 * (ti.x + k) + 1);
        if (kind == FTB_TEX_SCALE) { u = u / a; v = v / b; }  // Texture.fs:14-16
        else {                                                  // Texture.fs:18-22, a = cos, b = sin
            R x = a * u + R(0) * R(0) + b * v;
            R z = (-b) * u + R(0) * R(0) + a * v;
            u = x; v = z;
        }
    }
    const R ru = repeatOne(u), rv = repeatOne(v);
    if (ti.z == FTB_TEX_GRID) {  // Texture.fs:24-29
        const R4 c1 = ldg4<R>(S.tex_c1 + tex), c2 = ldg4<R>(S.tex_c2 + tex);
        const bool first = (ru < R(0.5) && rv < R(0.5)) || (!(ru < R(0.5)) && (ru > R(0.5) && rv > R(0.5)));
        return first ? mk<R>(c1.x, c1.y, c1.z) : mk<R>(c2.x, c2.y, c2.z);
    }
    const int4 im = __ldg(S.img_i + ti.w);
    int x = (int)floor_(ru * (R)im.y), y = (int)floor_(rv * (R)im.z);
    x = min(max(x, 0), im.y - 1);  // SURVEY.md A.8: repeat can return exactly 1.0; clamped (documented)
    y = min(max(y, 0), im.z - 1);
    const uchar4 px = __ldg(S.texels + im.x + y * im.y + x);
    return mk<R>((R)px.x / R(255), (R)px.y / R(255), (R)px.z / R(255));
}

// ---- Jitter.fs on the ftb_rng contract --------------------------------------------------------------------
template <typename R>
FTB_DEV Vec<R> jitterVector(unsigned long long seed, unsigned long long sample, unsigned depth, unsigned light, unsigned idx, R tanHalfAngle, Vec<R> vector)
{
    Vec<R> normalised = normalise(vector);
    Vec<R> generator = (normalised.x > R(0.9)) ? mk<R>(R(0), R(1), R(0)) : mk<R>(R(1), R(0), R(0));
    Vec<R> i = normalise(cross(generator, normalised));
    Vec<R> j = cross(i, normalised);
    R x, y;
    for (unsigned attempt = 0;; ++attempt) {  // Jitter.circle (Jitter.fs:15-21)
        // (2 bits - 2^24) / 2^24: exact in float and double, so every build sees the same offsets
        x = (R)(2 * (int)ftb_rng_bits24(seed, sample, depth, light, idx, attempt, 0) - 16777216) * R(5.9604644775390625e-08);
        y = (R)(2 * (int)ftb_rng_bits24(seed, sample, depth, light, idx, attempt, 1) - 16777216) * R(5.9604644775390625e-08);
        if (!((x * x + y * y) > R(1))) break;
    }
    return normalise((normalised + (tanHalfAngle * x) * i) + (tanHalfAngle * y) * j);
}

// ---- winner finalisation: p, n, uv, material of the nearest hit ---------------------------------------------
template <typename R>
struct Fragment {
    Vec<R> p, n;
    Vec<R> colour;
    R roughness, reflectance, shineyness;
    bool applyLighting;
    int planarLeaf;  // FP32 build: the hit is on a top-level planar leaf (index), else -1
};

template <typename R, unsigned FEAT>
FTB_DEV Fragment<R> finalise(const DevScene<R>& S, const Ray<R>& wr, const HitInfo<R>& h)
{
    typedef typename V4<R>::type R4;
    const int4 meta = __ldg(S.leaf_meta + h.leaf);
    const int kind = meta.x & 0xff;
    const bool identity = (meta.x >> 8) & 1;
    const Ray<R> r = toModel<PackedXform<R, FEAT>::value, R>(S, h.leaf, identity, wr);
    const Vec<R> pm = mk<R>(r.o.x + h.t * r.d.x, r.o.y + h.t * r.d.y, r.o.z + h.t * r.d.z);
    Vec<R> nm = mk<R>(R(0), R(1), R(0));
    R u = R(0), v = R(0);
    if (kind == LEAF_SPHERE) {
        nm = normalise(pm);
    } else if (kind == LEAF_PLANE || kind == LEAF_SQUARE || kind == LEAF_CIRCLE) {
        u = pm.x; v = pm.z;
    } else if (kind == LEAF_CUBE) {
        if constexpr ((FEAT & FT_CUBE) != 0) {
            const R x1 = pm.x + R(0.5), y1 = pm.y + R(0.5), z1 = pm.z + R(0.5);
            const int axis = h.sub >> 1;             // 0: y (bottom/top), 1: x (left/right), 2: z (front/back)
            const R sgn = (h.sub & 1) ? R(1) : R(-1);  // Cube.fs:18-23: outward normals
            nm = mk<R>(axis == 1 ? sgn : R(0), axis == 0 ? sgn : R(0), axis == 2 ? sgn : R(0));
            u = axis == 1 ? y1 : x1;
            v = axis == 2 ? y1 : z1;
        }
    } else if (kind == LEAF_CYLINDER || kind == LEAF_CONE || (kind == LEAF_SOLIDCYL && h.sub == 2)) {
        if constexpr ((FEAT & FT_ROUND) != 0) {
            Vec<R> n = normalise(mk<R>(pm.x, kind == LEAF_CONE ? -(pm.y - R(1)) : R(0), pm.z));
            nm = (dot(n, r.d) < R(0)) ? n : -n;  // Cylinder.fs:17, Cone.fs:24: always faces the ray
        }
    } else if (kind == LEAF_SOLIDCYL) {  // a cap: the circle's (0,1,0) and p.xz carried back into the cylinder's frame
        if constexpr ((FEAT & FT_ROUND) != 0) {
            if (h.sub == 0) { u = pm.x; v = pm.z; }  // translate (0,1,0): normal and p.xz unchanged
            else {                                    // rotate unitZ 180: n = transpose(R) (0,1,0) = (s, c, 0), p' = R p
                nm = normalise(mk<R>(S.cyl_s, S.cyl_c, R(0)));
                u = S.cyl_c * pm.x + (-S.cyl_s) * pm.y; v = pm.z;
            }
        }
    } else {  // LEAF_TRIANGLE, LEAF_MESH
        if constexpr ((FEAT & FT_MESH) != 0) {
            const int tri = (kind == LEAF_TRIANGLE) ? meta.w : h.sub;
            R4 a1 = ldg4<R>(S.tris + 3 * tri + 1), a2 = ldg4<R>(S.tris + 3 * tri + 2);
            nm = normalise(cross(mk<R>(a1.x, a1.y, a1.z), mk<R>(a2.x, a2.y, a2.z)));
        }
    }
    Fragment<R> f;
    f.planarLeaf = -1;
    const int4 si = __ldg(S.surf_i + meta.y);
    // n <- normalise(normalToWorld * n), normalToWorld = transpose(worldToModel) (Transform.fs:83,86)
    Vec<R> nw = nm;
    if (!identity) {
        R4 r0 = ldg4<R>(S.leaf_w2m + 3 * h.leaf), r1 = ldg4<R>(S.leaf_w2m + 3 * h.leaf + 1), r2 = ldg4<R>(S.leaf_w2m + 3 * h.leaf + 2);
        nw = normalise(mk<R>(r0.x * nm.x + r1.x * nm.y + r2.x * nm.z, r0.y * nm.x + r1.y * nm.y + r2.y * nm.z, r0.z * nm.x + r1.z * nm.y + r2.z * nm.z));
    }
    if (h.flip) nw = R(-1) * nw;  // Csg Flip (Csg.fs:87)
    f.n = nw;
    // p = modelToWorld * p_model == o + t d in exact arithmetic (t is invariant); the ray itself is used
    f.p = mk<R>(wr.o.x + h.t * wr.d.x, wr.o.y + h.t * wr.d.y, wr.o.z + h.t * wr.d.z);
    if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {
        // FP32 only: a hit on a planar leaf far from the origin (the horizon of a ground plane, |p| ~ 1e3) is off the plane
        // by |p| * 6e-8, which is more than the reference's fixed 1e-4 d / 1e-4 n offsets can absorb: reflection rays
        // re-hit the plane from below (seen as a 1 / (1 - reflectance) brightening).  Put p back on the plane: with
        // p0 a world point of the plane, p -= ((p - p0).n) n - exact for axis-aligned planes, harmless for the others.
        if (kind == LEAF_PLANE || kind == LEAF_SQUARE || kind == LEAF_CIRCLE) {
            const R4 q = ldg4<R>(S.leaf_p0 + h.leaf);
            const Vec<R> n1 = h.flip ? -nw : nw;
            const R off = (f.p.x - q.x) * n1.x + (f.p.y - q.y) * n1.y + (f.p.z - q.z) * n1.z;
            f.p = mk<R>(f.p.x - off * n1.x, f.p.y - off * n1.y, f.p.z - off * n1.z);
            if ((meta.x >> 9) & 1) f.planarLeaf = h.leaf;
        }
    }
    const R4 sa = ldg4<R>(S.surf_a + meta.y), sb = ldg4<R>(S.surf_b + meta.y);
    Vec<R> col = mk<R>(sa.x, sa.y, sa.z);
    if constexpr ((FEAT & FT_TEX) != 0) {
        if (si.x >= 0) {
            if (kind == LEAF_SPHERE) {  // Sphere.setUV (Sphere.fs:6-10), only needed when textured
                u = R(0.5) + (atan2_(nm.z, nm.x) / (R(2) * R(3.14159265358979323846)));
                v = R(0.5) - asin_(nm.y) / R(3.14159265358979323846);
            }
            col = evalTexture(S, si.x, u, v);
            for (int k = 0; k < si.y; ++k) col = mk<R>(col.z, col.x, col.y);  // Colour.hueShift (CommonTypes.fs:90)
        }
    }
    f.colour = col;
    f.roughness = sa.w; f.reflectance = sb.x; f.shineyness = sb.y;
    f.applyLighting = si.z != 0;
    return f;
}

// ---- Shading.fs ------------------------------------------------------------------------------------------------
template <typename R>
FTB_DEV Vec<R> roughDiffuse(const Fragment<R>& f, Vec<R> lightDir, Vec<R> viewD)  // Shading.fs:50-63
{
    R roughness = f.roughness * f.roughness;
    R A = R(1) - R(0.5) * roughness / (roughness + R(0.33));
    R B = R(0.45) * roughness / (roughness + R(0.09));
    Vec<R> tangentLight = normalise(perpendicularComponent(f.n, -lightDir));
    Vec<R> tangentRay = normalise(perpendicularComponent(f.n, -viewD));
    if constexpr (sizeof(R) == 4) {
        // FP32 product build: the model only wants cos(lightAngle), sin(alpha) and tan(beta) of the two angles, so the angles themselves
        // (two acos, then cos / sin / tan of their results: ~90 instructions and four more roundings) are never formed:
        // cos(lightAngle) is the clamped dot product angleBetween takes the acos of; alpha, the larger angle, has the smaller cosine
        // ca, beta the larger one cb; sin(alpha) = sqrt((1 - ca)(1 + ca)) >= 0 on [0, pi], tan(beta) = sqrt((1 - cb)(1 + cb)) / cb.
        // In real arithmetic the same value as the literal form (which the FP64 verification build keeps); in FP32 closer to it
        // (moon -0.9 %, 127 of 133 M frame bytes move by one step; profiles/r2ad_rough_trig_ab.txt).
        // fsmin / fsmax keep F#'s NaN propagation; |cb| is kept off zero so that the grazing case stays finite like tanf(fl(pi / 2)).
        const Vec<R> nn = normalise(f.n);
        const R cr = min_(R(1), max_(R(-1), dot(nn, normalise(-viewD))));
        const R cl = min_(R(1), max_(R(-1), dot(nn, normalise(-lightDir))));
        const R ca = fsmin(cr, cl);
        R cb = fsmax(cr, cl);
        if (abs_(cb) < R(4e-8)) cb = cb < R(0) ? R(-4e-8) : R(4e-8);
        const R sinAlpha = sqrt_((R(1) - ca) * (R(1) + ca));
        const R tanBeta = sqrt_((R(1) - cb) * (R(1) + cb)) / cb;
        const R intensity = cl * (A + (B * fsmax(R(0), dot(tangentLight, tangentRay)) * sinAlpha * tanBeta));
        return intensity * f.colour;
    }
    R rayAngle = angleBetween(f.n, -viewD);
    R lightAngle = angleBetween(f.n, -lightDir);
    R alpha = fsmax(rayAngle, lightAngle);
    R beta = fsmin(rayAngle, lightAngle);
    R intensity = cos_(lightAngle) * (A + (B * fsmax(R(0), dot(tangentLight, tangentRay)) * sin_(alpha) * tan_(beta)));
    return intensity * f.colour;
}

// One light's fragment colour (shadeIfRequired (multiPartShader [specular; diffuse]), Shading.fs:100-107)
// given its shadow intensity.  The reflection part is carried by the caller's running weight.
template <typename R, unsigned FEAT>
FTB_DEV Vec<R> shadeLight(const DevScene<R>& S, const Fragment<R>& f, Vec<R> viewD, int li, R intensity)
{
    typedef typename V4<R>::type R4;
    if (!f.applyLighting) return f.colour;  // shadeIfRequired (Shading.fs:100-104)
    const int2 lk = __ldg(S.light_i + li);
    const R4 la = ldg4<R>(S.light_a + li), lc = ldg4<R>(S.light_c + li);
    const Vec<R> lv = mk<R>(la.x, la.y, la.z);
    const Vec<R> ldir = (lk.x == FTB_LIGHT_POINT) ? normalise(f.p - lv) : lv;  // lightDirection (Shading.fs:44-48): uses p, not the offset origin
    const Vec<R> lightColour = mk<R>(intensity * lc.x, intensity * lc.y, intensity * lc.z);
    Vec<R> acc = mk<R>(R(0), R(0), R(0));
    {  // specularShader (Shading.fs:78-87)
        const Vec<R> normal = normalise(f.n);
        const Vec<R> reflectedLightDirection = normalise(reflect(normal, ldir));
        const Vec<R> viewDirection = normalise(viewD);
        if (f.shineyness > R(0)) {
            const R si = pow_(dot(viewDirection, -reflectedLightDirection), f.shineyness);
            if (!(si <= R(0))) acc = acc + mk<R>(lightColour.x * si, lightColour.y * si, lightColour.z * si);
        }
    }
    bool lambert = true;
    if constexpr ((FEAT & FT_ROUGH) != 0) {
        if (f.roughness != R(0)) { acc = acc + roughDiffuse(f, ldir, viewD); lambert = false; }
    }
    if (lambert) {  // lambertianDiffuse (Shading.fs:65-70), unclamped
        const R di = dot(-ldir, f.n);
        acc = acc + mk<R>(di * (f.colour.x * lightColour.x), di * (f.colour.y * lightColour.y), di * (f.colour.z * lightColour.z));
    }
    return acc;
}

// ---- Image.fs (sampling half) -----------------------------------------------------------------------------------
template <typename R, unsigned FEAT>
FTB_DEV Ray<R> primaryRay(const DevFrame<R>& F, int px, int py, int s, unsigned long long sampleIndex)
{
    const R jitterX = __ldg(F.jitter + 2 * s), jitterY = __ldg(F.jitter + 2 * s + 1);  // s: sample index within the pixel (corner mode: 0)
    // rayThroughPixel (Image.fs:83-89)
    const R centreX = F.tlx + (R)px * F.pw, centreY = F.tly - (R)py * F.ph;
    const R jx = centreX + jitterX * F.pw, jy = centreY + jitterY * F.ph;
    const Vec<R> k = mk<R>(F.cam_k[0], F.cam_k[1], F.cam_k[2]), i = mk<R>(F.cam_i[0], F.cam_i[1], F.cam_i[2]), j = mk<R>(F.cam_j[0], F.cam_j[1], F.cam_j[2]);
    Ray<R> r;
    r.o = mk<R>(F.cam_o[0], F.cam_o[1], F.cam_o[2]);
    r.d = (k + jx * i) + jy * j;
    if constexpr ((FEAT & FT_RNG) != 0) {
        if (F.has_focus) {  // depthOfFieldJitter (Image.fs:91-94, Ray.fs:15-18)
            r.o = r.o + F.focal * r.d;
            r.d = jitterVector<R>(F.seed, sampleIndex, 0u, FTB_RNG_STREAM_CAMERA, 0u, F.tan_half_aperture, r.d);
            r.o = r.o + (-F.focal) * r.d;
        }
    }
    return r;
}

// ---- the kernel ------------------------------------------------------------------------------------------------------
// Resident CTAs per SM, per variant (measured, profiles/r2a_*, r2m_*): 5 (<= 102 registers, 20 warps / SM) in general - 3-7 %
// faster than 4 on cfg2 and the simple scenes (moon +10 % at 4), faster than 6 / 8; 6 for the mesh-only variants, whose walks wait
// on dependent node fetches; 4 (128 registers) for the variants with the shared-copy pairs or the general CSG evaluator (the
// house family), which spill 550 bytes at 96 registers: house -11 %, night-house -7 %, repeat -2 % at 4.
// The FP64 verification build passes -DFTB_MIN_BLOCKS=1.
#ifdef FTB_MIN_BLOCKS
template <unsigned FEAT> struct MinBlocks { static constexpr int value = FTB_MIN_BLOCKS; };
#else
template <unsigned FEAT> struct MinBlocks {
    static constexpr int value = (FEAT == (unsigned)FT_MESH || FEAT == (unsigned)(FT_MESH | FT_MESHPK)) ? 6 : ((FEAT & (FT_PAIRG | FT_CSGN)) != 0 ? 4 : 5);
};
#endif
#ifndef FTB_PHASE_ALIGN
#define FTB_PHASE_ALIGN 1
#endif
enum Phase : int { PH_IDLE = 0, PH_NEAREST = 1, PH_SHADOW = 2, PH_START = 3 };

// Blend ring: every warp keeps up to kRingSlots units in flight; a unit is a run of pixels of one 8x4 block times the
// samples of this pass (<= UnitCap<R, FEAT> samples).  Lanes take SAMPLES, not pixels: the longest sequential chain a lane
// can be stuck with is one sample's bounce chain, not spp of them, which is what bounds the kernel's tail and its
// strong scaling.  Finished sample colours are parked in the unit's slot in shared memory; when the last sample of a
// unit lands, the warp folds each pixel's samples IN SAMPLE ORDER (Array.average folds from Zero, Image.fs:112-116),
// so the frame does not depend on which lane traced which sample, nor on timing.
#ifndef FTB_RING_SLOTS
#define FTB_RING_SLOTS 2  // measured: 1 starves cheap-sample scenes (moon +70 %), 2 beats 3 and 4 by 1-3 % (fewer warp-uniform registers)
#endif
constexpr int kRingSlots = FTB_RING_SLOTS;
#ifndef FTB_FAST_BOUNDS
#define FTB_FAST_BOUNDS 1
#endif

// Folds a completed unit: every pixel's samples of this pass, in sample order, onto the running sum of the earlier
// passes; the last pass divides by the frame's sample count (Array.average = fold (+) Zero, then DivideByInt;
// Image.fs:112-116, CommonTypes.fs:43).
//   quads == 0 (the FP64 verification build; units of more than two pixels): one (pixel, channel) per lane, the literal
//   left fold.
//   quads != 0 (FP32 product build, units of one or two pixels = passes of >= 43 / >= 86 samples): a unit of 64-spp pixels
//   is two pixels, i.e. six sums of 64 dependent additions with 26 lanes idle (5 % of the warp instructions of the 8K
//   repeat frame at 6.6 lanes).  The samples of a (pixel, channel) are cut into four consecutive segments, one lane each;
//   the segment sums are then added in segment order by the first lane of the four.  Whether and how a pixel's samples
//   are segmented depends on the pass's sample count and the variant's unit size ONLY (not on the block shape, the shard
//   or the band), so the frame is still bit-identical however it was dealt; against the literal fold the sum differs by
//   FP32 rounding of the association, 1e-7 relative.  Measured: repeat -3.8 %; two segments for four-pixel units (moon)
//   did not pay (+1.2 %).
template <typename R>
__device__ __noinline__ void foldUnit(const R* col, const int* hdr, R* out, int scount, int spp, int s_base, int lane, int quads)
{
    const int slot0 = hdr[0], w = hdr[1], p0 = hdr[2], np = hdr[3];
    if (quads) {
        const int seg = (scount + 3) >> 2;
        const int i = lane, task = i >> 2, part = i & 3;  // np <= 2: 6 tasks x 4 lanes fit one round
        R acc = R(0);
        long long o = 0;
        if (task < np * 3) {
            const int pix = task / 3, ch = task - 3 * pix;
            const int pj = p0 + pix;
            const int ly = pj / w;
            o = 3 * ((long long)slot0 + ly * FTB_TILE_W + (pj - ly * w)) + ch;
            if (part == 0 && s_base > 0) acc = out[o];  // a later pass continues the fold of the earlier ones
            const int q0 = part * seg, q1 = min(scount, q0 + seg);
            const R* c = col + 3 * (pix * scount) + ch;
#pragma unroll 4
            for (int q = q0; q < q1; ++q) acc = acc + c[3 * q];
        }
        R total = acc;
#pragma unroll
        for (int k = 1; k < 4; ++k) total = total + __shfl_sync(0xffffffffu, acc, (lane & ~3) + k);
        if (task < np * 3 && part == 0) {
            if (s_base + scount >= spp) total = total / (R)spp;
            out[o] = total;
        }
        return;
    }
    for (int i = lane; i < np * 3; i += 32) {
        const int pix = i / 3, ch = i - 3 * pix;
        const int pj = p0 + pix;
        const int ly = pj / w;
        const long long o = 3 * ((long long)slot0 + ly * FTB_TILE_W + (pj - ly * w)) + ch;
        R acc = s_base > 0 ? out[o] : R(0);  // a later pass continues the left fold of the earlier ones
        const R* c = col + 3 * (pix * scount) + ch;
#pragma unroll 4
        for (int q = 0; q < scount; ++q) acc = acc + c[3 * q];
        if (s_base + scount >= spp) acc = acc / (R)spp;
        out[o] = acc;
    }
}

template <typename R, unsigned FEAT, bool STATS>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<FEAT>::value) render_kernel(const __grid_constant__ DevScene<R> S, const __grid_constant__ DevFrame<R> F)
{
    typedef typename V4<R>::type R4;
    constexpr int CAP = UnitCap<R, FEAT>::value;
    constexpr int WARPS = kBlockThreads / 32;
    __shared__ R ring_col[WARPS][kRingSlots][CAP * 3];
    constexpr bool kTable = FTB_FAST_BOUNDS != 0 && (FEAT & FT_TABLE) != 0;
    __shared__ int ring_hdr[WARPS][kRingSlots][4];  // out slot of the block's pixel 0, block width, first pixel, pixel count
    __shared__ int mesh_stack[MeshWalks<FEAT>::kPacket ? WARPS : 1][MeshWalks<FEAT>::kPacket ? kBspStack : 1];  // packetMesh: one walk per warp
    __shared__ R4 origin_tab[kTable ? kOriginCap : 1];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    Counters<STATS> cn;

    // Common-origin bound table.  Most rays start at one of a handful of points: primary rays at the camera, shadow rays
    // (traced from the fragment towards the light) end at a point light.  For such a ray the object-level bound test
    // "the line passes within r of the centre and the bound is not behind the origin" is b >= sqrt(|oc|^2 - r^2) with
    // b = oc . unit(d): the right-hand side depends on (origin, item) only.  Row 0 = camera, row 1 + l = light l (sign
    // flipped, the ray points at it; a crossing between fragment and light is ahead of the light looking back).
    // Like the general form the test may keep a miss but never drops a hit.  Rounding budget (tests/test_bound_table_budget.py
    // replays it in float32 against exact geometry): (1) in FP32 b is off by <= 4.8e-7 |oc| (rsqrt 2 ulp, three products), the
    // row's |oc|^2 by 3.6e-7 |oc|^2 and the approximate sqrt moves the threshold by 2 ulp: together < 1.8e-6 |oc|^2 of the
    // 8e-6 |oc|^2 slack in the threshold.  (2) The traced line does not pass exactly through the common point: a primary ray
    // starts at fl(camera + 1e-4 d), g <= 1e-7 |camera| off the ideal line; a shadow ray's rounded direction (fl(L - P)
    // normalised: 1.7e-7 rad) misses the light by g <= 1.7e-7 tmax.  An offset g changes |oc|^2 - b^2 by <= 2 |oc| g + g^2,
    // of which the remaining 6e-6 |oc|^2 of the threshold slack absorbs all but 2 |oc| g - 6e-6 |oc|^2 <= g^2 / 6e-6 (the
    // maximum over |oc|): adding sqrt(g^2 / 6e-6) = 410 g to b covers it for every item, i.e. 4.1e-5 |camera| resp.
    // 7e-5 tmax.  The per-ray slack actually added is 2e-4 |camera| for primary rays and 4e-4 tmax for shadow rays (5x).
    // -inf = always a candidate (unbounded, or the origin inside the bound).
    const bool fastBounds = kTable && originTableFits(S);
    const bool fastPrimary = fastBounds && F.mode == 0 && !((FEAT & FT_RNG) != 0 && F.has_focus);
    if (fastBounds) buildOriginTable<R>(S, F, origin_tab);
    bool overflow = false;

    // warp-uniform cursors: the pixel block (or 32 rays) taken from the per-GPU queue, and the unit being dealt from it
    int blk_slot0 = 0, blk_x0 = 0, blk_y0 = 0, blk_w = 1, blk_npix = 0, blk_pos = 0;
    int u_slot = 0, u_p0 = 0, u_pos = 0, u_n = 0;  // u_pos / u_n count RUNS of F.run consecutive samples of one pixel
    int remaining[kRingSlots];
    bool busy[kRingSlots];
#pragma unroll
    for (int k = 0; k < kRingSlots; ++k) { remaining[k] = 0; busy[k] = false; }
    bool exhausted = false;

    // per-lane sample / path state
    // where this lane's sample is parked, in one register (the kernel is register-bound: every register saved is a spill less):
    // bits 0..11 = position in the slot, bits 12..15 = ring slot, bits 16.. = samples left in this lane's run
    int rpos = 0;
    int px = 0, py = 0, sj = 0;      // pixel, sample index within the pixel
    // Index of the sample in the reference's full-frame ray list (RNG key, explicit-ray index), also in a window.  Variants
    // with in-path randomness carry it (two registers); nothing else needs it.
    constexpr bool kCarryIndex = (FEAT & FT_RNG) != 0;
    unsigned long long sampleIndex = 0;
    bool retire = false;             // a sample of this lane finished in the previous iteration (for the unit's count)
    Vec<R> scol = mk<R>(R(0), R(0), R(0));
    int phase = PH_IDLE, limit = 0;  // limit: bounces left; the bounce depth (RNG key) is recursion_limit - limit
    R weight = R(1), tmax = R(0);
    Ray<R> ray;            // the ray to trace next: path ray (un-offset) in PH_NEAREST, shadow ray in PH_SHADOW
    Vec<R> pathD;          // direction of the current path ray (viewRay.d of the fragment being shaded)
    ray.o = mk<R>(R(0), R(0), R(0)); ray.d = ray.o; pathD = ray.o;
    Fragment<R> f;
    f.p = ray.o; f.n = ray.o; f.colour = ray.o; f.roughness = f.reflectance = f.shineyness = R(0); f.applyLighting = false;
    Vec<R> local = ray.o;  // sum over lights at the current level
    int li = 0, sk = 0, occluded = 0;
    const int scount = F.mode == 0 ? F.s_count : 1;  // samples per pixel in this pass
    const int spp = F.mode == 0 ? F.spp : 1;          // samples per pixel of the frame
    const int run = F.mode == 0 ? F.run : 1;          // consecutive samples of one pixel a lane takes at a time (divides scount)
    const int rpp = scount / run;                     // runs per pixel
    const int ppu = max(1, min(32, CAP / scount));    // pixels per unit
    const int foldQuads = (sizeof(R) == 4 && ppu <= 2) ? 1 : 0;  // see foldUnit

    for (;;) {
        // ---- fold units whose last sample has landed (colours were parked when each path ended) ---------------------
        if (__any_sync(full, retire)) {
            __syncwarp();  // the parked colours of every lane are visible to the lanes that fold
            unsigned doneSlots = 0;
#pragma unroll
            for (int k = 0; k < kRingSlots; ++k) {
                remaining[k] -= __popc(__ballot_sync(full, retire && ((rpos >> 12) & 0xf) == k));
                if (busy[k] && remaining[k] == 0) { doneSlots |= 1u << k; busy[k] = false; }
            }
            while (doneSlots) {  // rare relative to the trace: one out-of-line copy keeps the hot loop small
                const int k = __ffs(doneSlots) - 1;
                doneSlots &= doneSlots - 1;
                foldUnit<R>(&ring_col[wib][k][0], &ring_hdr[wib][k][0], F.out, scount, spp, F.s_base, lane, foldQuads);
            }
            retire = false;
            __syncwarp();
        }
        // ---- deal runs of samples to idle lanes (ballot + popc = warp scan) -------------------------------------------
        bool need = phase == PH_IDLE;
        unsigned m = __ballot_sync(full, need);
        while (m && !exhausted) {
            if (u_pos >= u_n) {  // open the next unit
                int freeSlot = -1;
#pragma unroll
                for (int k = kRingSlots - 1; k >= 0; --k) if (!busy[k]) freeSlot = k;
                if (freeSlot < 0) break;  // every slot still has a sample in flight: idle lanes wait one iteration
                if (blk_pos >= blk_npix) {  // the warp takes the next pixel block (32 rays) from the per-GPU queue
                    unsigned c = 0;
                    if (lane == 0) c = atomicAdd(F.tile_counter, 1u);
                    c = __shfl_sync(full, c, 0);
                    if (c >= (unsigned)F.n_blocks) { exhausted = true; break; }
                    blk_pos = 0;
                    if (F.mode == 0) {
                        openBlock<R>(F, c, blk_slot0, blk_x0, blk_y0, blk_w, blk_npix);
                    } else {
                        const long long first = (long long)c * 32;
                        blk_slot0 = (int)first;
                        blk_w = 32;
                        blk_npix = (int)min(32LL, F.n_rays - first);
                    }
                    if (blk_npix <= 0) continue;
                }
                const int np = min(ppu, blk_npix - blk_pos);
                u_slot = freeSlot; u_p0 = blk_pos; u_pos = 0; u_n = np * rpp;
                blk_pos += np;
#pragma unroll
                for (int k = 0; k < kRingSlots; ++k) if (k == freeSlot) { busy[k] = true; remaining[k] = np * scount; }
                if (lane == 0) {
                    ring_hdr[wib][u_slot][0] = blk_slot0; ring_hdr[wib][u_slot][1] = blk_w; ring_hdr[wib][u_slot][2] = u_p0; ring_hdr[wib][u_slot][3] = np;
                }
            }
            const int rank = __popc(m & lt_mask);
            const int avail = u_n - u_pos;
            if (need && rank < avail) {
                const int q = u_pos + rank;                                      // run index within the unit
                const int pu = rpp == 1 ? q : (int)__umulhi((unsigned)q, F.rpp_magic);  // pixel within the unit = q / rpp
                const int pj = u_p0 + pu;                                        // pixel within the block
                sj = F.s_base + (q - pu * rpp) * run;
                rpos = (q * run) | (u_slot << 12) | (run << 16);
                if (F.mode == 0) {
                    const int ly = blk_w == 8 ? (pj >> 3) : pj / blk_w;
                    px = blk_x0 + (pj - ly * blk_w); py = blk_y0 + ly;
                    if constexpr (kCarryIndex) sampleIndex = ((unsigned long long)py * (unsigned)F.gw + (unsigned)px) * (unsigned)spp + (unsigned)sj;
                } else {
                    px = blk_slot0 + pj; py = 0;  // the ray's index
                    if constexpr (kCarryIndex) sampleIndex = (unsigned long long)(unsigned)px;
                }
                phase = PH_START;
                need = false;
            }
            u_pos += min(__popc(m), avail);
            m = __ballot_sync(full, need);
        }
        if (phase == PH_START) {  // a new sample: dealt just now, or the next one of this lane's run
            if (F.mode == 0) ray = primaryRay<R, FEAT>(F, px, py, sj, sampleIndex);
            else {
                const double* q = F.rays + 6 * (size_t)(unsigned)px;
                ray.o = mk<R>((R)__ldg(q), (R)__ldg(q + 1), (R)__ldg(q + 2));
                ray.d = mk<R>((R)__ldg(q + 3), (R)__ldg(q + 4), (R)__ldg(q + 5));
            }
            phase = PH_NEAREST; limit = F.recursion_limit; weight = R(1);
            scol = mk<R>(R(0), R(0), R(0));
            cn.add(ST_PRIMARY);
        }
        if (!__any_sync(full, phase != PH_IDLE)) break;
        // Phase alignment.  A warp whose lanes are in different phases runs every iteration at the pace of its slowest kind
        // of work (a nearest-hit query on a mesh walks ~60 BVH nodes, a shadow query ~10, a miss none) and diverges in
        // the result handling below.  Shadow-phase lanes go first and nearest-phase lanes hold for that iteration, so
        // the lanes of a warp fall into step: everyone traces primary / bounce rays together, then everyone traces
        // shadow rays together.  Scheduling only: a held lane traces the same ray one iteration later.
        // Measured: -28 % on the full-size mesh, -12 % house, -8 % night-house, -5 % moon, +-0 cfg2.
        bool hold = false;
        if constexpr (FTB_PHASE_ALIGN != 0) hold = __any_sync(full, phase == PH_SHADOW) && phase == PH_NEAREST;
        // all lanes that trace in this iteration have a row in the common-origin table?  (warp-uniform)
        bool tabled = false;
        if (fastBounds) {
            const bool mine = phase == PH_NEAREST ? (fastPrimary && limit == F.recursion_limit) : tmax < realmax_<R>();  // finite tmax: a point light
            tabled = !__any_sync(full, phase != PH_IDLE && !hold && !mine);
        }
        unsigned tracing = full;  // variants with the packet walk: the lanes that trace a ray in this iteration
        if constexpr (MeshWalks<FEAT>::kPacket) tracing = __ballot_sync(full, !(phase == PH_IDLE || hold));
        if (phase == PH_IDLE || hold) continue;

        // ---- trace this lane's current ray: the one expensive step ------------------------------------------------
        Ray<R> tr = ray;
        if (phase == PH_NEAREST) {  // slightOffset (Shading.fs:129): d is NOT normalised
            tr.o = ray.o + R(0.0001) * ray.d;
            pathD = ray.d;
        } else cn.add(ST_SHADOW);
        // FP32 build: a ray that starts on a top-level plane / square / circle and heads away from it has no crossing with
        // that leaf at t >= 0 (the reference's 1e-4 offsets put the only crossing at t < 0).  Far from the origin FP32 cannot
        // represent those offsets (at the horizon of a ground plane 1e-4 * d.y ~ 1e-8 next to |y| ~ 2), the crossing lands
        // on t = 0 or beyond and the plane reflects / shadows itself.  Such rays skip that one leaf; nothing else changes.
        int skipLeaf = -1;
        if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {  // `f` is still the fragment this bounce / shadow ray starts from
            if (f.planarLeaf >= 0 && (phase == PH_NEAREST ? limit < F.recursion_limit : dot(ray.d, f.n) >= R(0))) skipLeaf = f.planarLeaf;
        }
        // A primary ray of a camera-grid frame traces only the items its tile's mask keeps (tiles.h): the others provably give
        // it no crossing that the trace would report.
        unsigned allow = ~0u;
        if constexpr (TileMasks<R, FEAT>::value) {
            if (F.tile_items && phase == PH_NEAREST && limit == F.recursion_limit)
                allow = __ldg(F.tile_items + ((py - F.wy0) / FTB_TILE_H) * F.tiles_x + (px - F.wx0) / FTB_TILE_W);
        }
        const HitInfo<R> h = traceScene<R, FEAT, STATS>(S, tr, phase == PH_NEAREST ? inf_<R>() : tmax, phase == PH_SHADOW, skipLeaf, allow,
                                                        tabled ? origin_tab + (phase == PH_NEAREST ? 0 : 1 + li) * tabStride(S.n_items) : nullptr,
                                                        phase == PH_NEAREST ? F.primary_slack : R(4e-4) * tmax,
                                                        overflow, cn, tracing, &mesh_stack[MeshWalks<FEAT>::kPacket ? wib : 0][0]);

        // ---- consume the result -----------------------------------------------------------------------------------------
        bool got = false;       // an intensity for light `li` is ready
        R intensity = R(0);
        if (phase == PH_NEAREST) {
            if (limit == F.recursion_limit && F.dbg_prim) {
                int prim = -1, sub = 0;
                if (h.leaf >= 0) {
                    const int4 meta = __ldg(S.leaf_meta + h.leaf);
                    const int kind = meta.x & 0xff;
                    prim = meta.z;
                    sub = (kind == LEAF_CUBE || kind == LEAF_MESH || kind == LEAF_SOLIDCYL) ? h.sub : ((kind == LEAF_TRIANGLE) ? 0 : meta.w);
                }
                const unsigned long long at = F.mode == 0 ? ((unsigned long long)(unsigned)(py - F.wy0) * (unsigned)F.dbg_w + (unsigned)(px - F.wx0)) * (unsigned)spp + (unsigned)sj
                                                          : (unsigned long long)(unsigned)px;
                F.dbg_prim[at] = prim;
                if (F.dbg_sub) F.dbg_sub[at] = sub;
                if (F.dbg_t) F.dbg_t[at] = h.leaf >= 0 ? (double)h.t : -1.0;
            }
            if (h.leaf < 0 || S.n_lights <= 0) {  // miss: empty sum (Shading.fs:137-139)
                R* c = &ring_col[wib][0][3 * (((rpos >> 12) & 0xf) * CAP + (rpos & 0xfff))];
                c[0] = scol.x; c[1] = scol.y; c[2] = scol.z;
                retire = true;
                rpos -= 0xffff;  // one sample fewer in the run, one position further
                if ((rpos >> 16) > 0) { ++sj; if constexpr (kCarryIndex) ++sampleIndex; phase = PH_START; } else phase = PH_IDLE;
                continue;
            }
            cn.add(ST_SHADED);
            f = finalise<R, FEAT>(S, tr, h);
            local = mk<R>(R(0), R(0), R(0));
            li = 0;
            ray.o = f.p + R(0.0001) * f.n;  // shadowRayOrigin (Shading.fs:111), the same for every light
        } else {
            const bool blocked = h.leaf >= 0;
            const int2 lk = __ldg(S.light_i + li);
            if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {  // softShadowLightIntensity (Shading.fs:24-31)
                if constexpr ((FEAT & FT_RNG) != 0) {
                    occluded += blocked ? 1 : 0;
                    ++sk;
                    if (sk < lk.y) {
                        const R4 la = ldg4<R>(S.light_a + li);
                        ray.d = jitterVector<R>(F.seed, sampleIndex, (unsigned)(F.recursion_limit - limit), (unsigned)li, (unsigned)sk, la.w, -mk<R>(la.x, la.y, la.z));
                        continue;  // next sample of the same light
                    }
                    intensity = (R)(lk.y - occluded) / (R)lk.y;
                }
            } else if (lk.x == FTB_LIGHT_POINT) {
                const R4 lb = ldg4<R>(S.light_b + li);
                intensity = blocked ? R(0) : R(1) / (lb.x + tmax * (lb.y + tmax * lb.z));  // Light.attenuate (Light.fs:16-17)
            } else {
                intensity = blocked ? R(0) : R(1);
            }
            got = true;
        }
        // advance through the lights until one needs a shadow ray or the level is complete
        for (;;) {
            if (got) { local = local + shadeLight<R, FEAT>(S, f, pathD, li, intensity); ++li; got = false; }
            if (li >= S.n_lights) break;
            // fragments whose colour ignores the light's intensity need no shadow ray: unlit surfaces
            // (shadeIfRequired) and Oren-Nayar surfaces without a specular term (Shading.fs:50-63, 85-86)
            bool needShadow = f.applyLighting;
            if constexpr ((FEAT & FT_ROUGH) != 0) needShadow = needShadow && !(f.roughness != R(0) && !(f.shineyness > R(0)));
            if (!needShadow) { intensity = R(1); got = true; continue; }
            const int2 lk = __ldg(S.light_i + li);
            if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {
                // A primary fragment on the ground of a lit tile (lit_tiles.h): the host proved this directional light's shadow
                // rays unblocked, so their traced intensity would be 1 exactly ((n - 0) / n for a soft light).  Counted as traced.
                if (F.lit_tiles && li < 8 && limit == F.recursion_limit && f.planarLeaf == F.lit_leaf && lk.x != FTB_LIGHT_POINT &&
                    ((__ldg(F.lit_tiles + ((py - F.wy0) / FTB_TILE_H) * F.tiles_x + (px - F.wx0) / FTB_TILE_W) >> li) & 1)) {
                    cn.add(ST_SHADOW, lk.x == FTB_LIGHT_SOFT_DIRECTIONAL ? (unsigned)lk.y : 1u);
                    intensity = R(1); got = true; continue;
                }
            }
            const R4 la = ldg4<R>(S.light_a + li);
            const Vec<R> lv = mk<R>(la.x, la.y, la.z);
            if (lk.x == FTB_LIGHT_POINT) {  // shadowLightIntensity (Shading.fs:33-42)
                const Vec<R> dvec = lv - ray.o;
                tmax = length(dvec);
                ray.d = normalise(dvec);
            } else if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {
                if (lk.y <= 0) { intensity = (R)(lk.y - 0) / (R)lk.y; got = true; continue; }  // 0/0: NaN like the reference
                if constexpr ((FEAT & FT_RNG) != 0) {
                    sk = 0; occluded = 0;
                    tmax = realmax_<R>();
                    ray.d = jitterVector<R>(F.seed, sampleIndex, (unsigned)(F.recursion_limit - limit), (unsigned)li, 0u, la.w, -lv);
                }
            } else {
                tmax = realmax_<R>();
                ray.d = -lv;
            }
            phase = PH_SHADOW;
            break;
        }
        if (li < S.n_lights) continue;  // a shadow ray is pending
        // ---- level complete (getColourForRay's Seq.sumBy, Shading.fs:139) -----------------------------------------------
        scol = scol + weight * local;
        // reflectionShader (Shading.fs:89-98) sits inside the per-light sum: L identical re-traces => weight L * reflectance
        if (f.applyLighting && f.reflectance > R(0) && limit > 0) {
            weight = weight * ((R)S.n_lights * f.reflectance);
            ray.o = f.p; ray.d = reflect(f.n, pathD);
            --limit;
            phase = PH_NEAREST;
            cn.add(ST_REFLECTION);
        } else {  // the sample is complete: park its colour in the unit's slot; take the next sample of the run, if any
            R* c = &ring_col[wib][0][3 * (((rpos >> 12) & 0xf) * CAP + (rpos & 0xfff))];
            c[0] = scol.x; c[1] = scol.y; c[2] = scol.z;
            retire = true;
            rpos -= 0xffff;  // one sample fewer in the run, one position further
            if ((rpos >> 16) > 0) { ++sj; if constexpr (kCarryIndex) ++sampleIndex; phase = PH_START; } else phase = PH_IDLE;
        }
    }
    if (overflow) atomicExch(F.overflow, 1u);
    if constexpr (STATS) {
        for (int i = 0; i < ST_COUNT; ++i) {
            unsigned long long v = cn.get(i);
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(full, v, o);
            if (lane == 0 && v) atomicAdd(F.stats + i, v);
        }
    }
}

template <typename R, unsigned FEAT, bool WITH_STATS>
cudaError_t launch_render_impl(const DevScene<R>& s, const DevFrame<R>& f, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    int per_sm = 0;
    cudaError_t e;
    if constexpr (WITH_STATS) {
        if (stats) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, render_kernel<R, FEAT, true>, kBlockThreads, 0);
        else e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, render_kernel<R, FEAT, false>, kBlockThreads, 0);
    } else {
        if (stats) return cudaErrorInvalidValue;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, render_kernel<R, FEAT, false>, kBlockThreads, 0);
    }
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent grid: a multiple of the SM count, never more warps than there are work units to hand out
    const long long units = f.n_blocks;
    long long want = (long long)sm_count * per_sm;
    long long cap = (units + (kBlockThreads / 32) - 1) / (kBlockThreads / 32);
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if constexpr (WITH_STATS) {
        if (stats) render_kernel<R, FEAT, true><<<grid, kBlockThreads, 0, stream>>>(s, f);
        else render_kernel<R, FEAT, false><<<grid, kBlockThreads, 0, stream>>>(s, f);
    } else {
        render_kernel<R, FEAT, false><<<grid, kBlockThreads, 0, stream>>>(s, f);
    }
    if (launches) ++*launches;
    return cudaGetLastError();
}

// ---- sample shading (ftb_shade_samples: explicit rays, spp samples per pixel, blended as a frame blends them) -------------
// render_kernel with a third mode, F.mode = 2: F.n_rays pixels of F.spp explicit rays each.  Sample s of pixel i is ray i * spp + s
// with RNG key keys[i * spp + s] (keys == nullptr: i * spp + s), and its debug entry is i * spp + s.  Warps take 32 pixels at a
// time from the per-device queue as mode 1 takes 32 rays (the pixels are flat: a block is one row of 32), and deal them in mode
// 0's passes, runs and units, so foldUnit folds every pixel with the segmentation a frame of that spp and variant uses.
// A kernel of its own, so that render_kernel's code stays exactly what it is (its register allocation moves with any edit to the
// code it inlines, DESIGN.md §8).  And a copy of render_kernel's body with only the lines of mode 2 changed, mode 0's code kept
// although mode 2 never runs it: in FP32 the compiler's choice of fused multiply-adds inside the inlined trace and shading code
// depends on the code around it, and a copy pared down to mode 2 rounded some hit distances of the house scene one ulp apart from
// the frame's.  Kept this way, the trace and shading compile to the same instructions as render_kernel's (DESIGN.md §3).
template <typename R, unsigned FEAT, bool STATS>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<FEAT>::value) samples_kernel(const __grid_constant__ DevScene<R> S, const __grid_constant__ DevFrame<R> F,
                                                                                        const unsigned long long* keys)
{
    typedef typename V4<R>::type R4;
    constexpr int CAP = UnitCap<R, FEAT>::value;
    constexpr int WARPS = kBlockThreads / 32;
    __shared__ R ring_col[WARPS][kRingSlots][CAP * 3];
    constexpr bool kTable = FTB_FAST_BOUNDS != 0 && (FEAT & FT_TABLE) != 0;
    __shared__ int ring_hdr[WARPS][kRingSlots][4];  // out slot of the block's pixel 0, block width, first pixel, pixel count
    __shared__ int mesh_stack[MeshWalks<FEAT>::kPacket ? WARPS : 1][MeshWalks<FEAT>::kPacket ? kBspStack : 1];  // packetMesh: one walk per warp
    __shared__ R4 origin_tab[kTable ? kOriginCap : 1];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    Counters<STATS> cn;

    // Common-origin bound table.  Most rays start at one of a handful of points: primary rays at the camera, shadow rays
    // (traced from the fragment towards the light) end at a point light.  For such a ray the object-level bound test
    // "the line passes within r of the centre and the bound is not behind the origin" is b >= sqrt(|oc|^2 - r^2) with
    // b = oc . unit(d): the right-hand side depends on (origin, item) only.  Row 0 = camera, row 1 + l = light l (sign
    // flipped, the ray points at it; a crossing between fragment and light is ahead of the light looking back).
    // Like the general form the test may keep a miss but never drops a hit.  Rounding budget (tests/test_bound_table_budget.py
    // replays it in float32 against exact geometry): (1) in FP32 b is off by <= 4.8e-7 |oc| (rsqrt 2 ulp, three products), the
    // row's |oc|^2 by 3.6e-7 |oc|^2 and the approximate sqrt moves the threshold by 2 ulp: together < 1.8e-6 |oc|^2 of the
    // 8e-6 |oc|^2 slack in the threshold.  (2) The traced line does not pass exactly through the common point: a primary ray
    // starts at fl(camera + 1e-4 d), g <= 1e-7 |camera| off the ideal line; a shadow ray's rounded direction (fl(L - P)
    // normalised: 1.7e-7 rad) misses the light by g <= 1.7e-7 tmax.  An offset g changes |oc|^2 - b^2 by <= 2 |oc| g + g^2,
    // of which the remaining 6e-6 |oc|^2 of the threshold slack absorbs all but 2 |oc| g - 6e-6 |oc|^2 <= g^2 / 6e-6 (the
    // maximum over |oc|): adding sqrt(g^2 / 6e-6) = 410 g to b covers it for every item, i.e. 4.1e-5 |camera| resp.
    // 7e-5 tmax.  The per-ray slack actually added is 2e-4 |camera| for primary rays and 4e-4 tmax for shadow rays (5x).
    // -inf = always a candidate (unbounded, or the origin inside the bound).
    const bool fastBounds = kTable && originTableFits(S);
    const bool fastPrimary = fastBounds && F.mode == 0 && !((FEAT & FT_RNG) != 0 && F.has_focus);
    if (fastBounds) buildOriginTable<R>(S, F, origin_tab);
    bool overflow = false;

    // warp-uniform cursors: the pixel block (or 32 rays) taken from the per-GPU queue, and the unit being dealt from it
    int blk_slot0 = 0, blk_x0 = 0, blk_y0 = 0, blk_w = 1, blk_npix = 0, blk_pos = 0;
    int u_slot = 0, u_p0 = 0, u_pos = 0, u_n = 0;  // u_pos / u_n count RUNS of F.run consecutive samples of one pixel
    int remaining[kRingSlots];
    bool busy[kRingSlots];
#pragma unroll
    for (int k = 0; k < kRingSlots; ++k) { remaining[k] = 0; busy[k] = false; }
    bool exhausted = false;

    // per-lane sample / path state
    // where this lane's sample is parked, in one register (the kernel is register-bound: every register saved is a spill less):
    // bits 0..11 = position in the slot, bits 12..15 = ring slot, bits 16.. = samples left in this lane's run
    int rpos = 0;
    int px = 0, py = 0, sj = 0;      // pixel, sample index within the pixel
    // Index of the sample in the reference's full-frame ray list (RNG key, explicit-ray index), also in a window.  Variants
    // with in-path randomness carry it (two registers); nothing else needs it.
    constexpr bool kCarryIndex = (FEAT & FT_RNG) != 0;
    unsigned long long sampleIndex = 0;
    bool retire = false;             // a sample of this lane finished in the previous iteration (for the unit's count)
    Vec<R> scol = mk<R>(R(0), R(0), R(0));
    int phase = PH_IDLE, limit = 0;  // limit: bounces left; the bounce depth (RNG key) is recursion_limit - limit
    R weight = R(1), tmax = R(0);
    Ray<R> ray;            // the ray to trace next: path ray (un-offset) in PH_NEAREST, shadow ray in PH_SHADOW
    Vec<R> pathD;          // direction of the current path ray (viewRay.d of the fragment being shaded)
    ray.o = mk<R>(R(0), R(0), R(0)); ray.d = ray.o; pathD = ray.o;
    Fragment<R> f;
    f.p = ray.o; f.n = ray.o; f.colour = ray.o; f.roughness = f.reflectance = f.shineyness = R(0); f.applyLighting = false;
    Vec<R> local = ray.o;  // sum over lights at the current level
    int li = 0, sk = 0, occluded = 0;
    const int scount = F.mode != 1 ? F.s_count : 1;  // samples per pixel in this pass
    const int spp = F.mode != 1 ? F.spp : 1;          // samples per pixel of the frame
    const int run = F.mode != 1 ? F.run : 1;          // consecutive samples of one pixel a lane takes at a time (divides scount)
    const int rpp = scount / run;                     // runs per pixel
    const int ppu = max(1, min(32, CAP / scount));    // pixels per unit
    const int foldQuads = (sizeof(R) == 4 && ppu <= 2) ? 1 : 0;  // see foldUnit

    for (;;) {
        // ---- fold units whose last sample has landed (colours were parked when each path ended) ---------------------
        if (__any_sync(full, retire)) {
            __syncwarp();  // the parked colours of every lane are visible to the lanes that fold
            unsigned doneSlots = 0;
#pragma unroll
            for (int k = 0; k < kRingSlots; ++k) {
                remaining[k] -= __popc(__ballot_sync(full, retire && ((rpos >> 12) & 0xf) == k));
                if (busy[k] && remaining[k] == 0) { doneSlots |= 1u << k; busy[k] = false; }
            }
            while (doneSlots) {  // rare relative to the trace: one out-of-line copy keeps the hot loop small
                const int k = __ffs(doneSlots) - 1;
                doneSlots &= doneSlots - 1;
                foldUnit<R>(&ring_col[wib][k][0], &ring_hdr[wib][k][0], F.out, scount, spp, F.s_base, lane, foldQuads);
            }
            retire = false;
            __syncwarp();
        }
        // ---- deal runs of samples to idle lanes (ballot + popc = warp scan) -------------------------------------------
        bool need = phase == PH_IDLE;
        unsigned m = __ballot_sync(full, need);
        while (m && !exhausted) {
            if (u_pos >= u_n) {  // open the next unit
                int freeSlot = -1;
#pragma unroll
                for (int k = kRingSlots - 1; k >= 0; --k) if (!busy[k]) freeSlot = k;
                if (freeSlot < 0) break;  // every slot still has a sample in flight: idle lanes wait one iteration
                if (blk_pos >= blk_npix) {  // the warp takes the next pixel block (32 rays) from the per-GPU queue
                    unsigned c = 0;
                    if (lane == 0) c = atomicAdd(F.tile_counter, 1u);
                    c = __shfl_sync(full, c, 0);
                    if (c >= (unsigned)F.n_blocks) { exhausted = true; break; }
                    blk_pos = 0;
                    if (F.mode == 0) {
                        openBlock<R>(F, c, blk_slot0, blk_x0, blk_y0, blk_w, blk_npix);
                    } else {
                        const long long first = (long long)c * 32;
                        blk_slot0 = (int)first;
                        blk_w = 32;
                        blk_npix = (int)min(32LL, F.n_rays - first);
                    }
                    if (blk_npix <= 0) continue;
                }
                const int np = min(ppu, blk_npix - blk_pos);
                u_slot = freeSlot; u_p0 = blk_pos; u_pos = 0; u_n = np * rpp;
                blk_pos += np;
#pragma unroll
                for (int k = 0; k < kRingSlots; ++k) if (k == freeSlot) { busy[k] = true; remaining[k] = np * scount; }
                if (lane == 0) {
                    ring_hdr[wib][u_slot][0] = blk_slot0; ring_hdr[wib][u_slot][1] = blk_w; ring_hdr[wib][u_slot][2] = u_p0; ring_hdr[wib][u_slot][3] = np;
                }
            }
            const int rank = __popc(m & lt_mask);
            const int avail = u_n - u_pos;
            if (need && rank < avail) {
                const int q = u_pos + rank;                                      // run index within the unit
                const int pu = rpp == 1 ? q : (int)__umulhi((unsigned)q, F.rpp_magic);  // pixel within the unit = q / rpp
                const int pj = u_p0 + pu;                                        // pixel within the block
                sj = F.s_base + (q - pu * rpp) * run;
                rpos = (q * run) | (u_slot << 12) | (run << 16);
                if (F.mode == 0) {
                    const int ly = blk_w == 8 ? (pj >> 3) : pj / blk_w;
                    px = blk_x0 + (pj - ly * blk_w); py = blk_y0 + ly;
                    if constexpr (kCarryIndex) sampleIndex = ((unsigned long long)py * (unsigned)F.gw + (unsigned)px) * (unsigned)spp + (unsigned)sj;
                } else {
                    px = blk_slot0 + pj; py = 0;  // the ray's index
                    if constexpr (kCarryIndex) sampleIndex = (unsigned long long)(unsigned)px;
                }
                phase = PH_START;
                need = false;
            }
            u_pos += min(__popc(m), avail);
            m = __ballot_sync(full, need);
        }
        if (phase == PH_START) {  // a new sample: dealt just now, or the next one of this lane's run
            if (F.mode == 0) ray = primaryRay<R, FEAT>(F, px, py, sj, sampleIndex);
            else {  // mode 2: sample sj of pixel px is ray px * spp + sj, with RNG key keys[that] (nullptr: the ray's index)
                const size_t ri = (size_t)(unsigned)px * (unsigned)spp + (unsigned)sj;
                if constexpr (kCarryIndex) sampleIndex = keys ? __ldg(keys + ri) : (unsigned long long)ri;
                const double* q = F.rays + 6 * ri;
                ray.o = mk<R>((R)__ldg(q), (R)__ldg(q + 1), (R)__ldg(q + 2));
                ray.d = mk<R>((R)__ldg(q + 3), (R)__ldg(q + 4), (R)__ldg(q + 5));
            }
            phase = PH_NEAREST; limit = F.recursion_limit; weight = R(1);
            scol = mk<R>(R(0), R(0), R(0));
            cn.add(ST_PRIMARY);
        }
        if (!__any_sync(full, phase != PH_IDLE)) break;
        // Phase alignment.  A warp whose lanes are in different phases runs every iteration at the pace of its slowest kind
        // of work (a nearest-hit query on a mesh walks ~60 BVH nodes, a shadow query ~10, a miss none) and diverges in
        // the result handling below.  Shadow-phase lanes go first and nearest-phase lanes hold for that iteration, so
        // the lanes of a warp fall into step: everyone traces primary / bounce rays together, then everyone traces
        // shadow rays together.  Scheduling only: a held lane traces the same ray one iteration later.
        // Measured: -28 % on the full-size mesh, -12 % house, -8 % night-house, -5 % moon, +-0 cfg2.
        bool hold = false;
        if constexpr (FTB_PHASE_ALIGN != 0) hold = __any_sync(full, phase == PH_SHADOW) && phase == PH_NEAREST;
        // all lanes that trace in this iteration have a row in the common-origin table?  (warp-uniform)
        bool tabled = false;
        if (fastBounds) {
            const bool mine = phase == PH_NEAREST ? (fastPrimary && limit == F.recursion_limit) : tmax < realmax_<R>();  // finite tmax: a point light
            tabled = !__any_sync(full, phase != PH_IDLE && !hold && !mine);
        }
        unsigned tracing = full;  // variants with the packet walk: the lanes that trace a ray in this iteration
        if constexpr (MeshWalks<FEAT>::kPacket) tracing = __ballot_sync(full, !(phase == PH_IDLE || hold));
        if (phase == PH_IDLE || hold) continue;

        // ---- trace this lane's current ray: the one expensive step ------------------------------------------------
        Ray<R> tr = ray;
        if (phase == PH_NEAREST) {  // slightOffset (Shading.fs:129): d is NOT normalised
            tr.o = ray.o + R(0.0001) * ray.d;
            pathD = ray.d;
        } else cn.add(ST_SHADOW);
        // FP32 build: a ray that starts on a top-level plane / square / circle and heads away from it has no crossing with
        // that leaf at t >= 0 (the reference's 1e-4 offsets put the only crossing at t < 0).  Far from the origin FP32 cannot
        // represent those offsets (at the horizon of a ground plane 1e-4 * d.y ~ 1e-8 next to |y| ~ 2), the crossing lands
        // on t = 0 or beyond and the plane reflects / shadows itself.  Such rays skip that one leaf; nothing else changes.
        int skipLeaf = -1;
        if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {  // `f` is still the fragment this bounce / shadow ray starts from
            if (f.planarLeaf >= 0 && (phase == PH_NEAREST ? limit < F.recursion_limit : dot(ray.d, f.n) >= R(0))) skipLeaf = f.planarLeaf;
        }
        const HitInfo<R> h = traceScene<R, FEAT, STATS>(S, tr, phase == PH_NEAREST ? inf_<R>() : tmax, phase == PH_SHADOW, skipLeaf, ~0u,
                                                        tabled ? origin_tab + (phase == PH_NEAREST ? 0 : 1 + li) * tabStride(S.n_items) : nullptr,
                                                        phase == PH_NEAREST ? F.primary_slack : R(4e-4) * tmax,
                                                        overflow, cn, tracing, &mesh_stack[MeshWalks<FEAT>::kPacket ? wib : 0][0]);

        // ---- consume the result -----------------------------------------------------------------------------------------
        bool got = false;       // an intensity for light `li` is ready
        R intensity = R(0);
        if (phase == PH_NEAREST) {
            if (limit == F.recursion_limit && F.dbg_prim) {
                int prim = -1, sub = 0;
                if (h.leaf >= 0) {
                    const int4 meta = __ldg(S.leaf_meta + h.leaf);
                    const int kind = meta.x & 0xff;
                    prim = meta.z;
                    sub = (kind == LEAF_CUBE || kind == LEAF_MESH || kind == LEAF_SOLIDCYL) ? h.sub : ((kind == LEAF_TRIANGLE) ? 0 : meta.w);
                }
                const unsigned long long at = F.mode == 0 ? ((unsigned long long)(unsigned)(py - F.wy0) * (unsigned)F.dbg_w + (unsigned)(px - F.wx0)) * (unsigned)spp + (unsigned)sj
                                                          : (unsigned long long)(unsigned)px * (unsigned)spp + (unsigned)sj;
                F.dbg_prim[at] = prim;
                if (F.dbg_sub) F.dbg_sub[at] = sub;
                if (F.dbg_t) F.dbg_t[at] = h.leaf >= 0 ? (double)h.t : -1.0;
            }
            if (h.leaf < 0 || S.n_lights <= 0) {  // miss: empty sum (Shading.fs:137-139)
                R* c = &ring_col[wib][0][3 * (((rpos >> 12) & 0xf) * CAP + (rpos & 0xfff))];
                c[0] = scol.x; c[1] = scol.y; c[2] = scol.z;
                retire = true;
                rpos -= 0xffff;  // one sample fewer in the run, one position further
                if ((rpos >> 16) > 0) { ++sj; if constexpr (kCarryIndex) ++sampleIndex; phase = PH_START; } else phase = PH_IDLE;
                continue;
            }
            cn.add(ST_SHADED);
            f = finalise<R, FEAT>(S, tr, h);
            local = mk<R>(R(0), R(0), R(0));
            li = 0;
            ray.o = f.p + R(0.0001) * f.n;  // shadowRayOrigin (Shading.fs:111), the same for every light
        } else {
            const bool blocked = h.leaf >= 0;
            const int2 lk = __ldg(S.light_i + li);
            if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {  // softShadowLightIntensity (Shading.fs:24-31)
                if constexpr ((FEAT & FT_RNG) != 0) {
                    occluded += blocked ? 1 : 0;
                    ++sk;
                    if (sk < lk.y) {
                        const R4 la = ldg4<R>(S.light_a + li);
                        ray.d = jitterVector<R>(F.seed, sampleIndex, (unsigned)(F.recursion_limit - limit), (unsigned)li, (unsigned)sk, la.w, -mk<R>(la.x, la.y, la.z));
                        continue;  // next sample of the same light
                    }
                    intensity = (R)(lk.y - occluded) / (R)lk.y;
                }
            } else if (lk.x == FTB_LIGHT_POINT) {
                const R4 lb = ldg4<R>(S.light_b + li);
                intensity = blocked ? R(0) : R(1) / (lb.x + tmax * (lb.y + tmax * lb.z));  // Light.attenuate (Light.fs:16-17)
            } else {
                intensity = blocked ? R(0) : R(1);
            }
            got = true;
        }
        // advance through the lights until one needs a shadow ray or the level is complete
        for (;;) {
            if (got) { local = local + shadeLight<R, FEAT>(S, f, pathD, li, intensity); ++li; got = false; }
            if (li >= S.n_lights) break;
            // fragments whose colour ignores the light's intensity need no shadow ray: unlit surfaces
            // (shadeIfRequired) and Oren-Nayar surfaces without a specular term (Shading.fs:50-63, 85-86)
            bool needShadow = f.applyLighting;
            if constexpr ((FEAT & FT_ROUGH) != 0) needShadow = needShadow && !(f.roughness != R(0) && !(f.shineyness > R(0)));
            if (!needShadow) { intensity = R(1); got = true; continue; }
            const int2 lk = __ldg(S.light_i + li);
            if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {
                // A primary fragment on the ground of a lit tile (lit_tiles.h): the host proved this directional light's shadow
                // rays unblocked, so their traced intensity would be 1 exactly ((n - 0) / n for a soft light).  Counted as traced.
                if (F.lit_tiles && li < 8 && limit == F.recursion_limit && f.planarLeaf == F.lit_leaf && lk.x != FTB_LIGHT_POINT &&
                    ((__ldg(F.lit_tiles + ((py - F.wy0) / FTB_TILE_H) * F.tiles_x + (px - F.wx0) / FTB_TILE_W) >> li) & 1)) {
                    cn.add(ST_SHADOW, lk.x == FTB_LIGHT_SOFT_DIRECTIONAL ? (unsigned)lk.y : 1u);
                    intensity = R(1); got = true; continue;
                }
            }
            const R4 la = ldg4<R>(S.light_a + li);
            const Vec<R> lv = mk<R>(la.x, la.y, la.z);
            if (lk.x == FTB_LIGHT_POINT) {  // shadowLightIntensity (Shading.fs:33-42)
                const Vec<R> dvec = lv - ray.o;
                tmax = length(dvec);
                ray.d = normalise(dvec);
            } else if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {
                if (lk.y <= 0) { intensity = (R)(lk.y - 0) / (R)lk.y; got = true; continue; }  // 0/0: NaN like the reference
                if constexpr ((FEAT & FT_RNG) != 0) {
                    sk = 0; occluded = 0;
                    tmax = realmax_<R>();
                    ray.d = jitterVector<R>(F.seed, sampleIndex, (unsigned)(F.recursion_limit - limit), (unsigned)li, 0u, la.w, -lv);
                }
            } else {
                tmax = realmax_<R>();
                ray.d = -lv;
            }
            phase = PH_SHADOW;
            break;
        }
        if (li < S.n_lights) continue;  // a shadow ray is pending
        // ---- level complete (getColourForRay's Seq.sumBy, Shading.fs:139) -----------------------------------------------
        scol = scol + weight * local;
        // reflectionShader (Shading.fs:89-98) sits inside the per-light sum: L identical re-traces => weight L * reflectance
        if (f.applyLighting && f.reflectance > R(0) && limit > 0) {
            weight = weight * ((R)S.n_lights * f.reflectance);
            ray.o = f.p; ray.d = reflect(f.n, pathD);
            --limit;
            phase = PH_NEAREST;
            cn.add(ST_REFLECTION);
        } else {  // the sample is complete: park its colour in the unit's slot; take the next sample of the run, if any
            R* c = &ring_col[wib][0][3 * (((rpos >> 12) & 0xf) * CAP + (rpos & 0xfff))];
            c[0] = scol.x; c[1] = scol.y; c[2] = scol.z;
            retire = true;
            rpos -= 0xffff;  // one sample fewer in the run, one position further
            if ((rpos >> 16) > 0) { ++sj; if constexpr (kCarryIndex) ++sampleIndex; phase = PH_START; } else phase = PH_IDLE;
        }
    }
    if (overflow) atomicExch(F.overflow, 1u);
    if constexpr (STATS) {
        for (int i = 0; i < ST_COUNT; ++i) {
            unsigned long long v = cn.get(i);
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(full, v, o);
            if (lane == 0 && v) atomicAdd(F.stats + i, v);
        }
    }
}

template <typename R, unsigned FEAT, bool WITH_STATS>
cudaError_t launch_samples_impl(const DevScene<R>& s, const DevFrame<R>& f, const unsigned long long* keys, bool stats, int sm_count, cudaStream_t stream,
                                int* launches)
{
    if (!WITH_STATS && stats) return cudaErrorInvalidValue;
    int per_sm = 0;
    cudaError_t e = stats ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, samples_kernel<R, FEAT, WITH_STATS>, kBlockThreads, 0)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, samples_kernel<R, FEAT, false>, kBlockThreads, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent grid: a multiple of the SM count, never more warps than there are blocks of 32 pixels
    const long long want = (long long)sm_count * per_sm, cap = ((long long)f.n_blocks + (kBlockThreads / 32) - 1) / (kBlockThreads / 32);
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (stats) samples_kernel<R, FEAT, WITH_STATS><<<grid, kBlockThreads, 0, stream>>>(s, f, keys);
    else samples_kernel<R, FEAT, false><<<grid, kBlockThreads, 0, stream>>>(s, f, keys);
    if (launches) ++*launches;
    return cudaGetLastError();
}

// ---- ray queries (Scene.closest / Scene.lightIsBocked on caller-supplied rays) -----------------------------------------
// A kernel of its own, so that render_kernel's code and register allocation stay exactly what they are.  Warps take groups of
// 32 rays from the per-device queue counter (like mode 1 of render_kernel); each lane traces its ray exactly as given: no
// slightOffset, no skipped leaf, no common-origin table (arbitrary rays share no origin).  Nearest queries (Q.max_t == nullptr)
// report the renderer's winner and, with Q.record, the fragment finalise builds for it; occlusion queries report whether some
// surface with applyLighting crosses the ray at 0 <= t < max_t.
template <typename R, unsigned FEAT, bool STATS>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<FEAT>::value) query_kernel(const __grid_constant__ DevScene<R> S, const __grid_constant__ DevQuery Q)
{
    constexpr int WARPS = kBlockThreads / 32;
    __shared__ int mesh_stack[MeshWalks<FEAT>::kPacket ? WARPS : 1][MeshWalks<FEAT>::kPacket ? kBspStack : 1];  // packetMesh: one walk per warp
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const bool any = Q.max_t != nullptr;
    Counters<STATS> cn;
    bool overflow = false;
    for (;;) {
        unsigned c = 0;
        if (lane == 0) c = atomicAdd(Q.group_counter, 1u);
        c = __shfl_sync(full, c, 0);
        if (c >= (unsigned)Q.n_groups) break;
        const long long i = (long long)c * 32 + lane;
        const bool have = i < Q.n;
        const unsigned tracing = __ballot_sync(full, have);  // the packet walk's lanes: those holding a ray
        if (!have) continue;
        const double* q = Q.rays + 6 * (size_t)i;
        Ray<R> r;
        r.o = mk<R>((R)__ldg(q), (R)__ldg(q + 1), (R)__ldg(q + 2));
        r.d = mk<R>((R)__ldg(q + 3), (R)__ldg(q + 4), (R)__ldg(q + 5));
        const R limit = any ? (R)__ldg(Q.max_t + i) : inf_<R>();
        cn.add(any ? ST_SHADOW : ST_PRIMARY);
        const HitInfo<R> h = traceScene<R, FEAT, STATS>(S, r, limit, any, -1, ~0u, (const typename V4<R>::type*)nullptr, R(0), overflow, cn, tracing,
                                                        &mesh_stack[MeshWalks<FEAT>::kPacket ? wib : 0][0]);
        if (any) {
            Q.blocked[i] = h.leaf >= 0 ? 1 : 0;
            continue;
        }
        // the debug planes' expression (render_kernel), written out again so that render_kernel's code stays as it is
        int prim = -1, sub = 0;
        if (h.leaf >= 0) {
            const int4 meta = __ldg(S.leaf_meta + h.leaf);
            const int kind = meta.x & 0xff;
            prim = meta.z;
            sub = (kind == LEAF_CUBE || kind == LEAF_MESH || kind == LEAF_SOLIDCYL) ? h.sub : ((kind == LEAF_TRIANGLE) ? 0 : meta.w);
        }
        if (Q.prim) Q.prim[i] = prim;
        if (Q.sub) Q.sub[i] = sub;
        if (Q.t) Q.t[i] = h.leaf >= 0 ? (double)h.t : -1.0;
        if (Q.record) {  // a kernel parameter: warp-uniform
            double rec[13];  // p, normal, colour, roughness, reflectance, shineyness, apply_lighting; a miss is all zero
#pragma unroll
            for (int k = 0; k < 13; ++k) rec[k] = 0.0;
            if (h.leaf >= 0) {
                const Fragment<R> f = finalise<R, FEAT>(S, r, h);
                rec[0] = f.p.x; rec[1] = f.p.y; rec[2] = f.p.z;
                rec[3] = f.n.x; rec[4] = f.n.y; rec[5] = f.n.z;
                rec[6] = f.colour.x; rec[7] = f.colour.y; rec[8] = f.colour.z;
                rec[9] = f.roughness; rec[10] = f.reflectance; rec[11] = f.shineyness; rec[12] = f.applyLighting ? 1.0 : 0.0;
            }
            if (Q.p) { Q.p[3 * i] = rec[0]; Q.p[3 * i + 1] = rec[1]; Q.p[3 * i + 2] = rec[2]; }
            if (Q.normal) { Q.normal[3 * i] = rec[3]; Q.normal[3 * i + 1] = rec[4]; Q.normal[3 * i + 2] = rec[5]; }
            if (Q.colour) { Q.colour[3 * i] = rec[6]; Q.colour[3 * i + 1] = rec[7]; Q.colour[3 * i + 2] = rec[8]; }
            if (Q.surface) { Q.surface[4 * i] = rec[9]; Q.surface[4 * i + 1] = rec[10]; Q.surface[4 * i + 2] = rec[11]; Q.surface[4 * i + 3] = rec[12]; }
        }
    }
    if (overflow) atomicExch(Q.overflow, 1u);
    if constexpr (STATS) {
        for (int k = 0; k < ST_COUNT; ++k) {
            unsigned long long v = cn.get(k);
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(full, v, o);
            if (lane == 0 && v) atomicAdd(Q.stats + k, v);
        }
    }
}

template <typename R, unsigned FEAT, bool WITH_STATS>
cudaError_t launch_query_impl(const DevScene<R>& s, const DevQuery& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    if (!WITH_STATS && stats) return cudaErrorInvalidValue;
    int per_sm = 0;
    cudaError_t e = stats ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, query_kernel<R, FEAT, WITH_STATS>, kBlockThreads, 0)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, query_kernel<R, FEAT, false>, kBlockThreads, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent grid: a multiple of the SM count, never more warps than there are groups of rays
    const long long want = (long long)sm_count * per_sm, cap = ((long long)q.n_groups + (kBlockThreads / 32) - 1) / (kBlockThreads / 32);
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (stats) query_kernel<R, FEAT, WITH_STATS><<<grid, kBlockThreads, 0, stream>>>(s, q);
    else query_kernel<R, FEAT, false><<<grid, kBlockThreads, 0, stream>>>(s, q);
    if (launches) ++*launches;
    return cudaGetLastError();
}

// ---- crossing queries (Scene.intersect on caller-supplied rays, sorted by t) -------------------------------------------
// One kept crossing: 16 bytes in FP32.  leaf carries the CSG flip in bit 30; sub is HitInfo's (cube face, solidCylinder part,
// triangle index); rank is a mesh triangle's seq (0 for every other crossing).
template <typename R>
struct Crossing {
    R t;
    int leaf, sub, rank;
};

// A lane's kept list: the first `cap` crossings with lo <= t < hi in the order (t, item, rank in the item's own list), and how many
// there were.  Items arrive in enumeration order and leaf and CSG items report their lists in their own order, so an insertion
// that passes only entries of strictly larger t keeps that order.  A mesh's crossings arrive in the BVH walk's order: they also
// pass the entries of the same mesh (= the same leaf) with equal t and a larger seq, so the list does not depend on the walk.
// The range test is in double on the t the caller receives, so that a narrower range returns exactly the sublist.
template <typename R>
struct CrossList {
    static constexpr bool kIsRay = false;
    Crossing<R>* e;
    int cap, n, count;
    double lo, hi;
    int cur;  // leaf being intersected (intersectLeaf's sink protocol)
    FTB_DEV bool before(R t, int leaf, int rank, bool mesh, const Crossing<R>& x) const
    {
        return t < x.t || (mesh && t == x.t && (x.leaf & 0x3fffffff) == leaf && rank < x.rank);
    }
    FTB_DEV void add(R t, int leaf, int sub, int rank, bool mesh)
    {
        const double td = (double)t;
        if (!(td >= lo && td < hi)) return;
        ++count;
        if (n == cap && !before(t, leaf & 0x3fffffff, rank, mesh, e[cap - 1])) return;
        int j = n < cap ? n : cap - 1;
        while (j > 0 && before(t, leaf & 0x3fffffff, rank, mesh, e[j - 1])) { e[j] = e[j - 1]; --j; }
        e[j].t = t; e[j].leaf = leaf; e[j].sub = sub; e[j].rank = rank;
        if (n < cap) ++n;
    }
    FTB_DEV void hit(R t, int hsub) { add(t, cur, hsub, 0, false); }
    FTB_DEV bool done() const { return false; }
};

// Every crossing of a mesh (BspMesh.intersect, BspMesh.fs:67-76): one private walk per lane over the device's BVH, which reports
// each triangle the ray crosses.  Boxes are culled by the interval [0, tmax] only (boxEntry2: a mesh crossing has t > 1e-7).
template <typename R, bool STATS>
FTB_DEV void meshCrossings(const DevScene<R>& S, int root, int leaf, const Ray<R>& r, R tmax, CrossList<R>& list, bool& overflow, Counters<STATS>& cn)
{
    typedef typename V4<R>::type R4;
    int stack[kBspStack];
    int sp = 0;
    int link = root;
    const Vec<R> inv = mk<R>(R(1) / r.d.x, R(1) / r.d.y, R(1) / r.d.z);
    for (;;) {
        while (link >= 0) {
            cn.add(ST_BSP_NODES);
            const R4 b0 = ldg4<R>(S.bvh_node + 4 * link), b1 = ldg4<R>(S.bvh_node + 4 * link + 1), b2 = ldg4<R>(S.bvh_node + 4 * link + 2);
            const int2 ch = nodeLinks<R>(ldg4<R>(S.bvh_node + 4 * link + 3));
            R tl, tr;
            boxEntry2<R>(b0, b1, b2, r.o, inv, tmax, tl, tr);
            const bool hl = tl < inf_<R>(), hr = tr < inf_<R>();
            if (hl && hr) {
                if (sp < kBspStack) stack[sp++] = ch.y; else overflow = true;
                link = ch.x;
            } else if (hl || hr) {
                link = hl ? ch.x : ch.y;
            } else {
                link = 0x7fffffff;  // nothing below: pop
                break;
            }
        }
        if (link < 0) {  // a run of <= 7 triangles
            const int code = ~link, first = code >> 3, count = code & 7;
            for (int i = 0; i < count; ++i) {
                R t; R4 a0, a1;
                cn.add(ST_TRI_TESTS_IN_MESH);
                if (triangleT<R>(S.bvh_tris + 3 * (first + i), r, t, a0, a1)) list.add(t, leaf, (int)a1.w, (int)a0.w, true);
            }
        }
        if (sp == 0) break;
        link = stack[--sp];
    }
}

// A kernel of its own (compiled in crossings.cu, generic FEAT only), so that render_kernel and query_kernel stay what they are.
// Warps take groups of 32 rays from the per-device queue counter, like query_kernel; each lane walks every item in enumeration
// order and skips only those whose bounding sphere the ray's LINE misses (traceScene's general test and slack; no behind-the-origin
// cull: crossings at t < 0 count too).  Leaf items report through the leaf intersectors, CSG items (pairs included) through
// evalCsg on the item's program, mesh items through meshCrossings.  With Q.record (warp-uniform) finalise builds each kept entry.
template <typename R, unsigned FEAT, bool STATS>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<FEAT>::value) crossings_kernel(const __grid_constant__ DevScene<R> S, const __grid_constant__ DevCrossings Q)
{
    typedef typename V4<R>::type R4;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    Counters<STATS> cn;
    bool overflow = false;
    Crossing<R> kept[FTB_MAX_CROSSINGS];
    HitRec<R> stack[kHitCap];
    for (;;) {
        unsigned c = 0;
        if (lane == 0) c = atomicAdd(Q.group_counter, 1u);
        c = __shfl_sync(full, c, 0);
        if (c >= (unsigned)Q.n_groups) break;
        const long long i = (long long)c * 32 + lane;
        if (i >= Q.n) continue;
        const double* q = Q.rays + 6 * (size_t)i;
        Ray<R> r;
        r.o = mk<R>((R)__ldg(q), (R)__ldg(q + 1), (R)__ldg(q + 2));
        r.d = mk<R>((R)__ldg(q + 3), (R)__ldg(q + 4), (R)__ldg(q + 5));
        cn.add(ST_PRIMARY);
        CrossList<R> list;
        list.e = kept; list.cap = Q.max_hits; list.n = 0; list.count = 0; list.lo = Q.t_min; list.hi = Q.t_max; list.cur = 0;
        const R tmax = (R)Q.t_max;
        const R inv_len = R(1) / sqrt_(dot(r.d, r.d));
        const Vec<R> du = mk<R>(r.d.x * inv_len, r.d.y * inv_len, r.d.z * inv_len);
        for (int it = 0; it < S.n_items; ++it) {
            const R4 bound = ldg4<R>(S.item_bound + it);  // xyz = centre, w = inflated radius^2 (+inf: unbounded)
            const Vec<R> oc = mk<R>(bound.x - r.o.x, bound.y - r.o.y, bound.z - r.o.z);
            const R b = dot(oc, du);
            const R oc2 = dot(oc, oc);
            cn.add(ST_BOUND_TESTS, bound.w < inf_<R>() ? 1u : 0u);
            if (oc2 - b * b > bound.w + R(1e-6) * oc2) continue;  // the ray's line misses the bound: no crossing at any t
            const int4 item = __ldg(S.items + it);
            if ((item.x & 0xff) == ITEM_LEAF) {
                const int kw = (item.x >> 12) & 0x1ff;
                if ((kw & 0xff) == LEAF_MESH) {
                    if constexpr ((FEAT & FT_MESH) != 0) {
                        const bool identity = (kw >> 8) & 1;
                        cn.add(ST_LEAF0 + LEAF_MESH);
                        if (!identity) cn.add(ST_XFORM);
                        const Ray<R> m = toModel<PackedXform<R, FEAT>::value, R>(S, item.y, identity, r);
                        meshCrossings<R, STATS>(S, __ldg(S.mesh_root + __ldg(&S.leaf_meta[item.y].w)), item.y, m, tmax, list, overflow, cn);
                    }
                } else {
                    list.cur = item.y;
                    intersectLeaf<R, FEAT, STATS>(S, item.y, kw, r, list, cn);
                }
            } else if constexpr ((FEAT & (FT_CSG | FT_CSGN)) != 0) {
                const int2 prog = __ldg(S.item_prog + it);  // every CSG item has its program, pairs too
                const int nh = evalCsg<R, FEAT, STATS>(S, prog.x, prog.y, r, stack, overflow, cn);
                for (int k = 0; k < nh; ++k) {  // sorted by t: the item's own list
                    const unsigned id = stack[k].id;
                    list.add(stack[k].t, (int)(id & kIdLeafMask) | ((id & kIdFlip) ? (1 << 30) : 0), (int)((id >> kIdSubShift) & 7u), 0, false);
                }
            }
        }
        Q.counts[i] = list.count;
        const size_t base = (size_t)i * (size_t)Q.max_hits;
        for (int k = 0; k < Q.max_hits; ++k) {
            const bool have = k < list.n;
            HitInfo<R> h;
            h.t = R(0); h.leaf = -1; h.sub = 0; h.flip = 0;
            if (have) { h.t = kept[k].t; h.leaf = kept[k].leaf & 0x3fffffff; h.sub = kept[k].sub; h.flip = (kept[k].leaf >> 30) & 1; }
            // the debug planes' expression, as in query_kernel
            int prim = -1, sub = 0;
            if (have) {
                const int4 meta = __ldg(S.leaf_meta + h.leaf);
                const int kind = meta.x & 0xff;
                prim = meta.z;
                sub = (kind == LEAF_CUBE || kind == LEAF_MESH || kind == LEAF_SOLIDCYL) ? h.sub : ((kind == LEAF_TRIANGLE) ? 0 : meta.w);
            }
            const size_t e = base + k;
            if (Q.prim) Q.prim[e] = prim;
            if (Q.sub) Q.sub[e] = sub;
            if (Q.t) Q.t[e] = have ? (double)h.t : -1.0;
            if (Q.record) {  // a kernel parameter: warp-uniform
                double rec[13];  // p, normal, colour, roughness, reflectance, shineyness, apply_lighting; an unused slot is all zero
#pragma unroll
                for (int j = 0; j < 13; ++j) rec[j] = 0.0;
                if (have) {
                    const Fragment<R> f = finalise<R, FEAT>(S, r, h);
                    rec[0] = f.p.x; rec[1] = f.p.y; rec[2] = f.p.z;
                    rec[3] = f.n.x; rec[4] = f.n.y; rec[5] = f.n.z;
                    rec[6] = f.colour.x; rec[7] = f.colour.y; rec[8] = f.colour.z;
                    rec[9] = f.roughness; rec[10] = f.reflectance; rec[11] = f.shineyness; rec[12] = f.applyLighting ? 1.0 : 0.0;
                }
                if (Q.p) { Q.p[3 * e] = rec[0]; Q.p[3 * e + 1] = rec[1]; Q.p[3 * e + 2] = rec[2]; }
                if (Q.normal) { Q.normal[3 * e] = rec[3]; Q.normal[3 * e + 1] = rec[4]; Q.normal[3 * e + 2] = rec[5]; }
                if (Q.colour) { Q.colour[3 * e] = rec[6]; Q.colour[3 * e + 1] = rec[7]; Q.colour[3 * e + 2] = rec[8]; }
                if (Q.surface) { Q.surface[4 * e] = rec[9]; Q.surface[4 * e + 1] = rec[10]; Q.surface[4 * e + 2] = rec[11]; Q.surface[4 * e + 3] = rec[12]; }
            }
        }
    }
    if (overflow) atomicExch(Q.overflow, 1u);
    if constexpr (STATS) {
        for (int k = 0; k < ST_COUNT; ++k) {
            unsigned long long v = cn.get(k);
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(full, v, o);
            if (lane == 0 && v) atomicAdd(Q.stats + k, v);
        }
    }
}

template <typename R, unsigned FEAT>
cudaError_t launch_crossings_impl(const DevScene<R>& s, const DevCrossings& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    int per_sm = 0;
    cudaError_t e = stats ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, crossings_kernel<R, FEAT, true>, kBlockThreads, 0)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, crossings_kernel<R, FEAT, false>, kBlockThreads, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent grid: a multiple of the SM count, never more warps than there are groups of rays
    const long long want = (long long)sm_count * per_sm, cap = ((long long)q.n_groups + (kBlockThreads / 32) - 1) / (kBlockThreads / 32);
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (stats) crossings_kernel<R, FEAT, true><<<grid, kBlockThreads, 0, stream>>>(s, q);
    else crossings_kernel<R, FEAT, false><<<grid, kBlockThreads, 0, stream>>>(s, q);
    if (launches) ++*launches;
    return cudaGetLastError();
}

}  // namespace ftb
