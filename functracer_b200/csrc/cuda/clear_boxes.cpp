// clear_boxes.cpp — see clear_boxes.h.
#include "clear_boxes.h"

#include <algorithm>
#include <cmath>

namespace ftb {
namespace {

double norm(V3 v) { return std::sqrt(dot(v, v)); }

// Plane.fs answers a ray parallel to a plane (|d.y| < 1e-7 in its frame) with a crossing at t = 0 at the ray's origin, and the
// square / circle test then looks at the origin's own coordinates: that crossing is at the camera, wherever the leaf's box is.
// It needs the origin within the face's extent in the face's frame: x, z in [0, 1] for a square, |p| < 1 for a circle (a cube
// face: two of the centred |x|, |y|, |z| <= 0.5; a solidCylinder cap: |p| < 1 about either cap's centre).  True when the
// camera may be there: its model-space position with a margin for the origin's offset 1e-4 d and for FP32 rounding.
bool mayHitAtCamera(const Leaf& lf, V3 o, double dMax)
{
    const double* m = lf.w2m;
    const V3 p = {m[0] * o.x + m[1] * o.y + m[2] * o.z + m[3], m[4] * o.x + m[5] * o.y + m[6] * o.z + m[7], m[8] * o.x + m[9] * o.y + m[10] * o.z + m[11]};
    double f = 0;
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) f += m[4 * r + k] * m[4 * r + k];
    const double e = 1e-4 * (1.0 + norm(p)) + 2e-4 * std::sqrt(f) * dMax;
    switch (lf.kind) {
    case LEAF_SQUARE: return p.x >= -e && p.x <= 1.0 + e && p.z >= -e && p.z <= 1.0 + e;
    case LEAF_CIRCLE: return norm(p) < 1.0 + e;
    case LEAF_CUBE: return (std::fabs(p.x) <= 0.5 + e) + (std::fabs(p.y) <= 0.5 + e) + (std::fabs(p.z) <= 0.5 + e) >= 2;
    case LEAF_SOLIDCYL: return norm(p) < 1.0 + e || norm({p.x, p.y - 1.0, p.z}) < 1.0 + e;
    default: return false;  // the quadrics and Moller-Trumbore report no crossing for a degenerate ray
    }
}

}  // namespace

std::vector<ImageRect> itemBoxRects(const Lowered& L, const ftb_camera& c, int width, int height)
{
    std::vector<ImageRect> rects(L.items.size(), ImageRect{false, 0, 0, 0, 0});
    const CameraBasis b = cameraBasis(c, width, height);
    if (c.has_focus || !std::isfinite(b.width) || !std::isfinite(b.height)) return rects;
    const double camR = norm(b.o);
    const double dMax = std::sqrt(1.0 + b.width * b.width + b.height * b.height);  // |k + x i + y j| over the frame, generously
    for (size_t n = 0; n < L.items.size(); ++n) {
        const Item& it = L.items[n];
        const ItemBoxes& ib = L.item_boxes[n];
        if (!ib.valid || it.bound_r < 0) continue;
        bool ok = true;
        if (it.kind == ITEM_LEAF) ok = !mayHitAtCamera(L.leaves[(size_t)it.a], b.o, dMax);
        else
            for (int q = it.prog_first; q < it.prog_first + it.prog_count && ok; ++q)
                if (L.ops[q].kind == OP_LEAF) ok = !mayHitAtCamera(L.leaves[(size_t)L.ops[q].arg], b.o, dMax);
        ImageRect r = {true, 1e300, -1e300, 1e300, -1e300};
        for (size_t k = 0; k < ib.boxes.size() && ok; ++k) {
            const WorldBox& w = ib.boxes[k];
            V3 cen = {0, 0, 0};
            for (int i = 0; i < 8; ++i) cen = {cen.x + w.corner[i][0] / 8, cen.y + w.corner[i][1] / 8, cen.z + w.corner[i][2] / 8};
            double size = 0;
            for (int i = 0; i < 8; ++i) size = std::max(size, norm(sub({w.corner[i][0], w.corner[i][1], w.corner[i][2]}, cen)));
            // Every crossing the FP32 intersectors report for a ray lies within `m` of the box: their model-space rounding
            // (quadric roots within 3e-6 of t relative, DESIGN.md §5; the in-range tests on the FP32 hit point) grows by the
            // transform's condition number in world space and stays below 1e-4 of the distances involved.  The ray's and the
            // corners' own FP32 rounding is a few 1e-8 of the magnitudes; carried into the leaf's frame (w2m o in FP32, which
            // may cancel between the camera and the leaf's origin) and back it grows by the condition number too, hence
            // 1e-5 cond of the magnitudes (as tiles.cpp kRel).  A ray whose line misses the box widened by m has no crossing
            // with the leaf at any t; all crossings of the item lie in its boxes.
            const double m = w.cond * (1e-4 * (norm(sub(cen, b.o)) + size) + 1e-5 * (camR + norm(cen)));
            double zmin = 1e300, xl = 1e300, xh = -1e300, yl = 1e300, yh = -1e300;
            for (int i = 0; i < 8 && ok; ++i) {
                const V3 v = sub({w.corner[i][0], w.corner[i][1], w.corner[i][2]}, b.o);
                const double z = dot(v, b.k);
                ok = z > 2.0 * m;  // the box wholly in front of the camera: then the line's t < 0 half misses it too
                zmin = std::min(zmin, z);
                const double x = dot(v, b.i) / z, y = dot(v, b.j) / z;
                xl = std::min(xl, x); xh = std::max(xh, x); yl = std::min(yl, y); yh = std::max(yh, y);
            }
            if (!ok) break;
            // The corners' rectangle holds the projection of the box (convex, in front).  A point within m of a point of the
            // box at depth z >= zmin projects at most m (1 + |x|) / (zmin - m) further along x, likewise along y.
            const double dx = m * (1.0 + std::max(std::fabs(xl), std::fabs(xh))) / (zmin - m);
            const double dy = m * (1.0 + std::max(std::fabs(yl), std::fabs(yh))) / (zmin - m);
            r.xl = std::min(r.xl, xl - dx); r.xh = std::max(r.xh, xh + dx);
            r.yl = std::min(r.yl, yl - dy); r.yh = std::max(r.yh, yh + dy);
        }
        if (ok) rects[n] = r;
    }
    return rects;
}

}  // namespace ftb
