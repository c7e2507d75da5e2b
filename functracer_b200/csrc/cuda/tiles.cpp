// tiles.cpp — see tiles.h.
#include "tiles.h"

#include <algorithm>
#include <cmath>

namespace ftb {

V3 normalise(V3 v)
{
    double l = std::sqrt(v.x * v.x + v.y * v.y + v.z * v.z);
    if (l < 0.0000001) return v;
    double s = 1.0 / l;
    return {s * v.x, s * v.y, s * v.z};
}

CameraBasis cameraBasis(const ftb_camera& c, int resH, int resV)
{
    const V3 o = {c.o[0], c.o[1], c.o[2]}, la = {c.look_at[0], c.look_at[1], c.look_at[2]}, up = {c.up[0], c.up[1], c.up[2]};
    const V3 k = normalise(sub(la, o));
    const V3 i = normalise(cross(up, k));
    const V3 j = cross(k, i);
    const double height = std::tan(c.fov_y_rad / 2.0) * 2.0;
    const double width = height * c.aspect_ratio;
    const double ph = height / (double)(resH - 1);  // the reference's swapped axes (Image.fs:71-72)
    const double pw = width / (double)(resV - 1);
    return {o, k, i, j, width, height, pw, ph, -width / 2.0 + pw / 2.0, height / 2.0 - ph / 2.0};
}

double sampleOffsetExtent(const ftb_render_params& p)
{
    if (p.sampling == FTB_SAMPLING_CORNER) return 0.5;  // CornerSampling.generateRays: (-0.5, +0.5)
    double e = 0;
    for (int k = 0; k < 2 * p.spp; ++k) e = std::max(e, std::fabs(p.jitter_xy[k]));
    return e;
}

// The kernels trace primary rays in FP32 (the camera basis, pixel pitch and jitter narrowed to float, d = k + jx i + jy j
// and the leaf transform evaluated in float): a few 1e-7 of the magnitudes involved.  Every margin below is 1e-5 of them.
constexpr double kRel = 1e-5;

bool estimateTiles(const Lowered& L, int n_lights, const ftb_camera& c, int width, int height, int recursion_limit, double offset, const TileGrid& g,
                   std::vector<float>& cost, std::vector<unsigned char>& clear, const std::vector<ImageRect>* box_rects, std::vector<unsigned>* items,
                   double* kept)
{
    const double kPiHalf = 1.5707963267948966;
    const CameraBasis b = cameraBasis(c, width, height);
    const size_t n_tiles = (size_t)g.tiles_x * g.tiles_y;
    cost.assign(n_tiles, 1.0f);
    clear.assign(n_tiles, 0);
    if (items) items->clear();
    const double slack = offset + 0.05;  // pixels: the samples' offsets from their pixel centres and FP32 rounding of the image-plane position
    const double camR = std::sqrt(dot(b.o, b.o));
    const double primarySlack = 2e-4 * camR;  // DevFrame::primary_slack
    auto range = [&](double a, double z, double r, double& lo, double& hi) {
        const double d2 = a * a + z * z;
        if (d2 <= r * r) { lo = -1e300; hi = 1e300; return true; }
        const double th = std::atan2(a, z), al = std::asin(r / std::sqrt(d2));
        const double t0 = th - al, t1 = th + al;
        if (t0 >= kPiHalf || t1 <= -kPiHalf) return false;  // entirely behind the image plane
        lo = t0 <= -kPiHalf ? -1e300 : std::tan(t0);
        hi = t1 >= kPiHalf ? 1e300 : std::tan(t1);
        return true;
    };
    // The per-tile item masks need the pinhole camera's rays (depth of field moves their origins) and an orthonormal basis (the
    // projection below assumes one).  An unbounded item keeps its bit everywhere unless it is a top-level plane:
    // (row . d, row . o + w) = the ray's y in the plane's frame.
    const bool pinhole = !c.has_focus && std::isfinite(b.pw) && std::isfinite(b.ph) && b.pw > 0 && b.ph > 0 && std::isfinite(b.tlx) && std::isfinite(b.tly) &&
                         std::isfinite(camR) && std::fabs(dot(b.i, b.i) - 1) < 1e-9 && std::fabs(dot(b.k, b.k) - 1) < 1e-9 && std::fabs(dot(b.i, b.k)) < 1e-9;
    struct Plane { V3 row; double w; unsigned bit; };
    std::vector<Plane> planes;
    // mask[t] bit min(i, 31): item i may have a crossing with a primary ray of tile t that the kernel would report (items past
    // the 31st share the last bit, so that mask == 0 still means "nothing")
    std::vector<unsigned> mask(n_tiles, 0u);
    // wide[t]: the bits the spheres alone keep, every unbounded item's included (the items phase A may keep for the tile)
    std::vector<unsigned> wide(n_tiles, 0u);
    bool any = false;
    for (size_t item = 0; item < L.items.size(); ++item) {
        const Item& it = L.items[item];
        const unsigned bit = 1u << std::min<size_t>(item, 31);
        if (it.bound_r < 0) {  // unbounded: the same cost everywhere
            const Leaf* lf = it.kind == ITEM_LEAF ? &L.leaves[(size_t)it.a] : nullptr;
            if (lf && lf->kind == LEAF_PLANE) planes.push_back(lf->identity ? Plane{{0, 1, 0}, 0, bit} : Plane{{lf->w2m[4], lf->w2m[5], lf->w2m[6]}, lf->w2m[7], bit});
            else for (unsigned& m : mask) m |= bit;
            for (unsigned& m : wide) m |= bit;
            continue;
        }
        double w = 1.0;
        bool reflective = false;
        auto leafWork = [&](int leaf) {
            const Leaf& lf = L.leaves[leaf];
            const Surface& sf = L.surfaces[lf.surface];
            if (sf.apply_lighting && sf.reflectance > 0.0) reflective = true;
        };
        if (it.kind == ITEM_LEAF) leafWork(it.a);
        else {
            w = 0.0;
            for (int q = it.prog_first; q < it.prog_first + it.prog_count; ++q)
                if (L.ops[q].kind == OP_LEAF) { leafWork(L.ops[q].arg); w += 2.0; }
        }
        w *= (1.0 + (double)n_lights);                                   // a shaded hit adds one shadow ray per light
        if (reflective) w *= 1.0 + (double)std::max(0, recursion_limit);  // and up to `limit` more generations
        const V3 cen = {it.bound_c[0], it.bound_c[1], it.bound_c[2]};
        const V3 v = sub(cen, b.o);
        const double x = dot(v, b.i), y = dot(v, b.j), z = dot(v, b.k), oc = std::sqrt(dot(v, v));
        // The tiles that the image-plane rectangle [xl, xh] x [yl, yh] touches, with `pad` pixels of slack: image-plane
        // coordinates -> sample-grid pixels (rayThroughPixel, Image.fs:83-89), relative to the window's origin.  False: none.
        int tx0, tx1, ty0, ty1;
        auto tilesOf = [&](double xl, double xh, double yl, double yh, double pad) {
            if (xl > xh || yl > yh) return false;
            const double px0 = (xl - b.tlx) / b.pw - pad - g.wx0, px1 = (xh - b.tlx) / b.pw + pad - g.wx0;
            const double py0 = (b.tly - yh) / b.ph - pad - g.wy0, py1 = (b.tly - yl) / b.ph + pad - g.wy0;
            if (px1 < 0 || py1 < 0 || px0 >= g.ww || py0 >= g.wh) return false;
            tx0 = (int)std::max(0.0, std::floor(px0 / FTB_TILE_W)); tx1 = (int)std::min((double)g.tiles_x - 1, std::floor(px1 / FTB_TILE_W));
            ty0 = (int)std::max(0.0, std::floor(py0 / FTB_TILE_H)); ty1 = (int)std::min((double)g.tiles_y - 1, std::floor(py1 / FTB_TILE_H));
            return true;
        };
        // ... and those a sphere of radius r can touch
        auto tileRect = [&](double r, double pad) {
            double xl, xh, yl, yh;
            return range(x, z, r, xl, xh) && range(y, z, r, yl, yh) && tilesOf(xl, xh, yl, yh, pad);
        };
        // the cost estimate: the item's bound, one pixel of slack for jitter
        if (tileRect(it.bound_r, 1.5)) {
            for (int ty = ty0; ty <= ty1; ++ty)
                for (int tx = tx0; tx <= tx1; ++tx) cost[(size_t)ty * g.tiles_x + tx] += (float)w;
            any = true;
        }
        // the tiles whose mask keeps the item: the radius beyond which the kernel's bound test drops the item for every primary
        // ray - the device's inflated radius (api.cu uploadScene), widened by the 1e-6 |oc|^2 of the general test or by the
        // 8e-6 |oc|^2 and the primary slack of the common-origin table (render.cuh), and by the FP32 rounding of the ray and of
        // the bound's centre - and the samples' largest offset from their pixel centres
        const double ri = it.bound_r * 1.002 + 1e-5;
        const double r = std::sqrt(ri * ri + 2e-5 * oc * oc + 2.0 * oc * primarySlack + primarySlack * primarySlack) + kRel * (oc + camR + std::sqrt(dot(cen, cen)));
        if (!tileRect(r, slack)) continue;
        for (int ty = ty0; ty <= ty1; ++ty)
            for (int tx = tx0; tx <= tx1; ++tx) wide[(size_t)ty * g.tiles_x + tx] |= bit;
        if (box_rects && (*box_rects)[item].valid) {  // and that the item's boxes leave traced
            const ImageRect& q = (*box_rects)[item];
            const int sx0 = tx0, sx1 = tx1, sy0 = ty0, sy1 = ty1;
            if (!tilesOf(q.xl, q.xh, q.yl, q.yh, slack)) continue;
            tx0 = std::max(tx0, sx0); tx1 = std::min(tx1, sx1); ty0 = std::max(ty0, sy0); ty1 = std::min(ty1, sy1);
        }
        for (int ty = ty0; ty <= ty1; ++ty)
            for (int tx = tx0; tx <= tx1; ++tx) mask[(size_t)ty * g.tiles_x + tx] |= bit;
    }
    if (!pinhole) return any;
    // A plane (y = 0 in its frame, Plane.fs) has no crossing at t >= 0 with a ray whose origin is strictly on one side and whose
    // direction leads away from it: t = -oy / dy < 0.  Plane.fs answers t = 0 for a ray parallel to it (|dy| < 1e-7) from below
    // or on it, so |dy| must stay clear of 1e-7 too.  dy is affine in the image-plane position (u, v) of the sample and the tile's
    // samples lie in a rectangle of (u, v): its corners bound dy over the whole tile.  The offset origin camera + 1e-4 d only
    // moves further away from the plane.
    for (int ty = 0; ty < g.tiles_y; ++ty)
        for (int tx = 0; tx < g.tiles_x; ++tx) {
            const size_t t = (size_t)ty * g.tiles_x + tx;
            const double c0 = g.wx0 + tx * FTB_TILE_W - slack, c1 = g.wx0 + tx * FTB_TILE_W + (FTB_TILE_W - 1) + slack;
            const double r0 = g.wy0 + ty * FTB_TILE_H - slack, r1 = g.wy0 + ty * FTB_TILE_H + (FTB_TILE_H - 1) + slack;
            const double us[2] = {b.tlx + c0 * b.pw, b.tlx + c1 * b.pw}, vs[2] = {b.tly - r0 * b.ph, b.tly - r1 * b.ph};
            // the scale of the rounding errors of d (absolute errors of jx, jy next to |tlx|, |tly|)
            const double dScale = std::sqrt(1.0 + std::max(us[0] * us[0], us[1] * us[1]) + std::max(vs[0] * vs[0], vs[1] * vs[1])) + std::fabs(b.tlx) + std::fabs(b.tly);
            for (const Plane& pl : planes) {
                const double n = std::sqrt(dot(pl.row, pl.row));
                const double oy = dot(pl.row, b.o) + pl.w;
                const double side = oy > 0 ? 1.0 : -1.0;
                bool ok = side * oy > kRel * (n * (camR + dScale) + std::fabs(pl.w));
                const double dk = dot(pl.row, b.k), di = dot(pl.row, b.i), dj = dot(pl.row, b.j);
                for (int a = 0; a < 2 && ok; ++a)
                    for (int e = 0; e < 2 && ok; ++e) ok = side * (dk + us[a] * di + vs[e] * dj) > 1.0001e-7 + kRel * n * dScale;
                if (!ok) mask[t] |= pl.bit;
            }
            clear[t] = mask[t] == 0 ? 1 : 0;
        }
    if (items && L.items.size() <= 32) {
        if (kept) {
            double k = 0, w = 0;
            for (size_t t = 0; t < n_tiles; ++t)
                if (!clear[t]) { k += __builtin_popcount(mask[t]); w += __builtin_popcount(wide[t]); }
            *kept = w > 0 ? k / w : 1.0;
        }
        items->swap(mask);
    }
    return any;
}

}  // namespace ftb
