// lit_tiles.cpp — see lit_tiles.h.
#include "lit_tiles.h"

#include <algorithm>
#include <cmath>

namespace ftb {
namespace {

double norm(V3 v) { return std::sqrt(dot(v, v)); }
V3 along(V3 o, double t, V3 d) { return {o.x + t * d.x, o.y + t * d.y, o.z + t * d.z}; }

constexpr double kRel = 1e-5;   // as tiles.cpp: FP32 rounding of the magnitudes involved, with a wide margin
constexpr int kMaxSplits = 3;   // a tile's sample rectangle is cut into up to 8 x 8 parts

struct Cone { V3 a; double theta; unsigned bit; };  // the directions a light's shadow rays can take: within theta of a
struct Caster { V3 c; double ri, cr; };             // an item's bounding sphere: centre, the device's inflated radius, |c|

struct Proof {
    const CameraBasis& b;
    V3 row;
    double oy, relT, camR;
    const std::vector<Cone>& cones;
    const std::vector<Caster>& casters;

    // The bits of `want` proven for the samples whose image-plane positions lie in [u0, u1] x [v0, v1], every one of whose
    // rays heads for the ground.
    unsigned bits(double u0, double u1, double v0, double v1, unsigned want, int depth) const
    {
        // The rays through the rectangle meet the ground in the convex quad of its corners' hits (a central projection of a
        // convex set onto a plane that all of its rays reach in front).  The ball (m, rho0) holds the quad.
        V3 p[4];
        for (int q = 0; q < 4; ++q) {
            const double u = (q & 1) ? u1 : u0, v = (q & 2) ? v1 : v0;
            const V3 d = {b.k.x + u * b.i.x + v * b.j.x, b.k.y + u * b.i.y + v * b.j.y, b.k.z + u * b.i.z + v * b.j.z};
            p[q] = along(b.o, -oy / dot(row, d), d);
        }
        const V3 m = {(p[0].x + p[1].x + p[2].x + p[3].x) / 4, (p[0].y + p[1].y + p[2].y + p[3].y) / 4, (p[0].z + p[1].z + p[2].z + p[3].z) / 4};
        double rho0 = 0, dist = 0, pMax = 0;
        for (const V3& q : p) { rho0 = std::max(rho0, norm(sub(q, m))); dist = std::max(dist, norm(sub(q, b.o))); pMax = std::max(pMax, norm(q)); }
        // A shadow ray's FP32 origin lies within e of the quad: the hit point's FP32 rounding (t relative relT, the position
        // kRel of the magnitudes, the projection back onto the plane) and the shadowRayOrigin offset 1e-4 n.
        const double e = kRel * (dist + pMax + camR) + relT * dist + 1.1e-4;
        const double rho = rho0 + e, oMax = pMax + e;
        unsigned ok = 0;
        for (const Cone& cn : cones) {
            if (!(want & cn.bit)) continue;
            bool clear = true;
            for (size_t k = 0; k < casters.size() && clear; ++k) {
                const Caster& s = casters[k];
                // The radius beyond which the general bound test drops the item for every such ray (tiles.cpp: the inflated
                // radius, the test's 1e-6 |oc|^2 and the FP32 rounding of the ray and of the centre), then widened by rho:
                // a half-line from any origin of the ball (m, rho) that meets the ball (c, rdev) has a parallel one from m
                // that meets the ball (c, rdev + rho).
                const V3 v = sub(s.c, m);
                const double oc = norm(v), ocMax = oc + rho;
                const double rdev = std::sqrt(s.ri * s.ri + 2e-5 * ocMax * ocMax) + kRel * (ocMax + oMax + s.cr);
                const double R = rdev + rho;
                if (oc <= R) { clear = false; break; }
                // every direction of the cone is more than asin(R / oc) away from the direction of the centre: the half-lines
                // from m miss the ball
                const double phi = std::acos(std::max(-1.0, std::min(1.0, dot(cn.a, v) / oc)));
                clear = phi > cn.theta + std::asin(R / oc) + 1e-6;
            }
            if (clear) ok |= cn.bit;
        }
        const unsigned rest = want & ~ok;
        if (rest && depth < kMaxSplits) {
            const double um = 0.5 * (u0 + u1), vm = 0.5 * (v0 + v1);
            unsigned sub = rest;
            sub &= bits(u0, um, v0, vm, sub, depth + 1);
            if (sub) sub &= bits(um, u1, v0, vm, sub, depth + 1);
            if (sub) sub &= bits(u0, um, vm, v1, sub, depth + 1);
            if (sub) sub &= bits(um, u1, vm, v1, sub, depth + 1);
            ok |= sub;
        }
        return ok;
    }
};

}  // namespace

int litTiles(const Lowered& L, const ftb_light* lights, int n_lights, const ftb_camera& c, int width, int height, double offset, const TileGrid& g,
             std::vector<unsigned char>& lit)
{
    lit.assign((size_t)g.tiles_x * g.tiles_y, 0);
    // the ground: the only unbounded item, a top-level plane
    int ground = -1, groundItem = -1;
    for (size_t n = 0; n < L.items.size(); ++n) {
        const Item& it = L.items[n];
        if (it.bound_r >= 0) continue;
        if (groundItem >= 0 || it.kind != ITEM_LEAF || L.leaves[(size_t)it.a].kind != LEAF_PLANE) return -1;
        ground = it.a; groundItem = (int)n;
    }
    if (ground < 0 || c.has_focus) return -1;
    const CameraBasis b = cameraBasis(c, width, height);
    const double camR = norm(b.o);
    if (!(std::isfinite(b.pw) && std::isfinite(b.ph) && b.pw > 0 && b.ph > 0 && std::isfinite(b.tlx) && std::isfinite(b.tly) && std::isfinite(camR) &&
          std::fabs(dot(b.i, b.i) - 1) < 1e-9 && std::fabs(dot(b.k, b.k) - 1) < 1e-9 && std::fabs(dot(b.i, b.k)) < 1e-9))
        return -1;
    const Leaf& lf = L.leaves[(size_t)ground];
    const V3 row = lf.identity ? V3{0, 1, 0} : V3{lf.w2m[4], lf.w2m[5], lf.w2m[6]};
    const double w = lf.identity ? 0.0 : lf.w2m[7];
    const double n = norm(row);
    const V3 nh = {row.x / n, row.y / n, row.z / n};  // the fragment's normal (transpose(w2m) (0, 1, 0), normalised)
    // The camera strictly on one side of the plane, as for clear tiles (tiles.cpp), with dScale over the whole frame
    const double dScale = std::sqrt(1.0 + b.width * b.width + b.height * b.height) + std::fabs(b.tlx) + std::fabs(b.tly);
    const double oy = dot(row, b.o) + w;
    const double side = oy > 0 ? 1.0 : -1.0;
    if (!(side * oy > kRel * (n * (camR + dScale) + std::fabs(w)))) return -1;
    // The FP32 model-space y of the primary ray's origin is off by ~1e-7 (n |o| + |w|): the hit's t by that much relative to oy
    const double relT = 1e-6 * (n * (camR + dScale) + std::fabs(w)) / std::fabs(oy) + 1e-6;
    // Light side: every direction the light can produce leaves the plane on the side of its normal by more than 1e-4 (in
    // FP32 the kernel's skipLeaf then drops the ground for the ray, and in the reference the crossing with the plane is
    // behind the offset origin).  A soft light's jitterVector lies within atan(tan(scatter / 2)) of -v (the unit disk scaled
    // by the tangent); 1e-6 relative and 1e-5 absolute cover its FP32 basis and normalisation.
    std::vector<Cone> cones;
    for (int k = 0; k < std::min(n_lights, 8); ++k) {
        const ftb_light& l = lights[k];
        if (l.kind != FTB_LIGHT_DIRECTIONAL && !(l.kind == FTB_LIGHT_SOFT_DIRECTIONAL && l.samples > 0)) continue;
        const V3 a = normalise({-l.v[0], -l.v[1], -l.v[2]});
        const double theta = (l.kind == FTB_LIGHT_DIRECTIONAL ? 0.0 : std::atan(std::fabs(std::tan(l.scatter_rad / 2.0))) * (1 + 1e-6)) + 1e-5;  // the cone
        const double alpha = std::acos(std::max(-1.0, std::min(1.0, dot(a, nh))));
        if (!std::isfinite(theta) || !std::isfinite(alpha) || !(alpha + theta < 1.5707963267948966) || !(std::cos(alpha + theta) > 1e-4)) continue;
        cones.push_back({a, theta, 1u << k});
    }
    if (cones.empty()) return -1;
    std::vector<Caster> casters;
    for (size_t k = 0; k < L.items.size(); ++k) {
        const Item& it = L.items[k];
        if ((int)k == groundItem || !it.casts_shadow) continue;  // shadow rays ignore items that cannot block (Scene.fs:121)
        const V3 cen = {it.bound_c[0], it.bound_c[1], it.bound_c[2]};
        casters.push_back({cen, it.bound_r * 1.002 + 1e-5, norm(cen)});  // api.cu uploadScene's inflated radius
    }
    unsigned all = 0;
    for (const Cone& cn : cones) all |= cn.bit;
    const Proof pr = {b, row, oy, relT, camR, cones, casters};
    const double slack = offset + 0.05;  // pixels, as clear tiles: the samples' offsets and the FP32 rounding of their directions
    bool any = false;
    for (int ty = 0; ty < g.tiles_y; ++ty)
        for (int tx = 0; tx < g.tiles_x; ++tx) {
            const double c0 = g.wx0 + tx * FTB_TILE_W - slack, c1 = g.wx0 + tx * FTB_TILE_W + (FTB_TILE_W - 1) + slack;
            const double r0 = g.wy0 + ty * FTB_TILE_H - slack, r1 = g.wy0 + ty * FTB_TILE_H + (FTB_TILE_H - 1) + slack;
            const double u0 = b.tlx + c0 * b.pw, u1 = b.tlx + c1 * b.pw, v0 = b.tly - r1 * b.ph, v1 = b.tly - r0 * b.ph;
            // Footprint: all four corner rays head for the ground, clear of the FP32 rounding of d.y (tiles.cpp); then every
            // ray of the rectangle does (d.y is affine in (u, v)) and meets it in front of the camera.  Tiles across the
            // horizon get no bit.
            bool ok = true;
            for (int q = 0; q < 4 && ok; ++q) {
                const double u = (q & 1) ? u1 : u0, v = (q & 2) ? v1 : v0;
                ok = -side * (dot(row, b.k) + u * dot(row, b.i) + v * dot(row, b.j)) > 1.0001e-7 + kRel * n * dScale;
            }
            if (!ok) continue;
            const unsigned bits = pr.bits(u0, u1, v0, v1, all, 0);
            lit[(size_t)ty * g.tiles_x + tx] = (unsigned char)bits;
            any = any || bits != 0;
        }
    return any ? ground : -1;
}

}  // namespace ftb
