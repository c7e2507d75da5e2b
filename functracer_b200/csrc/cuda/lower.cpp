// lower.cpp — see lower.h.
#include "lower.h"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <map>
#include <utility>

namespace ftb {
namespace {

struct M34 {
    double m[12];
};
const M34 kIdentity = {{1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0}};

// c = a * b as 4x4 affine matrices (last row 0 0 0 1)
M34 mul(const M34& a, const M34& b)
{
    M34 c;
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 4; ++k) {
            double s = a.m[4 * r + 0] * b.m[0 + k] + a.m[4 * r + 1] * b.m[4 + k] + a.m[4 * r + 2] * b.m[8 + k];
            if (k == 3) s += a.m[4 * r + 3];
            c.m[4 * r + k] = s;
        }
    return c;
}
bool isIdentity(const M34& a) { return std::memcmp(a.m, kIdentity.m, sizeof(a.m)) == 0; }

bool invertAffine(const M34& a, M34& inv)
{
    const double* m = a.m;
    double c00 = m[5] * m[10] - m[6] * m[9], c01 = m[6] * m[8] - m[4] * m[10], c02 = m[4] * m[9] - m[5] * m[8];
    double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
    if (!(std::fabs(det) > 0.0) || !std::isfinite(det)) return false;
    double id = 1.0 / det;
    double r[9] = {c00 * id, (m[2] * m[9] - m[1] * m[10]) * id, (m[1] * m[6] - m[2] * m[5]) * id,
                   c01 * id, (m[0] * m[10] - m[2] * m[8]) * id, (m[2] * m[4] - m[0] * m[6]) * id,
                   c02 * id, (m[1] * m[8] - m[0] * m[9]) * id,  (m[0] * m[5] - m[1] * m[4]) * id};
    for (int i = 0; i < 3; ++i) {
        inv.m[4 * i + 0] = r[3 * i + 0];
        inv.m[4 * i + 1] = r[3 * i + 1];
        inv.m[4 * i + 2] = r[3 * i + 2];
        inv.m[4 * i + 3] = -(r[3 * i + 0] * m[3] + r[3 * i + 1] * m[7] + r[3 * i + 2] * m[11]);
    }
    return true;
}

struct Sphere {
    double c[3];
    double r;  // < 0: unbounded; NaN-free
};
const Sphere kUnbounded = {{0, 0, 0}, -1.0};
const Sphere kEmpty = {{0, 0, 0}, 0.0};

Sphere enclose(const Sphere& a, const Sphere& b, bool aEmpty, bool bEmpty)
{
    if (aEmpty) return b;
    if (bEmpty) return a;
    if (a.r < 0 || b.r < 0) return kUnbounded;
    double d[3] = {b.c[0] - a.c[0], b.c[1] - a.c[1], b.c[2] - a.c[2]};
    double dist = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    if (dist + b.r <= a.r) return a;
    if (dist + a.r <= b.r) return b;
    double r = 0.5 * (dist + a.r + b.r);
    double k = (r - a.r) / dist;
    return {{a.c[0] + k * d[0], a.c[1] + k * d[1], a.c[2] + k * d[2]}, r};
}

Sphere boundOfPoints(const M34& m2w, const std::vector<std::array<double, 3>>& pts)
{
    if (pts.empty()) return kEmpty;
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    std::vector<std::array<double, 3>> w(pts.size());
    for (size_t i = 0; i < pts.size(); ++i) {
        for (int r = 0; r < 3; ++r) {
            w[i][r] = m2w.m[4 * r] * pts[i][0] + m2w.m[4 * r + 1] * pts[i][1] + m2w.m[4 * r + 2] * pts[i][2] + m2w.m[4 * r + 3];
            lo[r] = std::min(lo[r], w[i][r]);
            hi[r] = std::max(hi[r], w[i][r]);
        }
    }
    Sphere s;
    for (int r = 0; r < 3; ++r) s.c[r] = 0.5 * (lo[r] + hi[r]);
    double r2 = 0;
    for (auto& p : w) {
        double dx = p[0] - s.c[0], dy = p[1] - s.c[1], dz = p[2] - s.c[2];
        r2 = std::max(r2, dx * dx + dy * dy + dz * dz);
    }
    s.r = std::sqrt(r2);
    if (!std::isfinite(s.r) || !std::isfinite(s.c[0]) || !std::isfinite(s.c[1]) || !std::isfinite(s.c[2])) return kUnbounded;
    return s;
}

// ||A||_F ||A^-1||_F of the linear parts of a transform and its inverse: at least A's condition number in the 2-norm
double condition(const M34& a, const M34& inv)
{
    double s = 0, t = 0;
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) { s += a.m[4 * r + k] * a.m[4 * r + k]; t += inv.m[4 * r + k] * inv.m[4 * r + k]; }
    return std::sqrt(s * t);
}

// The box [lo, hi] carried to world space by m2w; invalid if not finite.
ItemBoxes worldBox(const M34& m2w, double cond, const double* lo, const double* hi)
{
    WorldBox w;
    w.cond = cond;
    for (int i = 0; i < 8; ++i) {
        const double p[3] = {(i & 1) ? hi[0] : lo[0], (i & 2) ? hi[1] : lo[1], (i & 4) ? hi[2] : lo[2]};
        for (int r = 0; r < 3; ++r) {
            w.corner[i][r] = m2w.m[4 * r] * p[0] + m2w.m[4 * r + 1] * p[1] + m2w.m[4 * r + 2] * p[2] + m2w.m[4 * r + 3];
            if (!std::isfinite(w.corner[i][r])) return ItemBoxes();
        }
    }
    if (!std::isfinite(cond)) return ItemBoxes();
    ItemBoxes b;
    b.valid = true;
    b.boxes.push_back(w);
    return b;
}

const ItemBoxes kNoBoxes = {true, {}};  // an item that reports nothing

ItemBoxes join(const ItemBoxes& a, const ItemBoxes& b)
{
    if (!a.valid || !b.valid) return ItemBoxes();
    ItemBoxes j = a;
    j.boxes.insert(j.boxes.end(), b.boxes.begin(), b.boxes.end());
    return j;
}

std::vector<std::array<double, 3>> boxCorners(double x0, double x1, double y0, double y1, double z0, double z1)
{
    std::vector<std::array<double, 3>> p;
    for (int i = 0; i < 8; ++i) p.push_back({(i & 1) ? x1 : x0, (i & 2) ? y1 : y0, (i & 4) ? z1 : z0});
    return p;
}

struct SurfaceOp {
    int32_t kind;  // ftb_node_kind of the SceneFunction
    int32_t arg;
};

struct Ctx {
    M34 w2m;
    std::vector<SurfaceOp> ops;  // outermost first
};

struct Lowerer {
    const ftb_scene_desc& d;
    Lowered& L;
    std::string& err;
    int status = FTB_OK;
    std::map<std::vector<double>, int> surfaceIndex;
    std::map<int, int> textureIndex;  // desc texture -> lowered texture
    std::vector<Sphere> leafBound;
    std::vector<ItemBoxes> leafBox;  // the model-space box of leafBound's points in world space
    std::vector<int> meshDepth;

    Lowerer(const ftb_scene_desc& dd, Lowered& ll, std::string& e) : d(dd), L(ll), err(e) {}

    bool fail(int code, const std::string& m)
    {
        if (status == FTB_OK) { status = code; err = m; }
        return false;
    }

    int lowerTexture(int t)
    {
        auto it = textureIndex.find(t);
        if (it != textureIndex.end()) return it->second;
        TexDef def = {};
        def.op_first = (int)L.tex_ops.size();
        int cur = t, guard = 0;
        for (;;) {
            if (cur < 0 || cur >= d.n_textures || ++guard > 4096) { fail(FTB_ERR_BAD_SCENE, "bad texture index"); return -1; }
            const ftb_texture& x = d.textures[cur];
            if (x.kind == FTB_TEX_SCALE) { L.tex_ops.push_back({FTB_TEX_SCALE, 0, x.p[0], x.p[1]}); cur = x.inner; }
            else if (x.kind == FTB_TEX_ROTATE) { L.tex_ops.push_back({FTB_TEX_ROTATE, 0, x.p[1], x.p[2]}); cur = x.inner; }
            else if (x.kind == FTB_TEX_GRID) {
                def.base_kind = FTB_TEX_GRID; def.image = -1;
                for (int i = 0; i < 3; ++i) { def.c1[i] = x.p[i]; def.c2[i] = x.p[3 + i]; }
                break;
            } else if (x.kind == FTB_TEX_IMAGE) {
                if (x.image < 0 || x.image >= d.n_images) { fail(FTB_ERR_BAD_SCENE, "bad image index"); return -1; }
                const ftb_image& im = d.images[x.image];
                if (!im.rgb24 || im.width < 1 || im.height < 1) { fail(FTB_ERR_BAD_SCENE, "empty image"); return -1; }
                def.base_kind = FTB_TEX_IMAGE; def.image = x.image;
                L.has_image = true;
                break;
            } else { fail(FTB_ERR_BAD_SCENE, "bad texture kind"); return -1; }
        }
        def.op_count = (int)L.tex_ops.size() - def.op_first;
        L.textures.push_back(def);
        L.has_texture = true;
        int idx = (int)L.textures.size() - 1;
        textureIndex[t] = idx;
        return idx;
    }

    // SURVEY.md A.5: ops applied innermost first; the outermost Material / colour source wins.
    int resolveSurface(const Ctx& cx)
    {
        Surface s = {};
        s.texture = -1; s.hue = 0; s.apply_lighting = 1;
        s.colour[0] = s.colour[1] = s.colour[2] = 1.0;  // mattWhite (Ray.fs:11)
        for (size_t i = cx.ops.size(); i-- > 0;) {
            const SurfaceOp& op = cx.ops[i];
            switch (op.kind) {
            case FTB_NODE_MATERIAL: {
                const ftb_material& m = d.materials[op.arg];
                s.texture = -1; s.hue = 0;
                for (int k = 0; k < 3; ++k) s.colour[k] = m.colour[k];
                s.roughness = m.roughness; s.reflectance = m.reflectance; s.shineyness = m.shineyness;
                s.apply_lighting = m.apply_lighting != 0;
                break;
            }
            case FTB_NODE_TEXTURE: s.texture = lowerTexture(op.arg); s.hue = 0; break;
            case FTB_NODE_HUESHIFT: s.hue = (s.hue + 1) % 3; break;
            case FTB_NODE_IGNORELIGHT: s.apply_lighting = 0; break;
            }
        }
        if (s.texture < 0 && s.hue) {  // fold the permutation into the constant colour
            for (int h = 0; h < s.hue; ++h) { double r = s.colour[0], g = s.colour[1], b = s.colour[2]; s.colour[0] = b; s.colour[1] = r; s.colour[2] = g; }
            s.hue = 0;
        }
        std::vector<double> key = {(double)s.texture, (double)s.hue, (double)s.apply_lighting, s.colour[0], s.colour[1], s.colour[2], s.roughness, s.reflectance, s.shineyness};
        auto it = surfaceIndex.find(key);
        if (it != surfaceIndex.end()) return it->second;
        L.surfaces.push_back(s);
        if (s.roughness != 0.0) L.has_rough = true;
        return surfaceIndex[key] = (int)L.surfaces.size() - 1;
    }

    int bspDepth(int link, int depth)
    {
        if (depth > 256) { fail(FTB_ERR_BAD_SCENE, "BSP tree too deep or cyclic"); return depth; }
        if (link < 0) {
            int li = ~link;
            if (li >= d.n_bsp_leaves) { fail(FTB_ERR_BAD_SCENE, "bad BSP leaf link"); return depth; }
            const ftb_bsp_leaf& lf = d.bsp_leaves[li];
            if (lf.tri_first < 0 || lf.tri_count < 0 || lf.tri_first + lf.tri_count > d.n_triangles) fail(FTB_ERR_BAD_SCENE, "bad BSP leaf triangle range");
            return depth;
        }
        if (link >= d.n_bsp_nodes) { fail(FTB_ERR_BAD_SCENE, "bad BSP node link"); return depth; }
        int a = bspDepth(d.bsp_nodes[link].right, depth + 1);
        if (status != FTB_OK) return a;
        int b = bspDepth(d.bsp_nodes[link].left, depth + 1);
        return std::max(a, b);
    }
    void bspRanges(int link, std::vector<std::pair<int, int>>& ranges)
    {
        if (link < 0) {
            const ftb_bsp_leaf& lf = d.bsp_leaves[~link];
            if (lf.tri_count > 0) ranges.push_back({lf.tri_first, lf.tri_count});
            return;
        }
        bspRanges(d.bsp_nodes[link].right, ranges);
        bspRanges(d.bsp_nodes[link].left, ranges);
    }
    // Bounding sphere of a mesh's vertices in world space (centre of their box, farthest vertex), straight off the triangle
    // table: two passes, nothing stored (a 355 k-triangle mesh has a million vertices).
    Sphere boundOfMesh(const M34& w2m, int root, ItemBoxes& box)
    {
        M34 m2w;
        box = ItemBoxes();
        if (!invertAffine(w2m, m2w)) return kUnbounded;
        std::vector<std::pair<int, int>> ranges;
        bspRanges(root, ranges);
        if (ranges.empty()) { box = kNoBoxes; return kEmpty; }
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        auto world = [&](const double* p, double* w) {
            for (int r = 0; r < 3; ++r) w[r] = m2w.m[4 * r] * p[0] + m2w.m[4 * r + 1] * p[1] + m2w.m[4 * r + 2] * p[2] + m2w.m[4 * r + 3];
        };
        for (auto& rg : ranges)
            for (int i = 0; i < 3 * rg.second; ++i) {
                double w[3];
                world(d.triangles + 9 * (size_t)rg.first + 3 * (size_t)i, w);
                for (int r = 0; r < 3; ++r) { lo[r] = std::min(lo[r], w[r]); hi[r] = std::max(hi[r], w[r]); }
            }
        Sphere s;
        for (int r = 0; r < 3; ++r) s.c[r] = 0.5 * (lo[r] + hi[r]);
        double r2 = 0;
        for (auto& rg : ranges)
            for (int i = 0; i < 3 * rg.second; ++i) {
                double w[3];
                world(d.triangles + 9 * (size_t)rg.first + 3 * (size_t)i, w);
                const double dx = w[0] - s.c[0], dy = w[1] - s.c[1], dz = w[2] - s.c[2];
                r2 = std::max(r2, dx * dx + dy * dy + dz * dz);
            }
        s.r = std::sqrt(r2);
        if (!std::isfinite(s.r) || !std::isfinite(s.c[0]) || !std::isfinite(s.c[1]) || !std::isfinite(s.c[2])) return kUnbounded;
        box = worldBox(kIdentity, condition(w2m, m2w), lo, hi);  // the vertices' world-space box
        return s;
    }

    int addLeaf(int kind, const Ctx& cx, const M34& w2m, int surface, int prim, int payload, const std::vector<std::array<double, 3>>& modelPts, bool bounded)
    {
        (void)cx;
        Leaf lf = {};
        lf.kind = kind; lf.surface = surface; lf.prim = prim; lf.payload = payload;
        lf.identity = isIdentity(w2m) ? 1 : 0;
        std::memcpy(lf.w2m, w2m.m, sizeof(lf.w2m));
        L.leaves.push_back(lf);
        Sphere b = kUnbounded;
        ItemBoxes box;
        M34 m2w;
        if (bounded && invertAffine(w2m, m2w)) {
            b = boundOfPoints(m2w, modelPts);
            if (b.r >= 0 && !modelPts.empty()) {
                double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
                for (auto& p : modelPts)
                    for (int r = 0; r < 3; ++r) { lo[r] = std::min(lo[r], p[r]); hi[r] = std::max(hi[r], p[r]); }
                box = worldBox(m2w, condition(w2m, m2w), lo, hi);
            }
        }
        leafBound.push_back(b);
        leafBox.push_back(box);
        return (int)L.leaves.size() - 1;
    }

    // Emits the leaves of one PRIMITIVE instance in the reference's enumeration order.
    bool primitiveLeaves(const ftb_node& n, const Ctx& cx, std::vector<int>& out)
    {
        int surface = resolveSurface(cx);
        if (status != FTB_OK) return false;
        int prim = L.n_prims++;
        switch (n.a) {
        case FTB_PRIM_SPHERE: out.push_back(addLeaf(LEAF_SPHERE, cx, cx.w2m, surface, prim, 0, boxCorners(-1, 1, -1, 1, -1, 1), true)); break;
        case FTB_PRIM_PLANE: out.push_back(addLeaf(LEAF_PLANE, cx, cx.w2m, surface, prim, 0, {}, false)); break;
        case FTB_PRIM_SQUARE: out.push_back(addLeaf(LEAF_SQUARE, cx, cx.w2m, surface, prim, 0, boxCorners(0, 1, 0, 0, 0, 1), true)); break;
        case FTB_PRIM_CIRCLE: out.push_back(addLeaf(LEAF_CIRCLE, cx, cx.w2m, surface, prim, 0, boxCorners(-1, 1, 0, 0, -1, 1), true)); break;
        case FTB_PRIM_CYLINDER: out.push_back(addLeaf(LEAF_CYLINDER, cx, cx.w2m, surface, prim, 0, boxCorners(-1, 1, 0, 1, -1, 1), true)); break;
        case FTB_PRIM_CONE: out.push_back(addLeaf(LEAF_CONE, cx, cx.w2m, surface, prim, 0, boxCorners(-1, 1, 0, 1, -1, 1), true)); break;
        case FTB_PRIM_CUBE: out.push_back(addLeaf(LEAF_CUBE, cx, cx.w2m, surface, prim, 0, boxCorners(-.5, .5, -.5, .5, -.5, .5), true)); break;
        case FTB_PRIM_SOLIDCYLINDER:
            // Cylinder.solidCylinder (Cylinder.fs:25-29): group [top; bottom; sides] - one fused leaf in the cylinder's frame,
            // the parts' own transforms (translate (0,1,0) / rotate unitZ 180) are applied inside the kernel (render.cuh)
            out.push_back(addLeaf(LEAF_SOLIDCYL, cx, cx.w2m, surface, prim, 0, boxCorners(-1, 1, 0, 1, -1, 1), true));
            break;
        case FTB_PRIM_TRIANGLE: {
            if (n.b < 0 || n.b >= d.n_triangles) return fail(FTB_ERR_BAD_SCENE, "bad triangle index");
            const double* t = d.triangles + 9 * (size_t)n.b;
            out.push_back(addLeaf(LEAF_TRIANGLE, cx, cx.w2m, surface, prim, n.b, {{t[0], t[1], t[2]}, {t[3], t[4], t[5]}, {t[6], t[7], t[8]}}, true));
            break;
        }
        case FTB_PRIM_BSPMESH: {
            if (n.b < 0 || n.b >= d.n_meshes) return fail(FTB_ERR_BAD_SCENE, "bad mesh index");
            int depth = bspDepth(d.meshes[n.b].root, 0);
            if (status != FTB_OK) return false;
            L.max_bsp_depth = std::max(L.max_bsp_depth, depth);
            if (L.mesh_used.size() < (size_t)d.n_meshes) L.mesh_used.resize((size_t)d.n_meshes, 0);
            L.mesh_used[n.b] = 1;
            out.push_back(addLeaf(LEAF_MESH, cx, cx.w2m, surface, prim, n.b, {}, false));
            leafBound.back() = boundOfMesh(cx.w2m, d.meshes[n.b].root, leafBox.back());
            L.has_mesh = true;
            break;
        }
        default: return fail(FTB_ERR_BAD_SCENE, "bad primitive kind");
        }
        return true;
    }

    bool checkNode(int node, int depth)
    {
        if (node < 0 || node >= d.n_nodes) return fail(FTB_ERR_BAD_SCENE, "node index out of range");
        if (depth > 2048) return fail(FTB_ERR_BAD_SCENE, "scene graph too deep or cyclic");
        return true;
    }

    // Post-order program of a subtree that sits under a CSG node.  Returns the bound of what the
    // subtree can report and the list-stack depth it needs.
    // closed: every line crosses the subtree's surface an even number of times (sphere, cube, solidCylinder and their
    // combinations).  The device culls an item whose bound lies entirely behind the ray origin; for `subtract A B`
    // (bound = A's) and `intersect A B` (bound = one operand's) that is only right if the bounding operand is closed: an open
    // one (cylinder, cone, square, circle, triangle) crossed once at t < 0 leaves Csg.constructedSolid's inA / inB state
    // true for all t > 0 (Csg.fs:74-94) and the reference then reports the OTHER operand's crossings ahead of the origin.
    // `boxes` follows the same rules as `bound`.
    bool emitProgram(int node, Ctx cx, int depth, Sphere& bound, ItemBoxes& boxes, bool& empty, int& lists, bool& casts, bool& closed)
    {
        if (!checkNode(node, depth)) return false;
        const ftb_node& n = d.nodes[node];
        switch (n.kind) {
        case FTB_NODE_PRIMITIVE: {
            if (n.a == FTB_PRIM_BSPMESH) return fail(FTB_ERR_UNSUPPORTED, "bspMesh as a CSG operand is not supported (meshes emit no t<0 crossings, Triangle.fs:62)");
            std::vector<int> lv;
            if (!primitiveLeaves(n, cx, lv)) return false;
            bound = kEmpty; boxes = kNoBoxes; empty = true;
            for (int l : lv) {
                L.ops.push_back({OP_LEAF, l});
                bound = enclose(bound, leafBound[l], empty, false); empty = false;
                boxes = join(boxes, leafBox[l]);
                if (L.surfaces[L.leaves[l].surface].apply_lighting) casts = true;
            }
            if (lv.size() != 1) L.ops.push_back({OP_GROUP, (int)lv.size()});
            lists = (int)lv.size();
            closed = n.a == FTB_PRIM_SPHERE || n.a == FTB_PRIM_CUBE || n.a == FTB_PRIM_SOLIDCYLINDER;
            return true;
        }
        case FTB_NODE_TRANSFORM:
            if (n.a < 0 || n.a >= d.n_transforms) return fail(FTB_ERR_BAD_SCENE, "bad transform index");
            { M34 t; std::memcpy(t.m, d.transforms[n.a].w2m, sizeof(t.m)); cx.w2m = mul(t, cx.w2m); }
            return emitProgram(n.b, cx, depth + 1, bound, boxes, empty, lists, casts, closed);
        case FTB_NODE_MATERIAL:
            if (n.a < 0 || n.a >= d.n_materials) return fail(FTB_ERR_BAD_SCENE, "bad material index");
            cx.ops.push_back({n.kind, n.a});
            return emitProgram(n.b, cx, depth + 1, bound, boxes, empty, lists, casts, closed);
        case FTB_NODE_TEXTURE: case FTB_NODE_HUESHIFT: case FTB_NODE_IGNORELIGHT:
            cx.ops.push_back({n.kind, n.a});
            return emitProgram(n.b, cx, depth + 1, bound, boxes, empty, lists, casts, closed);
        case FTB_NODE_GROUP: {
            if (n.b < 0 || n.a < 0 || n.a + n.b > d.n_children) return fail(FTB_ERR_BAD_SCENE, "bad group range");
            bound = kEmpty; boxes = kNoBoxes; empty = true; lists = 0; closed = true;
            if (n.b == 0) { L.ops.push_back({OP_EMPTY, 0}); lists = 1; return true; }
            for (int i = 0; i < n.b; ++i) {
                Sphere b; ItemBoxes bx; bool e; int l; bool c = false;
                if (!emitProgram(d.children[n.a + i], cx, depth + 1, b, bx, e, l, casts, c)) return false;
                bound = enclose(bound, b, empty, e); empty = empty && e;
                boxes = join(boxes, bx);
                lists = std::max(lists, i + l);
                closed = closed && c;
            }
            if (n.b != 1) L.ops.push_back({OP_GROUP, n.b});
            return true;
        }
        case FTB_NODE_UNION: case FTB_NODE_INTERSECT: case FTB_NODE_SUBTRACT: case FTB_NODE_EXCLUDE: {
            Sphere ba, bb; ItemBoxes xa, xb; bool ea, eb; int la, lb; bool ca = false, cb = false;
            if (!emitProgram(n.a, cx, depth + 1, ba, xa, ea, la, casts, ca)) return false;
            if (!emitProgram(n.b, cx, depth + 1, bb, xb, eb, lb, casts, cb)) return false;
            lists = std::max(la, 1 + lb);
            closed = ca && cb;
            switch (n.kind) {
            case FTB_NODE_UNION: L.ops.push_back({OP_UNION, 0}); bound = enclose(ba, bb, ea, eb); boxes = join(xa, xb); empty = ea && eb; break;
            case FTB_NODE_EXCLUDE: L.ops.push_back({OP_EXCLUDE, 0}); bound = enclose(ba, bb, ea, eb); boxes = join(xa, xb); empty = ea && eb; break;
            case FTB_NODE_SUBTRACT:  // every reported crossing lies inside A's bound - as long as A is closed (see above)
                L.ops.push_back({OP_SUBTRACT, 0});
                bound = ca ? ba : kUnbounded; boxes = ca ? xa : ItemBoxes(); empty = ea;
                break;
            default:  // intersect: every reported crossing lies inside both operands' bounds; the bounding operand must be closed
                L.ops.push_back({OP_INTERSECT, 0});
                if (ea || eb) { bound = kEmpty; boxes = kNoBoxes; empty = true; }
                else {
                    const bool useA = ca && ba.r >= 0, useB = cb && bb.r >= 0;
                    if (useA && useB) { bound = (ba.r <= bb.r) ? ba : bb; boxes = (ba.r <= bb.r) ? xa : xb; }
                    else if (useA) { bound = ba; boxes = xa; }
                    else if (useB) { bound = bb; boxes = xb; }
                    else { bound = kUnbounded; boxes = ItemBoxes(); }
                    empty = false;
                }
                break;
            }
            L.has_csg = true;
            return true;
        }
        default: return fail(FTB_ERR_BAD_SCENE, "bad node kind");
        }
    }

    void pushItem(int kind, int a, int b, bool casts, const Sphere& bound, const ItemBoxes& boxes, bool empty)
    {
        Item it = {};
        it.kind = kind; it.a = a; it.b = b; it.casts_shadow = casts ? 1 : 0;
        Sphere s = empty ? Sphere{{0, 0, 0}, 0.0} : bound;
        it.bound_c[0] = s.c[0]; it.bound_c[1] = s.c[1]; it.bound_c[2] = s.c[2]; it.bound_r = s.r;
        L.items.push_back(it);
        L.item_boxes.push_back(empty ? kNoBoxes : boxes);
    }

    // Top-level walk: everything outside CSG nodes is a flat, ordered list of items.
    bool walk(int node, Ctx cx, int depth)
    {
        if (!checkNode(node, depth)) return false;
        const ftb_node& n = d.nodes[node];
        switch (n.kind) {
        case FTB_NODE_PRIMITIVE: {
            std::vector<int> lv;
            if (!primitiveLeaves(n, cx, lv)) return false;
            for (int l : lv) {
                L.leaves[l].top_level = 1;
                pushItem(ITEM_LEAF, l, 0, L.surfaces[L.leaves[l].surface].apply_lighting != 0, leafBound[l], leafBox[l], false);
            }
            return true;
        }
        case FTB_NODE_TRANSFORM:
            if (n.a < 0 || n.a >= d.n_transforms) return fail(FTB_ERR_BAD_SCENE, "bad transform index");
            { M34 t; std::memcpy(t.m, d.transforms[n.a].w2m, sizeof(t.m)); cx.w2m = mul(t, cx.w2m); }
            return walk(n.b, cx, depth + 1);
        case FTB_NODE_MATERIAL:
            if (n.a < 0 || n.a >= d.n_materials) return fail(FTB_ERR_BAD_SCENE, "bad material index");
            cx.ops.push_back({n.kind, n.a});
            return walk(n.b, cx, depth + 1);
        case FTB_NODE_TEXTURE: case FTB_NODE_HUESHIFT: case FTB_NODE_IGNORELIGHT:
            cx.ops.push_back({n.kind, n.a});
            return walk(n.b, cx, depth + 1);
        case FTB_NODE_GROUP:
            if (n.b < 0 || n.a < 0 || n.a + n.b > d.n_children) return fail(FTB_ERR_BAD_SCENE, "bad group range");
            for (int i = 0; i < n.b; ++i)
                if (!walk(d.children[n.a + i], cx, depth + 1)) return false;
            return true;
        case FTB_NODE_UNION: case FTB_NODE_INTERSECT: case FTB_NODE_SUBTRACT: case FTB_NODE_EXCLUDE: {
            int first = (int)L.ops.size();
            Sphere b; ItemBoxes bx; bool e = true; int lists = 0; bool casts = false, closed = false;
            if (!emitProgram(node, cx, depth, b, bx, e, lists, casts, closed)) return false;
            L.max_csg_lists = std::max(L.max_csg_lists, lists);
            const int count = (int)L.ops.size() - first;
            pushItem(ITEM_CSG, first, count, casts, b, bx, e);
            L.items.back().prog_first = first; L.items.back().prog_count = count;
            if (count == 3 && L.ops[first].kind == OP_LEAF && L.ops[first + 1].kind == OP_LEAF && L.ops[first + 2].kind >= OP_UNION) {
                Item& it = L.items.back();
                it.kind = ITEM_CSG2 | (L.ops[first + 2].kind << 8);
                it.a = L.ops[first].arg; it.b = L.ops[first + 1].arg;
            }
            else {
                // An operand may also be a Group of consecutive leaves (solidCylinder = [top; bottom; sides],
                // Cylinder.fs:25-29): `LEAF l .. LEAF l+k-1, GROUP k`.  The item stays a pair, each operand a run of leaves:
                // a / b = first leaf | (leaves - 1) << 24 (kernel feature FT_PAIRG).  Every CSG item of the bundled scenes
                // has one of these two shapes.
                auto operand = [&](int& at, int& packed) -> bool {
                    if (at >= first + count || L.ops[at].kind != OP_LEAF) return false;
                    const int l0 = L.ops[at].arg;
                    int k = 1;
                    while (at + k < first + count && L.ops[at + k].kind == OP_LEAF && L.ops[at + k].arg == l0 + k) ++k;
                    if (k == 1) { packed = l0; at += 1; return true; }
                    // a run of k leaves must be closed by GROUP k (else the last leaf belongs to the next operand)
                    if (at + k < first + count && L.ops[at + k].kind == OP_GROUP && L.ops[at + k].arg == k && k <= 8 && l0 < (1 << 22)) {
                        packed = l0 | ((k - 1) << 24); at += k + 1; return true;
                    }
                    packed = l0; at += 1;
                    return true;
                };
                int at = first, pa = 0, pb = 0;
                if (operand(at, pa) && operand(at, pb) && at == first + count - 1 && L.ops[at].kind >= OP_UNION) {
                    Item& it = L.items.back();
                    it.kind = ITEM_CSG2 | (L.ops[at].kind << 8);
                    it.a = pa; it.b = pb;
                }
            }
            return true;
        }
        default: return fail(FTB_ERR_BAD_SCENE, "bad node kind");
        }
    }
};

}  // namespace

namespace {

// ---- BVH over a mesh's triangles (binned SAH, leaves of <= 4 triangles) ---------------------------------------
struct Box {
    double lo[3], hi[3];
    void reset() { for (int k = 0; k < 3; ++k) { lo[k] = 1e300; hi[k] = -1e300; } }
    void add(const double* p) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], p[k]); hi[k] = std::max(hi[k], p[k]); } }
    void add(const Box& b) { for (int k = 0; k < 3; ++k) { lo[k] = std::min(lo[k], b.lo[k]); hi[k] = std::max(hi[k], b.hi[k]); } }
    double area() const
    {
        double e[3] = {hi[0] - lo[0], hi[1] - lo[1], hi[2] - lo[2]};
        if (e[0] < 0) return 0;
        return 2.0 * (e[0] * e[1] + e[1] * e[2] + e[2] * e[0]);
    }
};

struct BvhBuilder {
    const double* tris;            // scene triangles, 9 doubles each
    std::vector<int32_t> ref;      // triangle indices being partitioned
    std::vector<Box> tbox;         // per ref position
    std::vector<double> cen;       // 3 per ref position
    Lowered& L;
    int slotBase;
    int maxDepth = 0;

    BvhBuilder(const double* t, Lowered& l) : tris(t), L(l), slotBase(0) {}

    Box boxOf(int b, int e) const
    {
        Box x; x.reset();
        for (int i = b; i < e; ++i) x.add(tbox[i]);
        return x;
    }
    void swapRef(int a, int b)
    {
        std::swap(ref[a], ref[b]); std::swap(tbox[a], tbox[b]);
        for (int k = 0; k < 3; ++k) std::swap(cen[3 * a + k], cen[3 * b + k]);
    }
    int build(int b, int e, int depth)
    {
        maxDepth = std::max(maxDepth, depth);
        const int n = e - b;
        if (n <= 4 || depth >= 60) {
            if (n > 7) {  // depth cap with a fat run: split it into a chain so that every leaf holds <= 4 (count has 3 bits)
                const int mid = b + 4;
                return makeNode(b, mid, e, depth);
            }
            return ~(((slotBase + b) << 3) | n);
        }
        Box cb; cb.reset();
        for (int i = b; i < e; ++i) cb.add(&cen[3 * i]);
        int axis = 0;
        double ext = -1;
        for (int k = 0; k < 3; ++k) if (cb.hi[k] - cb.lo[k] > ext) { ext = cb.hi[k] - cb.lo[k]; axis = k; }
        int mid = -1;
        if (ext > 0) {  // binned SAH on the widest centroid axis
            const int NB = 16;
            Box bb[NB]; int cnt[NB];
            for (int k = 0; k < NB; ++k) { bb[k].reset(); cnt[k] = 0; }
            const double scale = NB / ext;
            auto binOf = [&](int i) { int q = (int)((cen[3 * i + axis] - cb.lo[axis]) * scale); return q < 0 ? 0 : (q >= NB ? NB - 1 : q); };
            for (int i = b; i < e; ++i) { int q = binOf(i); bb[q].add(tbox[i]); ++cnt[q]; }
            double rightArea[NB]; int rightCnt[NB];
            Box acc; acc.reset(); int c = 0;
            for (int k = NB - 1; k > 0; --k) { acc.add(bb[k]); c += cnt[k]; rightArea[k] = acc.area(); rightCnt[k] = c; }
            acc.reset(); c = 0;
            double best = 1e300; int bestK = -1;
            for (int k = 0; k < NB - 1; ++k) {
                acc.add(bb[k]); c += cnt[k];
                if (c == 0 || rightCnt[k + 1] == 0) continue;
                const double cost = acc.area() * c + rightArea[k + 1] * rightCnt[k + 1];
                if (cost < best) { best = cost; bestK = k; }
            }
            if (bestK >= 0) {
                int i = b, j = e - 1;
                while (i <= j) { if (binOf(i) <= bestK) ++i; else { swapRef(i, j); --j; } }
                mid = i;
            }
        }
        if (mid <= b || mid >= e) {  // all centroids coincide (or SAH found nothing): split the run in half
            mid = b + n / 2;
        }
        return makeNode(b, mid, e, depth);
    }
    int makeNode(int b, int mid, int e, int depth)
    {
        const int idx = (int)L.bvh_nodes.size();
        L.bvh_nodes.push_back(BvhNode());
        const int l = build(b, mid, depth + 1);
        const int r = build(mid, e, depth + 1);
        const Box lb = boxOf(b, mid), rb = boxOf(mid, e);
        BvhNode& nd = L.bvh_nodes[idx];
        nd.child[0] = l; nd.child[1] = r;
        const Box* bx[2] = {&lb, &rb};
        for (int c = 0; c < 2; ++c)
            for (int k = 0; k < 3; ++k) {
                nd.dlo[c][k] = bx[c]->lo[k]; nd.dhi[c][k] = bx[c]->hi[k];
                float flo = (float)bx[c]->lo[k], fhi = (float)bx[c]->hi[k];  // round outward
                if ((double)flo > bx[c]->lo[k]) flo = std::nextafterf(flo, -INFINITY);
                if ((double)fhi < bx[c]->hi[k]) fhi = std::nextafterf(fhi, INFINITY);
                nd.lo[c][k] = flo; nd.hi[c][k] = fhi;
            }
        return idx;
    }
};

// triangles of a reference BSP in BspMesh.intersect's enumeration order: right subtree, then left (BspMesh.fs:72-75)
void enumerateBsp(const ftb_scene_desc& d, int link, std::vector<int32_t>& out, int depth)
{
    if (depth > 300) return;
    if (link < 0) {
        const ftb_bsp_leaf& lf = d.bsp_leaves[~link];
        for (int i = 0; i < lf.tri_count; ++i) out.push_back(lf.tri_first + i);
        return;
    }
    enumerateBsp(d, d.bsp_nodes[link].right, out, depth + 1);
    enumerateBsp(d, d.bsp_nodes[link].left, out, depth + 1);
}

void buildMeshIndex(const ftb_scene_desc& d, Lowered& L)
{
    std::vector<std::vector<int32_t>> order;
    enumerateMeshes(d, L, order);
    L.mesh_root.assign((size_t)std::max(0, d.n_meshes), ~0);
    for (int m = 0; m < d.n_meshes; ++m) {
        const std::vector<int32_t>& tri = order[(size_t)m];
        BvhBuilder bb(d.triangles, L);
        bb.slotBase = (int)L.bvh_tri.size();
        bb.ref = tri;
        const int n = (int)tri.size();
        std::vector<int32_t> seqOf((size_t)std::max(1, d.n_triangles), 0);
        bb.tbox.resize(n); bb.cen.resize(3 * (size_t)n);
        for (int i = 0; i < n; ++i) {
            const double* t = d.triangles + 9 * (size_t)tri[i];
            bb.tbox[i].reset();
            bb.tbox[i].add(t); bb.tbox[i].add(t + 3); bb.tbox[i].add(t + 6);
            for (int k = 0; k < 3; ++k) bb.cen[3 * i + k] = 0.5 * (bb.tbox[i].lo[k] + bb.tbox[i].hi[k]);
            seqOf[tri[i]] = i;
        }
        L.mesh_root[m] = n == 0 ? ~0 : bb.build(0, n, 0);
        for (int i = 0; i < n; ++i) { L.bvh_tri.push_back(bb.ref[i]); L.bvh_seq.push_back(seqOf[bb.ref[i]]); }
        L.max_bvh_depth = std::max(L.max_bvh_depth, bb.maxDepth);
    }
}

}  // namespace

void enumerateMeshes(const ftb_scene_desc& d, const Lowered& L, std::vector<std::vector<int32_t>>& order)
{
    order.assign((size_t)std::max(0, d.n_meshes), std::vector<int32_t>());
    for (int m = 0; m < d.n_meshes; ++m)
        if ((size_t)m < L.mesh_used.size() && L.mesh_used[m]) enumerateBsp(d, d.meshes[m].root, order[(size_t)m], 0);
}

void buildMeshIndexHost(const ftb_scene_desc& d, Lowered& L) { buildMeshIndex(d, L); }

int lower_scene(const ftb_scene_desc& d, Lowered& out, std::string& err, bool build_mesh_index)
{
    if (!d.nodes || d.n_nodes <= 0) { err = "scene has no nodes"; return FTB_ERR_BAD_SCENE; }
    if ((d.n_children > 0 && !d.children) || (d.n_transforms > 0 && !d.transforms) || (d.n_materials > 0 && !d.materials) ||
        (d.n_textures > 0 && !d.textures) || (d.n_images > 0 && !d.images) || (d.n_meshes > 0 && !d.meshes) ||
        (d.n_bsp_nodes > 0 && !d.bsp_nodes) || (d.n_bsp_leaves > 0 && !d.bsp_leaves) || (d.n_triangles > 0 && !d.triangles) ||
        (d.n_lights > 0 && !d.lights)) {
        err = "null table with non-zero count";
        return FTB_ERR_BAD_ARG;
    }
    for (int i = 0; i < d.n_children; ++i)
        if (d.children[i] < 0 || d.children[i] >= d.n_nodes) { err = "child index out of range"; return FTB_ERR_BAD_SCENE; }
    for (int i = 0; i < d.n_nodes; ++i) {
        const ftb_node& n = d.nodes[i];
        bool fn = n.kind >= FTB_NODE_TRANSFORM && n.kind <= FTB_NODE_IGNORELIGHT;
        bool csg = n.kind >= FTB_NODE_UNION && n.kind <= FTB_NODE_EXCLUDE;
        if ((fn && (n.b < 0 || n.b >= d.n_nodes)) || (csg && (n.a < 0 || n.a >= d.n_nodes || n.b < 0 || n.b >= d.n_nodes))) {
            err = "node link out of range";
            return FTB_ERR_BAD_SCENE;
        }
        if (n.kind == FTB_NODE_TEXTURE && (n.a < 0 || n.a >= d.n_textures)) { err = "bad texture index"; return FTB_ERR_BAD_SCENE; }
    }
    for (int i = 0; i < d.n_lights; ++i) {
        if (d.lights[i].kind < 0 || d.lights[i].kind > FTB_LIGHT_POINT) { err = "bad light kind"; return FTB_ERR_BAD_SCENE; }
        if (d.lights[i].kind == FTB_LIGHT_SOFT_DIRECTIONAL) {
            out.has_soft_light = true;
            if (d.lights[i].samples < 0) { err = "negative light sample count"; return FTB_ERR_BAD_SCENE; }
        }
    }
    Lowerer lw(d, out, err);
    Ctx cx;
    cx.w2m = kIdentity;
    lw.walk(d.root, cx, 0);
    if (lw.status != FTB_OK) return lw.status;
    unsigned f = 0;
    for (const Leaf& lf : out.leaves) {
        if (lf.kind == LEAF_CUBE) f |= 0x01;
        if (lf.kind == LEAF_SQUARE || lf.kind == LEAF_CIRCLE || lf.kind == LEAF_CYLINDER || lf.kind == LEAF_CONE || lf.kind == LEAF_SOLIDCYL) f |= 0x02;
        if (lf.kind == LEAF_TRIANGLE || lf.kind == LEAF_MESH) f |= 0x04;
    }
    for (const Item& it : out.items) {
        if ((it.kind & 0xff) == ITEM_CSG2) f |= 0x08;  // a two-operand CSG pair
        if ((it.kind & 0xff) == ITEM_CSG2 && ((it.a >> 24) || (it.b >> 24))) f |= 0x400;  // ... with a run of leaves as an operand
        if (it.kind == ITEM_CSG) f |= 0x80;            // a general CSG program
    }
    // pairs in a scene with the round leaf kinds share one copy of the (then large) leaf intersectors instead of inlining two
    if ((f & 0x08) && (f & 0x02)) f |= 0x400;
    if (out.has_texture) f |= 0x10;
    if (out.has_rough) f |= 0x20;
    if (out.has_soft_light) f |= 0x40;
    for (const Leaf& lf : out.leaves)
        if (lf.top_level && (lf.kind == LEAF_PLANE || lf.kind == LEAF_SQUARE || lf.kind == LEAF_CIRCLE)) f |= 0x100;
    if (wantsOriginTable((int)out.items.size(), d.n_lights)) f |= kFeatOriginTable;
    out.features = f;
    if (out.has_mesh && build_mesh_index) buildMeshIndex(d, out);
    return FTB_OK;
}

}  // namespace ftb
