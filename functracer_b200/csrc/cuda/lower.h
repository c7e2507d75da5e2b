// lower.h — host-side lowering of the reference's SceneGraph (as delivered through
// ftb_scene_desc) into the flat, leaf-centric form the CUDA kernels consume.
//
// What Scene.intersect (FuncTracer/Scene.fs:67-104) does by building closures is done here by
// building tables:
//   * every PRIMITIVE instance becomes one or more LEAVES with ONE pre-composed world->model
//     matrix (the product of the Transform nodes on its path; t is invariant under
//     Transform.transform, Transform.fs:84-86, so nearest-hit only ever needs this matrix);
//   * every leaf gets a statically RESOLVED SURFACE: the surface ops on its path
//     (Ray.fs:47-59) are maps over hits, applied innermost first, so their net effect per leaf
//     is known before any ray is traced (SURVEY.md A.5);
//   * the top-level object list is flattened into ITEMS in the reference's enumeration order
//     (Ray.group, Ray.fs:34), which is also the tie-break order of Scene.closest;
//   * each CSG subtree becomes a post-order PROGRAM over a per-ray hit stack (Csg.fs:74-94).
#pragma once

#include <cstdint>
#include <string>
#include <vector>

#include "../../../include/functracer_b200.h"

namespace ftb {

// The common-origin bound table (render.cuh) is used when the item list is long enough to matter and the table fits;
// such scenes carry the feature bit 0x200 (device_scene.h FT_TABLE).
constexpr int kOriginCap = 256;     // rows x items (4 KB of shared memory in FP32)
constexpr int kOriginMinItems = 8;  // measured again with the packed table walk: at 4 items (the moon scene) the table costs +4.2 %, sample +8 % (profiles/r2ae_table_min4_ab.txt)
constexpr unsigned kFeatOriginTable = 0x200;
inline bool wantsOriginTable(int n_items, int n_lights) { return n_items >= kOriginMinItems && (1 + n_lights) * ((n_items + 1) & ~1) <= kOriginCap; }  // an origin's rows: render.cuh tabStride

enum LeafKind : int32_t {
    LEAF_SPHERE = 0,
    LEAF_PLANE = 1,
    LEAF_SQUARE = 2,
    LEAF_CIRCLE = 3,
    LEAF_CYLINDER = 4,  // open side surface (Cylinder.cylinder)
    LEAF_CONE = 5,
    LEAF_CUBE = 6,  // the six squares of Cube.cube fused: sub = face
    LEAF_TRIANGLE = 7,
    LEAF_MESH = 8,
    LEAF_SOLIDCYL = 9  // the three parts of Cylinder.solidCylinder (top circle, bottom circle, sides) fused: sub = part
};
constexpr int kLeafKinds = 10;

// ITEM_CSG2: a CSG node whose two operands are single leaves (`subtract cube (scale .65 sphere)`) or Groups of
// consecutive leaves (`subtract (solidCylinder) (sphere)`): the device evaluates it in registers when neither operand
// yields more than two crossings; kind = ITEM_CSG2 | (CsgOpKind << 8), a / b = first leaf | (leaves - 1) << 24.
// Every CSG item also keeps its general post-order program (prog_first / prog_count).
enum ItemKind : int32_t { ITEM_LEAF = 0, ITEM_CSG = 1, ITEM_CSG2 = 2 };

enum CsgOpKind : int32_t {
    OP_LEAF = 0,   // arg = leaf index: push its hit list
    OP_GROUP = 1,  // arg = n: concatenate the top n lists (Ray.group)
    OP_EMPTY = 2,  // push an empty list (Group [])
    OP_UNION = 3,
    OP_INTERSECT = 4,
    OP_SUBTRACT = 5,
    OP_EXCLUDE = 6
};

struct Leaf {
    int32_t kind;
    int32_t surface;
    int32_t prim;     // depth-first PRIMITIVE-instance index (the debug plane's prim_id)
    int32_t payload;  // mesh index | triangle index | solidCylinder part (reported as sub_id)
    int32_t identity; // 1 = w2m is the identity (no transform on the path)
    int32_t top_level; // 1 = the leaf is an item of its own (not an operand of a CSG node)
    int32_t reserved[2];
    double w2m[12];   // composed world->model, row-major 3x4
};

struct Surface {
    int32_t texture;  // -1 = constant colour
    int32_t hue;      // number of (r,g,b)->(b,r,g) permutations applied after the colour source, mod 3
    int32_t apply_lighting;
    int32_t reserved;
    double colour[3];
    double roughness, reflectance, shineyness;
};

struct TexOp {
    int32_t kind;  // FTB_TEX_SCALE | FTB_TEX_ROTATE
    int32_t reserved;
    double a, b;  // scale: (x, y); rotate: (cos, sin)
};

struct TexDef {
    int32_t op_first, op_count;  // uv ops in application order (outermost first, Scene.fs:68-74)
    int32_t base_kind;           // FTB_TEX_GRID | FTB_TEX_IMAGE
    int32_t image;
    double c1[3], c2[3];
};

struct Item {
    int32_t kind;
    int32_t a;  // ITEM_LEAF: leaf index; ITEM_CSG: first op;  ITEM_CSG2: leaf A
    int32_t b;  // ITEM_CSG: op count;                          ITEM_CSG2: leaf B
    int32_t prog_first, prog_count;  // CSG items: the post-order program
    int32_t casts_shadow;  // 0 = every leaf under it has applyLighting = false (Scene.fs:121)
    // conservative world-space bounding sphere of everything the item can report (radius < 0: unbounded)
    double bound_c[3];
    double bound_r;
};

struct CsgOp {
    int32_t kind;
    int32_t arg;
};

// A leaf's model-space bounding box carried to world space (a parallelepiped: its 8 transformed corners), and the
// condition number of the leaf's transform, by which the intersectors' model-space rounding grows on the way to world space.
struct WorldBox {
    double corner[8][3];
    double cond;
};
// Boxes whose union holds every crossing an item can report, combined by the rules of its bounding sphere (DESIGN.md §2).
// valid = false: the item has no such boxes (its sphere is its only bound).  Host-only: tiles.h uses them to find clear tiles.
struct ItemBoxes {
    bool valid = false;
    std::vector<WorldBox> boxes;
};

// The device-side index over a mesh's triangles.  BspMesh.intersect (BspMesh.fs:67-76) visits every branch
// whose AABB the ray's line touches, right subtree before left, and Scene.closest then keeps the smallest
// t >= 0, first in that order on ties.  Which triangle that is does not depend on the shape of the tree,
// only on the triangle set and on the enumeration order; so the device traverses its own BVH (built here
// over the same - already clipped - triangles, front to back, culling against the best t so far) and
// breaks ties by `seq`, the triangle's rank in the reference's right-before-left enumeration.
struct BvhNode {
    float lo[2][3];  // child boxes, rounded outward from the double-precision triangle bounds
    float hi[2][3];
    int32_t child[2];  // >= 0: node index; < 0: ~((first << 3) | count), a run of `count` <= 4 slots in bvh_tri
    double dlo[2][3], dhi[2][3];  // the same boxes in double for the FP64 verification build
};

struct Lowered {
    std::vector<BvhNode> bvh_nodes;
    std::vector<int32_t> bvh_tri;    // slot -> index into the scene's triangles[]
    std::vector<int32_t> bvh_seq;    // slot -> enumeration rank within its mesh
    std::vector<int32_t> mesh_root;  // per mesh: link of the root (same encoding as BvhNode::child)
    std::vector<char> mesh_used;     // per mesh: referenced (and validated) by a bspMesh primitive
    int32_t max_bvh_depth = 0;
    std::vector<Leaf> leaves;
    std::vector<Surface> surfaces;
    std::vector<TexOp> tex_ops;
    std::vector<TexDef> textures;
    std::vector<Item> items;
    std::vector<ItemBoxes> item_boxes;  // per item
    std::vector<CsgOp> ops;
    int32_t n_prims = 0;
    int32_t max_csg_lists = 0;  // deepest list stack any program needs
    int32_t max_bsp_depth = 0;
    bool has_csg = false, has_mesh = false, has_texture = false, has_image = false;
    bool has_soft_light = false, has_rough = false;
    // Kernel features this scene needs, as device_scene.h `Feature` bits (cube 1, round 2, mesh 4, csg 8,
    // texture 16, Oren-Nayar 32, rng 64, general CSG 128, top-level planar leaf 256, bound table 512, shared-copy pairs 1024; api.cu adds 2048 for a large mesh);
    // camera depth of field adds rng at render time.
    unsigned features = 0;
};

// Returns FTB_OK or a negative ftb_status with a message in err.  build_mesh_index = false leaves the mesh index
// (bvh_nodes, bvh_tri, bvh_seq, mesh_root) to the caller: the device build of bvh_build.h, or buildMeshIndexHost.
int lower_scene(const ftb_scene_desc& d, Lowered& out, std::string& err, bool build_mesh_index = true);

// order[m] = the triangles of mesh m in BspMesh.intersect's enumeration order (right subtree before left,
// BspMesh.fs:72-75); empty for meshes no bspMesh primitive uses.
void enumerateMeshes(const ftb_scene_desc& d, const Lowered& L, std::vector<std::vector<int32_t>>& order);
// The host build of the mesh index (binned SAH), the fallback of the device build.
void buildMeshIndexHost(const ftb_scene_desc& d, Lowered& L);

}  // namespace ftb
