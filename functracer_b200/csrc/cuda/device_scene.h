// device_scene.h — the structure-of-arrays scene and frame descriptors the kernels consume.
// Templated on the arithmetic type: float for the product path, double for the FP64
// verification build.  Filled by api.cu from ftb::Lowered.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ftb {

constexpr int kHitCap = 32;    // per-ray CSG hit stack entries
constexpr int kMaxLists = 12;  // per-ray CSG list stack depth
constexpr int kBspStack = 64;  // per-ray mesh traversal stack
#ifndef FTB_BLOCK_THREADS
#define FTB_BLOCK_THREADS 128
#endif
constexpr int kBlockThreads = FTB_BLOCK_THREADS;
// Most samples of one unit of the blend ring (render.cuh): a launch covers at most this many samples per pixel, frames with
// more are rendered in several passes that continue the same left fold.  128 (FP32) / 64 (FP64) in general; 256 for the variants
// of simple scenes (spheres / planes only: no cube, round leaf, mesh or CSG), whose samples are cheap: at 64 spp a 128-sample unit
// is two pixels and its fold keeps 6 of 32 lanes busy (moon, 64 spp: -7.7 % with 256; the house family: +10 %, the larger ring
// takes shared memory away from the L1 those scenes need - hence per variant).
constexpr unsigned kHeavyFeatures = 0x01u | 0x02u | 0x04u | 0x08u | 0x80u;  // FT_CUBE | FT_ROUND | FT_MESH | FT_CSG | FT_CSGN
template <typename R, unsigned FEAT> struct UnitCap {
#ifdef FTB_UNIT_CAP
    static constexpr int value = sizeof(R) == 4 ? FTB_UNIT_CAP : 64;
#else
    static constexpr int value = sizeof(R) == 4 ? ((FEAT & kHeavyFeatures) == 0 ? 256 : 128) : 64;
#endif
};

// Tile -> shard dealing (multi-GPU).  The tiles of a frame are cut into groups of n consecutive tiles (row-major); group g gives
// one tile to every shard and is every shard's local tile g.  WHICH tile of the group a shard gets is rotated by a hash of g:
// dealing tile t to shard t % n hands every shard fixed tile COLUMNS whenever the tile row length is a multiple of n (an 8K
// frame is 480 tiles wide: 8 GPUs would each render vertical stripes, and a scene of upright objects then loads them unevenly).
__host__ __device__ inline int shardRot(int group, int n) { return n > 1 ? (int)((((unsigned)group * 2654435761u) >> 10) % (unsigned)n) : 0; }
__host__ __device__ inline int tileOfLocal(int ltile, int shard, int n)  // may be >= the frame's tile count in the last group: no such tile
{
    int k = shard - shardRot(ltile, n);
    if (k < 0) k += n;
    return ltile * n + k;
}
__host__ __device__ inline int shardOfTile(int tile, int n)  // its local index is tile / n
{
    const int g = tile / n;
    return (tile - g * n + shardRot(g, n)) % n;
}

template <typename R>
struct V4;
template <>
struct V4<float> {
    typedef float4 type;
};
template <>
struct V4<double> {
    typedef double4 type;
};

// Kernel feature mask: which primitive classes / shading terms a kernel variant contains.  A scene is
// rendered by the smallest compiled variant whose mask covers lower.h's Lowered::features.
enum Feature : unsigned {
    FT_CUBE = 0x01,   // LEAF_CUBE
    FT_ROUND = 0x02,  // LEAF_SQUARE, LEAF_CIRCLE, LEAF_CYLINDER, LEAF_CONE, LEAF_SOLIDCYL
    FT_MESH = 0x04,   // LEAF_TRIANGLE, LEAF_MESH (BSP traversal)
    FT_CSG = 0x08,    // CSG items that are a binary op of two single leaves (evaluated in registers)
    FT_TEX = 0x10,    // grid / image textures, sphere uv
    FT_ROUGH = 0x20,  // Oren-Nayar diffuse
    FT_RNG = 0x40,    // soft directional lights, depth of field
    FT_CSGN = 0x80,   // any other CSG item (general post-order program, inlined)
    FT_PLANAR = 0x100,  // a top-level plane / square / circle leaf exists (FP32 self-intersection guard, render.cuh)
    FT_TABLE = 0x200,  // enough top-level items for the common-origin bound table to pay (lower.h kFeatOriginTable, render.cuh)
    FT_PAIRG = 0x400,  // CSG pairs (FT_CSG) walk both operands through ONE copy of the leaf intersectors: scenes with many leaf kinds
                       // (instruction footprint) and pairs whose operand is a run of leaves (lower.cpp, render.cuh csgPair)
    FT_MESHPK = 0x800,  // a LARGE mesh: mesh leaves are walked by the whole warp (render.cuh packetMesh) instead of by each lane (intersectMesh);
                        // variants with FT_MESH but without this bit only contain the per-lane walk, FT_ALL contains both (DevScene::mesh_packet)
    FT_ALL = 0xfff,
    FT_TMASK = 0x1000  // not a scene feature: a variant that reads the per-tile item masks (DevFrame::tile_items, render.cuh TileMasks),
                       // compiled beside the plain one for the Makefile's F32_TMASK_FEATS; api.cu launches it when the masks pay
};

enum StatSlot : int {
    ST_PRIMARY = 0,
    ST_SHADOW,
    ST_REFLECTION,
    ST_SHADED,
    ST_LEAF0,  // 10 leaf kinds follow (ftb::LeafKind order)
    ST_XFORM = ST_LEAF0 + 10,
    ST_BSP_NODES,
    ST_BOUND_TESTS,
    ST_CSG_OPS,
    ST_TRI_TESTS_IN_MESH,
    ST_BOUND_FAST,  // bound tests answered from the common-origin table (one dot product + compare)
    ST_COUNT
};

template <typename R>
struct DevScene {
    typedef typename V4<R>::type R4;
    // leaves
    const R4* leaf_w2m;     // 3 rows per leaf
    const R4* leaf_p0;      // per leaf: the world point that maps to the model origin (a point of the plane for planar leaves)
    const int4* leaf_meta;  // x = kind | identity << 8, y = surface, z = prim, w = payload
    int n_leaves;
    // top-level items in enumeration order
    const int4* items;     // x = kind | CSG op << 8 | kind word of leaf a << 12 | of leaf b << 21 (kind word: leaf_meta.x & 0x1ff), y = a, z = b, w = casts_shadow
    const int2* item_prog; // CSG items: x = first op, y = op count of the general program
    const R4* item_bound;  // xyz = centre, w = (inflated radius)^2 of a conservative bounding sphere (+inf: unbounded)
    const R4* item_bound2; // FP32: the same bounds, two neighbouring items interleaved for the packed test: (x0 x1 y0 y1) (z0 z1 w0 w1), padded to an even count
    const unsigned* item_casts;  // bit j of word w: item 32 w + j can block light (something under it has applyLighting)
    const unsigned* item_mesh;   // bit j of word w: item 32 w + j is a mesh leaf
    int mesh_packet;             // 1: mesh leaves are walked by the whole warp (render.cuh packetMesh; large meshes), 0: by each lane (intersectMesh)
    int n_items;
    const int2* ops;  // CSG programs: x = kind, y = arg
    // surfaces
    const R4* surf_a;    // colour.rgb, roughness
    const R4* surf_b;    // reflectance, shineyness, 0, 0
    const int4* surf_i;  // texture, hue, apply_lighting, 0
    // textures
    const int4* tex_i;  // op_first, op_count, base_kind, image
    const R4* tex_c1;
    const R4* tex_c2;
    const int* texop_kind;
    const R* texop_ab;  // 2 per op
    const uchar4* texels;
    const int4* img_i;  // x = first texel, y = width, z = height
    // meshes: the device's own BVH over each mesh's triangles (lower.h BvhNode)
    const int* mesh_root;    // per mesh: root link (>= 0 node, < 0 ~((first << 3) | count))
    const R4* bvh_node;      // 4 per node (64 bytes): one row per axis, (L.lo, R.lo, L.hi, R.hi) of x, of y, of z (render.cuh boxEntry2: both children's
                             // slabs as packed pairs), then (child link L, child link R, -, -) as bits (FP32) or values (FP64)
    const R4* bvh_tris;      // 3 per slot: (v0, seq) (e1, triangle index) (e2, -); the ints stored as reals
    const R4* tris;          // 3 per scene triangle: v0, e1 = v1 - v0, e2 = v2 - v0 (LEAF_TRIANGLE, normals)
    // lights
    const int2* light_i;  // kind, samples
    const R4* light_a;    // v.xyz (dir or pos), tan(scatter / 2)
    const R4* light_b;    // falloff c, l, q
    const R4* light_c;    // colour
    int n_lights;
    R cyl_c, cyl_s;  // cos / sin of the -180 degree rotation about z that puts the bottom cap of a solidCylinder in place (Cylinder.fs:27), as the host computes them
};

template <typename R>
struct DevFrame {
    int mode;  // 0 = camera sample grid, 1 = explicit ray list (render_kernel); samples_kernel: explicit rays, spp per pixel (2)
    int gw, gh;  // the whole frame's sample grid (W x H, or (W+1) x (H+1) in corner mode): ray directions and RNG keys
    int spp;              // samples per pixel of the whole frame
    int s_base, s_count;  // this launch renders samples [s_base, s_base + s_count) of every pixel (s_count <= UnitCap)
    int run;              // consecutive samples of one pixel a lane takes at a time (divides s_count)
    unsigned rpp_magic;   // floor(2^32 / (s_count / run)) + 1: q / rpp == __umulhi(q, rpp_magic) for q < 65536
    int bw_log, bh_log;   // the work queue hands out blocks of (1 << bw_log) x (1 << bh_log) pixels (bw <= 8)
    int n_blocks;         // blocks (mode 0: of the traced tiles) or groups of 32 rays (mode 1) in the queue
    int tiles_x;             // 16 x 16 tiles per row of the WINDOW's tile grid, which starts at (wx0, wy0)
    unsigned tiles_x_magic;  // floor(2^32 / tiles_x) + 1: tile / tiles_x == __umulhi(tile, magic); 0 = frame too large for that, divide
    int n_local_tiles;  // tiles of the window this shard renders
    int shard_index, shard_count;
    long long n_rays;  // mode 1
    R cam_o[3], cam_k[3], cam_i[3], cam_j[3];
    R pw, ph, tlx, tly;
    R primary_slack;  // 2e-4 |cam_o|: see the common-origin bound table in render.cuh
    int has_focus;
    R focal, tan_half_aperture;
    const R* jitter;     // 2 * spp
    const double* rays;  // mode 1: o.xyz d.xyz
    int recursion_limit;
    unsigned long long seed;
    R* out;  // mode 0: tile-major [local tile][256][3]; mode 1: [ray][3]
    int* dbg_prim;
    int* dbg_sub;
    double* dbg_t;
    const int* tile_order;  // mode 0, optional: local tile indices, costliest first (longest-processing-time-first)
    unsigned int* tile_counter;
    unsigned int* overflow;
    unsigned long long* stats;  // ST_COUNT slots (stats kernels only)
    // Last, so that the fields above keep their offsets (and the 16-byte alignment of the camera rows, which the kernels load
    // as vectors) in the kernel's parameter block.
    int wx0, wy0, wx1, wy1;  // mode 0: the window [wx0, wx1) x [wy0, wy1) of the sample grid this frame renders (whole frame: 0, 0, gw, gh)
    int dbg_w;               // mode 0: row width of the debug planes (wx1 - wx0): they hold the window's samples only
    // mode 0: the clear tiles (tiles.h) are the last ones of tile_order; their blocks, n_blocks ... n_blocks + n_clear_blocks - 1,
    // are written without tracing by clear_kernel (api.cu), not by the render kernel
    int n_clear_blocks;
    // mode 0, FP32 kernels with top-level planar leaves: one byte per tile of the window's grid (global tile index), bit k =
    // every primary fragment of the tile on leaf lit_leaf sees directional light k unblocked (lit_tiles.h); nullptr: none
    const unsigned char* lit_tiles;
    int lit_leaf;
    // mode 0, FP32 kernels, scenes of <= 32 items: one word per tile of the window's grid (global tile index), bit i = item i may
    // be hit by a primary ray of the tile (tiles.h); the tile's primary rays trace no other item.  Set only for the FT_TMASK
    // variants (api.cu prepareFrame).  nullptr: every item
    const unsigned* tile_items;
};

// A batch of ray queries (query_kernel, render.cuh): caller-supplied rays traced exactly as given, nearest hit or occlusion.
// Every output pointer may be null (not wanted).
struct DevQuery {
    const double* rays;   // o.xyz d.xyz per ray
    const double* max_t;  // occlusion queries: the segment's end per ray; nullptr = nearest-hit queries
    long long n;          // rays
    int n_groups;         // groups of 32 rays in the queue
    int record;           // 1: some plane beyond t / prim / sub is wanted (finalise runs)
    double* t;
    int* prim;
    int* sub;
    double* p;        // 3 per ray
    double* normal;   // 3 per ray
    double* colour;   // 3 per ray
    double* surface;  // 4 per ray: roughness, reflectance, shineyness, apply_lighting
    int* blocked;     // occlusion queries
    unsigned int* group_counter;
    unsigned int* overflow;
    unsigned long long* stats;  // ST_COUNT slots (stats kernels only)
};

// A batch of crossing queries (crossings_kernel, render.cuh): every crossing of each ray with t_min <= t < t_max, sorted by t,
// the first max_hits of them kept.  Output planes are max_hits entries wide per ray; every output pointer but counts may be null.
struct DevCrossings {
    const double* rays;  // o.xyz d.xyz per ray
    long long n;         // rays
    int n_groups;        // groups of 32 rays in the queue
    int max_hits;        // 1 .. FTB_MAX_CROSSINGS
    int record;          // 1: some plane beyond t / prim / sub is wanted (finalise runs)
    double t_min, t_max;
    int* counts;
    double* t;
    int* prim;
    int* sub;
    double* p;        // 3 per entry
    double* normal;   // 3 per entry
    double* colour;   // 3 per entry
    double* surface;  // 4 per entry: roughness, reflectance, shineyness, apply_lighting
    unsigned int* group_counter;
    unsigned int* overflow;
    unsigned long long* stats;  // ST_COUNT slots (counting kernel only)
};

// A batch of path queries (path_kernel, paths.cu): getColourForRay on caller-supplied rays, every level and light recorded.
// Level planes are depth entries wide per ray, light planes depth * n_lights; every output pointer may be null.
struct DevPaths {
    const double* rays;                     // o.xyz d.xyz per ray
    const unsigned long long* sample_keys;  // RNG key per ray; nullptr = the ray's index (what ftb_shade_rays uses)
    long long n;                            // rays
    int n_groups;                           // groups of 32 rays in the queue
    int recursion_limit;                    // depth = recursion_limit + 1 levels
    unsigned long long seed;
    int record;  // 1: some hit plane beyond t / prim / sub is wanted
    int* levels;
    double* colour;        // 3 per ray
    double* ray_od;        // 6 per level
    double* weight;        // 1 per level
    double* t;             // 1 per level
    int* prim;             // 1 per level
    int* sub;              // 1 per level
    double* p;             // 3 per level
    double* normal;        // 3 per level
    double* hit_colour;    // 3 per level
    double* surface;       // 4 per level: roughness, reflectance, shineyness, apply_lighting
    double* intensity;     // 1 per (level, light)
    double* light_dir;     // 3 per (level, light)
    double* light_colour;  // 3 per (level, light)
    unsigned int* group_counter;
    unsigned int* overflow;
    unsigned long long* stats;  // ST_COUNT slots (counting kernel only)
};

#ifdef __CUDACC__
// Block c of a mode-0 frame's work queue: its first pixel's slot in the tile buffer, its origin in the whole frame's sample
// grid, its width and its pixel count (clipped to the window; 0 for a tile the last shard group lacks).
template <typename R>
__device__ __forceinline__ void openBlock(const DevFrame<R>& F, unsigned c, int& slot0, int& x0, int& y0, int& w, int& npix)
{
    // a 16x16 tile holds 2^(8 - bw_log - bh_log) blocks of (1 << bw_log) x (1 << bh_log) pixels
    const int bpt_log = 8 - F.bw_log - F.bh_log, bpr_log = 4 - F.bw_log;
    const int sub = (int)(c & ((1u << bpt_log) - 1u));
    const int tpos = (int)(c >> bpt_log);
    const int ltile = F.tile_order ? __ldg(F.tile_order + tpos) : tpos;  // costliest tiles first
    const int tile = tileOfLocal(ltile, F.shard_index, F.shard_count);
    const int sx = (sub & ((1 << bpr_log) - 1)) << F.bw_log, sy = (sub >> bpr_log) << F.bh_log;
    // the tile grid is the window's; px / py are whole-frame sample-grid coordinates
    const int tile_y = F.tiles_x_magic ? (int)__umulhi((unsigned)tile, F.tiles_x_magic) : tile / F.tiles_x;
    x0 = F.wx0 + (tile - tile_y * F.tiles_x) * FTB_TILE_W + sx;
    y0 = F.wy0 + tile_y * FTB_TILE_H + sy;
    slot0 = ltile * FTB_TILE_PIXELS + sy * FTB_TILE_W + sx;
    w = max(1, min(1 << F.bw_log, F.wx1 - x0));
    npix = max(0, min(1 << F.bw_log, F.wx1 - x0)) * max(0, min(1 << F.bh_log, F.wy1 - y0));
}
#endif

// A compiled kernel variant (render_variant.cu, one translation unit per FEAT mask / precision).
template <typename R>
struct Variant {
    unsigned feat;
    int unit_cap;    // UnitCap<R, feat>: samples per pixel one launch covers
    bool has_stats;  // the counting kernel is only compiled into the FT_ALL variants
    cudaError_t (*launch)(const DevScene<R>& s, const DevFrame<R>& f, bool stats, int sm_count, cudaStream_t stream, int* launches);
    cudaError_t (*query)(const DevScene<R>& s, const DevQuery& q, bool stats, int sm_count, cudaStream_t stream, int* launches);
    // samples_kernel (ftb_shade_samples): f in mode 2, f.n_rays pixels of f.spp rays each; keys may be null (the rays' indices)
    cudaError_t (*samples)(const DevScene<R>& s, const DevFrame<R>& f, const unsigned long long* keys, bool stats, int sm_count, cudaStream_t stream,
                           int* launches);
};

}  // namespace ftb
