/// P/Invoke face of libfunctracer_b200.so — field for field include/functracer_b200.h (ABI version 4;
/// tests/test_fsharp_binding.py lays these structs out by the CLR's rules and compares them with the header's).
/// Blittable structs, Sequential layout (the C compiler's natural alignment: 4-byte ints, 8-byte doubles / pointers).
module Native

open System
open System.Runtime.InteropServices

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbNode =
    val mutable kind: int
    val mutable a: int
    val mutable b: int
    val mutable reserved: int
    new (k, a, b) = { kind = k; a = a; b = b; reserved = 0 }

// ftb_transform = 12 + 12 doubles, row-major 3x4: m2w = matrix t, w2m = matrix (inverse t) (Transform.fs:55-71, 81-82).
// It is passed as a plain float[] of 24 doubles per transform (SceneFlatten), so no struct is declared for it.

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbMaterial =
    val mutable r: float
    val mutable g: float
    val mutable b: float
    val mutable roughness: float
    val mutable reflectance: float
    val mutable shineyness: float
    val mutable applyLighting: int
    val mutable reserved: int

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbTexture =
    val mutable kind: int      // 0 image, 1 grid, 2 scale, 3 rotate
    val mutable inner: int
    val mutable image: int
    val mutable reserved: int
    val mutable p0: float
    val mutable p1: float
    val mutable p2: float
    val mutable p3: float
    val mutable p4: float
    val mutable p5: float

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbImage =
    val mutable rgb24: nativeint
    val mutable width: int
    val mutable height: int

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbBspNode =
    val mutable minX: float
    val mutable minY: float
    val mutable minZ: float
    val mutable maxX: float
    val mutable maxY: float
    val mutable maxZ: float
    val mutable left: int      // >= 0: index into bsp_nodes; < 0: ~index into bsp_leaves
    val mutable right: int

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbBspLeaf =
    val mutable triFirst: int
    val mutable triCount: int

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbMesh =
    val mutable root: int
    val mutable reserved: int

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbLight =
    val mutable kind: int      // 0 directional, 1 soft directional, 2 point
    val mutable samples: int
    val mutable vx: float
    val mutable vy: float
    val mutable vz: float
    val mutable falloffC: float
    val mutable falloffL: float
    val mutable falloffQ: float
    val mutable scatterRad: float
    val mutable cr: float
    val mutable cg: float
    val mutable cb: float

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbSceneDesc =
    val mutable root: int
    val mutable nNodes: int
    val mutable nodes: nativeint
    val mutable nChildren: int
    val mutable children: nativeint
    val mutable nTransforms: int
    val mutable transforms: nativeint
    val mutable nMaterials: int
    val mutable materials: nativeint
    val mutable nTextures: int
    val mutable textures: nativeint
    val mutable nImages: int
    val mutable images: nativeint
    val mutable nMeshes: int
    val mutable meshes: nativeint
    val mutable nBspNodes: int
    val mutable bspNodes: nativeint
    val mutable nBspLeaves: int
    val mutable bspLeaves: nativeint
    val mutable nTriangles: int
    val mutable triangles: nativeint   // 9 doubles per triangle
    val mutable nLights: int
    val mutable lights: nativeint

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbCamera =
    val mutable ox: float
    val mutable oy: float
    val mutable oz: float
    val mutable lx: float
    val mutable ly: float
    val mutable lz: float
    val mutable ux: float
    val mutable uy: float
    val mutable uz: float
    val mutable fovYRad: float
    val mutable aspect: float
    val mutable hasFocus: int
    val mutable reserved: int
    val mutable focalLength: float
    val mutable apertureRad: float

[<Struct; StructLayout(LayoutKind.Sequential)>]
type FtbRenderParams =
    val mutable width: int
    val mutable height: int
    val mutable spp: int
    val mutable sampling: int        // 0 jitter, 1 corner
    val mutable jitterXy: nativeint  // 2 * spp doubles drawn on the host as Image.fs:101-105 does
    val mutable recursionLimit: int  // 8 (Shading.fs:142)
    val mutable precision: int       // 0 FP32, 1 FP64 verification build
    val mutable seed: uint64
    val mutable outFormat: int       // 0 RGB f64 (Bitmap.pixels), 1 RGB f32, 2 RGBA8 (Image.write's toByte)
    val mutable shardIndex: int
    val mutable shardCount: int
    val mutable nGpus: int
    val mutable collectStats: int
    val mutable bandIndex: int       // ftb_render_tiles_device only (ABI 4): one band of tile rows of the shard; 0 / 0 = all
    val mutable bandCount: int
    val mutable reserved: int

[<Literal>]
let Lib = "functracer_b200"
[<Literal>]
let AbiVersion = 4

[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_abi_version()
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_device_count()
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern nativeint ftb_last_error()
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_scene_create(FtbSceneDesc& desc, nativeint& scene)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern void ftb_scene_destroy(nativeint scene)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_render(nativeint scene, FtbCamera& camera, FtbRenderParams& p, nativeint outPixels, nativeint dbgOrNull, nativeint statsOrNull)
/// the pixels [x0, x1) x [y0, y1) of the frame p describes, bit-identical to ftb_render there; outPixels and the debug
/// planes hold the window only ((x1 - x0) * (y1 - y0) pixels, row-major)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_render_window(nativeint scene, FtbCamera& camera, FtbRenderParams& p, int x0, int y0, int x1, int y1, nativeint outPixels, nativeint dbgOrNull, nativeint statsOrNull)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_shade_rays(nativeint scene, nativeint raysOD, int64 n, FtbRenderParams& p, nativeint outRgb, nativeint dbgOrNull, nativeint statsOrNull)
/// Scene.closest (Scene.fs:112-118) on n caller-supplied rays (o.xyz d.xyz, traced exactly as given, no slightOffset).
/// hitOut is the address of a pinned nativeint[7]: the plane pointers of ftb_hit_out in its order (t, prim_id, sub_id, p,
/// normal, colour, surface; 0n = not wanted)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_intersect_rays(nativeint scene, nativeint raysOD, int64 n, FtbRenderParams& p, nativeint hitOut, nativeint statsOrNull)
/// Scene.intersect (Scene.fs:67-104) on n caller-supplied rays: every crossing with tMin <= t < tMax, sorted by t (equal t in the
/// reference's order), counts[i] crossings per ray (may exceed maxHits), the first maxHits of them written to the planes of
/// hitOut (as for ftb_intersect_rays, maxHits entries per ray: entry (i, k) at i * maxHits + k; unused slots read as a miss)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_intersect_all_rays(nativeint scene, nativeint raysOD, int64 n, int maxHits, float tMin, float tMax, FtbRenderParams& p, nativeint hitOut, int[] counts, nativeint statsOrNull)
/// Shading.getColourForRay (Shading.fs:109-147) level by level on n caller-supplied rays, shaded as ftb_shade_rays shades them.
/// pathOut is the address of a pinned nativeint[14]: the plane pointers of ftb_path_out in its order (levels, colour, ray_od,
/// weight, the 7 of ftb_hit_out, intensity, light_dir, light_colour; 0n = not wanted).  D = p.recursionLimit + 1 level entries
/// per ray (entry (i, k) at i * D + k), L lights per level (entry (i, k, l) at (i * D + k) * L + l).  keysOrNull: n uint64
/// sample keys of the soft lights' RNG, 0n = the ray's index (what ftb_shade_rays uses)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_trace_paths(nativeint scene, nativeint raysOD, nativeint keysOrNull, int64 n, FtbRenderParams& p, nativeint pathOut, nativeint statsOrNull)
/// SamplingStrategy.generateRays (Image.fs:100-111) as the render kernel runs it: the primary ray (o.xyz d.xyz, before
/// slightOffset, after depth-of-field jitter) and the RNG key ((py * gw + px) * spp + s) of every sample of the window
/// [x0, x1) x [y0, y1), in the debug planes' order (sample-major within a pixel; corner sampling: the corner grid).
/// raysODOrNull: 6 doubles per sample, keysOrNull: one uint64 per sample (0n = not wanted)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_frame_rays(nativeint scene, FtbCamera& camera, FtbRenderParams& p, int x0, int y0, int x1, int y1, nativeint raysODOrNull, nativeint keysOrNull)
/// Shading.shade + JitterSampling.blendPixels (Image.fs:112-116) on caller-supplied rays: nPixels * p.spp rays (sample s of pixel
/// i is ray i * p.spp + s), each shaded as ftb_shade_rays shades it with the RNG key keysOrNull[i * spp + s] (0n = the ray's
/// index), each pixel blended as ftb_render blends it; out = nPixels pixels in p.outFormat (2 = RGBA8: Image.write's bytes)
[<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
extern int ftb_shade_samples(nativeint scene, nativeint raysOD, nativeint keysOrNull, int64 nPixels, FtbRenderParams& p, nativeint out, nativeint dbgOrNull, nativeint statsOrNull)

let lastError () = Marshal.PtrToStringAnsi (ftb_last_error ())
let check rc = if rc <> 0 then failwithf "functracer_b200 status %d: %s" rc (lastError ())
/// the structs above are only valid against the ABI they were written for
let checkAbi () = if ftb_abi_version () <> AbiVersion then failwithf "libfunctracer_b200 has ABI %d, this binding is for %d" (ftb_abi_version ()) AbiVersion
