"""Scenes that land on each specialised FP32 kernel (csrc/Makefile F32_FEATS; api.cu pickVariant launches the compiled variant
with the fewest feature bits that covers a scene's mask, lower.cpp).  The bundled scenes and the fuzz suite reach most
variants with one scene family each; every generator here draws only on what its variant covers, so that the variant's own
code (packed transforms, the non-RUNS pair with its csgGeneral fallback, the RUNS pair walk, the inlined general CSG
evaluator, the per-lane mesh walk, the 256-sample blend units ...) meets rotated, mirrored, far-away, padded and nested cases.

tests/test_variant_cover_cpu.py pins where every scene lands with the real lowering; tests/test_gpu_variants.py renders them
against the oracle and checks the per-pixel fold exactly.

A scene is a VScene: options, a list of top-level objects and a list of lights, so that the fold test can wrap every top-level
object in an unlit material of its own (VScene.fold).  Meshes are PLY files written into a directory of the caller's."""
import os

import numpy as np

import large_mesh_scenes as lms
from functracer_b200 import scenes

RES = (96, 72)
LIGHTS_HARD = ["positional pos (3,6,-5) falloff (1,0.02,0.01) colour (0.9,0.85,0.8)", "directional dir (-0.4,-1,0.6) colour (0.4,0.45,0.5)"]
FOLD_LIGHT = "directional dir (0.3,-1,0.5) colour (1,1,1)"
OPS = ["union", "subtract", "intersect", "exclude"]


def _num(x):
    s = "%.4f" % x
    return s if not s.startswith("-0.0000") else "0.0000"


def _v(x):
    return "(" + ",".join(_num(c) for c in x) + ")"


def _colour(rng):
    return _v(rng.uniform(0.1, 1.0, size=3))


class VScene:
    """camera: the camera line; objects: top-level object texts; lights: light lines; files: {name: (verts, faces)} written
    as PLY next to the scene (assets then come from that directory)."""

    def __init__(self, name, variant, camera, objects, lights, spp=2, sampling=None, files=None):
        self.name, self.variant, self.camera, self.objects, self.lights = name, variant, camera, list(objects), list(lights)
        self.spp, self.sampling, self.files = spp, sampling, dict(files or {})

    def _assets(self, d):
        if not self.files:
            return scenes.asset_dir()
        for fn, (v, f) in self.files.items():
            p = os.path.join(d, fn)
            if not os.path.exists(p):
                lms.write_ply(p, v, f)
        return d

    def text(self, d, spp=None, res=RES, sampling=None):
        """(scene text, asset directory)."""
        samples = sampling or self.sampling or ("samples %d" % (spp or self.spp))
        head = "%s\n%s\nres %d %d\n\n" % (self.camera, samples, res[0], res[1])
        return head + "\n\n".join(self.objects) + "\n\n" + "\n".join(self.lights) + "\n", self._assets(d)

    def fold_colours(self):
        """A dyadic colour (multiples of 1/64) per top-level object: their sums over any sample count are exact."""
        rng = np.random.default_rng(len(self.objects) * 7919 + sum(map(ord, self.name)))
        return rng.integers(1, 64, size=(len(self.objects), 3)) / 64.0

    def fold(self, d, spp, res=RES, sampling=None):
        """The same geometry with every top-level object unlit in a dyadic colour of its own, under one directional light:
        every sample's colour is then exactly its object's colour (Shading.fs shadeIfRequired), or 0 for a miss.  The outer
        material replaces every inner one (Ray.setMaterial); `roughness` keeps a rough variant's feature bit.
        Returns (text, assets, colours)."""
        cols = self.fold_colours()
        rough = " roughness 0.5" if self.variant == 0x030 else ""
        exact = lambda c: "(%s)" % ",".join("%.6f" % x for x in c)  # a multiple of 1/64 has at most 6 decimals
        objs = ["(ignoreLight (material diffuse %s%s reflectance 0 shineyness 0 %s))" % (exact(c), rough, o) for c, o in zip(cols, self.objects)]
        fs = VScene(self.name, self.variant, self.camera, objs, [FOLD_LIGHT], files=self.files)
        text, assets = fs.text(d, spp=spp, res=res, sampling=sampling)
        return text, assets, cols


def _xform(rng, inner, mirror=True):
    """rotate about a random axis, scale non-uniformly, and (mirror) flip one axis."""
    s = rng.uniform(0.5, 1.3, size=3)
    if mirror and rng.random() < 0.5:
        s[int(rng.integers(0, 3))] *= -1.0
    axis = rng.uniform(-1, 1, size=3)
    axis[np.abs(axis) < 0.1] = 0.3
    return "(rotate %s %s (scale %s %s))" % (_v(axis), _num(rng.uniform(-170, 170)), _v(s), inner)


def _material(rng, reflect=True):
    refl = float(rng.choice([0.0, 0.3, 0.6])) if reflect else 0.0
    return "material diffuse %s reflectance %s shineyness %s" % (_colour(rng), _num(refl), _num(float(rng.choice([0, 5, 20]))))


# ---- 0x000 / 0x100: spheres (and a plane), packed world -> model transforms ---------------------------------------------
# FP32 cancellation in (world point - translation).  Much farther out the FP32 hit point's own rounding (ulp(4 600) = 4.9e-4)
# exceeds the reference's 1e-4 ray offsets: at (2400, -1300, 3700) the ids still agree but ~9 % of pixels miss 1/255 (B200).
FAR = np.array([60.5, -20.25, 50.75])


def spheres(seed, plane=False, far=True, n=6):
    rng = np.random.default_rng(seed)
    off = FAR if far else np.zeros(3)
    objs = []
    for _ in range(n):
        objs.append("(translate %s (%s %s))" % (_v(off + rng.uniform([-2, -1, -1.5], [2, 1.5, 2])), _material(rng), _xform(rng, "sphere")))
    if plane:  # a reflective ground plane whose horizon crosses the frame (the FP32 planar self-skip)
        objs.append("(material diffuse %s reflectance 0.5 shineyness 0 (translate %s plane))" % (_colour(rng), _v(off + [0, -1.5, 0])))
        cam = "camera pos %s lookat %s up (0,1,0) fov 60 ratio 1.3333" % (_v(off + [0.3, -0.9, -7]), _v(off + [0, -0.95, 0]))
    else:
        cam = "camera pos %s lookat %s up (0,1,0) fov 55 ratio 1.3333" % (_v(off + [rng.uniform(-1, 1), rng.uniform(0.5, 2), -6.5]), _v(off))
    lights = ["positional pos %s falloff (1,0.02,0.01) colour (0.9,0.85,0.8)" % _v(off + [3, 6, -5]), LIGHTS_HARD[1]]
    return VScene("%s%d" % ("plane" if plane else "spheres", seed), 0x100 if plane else 0x000, cam, objs, lights, spp=1 + seed % 3)


# ---- 0x209: cubes and single-leaf sphere / cube pairs, the common-origin table with scalar code --------------------------
CUBE_CAMERA = "camera pos (0.4,3.5,-9) lookat (0,0,1.5) up (0,1,0) fov 60 ratio 1.3333"
CUBE_LIGHTS = ["directional dir (-0.5,-1,0.4) colour (0.7,0.7,0.65)", "positional pos (-3,7,-4) falloff (1,0.01,0.005) colour (0.6,0.6,0.7)"]


def _cube_pair(rng, op):
    a = "(rotate %s %s (scale %s cube))" % (_v(rng.uniform(-1, 1, size=3) + 0.05), _num(rng.uniform(0, 90)), _v(rng.uniform(0.25, 0.45, size=3)))
    b = "(translate %s (scale %s sphere))" % (_v(rng.uniform(-0.25, 0.25, size=3)), _num(rng.uniform(0.3, 0.5)))
    return "(%s %s %s)" % (op, a, b) if rng.random() < 0.5 else "(%s %s %s)" % (op, b.replace("sphere", "cube"), a)


def cubes(n_items, seed=0, pad_to=None, reflect=True):
    """A flattened cube as the floor and n_items - 1 cubes and pairs (all four operators in turn) on a grid in view.
    pad_to: more cubes, far below and behind the camera where no ray of the frame reaches them, up to pad_to items."""
    rng = np.random.default_rng(seed + 100 * n_items)
    objs = ["(material diffuse (0.5,0.55,0.5) reflectance 0 shineyness 0 (translate (0,-0.6,2) (scale (9,0.1,9) cube)))"]
    cols = int(np.ceil(np.sqrt(n_items - 1)))
    for i in range(n_items - 1):
        x, z = i % cols, i // cols
        pos = [(x - (cols - 1) / 2.0) * 7.0 / cols, rng.uniform(-0.1, 0.6), z * 6.0 / cols - 0.5]
        geo = _cube_pair(rng, OPS[i % 4]) if i % 3 != 2 else "(rotate (0,1,0) %s (scale %s cube))" % (_num(rng.uniform(0, 90)), _num(3.0 / cols))
        if i % 3 != 2:
            geo = "(scale %s %s)" % (_num(min(1.0, 6.0 / cols)), geo)
        objs.append("(translate %s (%s %s))" % (_v(pos), _material(rng, reflect), geo))
    name = "cubes%d" % n_items + ("" if reflect else "_matte")
    if pad_to:
        for k in range(pad_to - n_items):
            objs.append("(translate %s (scale 0.5 cube))" % _v([k % 10 - 5.0, -500.0, -500.0 - k // 10]))
        name += "_pad%d" % pad_to
    return VScene(name, 0x209, CUBE_CAMERA, objs, CUBE_LIGHTS, spp=1 + n_items % 3)


def max_table_items(n_lights):
    """lower.h wantsOriginTable: (1 + lights) rows of the even-padded item count within kOriginCap = 256 slots."""
    n = 8
    while (1 + n_lights) * ((n + 2) & ~1) <= 256:
        n += 1
    return n


def cube_pairs_all_ops(seed):
    """Larger pairs, each operator several times, sphere-first and cube-first, with rays that leave A and enter B."""
    rng = np.random.default_rng(seed)
    objs = ["(material diffuse (0.5,0.5,0.55) reflectance 0.3 shineyness 0 (translate (0,-1.2,2) (scale (8,0.1,8) cube)))"]
    for i in range(8):
        op = OPS[i % 4]
        a = "(rotate %s %s (scale %s cube))" % (_v(rng.uniform(-1, 1, size=3) + 0.05), _num(rng.uniform(0, 90)), _v(rng.uniform(0.5, 0.8, size=3)))
        b = "(translate %s (scale %s sphere))" % (_v(rng.uniform(-0.5, 0.5, size=3)), _num(rng.uniform(0.55, 0.8)))
        geo = "(%s %s %s)" % (op, a, b) if i < 4 else "(%s %s %s)" % (op, b, a)
        objs.append("(translate %s (%s %s))" % (_v([(i % 4) * 2.2 - 3.3, 0.0, (i // 4) * 2.5]), _material(rng), geo))
    return VScene("pairs_ops%d" % seed, 0x209, CUBE_CAMERA, objs, CUBE_LIGHTS, spp=2)


# ---- 0x74b: pairs whose operands are runs of leaves (the RUNS pair walk) ---------------------------------------------------
RUN_LEAVES = ["sphere", "cube", "cylinder", "cone"]
SOFT = ["softdirectional dir (-0.6,-1,0.5) samples %d scatter 12 colour (0.5,0.5,0.45)", "directional dir (0.5,-1,0.3) colour (0.3,0.3,0.35)"]
FLOOR_PLANE = "(material diffuse (0.45,0.5,0.5) reflectance 0.2 shineyness 0 (translate (0,-1.2,0) plane))"
RUN_CAMERA = "camera pos (0.5,3,-9) lookat (0,0,1) up (0,1,0) fov 60 ratio 1.3333"


def _run(rng, k):
    """An operand: one leaf, or a group of k leaves (LEAF l .. LEAF l+k-1, GROUP k in the lowered program)."""
    leaves = ["(translate %s (scale %s %s))" % (_v(rng.uniform(-0.35, 0.35, size=3)), _num(rng.uniform(0.3, 0.5)), rng.choice(RUN_LEAVES)) for _ in range(k)]
    return leaves[0] if k == 1 else "(group %s)" % " ".join(leaves)


def runs(seed, soft_samples=2):
    """Pairs of runs of 1..8 leaves under all four operators, the closing-rule shapes (a leaf followed by a run whose first
    index continues it; a run followed by a leaf), solidCylinder operands, a plane floor and a soft light."""
    rng = np.random.default_rng(seed)
    objs, pos = [FLOOR_PLANE], []
    shapes = [(k, int(rng.integers(1, 9))) for k in range(1, 9)]
    shapes += [(1, 2), (2, 1), (1, 8), (8, 1)]
    for i, (ka, kb) in enumerate(shapes):
        geo = "(%s %s %s)" % (OPS[(i + seed) % 4], _run(rng, ka), _run(rng, kb))
        objs.append("(translate %s (%s %s))" % (_v([(i % 4) * 2.0 - 3.0, 0.0, (i // 4) * 2.0]), _material(rng), geo))
    objs.append("(translate (3.5,0,5) (%s (subtract solidCylinder (translate (0.2,0.4,-0.3) (scale 0.6 sphere)))))" % _material(rng))
    lights = [SOFT[0] % soft_samples, SOFT[1]]
    return VScene("runs%d_soft%d" % (seed, soft_samples), 0x74b, RUN_CAMERA, objs, lights, spp=1 + seed % 3)


# ---- 0x3c3: the inlined general CSG evaluator ---------------------------------------------------------------------------
def _nested(rng, depth):
    if depth == 0:
        return "(translate %s (scale %s %s))" % (_v(rng.uniform(-0.3, 0.3, size=3)), _num(rng.uniform(0.35, 0.6)), rng.choice(RUN_LEAVES + ["solidCylinder"]))
    return "(%s %s %s)" % (rng.choice(OPS), _nested(rng, depth - 1), _nested(rng, depth - 1 if rng.random() < 0.5 else 0))


def nested(seed, soft_samples=1):
    """General CSG programs (three or more leaves, not a pair of runs), a 9-leaf run (no longer a pair), a plane floor and a
    soft light."""
    rng = np.random.default_rng(seed)
    objs = [FLOOR_PLANE]
    for i in range(7):
        objs.append("(translate %s (%s %s))" % (_v([(i % 4) * 2.0 - 3.0, 0.0, (i // 4) * 2.2]), _material(rng), _nested(rng, 2 + i % 2)))
    objs.append("(translate (1,0,4.4) (%s (subtract %s (scale 0.5 sphere))))" % (_material(rng), _run(rng, 9)))
    lights = [SOFT[0] % soft_samples, SOFT[1]]
    return VScene("nested%d_soft%d" % (seed, soft_samples), 0x3c3, RUN_CAMERA, objs, lights, spp=1 + seed % 3)


def _row(n, left_deep):
    """A union of n disjoint spheres in a row along +z: a ray along the row crosses all of them, 2n crossings.  Left-deep
    ((a b) c) ... keeps two pending lists and stacks every crossing; right-deep (a (b (c ...))) keeps n lists."""
    leaves = ["(translate (0,0,%d) (scale 0.4 sphere))" % k for k in range(n)]
    if left_deep:
        g = leaves[0]
        for x in leaves[1:]:
            g = "(union %s %s)" % (g, x)
        return g
    g = leaves[-1]
    for x in reversed(leaves[:-1]):
        g = "(union %s %s)" % (x, g)
    return g


def csg_limit(n, left_deep):
    """render.cuh evalCsg: kHitCap = 32 stacked crossings (left-deep rows: 16 spheres fit, 17 overflow at run time) and
    kMaxLists = 12 pending lists (right-deep rows: 12 fit, 13 are refused when the scene is created).  The soft light has
    samples, so that the rows' lit pixels are finite and their colour is compared too."""
    cam = "camera pos (0.05,0.03,-4) lookat (0,0,8) up (0,1,0) fov 30 ratio 1.3333"
    objs = [FLOOR_PLANE, "(material diffuse (0.7,0.5,0.4) reflectance 0.3 shineyness 10 %s)" % _row(n, left_deep)]
    return VScene("row%d_%s" % (n, "left" if left_deep else "right"), 0x3c3, cam, objs, [SOFT[0] % 2, SOFT[1]], spp=2)


# ---- 0x050 / 0x030: textures on spheres; depth of field / Oren-Nayar ---------------------------------------------------
def _texture(rng):
    if rng.random() < 0.4:
        t = 'image "moon.ppm"'
    else:
        t = "grid %s %s" % (_colour(rng), _colour(rng))
    t = "(scale (%s,%s) %s)" % (_num(rng.uniform(0.1, 0.9)), _num(rng.uniform(0.1, 0.9)), t)
    if rng.random() < 0.6:
        t = "(rotate %s %s)" % (_num(rng.uniform(5, 85)), t)
    return t


def textured(seed, rough=False):
    """Textured spheres (grid and image, scaled and rotated) under rotated, mirrored transforms.  0x050: depth of field;
    0x030: Oren-Nayar surfaces, some with a specular term (a shadow ray) and some without (no shadow ray, render.cuh)."""
    rng = np.random.default_rng(seed)
    objs = []
    for i in range(6):
        mat = "material diffuse %s%s reflectance %s shineyness %s" % (_colour(rng), " roughness %s" % _num(rng.uniform(0.2, 0.8)) if rough else "",
                                                                      _num(float(rng.choice([0.0, 0.3]))), "0" if rough and i % 2 else "10")
        objs.append("(translate %s (%s (texture %s %s)))" % (_v(rng.uniform([-2.5, -1, -1], [2.5, 1.5, 2.5])), mat, _texture(rng), _xform(rng, "sphere")))
    cam = "camera pos (0.3,1.2,-6.5) lookat (0,0,0.5) up (0,1,0) fov 55 ratio 1.3333"
    if not rough:
        cam += " focus (6.5,1.2)"
    return VScene("%s%d" % ("rough" if rough else "dof", seed), 0x030 if rough else 0x050, cam, objs, LIGHTS_HARD, spp=2 + seed % 3)


# ---- 0x004: small meshes, the per-lane mesh walk -----------------------------------------------------------------------
def _mesh_material(refl=0.0):
    return "material diffuse (0.8,0.7,0.6) reflectance %g shineyness 10" % refl


MESH_CAMERA = "camera pos (1,2.5,-7) lookat (0,0.5,0) up (0,1,0) fov 60 ratio 1.3333"


def small_meshes(seed):
    """bspMesh and mesh (triangle items) instances of two small fields, rotated, mirrored and scaled, several instances of
    one file, and spheres."""
    rng = np.random.default_rng(seed)
    files = {"a.ply": lms.field(16, 8), "b.ply": lms.field(8, 8, planar=True)}
    objs = []
    for i, (kw, fn) in enumerate([("bspMesh 6", "a.ply"), ("bspMesh 0", "a.ply"), ("mesh", "b.ply"), ("bspMesh 3", "b.ply"), ("bspMesh 6", "a.ply")]):
        inner = '(scale 1.6 (translate (-1,-0.5,0) %s "%s"))' % (kw, fn)
        objs.append("(translate %s (%s %s))" % (_v([(i % 3) * 2.2 - 2.2, (i // 3) * 1.8 - 0.5, 0.4 * i]), _material(rng), _xform(rng, inner)))
    objs.append("(translate (2.5,1.5,2) (%s (scale 0.6 sphere)))" % _material(rng))
    return VScene("meshes%d" % seed, 0x004, MESH_CAMERA, objs, LIGHTS_HARD, spp=2, files=files)


def mesh_tie(mesh_first, n=1024, large=False):
    """A bspMesh of an n-triangle field and triangle items (`mesh`) that copy 31 of its triangles exactly: every ray
    through a copied triangle ties in t, and the earlier item wins (Scene.closest).  n < 32 768: the per-lane walk (0x004);
    n = 32 768: the warp's walk (0x804).  Hard lights only."""
    n = lms.LARGE_MESH if large else n
    v, f = lms.field(128, 128, n_tris=n)
    pick = np.linspace(0, n - 1, 31).astype(int)
    dup = [f[k] for k in pick]
    body = ['bspMesh 10 "big.ply"', 'mesh "dup.ply"']
    if not mesh_first:
        body.reverse()
    objs = ["(%s (group %s))" % (_mesh_material(), " ".join(body))]
    cam = "camera pos (8,1.5,-6) lookat (8,0.8,0) up (0,1,0) fov 60 ratio 1.3333"
    return VScene("tie%s_%s" % ("_large" if large else "", "mesh_first" if mesh_first else "copies_first"), 0x804 if large else 0x004, cam, objs,
                  lms.HARD_LIGHTS.strip().split("\n"), spp=1, files={"big.ply": (v, f), "dup.ply": (v, dup)})


# ---- 0x804: a large mesh, the warp's walk (tests/large_mesh_scenes.py geometry) -----------------------------------------
def large_meshes():
    """Two instances (one mirrored) of a 32 768-triangle field and a small mesh, hard lights only."""
    files = {"field.ply": lms.field(128, 128), "small.ply": lms.field(8, 4)}
    objs = ['(%s (translate (-4,-1,2) (rotate (1,0,0) 70 (scale 0.5 bspMesh 10 "field.ply"))))' % _mesh_material(0.3),
            '(%s (translate (4,-1,3) (rotate (1,0.2,0) -60 (scale (-0.4,0.4,0.4) bspMesh 10 "field.ply"))))' % _mesh_material(),
            '(%s (translate (-0.5,1,-1) bspMesh 3 "small.ply"))' % _mesh_material()]
    return VScene("large_meshes", 0x804, MESH_CAMERA, objs, lms.HARD_LIGHTS.strip().split("\n"), spp=2, files=files)


def all_scenes():
    """Every scene of the suite, in a fixed order: VScene.name is unique."""
    out = [spheres(s) for s in range(3)] + [spheres(3, far=False)]
    out += [spheres(10 + s, plane=True) for s in range(3)]
    nl = len(CUBE_LIGHTS)
    out += [cubes(n) for n in (8, 9, 31, 32, 33, 64, 65, max_table_items(nl) - 1, max_table_items(nl))]
    out += [cubes(33, reflect=False), cubes(33, reflect=False, pad_to=max_table_items(nl) + 16), cube_pairs_all_ops(1), cube_pairs_all_ops(2), edge_pairs()]
    out += [runs(s, soft_samples=k) for s, k in ((1, 2), (2, 0), (3, 3))]
    out += [nested(s, soft_samples=k) for s, k in ((1, 1), (2, 0), (3, 2))]
    out += [csg_limit(16, True), csg_limit(12, False)]
    out += [textured(s) for s in range(3)] + [textured(10 + s, rough=True) for s in range(3)]
    out += [small_meshes(s) for s in range(2)] + [mesh_tie(True), mesh_tie(False)]
    out += [large_meshes(), mesh_tie(True, large=True)]
    return out


# scenes past the limits: created and rendered, they must be refused with the given status (api.py FtbError)
def over_limit_scenes():
    return [csg_limit(17, True), csg_limit(13, False)]


# ---- 0x209 edge rays: axis-aligned pairs whose cube operand reports more than two crossings on its edges ---------------
EDGE_ITEMS = [((k % 4) * 3.0 - 4.5, 0.0, (k // 4) * 3.0) for k in range(8)]


def edge_pairs():
    """Every operator with the unit cube ([-0.5, 0.5]^3, Cube.fs) as A and as B and a sphere as the other operand, on a grid
    of dyadic positions: rays aimed at the cube's edges and corners from dyadic origins are exact, and the reference's cube
    (six squares) reports a crossing of each face it touches there, more than two in all (tests/test_gpu_variants.py)."""
    objs = []
    for k, c in enumerate(EDGE_ITEMS):
        a, b = "cube", "(translate (0.25,0.25,-0.25) (scale 0.5 sphere))"
        if k >= 4:
            a, b = b, a
        objs.append("(translate %s (material diffuse (0.7,0.6,0.5) reflectance 0 shineyness 5 (%s %s %s)))" % (_v(c), OPS[k % 4], a, b))
    return VScene("edge_pairs", 0x209, CUBE_CAMERA, objs, CUBE_LIGHTS, spp=1)


def edge_ray_candidates():
    """Rays [n, 6] from dyadic origins around each item at its cube's edge points and corners (world space), with the item
    centre of each."""
    rays, centres = [], []
    h = 0.5
    along = [-0.375, -0.125, 0.0, 0.25]
    targets = []
    for s1 in (-h, h):
        for s2 in (-h, h):
            for a in along:
                targets += [(a, s1, s2), (s1, a, s2), (s1, s2, a)]
            for s3 in (-h, h):
                targets.append((s1, s2, s3))
    offsets = [(-3.0, 2.0, -4.0), (2.5, 1.5, -3.5), (-1.25, 3.0, -2.0), (0.75, -2.0, -3.0), (4.0, 0.5, 1.0), (-2.0, 0.25, 3.5)]
    for c in EDGE_ITEMS:
        c = np.array(c)
        for t in targets:
            for off in offsets:
                o = c + np.array(t) + np.array(off)
                rays.append(np.concatenate([o, -np.array(off)]))
                centres.append(c)
    return np.array(rays), np.array(centres)
