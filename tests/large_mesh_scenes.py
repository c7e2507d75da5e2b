"""Generated meshes and scenes for the large-mesh tests (tests/test_gpu_large_mesh.py, tests/test_gpu_mesh_index.py).

Scenes whose bspMesh primitives hold 32 768 (api.cu kLargeMesh) or more triangles in all have their mesh index built on the
device (bvh_build.cu) and their meshes walked by the whole warp (render.cuh packetMesh).  The meshes here are written as PLY
text into a directory of the caller's; every scene function returns (scene text, that directory)."""
import os
import shutil

import numpy as np

from functracer_b200 import scenes

LARGE_MESH = 32768  # api.cu kLargeMesh
CELL = 0.125        # field cells; every field coordinate is a multiple of 1/64, exact in float and double
MARGIN = 1.0 / 64
# without the soft light (no RNG) a mesh-only scene runs on the FP32 large-mesh kernel 0x804, with it on the generic 0xfff
HARD_LIGHTS = "directional dir (0.3,0.2,1) colour (0.7,0.7,0.7)\npositional pos (6,10,-6) falloff (1,0.01,0.002) colour (0.8,0.8,0.6)\n"
LIGHTS = HARD_LIGHTS + "softdirectional dir (-1,-2,2) samples 1 scatter 5 colour (0.4,0.4,0.5)\n"
CAMERA = "camera pos (8,8,-12) lookat (8,8,0) up (0,1,0) fov 70 ratio 1.3333333333333333"


def write_ply(path, verts, faces):
    """PLY in the form the front end reads (x y z confidence intensity; faces `3 a b c`).  repr() writes each double exactly."""
    verts = np.asarray(verts, dtype=np.float64)
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n" % len(verts))
        f.write("property float confidence\nproperty float intensity\nelement face %d\nproperty list uchar int vertex_indices\nend_header\n" % len(faces))
        for v in verts:
            f.write("%r %r %r 1 0.5\n" % (float(v[0]), float(v[1]), float(v[2])))
        for a, b, c in faces:
            f.write("3 %d %d %d\n" % (a, b, c))
    return len(faces)


def field(nx, ny, n_tris=None, planar=False, origin=(0.0, 0.0, 0.0)):
    """nx x ny cells of CELL in the z = origin plane, each holding a quad inset by MARGIN and split into two triangles (tilted
    by multiples of 1/64 unless planar).  No triangle reaches a cell's border, so while the cell counts halve evenly (powers
    of two) the reference's BSP splits (bbox midpoints, BspMesh.fs:30-46) fall between cells and clip nothing: the mesh keeps
    exactly its triangles at any bspMesh depth.  n_tris: keep only the first n_tris triangles.  Returns (verts, faces)."""
    ox, oy, oz = origin
    verts, faces = [], []
    for j in range(ny):
        for i in range(nx):
            x0, y0, x1, y1 = ox + i * CELL + MARGIN, oy + j * CELL + MARGIN, ox + (i + 1) * CELL - MARGIN, oy + (j + 1) * CELL - MARGIN
            h = 0.0 if planar else ((3 * i + 5 * j) % 7) / 64.0
            dz = 0.0 if planar else 1.0 / 64
            k = len(verts)
            verts += [(x0, y0, oz + h), (x1, y0, oz + h + dz), (x1, y1, oz + h), (x0, y1, oz + h - dz)]
            faces += [(k, k + 1, k + 2), (k, k + 2, k + 3)]
    if n_tris is not None:
        faces = faces[:n_tris]
    return np.array(verts), faces


def blob(path, n_lon=128, n_lat=129, seed=13):
    """The bunny stand-in's closed blob (2 n_lon (n_lat - 1) triangles; 32 768 with the defaults)."""
    return scenes._blob_ply(path, n_lon, n_lat, seed)[1]


def _mat(refl=0.0):
    return "material diffuse (0.8,0.7,0.6) reflectance %g shineyness 10" % refl


def options(res=(128, 96), spp=1, camera=CAMERA):
    return "%s\nsamples %d\nres %d %d\n\n" % (camera, spp, res[0], res[1])


# ---- the tie: a bspMesh and later triangle items holding exact copies of some of its triangles ------------------------
def tie(d, n, mesh_first=True, soft=False):
    """bspMesh of an n-triangle field, then `mesh dup.ply`: 31 of its triangles again, as triangle items of the same batch of
    32 items (mesh_first=False: the other way round).  Returns (text, dir, the duplicated triangles [31, 3, 3])."""
    v, f = field(128, 128, n_tris=n)
    write_ply(os.path.join(d, "big.ply"), v, f)
    pick = np.linspace(0, n - 1, 31).astype(int)
    dup = [f[k] for k in pick]
    write_ply(os.path.join(d, "dup.ply"), v, dup)
    body = ['bspMesh 10 "big.ply"', 'mesh "dup.ply"']
    if not mesh_first:
        body.reverse()
    text = options() + "(%s (group %s))\n\n" % (_mat(), " ".join(body)) + (LIGHTS if soft else HARD_LIGHTS)
    return text, d, v[np.array(dup)]


def twin_instances(d):
    """The same 16 384-triangle field twice under one transform: two bspMesh items that tie everywhere."""
    v, f = field(128, 64)
    write_ply(os.path.join(d, "half.ply"), v, f)
    return options() + '(%s (translate (0,4,0) (group bspMesh 10 "half.ply" bspMesh 10 "half.ply")))\n\n' % _mat() + LIGHTS, d


# ---- several meshes in one scene -----------------------------------------------------------------------------------
def two_large_and_small(d):
    v, f = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), v, f)
    blob(os.path.join(d, "blob.ply"))
    shutil.copy(os.path.join(scenes.asset_dir(), "bunny_tiny.ply"), d)
    return (options() + "(%s (group\n" % _mat(0.3) + ' bspMesh 10 "field.ply"\n (translate (8,8,-3) (scale 24 bspMesh 8 "blob.ply"))\n'
            ' (translate (4,11,-4) (scale 10 bspMesh 3 "bunny_tiny.ply"))))\n\n' + LIGHTS), d


def many_small_meshes(d):
    """One field 100 triangles short of the threshold and 40 meshes of 1-4 triangles that make up the difference."""
    v, f = field(128, 128, n_tris=LARGE_MESH - 100)
    write_ply(os.path.join(d, "field.ply"), v, f)
    rng = np.random.default_rng(7)
    parts, total = [], len(f)
    for k in range(40):
        n = 1 + k % 4
        c = np.array([1.0 + (k % 8) * 1.75, 2.0 + (k // 8) * 3.0, -1.0 - (k % 3) * 0.5])
        verts = c + np.round(rng.uniform(-0.6, 0.6, size=(3 * n, 3)) * 64) / 64
        write_ply(os.path.join(d, "s%d.ply" % k), verts, [(3 * i, 3 * i + 1, 3 * i + 2) for i in range(n)])
        parts.append(' bspMesh 0 "s%d.ply"' % k)
        total += n
    assert total >= LARGE_MESH
    return options() + "(%s (group\n bspMesh 10 \"field.ply\"\n%s))\n\n" % (_mat(0.2), "\n".join(parts)) + LIGHTS, d


def transformed_instances(d):
    """A blob of 16 384 triangles three times: rotated, non-uniformly scaled, mirrored; a field behind them."""
    blob(os.path.join(d, "blob.ply"), 128, 65)
    v, f = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), v, f)
    return (options() + "(%s (group\n bspMesh 10 \"field.ply\"\n" % _mat(0.3) +
            ' (translate (3.5,8,-3) (rotate (0,1,0) 37 (rotate (1,0,0) -25 (scale 22 bspMesh 8 "blob.ply"))))\n'
            ' (translate (8,8,-3) (scale (30,14,22) bspMesh 8 "blob.ply"))\n'
            ' (translate (12.5,8,-3) (scale (-22,22,22) bspMesh 8 "blob.ply"))))\n\n' + LIGHTS), d


# ---- geometry that stresses the device build and the slab test -----------------------------------------------------
def planar_grid(d):
    """A field with zero extent in z, seen straight along z."""
    v, f = field(128, 128, planar=True)
    write_ply(os.path.join(d, "flat.ply"), v, f)
    cam = "camera pos (8,8,-10) lookat (8,8,0) up (0,1,0) fov 70 ratio 1.3333333333333333"
    return options(camera=cam) + '(%s bspMesh 10 "flat.ply")\n\n' % _mat() + LIGHTS, d


def fan(d, n=2048, centre=(8.0, 8.0, -1.0)):
    """n triangles with one centroid AND one box centre (each axis holds x, 0, -x about the centre), so one Morton key."""
    rng = np.random.default_rng(11)
    c = np.array(centre)
    verts = []
    for _ in range(n):
        a = np.round(rng.uniform(0.25, 2.0, size=3) * 64) / 64 * rng.choice([-1.0, 1.0], size=3)
        tri = np.zeros((3, 3))
        for ax in range(3):
            tri[rng.permutation(3), ax] = (a[ax], 0.0, -a[ax])
        verts += list(c + tri)
    write_ply(os.path.join(d, "fan.ply"), verts, [(3 * i, 3 * i + 1, 3 * i + 2) for i in range(n)])
    v, f = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), v, f)
    return options() + '(%s (group bspMesh 10 "field.ply" bspMesh 0 "fan.ply"))\n\n' % _mat(0.2) + LIGHTS, d


def slivers(d):
    """8 192 tiny triangles and 8 slivers across all of them in one mesh (bspMesh 0: the reference clips none), a field behind."""
    v, f = field(64, 64, origin=(4.0, 4.0, -1.0))
    v, f = v.tolist(), list(f)
    for k in range(8):
        y = 4.0 + k + 0.5
        base = len(v)
        v += [(4.0, y, -1.25), (12.0, y + 0.5 - k / 8.0, -1.125 - k / 64.0), (4.0, y + 1.0 / 64, -1.25)]
        f.append((base, base + 1, base + 2))
    write_ply(os.path.join(d, "mix.ply"), v, f)
    fv, ff = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), fv, ff)
    return options() + '(%s (group bspMesh 10 "field.ply" bspMesh 0 "mix.ply"))\n\n' % _mat() + LIGHTS, d


def coincident(d, n=5000):
    """n copies of one triangle (their boxes tie exactly in every clustering round), a field behind."""
    verts = [(6.0, 6.0, -1.0), (10.0, 6.5, -1.0), (7.0, 10.0, -1.5)]
    write_ply(os.path.join(d, "same.ply"), verts, [(0, 1, 2)] * n)
    v, f = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), v, f)
    return options() + '(%s (group bspMesh 10 "field.ply" bspMesh 0 "same.ply"))\n\n' % _mat() + LIGHTS, d


# ---- incoherent and secondary rays ---------------------------------------------------------------------------------
def shiny_blob(d):
    """A closed blob (32 768 triangles before the reference's clipping) over a field, both reflective, three kinds of light."""
    blob(os.path.join(d, "blob.ply"))
    v, f = field(128, 128)
    write_ply(os.path.join(d, "field.ply"), v, f)
    return (options(spp=2) + '(material diffuse (0.8,0.7,0.6) reflectance 0.5 shineyness 20 (group\n bspMesh 10 "field.ply"\n'
            ' (translate (8,5,-3) (scale 30 bspMesh 8 "blob.ply"))))\n\n' + LIGHTS), d


BLOB_CENTRE = np.array([8.0, 5.0, -3.0]) + 30 * np.array([-0.017, 0.11, 0.0])  # shiny_blob's blob: the centre its radii are drawn from


# ---- walk and tree must not change the picture ---------------------------------------------------------------------
def just_below_threshold(d, extra=False):
    """A 32 767-triangle field (host tree, per-lane walk); extra=True adds a one-triangle mesh of zero area, which takes
    the scene over the threshold (device tree, warp-packet walk) without adding anything that can be hit."""
    v, f = field(128, 128, n_tris=LARGE_MESH - 1)
    write_ply(os.path.join(d, "field.ply"), v, f)
    write_ply(os.path.join(d, "zero.ply"), [(8.0, 8.0, -1.0), (8.5, 8.5, -1.0), (9.0, 9.0, -1.0)], [(0, 1, 2)])
    return (options(spp=2) + '(%s (group bspMesh 10 "field.ply"%s))\n\n' % (_mat(0.4), ' bspMesh 0 "zero.ply"' if extra else "") + LIGHTS), d


def geometric_sequence(d, n=120):
    """Triangles whose sizes and distances from the origin shrink by half from one to the next: nested scales the
    clustering can only merge one level at a time, meant to give a tree deeper than the traversal stack."""
    verts = []
    for k in range(n):
        s = 2.0 ** -k
        verts += [(s, 0.0, 0.0), (s * 1.5, 0.0, 0.0), (s, s * 0.5, s * 0.25)]
    write_ply(os.path.join(d, "seq.ply"), verts, [(3 * i, 3 * i + 1, 3 * i + 2) for i in range(n)])
    return options() + '(%s bspMesh 0 "seq.ply")\n\n' % _mat() + LIGHTS, d
