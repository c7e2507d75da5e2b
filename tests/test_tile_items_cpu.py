"""Per-tile item masks (functracer_b200/csrc/cuda/tiles.h estimateTiles `items`), tested with the REAL host code (tiles.cpp,
clear_boxes.cpp and lower.cpp compiled with g++ into a throw-away probe, no device involved) against the CPU oracle.  CPU only.

A primary ray of a traced tile tests only the items whose bit its tile's mask keeps.  That is only right if no sample of the tile
has a crossing at t >= 0 with an item whose bit is clear, and, where the bit was cleared by the item's boxes rather than by its
bounding sphere, no crossing at any t.  Checked for every sample of every tile against the oracle's full hit lists (FP64, the
reference's algorithm): on every bundled config at small sizes, on the random scenes of the fuzz suite and on the scenes where
boxes and planes are easy to get wrong.  A clear tile is exactly a tile whose mask is 0, and the full-size clear tiles of every
bundled config are pinned to the classification the separate sphere / box / plane passes gave before the masks existed."""
import ctypes as C
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

from functracer_b200 import abi, frontend, scenes
from oracle import ftb_oracle as orc
from util import parse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "functracer_b200", "csrc")

# The hand-built cases of the clear-tile tests (test_clear_boxes_cpu.py, test_clear_tiles_cpu.py), run here against the masks.
BOX_GROUND = "(translate (0,-3,0) plane)\n\n"
BOX_LIGHT = "\ndirectional dir (0.3,-1,0.4) colour (1,1,1)\n"
BOX_CAM = "camera pos (0,0.5,-9) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.33\n"
BOX_CASES = [
    ("(rotate (0.3,1,0.2) 37 (scale (3,0.4,1) cube))", BOX_CAM),
    ("(rotate (1,0,1) 50 (scale (2,3,0.5) cone))", BOX_CAM),
    ("(rotate (0,0.2,1) -65 (scale (0.5,2,1.5) cylinder))", BOX_CAM),
    ("(scale (-2,1.5,1) (rotate (1,1,0) 30 solidCylinder))", BOX_CAM),                  # mirrored
    ("(scale (1,-1,-1) (translate (0.5,0.5,0) cone))", BOX_CAM),                        # mirrored twice
    ("(rotate (0,1,1) 20 (scale (2,1,3) square))", BOX_CAM),
    ("(rotate (1,0,0) 70 (scale (2,1,2) circle))", BOX_CAM),
    ('(translate (0,-1,0) (scale 12 (rotate (0,1,0) 40 (scale (1,-1.5,0.7) mesh "bunny_tiny.ply"))))', BOX_CAM),
    ('(translate (1,0,0) (scale (-9,9,9) (rotate (1,0,1) 25 bspMesh 3 "bunny_tiny.ply")))', BOX_CAM),
    # intersect / subtract with an open operand the camera's rays cross behind the origin
    ("(intersect (scale (2,2,40) cylinder) (scale 1.5 sphere))", BOX_CAM),
    ("(intersect (rotate (1,0,0) 90 (scale (1.5,20,1.5) cylinder)) (scale 1.2 cube))", BOX_CAM),
    ("(subtract (scale 2 cube) (rotate (1,0,0) 90 (scale (0.6,30,0.6) cone)))", BOX_CAM),
    ("(subtract (scale 20 square) (scale 1.5 sphere))", BOX_CAM),
    # the camera inside a box, and a box across the camera plane
    ("(scale (30,30,30) cube)", BOX_CAM),
    ("(translate (0,0.5,-9) (scale (4,1,0.2) cube))", BOX_CAM),
    ("(translate (3,0.5,-9) (rotate (0,1,0) 45 (scale (1,1,3) cylinder)))", BOX_CAM),
    # the camera over a cube's top face and over a disc, its rays level with them
    ("(translate (0,-2,0) (scale (8,1,40) cube))", "camera pos (0,3,-5) lookat (0,3,5) up (0,1,0) fov 40 ratio 1.33\n"),
    ("(translate (0,1,3) (scale 6 circle))", "camera pos (0,1,0) lookat (0,1,5) up (0,1,0) fov 40 ratio 1.33\n"),
    ("(translate (0,-3,6) (scale (4,4,4) solidCylinder))", "camera pos (0,1,6.5) lookat (0,1,20) up (0,1,0) fov 40 ratio 1.33\n"),
]
PLANE_SCENE = "(translate (0,-2.2,0) plane)\n\n(translate (0.3,0,0.5) sphere)\n\ndirectional dir (0.3,-1,0.4) colour (1,1,1)\n"
PLANE_CAMERAS = [
    "camera pos (0,-5,-6) lookat (0,-9,0) up (0,1,0) fov 55 ratio 1.33",     # below the plane, looking away from it
    "camera pos (0,-5,-6) lookat (0,0,0) up (0,1,0) fov 55 ratio 1.33",      # below the plane, looking up at it
    "camera pos (0,-5,-6) lookat (0,-5,0) up (0,1,0) fov 55 ratio 1.33",     # below the plane, its horizon across the frame
    "camera pos (0,0.5,-6) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.33",   # the horizon through the middle of a tile row
    "camera pos (0,-2.2,-6) lookat (0,-2.2,0) up (0,1,0) fov 55 ratio 1.33",  # in the plane, looking along it
    "camera pos (0,-2.19999,-6) lookat (0,-2.19999,0) up (0,1,0) fov 55 ratio 1.33",  # just above it, along it
    "camera pos (0,3,0) lookat (0,-5,0.001) up (0,1,0) fov 55 ratio 1.33",   # straight down at the plane
]

PROBE = r"""
#include "%(csrc)s/cuda/clear_boxes.h"
#include <string>
// The item masks and clear tiles of the window [x0, x1) x [y0, y1) as api.cu computeTileOrder builds them, row-major over the
// window's tiles (use_boxes = 0: the spheres and planes alone), and the item every PRIMITIVE instance belongs to.
// Returns 1 with masks, 0 without (depth of field, more than 32 items), < 0 on an error.
extern "C" int ftb_probe_items(const ftb_scene_desc* d, const ftb_camera* c, const ftb_render_params* p, int x0, int y0, int x1, int y1, int use_boxes,
                               unsigned* items, unsigned char* clear, int max_tiles, int* tiles_x, int* tiles_y, int* prim_item, int max_prims, int* n_items)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -1;
    const int corner = p->sampling == FTB_SAMPLING_CORNER ? 1 : 0;
    ftb::TileGrid g;
    g.wx0 = x0; g.wy0 = y0; g.ww = x1 - x0 + corner; g.wh = y1 - y0 + corner;
    g.tiles_x = (g.ww + FTB_TILE_W - 1) / FTB_TILE_W; g.tiles_y = (g.wh + FTB_TILE_H - 1) / FTB_TILE_H;
    *tiles_x = g.tiles_x; *tiles_y = g.tiles_y;
    if (g.tiles_x * g.tiles_y > max_tiles || L.n_prims > max_prims) return -2;
    *n_items = (int)L.items.size();
    for (int q = 0; q < L.n_prims; ++q) prim_item[q] = -1;
    for (size_t i = 0; i < L.items.size(); ++i) {
        const ftb::Item& it = L.items[i];
        if ((it.kind & 0xff) == ftb::ITEM_LEAF) prim_item[L.leaves[(size_t)it.a].prim] = (int)i;
        else
            for (int o = it.prog_first; o < it.prog_first + it.prog_count; ++o)
                if (L.ops[(size_t)o].kind == ftb::OP_LEAF) prim_item[L.leaves[(size_t)L.ops[(size_t)o].arg].prim] = (int)i;
    }
    std::vector<float> cost;
    std::vector<unsigned char> cl;
    std::vector<unsigned> m;
    const std::vector<ftb::ImageRect> boxes = ftb::itemBoxRects(L, *c, p->width, p->height);
    ftb::estimateTiles(L, d->n_lights, *c, p->width, p->height, p->recursion_limit, ftb::sampleOffsetExtent(*p), g, cost, cl, use_boxes ? &boxes : nullptr, &m);
    for (size_t t = 0; t < cl.size(); ++t) { clear[t] = cl[t]; items[t] = m.empty() ? ~0u : m[t]; }
    return m.empty() ? 0 : 1;
}
// estimateTiles' `kept` for the whole frame: the bits the masks keep in the traced tiles per bit the spheres alone keep; -1: no masks.
extern "C" double ftb_probe_kept(const ftb_scene_desc* d, const ftb_camera* c, const ftb_render_params* p)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -2;
    const int corner = p->sampling == FTB_SAMPLING_CORNER ? 1 : 0;
    ftb::TileGrid g;
    g.wx0 = 0; g.wy0 = 0; g.ww = p->width + corner; g.wh = p->height + corner;
    g.tiles_x = (g.ww + FTB_TILE_W - 1) / FTB_TILE_W; g.tiles_y = (g.wh + FTB_TILE_H - 1) / FTB_TILE_H;
    std::vector<float> cost;
    std::vector<unsigned char> cl;
    std::vector<unsigned> m;
    double kept = -1;
    const std::vector<ftb::ImageRect> boxes = ftb::itemBoxRects(L, *c, p->width, p->height);
    ftb::estimateTiles(L, d->n_lights, *c, p->width, p->height, p->recursion_limit, ftb::sampleOffsetExtent(*p), g, cost, cl, &boxes, &m, &kept);
    return m.empty() ? -1 : kept;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(str(tmp_path_factory.mktemp("items_probe")))


def build_probe(d):
    """The probe library, compiled into directory d."""
    src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe.so")
    open(src, "w").write(PROBE % dict(csrc=CSRC))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src] +
                          [os.path.join(CSRC, "cuda", f) for f in ("clear_boxes.cpp", "tiles.cpp", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_items.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 5 + [
        C.POINTER(C.c_uint), C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
    lib.ftb_probe_items.restype = C.c_int
    lib.ftb_probe_kept.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)]
    lib.ftb_probe_kept.restype = C.c_double
    return lib


def item_masks(lib, sc, params, window=None, use_boxes=True):
    """(masks [tiles_y, tiles_x] uint32 or None, clear [tiles_y, tiles_x] bool, prim -> item, number of items)."""
    x0, y0, x1, y1 = window or (0, 0, params.width, params.height)
    n = 1 << 20
    items, clear, prim_item = (C.c_uint * n)(), (C.c_ubyte * n)(), (C.c_int * (1 << 16))()
    tx, ty, ni = C.c_int(), C.c_int(), C.c_int()
    rc = lib.ftb_probe_items(sc.desc_ptr, sc.camera_ptr, C.byref(params), x0, y0, x1, y1, 1 if use_boxes else 0, items, clear, n,
                             C.byref(tx), C.byref(ty), prim_item, len(prim_item), C.byref(ni))
    assert rc >= 0, rc
    shape = (ty.value, tx.value)
    k = tx.value * ty.value
    masks = np.frombuffer(items, dtype=np.uint32, count=k).reshape(shape).copy() if rc == 1 else None
    cl = np.frombuffer(clear, dtype=np.uint8, count=k).reshape(shape).astype(bool)
    return masks, cl, np.array(prim_item[:]), ni.value


def samples(sc, params, x, y):
    """The primary samples of sample-grid pixel (x, y): (origin + 1e-4 d, d) as the kernel traces them."""
    corner = params.sampling == abi.SAMPLING_CORNER
    offs = [(-0.5, 0.5)] if corner else [(params.jitter_xy[2 * s], params.jitter_xy[2 * s + 1]) for s in range(params.spp)]
    for jx, jy in offs:
        r = orc.primary_ray(sc.camera, params.width, params.height, x, y, jx, jy)
        o, d = np.array(r[:3]), np.array(r[3:])
        yield o + 1e-4 * d, d


def check_against_oracle(lib, sc, params, window=None):
    """Every sample of every tile of the window: no crossing at t >= 0 with an item its tile's mask drops, and none at all with
    an item only the boxes drop.  Returns (masks or None, share of (tile, item) bits the boxes and planes clear in traced tiles)."""
    masks, clear, prim_item, n_items = item_masks(lib, sc, params, window)
    if masks is None:
        assert sc.camera.has_focus or n_items > 32
        return None, 0.0
    assert (clear == (masks == 0)).all(), "a clear tile is exactly a tile whose mask is 0"
    spheres, clear_s, _, _ = item_masks(lib, sc, params, window, use_boxes=False)
    assert not (masks & ~spheres).any(), "the boxes only clear bits"
    assert not (clear_s & ~clear).any()
    every = np.uint32((1 << n_items) - 1 if n_items < 32 else 0xffffffff)
    x0, y0 = (window or (0, 0))[:2]
    corner = params.sampling == abi.SAMPLING_CORNER
    gw, gh = (window[2] - x0 if window else params.width) + corner, (window[3] - y0 if window else params.height) + corner
    for ty, tx in zip(*np.nonzero((masks & every) != every)):
        m, ms = int(masks[ty, tx]), int(spheres[ty, tx])
        for y in range(ty * abi.TILE_H, min(gh, (ty + 1) * abi.TILE_H)):
            for x in range(tx * abi.TILE_W, min(gw, (tx + 1) * abi.TILE_W)):
                for o, d in samples(sc, params, x0 + x, y0 + y):
                    for h in orc.node_hits(sc, o, d, max_hits=4096):
                        it = int(prim_item[h["prim"]])
                        assert it >= 0
                        if (m >> it) & 1:
                            continue
                        assert h["t"] < 0, "tile (%d, %d), sample at pixel (%d, %d): item %d dropped, hit at t = %r" % (tx, ty, x0 + x, y0 + y, it, h["t"])
                        assert not (ms >> it) & 1, "tile (%d, %d): item %d dropped by its boxes, crossed at t = %r" % (tx, ty, it, h["t"])
    traced = masks[~clear]
    kept = sum(bin(int(v) & int(every)).count("1") for v in traced)
    return masks, 1.0 - kept / max(1, traced.size * n_items)


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_bundled_configs(probe, name):
    cfg = scenes.CONFIGS[name]
    W, H = (96, 54) if cfg["res"][0] > cfg["res"][1] else (60, 80)
    sc = parse(scenes.config_text(name, res=(W, H), spp=2))
    p = orc.make_params(W, H, 2, frontend.jitter_pattern(cfg["seed"], 2), sampling=sc.sampling)
    masks, dropped = check_against_oracle(probe, sc, p)
    print("%s: %.3f of the traced tiles' item bits clear" % (name, dropped))


@pytest.mark.parametrize("seed", range(40))
def test_random_scenes(probe, seed):
    from test_gpu_fuzz import _scene
    sc = parse(_scene(1000 + seed))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(seed + 1, sc.spp), sampling=sc.sampling, seed=77)
    masks, _ = check_against_oracle(probe, sc, p)
    if sc.camera.has_focus:
        assert masks is None  # depth of field moves the rays' origins: no masks


@pytest.mark.parametrize("obj, cam", [pytest.param(o, c, id="case%d" % i) for i, (o, c) in enumerate(BOX_CASES)])
@pytest.mark.parametrize("samples_line", ["samples 3", "samples corner"])
def test_shapes_boxes_get_wrong(probe, obj, cam, samples_line):
    """Rotated, non-uniformly scaled and mirrored leaves, open CSG operands crossed behind the camera, a camera inside a box or
    beside one that straddles the camera plane, a camera over a cube's face."""
    sc = parse(cam + samples_line + "\nres 80 60\n\n" + BOX_GROUND + obj + "\n" + BOX_LIGHT)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    check_against_oracle(probe, sc, p)


@pytest.mark.parametrize("camera", PLANE_CAMERAS)
@pytest.mark.parametrize("samples_line", ["samples 3", "samples corner"])
def test_ground_plane_cameras(probe, camera, samples_line):
    """Cameras below, in and just above the ground plane, and looking straight down at it."""
    sc = parse(camera + "\n" + samples_line + "\nres 80 60\n\n" + PLANE_SCENE)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    check_against_oracle(probe, sc, p)


def test_planes_drop_their_bit_where_the_rays_leave_them(probe):
    """The horizon through the frame: the ground plane's bit is clear in the tiles above it and kept below; the sphere's bit is
    kept only near it."""
    sc = parse("camera pos (0,0.5,-6) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.33\nsamples 3\nres 160 120\n\n" + PLANE_SCENE)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    masks, _, _, n = item_masks(probe, sc, p)
    assert n == 2
    ground = (masks & 1).astype(bool)
    assert not ground[0].any() and ground[-1].all()
    assert ((masks >> 1) & 1).any() and not ((masks >> 1) & 1).all()


def test_other_unbounded_items_keep_their_bit(probe):
    sc = parse("camera pos (0,1,-6) lookat (0,0,0) up (0,1,0) fov 55 ratio 1\nsamples 1\nres 128 96\n\n"
               "(intersect (translate (0,-2.2,0) plane) (scale (40,40,40) sphere))\n\n(translate (0,5,0) sphere)\n\n"
               "directional dir (0,-1,0) colour (1,1,1)\n")
    p = orc.make_params(128, 96, 1, frontend.jitter_pattern(1, 1))
    masks, clear, _, n = item_masks(probe, sc, p)
    assert n == 2 and (masks & 1).all() and not clear.any()
    assert not ((masks >> 1) & 1).all()


def test_more_than_32_items_have_no_masks_but_clear_tiles(probe):
    objs = "".join("(translate (%d,%d,0) (scale 0.3 sphere))\n\n" % (i % 7 - 3, i // 7 - 2) for i in range(33))
    sc = parse("camera pos (0,0,-12) lookat (0,0,0) up (0,1,0) fov 80 ratio 1\nsamples 1\nres 128 128\n\n" + objs +
               "directional dir (0,-1,0) colour (1,1,1)\n")
    p = orc.make_params(128, 128, 1, frontend.jitter_pattern(1, 1))
    masks, clear, _, n = item_masks(probe, sc, p)
    assert n == 33 and masks is None and clear.any() and not clear.all()
    sc = parse("camera pos (0,0,-12) lookat (0,0,0) up (0,1,0) fov 80 ratio 1\nsamples 1\nres 128 128\n\n" +
               objs.rsplit("(translate", 1)[0] + "directional dir (0,-1,0) colour (1,1,1)\n")
    masks32, clear32, _, n = item_masks(probe, sc, p)
    assert n == 32 and masks32 is not None and (clear32 == (masks32 == 0)).all()


def test_windows_agree_with_the_whole_frame(probe):
    sc = parse(scenes.config_text("cfg5-repeat", res=(384, 216), spp=2))
    p = orc.make_params(384, 216, 2, frontend.jitter_pattern(5, 2))
    whole = item_masks(probe, sc, p)[0]
    win = item_masks(probe, sc, p, (64, 32, 320, 160))[0]  # tile-aligned: the same tiles
    assert (win == whole[2:10, 4:20]).all()
    odd = (40, 24, 200, 120)  # not tile-aligned: its own tiles, each checked against the oracle
    check_against_oracle(probe, parse(scenes.config_text("cfg3-house", res=(240, 135), spp=1)),
                         orc.make_params(240, 135, 1, frontend.jitter_pattern(3, 1)), odd)


# Clear tiles of every bundled config at its full size: (clear tiles, tiles, md5 of the clear bytes, first 8 digits).  These are
# the tiles the separate sphere, box and plane passes classified as clear before the masks existed; mask == 0 must give
# exactly the same tiles.
FULL_SIZE_CLEAR = {
    "cfg1-sample": (0, 1200, "fb4aa89f"),
    "cfg2-hollow-sphere": (0, 8160, "405ea765"),
    "cfg3-house": (2656, 8160, "b745992f"),
    "cfg3-night-house": (1920, 8160, "cfbcbd6f"),
    "cfg4-bunny": (27528, 32400, "52ea429d"),
    "cfg4-bunny-d12": (27528, 32400, "52ea429d"),
    "cfg4-bunny-full-d14": (26793, 32400, "d273c5cb"),
    "cfg5-moon": (87526, 129600, "ce9134f5"),
    "cfg5-repeat": (93379, 129600, "b2d83d1f"),
}


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_full_size_clear_tiles_unchanged(probe, name):
    cfg = scenes.CONFIGS[name]
    sc = parse(scenes.config_text(name))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(cfg["seed"], sc.spp), sampling=sc.sampling)
    masks, clear, _, n = item_masks(probe, sc, p)
    if masks is not None:
        assert (clear == (masks == 0)).all()
    print("%s: %d items, %d of %d tiles clear (%.3f)" % (name, n, int(clear.sum()), clear.size, clear.mean()))
    digest = hashlib.md5(clear.astype(np.uint8).tobytes()).hexdigest()[:8]
    assert (int(clear.sum()), clear.size, digest) == FULL_SIZE_CLEAR[name]


# Which bundled frames launch the masked kernel instance: api.cu uses the masks when they keep at most kTileMaskKept (0.5) of
# the bits the spheres alone keep in the traced tiles.  Measured at full size: repeat keeps 0.41 (masked: -6.0 %), house 0.61
# and night-house 0.81 (+1.5 % and +5.0 % with the masks, so they run the plain instance).  None: no masks at all.
MASKED_AT_FULL_SIZE = {"cfg1-sample": None, "cfg2-hollow-sphere": False, "cfg3-house": False, "cfg3-night-house": False, "cfg4-bunny": False,
                       "cfg4-bunny-d12": False, "cfg4-bunny-full-d14": False, "cfg5-moon": False, "cfg5-repeat": True}


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_which_full_size_frames_use_the_masks(probe, name):
    api_cu = open(os.path.join(CSRC, "cuda", "api.cu")).read()
    limit = float(re.search(r"constexpr double kTileMaskKept = ([0-9.]+);", api_cu).group(1))
    cfg = scenes.CONFIGS[name]
    sc = parse(scenes.config_text(name))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(cfg["seed"], sc.spp), sampling=sc.sampling)
    kept = probe.ftb_probe_kept(sc.desc_ptr, sc.camera_ptr, C.byref(p))
    print("%s: kept %.4f" % (name, kept))
    assert (None if kept < 0 else kept <= limit) == MASKED_AT_FULL_SIZE[name]
