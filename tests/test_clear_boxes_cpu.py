"""Clear tiles by the items' world-space boxes (functracer_b200/csrc/cuda/clear_boxes.h), tested with the REAL host code
(clear_boxes.cpp, tiles.cpp and lower.cpp compiled with g++ into a throw-away probe, no device involved) against the CPU oracle.
CPU only.

A tile whose rays touch an item's bounding sphere is still clear when they miss the projection of the item's boxes.  For every
sample of every clear tile the oracle (FP64, the reference's algorithm) must report no hit: on every bundled config at small
sizes, on the random scenes of the fuzz suite, and on scenes where boxes are easy to get wrong (rotated, non-uniformly scaled
and mirrored leaves, open CSG operands crossed behind the camera, a camera inside a box or beside one that straddles the
camera plane, a camera over a cube's face).  The two guards that make an item keep its sphere (a box not wholly in front of
the camera; a planar face whose t = 0 answer to a parallel ray lies at the camera) each have a scene where the sphere stage
clears tiles and the guard decides the rest.  The headline frame's share of clear tiles is pinned."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from functracer_b200 import abi, frontend, scenes
from oracle import ftb_oracle as orc
from util import parse
import test_clear_tiles_cpu as sphere_stage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "functracer_b200", "csrc")

PROBE = r"""
#include "%(csrc)s/cuda/clear_boxes.h"
#include <string>
static int g_boxes = 1;
extern "C" void ftb_probe_use_boxes(int on) { g_boxes = on; }
// The clear-tile mask of the window [x0, x1) x [y0, y1) as api.cu computeTileOrder builds it, row-major over the window's tiles.
extern "C" int ftb_probe_clear(const ftb_scene_desc* d, const ftb_camera* c, const ftb_render_params* p, int x0, int y0, int x1, int y1,
                               unsigned char* clear, int max_tiles, int* tiles_x, int* tiles_y)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -1;
    if (L.item_boxes.size() != L.items.size()) return -3;
    const int corner = p->sampling == FTB_SAMPLING_CORNER ? 1 : 0;
    ftb::TileGrid g;
    g.wx0 = x0; g.wy0 = y0; g.ww = x1 - x0 + corner; g.wh = y1 - y0 + corner;
    g.tiles_x = (g.ww + FTB_TILE_W - 1) / FTB_TILE_W; g.tiles_y = (g.wh + FTB_TILE_H - 1) / FTB_TILE_H;
    *tiles_x = g.tiles_x; *tiles_y = g.tiles_y;
    if (g.tiles_x * g.tiles_y > max_tiles) return -2;
    std::vector<float> cost;
    std::vector<unsigned char> cl;
    const std::vector<ftb::ImageRect> boxes = ftb::itemBoxRects(L, *c, p->width, p->height);
    ftb::estimateTiles(L, d->n_lights, *c, p->width, p->height, p->recursion_limit, ftb::sampleOffsetExtent(*p), g, cost, cl, g_boxes ? &boxes : nullptr);
    for (size_t t = 0; t < cl.size(); ++t) clear[t] = cl[t];
    return 0;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(str(tmp_path_factory.mktemp("boxes_probe")))


def build_probe(d):
    """The probe library, compiled into directory d."""
    src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe.so")
    open(src, "w").write(PROBE % dict(csrc=CSRC))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src] +
                          [os.path.join(CSRC, "cuda", f) for f in ("clear_boxes.cpp", "tiles.cpp", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_clear.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 4 + [
        C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.ftb_probe_clear.restype = C.c_int
    lib.ftb_probe_use_boxes.argtypes = [C.c_int]
    return lib


def shares(lib, sc, params):
    """(share of clear tiles by the spheres alone, with the boxes); the boxes' tiles checked against the oracle."""
    lib.ftb_probe_use_boxes(0)
    spheres = sphere_stage.clear_mask(lib, sc, params)
    lib.ftb_probe_use_boxes(1)
    boxes = sphere_stage.clear_mask(lib, sc, params)
    assert not (spheres & ~boxes).any(), "the boxes must only add clear tiles"
    assert sphere_stage.check_against_oracle(lib, sc, params) == float(boxes.mean())
    return float(spheres.mean()), float(boxes.mean())


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_bundled_configs(probe, name):
    cfg = scenes.CONFIGS[name]
    W, H = (192, 108) if cfg["res"][0] > cfg["res"][1] else (120, 160)
    sc = parse(scenes.config_text(name, res=(W, H), spp=2))
    p = orc.make_params(W, H, 2, frontend.jitter_pattern(cfg["seed"], 2), sampling=sc.sampling)
    s, b = shares(probe, sc, p)
    print("%s: clear tiles %.3f by spheres, %.3f with boxes" % (name, s, b))


@pytest.mark.parametrize("seed", range(40))
def test_random_scenes(probe, seed):
    from test_gpu_fuzz import _scene
    sc = parse(_scene(1000 + seed))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(seed + 1, sc.spp), sampling=sc.sampling, seed=77)
    s, b = shares(probe, sc, p)
    if sc.camera.has_focus:
        assert b == 0.0


GROUND = "(translate (0,-3,0) plane)\n\n"
LIGHT = "\ndirectional dir (0.3,-1,0.4) colour (1,1,1)\n"
CAM = "camera pos (0,0.5,-9) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.33\n"


@pytest.mark.parametrize("obj, cam", [
    ("(rotate (0.3,1,0.2) 37 (scale (3,0.4,1) cube))", CAM),
    ("(rotate (1,0,1) 50 (scale (2,3,0.5) cone))", CAM),
    ("(rotate (0,0.2,1) -65 (scale (0.5,2,1.5) cylinder))", CAM),
    ("(scale (-2,1.5,1) (rotate (1,1,0) 30 solidCylinder))", CAM),                  # mirrored
    ("(scale (1,-1,-1) (translate (0.5,0.5,0) cone))", CAM),                        # mirrored twice
    ("(rotate (0,1,1) 20 (scale (2,1,3) square))", CAM),
    ("(rotate (1,0,0) 70 (scale (2,1,2) circle))", CAM),
    ('(translate (0,-1,0) (scale 12 (rotate (0,1,0) 40 (scale (1,-1.5,0.7) mesh "bunny_tiny.ply"))))', CAM),
    ('(translate (1,0,0) (scale (-9,9,9) (rotate (1,0,1) 25 bspMesh 3 "bunny_tiny.ply")))', CAM),
    # intersect / subtract with an open operand the camera's rays cross behind the origin
    ("(intersect (scale (2,2,40) cylinder) (scale 1.5 sphere))", CAM),
    ("(intersect (rotate (1,0,0) 90 (scale (1.5,20,1.5) cylinder)) (scale 1.2 cube))", CAM),
    ("(subtract (scale 2 cube) (rotate (1,0,0) 90 (scale (0.6,30,0.6) cone)))", CAM),
    ("(subtract (scale 20 square) (scale 1.5 sphere))", CAM),
    # the camera inside a box, and a box across the camera plane
    ("(scale (30,30,30) cube)", CAM),
    ("(translate (0,0.5,-9) (scale (4,1,0.2) cube))", CAM),
    ("(translate (3,0.5,-9) (rotate (0,1,0) 45 (scale (1,1,3) cylinder)))", CAM),
    # the camera over a cube's top face and over a disc, its rays level with them
    ("(translate (0,-2,0) (scale (8,1,40) cube))", "camera pos (0,3,-5) lookat (0,3,5) up (0,1,0) fov 40 ratio 1.33\n"),
    ("(translate (0,1,3) (scale 6 circle))", "camera pos (0,1,0) lookat (0,1,5) up (0,1,0) fov 40 ratio 1.33\n"),
    ("(translate (0,-3,6) (scale (4,4,4) solidCylinder))", "camera pos (0,1,6.5) lookat (0,1,20) up (0,1,0) fov 40 ratio 1.33\n"),
])
@pytest.mark.parametrize("samples", ["samples 3", "samples corner"])
def test_shapes_boxes_get_wrong(probe, obj, cam, samples):
    sc = parse(cam + samples + "\nres 160 120\n\n" + GROUND + obj + "\n" + LIGHT)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    s, b = shares(probe, sc, p)
    print("%s: %.3f -> %.3f" % (obj, s, b))


def _down_at_horizon_row(pos, heading):
    """A camera at `pos` (fov 100, 161 x 121 corner samples) pitched down so that the horizon falls exactly on the corner
    sample row 40: there d.y = k.y + v j.y = 0 (the reference's image plane swaps its axes: the row pitch is height / (W - 1))."""
    v = 0.5 * math.tan(math.radians(50))  # = height / 2 - 40 * height / 160
    at = (pos[0] + heading[0], pos[1] - v, pos[2] + heading[1])
    return ("camera pos (%r,%r,%r) lookat (%.17g,%.17g,%.17g) up (0,1,0) fov 100 ratio 1.33\nsamples corner\nres 161 121\n" %
            (tuple(pos) + at))


@pytest.mark.parametrize("text", [
    # A long box beside a wide-angle camera, reaching behind the camera plane, its sphere well clear of the camera.  Its
    # corners behind the camera would project to the other side of the image: the corners' rectangle would miss the rays
    # that see the box's near end towards the frame's right edge.  The box must not be used.
    "camera pos (0,0.5,0) lookat (0,0.5,1) up (0,1,0) fov 150 ratio 3\nsamples 2\nres 240 80\n\n(translate (0,-3,0) plane)\n\n"
    "(translate (17.5,2.5,0) (scale (25,2,10) cube))\n",
    # A camera above a tall solidCylinder's top cap, within 1 of the cap's centre in the cylinder's frame but outside its
    # sphere, looking down at it with the horizon in the frame: the rays level with the cap miss its box and touch its sphere,
    # and Plane.fs answers the horizon row (parallel to the cap) with a crossing at t = 0 at the camera.
    _down_at_horizon_row((2.4, 8.5, 0.0), (-1.0, 0.0)) + "\n(scale (4,5,4) solidCylinder)\n",
], ids=["box-across-camera-plane", "cap-answers-at-camera"])
def test_guards_that_keep_the_sphere(probe, text):
    sc = parse(text + LIGHT)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    s, b = shares(probe, sc, p)
    assert s > 0, "the sphere stage must clear some tiles, or the case shows nothing"
    print("%.3f -> %.3f" % (s, b))


def test_boxes_clear_more_of_a_tall_cone(probe):
    # a cone's sphere reaches far above its apex; the box stops at the apex
    sc = parse("camera pos (0,1,-12) lookat (0,1,0) up (0,1,0) fov 60 ratio 1\nsamples 1\nres 128 128\n\n" + GROUND +
               "(translate (0,-3,0) (scale (6,3,6) cone))\n" + LIGHT)
    p = orc.make_params(128, 128, 1, frontend.jitter_pattern(1, 1))
    s, b = shares(probe, sc, p)
    assert b > s + 0.1, (s, b)


def test_windows_agree_with_the_whole_frame(probe):
    sc = parse(scenes.config_text("cfg5-repeat", res=(384, 216), spp=2))
    p = orc.make_params(384, 216, 2, frontend.jitter_pattern(5, 2))
    whole = sphere_stage.clear_mask(probe, sc, p)
    win = sphere_stage.clear_mask(probe, sc, p, (64, 32, 320, 160))  # tile-aligned: the same tiles
    assert (win == whole[2:10, 4:20]).all()


def test_headline_share(probe):
    """cfg5-repeat at its full size (7680 x 4320 x 64): the sky above the roofs is clear too."""
    cfg = scenes.CONFIGS["cfg5-repeat"]
    sc = parse(scenes.config_text("cfg5-repeat"))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(cfg["seed"], sc.spp))
    probe.ftb_probe_use_boxes(0)
    spheres = float(sphere_stage.clear_mask(probe, sc, p).mean())
    probe.ftb_probe_use_boxes(1)
    mask = sphere_stage.clear_mask(probe, sc, p)
    share = float(mask.mean())
    print("cfg5-repeat: %d of %d tiles clear (%.3f; %.3f by the spheres alone)" % (int(mask.sum()), mask.size, share, spheres))
    assert 0.68 <= share <= 0.76, share
