"""Clear tiles (functracer_b200/csrc/cuda/tiles.h), tested with the REAL host code (tiles.cpp and lower.cpp compiled with g++
into a throw-away probe, no device involved) against the CPU oracle.  CPU only.

A tile is clear when no primary sample of it can have a crossing at t >= 0; the kernel then writes its pixels without tracing
them.  For every sample of every clear tile the oracle (FP64, the reference's algorithm) must report no hit: on every bundled
config at small sizes, on the random scenes of the fuzz suite and on cameras placed against the ground plane on purpose.  The
share of clear tiles of the headline frame is pinned, so that the path cannot switch itself off unnoticed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from functracer_b200 import abi, frontend, scenes
from oracle import ftb_oracle as orc
from util import parse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "functracer_b200", "csrc")

PROBE = r"""
#include "%(csrc)s/cuda/tiles.h"
#include <string>
// The clear-tile mask of the window [x0, x1) x [y0, y1) (api.cu frameGeom / computeTileOrder), row-major over the window's tiles.
extern "C" int ftb_probe_clear(const ftb_scene_desc* d, const ftb_camera* c, const ftb_render_params* p, int x0, int y0, int x1, int y1,
                               unsigned char* clear, int max_tiles, int* tiles_x, int* tiles_y)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -1;
    const int corner = p->sampling == FTB_SAMPLING_CORNER ? 1 : 0;
    ftb::TileGrid g;
    g.wx0 = x0; g.wy0 = y0; g.ww = x1 - x0 + corner; g.wh = y1 - y0 + corner;
    g.tiles_x = (g.ww + FTB_TILE_W - 1) / FTB_TILE_W; g.tiles_y = (g.wh + FTB_TILE_H - 1) / FTB_TILE_H;
    *tiles_x = g.tiles_x; *tiles_y = g.tiles_y;
    if (g.tiles_x * g.tiles_y > max_tiles) return -2;
    std::vector<float> cost;
    std::vector<unsigned char> cl;
    ftb::estimateTiles(L, d->n_lights, *c, p->width, p->height, p->recursion_limit, ftb::sampleOffsetExtent(*p), g, cost, cl);
    for (size_t t = 0; t < cl.size(); ++t) clear[t] = cl[t];
    return 0;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    d = tmp_path_factory.mktemp("tiles_probe")
    src, so = os.path.join(str(d), "probe.cpp"), os.path.join(str(d), "libprobe.so")
    open(src, "w").write(PROBE % dict(csrc=CSRC))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src, os.path.join(CSRC, "cuda", "tiles.cpp"),
                           os.path.join(CSRC, "cuda", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_clear.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 4 + [
        C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.ftb_probe_clear.restype = C.c_int
    return lib


def clear_mask(lib, sc, params, window=None):
    """[tiles_y, tiles_x] bool: the window's clear tiles."""
    x0, y0, x1, y1 = window or (0, 0, params.width, params.height)
    buf = (C.c_ubyte * (1 << 20))()
    tx, ty = C.c_int(), C.c_int()
    rc = lib.ftb_probe_clear(sc.desc_ptr, sc.camera_ptr, C.byref(params), x0, y0, x1, y1, buf, len(buf), C.byref(tx), C.byref(ty))
    assert rc == 0, rc
    return np.frombuffer(buf, dtype=np.uint8, count=tx.value * ty.value).reshape(ty.value, tx.value).astype(bool)


def check_against_oracle(lib, sc, params):
    """Every sample of every clear tile is a miss in the oracle; returns the share of clear tiles."""
    mask = clear_mask(lib, sc, params)
    if not mask.any():
        return 0.0
    corner = params.sampling == abi.SAMPLING_CORNER
    gw, gh = params.width + corner, params.height + corner
    spp = 1 if corner else params.spp
    ref = orc.render(sc, params)
    prim = ref["prim"].reshape(gh, gw, spp)
    tile_clear = np.repeat(np.repeat(mask, abi.TILE_H, axis=0), abi.TILE_W, axis=1)[:gh, :gw]
    hits = (prim[tile_clear] != -1).any(axis=-1)
    assert not hits.any(), "%d samples of clear tiles hit something" % int(hits.sum())
    return float(mask.mean())


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_bundled_configs(probe, name):
    cfg = scenes.CONFIGS[name]
    W, H = (192, 108) if cfg["res"][0] > cfg["res"][1] else (120, 160)
    sc = parse(scenes.config_text(name, res=(W, H), spp=2))
    p = orc.make_params(W, H, 2, frontend.jitter_pattern(cfg["seed"], 2), sampling=sc.sampling)
    share = check_against_oracle(probe, sc, p)
    print("%s: clear tiles %.3f" % (name, share))


@pytest.mark.parametrize("seed", range(40))
def test_random_scenes(probe, seed):
    from test_gpu_fuzz import _scene
    sc = parse(_scene(1000 + seed))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(seed + 1, sc.spp), sampling=sc.sampling, seed=77)
    share = check_against_oracle(probe, sc, p)
    if sc.camera.has_focus:
        assert share == 0.0  # depth of field moves the rays' origins: never clear


GROUND = "(translate (0,-2.2,0) plane)\n\n(translate (0.3,0,0.5) sphere)\n\ndirectional dir (0.3,-1,0.4) colour (1,1,1)\n"


@pytest.mark.parametrize("camera, some_clear", [
    ("camera pos (0,-5,-6) lookat (0,-9,0) up (0,1,0) fov 55 ratio 1.33", True),   # below the plane, looking away from it
    ("camera pos (0,-5,-6) lookat (0,0,0) up (0,1,0) fov 55 ratio 1.33", False),   # below the plane, looking up at it
    ("camera pos (0,-5,-6) lookat (0,-5,0) up (0,1,0) fov 55 ratio 1.33", True),   # below the plane, its horizon across the frame
    ("camera pos (0,0.5,-6) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.33", True),  # the horizon through the middle of a tile row
    ("camera pos (0,-2.2,-6) lookat (0,-2.2,0) up (0,1,0) fov 55 ratio 1.33", False),  # in the plane, looking along it
    ("camera pos (0,-2.19999,-6) lookat (0,-2.19999,0) up (0,1,0) fov 55 ratio 1.33", False),  # just above it, along it
    ("camera pos (0,3,0) lookat (0,-5,0.001) up (0,1,0) fov 55 ratio 1.33", False),  # straight down at the plane
])
@pytest.mark.parametrize("samples", ["samples 3", "samples corner"])
def test_ground_plane_cameras(probe, camera, some_clear, samples):
    sc = parse(camera + "\n" + samples + "\nres 160 120\n\n" + GROUND)
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    share = check_against_oracle(probe, sc, p)
    assert (share > 0) == some_clear, share


def test_other_unbounded_items_disable_it(probe):
    # a CSG item with a plane operand is unbounded and not a top-level plane leaf
    sc = parse("camera pos (0,1,-6) lookat (0,0,0) up (0,1,0) fov 55 ratio 1\nsamples 1\nres 128 96\n\n"
               "(intersect (translate (0,-2.2,0) plane) (scale (40,40,40) sphere))\n\ndirectional dir (0,-1,0) colour (1,1,1)\n")
    p = orc.make_params(128, 96, 1, frontend.jitter_pattern(1, 1))
    assert not clear_mask(probe, sc, p).any()


def test_windows_agree_with_the_whole_frame(probe):
    sc = parse(scenes.config_text("cfg5-repeat", res=(384, 216), spp=2))
    p = orc.make_params(384, 216, 2, frontend.jitter_pattern(5, 2))
    whole = clear_mask(probe, sc, p)
    win = clear_mask(probe, sc, p, (64, 32, 320, 160))  # tile-aligned: the same tiles
    assert (win == whole[2:10, 4:20]).all()


def test_headline_share(probe):
    """cfg5-repeat at its full size (7680 x 4320 x 64): the sky above the scene is clear."""
    cfg = scenes.CONFIGS["cfg5-repeat"]
    sc = parse(scenes.config_text("cfg5-repeat"))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(cfg["seed"], sc.spp))
    mask = clear_mask(probe, sc, p)
    share = float(mask.mean())
    print("cfg5-repeat: %d of %d tiles clear (%.3f)" % (int(mask.sum()), mask.size, share))
    assert 0.50 <= share <= 0.60, share
