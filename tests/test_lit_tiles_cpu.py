"""Lit ground tiles (functracer_b200/csrc/cuda/lit_tiles.h), tested with the REAL host code (lit_tiles.cpp, tiles.cpp and
lower.cpp compiled with g++ into a throw-away probe, no device involved) against the CPU oracle.  CPU only.

A lit bit says: every primary sample of the tile that lands on the ground sees directional light k unblocked.  For every lit
bit, every primary sample of the tile that the oracle (FP64, the reference's algorithm) reports on the ground gets its shadow
rays towards that light rebuilt from the RNG contract (the reference's shadowRayOrigin, jitterVector per soft sample), and
the oracle's node_hits must find no blocking crossing (t >= 0 on a lit surface) on any of them.  On every bundled config at
small sizes, on the random scenes of the fuzz suite, and on scenes built to be hard: an item grazing the edge of a light's
cone, wide scatter, a light nearly parallel to the ground, a camera below the ground, a tilted ground, a second unbounded item,
windows.  Two planted errors - dropping the soft light's scatter cone, dropping the inflation of the items' spheres by the
extent of the tile's footprint - must each make the check fail on a scene built for it."""
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
#include "%(csrc)s/cuda/lit_tiles.h"
#include <string>
// The lit-tile mask of the window [x0, x1) x [y0, y1) as api.cu computeTileOrder builds it, row-major over the window's
// tiles; *prim = the ground leaf's primitive index (-1: nothing lit).
extern "C" int ftb_probe_lit(const ftb_scene_desc* d, const ftb_camera* c, const ftb_render_params* p, int x0, int y0, int x1, int y1,
                             unsigned char* lit, int max_tiles, int* tiles_x, int* tiles_y, int* prim)
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
    std::vector<unsigned char> m;
    const int leaf = ftb::litTiles(L, d->lights, d->n_lights, *c, p->width, p->height, ftb::sampleOffsetExtent(*p), g, m);
    *prim = leaf >= 0 ? L.leaves[(size_t)leaf].prim : -1;
    for (size_t t = 0; t < m.size(); ++t) lit[t] = m[t];
    return 0;
}
"""

# Planted errors: (the line of lit_tiles.cpp, what it becomes)
PLANTS = {
    "no-scatter-cone": ("std::atan(std::fabs(std::tan(l.scatter_rad / 2.0))) * (1 + 1e-6)", "0.0"),
    "no-footprint-inflation": ("const double R = rdev + rho;", "const double R = rdev;"),
}


def _build(d, name, plant=None):
    src = open(os.path.join(CSRC, "cuda", "lit_tiles.cpp")).read()
    if plant:
        a, b = PLANTS[plant]
        assert src.count(a) == 1, a
        src = src.replace(a, b)
    lit_src = os.path.join(d, "lit_tiles_%s.cpp" % name)
    open(lit_src, "w").write(src.replace('#include "lit_tiles.h"', '#include "%s/cuda/lit_tiles.h"' % CSRC))
    probe_src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe_%s.so" % name)
    open(probe_src, "w").write(PROBE % dict(csrc=CSRC))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, probe_src, lit_src] +
                          [os.path.join(CSRC, "cuda", f) for f in ("tiles.cpp", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_lit.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 4 + [
        C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.ftb_probe_lit.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return _build(str(tmp_path_factory.mktemp("lit_probe")), "tree")


def lit_mask(lib, sc, params, window=None):
    """([tiles_y, tiles_x] uint8 light bits of the window's tiles, the ground's primitive index or -1)."""
    x0, y0, x1, y1 = window or (0, 0, params.width, params.height)
    buf = (C.c_ubyte * (1 << 20))()
    tx, ty, prim = C.c_int(), C.c_int(), C.c_int()
    rc = lib.ftb_probe_lit(sc.desc_ptr, sc.camera_ptr, C.byref(params), x0, y0, x1, y1, buf, len(buf), C.byref(tx), C.byref(ty), C.byref(prim))
    assert rc == 0, rc
    return np.frombuffer(buf, dtype=np.uint8, count=tx.value * ty.value).reshape(ty.value, tx.value).copy(), prim.value


def _blocked(sc, o, d):
    return any(h["t"] >= 0.0 and h["apply_lighting"] for h in orc.node_hits(sc, o, d))


def check_against_oracle(lib, sc, params, max_samples=None):
    """Every lit (tile, light) holds for every ground sample of the tile in the oracle.  Returns (share of the ground samples
    with every directional light of theirs proven, number of (sample, light) pairs checked, number found blocked)."""
    mask, ground = lit_mask(lib, sc, params)
    if ground < 0:
        assert not mask.any()
        return 0.0, 0, 0
    corner = params.sampling == abi.SAMPLING_CORNER
    W, H = params.width, params.height
    gw, gh = W + corner, H + corner
    spp = 1 if corner else params.spp
    jit = [(-0.5, 0.5)] if corner else [(params.jitter_xy[2 * s], params.jitter_xy[2 * s + 1]) for s in range(spp)]
    ref = orc.render(sc, params)
    prim = ref["prim"].reshape(gh, gw, spp)
    on_ground = prim == ground
    lights = [sc.desc.lights[k] for k in range(sc.desc.n_lights)]
    directional = sum(1 << k for k, l in enumerate(lights[:8]) if l.kind != abi.LIGHT_POINT)
    bits = np.repeat(np.repeat(mask, abi.TILE_H, axis=0), abi.TILE_W, axis=1)[:gh, :gw]
    proven = on_ground & ((bits & directional) == directional)[..., None] if directional else on_ground & False
    share = float(proven.sum()) / max(1, int(on_ground.sum()))
    ys, xs, ss = np.nonzero(on_ground & (bits != 0)[..., None])
    if max_samples is not None and len(ys) > max_samples:
        pick = np.random.default_rng(0).choice(len(ys), max_samples, replace=False)
        ys, xs, ss = ys[pick], xs[pick], ss[pick]
    checked = blocked = 0
    for y, x, s in zip(ys.tolist(), xs.tolist(), ss.tolist()):
        r = orc.primary_ray(sc.camera, W, H, x, y, *jit[s])
        o, d = r[:3] + 1e-4 * r[3:], r[3:]
        hs = [h for h in orc.node_hits(sc, o, d) if h["t"] >= 0.0]
        h = min(hs, key=lambda h: h["t"])
        assert h["prim"] == ground
        origin = np.array(h["p"]) + 1e-4 * np.array(h["n"])  # shadowRayOrigin (Shading.fs:111)
        sample = y * gw + x if corner else (y * W + x) * spp + s
        for k, l in enumerate(lights[:8]):
            if not (bits[y, x] >> k) & 1:
                continue
            v = -np.array(l.v)
            dirs = [v] if l.kind == abi.LIGHT_DIRECTIONAL else [
                orc.jitter_vector(params.seed, sample, 0, k, i, l.scatter_rad, v) for i in range(l.samples)]
            for dd in dirs:
                checked += 1
                blocked += _blocked(sc, origin, dd)
    return share, checked, blocked


def _assert_holds(lib, sc, params, **kw):
    share, checked, blocked = check_against_oracle(lib, sc, params, **kw)
    assert blocked == 0, "%d of %d shadow rays of lit ground samples are blocked" % (blocked, checked)
    return share, checked


@pytest.mark.parametrize("name", sorted(scenes.CONFIGS))
def test_bundled_configs(probe, name):
    cfg = scenes.CONFIGS[name]
    W, H = (192, 108) if cfg["res"][0] > cfg["res"][1] else (120, 160)
    sc = parse(scenes.config_text(name, res=(W, H), spp=2))
    p = orc.make_params(W, H, 2, frontend.jitter_pattern(cfg["seed"], 2), sampling=sc.sampling)
    share, checked = _assert_holds(probe, sc, p, max_samples=3000)
    print("%s: %.3f of the ground samples proven lit, %d shadow rays checked" % (name, share, checked))


@pytest.mark.parametrize("seed", range(40))
def test_random_scenes(probe, seed):
    from test_gpu_fuzz import _scene
    sc = parse(_scene(1000 + seed))
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(seed + 1, sc.spp), sampling=sc.sampling, seed=77)
    _assert_holds(probe, sc, p, max_samples=2000)
    if sc.camera.has_focus:
        assert not lit_mask(probe, sc, p)[0].any()  # depth of field moves the rays' origins


CAM = "camera pos (0,1.5,-9) lookat (0,-1,0) up (0,1,0) fov 60 ratio 1.33\n"
GROUND = "(translate (0,-2,0) plane)\n\n"

HARD = {
    # a sphere standing on the ground: its shadow's edge against a soft light's cone
    "grazing-soft": CAM + "samples 2\nres 160 120\n\n" + GROUND + "(translate (0.5,-1,1) sphere)\n\n"
                    "softdirectional dir (-0.5,-1,0.3) samples 4 scatter 20 colour (1,1,1)\n",
    # an item that floats above the ground, grazing the edge of a plain light's shadow rays
    "grazing-plain": CAM + "samples 3\nres 160 120\n\n" + GROUND + "(translate (-1,0.5,2) (scale 0.7 sphere))\n\n"
                     "directional dir (0.2,-1,0.1) colour (1,1,1)\n",
    # a sphere floating over the ground under a wide soft light: a broad penumbra
    "penumbra": CAM + "samples 2\nres 160 120\n\n" + GROUND + "(translate (0,0.5,1) sphere)\n\n"
                "softdirectional dir (-0.3,-1,0.2) samples 8 scatter 40 colour (1,1,1)\n",
    "wide-scatter": CAM + "samples 2\nres 160 120\n\n" + GROUND + "(translate (1,-1.3,3) (scale 0.7 cube))\n\n"
                    "softdirectional dir (0,-1,0) samples 3 scatter 120 colour (1,1,1)\n",
    "light-nearly-parallel": CAM + "samples 2\nres 160 120\n\n" + GROUND + "(translate (0,-1,4) sphere)\n\n"
                             "directional dir (1,-0.01,0.2) colour (1,1,1)\nsoftdirectional dir (0.3,-0.05,1) samples 2 scatter 4 colour (1,1,1)\n",
    "camera-below": "camera pos (0,-4,-9) lookat (0,-2,0) up (0,1,0) fov 60 ratio 1.33\nsamples 2\nres 160 120\n\n" + GROUND +
                    "(translate (0,-1,1) sphere)\n\n(translate (1,-3,1) sphere)\n\ndirectional dir (0.3,1,0.1) colour (1,1,1)\n"
                    "directional dir (0.3,-1,0.1) colour (1,1,1)\n",
    "tilted-ground": CAM + "samples 2\nres 160 120\n\n(translate (0,-2,0) (rotate (1,0,0.5) 12 plane))\n\n(translate (0.5,-1,1) sphere)\n\n"
                     "softdirectional dir (-0.5,-1,0.3) samples 3 scatter 10 colour (1,1,1)\ndirectional dir (0.4,-1,-0.2) colour (1,1,1)\n",
    "corner-sampling": CAM + "samples corner\nres 160 120\n\n" + GROUND + "(translate (0.5,-1,1) sphere)\n\n"
                       "directional dir (-0.5,-1,0.3) colour (1,1,1)\n",
    "point-light-only": CAM + "samples 2\nres 160 120\n\n" + GROUND + "(translate (0.5,-1,1) sphere)\n\n"
                        "positional pos (0,3,0) falloff (1,0,0) colour (1,1,1)\n",
}


@pytest.mark.parametrize("name", sorted(HARD))
def test_hard_scenes(probe, name):
    sc = parse(HARD[name])
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    share, checked = _assert_holds(probe, sc, p)
    mask, _ = lit_mask(probe, sc, p)
    print("%s: %.3f of the ground samples proven lit, %d shadow rays checked" % (name, share, checked))
    if name == "point-light-only":
        assert not mask.any()
    elif name == "camera-below":
        # the first light shines on the ground's underside (the camera's side): its shadow rays start above the plane (the
        # offset follows the plane's normal) and cross it; the second one's rays leave the plane
        assert not (mask & 1).any() and (mask & 2).any()
    elif name != "light-nearly-parallel":
        assert checked > 0, "the scene must have lit ground samples, or it shows nothing"


def test_second_unbounded_item_lights_nothing(probe):
    sc = parse(CAM + "samples 1\nres 128 96\n\n" + GROUND + "(translate (0,8,0) plane)\n\n(translate (0.5,-1,1) sphere)\n\n"
               "directional dir (0.2,-1,0.1) colour (1,1,1)\n")
    p = orc.make_params(128, 96, 1, frontend.jitter_pattern(1, 1))
    mask, ground = lit_mask(probe, sc, p)
    assert ground == -1 and not mask.any()


def test_windows_and_shards_agree_with_the_whole_frame(probe):
    """The mask is indexed by the window's tile; a shard reads the window's mask, so only windows need checking."""
    sc = parse(scenes.config_text("cfg5-repeat", res=(384, 216), spp=2))
    p = orc.make_params(384, 216, 2, frontend.jitter_pattern(5, 2))
    whole, g = lit_mask(probe, sc, p)
    assert g >= 0 and whole.any()
    win, g2 = lit_mask(probe, sc, p, (64, 96, 320, 216))  # tile-aligned: the same tiles
    assert g2 == g and win.any() and (win == whole[6:14, 4:20]).all()


@pytest.mark.parametrize("plant, scene", [("no-scatter-cone", "penumbra"), ("no-footprint-inflation", "penumbra")])
def test_planted_errors_are_caught(tmp_path, probe, plant, scene):
    sc = parse(HARD[scene])
    p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(5, sc.spp), sampling=sc.sampling)
    bad = _build(str(tmp_path), plant, plant)
    _, checked, blocked = check_against_oracle(bad, sc, p)
    assert blocked > 0, "the planted error %s went unnoticed (%d shadow rays checked)" % (plant, checked)


def test_headline_share(probe):
    """cfg5-repeat at a reduced size: the share of ground samples whose directional shadow is proven (tools/lit_tile_share.py
    prints it for every config)."""
    cfg = scenes.CONFIGS["cfg5-repeat"]
    sc = parse(scenes.config_text("cfg5-repeat", res=(768, 432), spp=1))
    p = orc.make_params(768, 432, 1, frontend.jitter_pattern(cfg["seed"], 1))
    share, checked = _assert_holds(probe, sc, p, max_samples=3000)
    print("cfg5-repeat 768x432: %.3f of the ground samples proven lit" % share)
    assert share > 0.5, share
