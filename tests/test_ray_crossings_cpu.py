"""CPU-side checks of the crossing queries (ftb_intersect_all_rays and its device form): the prototypes in the header and in
abi.EXPORTS, the ctypes signatures, the argument checks that need no device; and the one cull the crossings kernel makes - an
item whose bounding sphere the ray's LINE misses - against every crossing the oracle reports at any t.  No compute calls."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from functracer_b200 import abi, api, frontend, scenes
from test_lowering_cpu import _item_bounds, _rays, probe  # noqa: F401  (probe: the fixture of the real lowering)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "functracer_b200.h")
CROSSING_EXPORTS = {"ftb_intersect_all_rays": 10, "ftb_intersect_all_rays_device": 11}


def test_crossing_prototypes_are_declared_and_exported():
    raw = open(HEADER).read()
    assert int(re.search(r"#define FTB_MAX_CROSSINGS (\d+)\b", raw).group(1)) == api.MAX_CROSSINGS == 64
    text = re.sub(r"/\*.*?\*/", "", raw, flags=re.S)
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(ftb_[a-z_0-9]+)\s*\(([^)]*)\)\s*;", text)}
    for name, arity in CROSSING_EXPORTS.items():
        assert name in protos and name in abi.EXPORTS, name
        assert protos[name].count(",") + 1 == arity, name
    assert re.search(r"#define FTB_ABI_VERSION 4\b", text)  # additive: the ABI version stays
    L = api.lib()
    for name, arity in CROSSING_EXPORTS.items():
        assert len(getattr(L, name).argtypes) == arity, name
    assert L.ftb_intersect_all_rays.argtypes[3] is C.c_int32 and L.ftb_intersect_all_rays.argtypes[4:6] == [C.c_double, C.c_double]


def _calls(L, scene, rays, n, max_hits, t_min, t_max, counts, hit):
    """The host and the device entry with the same arguments."""
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    p = api.make_params(1, 1, 1, None)
    r = rays.ctypes.data_as(dp) if rays is not None else None
    c = counts.ctypes.data_as(ip) if counts is not None else None
    return (L.ftb_intersect_all_rays(scene, r, n, max_hits, t_min, t_max, C.byref(p), C.byref(hit), c, None),
            L.ftb_intersect_all_rays_device(scene, r, n, max_hits, t_min, t_max, C.byref(p), C.byref(hit), c, None, None))


def test_crossing_arguments_are_checked_before_any_device_is_needed():
    """Each bad argument alone is FTB_ERR_BAD_ARG, with a scene handle that is never dereferenced: the checks come before any
    device is looked for.  A valid call without a GPU is FTB_ERR_NO_DEVICE, n = 0 included (as for the other queries); with one, n = 0
    is OK."""
    L = api.lib()
    fake = C.c_void_p(0x10)  # never dereferenced by an argument check
    rays, counts, hit = np.zeros((4, 6)), np.zeros(4, np.int32), abi.HitOut()
    good = dict(scene=fake, rays=rays, n=4, max_hits=8, t_min=-math.inf, t_max=math.inf, counts=counts)
    bad = [dict(max_hits=0), dict(max_hits=-3), dict(max_hits=65), dict(t_min=math.nan), dict(t_max=math.nan), dict(t_min=1.0, t_max=1.0),
           dict(t_min=2.0, t_max=1.0), dict(t_min=math.inf, t_max=math.inf), dict(t_min=-math.inf, t_max=-math.inf), dict(rays=None),
           dict(counts=None), dict(scene=None), dict(n=-1)]
    for change in bad:
        args = dict(good, **change)
        assert _calls(L, hit=hit, **args) == (abi.ERR_BAD_ARG, abi.ERR_BAD_ARG), change
    empty = 0 if L.ftb_device_count() > 0 else abi.ERR_NO_DEVICE
    assert _calls(L, hit=hit, **dict(good, n=0, rays=None, counts=None)) == (empty, empty)
    assert _calls(L, hit=hit, **dict(good, max_hits=64, t_min=0.0, t_max=1.0, n=0)) == (empty, empty)
    if L.ftb_device_count() == 0:
        assert _calls(L, hit=hit, **good) == (abi.ERR_NO_DEVICE, abi.ERR_NO_DEVICE)
        assert b"no CUDA device" in L.ftb_last_error()


def test_python_crossing_planes_have_the_entry_width():
    out, hit = api._hit_planes(("t", "prim", "p", "surface"), 5, 8)
    assert out["t"].shape == (5, 8) and out["prim"].shape == (5, 8) and out["p"].shape == (5, 8, 3) and out["surface"].shape == (5, 8, 4)
    assert hit.t and hit.prim_id and not hit.sub_id and hit.p and not hit.normal and hit.surface


# ---- the crossings kernel's only cull, against every crossing at any t --------------------------------------------------------
def _check_line_cull(sc, bounds, prim_item, o, d, label):
    """Every crossing the oracle reports, at ANY t, belongs to an item whose bounding sphere the ray's line touches, and lies in that
    sphere.  Exempt and counted: Plane.fs's t = 0 crossing of a ray parallel to a planar face (DESIGN.md §6), which lies at the
    origin wherever the face is.  Returns (checked, behind the origin, t = 0 parallel crossings)."""
    from oracle import ftb_oracle as orc
    checked = behind = parallel = 0
    for k in range(o.shape[0]):
        du = d[k] / np.linalg.norm(d[k])
        for h in orc.node_hits(sc, o[k], d[k], max_hits=4096):
            if not np.isfinite(h["t"]):
                continue
            it = prim_item[h["prim"]]
            assert it >= 0, (label, "primitive %d belongs to no item" % h["prim"])
            c, r = bounds[it, :3], bounds[it, 3]
            if r < 0:
                continue  # unbounded: never culled
            if h["t"] == 0.0 and np.array_equal(np.array(h["p"]), o[k]):
                parallel += 1
                continue
            oc = c - o[k]
            b = float(oc @ du)
            dist2 = float(oc @ oc) - b * b
            assert dist2 <= r * r * (1 + 1e-9) + 1e-12, (label, k, h["prim"], h["t"], "line misses the bound by %g" % (math.sqrt(max(dist2, 0)) - r))
            p = o[k] + h["t"] * d[k]
            assert np.linalg.norm(p - c) <= r * (1 + 1e-9) + 1e-9, (label, k, h["prim"], h["t"], "crossing outside the bound")
            checked += 1
            behind += h["t"] < 0
    return checked, behind, parallel


@pytest.mark.parametrize("seed", range(24))
def test_no_crossing_at_any_t_lies_off_its_items_line_bound(probe, seed):  # noqa: F811
    """tests/test_lowering_cpu.py checks the renderer's cull (line miss, or sphere behind the origin) against the crossings with
    t >= 0.  The crossings kernel reports crossings behind the origin too and keeps only the line test: checked here on the same
    random scenes and rays, at every t."""
    from test_gpu_fuzz import _scene
    from util import parse
    sc = parse(_scene(1000 + seed))
    bounds, prim_item = _item_bounds(probe, sc)
    o, d = _rays(np.random.default_rng(seed), 400)
    checked, behind, parallel = _check_line_cull(sc, bounds, prim_item, o, d, seed)
    print("seed %d: %d items, %d crossings checked (%d behind the origin), %d parallel t = 0 crossings" % (seed, bounds.shape[0], checked, behind,
                                                                                                           parallel))


@pytest.mark.parametrize("name", ["cfg1-sample", "cfg2-hollow-sphere", "cfg3-house", "cfg3-night-house", "cfg4-bunny-d12", "cfg5-repeat", "cfg5-moon"])
def test_bundled_scenes_crossings_at_any_t_lie_inside_their_items_bounds(probe, name):  # noqa: F811
    sc = frontend.ParsedScene(scenes.config_text(name, res=(64, 48), spp=1), scenes.asset_dir())
    bounds, prim_item = _item_bounds(probe, sc)
    rng = np.random.default_rng(7)
    cam = np.array(sc.camera.o[:3])
    look = np.array(sc.camera.look_at[:3])
    n = 300
    fwd = (look - cam) / np.linalg.norm(look - cam)
    o = np.vstack([cam + rng.normal(scale=0.05, size=(n, 3)), rng.uniform([-20, 0.01, -5], [20, 6, 60], size=(n, 3))])
    d = np.vstack([fwd + rng.normal(scale=0.35, size=(n, 3)), rng.normal(size=(n, 3)) + np.array([0.0, 0.6, 0.0])])
    checked, behind, parallel = _check_line_cull(sc, bounds, prim_item, o, d, name)
    print("%s: %d items, %d crossings checked (%d behind the origin), %d parallel t = 0 crossings" % (name, bounds.shape[0], checked, behind, parallel))
    assert checked > 0 or name == "cfg1-sample"
