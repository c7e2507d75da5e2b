"""CPU-side checks of the path queries (ftb_trace_paths and its device form): ftb_path_out's layout against gcc, the prototypes
in the header and in abi.EXPORTS, the ctypes signatures and the argument checks that need no device.  And the test helper
itself (tests/path_oracle.py): its breakdown, summed the way the kernel sums it, must give the oracle's own getColourForRay
colour, whose summation order differs (the reflection inside each light's fragment)."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import path_oracle
from functracer_b200 import abi, api, frontend, scenes
from oracle import ftb_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "functracer_b200.h")
PATH_EXPORTS = {"ftb_trace_paths": 7, "ftb_trace_paths_device": 8}
BUNDLED = ["cfg1-sample", "cfg2-hollow-sphere", "cfg3-house", "cfg3-night-house", "cfg4-bunny-d12", "cfg5-repeat", "cfg5-moon"]


def _layout(struct, fields):
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "%s"' % HEADER, "int main(void){",
             'printf("size %%zu\\n", sizeof(%s));' % struct]
    for fname in fields:
        lines.append('printf("%s %%zu\\n", offsetof(%s, %s));' % (fname, struct, fname))
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "l.c"), os.path.join(d, "l")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-o", exe, src])
        return {k: int(v) for k, v in (l.split() for l in subprocess.check_output([exe], text=True).strip().splitlines())}


def test_path_out_layout_matches_header():
    names = [f for f, _ in abi.PathOut._fields_]
    assert names == ["levels", "colour", "ray_od", "weight", "hit", "intensity", "light_dir", "light_colour"]
    got = _layout("ftb_path_out", names + ["hit.surface"])
    assert got["size"] == C.sizeof(abi.PathOut) == 112
    for fname in names:
        assert got[fname] == getattr(abi.PathOut, fname).offset, fname
    assert got["hit.surface"] == abi.PathOut.hit.offset + abi.HitOut.surface.offset


def test_path_prototypes_are_declared_and_exported():
    raw = open(HEADER).read()
    assert int(re.search(r"#define FTB_MAX_PATH_LEVELS (\d+)\b", raw).group(1)) == api.MAX_PATH_LEVELS == 64
    text = re.sub(r"/\*.*?\*/", "", raw, flags=re.S)
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(ftb_[a-z_0-9]+)\s*\(([^)]*)\)\s*;", text)}
    for name, arity in PATH_EXPORTS.items():
        assert name in protos and name in abi.EXPORTS, name
        assert protos[name].count(",") + 1 == arity, name
    assert "const uint64_t* sample_keys" in protos["ftb_trace_paths"] and "const ftb_path_out* out" in protos["ftb_trace_paths"]
    assert re.search(r"#define FTB_ABI_VERSION 4\b", text)  # additive: the ABI version stays
    L = api.lib()
    for name, arity in PATH_EXPORTS.items():
        args = getattr(L, name).argtypes
        assert len(args) == arity, name
        assert args[2] is C.POINTER(C.c_uint64) and args[3] is C.c_int64 and args[5] is C.POINTER(abi.PathOut), name


def _calls(L, scene, rays, n, keys, params, out):
    """The host and the device entry with the same arguments."""
    r = rays.ctypes.data_as(C.POINTER(C.c_double)) if rays is not None else None
    k = keys.ctypes.data_as(C.POINTER(C.c_uint64)) if keys is not None else None
    p = C.byref(params) if params is not None else None
    return (L.ftb_trace_paths(scene, r, k, n, p, C.byref(out), None),
            L.ftb_trace_paths_device(scene, r, k, n, p, C.byref(out), None, None))


def test_path_arguments_are_checked_before_any_device_is_needed():
    """Each bad argument alone is FTB_ERR_BAD_ARG, with a scene handle that is never dereferenced: the checks come before any
    device is looked for.  A valid call without a GPU is FTB_ERR_NO_DEVICE, n = 0 included; with one, n = 0 is OK."""
    L = api.lib()
    fake = C.c_void_p(0x10)  # never dereferenced by an argument check
    rays, keys, out = np.zeros((4, 6)), np.arange(4, dtype=np.uint64), abi.PathOut()
    P = lambda **kw: api.make_params(1, 1, 1, None, **kw)  # noqa: E731
    good = dict(scene=fake, rays=rays, n=4, keys=keys, params=P())
    bad = [dict(scene=None), dict(params=None), dict(n=-1), dict(rays=None), dict(params=P(precision=2)), dict(params=P(precision=-1)),
           dict(params=P(recursion_limit=-1)), dict(params=P(recursion_limit=64)), dict(params=P(recursion_limit=1000))]
    for change in bad:
        args = dict(good, **change)
        assert _calls(L, out=out, **args) == (abi.ERR_BAD_ARG, abi.ERR_BAD_ARG), change
    empty = 0 if L.ftb_device_count() > 0 else abi.ERR_NO_DEVICE
    assert _calls(L, out=out, **dict(good, n=0, rays=None, keys=None)) == (empty, empty)
    assert _calls(L, out=out, **dict(good, n=0, params=P(recursion_limit=63))) == (empty, empty)
    if L.ftb_device_count() == 0:
        assert _calls(L, out=out, **dict(good, keys=None)) == (abi.ERR_NO_DEVICE, abi.ERR_NO_DEVICE)
        assert b"no CUDA device" in L.ftb_last_error()


def test_python_path_planes_are_validated():
    class Fake:
        pass
    s = api.Scene.__new__(api.Scene)  # never opened: trace_paths rejects the planes before it calls the library
    s.parsed = Fake()
    with pytest.raises(ValueError):
        s.trace_paths(np.zeros((2, 6)), planes=("colour", "depth"))
    with pytest.raises(ValueError):
        s.trace_paths_device(0, 2, {"rgb": 0})
    assert set(api.PATH_PLANES) == {"levels", "colour", "ray", "weight", "t", "prim", "sub", "p", "normal", "hit_colour", "surface",
                                    "intensity", "light_dir", "light_colour"}


# ---- the helper: its breakdown summed as the kernel sums it = the oracle's getColourForRay ----------------------------------------
def _rays(sc, rng, W=16, H=12, n=64):
    cam = np.array([orc.primary_ray(sc.camera, W, H, x, y) for y in range(H) for x in range(W)])
    o = cam[:, :3].mean(axis=0) + rng.normal(scale=2.0, size=(n, 3))
    d = rng.normal(size=(n, 3))
    return np.vstack([cam, np.hstack([o, d / np.linalg.norm(d, axis=1, keepdims=True)])])


def _check_helper(sc, rays, label, recursion_limit=8):
    r = path_oracle.paths(sc, rays, recursion_limit=recursion_limit)
    got = path_oracle.replay(r["levels"], r["weight"], r["light_colour"])
    ref = r["ref"]
    L = r["intensity"].shape[2]
    # the size of the terms the two orders add up: the bar is relative to them
    mag = np.abs(ref) + (np.abs(r["weight"])[..., None] * np.abs(np.nan_to_num(r["light_colour"])).sum(axis=2)).sum(axis=1)
    nan = np.isnan(ref) | np.isnan(got)
    assert (np.isnan(ref) == np.isnan(got)).all(), label
    err = np.where(nan, 0.0, np.abs(got - ref))
    assert (err <= 1e-12 * mag + 1e-300).all(), (label, float((err / np.maximum(mag, 1e-300)).max()))
    lv = r["levels"]
    assert ((lv >= 1) & (lv <= recursion_limit + 1)).all(), label
    D = recursion_limit + 1
    after = np.arange(D)[None, :] >= lv[:, None]
    assert (r["weight"][after] == 0).all() and (r["prim"][after] == -1).all() and (r["t"][after] == -1).all(), label
    print("%s: %d rays, %d lights, levels max %d mean %.2f, largest error %.3g of the terms" % (label, len(rays), L, lv.max(), lv.mean(),
                                                                                              float((err / np.maximum(mag, 1e-300)).max())))


@pytest.mark.parametrize("name", BUNDLED)
def test_helper_sums_to_the_oracles_colour_on_bundled_scenes(name):
    sc = frontend.ParsedScene(scenes.config_text(name, res=(64, 48), spp=1), scenes.asset_dir())
    _check_helper(sc, _rays(sc, np.random.default_rng(3)), name)


@pytest.mark.parametrize("seed", range(24))
def test_helper_sums_to_the_oracles_colour_on_random_scenes(seed):
    from test_gpu_fuzz import _scene
    from util import parse
    sc = parse(_scene(1000 + seed))
    _check_helper(sc, _rays(sc, np.random.default_rng(seed)), "fuzz %d" % seed)
