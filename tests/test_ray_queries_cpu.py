"""CPU-side checks of the ray-query entry points (ftb_intersect_rays, ftb_occluded_rays and their device forms): ftb_hit_out's
layout against gcc, the prototypes in the header and in abi.EXPORTS, the ctypes signatures, and the argument checks that
need no device.  No compute calls."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from functracer_b200 import abi, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "functracer_b200.h")
QUERY_EXPORTS = ["ftb_intersect_rays", "ftb_occluded_rays", "ftb_intersect_rays_device", "ftb_occluded_rays_device"]


def test_hit_out_layout_matches_header():
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "%s"' % HEADER, "int main(void){",
             'printf("size %zu\\n", sizeof(ftb_hit_out));']
    for fname, _ in abi.HitOut._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(ftb_hit_out, %s));' % (fname, fname))
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "l.c"), os.path.join(d, "l")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-o", exe, src])
        got = dict(l.split() for l in subprocess.check_output([exe], text=True).strip().splitlines())
    assert int(got["size"]) == C.sizeof(abi.HitOut) == 56
    for fname, _ in abi.HitOut._fields_:
        assert int(got[fname]) == getattr(abi.HitOut, fname).offset, fname
    assert [f for f, _ in abi.HitOut._fields_] == ["t", "prim_id", "sub_id", "p", "normal", "colour", "surface"]


def test_query_prototypes_are_declared_and_exported():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(ftb_[a-z_0-9]+)\s*\(([^)]*)\)\s*;", text)}
    want = {"ftb_intersect_rays": 6, "ftb_occluded_rays": 7, "ftb_intersect_rays_device": 7, "ftb_occluded_rays_device": 8}
    for name, arity in want.items():
        assert name in protos and name in abi.EXPORTS, name
        assert protos[name].count(",") + 1 == arity, name
    assert re.search(r"#define FTB_ABI_VERSION 4\b", text)  # additive: the ABI version stays
    L = api.lib()
    for name in QUERY_EXPORTS:
        assert getattr(L, name).argtypes is not None, name


def test_query_arguments_are_checked_before_any_device_is_needed():
    """A NULL scene, a negative count, NULL rays / max_t / blocked: FTB_ERR_BAD_ARG, with or without a GPU."""
    L = api.lib()
    p = api.make_params(1, 1, 1, None)
    rays = np.zeros((4, 6))
    mt = np.full(4, np.inf)
    blocked = np.zeros(4, np.int32)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    hit = abi.HitOut()
    calls = [
        lambda: L.ftb_intersect_rays(None, rays.ctypes.data_as(dp), 4, C.byref(p), C.byref(hit), None),
        lambda: L.ftb_intersect_rays(None, None, 0, C.byref(p), None, None),
        lambda: L.ftb_intersect_rays(None, rays.ctypes.data_as(dp), -1, C.byref(p), None, None),
        lambda: L.ftb_occluded_rays(None, rays.ctypes.data_as(dp), mt.ctypes.data_as(dp), 4, C.byref(p), blocked.ctypes.data_as(ip), None),
        lambda: L.ftb_intersect_rays_device(None, rays.ctypes.data_as(dp), 4, C.byref(p), C.byref(hit), None, None),
        lambda: L.ftb_occluded_rays_device(None, rays.ctypes.data_as(dp), mt.ctypes.data_as(dp), 4, C.byref(p), blocked.ctypes.data_as(ip), None, None),
    ]
    for call in calls:
        assert call() == abi.ERR_BAD_ARG
    assert b"null argument" in L.ftb_last_error()


def test_python_planes_are_validated():
    with pytest.raises(ValueError):
        api._hit_planes(("t", "depth"), 3)
    out, hit = api._hit_planes(("prim", "surface"), 5)
    assert set(out) == {"prim", "surface"} and out["surface"].shape == (5, 4) and out["prim"].dtype == np.int32
    assert not hit.t and hit.prim_id and not hit.p and hit.surface
