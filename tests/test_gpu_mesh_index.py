"""The mesh index built on the device (bvh_build.cu), checked like the host-built one (test_lowering_cpu.py
test_host_mesh_index_invariants) with the same checker (tests/mesh_index_check.h).  Needs a B200: run with `-m gpu`.

A probe compiled with the library's nvcc flags from bvh_build.cu, lower.cpp and a small entry lowers a scene, enumerates its
meshes and builds their index on the device exactly as ftb_scene_create does for large meshes (windows 16, 8, 4; the
64-entry traversal stack as the depth bound).  It then walks the result: every slot reached once, FP32 and FP64 child boxes
that contain every double-precision vertex below them, leaves of 1-4 triangles, `seq` = the enumeration rank and bvh_tri
naming the triangles of every mesh, and a depth the traversal stack holds."""
import ctypes as C
import os
import re
import subprocess

import pytest

import large_mesh_scenes as lms
from functracer_b200 import abi, frontend, scenes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "functracer_b200", "csrc")
TESTS = os.path.dirname(os.path.abspath(__file__))
STACK = 64  # device_scene.h kBspStack

ENTRY = r"""
#include "%(csrc)s/cuda/bvh_build.h"
#include "%(csrc)s/cuda/device_scene.h"
#include "%(tests)s/mesh_index_check.h"
#include <cstring>
// Returns the number of triangle slots checked (> 0), 0 when every window's build was refused (err says why), or a
// negative code: -1 the lowering failed, else mesh_index_check.h's codes.
extern "C" long ftb_probe_device_index(const ftb_scene_desc* d, int* reported_depth, int* walk_depth, int* radius, char* err, int errlen)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) { std::strncpy(err, e.c_str(), (size_t)errlen - 1); return -1; }
    std::vector<std::vector<int32_t>> order;
    ftb::enumerateMeshes(*d, L, order);
    const int radii[3] = {16, 8, 4};
    bool done = false;
    std::string why;
    for (int k = 0; k < 3 && !done; ++k) {
        ftb::DeviceBuildStats st;
        std::string w;
        done = ftb::buildMeshIndexDevice(d->triangles, d->n_triangles, order, ftb::kBspStack, radii[k], L, st, w);
        if (done) *radius = radii[k];
        else why += (why.empty() ? "" : "; ") + w;
    }
    std::strncpy(err, why.c_str(), (size_t)errlen - 1);
    err[errlen - 1] = 0;
    if (!done) return 0;
    *reported_depth = L.max_bvh_depth;
    return checkMeshIndex(d, L, order, 4, walk_depth);
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("device_index_probe"))
    src, so = os.path.join(d, "entry.cu"), os.path.join(d, "libprobe.so")
    open(src, "w").write(ENTRY % dict(csrc=CSRC, tests=TESTS))
    mk = open(os.path.join(CSRC, "Makefile")).read()
    arch = re.search(r"^ARCH := (.*)$", mk, flags=re.M).group(1).split()
    nvflags = re.search(r"^NVFLAGS := (.*)$", mk, flags=re.M).group(1).replace("$(ARCH)", " ".join(arch)).split()
    r = subprocess.run(["nvcc"] + nvflags + ["-shared", "-o", so, src, os.path.join(CSRC, "cuda", "bvh_build.cu"), os.path.join(CSRC, "cuda", "lower.cpp"),
                        "-lcudart"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-4000:]
    lib = C.CDLL(so)
    lib.ftb_probe_device_index.argtypes = [C.POINTER(abi.SceneDesc)] + [C.POINTER(C.c_int)] * 3 + [C.c_char_p, C.c_int]
    lib.ftb_probe_device_index.restype = C.c_long
    return lib


def _families():
    out = {"bunny_full": None, "geometric_sequence": lms.geometric_sequence}
    out.update({n: getattr(lms, n) for n in ("two_large_and_small", "many_small_meshes", "transformed_instances", "planar_grid",
                                              "fan", "slivers", "coincident", "shiny_blob", "twin_instances")})
    out["tie"] = lambda d: lms.tie(d, lms.LARGE_MESH)[:2]
    out["just_above_threshold"] = lambda d: lms.just_below_threshold(d, True)
    return out


FAMILIES = _families()


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_device_mesh_index_invariants(probe, tmp_path, family):
    if family == "bunny_full":
        sc = frontend.ParsedScene(scenes.config_text("cfg4-bunny-full-d14", res=(32, 24), spp=1), scenes.asset_dir())
    else:
        text, d = FAMILIES[family](str(tmp_path))
        sc = frontend.ParsedScene(text, d)
    reported, walked, radius = C.c_int(-1), C.c_int(-1), C.c_int(0)
    err = C.create_string_buffer(1024)
    n = probe.ftb_probe_device_index(sc.desc_ptr, C.byref(reported), C.byref(walked), C.byref(radius), err, 1024)
    why = err.value.decode()
    print("%s: %d meshes, %d triangles -> %d slots checked, window %d, depth reported %d, walked %d%s"
          % (family, sc.desc.n_meshes, sc.desc.n_triangles, n, radius.value, reported.value, walked.value, (" (" + why + ")") if why else ""))
    if family in ("geometric_sequence", "coincident") and n == 0:
        # refused by every window: too deep for the traversal stack, or (coincident boxes) no clustering progress
        assert ("deeper than the traversal stack" in why) or (family == "coincident" and "no progress" in why), why
        return
    assert n > 0, "violation %d (%s)" % (n, why)
    assert walked.value <= reported.value + 1  # the depth api.cu checks against the stack is the tree's own
    assert reported.value + 2 <= STACK and walked.value + 1 <= STACK
