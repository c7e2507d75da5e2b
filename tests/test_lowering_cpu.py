"""Host-side decisions of the product path, tested with the REAL lowering (lower.cpp compiled with g++ into a throw-away probe,
no device involved).  CPU only.

1. Which kernel a scene runs on: lower.cpp derives the scene's feature mask, api.cu launches the smallest compiled variant that
   covers it (csrc/Makefile F32_FEATS) and falls back to the generic 0xfff kernel - correct, but 1.3-2x slower - when no
   specialised variant does.  A drifting feature bit would cost the headline silently, so the variant every BASELINE.json config
   is documented to use (BENCH.md, DESIGN.md section 3) is pinned here.
2. The object-level cull: the kernel skips an item whose bounding sphere the ray's line misses or that lies behind the origin.
   Every crossing with t >= 0 that the reference's algorithm (the oracle's full hit lists) reports must belong to an item that
   passes both tests, for random rays on random and bundled scenes."""
import ctypes as C
import os
import re
import subprocess

import pytest

from functracer_b200 import abi, frontend, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "functracer_b200", "csrc")

PROBE = r"""
#include "%(csrc)s/cuda/lower.h"
#include <algorithm>
#include <cstring>
extern "C" int ftb_probe_lower(const ftb_scene_desc* d, unsigned* features, int* counts, char* err, int errlen)
{
    ftb::Lowered L;
    std::string e;
    const int rc = ftb::lower_scene(*d, L, e, true);  // with the host-built mesh index: its size decides the large-mesh walk
    std::strncpy(err, e.c_str(), (size_t)errlen - 1);
    err[errlen - 1] = 0;
    if (rc != 0) return rc;
    *features = L.features;
    counts[0] = (int)L.items.size();
    counts[1] = (int)L.leaves.size();
    counts[2] = (int)L.bvh_tri.size();
    counts[3] = (int)L.ops.size();
    return 0;
}
// The items' conservative bounding spheres (centre, radius; radius < 0 = unbounded) and the item each PRIMITIVE instance belongs to.
extern "C" int ftb_probe_bounds(const ftb_scene_desc* d, int max_items, double* bounds, int max_prims, int* prim_item, int* n_items, int* n_prims)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -1;
    *n_items = (int)L.items.size();
    *n_prims = L.n_prims;
    if (*n_items > max_items || *n_prims > max_prims) return -2;
    for (int p = 0; p < *n_prims; ++p) prim_item[p] = -1;
    for (int i = 0; i < *n_items; ++i) {
        const ftb::Item& it = L.items[(size_t)i];
        for (int k = 0; k < 3; ++k) bounds[4 * i + k] = it.bound_c[k];
        bounds[4 * i + 3] = it.bound_r;
        if ((it.kind & 0xff) == ftb::ITEM_LEAF) prim_item[L.leaves[(size_t)it.a].prim] = i;
        else
            for (int o = it.prog_first; o < it.prog_first + it.prog_count; ++o)
                if (L.ops[(size_t)o].kind == ftb::OP_LEAF) prim_item[L.leaves[(size_t)L.ops[(size_t)o].arg].prim] = i;
    }
    return 0;
}
// The host-built mesh index (buildMeshIndexHost, the builder of meshes below 32 768 triangles and the device build's fallback):
// tests/mesh_index_check.h's invariants with leaves of 1..7 slots, and a depth that agrees with the one the lowering reports
// (api.cu refuses a scene whose index the traversal stack cannot hold).
#include "%(tests)s/mesh_index_check.h"
extern "C" long ftb_probe_mesh_index(const ftb_scene_desc* d, int* depth_out)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, true) != 0) return -1;
    std::vector<std::vector<int32_t>> order;
    ftb::enumerateMeshes(*d, L, order);
    int maxDepth = 0;
    const long checked = checkMeshIndex(d, L, order, 7, &maxDepth);
    if (checked < 0) return checked;
    if (maxDepth != 0 && maxDepth > L.max_bvh_depth + 1) return -19;
    *depth_out = L.max_bvh_depth;
    return checked;
}
"""

FT_TABLE, FT_RNG, FT_MESHPK, FT_ALL = 0x200, 0x40, 0x800, 0xfff
LARGE_MESH = 32768  # api.cu kLargeMesh


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(str(tmp_path_factory.mktemp("lower_probe")))


def build_probe(d):
    """The probe library, compiled into directory d."""
    src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe.so")
    open(src, "w").write(PROBE % dict(csrc=CSRC, tests=os.path.dirname(os.path.abspath(__file__))))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src, os.path.join(CSRC, "cuda", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_lower.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(C.c_uint), C.POINTER(C.c_int), C.c_char_p, C.c_int]
    lib.ftb_probe_lower.restype = C.c_int
    lib.ftb_probe_bounds.argtypes = [C.POINTER(abi.SceneDesc), C.c_int, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.ftb_probe_bounds.restype = C.c_int
    lib.ftb_probe_mesh_index.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(C.c_int)]
    lib.ftb_probe_mesh_index.restype = C.c_long
    return lib


def compiled_variants():
    mk = open(os.path.join(CSRC, "Makefile")).read()
    return [int(x, 16) for x in re.search(r"^F32_FEATS := (.*)$", mk, flags=re.M).group(1).split()]


def constants_agree_with_the_sources():
    api_cu = open(os.path.join(CSRC, "cuda", "api.cu")).read()
    dev = open(os.path.join(CSRC, "cuda", "device_scene.h")).read()
    assert int(re.search(r"kLargeMesh = (\d+)", api_cu).group(1)) == LARGE_MESH
    for name, val in (("FT_TABLE", FT_TABLE), ("FT_RNG", FT_RNG), ("FT_MESHPK", FT_MESHPK), ("FT_ALL", FT_ALL)):
        assert int(re.search(r"\b%s = (0x[0-9a-f]+)" % name, dev).group(1), 16) == val, name


def pick(need, variants):
    """api.cu pickVariant: the cover with the fewest feature bits; the table bit is dropped rather than going generic."""
    def cover(n):
        best = None
        for v in variants:
            if v & n == n and (best is None or bin(v).count("1") < bin(best).count("1")):
                best = v
        return best
    v = cover(need)
    if need & FT_TABLE and (v is None or v == FT_ALL):
        w = cover(need & ~FT_TABLE)
        if w is not None and w != FT_ALL:
            return w
    return v


def lowered(probe, text, assets=None):
    sc = frontend.ParsedScene(text, assets or scenes.asset_dir())
    feats, counts, err = C.c_uint(0), (C.c_int * 4)(), C.create_string_buffer(256)
    rc = probe.ftb_probe_lower(sc.desc_ptr, C.byref(feats), counts, err, 256)
    assert rc == 0, err.value
    need = feats.value
    if counts[2] >= LARGE_MESH:
        need |= FT_MESHPK  # api.cu: a large mesh is walked by the whole warp
    if sc.camera.has_focus:
        need |= FT_RNG      # api.cu: depth of field draws random numbers
    return need, list(counts)


# the variant every BASELINE.json config is measured on (BENCH.md section 2)
EXPECTED = {
    "cfg1-sample": 0x050, "cfg2-hollow-sphere": 0x209, "cfg3-house": 0x74b, "cfg3-night-house": 0x74b, "cfg4-bunny": 0x004,
    "cfg4-bunny-d12": 0x004, "cfg4-bunny-full-d14": 0x804, "cfg5-repeat": 0x74b, "cfg5-moon": 0x030,
}


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_every_baseline_config_runs_on_its_specialised_kernel(probe, name):
    constants_agree_with_the_sources()
    variants = compiled_variants()
    assert FT_ALL in variants  # the generic kernel (also the counting kernel) must exist
    need, counts = lowered(probe, scenes.config_text(name, res=(64, 48), spp=1))  # the feature mask does not depend on the frame size
    v = pick(need, variants)
    print("%s: %d items, %d leaves, %d mesh slots, needs 0x%03x -> variant 0x%03x" % (name, counts[0], counts[1], counts[2], need, v))
    assert v == EXPECTED[name], "%s needs 0x%03x and would run on 0x%03x" % (name, need, v)
    assert v != FT_ALL


def test_the_table_is_only_asked_for_when_it_fits():
    """lower.h wantsOriginTable: at least 8 items, and (1 + lights) rows of the padded item count within 256 slots."""
    hdr = open(os.path.join(CSRC, "cuda", "lower.h")).read()
    assert re.search(r"kOriginCap = 256\b", hdr) and re.search(r"kOriginMinItems = 8\b", hdr)
    assert "((n_items + 1) & ~1)" in hdr  # the rows of an origin are padded to an even count (render.cuh tabStride)


# ---- the items' bounding spheres against every crossing the reference's algorithm reports ---------------------------------------
def _item_bounds(probe, sc):
    bounds, prim_item = (C.c_double * (4 * 4096))(), (C.c_int * 65536)()
    ni, npr = C.c_int(0), C.c_int(0)
    assert probe.ftb_probe_bounds(sc.desc_ptr, 4096, bounds, 65536, prim_item, C.byref(ni), C.byref(npr)) == 0
    import numpy as np
    return np.array(bounds[:4 * ni.value]).reshape(-1, 4), np.array(prim_item[:npr.value])


def _rays(rng, n):
    """Rays towards the scene from all around it, rays that start inside it, and near-parallel grazing rays."""
    import numpy as np
    o = rng.normal(size=(n, 3))
    o *= (rng.uniform(0.0, 9.0, size=(n, 1)) / np.linalg.norm(o, axis=1, keepdims=True))
    target = rng.uniform(-2.5, 2.5, size=(n, 3))
    d = target - o
    d *= rng.uniform(0.2, 3.0, size=(n, 1)) / np.linalg.norm(d, axis=1, keepdims=True)  # the reference never normalises d
    return o, d


@pytest.mark.parametrize("seed", range(24))
def test_no_crossing_the_reference_reports_lies_outside_its_items_bound(probe, seed):
    """The kernel skips an item when the ray's line misses the item's bounding sphere, or when the sphere lies entirely behind the
    origin (render.cuh traceScene).  That is only right if every crossing with t >= 0 that Scene.intersect reports for a primitive
    of the item passes both tests.  Checked here in double, against the oracle's full hit lists (ftbo_node_hits = the reference's
    sequence of hits), on the random scenes of the GPU fuzz suite and random rays - origins outside, inside and far away."""
    import numpy as np
    from oracle import ftb_oracle as orc
    from test_gpu_fuzz import _scene
    from util import parse
    sc = parse(_scene(1000 + seed))
    bounds, prim_item = _item_bounds(probe, sc)
    rng = np.random.default_rng(seed)
    o, d = _rays(rng, 400)
    checked = 0
    for k in range(o.shape[0]):
        du = d[k] / np.linalg.norm(d[k])
        for h in orc.node_hits(sc, o[k], d[k]):
            if not (h["t"] >= 0.0) or not np.isfinite(h["t"]):
                continue
            it = prim_item[h["prim"]]
            assert it >= 0, "primitive %d belongs to no item" % h["prim"]
            c, r = bounds[it, :3], bounds[it, 3]
            if r < 0:
                continue  # unbounded: never culled
            oc = c - o[k]
            b = float(oc @ du)
            dist2 = float(oc @ oc) - b * b
            assert dist2 <= r * r * (1 + 1e-9) + 1e-12, (seed, k, h["prim"], "line misses the bound by %g" % (np.sqrt(max(dist2, 0)) - r))
            assert b >= 0 or float(oc @ oc) <= r * r * (1 + 1e-9), (seed, k, h["prim"], "bound behind the origin but t = %g" % h["t"])
            p = o[k] + h["t"] * d[k]
            assert np.linalg.norm(p - c) <= r * (1 + 1e-9) + 1e-9, (seed, k, h["prim"], "hit point outside the bound")
            checked += 1
    print("seed %d: %d items, %d crossings checked" % (seed, bounds.shape[0], checked))


@pytest.mark.parametrize("name", ["cfg1-sample", "cfg2-hollow-sphere", "cfg3-house", "cfg3-night-house", "cfg4-bunny-d12", "cfg5-repeat", "cfg5-moon"])
def test_bundled_scenes_crossings_lie_inside_their_items_bounds(probe, name):
    """The same check on the BASELINE scenes, with rays from around the camera and from points on the ground towards the lights'
    side of the scene (the two kinds of rays the kernel's common-origin table serves)."""
    import numpy as np
    from oracle import ftb_oracle as orc
    sc = frontend.ParsedScene(scenes.config_text(name, res=(64, 48), spp=1), scenes.asset_dir())
    bounds, prim_item = _item_bounds(probe, sc)
    rng = np.random.default_rng(7)
    cam = np.array([sc.camera.o[0], sc.camera.o[1], sc.camera.o[2]])
    look = np.array([sc.camera.look_at[0], sc.camera.look_at[1], sc.camera.look_at[2]])
    n = 300
    fwd = (look - cam) / np.linalg.norm(look - cam)
    o = np.vstack([cam + rng.normal(scale=0.05, size=(n, 3)), rng.uniform([-20, 0.01, -5], [20, 6, 60], size=(n, 3))])
    d = np.vstack([fwd + rng.normal(scale=0.35, size=(n, 3)), rng.normal(size=(n, 3)) + np.array([0.0, 0.6, 0.0])])
    checked = 0
    for k in range(o.shape[0]):
        du = d[k] / np.linalg.norm(d[k])
        for h in orc.node_hits(sc, o[k], d[k], max_hits=4096):
            if not (h["t"] >= 0.0) or not np.isfinite(h["t"]):
                continue
            it = prim_item[h["prim"]]
            assert it >= 0
            c, r = bounds[it, :3], bounds[it, 3]
            if r < 0:
                continue
            oc = c - o[k]
            b = float(oc @ du)
            assert float(oc @ oc) - b * b <= r * r * (1 + 1e-9) + 1e-12, (name, k, h["prim"])
            assert b >= 0 or float(oc @ oc) <= r * r * (1 + 1e-9), (name, k, h["prim"], h["t"])
            checked += 1
    print("%s: %d items, %d crossings checked" % (name, bounds.shape[0], checked))
    assert checked > 0 or name == "cfg1-sample"


@pytest.mark.parametrize("name,kw", [("cfg4-bunny", {}), ("cfg4-bunny-d12", {}), ("cfg4-bunny", dict(depth=3, mesh="bunny_tiny.ply")),
                                     ("cfg4-bunny", dict(depth=4, mesh="bunny_res4.ply"))])
def test_host_mesh_index_invariants(probe, name, kw):
    """The host build of the device's mesh index (lower.cpp buildMeshIndexHost): every clipped triangle in exactly one leaf, boxes
    that contain their subtrees in both precisions, leaves within the slot-count encoding, a depth the 64-entry traversal stack
    can hold, and `seq` = the triangle's rank in BspMesh.intersect's right-before-left enumeration (BspMesh.fs:67-76) - the
    tie-break that makes the BVH's answer the reference's."""
    sc = frontend.ParsedScene(scenes.config_text(name, res=(32, 24), spp=1, **kw), scenes.asset_dir())
    depth = C.c_int(0)
    n = probe.ftb_probe_mesh_index(sc.desc_ptr, C.byref(depth))
    print("%s %s: %d triangle slots, index depth %d" % (name, kw, n, depth.value))
    assert n > 0, "violation %d" % n
    assert depth.value + 2 <= 64  # api.cu refuses deeper indices (kBspStack)
