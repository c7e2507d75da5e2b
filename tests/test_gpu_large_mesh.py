"""The large-mesh path against the CPU oracle.  Needs a B200: run with `-m gpu`.

Scenes whose bspMesh primitives hold 32 768 triangles or more in all (api.cu kLargeMesh) get a mesh index built on the device
(bvh_build.cu, PLOC) and have their meshes walked by the whole warp after each lane's other candidates of a batch of 32
items (render.cuh packetMesh, meshHit).  Every case here renders such a scene in both precisions and compares it with the
oracle: colour (FP64 within 1e-6, FP32 within 1/255, on >= 99.9 % of pixels or rays) and the primary primitive-id and sub-id
planes, mismatches classified by oracle/parity.py.  Scene.build_info() is asserted, so that a case which fell back to the
host build or to the small-mesh path does not pass as coverage.  The meshes are generated (tests/large_mesh_scenes.py)."""
import numpy as np
import pytest

import large_mesh_scenes as lms
from functracer_b200 import abi, api, frontend
from oracle import ftb_oracle as orc
from oracle import parity
from util import parse

pytestmark = pytest.mark.gpu

RNG_SEED = 1234
FP64, FP32 = abi.PRECISION_FP64_VERIFY, abi.PRECISION_FP32


def _colour_ok(got, ref, precision):
    d = np.abs(np.asarray(got, dtype=np.float64) - ref).max(axis=-1)
    return float((d <= (1e-6 if precision == FP64 else 1.0 / 255.0)).mean()), float(d.max())


def interior_rays(tris, rng, per_tri, spread=0.3):
    """per_tri rays at points well inside each triangle (barycentric weights >= 0.15), each from 12 units in front of its
    point along -z (and up to about `spread` aside): steep enough that no other cell of a field lies in the way."""
    w = rng.uniform(0.15, 1.0, size=(len(tris), per_tri, 3))
    w /= w.sum(axis=-1, keepdims=True)
    target = np.einsum("tkv,tvc->tkc", w, tris).reshape(-1, 3)
    o = target + np.column_stack([rng.normal(size=(len(target), 2)) * spread, np.full(len(target), -12.0)])
    return np.concatenate([o, target - o], axis=1)


def check_rays(sc, rays, expect_device, exact_ids=False, id_frac=(1e-3, 5e-3)):
    """Scene.shade against orc.shade_rays in both precisions.  Returns the oracle's result."""
    ref = orc.shade_rays(sc, rays, orc.make_params(1, 1, 1, [0.0, 0.0], seed=RNG_SEED))
    with api.Scene(sc) as scene:
        info = scene.build_info()
        print("build: %s" % info)
        if expect_device is not None:
            assert info["bvh_on_device"] == expect_device
        for precision, frac in zip((FP64, FP32), id_frac):
            got = scene.shade(rays, seed=RNG_SEED, precision=precision)
            within, worst = _colour_ok(got["rgb"], ref["rgb"], precision)
            mism = got["prim"] != ref["prim"]
            sub_mism = (~mism) & (got["sub"] != ref["sub"])
            print("precision %d: %d rays, colour within bar %.5f (max %.3g), prim mismatches %d, sub mismatches %d"
                  % (precision, len(rays), within, worst, int(mism.sum()), int(sub_mism.sum())))
            assert within >= 0.999
            if exact_ids:
                assert not mism.any(), list(zip(got["prim"][mism][:8], ref["prim"][mism][:8]))
                assert not sub_mism.any()
            else:
                assert mism.mean() <= frac
                assert sub_mism.mean() <= frac
    return ref


def check_frame(sc, expect_device, sub_frac=(1e-3, 5e-3), name=""):
    """A whole frame in both precisions against the oracle (jittered samples).  Returns (oracle result, {precision: render})."""
    W, H, spp = sc.width, sc.height, sc.spp
    jit = frontend.jitter_pattern(1, spp)
    ref = orc.render(sc, orc.make_params(W, H, spp, jit, seed=RNG_SEED))
    rp, rs = ref["prim"].reshape(H, W, spp), ref["sub"].reshape(H, W, spp)
    assert (rp >= 0).mean() > 0.2  # the frame sees the meshes
    out = {}
    with api.Scene(sc) as scene:
        info = scene.build_info()
        print("%s build: %s" % (name, info))
        if expect_device is not None:
            assert info["bvh_on_device"] == expect_device
        for precision, sf in zip((FP64, FP32), sub_frac):
            got = scene.render(W, H, spp, jit, seed=RNG_SEED, precision=precision, debug=True)
            out[precision] = got
            within, worst = _colour_ok(got["rgb"], ref["rgb"], precision)
            c = parity.compare_window(ref["rgb"], rp, got["rgb"], got["prim"].reshape(H, W, spp), ref_sub=rs, got_sub=got["sub"].reshape(H, W, spp))
            print("%s precision %d: colour within bar %.5f (max %.3g); prim mismatches %d of %d (edge leaks %d, unexplained %d), sub mismatches %d"
                  % (name, precision, within, worst, c["prim_mismatch"], c["samples"], c["prim_edge_leak"], c["prim_unexplained"], c["sub_mismatch"]))
            assert within >= 0.999
            assert c["prim_unexplained"] == 0, c.get("unexplained_samples")
            assert c["prim_mismatch"] <= (1e-3 if precision == FP64 else 5e-3) * c["samples"]
            if precision == FP64:
                assert c["prim_edge_leak"] == 0
            assert c["sub_mismatch"] <= sf * c["samples"]
    return ref, out


# ---- the tie ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("soft", [False, True], ids=["0x804", "0xfff"])
@pytest.mark.parametrize("n", [lms.LARGE_MESH - 1, lms.LARGE_MESH])
def test_mesh_wins_a_tie_against_a_later_item_of_its_batch(tmp_path, n, soft):
    """Scene.closest (and the oracle) give a tie in t to the item that comes first.  A bspMesh followed by triangle items that
    are exact copies of some of its triangles (dyadic coordinates: the same doubles, the same {v0, e1, e2} rows) ties on every
    ray through those triangles: the mesh must win.  In the other order the copies must win, so together the two orders show
    that the ties are exact in both builds.  At 32 767 triangles the mesh takes the host tree and the per-lane walk, at 32 768
    the device tree and the warp's walk (FP32: kernel 0x804 with hard lights only, 0xfff with a soft light)."""
    for mesh_first in (True, False):
        text, d, dup = lms.tie(str(tmp_path), n, mesh_first, soft)
        sc = parse(text, assets=d)
        rays = interior_rays(dup, np.random.default_rng(3), 16)
        ref = check_rays(sc, rays, n >= lms.LARGE_MESH, exact_ids=True)
        ids = np.unique(ref["prim"])
        assert ids.size == (1 if mesh_first else len(dup)), ids  # every ray hits the earlier item: the mesh, or each copy
        if mesh_first:
            assert np.unique(ref["sub"]).size == len(dup)  # at the duplicated triangles


def test_the_earlier_of_two_instances_of_a_mesh_wins(tmp_path):
    """The same mesh twice under one transform: every hit ties, the first instance wins."""
    text, d = lms.twin_instances(str(tmp_path))
    sc = parse(text, assets=d)
    v, f = lms.field(128, 64)
    tris = v[np.array(f)][np.random.default_rng(5).choice(len(f), 256, replace=False)] + np.array([0.0, 4.0, 0.0])
    ref = check_rays(sc, interior_rays(tris, np.random.default_rng(6), 4), True, exact_ids=True)
    assert np.unique(ref["prim"]).size == 1


# ---- several meshes in one scene: the offsets and root-leaf links of the device build, toModel before the packet walk --
@pytest.mark.parametrize("family", ["two_large_and_small", "many_small_meshes", "transformed_instances"])
def test_several_meshes_in_one_scene(tmp_path, family):
    text, d = getattr(lms, family)(str(tmp_path))
    check_frame(parse(text, assets=d), True, name=family)


# ---- geometry that stresses the device build and the slab test ------------------------------------------------------
def test_planar_grid_with_axis_parallel_rays(tmp_path):
    """Zero extent in z: the camera looks straight along z, and explicit rays run along each axis, in the mesh's plane too."""
    text, d = lms.planar_grid(str(tmp_path))
    sc = parse(text, assets=d)
    check_frame(sc, True, name="planar")
    rng = np.random.default_rng(9)
    n = 512
    xy = rng.uniform(-1.0, 17.0, size=(n, 2))
    rays = []
    for sign in (1.0, -1.0):  # along z, from either side
        rays.append(np.column_stack([xy, np.full(n, -5.0 * sign), np.zeros(n), np.zeros(n), np.full(n, sign)]))
    for z in (0.0, 1.0 / 1024, -1.0 / 1024):  # along x and y, in and next to the plane
        rays.append(np.column_stack([np.full(n, -2.0), xy[:, 1], np.full(n, z), np.ones(n), np.zeros(n), np.zeros(n)]))
        rays.append(np.column_stack([xy[:, 0], np.full(n, 18.0), np.full(n, z), np.zeros(n), -np.ones(n), np.zeros(n)]))
    rays = np.concatenate(rays)
    ref = check_rays(sc, rays, True)
    assert (ref["prim"][:2 * n] >= 0).mean() > 0.3  # the rays along z do hit the grid


@pytest.mark.parametrize("family", ["fan", "slivers", "coincident"])
def test_degenerate_clusters(tmp_path, family):
    """fan: 2 048 triangles with one centroid and one box centre (one Morton key); slivers: triangles that span a mesh of tiny
    ones; coincident: 5 000 copies of one triangle, whose boxes tie in every clustering round (PLOC merges one pair per round
    there and may give up after 4 096 rounds: the host tree is then used, which is also right - the test prints which)."""
    text, d = getattr(lms, family)(str(tmp_path))
    check_frame(parse(text, assets=d), None if family == "coincident" else True, name=family)


# ---- incoherent and secondary rays in one warp ----------------------------------------------------------------------
def test_incoherent_rays_inside_and_around_a_closed_mesh(tmp_path):
    """Random origins (in and around the blob's box, and inside the closed blob) and random directions: the warp's walk then
    mixes nearest-hit and shadow (any-hit) lanes whose rays share no path.  Reflective surfaces add secondary rays."""
    text, d = lms.shiny_blob(str(tmp_path))
    sc = parse(text, assets=d)
    rng = np.random.default_rng(21)
    n = 4096
    box_lo, box_hi = lms.BLOB_CENTRE - 4.0, lms.BLOB_CENTRE + 4.0
    o = np.concatenate([rng.uniform(box_lo, box_hi, size=(n, 3)), lms.BLOB_CENTRE + rng.normal(size=(n // 4, 3)) * 0.2])
    dirs = rng.normal(size=o.shape)
    # length 100: Moller-Trumbore's determinant threshold is absolute, and the blob's model-space triangles are small enough
    # that short directions would be rejected by it (in the reference too) rather than tested by the walk
    dirs *= 100.0 / np.linalg.norm(dirs, axis=1, keepdims=True)
    ref = check_rays(sc, np.concatenate([o, dirs], axis=1), True)
    inside = ref["prim"][n:]
    print("rays from inside the blob that hit something: %.4f" % (inside >= 0).mean())
    assert (inside >= 0).mean() > 0.99  # the origins are inside the closed mesh


def test_reflections_and_shadows_frame(tmp_path):
    """Reflection depth 8, point, directional and soft directional lights, a blob whose parts shadow each other."""
    text, d = lms.shiny_blob(str(tmp_path))
    check_frame(parse(text, assets=d), True, name="shiny_blob")


# ---- walk and tree do not change the picture (DESIGN.md section 3) ---------------------------------------------------
def test_walk_and_tree_do_not_change_the_picture(tmp_path):
    """A 32 767-triangle mesh (host tree, per-lane walk) and the same scene with one more mesh of a single zero-area triangle
    (device tree, warp-packet walk): FP64 frames and planes bit-identical.  FP32 runs different kernels (0x004, 0x804 are
    not compiled alike), so there each is compared with the oracle only."""
    frames = []
    for extra in (False, True):
        d = tmp_path / ("extra" if extra else "alone")
        d.mkdir()
        text, dd = lms.just_below_threshold(str(d), extra)
        _, out = check_frame(parse(text, assets=dd), extra, name="extra" if extra else "alone")
        frames.append(out[FP64])
    a, b = frames
    for k in ("rgb", "prim", "sub", "t"):
        assert np.array_equal(a[k], b[k]), k
