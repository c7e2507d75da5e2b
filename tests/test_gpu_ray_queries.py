"""Ray queries (ftb_intersect_rays, ftb_occluded_rays and their device forms) against the CPU oracle and against the renderer.
Needs a B200: run with `-m gpu`.

The oracle's answer to a nearest query is Scene.closest on the root's hit list (the first minimal t >= 0 of oracle.node_hits),
to an occlusion query Scene.lightIsBocked on the same list; tests/query_oracle.py answers whole batches of rays that way.
Scenes: the bundled builders at small size, one scene per kernel variant (tests/variant_scenes.py), a handful of
test_gpu_fuzz seeds and two large-mesh scenes (warp-packet walk).  Rays: the camera's (a full grid, classified by
oracle/parity.py), random rays from points in and around the scene's box, rays leaving the camera rays' hit points (offset by
1e-4 n), axis-aligned rays and directions scaled by 1e-3 .. 1e3.

Bars (every count is printed):
  - ids: camera rays have no unexplained primary-id mismatch (parity.compare_window); on the other rays, whose neighbours
    cannot be asked, at most 1e-3 (FP64) / 5e-3 (FP32) of the rays may differ, as tests/test_gpu_large_mesh.py allows.  Not
    counted: ties at t = 0, where a ray parallel to a plane, square or cube face meets it at its origin (Plane.fs:14-16) and
    several such crossings tie (axis-aligned rays; printed as t0_ties).
  - where prim and sub agree, on >= 99.9 % of the rays: t within 1e-9 relative (FP64), in FP32 t |d| within T_REL_BAR of the
    ray's scale |o| + t |d| + 1 (the FP32 origin alone is off by 6e-8 |o|, which a short t cannot absorb; t and p are held to
    >= 99 % in FP32: a grazing hit multiplies that error by 1 / sin of the angle between ray and surface); p within 1e-9
    (FP64) / 1e-4 (FP32) of that scale (in FP32 p = o + t d is as good as t, and a hit on a planar leaf is moved back onto its
    plane by up to |p| * 6e-8; a parallel hit at t = 0, whose p is the origin, is moved all the way); the normal within 1e-9 / 2e-3 (an FP32 normal is computed from the FP32
    model-space hit point, so it carries t's error over the primitive's size); colour and surface within 1e-9 / 1e-5 (FP32
    narrows the material and texel values to float).  Colour is held to >= 99.5 % in FP32: a u, v off by FP32 rounding at a
    texel or grid-cell boundary reads the neighbouring texel."""
import zlib

import numpy as np
import pytest

import large_mesh_scenes as lms
import query_oracle as qo
import variant_scenes as vs
from functracer_b200 import abi, api, scenes
from oracle import ftb_oracle as orc
from oracle import parity
from test_gpu_fuzz import _scene as fuzz_scene
from util import one_object_scene, parse

pytestmark = pytest.mark.gpu

FP32, FP64 = abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY
PRECISIONS = (FP64, FP32)
T_REL_BAR = 5e-5  # tests/test_gpu_variants.py
GRID = (48, 36)
ID_FRAC = {FP64: 1e-3, FP32: 5e-3}
BARS = {FP64: dict(t=1e-9, p=1e-9, normal=1e-9, colour=1e-9, surface=1e-9),
        FP32: dict(t=T_REL_BAR, p=1e-4, normal=2e-3, colour=1e-5, surface=1e-5)}
COVER = {FP64: dict(t=0.999, p=0.999, normal=0.999, colour=0.999, surface=0.999),
         FP32: dict(t=0.99, p=0.99, normal=0.999, colour=0.995, surface=0.999)}

VSCENES = {s.name: s for s in vs.all_scenes()}
# one scene per FP32 kernel variant (tests/test_variant_cover_cpu.py pins where they land)
VARIANT_SCENES = {0x000: "spheres0", 0x100: "plane10", 0x209: "cubes33", 0x74b: "runs1_soft2", 0x3c3: "nested1_soft1", 0x050: "dof0",
                  0x030: "rough10", 0x004: "meshes0", 0x804: "large_meshes"}
FUZZ_SEEDS = [0, 5, 17, 42, 77, 123]


def _bundled(name):
    return lambda d: parse(getattr(scenes, name)(res=GRID, spp=1))


def _variant(name):
    def make(d):
        text, assets = VSCENES[name].text(d)
        return parse(text, assets=assets)
    return make


def _fuzz(seed):
    return lambda d: parse(fuzz_scene(1000 + seed))


def _large(family):
    def make(d):
        text, assets = getattr(lms, family)(d)
        return parse(text, assets=assets)
    return make


CASES = {"bundled_" + n: _bundled(n) for n in ("sample", "hollow_sphere", "house", "night_house", "repeat", "moon", "bunny")}
CASES.update({"variant_0x%03x" % v: _variant(n) for v, n in VARIANT_SCENES.items()})
CASES.update({"fuzz_%d" % s: _fuzz(s) for s in FUZZ_SEEDS})
CASES.update({"large_" + f: _large(f) for f in ("shiny_blob", "two_large_and_small")})


def _open(sc):
    """api.Scene, or a skip for a fuzz scene the device path documents as unsupported."""
    try:
        return api.Scene(sc)
    except api.FtbError as e:
        assert e.status == abi.ERR_UNSUPPORTED
        pytest.skip("unsupported by the device path: %s" % e)


def camera_rays(sc, W, H):
    return np.array([orc.primary_ray(sc.camera, W, H, x, y) for y in range(H) for x in range(W)])


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def ray_sets(sc, rng, n=600):
    """{name: rays [m, 6]}: camera grid, random rays in and around the box of what the camera sees, rays leaving its hit points,
    axis-aligned rays, directions scaled by 1e-3 .. 1e3."""
    cam = camera_rays(sc, *GRID)
    ref = qo.nearest(sc, cam)
    hit = ref["prim"] >= 0
    pts = ref["p"][hit] if hit.any() else np.zeros((1, 3))
    lo, hi = np.percentile(pts, 2, axis=0), np.percentile(pts, 98, axis=0)
    pad = 0.2 * (hi - lo) + 0.5
    lo, hi = lo - pad, hi + pad
    o = rng.uniform(lo, hi, size=(n, 3))
    out = dict(camera=cam, random=np.hstack([o, _unit(rng.normal(size=(n, 3)))]))
    if hit.any():
        k = rng.integers(0, len(pts), size=n)
        nrm = ref["normal"][hit][k]
        d = _unit(rng.normal(size=(n, 3)))
        d = np.where((np.sum(d * nrm, axis=1) < 0)[:, None], -d, d)  # leaving the surface
        out["surface"] = np.hstack([pts[k] + 1e-4 * nrm, d])
    axes = np.eye(3)[rng.integers(0, 3, size=n)] * rng.choice([-1.0, 1.0], size=(n, 1))
    out["axis"] = np.hstack([rng.uniform(lo, hi, size=(n, 3)), axes])
    out["scaled"] = np.hstack([rng.uniform(lo, hi, size=(n, 3)), _unit(rng.normal(size=(n, 3))) * 10.0 ** rng.uniform(-3, 3, size=(n, 1))])
    return out


def compare_nearest(got, ref, rays, precision, label, grid=None):
    """Asserts the bars of the module docstring; returns the counts."""
    # Plane.fs:14-16: a ray parallel to a plane (|d.n| < 1e-7) on its front side meets it at t = 0, at the origin.  Axis rays
    # parallel to cube faces, squares and ground planes collect several such crossings at t = 0; which one comes first is a tie
    # decided by the 1e-7 tests in each implementation's own model space.
    zero = (ref["t"] == 0) | (got["t"] == 0)
    mism = got["prim"] != ref["prim"]
    same = ~mism & (ref["prim"] >= 0) & (got["sub"] == ref["sub"])
    sub_mism = ~mism & (got["sub"] != ref["sub"])
    res = dict(rays=len(rays), prim_mismatch=int(mism.sum()), sub_mismatch=int(sub_mism.sum()), t0_ties=int(((mism | sub_mism) & zero).sum()))
    mism, sub_mism = mism & ~zero, sub_mism & ~zero
    if grid is not None:
        W, H = grid
        z = np.zeros((H, W, 3))
        c = parity.compare_window(z, ref["prim"].reshape(H, W, 1), z, got["prim"].reshape(H, W, 1), ref_sub=ref["sub"].reshape(H, W, 1),
                                  got_sub=got["sub"].reshape(H, W, 1))
        res["prim_unexplained"] = c["prim_unexplained"]
        res["prim_edge_leak"] = c["prim_edge_leak"]
        assert c["prim_unexplained"] == 0, (label, c.get("unexplained_samples"))
    else:
        assert mism.mean() <= ID_FRAC[precision], (label, res)
    assert sub_mism.mean() <= ID_FRAC[precision], (label, res)
    miss = got["prim"] < 0
    assert (got["t"][miss] == -1).all() and (got["sub"][miss] == 0).all()
    for k in ("p", "normal", "colour", "surface"):
        assert (got[k][miss] == 0).all(), k
    if same.any():
        scale = np.linalg.norm(rays[same, :3], axis=1) + np.abs(ref["t"][same]) * np.linalg.norm(rays[same, 3:], axis=1) + 1.0
        dt = np.abs(got["t"][same] - ref["t"][same])
        perr = np.abs(got["p"][same] - ref["p"][same]).max(axis=1) / scale
        if precision == FP32:
            perr[ref["t"][same] == 0] = 0.0  # the parallel hit's p = o, which the FP32 fragment projects onto the plane
        errs = dict(t=dt / np.maximum(np.abs(ref["t"][same]), 1e-30) if precision == FP64 else dt * np.linalg.norm(rays[same, 3:], axis=1) / scale,
                    p=perr,
                    normal=np.abs(got["normal"][same] - ref["normal"][same]).max(axis=1),
                    colour=np.abs(got["colour"][same] - ref["colour"][same]).max(axis=1),
                    surface=np.abs(got["surface"][same] - ref["surface"][same]).max(axis=1) / np.maximum(np.abs(ref["surface"][same]).max(axis=1), 1.0))
        for k, e in errs.items():
            frac = float((e <= BARS[precision][k]).mean())
            res["%s_within" % k], res["%s_max" % k] = frac, float(e.max())
            assert frac >= COVER[precision][k], (label, k, frac, float(e.max()))
        assert np.array_equal(got["surface"][same, 3], ref["surface"][same, 3])  # apply_lighting is exact
    return res


# ---- 1. nearest against the oracle; 2. the same answer as the renderer -------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_nearest_against_the_oracle_and_the_renderer(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    sets = ray_sets(sc, np.random.default_rng(zlib.crc32(case.encode())))
    refs = {k: qo.nearest(sc, r) for k, r in sets.items()}
    with _open(sc) as scene:
        for precision in PRECISIONS:
            for k, rays in sets.items():
                try:
                    got = scene.intersect(rays, precision=precision)
                except api.FtbError as e:
                    assert e.status == abi.ERR_HIT_OVERFLOW and case.startswith("fuzz")
                    pytest.skip("hit-stack overflow reported: %s" % e)
                res = compare_nearest(got, refs[k], rays, precision, (case, k, precision), grid=GRID if k == "camera" else None)
                print("%s %s precision %d: %s" % (case, k, precision, res))
            # the renderer's primary trace is traceScene from o + 1e-4 d (slightOffset): a query of that ray is the same trace
            rays = sets["camera"]
            off = np.hstack([rays[:, :3] + 1e-4 * rays[:, 3:], rays[:, 3:]])
            q = scene.intersect(off, planes=("t", "prim", "sub"), precision=precision)
            try:
                s = scene.shade(rays, precision=precision)
            except api.FtbError as e:  # a bounce or shadow ray of the shader overflowed (fuzz scenes with deep CSG)
                assert e.status == abi.ERR_HIT_OVERFLOW and case.startswith("fuzz")
                print("%s: the renderer reports a hit-stack overflow; no comparison" % case)
                continue
            if precision == FP64:
                for k in ("t", "prim", "sub"):
                    assert np.array_equal(q[k], s[k]), (case, k)
            else:  # the FP32 kernel rounds o + 1e-4 d itself; the query's origin is that sum rounded in double, then narrowed
                W, H = GRID
                z = np.zeros((H, W, 3))
                c = parity.compare_window(z, s["prim"].reshape(H, W, 1), z, q["prim"].reshape(H, W, 1), ref_sub=s["sub"].reshape(H, W, 1),
                                          got_sub=q["sub"].reshape(H, W, 1))
                print("%s renderer vs query FP32: %d of %d primary ids differ (unexplained %d, edge leaks %d), %d sub-ids"
                      % (case, c["prim_mismatch"], c["samples"], c["prim_unexplained"], c["prim_edge_leak"], c["sub_mismatch"]))
                assert c["prim_unexplained"] == 0, (case, c.get("unexplained_samples"))


# ---- 3. occlusion against lightIsBocked from the same hit lists ---------------------------------------------------------
def _occlusion_cases(sc, rng, sets):
    """{name: (rays, max_t)}."""
    rays = np.concatenate([sets["random"], sets["scaled"], sets["axis"]] + ([sets["surface"]] if "surface" in sets else []))
    ts, lit, cnt = qo.hits(sc, rays)
    far = np.maximum(np.where(ts >= 0, ts, 0.0).max(axis=1), 1.0)  # the last crossing ahead (NaN pads compare false)
    out = {"inf": (rays, np.full(len(rays), np.inf)), "random": (rays, rng.uniform(0, 1, len(rays)) * far)}
    # shadow rays from the camera rays' hit points towards every light, as Shading.fs:33-48 builds them
    ref = qo.nearest(sc, sets["camera"])
    hit = ref["prim"] >= 0
    P = ref["p"][hit] + 1e-4 * ref["normal"][hit]
    d = sc.desc
    sr, sm = [], []
    for i in range(d.n_lights):
        L = d.lights[i]
        v = np.array(L.v[:])
        if L.kind == abi.LIGHT_POINT:
            dv = v - P
            sr.append(np.hstack([P, _unit(dv)]))
            sm.append(np.linalg.norm(dv, axis=1))
        else:
            sr.append(np.hstack([P, np.tile(-v, (len(P), 1))]))
            sm.append(np.full(len(P), np.finfo(np.float64).max))
    if sr:
        out["shadow"] = (np.concatenate(sr), np.concatenate(sm))
    return out


def _next_up(t, precision):
    """The next number above t in the kernel's working precision, as a double (FP32 t is a float widened to double)."""
    if precision == FP64:
        return np.nextafter(t, np.inf)
    return np.nextafter(t.astype(np.float32), np.float32(np.inf)).astype(np.float64)


@pytest.mark.parametrize("case", sorted(CASES))
def test_occlusion_is_strict_at_the_nearest_hit(case, tmp_path):
    """max_t equal to a ray's nearest hit, taken from the device's own answer: the crossing at max_t does not block (0 <= t <
    max_t, Scene.fs:121) and nothing lies before it; with the next number above it as max_t, the same crossing blocks.  Rays
    whose nearest surface has applyLighting and t > 0 (a hit at t = 0 leaves no number below it to test)."""
    sc = CASES[case](str(tmp_path))
    rays = np.concatenate(list(ray_sets(sc, np.random.default_rng(zlib.crc32(case.encode()) + 2), n=400).values()))
    with _open(sc) as scene:
        for precision in PRECISIONS:
            try:
                near = scene.intersect(rays, planes=("t", "surface"), precision=precision)
            except api.FtbError as e:
                assert e.status == abi.ERR_HIT_OVERFLOW and case.startswith("fuzz")
                pytest.skip("hit-stack overflow reported: %s" % e)
            sel = (near["t"] > np.finfo(np.float32).tiny) & (near["surface"][:, 3] == 1)
            r, t = rays[sel], near["t"][sel]
            at = scene.occluded(r, t, precision=precision)
            above = scene.occluded(r, _next_up(t, precision), precision=precision)
            print("%s precision %d: %d rays with a lit nearest hit; blocked at max_t = t: %d, at the next number above t: %d"
                  % (case, precision, len(r), int(at.sum()), int(above.sum())))
            assert len(r) >= 20
            assert not at.any() and above.all()


def _tie(sc, rays, max_t, tol):
    """Rays whose answer depends on the last bits of t: a lit crossing within tol (relative) of max_t or of 0."""
    ts, lit, _ = qo.hits(sc, rays)
    near = (lit == 1) & ((np.abs(ts - max_t[:, None]) <= tol * np.maximum(np.abs(max_t[:, None]), 1.0)) | (np.abs(ts) <= tol))
    return near.any(axis=1)


@pytest.mark.parametrize("case", sorted(CASES))
def test_occlusion_against_the_oracle(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    rng = np.random.default_rng(zlib.crc32(case.encode()) + 1)
    cases = _occlusion_cases(sc, rng, ray_sets(sc, rng, n=400))
    with _open(sc) as scene:
        for name, (rays, mt) in cases.items():
            ref = qo.occluded(sc, rays, mt)
            for precision in PRECISIONS:
                try:
                    got = scene.occluded(rays, mt, precision=precision)
                except api.FtbError as e:
                    assert e.status == abi.ERR_HIT_OVERFLOW and case.startswith("fuzz")
                    pytest.skip("hit-stack overflow reported: %s" % e)
                mism = got != ref
                tie = _tie(sc, rays, mt, 1e-9 if precision == FP64 else 1e-4) & mism
                print("%s %s precision %d: %d rays, %d blocked, %d differ (%d at a tie in t)" % (case, name, precision, len(rays), int(ref.sum()),
                                                                                          int(mism.sum()), int(tie.sum())))
                assert (mism & ~tie).mean() <= ID_FRAC[precision], (case, name, precision)


def test_ignore_light_surfaces_do_not_block():
    """A lit sphere behind an ignoreLight one: rays through both are blocked by the lit one only; rays through the ignoreLight
    sphere alone are not blocked, though their nearest hit is that sphere."""
    sc = parse(one_object_scene("(group (ignoreLight (translate (0,0,-2) (scale 0.5 sphere))) (translate (0,0,2) (scale 0.5 sphere)))",
                                "directional dir (0,0,1) colour (1,1,1)"))
    both = np.array([[0.0, y, -6.0, 0.0, 0.0, 1.0] for y in np.linspace(-0.3, 0.3, 31)])
    # tilted: through the ignoreLight sphere at z = -2, then above the lit one at z = 2 (the oracle picks the rays that do so)
    only = np.array([[0.0, y - 0.6, -6.0, 0.0, 0.15, 1.0] for y in np.linspace(-0.45, 0.45, 61)])
    only = only[(qo.nearest(sc, only)["prim"] == 0) & ~qo.occluded(sc, only, np.inf)]
    assert len(only) > 5 and qo.occluded(sc, both, np.inf).all() and not qo.occluded(sc, both, 6.0).any()
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            assert scene.occluded(both, np.inf, precision=precision).all()
            assert not scene.occluded(both, 6.0, precision=precision).any()  # before t = 6 lies only the ignoreLight sphere
            assert not scene.occluded(only, np.inf, precision=precision).any()
            assert (scene.intersect(only, planes=("prim",), precision=precision)["prim"] == 0).all()


# ---- 4. planes ------------------------------------------------------------------------------------------------------------
def test_each_plane_alone_equals_the_full_request(tmp_path):
    for make in (_bundled("sample"), _variant("runs1_soft2"), _variant("meshes0")):
        sc = make(str(tmp_path))
        rays = np.concatenate(list(ray_sets(sc, np.random.default_rng(4), n=300).values()))
        with api.Scene(sc) as scene:
            for precision in PRECISIONS:
                full = scene.intersect(rays, precision=precision)
                for k in api.HIT_PLANES:
                    alone = scene.intersect(rays, planes=(k,), precision=precision)
                    assert set(alone) == {k} and np.array_equal(alone[k], full[k]), k
                miss = full["prim"] < 0
                assert 0.02 < 1.0 - miss.mean() < 0.98  # hits and misses
                assert (full["t"][miss] == -1).all() and (full["sub"][miss] == 0).all()
                for k in ("p", "normal", "colour", "surface"):
                    assert (full[k][miss] == 0).all(), k


def _torch():
    import torch
    return torch


def test_planes_not_requested_stay_untouched(tmp_path):
    torch = _torch()
    sc = _bundled("house")(str(tmp_path))
    rays = np.concatenate(list(ray_sets(sc, np.random.default_rng(8), n=300).values()))
    n = len(rays)
    widths = dict(t=1, prim=1, sub=1, p=3, normal=3, colour=3, surface=4)
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            host = scene.intersect(rays, precision=precision)
            for want in (("t",), ("prim", "p"), ("sub", "colour", "surface"), ("normal",)):
                d_rays = torch.from_numpy(rays).cuda()
                bufs = {k: torch.full((n, w), -7, dtype=torch.int32 if k in ("prim", "sub") else torch.float64, device="cuda") for k, w in widths.items()}
                scene.intersect_device(d_rays.data_ptr(), n, {k: bufs[k].data_ptr() for k in want}, precision=precision)
                torch.cuda.synchronize()
                for k, b in bufs.items():
                    b = b.cpu().numpy().reshape(host[k].shape)
                    if k in want:
                        assert np.array_equal(b, host[k]), k
                    else:
                        assert (b == -7).all(), k


# ---- 5. device entries ----------------------------------------------------------------------------------------------------
def test_device_entries_on_a_side_stream_equal_the_host_entries(tmp_path):
    torch = _torch()
    for make in (_variant("cubes33"), _large("shiny_blob")):
        sc = make(str(tmp_path))
        sets = ray_sets(sc, np.random.default_rng(11), n=500)
        rays = np.concatenate(list(sets.values()))
        mt = np.random.default_rng(12).uniform(0, 20, len(rays))
        n = len(rays)
        with api.Scene(sc) as scene:
            side = torch.cuda.Stream()
            for precision in PRECISIONS:
                host = scene.intersect(rays, precision=precision)
                hb = scene.occluded(rays, mt, precision=precision)
                with torch.cuda.stream(side):
                    d_rays, d_mt = torch.from_numpy(rays).cuda(), torch.from_numpy(mt).cuda()
                    out = {k: torch.empty(v.shape, dtype=torch.int32 if v.dtype == np.int32 else torch.float64, device="cuda") for k, v in host.items()}
                    blocked = torch.full((n,), -1, dtype=torch.int32, device="cuda")
                    scene.intersect_device(d_rays.data_ptr(), n, {k: v.data_ptr() for k, v in out.items()}, stream=side.cuda_stream, precision=precision)
                    scene.occluded_device(d_rays.data_ptr(), d_mt.data_ptr(), n, blocked.data_ptr(), stream=side.cuda_stream, precision=precision)
                side.synchronize()
                scene.check_overflow(side.cuda_stream)
                for k, v in out.items():
                    assert np.array_equal(v.cpu().numpy(), host[k]), k
                assert np.array_equal(blocked.cpu().numpy() != 0, hb) and set(np.unique(blocked.cpu().numpy())) <= {0, 1}


# ---- 6. overflow ------------------------------------------------------------------------------------------------------------
def test_hit_stack_overflow_is_reported():
    torch = _torch()
    sc = parse(vs.csg_limit(17, True).text(".")[0])
    o = np.array(sc.camera.o[:])
    rays = np.array([np.concatenate([o, np.array([0.0, 0.0, 8.0]) - o])] * 40)
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            with pytest.raises(api.FtbError) as e:
                scene.intersect(rays, precision=precision)
            assert e.value.status == abi.ERR_HIT_OVERFLOW
            d_rays = torch.from_numpy(rays).cuda()
            t = torch.empty(len(rays), dtype=torch.float64, device="cuda")
            scene.intersect_device(d_rays.data_ptr(), len(rays), {"t": t.data_ptr()}, precision=precision)  # does not synchronise
            with pytest.raises(api.FtbError) as e:
                scene.check_overflow()
            assert e.value.status == abi.ERR_HIT_OVERFLOW
            scene.check_overflow()  # the flag was cleared


# ---- 7. batch size, repeats, stats ------------------------------------------------------------------------------------------
def test_a_batch_beyond_2_gib_of_rays_repeats_and_stats(tmp_path):
    sc = _variant("runs1_soft2")(str(tmp_path))
    base = np.concatenate(list(ray_sets(sc, np.random.default_rng(5), n=4000).values()))
    with api.Scene(sc) as scene:
        st = abi.Stats()
        small = scene.intersect(base, planes=("t", "prim", "sub"), stats=st, collect_stats=1)
        assert st.primary_rays == len(base) and st.shadow_rays == 0
        again = scene.intersect(base, planes=("t", "prim", "sub"))
        for k in small:
            assert np.array_equal(small[k], again[k]), k
        st = abi.Stats()
        b1 = scene.occluded(base, np.inf, stats=st, collect_stats=1)
        assert st.shadow_rays == len(base) and st.primary_rays == 0
        assert np.array_equal(b1, scene.occluded(base, np.inf))
        n = 45 * 1000 * 1000  # 45 M rays: 2.16 GB of rays, more than 2^31 bytes
        idx = np.arange(n, dtype=np.int64) % len(base)
        big_rays = base[idx]
        assert big_rays.nbytes > 2 ** 31
        big = scene.intersect(big_rays, planes=("t", "prim", "sub"))
        del big_rays
        pick = np.concatenate([np.random.default_rng(6).integers(0, n, 200000), np.arange(n - 1000, n)])
        for k in small:
            assert np.array_equal(big[k][pick], small[k][idx[pick]]), k
