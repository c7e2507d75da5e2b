"""Path queries (ftb_trace_paths and its device form) against the renderer and the CPU oracle.  Needs a B200: run with `-m gpu`.

Scenes: the bundled builders at small size, one scene per kernel variant (tests/variant_scenes.py), six fuzz seeds and the
reflective large-mesh frame with three kinds of light (tests/large_mesh_scenes.py shiny_blob).  Rays: the camera's, random rays
in and around the scene's box and rays leaving surface points, as tests/test_gpu_ray_queries.py builds them.

  1. FP64 is exact against the renderer: colour is bit-identical to ftb_shade_rays for the same rays, seed and recursion limit
     (0, 1, 8); a float64 replay of the kernel's sum from the planes is bit-identical to colour; level 0's prim, sub and t are
     ftb_shade_rays' debug planes; the counted rays and shaded hits equal ftb_shade_rays' counting kernel's, and so do its leaf and
     bound tests unless the scene has a point light (the frame's common-origin bound table answers some of ftb_shade_rays' bound
     tests for point-light shadow rays; the path query does not use it).
  2. FP64 against the oracle (tests/path_oracle.py): per level, on the rays whose earlier levels agree, the ids agree (level 0 of
     the camera grid classified by oracle/parity.py, elsewhere at most ID_FRAC of the entries may differ); intensities are equal
     where the ids agree for directional and soft lights (a ratio of integers: a difference is a shadow ray that grazes an
     occluder, allowed on at most ID_FRAC of the entries); a point light's intensity is Light.attenuate of the distance to the
     light, a real number that the two implementations round in their own order: blocked (0) exactly where the oracle's is, its
     value within the record bar.  Directions, light colours, weights and the hit records agree to the ray-query tests' FP64
     record bar, 1e-9 of their scale.
  3. FP32 (the generic kernel; ftb_shade_rays may run a specialised one): colour within 1/255 per channel of FP32 ftb_shade_rays
     on >= 99.9 % of the rays; level-0 ids of the camera grid agree with the FP32 debug planes up to parity.py's classification;
     the sum replayed in float64 from the FP32 planes within 1e-5 of colour's scale.
  4. Sample keys reproduce a frame: a window of a scene with soft lights and no depth of field, rendered in FP64, equals the
     literal mean of the path colours of its samples' primary rays with keys (py * gw + px) * spp + s; with the rays' own
     indices as keys the penumbra differs.
  5. Plumbing: each plane alone equals the full request, unrequested planes stay untouched, entries after levels[i] read as a
     miss with weight 0, L = 0 and n = 0 work, recursion_limit 63 works and 64 is refused, the device entry on a side stream is
     bit-identical to the host entry, and a hit-stack overflow returns FTB_ERR_HIT_OVERFLOW with the host arrays unwritten."""
import zlib

import numpy as np
import pytest

import path_oracle as po
import variant_scenes as vs
from functracer_b200 import abi, api, frontend, scenes
from oracle import ftb_oracle as orc
from oracle import parity
from test_gpu_ray_queries import CASES as QUERY_CASES
from test_gpu_ray_queries import GRID, _open, ray_sets
from util import one_object_scene, parse

pytestmark = pytest.mark.gpu

FP32, FP64 = abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY
ID_FRAC = 1e-3
REC_BAR = 1e-9
CASES = {k: v for k, v in QUERY_CASES.items() if k != "large_two_large_and_small"}  # large_shiny_blob: reflective, three kinds of light


def _sets(sc, case):
    s = ray_sets(sc, np.random.default_rng(zlib.crc32(case.encode())), n=400)
    return {k: s[k] for k in ("camera", "random", "surface") if k in s}


def _lights(sc):
    d = sc.desc
    return [d.lights[i].kind for i in range(d.n_lights)]


def _paths(scene, rays, **kw):
    """trace_paths, or None when a fuzz scene's deep CSG overflows the hit stack (reported, as by the other queries)."""
    try:
        return scene.trace_paths(rays, **kw)
    except api.FtbError as e:
        assert e.status == abi.ERR_HIT_OVERFLOW
        return None


def _shade(scene, rays, **kw):
    try:
        return scene.shade(rays, **kw)
    except api.FtbError as e:
        assert e.status == abi.ERR_HIT_OVERFLOW
        return None


STAT_EXACT = ("primary_rays", "shadow_rays", "reflection_rays", "shaded_hits")


# ---- 1. FP64: exact against the renderer ---------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_fp64_paths_are_the_renderers_colour(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    sets = _sets(sc, case)
    rays = np.concatenate(list(sets.values()))
    point = abi.LIGHT_POINT in _lights(sc)
    with _open(sc) as scene:
        for rl in (0, 1, 8):
            st_p, st_s = abi.Stats(), abi.Stats()
            got = _paths(scene, rays, recursion_limit=rl, precision=FP64, collect_stats=1, stats=st_p)
            sh = _shade(scene, rays, recursion_limit=rl, precision=FP64, collect_stats=1, stats=True)
            if got is None or sh is None:
                assert got is None and sh is None and case.startswith("fuzz"), case
                pytest.skip("hit-stack overflow reported by both")
            st_s = sh["stats"]
            assert np.array_equal(got["colour"], sh["rgb"], equal_nan=True), (case, rl, int((got["colour"] != sh["rgb"]).any(axis=1).sum()))
            assert np.array_equal(po.replay(got["levels"], got["weight"], got["light_colour"]), got["colour"], equal_nan=True), (case, rl)
            for k in ("prim", "sub", "t"):
                assert np.array_equal(got[k][:, 0], sh[k]), (case, rl, k)
            a, b = st_p.as_dict(), st_s.as_dict()
            for k in STAT_EXACT:
                assert a[k] == b[k], (case, rl, k, a[k], b[k])
            tests_equal = a["leaf_tests"] == b["leaf_tests"] and a["bound_tests"] == b["bound_tests"]
            assert tests_equal or point, (case, rl, a["leaf_tests"], b["leaf_tests"], a["bound_tests"], b["bound_tests"])
            assert a["primary_rays"] == len(rays) and int(got["levels"].sum()) == len(rays) + a["reflection_rays"]
            print("%s rl %d: %d rays, levels max %d, %d shadow rays, %d reflections, leaf/bound tests %s"
                  % (case, rl, len(rays), got["levels"].max(), a["shadow_rays"], a["reflection_rays"], "equal" if tests_equal else
                     "differ (point light: common-origin table) %d / %d vs %d / %d" % (sum(a["leaf_tests"]), a["bound_tests"],
                                                                                     sum(b["leaf_tests"]), b["bound_tests"])))


# ---- 2. FP64 against the oracle ---------------------------------------------------------------------------------------------
def _scale(v, axis=-1):
    return np.maximum(np.abs(v).max(axis=axis), 1.0)


def _within(e):
    """Every error below 1e-6 of its scale and >= 99.9 % of them below the record bar (an empty set passes)."""
    return e.size == 0 or ((e <= 1e-6).all() and (e <= REC_BAR).mean() >= 0.999)


def _same_intensity(g, r, point):
    """[m, L] bool: directional and soft lights exactly (NaN = NaN); point lights blocked alike and within the record bar."""
    exact = (g == r) | (np.isnan(g) & np.isnan(r))
    close = ((g == 0) == (r == 0)) & (np.abs(g - r) <= REC_BAR * np.abs(r))
    return np.where(point[None, :], close, exact)


@pytest.mark.parametrize("case", sorted(CASES))
def test_fp64_paths_against_the_oracle(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    sets = _sets(sc, case)
    point = np.array([kind == abi.LIGHT_POINT for kind in _lights(sc)], dtype=bool)
    with _open(sc) as scene:
        for name, rays in sets.items():
            got = _paths(scene, rays, precision=FP64)
            if got is None:
                assert case.startswith("fuzz")
                pytest.skip("hit-stack overflow reported")
            ref = po.paths(sc, rays)
            n, D = got["weight"].shape
            L = got["intensity"].shape[2]
            alive = np.ones(n, bool)  # the rays whose earlier levels agree
            counts = dict(entries=0, id_mismatch=0, intensity_mismatch=0)
            for k in range(D):
                live = alive & (got["levels"] > k) & (ref["levels"] > k)
                if not live.any():
                    break
                same = live & (got["prim"][:, k] == ref["prim"][:, k]) & (got["sub"][:, k] == ref["sub"][:, k])
                mism = live & ~same
                counts["entries"] += int(live.sum())
                counts["id_mismatch"] += int(mism.sum())
                if k == 0 and name == "camera":
                    W, H = GRID
                    z = np.zeros((H, W, 3))
                    c = parity.compare_window(z, ref["prim"][:, 0].reshape(H, W, 1), z, got["prim"][:, 0].reshape(H, W, 1),
                                              ref_sub=ref["sub"][:, 0].reshape(H, W, 1), got_sub=got["sub"][:, 0].reshape(H, W, 1))
                    assert c["prim_unexplained"] == 0, (case, c.get("unexplained_samples"))
                # the level's ray and weight follow from the earlier levels, which agree
                e = np.abs(got["ray"][live, k] - ref["ray"][live, k]).max(axis=1) / _scale(ref["ray"][live, k])
                assert _within(e), (case, name, k, "ray", float(e.max()))
                assert (np.abs(got["weight"][live, k] - ref["weight"][live, k]) <= REC_BAR * _scale(ref["weight"][live, k, None])).all(), (case, name, k)
                hit = same & (ref["prim"][:, k] >= 0)
                if hit.any():
                    s = np.abs(ref["ray"][hit, k, :3]).max(axis=1) + np.abs(ref["t"][hit, k]) * np.abs(ref["ray"][hit, k, 3:]).max(axis=1) + 1.0
                    for pl in ("p", "normal", "hit_colour", "surface"):
                        e = np.abs(got[pl][hit, k] - ref[pl][hit, k]).max(axis=1) / (s if pl == "p" else 1.0)
                        assert _within(e), (case, name, k, pl, float(e.max()))
                    if L:
                        ieq = _same_intensity(got["intensity"][hit, k], ref["intensity"][hit, k], point)
                        counts["intensity_mismatch"] += int((~ieq).sum())
                        ok = np.broadcast_to(ieq.all(axis=1)[:, None], ieq.shape)
                        for pl in ("light_dir", "light_colour"):
                            g, r = got[pl][hit, k][ok], ref[pl][hit, k][ok]
                            fin = np.isfinite(r).all(axis=1)
                            assert np.array_equal(np.isfinite(g).all(axis=1), fin), (case, name, k, pl)
                            e = np.abs(g[fin] - r[fin]).max(axis=1) / _scale(r[fin])
                            assert _within(e), (case, name, k, pl, float(e.max()) if e.size else 0)
                # a level that differs ends the comparison of its ray; so does a differing intensity (the colours that follow differ)
                alive = same.copy()
                if L:
                    alive &= _same_intensity(got["intensity"][:, k], ref["intensity"][:, k], point).all(axis=1)
            assert counts["id_mismatch"] <= ID_FRAC * counts["entries"] + (0 if name == "camera" else 1), (case, name, counts)
            assert counts["intensity_mismatch"] <= ID_FRAC * counts["entries"] * max(L, 1), (case, name, counts)
            print("%s %s: %s" % (case, name, counts))


# ---- 3. FP32 -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_fp32_paths_against_the_renderer(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    sets = _sets(sc, case)
    rays = np.concatenate(list(sets.values()))
    with _open(sc) as scene:
        got = _paths(scene, rays, precision=FP32)
        sh = _shade(scene, rays, precision=FP32)
        if got is None or sh is None:
            assert case.startswith("fuzz")
            pytest.skip("hit-stack overflow reported")
        d = np.abs(got["colour"] - sh["rgb"]).max(axis=1)
        frac = float((d <= 1.0 / 255.0).mean())
        assert frac >= 0.999, (case, frac, float(np.nanmax(d)))
        W, H = GRID
        m = W * H
        z = np.zeros((H, W, 3))
        c = parity.compare_window(z, sh["prim"][:m].reshape(H, W, 1), z, got["prim"][:m, 0].reshape(H, W, 1), ref_sub=sh["sub"][:m].reshape(H, W, 1),
                                  got_sub=got["sub"][:m, 0].reshape(H, W, 1))
        assert c["prim_unexplained"] == 0, (case, c.get("unexplained_samples"))
        rep = po.replay(got["levels"], got["weight"], got["light_colour"])
        mag = np.abs(got["colour"]) + (np.abs(got["weight"])[..., None] * np.abs(np.nan_to_num(got["light_colour"])).sum(axis=2)).sum(axis=1) + 1e-30
        fin = np.isfinite(rep).all(axis=1)
        assert np.array_equal(fin, np.isfinite(got["colour"]).all(axis=1)), case
        e = (np.abs(rep - got["colour"]) / mag)[fin]
        assert (e <= 1e-5).all(), (case, float(e.max()))
        print("%s FP32: colour within 1/255 on %.5f (max %.3g), level-0 ids differ on %d of %d (unexplained 0), replay max %.3g"
              % (case, frac, float(np.nanmax(d)), c["prim_mismatch"], m, float(e.max()) if e.size else 0.0))


# ---- 4. sample keys reproduce a frame ----------------------------------------------------------------------------------------
def test_sample_keys_reproduce_a_frame_window():
    W, H, spp = 40, 30, 4
    sc = parse(scenes.sample(res=(W, H), spp=spp, focus=False))
    assert abi.LIGHT_SOFT_DIRECTIONAL in _lights(sc) and not sc.camera.has_focus
    jit = frontend.jitter_pattern(5, spp)
    win = (8, 6, 32, 26)
    with api.Scene(sc) as scene:
        frame = scene.render_window(win, W, H, spp, jit, debug=True, precision=FP64)
        px = [(x, y) for y in range(win[1], win[3]) for x in range(win[0], win[2])]
        rays = np.array([orc.primary_ray(sc.camera, W, H, x, y, jit[2 * s], jit[2 * s + 1]) for x, y in px for s in range(spp)])
        keys = np.array([(y * W + x) * spp + s for x, y in px for s in range(spp)], dtype=np.uint64)
        got = scene.trace_paths(rays, sample_keys=keys, precision=FP64)
        assert np.array_equal(got["prim"][:, 0], frame["prim"]) and np.array_equal(got["sub"][:, 0], frame["sub"])
        col = got["colour"].reshape(-1, spp, 3)
        acc = np.zeros((col.shape[0], 3))
        for s in range(spp):  # Array.average: a left fold from zero, then the division
            acc = acc + col[:, s]
        mean = acc / spp
        want = frame["rgb"].reshape(-1, 3)
        assert (np.abs(mean - want) <= 1e-12 * np.maximum(np.abs(want), 1e-300)).all(), float(np.abs(mean - want).max())
        plain = scene.trace_paths(rays, precision=FP64, planes=("colour",))
        differ = int((plain["colour"] != got["colour"]).any(axis=1).sum())
        print("window %s: %d samples, %d differ with the rays' indices as keys" % (win, len(rays), differ))
        assert differ > 0


# ---- 5. plumbing --------------------------------------------------------------------------------------------------------------
def _plumbing_scene(d):
    return CASES["bundled_hollow_sphere"](d)


def test_each_plane_alone_equals_the_full_request(tmp_path):
    sc = _plumbing_scene(str(tmp_path))
    rays = np.concatenate(list(_sets(sc, "plumbing").values()))
    with api.Scene(sc) as scene:
        for precision in (FP64, FP32):
            full = scene.trace_paths(rays, precision=precision)
            for name in api.PATH_PLANES:
                one = scene.trace_paths(rays, precision=precision, planes=(name,))
                assert set(one) == {name} and np.array_equal(one[name], full[name], equal_nan=True), (precision, name)
            n, D = full["weight"].shape
            after = np.arange(D)[None, :] >= full["levels"][:, None]
            assert after.any()
            assert (full["weight"][after] == 0).all() and (full["t"][after] == -1).all() and (full["prim"][after] == -1).all()
            assert (full["sub"][after] == 0).all() and (full["ray"][after] == 0).all()
            for k in ("p", "normal", "hit_colour", "surface", "intensity", "light_dir", "light_colour"):
                assert (full[k][after] == 0).all(), k
            miss = (full["prim"] == -1) & ~after
            assert miss.any() and (full["t"][miss] == -1).all() and (full["intensity"][miss] == 0).all() and (full["light_colour"][miss] == 0).all()
            assert (full["weight"][miss] > 0).all()  # a level that misses keeps its weight


def test_unrequested_planes_stay_untouched(tmp_path):
    """Every plane gets an array filled with a sentinel; a call that requests one plane writes that one only."""
    import ctypes as C
    sc = _plumbing_scene(str(tmp_path))
    rays = _sets(sc, "plumbing")["camera"][:100]
    n, dims = len(rays), {"D": 9, "L": sc.desc.n_lights}
    with api.Scene(sc) as scene:
        full = scene.trace_paths(rays, precision=FP64)
        p = api.make_params(1, 1, 1, None, recursion_limit=8, precision=FP64)
        for want in api.PATH_PLANES:
            arrs = {name: np.full((n,) + tuple(dims.get(k, k) for k in shape), 77, dtype=dt) for name, (_, dt, shape) in api.PATH_PLANES.items()}
            out = api._path_out({want: arrs[want].ctypes.data_as(C.POINTER(api.PATH_PLANES[want][0]))})
            api._check(api.lib().ftb_trace_paths(scene._h, rays.ctypes.data_as(C.POINTER(C.c_double)), None, n, C.byref(p), C.byref(out), None))
            for name, a in arrs.items():
                assert np.array_equal(a, full[name], equal_nan=True) if name == want else (a == 77).all(), (want, name)
        api._check(api.lib().ftb_trace_paths(scene._h, rays.ctypes.data_as(C.POINTER(C.c_double)), None, n, C.byref(p), None, None))


def test_no_lights_and_no_rays():
    sc = parse(one_object_scene("(material diffuse (0.5,0.5,0.5) reflectance 0.5 sphere)"))
    assert sc.desc.n_lights == 0
    cam = np.array([orc.primary_ray(sc.camera, 16, 16, x, y) for y in range(16) for x in range(16)])
    with api.Scene(sc) as scene:
        for precision in (FP64, FP32):
            got = scene.trace_paths(cam, precision=precision)
            assert (got["levels"] == 1).all() and (got["colour"] == 0).all()
            assert got["intensity"].shape == (len(cam), 9, 0) and got["light_colour"].shape == (len(cam), 9, 0, 3)
            sh = scene.shade(cam, precision=precision)
            assert np.array_equal(got["prim"][:, 0], sh["prim"]) and (got["prim"][:, 0] >= 0).any()
            hit = got["prim"][:, 0] >= 0
            assert (got["surface"][hit, 0, 1] == 0.5).all() and (got["weight"][:, 0] == 1).all()
            empty = scene.trace_paths(np.zeros((0, 6)), precision=precision)
            assert empty["colour"].shape == (0, 3) and empty["weight"].shape == (0, 9)


def test_recursion_limit_63_works_and_64_is_refused(tmp_path):
    sc = _plumbing_scene(str(tmp_path))
    rays = _sets(sc, "plumbing")["camera"]
    with api.Scene(sc) as scene:
        got = scene.trace_paths(rays, recursion_limit=63, precision=FP64)
        sh = scene.shade(rays, recursion_limit=63, precision=FP64)
        assert got["weight"].shape == (len(rays), 64) and np.array_equal(got["colour"], sh["rgb"])
        print("recursion limit 63: levels max %d" % got["levels"].max())
        with pytest.raises(api.FtbError) as e:
            scene.trace_paths(rays, recursion_limit=64, precision=FP64)
        assert e.value.status == abi.ERR_BAD_ARG


def test_device_entry_on_a_side_stream_equals_the_host_entry(tmp_path):
    import torch
    sc = CASES["large_shiny_blob"](str(tmp_path))
    rays = np.concatenate(list(_sets(sc, "device").values()))
    n, L = len(rays), sc.desc.n_lights
    keys = np.arange(n, dtype=np.uint64)[::-1].copy() * 3 + 11
    with api.Scene(sc) as scene:
        for precision in (FP64, FP32):
            host = scene.trace_paths(rays, sample_keys=keys, recursion_limit=4, seed=99, precision=precision)
            side = torch.cuda.Stream()
            d_rays = torch.from_numpy(rays).cuda()
            d_keys = torch.from_numpy(keys.view(np.int64)).cuda()
            dims = {"D": 5, "L": L}
            dev = {}
            for name, (_, dt, shape) in api.PATH_PLANES.items():
                tdt = {np.int32: torch.int32, np.float64: torch.float64}[dt]
                dev[name] = torch.full((n,) + tuple(dims.get(k, k) for k in shape), -3, dtype=tdt, device="cuda")
            torch.cuda.synchronize()
            with torch.cuda.stream(side):
                scene.trace_paths_device(d_rays.data_ptr(), n, {k: v.data_ptr() for k, v in dev.items()}, d_keys_ptr=d_keys.data_ptr(),
                                         recursion_limit=4, seed=99, stream=side.cuda_stream, precision=precision)
            side.synchronize()
            scene.check_overflow(stream=side.cuda_stream)
            for name in api.PATH_PLANES:
                assert np.array_equal(dev[name].cpu().numpy(), host[name], equal_nan=True), (precision, name)


def test_hit_overflow_leaves_the_host_arrays_unwritten(tmp_path):
    row = vs.over_limit_scenes()[0]
    text, assets = row.text(str(tmp_path))
    sc = parse(text, assets=assets)
    rays = np.array([orc.primary_ray(sc.camera, 32, 24, x, y) for y in range(24) for x in range(32)])
    with api.Scene(sc) as scene:
        for precision in (FP64, FP32):
            colour = np.full((len(rays), 3), 5.0)
            import ctypes as C
            out = abi.PathOut()
            out.colour = colour.ctypes.data_as(C.POINTER(C.c_double))
            p = api.make_params(1, 1, 1, None, precision=precision)
            rc = api.lib().ftb_trace_paths(scene._h, rays.ctypes.data_as(C.POINTER(C.c_double)), None, len(rays), C.byref(p), C.byref(out), None)
            assert rc == abi.ERR_HIT_OVERFLOW and (colour == 5.0).all(), (precision, rc)
