"""Frames and queries at scene scales far from the unit.  Needs a B200: run with `-m gpu`.

Each family of tests/scale_scenes.py, enlarged by s and moved by T over tests/scale_scenes.py SWEEP (objects from 1e-3 to 1e4
units across, |p| up to 2e4), against the oracle rendered at the same s and T:

  (a) Shortcuts change no bit: ftb_render_window of the whole frame equals ftb_frame_rays -> ftb_shade_samples, colour and the
      prim / sub / t planes, in FP32 and FP64 at 4 spp.  The frame writes clear tiles without tracing them, skips the shadow rays
      of lit ground tiles and culls items with the inflated spheres, the common-origin table and its primary slack; the explicit
      path takes none of these.  A margin too small at some scale shows here as a differing bit, with no tolerance.  The host's
      clear and lit tiles of each frame are printed (the probes of tests/test_clear_boxes_cpu.py and tests/test_lit_tiles_cpu.py).
  (b) FP64 against the oracle with test_gpu_parity.check's bars, every primary-id mismatch classified by oracle/parity.py: an
      unexplained one is a cull or an absolute constant on the device that the oracle does not have.
  (c) FP32 against the oracle with the product bars (1/255 on >= 99.9 % of the pixels, ids <= 0.5 %), or within the envelope
      ENVELOPE measured for the cases where the float32 spacing next to |p| cannot hold the reference's absolute 1e-4 offsets
      (DESIGN.md section 6).  Printed per case: the share of hit samples whose level-0 shadow intensities differ from the
      oracle's (ftb_trace_paths on the frame's own primary rays and keys against tests/path_oracle.py: shadow acne).
  (d) Nearest-hit queries (ftb_intersect_rays) of the frame's primary rays in FP64 against tests/query_oracle.py, with
      test_gpu_ray_queries.compare_nearest's bars: ids agree except on classified ties.
  (e) Counters at the extreme scales: the counting kernel's primary, shadow and reflection rays and shaded hits agree with the
      oracle's as test_gpu_parity.test_stats_counters_against_oracle holds them."""
import functools
import tempfile

import numpy as np
import pytest

import path_oracle as po
import query_oracle as qo
import scale_scenes as ss
import test_clear_boxes_cpu as boxes_stage
import test_clear_tiles_cpu as sphere_stage
from functracer_b200 import abi, api, frontend
from oracle import ftb_oracle as orc
from oracle import parity
from test_gpu_parity import check
from test_gpu_ray_queries import _open, compare_nearest
from test_gpu_sample_shading import _assert_same, _probe
from util import colour_stats, parse

pytestmark = pytest.mark.gpu

FP32, FP64 = abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY
W, H = 192, 108
SPP_SHORTCUTS, SPP = 4, 2
SEED = 77
CASES = [(f, s, T) for f in sorted(ss.FAMILIES) for s, T in ss.SWEEP]
IDS = ["%s-%s" % (f, ss.case_id(s, T)) for f, s, T in CASES]
EXTREMES = ("s-10_T0", "s10_T0", "s-5_T1e3", "s0_T1e4", "s5_T1e4")

# (family, case id) -> (largest primary-id mismatch share, smallest share of pixels within 1/255): the FP32 frame's measured
# envelope where it misses the product bars (NVIDIA B200, see DESIGN.md section 6); every other case holds the product bars
ENVELOPE = {
    ("acne", "s10_T0"): (1e-4, 0.941), ("acne", "s0_T1e3"): (1e-4, 0.983), ("acne", "s-5_T1e3"): (1.2e-3, 0.972), ("acne", "s0_T1e4"): (3e-4, 0.901),
    ("acne", "s5_T1e4"): (1e-4, 0.893),
    ("hollow_sphere", "s10_T0"): (1e-4, 0.244), ("hollow_sphere", "s0_T1e3"): (1e-4, 0.960), ("hollow_sphere", "s-5_T1e3"): (2e-3, 0.980),
    ("hollow_sphere", "s0_T1e4"): (6e-4, 0.363), ("hollow_sphere", "s5_T1e4"): (1e-4, 0.297),
    ("house", "s10_T0"): (1e-4, 0.933), ("house", "s-5_T1e3"): (4e-4, 0.995), ("house", "s0_T1e4"): (1e-4, 0.939), ("house", "s5_T1e4"): (1e-4, 0.933),
    ("meshes", "s10_T0"): (1e-4, 0.981), ("meshes", "s0_T1e3"): (3e-4, 0.994), ("meshes", "s-5_T1e3"): (3e-3, 0.987), ("meshes", "s0_T1e4"): (1e-3, 0.978),
    ("meshes", "s5_T1e4"): (1e-4, 0.980),
    ("night_house", "s10_T0"): (1e-4, 0.953), ("night_house", "s-5_T1e3"): (2e-4, 0.995), ("night_house", "s0_T1e4"): (1e-4, 0.959),
    ("night_house", "s5_T1e4"): (1e-4, 0.958),
    ("repeat", "s10_T0"): (1e-4, 0.940), ("repeat", "s-5_T1e3"): (2e-4, 0.996), ("repeat", "s0_T1e4"): (1e-4, 0.942), ("repeat", "s5_T1e4"): (1e-4, 0.941),
}


def _scene(family, s, T, spp):
    d = tempfile.mkdtemp(prefix="ftb_scale_")
    return parse(*ss.family_text(family, d, (W, H), spp, s, T))


@functools.lru_cache(maxsize=4)
def _oracle(family, s, T):
    sc = _scene(family, s, T, SPP)
    return orc.render(sc, orc.make_params(W, H, SPP, frontend.jitter_pattern(3, SPP), sampling=sc.sampling, seed=SEED))


@pytest.fixture(scope="module")
def probes():
    return boxes_stage.build_probe(tempfile.mkdtemp(prefix="ftb_scale_boxes_")), _probe("lit")


# ---- (a) shortcuts change no bit -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family, s, T", CASES, ids=IDS)
def test_shortcuts_change_no_bit(probes, family, s, T):
    sc = _scene(family, s, T, SPP_SHORTCUTS)
    jit = frontend.jitter_pattern(3, SPP_SHORTCUTS)
    (clear_lib, (lit_lib, lit_mask)) = probes
    p = api.make_params(W, H, SPP_SHORTCUTS, jit, precision=FP32)
    clear = sphere_stage.clear_mask(clear_lib, sc, p)
    lit, ground = lit_mask(lit_lib, sc, p)
    print("%s %s: %d of %d tiles clear, %d lit (ground prim %d)" % (family, ss.case_id(s, T), int(clear.sum()), clear.size, int((lit != 0).sum()), ground))
    with _open(sc) as scene:
        for precision in (FP32, FP64):
            frame = scene.render_window((0, 0, W, H), W, H, SPP_SHORTCUTS, jit, precision=precision, out_format=abi.OUT_RGB_F64, seed=SEED, debug=True)
            rays, keys = scene.frame_rays((0, 0, W, H), W, H, SPP_SHORTCUTS, jit, precision=precision, seed=SEED)
            got = scene.shade_samples(rays, SPP_SHORTCUTS, sample_keys=keys, precision=precision, out_format=abi.OUT_RGB_F64, seed=SEED, debug=True)
            _assert_same(frame, got, (family, ss.case_id(s, T), precision))


def _render(sc, precision):
    with _open(sc) as scene:
        return scene.render(W, H, SPP, frontend.jitter_pattern(3, SPP), sampling=sc.sampling, seed=SEED, precision=precision, debug=True)


def _classified(ref, got):
    return parity.compare_window(ref["rgb"], ref["prim"].reshape(H, W, SPP), got["rgb"], got["prim"].reshape(H, W, SPP),
                                 ref_sub=ref["sub"].reshape(H, W, SPP), got_sub=got["sub"].reshape(H, W, SPP))


# ---- (b) FP64 against the oracle -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family, s, T", CASES, ids=IDS)
def test_fp64_against_the_oracle(family, s, T):
    ref, got = _oracle(family, s, T), _render(_scene(family, s, T, SPP), FP64)
    c = _classified(ref, got)
    print("%s %s FP64: %d of %d primary ids differ (unexplained %d, edge leaks %d)" % (family, ss.case_id(s, T), c["prim_mismatch"], c["samples"],
                                                                                    c["prim_unexplained"], c["prim_edge_leak"]))
    assert c["prim_unexplained"] == 0, c.get("unexplained_samples")
    check(ref, got, FP64, "%s %s" % (family, ss.case_id(s, T)))


# ---- (c) FP32 against the oracle -----------------------------------------------------------------------------------------------
def _acne(sc, scene, ref_intensity_of):
    """(share of the level-0 hits whose shadow intensities differ from the oracle's, hits compared, that share per primitive, the
    primitives from 5 on taken together) for the frame's own primary rays and keys: directional and soft lights exactly (a ratio
    of sample counts), point lights blocked alike."""
    rays, keys = scene.frame_rays((0, 0, W, H), W, H, SPP, frontend.jitter_pattern(3, SPP), precision=FP32, seed=SEED)
    got = scene.trace_paths(rays, sample_keys=keys, seed=SEED, precision=FP32, planes=("levels", "prim", "sub", "intensity"))
    ref = ref_intensity_of(rays, keys)
    hit = (got["prim"][:, 0] >= 0) & (got["prim"][:, 0] == ref["prim"][:, 0]) & (got["sub"][:, 0] == ref["sub"][:, 0])
    L = sc.desc.n_lights
    if not hit.any() or L == 0:
        return 0.0, int(hit.sum()), {}
    point = np.array([sc.desc.lights[k].kind == abi.LIGHT_POINT for k in range(L)])
    g, r = got["intensity"][hit, 0], ref["intensity"][hit, 0]
    differ = np.where(point[None, :], (g == 0) != (r == 0), np.abs(g - r) > 1e-6).any(axis=1)
    prim = np.minimum(ref["prim"][hit, 0], 5)
    per = {int(q): round(float(differ[prim == q].mean()), 5) for q in np.unique(prim)}
    return float(differ.mean()), int(hit.sum()), per


@pytest.mark.parametrize("family, s, T", CASES, ids=IDS)
def test_fp32_against_the_oracle(family, s, T):
    sc = _scene(family, s, T, SPP)
    ref = _oracle(family, s, T)
    with _open(sc) as scene:
        got = scene.render(W, H, SPP, frontend.jitter_pattern(3, SPP), sampling=sc.sampling, seed=SEED, precision=FP32, debug=True)
        acne, hits, per_prim = _acne(sc, scene, lambda rays, keys: po.paths(sc, rays, keys, seed=SEED))
    cs = colour_stats(got["rgb"], ref["rgb"])
    mism = float((got["prim"] != ref["prim"]).mean())
    c = _classified(ref, got)
    key = (family, ss.case_id(s, T))
    print("%s %s FP32: within 1/255 %.5f (max %.3g), primary ids differ %.2e (unexplained %d), level-0 shadow intensities differ on %.5f of %d hits"
          % (key + (cs["frac_within"], cs["max"], mism, c["prim_unexplained"], acne, hits)))
    if family == "acne":  # primitives 0 .. 5: ground plane, sphere, cube, solidCylinder, cone, the mesh's triangles
        print("    per primitive: %s" % per_prim)
    if key in ENVELOPE:
        max_id, min_within = ENVELOPE[key]
        assert mism <= max_id and cs["frac_within"] >= min_within, (key, mism, cs["frac_within"], ENVELOPE[key])
    else:
        check(ref, got, FP32, "%s %s" % key)


# ---- (d) nearest-hit queries ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family, s, T", CASES, ids=IDS)
def test_nearest_queries_of_the_primary_rays(family, s, T):
    sc = _scene(family, s, T, 1)
    with _open(sc) as scene:
        rays, _ = scene.frame_rays((0, 0, W, H), W, H, 1, frontend.jitter_pattern(3, 1), precision=FP64, seed=SEED)
        got = scene.intersect(rays, precision=FP64)
    res = compare_nearest(got, qo.nearest(sc, rays), rays, FP64, (family, ss.case_id(s, T)), grid=(W, H))
    print("%s %s: %s" % (family, ss.case_id(s, T), res))


# ---- (e) counters at the extreme scales ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("family, s, T", [c for c in CASES if ss.case_id(c[1], c[2]) in EXTREMES],
                         ids=[i for i, c in zip(IDS, CASES) if ss.case_id(c[1], c[2]) in EXTREMES])
def test_counters_against_the_oracle(family, s, T):
    Wc, Hc = 96, 54
    sc = parse(*ss.family_text(family, tempfile.mkdtemp(prefix="ftb_scale_"), (Wc, Hc), 1, s, T))
    jit = frontend.jitter_pattern(2, 1)
    a = orc.render(sc, orc.make_params(Wc, Hc, 1, jit))["stats"]
    with _open(sc) as scene:
        b = scene.render(Wc, Hc, 1, jit, precision=FP64, stats=True)["stats"]
    print("%s %s: primary %d / %d, shaded %d / %d, reflection %d / %d, shadow %d / %d" % (
        family, ss.case_id(s, T), b.primary_rays, a.primary_rays, b.shaded_hits, a.shaded_hits, b.reflection_rays, a.reflection_rays,
        b.shadow_rays, a.shadow_rays))
    assert b.primary_rays == a.primary_rays == Wc * Hc
    assert abs(int(b.shaded_hits) - int(a.shaded_hits)) <= 2
    assert abs(int(b.reflection_rays) - int(a.reflection_rays)) <= 4
    assert abs(int(b.shadow_rays) - int(a.shadow_rays)) <= 4
