"""The host's tile proofs at scene scales far from the unit, tested with the REAL host code (the probes of
tests/test_clear_tiles_cpu.py, tests/test_clear_boxes_cpu.py and tests/test_lit_tiles_cpu.py) against the CPU oracle.  CPU only.

Every scene of the other proof tests sits within about ten units of the origin, while the proofs mix absolute margins (tiles.cpp
`bound_r * 1.002 + 1e-5`, lit_tiles.cpp `1.1e-4`) with margins relative to the distance from the origin (tiles.cpp kRel and
primarySlack, clear_boxes.cpp `1e-4 (1 + |p|)`).  Here each family of tests/scale_scenes.py is enlarged by s and moved by T
over tests/scale_scenes.py SWEEP, and on every case:
  - no clear tile (sphere stage, then the box stage the frame uses) holds a sample the oracle reports as a hit;
  - no lit (tile, directional light) pair has a ground sample whose shadow ray the oracle finds blocked.
An empty mask passes both trivially, so SHARES pins what each case proves: the share of clear tiles and the share of ground
samples proven lit, each at least its entry less MARGIN and non-zero wherever the entry is.  Where an entry is lower than at
s = 1, T = 0, the relative margins have grown with the distance from the origin (house loses its clear tiles by the sphere stage
at T = (1e4, 0, 1e4), and the box stage keeps them).  Two planted errors in lit_tiles.cpp must each be caught on some case.

The oracle is FP64 and traces exact geometry: it refutes a proof that is wrong in exact arithmetic.  The margins that cover the
FP32 rounding of the device's rays (tiles.cpp `+ 1e-5` and kRel; with `+ 0` or kRel = 1e-7 this file still passes) are
held by tests/test_gpu_scale.py, where a frame whose clear tile hides an FP32 hit differs from its own samples traced plainly."""
import pytest

import scale_scenes as ss
import test_clear_boxes_cpu as boxes_stage
import test_lit_tiles_cpu as lit_tiles
from functracer_b200 import frontend
from oracle import ftb_oracle as orc
from util import parse

RES, SPP = (192, 108), 2
MAX_LIT_SAMPLES = 1500
MARGIN = 0.01
# the soft light's penumbra of test_lit_tiles_cpu, whose scatter cone the lit proof must widen by: checked on every sample
PENUMBRA = "penumbra"
FAMILIES = sorted(ss.FAMILIES) + [PENUMBRA]

# (family, tests/scale_scenes.case_id) -> (share of clear tiles with the boxes, share of ground samples proven lit), measured
# with this file at RES x SPP; the rows follow tests/scale_scenes.py SWEEP
SHARES = {
    ("acne", "s0_T0"): (0.0000, 0.5311), ("acne", "s-10_T0"): (0.0000, 0.5311), ("acne", "s10_T0"): (0.0000, 0.5288),
    ("acne", "s-5_T1e2"): (0.0000, 0.5311), ("acne", "s0_T1e2"): (0.0000, 0.5311), ("acne", "s0_T1e3"): (0.0000, 0.5311),
    ("acne", "s-5_T1e3"): (0.0000, 0.2749), ("acne", "s0_T1e4"): (0.0000, 0.4514), ("acne", "s5_T1e4"): (0.0000, 0.5311),
    ("hollow_sphere", "s0_T0"): (0.0000, 0.0000), ("hollow_sphere", "s-10_T0"): (0.0000, 0.0000),
    ("hollow_sphere", "s10_T0"): (0.0000, 0.0000), ("hollow_sphere", "s-5_T1e2"): (0.0000, 0.0000),
    ("hollow_sphere", "s0_T1e2"): (0.0000, 0.0000), ("hollow_sphere", "s0_T1e3"): (0.0000, 0.0000),
    ("hollow_sphere", "s-5_T1e3"): (0.0000, 0.0000), ("hollow_sphere", "s0_T1e4"): (0.0000, 0.0000),
    ("hollow_sphere", "s5_T1e4"): (0.0000, 0.0000),
    ("house", "s0_T0"): (0.2262, 0.2141), ("house", "s-10_T0"): (0.2262, 0.1828), ("house", "s10_T0"): (0.2262, 0.2141),
    ("house", "s-5_T1e2"): (0.2262, 0.1828), ("house", "s0_T1e2"): (0.2262, 0.2141), ("house", "s0_T1e3"): (0.2262, 0.1828),
    ("house", "s-5_T1e3"): (0.0000, 0.0762), ("house", "s0_T1e4"): (0.1786, 0.1583), ("house", "s5_T1e4"): (0.2262, 0.2141),
    ("meshes", "s0_T0"): (0.7738, 0.0000), ("meshes", "s-10_T0"): (0.7738, 0.0000), ("meshes", "s10_T0"): (0.7738, 0.0000),
    ("meshes", "s-5_T1e2"): (0.7143, 0.0000), ("meshes", "s0_T1e2"): (0.7738, 0.0000), ("meshes", "s0_T1e3"): (0.7381, 0.0000),
    ("meshes", "s-5_T1e3"): (0.0000, 0.0000), ("meshes", "s0_T1e4"): (0.6071, 0.0000), ("meshes", "s5_T1e4"): (0.7619, 0.0000),
    ("night_house", "s0_T0"): (0.1429, 0.6634), ("night_house", "s-10_T0"): (0.1429, 0.6448), ("night_house", "s10_T0"): (0.1429, 0.6634),
    ("night_house", "s-5_T1e2"): (0.1429, 0.6448), ("night_house", "s0_T1e2"): (0.1429, 0.6634),
    ("night_house", "s0_T1e3"): (0.1429, 0.6448), ("night_house", "s-5_T1e3"): (0.0000, 0.5940),
    ("night_house", "s0_T1e4"): (0.1429, 0.6313), ("night_house", "s5_T1e4"): (0.1429, 0.6634),
    ("repeat", "s0_T0"): (0.5357, 0.0000), ("repeat", "s-10_T0"): (0.5357, 0.0000), ("repeat", "s10_T0"): (0.5357, 0.0000),
    ("repeat", "s-5_T1e2"): (0.5357, 0.0000), ("repeat", "s0_T1e2"): (0.5357, 0.0000), ("repeat", "s0_T1e3"): (0.5357, 0.0000),
    ("repeat", "s-5_T1e3"): (0.2381, 0.0000), ("repeat", "s0_T1e4"): (0.5000, 0.0000), ("repeat", "s5_T1e4"): (0.5357, 0.0000),
    ("penumbra", "s0_T0"): (0.2500, 0.7053), ("penumbra", "s-10_T0"): (0.2500, 0.6846), ("penumbra", "s10_T0"): (0.2500, 0.7053),
    ("penumbra", "s-5_T1e2"): (0.2500, 0.6846), ("penumbra", "s0_T1e2"): (0.2500, 0.7053), ("penumbra", "s0_T1e3"): (0.2500, 0.6846),
    ("penumbra", "s-5_T1e3"): (0.0500, 0.4776), ("penumbra", "s0_T1e4"): (0.2125, 0.6639), ("penumbra", "s5_T1e4"): (0.2500, 0.7053),
}


def _scene(family, d, s, T):
    if family == PENUMBRA:
        sc = parse(ss.scaled(lit_tiles.HARD[PENUMBRA], s, T))
    else:
        sc = parse(*ss.family_text(family, d, RES, SPP, s, T))
    return sc, orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(3, sc.spp), sampling=sc.sampling)


@pytest.fixture(scope="module")
def probes(tmp_path_factory):
    return boxes_stage.build_probe(str(tmp_path_factory.mktemp("scale_boxes"))), lit_tiles._build(str(tmp_path_factory.mktemp("scale_lit")), "tree")


@pytest.mark.parametrize("s, T", ss.SWEEP, ids=[ss.case_id(s, T) for s, T in ss.SWEEP])
@pytest.mark.parametrize("family", FAMILIES)
def test_proofs_hold_at_every_scale(probes, family, s, T, tmp_path):
    clear_lib, lit_lib = probes
    sc, p = _scene(family, str(tmp_path), s, T)
    spheres, clear = boxes_stage.shares(clear_lib, sc, p)  # both stages against the oracle
    lit, checked, blocked = lit_tiles.check_against_oracle(lit_lib, sc, p, max_samples=None if family == PENUMBRA else MAX_LIT_SAMPLES)
    key = (family, ss.case_id(s, T))
    print("%-14s %-9s clear tiles %.4f (spheres %.4f), lit ground samples %.4f, %d shadow rays checked" % (key + (clear, spheres, lit, checked)))
    assert blocked == 0, "%d of %d shadow rays of lit ground samples are blocked" % (blocked, checked)
    want_clear, want_lit = SHARES[key]
    for got, want, what in ((clear, want_clear, "clear"), (lit, want_lit, "lit")):
        assert got >= want - MARGIN, (key, what, got, want)
        assert got > 0 or want == 0, (key, what, got, want)


@pytest.mark.parametrize("plant", sorted(lit_tiles.PLANTS))
def test_planted_lit_errors_are_caught_on_some_scale(tmp_path, plant):
    bad = lit_tiles._build(str(tmp_path), plant, plant)
    for s, T in ss.SWEEP:
        sc, p = _scene(PENUMBRA, str(tmp_path), s, T)
        _, checked, blocked = lit_tiles.check_against_oracle(bad, sc, p)
        if blocked:
            print("%s caught at %s: %d of %d shadow rays blocked" % (plant, ss.case_id(s, T), blocked, checked))
            return
    pytest.fail("the planted error %s went unnoticed at every scale" % plant)


def test_the_sweep_spans_small_far_and_large_near():
    far = lambda T: max(abs(x) for x in T)
    assert any(s < 1 and far(T) >= 1e2 for s, T in ss.SWEEP) and any(s > 1 and far(T) == 0 for s, T in ss.SWEEP)
    assert set(SHARES) == {(f, ss.case_id(s, T)) for f in FAMILIES for s, T in ss.SWEEP}


# ---- the scale transform itself ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", sorted(ss.FAMILIES) + ["sample"])
def test_scaled_maps_camera_lights_and_kernel_variant(family, tmp_path):
    """The front end reads the scaled text back with the camera and the lights mapped as scale_scenes states, and the lowering
    sends every scaled scene to the kernel variant of the unscaled one.  `sample` has depth of field: its focal length scales."""
    import numpy as np
    import test_lowering_cpu as low
    from functracer_b200 import abi, scenes
    lib = low.build_probe(str(tmp_path))
    variants = low.compiled_variants()
    if family == "sample":
        text, assets = scenes.sample(res=RES, spp=SPP), scenes.asset_dir()
    else:
        text, assets = ss.FAMILIES[family](str(tmp_path), RES, SPP)
    base = parse(text, assets)
    want = low.pick(low.lowered(lib, text, assets)[0], variants)
    for s, T in ss.SWEEP:
        out = ss.scaled(text, s, T)
        sc = parse(out, assets)
        root, root0 = sc.desc.nodes[sc.desc.root], base.desc.nodes[base.desc.root]
        assert root.b == root0.b and all(sc.desc.nodes[sc.desc.children[root.a + i]].kind == abi.NODE_TRANSFORM for i in range(root.b))
        c0, c = base.camera, sc.camera
        move = lambda p: s * np.asarray(p[:], dtype=np.float64) + np.asarray(T)
        assert np.allclose(c.o[:], move(c0.o), rtol=1e-15, atol=0) and np.allclose(c.look_at[:], move(c0.look_at), rtol=1e-15, atol=0)
        assert c.up[:] == c0.up[:] and c.fov_y_rad == c0.fov_y_rad and c.aspect_ratio == c0.aspect_ratio
        assert c.has_focus == c0.has_focus and c.focal_length == s * c0.focal_length and c.aperture_rad == c0.aperture_rad
        assert (sc.width, sc.height, sc.spp, sc.sampling) == (base.width, base.height, base.spp, base.sampling)
        assert sc.desc.n_lights == base.desc.n_lights
        for k in range(sc.desc.n_lights):
            a, b = base.desc.lights[k], sc.desc.lights[k]
            assert (b.kind, b.samples, b.scatter_rad, b.colour[:]) == (a.kind, a.samples, a.scatter_rad, a.colour[:])
            if a.kind == abi.LIGHT_POINT:
                assert np.allclose(b.v[:], move(a.v), rtol=1e-15, atol=0)
                assert b.falloff[:] == [a.falloff[0], a.falloff[1] / s, a.falloff[2] / (s * s)]
            else:
                assert b.v[:] == a.v[:]
        got = low.pick(low.lowered(lib, out, assets)[0], variants)
        assert got == want, (family, ss.case_id(s, T), hex(got), hex(want))
    print("%s: every scaled scene runs on variant 0x%03x" % (family, want))
