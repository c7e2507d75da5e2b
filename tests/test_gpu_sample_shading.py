"""A frame's own samples (ftb_frame_rays) shaded and blended on the explicit-ray path (ftb_shade_samples).  Needs a B200: run with
`-m gpu`.

  1. Frames equal their own samples, bit for bit: on the bundled scenes, one scene per kernel variant, six fuzz seeds and the two
     large-mesh scenes, ftb_frame_rays -> ftb_shade_samples with the frame's keys and params equals ftb_render_window, colour and
     the prim / sub / t planes, for a whole frame and an odd window, at spp across every unit, quad and pass boundary of the
     blend ring, in every out_format and both precisions.  The frame takes shortcuts the explicit path never takes (clear tiles
     written without tracing, lit ground tiles that skip shadow rays, the camera's row of the common-origin bound table, the
     costliest-first tile order); the house, night-house and repeat frames are checked to contain clear and lit tiles.
  2. Depth of field: FP64 bit-identical; FP32 (the frame runs the scene's variant with FT_RNG added) within 1/255 on >= 99.9 %
     of the pixels, every primary-id difference classified by oracle/parity.py.
  3. ftb_frame_rays against the oracle: rays equal orc.primary_ray (with the depth-of-field draw of the RNG contract) to FP
     rounding, keys exactly; the path query's reconstruction of a frame window is bit-exact with these rays.
  4. Against ftb_shade_rays: without keys the FP64 pixels are the literal left fold of ftb_shade_rays' colours divided by spp;
     at spp = 1 they are ftb_shade_rays' colours in both precisions.
  5. A custom camera: orthographic rays built here, shaded and blended, against the oracle's shade_rays averaged per pixel.
  6. Counters: primary, shadow and reflection rays and shaded hits equal the frame's counting kernel's.
  7. Plumbing: n_pixels = 0, unrequested debug planes untouched, the device entries on a side stream equal the host entries, a
     hit-stack overflow leaves the host arrays unwritten, and one batch of more than 2^24 samples equals smaller batches."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import variant_scenes as vs
from functracer_b200 import abi, api, frontend, scenes
from oracle import ftb_oracle as orc
from oracle import parity
from test_gpu_ray_queries import CASES, _open
from util import parse

pytestmark = pytest.mark.gpu

FP32, FP64 = abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY
FORMATS = (abi.OUT_RGB_F64, abi.OUT_RGB_F32, abi.OUT_RGBA8)
SPPS = (1, 3, 42, 43, 64, 86, 129, 130, 257)
W, H = 48, 36
WINDOW = (5, 3, 16, 10)  # 11 x 7 pixels, odd, off the tile grid
SEED = 77


def _frame_and_samples(scene, sc, window, spp, jit, precision, out_format, stats=False):
    """(ftb_render_window's dict, ftb_shade_samples' dict) for the same window, or None when both report a hit-stack overflow."""
    kw = dict(precision=precision, out_format=out_format, seed=SEED, debug=True)
    try:
        frame = scene.render_window(window, W, H, spp, jit, stats=stats, **kw)
    except api.FtbError as e:
        assert e.status == abi.ERR_HIT_OVERFLOW
        frame = None
    rays, keys = scene.frame_rays(window, W, H, spp, jit, precision=precision, seed=SEED)
    try:
        got = scene.shade_samples(rays, spp, sample_keys=keys, stats=stats, **kw)
    except api.FtbError as e:
        assert e.status == abi.ERR_HIT_OVERFLOW and frame is None
        return None
    assert frame is not None
    return frame, got


def _assert_same(frame, got, what):
    ch = frame["rgb"].shape[-1]
    a, b = frame["rgb"].reshape(-1, ch), got["rgb"].reshape(-1, ch)
    same = (a == b) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == "f" else a == b
    assert same.all(), "%s: %d of %d pixels differ" % (what, int((~same.all(axis=1)).sum()), len(a))
    for k in ("prim", "sub", "t"):
        assert np.array_equal(frame[k], got[k]), (what, k)


# ---- 1. frames equal their own samples ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_frames_equal_their_own_samples(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    with _open(sc) as scene:
        checked = 0
        for precision in (FP64, FP32):
            for spp in SPPS:
                jit = frontend.jitter_pattern(spp, spp)
                windows = [WINDOW] + ([(0, 0, W, H)] if spp in (1, 3) else [])
                for win in windows:
                    for fmt in FORMATS:
                        r = _frame_and_samples(scene, sc, win, spp, jit, precision, fmt)
                        if r is None:
                            pytest.skip("hit-stack overflow reported by both")
                        _assert_same(*r, what=(case, precision, spp, win, fmt))
                        checked += 1
        print("%s: %d frames equal their samples" % (case, checked))


def _probe(kind):
    """The host-side clear-tile / lit-tile probes of the CPU tests (compiled with g++ from the library's own sources)."""
    if kind == "clear":
        import test_clear_tiles_cpu as t
        d = tempfile.mkdtemp(prefix="ftb_clear_")
        src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe.so")
        open(src, "w").write(t.PROBE % dict(csrc=t.CSRC))
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src, os.path.join(t.CSRC, "cuda", "tiles.cpp"),
                               os.path.join(t.CSRC, "cuda", "lower.cpp")])
        lib = C.CDLL(so)
        lib.ftb_probe_clear.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 4 + [
            C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.ftb_probe_clear.restype = C.c_int
        return lib, t.clear_mask
    import test_lit_tiles_cpu as t
    return t._build(tempfile.mkdtemp(prefix="ftb_lit_"), "tree"), t.lit_mask


@pytest.mark.parametrize("name", ["house", "night_house", "repeat"])
def test_frame_shortcuts_change_no_bit(name):
    """Frames whose clear tiles are written without tracing and whose lit ground tiles skip shadow rays, against the same samples
    traced the plain way."""
    Wf, Hf = 256, 144  # repeat's first lit ground tiles appear at this size
    sc = parse(getattr(scenes, name)(res=(Wf, Hf), spp=1))
    clear_lib, clear_mask = _probe("clear")
    lit_lib, lit_mask = _probe("lit")
    with api.Scene(sc) as scene:
        for spp in (4, 64):
            jit = frontend.jitter_pattern(3, spp)
            p = api.make_params(Wf, Hf, spp, jit, precision=FP32)
            clear = clear_mask(clear_lib, sc, p)
            lit, ground = lit_mask(lit_lib, sc, p)
            print("%s %d spp: %d of %d tiles clear, %d lit (ground prim %d)" % (name, spp, int(clear.sum()), clear.size, int((lit != 0).sum()), ground))
            assert clear.any() and (lit != 0).any()
            for precision in (FP32, FP64):
                rays, keys = scene.frame_rays((0, 0, Wf, Hf), Wf, Hf, spp, jit, precision=precision, seed=SEED)
                for fmt in FORMATS if spp == 4 else (abi.OUT_RGB_F32,):
                    frame = scene.render(Wf, Hf, spp, jit, precision=precision, out_format=fmt, seed=SEED, debug=True)
                    got = scene.shade_samples(rays, spp, sample_keys=keys, precision=precision, out_format=fmt, seed=SEED, debug=True)
                    _assert_same(frame, got, (name, spp, precision, fmt))


# ---- 2. depth of field ----------------------------------------------------------------------------------------------------------
def test_depth_of_field():
    spp = 5
    sc = parse(scenes.sample(res=(W, H), spp=spp, focus=True))
    assert sc.camera.has_focus
    jit = frontend.jitter_pattern(4, spp)
    with api.Scene(sc) as scene:
        r = _frame_and_samples(scene, sc, (0, 0, W, H), spp, jit, FP64, abi.OUT_RGB_F64)
        _assert_same(*r, what="depth of field FP64")
        frame, got = _frame_and_samples(scene, sc, (0, 0, W, H), spp, jit, FP32, abi.OUT_RGB_F64)
    c = parity.compare_window(frame["rgb"], frame["prim"].reshape(H, W, spp), got["rgb"].reshape(H, W, 3), got["prim"].reshape(H, W, spp),
                              ref_sub=frame["sub"].reshape(H, W, spp), got_sub=got["sub"].reshape(H, W, spp))
    print("depth of field FP32: within 1/255 %d of %d, prim mismatches %d (unexplained %d)" % (c["within"], c["pixels"], c["prim_mismatch"], c["prim_unexplained"]))
    assert c["within"] >= 0.999 * c["pixels"] and c["prim_unexplained"] == 0


# ---- 3. ftb_frame_rays against the oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("focus", [False, True])
@pytest.mark.parametrize("sampling", [abi.SAMPLING_JITTER, abi.SAMPLING_CORNER])
def test_frame_rays_against_the_oracle(focus, sampling):
    spp = 3 if sampling == abi.SAMPLING_JITTER else 1
    sc = parse(scenes.sample(res=(W, H), spp=spp, focus=focus))
    cam = sc.camera
    jit = frontend.jitter_pattern(2, spp) if sampling == abi.SAMPLING_JITTER else np.array([-0.5, 0.5])
    win = (7, 4, 30, 21)
    gw = W + 1 if sampling == abi.SAMPLING_CORNER else W
    x1, y1 = (win[2] + 1, win[3] + 1) if sampling == abi.SAMPLING_CORNER else win[2:]
    want_rays, want_keys = [], []
    for y in range(win[1], y1):
        for x in range(win[0], x1):
            for s in range(spp):
                key = (y * gw + x) * spp + s
                r = orc.primary_ray(cam, W, H, x, y, jit[2 * s], jit[2 * s + 1])
                if focus:
                    o, d = r[:3] + cam.focal_length * r[3:], r[3:]
                    d = orc.jitter_vector(SEED, key, 0, 0xFFFF, 0, cam.aperture_rad, d)
                    r = np.concatenate([o - cam.focal_length * d, d])
                want_rays.append(r)
                want_keys.append(key)
    want_rays, want_keys = np.array(want_rays), np.array(want_keys, dtype=np.uint64)
    with api.Scene(sc) as scene:
        for precision, bar in ((FP64, 1e-12), (FP32, 2e-6)):
            rays, keys = scene.frame_rays(win, W, H, spp, jit if sampling == abi.SAMPLING_JITTER else None, precision=precision, seed=SEED,
                                          sampling=sampling)
            assert np.array_equal(keys, want_keys)
            scale = np.maximum(np.abs(want_rays).max(axis=1, keepdims=True), 1.0)
            err = float((np.abs(rays - want_rays) / scale).max())
            print("precision %d, sampling %d, focus %s: %d rays, max error %.3g" % (precision, sampling, focus, len(rays), err))
            assert err <= bar
            if precision == FP32:
                assert np.array_equal(rays.astype(np.float32).astype(np.float64), rays)  # the kernel's FP32 values, widened


def test_path_query_reproduces_a_frame_window_bit_for_bit():
    """test_gpu_path_queries' reconstruction with the frame's own rays: bit-exact instead of within 1e-12."""
    Wf, Hf, spp = 40, 30, 4
    sc = parse(scenes.sample(res=(Wf, Hf), spp=spp, focus=False))
    jit = frontend.jitter_pattern(5, spp)
    win = (8, 6, 32, 26)
    with api.Scene(sc) as scene:
        frame = scene.render_window(win, Wf, Hf, spp, jit, debug=True, precision=FP64)
        rays, keys = scene.frame_rays(win, Wf, Hf, spp, jit, precision=FP64)
        got = scene.trace_paths(rays, sample_keys=keys, precision=FP64)
        assert np.array_equal(got["prim"][:, 0], frame["prim"]) and np.array_equal(got["sub"][:, 0], frame["sub"])
        col = got["colour"].reshape(-1, spp, 3)
        acc = np.zeros((col.shape[0], 3))
        for s in range(spp):
            acc = acc + col[:, s]
        assert np.array_equal(acc / spp, frame["rgb"].reshape(-1, 3))


# ---- 4. against ftb_shade_rays ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["bundled_sample", "bundled_house", "variant_0x74b", "large_shiny_blob"])
def test_against_shade_rays(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    rng = np.random.default_rng(5)
    with _open(sc) as scene:
        rays, _ = scene.frame_rays((0, 0, 24, 18), W, H, 6, frontend.jitter_pattern(6, 6), precision=FP64)
        rays = rays[rng.permutation(len(rays))]  # any rays: a re-ordered batch
        for spp in (1, 2, 3, 6, 129):
            rr = rays[:(len(rays) // spp) * spp]
            ref = scene.shade(rr, debug=True, precision=FP64, seed=SEED)
            got = scene.shade_samples(rr, spp, debug=True, precision=FP64, seed=SEED)
            col = ref["rgb"].reshape(-1, spp, 3)
            acc = np.zeros((col.shape[0], 3))
            for s in range(spp):
                acc = acc + col[:, s]
            assert np.array_equal(acc / spp, got["rgb"]), (case, spp)
            for k in ("prim", "sub", "t"):
                assert np.array_equal(ref[k], got[k]), (case, spp, k)
        for precision in (FP64, FP32):
            ref = scene.shade(rays, debug=True, precision=precision, seed=SEED)
            got = scene.shade_samples(rays, 1, debug=True, precision=precision, seed=SEED)
            assert np.array_equal(ref["rgb"], got["rgb"]), (case, precision)


# ---- 5. a custom camera ---------------------------------------------------------------------------------------------------------
def test_orthographic_camera_against_the_oracle():
    """A SamplingStrategy the library does not fuse: an orthographic camera with 4 jittered samples per pixel."""
    Wo, Ho, spp = 64, 48, 4
    sc = parse(scenes.hollow_sphere(res=(Wo, Ho), spp=1))
    rng = np.random.default_rng(9)
    jx, jy = rng.uniform(-0.5, 0.5, (2, Ho, Wo, spp))
    xs = ((np.arange(Wo)[None, :, None] + 0.5 + jx) / Wo - 0.5) * 8.0
    ys = (0.5 - (np.arange(Ho)[:, None, None] + 0.5 + jy) / Ho) * 6.0
    eye, fwd, right, up = np.array([0.0, 1.0, -12.0]), np.array([0.0, -0.05, 1.0]), np.array([1.0, 0.0, 0.0]), np.array([0.0, 1.0, 0.0])
    fwd = fwd / np.linalg.norm(fwd)
    up = np.cross(fwd, right)
    o = eye + xs[..., None] * right + ys[..., None] * up
    rays = np.concatenate([o, np.broadcast_to(fwd, o.shape)], axis=-1).reshape(-1, 6)
    ref = orc.shade_rays(sc, rays, orc.make_params(1, 1, 1, None, seed=SEED))
    want = ref["rgb"].reshape(-1, spp, 3).mean(axis=1)
    with api.Scene(sc) as scene:
        for precision, frac in ((FP64, 1.0), (FP32, 0.999)):
            got = scene.shade_samples(rays, spp, precision=precision, seed=SEED, debug=True)
            d = np.abs(got["rgb"] - want).max(axis=-1)
            share = float((d <= 1.0 / 255.0).mean())
            ids = int((got["prim"] != ref["prim"]).sum())
            print("orthographic precision %d: within 1/255 %.5f, prim mismatches %d of %d" % (precision, share, ids, len(rays)))
            assert share >= frac and float((got["prim"] >= 0).mean()) > 0.1
            assert ids <= (0 if precision == FP64 else 8)
        rgba = scene.shade_samples(rays, spp, precision=FP32, seed=SEED, out_format=abi.OUT_RGBA8)["rgb"]
        assert rgba.shape == (Wo * Ho, 4) and (rgba[:, 3] == 255).all()


# ---- 6. counters ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["house", "night_house", "repeat", "sample", "bunny"])
def test_counters_equal_the_frames(name):
    spp = 3
    sc = parse(getattr(scenes, name)(res=(W, H), spp=spp))
    jit = frontend.jitter_pattern(6, spp)
    with api.Scene(sc) as scene:
        for precision in (FP32, FP64):
            r = _frame_and_samples(scene, sc, (0, 0, W, H), spp, jit, precision, abi.OUT_RGB_F64, stats=True)
            frame, got = r
            fs, gs = frame["stats"], got["stats"]
            for k in ("primary_rays", "shadow_rays", "reflection_rays", "shaded_hits"):
                assert getattr(fs, k) == getattr(gs, k), (name, precision, k, getattr(fs, k), getattr(gs, k))
            print("%s precision %d: rays %d / %d shadow, bound tests frame %d samples %d, leaf tests frame %d samples %d"
                  % (name, precision, gs.primary_rays, gs.shadow_rays, fs.bound_tests, gs.bound_tests, sum(fs.leaf_tests), sum(gs.leaf_tests)))


# ---- 7. plumbing -------------------------------------------------------------------------------------------------------------------
def _hollow():
    return parse(scenes.hollow_sphere(res=(W, H), spp=1))


def test_zero_pixels_and_untouched_planes():
    sc = _hollow()
    with api.Scene(sc) as scene:
        got = scene.shade_samples(np.zeros((0, 6)), 3, debug=True, stats=True)
        assert got["rgb"].shape == (0, 3) and got["stats"].primary_rays == 0
        rays, keys = scene.frame_rays((0, 0, 8, 8), W, H, 2, frontend.jitter_pattern(1, 2))
        n = len(rays)
        prim = np.full(n, -7, dtype=np.int32)
        sub = np.full(n, -7, dtype=np.int32)
        t = np.full(n, -7.0)
        out = np.zeros((n // 2, 3))
        dp = C.POINTER(C.c_double)
        p = api.make_params(1, 1, 2, None, seed=SEED)
        for planes in ((prim, None, None), (None, sub, t)):
            dbg = abi.DebugOut(*[a.ctypes.data_as(C.POINTER(C.c_int32 if a.dtype == np.int32 else C.c_double)) if a is not None else None for a in planes])
            rc = api.lib().ftb_shade_samples(scene._h, rays.ctypes.data_as(dp), keys.ctypes.data_as(C.POINTER(C.c_uint64)), n // 2, C.byref(p),
                                             out.ctypes.data_as(C.c_void_p), C.byref(dbg), None)
            assert rc == 0
        assert (sub == -7).all() and (t == -7.0).all() and (prim >= -1).all()  # without prim_id no plane is written


def test_device_entries_on_a_side_stream_equal_the_host_entries(tmp_path):
    import torch
    sc = CASES["large_shiny_blob"](str(tmp_path))
    spp, win = 5, (3, 2, 29, 19)
    jit = frontend.jitter_pattern(8, spp)
    with api.Scene(sc) as scene:
        for precision in (FP64, FP32):
            for fmt in FORMATS:
                rays, keys = scene.frame_rays(win, W, H, spp, jit, precision=precision, seed=SEED)
                host = scene.shade_samples(rays, spp, sample_keys=keys, precision=precision, out_format=fmt, seed=SEED, debug=True)
                n, npix = len(rays), len(rays) // spp
                side = torch.cuda.Stream()
                d_rays = torch.full((n, 6), -1.0, dtype=torch.float64, device="cuda")
                d_keys = torch.zeros(n, dtype=torch.int64, device="cuda")
                dt, ch = api._OUT_DTYPE[fmt]
                d_out = torch.zeros(npix * ch * np.dtype(dt).itemsize, dtype=torch.uint8, device="cuda")
                d_prim = torch.full((n,), -3, dtype=torch.int32, device="cuda")
                d_sub = torch.full((n,), -3, dtype=torch.int32, device="cuda")
                d_t = torch.full((n,), -3.0, dtype=torch.float64, device="cuda")
                p = api.make_params(W, H, spp, jit, precision=precision, out_format=fmt, seed=SEED)
                torch.cuda.synchronize()
                with torch.cuda.stream(side):
                    scene.frame_rays_device(p, win, d_rays.data_ptr(), d_keys.data_ptr(), stream=side.cuda_stream)
                    scene.shade_samples_device(d_rays.data_ptr(), npix, p, d_out.data_ptr(), d_keys_ptr=d_keys.data_ptr(),
                                               d_dbg=(d_prim.data_ptr(), d_sub.data_ptr(), d_t.data_ptr()), stream=side.cuda_stream)
                side.synchronize()
                scene.check_overflow(stream=side.cuda_stream)
                assert np.array_equal(d_rays.cpu().numpy(), rays) and np.array_equal(d_keys.cpu().numpy().view(np.uint64), keys)
                assert np.array_equal(d_out.cpu().numpy().view(dt).reshape(npix, ch), host["rgb"]), (precision, fmt)
                for k, d in (("prim", d_prim), ("sub", d_sub), ("t", d_t)):
                    assert np.array_equal(d.cpu().numpy(), host[k]), (precision, fmt, k)


def test_hit_overflow_leaves_the_host_arrays_unwritten(tmp_path):
    row = vs.over_limit_scenes()[0]
    text, assets = row.text(str(tmp_path))
    sc = parse(text, assets=assets)
    with api.Scene(sc) as scene:
        rays, keys = scene.frame_rays((0, 0, 32, 24), 32, 24, 2, frontend.jitter_pattern(1, 2))
        for precision in (FP64, FP32):
            out = np.full((len(rays) // 2, 3), 5.0)
            prim = np.full(len(rays), 5, dtype=np.int32)
            dbg = abi.DebugOut(prim.ctypes.data_as(C.POINTER(C.c_int32)), None, None)
            p = api.make_params(1, 1, 2, None, precision=precision)
            rc = api.lib().ftb_shade_samples(scene._h, rays.ctypes.data_as(C.POINTER(C.c_double)), None, len(rays) // 2, C.byref(p),
                                             out.ctypes.data_as(C.c_void_p), C.byref(dbg), None)
            assert rc == abi.ERR_HIT_OVERFLOW and (out == 5.0).all() and (prim == 5).all(), (precision, rc)


def test_a_batch_past_2_to_the_24_samples_equals_smaller_batches():
    Wb, Hb, spp = 1024, 256, 72  # 18.9 M samples in one batch
    sc = parse(scenes.sample(res=(Wb, Hb), spp=1, focus=False))
    jit = frontend.jitter_pattern(3, spp)
    with api.Scene(sc) as scene:
        rays, keys = scene.frame_rays((0, 0, Wb, Hb), Wb, Hb, spp, jit, precision=FP32)
        assert len(rays) > (1 << 24)
        whole = scene.shade_samples(rays, spp, sample_keys=keys, precision=FP32)["rgb"]
        cut = np.concatenate([scene.shade_samples(rays[a * spp:b * spp], spp, sample_keys=keys[a * spp:b * spp], precision=FP32)["rgb"]
                              for a, b in ((0, 100000), (100000, 200001), (200001, Wb * Hb))])
        assert np.array_equal(whole, cut)
