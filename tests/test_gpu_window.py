"""Window renders (ftb_render_window, ftb_render_window_tiles_device): the pixel rectangle [x0, x1) x [y0, y1) of a frame,
with outputs packed to the window, must equal the same pixels and debug-plane entries of the whole-frame render BIT FOR
BIT - every pixel's rays, RNG keys and blend order are the whole frame's (Shading.fs:141-147: pixels are independent).
Every comparison here is exact against the same call over the whole frame, except the full-size primitive-id planes,
which are checked against the CPU oracle with the bars of test_gpu_fullsize.py.  Needs a B200: run with `-m gpu`."""
import ctypes as C

import numpy as np
import pytest

from functracer_b200 import abi, api, frontend, scenes
from oracle import ftb_oracle as orc
from oracle import parity
from util import one_object_scene, parse

pytestmark = pytest.mark.gpu
SEED = 1234
W, H = 72, 56
FORMATS = (abi.OUT_RGB_F64, abi.OUT_RGB_F32, abi.OUT_RGBA8)
PRECISIONS = (abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY)


def windows(w, h):
    """The whole frame, 1x1 inside and at the last pixel, an 8-px full-height stripe at an x off the 16-px tile grid, 17x33 at
    an odd origin, a window of <= 16 columns (one tile column: the work queue's divide path) and exactly one aligned tile."""
    return [(0, 0, w, h), (w // 2 + 3, h // 3, w // 2 + 4, h // 3 + 1), (w - 1, h - 1, w, h), (21, 0, 29, h), (13, 7, 30, 40),
            (37, 5, 50, h - 3), (16, 16, 32, 32)]


def planes(res, shape):
    """The debug planes of a render as [rows, cols, samples] arrays."""
    return [np.asarray(res[k]).reshape(shape) for k in ("prim", "sub", "t")]


def assert_window_equals_whole(scene, whole, win, width, height, spp, jit, corner=False, **kw):
    """Renders `win` and compares it with `whole` (the whole-frame render of the same request, with debug planes)."""
    x0, y0, x1, y1 = win
    got = scene.render_window(win, width, height, spp, jit, debug=True, **kw)
    assert got["rgb"].shape[:2] == (y1 - y0, x1 - x0)
    assert np.array_equal(got["rgb"], whole["rgb"][y0:y1, x0:x1], equal_nan=True), win
    e = 1 if corner else 0  # corner sampling: the window's sample grid is the corners [x0, x1] x [y0, y1]
    s = 1 if corner else spp
    for a, b in zip(planes(got, (y1 - y0 + e, x1 - x0 + e, s)), planes(whole, (height + e, width + e, s))):
        assert np.array_equal(a, b[y0:y1 + e, x0:x1 + e], equal_nan=True), win
    return got


SMALL = ["cfg1-sample", "cfg2-hollow-sphere", "cfg3-house", "cfg5-moon", "cfg4-bunny", "cfg4-bunny-full-d14"]


@pytest.mark.parametrize("name", SMALL)
def test_windows_are_bit_identical_to_the_whole_frame(name):
    """cfg1-sample (depth of field, soft lights, an image texture) is the scene whose pixels depend on the RNG key of every
    sample; hollow-sphere has CSG pairs, house FT_PAIRG, moon Oren-Nayar and a texture, bunny the per-lane mesh walk and
    bunny-full-d14 the warp-packet walk over a device-built index."""
    spp = 2
    sc = parse(scenes.config_text(name, res=(W, H), spp=spp))
    jit = frontend.jitter_pattern(scenes.CONFIGS[name]["seed"], spp)
    with api.Scene(sc) as scene:
        for prec in PRECISIONS:
            for fmt in FORMATS:
                kw = dict(seed=SEED, precision=prec, out_format=fmt)
                whole = scene.render(W, H, spp, jit, debug=True, **kw)
                assert (whole["prim"] != -2).all()
                for win in windows(W, H):
                    assert_window_equals_whole(scene, whole, win, W, H, spp, jit, **kw)


@pytest.mark.parametrize("spp", [3, 130])
def test_window_sample_counts_and_multi_pass_blend(spp):
    """130 samples per pixel take more than one pass per launch (FP32: two of <= 128, FP64: three of <= 64); each pass
    continues the fold of the one before (s_base > 0), in a window as in the whole frame."""
    w, h = 40, 34
    sc = parse(scenes.house(res=(w, h), spp=spp))
    jit = frontend.jitter_pattern(7, spp)
    with api.Scene(sc) as scene:
        for prec in PRECISIONS:
            kw = dict(seed=SEED, precision=prec, out_format=abi.OUT_RGB_F64)
            whole = scene.render(w, h, spp, jit, debug=True, **kw)
            for win in [(0, 0, w, h), (3, 1, 4, 2), (11, 2, 30, 33), (17, 0, 25, h)]:
                assert_window_equals_whole(scene, whole, win, w, h, spp, jit, **kw)


def test_corner_sampling_windows():
    """Corner sampling (CornerSampling.blendPixels, Image.fs:134-144): a window's pixels average the corners [x0, x1] x
    [y0, y1] of the frame's corner grid, and its planes hold (w + 1) x (h + 1) entries."""
    sc = parse(scenes.hollow_sphere(res=(W, H), spp=1).replace("samples 1", "samples corner"))
    assert sc.sampling == abi.SAMPLING_CORNER
    with api.Scene(sc) as scene:
        for prec in PRECISIONS:
            for fmt in FORMATS:
                kw = dict(seed=SEED, precision=prec, out_format=fmt, sampling=abi.SAMPLING_CORNER)
                whole = scene.render(W, H, 1, None, debug=True, **kw)
                for win in windows(W, H):
                    assert_window_equals_whole(scene, whole, win, W, H, 1, None, corner=True, **kw)


def test_device_window_entry_with_shards_and_bands():
    """ftb_render_window_tiles_device renders the window's tiles into the tile buffer of a window-sized frame: two shards
    assembled with window_params equal the host window; so do two shards rendered band by band (band_count = 4), each band
    assembled over the rows ftb_band_rows gives for the window params."""
    import torch
    w, h, spp = 200, 150, 2
    win = (23, 9, 171, 140)  # 148 x 131 px: 9 tile rows, so four bands
    ww, wh = win[2] - win[0], win[3] - win[1]
    sc = parse(scenes.night_house(res=(w, h), spp=spp))
    jit = frontend.jitter_pattern(3, spp)
    s = torch.cuda.current_stream().cuda_stream
    with api.Scene(sc) as scene:
        host = scene.render_window(win, w, h, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32)["rgb"]
        bufs = []
        for k in range(2):
            p = api.make_params(w, h, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, shard_index=k, shard_count=2)
            bufs.append(torch.zeros(api.tile_buffer_bytes(api.window_params(p, win)), dtype=torch.uint8, device="cuda"))
            scene.render_window_tiles_device(p, win, bufs[k].data_ptr(), stream=s)
        frame = torch.zeros((wh, ww, 3), dtype=torch.float32, device="cuda")
        api.assemble_device(api.window_params(p, win), [b.data_ptr() for b in bufs], frame.data_ptr(), stream=s)
        torch.cuda.synchronize()
        scene.check_overflow(stream=s)
        assert np.array_equal(frame.cpu().numpy(), host)
        for b in bufs:
            b.zero_()
        frame.zero_()
        rows = []
        for c in range(4):
            for k in range(2):
                pk = api.make_params(w, h, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, shard_index=k, shard_count=2, band_index=c, band_count=4)
                scene.render_window_tiles_device(pk, win, bufs[k].data_ptr(), stream=s)
            wp = api.window_params(pk, win)
            y0, y1 = api.band_rows(wp, c, 4)
            rows.append((y0, y1))
            api.assemble_rows_device(wp, [b.data_ptr() for b in bufs], frame.data_ptr(), y0, y1, stream=s)
        torch.cuda.synchronize()
        scene.check_overflow(stream=s)
    assert rows[0][0] == 0 and rows[-1][1] == wh and all(a[1] == b[0] for a, b in zip(rows, rows[1:]))
    assert all(y1 > y0 for y0, y1 in rows)
    assert np.array_equal(frame.cpu().numpy(), host)


def test_device_window_debug_planes():
    """The device entry's debug planes are window-sized and equal the matching entries of the host whole-frame planes."""
    import torch
    spp = 2
    sc = parse(scenes.sample(res=(W, H), spp=spp))
    jit = frontend.jitter_pattern(1, spp)
    win = (13, 7, 30, 40)
    ww, wh = win[2] - win[0], win[3] - win[1]
    s = torch.cuda.current_stream().cuda_stream
    with api.Scene(sc) as scene:
        whole = scene.render(W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, debug=True)
        p = api.make_params(W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32)
        buf = torch.zeros(api.tile_buffer_bytes(api.window_params(p, win)), dtype=torch.uint8, device="cuda")
        prim = torch.full((wh, ww, spp), -2, dtype=torch.int32, device="cuda")
        sub = torch.full((wh, ww, spp), -2, dtype=torch.int32, device="cuda")
        t = torch.zeros((wh, ww, spp), dtype=torch.float64, device="cuda")
        scene.render_window_tiles_device(p, win, buf.data_ptr(), stream=s, d_dbg=(prim.data_ptr(), sub.data_ptr(), t.data_ptr()))
        frame = torch.zeros((wh, ww, 3), dtype=torch.float32, device="cuda")
        api.assemble_device(api.window_params(p, win), [buf.data_ptr()], frame.data_ptr(), stream=s)
        torch.cuda.synchronize()
    x0, y0, x1, y1 = win
    assert np.array_equal(frame.cpu().numpy(), whole["rgb"][y0:y1, x0:x1])
    for a, b in zip((prim, sub, t), planes(whole, (H, W, spp))):
        assert np.array_equal(a.cpu().numpy(), b[y0:y1, x0:x1])


def test_two_gpu_window_equals_one_gpu():
    if api.device_count() < 2:
        pytest.skip("needs two GPUs")
    w, h, spp = 320, 200, 2
    sc = parse(scenes.hollow_sphere(res=(w, h), spp=spp))
    jit = frontend.jitter_pattern(2, spp)
    with api.Scene(sc) as scene:
        for win in [(0, 0, w, h), (37, 21, 250, 190), (100, 0, 108, h)]:
            one = scene.render_window(win, w, h, spp, jit, out_format=abi.OUT_RGB_F32)["rgb"]
            two = scene.render_window(win, w, h, spp, jit, out_format=abi.OUT_RGB_F32, n_gpus=2)["rgb"]
            assert np.array_equal(two, one), win


def test_tile_order_cache_follows_the_window():
    """The cached tile order lists the local tiles of the window it was computed for.  Whole frame (four download bands),
    window A, window B, whole frame again on one scene: each equals a fresh scene's render of the same request."""
    w, h, spp = 640, 528, 1
    text = scenes.night_house(res=(w, h), spp=spp)
    jit = frontend.jitter_pattern(3, spp)
    reqs = [(0, 0, w, h), (100, 60, 420, 300), (5, 200, 77, 528), (0, 0, w, h)]
    kw = dict(seed=SEED, out_format=abi.OUT_RGBA8)
    with api.Scene(parse(text)) as scene:
        seq = [scene.render_window(win, w, h, spp, jit, **kw)["rgb"].copy() for win in reqs]
    for win, got in zip(reqs, seq):
        with api.Scene(parse(text)) as fresh:
            assert np.array_equal(got, fresh.render_window(win, w, h, spp, jit, **kw)["rgb"]), win


def test_window_ray_counts():
    """A window traces w * h * spp primary rays; four windows that tile the frame trace, between them, the whole frame's
    primary, shadow and reflection rays and shade its hits (counts that do not depend on how samples are dealt)."""
    w, h, spp = 96, 54, 2
    sc = parse(scenes.hollow_sphere(res=(w, h), spp=spp))
    jit = frontend.jitter_pattern(2, spp)
    keys = ("primary_rays", "shadow_rays", "reflection_rays", "shaded_hits")
    with api.Scene(sc) as scene:
        for prec in PRECISIONS:
            whole = scene.render(w, h, spp, jit, precision=prec, stats=True)["stats"]
            quads = [(0, 0, 37, 20), (37, 0, w, 20), (0, 20, 61, h), (61, 20, w, h)]
            tot = dict.fromkeys(keys, 0)
            for x0, y0, x1, y1 in quads:
                st = scene.render_window((x0, y0, x1, y1), w, h, spp, jit, precision=prec, stats=True)["stats"]
                assert st.primary_rays == (x1 - x0) * (y1 - y0) * spp
                for k in keys:
                    tot[k] += getattr(st, k)
            assert whole.primary_rays == w * h * spp
            assert tot == {k: getattr(whole, k) for k in keys}


def test_bad_windows_are_rejected():
    import torch
    sc = parse(scenes.hollow_sphere(res=(32, 24), spp=1))
    jit = [0.0, 0.0]
    p = api.make_params(32, 24, 1, jit, out_format=abi.OUT_RGB_F32)
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    with api.Scene(sc) as scene:
        out = np.zeros((24, 32, 3), dtype=np.float32)
        for win in [(-1, 0, 4, 4), (0, -1, 4, 4), (0, 0, 33, 24), (0, 0, 32, 25), (5, 5, 5, 9), (5, 5, 9, 5), (6, 0, 4, 4)]:
            rc = api.lib().ftb_render_window(scene._h, sc.camera_ptr, C.byref(p), *win, out.ctypes.data_as(C.c_void_p), None, None)
            assert rc == abi.ERR_BAD_ARG, win
            with pytest.raises(api.FtbError) as e:
                scene.render_window_tiles_device(p, win, buf.data_ptr())
            assert e.value.status == abi.ERR_BAD_ARG, win


def test_hit_overflow_is_reported_by_the_window_entries():
    """The overflow scene of test_gpu_parity.py: the host window entry reports it itself, the device one through
    ftb_check_overflow."""
    import torch
    col = lambda z0: " ".join("(translate (0,0,%g) sphere)" % (z0 + 0.1 * i) for i in range(10))
    sc = parse(one_object_scene("(union (group %s) (group %s))" % (col(0.0), col(1.0)), "directional dir (0,-1,1) colour 1"))
    s = torch.cuda.current_stream().cuda_stream
    with api.Scene(sc) as scene:
        with pytest.raises(api.FtbError) as e:
            scene.render_window((4, 4, 12, 12), 16, 16, 1, [0.0, 0.0])
        assert e.value.status == abi.ERR_HIT_OVERFLOW
        p = api.make_params(32, 32, 1, [0.0, 0.0], out_format=abi.OUT_RGB_F32)
        win = (8, 8, 24, 24)
        buf = torch.zeros(api.tile_buffer_bytes(api.window_params(p, win)), dtype=torch.uint8, device="cuda")
        scene.render_window_tiles_device(p, win, buf.data_ptr(), stream=s)
        with pytest.raises(api.FtbError) as e:
            scene.check_overflow(stream=s)
        assert e.value.status == abi.ERR_HIT_OVERFLOW


def test_full_size_stripes_and_probe():
    """cfg5-repeat at its full 7680 x 4320 x 64 spp: eight full-height stripes (8 px + one column of context either side)
    and a one-pixel probe, each with window-sized debug planes (a whole-frame prim plane alone would be 8.5 GB).  Colours
    equal the whole-frame f32 render bit for bit; the prim / sub planes meet test_gpu_fullsize.py's bars against the
    oracle; the probe's planes equal its stripe's."""
    import torch
    name = "cfg5-repeat"
    cfg = scenes.CONFIGS[name]
    sc = frontend.ParsedScene(scenes.config_text(name), scenes.asset_dir())
    w, h, spp = sc.width, sc.height, sc.spp
    assert (w, h, spp) == (7680, 4320, 64)
    jit = frontend.jitter_pattern(cfg["seed"], spp)
    s = torch.cuda.current_stream().cuda_stream
    margin = 1
    stripes = parity.stripe_windows(w, h, 8, 8, margin)
    sx0 = stripes[3][0]
    probe = (sx0 + 4, 2161, sx0 + 5, 2162)
    with api.Scene(sc) as scene:
        p = api.make_params(w, h, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32)
        tiles = torch.empty(api.tile_buffer_bytes(p), dtype=torch.uint8, device="cuda")
        scene.render_tiles_device(p, tiles.data_ptr(), stream=s)
        frame = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        api.assemble_device(p, [tiles.data_ptr()], frame.data_ptr(), stream=s)
        torch.cuda.synchronize()
        scene.check_overflow(stream=s)
        del tiles
        got = [scene.render_window(win, w, h, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, debug=True) for win in stripes + [probe]]
    frame = frame.cpu().numpy()
    for win, g in zip(stripes + [probe], got):
        x0, y0, x1, y1 = win
        assert np.array_equal(g["rgb"], frame[y0:y1, x0:x1]), win
    pr = [a.reshape(spp) for a in planes(got[-1], (1, 1, spp))]
    for a, b in zip(pr, planes(got[3], (h, stripes[3][2] - sx0, spp))):
        assert np.array_equal(a, b[probe[1], probe[0] - sx0], equal_nan=True)
    op = orc.make_params(w, h, spp, jit, seed=SEED)
    res = orc.render_windows(sc, op, stripes, debug=True)
    parts = []
    for ref, g in zip(res["windows"], got):
        x0, y0, x1, y1 = ref["rect"]
        gp, gs, _ = planes(g, (y1 - y0, x1 - x0, spp))
        parts.append(parity.compare_window(ref["rgb"], ref["prim"], g["rgb"], gp, margin, ref_sub=ref["sub"], got_sub=gs))
    m = parity.merge(parts)
    print("%s windows: %d samples, prim mismatches %d (unexplained %d), sub mismatches %d, colour within 1/255 on %.5f"
          % (name, m["samples"], m["prim_mismatch"], m["prim_unexplained"], m.get("sub_mismatch", 0), m["frac_within_1_255"]))
    assert m["nonfinite"] == 0
    assert m["frac_within_1_255"] >= 0.999
    assert m["prim_mismatch"] <= 2e-3 * m["samples"]
    assert m["prim_unexplained"] == 0, m.get("unexplained_samples")
    assert m.get("sub_mismatch", 0) <= 5e-3 * m["samples"]
