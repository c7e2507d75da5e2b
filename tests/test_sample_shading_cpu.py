"""CPU-side checks of a frame's own samples (ftb_frame_rays, ftb_shade_samples and their device forms): the prototypes in the
header and in abi.EXPORTS, the ctypes signatures, the argument checks that need no device (each made with a scene handle that is
never dereferenced), ftb_frame_rays' window checks against ftb_render_window's, and the flat pixel buffer of ftb_shade_samples as
the tile buffer of a 16-pixel-wide frame."""
import ctypes as C
import os
import re

import numpy as np

from functracer_b200 import abi, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "functracer_b200.h")
EXPORTS = {"ftb_frame_rays": 9, "ftb_frame_rays_device": 10, "ftb_shade_samples": 8, "ftb_shade_samples_device": 9}
RAY_LIMIT = 256 * 0x7fffff00 // 2  # ftb_shade_rays' ray limit (FTB_TILE_PIXELS * 0x7fffff00 / 2)
FAKE = C.c_void_p(0x10)  # never dereferenced by an argument check


def test_prototypes_are_declared_and_exported():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    protos = {m.group(1): m.group(2) for m in re.finditer(r"\b(ftb_[a-z_0-9]+)\s*\(([^)]*)\)\s*;", text)}
    for name, arity in EXPORTS.items():
        assert name in protos and name in abi.EXPORTS, name
        assert protos[name].count(",") + 1 == arity, name
    assert "uint64_t* sample_keys" in protos["ftb_frame_rays"] and "const uint64_t* sample_keys" in protos["ftb_shade_samples"]
    assert "int64_t n_pixels" in protos["ftb_shade_samples"] and "void* stream" in protos["ftb_shade_samples_device"]
    assert re.search(r"#define FTB_ABI_VERSION 4\b", text)  # additive: the ABI version stays
    assert len(abi.EXPORTS) == len(set(abi.EXPORTS)) == 30
    L = api.lib()
    for name, arity in EXPORTS.items():
        args = getattr(L, name).argtypes
        assert len(args) == arity and getattr(L, name).restype is C.c_int, name
    assert L.ftb_frame_rays.argtypes[3:7] == [C.c_int32] * 4 and L.ftb_frame_rays.argtypes[8] is C.POINTER(C.c_uint64)
    assert L.ftb_shade_samples.argtypes[2] is C.POINTER(C.c_uint64) and L.ftb_shade_samples.argtypes[3] is C.c_int64


def _samples(L, scene=FAKE, rays=np.zeros((8, 6)), keys=None, n=4, params=None, out=np.zeros((4, 3)), **pkw):
    """The host and the device entry with the same arguments."""
    p = params if params is not None else api.make_params(1, 1, pkw.pop("spp", 2), None, **pkw)
    r = rays.ctypes.data_as(C.POINTER(C.c_double)) if rays is not None else None
    k = keys.ctypes.data_as(C.POINTER(C.c_uint64)) if keys is not None else None
    o = out.ctypes.data_as(C.c_void_p) if out is not None else None
    pp = C.byref(p) if params is not False else None
    return (L.ftb_shade_samples(scene, r, k, n, pp, o, None, None), L.ftb_shade_samples_device(scene, r, k, n, pp, o, None, None, None))


def test_shade_samples_arguments_are_checked_before_any_device_is_needed():
    L = api.lib()
    bad = [dict(scene=None), dict(params=False), dict(n=-1), dict(rays=None), dict(out=None), dict(spp=0), dict(spp=-3),
           dict(precision=2), dict(precision=-1), dict(out_format=3), dict(out_format=-1),
           dict(n=1 << 62, spp=4),  # n_pixels * spp overflows int64
           dict(n=RAY_LIMIT // 256 + 1, spp=256),  # past ftb_shade_rays' ray limit
           dict(n=0x7fffff01, spp=1)]  # past the pixel limit
    for change in bad:
        assert _samples(L, **change) == (abi.ERR_BAD_ARG, abi.ERR_BAD_ARG), change
    empty = 0 if L.ftb_device_count() > 0 else abi.ERR_NO_DEVICE
    assert _samples(L, n=0, rays=None, out=None) == (empty, empty)
    assert _samples(L, n=0, sampling=7) == (empty, empty)  # sampling is not read
    if L.ftb_device_count() == 0:
        assert _samples(L, n=RAY_LIMIT // 256, spp=256) == (abi.ERR_NO_DEVICE, abi.ERR_NO_DEVICE)
        assert b"no CUDA device" in L.ftb_last_error()


def _frame_rays(L, window, scene=FAKE, camera=True, params=None, rays=True, keys=True):
    cam = C.byref(abi.Camera()) if camera else None
    buf = np.zeros((1, 6)), np.zeros(1, dtype=np.uint64)
    r = buf[0].ctypes.data_as(C.POINTER(C.c_double)) if rays else None
    k = buf[1].ctypes.data_as(C.POINTER(C.c_uint64)) if keys else None
    pp = C.byref(params) if params is not None else None
    return (L.ftb_frame_rays(scene, cam, pp, *window, r, k), L.ftb_frame_rays_device(scene, cam, pp, *window, r, k, None))


def test_frame_rays_checks_windows_as_render_window_does():
    """Every window and every params field ftb_frame_rays reads is refused exactly when ftb_render_window refuses it."""
    L = api.lib()
    jit = np.zeros(4)
    P = lambda **kw: api.make_params(20, 10, 2, jit, **kw)  # noqa: E731
    windows = [(0, 0, 20, 10), (3, 2, 4, 3), (-1, 0, 5, 5), (0, -1, 5, 5), (5, 0, 5, 5), (0, 5, 5, 5), (6, 0, 5, 5), (0, 0, 21, 10),
               (0, 0, 20, 11), (19, 9, 20, 10)]
    params = [P(), P(sampling=abi.SAMPLING_CORNER), P(sampling=5), P(precision=3), api.make_params(0, 10, 2, jit), api.make_params(20, 0, 2, jit),
              api.make_params(20, 10, 0, None), api.make_params(20, 10, 2, None), api.make_params(1 << 16, 1 << 15, 2, jit)]
    out = np.zeros(20 * 10 * 3)
    cam = abi.Camera()
    compared = 0
    for p in params:
        for w in windows:
            want = L.ftb_render_window(FAKE, C.byref(cam), C.byref(p), *w, out.ctypes.data_as(C.c_void_p), None, None)
            if want != abi.ERR_BAD_ARG and L.ftb_device_count() > 0:
                continue  # a valid call would look for the scene on the device
            assert _frame_rays(L, w, params=p) == (want, want), (w, p.width, p.height, p.spp, p.sampling, p.precision)
            compared += 1
    assert compared >= 40
    # fields ftb_frame_rays does not read are not checked
    for p in (P(out_format=9), P(shard_count=3, shard_index=5), P(band_count=99), P(n_gpus=64)):
        want = abi.ERR_NO_DEVICE if L.ftb_device_count() == 0 else None
        if want is not None:
            assert _frame_rays(L, (0, 0, 20, 10), params=p) == (want, want)
    for change in (dict(scene=None), dict(camera=False)):
        assert _frame_rays(L, (0, 0, 20, 10), params=P(), **change) == (abi.ERR_BAD_ARG, abi.ERR_BAD_ARG), change
    assert _frame_rays(L, (0, 0, 20, 10), params=None) == (abi.ERR_BAD_ARG, abi.ERR_BAD_ARG)
    if L.ftb_device_count() == 0:  # either output may be NULL
        assert _frame_rays(L, (0, 0, 20, 10), params=P(), rays=False, keys=False) == (abi.ERR_NO_DEVICE, abi.ERR_NO_DEVICE)


def test_flat_pixels_are_the_tile_buffer_of_a_16_wide_frame():
    """ftb_shade_samples writes pixel i at flat index i of a real buffer and assembles it as the frame of width 16 and ceil(n / 16)
    rows: the assembly reads pixel (x, y) from tile (y / 16) * tiles_x + x / 16 at (y % 16) * 16 + x % 16 (api.cu loadTilePixel),
    which for tiles_x = 1 is y * 16 + x = i, and the buffer that frame's tile_buffer_bytes sizes holds every row."""
    for n in (1, 15, 16, 17, 255, 256, 257, 1000, 4097, 123457):
        rows = (n + 15) // 16
        for precision, rs in ((abi.PRECISION_FP32, 4), (abi.PRECISION_FP64_VERIFY, 8)):
            p = api.make_params(16, rows, 1, np.zeros(2), precision=precision)
            assert api.tile_buffer_bytes(p) >= rows * 16 * 3 * rs
            assert api.tile_buffer_bytes(p) == -(-rows // 16) * 256 * 3 * rs
        assert api.band_rows(p, 0, 1) == (0, rows)
        i = np.arange(rows * 16)
        x, y = i % 16, i // 16
        tiles_x = (16 + 15) // 16
        slot = ((y // 16) * tiles_x + x // 16) * 256 + (y % 16) * 16 + (x % 16)
        assert tiles_x == 1 and np.array_equal(slot, i)
        # the kernel deals 32 pixels per queue block and writes block c's pixel j at 32 c + j (foldUnit with a block width of 32)
        c, j = i // 32, i % 32
        assert np.array_equal(32 * c + j, i)
