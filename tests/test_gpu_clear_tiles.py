"""Clear tiles on the device: tiles whose primary samples provably hit nothing (functracer_b200/csrc/cuda/tiles.h) are written
without tracing, by a kernel of their own.  Their pixels must be exactly what tracing gives (zero, folded over every pass), every
debug plane must hold a miss, the counted primary rays must still be every sample of the frame, and the rest of the frame
must agree with the oracle.  Windows, shards and bands of frames with clear tiles are compared bit for bit with the whole
frame by tests/test_gpu_window.py (its scenes have clear tiles: bunny 76 %, moon 33 % of the tiles at its sizes)."""
import numpy as np
import pytest

from functracer_b200 import abi, api, frontend
from oracle import ftb_oracle as orc
from test_gpu_window import assert_window_equals_whole, windows
from util import parse

W, H = 96, 80
# the horizon of the ground plane crosses the frame: sky above (clear tiles), the plane and a sphere below
SCENE = ("camera pos (0,0.5,-6) lookat (0,0.5,0) up (0,1,0) fov 55 ratio 1.2\nsamples %d\nres %d %d\n\n"
         "(translate (0,-2.2,0) plane)\n\n(translate (0.3,0,0.5) sphere)\n\ndirectional dir (0.3,-1,0.4) colour (1,1,1)\n"
         "positional pos (2,3,-2) falloff (1,0.02,0.01) colour (0.5,0.5,0.5)\n")
FORMATS = (abi.OUT_RGB_F64, abi.OUT_RGB_F32, abi.OUT_RGBA8)


SKY = slice(0, 16)  # the first tile row: clear (tests/test_clear_tiles_cpu.py checks the classification itself)


@pytest.mark.gpu
@pytest.mark.parametrize("spp", [3, 130])
def test_clear_tiles_against_the_oracle(spp):
    """130 samples take several passes (FP32: 128 + 2, FP64: 64 + 64 + 2): a clear pixel folds zero over each of them."""
    sc = parse(SCENE % (spp, W, H))
    jit = frontend.jitter_pattern(11, spp)
    ref = orc.render(sc, orc.make_params(W, H, spp, jit, seed=9))
    rp = ref["prim"].reshape(H, W, spp)
    assert (rp[SKY] == -1).all()  # the oracle sees sky there
    with api.Scene(sc) as scene:
        for prec in (abi.PRECISION_FP64_VERIFY, abi.PRECISION_FP32):
            for fmt in FORMATS:
                counted = scene.render(W, H, spp, jit, stats=True, seed=9, precision=prec, out_format=fmt)["stats"]
                assert counted.primary_rays == W * H * spp  # the clear tiles' samples count as primary rays
                got = scene.render(W, H, spp, jit, debug=True, seed=9, precision=prec, out_format=fmt)
                prim, sub, t = (np.asarray(got[k]).reshape(H, W, spp) for k in ("prim", "sub", "t"))
                assert (prim[SKY] == -1).all() and (sub[SKY] == 0).all() and (t[SKY] == -1.0).all()
                assert (got["rgb"][SKY][..., :3] == 0).all()
                assert int((prim != rp).sum()) <= 2, (prec, fmt)
                if fmt == abi.OUT_RGB_F64:
                    d = np.abs(got["rgb"] - ref["rgb"]).max(axis=-1)
                    bar = 1e-6 if prec == abi.PRECISION_FP64_VERIFY else 1.0 / 255.0
                    assert float((d <= bar).mean()) >= 0.999, (prec, spp)
                for win in windows(W, H):
                    assert_window_equals_whole(scene, got, win, W, H, spp, jit, seed=9, precision=prec, out_format=fmt)
