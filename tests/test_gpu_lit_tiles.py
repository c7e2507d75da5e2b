"""Lit ground tiles on the device: the FP32 kernels give a primary ground fragment of a lit tile (lit_tiles.h) the intensity 1
for the proven directional lights without tracing their shadow rays.  The frames, primary-id and sub-id planes must agree
with the oracle at the usual bars, the counted shadow rays must still be the oracle's (the skipped rays are counted as
traced), and windows, bands and two shards must be bit-identical to the whole frame.  tests/test_lit_tiles_cpu.py checks
the proof itself; these scenes are checked there to have lit tiles."""
import numpy as np
import pytest

from functracer_b200 import abi, api, frontend, scenes
from oracle import ftb_oracle as orc
from test_gpu_window import assert_window_equals_whole, windows
from test_lit_tiles_cpu import HARD, _build, lit_mask
from util import parse

SEED = 21
W, H = 160, 120


def _scenes():
    out = {"cfg5-repeat": scenes.config_text("cfg5-repeat", res=(W, H), spp=2)}
    for k in ("penumbra", "camera-below", "tilted-ground", "wide-scatter", "corner-sampling"):
        out[k] = HARD[k].replace("res 160 120", "res %d %d" % (W, H))
    return out


SCENES = _scenes()


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return _build(str(tmp_path_factory.mktemp("lit_gpu_probe")), "tree")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCENES))
def test_lit_tiles_against_the_oracle(probe, name):
    sc = parse(SCENES[name])
    corner = sc.sampling == abi.SAMPLING_CORNER
    spp = 1 if corner else sc.spp
    jit = None if corner else frontend.jitter_pattern(5, spp)
    kw = dict(seed=SEED, precision=abi.PRECISION_FP32, sampling=sc.sampling)
    assert lit_mask(probe, sc, orc.make_params(W, H, spp, jit, sampling=sc.sampling, seed=SEED))[0].any()
    ref = orc.render(sc, orc.make_params(W, H, spp, jit, sampling=sc.sampling, seed=SEED))
    gw, gh = W + corner, H + corner
    rp, rs = ref["prim"].reshape(gh, gw, spp), ref["sub"].reshape(gh, gw, spp)
    with api.Scene(sc) as scene:
        counted = scene.render(W, H, spp, jit, stats=True, **kw)["stats"]
        got = scene.render(W, H, spp, jit, debug=True, out_format=abi.OUT_RGB_F64, **kw)
        prim, sub = (np.asarray(got[k]).reshape(gh, gw, spp) for k in ("prim", "sub"))
        miss = int((prim != rp).sum())
        assert miss <= 0.005 * prim.size, (name, miss)
        assert int(((prim == rp) & (sub != rs)).sum()) <= 0.005 * prim.size
        d = np.abs(got["rgb"] - ref["rgb"]).max(axis=-1)
        assert float((d <= 1.0 / 255.0).mean()) >= 0.999, name
        # every shaded sample casts the same shadow rays in both; a sample whose primary id differs may cast others
        per_sample = sum(l.samples if l.kind == abi.LIGHT_SOFT_DIRECTIONAL else 1 for l in (sc.desc.lights[k] for k in range(sc.desc.n_lights)))
        assert abs(int(counted.shadow_rays) - int(ref["stats"].shadow_rays)) <= miss * per_sample * 9, name
        if miss == 0:
            assert counted.shadow_rays == ref["stats"].shadow_rays
        for fmt in (abi.OUT_RGB_F32, abi.OUT_RGBA8):
            whole = scene.render(W, H, spp, jit, debug=True, out_format=fmt, **kw)
            for win in windows(W, H):
                assert_window_equals_whole(scene, whole, win, W, H, spp, jit, corner=corner, out_format=fmt, **kw)


@pytest.mark.gpu
def test_shards_and_bands_equal_the_whole_frame():
    """Two shards, rendered whole and band by band, read the window's one mask: both assemble to the host frame."""
    import torch
    spp = 2
    win = (7, 21, 151, 120)
    ww, wh = win[2] - win[0], win[3] - win[1]
    sc = parse(SCENES["cfg5-repeat"])
    jit = frontend.jitter_pattern(3, spp)
    s = torch.cuda.current_stream().cuda_stream
    with api.Scene(sc) as scene:
        host = scene.render_window(win, W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32)["rgb"]
        whole = scene.render(W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32)["rgb"]
        assert np.array_equal(host, whole[win[1]:win[3], win[0]:win[2]])
        for bands in (1, 4):
            bufs = []
            for k in range(2):
                p = api.make_params(W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, shard_index=k, shard_count=2)
                bufs.append(torch.zeros(api.tile_buffer_bytes(api.window_params(p, win)), dtype=torch.uint8, device="cuda"))
            frame = torch.zeros((wh, ww, 3), dtype=torch.float32, device="cuda")
            for c in range(bands):
                for k in range(2):
                    pk = api.make_params(W, H, spp, jit, seed=SEED, out_format=abi.OUT_RGB_F32, shard_index=k, shard_count=2,
                                         band_index=c, band_count=bands)
                    scene.render_window_tiles_device(pk, win, bufs[k].data_ptr(), stream=s)
                wp = api.window_params(pk, win)
                y0, y1 = api.band_rows(wp, c, bands) if bands > 1 else (0, wh)
                api.assemble_rows_device(wp, [b.data_ptr() for b in bufs], frame.data_ptr(), y0, y1, stream=s)
            torch.cuda.synchronize()
            scene.check_overflow(stream=s)
            assert np.array_equal(frame.cpu().numpy(), host), bands
