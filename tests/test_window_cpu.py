"""The host-side arithmetic of window renders, which needs no GPU: window_params is the params copy with the window's size,
and the tile buffer and bands of a window are those of a frame of that size.  CPU only."""
from functracer_b200 import abi, api


def test_window_params_is_a_window_sized_copy():
    p = api.make_params(7680, 4320, 4, [0.1, -0.2, 0.3, 0.0, -0.4, 0.25, 0.0, 0.5], seed=99, out_format=abi.OUT_RGBA8,
                        shard_index=1, shard_count=3, band_index=2, band_count=4, precision=abi.PRECISION_FP64_VERIFY)
    q = api.window_params(p, (100, 7, 164, 4320))
    assert (q.width, q.height) == (64, 4313)
    assert (p.width, p.height) == (7680, 4320)  # the original is untouched
    for f, _ in abi.RenderParams._fields_:
        if f not in ("width", "height", "jitter_xy"):
            assert getattr(q, f) == getattr(p, f), f
    assert [q.jitter_xy[i] for i in range(8)] == [p.jitter_xy[i] for i in range(8)]


def test_window_buffer_and_bands_are_those_of_a_window_sized_frame():
    jit = [0.0, 0.0]
    for sampling in (abi.SAMPLING_JITTER, abi.SAMPLING_CORNER):
        p = api.make_params(1920, 1080, 1, jit, sampling=sampling, out_format=abi.OUT_RGB_F32, shard_count=2)
        for win in [(0, 0, 1920, 1080), (17, 33, 34, 66), (5, 0, 13, 1080), (1919, 1079, 1920, 1080)]:
            q = api.window_params(p, win)
            frame = api.make_params(win[2] - win[0], win[3] - win[1], 1, jit, sampling=sampling, out_format=abi.OUT_RGB_F32, shard_count=2)
            assert api.tile_buffer_bytes(q) == api.tile_buffer_bytes(frame)
            if sampling == abi.SAMPLING_JITTER:
                assert [api.band_rows(q, c, 4) for c in range(4)] == [api.band_rows(frame, c, 4) for c in range(4)]
