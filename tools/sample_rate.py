#!/usr/bin/env python
"""A frame rendered two ways, device times side by side: the render kernel's own path (ftb_render_window_tiles_device) and the
frame's own samples on the explicit-ray path (ftb_frame_rays_device + ftb_shade_samples_device, include/functracer_b200.h).

Scenes: repeat, house and the full-size bunny mesh (cfg4-bunny-full-d14) at 1920x1080, 64 spp, FP32, seed 1234, the jitter
pattern of the config.  Everything device-resident; CUDA events around each path, after a warm-up of both, over at least a second
of work per path.  The explicit path traces what the frame skips (clear tiles, the shadow rays of lit ground tiles), has no
camera row in its common-origin bound table, and reads 56 bytes of ray and key per sample.  The two outputs (RGB F32) are asserted
bit-identical in the same run.  The GPU's name and power limit are printed with the numbers.

usage: python tools/sample_rate.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from query_rate import gpu_info  # noqa: E402

W, H, SPP = 1920, 1080, 64
CONFIGS = ("cfg5-repeat", "cfg3-house", "cfg4-bunny-full-d14")


def main():
    import numpy as np
    import torch
    from functracer_b200 import abi, api, frontend, scenes

    if not torch.cuda.is_available():
        raise SystemExit("sample_rate.py measures on the GPU; no CUDA device is visible")
    stream = torch.cuda.current_stream()
    name, power = gpu_info()
    print("GPU: %s, power limit %s; %dx%d, %d spp, FP32, RGB F32 output" % (name, power, W, H, SPP))

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize()
        reps = max(2, int(1000.0 / max(e0.elapsed_time(e1), 1e-3)) + 1)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, reps

    print("%-22s %12s %14s %14s %8s" % ("scene", "frame ms", "rays ms", "samples ms", "ratio"))
    for cfg in CONFIGS:
        sc = frontend.ParsedScene(scenes.config_text(cfg, res=(W, H), spp=SPP), scenes.asset_dir())
        jit = frontend.jitter_pattern(scenes.CONFIGS[cfg]["seed"], SPP)
        p = api.make_params(W, H, SPP, jit, precision=abi.PRECISION_FP32, out_format=abi.OUT_RGB_F32, seed=1234)
        n = W * H * SPP
        with api.Scene(sc) as scene:
            d_tiles = torch.empty(api.tile_buffer_bytes(p), dtype=torch.uint8, device="cuda")
            d_frame = torch.empty((H * W, 3), dtype=torch.float32, device="cuda")
            d_out = torch.full((H * W, 3), -1.0, dtype=torch.float32, device="cuda")
            d_rays = torch.empty((n, 6), dtype=torch.float64, device="cuda")
            d_keys = torch.empty(n, dtype=torch.int64, device="cuda")
            s = stream.cuda_stream

            def frame():
                scene.render_tiles_device(p, d_tiles.data_ptr(), stream=s)

            def rays():
                scene.frame_rays_device(p, (0, 0, W, H), d_rays.data_ptr(), d_keys.data_ptr(), stream=s)

            def samples():
                scene.shade_samples_device(d_rays.data_ptr(), W * H, p, d_out.data_ptr(), d_keys_ptr=d_keys.data_ptr(), stream=s)

            t_frame, r_frame = timed(frame)
            t_rays, r_rays = timed(rays)
            t_samples, r_samples = timed(samples)
            api.assemble_device(p, [d_tiles.data_ptr()], d_frame.data_ptr(), stream=s)
            torch.cuda.synchronize()
            scene.check_overflow(stream=s)
            a, b = d_frame.cpu().numpy(), d_out.cpu().numpy()
            assert np.array_equal(a, b), "%s: %d pixels differ" % (cfg, int((a != b).any(axis=1).sum()))
            ratio = (t_rays + t_samples) / t_frame
            print("%-22s %12.2f %14.2f %14.2f %7.2fx   (%d / %d / %d timed calls; outputs bit-identical)"
                  % (cfg, t_frame, t_rays, t_samples, ratio, r_frame, r_rays, r_samples))


if __name__ == "__main__":
    main()
