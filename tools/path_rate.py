#!/usr/bin/env python
"""Path-query throughput (ftb_trace_paths, include/functracer_b200.h) next to ftb_shade_rays on the same rays, in Mrays/s.

Cases: the camera rays of the repeat scene and of the full-size bunny mesh scene at 1920x1080, 1 spp (one ray through each pixel
centre), recursion limit 8.  Host entries, timed with the host clock around the synchronous call (uploads and downloads
included): ftb_shade_rays, and ftb_trace_paths with only `colour` requested.  Device entry (rays and planes device-resident,
CUDA events): ftb_trace_paths_device with only `colour` and with every plane.  Every case is warmed up, then timed over enough
calls for at least a second of work.  The GPU's name and power limit are printed with the numbers.

usage: python tools/path_rate.py [precision: fp32 | fp64]"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from query_rate import gpu_info  # noqa: E402

W, H = 1920, 1080
RL = 8


def main():
    import numpy as np
    import torch
    from functracer_b200 import abi, api, frontend, scenes
    from oracle import ftb_oracle as orc

    if not torch.cuda.is_available():
        raise SystemExit("path_rate.py measures on the GPU; no CUDA device is visible")
    precision = abi.PRECISION_FP64_VERIFY if (len(sys.argv) > 1 and sys.argv[1] == "fp64") else abi.PRECISION_FP32
    stream = torch.cuda.current_stream()
    name, power = gpu_info()
    print("GPU: %s, power limit %s, precision %s" % (name, power, "fp64" if precision == abi.PRECISION_FP64_VERIFY else "fp32"))

    def camera_rays(sc):
        """One ray through every pixel centre (the rays of three pixels extended over the grid, as query_rate.py does)."""
        r00, r10, r01 = (np.array(orc.primary_ray(sc.camera, W, H, x, y)) for x, y in ((0, 0), (1, 0), (0, 1)))
        ys, xs = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
        d = r00[3:] + xs.reshape(-1, 1) * (r10[3:] - r00[3:]) + ys.reshape(-1, 1) * (r01[3:] - r00[3:])
        return np.ascontiguousarray(np.hstack([np.broadcast_to(r00[:3], d.shape), d]))

    def timed_host(fn):
        fn(); fn()  # warm-up
        t0 = time.perf_counter(); fn(); one = time.perf_counter() - t0
        reps = max(1, int(1.0 / max(one, 1e-6)) + 1)  # >= 1 s of work
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) * 1e3 / reps, reps

    def timed_device(fn):
        fn(); fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize()
        reps = max(1, int(1000.0 / max(e0.elapsed_time(e1), 1e-3)) + 1)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, reps

    def report(label, entry, planes, n, ms, reps, levels):
        print(json.dumps(dict(case=label, entry=entry, planes=planes, rays=n, recursion_limit=RL, mean_levels=levels, ms=round(ms, 3),
                              mrays_per_s=round(n / ms / 1e3, 2), reps=reps, gpu=name, power_limit=power)), flush=True)

    for cfg, label in (("cfg5-repeat", "repeat %dx%d camera rays" % (W, H)), ("cfg4-bunny-full-d14", "full-size bunny %dx%d camera rays" % (W, H))):
        sc = frontend.ParsedScene(scenes.config_text(cfg, spp=1), scenes.asset_dir())
        rays = camera_rays(sc)
        n, L = rays.shape[0], sc.desc.n_lights
        with api.Scene(sc) as scene:
            lv = scene.trace_paths(rays, recursion_limit=RL, precision=precision, planes=("levels",))["levels"]
            levels = round(float(lv.mean()), 4)
            ms, reps = timed_host(lambda: scene.shade(rays, debug=False, recursion_limit=RL, precision=precision))
            report(label, "ftb_shade_rays", "rgb", n, ms, reps, levels)
            ms, reps = timed_host(lambda: scene.trace_paths(rays, recursion_limit=RL, precision=precision, planes=("colour",)))
            report(label, "ftb_trace_paths", "colour", n, ms, reps, levels)
            d_rays = torch.from_numpy(rays).cuda()
            dims = {"D": RL + 1, "L": L}
            for mode, which in (("colour", ("colour",)), ("every plane", tuple(api.PATH_PLANES))):
                bufs = {}
                for p in which:
                    _, dt, shape = api.PATH_PLANES[p]
                    bufs[p] = torch.empty((n,) + tuple(dims.get(k, k) for k in shape), dtype=torch.int32 if dt == np.int32 else torch.float64, device="cuda")
                ptrs = {p: v.data_ptr() for p, v in bufs.items()}
                ms, reps = timed_device(lambda: scene.trace_paths_device(d_rays.data_ptr(), n, ptrs, recursion_limit=RL, stream=stream.cuda_stream,
                                                                         precision=precision))
                scene.check_overflow(stream.cuda_stream)
                report(label, "ftb_trace_paths_device", mode, n, ms, reps, levels)
                del bufs
                torch.cuda.empty_cache()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
