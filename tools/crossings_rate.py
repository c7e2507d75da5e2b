#!/usr/bin/env python
"""Crossing-query throughput (ftb_intersect_all_rays_device, include/functracer_b200.h) in Mrays/s: the counterpart of
tools/query_rate.py.

Cases: the camera rays of the repeat scene and of the full-size bunny mesh scene at 1920x1080, 1 spp (one ray through each pixel
centre).  Each case runs with max_hits = 8 and 64, as ids only (counts, t, prim, sub) and as full records (every plane), over the
whole list (t_min = -inf).  The frame is smaller than query_rate.py's: 64 full records per ray are 7.7 KB, 16 GB for two million
rays.  Rays and outputs are device-resident (torch tensors); every case is warmed up, then timed with CUDA events over enough
calls for at least a second of work.  The GPU's name and power limit are printed with the numbers.

usage: python tools/crossings_rate.py [precision: fp32 | fp64]"""
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from query_rate import gpu_info  # noqa: E402

W, H = 1920, 1080


def main():
    import torch
    from functracer_b200 import abi, api, frontend, scenes
    from oracle import ftb_oracle as orc

    if not torch.cuda.is_available():
        raise SystemExit("crossings_rate.py measures on the GPU; no CUDA device is visible")
    precision = abi.PRECISION_FP64_VERIFY if (len(sys.argv) > 1 and sys.argv[1] == "fp64") else abi.PRECISION_FP32
    stream = torch.cuda.current_stream()
    name, power = gpu_info()
    print("GPU: %s, power limit %s, precision %s" % (name, power, "fp64" if precision == abi.PRECISION_FP64_VERIFY else "fp32"))

    def camera_rays(sc):
        """One ray through every pixel centre, built on the device from the rays of three pixels (as query_rate.py does)."""
        r00, r10, r01 = (orc.primary_ray(sc.camera, W, H, x, y) for x, y in ((0, 0), (1, 0), (0, 1)))
        d00, dx, dy = (torch.tensor(v, dtype=torch.float64, device="cuda") for v in (r00[3:], r10[3:] - r00[3:], r01[3:] - r00[3:]))
        ys, xs = torch.meshgrid(torch.arange(H, device="cuda", dtype=torch.float64), torch.arange(W, device="cuda", dtype=torch.float64), indexing="ij")
        d = d00 + xs.reshape(-1, 1) * dx + ys.reshape(-1, 1) * dy
        o = torch.tensor(r00[:3], dtype=torch.float64, device="cuda").expand(d.shape[0], 3)
        return torch.cat([o, d], dim=1).contiguous()

    def timed(fn):
        fn(); fn()  # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize()
        reps = max(1, int(1000.0 / max(e0.elapsed_time(e1), 1e-3)) + 1)  # >= 1 s of work
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, reps

    def run(scene, label, rays):
        n = rays.shape[0]
        counts = torch.empty(n, dtype=torch.int32, device="cuda")
        s = stream.cuda_stream
        for k in (8, 64):
            w = dict(t=(), prim=(), sub=(), p=(3,), normal=(3,), colour=(3,), surface=(4,))
            for mode, which in (("ids", ("t", "prim", "sub")), ("records", api.HIT_PLANES)):
                planes = {p: torch.empty((n, k) + w[p], dtype=torch.int32 if p in ("prim", "sub") else torch.float64, device="cuda") for p in which}
                ptrs = {p: v.data_ptr() for p, v in planes.items()}
                ms, reps = timed(lambda: scene.intersect_all_device(rays.data_ptr(), n, k, counts.data_ptr(), ptrs, t_min=-math.inf, stream=s,
                                                                    precision=precision))
                scene.check_overflow(s)
                c = counts.to(torch.int64)
                r = dict(case=label, max_hits=k, mode=mode, rays=n, crossings_per_ray=round(float(c.float().mean()), 3), rays_over_max_hits=int((c > k).sum()),
                         ms=round(ms, 3), mrays_per_s=round(n / ms / 1e3, 1), reps=reps, gpu=name, power_limit=power)
                print(json.dumps(r), flush=True)
                del planes
                torch.cuda.empty_cache()

    for cfg, label in (("cfg5-repeat", "repeat %dx%d camera rays" % (W, H)), ("cfg4-bunny-full-d14", "full-size bunny %dx%d camera rays" % (W, H))):
        sc = frontend.ParsedScene(scenes.config_text(cfg, spp=1), scenes.asset_dir())
        with api.Scene(sc) as scene:
            run(scene, label, camera_rays(sc))
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
