#!/usr/bin/env python
"""Ray-query throughput (ftb_intersect_rays_device, ftb_occluded_rays_device, include/functracer_b200.h) in Mrays/s.

Cases: the camera rays of the repeat scene at 7680x4320, 1 spp (one ray through each pixel centre); random rays from points in
the box of what that camera sees; shadow rays from those camera rays' hit points (offset by 1e-4 n, as Shading.fs does)
towards each of its lights; the camera rays of the full-size bunny mesh scene at 3840x2160.  Each case runs as ids-only
queries (t, prim, sub), as full records (every plane) and as occlusion queries (max_t = +inf, the light's distance for the
shadow rays).  Rays and outputs are device-resident (torch tensors); every case is warmed up, then timed with CUDA events over
enough calls for at least a second of work.  The GPU's name and power limit are printed with the numbers.

usage: python tools/query_rate.py [precision: fp32 | fp64]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return "unknown", "unknown"


def main():
    import torch
    from functracer_b200 import abi, api, frontend, scenes

    if not torch.cuda.is_available():
        raise SystemExit("query_rate.py measures on the GPU; no CUDA device is visible")
    precision = abi.PRECISION_FP64_VERIFY if (len(sys.argv) > 1 and sys.argv[1] == "fp64") else abi.PRECISION_FP32
    stream = torch.cuda.current_stream()
    name, power = gpu_info()
    print("GPU: %s, power limit %s, precision %s" % (name, power, "fp64" if precision == abi.PRECISION_FP64_VERIFY else "fp32"))

    def camera_rays(sc, W, H):
        """One ray through every pixel centre: the image plane is planar, so the direction is linear in (x, y); built on the
        device from the rays of three pixels as Image.fs builds them (the oracle's rayThroughPixel)."""
        from oracle import ftb_oracle as orc
        r00, r10, r01 = (orc.primary_ray(sc.camera, W, H, x, y) for x, y in ((0, 0), (1, 0), (0, 1)))
        d00, dx, dy = (torch.tensor(v, dtype=torch.float64, device="cuda") for v in (r00[3:], r10[3:] - r00[3:], r01[3:] - r00[3:]))
        ys, xs = torch.meshgrid(torch.arange(H, device="cuda", dtype=torch.float64), torch.arange(W, device="cuda", dtype=torch.float64), indexing="ij")
        d = d00 + xs.reshape(-1, 1) * dx + ys.reshape(-1, 1) * dy
        o = torch.tensor(r00[:3], dtype=torch.float64, device="cuda").expand(d.shape[0], 3)
        return torch.cat([o, d], dim=1).contiguous()

    def planes_for(n, which):
        w = dict(t=1, prim=1, sub=1, p=3, normal=3, colour=3, surface=4)
        return {k: torch.empty((n, w[k]), dtype=torch.int32 if k in ("prim", "sub") else torch.float64, device="cuda") for k in which}

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

    def run(scene, label, rays, max_t):
        n = rays.shape[0]
        ids, full = planes_for(n, ("t", "prim", "sub")), planes_for(n, api.HIT_PLANES)
        blocked = torch.empty(n, dtype=torch.int32, device="cuda")
        s = stream.cuda_stream
        modes = [("ids", lambda: scene.intersect_device(rays.data_ptr(), n, {k: v.data_ptr() for k, v in ids.items()}, stream=s, precision=precision)),
                 ("records", lambda: scene.intersect_device(rays.data_ptr(), n, {k: v.data_ptr() for k, v in full.items()}, stream=s, precision=precision)),
                 ("occlusion", lambda: scene.occluded_device(rays.data_ptr(), max_t.data_ptr(), n, blocked.data_ptr(), stream=s, precision=precision))]
        for mode, fn in modes:
            ms, reps = timed(fn)
            scene.check_overflow(s)
            r = dict(case=label, mode=mode, rays=n, ms=round(ms, 3), mrays_per_s=round(n / ms / 1e3, 1), reps=reps, gpu=name, power_limit=power)
            print(json.dumps(r), flush=True)
        return full

    # repeat, 7680 x 4320
    sc = frontend.ParsedScene(scenes.config_text("cfg5-repeat", spp=1), scenes.asset_dir())
    with api.Scene(sc) as scene:
        cam = camera_rays(sc, 7680, 4320)
        n = cam.shape[0]
        full = run(scene, "repeat 7680x4320 camera rays", cam, torch.full((n,), float("inf"), dtype=torch.float64, device="cuda"))
        hit = full["prim"][:, 0] >= 0
        p, nrm = full["p"][hit], full["normal"][hit]
        lo, hi = torch.quantile(p[::97], 0.02, dim=0), torch.quantile(p[::97], 0.98, dim=0)
        g = torch.Generator(device="cuda").manual_seed(1)
        o = lo + (hi - lo) * torch.rand((n, 3), generator=g, dtype=torch.float64, device="cuda")
        d = torch.randn((n, 3), generator=g, dtype=torch.float64, device="cuda")
        rnd = torch.cat([o, d / d.norm(dim=1, keepdim=True)], dim=1).contiguous()
        run(scene, "repeat random rays in its box", rnd, torch.full((n,), float("inf"), dtype=torch.float64, device="cuda"))
        origin = p + 1e-4 * nrm
        srays, smax = [], []
        for i in range(sc.desc.n_lights):
            L = sc.desc.lights[i]
            v = torch.tensor(L.v[:], dtype=torch.float64, device="cuda")
            if L.kind == abi.LIGHT_POINT:
                dv = v - origin
                dist = dv.norm(dim=1)
                srays.append(torch.cat([origin, dv / dist[:, None]], dim=1)); smax.append(dist)
            else:
                srays.append(torch.cat([origin, (-v).expand_as(origin)], dim=1)); smax.append(torch.full((origin.shape[0],), float("inf"), dtype=torch.float64, device="cuda"))
        del full, cam, rnd
        run(scene, "repeat shadow rays towards its lights", torch.cat(srays).contiguous(), torch.cat(smax).contiguous())
    # full-size bunny mesh, 3840 x 2160
    torch.cuda.empty_cache()
    sc = frontend.ParsedScene(scenes.config_text("cfg4-bunny-full-d14", spp=1), scenes.asset_dir())
    with api.Scene(sc) as scene:
        cam = camera_rays(sc, 3840, 2160)
        run(scene, "full-size bunny 3840x2160 camera rays", cam, torch.full((cam.shape[0],), float("inf"), dtype=torch.float64, device="cuda"))


if __name__ == "__main__":
    main()
