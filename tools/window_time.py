#!/usr/bin/env python
"""What a window render costs next to the whole frame (ftb_render_window, include/functracer_b200.h).

For each scene at its BASELINE.json size: ftb_render of the whole frame, the whole frame as a window, the centred
quarter-frame window (half the width, half the height), an 8-px full-height stripe, a 64x64 window and a 1x1 window with
all three debug planes.  Every case renders into a pageable RGBA8 buffer with a stats block and no counting kernel, so the
library times the render kernel with its own CUDA events (ftb_stats.kernel_ms) and the call's wall time (total_ms): two
warm-up calls (the tile order of each window is computed once), then the mean and minimum of K.  The GPU's name and power
limit are printed with the numbers.

usage: python tools/window_time.py ["cfg5-repeat cfg2-hollow-sphere"] [K]"""
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


def cases(W, H):
    cx, cy = W // 2, H // 2
    return [("ftb_render whole frame", None, False), ("window: whole frame", (0, 0, W, H), False),
            ("window: centred quarter", (W // 4, H // 4, W // 4 + W // 2, H // 4 + H // 2), False), ("window: top quarter", (0, 0, W, H // 4), False),
            ("window: 8-px stripe", (cx - 4, 0, cx + 4, H), False), ("window: 64x64", (cx - 32, cy - 32, cx + 32, cy + 32), False),
            ("window: 1x1 + debug planes", (cx, cy, cx + 1, cy + 1), True)]


def main():
    import numpy as np
    from functracer_b200 import abi, api, frontend, scenes
    names = (sys.argv[1] if len(sys.argv) > 1 else "cfg5-repeat cfg2-hollow-sphere").split()
    k = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    gpu, power = gpu_info()
    print("GPU: %s, power limit %s" % (gpu, power), flush=True)
    for name in names:
        cfg = scenes.CONFIGS[name]
        sc = frontend.ParsedScene(scenes.config_text(name), scenes.asset_dir())
        W, H, spp = sc.width, sc.height, sc.spp
        jit = frontend.jitter_pattern(cfg["seed"], spp)
        with api.Scene(sc) as scene:
            p = api.make_params(W, H, spp, jit, seed=1234, out_format=abi.OUT_RGBA8)
            whole_ms = None
            for label, win, debug in cases(W, H):
                w, h = (W, H) if win is None else (win[2] - win[0], win[3] - win[1])
                out = np.empty((h, w, 4), dtype=np.uint8)
                kms, tms = [], []
                for it in range(2 + k):
                    st = scene.render_params(p, out=out, stats=True, debug=debug, window=win)["stats"]
                    if it >= 2:
                        kms.append(st.kernel_ms)
                        tms.append(st.total_ms)
                rec = dict(config=name, case=label, window=win, pixels=w * h, spp=spp, kernel_ms=sum(kms) / k, kernel_ms_min=min(kms),
                           total_ms=sum(tms) / k, total_ms_min=min(tms), gpu=gpu, power_limit=power)
                if whole_ms is None:
                    whole_ms = rec["kernel_ms"]
                rec["kernel_vs_whole"] = rec["kernel_ms"] / whole_ms
                print("%-20s %-28s %10d px  kernel %9.3f ms (min %9.3f, %6.3f x whole)  total %9.3f ms (min %9.3f)"
                      % (name, label, w * h, rec["kernel_ms"], rec["kernel_ms_min"], rec["kernel_vs_whole"], rec["total_ms"], rec["total_ms_min"]), flush=True)
                print("JSON " + json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
