#!/usr/bin/env python
"""Times ftb_scene_create for the mesh workloads (FTB_VERBOSE=1 prints the phases to stderr)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: F401  (creates the CUDA context first, as bench.py does)
from functracer_b200 import api, frontend, scenes

torch.zeros(1, device="cuda")
for name in sys.argv[1:] or ["cfg4-bunny", "cfg4-bunny-d12", "cfg4-bunny-full-d14"]:
    parsed = frontend.ParsedScene(scenes.config_text(name), scenes.asset_dir())
    for rep in range(3):
        t0 = time.perf_counter()
        sc = api.Scene(parsed)
        ms = 1e3 * (time.perf_counter() - t0)
        print(name, "create %.1f ms" % ms, sc.build_info(), flush=True)
        sc.close()
