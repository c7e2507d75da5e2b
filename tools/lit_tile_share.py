#!/usr/bin/env python
"""CPU estimate of what lit ground tiles (functracer_b200/csrc/cuda/lit_tiles.h) save, before any GPU run: per bundled config,
at a reduced size with one centred sample per pixel, the share of the primary samples that land on the ground and the share of
those whose every directional shadow ray is proven unblocked (their shadow rays are not traced).  The host proof is the real
lit_tiles.cpp (compiled by tests/test_lit_tiles_cpu.py's probe); which samples land on the ground comes from the CPU oracle.

usage: python tools/lit_tile_share.py [WIDTH]      (default 384; the height follows the config's aspect)"""
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from functracer_b200 import scenes  # noqa: E402
from oracle import ftb_oracle as orc  # noqa: E402
from test_lit_tiles_cpu import _build, check_against_oracle, lit_mask  # noqa: E402
from util import parse  # noqa: E402


def main():
    width = int(sys.argv[1]) if len(sys.argv) > 1 else 384
    lib = _build(tempfile.mkdtemp(prefix="ftb_lit_"), "tree")
    print("%-22s %11s %9s %12s %14s" % ("config", "size", "on ground", "tiles lit", "ground proven"))
    for name in sorted(scenes.CONFIGS):
        fw, fh = scenes.CONFIGS[name]["res"]
        w, h = width, max(16, round(width * fh / fw))
        sc = parse(scenes.config_text(name, res=(w, h), spp=1))
        p = orc.make_params(w, h, 1, [0.0, 0.0], sampling=sc.sampling)
        mask, ground = lit_mask(lib, sc, p)
        share, _, _ = check_against_oracle(lib, sc, p, max_samples=0)
        on = "-"
        if ground >= 0:
            prim = orc.render(sc, p)["prim"]
            on = "%.3f" % float((prim == ground).mean())
        print("%-22s %5dx%-5d %9s %12.3f %14.3f" % (name, w, h, on, float((mask != 0).mean()), share))


if __name__ == "__main__":
    main()
