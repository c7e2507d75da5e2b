#!/usr/bin/env python
"""CPU estimate for DESIGN.md section 3 "Per-tile item masks": how many phase-B candidate evaluations (render.cuh traceScene) of
primary rays the masks remove, by item kind, on every bundled config at its full size.  The masks come from the real host code
(tiles.cpp, clear_boxes.cpp, lower.cpp through the probe of tests/test_tile_items_cpu.py); a seeded sample of primary rays from
the traced tiles replays phase A (each item's bounding sphere against the ray's line, in double, with the kernel's slack) and
counts the candidates with no mask, with the 16 x 16 tile's mask and with the mask of the ray's 8 x 4 block (estimateTiles run
on that block as a window of its own); the oracle's hit lists give the candidates that have a crossing at t >= 0, which no mask
can remove.  usage: python tools/tile_item_mask_rate.py [RAYS_PER_CONFIG]"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from functracer_b200 import abi, frontend, scenes  # noqa: E402
from oracle import ftb_oracle as orc  # noqa: E402
from util import parse  # noqa: E402
import test_tile_items_cpu as T  # noqa: E402

KINDS = r"""
// Per item: kind (leaf kind, or 100 + item kind for CSG) and bounding sphere (centre, radius; < 0 = unbounded).
extern "C" int ftb_probe_item_kinds(const ftb_scene_desc* d, int max_items, int* kind, double* bound)
{
    ftb::Lowered L;
    std::string e;
    if (ftb::lower_scene(*d, L, e, false) != 0) return -1;
    if ((int)L.items.size() > max_items) return -2;
    for (size_t i = 0; i < L.items.size(); ++i) {
        const ftb::Item& it = L.items[i];
        kind[i] = (it.kind & 0xff) == ftb::ITEM_LEAF ? (int)L.leaves[(size_t)it.a].kind : 100 + (it.kind & 0xff);
        for (int k = 0; k < 3; ++k) bound[4 * i + k] = it.bound_c[k];
        bound[4 * i + 3] = it.bound_r;
    }
    return (int)L.items.size();
}
"""
NAMES = {0: "sphere", 1: "plane", 2: "square", 3: "circle", 4: "cylinder", 5: "cone", 6: "cube", 7: "triangle", 8: "mesh",
         9: "solidCylinder", 101: "CSG program", 102: "CSG pair"}


def build():
    d = tempfile.mkdtemp(prefix="ftb_mask_rate_")
    src, so = os.path.join(d, "probe.cpp"), os.path.join(d, "libprobe.so")
    open(src, "w").write(T.PROBE % dict(csrc=T.CSRC) + KINDS)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src] +
                          [os.path.join(T.CSRC, "cuda", f) for f in ("clear_boxes.cpp", "tiles.cpp", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_items.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int] * 5 + [
        C.POINTER(C.c_uint), C.POINTER(C.c_ubyte), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
    lib.ftb_probe_items.restype = C.c_int
    lib.ftb_probe_item_kinds.argtypes = [C.POINTER(abi.SceneDesc), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    lib.ftb_probe_item_kinds.restype = C.c_int
    return lib


def candidates(bound, o, d):
    """Phase A in double: the items whose bounding sphere the ray's line touches, not wholly behind the origin (the kernel's
    general test, radius inflated as uploadScene does, 1e-6 |oc|^2 slack)."""
    du = d / np.linalg.norm(d)
    oc = bound[:, :3] - o
    b = oc @ du
    oc2 = (oc * oc).sum(axis=1)
    w = (bound[:, 3] * 1.002 + 1e-5) ** 2
    keep = ~((oc2 - b * b > w + 1e-6 * oc2) | ((b < 0) & (oc2 > w)))
    return keep | (bound[:, 3] < 0)


def main():
    n_rays = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
    lib = build()
    print("phase-B candidate evaluations per primary ray of the traced tiles, by item kind: no mask / 16x16 tile mask / 8x4 block "
          "mask / with a crossing at t >= 0 (%d seeded rays per config, full size)" % n_rays)
    for name in sorted(scenes.CONFIGS):
        cfg = scenes.CONFIGS[name]
        sc = parse(scenes.config_text(name))
        p = orc.make_params(sc.width, sc.height, sc.spp, frontend.jitter_pattern(cfg["seed"], sc.spp), sampling=sc.sampling)
        masks, clear, prim_item, n_items = T.item_masks(lib, sc, p)
        kind, bound = (C.c_int * 64)(), (C.c_double * 256)()
        if masks is None:
            print("\n%s: %d items, no masks (more than 32 items or depth of field)" % (name, n_items))
            continue
        assert lib.ftb_probe_item_kinds(sc.desc_ptr, 64, kind, bound) == n_items
        kinds = [NAMES[kind[i]] for i in range(n_items)]
        bnd = np.array(bound[:4 * n_items]).reshape(-1, 4)
        rng = np.random.default_rng(7)
        traced = np.argwhere(~clear)
        corner = p.sampling == abi.SAMPLING_CORNER
        gw, gh = sc.width + corner, sc.height + corner
        tot = {k: np.zeros(4) for k in sorted(set(kinds))}
        rays = 0
        while rays < n_rays:
            ty, tx = traced[rng.integers(len(traced))]
            x, y = int(tx * abi.TILE_W + rng.integers(abi.TILE_W)), int(ty * abi.TILE_H + rng.integers(abi.TILE_H))
            if x >= gw or y >= gh:
                continue
            s = 0 if corner else int(rng.integers(p.spp))
            jx, jy = (-0.5, 0.5) if corner else (p.jitter_xy[2 * s], p.jitter_xy[2 * s + 1])
            r = orc.primary_ray(sc.camera, sc.width, sc.height, x, y, jx, jy)
            o, d = np.array(r[:3]) + 1e-4 * np.array(r[3:]), np.array(r[3:])
            bx, by = x // 8 * 8, y // 4 * 4
            # the block as a window of its own; estimateTiles tests planes on a 16 x 16 sample rectangle from the window's corner,
            # which reaches past the block, so what the block's tile proves holds for it as well
            block = int(T.item_masks(lib, sc, p, (bx, by, bx + 8 - corner, by + 4 - corner))[0][0, 0]) & int(masks[ty, tx])
            hit = set()
            for h in orc.node_hits(sc, o, d, max_hits=4096):
                if h["t"] >= 0:
                    hit.add(int(prim_item[h["prim"]]))
            cand = candidates(bnd, o, d)
            for i in np.nonzero(cand)[0]:
                k = kinds[i]
                tot[k] += [1, (int(masks[ty, tx]) >> i) & 1, (block >> i) & 1, i in hit]
            rays += 1
        print("\n%s: %d items, %d of %d tiles traced" % (name, n_items, len(traced), clear.size))
        all_ = sum(tot.values())
        for k, v in list(tot.items()) + [("all", all_)]:
            v = v / rays
            print("  %-14s %6.3f  %6.3f  %6.3f  %6.3f   (tile mask -%4.1f %%, block mask -%4.1f %%)" % (
                k, v[0], v[1], v[2], v[3], 100 * (1 - v[1] / v[0]) if v[0] else 0, 100 * (1 - v[2] / v[0]) if v[0] else 0))


if __name__ == "__main__":
    main()
