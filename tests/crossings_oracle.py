"""The CPU oracle's full crossing lists with their records (test infrastructure for tests/test_gpu_ray_crossings.py).

Scene.intersect (Scene.fs:67-104) is nodeHits at the root.  This compiles tests/query_oracle.py's SOURCE (oracle/ftb_oracle.cpp
unchanged, plus its batch entries) with one more batch entry and the same flags, and returns every crossing in the reference's
own order with t, prim, sub and the 13 record values of tests/query_oracle.nearest (p, n, colour, roughness, reflectance,
shineyness, applyLighting)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import query_oracle

SOURCE = query_oracle.SOURCE + r"""
// Scene.intersect on every ray, traced as given: the first cap crossings in the reference's order, and how many there are.
extern "C" int ftbq_crossings(const ftb_scene_desc* desc, const double* rays, int64_t n, int cap, double* ts, int32_t* prim, int32_t* sub, double* rec,
                              int32_t* count, int threads)
{
    Scene sc;
    if (!prepare(desc, sc)) return -1;
    forAll(n, threads, [&](int64_t i, Counters& cn) {
        const double* r = rays + 6 * i;
        Hits hs;
        nodeHits(sc, desc->root, 0, Ray{{r[0], r[1], r[2]}, {r[3], r[4], r[5]}}, hs, cn);
        count[i] = (int32_t)hs.size();
        for (int k = 0; k < (int)hs.size() && k < cap; ++k) {
            const Hit* h = &hs[k];
            const size_t e = (size_t)i * cap + k;
            ts[e] = h->t; prim[e] = h->prim; sub[e] = h->sub;
            const double v[13] = {h->p.x, h->p.y, h->p.z, h->n.x, h->n.y, h->n.z, h->material.colour.r, h->material.colour.g, h->material.colour.b,
                                  h->material.roughness, h->material.reflectance, h->material.shineyness, h->material.applyLighting ? 1.0 : 0.0};
            for (int j = 0; j < 13; ++j) rec[13 * e + j] = v[j];
        }
    });
    return 0;
}
"""

_LIB = None
_DIR = None


def lib():
    global _LIB, _DIR
    if _LIB is None:
        _DIR = tempfile.TemporaryDirectory(prefix="ftb_crossings_oracle_")
        src, so = os.path.join(_DIR.name, "x.cpp"), os.path.join(_DIR.name, "libx.so")
        open(src, "w").write(SOURCE % {"root": query_oracle.ROOT})
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fno-builtin-pow", "-pthread",
                               "-shared", "-o", so, src])
        L = C.CDLL(so)
        vp = C.c_void_p
        L.ftbq_crossings.argtypes = [vp, vp, C.c_int64, C.c_int, vp, vp, vp, vp, vp, C.c_int]
        _LIB = L
    return _LIB


def raw(scene, rays_od, cap=256, threads=0):
    """Scene.intersect per ray in the reference's order: dict(count [n], t [n, cap] (nan pad), prim, sub, p, normal, colour, surface)."""
    rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    t, prim, sub = np.full((n, cap), np.nan), np.full((n, cap), -1, np.int32), np.zeros((n, cap), np.int32)
    rec, cnt = np.zeros((n, cap, 13)), np.empty(n, np.int32)
    rc = lib().ftbq_crossings(C.cast(scene.desc_ptr, C.c_void_p), rays.ctypes.data, n, cap, t.ctypes.data, prim.ctypes.data, sub.ctypes.data,
                              rec.ctypes.data, cnt.ctypes.data, threads)
    assert rc == 0
    assert (cnt <= cap).all(), "raise cap: a ray has %d crossings" % cnt.max()
    return dict(count=cnt, t=t, prim=prim, sub=sub, p=rec[..., 0:3], normal=rec[..., 3:6], colour=rec[..., 6:9], surface=rec[..., 9:13])


def crossings(scene, rays_od, max_hits, t_min=-np.inf, t_max=np.inf, cap=256, threads=0):
    """What ftb_intersect_all_rays returns by definition: (counts [n], {plane: [n, max_hits(, k)]}), the crossings with
    t_min <= t < t_max stably sorted by t (Seq.sortBy), the first max_hits kept, unused slots filled as a miss."""
    r = raw(scene, rays_od, cap, threads)
    n = len(r["count"])
    out = dict(t=np.full((n, max_hits), -1.0), prim=np.full((n, max_hits), -1, np.int32), sub=np.zeros((n, max_hits), np.int32),
               p=np.zeros((n, max_hits, 3)), normal=np.zeros((n, max_hits, 3)), colour=np.zeros((n, max_hits, 3)), surface=np.zeros((n, max_hits, 4)))
    counts = np.zeros(n, np.int32)
    for i in range(n):
        t = r["t"][i, :r["count"][i]]
        idx = np.nonzero((t >= t_min) & (t < t_max))[0]
        idx = idx[np.argsort(t[idx], kind="stable")]
        counts[i] = len(idx)
        keep = idx[:max_hits]
        for k in out:
            out[k][i, :len(keep)] = r[k][i, keep]
    return counts, out
