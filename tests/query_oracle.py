"""Batch answers of the CPU oracle to ray queries (test infrastructure for tests/test_gpu_ray_queries.py).

oracle.node_hits answers one ray per ctypes call and prepares the scene each time; the query tests ask for hundreds of
thousands of rays.  This probe compiles oracle/ftb_oracle.cpp unchanged into a temporary library with two batch entry points
on the oracle's own functions (nodeHits at the root, then closest / lightIsBlocked, Scene.fs:112-121), threaded like
ftbo_shade_rays, and with the oracle's flags (oracle/Makefile)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SOURCE = r"""
#include "%(root)s/oracle/ftb_oracle.cpp"

namespace {
template <class Fn>
void forAll(int64_t n, int threads, Fn fn)
{
    std::atomic<int64_t> next(0);
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    auto work = [&]() {
        Counters cn;
        for (;;) {
            const int64_t b = next.fetch_add(256);
            if (b >= n) break;
            for (int64_t i = b; i < std::min(n, b + 256); ++i) fn(i, cn);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nt; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
}
}  // namespace

// Scene.closest on every ray, traced as given: t (-1 on a miss), prim (-1), sub (0), and 13 record values per ray (p, n, colour,
// roughness, reflectance, shineyness, applyLighting; 0 on a miss).
extern "C" int ftbq_nearest(const ftb_scene_desc* desc, const double* rays, int64_t n, double* t, int32_t* prim, int32_t* sub, double* rec, int threads)
{
    Scene sc;
    if (!prepare(desc, sc)) return -1;
    forAll(n, threads, [&](int64_t i, Counters& cn) {
        const double* r = rays + 6 * i;
        Hits hs;
        nodeHits(sc, desc->root, 0, Ray{{r[0], r[1], r[2]}, {r[3], r[4], r[5]}}, hs, cn);
        const Hit* h = closest(hs);
        double* q = rec + 13 * i;
        for (int k = 0; k < 13; ++k) q[k] = 0.0;
        if (!h) { t[i] = -1.0; prim[i] = -1; sub[i] = 0; return; }
        t[i] = h->t; prim[i] = h->prim; sub[i] = h->sub;
        const double v[13] = {h->p.x, h->p.y, h->p.z, h->n.x, h->n.y, h->n.z, h->material.colour.r, h->material.colour.g, h->material.colour.b,
                              h->material.roughness, h->material.reflectance, h->material.shineyness, h->material.applyLighting ? 1.0 : 0.0};
        for (int k = 0; k < 13; ++k) q[k] = v[k];
    });
    return 0;
}

// Scene.lightIsBocked on every ray: 1 iff a hit with applyLighting has 0 <= t < max_t.
extern "C" int ftbq_occluded(const ftb_scene_desc* desc, const double* rays, const double* max_t, int64_t n, int32_t* blocked, int threads)
{
    Scene sc;
    if (!prepare(desc, sc)) return -1;
    forAll(n, threads, [&](int64_t i, Counters& cn) {
        const double* r = rays + 6 * i;
        blocked[i] = lightIsBlocked(sc, max_t[i], Ray{{r[0], r[1], r[2]}, {r[3], r[4], r[5]}}, cn) ? 1 : 0;
    });
    return 0;
}

// every crossing of every ray (up to cap per ray) in the reference's order: t, applyLighting
extern "C" int ftbq_hits(const ftb_scene_desc* desc, const double* rays, int64_t n, int cap, double* ts, int32_t* lit, int32_t* count, int threads)
{
    Scene sc;
    if (!prepare(desc, sc)) return -1;
    forAll(n, threads, [&](int64_t i, Counters& cn) {
        const double* r = rays + 6 * i;
        Hits hs;
        nodeHits(sc, desc->root, 0, Ray{{r[0], r[1], r[2]}, {r[3], r[4], r[5]}}, hs, cn);
        count[i] = (int32_t)hs.size();
        for (int k = 0; k < (int)hs.size() && k < cap; ++k) { ts[(size_t)i * cap + k] = hs[k].t; lit[(size_t)i * cap + k] = hs[k].material.applyLighting ? 1 : 0; }
    });
    return 0;
}
"""

_LIB = None
_DIR = None


def lib():
    global _LIB, _DIR
    if _LIB is None:
        _DIR = tempfile.TemporaryDirectory(prefix="ftb_query_oracle_")
        src, so = os.path.join(_DIR.name, "q.cpp"), os.path.join(_DIR.name, "libq.so")
        open(src, "w").write(SOURCE % {"root": ROOT})
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fno-builtin-pow", "-pthread",
                               "-shared", "-o", so, src])
        L = C.CDLL(so)
        vp = C.c_void_p
        L.ftbq_nearest.argtypes = [vp, vp, C.c_int64, vp, vp, vp, vp, C.c_int]
        L.ftbq_occluded.argtypes = [vp, vp, vp, C.c_int64, vp, C.c_int]
        L.ftbq_hits.argtypes = [vp, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_int]
        _LIB = L
    return _LIB


def _desc(scene):
    return C.cast(scene.desc_ptr, C.c_void_p)


def nearest(scene, rays_od, threads=0):
    """The oracle's Scene.closest per ray: dict(t, prim, sub, p, normal, colour, surface) laid out like api.Scene.intersect's."""
    rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    t, prim, sub, rec = np.empty(n), np.empty(n, np.int32), np.empty(n, np.int32), np.empty((n, 13))
    rc = lib().ftbq_nearest(_desc(scene), rays.ctypes.data, n, t.ctypes.data, prim.ctypes.data, sub.ctypes.data, rec.ctypes.data, threads)
    assert rc == 0
    return dict(t=t, prim=prim, sub=sub, p=rec[:, 0:3], normal=rec[:, 3:6], colour=rec[:, 6:9], surface=rec[:, 9:13])


def occluded(scene, rays_od, max_t, threads=0):
    rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    mt = np.ascontiguousarray(np.broadcast_to(np.asarray(max_t, dtype=np.float64), (n,)))
    out = np.empty(n, np.int32)
    assert lib().ftbq_occluded(_desc(scene), rays.ctypes.data, mt.ctypes.data, n, out.ctypes.data, threads) == 0
    return out != 0


def hits(scene, rays_od, cap=64, threads=0):
    """Every crossing per ray: (t [n, cap] padded with nan, applyLighting [n, cap], count [n])."""
    rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    ts, lit, cnt = np.full((n, cap), np.nan), np.zeros((n, cap), np.int32), np.empty(n, np.int32)
    assert lib().ftbq_hits(_desc(scene), rays.ctypes.data, n, cap, ts.ctypes.data, lit.ctypes.data, cnt.ctypes.data, threads) == 0
    return ts, lit, cnt
