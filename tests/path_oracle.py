"""The CPU oracle's getColourForRay, level by level and light by light (test infrastructure for the path-query tests).

Shading.getColourForRay (Shading.fs:109-147) finds the nearest hit of a level, traces shadow rays towards every light, shades
one fragment per light and reflects.  This compiles tests/query_oracle.py's SOURCE (oracle/ftb_oracle.cpp unchanged, plus its
batch entries) with one more batch entry and the same flags.  The entry walks the levels with the oracle's own functions
(nodeHits / closest, shadowLightIntensity, lightDirection, specularShader, lambertianDiffuse / roughDiffuse, reflect) and
records what ftb_trace_paths reports: per level the ray (before slightOffset), the hit with its record and the running weight W;
per level and light the intensity, the direction and specular + diffuse (the unlit surface colour for a surface without
applyLighting).  The oracle's getColourForRay adds the reflection inside each light's fragment; the path form carries it in the
next level's W = W * L * reflectance instead.  For the same rays and keys the entry also returns getColourForRay's own colour,
so that the two summation orders can be checked against each other."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import query_oracle

SOURCE = query_oracle.SOURCE + r"""
// getColourForRay's levels on every ray, with sample key keys[i] (NULL: i), D = recursion_limit + 1 level entries per ray and L
// light entries per level.  Shadow rays a surface does not need (no applyLighting, or Oren-Nayar without a specular term) are
// not traced and report intensity 1, as the renderer does.  ref: getColourForRay's colour for the same ray and key.
extern "C" int ftbq_paths(const ftb_scene_desc* desc, const double* rays, const uint64_t* keys, int64_t n, int recursion_limit, uint64_t seed,
                          int32_t* levels, double* ray_od, double* weight, double* t, int32_t* prim, int32_t* sub, double* rec,
                          double* intensity, double* light_dir, double* light_colour, double* ref, int threads)
{
    Scene sc;
    if (!prepare(desc, sc)) return -1;
    const int D = recursion_limit + 1, L = desc->n_lights;
    forAll(n, threads, [&](int64_t i, Counters& cn) {
        const double* r = rays + 6 * i;
        const uint64_t key = keys ? keys[i] : (uint64_t)i;
        ShadeCtx cx = {&sc, seed, &cn};
        Ray ray = {{r[0], r[1], r[2]}, {r[3], r[4], r[5]}};
        const Col c = getColourForRay(cx, recursion_limit, ray, key, 0, nullptr);
        ref[3 * i] = c.r; ref[3 * i + 1] = c.g; ref[3 * i + 2] = c.b;
        for (int k = 0; k < D; ++k) {  // every entry starts as a miss with weight 0
            const size_t e = (size_t)i * D + k;
            for (int j = 0; j < 6; ++j) ray_od[6 * e + j] = 0.0;
            weight[e] = 0.0; t[e] = -1.0; prim[e] = -1; sub[e] = 0;
            for (int j = 0; j < 13; ++j) rec[13 * e + j] = 0.0;
            for (int l = 0; l < L; ++l) {
                const size_t q = e * L + l;
                intensity[q] = 0.0;
                for (int j = 0; j < 3; ++j) { light_dir[3 * q + j] = 0.0; light_colour[3 * q + j] = 0.0; }
            }
        }
        double W = 1.0;
        int limit = recursion_limit, k = 0;
        for (;; ++k) {
            const size_t e = (size_t)i * D + k;
            const double od[6] = {ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z};
            for (int j = 0; j < 6; ++j) ray_od[6 * e + j] = od[j];
            weight[e] = W;
            Ray off = {vadd(ray.o, vscale(ray.d, 0.0001)), ray.d};  // slightOffset (Shading.fs:129)
            Hits hs;
            nodeHits(sc, desc->root, 0, off, hs, cn);
            const Hit* hp = closest(hs);
            if (!hp) break;
            const Hit ix = *hp;
            t[e] = ix.t; prim[e] = ix.prim; sub[e] = ix.sub;
            const double v[13] = {ix.p.x, ix.p.y, ix.p.z, ix.n.x, ix.n.y, ix.n.z, ix.material.colour.r, ix.material.colour.g, ix.material.colour.b,
                                  ix.material.roughness, ix.material.reflectance, ix.material.shineyness, ix.material.applyLighting ? 1.0 : 0.0};
            for (int j = 0; j < 13; ++j) rec[13 * e + j] = v[j];
            if (L <= 0) break;
            const V3 shadowRayOrigin = vadd(ix.p, vscale(ix.n, 0.0001));
            const bool needShadow = ix.material.applyLighting && !(ix.material.roughness != 0.0 && !(ix.material.shineyness > 0.0));
            for (int l = 0; l < L; ++l) {
                const ftb_light& lt = desc->lights[l];
                const double in = needShadow ? shadowLightIntensity(cx, lt, l, shadowRayOrigin, key, (uint32_t)k) : 1.0;
                const Col lightColour = scaleColour(in, Col{lt.colour[0], lt.colour[1], lt.colour[2]});
                const V3 ldir = lightDirection(lt, ix.p);
                Col frag = ix.material.colour;
                if (ix.material.applyLighting) {
                    Col acc = {0, 0, 0};
                    acc = cadd(acc, specularShader(ix, lightColour, ldir, ray));
                    acc = cadd(acc, (ix.material.roughness == 0.0) ? lambertianDiffuse(ix, lightColour, ldir) : roughDiffuse(ix, ldir, ray));
                    frag = acc;
                }
                const size_t q = e * L + l;
                intensity[q] = in;
                light_dir[3 * q] = ldir.x; light_dir[3 * q + 1] = ldir.y; light_dir[3 * q + 2] = ldir.z;
                light_colour[3 * q] = frag.r; light_colour[3 * q + 1] = frag.g; light_colour[3 * q + 2] = frag.b;
            }
            if (!(ix.material.applyLighting && ix.material.reflectance > 0.0 && limit > 0)) break;
            W = W * ((double)L * ix.material.reflectance);  // reflectionShader inside each of the L fragments (Shading.fs:89-98)
            ray = Ray{ix.p, reflect(ix.n, ray.d)};
            --limit;
        }
        levels[i] = k + 1;
    });
    return 0;
}
"""

_LIB = None
_DIR = None


def lib():
    global _LIB, _DIR
    if _LIB is None:
        _DIR = tempfile.TemporaryDirectory(prefix="ftb_path_oracle_")
        src, so = os.path.join(_DIR.name, "p.cpp"), os.path.join(_DIR.name, "libp.so")
        open(src, "w").write(SOURCE % {"root": query_oracle.ROOT})
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fno-builtin-pow", "-pthread",
                               "-shared", "-o", so, src])
        L = C.CDLL(so)
        vp = C.c_void_p
        L.ftbq_paths.argtypes = [vp, vp, vp, C.c_int64, C.c_int, C.c_uint64] + [vp] * 11 + [C.c_int]
        _LIB = L
    return _LIB


def paths(scene, rays_od, sample_keys=None, recursion_limit=8, seed=1234, threads=0):
    """The oracle's breakdown, laid out like api.Scene.trace_paths' planes (without colour), plus ref [n, 3]: getColourForRay's
    own colour for the same rays and keys."""
    rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
    n, D, L = len(rays), recursion_limit + 1, scene.desc_ptr.contents.n_lights
    keys = None if sample_keys is None else np.ascontiguousarray(sample_keys, dtype=np.uint64)
    out = dict(levels=np.empty(n, np.int32), ray=np.empty((n, D, 6)), weight=np.empty((n, D)), t=np.empty((n, D)),
               prim=np.empty((n, D), np.int32), sub=np.empty((n, D), np.int32), rec=np.empty((n, D, 13)),
               intensity=np.empty((n, D, L)), light_dir=np.empty((n, D, L, 3)), light_colour=np.empty((n, D, L, 3)), ref=np.empty((n, 3)))
    rc = lib().ftbq_paths(C.cast(scene.desc_ptr, C.c_void_p), rays.ctypes.data, keys.ctypes.data if keys is not None else None, n,
                          recursion_limit, seed, *[out[k].ctypes.data for k in ("levels", "ray", "weight", "t", "prim", "sub", "rec",
                                                                                 "intensity", "light_dir", "light_colour", "ref")], threads)
    assert rc == 0
    rec = out.pop("rec")
    out.update(p=rec[..., 0:3], normal=rec[..., 3:6], hit_colour=rec[..., 6:9], surface=rec[..., 9:13])
    return out


def replay(levels, weight, light_colour):
    """The colour the kernel forms from a breakdown, in its order and in float64: per level local = 0, local += light_colour[l]
    in light order, then colour += W * local, over the levels traced."""
    n, D = weight.shape
    L = light_colour.shape[2]
    col = np.zeros((n, 3))
    for k in range(D):
        local = np.zeros((n, 3))
        for l in range(L):
            local = local + light_colour[:, k, l]
        col = np.where((k < levels)[:, None], col + weight[:, k, None] * local, col)
    return col
