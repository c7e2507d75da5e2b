"""ctypes face of libfunctracer_b200.so — the C ABI of include/functracer_b200.h.

This is the binding the F# shim makes with P/Invoke (INTEGRATION.md), restated for the Python
harness.  The names follow the reference's call site (Program.fs:54-64): `Scene.render` is
generateRays + shade + blendPixels, `Scene.shade` is Shading.shade on explicit rays.

There is no fallback: if the CUDA library is missing or no GPU is visible, every call raises.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class FtbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("functracer_b200 status %d: %s" % (status, message))
        self.status = status


def lib():
    """Loads libfunctracer_b200.so (built in-tree by __graft_entry__.build()).  Raises if absent."""
    global _LIB
    if _LIB is None:
        path = os.environ.get("FTB_LIB") or os.path.join(_HERE, "libfunctracer_b200.so")  # FTB_LIB: A/B builds of the same ABI
        if not os.path.exists(path):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)" % path)
        L = C.CDLL(path)
        vp = C.c_void_p
        L.ftb_abi_version.restype = C.c_int
        L.ftb_device_count.restype = C.c_int
        L.ftb_last_error.restype = C.c_char_p
        L.ftb_scene_create.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(vp)]
        L.ftb_scene_create.restype = C.c_int
        L.ftb_scene_destroy.argtypes = [vp]
        L.ftb_scene_destroy.restype = None
        L.ftb_render.argtypes = [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams), vp, C.POINTER(abi.DebugOut),
                                 C.POINTER(abi.Stats)]
        L.ftb_render.restype = C.c_int
        L.ftb_tile_buffer_bytes.argtypes = [C.POINTER(abi.RenderParams)]
        L.ftb_tile_buffer_bytes.restype = C.c_int64
        L.ftb_render_tiles_device.argtypes = [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams), vp,
                                              C.POINTER(abi.DebugOut), C.POINTER(abi.Stats), vp]
        L.ftb_render_tiles_device.restype = C.c_int
        L.ftb_assemble_device.argtypes = [C.POINTER(abi.RenderParams), C.POINTER(vp), vp, vp]
        L.ftb_assemble_device.restype = C.c_int
        L.ftb_shade_rays.argtypes = [vp, C.POINTER(C.c_double), C.c_int64, C.POINTER(abi.RenderParams),
                                     C.POINTER(C.c_double), C.POINTER(abi.DebugOut), C.POINTER(abi.Stats)]
        L.ftb_shade_rays.restype = C.c_int
        L.ftb_band_rows.argtypes = [C.POINTER(abi.RenderParams), C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.ftb_band_rows.restype = C.c_int
        L.ftb_assemble_rows_device.argtypes = [C.POINTER(abi.RenderParams), C.POINTER(vp), vp, C.c_int, C.c_int, vp]
        L.ftb_assemble_rows_device.restype = C.c_int
        L.ftb_host_copy_begin.argtypes = [vp, vp, vp, C.c_int64, vp]
        L.ftb_host_copy_begin.restype = C.c_int
        L.ftb_host_copy_finish.argtypes = [vp]
        L.ftb_host_copy_finish.restype = C.c_int
        L.ftb_check_overflow.argtypes = [vp, vp]
        L.ftb_check_overflow.restype = C.c_int
        if os.environ.get("FTB_LIB") and not hasattr(L, "ftb_scene_build_info"):
            L.ftb_scene_build_info = None  # an older A/B build of the same ABI (tools/ab_build.sh REV)
        else:
            L.ftb_scene_build_info.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_double)]
            L.ftb_scene_build_info.restype = C.c_int
        for name, args in (("ftb_render_window", [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int32] * 4
                            + [vp, C.POINTER(abi.DebugOut), C.POINTER(abi.Stats)]),
                           ("ftb_render_window_tiles_device", [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int32] * 4
                            + [vp, C.POINTER(abi.DebugOut), C.POINTER(abi.Stats), vp])):
            if os.environ.get("FTB_LIB") and not hasattr(L, name):
                setattr(L, name, None)  # an older A/B build of the same ABI without windows
            else:
                getattr(L, name).argtypes = args
                getattr(L, name).restype = C.c_int
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
        for name, args in (("ftb_intersect_rays", [vp, dp, C.c_int64, C.POINTER(abi.RenderParams), C.POINTER(abi.HitOut), C.POINTER(abi.Stats)]),
                           ("ftb_occluded_rays", [vp, dp, dp, C.c_int64, C.POINTER(abi.RenderParams), ip, C.POINTER(abi.Stats)]),
                           ("ftb_intersect_rays_device", [vp, dp, C.c_int64, C.POINTER(abi.RenderParams), C.POINTER(abi.HitOut),
                                                          C.POINTER(abi.Stats), vp]),
                           ("ftb_occluded_rays_device", [vp, dp, dp, C.c_int64, C.POINTER(abi.RenderParams), ip, C.POINTER(abi.Stats), vp]),
                           ("ftb_intersect_all_rays", [vp, dp, C.c_int64, C.c_int32, C.c_double, C.c_double, C.POINTER(abi.RenderParams),
                                                       C.POINTER(abi.HitOut), ip, C.POINTER(abi.Stats)]),
                           ("ftb_intersect_all_rays_device", [vp, dp, C.c_int64, C.c_int32, C.c_double, C.c_double, C.POINTER(abi.RenderParams),
                                                              C.POINTER(abi.HitOut), ip, C.POINTER(abi.Stats), vp]),
                           ("ftb_trace_paths", [vp, dp, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(abi.RenderParams), C.POINTER(abi.PathOut),
                                                C.POINTER(abi.Stats)]),
                           ("ftb_trace_paths_device", [vp, dp, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(abi.RenderParams),
                                                       C.POINTER(abi.PathOut), C.POINTER(abi.Stats), vp]),
                           ("ftb_frame_rays", [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int32] * 4
                            + [dp, C.POINTER(C.c_uint64)]),
                           ("ftb_frame_rays_device", [vp, C.POINTER(abi.Camera), C.POINTER(abi.RenderParams)] + [C.c_int32] * 4
                            + [dp, C.POINTER(C.c_uint64), vp]),
                           ("ftb_shade_samples", [vp, dp, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(abi.RenderParams), vp,
                                                  C.POINTER(abi.DebugOut), C.POINTER(abi.Stats)]),
                           ("ftb_shade_samples_device", [vp, dp, C.POINTER(C.c_uint64), C.c_int64, C.POINTER(abi.RenderParams), vp,
                                                         C.POINTER(abi.DebugOut), C.POINTER(abi.Stats), vp])):
            if os.environ.get("FTB_LIB") and not hasattr(L, name):
                setattr(L, name, None)  # an older A/B build of the same ABI without ray (crossing, path) queries or sample shading
            else:
                getattr(L, name).argtypes = args
                getattr(L, name).restype = C.c_int
        if L.ftb_abi_version() != abi.ABI_VERSION:
            raise RuntimeError("ABI version mismatch: library %d, bindings %d" % (L.ftb_abi_version(), abi.ABI_VERSION))
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise FtbError(rc, lib().ftb_last_error().decode(errors="replace"))


def make_params(width, height, spp, jitter_xy=None, sampling=abi.SAMPLING_JITTER, recursion_limit=8, seed=1234,
                precision=abi.PRECISION_FP32, out_format=abi.OUT_RGB_F64, shard_index=0, shard_count=1, n_gpus=0,
                collect_stats=0, band_index=0, band_count=0):
    p = abi.RenderParams()
    p.width, p.height, p.spp, p.sampling = width, height, spp, sampling
    keep = None
    if jitter_xy is not None:
        keep = np.ascontiguousarray(jitter_xy, dtype=np.float64)
        assert keep.size == 2 * spp
        p.jitter_xy = keep.ctypes.data_as(C.POINTER(C.c_double))
    p.recursion_limit, p.precision, p.seed, p.out_format = recursion_limit, precision, seed, out_format
    p.shard_index, p.shard_count, p.n_gpus, p.collect_stats = shard_index, shard_count, n_gpus, collect_stats
    p.band_index, p.band_count = band_index, band_count
    p._keep = keep
    return p


_OUT_DTYPE = {abi.OUT_RGB_F64: (np.float64, 3), abi.OUT_RGB_F32: (np.float32, 3), abi.OUT_RGBA8: (np.uint8, 4)}

MAX_CROSSINGS = 64  # FTB_MAX_CROSSINGS: the most crossings a crossing query keeps per ray

# the planes of a nearest-hit query (ftb_hit_out, in field order): ctypes element, numpy dtype, values per ray
HIT_PLANES = ("t", "prim", "sub", "p", "normal", "colour", "surface")
_PLANE_TYPES = ((C.c_double, np.float64, 1), (C.c_int32, np.int32, 1), (C.c_int32, np.int32, 1), (C.c_double, np.float64, 3),
                (C.c_double, np.float64, 3), (C.c_double, np.float64, 3), (C.c_double, np.float64, 4))

MAX_PATH_LEVELS = 64  # FTB_MAX_PATH_LEVELS: recursion_limit + 1 of a path query is at most this
# the planes of a path query (ftb_path_out; the hit planes are HIT_PLANES, with "hit_colour" for ftb_hit_out's colour):
# name -> (ctypes element, numpy dtype, shape after n: "D" = levels per ray, "L" = lights)
PATH_PLANES = {
    "levels": (C.c_int32, np.int32, ()), "colour": (C.c_double, np.float64, (3,)), "ray": (C.c_double, np.float64, ("D", 6)),
    "weight": (C.c_double, np.float64, ("D",)), "t": (C.c_double, np.float64, ("D",)), "prim": (C.c_int32, np.int32, ("D",)),
    "sub": (C.c_int32, np.int32, ("D",)), "p": (C.c_double, np.float64, ("D", 3)), "normal": (C.c_double, np.float64, ("D", 3)),
    "hit_colour": (C.c_double, np.float64, ("D", 3)), "surface": (C.c_double, np.float64, ("D", 4)),
    "intensity": (C.c_double, np.float64, ("D", "L")), "light_dir": (C.c_double, np.float64, ("D", "L", 3)),
    "light_colour": (C.c_double, np.float64, ("D", "L", 3)),
}


def _path_out(ptrs):
    """abi.PathOut from {plane name of PATH_PLANES: ctypes pointer} (missing = NULL)."""
    g = lambda name: ptrs.get(name)  # noqa: E731
    hit = abi.HitOut(g("t"), g("prim"), g("sub"), g("p"), g("normal"), g("hit_colour"), g("surface"))
    return abi.PathOut(g("levels"), g("colour"), g("ray"), g("weight"), hit, g("intensity"), g("light_dir"), g("light_colour"))


class Scene:
    """An ftb_scene: the flattened SceneGraph resident on the GPU(s)."""

    def __init__(self, parsed):
        """parsed: anything with .desc_ptr / .camera_ptr (functracer_b200.frontend.ParsedScene)."""
        self._h = C.c_void_p()
        self.parsed = parsed
        _check(lib().ftb_scene_create(parsed.desc_ptr, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().ftb_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- Program.fs:54-64: generateRays -> shade -> blendPixels ----------------------------------
    def render(self, width, height, spp, jitter_xy=None, debug=False, stats=False, out=None, camera=None, **kw):
        """Host-buffer render.  Returns dict(rgb[H,W,C], prim, sub, t, stats)."""
        if stats:
            kw.setdefault("collect_stats", 1)
        p = make_params(width, height, spp, jitter_xy, **kw)
        return self.render_params(p, debug=debug, stats=stats, out=out, camera=camera)

    def render_window(self, window, width, height, spp, jitter_xy=None, debug=False, stats=False, out=None, camera=None, **kw):
        """The pixels window = (x0, y0, x1, y1), i.e. [x0, x1) x [y0, y1), of the width x height frame, bit-identical to
        render() there.  Returns render()'s dict with rgb[y1 - y0, x1 - x0, C] and the window's debug planes."""
        if stats:
            kw.setdefault("collect_stats", 1)
        p = make_params(width, height, spp, jitter_xy, **kw)
        return self.render_params(p, debug=debug, stats=stats, out=out, camera=camera, window=window)

    def render_params(self, p, debug=False, stats=False, out=None, camera=None, window=None):
        """window: optional (x0, y0, x1, y1); the outputs then hold the window's pixels and samples only."""
        dt, ch = _OUT_DTYPE[p.out_format]
        W, H = p.width, p.height
        if window is not None:
            W, H = window[2] - window[0], window[3] - window[1]
        if out is None:
            out = np.empty((H, W, ch), dtype=dt)
        assert out.dtype == dt and out.size == W * H * ch and out.flags["C_CONTIGUOUS"]
        n = (W + 1) * (H + 1) if p.sampling == abi.SAMPLING_CORNER else W * H * p.spp
        prim = sub = t = dbg = None
        if debug:
            prim = np.full(n, -2, dtype=np.int32)
            sub = np.zeros(n, dtype=np.int32)
            t = np.zeros(n, dtype=np.float64)
            dbg = abi.DebugOut(prim.ctypes.data_as(C.POINTER(C.c_int32)), sub.ctypes.data_as(C.POINTER(C.c_int32)),
                               t.ctypes.data_as(C.POINTER(C.c_double)))
        st = abi.Stats() if stats else None
        cam = camera if camera is not None else self.parsed.camera_ptr
        args = (out.ctypes.data_as(C.c_void_p), C.byref(dbg) if dbg else None, C.byref(st) if st is not None else None)
        if window is None:
            _check(lib().ftb_render(self._h, cam, C.byref(p), *args))
        else:
            _check(_window_entry("ftb_render_window")(self._h, cam, C.byref(p), *[int(v) for v in window], *args))
        return dict(rgb=out, prim=prim, sub=sub, t=t, stats=st)

    # -- Shading.shade (Shading.fs:141-147) on explicit rays -----------------------------------------
    def shade(self, rays_od, debug=True, stats=False, **kw):
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        if stats:
            kw.setdefault("collect_stats", 1)
        p = make_params(1, 1, 1, None, **kw)
        rgb = np.zeros((n, 3), dtype=np.float64)
        prim = sub = t = dbg = None
        if debug:
            prim = np.full(n, -2, dtype=np.int32)
            sub = np.zeros(n, dtype=np.int32)
            t = np.zeros(n, dtype=np.float64)
            dbg = abi.DebugOut(prim.ctypes.data_as(C.POINTER(C.c_int32)), sub.ctypes.data_as(C.POINTER(C.c_int32)),
                               t.ctypes.data_as(C.POINTER(C.c_double)))
        st = abi.Stats() if stats else None
        dp = C.POINTER(C.c_double)
        _check(lib().ftb_shade_rays(self._h, rays.ctypes.data_as(dp), n, C.byref(p), rgb.ctypes.data_as(dp),
                                    C.byref(dbg) if dbg else None, C.byref(st) if st is not None else None))
        return dict(rgb=rgb, prim=prim, sub=sub, t=t, stats=st)

    # -- Scene.closest / Scene.lightIsBocked (Scene.fs:112-121) on explicit rays, traced exactly as given -------------------
    def intersect(self, rays_od, planes=HIT_PLANES, stats=None, **kw):
        """Nearest hit of every ray [n, 6] (o.xyz d.xyz; no slightOffset, d need not be unit length).  Returns {plane: array}
        for the requested planes of HIT_PLANES: t [n] (-1 on a miss), prim [n], sub [n], p / normal / colour [n, 3],
        surface [n, 4] (roughness, reflectance, shineyness, apply_lighting).  stats: an abi.Stats to fill (collect_stats=1
        for the counters).  kw: make_params' precision, collect_stats."""
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        out, hit = _hit_planes(planes, n)
        _check(_query_entry("ftb_intersect_rays")(self._h, rays.ctypes.data_as(C.POINTER(C.c_double)), n, C.byref(make_params(1, 1, 1, None, **kw)),
                                                   C.byref(hit), C.byref(stats) if stats is not None else None))
        return out

    def occluded(self, rays_od, max_t, stats=None, **kw):
        """Whether a surface with applyLighting crosses each ray [n, 6] at 0 <= t < max_t [n] (+inf allowed).  Returns bool [n]."""
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        mt = np.ascontiguousarray(np.broadcast_to(np.asarray(max_t, dtype=np.float64), (n,)))
        blocked = np.full(n, -1, dtype=np.int32)
        dp = C.POINTER(C.c_double)
        _check(_query_entry("ftb_occluded_rays")(self._h, rays.ctypes.data_as(dp), mt.ctypes.data_as(dp), n, C.byref(make_params(1, 1, 1, None, **kw)),
                                                  blocked.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(stats) if stats is not None else None))
        return blocked != 0

    def intersect_device(self, d_rays_ptr, n, d_planes, stream=0, stats=None, **kw):
        """intersect() on DEVICE memory of the current device, queued on `stream`: d_rays_ptr = n * 6 doubles, d_planes =
        {plane name of HIT_PLANES: device address} (missing / 0 = not wanted).  Does not synchronise unless stats is given."""
        hit = abi.HitOut(*[C.cast(C.c_void_p(d_planes.get(name) or None), C.POINTER(ct)) for name, (ct, _, _) in zip(HIT_PLANES, _PLANE_TYPES)])
        _check(_query_entry("ftb_intersect_rays_device")(self._h, C.cast(C.c_void_p(d_rays_ptr), C.POINTER(C.c_double)), n,
                                                          C.byref(make_params(1, 1, 1, None, **kw)), C.byref(hit),
                                                          C.byref(stats) if stats is not None else None, C.c_void_p(stream)))

    def occluded_device(self, d_rays_ptr, d_max_t_ptr, n, d_blocked_ptr, stream=0, stats=None, **kw):
        """occluded() on DEVICE memory: n * 6 ray doubles, n max_t doubles, n int32 results (1 = blocked)."""
        dp = C.POINTER(C.c_double)
        _check(_query_entry("ftb_occluded_rays_device")(self._h, C.cast(C.c_void_p(d_rays_ptr), dp), C.cast(C.c_void_p(d_max_t_ptr), dp), n,
                                                         C.byref(make_params(1, 1, 1, None, **kw)), C.cast(C.c_void_p(d_blocked_ptr), C.POINTER(C.c_int32)),
                                                         C.byref(stats) if stats is not None else None, C.c_void_p(stream)))

    # -- Scene.intersect (Scene.fs:67-104): every crossing of explicit rays, sorted by t -----------------------------------
    def intersect_all(self, rays_od, max_hits, t_min=-np.inf, t_max=np.inf, planes=HIT_PLANES, stats=None, **kw):
        """The crossings of every ray [n, 6] with t_min <= t < t_max, sorted by t (equal t in Scene.intersect's order), traced
        exactly as given.  Returns (counts [n], {plane: array}): counts may exceed max_hits (1 .. MAX_CROSSINGS), the planes hold
        the first max_hits crossings of each ray, [n, max_hits] for t / prim / sub, [n, max_hits, 3] for p / normal / colour,
        [n, max_hits, 4] for surface; unused slots read as a miss (t -1, prim -1, sub 0, 0 elsewhere).  kw: make_params'
        precision, collect_stats."""
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        out, hit = _hit_planes(planes, n, max_hits)
        counts = np.empty(n, dtype=np.int32)
        _check(_query_entry("ftb_intersect_all_rays")(self._h, rays.ctypes.data_as(C.POINTER(C.c_double)), n, max_hits, t_min, t_max,
                                                       C.byref(make_params(1, 1, 1, None, **kw)), C.byref(hit),
                                                       counts.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(stats) if stats is not None else None))
        return counts, out

    def intersect_all_device(self, d_rays_ptr, n, max_hits, d_counts_ptr, d_planes, t_min=-np.inf, t_max=np.inf, stream=0, stats=None, **kw):
        """intersect_all() on DEVICE memory of the current device, queued on `stream`: d_rays_ptr = n * 6 doubles, d_counts_ptr =
        n int32, d_planes = {plane name of HIT_PLANES: device address of n * max_hits entries} (missing / 0 = not wanted).
        Does not synchronise unless stats is given."""
        hit = abi.HitOut(*[C.cast(C.c_void_p(d_planes.get(name) or None), C.POINTER(ct)) for name, (ct, _, _) in zip(HIT_PLANES, _PLANE_TYPES)])
        _check(_query_entry("ftb_intersect_all_rays_device")(self._h, C.cast(C.c_void_p(d_rays_ptr), C.POINTER(C.c_double)), n, max_hits, t_min,
                                                              t_max, C.byref(make_params(1, 1, 1, None, **kw)), C.byref(hit),
                                                              C.cast(C.c_void_p(d_counts_ptr), C.POINTER(C.c_int32)),
                                                              C.byref(stats) if stats is not None else None, C.c_void_p(stream)))

    # -- Shading.getColourForRay (Shading.fs:109-147) on explicit rays, level by level and light by light -------------------
    def trace_paths(self, rays_od, sample_keys=None, recursion_limit=8, seed=1234, planes=tuple(PATH_PLANES), stats=None, **kw):
        """Why each ray [n, 6] has the colour ftb_shade_rays gives it.  The rays are shaded as shade() shades them (slightOffset
        included); sample_keys [n] uint64 are the soft lights' RNG keys (None: the ray's index, as shade() uses).  Returns
        {plane: array} for the requested planes of PATH_PLANES: levels [n], colour [n, 3], and per level (D = recursion_limit
        + 1) ray [n, D, 6], weight / t / prim / sub [n, D], p / normal / hit_colour [n, D, 3], surface [n, D, 4], and per level
        and light (L lights) intensity [n, D, L], light_dir / light_colour [n, D, L, 3].  kw: make_params' precision,
        collect_stats."""
        unknown = set(planes) - set(PATH_PLANES)
        if unknown:
            raise ValueError("unknown planes %s (choose from %s)" % (sorted(unknown), sorted(PATH_PLANES)))
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        keys = None
        if sample_keys is not None:
            keys = np.ascontiguousarray(sample_keys, dtype=np.uint64).reshape(-1)
            if keys.size != n:
                raise ValueError("sample_keys must hold one key per ray")
        dims = {"D": max(0, recursion_limit) + 1, "L": self.parsed.desc_ptr.contents.n_lights}
        out, ptrs = {}, {}
        for name in planes:
            ct, dt, shape = PATH_PLANES[name]
            out[name] = np.empty((n,) + tuple(dims.get(k, k) for k in shape), dtype=dt)
            ptrs[name] = out[name].ctypes.data_as(C.POINTER(ct))
        po = _path_out(ptrs)
        p = make_params(1, 1, 1, None, recursion_limit=recursion_limit, seed=seed, **kw)
        _check(_query_entry("ftb_trace_paths")(self._h, rays.ctypes.data_as(C.POINTER(C.c_double)),
                                                keys.ctypes.data_as(C.POINTER(C.c_uint64)) if keys is not None else None, n,
                                                C.byref(p), C.byref(po), C.byref(stats) if stats is not None else None))
        return out

    def trace_paths_device(self, d_rays_ptr, n, d_planes, d_keys_ptr=0, recursion_limit=8, seed=1234, stream=0, stats=None, **kw):
        """trace_paths() on DEVICE memory of the current device, queued on `stream`: d_rays_ptr = n * 6 doubles, d_keys_ptr =
        n uint64 (0 = the ray's index), d_planes = {plane name of PATH_PLANES: device address} (missing / 0 = not wanted),
        sized as trace_paths() returns them.  Does not synchronise unless stats is given."""
        unknown = set(d_planes) - set(PATH_PLANES)
        if unknown:
            raise ValueError("unknown planes %s (choose from %s)" % (sorted(unknown), sorted(PATH_PLANES)))
        po = _path_out({name: C.cast(C.c_void_p(d_planes.get(name) or None), C.POINTER(PATH_PLANES[name][0])) for name in PATH_PLANES})
        p = make_params(1, 1, 1, None, recursion_limit=recursion_limit, seed=seed, **kw)
        _check(_query_entry("ftb_trace_paths_device")(self._h, C.cast(C.c_void_p(d_rays_ptr), C.POINTER(C.c_double)),
                                                       C.cast(C.c_void_p(d_keys_ptr or None), C.POINTER(C.c_uint64)), n, C.byref(p),
                                                       C.byref(po), C.byref(stats) if stats is not None else None, C.c_void_p(stream)))

    # -- a frame's own samples (SamplingStrategy.generateRays / blendPixels, Image.fs:100-116) in the caller's hands ------------
    def frame_rays(self, window, width, height, spp, jitter_xy=None, camera=None, **kw):
        """The primary ray and RNG key of every sample of window (x0, y0, x1, y1) of the width x height frame, as render_window
        generates them.  Returns (rays [n, 6] o.xyz d.xyz before slightOffset, keys [n] uint64), n entries in the debug planes'
        order: (x1-x0)*(y1-y0)*spp in jitter sampling, (x1-x0+1)*(y1-y0+1) corners in corner sampling.  kw: make_params'
        sampling, precision, seed."""
        p = make_params(width, height, spp, jitter_xy, **kw)
        x0, y0, x1, y1 = (int(v) for v in window)
        n = max(0, x1 - x0 + 1) * max(0, y1 - y0 + 1) if p.sampling == abi.SAMPLING_CORNER else max(0, x1 - x0) * max(0, y1 - y0) * spp
        rays = np.empty((n, 6), dtype=np.float64)
        keys = np.empty(n, dtype=np.uint64)
        cam = camera if camera is not None else self.parsed.camera_ptr
        _check(_query_entry("ftb_frame_rays")(self._h, cam, C.byref(p), x0, y0, x1, y1, rays.ctypes.data_as(C.POINTER(C.c_double)),
                                               keys.ctypes.data_as(C.POINTER(C.c_uint64))))
        return rays, keys

    def frame_rays_device(self, p, window, d_rays_ptr, d_keys_ptr, stream=0, camera=None):
        """frame_rays() into DEVICE memory of the current device, queued on `stream`: d_rays_ptr = n * 6 doubles, d_keys_ptr = n
        uint64 (either 0 = not wanted); p: make_params(...)."""
        cam = camera if camera is not None else self.parsed.camera_ptr
        _check(_query_entry("ftb_frame_rays_device")(self._h, cam, C.byref(p), *[int(v) for v in window],
                                                      C.cast(C.c_void_p(d_rays_ptr or None), C.POINTER(C.c_double)),
                                                      C.cast(C.c_void_p(d_keys_ptr or None), C.POINTER(C.c_uint64)), C.c_void_p(stream)))

    def shade_samples(self, rays_od, spp, sample_keys=None, debug=False, stats=False, out=None, **kw):
        """Shades n_pixels * spp rays [n_pixels * spp, 6] (sample s of pixel i = ray i * spp + s) and blends each pixel as
        render() blends a jitter-mode pixel.  sample_keys [n_pixels * spp] uint64 are the RNG keys (None: the ray's index).
        Returns render()'s dict with rgb [n_pixels, C] and debug planes of n_pixels * spp entries.  kw: make_params' precision,
        seed, recursion_limit, out_format, collect_stats."""
        rays = np.ascontiguousarray(rays_od, dtype=np.float64).reshape(-1, 6)
        if spp < 1 or rays.shape[0] % spp:
            raise ValueError("the ray count must be a multiple of spp >= 1")
        n_pix, n = rays.shape[0] // spp, rays.shape[0]
        keys = None
        if sample_keys is not None:
            keys = np.ascontiguousarray(sample_keys, dtype=np.uint64).reshape(-1)
            if keys.size != n:
                raise ValueError("sample_keys must hold one key per ray")
        if stats:
            kw.setdefault("collect_stats", 1)
        p = make_params(1, 1, spp, None, **kw)
        dt, ch = _OUT_DTYPE[p.out_format]
        if out is None:
            out = np.empty((n_pix, ch), dtype=dt)
        assert out.dtype == dt and out.size == n_pix * ch and out.flags["C_CONTIGUOUS"]
        prim = sub = t = dbg = None
        if debug:
            prim = np.full(n, -2, dtype=np.int32)
            sub = np.zeros(n, dtype=np.int32)
            t = np.zeros(n, dtype=np.float64)
            dbg = abi.DebugOut(prim.ctypes.data_as(C.POINTER(C.c_int32)), sub.ctypes.data_as(C.POINTER(C.c_int32)),
                               t.ctypes.data_as(C.POINTER(C.c_double)))
        st = abi.Stats() if stats else None
        _check(_query_entry("ftb_shade_samples")(self._h, rays.ctypes.data_as(C.POINTER(C.c_double)),
                                                  keys.ctypes.data_as(C.POINTER(C.c_uint64)) if keys is not None else None, n_pix, C.byref(p),
                                                  out.ctypes.data_as(C.c_void_p), C.byref(dbg) if dbg else None,
                                                  C.byref(st) if st is not None else None))
        return dict(rgb=out, prim=prim, sub=sub, t=t, stats=st)

    def shade_samples_device(self, d_rays_ptr, n_pixels, p, d_out_ptr, d_keys_ptr=0, d_dbg=None, stream=0, stats=None):
        """shade_samples() on DEVICE memory of the current device, queued on `stream`: d_rays_ptr = n_pixels * p.spp * 6 doubles,
        d_keys_ptr = n_pixels * p.spp uint64 (0 = the ray's index), d_out_ptr = n_pixels pixels in p.out_format, d_dbg = optional
        (prim_ptr, sub_ptr, t_ptr) of n_pixels * p.spp entries (0 = not wanted).  Does not synchronise unless stats is given."""
        dbg = None
        if d_dbg is not None:
            dbg = abi.DebugOut(C.cast(C.c_void_p(d_dbg[0] or None), C.POINTER(C.c_int32)), C.cast(C.c_void_p(d_dbg[1] or None), C.POINTER(C.c_int32)),
                               C.cast(C.c_void_p(d_dbg[2] or None), C.POINTER(C.c_double)))
        _check(_query_entry("ftb_shade_samples_device")(self._h, C.cast(C.c_void_p(d_rays_ptr or None), C.POINTER(C.c_double)),
                                                         C.cast(C.c_void_p(d_keys_ptr or None), C.POINTER(C.c_uint64)), n_pixels, C.byref(p),
                                                         C.c_void_p(d_out_ptr or None), C.byref(dbg) if dbg is not None else None,
                                                         C.byref(stats) if stats is not None else None, C.c_void_p(stream)))

    # -- device-buffer entry points (one process per GPU; pointers are raw device addresses) -----
    def render_tiles_device(self, p, d_tiles_ptr, stream=0, stats=False, camera=None, d_dbg=None, window=None):
        """d_dbg: optional (prim_ptr, sub_ptr, t_ptr) DEVICE addresses of per-sample debug planes (0 / None = not wanted).
        window: optional (x0, y0, x1, y1), see render_window_tiles_device."""
        st = abi.Stats() if stats else None
        cam = camera if camera is not None else self.parsed.camera_ptr
        dbg = None
        if d_dbg is not None:
            dbg = abi.DebugOut(C.cast(C.c_void_p(d_dbg[0] or None), C.POINTER(C.c_int32)), C.cast(C.c_void_p(d_dbg[1] or None), C.POINTER(C.c_int32)),
                               C.cast(C.c_void_p(d_dbg[2] or None), C.POINTER(C.c_double)))
        args = (C.c_void_p(d_tiles_ptr), C.byref(dbg) if dbg is not None else None, C.byref(st) if st is not None else None, C.c_void_p(stream))
        if window is None:
            _check(lib().ftb_render_tiles_device(self._h, cam, C.byref(p), *args))
        else:
            _check(_window_entry("ftb_render_window_tiles_device")(self._h, cam, C.byref(p), *[int(v) for v in window], *args))
        return st

    def render_window_tiles_device(self, p, window, d_tiles_ptr, stream=0, stats=False, camera=None, d_dbg=None):
        """This shard's (band's) tiles of the window (x0, y0, x1, y1) of the frame p describes.  The buffer is that of a frame
        of the window's size: size it, band it and assemble it with window_params(p, window)."""
        return self.render_tiles_device(p, d_tiles_ptr, stream=stream, stats=stats, camera=camera, d_dbg=d_dbg, window=window)

    def build_info(self):
        """dict(bvh_on_device, bvh_build_ms, bvh_total_ms): how the scene's mesh index was built at create time."""
        on, b, t = C.c_int32(), C.c_double(), C.c_double()
        if lib().ftb_scene_build_info is None:
            return dict(bvh_on_device=False, bvh_build_ms=0.0, bvh_total_ms=0.0)
        _check(lib().ftb_scene_build_info(self._h, C.byref(on), C.byref(b), C.byref(t)))
        return dict(bvh_on_device=bool(on.value), bvh_build_ms=b.value, bvh_total_ms=t.value)

    def check_overflow(self, stream=0):
        """Waits for `stream`; raises FtbError(ERR_HIT_OVERFLOW) if a frame rendered through the device entry points on the
        current device overflowed a per-ray stack since the last check."""
        _check(lib().ftb_check_overflow(self._h, C.c_void_p(stream)))

    def host_copy_begin(self, d_src_ptr, host_array, stream=0, offset=0, nbytes=None):
        """Queues device -> host_array[offset : offset + nbytes] (bytes) behind `stream`; pageable destinations are staged
        through the scene's page-locked ring.  Complete with host_copy_finish()."""
        n = host_array.nbytes - offset if nbytes is None else nbytes
        _check(lib().ftb_host_copy_begin(self._h, C.c_void_p(d_src_ptr), C.c_void_p(host_array.ctypes.data + offset), n, C.c_void_p(stream)))

    def host_copy_finish(self):
        _check(lib().ftb_host_copy_finish(self._h))


def _hit_planes(planes, n, width=None):
    """({name: host array}, abi.HitOut pointing at them) for the requested planes; width: entries per ray (crossing queries)."""
    unknown = set(planes) - set(HIT_PLANES)
    if unknown:
        raise ValueError("unknown planes %s (choose from %s)" % (sorted(unknown), HIT_PLANES))
    out, ptrs = {}, []
    for name, (ct, dt, k) in zip(HIT_PLANES, _PLANE_TYPES):
        if name in planes:
            out[name] = np.empty((n,) + ((width,) if width else ()) + ((k,) if k > 1 else ()), dtype=dt)
            ptrs.append(out[name].ctypes.data_as(C.POINTER(ct)))
        else:
            ptrs.append(None)
    return out, abi.HitOut(*ptrs)


def _query_entry(name):
    fn = getattr(lib(), name)
    if fn is None:
        raise RuntimeError("%s has no %s (an older build)" % (os.environ.get("FTB_LIB"), name))
    return fn


def _window_entry(name):
    fn = getattr(lib(), name)
    if fn is None:
        raise RuntimeError("%s has no %s (an older build)" % (os.environ.get("FTB_LIB"), name))
    return fn


def window_params(p, window):
    """A copy of params p with the width / height of window (x0, y0, x1, y1): the params that size (tile_buffer_bytes),
    band (band_rows) and assemble (assemble_device, assemble_rows_device) a window's tile buffer."""
    q = abi.RenderParams.from_buffer_copy(p)
    q.width, q.height = window[2] - window[0], window[3] - window[1]
    q._keep = getattr(p, "_keep", None)
    return q


def band_rows(p, band_index, band_count):
    y0, y1 = C.c_int(), C.c_int()
    _check(lib().ftb_band_rows(C.byref(p), band_index, band_count, C.byref(y0), C.byref(y1)))
    return y0.value, y1.value


def assemble_rows_device(p, d_tile_ptrs, d_out_ptr, y0, y1, stream=0):
    arr = (C.c_void_p * len(d_tile_ptrs))(*[C.c_void_p(x) for x in d_tile_ptrs])
    _check(lib().ftb_assemble_rows_device(C.byref(p), arr, C.c_void_p(d_out_ptr), y0, y1, C.c_void_p(stream)))


def tile_buffer_bytes(p):
    n = lib().ftb_tile_buffer_bytes(C.byref(p))
    if n < 0:
        _check(int(n))
    return int(n)


def assemble_device(p, d_tile_ptrs, d_out_ptr, stream=0):
    arr = (C.c_void_p * len(d_tile_ptrs))(*[C.c_void_p(x) for x in d_tile_ptrs])
    _check(lib().ftb_assemble_device(C.byref(p), arr, C.c_void_p(d_out_ptr), C.c_void_p(stream)))


def device_count():
    return lib().ftb_device_count()
