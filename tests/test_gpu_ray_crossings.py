"""Crossing queries (ftb_intersect_all_rays and its device form) against the CPU oracle and against the other queries.  Needs a
B200: run with `-m gpu`.

The oracle's answer is Scene.intersect (nodeHits at the root, tests/crossings_oracle.py) filtered to t_min <= t < t_max and
stably sorted by t; the scenes and ray sets are tests/test_gpu_ray_queries.py's (bundled scenes, one scene per kernel variant,
six fuzz seeds, two large-mesh scenes; camera, random, surface-leaving, axis-aligned and scaled rays).

Bars (every count is printed):
  - counts equal to the oracle's on >= 99.9 % of the rays in FP64 and >= 99 % in FP32 (a grazing ray, or one through a cube's edge,
    meets a different number of faces with the last bits of t; DESIGN.md §6); every ray whose count differs is printed.  Not counted:
    rays for which the oracle lists a crossing at t = 0 and the kernel fewer crossings (a ray parallel to a planar face meets it at
    its origin, Plane.fs:14-16, where the ray's line can miss the item's bound: DESIGN.md §6);
  - where the counts agree, prim and sub entry by entry.  Not counted as a difference: two entries whose oracle t agree to 1e-9
    (FP64) / 1e-4 (FP32) relative and that appear in the other order (ties at cube edges, coincident surfaces), and crossings at
    t = 0 of rays parallel to a planar face (Plane.fs:14-16).  What remains may touch 1e-3 (FP64) / 5e-3 (FP32) of the rays,
    as for the nearest queries;
  - t and the records of the entries whose ids agree: test_gpu_ray_queries.py's BARS and COVER, computed as there, except that the
    normal is held relative to the scale |o| + |t| |d| + 1 that p is held to (a crossing far along the ray, or behind its origin,
    has its model-space point - from which its normal is made - as far off as its p); unused slots a miss."""
import math
import zlib

import numpy as np
import pytest

import crossings_oracle as co
import large_mesh_scenes as lms
import test_gpu_ray_queries as rq
import variant_scenes as vs
from functracer_b200 import abi, api
from oracle import parity
from util import parse

pytestmark = pytest.mark.gpu

FP32, FP64 = abi.PRECISION_FP32, abi.PRECISION_FP64_VERIFY
PRECISIONS = (FP64, FP32)
K = api.MAX_CROSSINGS
COUNT_FRAC = {FP64: 0.999, FP32: 0.99}
TIE_REL = {FP64: 1e-9, FP32: 1e-4}
CASES = rq.CASES


def _intersect_all(scene, rays, case, **kw):
    try:
        return scene.intersect_all(rays, **kw)
    except api.FtbError as e:
        assert e.status == abi.ERR_HIT_OVERFLOW and case.startswith("fuzz")
        pytest.skip("hit-stack overflow reported: %s" % e)


def check_unused_slots(counts, got):
    used = np.arange(got["t"].shape[1])[None, :] < np.minimum(counts, got["t"].shape[1])[:, None]
    if "t" in got:
        assert (got["t"][~used] == -1).all()
    if "prim" in got:
        assert (got["prim"][~used] == -1).all() and (got["prim"][used] >= 0).all()
    if "sub" in got:
        assert (got["sub"][~used] == 0).all()
    for k in ("p", "normal", "colour", "surface"):
        if k in got:
            assert (got[k][~used] == 0).all(), k


def _explained(gr, rr, gt, rt, k, tol):
    """Entry k of one ray differs in ids: a tie in t with an entry that carries the device's ids, or a t = 0 parallel crossing."""
    if rt[k] == 0 or gt[k] == 0:
        return True
    near = np.abs(rt - rt[k]) <= tol * max(abs(rt[k]), 1.0)
    return bool((near & (rr[:, 0] == gr[k, 0]) & (rr[:, 1] == gr[k, 1])).any())


def compare_crossings(gc, got, rc, ref, rays, precision, label):
    """Asserts the bars of the module docstring; returns the counts."""
    n = len(rays)
    check_unused_slots(gc, got)
    cmism = gc != rc
    # Plane.fs:14-16 (DESIGN.md §6): a ray parallel to a planar face meets it at t = 0 wherever the face is; where the ray's line
    # misses the item's bound the kernel does not see that crossing
    parallel = ((ref["t"] == 0) & (ref["prim"] >= 0)).any(axis=1) & (gc < rc)
    res = dict(rays=n, count_mismatch=int(cmism.sum()), count_t0_parallel=int((cmism & parallel).sum()), crossings=int(rc.sum()),
               behind=int(((ref["t"] < 0) & (ref["prim"] >= 0)).sum()))
    for i in np.nonzero(cmism)[0]:
        print("  %s ray %d%s: %d crossings, oracle %d; t %s / oracle %s" % (label, i, " (t = 0 parallel)" if parallel[i] else "", gc[i], rc[i],
                                                                         got["t"][i, :min(gc[i], 8)], ref["t"][i, :min(rc[i], 8)]))
    assert 1.0 - (cmism & ~parallel).mean() >= COUNT_FRAC[precision], (label, res)
    idm = (got["prim"] != ref["prim"]) | (got["sub"] != ref["sub"])
    bad_rays, ties = set(), 0
    for i in np.nonzero(~cmism & idm.any(axis=1))[0]:
        gr, rr = np.stack([got["prim"][i], got["sub"][i]], 1), np.stack([ref["prim"][i], ref["sub"][i]], 1)
        for k in np.nonzero(idm[i])[0]:
            if _explained(gr, rr, got["t"][i], ref["t"][i], k, TIE_REL[precision]):
                ties += 1
            else:
                bad_rays.add(int(i))
    res.update(id_ties=ties, id_unexplained_rays=len(bad_rays))
    for i in sorted(bad_rays):
        print("  %s ray %d: ids %s / oracle %s" % (label, i, list(zip(got["prim"][i, :gc[i]], got["sub"][i, :gc[i]])),
                                                   list(zip(ref["prim"][i, :rc[i]], ref["sub"][i, :rc[i]]))))
    assert len(bad_rays) <= rq.ID_FRAC[precision] * n, (label, res)
    # records: every used entry of the rays whose counts and ids agree, held to the nearest queries' bars (errors as there)
    same = (~cmism & ~idm.any(axis=1))[:, None] & (ref["prim"] >= 0)
    if same.any():
        r = np.broadcast_to(rays[:, None, :], ref["t"].shape + (6,))[same]
        t_ref, t_got = ref["t"][same], got["t"][same]
        dlen = np.linalg.norm(r[:, 3:], axis=1)
        scale = np.linalg.norm(r[:, :3], axis=1) + np.abs(t_ref) * dlen + 1.0
        d = {k: np.abs(got[k][same] - ref[k][same]).max(axis=1) for k in ("p", "normal", "colour", "surface")}
        perr = d["p"] / scale
        if precision == FP32:
            perr[t_ref == 0] = 0.0  # the parallel hit's p = o, which the FP32 fragment projects onto the plane
        # A crossing far along the ray (or behind its origin) has a model-space point as far off as its p, and its normal is made
        # from that point: the normal is held relative to the same scale as p.  The nearest queries' first hits have scale ~ 1.
        errs = dict(t=np.abs(t_got - t_ref) / np.maximum(np.abs(t_ref), 1e-30) if precision == FP64 else np.abs(t_got - t_ref) * dlen / scale,
                    p=perr, normal=d["normal"] / scale, colour=d["colour"],
                    surface=d["surface"] / np.maximum(np.abs(ref["surface"][same]).max(axis=1), 1.0))
        for k, e in errs.items():
            frac = float((e <= rq.BARS[precision][k]).mean())
            res["%s_within" % k], res["%s_max" % k] = frac, float(e.max())
            assert frac >= rq.COVER[precision][k], (label, k, frac, float(e.max()))
        assert np.array_equal(got["surface"][same][:, 3], ref["surface"][same][:, 3])  # apply_lighting is exact
    return res


# ---- 1. against the oracle's sorted lists ----------------------------------------------------------------------------------
@pytest.mark.parametrize("case", sorted(CASES))
def test_crossings_against_the_oracle(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    sets = rq.ray_sets(sc, np.random.default_rng(zlib.crc32(case.encode()) + 5))
    refs = {k: co.crossings(sc, r, K) for k, r in sets.items()}
    with rq._open(sc) as scene:
        for precision in PRECISIONS:
            for k, rays in sets.items():
                gc, got = _intersect_all(scene, rays, case, max_hits=K, precision=precision)
                res = compare_crossings(gc, got, refs[k][0], refs[k][1], rays, precision, (case, k, precision))
                print("%s %s precision %d: %s" % (case, k, precision, res))


# ---- 2. against the other queries: the first crossing ahead is the nearest hit; occlusion is a lit crossing before max_t -------
@pytest.mark.parametrize("case", sorted(CASES))
def test_first_crossing_ahead_is_the_nearest_hit_and_decides_occlusion(case, tmp_path):
    sc = CASES[case](str(tmp_path))
    rng = np.random.default_rng(zlib.crc32(case.encode()) + 6)
    sets = rq.ray_sets(sc, rng, n=400)
    with rq._open(sc) as scene:
        for precision in PRECISIONS:
            for k, rays in sets.items():
                gc, got = _intersect_all(scene, rays, case, max_hits=K, t_min=0.0, precision=precision)
                near = scene.intersect(rays, precision=precision)
                first = {p: v[:, 0] for p, v in got.items()}
                if precision == FP64:  # the same trace in the same kernel family: bit for bit, every plane
                    for p in api.HIT_PLANES:
                        assert np.array_equal(first[p], near[p]), (case, k, p)
                elif k == "camera":  # FP32: the crossings run the generic kernel, the queries the scene's own variant
                    W, H = rq.GRID
                    z = np.zeros((H, W, 3))
                    c = parity.compare_window(z, near["prim"].reshape(H, W, 1), z, first["prim"].reshape(H, W, 1),
                                              ref_sub=near["sub"].reshape(H, W, 1), got_sub=first["sub"].reshape(H, W, 1))
                    print("%s camera FP32: %d of %d first ids differ from the nearest query's (unexplained %d)" % (case, c["prim_mismatch"], c["samples"],
                                                                                                              c["prim_unexplained"]))
                    assert c["prim_unexplained"] == 0, (case, c.get("unexplained_samples"))
                else:
                    print("%s %s FP32: %d of %d first ids differ from the nearest query's" % (case, k, int((first["prim"] != near["prim"]).sum()), len(rays)))
                # occlusion: a crossing with applyLighting at 0 <= t < max_t (decided by the list unless it was cut at K crossings)
                ahead = np.where(got["prim"] >= 0, got["t"], 0.0).max(axis=1)
                mt = np.where(rng.random(len(rays)) < 0.2, np.inf, rng.uniform(0.0, 1.2, len(rays)) * np.maximum(ahead, 1e-3))
                lit = (got["prim"] >= 0) & (got["t"] < mt[:, None]) & (got["surface"][..., 3] == 1)
                want, known = lit.any(axis=1), (gc <= K) | lit.any(axis=1)
                blocked = scene.occluded(rays, mt, precision=precision)
                mism = (blocked != want) & known
                print("%s %s precision %d: %d rays, %d blocked, %d differ from the crossing list" % (case, k, precision, int(known.sum()), int(blocked.sum()),
                                                                                                 int(mism.sum())))
                if precision == FP64:
                    assert not mism.any(), (case, k)
                else:
                    tie = rq._tie(sc, rays, mt, 1e-4) & mism
                    assert (mism & ~tie).mean() <= rq.ID_FRAC[FP32], (case, k)


# ---- 3. range, truncation, planes -------------------------------------------------------------------------------------------
RANGES = [(0.0, math.inf), (-math.inf, 0.0), (0.5, 3.0), (-2.0, 1.0), (1e-7, 7.25)]


@pytest.mark.parametrize("make", [rq._bundled("house"), rq._variant("cubes33"), rq._variant("nested1_soft1"), rq._variant("meshes0"),
                                  rq._large("shiny_blob")], ids=["house", "cubes33", "nested1_soft1", "meshes0", "shiny_blob"])
def test_range_and_truncation_return_sublists(make, tmp_path):
    """An [t_min, t_max) call returns exactly the in-range sublist of the (-inf, inf) call, and max_hits = k the first k entries of
    the 64-wide call with the same counts, in every plane and both precisions."""
    sc = make(str(tmp_path))
    rays = np.concatenate(list(rq.ray_sets(sc, np.random.default_rng(21), n=300).values()))
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            fc, full = scene.intersect_all(rays, K, precision=precision)
            fits = fc <= K
            assert fits.mean() > 0.99 and (fc > 1).sum() > 50
            for t_min, t_max in RANGES:
                c, part = scene.intersect_all(rays, K, t_min, t_max, precision=precision)
                inr = (full["prim"] >= 0) & (full["t"] >= t_min) & (full["t"] < t_max)
                assert np.array_equal(c[fits], inr.sum(axis=1)[fits]), (t_min, t_max)
                for i in np.nonzero(fits)[0]:
                    sel = np.nonzero(inr[i])[0]
                    for p in api.HIT_PLANES:
                        assert np.array_equal(part[p][i, :len(sel)], full[p][i, sel]), (t_min, t_max, i, p)
                check_unused_slots(c, part)
                print("precision %d [%g, %g): %d crossings" % (precision, t_min, t_max, int(c.sum())))
            for k in (1, 2, 3, 8, 17, 63):
                c, part = scene.intersect_all(rays, k, precision=precision)
                assert np.array_equal(c, fc), k
                for p in api.HIT_PLANES:
                    assert np.array_equal(part[p], full[p][:, :k]), (k, p)


def test_planes_not_requested_stay_untouched(tmp_path):
    import torch
    sc = rq._bundled("house")(str(tmp_path))
    rays = np.concatenate(list(rq.ray_sets(sc, np.random.default_rng(8), n=300).values()))
    n, k = len(rays), 5
    widths = dict(t=(), prim=(), sub=(), p=(3,), normal=(3,), colour=(3,), surface=(4,))
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            hc, host = scene.intersect_all(rays, k, precision=precision)
            d_rays = torch.from_numpy(rays).cuda()
            for want in ((), ("t",), ("prim", "p"), ("sub", "colour", "surface"), ("normal",)):
                counts = torch.full((n,), -7, dtype=torch.int32, device="cuda")
                bufs = {p: torch.full((n, k) + w, -7, dtype=torch.int32 if p in ("prim", "sub") else torch.float64, device="cuda") for p, w in widths.items()}
                scene.intersect_all_device(d_rays.data_ptr(), n, k, counts.data_ptr(), {p: bufs[p].data_ptr() for p in want}, precision=precision)
                torch.cuda.synchronize()
                assert np.array_equal(counts.cpu().numpy(), hc)
                for p, b in bufs.items():
                    b = b.cpu().numpy()
                    if p in want:
                        assert np.array_equal(b, host[p]), p
                    else:
                        assert (b == -7).all(), p


# ---- 4. order on ties, exact in FP64 ----------------------------------------------------------------------------------------
def _exact_against_oracle(sc, rays, label, cap=256):
    rc, ref = co.crossings(sc, rays, K, cap=cap)
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            gc, got = scene.intersect_all(rays, K, precision=precision)
            if precision == FP64:
                assert np.array_equal(gc, rc), label
                assert np.array_equal(got["prim"], ref["prim"]) and np.array_equal(got["sub"], ref["sub"]), label
            else:
                res = compare_crossings(gc, got, rc, ref, rays, precision, (label, precision))
                print("%s FP32: %s" % (label, res))
    return rc, ref


def test_coincident_triangles_keep_their_mesh_order(tmp_path):
    """5 000 copies of one triangle: 5 000 crossings at one t, which Scene.intersect lists in the mesh's enumeration order."""
    text, d = lms.coincident(str(tmp_path))
    sc = parse(text, assets=d)
    tri = np.array([(6.0, 6.0, -1.0), (10.0, 6.5, -1.0), (7.0, 10.0, -1.5)])
    w = np.random.default_rng(3).dirichlet((2, 2, 2), size=100)
    o = np.array([8.0, 8.0, -12.0])
    rays = np.hstack([np.tile(o, (100, 1)), w @ tri - o])
    rc, ref = _exact_against_oracle(sc, rays, "coincident", cap=8192)
    assert (rc >= 5000).all() and (ref["t"][:, 1:K] == ref["t"][:, :1]).all()


@pytest.mark.parametrize("n_tris", [32767, 32768])
@pytest.mark.parametrize("mesh_first", [True, False])
def test_mesh_tied_with_triangle_items(tmp_path, n_tris, mesh_first):
    """A mesh and triangle items holding exact copies of 31 of its triangles: both crossings at one t, in item order."""
    text, d, dup = lms.tie(str(tmp_path), n_tris, mesh_first=mesh_first)
    sc = parse(text, assets=d)
    o = np.array([8.0, 8.0, -12.0])
    w = np.random.default_rng(4).dirichlet((3, 3, 3), size=(31, 4))
    pts = np.einsum("tkc,tcx->tkx", w, dup).reshape(-1, 3)
    rays = np.hstack([np.tile(o, (len(pts), 1)), pts - o])
    rc, ref = _exact_against_oracle(sc, rays, "tie %d %s" % (n_tris, mesh_first))
    # each ray's list holds the tie: two neighbouring entries at one t (a tilted neighbouring cell may come first)
    tie = ((ref["t"][:, :-1] == ref["t"][:, 1:]) & (ref["prim"][:, 1:] >= 0)).any(axis=1)
    assert (rc >= 2).all() and tie.all()


def test_crossings_behind_the_origin_of_open_csg_operands():
    """tests/test_gpu_parity.py's open operands seen from beyond the open end: the crossings behind the origin that set
    Csg.constructedSolid's inside state are listed too (t_min = -inf), and the phantom crossings ahead follow them."""
    cam = "camera pos (0.3,3,0) lookat (-1.0,7,0) up (0,0,1) fov 40 ratio 1"
    obj = "(material diffuse (0.8,0.6,0.4) reflectance 0 shineyness 0 (subtract cylinder (translate (-1.6,7,0.7) sphere)))"
    obj2 = "(material diffuse (0.3,0.6,0.9) reflectance 0 shineyness 0 (intersect (translate (-0.4,7,-0.7) (scale 0.8 sphere)) (scale (3,1,3) cone)))"
    sc = parse(cam + "\nsamples 1\n\n" + obj + "\n" + obj2 + "\n\ndirectional dir (0,1,0.2) colour 1\n")
    rays = rq.camera_rays(sc, 48, 48)
    rc, ref = _exact_against_oracle(sc, rays, "open-operand")
    behind = (ref["prim"] >= 0) & (ref["t"] < 0)
    assert behind.any(axis=1).sum() > 100 and ((ref["prim"] >= 1) & (ref["t"] > 0)).any(axis=1).sum() > 100


# ---- 5. errors, device entry, counters --------------------------------------------------------------------------------------
def test_hit_stack_overflow_leaves_the_host_arrays_unwritten():
    import ctypes as C
    sc = parse(vs.csg_limit(17, True).text(".")[0])
    o = np.array(sc.camera.o[:])
    rays = np.array([np.concatenate([o, np.array([0.0, 0.0, 8.0]) - o])] * 40)
    with api.Scene(sc) as scene:
        for precision in PRECISIONS:
            with pytest.raises(api.FtbError) as e:
                scene.intersect_all(rays, 8, precision=precision)
            assert e.value.status == abi.ERR_HIT_OVERFLOW
            counts, t = np.full(40, -5, np.int32), np.full((40, 8), 7.0)
            hit = abi.HitOut(t.ctypes.data_as(C.POINTER(C.c_double)))
            rc = api.lib().ftb_intersect_all_rays(scene._h, rays.ctypes.data_as(C.POINTER(C.c_double)), 40, 8, -math.inf, math.inf,
                                                  C.byref(api.make_params(1, 1, 1, None, precision=precision)), C.byref(hit),
                                                  counts.ctypes.data_as(C.POINTER(C.c_int32)), None)
            assert rc == abi.ERR_HIT_OVERFLOW and (counts == -5).all() and (t == 7.0).all()
            scene.check_overflow()  # the host entry read (and cleared) the flag


def test_device_entry_on_a_side_stream_equals_the_host_entry_and_counts_primary_rays(tmp_path):
    import torch
    for make in (rq._variant("cubes33"), rq._large("shiny_blob")):
        sc = make(str(tmp_path))
        rays = np.concatenate(list(rq.ray_sets(sc, np.random.default_rng(11), n=500).values()))
        n = len(rays)
        with api.Scene(sc) as scene:
            side = torch.cuda.Stream()
            for precision in PRECISIONS:
                st = abi.Stats()
                hc, host = scene.intersect_all(rays, 16, -1.0, 50.0, stats=st, collect_stats=1, precision=precision)
                assert st.primary_rays == n and st.shadow_rays == 0 and st.reflection_rays == 0
                hc2, host2 = scene.intersect_all(rays, 16, -1.0, 50.0, precision=precision)
                assert np.array_equal(hc, hc2) and all(np.array_equal(host[p], host2[p]) for p in host)
                with torch.cuda.stream(side):
                    d_rays = torch.from_numpy(rays).cuda()
                    counts = torch.empty(n, dtype=torch.int32, device="cuda")
                    out = {p: torch.empty(v.shape, dtype=torch.int32 if v.dtype == np.int32 else torch.float64, device="cuda") for p, v in host.items()}
                    scene.intersect_all_device(d_rays.data_ptr(), n, 16, counts.data_ptr(), {p: v.data_ptr() for p, v in out.items()},
                                               t_min=-1.0, t_max=50.0, stream=side.cuda_stream, precision=precision)
                side.synchronize()
                scene.check_overflow(side.cuda_stream)
                assert np.array_equal(counts.cpu().numpy(), hc)
                for p, v in out.items():
                    assert np.array_equal(v.cpu().numpy(), host[p]), p
