"""Shared helpers for the parity tests."""
import os

import numpy as np

from functracer_b200 import abi, frontend, scenes
from oracle import ftb_oracle as orc


def parse(text, assets=None):
    return frontend.ParsedScene(text, assets or scenes.asset_dir())


def one_object_scene(obj, lights="", camera="camera pos (0,0,-5) lookat (0,0,0) up (0,1,0) fov 60 ratio 1"):
    return camera + "\nsamples 1\n\n" + obj + "\n\n" + lights + ("\n" if lights else "")


def oracle_render(sc, width=None, height=None, spp=None, seed=1, rng_seed=1234, sampling=None, **kw):
    width = width or sc.width
    height = height or sc.height
    spp = spp or sc.spp
    sampling = sc.sampling if sampling is None else sampling
    jit = frontend.jitter_pattern(seed, spp)
    p = orc.make_params(width, height, spp, jit, sampling=sampling, seed=rng_seed, **kw)
    return orc.render(sc, p), p


def colour_stats(a, b):
    """Per-pixel max-channel error statistics in 1/255 units."""
    d = np.abs(np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)).max(axis=-1)
    return dict(max=float(d.max()), frac_within=float((d <= 1.0 / 255.0).mean()))


# ---- the reference's own scene files: Scenes/ of an antonburger/FuncTracer checkout named by FTB_REFERENCE_DIR ----
# (not part of this repository; the tests that read them skip without it)
REFERENCE_SCENES = os.path.join(os.environ["FTB_REFERENCE_DIR"], "Scenes") if os.environ.get("FTB_REFERENCE_DIR") else None
# the three assets the reference does not ship -> the generated stand-ins (functracer_b200/scenes.py)
ASSET_SUBSTITUTES = {
    "c:\\Temp\\env4.jpg": "env4.ppm",
    "http://richardandersson.net/wp-content/uploads/2016/08/Moon.Diffuse_21600x10800-1024x512.jpg": "moon.ppm",
    "..\\stanford bunny\\reconstruction\\bun_zipper_res4.ply": "bunny_res4.ply",
}


def reference_scene_text(file_name, res=None, spp=None, mesh=None, depth=None):
    """The text of the reference's Scenes/<file_name> with only what BASELINE.md §3 allows changed: `res` / `samples`
    option lines inserted after the scene's own option lines (the grammar is options -> objects -> lights and later
    setters win, SceneParser.fs:357-364), the three missing asset paths substituted, and house.scene:17 (a comment
    inside a group: a parse error at HEAD) dropped."""
    import re
    lines = open(os.path.join(REFERENCE_SCENES, file_name), encoding="utf-8").read().splitlines()
    if file_name == "house.scene":
        assert lines[16].lstrip().startswith(";Bug"), lines[16]
        del lines[16]
    last_option = max(i for i, l in enumerate(lines) if re.match(r"\s*(camera|samples|res)\b", l, re.I))
    extra = []
    if spp is not None:
        extra.append("samples %s" % spp)
    if res is not None:
        extra.append("res %d %d" % tuple(res))
    lines[last_option + 1:last_option + 1] = extra
    text = "\n".join(lines) + "\n"
    for old, new in ASSET_SUBSTITUTES.items():
        text = text.replace('"%s"' % old, '"%s"' % new)
    if mesh is not None:
        text = text.replace('"bunny_res4.ply"', '"%s"' % mesh)
    if depth is not None:
        text, n = re.subn(r"bspMesh\s+\d+", "bspMesh %d" % depth, text)
        assert n == 1
    return text


def desc_tables(sc):
    """Every table of a ParsedScene's ftb_scene_desc (+ camera and options) as plain Python / numpy values, for
    field-by-field comparison."""
    import ctypes as C
    d = sc.desc

    def rows(ptr, n, fields):
        out = []
        for i in range(n):
            r = ptr[i]
            out.append(tuple(tuple(getattr(r, f)) if hasattr(getattr(r, f), "__len__") else getattr(r, f) for f in fields))
        return out

    t = {
        "root": d.root,
        "nodes": rows(d.nodes, d.n_nodes, ["kind", "a", "b"]),
        "children": [d.children[i] for i in range(d.n_children)],
        "transforms": rows(d.transforms, d.n_transforms, ["m2w", "w2m"]),
        "materials": rows(d.materials, d.n_materials, ["colour", "roughness", "reflectance", "shineyness", "apply_lighting"]),
        "textures": rows(d.textures, d.n_textures, ["kind", "inner", "image", "p"]),
        "images": [(d.images[i].width, d.images[i].height, C.string_at(d.images[i].rgb24, 3 * d.images[i].width * d.images[i].height)) for i in range(d.n_images)],
        "meshes": rows(d.meshes, d.n_meshes, ["root"]),
        "bsp_nodes": rows(d.bsp_nodes, d.n_bsp_nodes, ["aabb_min", "aabb_max", "left", "right"]),
        "bsp_leaves": rows(d.bsp_leaves, d.n_bsp_leaves, ["tri_first", "tri_count"]),
        "triangles": np.ctypeslib.as_array(d.triangles, shape=(d.n_triangles, 9)).copy() if d.n_triangles else np.zeros((0, 9)),
        "lights": rows(d.lights, d.n_lights, ["kind", "samples", "v", "falloff", "scatter_rad", "colour"]),
        "camera": tuple(tuple(getattr(sc.camera, f)) if hasattr(getattr(sc.camera, f), "__len__") else getattr(sc.camera, f)
                        for f in ["o", "look_at", "up", "fov_y_rad", "aspect_ratio", "has_focus", "focal_length", "aperture_rad"]),
        "options": (sc.width, sc.height, sc.spp, sc.sampling),
    }
    return t
