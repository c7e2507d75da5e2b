"""Scene texts enlarged by s and moved by T (test infrastructure for tests/test_scale_proofs_cpu.py and tests/test_gpu_scale.py).

scaled(text, s, T) wraps each top-level object as (translate T (scale s OBJ)), maps the camera's pos and lookat and a positional
light's pos to s p + T, scales the camera's focal length by s and a positional light's falloff (c, l, q) to (c, l / s, q / s^2);
directional and soft-directional lights keep their direction.  In exact arithmetic the picture does not change (attenuation
c + l d + q d^2 is the same at the distance s d).  The reference's own offsets are absolute (slightOffset 1e-4 d, the shadow
ray's origin 1e-4 n, the plane's |d.n| < 1e-7), so the oracle's picture at the extremes differs slightly from the unscaled one;
every case is compared with the oracle rendered at the same s and T.

SWEEP holds the (s, T) pairs: s a power of two (the scaling itself is exact), T up to 1.4e4 from the origin; small objects far out
and large objects near the origin both appear.  FAMILIES builds the scenes: house, night-house and repeat (ground plane,
directional and point lights, clear and lit tiles), hollow-sphere (reflections and CSG), one small-mesh scene of the 0x004 variant
and ACNE, five primitive classes on a matte ground under a 40-degree directional light and a point light."""
import re

import variant_scenes as vs
from functracer_b200 import scenes

OPTIONS = ("camera", "samples", "res")
LIGHTS = ("directional", "softdirectional", "positional")

_TRIPLE = r"\(\s*([^,()]+?)\s*,\s*([^,()]+?)\s*,\s*([^,()]+?)\s*\)"


def _g(x):
    return "%.17g" % x


def _triple(v):
    return "(%s)" % ",".join(_g(float(x)) for x in v)


def _keyword_triple(line, kw, f):
    """`kw (x,y,z)` in line with its triple replaced by f([x, y, z])."""
    return re.sub(r"(%s\s*)" % kw + _TRIPLE, lambda m: m.group(1) + _triple(f([float(m.group(i)) for i in (2, 3, 4)])), line, flags=re.I)


def _first_word(line):
    m = re.match(r"\s*([A-Za-z]+)", line)
    return m.group(1).lower() if m else ""


def split_objects(text):
    """The top-level object forms of an object section: balanced (...) forms, and a bare primitive on a line of its own."""
    out, i, n = [], 0, len(text)
    while i < n:
        if text[i].isspace():
            i += 1
            continue
        if text[i] == "(":
            depth, j = 0, i
            while True:
                if text[j] == "(":
                    depth += 1
                elif text[j] == ")":
                    depth -= 1
                    if depth == 0:
                        break
                j += 1
            out.append(text[i:j + 1])
            i = j + 1
        else:
            j = text.find("\n", i)
            j = n if j < 0 else j
            out.append(text[i:j].strip())
            i = j
    return out


def _camera(line, s, T):
    move = lambda p: [s * p[i] + T[i] for i in range(3)]
    line = _keyword_triple(_keyword_triple(line, "pos", move), "lookat", move)
    return re.sub(r"(focus\s*)\(\s*([^,()]+?)\s*,\s*([^,()]+?)\s*\)",
                  lambda m: "%s(%s,%s)" % (m.group(1), _g(s * float(m.group(2))), m.group(3)), line, flags=re.I)


def _light(line, s, T):
    if _first_word(line) != "positional":
        return line
    line = _keyword_triple(line, "pos", lambda p: [s * p[i] + T[i] for i in range(3)])
    return _keyword_triple(line, "falloff", lambda f: [f[0], f[1] / s, f[2] / (s * s)])


def scaled(text, s, T=(0.0, 0.0, 0.0)):
    """The scene of `text` enlarged by s about the origin, then moved by T."""
    s, T = float(s), [float(x) for x in T]
    options, objects, lights = [], [], []
    for line in text.splitlines():
        line = line.split(";", 1)[0].rstrip()
        w = _first_word(line)
        if w in OPTIONS:
            options.append(_camera(line, s, T) if w == "camera" else line)
        elif w in LIGHTS:
            lights.append(_light(line, s, T))
        else:
            objects.append(line)
    wrapped = ["(translate %s (scale %s %s))" % (_triple(T), _g(s), " ".join(o.split())) for o in split_objects("\n".join(objects))]
    return "\n".join(options) + "\n\n" + "\n\n".join(wrapped) + "\n\n" + "\n".join(lights) + "\n"


# ---- the sweep ---------------------------------------------------------------------------------------------------------------
ORIGIN = (0.0, 0.0, 0.0)
SWEEP = [
    (1.0, ORIGIN),
    (2.0 ** -10, ORIGIN),              # small objects near the origin
    (2.0 ** 10, ORIGIN),               # large objects: the camera 2e4 out
    (2.0 ** -5, (1e2, 0.0, 0.0)),      # small objects far out
    (1.0, (1e2, 0.0, 0.0)),
    (1.0, (1e3, 1e3, -1e3)),
    (2.0 ** -5, (1e3, 1e3, -1e3)),     # small objects farther out
    (1.0, (1e4, 0.0, 1e4)),
    (2.0 ** 5, (1e4, 0.0, 1e4)),       # large objects far out
]


def case_id(s, T):
    """A short id: s as a power of two, T by its largest component, e.g. 's-5_T1e2'."""
    import math
    e = int(round(math.log2(s)))
    t = max(abs(x) for x in T)
    return "s%d_T%s" % (e, "0" if t == 0 else "1e%d" % int(round(math.log10(t))))


# ---- the families ------------------------------------------------------------------------------------------------------------
ACNE = """camera pos (0,1.5,-7) lookat (-2.5,-1.4,0) up (0,1,0) fov 50 ratio 1
samples 2

(material diffuse (0.8,0.8,0.75) reflectance 0 shineyness 0 (translate (0,-1,0) plane))
(material diffuse (0.9,0.3,0.2) reflectance 0.5 shineyness 20 (translate (-2,0,0.5) sphere))
(material diffuse (0.2,0.6,0.9) reflectance 0 shineyness 10 (translate (0,-0.3,1) (rotate (0,1,0) 30 (scale 0.7 cube))))
(material diffuse (0.3,0.8,0.3) reflectance 0.5 shineyness 0 (translate (2,-1,0.5) (scale (0.6,1.4,0.6) solidCylinder)))
(material diffuse (0.9,0.8,0.2) reflectance 0 shineyness 20 (translate (-0.8,-1,-1.6) (scale (0.6,1.2,0.6) cone)))
(material diffuse (0.7,0.6,0.8) reflectance 0.5 shineyness 10 (translate (1,-1.05,-1.8) (scale 9 (translate (0.017,-0.11,0) mesh "bunny_tiny.ply"))))

directional dir (0.6128,-0.6428,0.4596) colour (0.8,0.8,0.8)
positional pos (-2,4,-3) falloff (1,0.05,0.01) colour (0.7,0.7,0.6)
"""


def _bundled(name):
    return lambda d, res, spp: (getattr(scenes, name)(res=res, spp=spp), scenes.asset_dir())


def _meshes(d, res, spp):
    return vs.small_meshes(0).text(d, spp=spp, res=res)


def _acne(d, res, spp):
    return ACNE.replace("samples 2", "samples %d\nres %d %d" % (spp, res[0], res[1])), scenes.asset_dir()


# family -> builder(directory, res, spp) -> (unscaled scene text, asset directory)
FAMILIES = {
    "house": _bundled("house"),
    "night_house": _bundled("night_house"),
    "repeat": _bundled("repeat"),
    "hollow_sphere": _bundled("hollow_sphere"),
    "meshes": _meshes,
    "acne": _acne,
}


def family_text(family, d, res, spp, s=1.0, T=ORIGIN):
    """(the family's scene text scaled by s and moved by T, asset directory)."""
    text, assets = FAMILIES[family](d, res, spp)
    return scaled(text, s, T), assets
