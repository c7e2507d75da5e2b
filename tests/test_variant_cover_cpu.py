"""Which FP32 kernel each scene of tests/variant_scenes.py runs on, with the real lowering (lower.cpp compiled into the probe of
tests/test_lowering_cpu.py) and api.cu pickVariant over the variants the Makefile compiles.  CPU only.

tests/test_gpu_variants.py holds each specialised kernel to the oracle and to the exact fold on these scenes; that is only
coverage while each scene still lands on the kernel it was written for.  So every scene (and its unlit fold twin) must land
there, and every specialised variant must be reached by at least MIN_SCENES of them."""
import collections
import ctypes as C
import os
import subprocess

import pytest

import test_lowering_cpu as low
import variant_scenes as vs
from functracer_b200 import abi

MIN_SCENES = 2


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    d = tmp_path_factory.mktemp("variant_probe")
    src, so = os.path.join(str(d), "probe.cpp"), os.path.join(str(d), "libprobe.so")
    open(src, "w").write(low.PROBE % dict(csrc=low.CSRC, tests=os.path.dirname(os.path.abspath(__file__))))
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-o", so, src, os.path.join(low.CSRC, "cuda", "lower.cpp")])
    lib = C.CDLL(so)
    lib.ftb_probe_lower.argtypes = [C.POINTER(abi.SceneDesc), C.POINTER(C.c_uint), C.POINTER(C.c_int), C.c_char_p, C.c_int]
    lib.ftb_probe_lower.restype = C.c_int
    return lib


def test_every_variant_scene_lands_on_its_kernel(probe, tmp_path):
    low.constants_agree_with_the_sources()
    variants = low.compiled_variants()
    specialised = [v for v in variants if v != low.FT_ALL]
    per = collections.Counter()
    rows = []
    for s in vs.all_scenes() + vs.over_limit_scenes():
        d = tmp_path / s.name
        d.mkdir()
        text, assets = s.text(str(d))
        need, counts = low.lowered(probe, text, assets)
        got = low.pick(need, variants)
        ftext, fassets, _ = s.fold(str(d), 3)
        fneed, _ = low.lowered(probe, ftext, fassets)
        fgot = low.pick(fneed, variants)
        rows.append("%-24s needs 0x%03x -> 0x%03x (fold twin 0x%03x -> 0x%03x), %4d items %5d leaves" % (s.name, need, got, fneed, fgot, counts[0], counts[1]))
        assert got == s.variant, rows[-1]
        assert fgot == s.variant, rows[-1]
        per[got] += 1
    print("\n".join(rows))
    print("scenes per variant: " + ", ".join("0x%03x: %d" % (v, per[v]) for v in specialised))
    assert set(per) <= set(specialised)
    for v in specialised:
        assert per[v] >= MIN_SCENES, "variant 0x%03x is reached by %d scenes" % (v, per[v])


def test_the_table_scenes_cross_its_batch_and_padding_boundaries(probe, tmp_path):
    """The 0x209 item counts: both sides of a 32-item batch and of the odd-count padding row, the largest count whose table
    fits with the scene's lights (lower.h wantsOriginTable), and a scene padded past it, which keeps the variant (the table
    bit is dropped, not the kernel) but runs without the table."""
    hdr = open(os.path.join(low.CSRC, "cuda", "lower.h")).read()
    assert "kOriginCap = 256;" in hdr and "((n_items + 1) & ~1)" in hdr
    nl = len(vs.CUBE_LIGHTS)
    top = vs.max_table_items(nl)
    assert (1 + nl) * ((top + 1) & ~1) <= 256 < (1 + nl) * ((top + 2) & ~1)
    seen = {}
    for s in vs.all_scenes():
        if s.variant != 0x209:
            continue
        need, counts = low.lowered(probe, s.text(str(tmp_path))[0])
        seen[s.name] = (counts[0], bool(need & low.FT_TABLE))
    print(seen)
    counts = {n for n, table in seen.values() if table}
    assert {8, 9, 31, 32, 33, 64, 65, top - 1, top} <= counts
    assert any(n > top and not table for n, table in seen.values())
