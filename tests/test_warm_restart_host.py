"""Host-side parts of the warm restart: remap_bands, the argument checks of the Python surface, and the C-ABI declarations."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_remap_bands_keeps_survivors_and_seeds_new_triangles_with_E():
    from daisyriot_b200 import remap_bands
    B = np.arange(12, dtype=np.float32).reshape(3, 4)
    E = np.full((3, 5), -1.0, np.float32)
    prev = np.array([3, -1, 0, 0, -1])
    out = remap_bands(B, prev, E)
    assert out.dtype == np.float32 and out.shape == (3, 5) and out.flags.c_contiguous
    assert np.array_equal(out[:, 0], B[:, 3]) and np.array_equal(out[:, 2], B[:, 0]) and np.array_equal(out[:, 3], B[:, 0])
    assert np.array_equal(out[:, 1], E[:, 1]) and np.array_equal(out[:, 4], E[:, 4])
    assert np.array_equal(B, np.arange(12, dtype=np.float32).reshape(3, 4)), "B_old is not modified"


def test_remap_bands_with_scenes_edit_scene():
    from daisyriot_b200 import remap_bands, scenes
    sc = scenes.cornell_box(512)
    sc_new, prev = scenes.edit_scene(sc, remove=np.arange(10, 40), add=scenes.cornell_panel(512), insert_at=100)
    K = 3
    B = np.random.RandomState(0).uniform(0, 1, (K, sc.numtriangles)).astype(np.float32)
    E = np.random.RandomState(1).uniform(0, 1, (K, sc_new.numtriangles)).astype(np.float32)
    out = remap_bands(B, prev, E)
    kept = prev >= 0
    assert np.array_equal(out[:, kept], B[:, prev[kept]])
    assert np.array_equal(out[:, ~kept], E[:, ~kept])
    assert (~kept).sum() == scenes.cornell_panel(512).numtriangles


@pytest.mark.parametrize("bad", ["length", "range_hi", "range_lo", "float", "bands"])
def test_remap_bands_refuses(bad):
    from daisyriot_b200 import remap_bands
    B = np.zeros((2, 4), np.float32)
    E = np.zeros((2, 3), np.float32)
    prev = np.array([0, 1, -1])
    if bad == "length":
        prev = np.array([0, 1])
    elif bad == "range_hi":
        prev = np.array([0, 4, -1])
    elif bad == "range_lo":
        prev = np.array([0, -2, 1])
    elif bad == "float":
        prev = np.array([0.0, 1.0, -1.0])
    else:
        E = np.zeros((3, 3), np.float32)
    with pytest.raises(ValueError):
        remap_bands(B, prev, E)


def test_material_arrays_check_shapes():
    from daisyriot_b200.api import _material_arrays
    M, mat = _material_arrays(np.zeros((2, 3, 3)), [0, 1, 1], 3, 3)
    assert M.dtype == np.float32 and mat.dtype == np.int32
    with pytest.raises(ValueError):
        _material_arrays(np.zeros((2, 3, 3)), [0, 1], 3, 3)
    with pytest.raises(ValueError):
        _material_arrays(np.zeros((2, 2, 3)), [0, 1, 1], 3, 3)


def test_entry_points_declared_and_bound():
    from daisyriot_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "daisy_b200.h")).read()
    for name, nargs in (("daisy_solver_restart", 2), ("daisy_solver_set_emission", 2), ("daisy_solver_set_materials", 4),
                        ("daisy_group_solver_restart", 2), ("daisy_group_solver_set_emission", 2), ("daisy_group_solver_set_materials", 4)):
        m = re.search(r"\bint\s+%s\s*\(([^)]*)\)" % name, hdr)
        assert m, name
        assert len(m.group(1).split(",")) == nargs, name
        assert len(_lib.SYMBOLS[name][1]) == nargs, name


def test_shim_exposes_restart():
    src = open(os.path.join(ROOT, "shim", "Lightning.h")).read()
    assert "void restart()" in src and "void reconverge_lightning()" in src
    assert "daisy_group_solver_restart" in src
