"""CPU suite for mesh edits: scenes.edit_scene (the map it returns, the renumbering, the materials) and the argument checks made
before the library is called (no device needed: every one of them is rejected before any CUDA call)."""
import ctypes as C

import numpy as np
import pytest

from daisyriot_b200 import _lib, scenes
from daisyriot_b200.api import DeviceGroup, MeshS, OptixPrimeFunctionality


def _positions(sc):
    """per triangle: its 3 vertex positions and 3 normals (what a triangle IS, independent of the numbering)"""
    return np.concatenate([sc.vertices[sc.tri[:, :3]].reshape(-1, 9), sc.normals[sc.tri[:, 3:]].reshape(-1, 9)], 1)


def _panel():
    V, VN, T, M = [], [], [], []
    scenes._quad((0.6, 1.2, 4.6), (1.1, 0, 0), (0, 1.4, 0), 2, 2, (0, 0, 1), V, VN, T, M, 0)
    mats = [{"name": "green", "Kd": np.array([0, 1, 0], np.float32), "Ke": np.zeros(3, np.float32), "Ks": np.zeros(3, np.float32)}]
    return scenes.Scene(np.asarray(V, np.float32), np.asarray(VN, np.float32), np.asarray(T, np.int32), np.asarray(M, np.int32), mats, "panel")


def test_remove_keeps_order_and_compacts():
    sc = scenes.cornell_box(512)
    per = 512 // 16
    remove = np.arange(5 * per, 10 * per)  # the short block
    out, prev = scenes.edit_scene(sc, remove=remove)
    assert out.numtriangles == 512 - remove.size and prev.dtype == np.int32
    assert np.array_equal(prev, np.setdiff1d(np.arange(512), remove))
    assert np.all(np.diff(prev) > 0)
    assert np.array_equal(_positions(out), _positions(sc)[prev])
    assert np.array_equal(out.mat_idx, sc.mat_idx[prev])
    # compacted: every vertex and normal is used, none is lost
    assert np.array_equal(np.unique(out.tri[:, :3]), np.arange(out.vertices.shape[0]))
    assert np.array_equal(np.unique(out.tri[:, 3:]), np.arange(out.normals.shape[0]))
    assert out.normals.shape[0] == 16 - 5


@pytest.mark.parametrize("insert_at", [None, 0, 100])
def test_insert_marks_new_triangles_and_carries_materials(insert_at):
    sc = scenes.cornell_box(512)
    add = _panel()
    out, prev = scenes.edit_scene(sc, remove=[3, 4, 500], add=add, insert_at=insert_at)
    at = 509 if insert_at is None else insert_at
    assert out.numtriangles == 509 + add.numtriangles
    assert np.all(prev[at:at + add.numtriangles] == -1) and (prev >= 0).sum() == 509
    old = prev >= 0
    assert np.all(np.diff(prev[old]) > 0), "survivors keep their relative order"
    assert np.array_equal(_positions(out)[old], _positions(sc)[prev[old]])
    assert np.array_equal(_positions(out)[~old], _positions(add))
    assert np.array_equal(out.mat_idx[old], sc.mat_idx[prev[old]])
    # the added material is appended by name, the existing ones keep their ids
    assert [m["name"] for m in out.materials] == [m["name"] for m in sc.materials] + ["green"]
    assert np.all(out.mat_idx[~old] == len(sc.materials))


def test_material_matched_by_name():
    sc = scenes.cornell_box(512)
    add = _panel()
    add.materials = [dict(sc.materials[3])]  # "white"
    out, prev = scenes.edit_scene(sc, add=add)
    assert len(out.materials) == len(sc.materials) and np.all(out.mat_idx[prev < 0] == 3)


def test_bad_edits_raise():
    sc = scenes.cornell_box(512)
    with pytest.raises(ValueError):
        scenes.edit_scene(sc, remove=[512])
    with pytest.raises(ValueError):
        scenes.edit_scene(sc, add=_panel(), insert_at=600)


def _mesh(ntri):
    m = MeshS()
    m.vertices = np.zeros((4, 3), np.float32)
    m.normals = np.zeros((2, 3), np.float32)
    m.triangleIndices = np.array([[0, 1, 2, 0, 0, 0], [1, 2, 3, 1, 1, 1]] * ntri, np.int32)[:ntri]
    m.numtriangles = ntri
    return m


@pytest.mark.parametrize("cls", [OptixPrimeFunctionality, DeviceGroup])
@pytest.mark.parametrize("bad", [[0], [0, 1, 2], [0.0, 1.0], [[0, 1]]])
def test_python_mirror_checks_previous(cls, bad):
    obj = cls.__new__(cls)
    obj.mesh, obj.N = _mesh(2), 2
    obj._ctx = obj._g = None
    fn = obj.replaceMesh if cls is OptixPrimeFunctionality else obj.replace_mesh
    with pytest.raises(ValueError):
        fn(_mesh(2), np.asarray(bad))
    assert obj.N == 2 and obj.mesh.numtriangles == 2  # untouched


def test_null_context_and_group_are_rejected():
    L = _lib.lib()
    v = np.zeros((3, 3), np.float32)
    t = np.zeros((1, 6), np.int32)
    p = np.zeros(1, np.int32)
    assert L.daisy_ctx_replace_mesh(None, _lib.fptr(v), 3, _lib.fptr(v), 3, _lib.iptr(t), 1, _lib.iptr(p)) == -1
    assert L.daisy_group_replace_mesh(None, _lib.fptr(v), 3, _lib.fptr(v), 3, _lib.iptr(t), 1, _lib.iptr(p)) == -1
    assert b"null" in L.daisy_last_error()


def test_python_mirror_raises_on_a_failed_call():
    obj = OptixPrimeFunctionality.__new__(OptixPrimeFunctionality)
    obj.mesh, obj.N = _mesh(2), 2
    obj._ctx = None
    with pytest.raises(_lib.DaisyError):
        obj.replaceMesh(_mesh(1), [0])
    assert obj.N == 2
