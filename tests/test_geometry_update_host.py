"""CPU suite: argument and state errors of the geometry-update entry points (no device needed: every one of them is rejected
before any CUDA call), and the Python mirror raising on them."""
import ctypes as C

import numpy as np
import pytest

from daisyriot_b200 import _lib
from daisyriot_b200.api import DeviceGroup, MeshS, OptixPrimeFunctionality


def test_null_context_and_group_are_rejected():
    L = _lib.lib()
    v = np.zeros((3, 3), np.float32)
    i64, d = C.c_int64(), C.c_double()
    assert L.daisy_ctx_update_geometry(None, _lib.fptr(v), 3, _lib.fptr(v), 3) == -1
    assert L.daisy_formfactors_update(None, 0) == -1
    assert L.daisy_formfactors_update_stats(None, C.byref(i64), C.byref(i64), C.byref(i64), C.byref(d)) == -1
    assert L.daisy_group_update_geometry(None, _lib.fptr(v), 3, _lib.fptr(v), 3) == -1
    assert L.daisy_group_formfactors_update(None, 0) == -1
    assert b"null" in L.daisy_last_error()


def _mesh():
    m = MeshS()
    m.vertices = np.zeros((4, 3), np.float32)
    m.normals = np.zeros((2, 3), np.float32)
    m.triangleIndices = np.array([[0, 1, 2, 0, 0, 0], [1, 2, 3, 1, 1, 1]], np.int32)
    m.numtriangles = 2
    return m


@pytest.mark.parametrize("cls", [OptixPrimeFunctionality, DeviceGroup])
@pytest.mark.parametrize("bad", ["vertices", "normals"])
def test_python_mirror_raises_on_count_mismatch(cls, bad):
    obj = cls.__new__(cls)
    obj.mesh = _mesh()
    obj._ctx = obj._g = None
    kw = {bad: np.zeros((5, 3), np.float32)}
    fn = obj.updateGeometry if cls is OptixPrimeFunctionality else obj.update_geometry
    with pytest.raises(ValueError):
        fn(**kw)
    assert obj.mesh.vertices.shape == (4, 3) and obj.mesh.normals.shape == (2, 3)  # the mesh is untouched


def test_python_mirror_raises_on_a_failed_call():
    obj = OptixPrimeFunctionality.__new__(OptixPrimeFunctionality)
    obj.mesh = _mesh()
    obj._ctx = None
    with pytest.raises(_lib.DaisyError):
        obj.updateGeometry()
    with pytest.raises(_lib.DaisyError):
        obj.updateRadiosityMatrix()
