"""CPU suite: the device-converge entry points reject a null solver before touching any device."""
import ctypes as C

from daisyriot_b200 import _lib


def test_converge_device_null_solver_is_invalid():
    L = _lib.lib()
    n = C.c_int(-7)
    assert L.daisy_solver_converge_device(None, 1.0, 0, 0, C.byref(n)) == -1            # DAISY_E_INVALID
    assert L.daisy_group_solver_converge_device(None, 1.0, 1, 5, C.byref(n)) == -1
    assert n.value == -7
