"""Small-N runs of the three hot kernels for compute-sanitizer (tools/sanitize.sh): k_ff_tiles (form factors + masks),
k_gather_tma<9> (fused epilogue, several column splits), k_gather_mma<32> and k_gather_mma<64> (tcgen05).  Results are checked against the
oracle so that a sanitizer run is also a parity run."""
import ctypes as C
import sys

import numpy as np

sys.path.insert(0, ".")
import daisyriot_b200 as dz  # noqa: E402
from daisyriot_b200 import _lib, scenes  # noqa: E402

what = sys.argv[1] if len(sys.argv) > 1 else "ff"
uv = scenes.msvc_sample_pattern(1)
L = dz.lib()
if what == "ff":
    from oracle import pyoracle
    sc = scenes.cornell_box(512)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), rands=uv)
    F = p.cudaCalculateRadiosityMatrix().rows()
    m = p.visibilityMasks(0, 64)
    F_ref, m_ref, _ = pyoracle.Oracle.from_scene(sc).radmat_rows(uv, 0, 64)
    assert np.array_equal(F[:64].view(np.uint32), F_ref.view(np.uint32)) and np.array_equal(m, m_ref)
    print("ff ok", p.stats())
    p.close()
else:
    K = {"gather9": 9, "gather32": 32, "gather64": 64}[what]
    N = 4096 if K == 9 else 1024
    sc = scenes.cornell_box(N)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), rands=uv)
    rng = np.random.RandomState(1)
    F = (rng.uniform(0, 1, (N, N)) * (rng.uniform(0, 1, (N, N)) < 0.3) / N).astype(np.float32)
    p.loadRadiosityMatrix(F)
    M = rng.uniform(0, 0.05, (len(sc.materials), K, K)).astype(np.float32)
    E = np.ascontiguousarray(rng.uniform(0, 3, (K, N)).astype(np.float32))
    s = C.c_void_p()
    _lib.check(L.daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(sc.mat_idx), C.byref(s)))
    sums = np.zeros(K)
    for _ in range(2):
        _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
    B, R = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
    b1 = np.einsum("pji,jp->ip", M.astype(np.float64)[sc.mat_idx], E.astype(np.float64) @ F.astype(np.float64).T)
    b2 = np.einsum("pji,jp->ip", M.astype(np.float64)[sc.mat_idx], b1 @ F.astype(np.float64).T)
    assert np.allclose(R, b2, rtol=1e-5, atol=1e-12), np.abs(R - b2).max()
    print(what, "ok, launches per pass", L.daisy_solver_launches_per_pass(s))
    L.daisy_solver_destroy(s)
    p.close()
