"""Tile skipping in the fused K <= 9 gather (csrc/gather.cu: k_tile_scan, build_skip_plan, next_piece): a pass streams only the
64 x 256 tiles of F that hold a non-zero entry.  Every case runs the same passes with skipping and with the dense plan
(DAISY_GATHER_SKIP=0) and against an FP64 numpy pass."""
import ctypes as C

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu

N = 2048


@pytest.fixture(scope="module")
def scene():
    from daisyriot_b200 import scenes
    return scenes.cornell_box(N)


@pytest.fixture(scope="module")
def built(scene):
    """The Cornell box's own matrix with a band of zero rows (whole row blocks) and a band of zero columns (whole column
    steps) cut into it, on a context of its own."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(scene), rands=scenes.msvc_sample_pattern(1))
    F = p.cudaCalculateRadiosityMatrix().rows()
    F[256:512] = 0.0
    F[:, 1024:1536] = 0.0
    p.loadRadiosityMatrix(F)
    yield p, F
    p.close()


def _inputs(scene, K, seed):
    rng = np.random.RandomState(seed)
    M = rng.uniform(0, 0.6 / K, (len(scene.materials), K, K)).astype(np.float32)  # contracting: converge stops
    E = (rng.uniform(0, 5, (K, N)) * (rng.uniform(0, 1, (K, N)) < 0.2)).astype(np.float32)
    E[:, scene.mat_idx == 0] = 5.0
    return np.ascontiguousarray(E), M


def _solver(p, K, E, M, mat, skip, monkeypatch):
    from daisyriot_b200 import _lib
    monkeypatch.setenv("DAISY_GATHER_SKIP", "1" if skip else "0")
    s = C.c_void_p()
    _lib.check(_lib.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)))
    dims = np.zeros(2, np.int32)
    _lib.check(_lib.lib().daisy_solver_tile_map(s, _lib.iptr(dims), None, 0, None, None))
    assert (dims[0] > 0) == skip  # the switch selects the plan
    return s


def _dp(x):
    return x.ctypes.data_as(C.POINTER(C.c_double))


def _fp64_pass(F, R, B, M, mat):
    """residual <- M[mat] (F residual), B += residual, in FP64"""
    b = F.astype(np.float64) @ R.T                       # N x K
    y = np.einsum("ijk,ij->ik", M.astype(np.float64)[mat], b)  # column-major K x K: y[k] = sum_j M[j, k] b[j]
    R = y.T.copy()
    return R, B + R, R.sum(axis=1)


def _run(p, K, E, M, mat, skip, chained, passes, monkeypatch):
    from daisyriot_b200 import _lib
    L = _lib.lib()
    s = _solver(p, K, E, M, mat, skip, monkeypatch)
    _lib.check(L.daisy_solver_set_chained(s, int(chained)))
    sums = np.zeros(K)
    for _ in range(passes):
        _lib.check(L.daisy_solver_step(s, None if chained else _dp(sums)))
    _lib.check(L.daisy_solver_band_sums(s, _dp(sums)))
    B, R = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
    return s, B, R, sums.copy()


def _close(got, want, tol, what):
    for k in range(got.shape[0]):
        rel, small, floor = rel_err(got[k], want[k])  # over the entries above 1e-6 of the band's largest
        assert rel <= tol, (what, k, rel, floor)


@pytest.mark.parametrize("chained", [0, 1])
@pytest.mark.parametrize("K", [1, 3, 9])
def test_skip_matches_dense_and_fp64(built, scene, K, chained, monkeypatch):
    from daisyriot_b200 import _lib
    p, F = built
    L = _lib.lib()
    E, M = _inputs(scene, K, 11 + K)
    s1, B1, R1, S1 = _run(p, K, E, M, scene.mat_idx, True, chained, 4, monkeypatch)
    s0, B0, R0, S0 = _run(p, K, E, M, scene.mat_idx, False, chained, 4, monkeypatch)
    # the map has whole zero row blocks (rows 256..511) and whole zero column steps (columns 1024..1535)
    dims = np.zeros(2, np.int32)
    occ = np.zeros(32 * 8, np.uint8)
    occupied = C.c_int64()
    _lib.check(L.daisy_solver_tile_map(s1, _lib.iptr(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, C.byref(occupied), None))
    occ = occ.reshape(dims[0], dims[1])
    want = np.array([[np.any(F[r:r + 64, c:c + 256] != 0) for c in range(0, N, 256)] for r in range(0, N, 64)])
    assert np.array_equal(occ.astype(bool), want) and occupied.value == want.sum()
    assert not occ[4:8].any() and not occ[:, 4:6].any() and 0 < occupied.value < occ.size
    _close(B1, B0, 1e-6, "B skip vs dense")
    _close(R1, R0, 1e-6, "residual skip vs dense")
    assert np.allclose(S1, S0, rtol=1e-7, atol=0)
    R, B = E.astype(np.float64), E.astype(np.float64)
    for _ in range(4):
        R, B, sums = _fp64_pass(F, R, B, M, scene.mat_idx)
    _close(B1, B, 1e-5, "B vs fp64")
    _close(R1, R, 1e-5, "residual vs fp64")
    assert np.allclose(S1, sums, rtol=1e-5)
    # the same stop decision
    n = {}
    for key, s in (("skip", s1), ("dense", s0)):
        _lib.check(L.daisy_solver_reset(s))
        c = C.c_int()
        _lib.check(L.daisy_solver_converge(s, 1e-2 * float(E.sum()), 0, 200, C.byref(c)))
        n[key] = c.value
        L.daisy_solver_destroy(s)
    assert n["skip"] == n["dense"] and n["skip"] > 1


@pytest.mark.parametrize("case", ["all_zero", "last_entry_only"])
def test_degenerate_matrices(scene, case, monkeypatch):
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    K = 3
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(scene), rands=scenes.msvc_sample_pattern(1))
    F = np.zeros((N, N), np.float32)
    if case == "last_entry_only":
        F[N - 1, N - 1] = 0.5  # the last column of the last tile
    p.loadRadiosityMatrix(F)
    E, M = _inputs(scene, K, 5)
    E[:, N - 1] = 2.0
    got = {}
    for skip in (True, False):
        s, B, R, S = _run(p, K, E, M, scene.mat_idx, skip, 0, 2, monkeypatch)
        got[skip] = (B, R, S)
        from daisyriot_b200 import _lib
        _lib.lib().daisy_solver_destroy(s)
    R, B = E.astype(np.float64), E.astype(np.float64)
    for _ in range(2):
        R, B, sums = _fp64_pass(F, R, B, M, scene.mat_idx)
    for skip in (True, False):
        Bg, Rg, Sg = got[skip]
        _close(Bg, B, 1e-5, (case, skip, "B"))
        _close(Rg, R, 1e-5, (case, skip, "residual"))
        assert np.allclose(Sg, sums, rtol=1e-5, atol=1e-30)
    if case == "all_zero":
        assert not got[True][1].any() and np.array_equal(got[True][0], E)
    else:
        assert got[True][1][:, N - 1].all() and not got[True][1][:, :N - 1].any()
    p.close()


def test_write_rows_after_solver_exists(scene, monkeypatch):
    """A row block zeroed and an entry put into an empty tile after the solver was created: the next pass sees both."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    L = _lib.lib()
    K = 3
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(scene), rands=scenes.msvc_sample_pattern(1))
    F = p.cudaCalculateRadiosityMatrix().rows()
    F[:64, 1792:] = 0.0  # an empty tile: row block 0, column step 7
    p.loadRadiosityMatrix(F)
    E, M = _inputs(scene, K, 21)
    E[:] = 1.0
    s = _solver(p, K, E, M, scene.mat_idx, True, monkeypatch)
    _lib.check(L.daisy_solver_step(s, None))
    dims = np.zeros(2, np.int32)
    occ = np.zeros(32 * 8, np.uint8)
    _lib.check(L.daisy_solver_tile_map(s, _lib.iptr(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, None, None))
    occ = occ.reshape(dims[0], dims[1])
    assert occ[2].any()
    rb, cs = map(int, np.argwhere(occ == 0)[0])
    F[128:192] = 0.0                                    # row block 2
    F[rb * 64 + 5, cs * 256 + 7] = 0.25                 # one entry into a tile that was empty
    p.loadRadiosityMatrix(F[128:192], row0=128)
    p.loadRadiosityMatrix(F[rb * 64 + 5:rb * 64 + 6], row0=rb * 64 + 5)
    Bg, Rg = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
    _lib.check(L.daisy_solver_step(s, None))
    B2, R2 = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B2), _lib.fptr(R2)))
    R, B, _ = _fp64_pass(F, Rg.astype(np.float64), Bg.astype(np.float64), M, scene.mat_idx)
    _close(R2, R, 1e-5, "residual after write_rows")
    _close(B2, B, 1e-5, "B after write_rows")
    assert not R2[:, 128:192].any() and R2[:, rb * 64 + 5].all()
    _lib.check(L.daisy_solver_tile_map(s, _lib.iptr(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, None, None))
    assert not occ[2].any() and occ[rb, cs] == 1
    L.daisy_solver_destroy(s)
    p.close()


def test_two_gpus_rank_without_tiles_in_a_peer_block(scene, monkeypatch):
    """Fused exchange on two GPUs with a matrix in which rank 0 has no occupied tile in rank 1's column block: its CTAs never
    wait on rank 1's flag while streaming, yet must not overwrite the buffer rank 1 is still reading.  Pass counts and B equal
    the single GPU's, and no exchange timeout fires."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    L = _lib.lib()
    if L.daisy_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setenv("DAISY_GATHER_SKIP", "1")
    monkeypatch.setenv("DAISY_EXCHANGE_TIMEOUT_MS", "20000")
    uv = scenes.msvc_sample_pattern(1)
    mesh = dz.MeshS.from_scene(scene)
    p = dz.OptixPrimeFunctionality(mesh, rands=uv)
    F = p.cudaCalculateRadiosityMatrix().rows()
    F[:N // 2, N // 2:] = 0.0
    p.loadRadiosityMatrix(F)
    grp = dz.DeviceGroup(mesh, devices=[0, 1], rands=uv)
    _lib.check(L.daisy_group_formfactors_write_rows(grp._g, 0, N, _lib.fptr(F)))
    K = 9
    E, M = _inputs(scene, K, 31)
    s = _solver(p, K, E, M, scene.mat_idx, True, monkeypatch)
    gs = dz.GroupSolver(grp, K, E, M, scene.mat_idx)
    for _ in range(3):
        t = np.zeros(K)
        _lib.check(L.daisy_solver_step(s, _dp(t)))
        assert np.allclose(gs.step(True), t, rtol=1e-6)
    for _ in range(20):  # back to back: rank 0 finishes its passes quickly and would run ahead without the flag wait
        gs.step(False)
        _lib.check(L.daisy_solver_step(s, None))
    B1, R1 = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B1), _lib.fptr(R1)))
    B2, R2 = gs.read()
    _close(B2, B1, 1e-5, "B 2 GPUs vs 1")
    _close(R2, R1, 1e-5, "residual 2 GPUs vs 1")
    _lib.check(L.daisy_solver_reset(s))
    gs.reset()
    n1 = C.c_int()
    thr = 1e-3 * float(E.sum())
    _lib.check(L.daisy_solver_converge(s, thr, 0, 500, C.byref(n1)))
    assert gs.converge(thr, False, 500) == n1.value and n1.value > 3
    gs.close()
    grp.close()
    L.daisy_solver_destroy(s)
    p.close()
