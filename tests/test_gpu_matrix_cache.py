"""The matrix cache on the device: F handed back as CSC (daisy_formfactors_to_csc, daisy_group_formfactors_to_csc) and a CSC
matrix loaded into F (daisy_formfactors_write_csc, daisy_group_formfactors_write_csc).

Export: bit-identical to the host conversion (DAISY_CSC_HOST=1) and to a numpy statement of the rule -- entry (r, c) is listed
exactly when its bits other than the sign are not all zero -- on built matrices of several sizes, both variants, with small
staging buffers (many column chunks) too, and on special values.  Import: the rows read back and the device row digests equal
the expected dense matrix bit for bit; solvers, updates and partitions see what a dense load gives them; invalid input changes
nothing."""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FFD, FFH = 0, 1
E_INVALID = -1
SMALL_STAGE = "65536"  # bytes: a few thousand entries per staging chunk


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


@pytest.fixture(scope="module")
def uv():
    from daisyriot_b200 import scenes
    return scenes.msvc_sample_pattern(1)


def sub_scene(N):
    """The first N triangles of a Cornell box of 32 * ceil(N / 32) patches."""
    from daisyriot_b200 import scenes
    from daisyriot_b200.scenes import Scene
    sc = scenes.cornell_box(32 * math.ceil(N / 32))
    return Scene(sc.vertices, sc.normals, sc.tri[:N], sc.mat_idx[:N], sc.materials, "cornell_first_%d" % N)


def scene(name):
    import os
    from daisyriot_b200 import scenes
    from conftest import GOLDEN
    if name in ("cornellbox_blacklight", "colorballs"):
        return scenes.load_scene_npz(os.path.join(GOLDEN, name + ".npz"))
    if name.startswith("cornell_box_"):
        return scenes.cornell_box(int(name.split("_")[-1]))
    return sub_scene(int(name.split("_")[-1]))


def ctx(dz, sc, uv, **kw):
    return dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv, **kw)


def csc_rule(F):
    """numpy statement of the export: columns ascending, rows ascending within a column, listed iff (bits & 0x7fffffff) != 0"""
    F = np.ascontiguousarray(F, np.float32)
    mask = (F.view(np.uint32) & np.uint32(0x7fffffff)) != 0
    cols, rows = np.nonzero(mask.T)
    outer = np.concatenate([[0], np.cumsum(mask.sum(axis=0))]).astype(np.int32)
    return F[rows, cols], rows.astype(np.int32), outer


def dense_of(vals, inner, outer, N):
    """expected F after an import: listed values bit for bit, +0.0 elsewhere"""
    D = np.zeros((N, N), np.float32)
    for c in range(N):
        s, e = outer[c], outer[c + 1]
        D[inner[s:e], c] = vals[s:e]
    return D


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32 if a.dtype == np.float32 else a.dtype), b.view(np.uint32 if b.dtype == np.float32 else b.dtype))


def assert_csc(got, want, what):
    for k, name in enumerate(("values", "inner", "outer")):
        assert bits_equal(got[k], want[k]), (what, name)


def count_only(dz, p):
    nnz = C.c_int64(-1)
    dz.lib().daisy_formfactors_to_csc(p._ctx, C.byref(nnz), None, None, None)
    return nnz.value


def write_csc_rc(dz, p, vals, inner, outer):
    from daisyriot_b200 import _lib
    v = np.ascontiguousarray(vals, np.float32)
    i = np.ascontiguousarray(inner, np.int32)
    o = np.ascontiguousarray(outer, np.int32)
    return dz.lib().daisy_formfactors_write_csc(p._ctx, v.size, _lib.fptr(v), _lib.iptr(i), _lib.iptr(o))


def assert_holds(p, want, what):
    """rows read back and device digests of p's row range equal want's rows bit for bit"""
    from daisyriot_b200 import api
    r0, r1 = p.row_range
    assert bits_equal(_rows(p), want[r0:r1]), (what, "rows")
    if r1 > r0:
        x, w = _radmat(p).row_digest()
        hx, hw = api.row_digest_host(want[r0:r1])
        assert np.array_equal(x, hx) and np.array_equal(w, hw), (what, "digests")


def _radmat(p):
    from daisyriot_b200.api import RadMat
    return RadMat(p)


def _rows(p):
    return _radmat(p).rows()


def random_csc(N, density, seed, specials=True):
    rng = np.random.RandomState(seed)
    mask = rng.uniform(0, 1, (N, N)) < density
    F = np.where(mask, rng.uniform(1e-6, 1.0, (N, N)), 0.0).astype(np.float32)
    cols, rows = np.nonzero(mask.T)
    vals = F[rows, cols].copy()
    if specials and vals.size >= 4:  # listed -0.0, explicit +0.0, a NaN with a payload, a denormal: all stored bit for bit
        vals.view(np.uint32)[:4] = [0x80000000, 0x00000000, 0x7fc01234, 0x00000007]
    outer = np.concatenate([[0], np.cumsum(mask.sum(axis=0))]).astype(np.int32)
    return vals, rows.astype(np.int32), outer


# ---- export --------------------------------------------------------------------------------------------------------------
EXPORT_SCENES = ["cornell_box_512", "cornell_box_2048", "cornellbox_blacklight", "colorballs",
                 "first_1", "first_2", "first_33", "first_257", "first_1000"]


@pytest.mark.parametrize("variant", [FFD, FFH])
@pytest.mark.parametrize("name", EXPORT_SCENES)
def test_export_matches_host_and_rule(dz, uv, name, variant, monkeypatch):
    p = ctx(dz, scene(name), uv)
    F = (p.cudaCalculateRadiosityMatrix() if variant == FFD else p.calculateRadiosityMatrix()).rows()
    want = csc_rule(F)
    monkeypatch.delenv("DAISY_CSC_STAGE_BYTES", raising=False)
    monkeypatch.setenv("DAISY_CSC_HOST", "1")
    host = _radmat(p).to_csc()
    n_host = count_only(dz, p)
    monkeypatch.delenv("DAISY_CSC_HOST")
    dev = _radmat(p).to_csc()
    assert_csc(host, want, (name, "host"))
    assert_csc(dev, want, (name, "device"))
    assert count_only(dz, p) == n_host == want[0].size
    if name in ("cornell_box_2048", "cornellbox_blacklight", "first_257"):  # many column chunks through the two staging buffers
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", SMALL_STAGE)
        assert_csc(_radmat(p).to_csc(), want, (name, "small staging"))
    p.close()


def special_matrix(N=70):
    rng = np.random.RandomState(5)
    F = np.where(rng.uniform(0, 1, (N, N)) < 0.3, rng.uniform(0, 1, (N, N)), 0.0).astype(np.float32)
    b = F.view(np.uint32)
    b[3, 1] = 0x7fc0beef    # quiet NaN with a payload
    b[4, 1] = 0xffa00001    # negative signalling NaN pattern
    b[5, 2] = 0x7f800000    # +inf
    b[6, 2] = 0xff800000    # -inf
    b[7, 3] = 0x00000001    # smallest denormal
    b[8, 3] = 0x807fffff    # largest negative denormal
    b[9, 4] = 0x80000000    # -0.0: not listed
    b[10, 4] = 0x00000000   # +0.0: not listed
    F[:, 10] = 0.0          # empty columns
    F[:, 11] = -0.0
    F[:, 12] = rng.uniform(0.5, 1, N).astype(np.float32)  # a full column
    F[:, N - 1] = 0.0       # empty last column
    return F


def test_export_special_values(dz, uv, monkeypatch):
    N = 70
    F = special_matrix(N)
    p = ctx(dz, sub_scene(N), uv)
    p.loadRadiosityMatrix(F)
    want = csc_rule(F)
    o = want[2]
    assert o[11] == o[10] and o[12] == o[11] and o[13] - o[12] == N and o[N] == o[N - 1]  # empty columns, a full column
    assert np.isnan(want[0]).sum() == 2 and np.isinf(want[0]).sum() == 2
    assert_csc(_radmat(p).to_csc(), want, "device")
    monkeypatch.setenv("DAISY_CSC_HOST", "1")
    assert_csc(_radmat(p).to_csc(), want, "host")
    p.close()


# ---- import --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stage", [None, SMALL_STAGE])
def test_import_round_trip_of_built_matrix(dz, uv, cornell2048, stage, monkeypatch):
    if stage:
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", stage)
    a = ctx(dz, cornell2048, uv)
    F = a.cudaCalculateRadiosityMatrix().rows()
    vals, inner, outer = _radmat(a).to_csc()
    b = ctx(dz, cornell2048, uv)
    b.loadRadiosityMatrix(np.full_like(F, 3.0))  # the import must clear what was there
    b.loadRadiosityMatrixCSC(vals, inner, outer)
    assert_holds(b, F, "built matrix")
    # small staging: uploaded twice in chunks (rows only for the validation); default: one upload kept resident
    assert dz.lib().daisy_formfactors_csc_uploads(b._ctx) == (2 if stage else 1)
    a.close(); b.close()


@pytest.mark.parametrize("stage", [None, SMALL_STAGE])
@pytest.mark.parametrize("N", [1, 2, 33, 257, 1000])
def test_import_random_sparse(dz, uv, N, stage, monkeypatch):
    if stage:
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", stage)
    vals, inner, outer = random_csc(N, 0.3, N)
    want = dense_of(vals, inner, outer, N)
    p = ctx(dz, sub_scene(N), uv)
    p.loadRadiosityMatrix(np.full((N, N), -2.5, np.float32))
    p.loadRadiosityMatrixCSC(vals, inner, outer)
    assert_holds(p, want, ("random", N))
    # an empty matrix loads as all +0.0
    p.loadRadiosityMatrixCSC(np.zeros(0, np.float32), np.zeros(0, np.int32), np.zeros(N + 1, np.int32))
    assert_holds(p, np.zeros((N, N), np.float32), ("empty", N))
    p.close()


def test_import_special_values_round_trip(dz, uv):
    N = 70
    F = special_matrix(N)
    p = ctx(dz, sub_scene(N), uv)
    p.loadRadiosityMatrix(F)
    csc = _radmat(p).to_csc()
    q = ctx(dz, sub_scene(N), uv)
    q.loadRadiosityMatrixCSC(*csc)
    want = F.copy()
    want.view(np.uint32)[(want.view(np.uint32) & 0x7fffffff) == 0] = 0  # -0.0 is not listed, so it comes back as +0.0
    assert_holds(q, want, "special values")
    p.close(); q.close()


def _solver(dz, p, K, E, M, mat):
    from daisyriot_b200 import _lib
    s = C.c_void_p()
    _lib.check(dz.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)), "solver_create")
    return s


def _read(dz, s, K, N):
    from daisyriot_b200 import _lib
    B = np.empty((K, N), np.float32); R = np.empty((K, N), np.float32)
    _lib.check(dz.lib().daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
    sums = np.zeros(K)
    _lib.check(dz.lib().daisy_solver_band_sums(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
    return B, R, sums


def _inputs(sc, K, seed):
    rng = np.random.RandomState(seed)
    N = sc.numtriangles
    E = np.zeros((K, N), np.float32)
    E[:, sc.mat_idx == 0] = 7.0
    E[:, :3] = 1.0
    M = rng.uniform(0, 0.25, (len(sc.materials), K, K)).astype(np.float32)
    return E, M, np.ascontiguousarray(sc.mat_idx, np.int32)


def test_import_solve_matches_dense_load(dz, uv, cornell2048):
    from daisyriot_b200 import _lib
    a = ctx(dz, cornell2048, uv)
    F = a.cudaCalculateRadiosityMatrix().rows()
    csc = _radmat(a).to_csc()
    N, K = cornell2048.numtriangles, 3
    E, M, mat = _inputs(cornell2048, K, 1)
    dense, sparse = ctx(dz, cornell2048, uv), ctx(dz, cornell2048, uv)
    dense.loadRadiosityMatrix(F)
    # a solver that exists before the import must rescan F
    other = np.ascontiguousarray(F[::-1].copy())
    sparse.loadRadiosityMatrix(other)
    s_pre = _solver(dz, sparse, K, E, M, mat)
    sparse.loadRadiosityMatrixCSC(*csc)
    s_dense, s_sparse = _solver(dz, dense, K, E, M, mat), _solver(dz, sparse, K, E, M, mat)
    passes = []
    for s in (s_dense, s_sparse, s_pre):
        _lib.check(dz.lib().daisy_solver_reset(s))
        n = C.c_int()
        _lib.check(dz.lib().daisy_solver_converge(s, 1e-4, 1, 200, C.byref(n)))
        passes.append(n.value)
    assert passes[0] == passes[1] == passes[2] > 1
    want = _read(dz, s_dense, K, N)
    for s, what in ((s_sparse, "fresh solver"), (s_pre, "solver created before the import")):
        got = _read(dz, s, K, N)
        assert bits_equal(got[0], want[0]) and bits_equal(got[1], want[1]), what
        assert np.array_equal(got[2], want[2]), what
    for s in (s_dense, s_sparse, s_pre):
        dz.lib().daisy_solver_destroy(s)
    a.close(); dense.close(); sparse.close()


def test_update_after_import_retraces_everything(dz, uv, cornell512):
    a = ctx(dz, cornell512, uv)
    F = a.cudaCalculateRadiosityMatrix().rows()
    csc = _radmat(a).to_csc()
    stats = []
    for load in ("rows", "csc"):
        p = ctx(dz, cornell512, uv)
        if load == "rows":
            p.loadRadiosityMatrix(F)
        else:
            p.loadRadiosityMatrixCSC(*csc)
        got = p.updateRadiosityMatrix().rows()
        assert bits_equal(got, F), load
        stats.append(p.update_stats())
        p.close()
    assert stats[0] == stats[1] and stats[1]["tris_changed"] == cornell512.numtriangles
    a.close()


def _invalid_cases(vals, inner, outer, N):
    c = int(np.argmax(np.diff(outer) >= 2))  # a column with at least two entries
    s = outer[c]
    cases = {}
    i = inner.copy(); i[s], i[s + 1] = i[s + 1], i[s]; cases["unsorted"] = (vals, i, outer)
    i = inner.copy(); i[s + 1] = i[s]; cases["duplicate"] = (vals, i, outer)
    i = inner.copy(); i[-1] = N; cases["row N"] = (vals, i, outer)
    i = inner.copy(); i[0] = -1; cases["row -1"] = (vals, i, outer)
    o = outer.copy(); o[c + 1] = o[c] - 1 if o[c] > 0 else o[c + 2] + 1; cases["decreasing outer"] = (vals, inner, o)
    o = outer.copy(); o[-1] -= 1; cases["outer[N] != nnz"] = (vals, inner, o)
    o = outer.copy(); o[0] = 1; cases["outer[0] != 0"] = (vals, inner, o)
    return cases


@pytest.mark.parametrize("stage", [None, SMALL_STAGE])
def test_import_invalid_input_changes_nothing(dz, uv, stage, monkeypatch):
    if stage:
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", stage)
    N = 257
    vals, inner, outer = random_csc(N, 0.3, 11, specials=False)
    before = np.random.RandomState(3).uniform(0, 1, (N, N)).astype(np.float32)
    p = ctx(dz, sub_scene(N), uv)
    p.loadRadiosityMatrix(before)
    for what, (v, i, o) in _invalid_cases(vals, inner, outer, N).items():
        assert write_csc_rc(dz, p, v, i, o) == E_INVALID, what
        assert_holds(p, before, what)
    p.close()


@pytest.mark.parametrize("N,G", [(300, 3), (1000, 2), (600, 4)])
def test_partitioned_contexts_keep_their_rows(dz, uv, N, G):
    vals, inner, outer = random_csc(N, 0.3, N + G)
    want = dense_of(vals, inner, outer, N)
    mesh_sc = sub_scene(N)
    ranges = []
    for g in range(G):
        p = ctx(dz, mesh_sc, uv, rank=g, nranks=G)
        r0, r1 = p.row_range
        ranges.append((r0, r1))
        p.loadRadiosityMatrixCSC(vals, inner, outer)
        assert_holds(p, want, ("rank", g, "of", G))
        p.close()
    assert any(r0 == r1 for r0, r1 in ranges) or G < 3, ranges  # (300, 3) and (600, 4) have a rank without rows


# ---- device group ----------------------------------------------------------------------------------------------------------
def _need_two(dz):
    if dz.lib().daisy_device_count() < 2:
        pytest.skip("needs 2 GPUs")


@pytest.mark.parametrize("stage", [None, SMALL_STAGE])
def test_group_export_matches_single_gpu(dz, uv, cornell2048, stage, monkeypatch):
    _need_two(dz)
    single = ctx(dz, cornell2048, uv)
    single.cudaCalculateRadiosityMatrix()
    want = _radmat(single).to_csc()
    if stage:
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", stage)
    g = dz.DeviceGroup(dz.MeshS.from_scene(cornell2048), devices=[0, 1], rands=uv)
    g.cudaCalculateRadiosityMatrix()
    assert_csc(g.to_csc(), want, "group")
    monkeypatch.setenv("DAISY_CSC_HOST", "1")
    assert_csc(g.to_csc(), want, "group, host conversion")
    g.close(); single.close()


@pytest.mark.parametrize("N", [200, 1000])
def test_group_import_matches_group_dense_load(dz, uv, N):
    """N = 200: device 1 owns no rows (blocks of 256)"""
    _need_two(dz)
    from daisyriot_b200.api import GroupSolver
    vals, inner, outer = random_csc(N, 0.3, 7 * N, specials=False)
    vals = (vals * np.float32(0.5 / (0.3 * N))).astype(np.float32)  # a contracting matrix for the solve
    want = dense_of(vals, inner, outer, N)
    sc = sub_scene(N)
    gs = []
    for load in ("rows", "csc"):
        g = dz.DeviceGroup(dz.MeshS.from_scene(sc), devices=[0, 1], rands=uv)
        if load == "rows":
            from daisyriot_b200 import _lib
            _lib.check(dz.lib().daisy_group_formfactors_write_rows(g._g, 0, N, _lib.fptr(want)))
        else:
            g.loadRadiosityMatrixCSC(vals, inner, outer)
        assert bits_equal(g.rows(), want), load
        for i in range(2):
            assert_holds(g.device(i), want, (load, "device", i))
        gs.append(g)
    K = 3
    E, M, mat = _inputs(sc, K, 2)
    res = []
    for g in gs:
        s = GroupSolver(g, K, E, M, mat)
        s.reset()
        n = s.converge(1e-4, True, 100)
        res.append((n, *s.read(), s.band_sums()))
        s.close()
    assert res[0][0] == res[1][0]
    assert bits_equal(res[0][1], res[1][1]) and bits_equal(res[0][2], res[1][2]) and np.array_equal(res[0][3], res[1][3])
    for g in gs:
        g.close()
