"""Matrix updates after a geometry change (daisy_ctx_update_geometry + daisy_formfactors_update).

Every case compares the updated context with a FRESH context built on the moved scene: F bit for bit (whole matrix), both
variants where it matters, and on small scenes the visibility masks and the brute-force oracle too.  The update statistics
show that only part of the matrix was re-traced where the contract says so (no-op, return to the recorded geometry,
normals-only change) and that everything was re-traced where nothing can be reused (loaded matrix, other variant, other
samples, samples outside the triangle)."""
import ctypes as C

import numpy as np
import pytest

import geometry_scenes as gs
from oracle.pyoracle import Oracle

pytestmark = pytest.mark.gpu

FFD, FFH = 0, 1


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


def _scene_with(sc, V, VN):
    from daisyriot_b200.scenes import Scene
    return Scene(np.ascontiguousarray(V, np.float32), np.ascontiguousarray(VN, np.float32), sc.tri, sc.mat_idx, sc.materials, sc.name + "*")


def _fresh_F(dz, sc, uv, variant, **kw):
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv, **kw)
    F = (p.cudaCalculateRadiosityMatrix() if variant == FFD else p.calculateRadiosityMatrix()).rows()
    stats = p.stats()
    p.close()
    return F, stats


def _build(dz, sc, uv, variant):
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv)
    (p.cudaCalculateRadiosityMatrix() if variant == FFD else p.calculateRadiosityMatrix())
    return p


def _assert_bits(got, want, what):
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), (what, int(bad.sum()), "entries differ; first", np.argwhere(bad)[:6].tolist())


def _update_and_check(dz, p, sc_new, uv, variant, what):
    """update p's matrix to sc_new's geometry (already set) and compare with a fresh build; returns the update stats"""
    F = p.updateRadiosityMatrix(variant).rows()
    want, _ = _fresh_F(dz, sc_new, uv, variant)
    _assert_bits(F, want, what)
    return p.update_stats()


def _touching_pairs(n_changed, N):
    return n_changed * (N - n_changed) + n_changed * (n_changed - 1) // 2


# ---- the Cornell box: lamp, short block, rotated block --------------------------------------------------------------------
MOVES = {
    "lamp": lambda sc, s: s.cornell_moved(sc, s.CORNELL_LAMP, offset=(0.25, 0.0, 0.0)),
    "short_block": lambda sc, s: s.cornell_moved(sc, s.CORNELL_SHORT_BLOCK, offset=(0.0, 0.0, 0.3)),
    "rotated_block": lambda sc, s: s.cornell_moved(sc, s.CORNELL_TALL_BLOCK, angle_y=0.2),
}


@pytest.mark.parametrize("variant", [FFD, FFH])
@pytest.mark.parametrize("move", list(MOVES))
@pytest.mark.parametrize("n", [512, 2048])
def test_cornell_moves_match_fresh_build(dz, uv50, n, move, variant):
    from daisyriot_b200 import scenes
    sc = scenes.cornell_box(n)
    V, VN = MOVES[move](sc, scenes)
    sc_new = _scene_with(sc, V, VN)
    p = _build(dz, sc, uv50, variant)
    full_pairs = p.stats()["pairs_traced"]
    p.updateGeometry(V, VN)
    st = _update_and_check(dz, p, sc_new, uv50, variant, f"cornell{n} {move}")
    quads = {"lamp": 1, "short_block": 5, "rotated_block": 5}[move]
    assert st["tris_changed"] == quads * n // 16, st
    assert 0 < st["pairs_retraced"] <= full_pairs, (st, full_pairs)
    if move == "lamp":
        assert st["pairs_retraced"] < full_pairs, ("a lamp move re-traced every pair", st, full_pairs)
    if n == 512:
        _assert_bits(p.visibilityMasks(variant=variant), dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc_new), rands=uv50).visibilityMasks(variant=variant),
                     "masks")
    p.close()


def test_cornell512_lamp_move_vs_bruteforce(dz, uv50):
    from daisyriot_b200 import scenes
    sc = scenes.cornell_box(512)
    V, VN = scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    sc_new = _scene_with(sc, V, VN)
    p = _build(dz, sc, uv50, FFD)
    p.updateGeometry(V, VN)
    F = p.updateRadiosityMatrix(FFD).rows()
    F_ref, masks_ref = Oracle.from_scene(sc_new).radmat_rows(uv50, 0, sc.numtriangles, brute=True)[:2]
    _assert_bits(F, F_ref, "brute force")
    _assert_bits(p.visibilityMasks(), masks_ref, "masks vs brute force")
    p.close()


def test_normals_only_change(dz, uv50, cornell512):
    sc = cornell512
    VN = np.array(sc.normals, np.float32)
    per = sc.numtriangles // 16
    ni = np.unique(sc.tri[3 * per:4 * per, 3:])  # the left wall's normal, tilted
    VN[ni] = (VN[ni] + np.float32(0.05) * np.array([0, 1, 0], np.float32)).astype(np.float32)
    p = _build(dz, sc, uv50, FFD)
    p.updateGeometry(normals=VN)
    st = _update_and_check(dz, p, _scene_with(sc, sc.vertices, VN), uv50, FFD, "normals only")
    assert st["tris_changed"] == per
    assert st["pairs_retraced"] <= _touching_pairs(per, sc.numtriangles), st
    p.close()


def test_noop_update(dz, uv50, cornell512):
    p = _build(dz, cornell512, uv50, FFD)
    before = p.cudaCalculateRadiosityMatrix().row_digest()
    p.updateGeometry(cornell512.vertices, cornell512.normals)
    p.updateRadiosityMatrix(FFD)
    st = p.update_stats()
    assert st["tris_changed"] == 0 and st["tiles_retraced"] == 0 and st["pairs_retraced"] == 0, st
    after = dz.RadMat(p).row_digest()
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    p.close()


def test_several_geometry_updates_then_back_to_the_record(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    sc = cornell512
    A = (sc.vertices, sc.normals)
    B = scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.3, 0.0, 0.0))
    Cg = scenes.cornell_moved(sc, scenes.CORNELL_SHORT_BLOCK, offset=(0.0, 0.0, -0.2))
    p = _build(dz, sc, uv50, FFD)
    # A -> B -> A: F still is A's matrix, nothing to trace
    p.updateGeometry(*B)
    p.updateGeometry(*A)
    p.updateRadiosityMatrix(FFD)
    assert p.update_stats()["tiles_retraced"] == 0
    # A -> B -> C, one update: C's matrix
    p.updateGeometry(*B)
    p.updateGeometry(*Cg)
    _update_and_check(dz, p, _scene_with(sc, *Cg), uv50, FFD, "A->B->C")
    # C -> A -> C: back to the recorded geometry, nothing to trace
    p.updateGeometry(*A)
    p.updateGeometry(*Cg)
    p.updateRadiosityMatrix(FFD)
    st = p.update_stats()
    assert st["tris_changed"] == 0 and st["tiles_retraced"] == 0, st
    # C -> A with one update: A's matrix
    p.updateGeometry(*A)
    _update_and_check(dz, p, sc, uv50, FFD, "C->A")
    p.close()


# ---- adversarial moves on the irregular walls ------------------------------------------------------------------------------
def _walls_parts(sc):
    """vertex ids of the occluder wall (the third wall: triangles 270..309) and of the floor"""
    occ = np.unique(sc.tri[270:310, :3])
    floor = np.unique(sc.tri[:144, :3])
    return occ, floor


@pytest.mark.parametrize("seed", [1, 2])
def test_irregular_walls_occluder_in_and_out_of_sight(dz, uv50, seed):
    sc = gs.irregular_walls(seed)
    occ, _ = _walls_parts(sc)
    V0 = np.array(sc.vertices, np.float32)
    # slide the occluder along its longest extent: far out of the walls' line of sight, back, part way, home
    e = V0[occ].max(axis=0) - V0[occ].min(axis=0)
    side = np.eye(3)[int(np.argmax(e))].astype(np.float32)
    p = _build(dz, sc, uv50, FFD)
    for k, shift in enumerate([8.0, -8.0, 0.7, 0.0]):  # far out of sight, back, partly, home
        V = V0.copy()
        V[occ] = (V0[occ] + np.float32(shift) * side).astype(np.float32)
        p.updateGeometry(V)
        sc_new = _scene_with(sc, V, sc.normals)
        _update_and_check(dz, p, sc_new, uv50, FFD, f"occluder step {k}")
        if k == 2:
            F_ref = Oracle.from_scene(sc_new).radmat_rows(uv50, 0, sc.numtriangles, brute=True)[0]
            _assert_bits(dz.RadMat(p).rows(), F_ref, "brute force")
    p.close()


def test_irregular_walls_one_ulp_and_plane_changes(dz, uv50):
    sc = gs.irregular_walls(1)
    occ, floor = _walls_parts(sc)
    V0 = np.array(sc.vertices, np.float32)
    p = _build(dz, sc, uv50, FFH)
    # one ulp
    V = V0.copy()
    V[occ] = np.nextafter(V0[occ], np.float32(np.inf))
    p.updateGeometry(V)
    _update_and_check(dz, p, _scene_with(sc, V, sc.normals), uv50, FFH, "one ulp")
    # one floor vertex out of the floor's plane (its triangles lose their plane id), then back into it
    inner = floor[len(floor) // 2]
    n = np.cross(V0[sc.tri[0, 1]] - V0[sc.tri[0, 0]], V0[sc.tri[0, 2]] - V0[sc.tri[0, 0]])
    n = (n / np.linalg.norm(n)).astype(np.float32)
    for lift in (0.05, 1e-3, 0.0):
        V2 = V.copy()
        V2[inner] = (V0[inner] + np.float32(lift) * n).astype(np.float32)
        p.updateGeometry(V2)
        sc_new = _scene_with(sc, V2, sc.normals)
        _update_and_check(dz, p, sc_new, uv50, FFH, f"lift {lift}")
        q = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc_new), rands=uv50)
        assert dz.lib().daisy_ctx_face_count(p._ctx) == dz.lib().daisy_ctx_face_count(q._ctx)
        q.close()
    p.close()


def test_irregular_walls_random_move_sequence(dz, uv50):
    sc = gs.irregular_walls(2)
    rng = np.random.RandomState(7)
    V = np.array(sc.vertices, np.float32)
    p = _build(dz, sc, uv50, FFD)
    for step in range(5):
        ids = rng.choice(V.shape[0], size=rng.randint(1, 12), replace=False)
        V = V.copy()
        V[ids] = (V[ids] + rng.normal(scale=0.05, size=(len(ids), 3))).astype(np.float32)
        p.updateGeometry(V)
        st = _update_and_check(dz, p, _scene_with(sc, V, sc.normals), uv50, FFD, f"random step {step}")
        assert st["tris_changed"] > 0
    p.close()


def test_blacklight_fixture_one_material_moved(dz, uv50, fixture_scenes):
    sc = fixture_scenes["cornellbox_blacklight"]
    mat = int(np.bincount(sc.mat_idx).argmin())
    vi = np.unique(sc.tri[sc.mat_idx == mat, :3])
    V = np.array(sc.vertices, np.float32)
    V[vi] = (V[vi] + np.array([0.02, 0.0, -0.03], np.float32)).astype(np.float32)
    for variant in (FFD, FFH):
        p = _build(dz, sc, uv50, variant)
        p.updateGeometry(V)
        _update_and_check(dz, p, _scene_with(sc, V, sc.normals), uv50, variant, f"blacklight material {mat}")
        p.close()


# ---- modes ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env", ["DAISY_FF_FACES", "DAISY_FF_RING"])
def test_modes_off(dz, uv50, cornell512, monkeypatch, env):
    from daisyriot_b200 import scenes
    monkeypatch.setenv(env, "0")
    V, VN = scenes.cornell_moved(cornell512, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    p = _build(dz, cornell512, uv50, FFD)
    p.updateGeometry(V, VN)
    _update_and_check(dz, p, _scene_with(cornell512, V, VN), uv50, FFD, env + "=0")
    p.close()


def test_samples_outside_the_triangle_trace_everything(dz, cornell512):
    from daisyriot_b200 import scenes
    uv = np.array(scenes.msvc_sample_pattern(3, 16), np.float32)
    uv[0] = (0.9, 0.4)  # u + v > 1
    V, VN = scenes.cornell_moved(cornell512, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    p = _build(dz, cornell512, uv, FFD)
    p.updateGeometry(V, VN)
    sc_new = _scene_with(cornell512, V, VN)
    st = _update_and_check(dz, p, sc_new, uv, FFD, "outside pattern")
    _, fresh = _fresh_F(dz, sc_new, uv, FFD)
    assert st["pairs_retraced"] == fresh["pairs_traced"], (st, fresh)


@pytest.mark.parametrize("why", ["write_rows", "variant", "set_samples"])
def test_fallback_to_full_tracing(dz, uv50, cornell512, why):
    from daisyriot_b200 import scenes
    V, VN = scenes.cornell_moved(cornell512, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    sc_new = _scene_with(cornell512, V, VN)
    p = _build(dz, cornell512, uv50, FFD)
    uv = uv50
    variant = FFD
    if why == "write_rows":
        p.loadRadiosityMatrix(dz.RadMat(p).rows())
    elif why == "variant":
        variant = FFH
    else:
        uv = np.ascontiguousarray(scenes.msvc_sample_pattern(2), np.float32)
        dz._lib.check(dz.lib().daisy_ctx_set_samples(p._ctx, dz._lib.fptr(uv), uv.shape[0]))
    p.updateGeometry(V, VN)
    st = _update_and_check(dz, p, sc_new, uv, variant, "fallback " + why)
    _, fresh = _fresh_F(dz, sc_new, uv, variant)
    assert st["pairs_retraced"] == fresh["pairs_traced"] and st["tris_changed"] == cornell512.numtriangles, (st, fresh)
    p.close()


def test_row_partition_without_peers(dz, uv50, cornell2048):
    from daisyriot_b200 import scenes
    sc = cornell2048
    V, VN = scenes.cornell_moved(sc, scenes.CORNELL_SHORT_BLOCK, offset=(0.0, 0.0, 0.3))
    want, _ = _fresh_F(dz, _scene_with(sc, V, VN), uv50, FFD)
    for rank in range(3):
        p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv50, rank=rank, nranks=3)
        p.cudaCalculateRadiosityMatrix()
        p.updateGeometry(V, VN)
        r0, r1 = p.row_range
        got = p.updateRadiosityMatrix(FFD).rows()
        _assert_bits(got, want[r0:r1], f"rank {rank}")
        p.close()


# ---- downstream ------------------------------------------------------------------------------------------------------------
def test_queries_follow_the_geometry_and_F_waits(dz, uv50, cornell512):
    from daisyriot_b200 import api, scenes
    sc = cornell512
    V, VN = scenes.cornell_moved(sc, scenes.CORNELL_SHORT_BLOCK, offset=(0.0, 0.0, 0.3))
    sc_new = _scene_with(sc, V, VN)
    p = _build(dz, sc, uv50, FFD)
    F_old = dz.RadMat(p).rows()
    p.updateGeometry(V, VN)
    q = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc_new), rands=uv50)
    rays = np.ascontiguousarray(gs.closest_hit_rays(sc_new, 5), np.float32)
    got, want = p.optixQuery(rays.shape[0], rays), q.optixQuery(rays.shape[0], rays)
    assert (got.view(np.uint8) == want.view(np.uint8)).all()
    cam = api.Camera(64, 48, 2)
    colors = np.random.RandomState(0).uniform(0, 1, (sc.numtriangles, 3)).astype(np.float32)
    _assert_bits(api.traceScreen(p, cam, colors), api.traceScreen(q, cam, colors), "traceScreen")
    assert dz.lib().daisy_ctx_face_count(p._ctx) == dz.lib().daisy_ctx_face_count(q._ctx)
    _assert_bits(dz.RadMat(p).rows(), F_old, "F before the matrix update")
    p.close(); q.close()


def _solver(dz, p, sc, K=3):
    from daisyriot_b200 import _lib
    rng = np.random.RandomState(1)
    nmat = int(sc.mat_idx.max()) + 1
    M = rng.uniform(0, 0.25, (nmat, K, K)).astype(np.float32)
    E = np.zeros((K, sc.numtriangles), np.float32)
    E[:, sc.mat_idx == 0] = 5.0
    s = C.c_void_p()
    _lib.check(dz.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), nmat, _lib.iptr(np.ascontiguousarray(sc.mat_idx, np.int32)), C.byref(s)))
    return s


def _converge(dz, s, K=3):
    from daisyriot_b200 import _lib
    L = dz.lib()
    _lib.check(L.daisy_solver_reset(s))
    passes = C.c_int()
    _lib.check(L.daisy_solver_converge(s, 1e-3, 1, 200, C.byref(passes)))
    dims = np.zeros(2, np.int32)
    _lib.check(L.daisy_solver_tile_map(s, _lib.iptr(dims), None, 0, None, None))
    occ = np.zeros(max(1, int(dims[0] * dims[1])), np.uint8)
    _lib.check(L.daisy_solver_tile_map(s, _lib.iptr(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, None, None))
    return passes.value, occ


def test_solver_on_the_updated_matrix(dz, uv50, cornell2048):
    from daisyriot_b200 import _lib, scenes
    sc = cornell2048
    # the lamp starts above the ceiling, facing the ceiling's back: its rows and columns are empty; the update brings it home
    Va, VNa = scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.0, 3.0, 0.0))
    sc_a = _scene_with(sc, Va, VNa)
    p = _build(dz, sc_a, uv50, FFD)
    s = _solver(dz, p, sc)
    _, occ_a = _converge(dz, s)
    p.updateGeometry(sc.vertices, sc.normals)
    p.updateRadiosityMatrix(FFD)
    passes, occ = _converge(dz, s)
    q = _build(dz, sc, uv50, FFD)
    s2 = _solver(dz, q, sc)
    passes2, occ2 = _converge(dz, s2)
    assert passes == passes2
    assert np.array_equal(occ, occ2)
    assert (occ.astype(bool) & ~occ_a.astype(bool)).any(), "no tile went from empty to occupied"
    K, N = 3, sc.numtriangles
    B1, R1, B2, R2 = (np.empty((K, N), np.float32) for _ in range(4))
    _lib.check(dz.lib().daisy_solver_read(s, _lib.fptr(B1), _lib.fptr(R1)))
    _lib.check(dz.lib().daisy_solver_read(s2, _lib.fptr(B2), _lib.fptr(R2)))
    _assert_bits(B1, B2, "B")
    dz.lib().daisy_solver_destroy(s); dz.lib().daisy_solver_destroy(s2)
    p.close(); q.close()


# ---- several GPUs ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ndev", [2, 8])
def test_group_update(dz, uv50, cornell2048, ndev):
    from daisyriot_b200 import scenes
    if dz.lib().daisy_device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    sc = cornell2048
    V, VN = scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    g = dz.DeviceGroup(dz.MeshS.from_scene(sc), ndev=ndev, rands=uv50)
    g.cudaCalculateRadiosityMatrix()
    g.update_geometry(V, VN)
    got = g.updateRadiosityMatrix(FFD).rows()
    want, _ = _fresh_F(dz, _scene_with(sc, V, VN), uv50, FFD)
    _assert_bits(got, want, f"group of {ndev}")
    g.close()
