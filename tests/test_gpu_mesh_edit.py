"""Mesh edits (daisy_ctx_replace_mesh + daisy_formfactors_update): triangles removed, added, inserted, renumbered.

Unless stated otherwise every case compares the edited context's whole F bit for bit with a FRESH context built on the edited
scene, and checks that the update re-traced fewer pairs than the fresh build traced where the edit leaves most of the matrix as
it was."""
import ctypes as C

import numpy as np
import pytest

import geometry_scenes as gs
from oracle.pyoracle import Oracle

pytestmark = pytest.mark.gpu

FFD, FFH = 0, 1
E_INVALID, E_STATE = -1, -3


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


def _mesh(dz, sc):
    return dz.MeshS.from_scene(sc)


def _build(dz, sc, uv, variant, **kw):
    p = dz.OptixPrimeFunctionality(_mesh(dz, sc), device=0, rands=uv, **kw)
    (p.cudaCalculateRadiosityMatrix() if variant == FFD else p.calculateRadiosityMatrix())
    return p


def _fresh(dz, sc, uv, variant):
    p = _build(dz, sc, uv, variant)
    F, st = dz.RadMat(p).rows(), p.stats()
    p.close()
    return F, st


def _assert_bits(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = got.view(np.uint32) != want.view(np.uint32) if got.dtype == np.float32 else got != want
    assert not bad.any(), (what, int(bad.sum()), "entries differ; first", np.argwhere(bad)[:6].tolist())


def _quads(sc, quads):
    per = sc.numtriangles // 16
    return np.concatenate([np.arange(q * per, (q + 1) * per) for q in quads])


def _subscene(sc, tris, offset=(0.0, 0.0, 0.0)):
    """the listed triangles of sc as a scene of their own, translated by offset"""
    from daisyriot_b200 import scenes
    keep = np.zeros(sc.numtriangles, bool)
    keep[tris] = True
    sub, _ = scenes.edit_scene(sc, remove=np.nonzero(~keep)[0])
    sub.vertices = (sub.vertices.astype(np.float64) + np.asarray(offset, np.float64)).astype(np.float32)
    return sub


def _edit(sc, name):
    from daisyriot_b200 import scenes
    n = sc.numtriangles
    if name == "remove_short_block":
        return scenes.edit_scene(sc, remove=_quads(sc, scenes.CORNELL_SHORT_BLOCK))
    if name == "remove_lamp":
        return scenes.edit_scene(sc, remove=_quads(sc, scenes.CORNELL_LAMP))
    if name == "append_panel":
        return scenes.edit_scene(sc, add=scenes.cornell_panel(n))
    if name == "insert_panel":
        return scenes.edit_scene(sc, add=scenes.cornell_panel(n), insert_at=n // 2 + 7)
    if name == "move_tall_block":  # the tall block removed and a block added elsewhere, in one edit
        tall = _quads(sc, scenes.CORNELL_TALL_BLOCK)
        return scenes.edit_scene(sc, remove=tall, add=_subscene(sc, tall, offset=(-2.0, 0.0, 0.6)), insert_at=3 * n // 16)
    raise KeyError(name)


def _replace_update_check(dz, p, sc_new, prev, uv, variant, what):
    p.replaceMesh(_mesh(dz, sc_new), prev)
    F = p.updateRadiosityMatrix(variant).rows()
    want, fresh = _fresh(dz, sc_new, uv, variant)
    _assert_bits(F, want, what)
    return p.update_stats(), fresh


EDITS = ["remove_short_block", "remove_lamp", "append_panel", "insert_panel", "move_tall_block"]


@pytest.mark.parametrize("variant", [FFD, FFH])
@pytest.mark.parametrize("edit", EDITS)
@pytest.mark.parametrize("n", [512, 2048])
def test_cornell_edits_match_fresh_build(dz, uv50, n, edit, variant):
    from daisyriot_b200 import scenes
    sc = scenes.cornell_box(n)
    sc_new, prev = _edit(sc, edit)
    p = _build(dz, sc, uv50, variant)
    st, fresh = _replace_update_check(dz, p, sc_new, prev, uv50, variant, f"cornell{n} {edit}")
    assert p.N == sc_new.numtriangles
    assert st["tris_changed"] == int((prev < 0).sum()), st
    assert st["pairs_retraced"] < fresh["pairs_traced"], (edit, st, fresh)
    if n == 512:
        q = dz.OptixPrimeFunctionality(_mesh(dz, sc_new), rands=uv50)
        _assert_bits(p.visibilityMasks(variant=variant), q.visibilityMasks(variant=variant), "masks")
        q.close()
    p.close()


def test_noop_edits_trace_nothing(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    sc = cornell512
    p = _build(dz, sc, uv50, FFD)
    before = dz.RadMat(p).row_digest()
    # the same mesh, every triangle continued
    p.replaceMesh(_mesh(dz, sc), np.arange(sc.numtriangles))
    p.updateRadiosityMatrix(FFD)
    st = p.update_stats()
    assert st["tris_changed"] == 0 and st["pairs_retraced"] == 0 and st["tiles_retraced"] == 0, st
    # the same triangles over a permuted vertex array with duplicated entries, and a permuted normal array
    rng = np.random.RandomState(3)
    nv, nn = sc.vertices.shape[0], sc.normals.shape[0]
    vperm, nperm = rng.permutation(nv), rng.permutation(nn)
    dups = rng.choice(nv, 40, replace=False)  # these vertices appear twice; every other triangle uses the copy
    vinv = np.empty(nv, np.int64); vinv[vperm] = np.arange(nv)
    ninv = np.empty(nn, np.int64); ninv[nperm] = np.arange(nn)
    T = np.concatenate([vinv[sc.tri[:, :3]], ninv[sc.tri[:, 3:]]], 1)
    copy_of = np.full(nv, -1, np.int64); copy_of[dups] = nv + np.arange(dups.size)
    odd = np.zeros_like(T[:, :3], bool); odd[1::2] = True
    T[:, :3] = np.where(odd & (copy_of[sc.tri[:, :3]] >= 0), copy_of[sc.tri[:, :3]], T[:, :3])
    sc2 = scenes.Scene(np.concatenate([sc.vertices[vperm], sc.vertices[dups]]), sc.normals[nperm], T.astype(np.int32), sc.mat_idx,
                       sc.materials, "renumbered")
    p.replaceMesh(_mesh(dz, sc2), np.arange(sc.numtriangles))
    p.updateRadiosityMatrix(FFD)
    st = p.update_stats()
    assert st["tris_changed"] == 0 and st["pairs_retraced"] == 0 and st["tiles_retraced"] == 0, st
    after = dz.RadMat(p).row_digest()
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    p.close()


def test_order_not_kept_traces_every_facing_pair(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    sc = cornell512
    prev = np.arange(sc.numtriangles)
    prev[[40, 300]] = prev[[300, 40]]
    sc_new = scenes.Scene(sc.vertices, sc.normals, sc.tri[prev], sc.mat_idx[prev], sc.materials, "swapped")
    p = _build(dz, sc, uv50, FFD)
    st, fresh = _replace_update_check(dz, p, sc_new, prev, uv50, FFD, "swap")
    assert st["pairs_retraced"] == fresh["pairs_traced"], (st, fresh)
    p.close()


@pytest.mark.parametrize("which", ["shaft_cap", "occluded_walls"])
def test_removing_occluders_vs_bruteforce(dz, uv50, which):
    from daisyriot_b200 import scenes
    sc = gs.shaft_cap_scene(40) if which == "shaft_cap" else gs.occluded_walls(4, 4, n_occ=60)
    n_occ = 40 if which == "shaft_cap" else 60
    first = sc.numtriangles - n_occ
    sc_new, prev = scenes.edit_scene(sc, remove=np.arange(first, sc.numtriangles, 2))
    p = _build(dz, sc, uv50, FFD)
    st, fresh = _replace_update_check(dz, p, sc_new, prev, uv50, FFD, which)
    F_ref, masks_ref = Oracle.from_scene(sc_new).radmat_rows(uv50, 0, sc_new.numtriangles, brute=True)[:2]
    _assert_bits(dz.RadMat(p).rows(), F_ref, "brute force")
    _assert_bits(p.visibilityMasks(), masks_ref, "masks vs brute force")
    p.close()


def test_ties_survive_renumbering(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    sc = gs.with_ties(cornell512)
    sc_new, prev = scenes.edit_scene(sc, remove=np.arange(0, 12))  # low ids gone: every tied survivor shifts, in order
    for variant in (FFD, FFH):
        p = _build(dz, sc, uv50, variant)
        st, fresh = _replace_update_check(dz, p, sc_new, prev, uv50, variant, f"ties variant {variant}")
        assert st["pairs_retraced"] < fresh["pairs_traced"], (st, fresh)
        p.close()


def test_sequences_of_edits(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    sc = cornell512
    p = _build(dz, sc, uv50, FFD)
    # remove the short block; move the lamp; add a panel; one update
    s1, prev1 = _edit(sc, "remove_short_block")
    p.replaceMesh(_mesh(dz, s1), prev1)
    lamp = np.nonzero(s1.mat_idx == 0)[0]
    vi = np.unique(s1.tri[lamp, :3])
    V = np.array(s1.vertices, np.float32)
    V[vi] = (V[vi] + np.array([0.25, 0.0, 0.0], np.float32)).astype(np.float32)
    p.updateGeometry(V)
    s2 = scenes.Scene(V, s1.normals, s1.tri, s1.mat_idx, s1.materials, "moved")
    s3, prev3 = scenes.edit_scene(s2, add=scenes.cornell_panel(512))
    _replace_update_check(dz, p, s3, prev3, uv50, FFD, "replace, move, replace")
    # a triangle added in one replace and removed in the next leaves nothing behind
    s4, prev4 = scenes.edit_scene(s3, add=_subscene(s3, np.arange(0, 6), offset=(0.5, 2.0, 0.5)), insert_at=100)
    p.replaceMesh(_mesh(dz, s4), prev4)
    s5, prev5 = scenes.edit_scene(s4, remove=np.arange(100, 106))
    st, fresh = _replace_update_check(dz, p, s5, prev5, uv50, FFD, "add then remove")
    assert st["tris_changed"] == 0 and st["pairs_retraced"] == 0, st
    p.close()


def test_between_replace_and_update(dz, uv50, cornell512):
    from daisyriot_b200 import api
    sc = cornell512
    sc_new, prev = _edit(sc, "move_tall_block")
    p = _build(dz, sc, uv50, FFD)
    F_old = dz.RadMat(p).rows()
    p.replaceMesh(_mesh(dz, sc_new), prev)
    q = dz.OptixPrimeFunctionality(_mesh(dz, sc_new), rands=uv50)
    rays = np.ascontiguousarray(gs.closest_hit_rays(sc_new, 5), np.float32)
    got, want = p.optixQuery(rays.shape[0], rays), q.optixQuery(rays.shape[0], rays)
    assert (got.view(np.uint8) == want.view(np.uint8)).all()
    cam = api.Camera(64, 48, 2)
    colors = np.random.RandomState(0).uniform(0, 1, (sc_new.numtriangles, 3)).astype(np.float32)
    _assert_bits(api.traceScreen(p, cam, colors), api.traceScreen(q, cam, colors), "traceScreen")
    assert p.row_range == q.row_range
    ld_p, ld_q = C.c_int64(), C.c_int64()
    dz.lib().daisy_formfactors_ld(p._ctx, C.byref(ld_p)); dz.lib().daisy_formfactors_ld(q._ctx, C.byref(ld_q))
    assert ld_p.value == ld_q.value
    F = dz.RadMat(p).rows()
    old = prev >= 0
    _assert_bits(F[np.ix_(old, old)], F_old[np.ix_(prev[old], prev[old])], "surviving entries")
    assert not F[~old].view(np.uint32).any() and not F[:, ~old].view(np.uint32).any(), "rows / columns of new triangles"
    p.close(); q.close()


def _solver(dz, p, sc, K=3):
    from daisyriot_b200 import _lib
    rng = np.random.RandomState(1)
    nmat = len(sc.materials)
    M = rng.uniform(0, 0.25, (nmat, K, K)).astype(np.float32)
    E = np.zeros((K, sc.numtriangles), np.float32)
    E[:, sc.mat_idx == 0] = 5.0
    s = C.c_void_p()
    _lib.check(dz.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), nmat, _lib.iptr(np.ascontiguousarray(sc.mat_idx, np.int32)), C.byref(s)))
    return s


def _converge(dz, s, K, N):
    from daisyriot_b200 import _lib
    L = dz.lib()
    passes = C.c_int()
    _lib.check(L.daisy_solver_converge(s, 1e-3, 1, 200, C.byref(passes)))
    B, R = np.empty((K, N), np.float32), np.empty((K, N), np.float32)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
    return passes.value, B, R


def test_solvers(dz, uv50, cornell2048):
    from daisyriot_b200 import _lib
    sc = cornell2048
    sc_new, prev = _edit(sc, "append_panel")
    p = _build(dz, sc, uv50, FFD)
    old = _solver(dz, p, sc)
    L = dz.lib()
    p.replaceMesh(_mesh(dz, sc_new), prev)
    K, N = 3, sc_new.numtriangles
    B, R = np.empty((K, N), np.float32), np.empty((K, N), np.float32)
    passes, sums = C.c_int(), np.zeros(K)
    assert L.daisy_solver_step(old, sums.ctypes.data_as(C.POINTER(C.c_double))) == E_STATE
    assert b"create a new solver" in L.daisy_last_error()
    assert L.daisy_solver_read(old, _lib.fptr(B), _lib.fptr(R)) == E_STATE
    assert L.daisy_solver_converge(old, 1e-3, 1, 10, C.byref(passes)) == E_STATE
    assert L.daisy_solver_converge_device(old, 1e-3, 1, 10, C.byref(passes)) == E_STATE
    assert L.daisy_solver_reset(old) == E_STATE
    L.daisy_solver_destroy(old)
    p.updateRadiosityMatrix(FFD)
    q = _build(dz, sc_new, uv50, FFD)
    s1, s2 = _solver(dz, p, sc_new), _solver(dz, q, sc_new)
    p1, B1, R1 = _converge(dz, s1, K, N)
    p2, B2, R2 = _converge(dz, s2, K, N)
    assert p1 == p2 and p1 > 1
    _assert_bits(B1, B2, "B")
    _assert_bits(R1, R2, "residual")
    L.daisy_solver_destroy(s1); L.daisy_solver_destroy(s2)
    p.close(); q.close()


def test_invalid_input_leaves_the_context_unchanged(dz, uv50, cornell512):
    from daisyriot_b200 import _lib
    sc = cornell512
    sc_new, prev = _edit(sc, "remove_lamp")
    p = _build(dz, sc, uv50, FFD)
    digest = dz.RadMat(p).row_digest()
    L = dz.lib()
    with pytest.raises(ValueError):
        p.replaceMesh(_mesh(dz, sc_new), prev[:-1])  # too short
    v, n = np.ascontiguousarray(sc_new.vertices), np.ascontiguousarray(sc_new.normals)

    def call(tri, pv):
        return L.daisy_ctx_replace_mesh(p._ctx, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(tri), tri.shape[0], _lib.iptr(pv))

    tri = np.ascontiguousarray(sc_new.tri, np.int32)
    bad = np.array(prev, np.int32); bad[3] = sc.numtriangles
    assert call(tri, bad) == E_INVALID
    bad = np.array(prev, np.int32); bad[3] = -2
    assert call(tri, bad) == E_INVALID
    bad = np.array(prev, np.int32); bad[5] = bad[4]
    assert call(tri, bad) == E_INVALID and b"twice" in L.daisy_last_error()
    badtri = tri.copy(); badtri[7, 1] = v.shape[0]
    assert call(badtri, np.ascontiguousarray(prev, np.int32)) == E_INVALID
    assert p.N == sc.numtriangles and p.row_range == (0, sc.numtriangles)
    after = dz.RadMat(p).row_digest()
    assert np.array_equal(digest[0], after[0]) and np.array_equal(digest[1], after[1])
    # the context still works: the valid edit goes through
    _replace_update_check(dz, p, sc_new, prev, uv50, FFD, "after invalid calls")
    p.close()
    # a two-rank partition
    q = dz.OptixPrimeFunctionality(_mesh(dz, sc), rands=uv50, rank=0, nranks=2)
    assert L.daisy_ctx_replace_mesh(q._ctx, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(tri), tri.shape[0],
                                    _lib.iptr(np.ascontiguousarray(prev, np.int32))) == E_STATE
    q.close()


@pytest.mark.parametrize("mode", ["DAISY_FF_FACES", "DAISY_FF_RING", "outside_pattern"])
def test_culling_switches(dz, uv50, cornell512, monkeypatch, mode):
    from daisyriot_b200 import scenes
    uv = uv50
    if mode == "outside_pattern":
        uv = np.array(scenes.msvc_sample_pattern(3, 16), np.float32)
        uv[0] = (0.9, 0.4)  # u + v > 1
    else:
        monkeypatch.setenv(mode, "0")
    sc_new, prev = _edit(cornell512, "move_tall_block")
    p = _build(dz, cornell512, uv, FFD)
    st, fresh = _replace_update_check(dz, p, sc_new, prev, uv, FFD, mode)
    if mode == "outside_pattern":
        assert st["pairs_retraced"] == fresh["pairs_traced"], (st, fresh)
    else:
        assert st["pairs_retraced"] < fresh["pairs_traced"], (st, fresh)
    p.close()


@pytest.mark.parametrize("ndev", [2, 8])
def test_group_edit(dz, uv50, cornell2048, ndev):
    from daisyriot_b200 import scenes
    if dz.lib().daisy_device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    sc = cornell2048
    # triangles of device 0's block removed: every later row moves down, across the block boundaries
    sc_new, prev = scenes.edit_scene(sc, remove=np.arange(0, 300), add=scenes.cornell_panel(sc.numtriangles))
    g = dz.DeviceGroup(_mesh(dz, sc), ndev=ndev, rands=uv50)
    g.cudaCalculateRadiosityMatrix()
    g.replace_mesh(_mesh(dz, sc_new), prev)
    assert g.N == sc_new.numtriangles
    got = g.updateRadiosityMatrix(FFD).rows()
    want, _ = _fresh(dz, sc_new, uv50, FFD)
    _assert_bits(got, want, f"group of {ndev}")
    h = dz.DeviceGroup(_mesh(dz, sc_new), ndev=ndev, rands=uv50)
    h.cudaCalculateRadiosityMatrix()
    K = 3
    rng = np.random.RandomState(1)
    M = rng.uniform(0, 0.25, (len(sc_new.materials), K, K)).astype(np.float32)
    E = np.zeros((K, sc_new.numtriangles), np.float32)
    E[:, sc_new.mat_idx == 0] = 5.0
    res = []
    for grp in (g, h):
        s = dz.GroupSolver(grp, K, E, M, sc_new.mat_idx)
        s.reset()
        passes = s.converge(1e-3, True, 200)
        res.append((passes, *s.read()))
        s.close()
    assert res[0][0] == res[1][0]
    _assert_bits(res[0][1], res[1][1], "group B")
    g.close(); h.close()
