"""GPU parity tests proper: the CUDA path, called through the C-ABI, against the CPU oracle on the same inputs.
Integer / mask / index results and the form factors are compared BIT-EXACT; the gather within 1e-5 relative
(the tolerance BASELINE.json's north_star states) against the FP64-accumulating oracle."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_rel, two_triangle_scene
from geometry_scenes import irregular_walls, perforated_plate

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


def _ctx(dz, sc, uv):
    return dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv)


def _oracle(sc):
    from oracle.pyoracle import Oracle
    return Oracle.from_scene(sc)


def _random_rays(sc, n, seed):
    rng = np.random.RandomState(seed)
    lo, hi = sc.vertices.min(0), sc.vertices.max(0)
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    return np.concatenate([o, d], 1).astype(np.float32)


@pytest.mark.parametrize("scene_name", ["cornell512", "cornell2048"])
def test_closest_hit_bitexact(dz, request, uv50, scene_name):
    sc = request.getfixturevalue(scene_name)
    p, orc = _ctx(dz, sc, uv50), _oracle(sc)
    rays = _random_rays(sc, 20000, 1)
    pair = np.concatenate([orc.pair_rays(i, j, uv50) for i, j in [(0, sc.numtriangles - 1), (3, 100), (17, 300), (40, 41)]])
    # axis-aligned and degenerate directions exercise the 0*inf paths of the slab test
    axis = np.array([[2.7, 2.7, 2.7, 1, 0, 0], [2.7, 2.7, 2.7, 0, -1, 0], [2.7, 2.7, 2.7, 0, 0, 1], [1, 1, 1, 0, 0, 0]], np.float32)
    rays = np.concatenate([rays, pair, axis])
    got = p.optixQuery(rays.shape[0], rays)
    want = orc.query_closest(rays, brute=True)
    assert np.array_equal(got["triangleId"], want["triangleId"])
    assert np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32))
    assert np.array_equal(got["u"].view(np.uint32), want["u"].view(np.uint32))
    assert np.array_equal(got["v"].view(np.uint32), want["v"].view(np.uint32))
    assert (got["triangleId"] >= 0).mean() > 0.5
    p.close()


def test_closest_hit_known_answers(dz, uv50):
    sc = two_triangle_scene()
    p = _ctx(dz, sc, uv50)
    rays = np.array([[0.25, 0.25, -1, 0, 0, 1],    # hits tri 0 at t=1, then tri 1 behind it
                     [0.25, 0.25, 0.5, 0, 0, 1],   # between them: hits tri 1 at t=0.5
                     [0.25, 0.25, 2.0, 0, 0, 1],   # beyond both: miss
                     [0.9, 0.9, -1, 0, 0, 1]], np.float32)  # outside both triangles: miss
    h = p.optixQuery(4, rays)
    assert list(h["triangleId"]) == [0, 1, -1, -1]
    assert h["t"][0] == np.float32(1.0) and h["t"][1] == np.float32(0.5) and h["t"][2] < 0 and h["t"][3] < 0
    assert h["u"][0] == np.float32(0.25) and h["v"][0] == np.float32(0.25)  # weights of vertices 1 and 2
    p.close()


def test_empty_and_single_triangle(dz, uv50):
    from daisyriot_b200.scenes import Scene
    sc1 = two_triangle_scene()
    one = Scene(sc1.vertices, sc1.normals, sc1.tri[:1], sc1.mat_idx[:1], sc1.materials, "one")
    p = _ctx(dz, one, uv50)
    h = p.optixQuery(2, np.array([[0.25, 0.25, -1, 0, 0, 1], [5, 5, -1, 0, 0, 1]], np.float32))
    assert list(h["triangleId"]) == [0, -1]
    F = p.cudaCalculateRadiosityMatrix().rows()
    assert F.shape == (1, 1) and F[0, 0] == 0
    assert p.optixQuery(0, np.zeros((0, 6), np.float32)).shape == (0,)
    p.close()


@pytest.mark.parametrize("variant", [0, 1])
def test_unoccluded_rows_bitexact(dz, cornell512, uv50, variant):
    p, orc = _ctx(dz, cornell512, uv50), _oracle(cornell512)
    got = p.runCalculateRadiosityMatrix(0, 512, variant)
    want = orc.unoccluded_rows(0, 512, variant)
    assert np.array_equal(got["m_row"], np.repeat(np.arange(512), 512).reshape(512, 512))
    assert np.array_equal(got["m_col"], np.tile(np.arange(512), (512, 1)))
    assert np.array_equal(got["m_value"].astype(np.float32).view(np.uint32), want.view(np.uint32))
    assert np.array_equal(got["m_value"], want.astype(np.float64))  # stored as the float widened to double
    p.close()


@pytest.mark.parametrize("variant", [0, 1])
def test_radmat_small_bitexact_vs_bruteforce(dz, cornell512, uv50, variant):
    p, orc = _ctx(dz, cornell512, uv50), _oracle(cornell512)
    rm = p.cudaCalculateRadiosityMatrix() if variant == 0 else p.calculateRadiosityMatrix()
    F = rm.rows()
    masks = p.visibilityMasks(variant=variant)
    F_ref, m_ref, rays = orc.radmat_rows(uv50, 0, 512, variant=variant, reciprocity=bool(variant), brute=True)
    if variant == 0:
        assert np.array_equal(masks, m_ref)
    else:  # the per-pair path traces every pair; the fused kernel skips pairs whose factor is zero anyway
        traced = masks != 0
        assert np.array_equal(masks[traced], m_ref[traced])
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    st = p.stats()
    assert st["rays"] == st["pairs_traced"] * 50 and st["pairs_traced"] > 0 and st["pairs_owned"] == st["pairs_traced"]
    # masks are symmetric, the matrix has an empty diagonal, a closed-ish box keeps row sums bounded
    assert np.array_equal(masks, masks.T) and not F.diagonal().any()
    # CSC hand-back equals the dense matrix
    vals, inner, outer = rm.to_csc()
    dense = np.zeros_like(F)
    for c in range(512):
        dense[inner[outer[c]:outer[c + 1]], c] = vals[outer[c]:outer[c + 1]]
    assert np.array_equal(dense, F) and np.all(np.diff(inner[outer[3]:outer[4]]) > 0)
    p.close()


def test_radmat_2048_rows_bitexact(dz, cornell2048, uv50):
    p, orc = _ctx(dz, cornell2048, uv50), _oracle(cornell2048)
    F = p.cudaCalculateRadiosityMatrix().rows()
    rows = [0, 1, 63, 64, 65, 700, 1023, 1024, 1999, 2047]
    masks_all = p.visibilityMasks(0, 2048)
    for r in rows:
        F_ref, m_ref, _ = orc.radmat_rows(uv50, r, r + 1)
        assert np.array_equal(masks_all[r], m_ref[0]), r
        assert np.array_equal(F[r].view(np.uint32), F_ref[0].view(np.uint32)), r
    # partial occlusion really occurs in this scene (not just all-or-nothing masks)
    full = np.uint64((1 << 50) - 1)
    assert ((masks_all != 0) & (masks_all != full)).sum() > 1000
    p.close()


@pytest.mark.parametrize("name", ["cornellbox_blacklight", "colorballs"])
def test_fixture_scene_rows_bitexact(dz, fixture_scenes, uv50, name):
    sc = fixture_scenes[name]
    p, orc = _ctx(dz, sc, uv50), _oracle(sc)
    F = p.cudaCalculateRadiosityMatrix().rows()
    N = sc.numtriangles
    rows = [0, 1, 2, 777, 2560, 5119, 5120, N - 33, N - 1]
    for r in rows:
        F_ref, m_ref, _ = orc.radmat_rows(uv50, r, r + 1)
        m = p.visibilityMasks(r, 1)
        assert np.array_equal(m[0], m_ref[0]), (name, r)
        assert np.array_equal(F[r].view(np.uint32), F_ref[0].view(np.uint32)), (name, r)
    st = p.stats()
    expect = {"cornellbox_blacklight": 9322918, "colorballs": 7587047}[name]  # SURVEY.md section 6
    assert abs(st["pairs_traced"] - expect) <= 0.002 * expect, st
    p.close()


def _solver(dz, p, K, E, M, mat):
    from daisyriot_b200 import _lib
    s = C.c_void_p()
    _lib.check(_lib.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)))
    return s


@pytest.mark.parametrize("K", [1, 3, 9, 12, 32])
def test_gather_pass_vs_oracle(dz, cornell2048, uv50, K):
    from daisyriot_b200 import _lib
    from oracle import pyoracle
    sc = cornell2048
    p = _ctx(dz, sc, uv50)
    N = sc.numtriangles
    rng = np.random.RandomState(K)
    F = (rng.uniform(0, 1, (N, N)) * (rng.uniform(0, 1, (N, N)) < 0.3) / N).astype(np.float32)
    np.fill_diagonal(F, 0)
    p.loadRadiosityMatrix(F)
    nmat = len(sc.materials)
    M = rng.uniform(0, 0.4, (nmat, K, K)).astype(np.float32)
    E = rng.uniform(0, 3, (K, N)).astype(np.float32) * (rng.uniform(0, 1, (K, N)) < 0.2)
    E = np.ascontiguousarray(E, np.float32)
    s = _solver(dz, p, K, E, M, sc.mat_idx)
    L = _lib.lib()
    res, B = E.copy(), E.copy()
    for it in range(3):
        sums = np.zeros(K)
        _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        sums_ref = pyoracle.gather_pass(F, res, B, M, sc.mat_idx, accum=1)
        Bg, Rg = np.empty_like(E), np.empty_like(E)
        _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
        # tolerance: TRUE relative error <= 1e-5 (north_star) for every entry above 1e-6 of its band's largest value
        for k in range(K):
            assert_rel(Rg[k], res[k], ("residual", K, it, k))
            assert_rel(Bg[k], B[k], ("B", K, it, k))
        assert np.allclose(sums, sums_ref, rtol=1e-6)
    assert L.daisy_solver_numpasses(s) == 3
    _lib.check(L.daisy_solver_reset(s))
    Bg, Rg = np.empty_like(E), np.empty_like(E)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
    assert np.array_equal(Bg, E) and np.array_equal(Rg, E) and L.daisy_solver_numpasses(s) == 0
    L.daisy_solver_destroy(s)
    p.close()


@pytest.mark.parametrize("K", [3, 9])
def test_chained_passes_change_nothing(dz, cornell2048, uv50, K):
    """daisy_solver_set_chained: passes issued back to back without reading the band sums overlap (programmatic dependent
    launch: the next pass streams its first F tiles while the previous one finishes).  Twelve chained passes must leave exactly
    the B, residual and band sums that twelve passes with a host synchronisation after each one leave."""
    from daisyriot_b200 import _lib
    sc = cornell2048
    p = _ctx(dz, sc, uv50)
    p.cudaCalculateRadiosityMatrix()
    rng = np.random.RandomState(40 + K)
    M = rng.uniform(0, 0.3, (len(sc.materials), K, K)).astype(np.float32)
    E = np.zeros((K, sc.numtriangles), np.float32)
    E[:, sc.mat_idx == 0] = 5.0
    L = _lib.lib()
    got = {}
    for chained in (0, 1):
        s = _solver(dz, p, K, E, M, sc.mat_idx)
        _lib.check(L.daisy_solver_set_chained(s, chained))
        sums = np.zeros(K)
        for it in range(12):
            if chained:
                _lib.check(L.daisy_solver_step(s, None))
            else:
                _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        _lib.check(L.daisy_solver_band_sums(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        B, R = np.empty_like(E), np.empty_like(E)
        _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
        got[chained] = (B, R, sums.copy())
        L.daisy_solver_destroy(s)
    assert np.array_equal(got[0][0], got[1][0]) and np.array_equal(got[0][1], got[1][1]) and np.array_equal(got[0][2], got[1][2])
    assert got[0][2].sum() > 0
    p.close()


def test_lightning_classes_match_oracle_loop(dz, cornell2048, uv50, coeff_model):
    """Spectral / RGB / BW flavours end to end on a built matrix: same pass count under the reference's stop rule and
    converged radiosity within 1e-5 of the FP64-accumulating oracle iteration."""
    from daisyriot_b200 import materials
    from oracle import pyoracle
    model, _ = coeff_model
    sc = cornell2048
    wl = np.arange(200, 601, 50).astype(np.float32)
    mesh = dz.MeshS.from_scene(sc, wl, model)
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv50)
    # RGB/BW emitters: the lamp has no RGB emission (UVLightMaterial zeroes it), so let the white paint glow a little;
    # the spectral flavour reads spectral_emission and is unaffected
    mesh.materials[3].emission[:] = (0.2, 0.1, 0.05)
    for method, thr, per_band in [(2, 200.0, 0), (1, 1e-4, 1), (0, 1e-4, 1)]:
        ev = 7.0 if method == 2 else 500.0
        lt = dz.Lightning.get_lightning(method, mesh, p, ev, wl, True, None, converge=False)
        F = lt.RadMat.rows()  # BW rebuilds with the per-pair variant, as the reference does
        inputs = {2: materials.spectral_inputs, 1: materials.rgb_inputs, 0: materials.bw_inputs}[method]
        E, M = inputs(mesh.materials, mesh.materialIndexPerTriangle, ev)
        res, B = E.copy(), E.copy()
        sums = res.astype(np.float64).sum(1)
        passes = 0
        crit = (lambda s: s.sum() > thr) if not per_band else (lambda s: (s > thr).any())
        while crit(sums) and passes < 400:
            sums = pyoracle.gather_pass(F, res, B, M, mesh.materialIndexPerTriangle, accum=1)
            passes += 1
        got = lt.converge_lightning(400)
        assert got == passes and passes > 0, (method, got, passes)
        Bg, Rg = lt.read()
        for k in range(B.shape[0]):
            assert_rel(Bg[k], B[k], ("converged B", method, k))
        c = lt.get_color_of_patch(5)
        assert c.shape == (3,) and np.isfinite(c).all()
        lt.close()
    p.close()


@pytest.mark.parametrize("name", ["cornellbox_blacklight", "colorballs"])
def test_fixture_scene_whole_matrix_digests(dz, fixture_scenes, name):
    """Every entry of the reference scenes' matrices and every visibility mask, against the whole-matrix digests the CPU
    oracle froze in tests/golden/<scene>_full_golden.npz (mask hash and F bit-xor per row are exact, row sums to 1e-12)."""
    import os
    from conftest import GOLDEN
    from oracle.pyoracle import row_checksums
    g = np.load(os.path.join(GOLDEN, name + "_full_golden.npz"))
    sc = fixture_scenes[name]
    N = sc.numtriangles
    p = _ctx(dz, sc, g["uv"])
    rm = p.cudaCalculateRadiosityMatrix()
    assert p.stats()["pairs_traced"] == int(g["pairs"]) == {"cornellbox_blacklight": 9322918, "colorballs": 7587047}[name]
    CH = 512
    for r0 in range(0, N, CH):
        nr = min(CH, N - r0)
        F = rm.rows(r0, nr)
        m = p.visibilityMasks(r0, nr)
        mh, fs, fx = row_checksums(F, m)
        assert np.array_equal(mh, g["mask_hash"][r0:r0 + nr]), (name, r0)
        assert np.array_equal(fx, g["F_xor"][r0:r0 + nr]), (name, r0)
        assert np.allclose(fs, g["F_sum"][r0:r0 + nr], rtol=1e-12, atol=1e-15), (name, r0)
    p.close()


def test_unoccluded_vs_reference_cuda_kernel(dz, cornell2048, fixture_scenes, uv50):
    """The reference's own calculateRow kernel (parallellism.cu, compiled unmodified for sm_100a into oracle/_ref).
    Its only arithmetic we do not restate is `powf(length, 2)`: nvcc 12.9 expands that into libdevice's polynomial powf
    (a few ulp off the exact square, and toolkit-version dependent), where we compute length*length.  Built with
    -fmad=false everything else is the same operation sequence, so the two agree to a few ulp (< 1e-6 relative);
    built with nvcc's default FMA contraction they agree to 1e-5 wherever the value is not rounding noise."""
    from oracle import pyref
    if not pyref.cuda_kernel_available(True):
        pytest.skip("oracle/_ref/libdaisy_ref_cuda*.so not built (needs /root/reference at build time)")
    for sc in (cornell2048, fixture_scenes["colorballs"]):
        N = sc.numtriangles
        p = _ctx(dz, sc, uv50)
        ours = p.runCalculateRadiosityMatrix(0, N, 0)["m_value"]
        for nofma in (True, False):
            ref, secs = pyref.cuda_run_calculate_radiosity_matrix(sc.vertices, sc.normals, sc.tri, nofma=nofma)
            assert not ((ours > 0) != (ref > 0)).any()  # the set of mutually facing pairs is identical
            if nofma:
                # same operation sequence except powf: a few ulp at most, and most entries identical to the last bit
                nz = ours > 0
                assert (np.abs(ours - ref)[nz] / ours[nz]).max() < 1e-6, (sc.name, "nofma")
                assert (ours[nz] == ref[nz]).mean() > 0.9
            else:
                # nvcc's FMA contraction reorders roundings inside the dot products; entries that are themselves
                # cancellation residue (1e-9 and below, against typical 1e-5..1e-2) carry that noise in full, hence
                # the absolute floor of 1e-10 next to the 1e-5 relative bar
                assert np.allclose(ours, ref, rtol=1e-5, atol=1e-10), (sc.name, np.abs(ours - ref).max())
        p.close()


def test_trace_screen_matches_literal_restatement(dz, cornell2048, uv50):
    """traceScreen (camera rays -> closest hit on the GPU -> isFacingBack -> Drawer::interpolate -> clamp) against a literal
    per-pixel loop over the oracle's closest hits (reference OptixPrimeFunctionality.cpp:83-131, Drawer.cpp:161-186)."""
    from daisyriot_b200 import api
    sc = cornell2048
    mesh = dz.MeshS.from_scene(sc)
    p = dz.OptixPrimeFunctionality(mesh, rands=uv50)
    cam = api.Camera(48, 36, 4)
    cam.eye = np.array([2.75, 2.75, 14.0], np.float32)   # look into the box from its open side
    cam.dir = np.array([2.75, 2.75, 0.0], np.float32)
    rng = np.random.RandomState(2)
    colors = rng.uniform(0, 1.2, (sc.numtriangles, 3)).astype(np.float32)
    img = api.traceScreen(p, cam, colors, True, True)
    rays = cam.gen_rays_for_screen(True)
    hits = _oracle(sc).query_closest(rays)
    tpv = [[] for _ in range(len(sc.vertices))]
    for t in range(sc.numtriangles):
        for k in range(3):
            tpv[sc.tri[t, k]].append(t)
    want = np.zeros((36, 48, 3), np.float32)
    for y in range(36):
        for x in range(48):
            col = np.zeros(3, np.float32)
            for s_ in range(4):
                h = hits[(y * 48 + x) * 4 + s_]
                if h["t"] > 0:
                    tid = h["triangleId"]
                    a, b, c = (sc.vertices[sc.tri[tid, k]] for k in range(3))
                    centre = (a + b + c) / np.float32(3)
                    n = sc.normals[sc.tri[tid, 3:]].sum(0) / np.float32(3)
                    n = n / np.linalg.norm(n)
                    d = centre - cam.eye
                    d = d / np.linalg.norm(d)
                    if not (np.dot(d, n) >= 0):
                        va, vb, vc = (np.mean(colors[tpv[sc.tri[tid, k]]], axis=0) for k in range(3))
                        col += h["u"] * va + h["v"] * vb + (1 - h["u"] - h["v"]) * vc
            want[y, x] = np.clip(col / np.float32(4), 0, 1)
    assert (img > 0).mean() > 0.15  # the box fills a good part of the frame
    assert np.allclose(img, want, rtol=1e-5, atol=2e-6)
    p.close()


def test_coplanar_skipping_changes_nothing(dz, uv50, monkeypatch):
    """Coplanar skipping (formfactor.cu: k_tri_planes / shaft_candidates) is a pure optimisation: with it switched off
    (DAISY_FF_RING=0) every triangle of a candidate list is tested by every sample.  Matrix and masks must be identical
    bit for bit at a size where most pairs take the skipping path."""
    from daisyriot_b200 import scenes
    sc = scenes.cornell_box(8192)
    got = {}
    for ring in ("1", "0"):
        monkeypatch.setenv("DAISY_FF_RING", ring)
        p = _ctx(dz, sc, uv50)
        got[ring] = (p.cudaCalculateRadiosityMatrix().rows().copy(), p.visibilityMasks(3000, 256).copy())
        p.close()
    assert np.array_equal(got["1"][0].view(np.uint32), got["0"][0].view(np.uint32))
    assert np.array_equal(got["1"][1], got["0"][1])


def test_face_grids_change_nothing(dz, uv50, monkeypatch):
    """The planar face grids (faces.cu; formfactor.cu: shaft_candidates / pair_mask_warp) are a pure optimisation: with them
    switched off (DAISY_FF_FACES=0) the triangles of a face are ordinary candidates again.  Matrix and masks must be
    identical bit for bit."""
    from daisyriot_b200 import scenes
    sc = scenes.cornell_box(8192)
    got = {}
    for faces in ("1", "0"):
        monkeypatch.setenv("DAISY_FF_FACES", faces)
        p = _ctx(dz, sc, uv50)
        got[faces] = (p.cudaCalculateRadiosityMatrix().rows().copy(), p.visibilityMasks(3000, 256).copy())
        p.close()
    assert np.array_equal(got["1"][0].view(np.uint32), got["0"][0].view(np.uint32))
    assert np.array_equal(got["1"][1], got["0"][1])


def test_edge_heavy_pattern_and_coplanar_decal_vs_bruteforce(dz):
    """Stress for the skipping premises, against the brute-force oracle (every ray against every triangle):
    * a sample pattern with samples ON the triangle edges and vertices (u = 0, v = 0, u + v = 1) next to random ones --
      edge samples must still test the coplanar neighbours;
    * a decal: two triangles lying IN the floor plane and overlapping floor patches -- k_tri_planes must disqualify the
      patches they overlap, because a ray leaving such a patch can start inside the decal."""
    from daisyriot_b200 import scenes
    from daisyriot_b200.scenes import Scene
    base = scenes.cornell_box(512)
    V = np.concatenate([base.vertices, np.array([[1.0, 0.0, 3.0], [2.1, 0.0, 3.0], [1.0, 0.0, 4.3], [2.1, 0.0, 4.3]], np.float32)])
    nv0, nn0 = len(base.vertices), len(base.normals)
    VN = np.concatenate([base.normals, np.array([[0, 1, 0]], np.float32)])
    T = np.concatenate([base.tri, np.array([[nv0, nv0 + 2, nv0 + 1, nn0, nn0, nn0], [nv0 + 1, nv0 + 2, nv0 + 3, nn0, nn0, nn0]], np.int32)])
    sc = Scene(V, VN, T, np.concatenate([base.mat_idx, [3, 3]]).astype(np.int32), base.materials, "cornell512_decal")
    rng = np.random.RandomState(11)
    u = rng.uniform(0, 1, 50).astype(np.float32)
    v = (rng.uniform(0, 1, 50).astype(np.float32) * (1 - u)).astype(np.float32)
    u[:6] = [0, 0, 1, 0.5, 0.25, 0]
    v[:6] = [0, 1, 0, 0.5, 0, 0.75]
    uv = np.stack([u, v], 1).astype(np.float32)
    p = _ctx(dz, sc, uv)
    F = p.cudaCalculateRadiosityMatrix().rows()
    masks = p.visibilityMasks()
    F_ref, masks_ref, _ = _oracle(sc).radmat_rows(uv, 0, sc.numtriangles, brute=True)
    assert np.array_equal(masks, masks_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    p.close()


def test_gather_tensor_core_path_at_scale(dz, uv50):
    """K = 32 on the tcgen05 3xTF32 path with 8192 columns per row (256 accumulator drains per item): the truncating
    tensor-core accumulator must not show up as a bias -- 1e-5 relative against the FP64-accumulating oracle, and the
    band sums (which expose any systematic bias directly) within 2e-6."""
    from daisyriot_b200 import _lib, scenes
    from oracle import pyoracle
    sc = scenes.cornell_box(8192)
    p = _ctx(dz, sc, uv50)
    N, K = sc.numtriangles, 32
    rng = np.random.RandomState(5)
    F = (rng.uniform(0, 1, (N, N)).astype(np.float32) * (rng.uniform(0, 1, (N, N)) < 0.3) / N).astype(np.float32)
    np.fill_diagonal(F, 0)
    p.loadRadiosityMatrix(F)
    M = rng.uniform(0, 0.06, (len(sc.materials), K, K)).astype(np.float32)
    E = np.ascontiguousarray(rng.uniform(0, 3, (K, N)).astype(np.float32))
    s = _solver(dz, p, K, E, M, sc.mat_idx)
    L = _lib.lib()
    res, B = E.copy(), E.copy()
    for it in range(2):
        sums = np.zeros(K)
        _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        sums_ref = pyoracle.gather_pass(F, res, B, M, sc.mat_idx, accum=1)
        Bg, Rg = np.empty_like(E), np.empty_like(E)
        _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
        for k in range(K):
            assert_rel(Rg[k], res[k], ("residual", it, k))
        assert np.allclose(sums, sums_ref, rtol=2e-6), (it, np.abs(sums / sums_ref - 1).max())
    L.daisy_solver_destroy(s)
    p.close()


@pytest.mark.parametrize("S,kind", [(7, "random"), (64, "random"), (33, "all_inner"), (20, "all_edge")])
def test_sample_counts_and_inner_edge_splits_vs_bruteforce(dz, cornell512, S, kind):
    """Sample counts other than 50 (one pass, two full passes, a one-lane second pass) and patterns that are all inner
    or all edge samples: masks (bit position = the caller's sample index) and matrix against the brute-force oracle."""
    rng = np.random.RandomState(100 + S)
    if kind == "all_inner":
        u = rng.uniform(0.05, 0.4, S)
        v = rng.uniform(0.05, 0.4, S)
    elif kind == "all_edge":
        u = rng.uniform(0, 1, S)
        v = (1 - u) * rng.choice([0.0, 0.003, 0.999], S)
    else:
        u = rng.uniform(0, 1, S)
        v = rng.uniform(0, 1, S) * (1 - u)
    uv = np.stack([u, v], 1).astype(np.float32)
    sc = cornell512
    p = _ctx(dz, sc, uv)
    F = p.cudaCalculateRadiosityMatrix().rows()
    masks = p.visibilityMasks()
    F_ref, masks_ref, _ = _oracle(sc).radmat_rows(uv, 0, sc.numtriangles, brute=True)
    assert np.array_equal(masks, masks_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    p.close()


@pytest.mark.parametrize("mode,K", [("fp32", 32), ("fp32", 12), ("ldg", 9)])
def test_gather_alternative_kernels_vs_oracle(dz, cornell2048, uv50, monkeypatch, mode, K):
    """The kernels behind DAISY_GATHER (CUDA-core TMA kernel for wide band counts, first-generation register-prefetch
    kernel) stay selectable as reference points; they must meet the same 1e-5 bar."""
    from daisyriot_b200 import _lib
    from oracle import pyoracle
    monkeypatch.setenv("DAISY_GATHER", mode)
    sc = cornell2048
    p = _ctx(dz, sc, uv50)
    N = sc.numtriangles
    rng = np.random.RandomState(40 + K)
    F = (rng.uniform(0, 1, (N, N)) * (rng.uniform(0, 1, (N, N)) < 0.3) / N).astype(np.float32)
    p.loadRadiosityMatrix(F)
    M = rng.uniform(0, 0.3, (len(sc.materials), K, K)).astype(np.float32)
    E = np.ascontiguousarray(rng.uniform(0, 3, (K, N)).astype(np.float32))
    s = _solver(dz, p, K, E, M, sc.mat_idx)
    L = _lib.lib()
    res, B = E.copy(), E.copy()
    for it in range(2):
        sums = np.zeros(K)
        _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        sums_ref = pyoracle.gather_pass(F, res, B, M, sc.mat_idx, accum=1)
        Bg, Rg = np.empty_like(E), np.empty_like(E)
        _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
        assert np.allclose(Rg, res, rtol=1e-5, atol=1e-5 * np.abs(res).max())
        assert np.allclose(sums, sums_ref, rtol=1e-6)
    L.daisy_solver_destroy(s)
    p.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_irregular_walls_vs_bruteforce(dz, uv50, seed):
    """Adversarial input for coplanar skipping: two facing walls and a tilted occluder triangulated irregularly (jittered grids,
    random diagonals, slivers, triangles 20x larger than their neighbours), vertex heights perturbed by rounding-sized noise
    on part of each wall, arbitrary wall orientation.  Masks and matrix must equal the brute-force oracle bit for bit."""
    sc = irregular_walls(seed)
    p = _ctx(dz, sc, uv50)
    F = p.cudaCalculateRadiosityMatrix().rows()
    masks = p.visibilityMasks()
    F_ref, masks_ref, _ = _oracle(sc).radmat_rows(uv50, 0, sc.numtriangles, brute=True)
    assert (masks_ref != 0).sum() > 1000  # the walls do see each other
    assert np.array_equal(masks, masks_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    p.close()


def test_samples_outside_the_triangle_vs_bruteforce(dz, cornell512):
    """The reference's pattern keeps (u, v) inside the triangle (OptixPrimeFunctionality.cpp:55-63) and every culling step of
    the kernel relies on it.  A caller's pattern that does not (u + v > 1, negative v) still has to give the closest-hit
    answer: the kernel then culls nothing and walks the LBVH per ray."""
    rng = np.random.RandomState(5)
    uv = rng.uniform(-0.3, 1.2, (50, 2)).astype(np.float32)
    assert ((uv.sum(1) > 1) | (uv.min(1) < 0)).sum() > 10
    sc = cornell512
    p = _ctx(dz, sc, uv)
    F = p.cudaCalculateRadiosityMatrix().rows()
    masks = p.visibilityMasks()
    F_ref, masks_ref, _ = _oracle(sc).radmat_rows(uv, 0, sc.numtriangles, brute=True)
    assert (masks_ref != 0).sum() > 1000
    assert np.array_equal(masks, masks_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    p.close()


@pytest.mark.parametrize("seed", [1, 2])
def test_perforated_faces_vs_bruteforce(dz, uv50, seed):
    """Adversarial input for the planar face grids (csrc/faces.cu): between a floor and a ceiling hangs a tilted plate with
    holes, a ragged outline, T-junctions (cells cut in four next to uncut neighbours) and a second, overlapping sheet in the
    very same plane; a fin stands ON the floor (its lower edge lies in the floor's plane, so rays leave and reach it flatly
    and skim the floor); the sample pattern holds samples exactly on triangle edges and vertices.  Everything is rotated
    arbitrarily.  Covered / mixed / empty cells, flat stretches and end-point margins all come into play; masks and matrix
    must equal the brute-force oracle (every ray against every triangle) bit for bit."""
    sc = perforated_plate(seed)
    # the usual pattern with eight samples moved onto edges and vertices
    uv = uv50.copy()
    uv[:8] = np.array([[0, 0], [1, 0], [0, 1], [0.5, 0], [0, 0.5], [0.5, 0.5], [0.25, 0.75], [1e-4, 0.3]], np.float32)
    p = _ctx(dz, sc, uv)
    assert p.stats().get("faces", 1) >= 1
    F = p.cudaCalculateRadiosityMatrix().rows()
    masks = p.visibilityMasks()
    F_ref, masks_ref, _ = _oracle(sc).radmat_rows(uv, 0, sc.numtriangles, brute=True)
    vis = np.array([bin(int(m)).count("1") for m in masks_ref.ravel()])
    assert (vis >= 40).sum() > 1000 and ((vis > 0) & (vis < 40)).sum() > 1000  # open and partially hidden pairs both occur
    assert np.array_equal(masks, masks_ref)
    assert np.array_equal(F.view(np.uint32), F_ref.view(np.uint32))
    p.close()


def test_per_pair_debug_entry_points_vs_oracle(dz, cornell512, uv50):
    """p2pFormfactorNusselt / p2pFormfactor / shootPatchRay (OptixPrimeFunctionality.cpp:273-306, :133-167, :456-469): host
    arithmetic around the GPU closest-hit query, against the same arithmetic around the oracle's closest hit."""
    from daisyriot_b200 import api
    sc = cornell512
    p = _ctx(dz, sc, uv50)
    orc = _oracle(sc)
    rng = np.random.RandomState(9)
    real_query = p.optixQuery
    checked = 0
    for _ in range(24):
        a, b = (int(x) for x in rng.randint(0, sc.numtriangles, 2))
        if a == b:
            continue
        got = (p.p2pFormfactorNusselt(a, b), p.p2pFormfactor(a, b))
        p.optixQuery = lambda n, rays, hits=None: orc.query_closest(np.asarray(rays, np.float32).reshape(-1, 6)[:n])
        want = (p.p2pFormfactorNusselt(a, b), p.p2pFormfactor(a, b))
        picks = np.zeros(2, api.HIT_DTYPE)
        picks["triangleId"] = [a, b]
        picks["u"], picks["v"] = rng.uniform(0, 0.5, 2), rng.uniform(0, 0.5, 2)
        shot_want = p.shootPatchRay(picks)
        p.optixQuery = real_query
        assert got == want and p.shootPatchRay(picks) == shot_want
        checked += got[0] > 0
    assert checked >= 3
    p.close()
