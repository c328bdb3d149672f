"""Geometry far from the origin, against brute force.

Every conservative tolerance of the LBVH and the form-factor kernel (box padding, face-grid margins, coplanar thresholds) is
a fraction of the scene extent, while float32 coordinates round at ulp(max |coord|).  These tests move and scale scenes until
that ulp passes the 1e-4 x extent box padding, and compare closest hits (optixQuery, daisy_query_closest_device, traceScreen)
and the form-factor build (matrix and visibility masks, both variants, every culling path) bit for bit with the brute-force
oracle on the SAME float32 scene: far from the origin the reference algorithm itself gives different numbers (the 1e-6
origin nudge and the sample points round away), so only brute force on the translated scene is a valid reference."""
import ctypes as C

import numpy as np
import pytest

import geometry_scenes as gs
from oracle.pyoracle import Oracle

pytestmark = pytest.mark.gpu

CORNELL_KEYS = list(gs.OFFSETS) + list(gs.SCALES)
WALLS = ["irregular1", "irregular2", "perforated1", "perforated2"]


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


_SCENES, _BRUTE = {}, {}


def _scene(name, ties=False):
    key = (name, ties)
    if key not in _SCENES:
        if name in WALLS:
            base = gs.irregular_walls(int(name[-1])) if name.startswith("irregular") else gs.perforated_plate(int(name[-1]))
            sc = gs.moved(base, offset=gs.FAR_DIRECTION_32768, name=name + "@32768")
        else:
            sc = gs.cornell512_at(name)
        _SCENES[key] = gs.with_ties(sc) if ties else sc
    return _SCENES[key]


def _brute_ff(name, uv, variant):
    """Whole matrix and masks of the brute-force oracle, cached per (scene, pattern, variant)."""
    key = (name, uv.tobytes(), variant)
    if key not in _BRUTE:
        sc = _scene(name)
        _BRUTE[key] = Oracle.from_scene(sc).radmat_rows(uv, 0, sc.numtriangles, variant=variant, reciprocity=bool(variant), brute=True)[:2]
    return _BRUTE[key]


def _ctx(dz, sc, uv):
    return dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv)


def _assert_same_hits(got, want, what):
    bad = ((got["triangleId"] != want["triangleId"]) | (got["t"].view(np.uint32) != want["t"].view(np.uint32))
           | (got["u"].view(np.uint32) != want["u"].view(np.uint32)) | (got["v"].view(np.uint32) != want["v"].view(np.uint32)))
    assert not bad.any(), (what, int(bad.sum()), "of", bad.size, "rays differ; first", np.flatnonzero(bad)[:8])


def _rays(sc, uv, seed):
    orc = Oracle.from_scene(sc)
    N = sc.numtriangles
    pair = np.concatenate([orc.pair_rays(i, j, uv) for i, j in [(0, N - 1), (3, 100), (17, 300), (40, 41), (200, N // 2)]])
    return np.ascontiguousarray(np.concatenate([gs.closest_hit_rays(sc, seed), pair]), np.float32)


# ---- closest hit ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CORNELL_KEYS + WALLS)
def test_closest_hit_far_vs_bruteforce(dz, uv50, name):
    """optixQuery: random and pair rays, axis-parallel rays through vertices (every axis, both signs), rays along edges and
    rays starting on a triangle, over a scene with flipped duplicates and zero-area triangles (ties on t)."""
    sc = _scene(name, ties=True)
    rays = _rays(sc, uv50, 1)
    p = _ctx(dz, sc, uv50)
    got = p.optixQuery(rays.shape[0], rays)
    p.close()
    want = Oracle.from_scene(sc).query_closest(rays, brute=True)
    assert (want["triangleId"] >= 0).mean() > 0.3
    _assert_same_hits(got, want, name)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 1037])
@pytest.mark.parametrize("name", ["o0", "o32768", "s1e3"])
def test_query_closest_device_vs_bruteforce(dz, uv50, name, n):
    """daisy_query_closest_device on torch CUDA tensors, at ray counts around the 128-thread block of k_closest."""
    import torch
    from daisyriot_b200 import _lib
    from daisyriot_b200.api import HIT_DTYPE
    sc = _scene(name, ties=True)
    allr = _rays(sc, uv50, 3)
    rays = np.ascontiguousarray(allr[np.random.RandomState(n).choice(allr.shape[0], n, replace=False)])
    p = _ctx(dz, sc, uv50)
    d_rays = torch.from_numpy(rays).cuda()
    d_hits = torch.full((n, 4), -7.0, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    _lib.check(_lib.lib().daisy_query_closest_device(p._ctx, n, C.c_void_p(d_rays.data_ptr()), C.c_void_p(d_hits.data_ptr())))
    got = d_hits.cpu().numpy().view(HIT_DTYPE).reshape(n)
    p.close()
    _assert_same_hits(got, Oracle.from_scene(sc).query_closest(rays, brute=True), (name, n))


def _literal_trace(sc, eye, hits, colors, W, H, samples, interpolate):
    """OptixPrimeFunctionality::traceScreen's per-pixel loop (.cpp:83-131, Drawer.cpp:161-186) over given hit records."""
    tpv = [[] for _ in range(len(sc.vertices))]
    for t in range(sc.numtriangles):
        for k in range(3):
            tpv[sc.tri[t, k]].append(t)
    want = np.zeros((H, W, 3), np.float32)
    for y in range(H):
        for x in range(W):
            col = np.zeros(3, np.float32)
            for s_ in range(samples):
                h = hits[(y * W + x) * samples + s_]
                if h["t"] > 0:
                    tid = h["triangleId"]
                    a, b, c = (sc.vertices[sc.tri[tid, k]] for k in range(3))
                    centre = (a + b + c) / np.float32(3)
                    n = sc.normals[sc.tri[tid, 3:]].sum(0) / np.float32(3)
                    n = n / np.linalg.norm(n)
                    d = centre - eye
                    d = d / np.linalg.norm(d)
                    if not (np.dot(d, n) >= 0):
                        if interpolate:
                            va, vb, vc = (np.mean(colors[tpv[sc.tri[tid, k]]], axis=0) for k in range(3))
                            col += h["u"] * va + h["v"] * vb + (1 - h["u"] - h["v"]) * vc
                        else:
                            col += colors[tid]
            want[y, x] = np.clip(col / np.float32(samples), 0, 1)
    return want


@pytest.mark.parametrize("W,H,interpolate,with_hits", [(48, 36, True, True), (37, 5, False, True), (37, 5, True, False)])
@pytest.mark.parametrize("name", ["o0", "o16384", "o32768", "o3e5"])
def test_trace_screen_far_vs_literal_restatement(dz, uv50, name, W, H, interpolate, with_hits):
    """traceScreen on the translated box, camera translated alike: the camera rays of the untranslated view with their
    origins moved by the same offset (the reference passes the far-plane point as the direction, so the direction stays),
    the eye moved too.  Hit records bit for bit against brute force; the frame against the literal per-pixel loop over the
    brute-force hits, with interpolation on and off and a ragged frame."""
    from daisyriot_b200 import api
    sc = _scene(name)
    off = np.asarray(gs.OFFSETS[name], np.float64)
    cam = api.Camera(W, H, 4)
    cam.eye = np.array([2.75, 2.75, 14.0], np.float32)
    cam.dir = np.array([2.75, 2.75, 0.0], np.float32)
    rays = cam.gen_rays_for_screen(True)
    rays[:, :3] = (rays[:, :3].astype(np.float64) + off).astype(np.float32)
    cam.eye = (cam.eye.astype(np.float64) + off).astype(np.float32)
    mesh = dz.MeshS.from_scene(sc)
    p = dz.OptixPrimeFunctionality(mesh, rands=uv50)
    colors = np.random.RandomState(2).uniform(0, 1.2, (sc.numtriangles, 3)).astype(np.float32)
    mat_colors = np.random.RandomState(3).uniform(0, 1, (int(mesh.materialIndexPerTriangle.max()) + 1, 3)).astype(np.float32)
    out = api.traceScreen(p, cam, colors, interpolate, True, material_colors=mat_colors, rays=rays, return_hits=with_hits)
    p.close()
    img = out[0] if with_hits else out
    hits = Oracle.from_scene(sc).query_closest(rays, brute=True)
    assert (hits["t"] > 0).mean() > 0.03  # a quarter of the 48 x 36 frame, a twentieth of the wide 37 x 5 one
    if with_hits:
        _assert_same_hits(out[1], hits, (name, W, H))
    shade = colors if interpolate else mat_colors[mesh.materialIndexPerTriangle]
    want = _literal_trace(sc, cam.eye, hits, shade, W, H, 4, interpolate)
    assert (img > 0).mean() > 0.03
    assert np.allclose(img, want, rtol=1e-5, atol=2e-6), (name, np.abs(img - want).max())


# ---- form factors ---------------------------------------------------------------------------------------------------------
FF_KEYS = ["o0", "o16", "o4096", "o16384", "o32768", "o3e5", "s1e-3", "s1e3", "s0.37"]
MODES = {"default": {}, "no_faces": {"DAISY_FF_FACES": "0"}, "no_ring": {"DAISY_FF_RING": "0"}}


def _check_ff(dz, sc, uv, name, variant):
    p = _ctx(dz, sc, uv)
    rm = p.cudaCalculateRadiosityMatrix() if variant == 0 else p.calculateRadiosityMatrix()
    F = rm.rows()
    masks = p.visibilityMasks(variant=variant)
    p.close()
    F_ref, m_ref = _brute_ff(name, uv, variant)
    assert (m_ref != 0).sum() > 1000
    if variant == 0:
        assert np.array_equal(masks, m_ref), (name, int((masks != m_ref).sum()), "masks differ")
    else:  # the per-pair path traces every pair; the fused kernel skips pairs whose factor is zero anyway
        traced = masks != 0
        assert np.array_equal(masks[traced], m_ref[traced]), (name, "masks differ")
    bad = F.view(np.uint32) != F_ref.view(np.uint32)
    assert not bad.any(), (name, int(bad.sum()), "matrix entries differ")


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("name", FF_KEYS)
def test_form_factors_far_vs_bruteforce(dz, uv50, monkeypatch, name, mode):
    """Whole matrix and masks (fused kernel, device variant) with face grids and coplanar skipping on and off."""
    for k, v in MODES[mode].items():
        monkeypatch.setenv(k, v)
    _check_ff(dz, _scene(name), uv50, name, 0)


@pytest.mark.parametrize("name", ["o16", "o32768", "s0.37"])
def test_form_factors_far_host_variant_vs_bruteforce(dz, uv50, name):
    """The per-pair variant (float pi, reciprocity) on the same scenes."""
    _check_ff(dz, _scene(name), uv50, name, 1)


@pytest.mark.parametrize("name", ["o16384", "o32768", "s1e3"])
def test_form_factors_far_samples_outside_the_triangle(dz, name):
    """A pattern with samples outside the triangle: every pair takes the per-ray LBVH walk (ray_sees)."""
    uv = np.random.RandomState(5).uniform(-0.3, 1.2, (50, 2)).astype(np.float32)
    _check_ff(dz, _scene(name), uv, name, 0)


@pytest.mark.parametrize("name", WALLS)
def test_form_factors_far_walls_vs_bruteforce(dz, uv50, name):
    """The adversarial wall scenes of the parity suite (irregular triangulations, a perforated plate with coplanar sheets)
    moved 32768 along an arbitrary direction; the perforated plates keep their samples on edges and vertices."""
    uv = uv50.copy()
    if name.startswith("perforated"):
        uv[:8] = np.array([[0, 0], [1, 0], [0, 1], [0.5, 0], [0, 0.5], [0.5, 0.5], [0.25, 0.75], [1e-4, 0.3]], np.float32)
    _check_ff(dz, _scene(name), uv, name, 0)


@pytest.mark.parametrize("name", ["o0", "o32768"])
def test_visibility_masks_ragged_windows_far(dz, uv50, name):
    """visibilityMasks over row windows that start and end off the 64-patch tiles, against the brute-force masks."""
    sc = _scene(name)
    _, m_ref = _brute_ff(name, uv50, 0)
    p = _ctx(dz, sc, uv50)
    for r0, nr in [(0, 1), (1, 62), (63, 66), (129, 127), (300, 211), (511, 1)]:
        m = p.visibilityMasks(r0, nr)
        assert np.array_equal(m, m_ref[r0:r0 + nr]), (name, r0, nr)
    p.close()
