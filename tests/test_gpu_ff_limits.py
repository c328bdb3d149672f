"""The form-factor kernel past its fixed capacities, against the brute-force oracle (every ray against every triangle), bit for
bit: F as uint32 patterns, masks as uint64.  Scenes and their CPU premises: geometry_scenes.py, test_ff_limits_scenes.py.
* SHAFT_CAP = 256 shaft candidates: a pair with more is resolved by phase 2b (one LBVH walk per ray, its own coplanar
  skipping and mask assembly), next to list pairs of the same tile, in updates and in row partitions;
* DAISY_MAX_FACES = 64 face grids: faces 32-63 (the upper word of the 64-bit face mask) and planes left without a grid;
* NBR_CAP = 32 (31 neighbours): patches on both sides of a full neighbour list."""
import numpy as np
import pytest

from daisyriot_b200 import scenes
from geometry_scenes import (edge_pattern, facing_pairs, fan_floor, lifted, many_planes, occluded_walls, random_pattern,
                             shaft_cap_scene)
from oracle.pyoracle import Oracle
from test_ff_limits_scenes import wall_overflow_lower_bound

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


def _ctx(dz, sc, uv, **kw):
    return dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv, **kw)


def _same_F(got, want, what=""):
    assert got.shape == want.shape, what
    bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))
    assert bad[0].size == 0, (what, "entries differ", bad[0].size, list(zip(bad[0][:5], bad[1][:5])))


def _same_masks(got, want, what=""):
    bad = np.nonzero(got != want)
    assert bad[0].size == 0, (what, "masks differ", bad[0].size, list(zip(bad[0][:5], bad[1][:5])))


def _build_vs_brute(dz, sc, uv, variant=0):
    """Whole matrix and masks of one build against the oracle; returns the build's stats."""
    p = _ctx(dz, sc, uv)
    F = (p.cudaCalculateRadiosityMatrix() if variant == 0 else p.calculateRadiosityMatrix()).rows()
    masks = p.visibilityMasks(variant=variant)
    st = p.stats()
    p.close()
    F_ref, m_ref, _ = Oracle.from_scene(sc).radmat_rows(uv, 0, sc.numtriangles, variant=variant, reciprocity=bool(variant), brute=True)
    _same_F(F, F_ref, sc.name)
    if variant == 0:
        _same_masks(masks, m_ref, sc.name)
    else:  # the per-pair path traces every pair; the fused kernel skips pairs whose factor is zero anyway
        traced = masks != 0
        _same_masks(masks[traced], m_ref[traced], sc.name)
    return st, masks


# ---- 1. the 256 / 257 boundary of the shaft lists ------------------------------------------------------------------------------
@pytest.mark.parametrize("n_occ", [0, 1, 15, 16, 17, 255, 256, 257])
def test_shaft_cap_boundary(dz, uv50, n_occ):
    """(A, B) has exactly n_occ candidates (test_shaft_cap_scene_candidates), every other pair fewer than 257: the pair falls
    back to phase 2b exactly when n_occ > 256, and nothing else does.  The small counts cover the 16-entry candidate staging."""
    sc = shaft_cap_scene(n_occ)
    st, masks = _build_vs_brute(dz, sc, uv50)
    assert st["pairs_fallback"] == (1 if n_occ > 256 else 0), st
    assert st["pairs_traced"] == len(facing_pairs(Oracle.from_scene(sc)))
    if n_occ >= 255:
        assert 0 < bin(int(masks[0, 1])).count("1") < 50  # partly hidden
    if n_occ >= 256:
        st_h, _ = _build_vs_brute(dz, sc, uv50, variant=1)
        assert st_h["pairs_fallback"] == st["pairs_fallback"]


# ---- 2. many fallback pairs with coplanar walls ---------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["default", "ring0", "faces0"])
@pytest.mark.parametrize("pattern", ["edge50", "random64", "random33"])
@pytest.mark.parametrize("nu,nv", [(4, 3), (6, 6)])
def test_mass_fallback_with_coplanar_walls(dz, uv50, monkeypatch, nu, nv, pattern, mode):
    """Hundreds of wall-to-wall pairs overflow and share tiles with list pairs.  Their inner samples skip the walls' own planes
    in phase 2b while edge samples (edge50: eight samples on edges and vertices) must test them: rays that end on an edge
    shared with a lower-id neighbour lose the tie.  64 samples fill both 32-lane passes, 33 leave one lane in the second."""
    if mode == "ring0":
        monkeypatch.setenv("DAISY_FF_RING", "0")
    if mode == "faces0":
        monkeypatch.setenv("DAISY_FF_FACES", "0")
    uv = {"edge50": edge_pattern(uv50), "random64": random_pattern(64, 64), "random33": random_pattern(33, 33)}[pattern]
    sc = occluded_walls(nu, nv)
    st, _ = _build_vs_brute(dz, sc, uv)
    heavy, _ = wall_overflow_lower_bound(sc, nu, nv)
    assert len(heavy) <= st["pairs_fallback"] <= st["pairs_traced"], (len(heavy), st)


# ---- 3. mask windows ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene", ["shaft_cap257", "walls4x3"])
def test_mask_windows_through_the_fallback(dz, uv50, scene):
    sc = shaft_cap_scene(257) if scene == "shaft_cap257" else occluded_walls(4, 3)
    uv = edge_pattern(uv50)
    p = _ctx(dz, sc, uv)
    full = p.visibilityMasks()
    _, m_ref, _ = Oracle.from_scene(sc).radmat_rows(uv, 0, sc.numtriangles, brute=True)
    _same_masks(full, m_ref, "full")
    for row0, nrows in [(1, 37), (250, 9), (0, 1), (sc.numtriangles - 1, 1)]:
        w = p.visibilityMasks(row0, nrows)
        _same_masks(w, full[row0:row0 + nrows], (row0, nrows))
    p.close()


# ---- 4. row partitions ----------------------------------------------------------------------------------------------------------
def test_row_partitions_through_the_fallback(dz, uv50):
    """A = triangle 0, B = the last triangle (258).  Two ranks: rank 1 owns rows 256-258.  Three ranks: rank 2 owns none.  Both
    ranks that hold A or B trace the heavy pair."""
    sc0 = shaft_cap_scene(257)
    order = np.r_[0, 2:sc0.numtriangles, 1]
    sc = scenes.Scene(sc0.vertices, sc0.normals, sc0.tri[order], sc0.mat_idx[order], sc0.materials, "shaft_cap257_reordered")
    N = sc.numtriangles
    p = _ctx(dz, sc, uv50)
    F1 = p.cudaCalculateRadiosityMatrix().rows()
    st1 = p.stats()
    p.close()
    assert st1["pairs_fallback"] == 1
    F_ref, _, _ = Oracle.from_scene(sc).radmat_rows(uv50, 0, N, brute=True)
    _same_F(F1, F_ref, "single")
    for nranks in (2, 3):
        rows, owned = [], 0
        for rank in range(nranks):
            q = _ctx(dz, sc, uv50, rank=rank, nranks=nranks)
            r0, r1 = q.row_range
            R = q.cudaCalculateRadiosityMatrix().rows()
            st = q.stats()
            q.close()
            assert R.shape == (r1 - r0, N)
            rows.append(R)
            owned += st["pairs_owned"]
            holds_ab = r0 <= 0 < r1 or r0 <= N - 1 < r1
            assert st["pairs_fallback"] == (1 if holds_ab else 0), (nranks, rank, st)
            if nranks == 2 and rank == 1:
                assert (r0, r1) == (256, N)
            if nranks == 3 and rank == 2:
                assert r0 == r1
        _same_F(np.concatenate(rows), F1, nranks)
        assert owned == st1["pairs_traced"], (nranks, owned, st1)


# ---- 5. updates ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("direction", ["257_to_256", "256_to_257"])
def test_update_across_the_cap(dz, uv50, direction):
    """Lifting occluder 2 above B (same x, y; z in [1.5, 2.5]) takes (A, B) from 257 candidates to 256; moving the parked one
    back in goes the other way.  The extent, and with it the box padding, stays the same.  The update re-traces (A, B): the
    result equals a fresh build and brute force, and the stats show the update's own pass."""
    sc = shaft_cap_scene(257)
    V_in, V_up = sc.vertices.copy(), lifted(sc, 2)
    V0, V1 = (V_in, V_up) if direction == "257_to_256" else (V_up, V_in)
    start = scenes.Scene(V0, sc.normals, sc.tri, sc.mat_idx, sc.materials, "start")
    end = scenes.Scene(V1, sc.normals, sc.tri, sc.mat_idx, sc.materials, "end")
    p = _ctx(dz, start, uv50)
    p.cudaCalculateRadiosityMatrix()
    assert p.stats()["pairs_fallback"] == (1 if direction == "257_to_256" else 0)
    p.updateGeometry(vertices=V1)
    F = p.updateRadiosityMatrix().rows()
    st, ust = p.stats(), p.update_stats()
    p.close()
    assert ust["tris_changed"] == 1 and ust["pairs_retraced"] > 0, ust
    assert st["pairs_fallback"] == (0 if direction == "257_to_256" else 1), st
    q = _ctx(dz, end, uv50)
    F_fresh = q.cudaCalculateRadiosityMatrix().rows()
    q.close()
    F_ref, _, _ = Oracle.from_scene(end).radmat_rows(uv50, 0, end.numtriangles, brute=True)
    _same_F(F_fresh, F_ref, "fresh")
    _same_F(F, F_ref, "update")


# ---- 6. 64 face grids ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nplates", [63, 64, 65, 70])
def test_64_face_grids(dz, uv50, monkeypatch, nplates):
    """Plate q is face q up to 64 faces (test_many_planes_faces); vertical plates among faces 32-63 and among the planes left
    without a grid block floor-to-ceiling rays.  The whole matrix equals the build without grids; sampled rows -- first,
    middle and last face, every plane left over, the occluders -- equal brute force."""
    sc = many_planes(nplates)
    uv = edge_pattern(uv50)
    got = {}
    for faces in ("1", "0"):
        monkeypatch.setenv("DAISY_FF_FACES", faces)
        p = _ctx(dz, sc, uv)
        F = p.cudaCalculateRadiosityMatrix().rows()
        got[faces] = (F, p.visibilityMasks(), p.stats())
        p.close()
    assert got["1"][2]["faces"] == min(nplates, 64) and got["0"][2]["faces"] == 0
    _same_F(got["1"][0], got["0"][0], "faces on / off")
    _same_masks(got["1"][1], got["0"][1], "faces on / off")
    rows = [32 * q + k for q in [0, 32, min(nplates, 64) - 1] + list(range(64, nplates)) for k in (0, 13, 31)]
    rows += [32 * nplates + k for k in (0, 17, 39)]
    F_ref, m_ref, _ = Oracle.from_scene(sc).radmat_rowlist(uv, rows, brute=True)
    _same_F(got["1"][0][rows], F_ref, "sampled rows")
    _same_masks(got["1"][1][rows], m_ref, "sampled rows")


# ---- 7. full neighbour lists ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("faces", ["1", "0"])
@pytest.mark.parametrize("n", [32, 33, 40])
def test_fan_neighbour_cap(dz, uv50, monkeypatch, n, faces):
    """Every fan triangle has n - 1 coplanar neighbours: 31 fill the list, 32 and 39 are past it and the patch loses coplanar
    skipping.  Edge samples end on shared edges and on the centre vertex, where a lower-id neighbour wins the tie."""
    monkeypatch.setenv("DAISY_FF_FACES", faces)
    _build_vs_brute(dz, fan_floor(n), edge_pattern(uv50))
