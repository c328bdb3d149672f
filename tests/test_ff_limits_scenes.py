"""CPU premises of the capacity-limit scenes (geometry_scenes.py; GPU comparisons in test_gpu_ff_limits.py).  Each test states
what a GPU test relies on -- shaft candidate counts on either side of SHAFT_CAP = 256, plane ids, 64 face grids with planes
left over, neighbour counts on either side of NBR_CAP - 1 = 31 -- and that the oracle can see the difference, so that a
scene that misses its purpose fails here instead of letting the GPU test pass vacuously.  Host only: the C oracle and the
library's host-side diagnostics (daisy_plane_ids, daisy_face_grid_stats), no device."""
import ctypes as C

import numpy as np
import pytest

from daisyriot_b200 import _lib, scenes
from geometry_scenes import (MANY_PLANES_KINDS, edge_pattern, facing_pairs, fan_floor, lifted, many_planes, occluded_walls,
                             padded_boxes, shaft_cap_scene, shaft_meets)
from oracle.pyoracle import Oracle

SHAFT_CAP = 256


def _ext(V):
    return float((V.max(0) - V.min(0)).max())


def plane_ids(sc):
    v, t = np.ascontiguousarray(sc.vertices, np.float32), np.ascontiguousarray(sc.tri, np.int32)
    out = np.zeros(t.shape[0], np.int32)
    _lib.check(_lib.lib().daisy_plane_ids(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], _lib.iptr(out)))
    return out


def face_grids(sc):
    """(number of face grids, plane ids as the kernel sees them: face f = id f + 1, other planes above)."""
    v, t = np.ascontiguousarray(sc.vertices, np.float32), np.ascontiguousarray(sc.tri, np.int32)
    st = np.zeros((64, 6), np.int64)
    nf = C.c_int(0)
    pid = np.zeros(t.shape[0], np.int32)
    _lib.check(_lib.lib().daisy_face_grid_stats(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], 64, st.ctypes.data_as(C.POINTER(C.c_int64)),
                                                C.byref(nf), _lib.iptr(pid)))
    return nf.value, pid


def occluder_counts(sc, pairs, occluders, pad):
    """Per pair: occluders (other than the pair's own triangles) whose box, grown by pad, meets the pair's shaft."""
    m = shaft_meets(sc, pairs, padded_boxes(sc, occluders, pad))
    own = np.asarray(pairs)[:, :, None] == np.asarray(occluders)[None, None, :]
    return (m & ~own.any(1)).sum(1)


def shaft_cap_counts(sc, a, b, occluders):
    """(candidates of (a, b), most candidates of any other facing pair), each with the box padding of the kernel (1e-4 x
    extent) and both halved and doubled: the float32 kernel rounds far inside that range."""
    fp = facing_pairs(Oracle.from_scene(sc))
    ab = np.nonzero((fp[:, 0] == min(a, b)) & (fp[:, 1] == max(a, b)))[0]
    assert len(ab) == 1, "A and B must face each other"
    out = []
    for k in (0.5, 1.0, 2.0):
        c = occluder_counts(sc, fp, occluders, k * 1e-4 * _ext(sc.vertices))
        out.append((int(c[ab[0]]), int(np.delete(c, ab).max(initial=0))))
    assert out[0] == out[1] == out[2], out
    return out[1]


def wall_overflow_lower_bound(sc, nu, nv):
    """Wall-to-wall pairs (lo on the z = 0 wall, hi on the z = 1 wall) that must overflow: counting only occluders, with half
    the kernel's box padding, their shafts already hold more than SHAFT_CAP."""
    w = 2 * nu * nv
    fp = facing_pairs(Oracle.from_scene(sc))
    ww = fp[(fp[:, 0] < w) & (fp[:, 1] >= w) & (fp[:, 1] < 2 * w)]
    c = occluder_counts(sc, ww, np.arange(2 * w, sc.numtriangles), 0.5e-4 * _ext(sc.vertices))
    return ww[c > SHAFT_CAP], len(ww)


@pytest.mark.parametrize("n_occ", [0, 1, 16, 255, 256, 257])
def test_shaft_cap_scene_candidates(n_occ):
    sc = shaft_cap_scene(n_occ)
    ab, other = shaft_cap_counts(sc, 0, 1, np.arange(2, sc.numtriangles))
    assert ab == n_occ and other < SHAFT_CAP + 1 and (n_occ < 2 or other <= n_occ - 1)
    pid = plane_ids(sc)
    assert (pid[2:] == 0).all() and pid[0] > 0 and pid[1] > 0 and pid[0] != pid[1]


def test_shaft_cap_scene_mask_is_partial(uv50):
    sc = shaft_cap_scene(257)
    orc = Oracle.from_scene(sc)
    hits = orc.query_closest(orc.pair_rays(0, 1, uv50), brute=True)
    seen = int((hits["triangleId"] == 1).sum())
    assert 10 <= seen <= 40, seen


def test_shaft_cap_scene_moves():
    """The update cases: lifting one occluder above B (z in [1.5, 2.5], same x and y) takes (A, B) from 257 to 256 candidates
    and keeps the extent, so the box padding stays the same; parking it there and moving it back goes the other way."""
    sc = shaft_cap_scene(257)
    up = scenes.Scene(lifted(sc, 2), sc.normals, sc.tri, sc.mat_idx, sc.materials, "lifted")
    assert _ext(up.vertices) == _ext(sc.vertices) == 10.0
    assert up.vertices[up.tri[2, :3], 2].min() > 1.5 and up.vertices[up.tri[2, :3], 2].max() < 2.5
    assert shaft_cap_counts(up, 0, 1, np.arange(2, sc.numtriangles))[0] == 256
    assert shaft_cap_counts(sc, 0, 1, np.arange(2, sc.numtriangles))[0] == 257


def test_shaft_cap_scene_reordered():
    """The row-partition case: A is triangle 0 and B the last one; the counts do not depend on the order."""
    sc = shaft_cap_scene(257)
    order = np.r_[0, 2:sc.numtriangles, 1]
    ro = scenes.Scene(sc.vertices, sc.normals, sc.tri[order], sc.mat_idx[order], sc.materials, "reordered")
    assert shaft_cap_counts(ro, 0, ro.numtriangles - 1, np.arange(1, ro.numtriangles - 1))[0] == 257


@pytest.mark.parametrize("nu,nv,gridded", [(4, 3, False), (6, 6, True)])
def test_occluded_walls_premises(uv50, nu, nv, gridded):
    sc = occluded_walls(nu, nv)
    w = 2 * nu * nv
    heavy, nww = wall_overflow_lower_bound(sc, nu, nv)
    assert len(heavy) >= 100, len(heavy)
    pid = plane_ids(sc)
    assert (pid[2 * w:] == 0).all() and len(set(pid[:w])) == 1 and len(set(pid[w:2 * w])) == 1 and pid[0] != pid[w] and pid[0] > 0
    nf, _ = face_grids(sc)
    assert nf == (2 if gridded else 0)
    # an edge sample's ray may end on the destination's coplanar neighbour (a tie on a shared edge or vertex, lower id wins):
    # skipping the own plane for such a sample would change the mask
    orc = Oracle.from_scene(sc)
    uv = edge_pattern(uv50)
    on_nbr = 0
    for lo, hi in heavy[::max(1, len(heavy) // 40)]:
        h = orc.query_closest(orc.pair_rays(lo, hi, uv), brute=True)["triangleId"]
        on_nbr += int(((h >= w) & (h < 2 * w) & (h != hi)).sum())
    assert on_nbr > 0


@pytest.mark.parametrize("nplates,nfaces,left", [(63, 63, 0), (64, 64, 0), (65, 64, 1), (70, 64, 6)])
def test_many_planes_faces(nplates, nfaces, left):
    sc = many_planes(nplates)
    nf, pid = face_grids(sc)
    ids, cnt = np.unique(pid[pid > 0], return_counts=True)
    assert nf == nfaces and ((ids > nf) & (cnt >= 32)).sum() == left
    assert (pid[32 * nplates:] == 0).all()
    # plate q is face q (all plates have 32 triangles; ties keep the order), planes after the 64th have no grid
    assert all((pid[32 * q:32 * q + 32] == q + 1).all() for q in range(min(nplates, 64)))
    assert all((pid[32 * q:32 * q + 32] > 64).all() for q in range(64, nplates))


def many_planes_blockers(sc, uv, pairs):
    """Plane ids (kernel numbering) of the triangles that end the pairs' rays short of the destination."""
    orc = Oracle.from_scene(sc)
    _, pid = face_grids(sc)
    out = []
    for lo, hi in pairs:
        h = orc.query_closest(orc.pair_rays(lo, hi, uv), brute=True)["triangleId"]
        out += [int(pid[k]) for k in h if k >= 0 and k != hi and k != lo]
    return np.asarray(out, np.int64)


def many_planes_sample_pairs(nplates, seed=1):
    """Floor-to-ceiling plate pairs: the rays the vertical plates stand in."""
    kinds = [MANY_PLANES_KINDS[(q + 1) % 3] for q in range(nplates)]
    floor = [q for q in range(nplates) if kinds[q] == "floor"]
    ceil = [q for q in range(nplates) if kinds[q] == "ceiling"]
    rng = np.random.RandomState(seed)
    f = rng.choice(floor, 400) * 32 + rng.randint(0, 32, 400)
    c = rng.choice(ceil, 400) * 32 + rng.randint(0, 32, 400)
    return np.stack([np.minimum(f, c), np.maximum(f, c)], 1)


def test_many_planes_upper_faces_and_ungridded_planes_block_rays(uv50):
    sc = many_planes(70)
    nf, pid = face_grids(sc)
    blk = many_planes_blockers(sc, uv50, many_planes_sample_pairs(70))
    assert ((blk >= 33) & (blk <= 64)).sum() > 0   # faces 32-63: the upper half of the 64-bit face mask
    assert ((blk >= 1) & (blk <= 32)).sum() > 0    # and the lower half
    assert (blk > nf).sum() > 0                     # a plane of 32 triangles without a grid


@pytest.mark.parametrize("n", [32, 33, 40])
def test_fan_floor_neighbours(uv50, n):
    sc = fan_floor(n)
    fan = np.arange(3, 3 + n)
    pid = plane_ids(sc)
    assert len(set(pid[fan])) == 1 and pid[3] > 0 and pid[2] != pid[3]
    # every fan triangle holds the centre vertex: each has n - 1 coplanar neighbours whose boxes meet its own
    assert (sc.tri[fan, 0] == sc.tri[3, 0]).all()
    # sliver rule of k_tri_planes: 8 x smallest altitude >= longest edge
    P = sc.vertices[sc.tri[fan, :3]].astype(np.float64)
    e = np.stack([P[:, 1] - P[:, 0], P[:, 2] - P[:, 0], P[:, 2] - P[:, 1]], 1)
    L = np.linalg.norm(e, axis=2).max(1)
    h = np.linalg.norm(np.cross(e[:, 0], e[:, 1]), axis=1) / L
    assert (8 * h >= L).all()
    # rays from the plate may end on a fan neighbour of the destination (shared edges and the centre vertex)
    orc = Oracle.from_scene(sc)
    uv = edge_pattern(uv50)
    on_nbr = 0
    for lo in (0, 1):
        for hi in fan:
            k = orc.query_closest(orc.pair_rays(lo, hi, uv), brute=True)["triangleId"]
            on_nbr += int(((k >= 3) & (k != hi)).sum())
    assert on_nbr > 0
