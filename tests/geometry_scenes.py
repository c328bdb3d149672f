"""Scene builders shared by the geometry tests: the adversarial walls of test_gpu_parity.py, translated / scaled copies of
any scene for the far-from-origin tests (test_far_geometry_oracle.py, test_gpu_far_geometry.py), and the scenes that push
the form-factor kernel past its fixed capacities (test_ff_limits_scenes.py, test_gpu_ff_limits.py)."""
import numpy as np

from daisyriot_b200 import scenes
from daisyriot_b200.scenes import Scene


def _rot(axis, ang):
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def _one_material():
    return [{"name": "w", "Kd": np.ones(3, np.float32), "Ke": np.zeros(3, np.float32), "Ks": np.zeros(3, np.float32)}]


def irregular_walls(seed):
    """Two facing walls and a tilted occluder triangulated irregularly (jittered grids, random diagonals, slivers, triangles
    20x larger than their neighbours), vertex heights perturbed by rounding-sized noise on part of each wall, arbitrary wall
    orientation."""
    rng = np.random.RandomState(seed)
    R = _rot(rng.normal(size=3), rng.uniform(0, 3))
    V, T, VN = [], [], []

    def wall(origin, eu, ev, n, nu, nv, flip):
        base = len(V)
        us = np.sort(np.concatenate([[0, 1], rng.uniform(0, 1, nu - 1)]))
        vs = np.sort(np.concatenate([[0, 1], rng.uniform(0, 1, nv - 1)]))
        if seed == 2:
            us[1] = us[0] + 1e-3  # a column of slivers
        for j in range(nv + 1):
            for i in range(nu + 1):
                p = origin + us[i] * eu + vs[j] * ev
                if rng.uniform() < 0.3:
                    p = p + n * rng.uniform(-2e-7, 2e-7) * 6.0
                V.append(p)
        ni = len(VN)
        VN.append(n)
        for j in range(nv):
            for i in range(nu):
                a, b, c, d = base + j * (nu + 1) + i, base + j * (nu + 1) + i + 1, base + (j + 1) * (nu + 1) + i, base + (j + 1) * (nu + 1) + i + 1
                tris = [(a, b, d), (a, d, c)] if rng.uniform() < 0.5 else [(a, b, c), (b, d, c)]
                for t in tris:
                    T.append([*(t[::-1] if flip else t), ni, ni, ni])

    ex, ey, ez = np.eye(3)
    wall(np.zeros(3), 6 * ex, 6 * ez, ey, 9, 8, True)                       # floor, facing +y
    wall(np.array([0, 4.0, 0]), 6 * ex, 6 * ez, -ey, 7, 9, False)           # ceiling, facing -y
    wall(np.array([1.5, 1.7, 1.0]), 2.5 * ex + 0.4 * ey, 3 * ez, np.cross(2.5 * ex + 0.4 * ey, 3 * ez) / np.linalg.norm(np.cross(2.5 * ex + 0.4 * ey, 3 * ez)), 4, 5, False)
    big = len(V)                                                            # one triangle much larger than its neighbours
    V += [np.array([6.0, 0, 0]), np.array([9.0, 0, 0]), np.array([6.0, 0, 6.0])]
    T.append([big, big + 2, big + 1, 0, 0, 0])
    V = (np.asarray(V) @ R.T).astype(np.float32)
    VN = (np.asarray(VN) @ R.T).astype(np.float32)
    T = np.asarray(T, np.int32)
    return Scene(V, VN, T, np.zeros(len(T), np.int32), _one_material(), f"irregular{seed}")


def perforated_plate(seed):
    """Between a floor and a ceiling hangs a tilted plate with holes, a ragged outline, T-junctions (cells cut in four next to
    uncut neighbours) and a second, overlapping sheet in the very same plane; a fin stands ON the floor (its lower edge lies in
    the floor's plane).  Seed 2 rotates everything arbitrarily."""
    rng = np.random.RandomState(100 + seed)
    R = _rot(rng.normal(size=3), rng.uniform(0, 3)) if seed == 2 else np.eye(3)
    V, T, VN = [], [], []

    def sheet(origin, eu, ev, n, nu, nv, flip, keep=None, split=None):
        """nu x nv cells; keep(i, j) False = hole; split(i, j) True = the cell is cut into four sub-cells (T-junctions)."""
        ni = len(VN)
        VN.append(n)

        def vid(s, t):
            V.append(origin + s * eu + t * ev)
            return len(V) - 1

        grid = [[vid(i / nu, j / nv) for i in range(nu + 1)] for j in range(nv + 1)]

        def quad(a, b, c, d):  # a b / c d
            tris = [(a, b, d), (a, d, c)] if rng.uniform() < 0.5 else [(a, b, c), (b, d, c)]
            for t in tris:
                T.append([*(t[::-1] if flip else t), ni, ni, ni])

        for j in range(nv):
            for i in range(nu):
                if keep is not None and not keep(i, j):
                    continue
                a, b, c, d = grid[j][i], grid[j][i + 1], grid[j + 1][i], grid[j + 1][i + 1]
                if split is not None and split(i, j):
                    m = [[a, vid((i + .5) / nu, j / nv), b], [vid(i / nu, (j + .5) / nv), vid((i + .5) / nu, (j + .5) / nv), vid((i + 1) / nu, (j + .5) / nv)],
                         [c, vid((i + .5) / nu, (j + 1) / nv), d]]
                    for jj in range(2):
                        for ii in range(2):
                            quad(m[jj][ii], m[jj][ii + 1], m[jj + 1][ii], m[jj + 1][ii + 1])
                else:
                    quad(a, b, c, d)

    ex, ey, ez = np.eye(3)
    sheet(np.zeros(3), 6 * ex, 6 * ez, ey, 7, 6, True)                       # floor, facing +y
    sheet(np.array([0, 4.0, 0]), 6 * ex, 6 * ez, -ey, 6, 7, False)           # ceiling, facing -y
    holes = rng.uniform(size=(9, 9)) < 0.25
    splits = rng.uniform(size=(9, 9)) < 0.2
    pu, pv = 4.2 * ex + 0.5 * ey, 4.0 * ez + 0.3 * ey
    pn = np.cross(pu, pv) / np.linalg.norm(np.cross(pu, pv))
    sheet(np.array([0.8, 1.8, 0.9]), pu, pv, pn, 9, 9, False, keep=lambda i, j: not holes[j, i] and not (i > 5 and j > 6), split=lambda i, j: splits[j, i])
    # a second sheet in the same plane, overlapping part of the first (its vertices are points of the first sheet's plane)
    sheet(np.array([0.8, 1.8, 0.9]) + 0.31 * pu + 0.27 * pv, 0.45 * pu, 0.4 * pv, pn, 4, 4, False)
    # a fin standing on the floor: its lower edge lies in the floor's plane
    sheet(np.array([1.0, 0.0, 5.2]), 4.0 * ex + 0.3 * ez, 0.9 * ey, np.cross(4.0 * ex + 0.3 * ez, 0.9 * ey) / np.linalg.norm(np.cross(4.0 * ex + 0.3 * ez, 0.9 * ey)), 8, 2, False)
    V = (np.asarray(V) @ R.T).astype(np.float32)
    VN = (np.asarray(VN) @ R.T).astype(np.float32)
    T = np.asarray(T, np.int32)
    return Scene(V, VN, T, np.zeros(len(T), np.int32), _one_material(), f"perforated{seed}")


# ---- far from the origin ------------------------------------------------------------------------------------------------
# Translations and scales of the far-geometry tests.  Every conservative margin of the LBVH and the form-factor kernel is a
# fraction of the scene extent, while float32 coordinates round at ulp(max |coord|): the translations move a room about 5.5
# wide from coordinates of its own size (0) to where that ulp is a fraction of the 1e-4 x extent box padding (16, 64, 4096)
# and beyond it (16384 and up).  The scales keep the ratio and move everything else.
OFFSETS = {
    "o0": (0.0, 0.0, 0.0),
    "o16": (16.0, 16.0, 16.0),
    "o64": (64.0, 64.0, 64.0),
    "o4096": (4096.0, 4096.0, 4096.0),
    "o16384": (16384.0, 0.0, 0.0),
    "o32768": (32768.0, 32768.0, -32768.0),
    "o3e5": (3e5, -3e5, 0.0),
}
SCALES = {"s1e-3": 1e-3, "s1e3": 1e3, "s0.37": 0.37}
# the adversarial wall scenes go to 32768 along an arbitrary direction
FAR_DIRECTION_32768 = 32768.0 * np.array([0.48, -0.6, 0.64])


def moved(sc, offset=(0.0, 0.0, 0.0), scale=1.0, name=None):
    """The scene with every vertex mapped to float32(scale * v + offset) (float64 arithmetic, one rounding)."""
    V = (sc.vertices.astype(np.float64) * scale + np.asarray(offset, np.float64)).astype(np.float32)
    return Scene(V, sc.normals.copy(), sc.tri.copy(), sc.mat_idx.copy(), sc.materials, name or sc.name)


def with_ties(sc):
    """The scene plus triangles that make the (t, id) tie rule decide hits: every seventh triangle again with its winding
    flipped (same vertices), and zero-area triangles on every eleventh triangle's first edge (a repeated vertex)."""
    t = sc.tri
    dup = t[::7][:, [0, 2, 1, 3, 5, 4]]
    flat = t[::11][:, [0, 1, 1, 3, 4, 4]]
    T = np.concatenate([t, dup, flat]).astype(np.int32)
    mat = np.concatenate([sc.mat_idx, sc.mat_idx[::7], sc.mat_idx[::11]]).astype(np.int32)
    return Scene(sc.vertices, sc.normals, T, mat, sc.materials, sc.name + "+ties")


def cornell512_at(key):
    sc = scenes.cornell_box(512)
    if key in OFFSETS:
        return moved(sc, offset=OFFSETS[key], name=f"cornell512@{key}")
    return moved(sc, scale=SCALES[key], name=f"cornell512@{key}")


def closest_hit_rays(sc, seed, n_random=3000, n_axis=4000):
    """Rays for the closest-hit comparisons, all float32:
    * random origins inside the bounding box, random directions;
    * axis-parallel rays through every third vertex, all three axes and both signs, starting outside the box;
    * axis-parallel rays through random vertices, starting at a random point of the vertex's axis line inside the box;
    * rays along triangle edges (from behind the first vertex towards the second);
    * rays starting on a triangle (a point of its surface), in random directions -- its own t = 0 must not count."""
    rng = np.random.RandomState(seed)
    V = sc.vertices
    lo, hi = V.min(0).astype(np.float64), V.max(0).astype(np.float64)
    ext = float((hi - lo).max())
    out = []

    def unit(d):
        d = np.asarray(d, np.float64)
        return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)

    o = rng.uniform(lo, hi, (n_random, 3)).astype(np.float32)
    out.append(np.concatenate([o, unit(rng.normal(size=(n_random, 3)))], 1))
    for a in range(3):
        for s in (1.0, -1.0):
            o = V[::3].astype(np.float64).copy()
            o[:, a] = (lo[a] - 0.5 * ext) if s > 0 else (hi[a] + 0.5 * ext)
            d = np.zeros_like(o)
            d[:, a] = s
            out.append(np.concatenate([o.astype(np.float32), d.astype(np.float32)], 1))
    vi = rng.randint(0, len(V), n_axis)
    ax = rng.randint(0, 3, n_axis)
    sg = rng.choice([-1.0, 1.0], n_axis)
    o = V[vi].astype(np.float64).copy()
    o[np.arange(n_axis), ax] = rng.uniform(lo[ax], hi[ax])
    d = np.zeros((n_axis, 3))
    d[np.arange(n_axis), ax] = sg
    out.append(np.concatenate([o.astype(np.float32), d.astype(np.float32)], 1))
    tri = sc.tri[::2]
    a, b = V[tri[:, 0]].astype(np.float64), V[tri[:, 1]].astype(np.float64)
    out.append(np.concatenate([(a - 0.25 * (b - a)).astype(np.float32), unit(b - a)], 1))
    tri = sc.tri[::3]
    u = rng.uniform(0, 1, len(tri))
    v = rng.uniform(0, 1, len(tri)) * (1 - u)
    a, b, c = (V[tri[:, k]].astype(np.float64) for k in range(3))
    p = a + u[:, None] * (b - a) + v[:, None] * (c - a)
    out.append(np.concatenate([p.astype(np.float32), unit(rng.normal(size=(len(tri), 3)))], 1))
    return np.ascontiguousarray(np.concatenate(out), np.float32)


# ---- capacity limits of the form-factor kernel ----------------------------------------------------------------------------
# formfactor.cu has three fixed capacities, and a scene past any of them takes another code path:
# * SHAFT_CAP = 256 candidates per pair: a longer shaft list flags the pair heavy, and phase 2b traces its rays one LBVH walk each;
# * DAISY_MAX_FACES = 64 face grids: further planes of 32 or more triangles stay ordinary candidates, with plane ids above nfaces;
# * NBR_CAP = 32 ints of neighbour list (31 neighbours): a patch with more coplanar neighbours loses coplanar skipping.
# The builders below put small scenes on both sides of each limit.  Their premises are checked in test_ff_limits_scenes.py.

class _Builder:
    """Triangles with one normal each (the normal array holds one entry per triangle)."""

    def __init__(self):
        self.V, self.VN, self.T = [], [], []

    def tri(self, a, b, c, n):
        base, ni = len(self.V), len(self.VN)
        self.V += [np.asarray(a, np.float64), np.asarray(b, np.float64), np.asarray(c, np.float64)]
        self.VN.append(np.asarray(n, np.float64) / np.linalg.norm(n))
        self.T.append([base, base + 1, base + 2, ni, ni, ni])

    def grid(self, origin, eu, ev, n, nu, nv):
        """nu x nv quads of two triangles each; shared edges are bit-identical (one vertex array per grid)."""
        base, ni = len(self.V), len(self.VN)
        origin, eu, ev = (np.asarray(x, np.float64) for x in (origin, eu, ev))
        for j in range(nv + 1):
            for i in range(nu + 1):
                self.V.append(origin + (i / nu) * eu + (j / nv) * ev)
        self.VN.append(np.asarray(n, np.float64) / np.linalg.norm(n))
        for j in range(nv):
            for i in range(nu):
                a, b = base + j * (nu + 1) + i, base + j * (nu + 1) + i + 1
                c, d = a + nu + 1, b + nu + 1
                self.T += [[a, b, d, ni, ni, ni], [a, d, c, ni, ni, ni]]

    def scene(self, name):
        V = np.asarray(self.V, np.float64).astype(np.float32)
        VN = np.asarray(self.VN, np.float64).astype(np.float32)
        T = np.asarray(self.T, np.int32).reshape(-1, 6)
        return Scene(V, VN, T, np.zeros(len(T), np.int32), _one_material(), name)


def _random_triangles(b, rng, centres, radius, tilt=(0.3, 2.8)):
    """One equilateral triangle of circumradius `radius` around each centre, each in its own random orientation: the xy-plane
    turned about a random axis by an angle drawn from `tilt` (radians)."""
    ang = np.array([0.0, 2 * np.pi / 3, 4 * np.pi / 3])
    flat = radius * np.stack([np.cos(ang), np.sin(ang), np.zeros(3)], 1)
    for c in centres:
        R = _rot(rng.normal(size=3), rng.uniform(*tilt))
        p = flat @ R.T + c
        b.tri(p[0], p[1], p[2], np.cross(p[1] - p[0], p[2] - p[0]))


def lifted(sc, k, dz=1.5):
    """The vertex array of sc with triangle k's three vertices raised by dz along z (the builders give every occluder
    vertices of its own)."""
    V = sc.vertices.copy()
    V[sc.tri[k, :3], 2] += np.float32(dz)
    return V


def edge_pattern(uv):
    """The pattern with its first eight samples moved onto triangle edges and vertices (u = 0, v = 0, u + v = 1)."""
    uv = np.array(uv, np.float32)
    uv[:8] = np.array([[0, 0], [1, 0], [0, 1], [0.5, 0], [0, 0.5], [0.5, 0.5], [0.25, 0.75], [1e-4, 0.3]], np.float32)
    return uv


def random_pattern(S, seed):
    rng = np.random.RandomState(seed)
    u = rng.uniform(0, 1, S)
    v = rng.uniform(0, 1, S) * (1 - u)
    return np.stack([u, v], 1).astype(np.float32)


def shaft_cap_scene(n_occ, seed=0):
    """Two single-triangle plates one unit apart, facing each other -- A (triangle 0) at z = 0 with normal +z, B (triangle 1) the
    same triangle at z = 1 with normal -z -- and n_occ small triangles between them (triangles 2 ...), each in its own random
    orientation (tilted 0.1-0.8 rad): centres with x, y in [1, 8], x + y < 8.5, z in [0.4, 0.6], vertices 0.35 from the centre.  Every occluder's
    box lies inside the hull of A and B by at least 0.05, far above the 1e-3 box padding, so the pair (A, B) has exactly n_occ
    shaft candidates; any other pair has fewer."""
    rng = np.random.RandomState(1000 + seed)
    b = _Builder()
    b.tri((0, 0, 0), (10, 0, 0), (0, 10, 0), (0, 0, 1))
    b.tri((0, 0, 1), (10, 0, 1), (0, 10, 1), (0, 0, -1))
    centres = []
    while len(centres) < n_occ:
        x, y = rng.uniform(1.0, 8.0, 2)
        if x + y < 8.5:
            centres.append((x, y, rng.uniform(0.4, 0.6)))
    _random_triangles(b, rng, centres, 0.35, tilt=(0.1, 0.8))  # nearly face-on: they hide part of A from B
    return b.scene(f"shaft_cap{n_occ}")


def occluded_walls(nu, nv, seed=0, n_occ=360):
    """Two facing 10 x 10 walls, z = 0 (normal +z) and z = 1 (normal -z), each cut into nu x nv quads, and n_occ small occluders
    (circumradius 0.12) clustered in x, y in [4.3, 5.7], z in [0.3, 0.7].  Hundreds of wall-to-wall pairs see more than 256
    occluders in their shafts; the walls' own triangles are coplanar neighbours of every wall patch."""
    rng = np.random.RandomState(2000 + seed)
    b = _Builder()
    b.grid((0, 0, 0), (10, 0, 0), (0, 10, 0), (0, 0, 1), nu, nv)
    b.grid((0, 0, 1), (0, 10, 0), (10, 0, 0), (0, 0, -1), nv, nu)
    centres = np.stack([rng.uniform(4.3, 5.7, n_occ), rng.uniform(4.3, 5.7, n_occ), rng.uniform(0.3, 0.7, n_occ)], 1)
    _random_triangles(b, rng, centres, 0.12)
    return b.scene(f"occluded_walls{nu}x{nv}")


MANY_PLANES_KINDS = ("floor", "ceiling", "vertical")


def many_planes(nplates, seed=0):
    """nplates plates of 4 x 4 quads (32 triangles each), every plate in its own axis-aligned plane, in this order: plate q is
    MANY_PLANES_KINDS[(q + 1) % 3] -- a floor plate at y = 1e-3 q, a ceiling plate at y = 4 - 1e-3 q (both 1 x 1, on a 5 x 5
    layout of x, z cells), or a vertical plate in the plane x = 0.3 + 0.2 j (y in [1.5, 2.5], z over one cell) that blocks
    rays between floor and ceiling.  Then 40 small tilted occluders between them.  All plates have the same size, so the
    face grids go to the first 64 plates in order (face f = plate f), and vertical plates sit among faces 32-63 and among the
    planes left without a grid."""
    rng = np.random.RandomState(3000 + seed)
    b = _Builder()
    seen = {k: 0 for k in MANY_PLANES_KINDS}
    for q in range(nplates):
        kind = MANY_PLANES_KINDS[(q + 1) % 3]
        j = seen[kind]
        seen[kind] += 1
        cx, cz = float(j % 5), float((j // 5) % 5)
        if kind == "floor":
            b.grid((cx, 1e-3 * q, cz), (0, 0, 1), (1, 0, 0), (0, 1, 0), 4, 4)
        elif kind == "ceiling":
            b.grid((cx, 4 - 1e-3 * q, cz), (1, 0, 0), (0, 0, 1), (0, -1, 0), 4, 4)
        else:
            x = 0.3 + 0.2 * j
            b.grid((x, 1.5, float((3 * j) % 5)), (0, 1, 0), (0, 0, 1), (1 if j % 2 else -1, 0, 0), 4, 4)
    centres = np.stack([rng.uniform(0.2, 4.8, 40), rng.uniform(0.8, 3.2, 40), rng.uniform(0.2, 4.8, 40)], 1)
    _random_triangles(b, rng, centres, 0.3)
    return b.scene(f"many_planes{nplates}")


def fan_floor(n):
    """A plate (triangles 0 and 1: a 2 x 2 square at y = 1.5, normal -y), a tilted occluder (triangle 2) and a floor at y = 0 made
    of ONE fan of n triangles around a centre vertex (triangles 3 ...): a closed disk of radius 2, apex angle 360 / n degrees
    (11.25 for n = 32, 9 for n = 40: all pass the sliver rule 8 h >= longest edge).  Every fan triangle contains the centre, so
    each has n - 1 coplanar neighbours: n = 32 fills the neighbour list exactly, n = 33 is one past it."""
    b = _Builder()
    b.tri((-1, 1.5, -1), (1, 1.5, -1), (1, 1.5, 1), (0, -1, 0))
    b.tri((-1, 1.5, -1), (1, 1.5, 1), (-1, 1.5, 1), (0, -1, 0))
    p = np.array([[-0.4, 0.7, -0.3], [0.6, 0.8, 0.1], [-0.1, 0.9, 0.7]])
    b.tri(p[0], p[1], p[2], np.cross(p[1] - p[0], p[2] - p[0]))
    base = len(b.V)
    b.V.append(np.zeros(3))
    for i in range(n):
        a = 2 * np.pi * i / n
        b.V.append(np.array([2 * np.cos(a), 0.0, 2 * np.sin(a)]))
    b.VN.append(np.array([0.0, 1.0, 0.0]))
    ni = len(b.VN) - 1
    for i in range(n):
        b.T.append([base, base + 1 + (i + 1) % n, base + 1 + i, ni, ni, ni])
    return b.scene(f"fan{n}")


def padded_boxes(sc, tris, pad):
    """float64 boxes (len(tris), 6) = (lo xyz, hi xyz) of the listed triangles, grown by pad on every side."""
    P = sc.vertices[sc.tri[np.asarray(tris), :3]].astype(np.float64)  # (M, 3 vertices, 3)
    return np.concatenate([P.min(1) - pad, P.max(1) + pad], 1)


def shaft_meets(sc, pairs, boxes):
    """float64 statement of formfactor.cu's shaft_box: (len(pairs), len(boxes)) bool, True where the box may meet the hull of
    the pair's two triangles (six separating axes: x, y, z and D x {x, y, z}, D = centroid difference x 3, the kernel's slack)."""
    pairs = np.asarray(pairs).reshape(-1, 2)
    P = sc.vertices[sc.tri[pairs.reshape(-1), :3]].astype(np.float64).reshape(len(pairs), 6, 3)
    lo, hi = P.min(1)[:, None, :], P.max(1)[:, None, :]
    D = (P[:, 3:].sum(1) - P[:, :3].sum(1))[:, None, :]
    blo, bhi = boxes[None, :, :3], boxes[None, :, 3:]
    ok = ~((blo > hi) | (bhi < lo)).any(2)
    c, h = 0.5 * (blo + bhi), 0.5 * (bhi - blo)
    aD = np.abs(D)
    for a, b in ((1, 2), (2, 0), (0, 1)):  # axis D x e: projection p = c_a D_b - c_b D_a, as q0 / q1 / q2 of make_shaft
        q = P[:, :, a] * D[:, :, b] - P[:, :, b] * D[:, :, a]
        p = c[..., a] * D[..., b] - c[..., b] * D[..., a]
        r = h[..., a] * aD[..., b] + h[..., b] * aD[..., a]
        r = r + 1e-5 * (np.abs(p) + r)
        ok &= ~((p - r > q.max(1)[:, None]) | (p + r < q.min(1)[:, None]))
    return ok


def facing_pairs(orc):
    """(lo, hi) pairs the kernel traces: the unoccluded factor from the lower to the higher triangle id is > 0."""
    U = orc.unoccluded_rows(0, orc.N)
    lo, hi = np.nonzero(np.triu(U > 0, 1))
    return np.stack([lo, hi], 1)
