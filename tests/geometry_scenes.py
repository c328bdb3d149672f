"""Scene builders shared by the geometry tests: the adversarial walls of test_gpu_parity.py, and translated / scaled copies of
any scene for the far-from-origin tests (test_far_geometry_oracle.py, test_gpu_far_geometry.py)."""
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
