"""Scene inputs for the form-factor / radiosity hot path (host side, numpy only).

* :func:`load_obj` -- the patch layout ``MeshS::loadFromFile`` produces
  (reference ``visual studio/MeshS.cpp:22-128``): unique vertices / normals, one patch per ``f`` line
  with six indices ``{v0,v1,v2,n0,n1,n2}`` (``visual studio/Vertex.h:11-14``) and a material id per patch.
* :func:`cornell_box` -- the synthetic subdivided Cornell boxes named in ``BASELINE.json`` configs 3-5.
* :func:`msvc_sample_pattern` -- the 50-sample ``rands`` pattern of
  ``visual studio/OptixPrimeFunctionality.cpp:55-63`` with the MSVC CRT ``rand()`` restated and a fixed seed
  (the reference seeds with wall-clock time, so the pattern has to be an explicit input).
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field

import numpy as np

RAYS_PER_PATCH = 50  # visual studio/Defines.h:25


@dataclass
class Scene:
    """Plain arrays in the reference's ``MeshS`` layout (``visual studio/MeshS.h:14-20``)."""

    vertices: np.ndarray  # (nv,3) float32
    normals: np.ndarray  # (nn,3) float32
    tri: np.ndarray  # (N,6) int32  v0 v1 v2 n0 n1 n2
    mat_idx: np.ndarray  # (N,) int32
    materials: list = field(default_factory=list)  # dicts: name, Kd, Ke, Ks (float32[3])
    name: str = ""

    @property
    def numtriangles(self) -> int:
        return int(self.tri.shape[0])


def _parse_mtl(path):
    mats = []
    cur = None
    with open(path) as f:
        for line in f:
            p = line.split()
            if not p or p[0].startswith("#"):
                continue
            if p[0] == "newmtl":
                cur = {"name": p[1], "Kd": np.zeros(3, np.float32), "Ke": np.zeros(3, np.float32),
                       "Ks": np.zeros(3, np.float32)}
                mats.append(cur)
            elif cur is not None and p[0] in ("Kd", "Ke", "Ks"):
                cur[p[0]] = np.array([float(x) for x in p[1:4]], np.float32)
    return mats


def load_obj(obj_path: str, mtl_dir: str | None = None) -> Scene:
    """OBJ/MTL -> patch arrays, one patch per face (faces must be triangles, as the reference requires:
    it calls tinyobj with ``triangulate=false``, ``visual studio/MeshS.cpp:29``)."""
    V, VN, T, M = [], [], [], []
    mats, names, cur = [], {}, -1
    base = mtl_dir if mtl_dir is not None else os.path.dirname(obj_path)
    with open(obj_path) as f:
        for line in f:
            p = line.split()
            if not p:
                continue
            if p[0] == "v":
                V.append([float(x) for x in p[1:4]])
            elif p[0] == "vn":
                VN.append([float(x) for x in p[1:4]])
            elif p[0] == "mtllib":
                mats = _parse_mtl(os.path.join(base, p[1]))
                names = {m["name"]: i for i, m in enumerate(mats)}
            elif p[0] == "usemtl":
                cur = names.get(p[1], -1)
            elif p[0] == "f":
                if len(p) != 4:
                    raise ValueError("only triangle faces are supported (reference loads with triangulate=false)")
                vi, ni = [], []
                for q in p[1:]:
                    s = q.split("/")
                    vi.append(int(s[0]) - 1)
                    ni.append(int(s[2]) - 1 if len(s) > 2 and s[2] else -1)
                T.append(vi + ni)
                M.append(cur)
    return Scene(np.asarray(V, np.float32).reshape(-1, 3), np.asarray(VN, np.float32).reshape(-1, 3),
                 np.asarray(T, np.int32).reshape(-1, 6), np.asarray(M, np.int32), mats,
                 os.path.basename(obj_path))


def save_scene_npz(scene: Scene, path: str) -> None:
    np.savez_compressed(
        path, vertices=scene.vertices, normals=scene.normals, tri=scene.tri, mat_idx=scene.mat_idx,
        mat_names=np.array([m["name"] for m in scene.materials]),
        Kd=np.array([m["Kd"] for m in scene.materials], np.float32).reshape(-1, 3),
        Ke=np.array([m["Ke"] for m in scene.materials], np.float32).reshape(-1, 3),
        Ks=np.array([m["Ks"] for m in scene.materials], np.float32).reshape(-1, 3), name=scene.name)


def load_scene_npz(path: str) -> Scene:
    z = np.load(path, allow_pickle=False)
    mats = [{"name": str(n), "Kd": kd, "Ke": ke, "Ks": ks}
            for n, kd, ke, ks in zip(z["mat_names"], z["Kd"], z["Ke"], z["Ks"])]
    return Scene(z["vertices"], z["normals"], z["tri"], z["mat_idx"], mats, str(z["name"]))


# ---------------------------------------------------------------------------------------------
def msvc_sample_pattern(seed: int = 1, S: int = RAYS_PER_PATCH) -> np.ndarray:
    """``rands`` of ``visual studio/OptixPrimeFunctionality.cpp:55-63`` with MSVC's ``rand()``
    (``x = x*214013 + 2531011; return (x >> 16) & 0x7fff``, ``RAND_MAX = 32767``) and ``srand(seed)``::

        uv.u = ((float)(rand() % RAND_MAX)) / RAND_MAX;
        uv.v = ((float)(rand() % RAND_MAX)) / RAND_MAX;
        uv.v = uv.v * (1 - uv.u);
    """
    state = seed & 0xFFFFFFFF

    def rand():
        nonlocal state
        state = (state * 214013 + 2531011) & 0xFFFFFFFF
        return (state >> 16) & 0x7FFF

    RAND_MAX = 32767
    out = np.zeros((S, 2), np.float32)
    for i in range(S):
        u = np.float32(rand() % RAND_MAX) / np.float32(RAND_MAX)
        v = np.float32(rand() % RAND_MAX) / np.float32(RAND_MAX)
        v = np.float32(v * np.float32(np.float32(1) - u))
        out[i] = (u, v)
    return out


# ---------------------------------------------------------------------------------------------
def _quad(p0, pu, pv, nu, nv, normal, V, VN, T, M, mat):
    """Append a parallelogram p0 + s*pu + t*pv subdivided nu x nv, two triangles per cell."""
    p0, pu, pv = (np.asarray(x, np.float64) for x in (p0, pu, pv))
    base = len(V)
    for j in range(nv + 1):
        for i in range(nu + 1):
            V.append((p0 + pu * (i / nu) + pv * (j / nv)).astype(np.float32))
    ni = len(VN)
    n = np.asarray(normal, np.float64)
    VN.append((n / np.linalg.norm(n)).astype(np.float32))
    # winding chosen so that cross(b-a, c-a) points along `normal`
    flip = np.dot(np.cross(pu, pv), n) < 0
    for j in range(nv):
        for i in range(nu):
            a = base + j * (nu + 1) + i
            b = a + 1
            c = a + (nu + 1)
            d = c + 1
            t1, t2 = (a, b, d), (a, d, c)
            if flip:
                t1, t2 = (a, d, b), (a, c, d)
            T.append([*t1, ni, ni, ni])
            T.append([*t2, ni, ni, ni])
            M.extend([mat, mat])


CORNELL_MATERIALS = [
    # same four classes as example_scenes/cornellbox_blacklight.mtl (lamp / two fluorescent paints / white)
    {"name": "Blacklight", "Kd": (0, 0, 0), "Ke": (1, 1, 1), "Ks": (0, 0, 0)},
    {"name": "Blacklight_Pink", "Kd": (0, 0, 1), "Ke": (0, 0, 0), "Ks": (0, 0.787117, 1)},
    {"name": "Blacklight_blue", "Kd": (1, 0, 0.099734), "Ke": (0, 0, 0), "Ks": (1, 0.110627, 0.991776)},
    {"name": "white", "Kd": (1, 1, 1), "Ke": (0, 0, 0), "Ks": (0, 0, 0)},
]


def cornell_subdivision(n_patches: int):
    """(nu, nv) per quad such that 16 quads * 2 * nu * nv == n_patches."""
    cells = n_patches // 32
    if cells * 32 != n_patches or cells < 1:
        raise ValueError("synthetic Cornell box needs n_patches = 32 * nu * nv")
    nu = 1
    while nu * nu * 2 <= cells and cells % (nu * 2) == 0:
        nu *= 2
    nv = cells // nu
    return max(nu, nv), min(nu, nv)


def cornell_box(n_patches: int, n_fluorescent: int = 2, seed: int = 0x5EED) -> Scene:
    """Synthetic Cornell box: 5 walls + short block (5 faces) + tall block (5 faces) + lamp quad = 16 quads,
    each uniformly subdivided; all triangles, one ``vn`` per face (like the fixture scenes).
    ``n_patches`` must be ``32*nu*nv`` (32768 -> 32x32, 65536 -> 64x32, 131072 -> 64x64 cells per quad).
    ``n_fluorescent`` > 2 adds further fluorescent paints on the block faces (config 5 asks for >= 8)."""
    nu, nv = cornell_subdivision(n_patches)
    V, VN, T, M = [], [], [], []
    L = 5.5
    mats = [dict(m) for m in CORNELL_MATERIALS]
    rng = np.random.RandomState(seed)
    extra = []
    for i in range(max(0, n_fluorescent - 2)):
        kd = rng.uniform(0.1, 0.9, 3)
        ks = rng.uniform(0.2, 1.0, 3)
        mats.append({"name": f"Fluor_{i}", "Kd": tuple(kd), "Ke": (0, 0, 0), "Ks": tuple(ks)})
        extra.append(len(mats) - 1)
    LAMP, PINK, BLUE, WHITE = 0, 1, 2, 3
    # room (normals point inward)
    _quad((0, 0, 0), (L, 0, 0), (0, 0, L), nu, nv, (0, 1, 0), V, VN, T, M, WHITE)  # floor
    _quad((0, L, 0), (L, 0, 0), (0, 0, L), nu, nv, (0, -1, 0), V, VN, T, M, WHITE)  # ceiling
    _quad((0, 0, 0), (L, 0, 0), (0, L, 0), nu, nv, (0, 0, 1), V, VN, T, M, WHITE)  # back wall
    _quad((0, 0, 0), (0, 0, L), (0, L, 0), nu, nv, (1, 0, 0), V, VN, T, M, PINK)  # left wall
    _quad((L, 0, 0), (0, 0, L), (0, L, 0), nu, nv, (-1, 0, 0), V, VN, T, M, BLUE)  # right wall

    def block(corners, h, face_mats):
        c = [np.array([x, 0.0, z]) for x, z in corners]
        up = np.array([0.0, h, 0.0])
        centre = sum(c) / 4.0
        _quad(c[0] + up, c[1] - c[0], c[3] - c[0], nu, nv, (0, 1, 0), V, VN, T, M, face_mats[0])  # top
        for k in range(4):
            a, b = c[k], c[(k + 1) % 4]
            e = b - a
            n = np.array([e[2], 0.0, -e[0]])
            if np.dot(n, (a + b) / 2 - centre) < 0:
                n = -n
            _quad(a, e, up, nu, nv, n, V, VN, T, M, face_mats[1 + k])

    fm_short = [WHITE] * 5
    fm_tall = [WHITE] * 5
    slots = [(fm_short, i) for i in range(5)] + [(fm_tall, i) for i in range(5)]
    for s, mi in zip(slots, extra):
        s[0][s[1]] = mi
    block([(1.30, 0.65), (0.82, 2.25), (2.40, 2.72), (2.90, 1.14)], 1.65, fm_short)
    block([(4.23, 2.47), (2.65, 2.96), (3.14, 4.56), (4.72, 4.06)], 3.30, fm_tall)
    # lamp just under the ceiling, facing down
    _quad((2.13, L - 0.012, 2.27), (1.30, 0, 0), (0, 0, 1.05), nu, nv, (0, -1, 0), V, VN, T, M, LAMP)
    for m in mats:
        for k in ("Kd", "Ke", "Ks"):
            m[k] = np.asarray(m[k], np.float32)
    sc = Scene(np.asarray(V, np.float32), np.asarray(VN, np.float32), np.asarray(T, np.int32),
               np.asarray(M, np.int32), mats, f"cornell_{n_patches}")
    assert sc.numtriangles == n_patches, (sc.numtriangles, n_patches)
    return sc


CORNELL_LAMP, CORNELL_SHORT_BLOCK, CORNELL_TALL_BLOCK = [15], [5, 6, 7, 8, 9], [10, 11, 12, 13, 14]  # quads of cornell_box


def cornell_moved(scene: Scene, quads, offset=(0.0, 0.0, 0.0), angle_y: float = 0.0):
    """(vertices, normals) of a :func:`cornell_box` scene with the given quads rotated by ``angle_y`` radians about the
    vertical axis through their centre, then translated by ``offset``.  Quad q holds triangles [q*2*nu*nv, (q+1)*2*nu*nv) and
    its own vertices and normal, so nothing else moves."""
    per = scene.numtriangles // 16
    tri = np.concatenate([scene.tri[q * per:(q + 1) * per] for q in quads])
    vi, ni = np.unique(tri[:, :3]), np.unique(tri[:, 3:])
    V = np.array(scene.vertices, np.float64)
    VN = np.array(scene.normals, np.float64)
    c, s_ = np.cos(angle_y), np.sin(angle_y)
    R = np.array([[c, 0, s_], [0, 1, 0], [-s_, 0, c]])
    centre = V[vi].mean(axis=0)
    V[vi] = (V[vi] - centre) @ R.T + centre + np.asarray(offset, np.float64)
    VN[ni] = VN[ni] @ R.T
    V32, VN32 = np.array(scene.vertices, np.float32), np.array(scene.normals, np.float32)
    V32[vi] = V[vi].astype(np.float32)
    if angle_y:
        VN32[ni] = VN[ni].astype(np.float32)
    return V32, VN32


def cornell_panel(n_patches: int) -> Scene:
    """A free-standing white panel for :func:`cornell_box` scenes of ``n_patches``: 1.1 x 1.4 at z = 4.6, facing the room (+z),
    subdivided like one quad of the box (``n_patches / 16`` triangles).  The object the mesh-edit tests and tools add."""
    nu, nv = cornell_subdivision(n_patches)
    V, VN, T, M = [], [], [], []
    _quad((0.6, 1.2, 4.6), (1.1, 0, 0), (0, 1.4, 0), nu, nv, (0, 0, 1), V, VN, T, M, 0)
    white = next(m for m in CORNELL_MATERIALS if m["name"] == "white")
    mats = [{k: (np.asarray(v, np.float32) if k != "name" else v) for k, v in white.items()}]
    return Scene(np.asarray(V, np.float32), np.asarray(VN, np.float32), np.asarray(T, np.int32), np.asarray(M, np.int32), mats, "panel")


def edit_scene(scene: Scene, remove=(), add: Scene | None = None, insert_at: int | None = None):
    """``(edited scene, previous)``: ``scene`` without the triangles listed in ``remove``, with the triangles of ``add`` inserted
    before surviving triangle ``insert_at`` (appended when ``None``); the vertex and normal arrays are compacted to the entries
    the triangles use and renumbered (survivors keep their relative order).  Materials follow their triangles; a material of
    ``add`` is matched to one of ``scene`` by name or appended.  ``previous[t]`` = the index in ``scene`` of the triangle new
    triangle t continues, -1 for an added one: the ``previous`` argument of ``replaceMesh``."""
    N = scene.numtriangles
    remove = np.asarray(remove, np.int64).reshape(-1)
    if remove.size and (remove.min() < 0 or remove.max() >= N):
        raise ValueError("edit_scene: a removed triangle is not in the scene")
    keep = np.ones(N, bool)
    keep[remove] = False
    kept = np.nonzero(keep)[0]
    V = [np.asarray(scene.vertices, np.float32).reshape(-1, 3)]
    VN = [np.asarray(scene.normals, np.float32).reshape(-1, 3)]
    tri, mat, prev = scene.tri[kept].astype(np.int64), scene.mat_idx[kept].astype(np.int64), kept.astype(np.int64)
    mats = list(scene.materials)
    if add is not None:
        names = {m["name"]: i for i, m in enumerate(mats)}
        mat_map = []
        for m in add.materials:
            if m["name"] not in names:
                names[m["name"]] = len(mats)
                mats.append(m)
            mat_map.append(names[m["name"]])
        add_tri = add.tri.astype(np.int64) + np.array([V[0].shape[0]] * 3 + [VN[0].shape[0]] * 3, np.int64)
        add_mat = np.asarray(mat_map, np.int64)[add.mat_idx] if len(mat_map) else np.asarray(add.mat_idx, np.int64)
        at = len(kept) if insert_at is None else int(insert_at)
        if not 0 <= at <= len(kept):
            raise ValueError("edit_scene: insert_at is not a position in the surviving triangles")
        tri = np.concatenate([tri[:at], add_tri, tri[at:]])
        mat = np.concatenate([mat[:at], add_mat, mat[at:]])
        prev = np.concatenate([prev[:at], np.full(add.numtriangles, -1, np.int64), prev[at:]])
        V.append(np.asarray(add.vertices, np.float32).reshape(-1, 3))
        VN.append(np.asarray(add.normals, np.float32).reshape(-1, 3))
    V, VN = np.concatenate(V), np.concatenate(VN)
    used_v, used_n = np.unique(tri[:, :3]), np.unique(tri[:, 3:])
    vmap, nmap = np.full(V.shape[0], -1, np.int64), np.full(VN.shape[0], -1, np.int64)
    vmap[used_v], nmap[used_n] = np.arange(used_v.size), np.arange(used_n.size)
    tri = np.concatenate([vmap[tri[:, :3]], nmap[tri[:, 3:]]], 1)
    out = Scene(np.ascontiguousarray(V[used_v]), np.ascontiguousarray(VN[used_n]), tri.astype(np.int32).reshape(-1, 6), mat.astype(np.int32),
                mats, scene.name)
    return out, prev.astype(np.int32)


def write_obj(scene: Scene, directory: str, stem: str | None = None):
    """Write ``scene`` as OBJ + MTL (the inverse of :func:`load_obj`; float32 values survive the round trip).
    Lets the reference's own loader (``MeshS::loadFromFile``) read the synthetic scenes."""
    stem = stem or (scene.name or "scene").replace(".obj", "")
    obj, mtl = os.path.join(directory, stem + ".obj"), os.path.join(directory, stem + ".mtl")
    with open(mtl, "w") as f:
        for m in scene.materials:
            f.write(f"newmtl {m['name']}\n")
            for key in ("Kd", "Ks", "Ke"):
                f.write(f"{key} {float(m[key][0]):.9g} {float(m[key][1]):.9g} {float(m[key][2]):.9g}\n")
            f.write("\n")
    with open(obj, "w") as f:
        f.write(f"mtllib {stem}.mtl\no {stem}\n")
        for v in scene.vertices:
            f.write(f"v {float(v[0]):.9g} {float(v[1]):.9g} {float(v[2]):.9g}\n")
        for v in scene.normals:
            f.write(f"vn {float(v[0]):.9g} {float(v[1]):.9g} {float(v[2]):.9g}\n")
        cur = None
        for t, mi in zip(scene.tri, scene.mat_idx):
            if mi != cur:
                f.write(f"usemtl {scene.materials[mi]['name']}\n")
                cur = mi
            f.write(f"f {t[0]+1}//{t[3]+1} {t[1]+1}//{t[4]+1} {t[2]+1}//{t[5]+1}\n")
    return obj, mtl
