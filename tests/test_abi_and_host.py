"""CPU suite: the C-ABI library loads and exports exactly what include/daisy_b200.h declares (no compute calls
without a GPU), plus the host-side logic around it."""
import os
import re
import struct

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from daisyriot_b200 import _lib, api, dist, materials, rgb2spec, scenes


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "daisy_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return set(re.findall(r"\b(daisy_[a-z0-9_]+)\s*\(", txt))


def test_library_exports_every_declared_symbol():
    import ctypes
    assert os.path.exists(_lib.SO_PATH), "build the CUDA library first (python -c 'import __graft_entry__ as g; g.build()')"
    L = ctypes.CDLL(_lib.SO_PATH)
    declared = _header_symbols()
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(L, name), name
    assert _lib.lib().daisy_version() >= 100


def test_library_is_sm100a_cuda_with_tma():
    # the product is the CUDA library: its SASS must be sm_100a and contain the TMA bulk copy of the gather kernel
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    out = subprocess.run(["cuobjdump", "-sass", _lib.SO_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out and "k_gather_partial" in out and "k_ff_tiles" in out


def test_errors_without_a_gpu_are_reported_not_faked():
    import ctypes as C
    L = _lib.lib()
    if L.daisy_device_count() > 0:
        pytest.skip("a GPU is present")
    ctx = C.c_void_p()
    v = np.zeros((3, 3), np.float32); n = np.zeros((1, 3), np.float32); t = np.array([[0, 1, 2, 0, 0, 0]], np.int32)
    rc = L.daisy_ctx_create(_lib.fptr(v), 3, _lib.fptr(n), 1, _lib.iptr(t), 1, 0, C.byref(ctx))
    assert rc != 0 and not ctx.value and L.daisy_last_error()
    with pytest.raises(_lib.DaisyError):
        api.OptixPrimeFunctionality(api.MeshS.from_scene(scenes.cornell_box(32)))  # no silent CPU fallback
    bad = np.array([[0, 1, 7, 0, 0, 0]], np.int32)
    assert L.daisy_ctx_create(_lib.fptr(v), 3, _lib.fptr(n), 1, _lib.iptr(bad), 1, 0, C.byref(ctx)) == -1


def test_msvc_sample_pattern():
    uv = scenes.msvc_sample_pattern(1)
    assert uv.shape == (50, 2) and uv.dtype == np.float32
    # MSVC rand() with srand(1) starts 41, 18467, 6334, ...
    assert uv[0, 0] == np.float32(41) / np.float32(32767)
    assert uv[0, 1] == np.float32(np.float32(18467) / np.float32(32767)) * np.float32(np.float32(1) - uv[0, 0])
    assert (uv >= 0).all() and (uv.sum(1) < 1).all()
    assert not np.array_equal(uv, scenes.msvc_sample_pattern(2))


def test_cornell_generator_and_obj_roundtrip(tmp_path):
    for n in (32, 512, 2048):
        sc = scenes.cornell_box(n)
        assert sc.numtriangles == n and sc.tri.max() < len(sc.vertices) and sc.tri[:, 3:].max() < len(sc.normals)
        a, b, c = (sc.vertices[sc.tri[:, k]] for k in range(3))
        geo = np.cross(b - a, c - a)
        nrm = sc.normals[sc.tri[:, 3]]
        assert ((geo * nrm).sum(1) > 0).all()  # winding agrees with the stored normals
        assert (np.linalg.norm(geo, axis=1) > 0).all()
    with pytest.raises(ValueError):
        scenes.cornell_box(1000)
    sc = scenes.cornell_box(512, n_fluorescent=5)
    obj, _ = scenes.write_obj(sc, str(tmp_path))
    s2 = scenes.load_obj(obj, str(tmp_path))
    assert np.array_equal(sc.vertices, s2.vertices) and np.array_equal(sc.tri, s2.tri) and np.array_equal(sc.mat_idx, s2.mat_idx)
    scenes.save_scene_npz(sc, str(tmp_path / "s.npz"))
    s3 = scenes.load_scene_npz(str(tmp_path / "s.npz"))
    assert np.array_equal(sc.tri, s3.tri) and [m["name"] for m in s3.materials] == [m["name"] for m in sc.materials]


def test_fixture_scenes_have_the_surveyed_shape(fixture_scenes):
    cb, balls = fixture_scenes["cornellbox_blacklight"], fixture_scenes["colorballs"]
    assert (cb.numtriangles, len(cb.vertices), len(cb.normals)) == (7712, 4360, 304)
    assert (balls.numtriangles, len(balls.vertices), len(balls.normals)) == (6400, 3373, 2551)
    assert list(np.bincount(cb.mat_idx)) == [32, 2560, 2560, 2560]


def test_material_classification_and_matrices(coeff_model, fixture_scenes):
    model, _ = coeff_model
    wl = np.arange(200, 601, 50).astype(np.float32)
    mats = materials.make_materials(fixture_scenes["cornellbox_blacklight"].materials, wl, model)
    assert [m.kind for m in mats] == ["uvlight", "fluorescent", "fluorescent", "diffuse"]
    lamp, pink, _, white = mats
    assert not lamp.M.any() and lamp.spectral_emission[3] == 1.0 and lamp.spectral_emission[0] < 1e-30  # bell curve at 350 nm
    assert np.array_equal(np.diag(white.M), white.spectral_values) and not (white.M - np.diag(np.diag(white.M))).any()
    uvcol = 3  # 350 nm is the only band inside (300, 400)
    off = pink.M.copy(); off[:, uvcol] = 0
    assert np.array_equal(off, np.eye(9, dtype=np.float32) * (np.arange(9) != uvcol))
    assert np.isnan(white.spectral_emission).all()  # Ke = 0 -> 0*inf in rgb2spec_fetch; filtered by `> 0` downstream
    E, M = materials.spectral_inputs(mats, fixture_scenes["cornellbox_blacklight"].mat_idx, 7.0)
    assert E.shape == (9, 7712) and np.isfinite(E).all() and E[3, 0] == 0 and E[3].max() == 7.0
    assert M.shape == (4, 9, 9) and M[1, uvcol, 0] == pink.M[0, uvcol]  # column-major per material
    balls = materials.make_materials(fixture_scenes["colorballs"].materials, wl, model)
    assert [m.kind for m in balls] == ["diffuse"] * 4 + ["fluorescent"]  # "white" has Ks = 0.5 => fluorescent
    Ergb, Mrgb = materials.rgb_inputs(balls, fixture_scenes["colorballs"].mat_idx, 2.0)
    assert Ergb.shape == (3, 6400) and Ergb.max() == np.float32(1.6) * np.float32(2.0) and Mrgb[1, 0, 0] == np.float32(0.8)


def test_rgb2spec_table_roundtrip(tmp_path):
    p = str(tmp_path / "t.coeff")
    rgb2spec.write_surrogate_table(p, 8)
    m = rgb2spec.RGB2Spec.load(p)
    assert m.res == 8 and m.scale[0] == 0 and m.scale[-1] == 1 and m.data.size == 3 * 8 ** 3 * 3
    s = [rgb2spec.eval_precise(m.fetch([0.2, 0.5, 0.9]), w) for w in (400, 500, 600)]
    assert all(0 < v < 1 for v in s)
    with open(p, "r+b") as f:
        f.write(b"XXXX")
    with pytest.raises(ValueError):
        rgb2spec.RGB2Spec.load(p)


def test_matrix_cache_file_format(tmp_path):
    # Lightning::SerializeMat layout (Lightning.h:21-50): 5 ints, values, outerIndex[outerSize], innerIndex
    rng = np.random.RandomState(0)
    D = (rng.uniform(0, 1, (7, 7)) * (rng.uniform(0, 1, (7, 7)) < 0.4)).astype(np.float32)
    vals, inner, outer = [], [], [0]
    for c in range(7):
        nz = np.nonzero(D[:, c])[0]
        vals += list(D[nz, c]); inner += list(nz); outer.append(len(vals))
    p = str(tmp_path / "m")
    api.serialize_mat(p, np.array(vals, np.float32), np.array(inner, np.int32), np.array(outer, np.int32), 7)
    raw = open(p, "rb").read()
    assert struct.unpack("<5i", raw[:20]) == (7, 7, len(vals), 7, 7) and len(raw) == 20 + 4 * len(vals) * 2 + 4 * 7
    assert np.array_equal(api.deserialize_mat(p), D)


def test_partition_and_exchange_layout():
    assert dist.partition(131072, 3, 8) == (49152, 65536, 16384)
    assert dist.partition(7712, 7, 8) == (7168, 7712, 1024)  # 964 rounded up to a multiple of 256; last block is short
    assert dist.partition(6401, 0, 1) == (0, 6401, 6404)     # single block: multiple of 4
    assert dist.partition(10, 3, 4) == (10, 10, 256)         # more blocks than rows: empty tail ranks
    assert dist.block_layout(9, 964) == (8696, 8676)         # K*n floats + K doubles, padded to 16 B
    assert [dist.padded_K(k) for k in (1, 2, 3, 9, 12, 17, 32)] == [1, 3, 3, 9, 16, 32, 32]
    x = api.cie1931WavelengthToXYZFit(550.0)
    assert x.dtype == np.float32 and abs(x[1] - 0.99) < 0.02


def test_camera_rays_match_reference_camera_h():
    """Camera::gen_rays_for_screen restated in float32 (glm lookAt / perspective / inverse / unProject order) against the
    reference's own Camera.h compiled in oracle/_ref: bit-exact, with and without supersampling.  Where oracle/_ref is not
    built, against a seeded sample of rays recorded in tests/golden/reference_record.npz: this restatement's own output, not
    Camera.h's, which DESIGN.md section 5 records as bit-identical to it; the committed file was written without oracle/_ref
    to check it."""
    from oracle import pyref
    rec = None if pyref.available() else np.load(os.path.join(GOLDEN, "reference_record.npz"))
    for c, (w, h, ss, aa) in enumerate([(80, 60, 4, True), (80, 60, 4, False), (33, 17, 9, True)]):
        mine = api.Camera(w, h, ss).gen_rays_for_screen(aa)
        if rec is None:
            ref = pyref.camera_rays(w, h, ss, aa)
            assert mine.shape == ref.shape and np.array_equal(mine.view(np.uint32), ref.view(np.uint32))
        else:
            idx = rec[f"camera_{c}_idx"]
            assert mine.shape == (int(rec[f"camera_{c}_count"]), 6)
            assert np.array_equal(mine[idx].view(np.uint32), rec[f"camera_{c}_rays"].view(np.uint32))


def test_product_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under daisyriot_b200/ (Python or CUDA/C++), include/ or shim/ may import,
    include, link or execute it; bench.py may only do so inside its CPU-baseline / reference-arm functions."""
    import re
    bad = []
    for base in ("daisyriot_b200", "include", "shim"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            if "_build" in dirpath or "__pycache__" in dirpath:
                continue
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", "Makefile")):
                    continue
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                if re.search(r"(from|import)\s+oracle|oracle/|liboracle|pyoracle|pyref|daisy_oracle", text):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad
    # bench.py: the oracle is imported only inside the functions that CHECK or serve as the reported CPU baseline, never in the
    # measured path (run_ours calls them outside every timed region)
    src = open(os.path.join(ROOT, "bench.py")).read()
    allowed = {"cpu_reference_run", "parity_block", "incumbent_block"}
    uses = [m.start() for m in re.finditer(r"from oracle import", src)]
    assert uses
    for u in uses:
        owner = re.findall(r"^def (\w+)", src[:u], flags=re.M)[-1]
        assert owner in allowed, owner


def test_library_carries_tcgen05_tmem_and_tensor_tma_code():
    """The wide-band gather must be the tcgen05 kernel (UTCHMMA + TMEM loads/stores) and the loads tensor-map TMA."""
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.SO_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "STTM", "LDTM", "UTMALDG", "UTCBAR"):
        assert mnemonic in sass, mnemonic


def test_plane_ids_host_side(fixture_scenes):
    """daisy_plane_ids (host only): the plane ids the form-factor kernel's coplanar skipping relies on.  The synthetic Cornell
    box has 16 planar quads -- 8 axis-aligned (exact ids) and 8 rotated block faces (fitted in double precision) -- and every
    triangle of a quad must carry the quad's id; vertices moved off their plane by more than the tolerance lose it."""
    from daisyriot_b200 import scenes
    L = _lib.lib()

    def ids(sc):
        v = np.ascontiguousarray(sc.vertices, np.float32)
        t = np.ascontiguousarray(sc.tri, np.int32)
        out = np.zeros(t.shape[0], np.int32)
        _lib.check(L.daisy_plane_ids(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], _lib.iptr(out)))
        return out

    sc = scenes.cornell_box(2048)
    pid = ids(sc).reshape(16, -1)
    assert (pid > 0).all() and all(len(set(q.tolist())) == 1 for q in pid) and len(set(pid[:, 0].tolist())) == 16
    # the same face split over two parallel planes 1e-3 apart: two ids
    sc2 = scenes.cornell_box(2048)
    quad5 = np.unique(sc2.tri[5 * 128:5 * 128 + 64, :3])
    only5 = np.setdiff1d(quad5, np.unique(np.delete(sc2.tri[:, :3], np.s_[5 * 128:5 * 128 + 64], axis=0)))
    sc2.vertices[only5, 1] += 1e-3
    pid2 = ids(sc2)
    assert len(set(pid2[5 * 128:6 * 128].tolist()) - {0}) >= 2
    # curved geometry: the sphere quads of colorballs pair up, nothing larger
    pc = ids(fixture_scenes["colorballs"])
    _, counts = np.unique(pc[pc > 0], return_counts=True)
    assert counts.max() <= 512 and (pc == 0).sum() > 0


def test_face_grids_host_side(fixture_scenes):
    """daisy_face_grid_stats (host only): the planar face grids of csrc/faces.cu.  Every quad of the synthetic Cornell box is a
    face; its cells split into empty (the apron), covered (the inside) and mixed (the outline) and only a thin band is mixed.
    A hole in a face turns the cells around it mixed; T-junctions (an edge not shared by exactly two triangles) do the same."""
    import ctypes as C
    from daisyriot_b200 import scenes
    L = _lib.lib()

    def grids(sc):
        v = np.ascontiguousarray(sc.vertices, np.float32)
        t = np.ascontiguousarray(sc.tri, np.int32)
        st = np.zeros((64, 6), np.int64)
        nf = C.c_int(0)
        pid = np.zeros(t.shape[0], np.int32)
        _lib.check(L.daisy_face_grid_stats(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], 64, st.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(nf), _lib.iptr(pid)))
        return st[:nf.value], pid

    sc = scenes.cornell_box(8192)
    st, pid = grids(sc)
    assert st.shape[0] == 16 and (st[:, 0] == 512).all()
    assert sorted(set(pid.tolist())) == list(range(1, 17))          # face f carries plane id f + 1
    assert (st[:, 2] + st[:, 3] + st[:, 4] == st[:, 1]).all()        # empty + covered + mixed = cells
    assert (st[:, 3] > 10 * st[:, 4]).all() and (st[:, 4] > 0).all()  # a thin mixed band around a covered inside
    assert (st[:, 5] >= st[:, 3] + st[:, 4]).all()                   # every non-empty cell lists at least one triangle
    # remove a block of 4 x 4 cells from the floor (quad 0): the hole's rim becomes mixed, its inside empty
    keep = np.ones(sc.numtriangles, bool)
    for j in range(6, 10):
        keep[(j * 16 + 6) * 2:(j * 16 + 10) * 2] = False
    sc2 = scenes.Scene(sc.vertices, sc.normals, sc.tri[keep], sc.mat_idx[keep], sc.materials, "holed")
    st2, _ = grids(sc2)
    f0 = int(np.argmin(st2[:, 0]))                                   # the face that lost 32 triangles
    assert st2[f0, 0] == 512 - 32 and st2[f0, 4] > st[0, 4] and st2[f0, 2] > st[0, 2]
    # T-junctions: one 8 x 8 sheet with a cell cut in four next to uncut neighbours.  The halves of the uncut neighbours' edges are
    # not shared by exactly two triangles, so the cells along them turn mixed although the sheet has no hole
    def sheet(split):
        V, T = [], []

        def vid(x, z):
            V.append((x, 0.0, z))
            return len(V) - 1

        g = [[vid(i, j) for i in range(9)] for j in range(9)]
        for j in range(8):
            for i in range(8):
                a, b, c, d = g[j][i], g[j][i + 1], g[j + 1][i], g[j + 1][i + 1]
                if split and (i, j) == (3, 4):
                    m = [[a, vid(i + .5, j), b], [vid(i, j + .5), vid(i + .5, j + .5), vid(i + 1, j + .5)], [c, vid(i + .5, j + 1), d]]
                    for jj in range(2):
                        for ii in range(2):
                            q = (m[jj][ii], m[jj][ii + 1], m[jj + 1][ii], m[jj + 1][ii + 1])
                            T += [[q[0], q[3], q[1], 0, 0, 0], [q[0], q[2], q[3], 0, 0, 0]]
                else:
                    T += [[a, d, b, 0, 0, 0], [a, c, d, 0, 0, 0]]
        return scenes.Scene(np.asarray(V, np.float32), np.array([[0, 1, 0]], np.float32), np.asarray(T, np.int32),
                            np.zeros(len(T), np.int32), sc.materials, "sheet")

    plain, cut = grids(sheet(False))[0], grids(sheet(True))[0]
    assert plain.shape[0] == 1 and cut.shape[0] == 1 and cut[0, 0] == plain[0, 0] + 6
    # (six more, smaller triangles: the cell size differs a little, so fractions are compared) a larger share of mixed cells
    assert cut[0, 4] / cut[0, 1] > 1.03 * plain[0, 4] / plain[0, 1]
    # curved geometry has no faces to speak of; the box around the balls does
    stc, _ = grids(fixture_scenes["colorballs"])
    assert 1 <= stc.shape[0] <= 64


def test_face_grid_cells_mean_what_they_say():
    """The two claims the form-factor kernel builds on (csrc/faces.cu), checked on the CPU against plain geometry for a ragged,
    perforated, T-junctioned, arbitrarily rotated sheet: every point of a COVERED cell (grown by delta) lies in some triangle of
    the face, and no triangle of the face comes within delta of an EMPTY cell.  The cell lists must name every triangle that
    touches the grown cell."""
    import ctypes as C
    from daisyriot_b200 import scenes
    L = _lib.lib()
    rng = np.random.RandomState(7)
    V, T = [], []

    def vid(s, t):
        V.append((s, t))
        return len(V) - 1

    nu = nv = 10
    holes = rng.uniform(size=(nv, nu)) < 0.2
    splits = rng.uniform(size=(nv, nu)) < 0.2
    g = [[vid(i / nu, j / nv) for i in range(nu + 1)] for j in range(nv + 1)]
    for j in range(nv):
        for i in range(nu):
            if holes[j, i] or (i > 6 and j > 7):
                continue
            a, b, c, d = g[j][i], g[j][i + 1], g[j + 1][i], g[j + 1][i + 1]
            quads = [(a, b, c, d)]
            if splits[j, i]:
                m = [[a, vid((i + .5) / nu, j / nv), b], [vid(i / nu, (j + .5) / nv), vid((i + .5) / nu, (j + .5) / nv), vid((i + 1) / nu, (j + .5) / nv)],
                     [c, vid((i + .5) / nu, (j + 1) / nv), d]]
                quads = [(m[jj][ii], m[jj][ii + 1], m[jj + 1][ii], m[jj + 1][ii + 1]) for jj in range(2) for ii in range(2)]
            for q in quads:
                T += [[q[0], q[1], q[3], 0, 0, 0], [q[0], q[3], q[2], 0, 0, 0]] if rng.uniform() < 0.5 else [[q[0], q[1], q[2], 0, 0, 0], [q[1], q[3], q[2], 0, 0, 0]]
    st2 = np.asarray(V, np.float64)
    # place the sheet in space: origin + s * eu + t * ev, rotated arbitrarily
    ax = rng.normal(size=3); ax /= np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    R = np.eye(3) + np.sin(1.1) * K + (1 - np.cos(1.1)) * K @ K
    P3 = (np.array([0.3, 1.0, -0.4]) + st2[:, :1] * np.array([4.0, 0, 0]) + st2[:, 1:] * np.array([0, 0.2, 3.0])) @ R.T
    v = np.ascontiguousarray(P3, np.float32)
    t = np.ascontiguousarray(T, np.int32)
    assert len(t) >= 32
    frame = np.zeros(16, np.float32)
    _lib.check(L.daisy_face_grid_dump(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], 0, _lib.fptr(frame), None, None, 0))
    nx, ny, ntri = int(frame[12]), int(frame[13]), int(frame[14])
    assert ntri == len(t)
    state = np.zeros(nx * ny, np.int8)
    count = np.zeros(nx * ny, np.int32)
    _lib.check(L.daisy_face_grid_dump(_lib.fptr(v), v.shape[0], _lib.iptr(t), t.shape[0], 0, _lib.fptr(frame), state.ctypes.data_as(C.POINTER(C.c_int8)),
                                      _lib.iptr(count), nx * ny))
    state, count = state.reshape(ny, nx), count.reshape(ny, nx)
    assert (state == 1).sum() > 200 and (state == 2).sum() > 50 and (state == 0).sum() > 20
    # triangles in cell coordinates (a, b)
    vd = v.astype(np.float64)
    ex, ey = frame[4:8].astype(np.float64), frame[8:12].astype(np.float64)
    ab = np.stack([vd @ ex[:3] + ex[3], vd @ ey[:3] + ey[3]], 1)
    tri = ab[t[:, :3]]                                                   # (ntri, 3, 2)
    cs = 1.0 / np.linalg.norm(ex[:3])                                    # world units per cell
    used = np.unique(t[:, :3])                                           # the scene extent runs over the vertices the triangles use
    ext = float((v[used].max(0) - v[used].min(0)).max())
    dl = 0.999 * 2.5e-4 * ext / cs                                       # delta in cell units (a hair inside: the frame is float32)

    def inside_any(p, tol):
        d0 = tri[:, 1] - tri[:, 0]; d1 = tri[:, 2] - tri[:, 1]; d2 = tri[:, 0] - tri[:, 2]
        c0 = d0[:, 0] * (p[1] - tri[:, 0, 1]) - d0[:, 1] * (p[0] - tri[:, 0, 0])
        c1 = d1[:, 0] * (p[1] - tri[:, 1, 1]) - d1[:, 1] * (p[0] - tri[:, 1, 0])
        c2 = d2[:, 0] * (p[1] - tri[:, 2, 1]) - d2[:, 1] * (p[0] - tri[:, 2, 0])
        sgn = np.sign(d0[:, 0] * (tri[:, 2, 1] - tri[:, 0, 1]) - d0[:, 1] * (tri[:, 2, 0] - tri[:, 0, 0]))
        return ((c0 * sgn >= -tol) & (c1 * sgn >= -tol) & (c2 * sgn >= -tol)).any()

    def seg_dist(p, a, b):
        ab_, ap = b - a, p - a
        s_ = np.clip((ap * ab_).sum(-1) / np.maximum((ab_ * ab_).sum(-1), 1e-300), 0, 1)
        return np.linalg.norm(ap - s_[:, None] * ab_, axis=-1)

    def dist_to_faces(p):
        if inside_any(p, 0.0):
            return 0.0
        return min(seg_dist(p, tri[:, k], tri[:, (k + 1) % 3]).min() for k in range(3))

    checked = [0, 0]
    for j in range(ny):
        for i in range(nx):
            pts = [(i + fx, j + fy) for fx in (-dl, 0.5, 1 + dl) for fy in (-dl, 0.5, 1 + dl)]   # corners of the grown cell, mid points, centre
            if state[j, i] == 1:
                assert all(inside_any(np.array(p), 1e-9) for p in pts), ("covered cell leaves the face", i, j)
                checked[0] += 1
            elif state[j, i] == 0:
                assert min(dist_to_faces(np.array(p)) for p in pts) > 0.0 and dist_to_faces(np.array((i + .5, j + .5))) > dl, ("triangle near an empty cell", i, j)
                assert count[j, i] == 0
                checked[1] += 1
            if state[j, i] != 0:
                # the list names every triangle that overlaps the cell (at least those containing one of the sample points)
                touching = set()
                for p in pts:
                    p = np.array(p)
                    d0 = tri[:, 1] - tri[:, 0]
                    sgn = np.sign(d0[:, 0] * (tri[:, 2, 1] - tri[:, 0, 1]) - d0[:, 1] * (tri[:, 2, 0] - tri[:, 0, 0]))
                    ok = np.ones(len(tri), bool)
                    for k in range(3):
                        dk = tri[:, (k + 1) % 3] - tri[:, k]
                        ok &= (dk[:, 0] * (p[1] - tri[:, k, 1]) - dk[:, 1] * (p[0] - tri[:, k, 0])) * sgn >= 0
                    touching |= set(np.nonzero(ok)[0].tolist())
                assert count[j, i] >= len(touching), ("cell list too short", i, j, count[j, i], len(touching))
    assert checked[0] > 200 and checked[1] > 20


def test_committed_row_digests_cover_the_bench_workloads():
    import bench
    for name, (N, K, _) in bench.WORKLOADS.items():
        path = os.path.join(GOLDEN, f"rowdigest_{name}.npz")
        if name == "cornell_8k" or name in bench.SAME_MATRIX_AS:
            continue
        assert os.path.exists(path), path
        g = np.load(path)
        assert g["digest"].shape == (N,) and g["digest"].dtype == np.uint32 and int(g["patches"]) == N and int(g["pairs"]) > N
