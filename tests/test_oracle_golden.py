"""CPU suite: the oracle against (a) the reference's only known-answer test, (b) analytic identities,
(c) the reference's own sources compiled in oracle/_ref when present, else what they were recorded to produce,
(d) the committed golden vectors."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, two_triangle_scene
from daisyriot_b200 import scenes
from oracle import pyoracle, pyref


def test_reference_known_answer_surface():
    # the reference's single unit test: calculateSurface((0,0,0),(1,0,0),(0,1,0)) == 0.5f   (unittest1.cpp:15)
    L = pyoracle.lib()
    a, b, c = (np.array(v, np.float32) for v in ([0, 0, 0], [1, 0, 0], [0, 1, 0]))
    assert L.orc_surface3(pyoracle._fp(a), pyoracle._fp(b), pyoracle._fp(c)) == np.float32(0.5)
    if pyref.available():
        assert pyref.calculate_surface3(a, b, c) == np.float32(0.5)


def test_two_facing_triangles_by_hand():
    """F for two parallel unit right triangles one unit apart equals the 16-term sum evaluated in float64."""
    sc = two_triangle_scene()
    orc = pyoracle.Oracle.from_scene(sc)
    V, T = sc.vertices.astype(np.float64), sc.tri

    def subs(t):
        a, b, c = V[T[t, 0]], V[T[t, 1]], V[T[t, 2]]
        iA, iC, iB = (b - a) / 2 + a, (c - a) / 2 + a, (b - c) / 2 + c
        tr = [(a, iC, iA), (iC, c, iB), (iA, iB, b), (iA, iB, iC)]
        return [(sum(x) / 3, 0.5 * np.linalg.norm(np.cross(x[1] - x[0], x[2] - x[0]))) for x in tr]

    n0, n1 = np.array([0, 0, 1.0]), np.array([0, 0, -1.0])
    tot = 0.0
    for p, ap in subs(0):
        for q, aq in subs(1):
            d = q - p
            ln = np.linalg.norm(d)
            tot += (n0 @ d / ln) * (n1 @ -d / ln) / (np.pi * ln * ln) * ap * aq
    want = tot / 0.5
    got = orc.p2p_ff(0, 1, 0)
    assert abs(got - want) < 2e-6 * want
    assert abs(orc.p2p_ff(0, 1, 1) - want) < 2e-6 * want
    # reciprocity A_i F_ij = A_j F_ji (equal areas here) and an empty diagonal
    assert abs(orc.p2p_ff(1, 0, 0) - got) < 1e-6 * want
    uv = scenes.msvc_sample_pattern(1)
    F, m, rays = orc.radmat_rows(uv, 0, 2, brute=True)
    assert rays == 2 * 50 and F[0, 0] == 0 and F[1, 1] == 0
    assert m[0, 1] == m[1, 0] == np.uint64((1 << 50) - 1)  # nothing in between: every sample sees the other patch
    assert F[0, 1] == got


def test_watertight_known_answers():
    a, b, c = [0, 0, 0], [1, 0, 0], [0, 1, 0]
    ok, t, u, v = pyoracle.ray_tri([0.25, 0.5, -2, 0, 0, 1], a, b, c)
    assert ok and t == 2.0 and u == 0.25 and v == 0.5
    assert not pyoracle.ray_tri([0.25, 0.5, 2, 0, 0, 1], a, b, c)[0]      # behind the origin
    assert not pyoracle.ray_tri([0.75, 0.75, -1, 0, 0, 1], a, b, c)[0]    # outside
    assert not pyoracle.ray_tri([0.25, 0.25, 0, 0, 0, 1], a, b, c)[0]     # t == 0 is not a hit (t > 0 rule)
    assert not pyoracle.ray_tri([0.25, 0.25, -1, 1, 0, 0], a, b, c)[0]    # parallel to the plane
    # a ray through a shared edge hits exactly one... or both: never neither (watertightness)
    d = [1, 1, 0]
    h1 = pyoracle.ray_tri([0.5, 0.5, -1, 0, 0, 1], a, b, c)[0]
    h2 = pyoracle.ray_tri([0.5, 0.5, -1, 0, 0, 1], b, d, c)[0]
    assert h1 or h2


def test_bvh_equals_bruteforce(cornell512, uv50):
    orc = pyoracle.Oracle.from_scene(cornell512)
    rng = np.random.RandomState(3)
    o = rng.uniform(0, 5.5, (3000, 3)).astype(np.float32)
    d = rng.normal(size=(3000, 3)).astype(np.float32)
    rays = np.concatenate([o, d], 1)
    a, b = orc.query_closest(rays), orc.query_closest(rays, brute=True)
    assert np.array_equal(a, b)
    assert (a["triangleId"] >= 0).mean() > 0.7
    Fa, ma, _ = orc.radmat_rows(uv50, 100, 104)
    Fb, mb, _ = orc.radmat_rows(uv50, 100, 104, brute=True)
    assert np.array_equal(ma, mb) and np.array_equal(Fa, Fb)


def test_oracle_vs_compiled_reference_sources(fixture_scenes, uv50):
    """Bit-exact against triangle_math.cpp compiled in oracle/_ref; where that is not built, against the same quantities on the
    same inputs recorded in tests/golden/reference_record.npz.  That record is this oracle's own output, not the reference's;
    DESIGN.md section 5 records the two as bit-identical, and the committed file was written without oracle/_ref to check it."""
    rec = None if pyref.available() else np.load(os.path.join(GOLDEN, "reference_record.npz"))
    for name, sc in fixture_scenes.items():
        orc = pyoracle.Oracle.from_scene(sc)
        rs = pyref.RefScene.from_arrays(sc.vertices, sc.normals, sc.tri) if rec is None else None
        rng = np.random.RandomState(1)
        for n in range(600):
            i, j = rng.randint(0, sc.numtriangles, 2)
            k = rng.randint(50)
            if rs is not None:  # triangle_math.cpp, float pi
                want = rs.p2p_unoccluded(i, j), rs.pair_ray(i, j, uv50[k, 0], uv50[k, 1]), rs.surface(i)
            else:
                assert tuple(rec[name + "_ij"][n]) == (i, j) and rec[name + "_k"][n] == k
                want = rec[name + "_p2p"][n], rec[name + "_pair_ray"][n], rec[name + "_surface"][n]
            a = orc.p2p_ff(i, j, 1)
            assert a == want[0] or (np.isnan(a) and np.isnan(want[0])), (name, i, j)
            assert np.array_equal(orc.pair_ray(i, j, uv50[k, 0], uv50[k, 1]), want[1], equal_nan=True)
            assert np.float32(orc.surface(i)) == want[2]
        if rs is not None:
            rs.close()


def test_gather_vs_reference_lightning(cornell512, uv50, coeff_model):
    """The reference's unmodified Lightning.h + Eigen 3.2.10 against the oracle pass on the same matrix:
    identical pass count under the stop rule; FP32-sequential oracle within 1e-6, FP64 oracle within 1e-5.  Where oracle/_ref
    is not built, against the materials, pass counts and B recorded in tests/golden/reference_record.npz: this project's own
    output, not the reference's, which DESIGN.md section 5 records as matching it (same pass counts, B within 2e-6); the
    committed file was written without oracle/_ref to check it."""
    from daisyriot_b200 import materials
    model, cwd = coeff_model
    sc = cornell512
    wl = np.arange(200, 601, 50).astype(np.float32)
    mats = materials.make_materials(sc.materials, wl, model)
    g = np.load(os.path.join(GOLDEN, "cornell512_golden.npz"))
    F = g["F_device"]
    rec = rs = None
    if pyref.available():
        obj, _ = scenes.write_obj(sc, cwd, "c512")
        rs = pyref.RefScene.load(obj, cwd + "/", wl, cwd)
    else:
        rec = np.load(os.path.join(GOLDEN, "reference_record.npz"))
    for i, m in enumerate(mats):  # material restatement is bit-exact, except the lamp's undefined M
        r = rs.material(i) if rs is not None else {"spectral_values": rec["material_spectral_values"][i],
                                                   "spectral_emission": rec["material_spectral_emission"][i], "M": rec["material_M"][i]}
        assert np.array_equal(r["spectral_values"], m.spectral_values, equal_nan=True)
        assert np.array_equal(r["spectral_emission"], m.spectral_emission, equal_nan=True)
        if m.kind == "uvlight":
            if rs is not None:
                rs.set_material_M(i, m.M)
        else:
            assert np.array_equal(r["M"], m.M, equal_nan=True)
    if rs is not None:
        rs.set_triplets_from_dense(F)
    for method, inputs in [(2, materials.spectral_inputs), (1, materials.rgb_inputs), (0, materials.bw_inputs)]:
        ev = 7.0
        if rs is not None:
            passes_ref = rs.lightning_create(method, ev)  # constructor converges
            B_ref, R_ref = rs.lightning_read()
        else:
            passes_ref, B_ref = int(rec[f"lightning_passes_{method}"]), rec[f"lightning_B_{method}"]
        E, M = inputs(mats, sc.mat_idx, ev)
        thr, per_band = (200.0, False) if method == 2 else (1e-4, True)
        for accum, tol in [(0, 2e-6), (1, 1e-5)]:
            res, B = E.copy(), E.copy()
            sums = res.astype(np.float64).sum(1)
            passes = 0
            while ((sums > thr).any() if per_band else sums.sum() > thr) and passes < 1000:
                sums = pyoracle.gather_pass(F, res, B, M, sc.mat_idx, accum=accum)
                passes += 1
            assert passes == passes_ref, (method, accum, passes, passes_ref)
            scale = max(np.abs(B_ref).max(), 1e-30)
            assert np.allclose(B, B_ref, rtol=tol, atol=tol * scale), (method, accum, np.abs(B - B_ref).max() / scale)
    if rs is not None:
        rs.close()


def test_oracle_reproduces_golden_vectors(cornell512):
    g = np.load(os.path.join(GOLDEN, "cornell512_golden.npz"))
    uv = g["uv"]
    assert np.array_equal(uv, scenes.msvc_sample_pattern(1))
    orc = pyoracle.Oracle.from_scene(cornell512)
    rows = [0, 5, 97, 256, 400, 511]
    assert list(g["F_host_reciprocity_rows"]) == rows  # the host-variant matrix is stored for these rows only
    for i, r in enumerate(rows):
        F, m, _ = orc.radmat_rows(uv, r, r + 1)
        assert np.array_equal(F[0].view(np.uint32), g["F_device"][r].view(np.uint32))
        assert np.array_equal(m[0], g["masks_device"][r])
        F1, _, _ = orc.radmat_rows(uv, r, r + 1, variant=1, reciprocity=True)
        assert np.array_equal(F1[0].view(np.uint32), g["F_host_reciprocity"][i].view(np.uint32))
    U = orc.unoccluded_rows(0, 8, 0)
    assert np.array_equal(U.view(np.uint32), g["unoccluded_device"][:8].view(np.uint32))
    assert np.array_equal(orc.query_closest(g["hit_rays"]), g["hits"])
    res, B = g["gather_E"].copy(), g["gather_E"].copy()
    for it in range(3):
        sums = pyoracle.gather_pass(g["F_device"], res, B, g["gather_M"], cornell512.mat_idx, accum=1)
        assert np.allclose(sums, g["gather_sums"][it], rtol=1e-12)
    assert np.array_equal(B, g["gather_B3"]) and np.array_equal(res, g["gather_res3"])
    # whole-matrix invariants of the frozen matrix: symmetric masks, empty diagonal, reciprocity A_i F_ij = A_j F_ji
    F = g["F_device"]
    A = np.array([orc.surface(i) for i in range(512)])
    assert np.array_equal(g["masks_device"], g["masks_device"].T) and not F.diagonal().any()
    AF = A[:, None] * F.astype(np.float64)
    assert np.abs(AF - AF.T).max() < 1e-6 * AF.max()


@pytest.mark.parametrize("name", ["cornellbox_blacklight", "colorballs"])
def test_oracle_reproduces_fixture_rows(fixture_scenes, name):
    g = np.load(os.path.join(GOLDEN, name + "_rows_golden.npz"))
    orc = pyoracle.Oracle.from_scene(fixture_scenes[name])
    for k in (0, 4, 8):  # three of the nine frozen rows keep the CPU suite quick
        r = int(g["rows"][k])
        F, m, _ = orc.radmat_rows(g["uv"], r, r + 1)
        assert np.array_equal(F[0].view(np.uint32), g["F"][k].view(np.uint32))
        assert np.array_equal(m[0], g["masks"][k])


@pytest.mark.parametrize("name,pairs", [("cornellbox_blacklight", 9322918), ("colorballs", 7587047)])
def test_full_golden_matches_surveyed_workload(name, pairs, fixture_scenes):
    """The whole-matrix goldens were produced by the oracle over every pair of the reference scenes; their facing-pair
    counts equal the independently surveyed ones (SURVEY.md section 6), and a re-derived row matches its digest."""
    g = np.load(os.path.join(GOLDEN, name + "_full_golden.npz"))
    assert int(g["pairs"]) == pairs
    sc = fixture_scenes[name]
    orc = pyoracle.Oracle.from_scene(sc)
    r = sc.numtriangles - 7
    F, m, _ = orc.radmat_rows(g["uv"], r, r + 1)
    mh, fs, fx = pyoracle.row_checksums(F, m)
    assert mh[0] == g["mask_hash"][r] and fx[0] == g["F_xor"][r] and abs(fs[0] - g["F_sum"][r]) <= 1e-12 * max(1.0, abs(fs[0]))
