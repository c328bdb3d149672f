"""Solves with 33-64 bands: the K = 64 instantiation of the tcgen05 3xTF32 gather (csrc/gather_mma.cuh), the only kernel
for K > 32, against FP64.

K = 33..63 run padded to 64 with inert zero bands.  Ragged sizes exercise a partial last 128-row block, a last column step
clipped at ldF and residual columns between N and n; the matrices are built tile by tile (64 x 256) so that a dropped or
double-counted tile moves the results far beyond the 1e-5 tolerance.  Partitions on one GPU are exchanged by hand; the
fused exchange with real peers needs two GPUs.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_rel

pytestmark = pytest.mark.gpu

SIZES = [1, 5, 127, 129, 257, 1000, 7712]
KS = [33, 41, 47, 63, 64]
ALL_K_SIZES = (257, 7712)
CASES = [(N, K) for N in SIZES for K in KS] + [(N, K) for N in ALL_K_SIZES for K in range(33, 65) if K not in KS]
NMAT = 13
PASSES = 3
ENV_VARS = ("DAISY_GATHER", "DAISY_GATHER_EPI", "DAISY_GATHER_SKIP")


def _L():
    from daisyriot_b200 import _lib
    return _lib.lib()


def _check(rc, what=""):
    from daisyriot_b200 import _lib
    _lib.check(rc, what)


def _fp(a):
    from daisyriot_b200 import _lib
    return _lib.fptr(a)


def _ip(a):
    from daisyriot_b200 import _lib
    return _lib.iptr(a)


def _dp(x):
    return x.ctypes.data_as(C.POINTER(C.c_double))


# ---- inputs (the same construction as the narrow-band shape tests) ------------------------------------------------------
def make_matrix(N, seed):
    """N x N FP32 built at 64 x 256 tile granularity: about half the tiles occupied, a few whole zero row blocks and column
    steps, non-zeros guaranteed in row N-1 and column N-1; values in (0, 2/N)."""
    rng = np.random.RandomState(seed)
    nrb, ncs = -(-N // 64), -(-N // 256)
    occ = rng.uniform(0, 1, (nrb, ncs)) < 0.5
    zero_rb = set(rng.choice(nrb - 1, min(2, nrb - 1), replace=False).tolist()) if nrb > 2 else set()
    zero_cs = {int(rng.randint(0, ncs - 1))} if ncs > 2 else set()
    for rb in zero_rb:
        occ[rb] = False
    for cs in zero_cs:
        occ[:, cs] = False
    free_rows = np.array([r for r in range(N) if r // 64 not in zero_rb])
    free_cols = np.array([c for c in range(N) if c // 256 not in zero_cs])
    mask = np.repeat(np.repeat(occ, 64, axis=0), 256, axis=1)[:N, :N] & (rng.uniform(0, 1, (N, N)) < 0.5)
    F = np.where(mask, rng.uniform(0, 2.0 / N, (N, N)), 0.0).astype(np.float32)
    for rb, cs in zip(*np.nonzero(occ)):
        r = rng.randint(rb * 64, min(N, rb * 64 + 64))
        c = rng.randint(cs * 256, min(N, cs * 256 + 256))
        F[r, c] = rng.uniform(0.5, 2.0) / N
    F[N - 1, N - 1] = 1.5 / N
    F[N - 1, rng.choice(free_cols, min(8, len(free_cols)))] = 1.0 / N
    F[rng.choice(free_rows, min(8, len(free_rows))), N - 1] = 1.0 / N
    return F


def make_inputs(N, K, seed):
    """E positive in every band and column; 13 random non-symmetric, contracting K x K material matrices."""
    rng = np.random.RandomState(seed)
    E = np.ascontiguousarray(rng.uniform(0.5, 2.0, (K, N)).astype(np.float32))
    M = np.ascontiguousarray(rng.uniform(0, 0.9 / K, (NMAT, K, K)).astype(np.float32))
    mat = np.ascontiguousarray(rng.randint(0, NMAT, N).astype(np.int32))
    return E, M, mat


def fp64_pass(F, R, B, M, mat):
    """residual <- M[mat] (F residual), B += residual, in FP64 (M column-major: y[k] = sum_j M[j, k] b[j])"""
    b = np.asarray(F, np.float64) @ R.T
    y = np.einsum("ijk,ij->ik", M.astype(np.float64)[mat], b)
    R = y.T.copy()
    return R, B + R, R.sum(axis=1)


def fp64_passes(F, E, M, mat, passes):
    R, B = E.astype(np.float64), E.astype(np.float64)
    out = []
    for _ in range(passes):
        R, B, sums = fp64_pass(F, R, B, M, mat)
        out.append((R, B, sums))
    return out


def sub_scene(N):
    """The first N triangles of a Cornell box of 32 * ceil(N / 32) patches."""
    from daisyriot_b200 import scenes
    from daisyriot_b200.scenes import Scene
    sc = scenes.cornell_box(32 * math.ceil(N / 32))
    return Scene(sc.vertices, sc.normals, sc.tri[:N], sc.mat_idx[:N], sc.materials, "cornell_first_%d" % N)


def create_solver(ctx, K, E, M, mat, monkeypatch):
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    L = _L()
    s = C.c_void_p()
    _check(L.daisy_solver_create(ctx, K, _fp(E), _fp(M), M.shape[0], _ip(mat), C.byref(s)), "solver_create K=%d" % K)
    assert L.daisy_solver_launches_per_pass(s) == 3, K  # residual split, tcgen05 pass, epilogue
    return s


def read_guarded(s, K, nloc):
    """daisy_solver_read into buffers one band and a few columns larger, pre-filled with a sentinel that must survive."""
    sentinel = np.float32(-7.25e30)
    bufB = np.full((K + 1) * (nloc + 3), sentinel, np.float32)
    bufR = np.full((K + 1) * (nloc + 3), sentinel, np.float32)
    _check(_L().daisy_solver_read(s, _fp(bufB), _fp(bufR)))
    assert np.all(bufB[K * nloc:] == sentinel) and np.all(bufR[K * nloc:] == sentinel), "read wrote past K x nloc"
    return bufB[:K * nloc].reshape(K, nloc).copy(), bufR[:K * nloc].reshape(K, nloc).copy()


def run_passes(s, K, N, passes):
    sums = []
    for _ in range(passes):
        t = np.zeros(K)
        _check(_L().daisy_solver_step(s, _dp(t)), "solver_step")
        sums.append(t)
    B, R = read_guarded(s, K, N)
    return B, R, sums


def compare(B, R, sums, ref, what):
    Rw, Bw, Sw = ref
    for k in range(B.shape[0]):
        assert_rel(R[k], Rw[k], (what, "residual", k))
        assert_rel(B[k], Bw[k], (what, "B", k))
    assert np.allclose(sums, Sw, rtol=1e-5, atol=0), (what, "band sums", sums, Sw)


def bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a.view(np.uint64)


class _Contexts:
    """One context per N (and per partition), F loaded from make_matrix, built on first use."""

    def __init__(self):
        self.single, self.parts, self.F, self.F64 = {}, {}, {}, {}

    def matrix(self, N):
        if N not in self.F:
            self.F[N] = make_matrix(N, 3000 + N)
            self.F64[N] = self.F[N].astype(np.float64)
        return self.F[N]

    def get(self, N):
        import daisyriot_b200 as dz
        from daisyriot_b200 import scenes
        if N not in self.single:
            p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sub_scene(N)), device=0, rands=scenes.msvc_sample_pattern(1))
            p.loadRadiosityMatrix(self.matrix(N))
            self.single[N] = p
        return self.single[N], self.F[N]

    def partition(self, N, G):
        import daisyriot_b200 as dz
        from daisyriot_b200 import scenes
        if (N, G) not in self.parts:
            F = self.matrix(N)
            mesh = dz.MeshS.from_scene(sub_scene(N))
            ps = []
            for g in range(G):
                p = dz.OptixPrimeFunctionality(mesh, device=0, rands=scenes.msvc_sample_pattern(1), rank=g, nranks=G)
                r0, r1 = p.row_range
                p.loadRadiosityMatrix(F[r0:r1], r0)
                ps.append(p)
            self.parts[(N, G)] = ps
        return self.parts[(N, G)], self.F[N]

    def reference(self, N, K, passes=PASSES):
        E, M, mat = make_inputs(N, K, 5 * N + K)
        self.matrix(N)
        return E, M, mat, fp64_passes(self.F64[N], E, M, mat, passes)

    def close(self):
        for p in self.single.values():
            p.close()
        for ps in self.parts.values():
            for p in ps:
                p.close()


@pytest.fixture(scope="module")
def contexts():
    import daisyriot_b200 as dz
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    c = _Contexts()
    yield c
    c.close()


# ---- 1. ragged sizes ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,K", CASES)
def test_wide_bands_vs_fp64(contexts, N, K, monkeypatch):
    """3 passes with band sums against FP64; reads stay inside K x N; the same passes after daisy_solver_reset are
    bit-identical."""
    L = _L()
    p, F = contexts.get(N)
    E, M, mat, ref = contexts.reference(N, K)
    s = create_solver(p._ctx, K, E, M, mat, monkeypatch)
    try:
        B, R, sums = run_passes(s, K, N, PASSES)
        for i in range(PASSES):
            assert np.allclose(sums[i], ref[i][2], rtol=1e-5, atol=0), (N, K, "band sums of pass", i)
        compare(B, R, sums[-1], ref[-1], (N, K))
        _check(L.daisy_solver_reset(s))
        B2, R2, sums2 = run_passes(s, K, N, PASSES)
        assert np.array_equal(bits(B2), bits(B)) and np.array_equal(bits(R2), bits(R)), (N, K, "not deterministic")
        assert all(np.array_equal(a, b) for a, b in zip(sums, sums2)), (N, K, "band sums not deterministic")
    finally:
        L.daisy_solver_destroy(s)


# ---- 2. padding ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [257, 7712])
def test_padded_bands_are_inert(contexts, N, monkeypatch):
    """K = 41 (run padded to 64) and the same problem padded to K = 64 by hand -- zero emission, zero rows and columns of M
    -- give bit-identical bands 0-40, and the hand-padded bands stay exactly zero.  This guards the host's padding of E and M
    to 64 bands (daisy_solver_create) and the reads, sums and stop rule restricted to the first K bands; both runs feed the
    same kernel the same device data, so the kernel's arithmetic is covered by the FP64 tests, not here."""
    L = _L()
    p, F = contexts.get(N)
    K, Kp = 41, 64
    E, M, mat = make_inputs(N, K, 17 + N)
    E64 = np.zeros((Kp, N), np.float32)
    E64[:K] = E
    M64 = np.zeros((NMAT, Kp, Kp), np.float32)
    M64[:, :K, :K] = M
    got = []
    for k, e, m in ((K, E, M), (Kp, E64, M64)):
        s = create_solver(p._ctx, k, e, m, mat, monkeypatch)
        got.append(run_passes(s, k, N, PASSES))
        L.daisy_solver_destroy(s)
    (B1, R1, S1), (B2, R2, S2) = got
    assert np.array_equal(bits(B1), bits(B2[:K])) and np.array_equal(bits(R1), bits(R2[:K]))
    assert all(np.array_equal(a, b[:K]) for a, b in zip(S1, S2))
    assert not B2[K:].any() and not R2[K:].any() and all(not b[K:].any() for b in S2)


# ---- 3. long rows ------------------------------------------------------------------------------------------------------------
def test_k64_tensor_core_gather_at_65536_columns(uv50):
    """65 536 patches, K = 64: a context owning 2 048 rows x 65 536 columns (1 024 accumulator drains per row), one pass
    against an FP64 restatement of Lightning.h:196-226 on those rows, without the bias of a truncating accumulator."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    N, K, G = 65536, 64, 32
    sc = scenes.cornell_box(N, n_fluorescent=10)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv50, rank=5, nranks=G)
    r0, r1 = p.row_range
    nloc = r1 - r0
    assert nloc == 2048
    rng = np.random.RandomState(64)
    F = (rng.uniform(0, 1, (nloc, N)).astype(np.float32) * (rng.uniform(0, 1, (nloc, N)) < 0.3) / np.float32(N)).astype(np.float32)
    p.loadRadiosityMatrix(F, r0)
    nmat = len(sc.materials)
    M = rng.uniform(0, 0.03, (nmat, K, K)).astype(np.float32)
    E = np.ascontiguousarray(rng.uniform(0, 3, (K, N)).astype(np.float32))
    L = _lib.lib()
    s = C.c_void_p()
    _lib.check(L.daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), nmat, _lib.iptr(sc.mat_idx), C.byref(s)))
    _lib.check(L.daisy_solver_step_local(s))
    _lib.check(L.daisy_solver_step_finish(s, None))
    Bg, Rg = np.empty((K, nloc), np.float32), np.empty((K, nloc), np.float32)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(Bg), _lib.fptr(Rg)))
    bounced = E.astype(np.float64) @ F.astype(np.float64).T
    Mr = M.astype(np.float64)[sc.mat_idx[r0:r1]]
    want = np.einsum("pji,jp->ip", Mr, bounced)
    for k in range(K):
        assert_rel(Rg[k], want[k], ("residual", k))
        assert_rel(Bg[k], E[k, r0:r1].astype(np.float64) + want[k], ("B", k))
    assert abs(Rg.astype(np.float64).sum() / want.sum() - 1) < 2e-6  # no systematic bias from the truncating accumulator
    L.daisy_solver_destroy(s)
    p.close()


# ---- 4. device converge ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_band", [0, 1])
def test_converge_device_matches_host_loop(contexts, per_band, monkeypatch):
    """daisy_solver_converge_device against daisy_solver_converge at K = 64: the same pass count (the FP64 one) and
    bit-identical B, residual and band sums; then a max_passes cut below the deciding pass."""
    L = _L()
    N, K = 2050, 64
    p, F = contexts.get(N)
    E, M, mat, ref = contexts.reference(N, K, 12)
    stat = (lambda v: float(np.max(v))) if per_band else (lambda v: float(np.sum(v)))
    vals = [stat(E.astype(np.float64).sum(axis=1))] + [stat(r[2]) for r in ref]
    assert all(b < a for a, b in zip(vals, vals[1:]))
    j = 6
    thr = math.sqrt(vals[j] * vals[j + 1])
    assert min(abs(v / thr - 1) for v in vals) > 1e-3
    for cut in (0, 4):
        got = []
        for fn in (L.daisy_solver_converge, L.daisy_solver_converge_device):
            s = create_solver(p._ctx, K, E, M, mat, monkeypatch)
            n = C.c_int()
            _check(fn(s, thr, per_band, cut, C.byref(n)))
            sums = np.zeros(K)
            _check(L.daisy_solver_band_sums(s, _dp(sums)))
            B, R = read_guarded(s, K, N)
            got.append((n.value, B, R, sums))
            L.daisy_solver_destroy(s)
        (n1, B1, R1, S1), (n2, B2, R2, S2) = got
        assert n1 == n2 == (j + 1 if cut == 0 else cut), (per_band, cut, n1, n2)
        assert np.array_equal(bits(B1), bits(B2)) and np.array_equal(bits(R1), bits(R2)) and np.array_equal(S1, S2), (per_band, cut)
        compare(B2, R2, S2, ref[n2 - 1], (per_band, cut))


# ---- 5. partitions -------------------------------------------------------------------------------------------------------------
def _exchange_views(solvers):
    """torch views of every rank's next exchange buffer, and the block length in floats"""
    import torch
    from daisyriot_b200.dist import _DevMem
    views, blk = [], None
    for s in solvers:
        ptr, b, tot = C.c_void_p(), C.c_int64(), C.c_int64()
        _check(_L().daisy_solver_exchange_info(s, C.byref(ptr), C.byref(b), C.byref(tot)))
        views.append(torch.as_tensor(_DevMem(ptr.value, tot.value), device="cuda:0"))
        blk = b.value // 4
    return views, blk


@pytest.mark.parametrize("N,G", [(300, 2), (300, 3)])
def test_partition_on_one_gpu(contexts, N, G, monkeypatch):
    """G ranks on device 0 (N = 300 on 3 ranks leaves the last one without rows), exchanged by hand: the concatenated B,
    the residual and the totals equal the single context and FP64."""
    import torch
    L = _L()
    K = 64
    ps, F = contexts.partition(N, G)
    ranges = [p.row_range for p in ps]
    assert ranges[-1][1] == N and (G < 3 or ranges[-1][0] == ranges[-1][1])
    E, M, mat, ref = contexts.reference(N, K)
    p1, _ = contexts.get(N)
    s1 = create_solver(p1._ctx, K, E, M, mat, monkeypatch)
    B1, R1, S1 = run_passes(s1, K, N, PASSES)
    L.daisy_solver_destroy(s1)
    solvers = [create_solver(p._ctx, K, E, M, mat, monkeypatch) for p in ps]
    try:
        for it in range(PASSES):
            for s in solvers:
                _check(L.daisy_solver_step_local(s), "step_local")
            torch.cuda.synchronize(0)
            views, blk = _exchange_views(solvers)
            for g in range(G):
                for h in range(G):
                    if h != g:
                        views[h][g * blk:(g + 1) * blk].copy_(views[g][g * blk:(g + 1) * blk])
            torch.cuda.synchronize(0)
            for g, s in enumerate(solvers):
                t = np.zeros(K)
                _check(L.daisy_solver_step_finish(s, _dp(t)), "step_finish")
                assert np.allclose(t, S1[it], rtol=1e-5, atol=0) and np.allclose(t, ref[it][2], rtol=1e-5, atol=0), (N, G, it, g)
        B = np.zeros((K, N), np.float32)
        R = np.zeros((K, N), np.float32)
        for (r0, r1), s in zip(ranges, solvers):
            if r1 > r0:
                B[:, r0:r1], R[:, r0:r1] = read_guarded(s, K, r1 - r0)
        for k in range(K):
            assert_rel(B[k], B1[k], (N, G, "B against one context", k))
            assert_rel(R[k], R1[k], (N, G, "residual against one context", k))
        compare(B, R, t, ref[-1], (N, G))
    finally:
        torch.cuda.synchronize(0)
        for s in solvers:
            L.daisy_solver_destroy(s)


@pytest.mark.parametrize("N", [224, 2050])
def test_device_group_fused_exchange(N, monkeypatch):
    """DeviceGroup over 2 GPUs (N = 224 leaves rank 1 without rows), K = 64 with the fused exchange: step against FP64 and
    one GPU, converge(on_device=True) against the host group loop, bit for bit."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    L = _L()
    if L.daisy_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setenv("DAISY_EXCHANGE_TIMEOUT_MS", "20000")
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    K = 64
    uv = scenes.msvc_sample_pattern(1)
    mesh = dz.MeshS.from_scene(sub_scene(N))
    F = make_matrix(N, 4000 + N)
    E, M, mat = make_inputs(N, K, 13 * N)
    ref = fp64_passes(F.astype(np.float64), E, M, mat, PASSES)
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv)
    grp = dz.DeviceGroup(mesh, devices=[0, 1], rands=uv)
    try:
        p.loadRadiosityMatrix(F)
        _check(L.daisy_group_formfactors_write_rows(grp._g, 0, N, _lib.fptr(F)))
        s = create_solver(p._ctx, K, E, M, mat, monkeypatch)
        gs = dz.GroupSolver(grp, K, E, M, mat)
        for it in range(PASSES):
            t = np.zeros(K)
            _check(L.daisy_solver_step(s, _dp(t)))
            got = gs.step(True)
            assert np.allclose(got, ref[it][2], rtol=1e-5, atol=0) and np.allclose(got, t, rtol=1e-6, atol=0), (N, it)
        B2, R2 = gs.read()
        compare(B2, R2, got, ref[-1], (N, "group"))
        thr = 1e-3 * float(E.astype(np.float64).sum())
        res = []
        for on_device in (False, True):
            gs.reset()
            n = gs.converge(thr, False, 200, on_device=on_device)
            res.append((n, *gs.read(), gs.band_sums()))
        (n1, Bh, Rh, Sh), (n2, Bd, Rd, Sd) = res
        assert n1 == n2 and n1 > 2, (n1, n2)
        assert np.array_equal(bits(Bh), bits(Bd)) and np.array_equal(bits(Rh), bits(Rd)) and np.array_equal(Sh, Sd)
        gs.close()
        L.daisy_solver_destroy(s)
    finally:
        grp.close()
        p.close()


# ---- 6. spectral end to end ----------------------------------------------------------------------------------------------------
def test_spectral_lightning_41_wavelengths(uv50, coeff_model):
    """SpectralLightning on the cornellbox_blacklight scene sampled every 10 nm from 200 to 600 nm (41 bands, 9 of them in the
    UV window the fluorescent material rewrites): the pass count of an FP64 restatement of increment_light_fluorescent with
    the threshold-200 rule on the read-back F, B within 1e-5, finite colours."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import materials, scenes
    model, _ = coeff_model
    sc = scenes.load_scene_npz(os.path.join(GOLDEN, "cornellbox_blacklight.npz"))
    wl = np.arange(200, 601, 10).astype(np.float32)
    assert len(wl) == 41 and int(((wl > 300) & (wl < 400)).sum()) == 9
    mesh = dz.MeshS.from_scene(sc, wl, model)
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv50)
    ev = 7.0
    lt = dz.Lightning.get_lightning(2, mesh, p, ev, wl, True, None, converge=False)
    try:
        assert lt.K == 41
        F = lt.RadMat.rows().astype(np.float64)
        E, M = materials.spectral_inputs(mesh.materials, mesh.materialIndexPerTriangle, ev)
        assert np.any(M[:, :, :] * (1 - np.eye(41))[None]), "no material mixes bands"
        R, B = E.astype(np.float64), E.astype(np.float64)
        crit = [float(R.sum())]
        while crit[-1] > 200.0 and len(crit) <= 400:
            R, B, sums = fp64_pass(F, R, B, M, mesh.materialIndexPerTriangle)
            crit.append(float(sums.sum()))
        passes = len(crit) - 1
        assert passes >= 1
        assert abs(crit[-1] / 200.0 - 1) > 1e-5 and abs(crit[-2] / 200.0 - 1) > 1e-5, crit[-2:]  # no decision within rounding
        got = lt.converge_lightning(400)
        assert got == passes, (got, passes)
        Bg, _ = lt.read()
        for k in range(41):
            assert_rel(Bg[k], B[k], ("converged B", k))
        lt.update_color_cache()
        assert np.isfinite(lt._cache).all() and lt._cache.shape == (sc.numtriangles, 3)
    finally:
        lt.close()
        p.close()


# ---- 7. refusals ---------------------------------------------------------------------------------------------------------------
def test_band_count_limits(contexts, monkeypatch):
    """K = 65 and K = 0 are refused; K > 32 has no FP32 or ldg kernel, so those settings are refused too; K = 64 launches the
    residual split, the tensor-core pass and the epilogue."""
    L = _L()
    N = 129
    p, F = contexts.get(N)
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    for K in (65, 0):
        E, M, mat = make_inputs(N, max(K, 1), 1)
        s = C.c_void_p()
        assert L.daisy_solver_create(p._ctx, K, _fp(E), _fp(M), NMAT, _ip(mat), C.byref(s)) == -1, K  # DAISY_E_INVALID
    E, M, mat = make_inputs(N, 40, 2)
    for path in ("fp32", "ldg"):
        monkeypatch.setenv("DAISY_GATHER", path)
        s = C.c_void_p()
        assert L.daisy_solver_create(p._ctx, 40, _fp(E), _fp(M), NMAT, _ip(mat), C.byref(s)) == -1, path
        assert b"tensor-core" in L.daisy_last_error()
    E, M, mat = make_inputs(N, 64, 3)
    s = create_solver(p._ctx, 64, E, M, mat, monkeypatch)
    L.daisy_solver_destroy(s)
