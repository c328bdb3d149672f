"""Every gather kernel at sizes that do not divide its tiles, against an FP64 numpy pass.

The kernels (csrc/gather.cu, gather_mma.cuh) have edge logic that only runs when the sizes are ragged: a partial last row
block (64 rows, 32 for the FP32 K = 32 kernel, 128 for tcgen05), a last column step clipped by the F tensor map at ldF (N
rounded up to 32), residual columns between N and n (N rounded up to 4), stream-K grids smaller than the SM count with row
blocks shared by several CTAs, and padded band counts (K = 2 runs the K = 3 kernel, 4-8 run 9, 10-15 run 16, 17-31 run 32).
The matrices here are built tile by tile (64 x 256) so that a dropped or double-counted tile, or a wrong edge, moves the
results far beyond the 1e-5 tolerance.

Single GPU: contexts of any N (the first N triangles of a Cornell box), every kernel path, every band count class.
Partitions on one GPU: G contexts with rank g of G on device 0, exchanged by hand -- ragged and empty ranks.
Fused exchange with real peers (DeviceGroup, needs 2 / 8 GPUs): ranks that own few or no rows.
"""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import assert_rel

pytestmark = pytest.mark.gpu

SIZES = [1, 5, 63, 65, 127, 129, 255, 257, 1000, 2050, 6400, 7712]
KS = [1, 2, 5, 9, 13, 16, 23, 32]
ALL_K_SIZES = (257, 7712)
CASES = [(N, K) for N in SIZES for K in KS] + [(N, K) for N in ALL_K_SIZES for K in range(1, 33) if K not in KS]
NMAT = 13
PASSES = 3

# kernel paths: environment of daisy_solver_create, and what the solver must report (launches per pass, tile map or not)
#   K <= 9:  fused TMA kernel with tile skipping / dense stream-K / TMA kernel + separate epilogue / ldg kernel + epilogue
#   K >= 10: tcgen05 3xTF32 (+ residual split + epilogue) / fused FP32 TMA / FP32 TMA + separate epilogue / ldg
ENV_VARS = ("DAISY_GATHER", "DAISY_GATHER_EPI", "DAISY_GATHER_SKIP")
PATHS_NARROW = {
    "skip": ({}, 1, True),
    "dense": ({"DAISY_GATHER_SKIP": "0"}, 1, False),
    "split": ({"DAISY_GATHER_EPI": "split"}, 2, False),
    "ldg": ({"DAISY_GATHER": "ldg"}, 2, False),
}
PATHS_WIDE = {
    "mma": ({}, 3, False),
    "fp32": ({"DAISY_GATHER": "fp32"}, 1, False),
    "fp32_split": ({"DAISY_GATHER": "fp32", "DAISY_GATHER_EPI": "split"}, 2, False),
    "ldg": ({"DAISY_GATHER": "ldg"}, 2, False),
}


def paths_for(K):
    return PATHS_NARROW if K <= 9 else PATHS_WIDE


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


# ---- inputs --------------------------------------------------------------------------------------------------------
def make_matrix(N, seed):
    """N x N FP32 built at 64 x 256 tile granularity: about half the tiles occupied, a few whole zero row blocks and column
    steps, non-zeros guaranteed in row N-1, column N-1 (so in the last, partial, row block and column step); values in
    (0, 2/N)."""
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
    for rb, cs in zip(*np.nonzero(occ)):  # every occupied tile holds at least one entry
        r = rng.randint(rb * 64, min(N, rb * 64 + 64))
        c = rng.randint(cs * 256, min(N, cs * 256 + 256))
        F[r, c] = rng.uniform(0.5, 2.0) / N
    F[N - 1, N - 1] = 1.5 / N
    F[N - 1, rng.choice(free_cols, min(8, len(free_cols)))] = 1.0 / N
    F[rng.choice(free_rows, min(8, len(free_rows))), N - 1] = 1.0 / N
    return F


def tile_map(F, trows=64, tcols=256):
    N = F.shape[0]
    return np.array([[np.any(F[r:r + trows, c:c + tcols] != 0) for c in range(0, N, tcols)] for r in range(0, N, trows)])


def make_inputs(N, K, seed):
    """E positive in every band and column; 13 random non-symmetric K x K material matrices (contracting); a material per
    patch drawn independently of the mesh."""
    rng = np.random.RandomState(seed)
    E = np.ascontiguousarray(rng.uniform(0.5, 2.0, (K, N)).astype(np.float32))
    M = np.ascontiguousarray(rng.uniform(0, 0.9 / K, (NMAT, K, K)).astype(np.float32))
    mat = np.ascontiguousarray(rng.randint(0, NMAT, N).astype(np.int32))
    return E, M, mat


def _fp64_pass(F, R, B, M, mat):
    """residual <- M[mat] (F residual), B += residual, in FP64"""
    b = np.asarray(F, np.float64) @ R.T                  # N x K
    y = np.einsum("ijk,ij->ik", M.astype(np.float64)[mat], b)  # column-major K x K: y[k] = sum_j M[j, k] b[j]
    R = y.T.copy()
    return R, B + R, R.sum(axis=1)


def fp64_passes(F, E, M, mat, passes):
    R, B = E.astype(np.float64), E.astype(np.float64)
    out = []
    for _ in range(passes):
        R, B, sums = _fp64_pass(F, R, B, M, mat)
        out.append((R, B, sums))
    return out


def sub_scene(N):
    """The first N triangles of a Cornell box of 32 * ceil(N / 32) patches."""
    from daisyriot_b200 import scenes
    from daisyriot_b200.scenes import Scene
    sc = scenes.cornell_box(32 * math.ceil(N / 32))
    return Scene(sc.vertices, sc.normals, sc.tri[:N], sc.mat_idx[:N], sc.materials, "cornell_first_%d" % N)


# ---- solver helpers ----------------------------------------------------------------------------------------------------
def set_path(monkeypatch, env):
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def create_solver(ctx, K, E, M, mat, path, monkeypatch):
    env, launches, skip = paths_for(K)[path]
    set_path(monkeypatch, env)
    L = _L()
    s = C.c_void_p()
    _check(L.daisy_solver_create(ctx, K, _fp(E), _fp(M), M.shape[0], _ip(mat), C.byref(s)), "solver_create %s K=%d" % (path, K))
    dims = np.zeros(2, np.int32)
    _check(L.daisy_solver_tile_map(s, _ip(dims), None, 0, None, None))
    assert (dims[0] > 0) == skip, (path, K, dims)                     # tile skipping on exactly where intended
    assert L.daisy_solver_launches_per_pass(s) == launches, (path, K)  # fused / split / tcgen05 as intended
    return s


def read_guarded(s, K, nloc):
    """daisy_solver_read into buffers one band and a few columns larger, pre-filled with a sentinel that must survive."""
    L = _L()
    sentinel = np.float32(-7.25e30)
    bufB = np.full((K + 1) * (nloc + 3), sentinel, np.float32)
    bufR = np.full((K + 1) * (nloc + 3), sentinel, np.float32)
    _check(L.daisy_solver_read(s, _fp(bufB), _fp(bufR)))
    assert np.all(bufB[K * nloc:] == sentinel) and np.all(bufR[K * nloc:] == sentinel), "read wrote past K x nloc"
    return bufB[:K * nloc].reshape(K, nloc).copy(), bufR[:K * nloc].reshape(K, nloc).copy()


def run_passes(s, K, N, passes):
    L = _L()
    sums = []
    for _ in range(passes):
        t = np.zeros(K)
        _check(L.daisy_solver_step(s, _dp(t)), "solver_step")
        sums.append(t)
    B, R = read_guarded(s, K, N)
    return B, R, sums


def compare(B, R, sums, ref, what):
    Rw, Bw, Sw = ref
    for k in range(B.shape[0]):
        assert_rel(R[k], Rw[k], (what, "residual", k))
        assert_rel(B[k], Bw[k], (what, "B", k))
    assert np.allclose(sums, Sw, rtol=1e-5, atol=0), (what, "band sums", sums, Sw)


# ---- fixtures ----------------------------------------------------------------------------------------------------------
class _Contexts:
    """One context per N (and per partition), F loaded from make_matrix, built on first use."""

    def __init__(self):
        self.single, self.parts, self.F, self.F64 = {}, {}, {}, {}

    def matrix(self, N):
        if N not in self.F:
            self.F[N] = make_matrix(N, 1000 + N)
            self.F64[N] = self.F[N].astype(np.float64)
        return self.F[N]

    def get(self, N):
        import daisyriot_b200 as dz
        from daisyriot_b200 import scenes
        if N not in self.single:
            p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sub_scene(N)), device=0, rands=scenes.msvc_sample_pattern(1))
            assert p.row_range == (0, N)
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
        """inputs of case (N, K) and the FP64 results of its first passes"""
        E, M, mat = make_inputs(N, K, 7 * N + K)
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


# ---- 1. single GPU ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,K", CASES)
def test_every_path_vs_fp64(contexts, N, K, monkeypatch):
    """3 passes with band sums on every kernel path: B, residual and band sums against FP64; the same passes again from
    daisy_solver_reset are bit-identical; the tile map of the skip plan is exactly the matrix's."""
    L = _L()
    p, F = contexts.get(N)
    E, M, mat, ref = contexts.reference(N, K)
    for path in paths_for(K):
        what = (N, K, path)
        s = create_solver(p._ctx, K, E, M, mat, path, monkeypatch)
        try:
            if path == "skip":
                want = tile_map(np.pad(F, ((0, 0), (0, (-N) % 32))))  # the map covers the F tensor map: ldF columns
                dims = np.zeros(2, np.int32)
                occ = np.zeros(want.size, np.uint8)
                occupied = C.c_int64()
                _check(L.daisy_solver_tile_map(s, _ip(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, C.byref(occupied), None))
                assert tuple(dims) == want.shape and np.array_equal(occ.reshape(want.shape).astype(bool), want), what
                assert occupied.value == want.sum(), what
            B, R, sums = run_passes(s, K, N, PASSES)
            for i in range(PASSES):
                assert np.allclose(sums[i], ref[i][2], rtol=1e-5, atol=0), (what, "band sums of pass", i, sums[i], ref[i][2])
            compare(B, R, sums[-1], ref[-1], what)
            _check(L.daisy_solver_reset(s))
            B2, R2, sums2 = run_passes(s, K, N, PASSES)
            assert np.array_equal(B2.view(np.uint32), B.view(np.uint32)) and np.array_equal(R2.view(np.uint32), R.view(np.uint32)), (what, "not deterministic")
            assert all(np.array_equal(a, b) for a, b in zip(sums, sums2)), (what, "band sums not deterministic")
        finally:
            L.daisy_solver_destroy(s)


@pytest.mark.parametrize("N", [65, 7712])
@pytest.mark.parametrize("K", [1, 9])
@pytest.mark.parametrize("path", ["skip", "dense"])
def test_fused_chained_is_bit_identical(contexts, N, K, path, monkeypatch):
    """The fused kernel's chained passes (programmatic dependent launch, no events in between) give the very same bits."""
    L = _L()
    p, F = contexts.get(N)
    E, M, mat, ref = contexts.reference(N, K)
    got = {}
    for chained in (0, 1):
        s = create_solver(p._ctx, K, E, M, mat, path, monkeypatch)
        _check(L.daisy_solver_set_chained(s, chained))
        for _ in range(PASSES):
            _check(L.daisy_solver_step(s, None))
        sums = np.zeros(K)
        _check(L.daisy_solver_band_sums(s, _dp(sums)))
        B, R = read_guarded(s, K, N)
        got[chained] = (B, R, sums)
        L.daisy_solver_destroy(s)
    for a, b in zip(got[0], got[1]):
        assert np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b), (N, K, path)
    compare(*got[1], ref[-1], (N, K, path, "chained"))


@pytest.mark.parametrize("N", [65, 7712])
@pytest.mark.parametrize("K", [3, 32])
@pytest.mark.parametrize("per_band", [0, 1])
def test_converge_pass_count(contexts, N, K, per_band, monkeypatch):
    """daisy_solver_converge stops after as many passes as FP64 does; the threshold is the geometric mean of two consecutive
    FP64 values of the stop quantity, so no decision sits within rounding."""
    L = _L()
    p, F = contexts.get(N)
    E, M, mat, ref = contexts.reference(N, K, 12)
    stat = (lambda s: float(np.max(s))) if per_band else (lambda s: float(np.sum(s)))
    vals = [stat(E.astype(np.float64).sum(axis=1))] + [stat(r[2]) for r in ref]
    assert all(b < a for a, b in zip(vals, vals[1:]))
    j = 4
    thr = math.sqrt(vals[j] * vals[j + 1])
    want = next(i for i, v in enumerate(vals) if v <= thr)
    assert want == j + 1 and min(abs(v / thr - 1) for v in vals) > 1e-3
    for path in paths_for(K):
        s = create_solver(p._ctx, K, E, M, mat, path, monkeypatch)
        n = C.c_int()
        _check(L.daisy_solver_converge(s, thr, per_band, 100, C.byref(n)))
        assert n.value == want, (N, K, per_band, path, n.value, want)
        L.daisy_solver_destroy(s)


@pytest.mark.parametrize("N", [257, 1000])
@pytest.mark.parametrize("K", [5, 23])
def test_write_then_pass_then_reset(contexts, N, K, monkeypatch):
    """daisy_solver_write with arbitrary B and residual, one pass against FP64 from those values, then reset gives back
    exactly E."""
    L = _L()
    p, F = contexts.get(N)
    E, M, mat, _ = contexts.reference(N, K)
    rng = np.random.RandomState(N + K)
    Bw = np.ascontiguousarray(rng.uniform(0, 3, (K, N)).astype(np.float32))
    Rw = np.ascontiguousarray(rng.uniform(0.1, 1, (K, N)).astype(np.float32))
    want = _fp64_pass(contexts.F64[N], Rw.astype(np.float64), Bw.astype(np.float64), M, mat)
    for path in paths_for(K):
        s = create_solver(p._ctx, K, E, M, mat, path, monkeypatch)
        _check(L.daisy_solver_step(s, None))  # something in the buffers before the write
        _check(L.daisy_solver_write(s, _fp(Bw), _fp(Rw)))
        sums = np.zeros(K)
        _check(L.daisy_solver_band_sums(s, _dp(sums)))
        assert np.allclose(sums, Rw.astype(np.float64).sum(axis=1), rtol=1e-12), (N, K, path)
        _check(L.daisy_solver_step(s, _dp(sums)))
        B, R = read_guarded(s, K, N)
        compare(B, R, sums, want, (N, K, path, "after write"))
        _check(L.daisy_solver_reset(s))
        B0, R0 = read_guarded(s, K, N)
        assert np.array_equal(B0, E) and np.array_equal(R0, E), (N, K, path, "reset")
        L.daisy_solver_destroy(s)


# ---- 2. partitions on one GPU ------------------------------------------------------------------------------------------
PARTITIONS = [(300, 2), (200, 2), (6400, 8)]
PART_KS = [1, 2, 5, 9, 13, 32]


def _exchange_views(solvers):
    """torch views of every rank's next exchange buffer (as dist.py aliases them), and the block length in floats"""
    import torch
    from daisyriot_b200.dist import _DevMem
    L = _L()
    views, blk = [], None
    for s in solvers:
        ptr, b, tot = C.c_void_p(), C.c_int64(), C.c_int64()
        _check(L.daisy_solver_exchange_info(s, C.byref(ptr), C.byref(b), C.byref(tot)))
        views.append(torch.as_tensor(_DevMem(ptr.value, tot.value), device="cuda:0"))
        blk = b.value // 4
    return views, blk


@pytest.mark.parametrize("N,G", PARTITIONS)
@pytest.mark.parametrize("K", PART_KS)
def test_partition_on_one_gpu(contexts, N, G, K, monkeypatch):
    """G ranks on device 0, driven by step_local / hand exchange / step_finish: the concatenated B, the residual and the
    totals equal FP64, including ranks with a partial last row block and ranks that own no rows."""
    import torch
    L = _L()
    ps, F = contexts.partition(N, G)
    ranges = [p.row_range for p in ps]
    n = -(-N // G)
    n = -(-n // 256) * 256
    assert ranges == [(min(N, g * n), min(N, (g + 1) * n)) for g in range(G)]
    E, M, mat, ref = contexts.reference(N, K)
    for path in paths_for(K):
        what = (N, G, K, path)
        solvers = [create_solver(p._ctx, K, E, M, mat, path, monkeypatch) for p in ps]
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
                    assert np.allclose(t, ref[it][2], rtol=1e-5, atol=0), (what, "band sums of pass", it, "rank", g)
            B = np.zeros((K, N), np.float32)
            R = np.zeros((K, N), np.float32)
            for (r0, r1), s in zip(ranges, solvers):
                if r1 > r0:
                    B[:, r0:r1], R[:, r0:r1] = read_guarded(s, K, r1 - r0)
            compare(B, R, t, ref[-1], what)
        finally:
            torch.cuda.synchronize(0)
            for s in solvers:
                L.daisy_solver_destroy(s)


# ---- 3. fused exchange with real peers ---------------------------------------------------------------------------------
@pytest.mark.parametrize("N,G", [(224, 2), (288, 2), ("colorballs", 8)])
@pytest.mark.parametrize("K", [1, 3, 9, 16])
def test_fused_exchange_small_and_empty_ranks(contexts, fixture_scenes, N, G, K, monkeypatch):
    """DeviceGroup on G GPUs where the last rank owns few (N = 288: 32 rows) or no rows (N = 224; colorballs on 8 GPUs:
    rank 7).  Such a rank must still publish every pass -- or its peers wait for its flag until the exchange times out."""
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    L = _L()
    if L.daisy_device_count() < G:
        pytest.skip("needs %d GPUs" % G)
    monkeypatch.setenv("DAISY_EXCHANGE_TIMEOUT_MS", "20000")
    set_path(monkeypatch, {})
    sc = fixture_scenes["colorballs"] if N == "colorballs" else sub_scene(N)
    N = sc.numtriangles
    uv = scenes.msvc_sample_pattern(1)
    mesh = dz.MeshS.from_scene(sc)
    F = make_matrix(N, 2000 + N)
    E, M, mat = make_inputs(N, K, 11 * N + K)
    ref = fp64_passes(F, E, M, mat, PASSES)
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv)
    grp = dz.DeviceGroup(mesh, devices=list(range(G)), rands=uv)
    try:
        if N == 224 and K == 1:  # the group's own build with an empty rank equals one GPU's, bit for bit
            F1 = p.cudaCalculateRadiosityMatrix().rows()
            F2 = grp.cudaCalculateRadiosityMatrix().rows()
            assert np.array_equal(F2.view(np.uint32), F1.view(np.uint32))
        p.loadRadiosityMatrix(F)
        from daisyriot_b200 import _lib
        _check(L.daisy_group_formfactors_write_rows(grp._g, 0, N, _lib.fptr(F)))
        s = create_solver(p._ctx, K, E, M, mat, next(iter(paths_for(K))), monkeypatch)
        gs = dz.GroupSolver(grp, K, E, M, mat)
        for it in range(PASSES):
            t = np.zeros(K)
            _check(L.daisy_solver_step(s, _dp(t)))
            got = gs.step(True)
            assert np.allclose(got, ref[it][2], rtol=1e-5, atol=0) and np.allclose(got, t, rtol=1e-6, atol=0), (N, G, K, it)
        B2, R2 = gs.read()
        compare(B2, R2, got, ref[-1], (N, G, K, "group"))
        for _ in range(10):
            gs.step(False)
            _check(L.daisy_solver_step(s, None))
        B1, R1 = read_guarded(s, K, N)
        B2, R2 = gs.read()
        for k in range(K):
            assert_rel(B2[k], B1[k], (N, G, K, "B group vs one GPU", k))
            assert_rel(R2[k], R1[k], (N, G, K, "residual group vs one GPU", k))
        _check(L.daisy_solver_reset(s))
        gs.reset()
        thr = 1e-3 * float(E.sum())
        n1 = C.c_int()
        _check(L.daisy_solver_converge(s, thr, 0, 200, C.byref(n1)))
        assert gs.converge(thr, False, 200) == n1.value and n1.value > 2
        gs.close()
        L.daisy_solver_destroy(s)
    finally:
        grp.close()
        p.close()
