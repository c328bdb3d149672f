"""Every entry point on a caller's non-blocking stream, and two contexts driven from two host threads.

PyTorch creates its side streams non-blocking: they take no ordering from the legacy default stream.  A context bound to one
(OptixPrimeFunctionality(..., stream=...) -> daisy_ctx_set_stream) must still see every upload it made before the kernels
that read it, and a context's sample pattern must be its own while another context on the same device builds with another.

The reference of each case is the same call sequence on a twin context on the default stream, compared bit for bit (F,
masks, hits, frames, CSC arrays, B, residual, band sums); the small scenes are also compared with the oracle's brute force,
the solver with the FP64 passes of test_gpu_gather_shapes.  A race may be won by luck on any one run, so
test_streams_host.py checks the properties these tests rely on in the library and the sources as well."""
import ctypes as C
import threading

import numpy as np
import pytest

import geometry_scenes as gs
from oracle.pyoracle import Oracle
from test_gpu_far_geometry import _assert_same_hits
from test_gpu_gather_shapes import compare, create_solver, fp64_passes, make_inputs, make_matrix, paths_for, sub_scene

pytestmark = pytest.mark.gpu

FFD, FFH = 0, 1


@pytest.fixture(scope="module")
def dz():
    import daisyriot_b200 as dz
    dz.lib()  # raises if libdaisy_b200.so is missing: no CPU fallback
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    return dz


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


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(-1)


def _assert_bits(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape, got.dtype, want.dtype)
    bad = _bits(got) != _bits(want)
    assert not bad.any(), (what, int(bad.sum()), "bytes differ")


def _side_stream():
    import torch
    return torch.cuda.Stream(device=0)


def _ctx(dz, sc, uv, stream=None):
    """a context on `stream` (a torch.cuda.Stream, kept alive with the context) or on the default stream"""
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv, stream=None if stream is None else stream.cuda_stream)
    p._torch_stream = stream
    return p


def _twins(dz, sc, uv):
    """(context on a fresh non-blocking stream, twin on the default stream)"""
    return _ctx(dz, sc, uv, _side_stream()), _ctx(dz, sc, uv)


def _both(fn, ps, ref, what):
    """fn on both twins: bit-identical, and returned"""
    got, want = fn(ps), fn(ref)
    if isinstance(got, tuple):
        for i, (g, w) in enumerate(zip(got, want)):
            _assert_bits(g, w, (what, i))
    else:
        _assert_bits(got, want, what)
    return got


def _build(p, variant):
    return (p.cudaCalculateRadiosityMatrix() if variant == FFD else p.calculateRadiosityMatrix()).rows()


def _scene(name):
    from daisyriot_b200 import scenes
    return scenes.cornell_box(512) if name == "cornell512" else gs.irregular_walls(1)


def _sleep_cycles(ms):
    """cycles of torch.cuda._sleep that take about `ms` on device 0 (SM clock as the device reports it, else 2 GHz)"""
    import torch
    khz = getattr(torch.cuda.get_device_properties(0), "clock_rate", 0) or 2_000_000
    return int(ms * khz)


# ---- geometry and queries ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [FFD, FFH])
@pytest.mark.parametrize("name", ["cornell512", "irregular_walls"])
def test_geometry_queries_on_a_side_stream(dz, uv50, name, variant):
    import torch
    from daisyriot_b200 import api
    from daisyriot_b200.api import HIT_DTYPE
    sc = _scene(name)
    N = sc.numtriangles
    ps, ref = _twins(dz, sc, uv50)
    F = _both(lambda p: _build(p, variant), ps, ref, "F")
    orc = Oracle.from_scene(sc)
    if variant == FFD:
        F_brute, masks_brute = orc.radmat_rows(uv50, 0, N, brute=True)[:2]
        _assert_bits(F, F_brute, "F vs brute force")
    # masks over ragged row windows
    for r0, nr in ((0, 37), (129, 70), (N - 5, 5)):
        m = _both(lambda p: p.visibilityMasks(r0, nr, variant=variant), ps, ref, ("masks", r0, nr))
        if variant == FFD:
            _assert_bits(m, masks_brute[r0:r0 + nr], ("masks vs brute force", r0, nr))
    _both(lambda p: p.runCalculateRadiosityMatrix(3, 61, variant=variant), ps, ref, "daisy_unoccluded_rows")
    _both(lambda p: p.runCalculateRadiosityMatrix(N - 40, 40, variant=variant), ps, ref, "daisy_unoccluded_rows, last rows")
    _both(lambda p: dz.RadMat(p).rows(5, 77), ps, ref, "read rows")
    _both(lambda p: dz.RadMat(p).row_digest(), ps, ref, "row digests")
    # closest hit: host buffers, then torch tensors allocated on the context's stream
    rays = gs.closest_hit_rays(sc, 4)
    n = rays.shape[0]
    hits = _both(lambda p: p.optixQuery(n, rays), ps, ref, "optixQuery")
    _assert_same_hits(hits, orc.query_closest(rays, brute=True), "optixQuery vs brute force")
    with torch.cuda.stream(ps._torch_stream):
        d_rays = torch.from_numpy(rays).to("cuda")
        d_hits = torch.full((n, 4), -7.0, dtype=torch.float32, device="cuda")
    ps._torch_stream.synchronize()
    _check(_L().daisy_query_closest_device(ps._ctx, n, C.c_void_p(d_rays.data_ptr()), C.c_void_p(d_hits.data_ptr())), "closest_device")
    with torch.cuda.stream(ps._torch_stream):
        got = d_hits.cpu().numpy().view(HIT_DTYPE).reshape(n)
    _assert_bits(got, hits, "daisy_query_closest_device")
    # traceScreen with hit records
    cam = api.Camera(37, 29, 4)
    cam.eye = np.array([2.75, 2.75, 14.0], np.float32) if name == "cornell512" else np.asarray(sc.vertices.mean(0) + [0, 0, 9], np.float32)
    cam.dir = np.asarray(sc.vertices.mean(0), np.float32)
    colors = np.random.RandomState(2).uniform(0, 1.2, (N, 3)).astype(np.float32)
    _both(lambda p: api.traceScreen(p, cam, colors, True, True, return_hits=True), ps, ref, "traceScreen")
    ps.close(); ref.close()


# ---- geometry changes ------------------------------------------------------------------------------------------------------
def test_move_then_update_matches_fresh_build(dz, uv50, cornell512):
    from daisyriot_b200 import scenes
    from test_gpu_geometry_update import _scene_with
    sc = cornell512
    V, VN = scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0))
    ps, ref = _twins(dz, sc, uv50)
    _both(lambda p: _build(p, FFD), ps, ref, "F before")
    for p in (ps, ref):
        p.updateGeometry(V, VN)
    F = _both(lambda p: p.updateRadiosityMatrix(FFD).rows(), ps, ref, "F after the move")
    assert ps.update_stats()["pairs_retraced"] == ref.update_stats()["pairs_retraced"]
    fresh = _ctx(dz, _scene_with(sc, V, VN), uv50)
    _assert_bits(F, _build(fresh, FFD), "updated vs fresh build")
    fresh.close(); ps.close(); ref.close()


def test_replace_mesh_then_update_matches_fresh_build(dz, uv50, cornell512):
    from test_gpu_mesh_edit import _edit
    sc = cornell512
    sc_new, prev = _edit(sc, "insert_panel")
    ps, ref = _twins(dz, sc, uv50)
    _both(lambda p: _build(p, FFD), ps, ref, "F before")
    for p in (ps, ref):
        p.replaceMesh(dz.MeshS.from_scene(sc_new), prev)
    _both(lambda p: dz.RadMat(p).rows(), ps, ref, "F remapped")
    F = _both(lambda p: p.updateRadiosityMatrix(FFD).rows(), ps, ref, "F after the edit")
    fresh = _ctx(dz, sc_new, uv50)
    _assert_bits(F, _build(fresh, FFD), "edited vs fresh build")
    _assert_bits(ps.visibilityMasks(0, 50), fresh.visibilityMasks(0, 50), "masks after the edit")
    fresh.close(); ps.close(); ref.close()


# ---- matrix cache ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stage", [None, "65536"])
def test_matrix_cache_on_a_side_stream(dz, uv50, cornell2048, stage, monkeypatch):
    """to_csc, write_csc resident (default staging) and chunked (64 KB staging), then write_rows"""
    if stage is None:
        monkeypatch.delenv("DAISY_CSC_STAGE_BYTES", raising=False)
    else:
        monkeypatch.setenv("DAISY_CSC_STAGE_BYTES", stage)
    sc = cornell2048
    ps, ref = _twins(dz, sc, uv50)
    F = _both(lambda p: _build(p, FFD), ps, ref, "F")
    vals, inner, outer = _both(lambda p: dz.RadMat(p).to_csc(), ps, ref, "to_csc")
    qs, qref = _twins(dz, sc, uv50)
    _both(lambda p: p.loadRadiosityMatrixCSC(vals, inner, outer).rows(), qs, qref, "write_csc")
    _assert_bits(dz.RadMat(qs).rows(), F, "write_csc round trip")
    G = make_matrix(sc.numtriangles, 5)
    _both(lambda p: p.loadRadiosityMatrix(G).rows(), qs, qref, "write_rows")
    _assert_bits(dz.RadMat(qs).rows(), G, "write_rows round trip")
    for p in (ps, ref, qs, qref):
        p.close()


# ---- solver -----------------------------------------------------------------------------------------------------------------
class _Solver:
    def __init__(self, p, K, E, M, mat, path, monkeypatch):
        self.p, self.K, self.N = p, K, E.shape[1]
        self.s = create_solver(p._ctx, K, E, M, mat, path, monkeypatch)

    def state(self):
        B, R = np.empty((self.K, self.N), np.float32), np.empty((self.K, self.N), np.float32)
        _check(_L().daisy_solver_read(self.s, _fp(B), _fp(R)), "read")
        sums = np.zeros(self.K)
        _check(_L().daisy_solver_band_sums(self.s, _dp(sums)), "band_sums")
        return B, R, sums, np.array([_L().daisy_solver_numpasses(self.s)])

    def step(self, want_sums=True):
        t = np.zeros(self.K)
        _check(_L().daisy_solver_step(self.s, _dp(t) if want_sums else None), "step")
        return t

    def converge(self, device, thr, per_band, max_passes):
        n = C.c_int(-1)
        fn = _L().daisy_solver_converge_device if device else _L().daisy_solver_converge
        _check(fn(self.s, float(thr), int(per_band), int(max_passes), C.byref(n)), "converge")
        return np.array([n.value])

    def close(self):
        _L().daisy_solver_destroy(self.s)


class _Twin:
    """a solver on the side-stream context and one on its default-stream twin, driven alike and compared after every call"""

    def __init__(self, ps, ref, K, E, M, mat, path, monkeypatch):
        self.a = _Solver(ps, K, E, M, mat, path, monkeypatch)
        self.b = _Solver(ref, K, E, M, mat, path, monkeypatch)

    def both(self, fn, what):
        x, y = fn(self.a), fn(self.b)
        if x is not None:
            _assert_bits(np.asarray(x), np.asarray(y), (what, "returned"))
        sa, sb = self.a.state(), self.b.state()
        for i, (u, v) in enumerate(zip(sa, sb)):
            _assert_bits(u, v, (what, ("B", "residual", "band sums", "numpasses")[i]))
        return sa

    def close(self):
        self.a.close(); self.b.close()


class _SolverContexts:
    """per N: the side-stream context and its twin, both holding make_matrix(N)"""

    def __init__(self):
        self.ctx, self.F = {}, {}

    def get(self, dz, N):
        from daisyriot_b200 import scenes
        if N not in self.ctx:
            self.F[N] = make_matrix(N, 1000 + N)
            ps, ref = _twins(dz, sub_scene(N), scenes.msvc_sample_pattern(1))
            for p in (ps, ref):
                p.loadRadiosityMatrix(self.F[N])
            self.ctx[N] = (ps, ref)
        return self.ctx[N] + (self.F[N],)

    def close(self):
        for ps, ref in self.ctx.values():
            ps.close(); ref.close()


@pytest.fixture(scope="module")
def solver_ctxs():
    c = _SolverContexts()
    yield c
    c.close()


SOLVER_CASES = [(N, K, path) for N in (2050, 7712) for K in (1, 3, 9, 16, 32, 64) for path in paths_for(K) if K <= 32 or path == "mma"]


@pytest.mark.parametrize("N,K,path", SOLVER_CASES)
def test_solver_on_a_side_stream(dz, solver_ctxs, N, K, path, monkeypatch):
    ps, ref, F = solver_ctxs.get(dz, N)
    E, M, mat = make_inputs(N, K, 7 * N + K)
    t = _Twin(ps, ref, K, E, M, mat, path, monkeypatch)
    what = (N, K, path)
    # three passes with band sums, against FP64 too
    for i, (Rw, Bw, Sw) in enumerate(fp64_passes(F.astype(np.float64), E, M, mat, 3)):
        sums = t.both(lambda s: s.step(), (what, "pass", i))[2]
    B, R = t.a.state()[:2]
    compare(B, R, sums, (Rw, Bw, Sw), what)
    # chained passes issued without band sums
    for s in (t.a, t.b):
        _check(_L().daisy_solver_set_chained(s.s, 1), "set_chained")
    t.both(lambda s: [s.step(False) for _ in range(3)][-1], (what, "chained"))
    for s in (t.a, t.b):
        _check(_L().daisy_solver_set_chained(s.s, 0), "set_chained")
    thr = float(np.sum(sums)) * 0.05
    t.both(lambda s: s.converge(False, thr, 0, 6), (what, "converge"))
    t.both(lambda s: s.converge(True, thr * 0.2, 1, 6), (what, "converge_device"))
    t.both(lambda s: _check(_L().daisy_solver_restart(s.s, None), "restart"), (what, "restart"))
    t.both(lambda s: s.step(), (what, "pass after restart"))
    E2, M2, mat2 = make_inputs(N, K, 7 * N + K + 1)
    t.both(lambda s: _check(_L().daisy_solver_set_emission(s.s, _fp(E2)), "set_emission"), (what, "set_emission"))
    t.both(lambda s: _check(_L().daisy_solver_restart(s.s, None), "restart"), (what, "restart after set_emission"))
    t.both(lambda s: _check(_L().daisy_solver_set_materials(s.s, _fp(M2), M2.shape[0], _ip(mat2)), "set_materials"), (what, "set_materials"))
    t.both(lambda s: s.step(), (what, "pass after set_materials"))
    # F replaced under a live solver: the next pass rescans it and uploads a new tile plan
    G = make_matrix(N, 2000 + N)
    for p in (ps, ref):
        p.loadRadiosityMatrix(G)
    t.both(lambda s: _check(_L().daisy_solver_reset(s.s), "reset"), (what, "reset"))
    for i, (Rw, Bw, Sw) in enumerate(fp64_passes(G.astype(np.float64), E2, M2, mat2, 2)):
        sums = t.both(lambda s: s.step(), (what, "pass on the new F", i))[2]
    B, R = t.a.state()[:2]
    compare(B, R, sums, (Rw, Bw, Sw), (what, "new F"))
    t.close()
    for p in (ps, ref):
        p.loadRadiosityMatrix(F)


def test_switching_streams_mid_solve(dz, solver_ctxs, monkeypatch):
    """stream A -> stream B -> default stream under one solver: the passes do not change"""
    N, K = 2050, 9
    ps, ref, F = solver_ctxs.get(dz, N)
    E, M, mat = make_inputs(N, K, 11)
    t = _Twin(ps, ref, K, E, M, mat, "skip", monkeypatch)
    t.both(lambda s: s.step(), "stream A")
    sb = _side_stream()
    _check(_L().daisy_ctx_set_stream(ps._ctx, C.c_void_p(sb.cuda_stream)), "set_stream B")
    t.both(lambda s: [s.step() for _ in range(2)][-1], "stream B")
    t.both(lambda s: s.converge(True, 1e-3, 0, 4), "stream B, converge_device")
    _check(_L().daisy_ctx_set_stream(ps._ctx, None), "set_stream default")
    t.both(lambda s: [s.step() for _ in range(2)][-1], "default stream")
    _check(_L().daisy_ctx_set_stream(ps._ctx, C.c_void_p(ps._torch_stream.cuda_stream)), "set_stream A")
    t.both(lambda s: s.step(), "stream A again")
    t.close()


# ---- ordering with the caller's own work ----------------------------------------------------------------------------------
def test_call_waits_for_the_callers_work_on_its_stream(dz, uv50, cornell512):
    """The caller's stream is busy (~50 ms sleep), then a torch copy writes the rays; the call, made at once, must trace the
    written rays.  Its hits are then read by torch work enqueued after it returns, with no synchronisation in between."""
    import torch
    from daisyriot_b200.api import HIT_DTYPE
    sc = cornell512
    rays = gs.closest_hit_rays(sc, 9)
    n = rays.shape[0]
    want = Oracle.from_scene(sc).query_closest(rays, brute=True)
    p = _ctx(dz, sc, uv50, _side_stream())
    s = p._torch_stream
    src = torch.from_numpy(rays).to("cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        d_rays = torch.zeros((n, 6), dtype=torch.float32, device="cuda")  # rays that hit nothing
        d_hits = torch.full((n, 4), -7.0, dtype=torch.float32, device="cuda")
        torch.cuda._sleep(_sleep_cycles(50))
        d_rays.copy_(src)
        _check(_L().daisy_query_closest_device(p._ctx, n, C.c_void_p(d_rays.data_ptr()), C.c_void_p(d_hits.data_ptr())), "closest_device")
        on_stream = d_hits.clone()
    on_default = d_hits.clone()  # the current stream outside the block: torch's default stream
    torch.cuda.synchronize()
    _assert_same_hits(on_stream.cpu().numpy().view(HIT_DTYPE).reshape(n), want, "hits read on the context's stream")
    _assert_same_hits(on_default.cpu().numpy().view(HIT_DTYPE).reshape(n), want, "hits read on the default stream")
    p.close()


# ---- two contexts, two host threads ---------------------------------------------------------------------------------------
def _sequence(dz, sc, uv, V):
    """build -> masks -> move + update -> solver passes on a fresh side-stream context; every result"""
    p = _ctx(dz, sc, uv, _side_stream())
    out = [_build(p, FFD), p.visibilityMasks(0, min(sc.numtriangles, 150))]
    p.updateGeometry(V, None)
    out.append(p.updateRadiosityMatrix(FFD).rows())
    K = 3
    E, M, mat = make_inputs(sc.numtriangles, K, 3)
    s = C.c_void_p()
    _check(_L().daisy_solver_create(p._ctx, K, _fp(E), _fp(M), M.shape[0], _ip(mat), C.byref(s)), "solver_create")
    for _ in range(3):
        t = np.zeros(K)
        _check(_L().daisy_solver_step(s, _dp(t)), "step")
        out.append(t)
    B, R = np.empty((K, sc.numtriangles), np.float32), np.empty((K, sc.numtriangles), np.float32)
    _check(_L().daisy_solver_read(s, _fp(B), _fp(R)), "read")
    out += [B, R]
    _L().daisy_solver_destroy(s)
    p.close()
    return out


def test_two_contexts_two_threads(dz, uv50):
    """Different scenes and sample patterns (S = 50, and S = 37 with samples on the edges, which changes the inner / edge
    permutation), each context on its own stream and host thread: every result as when the sequence runs alone."""
    from daisyriot_b200 import scenes
    a = scenes.cornell_box(512)
    b = gs.irregular_walls(1)
    jobs = [(a, np.ascontiguousarray(uv50), gs.lifted(a, 40)), (b, np.ascontiguousarray(gs.edge_pattern(uv50)[:37]), gs.lifted(b, 11))]
    alone = [_sequence(dz, *j) for j in jobs]
    for rnd in range(3):
        res, err = [None, None], [None, None]

        def run(i):
            try:
                res[i] = _sequence(dz, *jobs[i])
            except BaseException as e:  # re-raised in the main thread
                err[i] = e

        th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        for i in range(2):
            if err[i] is not None:
                raise err[i]
            for k, (g, w) in enumerate(zip(res[i], alone[i])):
                _assert_bits(np.asarray(g), np.asarray(w), ("round", rnd, "context", i, "result", k))
