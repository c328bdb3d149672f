"""Warm restart of the gather solver (daisy_solver_restart, the emission / material setters, restart mode's |r| band sums).

A restart pass streams F once with B_old as its input: B = E + M F B_old, residual = B - B_old.  The cases check that identity
bit for bit on every kernel path, the FP64 value of B, the padded bands, the fixed point of a converged solve, warm solves after
geometry moves, emission and material changes and mesh edits against cold solves of the new inputs, the device converge
against the host loop, the way back to the cold path, the refusals, and the multi-GPU forms.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, assert_rel
from test_gpu_gather_shapes import make_inputs, paths_for, set_path

pytestmark = pytest.mark.gpu

E_INVALID, E_STATE = -1, -3
N_BOX = 2048
WL = np.array([330, 350, 370, 450, 550, 650], np.float32)  # UV bands under the lamp's bell curve + three visible ones


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


def padded_K(K):
    from daisyriot_b200 import dist
    return dist.padded_K(K)


@pytest.fixture(scope="module")
def box(uv50):
    """Cornell box of 2048 patches with its form factors built, and F read back"""
    import daisyriot_b200 as dz
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    sc = dz.cornell_box(N_BOX)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv50)
    F = p.cudaCalculateRadiosityMatrix().rows()
    yield sc, p, F
    p.close()


class Solver:
    """a raw daisy_solver on a context, created under the given kernel-path environment"""

    def __init__(self, p, K, E, M, mat):
        self.K, self.N = K, E.shape[1]
        self.E, self.M, self.mat = E, M, mat
        self.s = C.c_void_p()
        _check(_L().daisy_solver_create(p._ctx, K, _fp(E), _fp(M), M.shape[0], _ip(mat), C.byref(self.s)), "create")

    def restart(self, B0=None):
        b = None if B0 is None else np.ascontiguousarray(B0, np.float32)
        return _L().daisy_solver_restart(self.s, None if b is None else _fp(b))

    def read(self):
        B, R = np.empty((self.K, self.N), np.float32), np.empty((self.K, self.N), np.float32)
        _check(_L().daisy_solver_read(self.s, _fp(B), _fp(R)), "read")
        return B, R

    def sums(self):
        out = np.zeros(self.K)
        _check(_L().daisy_solver_band_sums(self.s, _dp(out)), "band_sums")
        return out

    def step(self):
        out = np.zeros(self.K)
        _check(_L().daisy_solver_step(self.s, _dp(out)), "step")
        return out

    def converge(self, thr, per_band, on_device=False, max_passes=0):
        n = C.c_int(-1)
        fn = _L().daisy_solver_converge_device if on_device else _L().daisy_solver_converge
        _check(fn(self.s, float(thr), int(per_band), int(max_passes), C.byref(n)), "converge")
        return n.value

    @property
    def numpasses(self):
        return int(_L().daisy_solver_numpasses(self.s))

    def state(self):
        B, R = self.read()
        return B, R, self.sums(), self.numpasses

    def close(self):
        _L().daisy_solver_destroy(self.s)


def fp64_restart(F, B0, E, M, mat):
    """E + M F B0 in FP64 (column-major K x K per material), K x N"""
    b = np.asarray(F, np.float64) @ np.asarray(B0, np.float64).T            # N x K
    y = np.einsum("ijk,ij->ik", M.astype(np.float64)[mat], b)              # y[i, k] = sum_j M[mat_i][j, k] b[i, j]
    return E.astype(np.float64) + y.T


def ulp(x):
    x = np.abs(np.asarray(x, np.float32))
    return np.spacing(x).astype(np.float64)


def lamp_inputs(sc, K, seed, ev=7.0):
    """E on the lamp's patches, random contracting material matrices (the smoke test's kind of input)"""
    rng = np.random.RandomState(seed)
    M = rng.uniform(0, 0.5 / K, (len(sc.materials), K, K)).astype(np.float32)
    E = np.zeros((K, sc.numtriangles), np.float32)
    E[:, sc.mat_idx == 0] = ev
    return E, M, np.ascontiguousarray(sc.mat_idx, np.int32)


def exchange_block(s, K, n):
    """this rank's block of the buffer daisy_solver_exchange_info names, read from the device: (Kp x n body)"""
    import torch
    from daisyriot_b200.dist import _DevMem
    ptr, blk, tot = C.c_void_p(), C.c_int64(), C.c_int64()
    _check(_L().daisy_solver_exchange_info(s, C.byref(ptr), C.byref(blk), C.byref(tot)))
    host = torch.as_tensor(_DevMem(ptr.value, tot.value), device="cuda").cpu().numpy()
    Kp = padded_K(K)
    return host[:Kp * n].reshape(Kp, n)


def converge_tolerance(sums_traj, thr, B):
    """largest per-band distance of two solutions that each stopped at a band sum <= thr: the untaken tail of the residual
    series (thr rho / (1 - rho)) of both, plus the FP32 floor -- increments below half an ulp of B are lost, up to
    ulp(B) / (1 - rho) per entry over both solutions; rho = the cold solve's contraction over its last passes"""
    a = np.array([float(np.max(s)) for s in sums_traj[-4:]])
    rho = float(np.max(a[1:] / a[:-1]))
    assert 0.0 < rho < 1.0, ("no contraction to bound the tail", a)
    return (2.0 * thr + ulp(B).sum(axis=1)) / (1.0 - rho), rho


def cold_trajectory(sv, thr, per_band):
    """converge from reset with host steps, keeping every pass's band sums"""
    _check(_L().daisy_solver_reset(sv.s))
    traj = [sv.sums()]
    crit = (lambda v: (v > thr).any()) if per_band else (lambda v: v.sum() > thr)
    while crit(traj[-1]):
        traj.append(sv.step())
        assert len(traj) < 2000
    return traj


# ---- 1. restart identity on every kernel path ---------------------------------------------------------------------------
RESTART_CASES = [(K, path) for K in (1, 3, 9) for path in paths_for(K)] + \
                [(K, path) for K in (16, 32) for path in paths_for(K)] + [(64, "mma"), (41, "mma")]


@pytest.mark.parametrize("K,path", RESTART_CASES)
def test_restart_identity(box, K, path, monkeypatch):
    sc, p, F = box
    N = sc.numtriangles
    E, M, mat = make_inputs(N, K, 31 * K + 5)
    set_path(monkeypatch, paths_for(K)[path][0])
    s = Solver(p, K, E, M, mat)
    try:
        assert _L().daisy_solver_launches_per_pass(s.s) == paths_for(K)[path][1]
        rng = np.random.RandomState(K)
        B0 = rng.uniform(0.0, 3.0, (K, N)).astype(np.float32)
        s.step()  # a pass before: the restart reads B0, not the state
        _check(s.restart(B0), "restart")
        assert s.numpasses == 1
        B, R = s.read()
        want = (B - B0).astype(np.float32)
        assert np.array_equal(R.view(np.uint32), want.view(np.uint32)), (K, path, "residual != B_after - B0")
        assert_rel(B, fp64_restart(F, B0, E, M, mat), "B after restart K=%d %s" % (K, path))
        sums = s.sums()
        assert np.allclose(sums, np.abs(R.astype(np.float64)).sum(axis=1), rtol=1e-9, atol=0), (sums,)
        # padded bands: the staged input (the buffer the restart read) holds B0 and zeros; after one more pass the restart's
        # own output block is that buffer again, with r in the first K bands and zeros in the others
        Kp = padded_K(K)
        inp = exchange_block(s.s, K, N if N % 4 == 0 else N + 4 - N % 4)
        assert np.array_equal(inp[:K, :N], B0) and not inp[K:Kp].any()
        s.step()
        out = exchange_block(s.s, K, inp.shape[1])
        assert np.array_equal(out[:K, :N].view(np.uint32), R.view(np.uint32)) and not out[K:Kp].any()
    finally:
        s.close()


# ---- 2. fixed point ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [3, 9, 32])
def test_restart_at_the_fixed_point(box, K, monkeypatch):
    """a converged solve restarted with unchanged inputs: per band, sum |r| is the next pass's band sum (M F r_n, computed by
    a copy of the solver that takes one more step) plus the rounding floor sum_p ulp(B_p)"""
    sc, p, F = box
    set_path(monkeypatch, {})
    E, M, mat = lamp_inputs(sc, K, 3 + K)
    s = Solver(p, K, E, M, mat)
    t = Solver(p, K, E, M, mat)
    try:
        s.converge(1e-4, 1)
        B, R = s.read()
        _check(_L().daisy_solver_write(t.s, _fp(B), _fp(R)))
        nxt = t.step()
        _check(s.restart(), "restart")
        got = s.sums()
        floor = ulp(B).sum(axis=1)
        assert (got <= nxt + floor).all(), ("sum |r| of the restart", got, "next step", nxt, "floor", floor)
    finally:
        s.close(); t.close()


# ---- 3. geometry moves ---------------------------------------------------------------------------------------------------
MOVES = [("noop", None, (0.0, 0.0, 0.0)), ("lamp_small", "lamp", (0.03, 0.0, 0.02)), ("lamp", "lamp", (0.4, 0.0, -0.3)),
         ("short_block_small", "short", (0.03, 0.0, 0.0)), ("short_block", "short", (0.5, 0.0, 0.4))]


@pytest.mark.parametrize("name,quads,offset", MOVES)
def test_warm_solve_after_a_geometry_move(uv50, name, quads, offset, monkeypatch):
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    set_path(monkeypatch, {})
    sc = dz.cornell_box(N_BOX)
    K, thr = 3, 1e-4
    E, M, mat = lamp_inputs(sc, K, 11)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv50)
    p.cudaCalculateRadiosityMatrix()
    s = Solver(p, K, E, M, mat)
    c = None
    try:
        s.converge(thr, 1)
        if quads is not None:
            v, n = scenes.cornell_moved(sc, scenes.CORNELL_LAMP if quads == "lamp" else scenes.CORNELL_SHORT_BLOCK, offset=offset)
            p.updateGeometry(v, n)
            p.updateRadiosityMatrix()
        _check(s.restart(), "restart")
        warm = s.converge(thr, 1)
        Bw, _ = s.read()
        c = Solver(p, K, E, M, mat)
        traj = cold_trajectory(c, thr, 1)
        cold = len(traj) - 1
        Bc, _ = c.read()
        tol, rho = converge_tolerance(traj, thr, Bc)
        dist = np.abs(Bw.astype(np.float64) - Bc.astype(np.float64)).sum(axis=1)
        print("%s: warm %d passes, cold %d, rho %.3f, distance %s, tolerance %s" % (name, warm, cold, rho, dist, tol))
        assert (dist <= tol).all(), (name, dist, tol)
        if name == "noop" or name.endswith("_small"):
            assert warm <= cold, (name, "warm", warm, "cold", cold)
    finally:
        s.close()
        if c is not None:
            c.close()
        p.close()


# ---- 4. signed residual -------------------------------------------------------------------------------------------------
def test_lamp_turned_off_needs_the_absolute_sums(box, monkeypatch):
    """half of the lamp switched off: the restart residual is negative there, its signed band sums pass the RGB rule at once,
    the absolute ones do not; the warm solve goes on and matches a cold solve with the new emission"""
    sc, p, F = box
    set_path(monkeypatch, {})
    K, thr = 3, 1e-4
    E, M, mat = lamp_inputs(sc, K, 5)
    s = Solver(p, K, E, M, mat)
    c = None
    try:
        s.converge(thr, 1)
        lamp = np.nonzero(sc.mat_idx == 0)[0]
        E2 = E.copy()
        E2[:, lamp[: lamp.size // 2]] = 0.0
        _check(_L().daisy_solver_set_emission(s.s, _fp(E2)), "set_emission")
        _check(s.restart(), "restart")
        B1, R1 = s.read()
        sums = s.sums()
        absref = np.abs(R1.astype(np.float64)).sum(axis=1)
        assert np.allclose(sums, absref, rtol=1e-12, atol=0), (sums, absref)
        assert (R1.astype(np.float64).sum(axis=1) <= thr).all(), "the signed sums would not have stopped the solve"
        assert (sums > thr).any()
        warm = s.converge(thr, 1)
        assert warm > 1
        Bw, _ = s.read()
        c = Solver(p, K, E2, M, mat)
        traj = cold_trajectory(c, thr, 1)
        Bc, _ = c.read()
        tol, _ = converge_tolerance(traj, thr, Bc)
        dist = np.abs(Bw.astype(np.float64) - Bc.astype(np.float64)).sum(axis=1)
        assert (dist <= tol).all(), (dist, tol)
    finally:
        s.close()
        if c is not None:
            c.close()


# ---- 5. materials -------------------------------------------------------------------------------------------------------
def test_recoloured_material_and_refusals(box, monkeypatch):
    sc, p, F = box
    set_path(monkeypatch, {})
    K, thr = 3, 1e-4
    E, M, mat = lamp_inputs(sc, K, 9)
    s = Solver(p, K, E, M, mat)
    c = None
    try:
        s.converge(thr, 1)
        before = s.state()
        # refusals: nothing changes
        assert _L().daisy_solver_set_materials(s.s, _fp(M), 0, _ip(mat)) == E_INVALID
        bad = mat.copy()
        bad[17] = M.shape[0]
        assert _L().daisy_solver_set_materials(s.s, _fp(M), M.shape[0], _ip(bad)) == E_INVALID
        bad[17] = -1
        assert _L().daisy_solver_set_materials(s.s, _fp(M), M.shape[0], _ip(bad)) == E_INVALID
        assert _L().daisy_solver_set_emission(s.s, None) == E_INVALID
        after = s.state()
        for a, b, what in zip(before, after, ("B", "residual", "sums", "passes")):
            assert np.array_equal(np.asarray(a), np.asarray(b)), what
        # one material recoloured, and one more material (nmat grows) given to a few patches
        M2 = np.concatenate([M, (M[2:3] * 0.5).astype(np.float32)])
        M2[3] = (M2[3] * np.float32(0.3)).astype(np.float32)
        mat2 = mat.copy()
        mat2[np.nonzero(mat == 2)[0][::3]] = M2.shape[0] - 1
        _check(_L().daisy_solver_set_materials(s.s, _fp(M2), M2.shape[0], _ip(mat2)), "set_materials")
        _check(s.restart(), "restart")
        s.converge(thr, 1)
        Bw, _ = s.read()
        c = Solver(p, K, E, M2, mat2)
        traj = cold_trajectory(c, thr, 1)
        Bc, _ = c.read()
        tol, _ = converge_tolerance(traj, thr, Bc)
        dist = np.abs(Bw.astype(np.float64) - Bc.astype(np.float64)).sum(axis=1)
        assert (dist <= tol).all(), (dist, tol)
    finally:
        s.close()
        if c is not None:
            c.close()


# ---- 6. device converge after a restart ---------------------------------------------------------------------------------
DEVICE_CASES = [(K, path) for K in (3, 9) for path in paths_for(K)] + [(K, path) for K in (16, 32) for path in paths_for(K)] + [(41, "mma")]


@pytest.mark.parametrize("K,path", DEVICE_CASES)
def test_device_converge_after_restart(box, K, path, monkeypatch):
    sc, p, F = box
    N = sc.numtriangles
    set_path(monkeypatch, paths_for(K)[path][0])
    E, M, mat = make_inputs(N, K, 77 + K)
    h, d = Solver(p, K, E, M, mat), Solver(p, K, E, M, mat)
    try:
        rng = np.random.RandomState(3 * K)
        B0 = (E * rng.uniform(0.5, 1.5, E.shape)).astype(np.float32)
        for thr, per_band in ((1e-3, 1), (float(K), 0)):
            _check(h.restart(B0)); _check(d.restart(B0))
            ph, pd = h.converge(thr, per_band), d.converge(thr, per_band, on_device=True)
            assert ph == pd and ph > 2, (ph, pd)
            (Bh, Rh, Sh, nh), (Bd, Rd, Sd, nd) = h.state(), d.state()
            assert nh == nd
            assert np.array_equal(Bh.view(np.uint32), Bd.view(np.uint32))
            assert np.array_equal(Rh.view(np.uint32), Rd.view(np.uint32))
            assert np.array_equal(Sh, Sd)
            assert np.allclose(Sh, np.abs(Rh.astype(np.float64)).sum(axis=1), rtol=1e-9, atol=0)
    finally:
        h.close(); d.close()


# ---- 7. back to the cold path -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [3, 16])
def test_reset_returns_to_the_cold_path(box, K, monkeypatch):
    sc, p, F = box
    set_path(monkeypatch, {})
    E, M, mat = lamp_inputs(sc, K, 21)
    s, f = Solver(p, K, E, M, mat), Solver(p, K, E, M, mat)
    try:
        s.converge(1e-4, 1)
        _check(s.restart((s.read()[0] * np.float32(1.25)).astype(np.float32)))
        s.converge(1e-4, 1)
        _check(_L().daisy_solver_reset(s.s))
        ps, pf = s.converge(1e-4, 1), f.converge(1e-4, 1)
        assert ps == pf
        (Bs, Rs, Ss, ns), (Bf, Rf, Sf, nf) = s.state(), f.state()
        assert ns == nf
        assert np.array_equal(Bs.view(np.uint32), Bf.view(np.uint32))
        assert np.array_equal(Rs.view(np.uint32), Rf.view(np.uint32))
        assert np.array_equal(Ss.view(np.uint64), Sf.view(np.uint64))
    finally:
        s.close(); f.close()


# ---- 8. Python surface: emission value, materials, mesh edit ---------------------------------------------------------
def _spectral(dz, sc, p, model, converge=True, thr=1e-3):
    mesh = dz.MeshS.from_scene(sc, WL, model)
    p.mesh = mesh
    l = dz.SpectralLightning(mesh, p, 7.0, WL, cuda_enabled=True, converge=False)
    l.threshold = thr
    if converge:
        l.converge_lightning()
    return l


def _tail_tolerance(aw, ac0, ac1, Bc):
    """distance two stopped solves may have (sum over bands and patches): the untaken tails of both residual series, a / (1 - rho)
    with rho = one more cold pass's contraction ac1 / ac0, plus the FP32 floor ulp(B) / (1 - rho)"""
    rho = ac1 / ac0
    assert 0.0 < rho < 1.0, (ac0, ac1)
    return (aw + ac0 + ulp(Bc).sum()) / (1.0 - rho)


def _assert_close_solutions(lw, lc, what):
    Bw, Bc = lw.lightningvalues, lc.lightningvalues
    ac0 = float(lc.band_sums().sum())
    ac1 = float(lc.increment_lightpass().sum())
    tol = _tail_tolerance(float(lw.band_sums().sum()), ac0, ac1, Bc)
    dist = np.abs(Bw.astype(np.float64) - Bc.astype(np.float64)).sum()
    assert dist <= tol, (what, dist, tol)


def test_lightning_mesh_edit_and_setters(uv50, coeff_model):
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    model = coeff_model[0]
    sc = dz.cornell_box(N_BOX)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc, WL, model), device=0, rands=uv50)
    l = _spectral(dz, sc, p, model)
    cold_passes = l.numpasses
    assert l.reconverge() <= cold_passes  # nothing changed: the warm solve is no longer than the cold one
    # emission value
    l.set_emission_value(3.5)
    l.reconverge()
    q = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc, WL, model), device=0, rands=uv50)
    lc = _spectral(dz, sc, q, model, converge=False)
    lc.set_emission_value(3.5)
    lc.reset()
    lc.converge_lightning()
    _assert_close_solutions(l, lc, "emission value")
    lc.close()
    # a material recoloured
    i = next(k for k, m in enumerate(l.mesh_.materials) if m.kind == "diffuse")
    l.mesh_.materials[i].M = (l.mesh_.materials[i].M * np.float32(0.5)).astype(np.float32)
    l.set_materials()
    l.reconverge()
    E2, M2 = l._derive_inputs(3.5)
    c = Solver(q, l.K, E2, M2, np.ascontiguousarray(sc.mat_idx, np.int32))
    c.converge(l.threshold, 0)
    Bc, _ = c.read()
    ac0 = float(c.sums().sum())
    tol = _tail_tolerance(float(l.band_sums().sum()), ac0, float(c.step().sum()), Bc)
    dist = np.abs(l.lightningvalues.astype(np.float64) - Bc.astype(np.float64)).sum()
    assert dist <= tol, ("material", dist, tol)
    c.close()
    q.close()
    # mesh edit: the short block removed
    B_before = l.lightningvalues
    sc_new, prev = scenes.edit_scene(sc, remove=np.arange(5 * N_BOX // 16, 10 * N_BOX // 16))
    mesh_new = dz.MeshS.from_scene(sc_new, WL, model)
    mesh_new.materials = l.mesh_.materials  # the recoloured material carries over
    p.replaceMesh(mesh_new, prev)
    p.updateRadiosityMatrix()
    warm = l.after_mesh_edit(mesh_new, prev, B_before)
    r = dz.OptixPrimeFunctionality(mesh_new, device=0, rands=uv50)
    lc = dz.SpectralLightning(mesh_new, r, 3.5, WL, cuda_enabled=True, converge=False)
    lc.threshold = l.threshold
    cold = lc.converge_lightning()
    print("mesh edit: warm %d passes, cold %d" % (warm, cold))
    _assert_close_solutions(l, lc, "mesh edit")
    lc.close(); r.close(); l.close(); p.close()


# ---- 9. multi-GPU forms -------------------------------------------------------------------------------------------------
def test_host_exchanged_partition_refuses(uv50):
    import daisyriot_b200 as dz
    sc = dz.cornell_box(512)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=uv50, rank=0, nranks=2)
    try:
        r0, r1 = p.row_range
        F = np.zeros((r1 - r0, sc.numtriangles), np.float32)
        p.loadRadiosityMatrix(F, r0)
        E, M, mat = lamp_inputs(sc, 3, 1)
        s = Solver(p, 3, E, M, mat)
        assert s.restart() == E_STATE
        assert b"fused exchange" in _L().daisy_last_error()
        s.close()
    finally:
        p.close()


@pytest.mark.parametrize("ndev", [2, 8])
def test_group_restart_matches_single_gpu(box, uv50, ndev):
    import daisyriot_b200 as dz
    if dz.lib().daisy_device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    sc, p, F = box
    K = 9
    E, M, mat = make_inputs(sc.numtriangles, K, 5)
    B0 = (E * np.float32(1.5)).astype(np.float32)
    g = dz.DeviceGroup(dz.MeshS.from_scene(sc), ndev=ndev, rands=uv50)
    g.cudaCalculateRadiosityMatrix()
    gs = dz.GroupSolver(g, K, E, M, mat)
    s = Solver(p, K, E, M, mat)
    try:
        gs.restart(B0)
        _check(s.restart(B0))
        Bg, Rg = gs.read()
        Bs, Rs = s.read()
        assert_rel(Bg, Bs, "group restart B")
        assert np.allclose(gs.band_sums(), s.sums(), rtol=1e-5)
        for on_device in (False, True):
            gs.restart(B0)
            _check(s.restart(B0))
            pg = gs.converge(1e-3, True, on_device=on_device)
            ps = s.converge(1e-3, 1)
            assert abs(pg - ps) <= 1, (pg, ps)
            assert_rel(gs.read()[0], s.read()[0], "group converge after restart")
        gs.set_emission((E * np.float32(0.5)).astype(np.float32))
        gs.set_materials(M, mat)
        gs.restart()
        assert gs.numpasses == 1
    finally:
        s.close(); gs.close(); g.close()


# ---- 10. the C++ shim ---------------------------------------------------------------------------------------------------
DEMO = os.path.join(ROOT, "shim", "_build", "shim_demo")


@pytest.mark.skipif(not os.path.exists(DEMO), reason="shim demo is built where /root/reference exists (make -C shim)")
def test_shim_reconverge(tmp_path, coeff_model, uv50):
    """shim_demo with DAISY_DEMO_RECONVERGE: one restart after the converge, through Lightning::reconverge_lightning()"""
    import subprocess
    from daisyriot_b200 import scenes
    model, cwd = coeff_model
    sc = scenes.cornell_box(2048)
    obj, _ = scenes.write_obj(sc, cwd, "shim_restart")
    rands = os.path.join(cwd, "rands_restart.bin")
    uv50.astype(np.float32).tofile(rands)
    out = subprocess.run([DEMO, obj, cwd + "/", "2", "7.0", "1", rands], cwd=cwd, capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, DAISY_DEMO_RECONVERGE="1", DAISY_DEMO_SOLVE_ONLY="1"))
    assert out.returncode == 0, out.stderr[-2000:]
    m = re.search(r"RESTART passes=(\d+) sumB=(\S+)", out.stdout)
    s = re.search(r"SOLVE patches=\d+ gpus=\d+ passes=(\d+) sumB=(\S+)", out.stdout)
    assert m and s, out.stdout[-2000:]
    assert int(m.group(1)) >= 1 and int(s.group(1)) == int(m.group(1))
    assert abs(float(m.group(2)) - float(s.group(2))) <= 1e-12 * abs(float(s.group(2)))
