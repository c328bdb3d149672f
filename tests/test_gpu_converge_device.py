"""daisy_solver_converge_device (the stop rule evaluated by the pass kernels) against daisy_solver_converge (the host loop).

Every case runs both on twin solvers -- same context, inputs, kernel path and state -- and requires the same pass count and
B, residual and band sums equal bit for bit.  Thresholds are placed on the band-sum trajectory the host loop sees, so that
the decision falls before the first pass, on the first and second decision a kernel takes, exactly on a band total (the
strict '>'), after several batches of launches, and at max_passes.
"""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_gather_shapes import make_inputs, make_matrix, paths_for, set_path, sub_scene

pytestmark = pytest.mark.gpu

NS = [65, 257, 2050, 7712]
KS = [1, 2, 5, 9, 13, 16, 23, 32]
DEMO = os.path.join(ROOT, "shim", "_build", "shim_demo")


def _L():
    from daisyriot_b200 import _lib
    return _lib.lib()


def _check(rc, what=""):
    from daisyriot_b200 import _lib
    _lib.check(rc, what)


def _dp(x):
    return x.ctypes.data_as(C.POINTER(C.c_double))


def stat(sums, per_band):
    """the host loop's criterion: largest band total, or the total over bands added in band order"""
    if per_band:
        return max(float(v) for v in sums)
    t = 0.0
    for v in sums:
        t += float(v)
    return t


class _Ctx:
    def __init__(self):
        self.ctx = {}

    def get(self, N, fresh=False):
        import daisyriot_b200 as dz
        from daisyriot_b200 import scenes
        key = (N, fresh)
        if key not in self.ctx:
            p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sub_scene(N)), device=0, rands=scenes.msvc_sample_pattern(1))
            p.loadRadiosityMatrix(make_matrix(N, 1000 + N))
            self.ctx[key] = p
        return self.ctx[key]

    def close(self):
        for p in self.ctx.values():
            p.close()


@pytest.fixture(scope="module")
def ctxs():
    import daisyriot_b200 as dz
    assert dz.lib().daisy_device_count() >= 1, "no CUDA device visible"
    c = _Ctx()
    yield c
    c.close()


class Twin:
    """Two solvers built identically: `h` is driven by the host loop, `d` by the device converge."""

    def __init__(self, p, K, E, M, mat, path, monkeypatch):
        set_path(monkeypatch, paths_for(K)[path][0])
        from daisyriot_b200 import _lib
        self.K, self.N = K, E.shape[1]
        self.h, self.d = C.c_void_p(), C.c_void_p()
        for s in (self.h, self.d):
            _check(_L().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)), "create")
        assert _L().daisy_solver_launches_per_pass(self.h) == paths_for(K)[path][1]

    def both(self, fn):
        fn(self.h)
        fn(self.d)

    def converge(self, thr, per_band, max_passes=0):
        ph, pd = C.c_int(-1), C.c_int(-1)
        _check(_L().daisy_solver_converge(self.h, float(thr), int(per_band), int(max_passes), C.byref(ph)), "converge")
        _check(_L().daisy_solver_converge_device(self.d, float(thr), int(per_band), int(max_passes), C.byref(pd)), "converge_device")
        return ph.value, pd.value

    def state(self, s):
        from daisyriot_b200 import _lib
        B, R = np.empty((self.K, self.N), np.float32), np.empty((self.K, self.N), np.float32)
        sums = np.zeros(self.K)
        _check(_L().daisy_solver_band_sums(s, _dp(sums)))
        _check(_L().daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
        return B, R, sums, _L().daisy_solver_numpasses(s)

    def assert_same(self, what):
        (Bh, Rh, Sh, nh), (Bd, Rd, Sd, nd) = self.state(self.h), self.state(self.d)
        assert nh == nd, (what, "numpasses", nh, nd)
        assert np.array_equal(Bh.view(np.uint32), Bd.view(np.uint32)), (what, "B")
        assert np.array_equal(Rh.view(np.uint32), Rd.view(np.uint32)), (what, "residual")
        assert np.array_equal(Sh, Sd), (what, "band sums", Sh, Sd)
        return nh

    def check(self, thr, per_band, what, max_passes=0):
        ph, pd = self.converge(thr, per_band, max_passes)
        assert ph == pd, (what, "passes_out", ph, pd)
        self.assert_same(what)
        return ph

    def close(self):
        self.both(_L().daisy_solver_destroy)


def trajectory(s, K, passes):
    """band sums before the first pass and after each of `passes` passes (daisy_solver_step from reset)"""
    _check(_L().daisy_solver_reset(s))
    out = [np.zeros(K)]
    _check(_L().daisy_solver_band_sums(s, _dp(out[0])))
    for _ in range(passes):
        t = np.zeros(K)
        _check(_L().daisy_solver_step(s, _dp(t)))
        out.append(t)
    _check(_L().daisy_solver_reset(s))
    return out


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("K", KS)
def test_every_path_and_decision_point(ctxs, N, K, monkeypatch):
    """Both rules on every kernel path, with the decision before the first pass (nothing launched, B unchanged), after one and
    two passes, on a threshold equal to a band total, after eight passes; max_passes cuts an unfinished converge exactly."""
    p = ctxs.get(N)
    E, M, mat = make_inputs(N, K, 7 * N + K)
    for path in paths_for(K):
        t = Twin(p, K, E, M, mat, path, monkeypatch)
        try:
            traj = trajectory(t.h, K, 9)
            for per_band in (0, 1):
                v = [stat(s, per_band) for s in traj]
                assert all(b < a for a, b in zip(v, v[1:])), v
                cases = [(v[0] * 1.5, 0), (math.sqrt(v[0] * v[1]), 1), (math.sqrt(v[1] * v[2]), 2), (v[3], 3), (math.sqrt(v[7] * v[8]), 8)]
                for thr, want in cases:
                    what = (N, K, path, per_band, want)
                    t.both(lambda s: _check(_L().daisy_solver_reset(s)))
                    assert t.check(thr, per_band, what) == want, what
                    if want == 0:
                        B, _, _, n = t.state(t.d)
                        assert n == 0 and np.array_equal(B, E), what
                for mp in (1, 5):  # not finished at max_passes
                    t.both(lambda s: _check(_L().daisy_solver_reset(s)))
                    assert t.check(0.0, per_band, (N, K, path, per_band, "max", mp), max_passes=mp) == mp
        finally:
            t.close()


@pytest.mark.parametrize("K", [1, 9, 16])
@pytest.mark.parametrize("per_band", [0, 1])
def test_slow_contraction_crosses_batches(ctxs, K, per_band, monkeypatch):
    """about 0.97 per pass: a converge of more than 200 passes, many batches of launches, on every path"""
    N = 2050
    p = ctxs.get(N)
    F = make_matrix(N, 1000 + N).astype(np.float64)
    x = np.ones(N)
    for _ in range(200):  # power iteration: spectral radius of F (non-negative)
        y = F @ x
        rho = np.linalg.norm(y) / np.linalg.norm(x)
        x = y / np.linalg.norm(y)
    E, _, mat = make_inputs(N, K, 11 * K)
    M = np.ascontiguousarray(np.broadcast_to(np.eye(K, dtype=np.float32) * np.float32(0.97 / rho), (13, K, K)))
    s0 = stat(E.astype(np.float64).sum(axis=1), per_band)
    thr = s0 * 0.97 ** 230
    for path in paths_for(K):
        t = Twin(p, K, E, M, mat, path, monkeypatch)
        try:
            n = t.check(thr, per_band, (K, per_band, path))
            assert n > 200, n
        finally:
            t.close()


@pytest.mark.parametrize("K", [3, 9, 16, 32])
def test_continuation_matches_host_twin(ctxs, K, monkeypatch):
    """converge, 2 steps, converge lower, reset, converge; then after daisy_solver_write and after daisy_formfactors_write_rows
    (which makes the skip plan rescan F) -- each step on both twins, bit-identical throughout"""
    from daisyriot_b200 import _lib
    N = 2050
    p = ctxs.get(N, fresh=True)
    E, M, mat = make_inputs(N, K, 5 + K)
    path = "skip" if K <= 9 else "mma"
    t = Twin(p, K, E, M, mat, path, monkeypatch)
    try:
        v = [stat(s, 0) for s in trajectory(t.h, K, 10)]
        t.check(math.sqrt(v[3] * v[4]), 0, "first")
        t.both(lambda s: _check(_L().daisy_solver_step(s, None)))
        t.both(lambda s: _check(_L().daisy_solver_step(s, None)))
        t.assert_same("steps")
        assert t.check(math.sqrt(v[8] * v[9]), 0, "lower") == 9
        t.both(lambda s: _check(_L().daisy_solver_reset(s)))
        t.check(math.sqrt(v[2] * v[3]), 0, "after reset")
        rng = np.random.RandomState(K)
        B = np.ascontiguousarray(rng.uniform(0, 1, (K, N)).astype(np.float32))
        R = np.ascontiguousarray(rng.uniform(0, 1, (K, N)).astype(np.float32))
        t.both(lambda s: _check(_L().daisy_solver_write(s, _lib.fptr(B), _lib.fptr(R))))
        t.check(stat(R.astype(np.float64).sum(axis=1), 1) * 1e-3, 1, "after write")
        rows = make_matrix(N, 77)[:300] * np.float32(0.5)
        _check(_L().daisy_formfactors_write_rows(p._ctx, 100, 300, _lib.fptr(np.ascontiguousarray(rows))), "write_rows")
        t.both(lambda s: _check(_L().daisy_solver_reset(s)))
        t.check(math.sqrt(v[4] * v[5]), 0, "after write_rows")
        t.both(lambda s: _check(_L().daisy_solver_reset(s)))
        t.check(0.0, 1, "after write_rows, max_passes", max_passes=6)
    finally:
        t.close()


def test_partition_exchanged_by_host_is_refused(monkeypatch):
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    set_path(monkeypatch, {})
    N, K = 300, 3
    mesh = dz.MeshS.from_scene(sub_scene(N))
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=scenes.msvc_sample_pattern(1), rank=0, nranks=2)
    r0, r1 = p.row_range
    p.loadRadiosityMatrix(make_matrix(N, 3)[r0:r1], r0)
    E, M, mat = make_inputs(N, K, 1)
    s = C.c_void_p()
    _check(_L().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)))
    n = C.c_int()
    assert _L().daisy_solver_converge_device(s, 1.0, 0, 0, C.byref(n)) == -3  # DAISY_E_STATE
    _L().daisy_solver_destroy(s)
    p.close()


def test_lightning_mirror_on_device(cornell2048, uv50, coeff_model):
    """Spectral / RGB / BW Lightning on the 2 048-patch box: converge_lightning(on_device=True) gives the default's passes and
    bit-identical read()"""
    import daisyriot_b200 as dz
    model, _ = coeff_model
    wl = np.arange(200, 601, 50).astype(np.float32)
    mesh = dz.MeshS.from_scene(cornell2048, wl, model)
    p = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv50)
    mesh.materials[3].emission[:] = (0.2, 0.1, 0.05)
    for method in (2, 1, 0):
        ev = 7.0 if method == 2 else 500.0
        lt = dz.Lightning.get_lightning(method, mesh, p, ev, wl, True, None, converge=False)
        n_host = lt.converge_lightning(400)
        B_host, R_host = (a.copy() for a in lt.read())
        lt.reset()
        n_dev = lt.converge_lightning(400, on_device=True)
        B_dev, R_dev = lt.read()
        assert n_host == n_dev and n_host > 0, (method, n_host, n_dev)
        assert np.array_equal(B_host.view(np.uint32), B_dev.view(np.uint32)) and np.array_equal(R_host.view(np.uint32), R_dev.view(np.uint32)), method
        lt.close()
    p.close()


@pytest.mark.parametrize("ndev,N", [(2, 224), (2, 2050), (8, 6400)])
def test_group_converge_on_device(ndev, N):
    """DeviceGroup over 2 / 8 GPUs (N = 224 on 2 and 6400 on 8 leave the last rank without rows): on_device=True against the
    host group converge, bit-identical"""
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    if dz.lib().daisy_device_count() < ndev:
        pytest.skip("needs %d GPUs" % ndev)
    mesh = dz.MeshS.from_scene(sub_scene(N))
    from daisyriot_b200 import _lib
    g = dz.DeviceGroup(mesh, devices=list(range(ndev)), rands=scenes.msvc_sample_pattern(1))
    F = make_matrix(N, 1000 + N)
    _check(_L().daisy_group_formfactors_write_rows(g._g, 0, N, _lib.fptr(F)))
    for K in (3, 9, 16):
        E, M, mat = make_inputs(N, K, 3 * K)
        res = []
        for on_device in (False, True):
            gs = dz.GroupSolver(g, K, E, M, mat)
            traj = [stat(gs.band_sums(), 0)] + [stat(gs.step(True), 0) for _ in range(6)]
            gs.reset()
            n = gs.converge(math.sqrt(traj[5] * traj[6]), False, on_device=on_device)
            B, R = gs.read()
            res.append((n, B, R, gs.band_sums()))
            gs.close()
        assert res[0][0] == res[1][0] == 6, (ndev, N, K, res[0][0], res[1][0])
        assert all(np.array_equal(a, b) for a, b in zip(res[0][1:], res[1][1:])), (ndev, N, K)
    g.close()


WORKER = r'''
import os, sys, numpy as np, torch
sys.path.insert(0, os.environ["DAISY_ROOT"]); sys.path.insert(0, os.path.join(os.environ["DAISY_ROOT"], "tests"))
import daisyriot_b200 as dz
from daisyriot_b200 import dist as ddist, scenes
from test_gpu_gather_shapes import make_inputs, make_matrix, sub_scene
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", rank))
N = 2050
p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sub_scene(N)), device=rank, rands=scenes.msvc_sample_pattern(1), rank=rank, nranks=world)
r0, r1 = p.row_range
p.loadRadiosityMatrix(make_matrix(N, 1000 + N)[r0:r1], r0)
torch.distributed.barrier()
out = {}
for K in (9, 16):
    E, M, mat = make_inputs(N, K, 3 * K)
    s = ddist.PartitionedSolver(p, K, E, M, mat, fused=True)
    thr = float(np.sum(s.band_sums())) * 1e-4
    for on_device in (0, 1):
        s.reset()
        torch.distributed.barrier()
        n = s.converge(thr, False, on_device=bool(on_device))
        B, R = s.read_local()
        out["K%d_%d" % (K, on_device)] = np.array([n])
        out["B%d_%d" % (K, on_device)] = B; out["R%d_%d" % (K, on_device)] = R; out["S%d_%d" % (K, on_device)] = s.band_sums()
    s.close()
np.savez(os.path.join(os.environ["DAISY_OUT"], "rank%d.npz" % rank), **out)
p.close()
torch.distributed.destroy_process_group()
'''


def test_two_process_fused_converge_on_device(tmp_path):
    import sys
    import daisyriot_b200 as dz
    if dz.lib().daisy_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    wf = tmp_path / "worker.py"
    wf.write_text(WORKER)
    env = dict(os.environ, DAISY_ROOT=ROOT, DAISY_OUT=str(tmp_path))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", "29641", str(wf)], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    for r in range(2):
        o = np.load(tmp_path / ("rank%d.npz" % r))
        for K in (9, 16):
            assert o["K%d_0" % K][0] == o["K%d_1" % K][0] > 0, (r, K)
            for a in "BRS":
                assert np.array_equal(o["%s%d_0" % (a, K)], o["%s%d_1" % (a, K)]), (r, K, a)


def _demo_solve(args, cwd, **env):
    out = subprocess.run([DEMO] + args, cwd=cwd, capture_output=True, text=True, timeout=600, env=dict(os.environ, DAISY_DEMO_SOLVE_ONLY="1", **env))
    assert out.returncode == 0, out.stderr[-2000:]
    m = re.search(r"SOLVE patches=\d+ gpus=\d+ passes=(\d+) sumB=(\S+)", out.stdout)
    assert m, out.stdout[-2000:]
    return m.group(1), m.group(2)


@pytest.mark.skipif(not os.path.exists(DEMO), reason="shim demo is built where /root/reference exists (make -C shim)")
@pytest.mark.parametrize("ndev", [1, 2])
def test_shim_demo_converge_on_device(tmp_path, coeff_model, uv50, ndev):
    import daisyriot_b200 as dz
    from daisyriot_b200 import scenes
    if dz.lib().daisy_device_count() < ndev:
        pytest.skip("needs %d GPUs" % ndev)
    _, cwd = coeff_model
    sc = scenes.cornell_box(2048)
    obj, _ = scenes.write_obj(sc, cwd, "conv_dev_scene")
    rands = os.path.join(cwd, "rands_conv.bin")
    uv50.astype(np.float32).tofile(rands)
    args = [obj, cwd + "/", "2", "7.0", "1", rands]
    host = _demo_solve(args, cwd, DAISY_DEMO_NDEV=str(ndev))
    dev = _demo_solve(args, cwd, DAISY_DEMO_NDEV=str(ndev), DAISY_DEMO_CONVERGE="device")
    assert host == dev and int(host[0]) > 0, (host, dev)
