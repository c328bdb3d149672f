#!/usr/bin/env python
"""bench.py -- radiosity gather iterations/s (+ form-factor visibility rays/s) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path on the host cores
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR  # also write B / residual / band sums of the last timed pass

A step is ONE gather pass (residual <- M (F residual); B += residual, reference Lightning.h:196-226) over the
resident dense FP32 form-factor matrix of the workload.  Before the timed passes the matrix is built by the fused
form-factor/visibility kernel; that build is timed too and reported under "formfactor" (rays/s, BASELINE.json's other
metric).  Inputs are synthetic (subdivided Cornell box, BASELINE.json configs 3-5).  F is >= 4 GB, far larger than the
126 MB L2, so successive passes cannot be served from cache.

One JSON line is printed by rank 0.  Keys: see the contract in the task statement; extra: "formfactor",
"roofline" (gather kernel, HBM), "cpu_baseline".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (patches, bands, n_fluorescent)   -- BASELINE.json configs
    "cornell_32k": (32768, 9, 2),        # config 3: 32K patches, dense F ~4 GB, 1 B200
    "cornell_128k": (131072, 9, 2),      # config 4 / north-star target: 128K patches, F 68.7 GB, row-sharded
    "fluor_64k_k32": (65536, 32, 10),    # config 5: 64K patches, 32 bands, >= 8 fluorescent materials
    "fluor_32k_k16": (32768, 16, 6),     # 16 bands: the narrower instance of the tcgen05 gather (same geometry as cornell_32k)
    "cornell_8k": (8192, 9, 2),          # small smoke size
    # the reference's own example scenes (BASELINE.json configs 1-2), read from the committed fixtures in tests/golden/
    "cornellbox_blacklight": (7712, 9, 0),
    "colorballs": (6400, 9, 0),
}
FIXTURE_SCENES = ("cornellbox_blacklight", "colorballs")
# the matrix depends on the geometry only: workloads that differ in bands / materials share the committed digests and ncu captures
SAME_MATRIX_AS = {"fluor_32k_k16": "cornell_32k"}


def row_digest32(wsum):
    """One uint32 per matrix row, as committed in tests/golden/rowdigest_<workload>.npz: the low 32 bits of the device's
    position-weighted sum of the row's bit patterns (sum of bits_c * (2c + 1) mod 2^64).  Every weight is odd, hence invertible
    mod 2^32, so a change of any single entry always changes it; 4 bytes per row keep the largest workload's file under 1 MB.
    The device's xor digest is not used: xor-ing it in lets the two cancel for a one-ulp change of the same entry."""
    return (np.asarray(wsum, np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.uint32)


def parity_rows(N):
    """The constant set of 16 matrix rows that stand for the whole matrix wherever the CPU oracle is involved (parity block,
    cpu_baseline sample, --impl reference): first / last rows, 64-row tile boundaries, the row-block boundaries of 2/4/8-GPU
    partitions and a few fixed pseudo-random rows."""
    rows = {0, 1, 63, 64, N // 2 - 1, N // 2, N - 64, N - 1, N // 8, 3 * (N // 8), 5 * (N // 8), 7 * (N // 8) - 1}
    rng = np.random.RandomState(12345)
    while len(rows) < 16:
        rows.add(int(rng.randint(0, N)))
    return np.array(sorted(rows), np.int32)


def wavelengths_for(K):
    if K == 9:
        return np.arange(200, 601, 50).astype(np.float32)  # reference main.cpp:94
    return (200.0 + (400.0 / (K - 1)) * np.arange(K)).astype(np.float32) if K > 1 else np.array([350.0], np.float32)


def make_workload(name):
    from daisyriot_b200 import materials, rgb2spec, scenes
    N, K, nfl = WORKLOADS[name]
    if name in FIXTURE_SCENES:
        sc = scenes.load_scene_npz(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        assert sc.numtriangles == N
    else:
        sc = scenes.cornell_box(N, n_fluorescent=nfl)
    wl = wavelengths_for(K)
    tmp = tempfile.mkdtemp(prefix="daisy_bench_")
    os.makedirs(os.path.join(tmp, "color_tables"))
    coeff = os.path.join(tmp, "color_tables", "srgb.coeff")
    rgb2spec.write_surrogate_table(coeff, 16)
    mats = materials.make_materials(sc.materials, wl, rgb2spec.RGB2Spec.load(coeff))
    if K >= 16:
        # config 5: full 32x32 re-emission matrices -- the Material.cpp:90-100 rule plus a dense perturbation
        rng = np.random.RandomState(0x5EED)
        for m in mats:
            if m.kind == "fluorescent":
                m.M = (m.M * 0.6 + rng.uniform(0, 0.4 / K, (K, K))).astype(np.float32)
    E, M = materials.spectral_inputs(mats, sc.mat_idx, 7.0)  # emission_value 7.0, config_example.ini:18
    return sc, wl, E, M, tmp


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_run(sc, wl, K, budget_s, steps, coeff_dir, log=lambda *a: None):
    """The reference's CPU path on the host cores, on the constant row sample `parity_rows` of the workload.

    form factors + visibility: the oracle's restatement of calculateAllVisibility (OptiX Prime itself is closed source) on
    an explicit number of OpenMP threads (all host cores, whatever OMP_NUM_THREADS the launcher exported); gather: the
    reference's UNMODIFIED Lightning.h + vendored Eigen 3.2.10 compiled into oracle/_ref (single-threaded, as in the
    reference), fed the sampled rows; full-pass time = SpMV time scaled by N/rows + the measured per-patch loop.
    The rows are processed in a fixed order, one batch of `threads` rows at a time; if the time budget runs out the
    remaining batches are dropped (the sample string says how many rows were done)."""
    from daisyriot_b200 import scenes
    from oracle import pyoracle, pyref
    N = sc.numtriangles
    uv = scenes.msvc_sample_pattern(1)
    orc = pyoracle.Oracle.from_scene(sc)
    cores = max(1, pyoracle.num_procs())
    orc.bvh
    rows = parity_rows(N)
    rows_done, rays_done, t_ff, Fs = [], 0, 0.0, []
    for b0 in range(0, len(rows), cores):
        if rows_done and t_ff >= budget_s:
            break
        batch = rows[b0:b0 + cores]
        t0 = time.time()
        F_b, _, rays = orc.radmat_rowlist(uv, batch, want_masks=False, nthreads=cores)
        t_ff += time.time() - t0
        rays_done += rays
        rows_done += [int(r) for r in batch]
        Fs += [F_b[i] for i in range(len(batch))]
    rays_per_s = rays_done / t_ff if t_ff > 0 else 0.0
    log(f"cpu ff: {len(rows_done)} rows, {rays_done} rays in {t_ff:.1f}s on {cores} threads")
    out = {"ff_rays_per_s": rays_per_s, "ff_rows": len(rows_done), "ff_rays": rays_done, "ff_seconds": t_ff, "cores_ff": cores,
           "gather_kind": None, "it_per_s": None}
    # --- gather: reference Lightning.h + Eigen on the sampled rows
    R = len(rows_done)
    if pyref.available():
        obj, _ = scenes.write_obj(sc, coeff_dir, "bench_scene")
        rs = pyref.RefScene.load(obj, coeff_dir + "/", wl, coeff_dir)
        for i in range(rs.nmat):  # the lamp's M is undefined behaviour in the reference; use the documented restatement
            m = rs.material(i)
            if not np.isfinite(m["M"]).all() or (m["spectral_values"] == 0).all():
                rs.set_material_M(i, np.zeros((K, K), np.float32))
        def run(rows_idx, rows_val):
            r_i, c_i, v = [], [], []
            for r, row in zip(rows_idx, rows_val):
                nz = np.nonzero(row)[0]
                r_i.append(np.full(nz.size, r, np.int32)); c_i.append(nz.astype(np.int32)); v.append(row[nz].astype(np.float64))
            r_i = np.concatenate(r_i) if r_i else np.zeros(0, np.int32)
            c_i = np.concatenate(c_i) if c_i else np.zeros(0, np.int32)
            v = np.concatenate(v) if v else np.zeros(0, np.float64)
            rs.L.ref_set_triplets(rs.h, r_i.ctypes.data_as(C.POINTER(C.c_int)), c_i.ctypes.data_as(C.POINTER(C.c_int)),
                                  v.ctypes.data_as(C.POINTER(C.c_double)), v.size)
            rs.lightning_create(2 if K > 3 else (1 if K == 3 else 0), 7.0)
            rs.lightning_reset()
            ts = []
            for _ in range(max(1, steps)):
                t0 = time.time(); rs.lightning_pass_only(); ts.append(time.time() - t0)
            return float(np.median(ts)), v.size
        t_empty, _ = run([], [])
        t_samp, nnz = run(rows_done, Fs)
        t_full = max(t_samp - t_empty, 1e-9) * (N / max(R, 1)) + t_empty
        out.update({"gather_kind": "reference", "it_per_s": 1.0 / t_full, "gather_sample_nnz": int(nnz), "t_pass_sample_s": t_samp,
                    "t_pass_empty_s": t_empty})
        rs.close()
    else:
        out.update({"gather_kind": "port", "it_per_s": None})  # oracle/_ref was not built: no Eigen pass to time
    return out


def bench_config(name, N, K, S, world):
    """The `config` object, identical in both arms (the driver compares them key by key)."""
    nloc = -(-N // world)
    return {"workload": name, "patches": N, "bands": K, "rays_per_pair": int(S), "parallelism": f"rowshard{world}",
            "cache": "F rows per GPU %.2f GB > 126 MB L2 (inputs larger than L2, no flush needed)" % (4.0 * nloc * N / 1e9)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    sc, wl, E, M, tmp = make_workload(name)
    N, K, _ = WORKLOADS[name]
    t0 = time.time()
    r = cpu_reference_run(sc, wl, K, budget_s=min(60.0, 3.0 * args.cpu_budget), steps=args.steps + args.warmup, coeff_dir=tmp,
                          log=lambda *a: print(*a, file=sys.stderr))
    val = r["it_per_s"]
    line = {"impl": "reference", "metric": "radiosity_gather_iterations_per_s", "value": val, "unit": "iterations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": (1e3 / val) if val else None, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(name, N, K, 50, args.gpus),
            "cpu_baseline": {"value": val, "unit": "iterations/s", "cores": 1, "kind": r["gather_kind"],
                             "sample": f"Lightning.h+Eigen pass on {r['ff_rows']} fixed rows of {N} ({r.get('gather_sample_nnz')} nnz), SpMV time scaled by N/rows"},
            "e2e": {"value": val, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "formfactor": {"metric": "formfactor_visibility_rays_per_s", "value": r["ff_rays_per_s"], "unit": "rays/s", "cores": r["cores_ff"],
                           "kind": "port", "threads": r["cores_ff"], "sample": f"{r['ff_rows']} fixed rows, {r['ff_rays']} rays in {r['ff_seconds']:.1f} s"},
            "wall_s": time.time() - t0}
    print(json.dumps(line))



# ---------------------------------------------------------------------------------------------------------------
def parity_block(optixP, solver, sc, uv, E, M, K, world, rank, torch, name, stop_threshold=200.0):
    """Parity evidence reported with the numbers (SURVEY 8(d)): the constant row sample `parity_rows` of the matrix the
    bench just built, against the CPU oracle (rank 0 computes the oracle rows once, every rank compares the rows it owns):

    * mask_mismatches / F_bit_mismatches: visibility masks and matrix entries that differ (bit-exact bar => 0);
    * ties: rays of those rows whose closest-hit distance is shared bit for bit by two different triangles, i.e. where the
      (t, triangle id) tie rule and not geometry decides (OptiX Prime's own rule is unpinned);
    * digest: every row of the resident matrix against the committed per-row digests of this workload
      (tests/golden/rowdigest_<workload>.npz, exact integer digests) -- proves that 1, 2, 4 and 8 GPUs build the same matrix;
    * gather: the whole solve is repeated with the residual vector read back after every pass; for the sampled rows each new
      residual entry is recomputed in FP64 from the ORACLE's matrix row and the device's previous residual vector
      (Lightning.h:196-226), B is accumulated alongside; max_rel_* are true relative errors over entries above 1e-6 of
      the band's largest value; passes / passes_from_host_sums apply the reference's stop rule to the device's band sums and
      to FP64 sums of the read-back residuals."""
    import torch.distributed as tdist
    from daisyriot_b200 import _lib, api
    N = sc.numtriangles
    rows = parity_rows(N)
    r0, r1 = optixP.row_range
    t0 = time.time()
    dev = torch.device("cuda", torch.cuda.current_device())
    F_ref = np.zeros((len(rows), N), np.float32)
    m_ref = np.zeros((len(rows), N), np.uint64)
    ties = rays = 0
    if rank == 0:
        from oracle import pyoracle
        orc = pyoracle.Oracle.from_scene(sc)
        nth = max(1, pyoracle.num_procs())
        F_ref, m_ref, rays = orc.radmat_rowlist(uv, rows, nthreads=nth)
        ties = orc.count_ties(uv, rows, nthreads=nth)
    if world > 1:
        tF = torch.from_numpy(F_ref).to(dev); tm = torch.from_numpy(m_ref.view(np.int64)).to(dev)
        tdist.broadcast(tF, 0); tdist.broadcast(tm, 0)
        F_ref = tF.cpu().numpy(); m_ref = tm.cpu().numpy().view(np.uint64)
    oracle_s = time.time() - t0

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        tdist.all_reduce(t, op=tdist.ReduceOp.SUM)
        return float(t.item())

    def allmaxf(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())

    mine = [i for i, r in enumerate(rows) if r0 <= r < r1]
    rm = api.RadMat(optixP)
    f_mis = m_mis = 0
    for i in mine:
        r = int(rows[i])
        f_mis += int(np.count_nonzero(rm.rows(r, 1)[0].view(np.uint32) != F_ref[i].view(np.uint32)))
        m_mis += int(np.count_nonzero(optixP.visibilityMasks(r, 1)[0] != m_ref[i]))
    out = {"rows": [int(r) for r in rows], "rows_checked": int(allsum(len(mine))), "rays_checked": int(rays),
           "mask_mismatches": int(allsum(m_mis)), "F_bit_mismatches": int(allsum(f_mis)), "max_rel_F": 0.0, "ties": int(ties),
           "oracle_seconds": oracle_s}
    if out["F_bit_mismatches"]:
        out["max_rel_F"] = None
    # ---- committed per-row digests of the whole matrix
    dpath = os.path.join(ROOT, "tests", "golden", f"rowdigest_{SAME_MATRIX_AS.get(name, name)}.npz")
    if os.path.exists(dpath) and r1 > r0:
        g = np.load(dpath)
        _, dw = rm.row_digest()
        bad = int(np.count_nonzero(row_digest32(dw) != g["digest"][r0:r1]))
        out["digest"] = {"file": os.path.relpath(dpath, ROOT), "rows_checked": int(allsum(r1 - r0)), "row_mismatches": int(allsum(bad))}
    elif os.path.exists(dpath):
        out["digest"] = {"file": os.path.relpath(dpath, ROOT), "rows_checked": int(allsum(0)), "row_mismatches": int(allsum(0))}
    else:
        out["digest"] = None
    # ---- the solve, pass by pass, on the sampled rows
    solver.reset()
    nloc = r1 - r0
    mat = sc.mat_idx
    Mr = {i: M.astype(np.float64)[mat[int(rows[i])]] for i in mine}          # column-major: M[m][j, i] = M(i, j)
    Bchk = {i: E[:, int(rows[i])].astype(np.float64) for i in mine}
    res_prev = np.ascontiguousarray(E, np.float32)
    sums = res_prev.astype(np.float64).sum(1)
    host_sums = sums.copy()
    passes = host_passes = 0
    host_done = False
    max_rel_res = max_rel_B = 0.0
    FLOOR = 1e-6
    while sums.sum() > stop_threshold and passes < 2000:
        sums = solver.step(True)
        passes += 1
        Bl, Rl = solver.read_local()
        if world > 1:
            parts = [torch.zeros((K, optixP_rows_per_rank(optixP)), dtype=torch.float32, device=dev) for _ in range(world)]
            mineT = torch.zeros((K, optixP_rows_per_rank(optixP)), dtype=torch.float32, device=dev)
            mineT[:, :nloc] = torch.from_numpy(Rl).to(dev)
            tdist.all_gather(parts, mineT)
            res_new = torch.cat(parts, 1)[:, :N].cpu().numpy()
        else:
            res_new = Rl
        if not host_done:
            if host_sums.sum() > stop_threshold:
                host_passes += 1
                host_sums = res_new.astype(np.float64).sum(1)
            if not (host_sums.sum() > stop_threshold):
                host_done = True
        band_max = np.abs(res_new).max(1).astype(np.float64) + 1e-300
        band_max_B = np.abs(Bl).max(1).astype(np.float64) + 1e-300
        for i in mine:
            r = int(rows[i])
            want = Mr[i].T @ (res_prev.astype(np.float64) @ F_ref[i].astype(np.float64))   # M_p (F[r,:] . residual_k)_k
            got = Rl[:, r - r0].astype(np.float64)
            Bchk[i] = Bchk[i] + want
            big = np.abs(want) > FLOOR * band_max
            if big.any():
                max_rel_res = max(max_rel_res, float((np.abs(got - want)[big] / np.abs(want)[big]).max()))
            gotB = Bl[:, r - r0].astype(np.float64)
            bigB = np.abs(Bchk[i]) > FLOOR * band_max_B  # same floor as for the residual: FP64 keeps values FP32 flushes to zero
            if bigB.any():
                max_rel_B = max(max_rel_B, float((np.abs(gotB - Bchk[i])[bigB] / np.abs(Bchk[i])[bigB]).max()))
        res_prev = res_new
    out["gather"] = {"passes": int(passes), "passes_from_host_sums": int(host_passes), "max_rel_residual": allmaxf(max_rel_res),
                     "max_rel_B": allmaxf(max_rel_B), "tolerance": 1e-5, "floor": "1e-6 of the band's largest entry",
                     "rows": "the sampled rows; FP64 products of the oracle's matrix rows with the device's residual vectors"}
    out["max_rel_B"] = out["gather"]["max_rel_B"]
    out["passes"] = int(passes)
    out["seconds"] = time.time() - t0
    return out


def incumbent_block(dz, uv):
    """The one GPU kernel the reference already has -- parallellism::runCalculateRadiosityMatrix / calculateRow
    (parallellism.cu:4-111), compiled UNMODIFIED for sm_100a into oracle/_ref -- against this library's counterpart
    (daisy_unoccluded_rows) on the same scenes.  Both deliver the dense N x N list of 16-byte triplets in host memory, which
    is what the reference's entry point returns; seconds are wall clock around the whole call (the reference's managed-memory
    chunks and host copies included, ours with its device-to-host copies included)."""
    from daisyriot_b200 import scenes
    from oracle import pyref
    if not pyref.cuda_kernel_available(False):
        return {"unavailable": "oracle/_ref/libdaisy_ref_cuda.so not built (needs /root/reference at build time)"}
    out = {"kernel": "parallellism::calculateRow (reference, recompiled for sm_100a)", "ours": "k_unoccluded via daisy_unoccluded_rows", "cases": []}
    cases = [("cornellbox_blacklight", scenes.load_scene_npz(os.path.join(ROOT, "tests", "golden", "cornellbox_blacklight.npz"))),
             ("cornell_15k", scenes.cornell_box(15360))]  # the reference's launch geometry divides by zero from N = 16 001 patches on
    for nm, sc in cases:
        N = sc.numtriangles
        p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), rands=uv)
        p.runCalculateRadiosityMatrix(0, min(N, 256), 0)  # warm-up (module load, allocation)
        t0 = time.time()
        ours = p.runCalculateRadiosityMatrix(0, N, 0)["m_value"]
        t_ours = time.time() - t0
        if not out["cases"]:  # warm-up (module load, managed-memory set-up); the reference's launch geometry needs a few thousand patches
            pyref.cuda_run_calculate_radiosity_matrix(sc.vertices, sc.normals, sc.tri)
        ref, t_ref = pyref.cuda_run_calculate_radiosity_matrix(sc.vertices, sc.normals, sc.tri)
        nz = ours > 0
        same_support = bool(((ref > 0) == nz).all())
        # the reference binary is nvcc's default build (FMA contraction, libdevice powf): entries that are cancellation residue
        # (1e-9 and below, against typical 1e-5 .. 1e-2) carry that rounding noise in full, hence the floor
        big = ours > 1e-6 * float(ours.max())
        rel = float((np.abs(ours - ref)[big] / ours[big]).max()) if big.any() else 0.0
        out["cases"].append({"scene": nm, "patches": int(N), "reference_seconds": t_ref, "ours_seconds": t_ours, "speedup": t_ref / t_ours,
                             "pairs_per_s_reference": N * N / t_ref, "pairs_per_s_ours": N * N / t_ours,
                             "same_facing_pairs": same_support, "max_abs_diff": float(np.abs(ours - ref).max()),
                             "max_rel_diff_above_1e-6_of_max": rel})
        p.close()
        del ours, ref
    return out



def peaks_sm_mhz():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("sm_max_mhz", 1965.0))
    except Exception:
        return 1965.0


def optixP_rows_per_rank(optixP):
    from daisyriot_b200 import _lib
    n = C.c_int()
    _lib.check(_lib.lib().daisy_ctx_row_range(optixP._ctx, None, None, C.byref(n)))
    return n.value


def dump_outputs(out_dir, optixP, solver, K, N, world, rank, torch):
    """Writes what a caller of the solver receives after the last timed pass: B.npy and residual.npy (K x N float32, every
    patch, gathered from all ranks) and band_sums.npy (K float64).  The inputs are fixed by the workload, so two builds run
    with the same arguments can be compared array for array.  The largest workload (65536 patches, K = 32) writes 16 MB."""
    B, R = solver.read_local()
    sums = solver.band_sums()
    if world > 1:
        n = optixP_rows_per_rank(optixP)

        def gather(X):
            mine = torch.zeros((K, n), dtype=torch.float32, device="cuda")
            mine[:, :X.shape[1]] = torch.from_numpy(X).cuda()
            parts = [torch.empty_like(mine) for _ in range(world)]
            torch.distributed.all_gather(parts, mine)
            return torch.cat(parts, 1)[:, :N].cpu().numpy()

        B, R = gather(B), gather(R)
    if rank == 0:
        assert B.nbytes + R.nbytes + sums.nbytes <= 64 << 20
        os.makedirs(out_dir, exist_ok=True)
        for name, a in (("B", B), ("residual", R), ("band_sums", sums)):
            np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, dist as ddist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = dz.lib()  # raises without the CUDA library: there is no CPU fallback

    name = args.workload
    sc, wl, E, M, tmp = make_workload(name)
    N, K, _ = WORKLOADS[name]
    uv = dz.msvc_sample_pattern(1)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM)
        return float(t.item())

    # ---- form-factor stage (timed once; it is seconds long, so self-warming): host mesh -> LBVH -> fused FF/visibility
    barrier()
    ff_sampler = ClockSampler(local)
    if rank == 0:
        ff_sampler.start()
    t0 = time.time()
    mesh = dz.MeshS.from_scene(sc)
    optixP = dz.OptixPrimeFunctionality(mesh, device=local, rands=uv, rank=rank, nranks=world)
    if world > 1:
        ddist.build_formfactors_sharded(optixP, peer_tiles=not args.no_peer_tiles)  # mirrored tiles go to the peer's F over NVLink
    else:
        optixP.cudaCalculateRadiosityMatrix()
    torch.cuda.synchronize()
    ff_wall = allmax(time.time() - t0)
    ff_clocks = ff_sampler.stop() if rank == 0 else None
    st = optixP.stats()
    ff_ms = allmax(st["ff_ms"])
    lbvh_ms = allmax(st["lbvh_ms"])
    r0, r1 = optixP.row_range
    # unique facing pairs of the whole matrix: every rank counts pairs whose lower index it owns
    pairs_unique = allsum(float(st["pairs_owned"]))
    pairs_traced = allsum(float(st["pairs_traced"]))
    rays = pairs_unique * uv.shape[0]

    solver = ddist.PartitionedSolver(optixP, K, E, M, sc.mat_idx, fused=not args.no_fused)
    nloc = r1 - r0

    def one_step():
        solver.step(False)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi needs a moment to start: sample from the warm-up through the kernel-timing loop
    # one GPU: back-to-back passes are chained (no per-pass events, programmatic dependent launch: the next pass's grid moves
    # onto SMs as the previous one leaves them) -- what a caller running passes without reading the band sums gets
    chained = world == 1 and not args.no_chained
    if chained:
        _lib.check(L.daisy_solver_set_chained(solver._s, 1))
    for _ in range(max(3, args.warmup)):
        one_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        one_step()
    e1.record()
    barrier()
    ms_total = allmax(e0.elapsed_time(e1))
    ms_step = ms_total / args.steps
    value = 1e3 / ms_step
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, optixP, solver, K, N, world, rank, torch)
    if chained:
        _lib.check(L.daisy_solver_set_chained(solver._s, 0))

    # ---- kernel-only duration of the gather pass for the roofline (library's CUDA events around the pass's kernels)
    kms = []
    for _ in range(min(args.steps, 50)):
        solver.step(True)
        m = C.c_double()
        L.daisy_solver_last_step_ms(solver._s, C.byref(m))
        kms.append(m.value)
    k_ms_isolated = allmax(float(np.mean(kms)))  # one pass alone: launch, ramp and tail exposed
    # roofline: the kernel's average launch duration over the TIMED region -- with chained passes (one launch per pass, grids
    # overlapping their neighbours' ramp and tail) that is the timed region divided by its launches
    k_ms = ms_step if (chained and K <= 9) else k_ms_isolated
    # keep the same load up for ~0.6 s so that nvidia-smi (50 ms period) sees it; the pass count is derived from the
    # all-reduced step time, i.e. identical on every rank (the fused exchange needs all ranks to step in lockstep)
    for _ in range(int(min(20000, max(0, 600.0 / max(ms_step, 1e-3) - args.steps)))):
        solver.step(False)
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    alg_bytes = 4.0 * nloc * N + 16.0 * N * K  # F rows streamed once + residual in/out + B read/write (SURVEY 8(d))
    alg_bytes = allmax(alg_bytes)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    # measured DRAM bytes per launch of the gather kernel (one ncu --set full capture per workload, profiles/gather_traffic.json)
    # form-factor stage roofline: instruction issue.  The warp-instruction count of k_ff_tiles is a property of the workload
    # (same tiles, same candidate lists whatever the schedule), taken from the committed ncu capture of THIS workload
    # (profiles/ff_ncu.json, keyed by workload); the kernel time and the SM clock are measured in this run.
    ff_ncu = ff_roof = None
    try:
        ff_ncu = json.load(open(os.path.join(ROOT, "profiles", "ff_ncu.json"))).get(SAME_MATRIX_AS.get(name, name))
    except Exception:
        pass
    if ff_ncu and ff_ncu.get("warp_instructions"):
        clk = ((ff_clocks or {}).get("sm_mhz") or peaks_sm_mhz()) * 1e6
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        wi = float(ff_ncu["warp_instructions"])  # whole matrix; with N ranks every rank issues 1/N of it (tiles are hashed over the ranks)
        ach = wi / world / (ff_ms * 1e-3)
        pk = sms * 4 * clk
        ff_roof = {"bound": "issue", "achieved": ach, "peak": pk, "unit": "warp-instructions/s per GPU", "frac": ach / pk,
                   "warp_instructions": wi, "warp_instructions_per_ray": wi / max(rays, 1.0), "sm_clock_mhz": clk / 1e6,
                   "threads_per_warp_instruction": ff_ncu.get("threads_active_per_warp_instruction"),
                   "source": ff_ncu.get("source"), "peak_note": "SMs x 4 schedulers x SM clock sampled during the build"}
    elif ff_ncu is None:
        ff_roof = {"unavailable": f"no ncu capture of k_ff_tiles for workload {name} under profiles/ff_ncu.json"}
    # measured DRAM bytes per launch of the gather kernel (one ncu capture per workload and GPU count, profiles/gather_traffic.json;
    # the N-GPU entries were captured on one GPU holding rank 0's row block of an N-way partition: same kernel, same rows x columns)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "gather_traffic.json")))
        t = tj.get(name if world == 1 else f"{name}@{world}")
        if t:
            traffic = t["dram_bytes_per_launch"]
    except Exception:
        pass

    # ---- end to end through the C-ABI with HOST buffers (single GPU): H2D residual+B, pass, D2H residual+B
    e2e = None
    if world == 1:
        hB = torch.empty((K, N), dtype=torch.float32, pin_memory=True).numpy()
        hR = torch.empty((K, N), dtype=torch.float32, pin_memory=True).numpy()
        hB[:] = E; hR[:] = E
        for _ in range(2):
            _lib.check(L.daisy_solver_write(solver._s, _lib.fptr(hB), _lib.fptr(hR)))
            _lib.check(L.daisy_solver_step(solver._s, None))
            _lib.check(L.daisy_solver_read(solver._s, _lib.fptr(hB), _lib.fptr(hR)))
        hB[:] = E; hR[:] = E
        torch.cuda.synchronize()
        nst = min(args.steps, 50)
        t0 = time.time()
        for _ in range(nst):
            _lib.check(L.daisy_solver_write(solver._s, _lib.fptr(hB), _lib.fptr(hR)))
            _lib.check(L.daisy_solver_step(solver._s, None))
            _lib.check(L.daisy_solver_read(solver._s, _lib.fptr(hB), _lib.fptr(hR)))
        torch.cuda.synchronize()
        e2e_s = (time.time() - t0) / nst
        e2e = {"value": 1.0 / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": int(2 * K * N * 4), "d2h_bytes_per_step": int(2 * K * N * 4)}
    else:
        # multi-GPU: every rank uploads ONLY its own rows of B and of the residual from pinned host memory (the residual slices
        # reach the other ranks over NVLink like the output of a pass), runs one pass through the public API (exchange
        # included) and reads back its slices plus the band sums
        hBl = torch.empty((K, nloc), dtype=torch.float32, pin_memory=True).numpy()
        hRl = torch.empty((K, nloc), dtype=torch.float32, pin_memory=True).numpy()
        hRin = torch.empty((K, nloc), dtype=torch.float32, pin_memory=True).numpy()
        hR = torch.empty((K, N), dtype=torch.float32, pin_memory=True).numpy()
        hBl[:] = E[:, r0:r1]; hRin[:] = E[:, r0:r1]; hR[:] = E
        sliced = not args.no_fused
        def e2e_step():
            if sliced:
                _lib.check(L.daisy_solver_write_slices(solver._s, _lib.fptr(hBl), _lib.fptr(hRin)))
            else:
                _lib.check(L.daisy_solver_write_partitioned(solver._s, _lib.fptr(hBl), _lib.fptr(hR)))
            solver.step(True)
            _lib.check(L.daisy_solver_read(solver._s, _lib.fptr(hBl), _lib.fptr(hRl)))
        for _ in range(2):
            e2e_step()
        hBl[:] = E[:, r0:r1]; hR[:] = E
        barrier()
        t0 = time.time()
        nst = min(args.steps, 50)
        for _ in range(nst):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = allmax((time.time() - t0) / nst)
        h2d = (2 * K * N * 4) if sliced else int(world * (K * N + K * nloc) * 4)
        e2e = {"value": 1.0 / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(world * (2 * K * nloc * 4 + 8 * K * world))}

    # ---- whole solve with the reference's stop rule (SpectralLightning::converge_lightning, Lightning.h:145-151:
    # iterate while the residual summed over bands and patches exceeds 200), band sums read back every pass
    barrier()
    solver.reset()
    t0 = time.time()
    conv_passes = solver.converge(200.0, per_band=False, max_passes=2000)
    torch.cuda.synchronize()
    conv_s = allmax(time.time() - t0)

    parity = None
    if not args.no_parity:
        try:
            parity = parity_block(optixP, solver, sc, uv, E, M, K, world, rank, torch, name)
        except Exception as ex:
            if world > 1:
                raise  # a rank that drops out of the collectives would hang the others
            parity = {"failed": repr(ex)}
    incumbent = None
    if world == 1 and rank == 0 and not args.no_incumbent:
        try:
            incumbent = incumbent_block(dz, uv)
        except Exception as ex:
            incumbent = {"unavailable": repr(ex)}

    # ---- closest hit (optixQuery) through host buffers: the camera rays of an 800 x 600 window, 4 samples per pixel
    closest = None
    if world == 1 and rank == 0:
        try:
            from daisyriot_b200 import api as dzapi
            cam = dzapi.Camera(800, 600, 4)
            lo, hi = sc.vertices.min(0), sc.vertices.max(0)
            mid = (np.float32(0.5) * (lo + hi)).astype(np.float32)
            cam.dir = mid.copy()
            cam.eye = np.array([mid[0], mid[1], hi[2] + np.float32(1.6) * (hi[2] - lo[2])], np.float32)
            gen = np.ascontiguousarray(cam.gen_rays_for_screen(True), np.float32)
            nr = gen.reshape(-1, 6).shape[0]
            # pinned host buffers on both sides, as for the gather's host-buffer steps
            from daisyriot_b200.api import HIT_DTYPE
            cam_rays = torch.empty(gen.size, dtype=torch.float32, pin_memory=True).numpy()
            cam_rays[:] = gen.reshape(-1)
            hits = torch.empty(nr * HIT_DTYPE.itemsize, dtype=torch.uint8, pin_memory=True).numpy().view(HIT_DTYPE)
            optixP.optixQuery(nr, cam_rays, hits)
            ts = []
            for _ in range(3):
                t0 = time.time(); optixP.optixQuery(nr, cam_rays, hits); ts.append(time.time() - t0)
            closest = {"metric": "closest_hit_rays_per_s through pinned host buffers (daisy_query_closest: H2D 24 B/ray, D2H 16 B/ray)", "rays": int(nr),
                       "value": nr / min(ts), "seconds": min(ts), "hit_fraction": float((hits["t"] > 0).mean())}
        except Exception as ex:
            closest = {"failed": repr(ex)}

    cpu_baseline = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        try:
            r = cpu_reference_run(sc, wl, K, budget_s=args.cpu_budget, steps=3, coeff_dir=tmp)
            cpu_baseline = {"value": r["it_per_s"], "unit": "iterations/s", "cores": 1, "kind": r["gather_kind"],
                            "sample": f"Lightning.h+Eigen pass on {r['ff_rows']} of {N} matrix rows ({r.get('gather_sample_nnz')} nnz), SpMV time scaled by N/rows",
                            "formfactor": {"value": r["ff_rays_per_s"], "unit": "rays/s", "cores": r["cores_ff"], "kind": "port",
                                           "sample": f"{r['ff_rows']} rows, {r['ff_rays']} rays in {r['ff_seconds']:.1f} s"}}
        except Exception as ex:  # the baseline is a reported extra; never let it kill the measurement
            cpu_baseline = {"value": None, "unit": "iterations/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        line = {
            "metric": "radiosity_gather_iterations_per_s", "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "reference example scene (tests/golden fixture)" if name in FIXTURE_SCENES else "synthetic",
            "config": bench_config(name, N, K, uv.shape[0], world),
            "e2e": e2e, "gpu_launches": int(L.daisy_solver_launches_per_pass(solver._s) * args.steps),
            "clocks": clocks,
            "roofline": {"kernel": ("k_split_residual+k_gather_mma+k_gather_epilogue" if K > 9 else "k_gather_tma (epilogue fused)"), "bound": "hbm", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_note": "hbm_gbs is a copy (read+write) bandwidth; this kernel only reads, so frac can exceed 1", "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback",
                         "kernel_ms": k_ms, "kernel_ms_isolated_launch": k_ms_isolated, "chained_passes": bool(chained and K <= 9),
                         "algorithmic_bytes": alg_bytes},
            "cpu_baseline": cpu_baseline,
            "formfactor": {"metric": "formfactor_visibility_rays_per_s", "value": rays / (ff_ms * 1e-3), "unit": "rays/s",
                           "pairs_facing": int(pairs_unique), "pairs_traced_all_ranks": int(pairs_traced), "rays": int(rays), "kernel_ms": ff_ms,
                           "lbvh_build_ms": lbvh_ms, "e2e_wall_s": ff_wall,
                           "e2e_rays_per_s": rays / ff_wall,
                           "roofline": ff_roof, "clocks": ff_clocks,
                           "ncu": ff_ncu},  # pipe / cache utilisation of the traversal kernel from the committed ncu capture of this workload
            "parity": parity, "incumbent": incumbent, "closest_hit": closest,
            "converge": {"rule": "sum of residual over bands and patches <= 200 (Lightning.h:145-151)", "passes": int(conv_passes),
                         "seconds": conv_s, "total_with_formfactors_s": conv_s + ff_wall},
        }
        print(json.dumps(line))
    solver.close()
    optixP.close()
    if world > 1:
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DAISY_WORKLOAD", "cornell_128k"), choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU form-factor sampling for the baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison of the sampled rows")
    ap.add_argument("--no-incumbent", action="store_true", help="skip the timing of the reference's own calculateRow kernel")
    ap.add_argument("--no-chained", action="store_true", help="one GPU: per-pass events and plain stream order between passes (no programmatic dependent launch)")
    ap.add_argument("--no-fused", action="store_true", help="multi-GPU: NCCL all-gather per pass instead of the epilogue kernel's peer stores")
    ap.add_argument("--no-peer-tiles", action="store_true", help="multi-GPU: trace every tile touching this rank's rows instead of exchanging mirrored tiles")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write B, residual and band sums after the last timed pass as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
