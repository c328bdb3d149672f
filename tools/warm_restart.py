"""Warm restart (daisy_solver_restart + converge) against a cold converge (daisy_solver_reset + converge) after a scene change.

For every workload (cornell_32k, cornell_128k, fluor_64k_k32: the benchmark's inputs, spectral rule: total over bands <= 200),
starting from the converged solve of the unchanged scene, four changes:
  (a) lamp:    the lamp moved (scenes.cornell_moved on CORNELL_LAMP) + daisy_formfactors_update
  (b) block:   the short block moved (CORNELL_SHORT_BLOCK) + daisy_formfactors_update
  (c) emission: the emission halved (daisy_solver_set_emission)
  (d) material: one material's matrix darkened to half (daisy_solver_set_materials)
and for each the passes and wall time (host clock around the blocking calls; the matrix update is not part of it) of
  cold: reset + converge,   warm: restart from the converged B of the old scene + converge,
both through the host loop (daisy_solver_converge) and the device converge (daisy_solver_converge_device), the distance between
the warm and the cold result, sum |r0| of the restart pass against sum E, and the contraction estimate of the passes saved,
log(sum E / sum |r0|) / log(1 / rho) with rho = (threshold / sum E)^(1 / cold passes).  Prints one JSON line; --out writes it.
A workload whose cold solve does not converge (B overflows to Inf / NaN, and the reference's rule, NaN > 200 being false, stops
it) is recorded with the count of non-finite entries of the old solution; its warm numbers mean nothing.

    python tools/warm_restart.py [--workloads cornell_32k,cornell_128k,fluor_64k_k32] [--rounds 1] [--out profiles/x.json]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MAX_PASSES = 2000
THRESHOLD, PER_BAND = 200.0, 0
CASES = ("lamp", "block", "emission", "material")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cornell_32k,cornell_128k,fluor_64k_k32")
    ap.add_argument("--rounds", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, scenes
    L = _lib.lib()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    dp = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
    results = []
    for name in args.workloads.split(","):
        sc, wl, E, M, _ = bench.make_workload(name)
        E = np.ascontiguousarray(E, np.float32)
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(sc.mat_idx, np.int32)
        N, K = sc.numtriangles, E.shape[0]
        p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=dz.msvc_sample_pattern(1))
        p.cudaCalculateRadiosityMatrix()
        s = C.c_void_p()
        _lib.check(L.daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)))

        def read():
            B, R = np.empty((K, N), np.float32), np.empty((K, N), np.float32)
            _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
            return B, R

        def converge(device):
            n = C.c_int()
            fn = L.daisy_solver_converge_device if device else L.daisy_solver_converge
            _lib.check(fn(s, THRESHOLD, PER_BAND, MAX_PASSES, C.byref(n)))
            return n.value

        def arm(warm, device, B0):
            t0 = time.perf_counter()
            if warm:
                _lib.check(L.daisy_solver_restart(s, _lib.fptr(B0)))
            else:
                _lib.check(L.daisy_solver_reset(s))
            n = converge(device)
            return n, (time.perf_counter() - t0) * 1e3

        _lib.check(L.daisy_solver_reset(s))
        converge(False)
        B_old, _ = read()
        nonfinite = int(np.count_nonzero(~np.isfinite(B_old)))  # a cold solve that overflowed: the stop rule's NaN > 200 is false
        diffuse = [i for i in range(M.shape[0]) if i != 0 and np.count_nonzero(mat == i) > 0]
        recolour = max(diffuse, key=lambda i: np.count_nonzero(mat == i))  # the most common non-lamp material
        M2 = M.copy()
        M2[recolour] = (M2[recolour] * np.float32(0.5)).astype(np.float32)
        for case in CASES:
            if case in ("lamp", "block"):
                v, nrm = scenes.cornell_moved(sc, scenes.CORNELL_LAMP if case == "lamp" else scenes.CORNELL_SHORT_BLOCK,
                                              offset=(0.3, 0.0, 0.2) if case == "lamp" else (0.3, 0.0, 0.3))
                p.updateGeometry(v, nrm)
                p.updateRadiosityMatrix()
            elif case == "emission":
                _lib.check(L.daisy_solver_set_emission(s, _lib.fptr(np.ascontiguousarray(E * np.float32(0.5)))))
            else:
                _lib.check(L.daisy_solver_set_materials(s, _lib.fptr(M2), M2.shape[0], _lib.iptr(mat)))
            arm(False, False, None)  # warm-up: the tile scan of a changed matrix, first launches
            r0 = np.zeros(K)
            _lib.check(L.daisy_solver_restart(s, _lib.fptr(B_old)))
            _lib.check(L.daisy_solver_band_sums(s, dp(r0)))
            res = {}
            for warm in (False, True):
                for device in (False, True):
                    runs = [arm(warm, device, B_old) for _ in range(args.rounds)]
                    res[("warm" if warm else "cold") + ("_device" if device else "_host")] = {
                        "passes": runs[0][0], "wall_ms": float(np.median([r[1] for r in runs])), "wall_ms_rounds": [round(r[1], 3) for r in runs]}
                    B, _ = read()
                    if warm and not device:
                        Bw = B.astype(np.float64)
                    if not warm and not device:
                        Bc = B.astype(np.float64)
            e_sum = float(_lib_sum(L, s, K, dp))
            pc = res["cold_host"]["passes"]
            rho = (THRESHOLD / e_sum) ** (1.0 / pc) if pc > 0 and e_sum > THRESHOLD else None
            r0_sum = float(r0.sum())
            est = math.log(e_sum / r0_sum) / math.log(1.0 / rho) if rho and 0 < rho < 1 and r0_sum > 0 else None
            r = {"workload": name, "case": case, "N": N, "K": K, "threshold": THRESHOLD, "per_band": PER_BAND,
                 "old_solution_nonfinite_entries": nonfinite, **res,
                 "passes_saved_host": res["cold_host"]["passes"] - res["warm_host"]["passes"],
                 "sum_E": e_sum, "sum_abs_r0": r0_sum, "rho_estimate": rho, "passes_saved_estimate": est,
                 "warm_vs_cold": {"max_abs": float(np.abs(Bw - Bc).max()), "max_abs_rel_to_max_B": float(np.abs(Bw - Bc).max() / np.abs(Bc).max()),
                                  "sum_abs_rel": float(np.abs(Bw - Bc).sum() / np.abs(Bc).sum())}}
            print(json.dumps(r), flush=True)
            results.append(r)
            # back to the unchanged scene
            if case in ("lamp", "block"):
                p.updateGeometry(sc.vertices, sc.normals)
                p.updateRadiosityMatrix()
            elif case == "emission":
                _lib.check(L.daisy_solver_set_emission(s, _lib.fptr(E)))
            else:
                _lib.check(L.daisy_solver_set_materials(s, _lib.fptr(M), M.shape[0], _lib.iptr(mat)))
        L.daisy_solver_destroy(s)
        p.close()
    out = {"tool": "tools/warm_restart.py", "device": smi, "rounds": args.rounds, "timer": "host clock around the blocking calls",
           "results": results}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def _lib_sum(L, s, K, dp):
    """sum over bands of the current emission's band sums: the band sums right after a reset"""
    from daisyriot_b200 import _lib
    v = np.zeros(K)
    _lib.check(L.daisy_solver_reset(s))
    _lib.check(L.daisy_solver_band_sums(s, dp(v)))
    return v.sum()


if __name__ == "__main__":
    main()
