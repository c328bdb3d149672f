"""The device converge (daisy_solver_converge_device) against the host loop (daisy_solver_converge) on one GPU.

For every workload: both arms alternate from daisy_solver_reset --rounds times in this process, each converge timed with a host
clock around the blocking call.  Prints one JSON line with, per workload:
  * passes of both arms and whether B and the residual are bit-identical between them;
  * the wall time of both arms (median over the rounds, and every round);
  * the chained pass time (daisy_solver_set_chained, back-to-back passes, host clock over --chained passes) and passes times it;
  * pass-kernel launches of one device converge (torch.profiler), i.e. how many launches found the residual converged;
and the device name and power limit, read in the same run.

Workloads: colorballs and cornellbox_blacklight in spectral (K = 9, total over bands <= 200), RGB (K = 3, every band <= 1e-4)
and BW (K = 1, 1e-4) mode with materials.*_inputs (cornellbox_blacklight has no RGB emitter: its most common material glows
(0.2, 0.1, 0.05), as the 2 048-patch box of test_gpu_parity.py does), then cornell_32k, cornell_128k and fluor_64k_k32.

    python tools/converge_device.py [--rounds 3] [--workloads colorballs,cornell_32k] [--out profiles/x.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCENES = ("colorballs", "cornellbox_blacklight")
LARGE = ("cornell_32k", "cornell_128k", "fluor_64k_k32")
MAX_PASSES = 1000


def modes_for(bench, name):
    """(mode, K, E, M, threshold, per_band) of a workload"""
    import bench as _b
    from daisyriot_b200 import materials, rgb2spec
    sc, wl, E, M, tmp = _b.make_workload(name)
    out = [("spectral", E.shape[0], E, M, 200.0, 0)]
    if name in SCENES:
        mats = materials.make_materials(sc.materials, wl, rgb2spec.RGB2Spec.load(os.path.join(tmp, "color_tables", "srgb.coeff")))
        if not any(np.any(m.emission > 0) for m in mats):
            mats[int(np.bincount(sc.mat_idx).argmax())].emission[:] = (0.2, 0.1, 0.05)
        Er, Mr = materials.rgb_inputs(mats, sc.mat_idx, 500.0)
        Eb, Mb = materials.bw_inputs(mats, sc.mat_idx, 500.0)
        out += [("rgb", 3, Er, Mr, 1e-4, 1), ("bw", 1, Eb, Mb, 1e-4, 1)]
    return sc, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chained", type=int, default=60, help="passes of the chained-pass timing")
    ap.add_argument("--workloads", default=",".join(SCENES + LARGE))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib
    L = _lib.lib()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    dp = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
    results = []
    for name in args.workloads.split(","):
        sc, modes = modes_for(bench, name)
        p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=dz.msvc_sample_pattern(1))
        p.cudaCalculateRadiosityMatrix()
        N = sc.numtriangles
        for mode, K, E, M, thr, per_band in modes:
            E = np.ascontiguousarray(E, np.float32)
            M = np.ascontiguousarray(M, np.float32)
            s = C.c_void_p()
            _lib.check(L.daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(sc.mat_idx), C.byref(s)))

            def run(fn):
                _lib.check(L.daisy_solver_reset(s))
                n = C.c_int()
                t0 = time.perf_counter()
                _lib.check(fn(s, thr, per_band, MAX_PASSES, C.byref(n)))
                ms = (time.perf_counter() - t0) * 1e3
                B, R = np.empty((K, N), np.float32), np.empty((K, N), np.float32)
                _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
                return n.value, ms, B, R

            run(L.daisy_solver_converge)  # warm-up: module load, tile scan, first launches
            run(L.daisy_solver_converge_device)
            arms = {"host": [], "device": []}
            identical = True
            for _ in range(args.rounds):
                nh, mh, Bh, Rh = run(L.daisy_solver_converge)
                nd, md, Bd, Rd = run(L.daisy_solver_converge_device)
                arms["host"].append((nh, mh))
                arms["device"].append((nd, md))
                identical = identical and nh == nd and np.array_equal(Bh.view(np.uint32), Bd.view(np.uint32)) and \
                    np.array_equal(Rh.view(np.uint32), Rd.view(np.uint32))
            passes = arms["host"][0][0]
            # chained pass: back-to-back passes without a host decision, host clock over the whole run (band_sums synchronises)
            _lib.check(L.daisy_solver_set_chained(s, 1))
            sums = np.zeros(K)
            _lib.check(L.daisy_solver_reset(s))
            for _ in range(5):
                _lib.check(L.daisy_solver_step(s, None))
            _lib.check(L.daisy_solver_band_sums(s, dp(sums)))
            t0 = time.perf_counter()
            for _ in range(args.chained):
                _lib.check(L.daisy_solver_step(s, None))
            _lib.check(L.daisy_solver_band_sums(s, dp(sums)))
            chained_ms = (time.perf_counter() - t0) * 1e3 / args.chained
            _lib.check(L.daisy_solver_set_chained(s, 0))
            launches = None
            try:  # pass-kernel launches of one device converge
                import torch
                from torch.profiler import ProfilerActivity, profile
                _lib.check(L.daisy_solver_reset(s))
                n = C.c_int()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    _lib.check(L.daisy_solver_converge_device(s, thr, per_band, MAX_PASSES, C.byref(n)))
                    torch.cuda.synchronize()
                pass_kernels = ("k_gather_tma", "k_split_residual", "k_gather_partial")
                launches = sum(e.count for e in prof.key_averages() if any(k in e.key for k in pass_kernels) and "k_gather_epilogue" not in e.key)
            except Exception as e:  # the measurement is optional; say why it is missing
                launches = "unavailable: %s" % e
            med = lambda xs: float(np.median([x[1] for x in xs]))
            r = {"workload": name, "mode": mode, "K": K, "N": N, "threshold": thr, "per_band": per_band,
                 "launches_per_pass": L.daisy_solver_launches_per_pass(s),
                 "passes": {"host": [x[0] for x in arms["host"]], "device": [x[0] for x in arms["device"]]},
                 "hit_max_passes": passes >= MAX_PASSES,
                 "wall_ms": {"host": med(arms["host"]), "device": med(arms["device"])},
                 "wall_ms_rounds": {"host": [round(x[1], 4) for x in arms["host"]], "device": [round(x[1], 4) for x in arms["device"]]},
                 "chained_pass_ms": chained_ms, "passes_x_chained_ms": passes * chained_ms,
                 "speedup": med(arms["host"]) / med(arms["device"]) if med(arms["device"]) > 0 else None,
                 "device_converge_pass_launches": launches,
                 "launches_after_deciding_pass": (launches - passes - 1) if isinstance(launches, int) and passes < MAX_PASSES else None,
                 "bit_identical": bool(identical)}
            print(json.dumps(r), flush=True)
            results.append(r)
            L.daisy_solver_destroy(s)
        p.close()
    out = {"tool": "tools/converge_device.py", "device": smi, "rounds": args.rounds, "timer": "host clock around the blocking call",
           "results": results}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
