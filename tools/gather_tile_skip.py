"""Tile skipping in the fused K <= 9 gather: how much of F a pass streams, and what that buys.

Prints, for one workload of bench.py on one GPU:
  * tile occupancy of the 64-row x 256-column tiles the kernel loads (from the solver's own scan): overall, per band of rows
    (--band rows, default 8192 = one quad of the Cornell box at 128K), and per rank of 2- and 8-way row partitions;
  * F bytes streamed per pass with skipping against the dense matrix, and the device time of the scan;
  * ms per pass (daisy_solver_last_step_ms: CUDA events around one pass) of a skipping and a dense solver on the same matrix,
    alternated --rounds times in this process;
  * the device name and power limit, read in the same run.

    python tools/gather_tile_skip.py [--workload cornell_128k] [--rounds 3] [--passes 30]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TROWS, TCOLS = 64, 256


def solver(dz, _lib, p, K, E, M, mat, skip):
    os.environ["DAISY_GATHER_SKIP"] = "1" if skip else "0"  # read when the solver is planned
    s = C.c_void_p()
    _lib.check(_lib.lib().daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(s)))
    return s


def pass_ms(_lib, s, K, passes):
    L = _lib.lib()
    sums = np.zeros(K)
    ms = []
    for _ in range(passes):
        _lib.check(L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double))))
        m = C.c_double()
        _lib.check(L.daisy_solver_last_step_ms(s, C.byref(m)))
        ms.append(m.value)
    return float(np.mean(ms[len(ms) // 3:]))  # the first third warms up


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cornell_128k")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--passes", type=int, default=30)
    ap.add_argument("--band", type=int, default=8192, help="rows per band of the per-band occupancy")
    args = ap.parse_args()
    import bench
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, dist
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    sc, _, E, M, _ = bench.make_workload(args.workload)
    N, K, _ = bench.WORKLOADS[args.workload]
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=dz.msvc_sample_pattern(1))
    p.cudaCalculateRadiosityMatrix()
    L = _lib.lib()
    s_skip = solver(dz, _lib, p, K, E, M, sc.mat_idx, True)
    s_dense = solver(dz, _lib, p, K, E, M, sc.mat_idx, False)
    dims = np.zeros(2, np.int32)
    _lib.check(L.daisy_solver_tile_map(s_skip, _lib.iptr(dims), None, 0, None, None))
    nrb, S = int(dims[0]), int(dims[1])
    occ = np.zeros(nrb * S, np.uint8)
    occupied, scan_ms = C.c_int64(), C.c_double()
    _lib.check(L.daisy_solver_tile_map(s_skip, _lib.iptr(dims), occ.ctypes.data_as(C.POINTER(C.c_uint8)), occ.size, C.byref(occupied),
                                       C.byref(scan_ms)))
    occ = occ.reshape(nrb, S).astype(bool)
    ld = C.c_int64()
    _lib.check(L.daisy_formfactors_ld(p._ctx, C.byref(ld)))
    # bytes inside the matrix extent (nloc x ldF) of every tile: what the TMA unit reads from memory
    h = np.minimum(TROWS, N - np.arange(nrb) * TROWS)
    w = np.minimum(TCOLS, ld.value - np.arange(S) * TCOLS)
    tile_bytes = 4.0 * h[:, None] * w[None, :]
    streamed, dense = float((tile_bytes * occ).sum()), float(tile_bytes.sum())
    bands = [float(occ[b // TROWS:(b + args.band) // TROWS].mean()) for b in range(0, N, args.band)]
    ranks = {}
    for G in (2, 8):
        fr = []
        for r in range(G):
            r0, r1, _ = dist.partition(N, r, G)
            fr.append(float(occ[r0 // TROWS:(r1 + TROWS - 1) // TROWS].mean()) if r1 > r0 else 0.0)
        ranks[G] = fr
    timings = {"skip": [], "dense": []}
    for _ in range(args.rounds):
        timings["skip"].append(pass_ms(_lib, s_skip, K, args.passes))
        timings["dense"].append(pass_ms(_lib, s_dense, K, args.passes))
    ms_skip, ms_dense = float(np.median(timings["skip"])), float(np.median(timings["dense"]))
    out = {
        "workload": args.workload, "device": smi, "tiles": [nrb, S], "tile": [TROWS, TCOLS],
        "occupancy": float(occ.mean()), "occupied_tiles": int(occupied.value),
        "occupancy_per_band": {"rows_per_band": args.band, "values": [round(b, 4) for b in bands]},
        "occupancy_per_rank": {str(G): [round(v, 4) for v in fr] for G, fr in ranks.items()},
        "F_bytes_streamed": streamed, "F_bytes_dense": dense, "scan_ms": scan_ms.value,
        "ms_per_pass": timings, "ms_per_pass_median": {"skip": ms_skip, "dense": ms_dense}, "speedup": ms_dense / ms_skip,
        "streamed_GBs": {"skip": streamed / (ms_skip * 1e-3) / 1e9, "dense": dense / (ms_dense * 1e-3) / 1e9},
    }
    print(json.dumps(out))
    L.daisy_solver_destroy(s_skip)
    L.daisy_solver_destroy(s_dense)
    p.close()


if __name__ == "__main__":
    main()
