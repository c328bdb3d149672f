"""Pass time of the tcgen05 3xTF32 gather at K = 32, 41 and 64 bands on one matrix.

For each size (Cornell box with 10 fluorescent materials, form factors built on the GPU) three solvers share the matrix and
are alternated --rounds times in this process: reset, --warmup passes, then --passes passes each timed by CUDA events
(daisy_solver_last_step_ms: residual split + tensor-core pass + epilogue).  Reported per K:
  * ms per pass (median over the rounds of each round's median);
  * F bytes streamed per pass over that time, and its fraction of the 6.55 TB/s copy peak (F is read once per pass, so
    a pass that streamed it twice would show half the rate);
  * tensor FLOP/s of the three TF32 products over the padded band count the kernel runs (K = 41 runs as 64), against the
    data sheet's 1 125 TFLOP/s dense TF32;
  * the split residual [Rh;Rl] that every stage reads from L2 (2 x Kp x 4 bytes per column);
  * parity: one pass from E on a fresh reset, sampled rows against FP64 (max relative error above 1e-6 of the band maximum).
The device name, power limit and maximum SM clock are read in the same run.  Writes one JSON line to stdout and, with --out,
to that file.

    python tools/gather_wide_bands.py [--sizes 65536,131072] [--rounds 3] [--warmup 5] [--passes 25] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KS = (32, 41, 64)
COPY_PEAK = 6.55e12
TF32_PEAK = 1.125e15
SAMPLE_ROWS = 96


def inputs(sc, K, model):
    """E and M as bench.py builds them for its spectral workloads: the materials' spectra at K wavelengths from 200 to 600 nm,
    fluorescent materials with a dense perturbation of their re-emission matrix"""
    import bench
    from daisyriot_b200 import materials
    wl = bench.wavelengths_for(K)
    mats = materials.make_materials(sc.materials, wl, model)
    rng = np.random.RandomState(0x5EED)
    for m in mats:
        if m.kind == "fluorescent":
            m.M = (m.M * 0.6 + rng.uniform(0, 0.4 / K, (K, K))).astype(np.float32)
    return materials.spectral_inputs(mats, sc.mat_idx, 7.0)


def pass_ms(L, s, K, warmup, passes):
    sums = np.zeros(K)
    L.daisy_solver_reset(s)
    ms = []
    for i in range(warmup + passes):
        rc = L.daisy_solver_step(s, sums.ctypes.data_as(C.POINTER(C.c_double)))
        assert rc == 0, (K, rc, L.daisy_last_error())
        m = C.c_double()
        L.daisy_solver_last_step_ms(s, C.byref(m))
        if i >= warmup:
            ms.append(m.value)
    return float(np.median(ms))


def parity(L, _lib, s, K, E, M, mat, F_rows, rows):
    """one pass from E: residual of the sampled rows against FP64, max relative error over entries above 1e-6 of the max"""
    assert L.daisy_solver_reset(s) == 0
    assert L.daisy_solver_step(s, None) == 0
    N = E.shape[1]
    B, R = np.empty((K, N), np.float32), np.empty((K, N), np.float32)
    _lib.check(L.daisy_solver_read(s, _lib.fptr(B), _lib.fptr(R)))
    b = F_rows.astype(np.float64) @ E.astype(np.float64).T                 # rows x K
    want = np.einsum("pjk,pj->pk", M.astype(np.float64)[mat[rows]], b).T   # K x rows (M column-major)
    got = R[:, rows].astype(np.float64)
    floor = 1e-6 * float(np.abs(want).max())
    big = np.abs(want) > floor
    return float((np.abs(got - want)[big] / np.abs(want)[big]).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="65536,131072")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--passes", type=int, default=25)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import daisyriot_b200 as dz
    from daisyriot_b200 import _lib, dist, rgb2spec, scenes
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    with tempfile.TemporaryDirectory(prefix="daisy_wide_") as tmp:
        os.makedirs(os.path.join(tmp, "color_tables"))
        coeff = os.path.join(tmp, "color_tables", "srgb.coeff")
        rgb2spec.write_surrogate_table(coeff, 16)
        model = rgb2spec.RGB2Spec.load(coeff)
    L = _lib.lib()
    out = {"device": smi, "rounds": args.rounds, "warmup": args.warmup, "passes_timed": args.passes, "copy_peak_Bs": COPY_PEAK,
           "tf32_peak_flops": TF32_PEAK, "sizes": {}}
    for N in [int(x) for x in args.sizes.split(",")]:
        sc = scenes.cornell_box(N, n_fluorescent=10)
        p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), device=0, rands=scenes.msvc_sample_pattern(1))
        rm = p.cudaCalculateRadiosityMatrix()
        ld = C.c_int64()
        _lib.check(L.daisy_formfactors_ld(p._ctx, C.byref(ld)))
        rows = np.unique(np.linspace(0, N - 1, SAMPLE_ROWS).astype(np.int64))
        F_rows = np.concatenate([rm.rows(int(r), 1) for r in rows])
        solvers, ins = {}, {}
        for K in KS:
            E, M = inputs(sc, K, model)
            ins[K] = (E, M)
            s = C.c_void_p()
            _lib.check(L.daisy_solver_create(p._ctx, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(sc.mat_idx), C.byref(s)))
            assert L.daisy_solver_launches_per_pass(s) == 3
            solvers[K] = s
        times = {K: [] for K in KS}
        for _ in range(args.rounds):
            for K in KS:
                times[K].append(pass_ms(L, solvers[K], K, args.warmup, args.passes))
        fbytes = 4.0 * N * ld.value
        res = {"patches": N, "ldF": ld.value, "F_bytes": fbytes, "per_K": {}}
        for K in KS:
            Kp = dist.padded_K(K)
            ms = float(np.median(times[K]))
            flops = 3 * 2.0 * N * ld.value * Kp
            res["per_K"][str(K)] = {
                "padded_K": Kp, "ms_per_pass": ms, "ms_per_pass_rounds": times[K],
                "F_Bs": fbytes / (ms * 1e-3), "frac_copy_peak": fbytes / (ms * 1e-3) / COPY_PEAK,
                "tensor_flops": flops / (ms * 1e-3), "frac_tf32_peak": flops / (ms * 1e-3) / TF32_PEAK,
                "split_residual_bytes": 2.0 * Kp * 4 * ((N + 63) // 64 * 64),
                "parity_max_rel": parity(L, _lib, solvers[K], K, *ins[K], sc.mat_idx, F_rows, rows),
            }
        k32 = res["per_K"]["32"]["ms_per_pass"]
        res["ms_ratio_to_k32"] = {str(K): res["per_K"][str(K)]["ms_per_pass"] / k32 for K in KS}
        out["sizes"][str(N)] = res
        for s in solvers.values():
            L.daisy_solver_destroy(s)
        p.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
