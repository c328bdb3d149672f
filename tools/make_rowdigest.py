"""GPU box: build the matrix of a bench workload and save its per-row digests (exact integer digests computed on the device,
daisy_formfactors_row_digest) as gpurun_out/rowdigest_<workload>.npz -- committed under tests/golden/ and checked by every rank of
every bench run (bench.py parity.digest), so that 1-, 2-, 4- and 8-GPU builds are proven to produce the same matrix.

    python tools/make_rowdigest.py cornell_32k cornell_128k ...
"""
import os
import sys

import numpy as np

sys.path.insert(0, ".")
import bench  # noqa: E402
import daisyriot_b200 as dz  # noqa: E402

for name in sys.argv[1:]:
    sc, wl, E, M, tmp = bench.make_workload(name)
    uv = dz.msvc_sample_pattern(1)
    p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), rands=uv)
    rm = p.cudaCalculateRadiosityMatrix()
    _, w = rm.row_digest()
    st = p.stats()
    out = os.path.join("gpurun_out", f"rowdigest_{name}.npz")
    np.savez_compressed(out, digest=bench.row_digest32(w), pairs=np.int64(st["pairs_traced"]), patches=np.int64(sc.numtriangles))
    print(name, "pairs", st["pairs_traced"], "ff_ms %.1f" % st["ff_ms"], "->", out, os.path.getsize(out), "bytes", flush=True)
    p.close()
