"""GPU box: matrix updates after a geometry change against a full build on the same moved geometry.

    python tools/ff_update.py OUT.json [--sizes 32768 131072] [--gpus 1 8]

Scenarios on the synthetic Cornell box (scenes.cornell_box): the lamp moved 0.25 in x, the short block moved 0.3 in z, and
a no-op update.  For each: triangles changed, tiles and pairs re-traced and their share of the facing pairs, host rebuild
(daisy_ctx_update_geometry wall time), LBVH, classification and kernel milliseconds, update wall time against a fresh full
build of the moved geometry, and whether the row digests of the two matrices are equal."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402

import daisyriot_b200 as dz  # noqa: E402
from daisyriot_b200 import scenes  # noqa: E402

SCENARIOS = {
    "lamp_x+0.25": lambda sc: scenes.cornell_moved(sc, scenes.CORNELL_LAMP, offset=(0.25, 0.0, 0.0)),
    "short_block_z+0.3": lambda sc: scenes.cornell_moved(sc, scenes.CORNELL_SHORT_BLOCK, offset=(0.0, 0.0, 0.3)),
    "noop": lambda sc: (np.array(sc.vertices, np.float32), np.array(sc.normals, np.float32)),
}


def _digest(obj, ndev):
    if ndev == 1:
        return dz.RadMat(obj).row_digest()
    xs, ws = [], []
    for i in range(ndev):
        v = obj.device(i)
        r0, r1 = v.row_range
        if r1 > r0:
            x, w = dz.RadMat(v).row_digest()
            xs.append(x); ws.append(w)
    return np.concatenate(xs), np.concatenate(ws)


def _make(mesh, uv, ndev):
    return dz.OptixPrimeFunctionality(mesh, rands=uv) if ndev == 1 else dz.DeviceGroup(mesh, ndev=ndev, rands=uv)


def _sync_wall(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3  # every entry point is blocking


def run(n, ndev):
    uv = scenes.msvc_sample_pattern(1)
    sc = scenes.cornell_box(n)
    out = []
    for name, move in SCENARIOS.items():
        V, VN = move(sc)
        moved = scenes.Scene(V, VN, sc.tri, sc.mat_idx, sc.materials, sc.name + "*")
        # full build on the moved geometry: the reference numbers and digests
        fresh = _make(dz.MeshS.from_scene(moved), uv, ndev)
        full_ms = _sync_wall(fresh.cudaCalculateRadiosityMatrix)
        st_full = fresh.stats()
        d_full = _digest(fresh, ndev)
        fresh.close()
        # build on the original geometry, move, update
        obj = _make(dz.MeshS.from_scene(sc), uv, ndev)
        obj.cudaCalculateRadiosityMatrix()
        if ndev == 1:
            rebuild_ms = _sync_wall(lambda: obj.updateGeometry(V, VN))
            upd_ms = _sync_wall(lambda: obj.updateRadiosityMatrix(dz.FF_DEVICE))
            us, st = obj.update_stats(), obj.stats()
            tiles, pairs, cls_ms, lbvh_ms, ff_ms = us["tiles_retraced"], us["pairs_retraced"], us["classify_ms"], st["lbvh_ms"], st["ff_ms"]
        else:
            rebuild_ms = _sync_wall(lambda: obj.update_geometry(V, VN))
            upd_ms = _sync_wall(lambda: obj.updateRadiosityMatrix(dz.FF_DEVICE))
            per = [obj.device(i) for i in range(ndev)]
            ups = [v.update_stats() for v in per]
            sts = [v.stats() for v in per]
            tiles = sum(u["tiles_retraced"] for u in ups)
            pairs = sum(u["pairs_retraced"] for u in ups)
            cls_ms = max(u["classify_ms"] for u in ups)
            lbvh_ms = max(s["lbvh_ms"] for s in sts)
            ff_ms = max(s["ff_ms"] for s in sts)
            us = ups[0]
        d_upd = _digest(obj, ndev)
        facing = st_full["pairs_traced"] if ndev == 1 else st_full["pairs"]
        rec = {"scenario": name, "patches": n, "gpus": ndev, "tris_changed": us["tris_changed"], "tiles_retraced": tiles,
               "pairs_retraced": pairs, "facing_pairs": facing, "fraction_of_facing_pairs": pairs / facing if facing else 0.0,
               "host_rebuild_ms": rebuild_ms, "lbvh_ms": lbvh_ms, "classify_ms": cls_ms, "kernel_ms": ff_ms,
               "update_wall_ms": upd_ms, "full_build_wall_ms": full_ms, "full_build_kernel_ms": st_full["ff_ms"],
               "digest_equal": bool(np.array_equal(d_upd[0], d_full[0]) and np.array_equal(d_upd[1], d_full[1]))}
        print(json.dumps(rec), flush=True)
        out.append(rec)
        obj.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--sizes", type=int, nargs="+", default=[32768, 131072])
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 8])
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else "unknown", "gpus_visible": int(dz.lib().daisy_device_count()), "runs": []}
    for ndev in a.gpus:
        if ndev > res["gpus_visible"]:
            continue
        for n in a.sizes:
            res["runs"] += run(n, ndev)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
