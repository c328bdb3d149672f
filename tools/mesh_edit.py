"""GPU box: mesh edits (daisy_ctx_replace_mesh + daisy_formfactors_update) against a full build of the edited scene.

    python tools/mesh_edit.py [OUT.json] [--sizes 32768 131072] [--rounds 3]

Edits on the synthetic Cornell box (scenes.cornell_box): the lamp removed, the short block removed, a panel added
(scenes.cornell_panel).  The two arms -- a fresh context built on the edited scene, and a context built on the original scene,
edited and updated -- alternate over the rounds.  Per edit: the fresh build's wall and kernel time and facing pairs; the
replace split into allocation, remap kernel (k_remap_F) and host rebuild (DAISY_TIMING, read from the library's stderr); the
update split into classification and partial kernel; pairs re-traced; and whether the row digests of the two matrices are
equal.  The card's name and power limit are read in the same call."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402

import daisyriot_b200 as dz  # noqa: E402
from daisyriot_b200 import scenes  # noqa: E402


def _quads(sc, quads):
    per = sc.numtriangles // 16
    return np.concatenate([np.arange(q * per, (q + 1) * per) for q in quads])


EDITS = {
    "remove_lamp": lambda sc: scenes.edit_scene(sc, remove=_quads(sc, scenes.CORNELL_LAMP)),
    "remove_short_block": lambda sc: scenes.edit_scene(sc, remove=_quads(sc, scenes.CORNELL_SHORT_BLOCK)),
    "add_panel": lambda sc: scenes.edit_scene(sc, add=scenes.cornell_panel(sc.numtriangles)),
}


def _wall_ms(fn):
    t = time.perf_counter()
    fn()
    return (time.perf_counter() - t) * 1e3  # every entry point is blocking


def _replace_timed(p, mesh, prev):
    """replaceMesh with DAISY_TIMING on, the library's stderr captured: (wall ms, allocation ms, remap ms, host rebuild ms)"""
    os.environ["DAISY_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            wall = _wall_ms(lambda: p.replaceMesh(mesh, prev))
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["DAISY_TIMING"]
        f.seek(0)
        text = f.read()
    m = re.search(r"daisy_ctx_replace_mesh: allocation ([0-9.]+) s, k_remap_F ([0-9.]+) s, host rebuild ([0-9.]+) s", text)
    if not m:
        raise RuntimeError("no timing line from daisy_ctx_replace_mesh: " + text[-400:])
    return wall, 1e3 * float(m.group(1)), 1e3 * float(m.group(2)), 1e3 * float(m.group(3))


def run(n, rounds):
    uv = scenes.msvc_sample_pattern(1)
    sc = scenes.cornell_box(n)
    out = []
    for name, edit in EDITS.items():
        sc_new, prev = edit(sc)
        recs = {"fresh": [], "edit": []}
        digests = {}
        for r in range(rounds):
            # arm 1: a fresh context on the edited scene
            fresh = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc_new), rands=uv)
            ms = _wall_ms(fresh.cudaCalculateRadiosityMatrix)
            st = fresh.stats()
            recs["fresh"].append({"build_wall_ms": ms, "build_kernel_ms": st["ff_ms"], "pairs_traced": st["pairs_traced"]})
            digests["fresh"] = dz.RadMat(fresh).row_digest()
            fresh.close()
            # arm 2: build on the original scene (not timed), replace, update
            p = dz.OptixPrimeFunctionality(dz.MeshS.from_scene(sc), rands=uv)
            p.cudaCalculateRadiosityMatrix()
            wall, alloc_ms, remap_ms, host_ms = _replace_timed(p, dz.MeshS.from_scene(sc_new), prev)
            upd_ms = _wall_ms(lambda: p.updateRadiosityMatrix(dz.FF_DEVICE))
            us, st = p.update_stats(), p.stats()
            recs["edit"].append({"replace_wall_ms": wall, "replace_alloc_ms": alloc_ms, "replace_remap_ms": remap_ms, "replace_host_rebuild_ms": host_ms,
                                 "update_wall_ms": upd_ms, "update_classify_ms": us["classify_ms"], "update_kernel_ms": st["ff_ms"],
                                 "tris_changed": us["tris_changed"], "tiles_retraced": us["tiles_retraced"], "pairs_retraced": us["pairs_retraced"]})
            digests["edit"] = dz.RadMat(p).row_digest()
            p.close()
            print(json.dumps({"edit": name, "patches": n, "round": r, "fresh": recs["fresh"][-1], "edited": recs["edit"][-1]}), flush=True)
        med = lambda arm, k: float(np.median([x[k] for x in recs[arm]]))  # noqa: E731
        facing = recs["fresh"][0]["pairs_traced"]
        rec = {"edit": name, "patches": n, "patches_after": sc_new.numtriangles, "rounds": rounds,
               "tris_added": int((prev < 0).sum()), "tris_removed": n - int((prev >= 0).sum()),
               "fresh_build_wall_ms": med("fresh", "build_wall_ms"), "fresh_build_kernel_ms": med("fresh", "build_kernel_ms"), "facing_pairs": facing,
               **{k: med("edit", k) for k in ("replace_wall_ms", "replace_alloc_ms", "replace_remap_ms", "replace_host_rebuild_ms",
                                               "update_wall_ms", "update_classify_ms", "update_kernel_ms")},
               "pairs_retraced": recs["edit"][0]["pairs_retraced"], "tiles_retraced": recs["edit"][0]["tiles_retraced"],
               "fraction_of_facing_pairs": recs["edit"][0]["pairs_retraced"] / facing if facing else 0.0,
               "digest_equal": bool(np.array_equal(digests["fresh"][0], digests["edit"][0]) and np.array_equal(digests["fresh"][1], digests["edit"][1])),
               "per_round": recs}
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "r09_mesh_edit.json"))
    ap.add_argument("--sizes", type=int, nargs="+", default=[32768, 131072])
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": gpu[0] if gpu else "unknown", "method": "medians over alternating rounds of the two arms; wall times are host clocks around "
           "blocking calls, kernel / classification times CUDA events, remap and host rebuild the library's DAISY_TIMING split", "runs": []}
    for n in a.sizes:
        res["runs"] += run(n, a.rounds)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
