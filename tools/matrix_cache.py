"""GPU box: the matrix-cache path (the reference's matfile, Lightning.h:84-96) timed on the device against the host conversion.

    python tools/matrix_cache.py OUT.json [--rounds 5] [--workloads colorballs cornellbox_blacklight cornell_32k cornell_32k_2gpu]

Per workload, after one form-factor build (device variant):
  * export, daisy_formfactors_to_csc (daisy_group_formfactors_to_csc for the 2-GPU group): the count-only call and the fill
    call, each on the device and with DAISY_CSC_HOST=1 (dense row read-backs converted on the host);
  * import: deserialize_csc + write_csc against deserialize_mat + write_rows, from the same matrix file;
  * the bytes each arm moves over PCIe, computed from N, nnz and the device count;
  * whether both exports and both imports give bit-identical results.
Wall times are medians of alternated rounds (device arm, host arm, device arm, ...), one warm-up call of each arm first.
With shim/_build/shim_demo present (it needs the reference's sources to build), the demo is also timed with a matfile on
cornellbox_blacklight: the first run (build, export, write) and the second (read, import), DAISY_CSC_HOST=1 against default.
That switch selects the export only, so it compares the first runs; the second run loads through write_csc in both arms."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402

import daisyriot_b200 as dz  # noqa: E402
from daisyriot_b200 import _lib, api, scenes  # noqa: E402

WORKLOADS = {  # name: (scene, devices)
    "colorballs": ("colorballs", 1),
    "cornellbox_blacklight": ("cornellbox_blacklight", 1),
    "cornell_32k": ("cornell_32k", 1),
    "cornell_32k_2gpu": ("cornell_32k", 2),
}


def load_scene(name):
    if name in ("colorballs", "cornellbox_blacklight"):
        return scenes.load_scene_npz(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return scenes.cornell_box(32768, n_fluorescent=2)


def set_host(on):
    if on:
        os.environ["DAISY_CSC_HOST"] = "1"
    else:
        os.environ.pop("DAISY_CSC_HOST", None)


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def alternate(arms, rounds):
    """arms: {name: fn}; one warm-up call of each, then `rounds` rounds calling every arm in turn; medians in seconds"""
    for fn in arms.values():
        fn()
    t = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            t[k].append(timed(fn)[0])
    return {k: {"median_s": statistics.median(v), "all_s": v} for k, v in t.items()}


def run_workload(name, rounds, tmp):
    scene_name, ndev = WORKLOADS[name]
    sc = load_scene(scene_name)
    N = sc.numtriangles
    uv = scenes.msvc_sample_pattern(1)
    mesh = dz.MeshS.from_scene(sc)
    L = _lib.lib()
    if ndev == 1:
        obj = dz.OptixPrimeFunctionality(mesh, device=0, rands=uv)
        obj.cudaCalculateRadiosityMatrix()
        to_csc_fn, handle = L.daisy_formfactors_to_csc, obj._ctx
        load_csc = obj.loadRadiosityMatrixCSC
        write_rows = lambda D: _lib.check(L.daisy_formfactors_write_rows(obj._ctx, 0, N, _lib.fptr(D)))  # noqa: E731
    else:
        obj = dz.DeviceGroup(mesh, devices=list(range(ndev)), rands=uv)
        obj.cudaCalculateRadiosityMatrix()
        to_csc_fn, handle = L.daisy_group_formfactors_to_csc, obj._g
        load_csc = obj.loadRadiosityMatrixCSC
        write_rows = lambda D: _lib.check(L.daisy_group_formfactors_write_rows(obj._g, 0, N, _lib.fptr(D)))  # noqa: E731
    nnz = C.c_int64()
    _lib.check(to_csc_fn(handle, C.byref(nnz), None, None, None))
    nnz = nnz.value
    vals = np.empty(nnz, np.float32)
    inner = np.empty(nnz, np.int32)
    outer = np.empty(N + 1, np.int32)

    def count(host):
        set_host(host)
        n = C.c_int64()
        _lib.check(to_csc_fn(handle, C.byref(n), None, None, None))
        return n.value

    def fill(host):
        set_host(host)
        n = C.c_int64()
        _lib.check(to_csc_fn(handle, C.byref(n), _lib.fptr(vals), _lib.iptr(inner), _lib.iptr(outer)))

    export = {
        "count": alternate({"device": lambda: count(False), "host": lambda: count(True)}, rounds),
        "fill": alternate({"device": lambda: fill(False), "host": lambda: fill(True)}, rounds),
    }
    set_host(True)
    fill(True)
    ref = (vals.copy(), inner.copy(), outer.copy())
    fill(False)
    export_identical = all(np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b)
                           for a, b in zip((vals, inner, outer), ref))
    set_host(False)
    path = os.path.join(tmp, name + ".bin")
    api.serialize_mat(path, vals, inner, outer, N)
    del ref

    def import_csc():
        t_read, arrs = timed(lambda: api.deserialize_csc(path))
        t_load, _ = timed(lambda: load_csc(*arrs))
        return t_read, t_load

    def import_dense():
        t_read, D = timed(lambda: api.deserialize_mat(path))
        t_load, _ = timed(lambda: write_rows(D))
        return t_read, t_load

    parts = {"csc": [], "dense": []}
    arms = {"csc": lambda: parts["csc"].append(import_csc()), "dense": lambda: parts["dense"].append(import_dense())}
    imp = alternate(arms, rounds)
    for k in arms:
        imp[k]["read_file_median_s"] = statistics.median(p[0] for p in parts[k][1:])
        imp[k]["load_median_s"] = statistics.median(p[1] for p in parts[k][1:])
    # bit-identical imports: digests of every device's rows after each arm
    digests = []
    for arm in (import_dense, import_csc):
        arm()
        views = [obj] if ndev == 1 else [obj.device(i) for i in range(ndev)]
        digests.append([tuple(a.tobytes() for a in dz.RadMat(v).row_digest()) for v in views if v.row_range[1] > v.row_range[0]])
    # how the library staged the last import (1: resident, 2: uploaded twice), as the first device's context records it
    uploads = int(L.daisy_formfactors_csc_uploads(obj._ctx if ndev == 1 else C.c_void_p(L.daisy_group_ctx(obj._g, 0))))
    resident = uploads == 1
    dense_b, csc_b = 4 * N * N, 8 * nnz
    res = {
        "workload": name, "N": N, "devices": ndev, "nnz": nnz, "density": nnz / float(N * N),
        "export": export, "export_bit_identical": bool(export_identical),
        "import": imp, "import_bit_identical": digests[0] == digests[1],
        "import_staging": {1: "resident (one upload)", 2: "two uploads"}.get(uploads, "unknown (%d)" % uploads),
        "pcie_bytes": {
            "export_count_device": 4 * N * ndev, "export_count_host": dense_b,
            "export_fill_device": 4 * N * ndev + 8 * N * ndev + csc_b, "export_fill_host": 2 * dense_b,
            "import_csc": ndev * (csc_b + 4 * (N + 1) + (0 if resident else 4 * nnz)), "import_dense": dense_b,
        },
    }
    obj.close()
    return res


def shim_demo(tmp, rounds):
    demo = os.path.join(ROOT, "shim", "_build", "shim_demo")
    if not os.path.exists(demo):
        return {"measured": False, "why": "shim/_build/shim_demo is not built (it compiles against the reference's sources)"}
    from daisyriot_b200 import rgb2spec
    sc = load_scene("cornellbox_blacklight")
    obj, _ = scenes.write_obj(sc, tmp, "shim_cache_scene")
    os.makedirs(os.path.join(tmp, "color_tables"), exist_ok=True)
    rgb2spec.write_surrogate_table(os.path.join(tmp, "color_tables", "srgb.coeff"), 16)
    rands = os.path.join(tmp, "rands.bin")
    scenes.msvc_sample_pattern(1).astype(np.float32).tofile(rands)

    def pair(host):
        env = dict(os.environ)
        env.pop("DAISY_CSC_HOST", None)
        if host:
            env["DAISY_CSC_HOST"] = "1"
        matfile = os.path.join(tmp, "radmat_%d.bin" % host)
        if os.path.exists(matfile):
            os.remove(matfile)
        out = []
        for _ in range(2):
            t, r = timed(lambda: subprocess.run([demo, obj, tmp + "/", "2", "7.0", "1", rands, matfile], cwd=tmp, capture_output=True, text=True, timeout=900, env=env))
            assert r.returncode == 0, r.stderr[-2000:]
            out.append(t)
        return out

    res = {"device": [], "host": []}
    for _ in range(rounds):
        res["device"].append(pair(False))
        res["host"].append(pair(True))
    return {"measured": True, "note": "DAISY_CSC_HOST=1 changes the export (first run) only; both second runs load through write_csc",
            **{k: {"first_run_median_s": statistics.median(p[0] for p in v), "second_run_median_s": statistics.median(p[1] for p in v)}
                                 for k, v in res.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    ndev = dz.lib().daisy_device_count()
    out = {"gpu": gpu, "rounds": args.rounds, "workloads": []}
    with tempfile.TemporaryDirectory(prefix="daisy_matrix_cache_") as tmp:
        for w in args.workloads:
            if WORKLOADS[w][1] > ndev:
                out["workloads"].append({"workload": w, "measured": False, "why": "%d GPU(s) visible" % ndev})
                continue
            r = run_workload(w, args.rounds, tmp)
            print(json.dumps({k: r[k] for k in ("workload", "nnz", "export_bit_identical", "import_bit_identical")}), flush=True)
            out["workloads"].append(r)
        out["shim_demo_cornellbox_blacklight"] = shim_demo(tmp, args.rounds)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
