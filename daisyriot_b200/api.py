"""Host-side mirror of the reference's entry points for the form-factor + gather path, over the C-ABI.

Same names, argument meaning and (print-and-continue vs. raise aside) behaviour as the reference classes:

* :class:`MeshS`                     -- ``visual studio/MeshS.h:7-26`` (patch layout + materials)
* :class:`OptixPrimeFunctionality`   -- ``visual studio/OptixPrimeFunctionality.h:24-48``
* :class:`Lightning` and its three flavours -- ``visual studio/Lightning.h``

The heavy lifting is in ``libdaisy_b200.so`` (hand-written sm_100a kernels); nothing here computes on the CPU
except O(N*K) input preparation and the colour cache.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import struct

import numpy as np

from . import _lib
from . import materials as _mat
from . import rgb2spec as _r2s
from .scenes import RAYS_PER_PATCH, Scene, load_obj, msvc_sample_pattern

HIT_DTYPE = _lib.HIT_DTYPE


class MeshS:
    """Reference ``MeshS``: public arrays ``vertices``, ``normals``, ``triangleIndices``, ``materials``,
    ``materialIndexPerTriangle``, ``numtriangles`` (``MeshS.h:14-20``)."""

    def __init__(self, filepath=None, mtlpath=None, wavelengths=None, coeff_table=None):
        self.vertices = np.zeros((0, 3), np.float32)
        self.normals = np.zeros((0, 3), np.float32)
        self.triangleIndices = np.zeros((0, 6), np.int32)
        self.materials = []
        self.materialIndexPerTriangle = np.zeros(0, np.int32)
        self.numtriangles = 0
        self.wavelengths = None if wavelengths is None else np.asarray(wavelengths, np.float32)
        if filepath is not None:
            self.loadFromFile(filepath, mtlpath, wavelengths, coeff_table)

    def loadFromFile(self, filepath, mtldirpath, wavelengths, coeff_table="color_tables/srgb.coeff"):
        """``MeshS::loadFromFile`` (``MeshS.cpp:22-128``)."""
        self._from_scene(load_obj(filepath, mtldirpath), wavelengths, coeff_table)

    @classmethod
    def from_scene(cls, scene: Scene, wavelengths=None, coeff_table=None):
        m = cls()
        m._from_scene(scene, wavelengths, coeff_table)
        return m

    def _from_scene(self, scene: Scene, wavelengths, coeff_table):
        self.vertices = np.ascontiguousarray(scene.vertices, np.float32)
        self.normals = np.ascontiguousarray(scene.normals, np.float32)
        self.triangleIndices = np.ascontiguousarray(scene.tri, np.int32)
        self.materialIndexPerTriangle = np.ascontiguousarray(scene.mat_idx, np.int32)
        self.numtriangles = int(self.triangleIndices.shape[0])
        self.scene_materials = scene.materials
        if wavelengths is not None:
            self.wavelengths = np.asarray(wavelengths, np.float32)
            if coeff_table is None:
                raise ValueError("a rgb2spec coefficient table is needed to build spectral materials")
            model = coeff_table if isinstance(coeff_table, _r2s.RGB2Spec) else _r2s.RGB2Spec.load(coeff_table)
            self.materials = _mat.make_materials(scene.materials, self.wavelengths, model)


class RadMat:
    """Stand-in for the reference's ``SpMat RadMat`` (``Eigen::SparseMatrix<float>``, ``Lightning.h:19``): the
    matrix stays on the GPU as dense FP32 rows; this handle reads it back in either form."""

    def __init__(self, optixP: "OptixPrimeFunctionality"):
        self._p = optixP

    @property
    def shape(self):
        return (self._p.N, self._p.N)

    def rows(self, row0=None, nrows=None) -> np.ndarray:
        r0, r1 = self._p.row_range
        row0 = r0 if row0 is None else row0
        nrows = (r1 - row0) if nrows is None else nrows
        out = np.empty((nrows, self._p.N), np.float32)
        _lib.check(_lib.lib().daisy_formfactors_read_rows(self._p._ctx, row0, nrows, _lib.fptr(out)), "formfactors_read_rows")
        return out

    def row_digest(self, row0=None, nrows=None):
        """Exact per-row digests computed on the device (no read-back of the rows): (xor of the float bit patterns,
        sum of bits*(2c+1) mod 2^64).  :func:`row_digest_host` gives the same from host rows."""
        r0, r1 = self._p.row_range
        row0 = r0 if row0 is None else row0
        nrows = (r1 - row0) if nrows is None else nrows
        x = np.empty(nrows, np.uint32)
        w = np.empty(nrows, np.uint64)
        _lib.check(_lib.lib().daisy_formfactors_row_digest(self._p._ctx, row0, nrows, x.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                           w.ctypes.data_as(C.POINTER(C.c_uint64))), "formfactors_row_digest")
        return x, w

    def to_csc(self):
        """(values, innerIndices, outerStarts) exactly as ``setFromTriplets`` leaves a column-major SparseMatrix."""
        L = _lib.lib()
        nnz = C.c_int64()
        _lib.check(L.daisy_formfactors_to_csc(self._p._ctx, C.byref(nnz), None, None, None), "formfactors_to_csc")
        vals = np.empty(nnz.value, np.float32)
        inner = np.empty(nnz.value, np.int32)
        outer = np.empty(self._p.N + 1, np.int32)
        _lib.check(L.daisy_formfactors_to_csc(self._p._ctx, C.byref(nnz), _lib.fptr(vals), _lib.iptr(inner), _lib.iptr(outer)),
                   "formfactors_to_csc")
        return vals, inner, outer


class OptixPrimeFunctionality:
    """Reference ``OptixPrimeFunctionality`` (``OptixPrimeFunctionality.h:24-48``) on a B200.

    The constructor uploads the mesh and builds the LBVH (the reference builds an OptiX Prime model,
    ``OptixPrimeFunctionality.cpp:36-47``) and fixes the ``rands`` sample pattern (``:55-63``; the reference seeds
    it with wall-clock time -- pass ``rands`` or ``seed`` to choose it)."""

    def __init__(self, mesh: MeshS, device: int = 0, rands=None, seed: int = 1, rank: int = 0, nranks: int = 1, stream=None):
        L = _lib.lib()
        self.mesh = mesh
        self.N = mesh.numtriangles
        self._ctx = C.c_void_p()
        v = np.ascontiguousarray(mesh.vertices, np.float32)
        n = np.ascontiguousarray(mesh.normals, np.float32)
        t = np.ascontiguousarray(mesh.triangleIndices, np.int32)
        _lib.check(L.daisy_ctx_create(_lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(t), t.shape[0], device,
                                      C.byref(self._ctx)), "ctx_create")
        self.rands = np.ascontiguousarray(msvc_sample_pattern(seed, RAYS_PER_PATCH) if rands is None else rands, np.float32)
        _lib.check(L.daisy_ctx_set_samples(self._ctx, _lib.fptr(self.rands), self.rands.shape[0]), "ctx_set_samples")
        if nranks > 1:
            _lib.check(L.daisy_ctx_set_partition(self._ctx, rank, nranks), "ctx_set_partition")
        if stream is not None:
            _lib.check(L.daisy_ctx_set_stream(self._ctx, C.c_void_p(stream)), "ctx_set_stream")
        self.rank, self.nranks = rank, nranks

    def close(self):
        if getattr(self, "_ctx", None):
            _lib.lib().daisy_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def row_range(self):
        r0, r1, n = C.c_int(), C.c_int(), C.c_int()
        _lib.check(_lib.lib().daisy_ctx_row_range(self._ctx, C.byref(r0), C.byref(r1), C.byref(n)))
        return r0.value, r1.value

    # -- optixQuery(int number_of_rays, vector<float3>& rays, vector<Hit>& hits)              .cpp:66-81
    def optixQuery(self, number_of_rays: int, rays, hits=None) -> np.ndarray:
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1)
        if rays.size < 6 * number_of_rays:
            raise ValueError("rays holds fewer than number_of_rays origin/direction pairs")
        if hits is None:
            hits = np.empty(number_of_rays, HIT_DTYPE)
        _lib.check(_lib.lib().daisy_query_closest(self._ctx, number_of_rays, _lib.fptr(rays), hits.ctypes.data), "query_closest")
        return hits

    # -- parallellism::runCalculateRadiosityMatrix(SimpleMesh&)                      parallellism.cu:4-89
    def runCalculateRadiosityMatrix(self, row0=0, nrows=None, variant=_lib.FF_DEVICE) -> np.ndarray:
        nrows = self.N - row0 if nrows is None else nrows
        out = np.empty((nrows, self.N), _lib.TRIPL_DTYPE)
        _lib.check(_lib.lib().daisy_unoccluded_rows(self._ctx, variant, row0, nrows, out.ctypes.data), "unoccluded_rows")
        return out

    # -- cudaCalculateRadiosityMatrix(SpMat&, MeshS&)                                        .cpp:6-34
    def cudaCalculateRadiosityMatrix(self, RadMat_=None, mesh=None) -> RadMat:
        _lib.check(_lib.lib().daisy_formfactors_build(self._ctx, _lib.FF_DEVICE), "formfactors_build")
        return RadMat(self)

    # -- calculateRadiosityMatrix(SpMat&, MeshS&)   (cuda_on = false: float pi, reciprocity)  .cpp:311-366
    def calculateRadiosityMatrix(self, RadMat_=None, mesh=None) -> RadMat:
        _lib.check(_lib.lib().daisy_formfactors_build(self._ctx, _lib.FF_HOST), "formfactors_build")
        return RadMat(self)

    def updateGeometry(self, vertices=None, normals=None) -> None:
        """Move the mesh: new vertex positions and/or normals (same counts, same triangles; ``None`` keeps an array).  The
        hierarchy and every derived record are rebuilt, so queries answer for the new geometry at once; the matrix changes
        only at :meth:`updateRadiosityMatrix`.  ``self.mesh`` takes the new arrays."""
        v, n = _geometry_arrays(self.mesh, vertices, normals)
        _lib.check(_lib.lib().daisy_ctx_update_geometry(self._ctx, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0]), "ctx_update_geometry")
        self.mesh.vertices, self.mesh.normals = v, n

    def replaceMesh(self, mesh: MeshS, previous) -> None:
        """Replace the mesh (objects removed or added, vertices renumbered): ``previous[t]`` = index in the current mesh of the
        triangle new triangle t continues, or -1 for a new one.  Queries answer for the new mesh at once; the matrix is remapped
        at once (entries of new triangles +0.0) and traced where the edit reaches it at :meth:`updateRadiosityMatrix`.  Solvers
        created before are stale: create new ones.  ``self.mesh`` and ``self.N`` follow."""
        v, n, t, prev = _mesh_edit_arrays(mesh, previous)
        _lib.check(_lib.lib().daisy_ctx_replace_mesh(self._ctx, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(t), t.shape[0],
                                                     _lib.iptr(prev)), "ctx_replace_mesh")
        self.mesh, self.N = mesh, t.shape[0]

    def updateRadiosityMatrix(self, variant=_lib.FF_DEVICE) -> RadMat:
        """Bring the matrix to the current geometry, bit-identical to a fresh build, re-tracing only the pairs a change can
        reach (everything when the matrix was loaded, built with another variant or other samples, or not built yet)."""
        _lib.check(_lib.lib().daisy_formfactors_update(self._ctx, variant), "formfactors_update")
        return RadMat(self)

    def update_stats(self):
        t, k, p, ms = C.c_int64(), C.c_int64(), C.c_int64(), C.c_double()
        _lib.check(_lib.lib().daisy_formfactors_update_stats(self._ctx, C.byref(t), C.byref(k), C.byref(p), C.byref(ms)))
        return {"tris_changed": t.value, "tiles_retraced": k.value, "pairs_retraced": p.value, "classify_ms": ms.value}

    def loadRadiosityMatrix(self, dense_rows: np.ndarray, row0: int = 0) -> RadMat:
        """The reference's matrix-cache path (``Lightning.h:84-96``): load instead of build."""
        a = np.ascontiguousarray(dense_rows, np.float32)
        _lib.check(_lib.lib().daisy_formfactors_write_rows(self._ctx, row0, a.shape[0], _lib.fptr(a)), "formfactors_write_rows")
        return RadMat(self)

    def loadRadiosityMatrixCSC(self, values, inner, outer) -> RadMat:
        """The matrix-cache path from the CSC arrays themselves (``DeserializeMat``'s ``SpMat``, :func:`deserialize_csc`):
        validated and scattered on the device, no dense matrix on the host.  ``outer`` holds N + 1 column starts.  Entries
        not listed become +0.0; partitioned contexts keep the rows of their range."""
        v, i, o = _csc_arrays(values, inner, outer, self.N)
        _lib.check(_lib.lib().daisy_formfactors_write_csc(self._ctx, v.size, _lib.fptr(v), _lib.iptr(i), _lib.iptr(o)), "formfactors_write_csc")
        return RadMat(self)

    def visibilityMasks(self, row0=0, nrows=None, variant=_lib.FF_DEVICE) -> np.ndarray:
        nrows = self.N - row0 if nrows is None else nrows
        out = np.empty((nrows, self.N), np.uint64)
        _lib.check(_lib.lib().daisy_visibility_masks(self._ctx, variant, row0, nrows, out.ctypes.data_as(C.POINTER(C.c_uint64))),
                   "visibility_masks")
        return out

    # -- float calculateVisibility(int originPatch, int destPatch, MeshS&, ...)               .cpp:244-271
    def calculateVisibility(self, originPatch: int, destPatch: int, mesh=None) -> float:
        lo, hi = (originPatch, destPatch)
        rays = self.pair_rays(lo, hi)
        hits = self.optixQuery(rays.shape[0], rays)
        seen = np.count_nonzero((hits["t"] > 0) & (hits["triangleId"] == destPatch))
        return float(np.float32(seen) / np.float32(rays.shape[0]))

    # -- float p2pFormfactor(int originPatch, int destPatch, MeshS&)     (4x4 rule, host arithmetic, x visibility)   .cpp:133-167
    def p2pFormfactor(self, originPatch: int, destPatch: int, mesh=None) -> float:
        row = self.runCalculateRadiosityMatrix(originPatch, 1, _lib.FF_HOST)[0]
        return float(np.float32(row["m_value"][destPatch]) * np.float32(self.calculateVisibility(originPatch, destPatch)))

    # triangle_math helpers in the reference's float32 operation order                         triangle_math.cpp:16-29, 31-35, 76-86
    def _centre(self, tri: int) -> np.ndarray:
        m = self.mesh
        a, b, c = (m.vertices[m.triangleIndices[tri, k]] for k in range(3))
        return ((a + b + c) / np.float32(3)).astype(np.float32)

    def _avg_normal(self, tri: int) -> np.ndarray:
        m = self.mesh
        n = (m.normals[m.triangleIndices[tri, 3]] + m.normals[m.triangleIndices[tri, 4]] + m.normals[m.triangleIndices[tri, 5]]) / np.float32(3)
        return _normalize32(n.astype(np.float32))

    def _is_facing_back(self, origin: np.ndarray, destPatch: int) -> bool:
        d = _normalize32((self._centre(destPatch) - origin).astype(np.float32))
        return bool(_dot32(d, self._avg_normal(destPatch)) >= 0)

    # -- float p2pFormfactorNusselt(int originPatch, int destPatch, MeshS&)                                  .cpp:273-306
    def p2pFormfactorNusselt(self, originPatch: int, destPatch: int, mesh=None) -> float:
        """Nusselt analogue: the destination triangle projected onto the unit hemisphere around the origin patch's centre
        and then onto its plane, area / pi, times the sampled visibility.  The reference guards with
        ``if (isFacingBack(a), isFacingBack(b))`` -- a comma expression, so only the second test counts; kept as is."""
        m = self.mesh
        co, cd = self._centre(originPatch), self._centre(destPatch)
        no = self._avg_normal(originPatch)
        if self._is_facing_back(cd, originPatch):
            return 0.0
        proj = []
        for i in range(3):
            v = m.vertices[m.triangleIndices[destPatch, i]]
            h = (co + _normalize32((v - co).astype(np.float32))).astype(np.float32)
            proj.append((h - _dot32(no, (h - co).astype(np.float32)) * no).astype(np.float32))
        ab, ac = (proj[1] - proj[0]).astype(np.float32), (proj[2] - proj[0]).astype(np.float32)
        cr = np.array([ab[1] * ac[2] - ac[1] * ab[2], ab[2] * ac[0] - ac[2] * ab[0], ab[0] * ac[1] - ac[0] * ab[1]], np.float32)
        surface = np.float32(0.5 * float(np.sqrt(_dot32(cr, cr), dtype=np.float32)))
        ff = np.float32(surface / np.float32(math.pi))
        return float(np.float32(ff * np.float32(self.calculateVisibility(originPatch, destPatch))))

    # -- bool shootPatchRay(vector<Hit>& patches, MeshS&)     one ray between two picked surface points              .cpp:456-469
    def shootPatchRay(self, patches, mesh=None) -> bool:
        m = self.mesh
        f = np.float32

        def uv2xyz(h):
            a, b, c = (m.vertices[m.triangleIndices[int(h["triangleId"]), k]] for k in range(3))
            return ((a + f(h["u"]) * (b - a)) + f(h["v"]) * (c - a)).astype(np.float32)

        pa, pb = uv2xyz(patches[0]), uv2xyz(patches[1])
        n = _normalize32((pb - pa).astype(np.float32))
        ray = np.concatenate([(pa + n * f(0.000001)).astype(np.float32), n]).astype(np.float32)
        hit = self.optixQuery(1, ray)
        return bool(hit[0]["triangleId"] == patches[1]["triangleId"])

    def pair_rays(self, originPatch: int, destPatch: int) -> np.ndarray:
        """The S rays of ``.cpp:253-258`` (float32, reference operation order)."""
        m = self.mesh
        f = np.float32

        def uv2xyz(tri, u, v):
            a, b, c = (m.vertices[m.triangleIndices[tri, k]] for k in range(3))
            return (a + u * (b - a)) + v * (c - a)

        out = np.empty((self.rands.shape[0], 6), np.float32)
        for i, (u, v) in enumerate(self.rands):
            o = uv2xyz(originPatch, f(u), f(v))
            d = uv2xyz(destPatch, f(u), f(v))
            diff = (d - o).astype(np.float32)
            t = diff * diff
            inv = f(1.0) / np.sqrt(f(f(t[0] + t[1]) + t[2]), dtype=np.float32)
            n = (diff * inv).astype(np.float32)
            out[i, :3] = o + n * f(0.000001)
            out[i, 3:] = n
        return out

    def stats(self):
        p, o, r, a, b = C.c_int64(), C.c_int64(), C.c_int64(), C.c_double(), C.c_double()
        _lib.check(_lib.lib().daisy_formfactors_stats(self._ctx, C.byref(p), C.byref(o), C.byref(r), C.byref(a), C.byref(b)))
        return {"pairs_traced": p.value, "pairs_owned": o.value, "rays": r.value, "lbvh_ms": a.value, "ff_ms": b.value,
                "pairs_fallback": int(_lib.lib().daisy_formfactors_pairs_fallback(self._ctx)),
                "faces": int(_lib.lib().daisy_ctx_face_count(self._ctx))}



class DeviceGroup:
    """All GPUs of the box behind ONE host process (``daisy_group_*``): the reference's ``OptixPrimeFunctionality`` surface
    for the matrix build over several devices -- row block g on ``devices[g]``, mesh and LBVH replicated, mirrored tiles
    stored into the owners' matrices over NVLink.  ``device(i)`` gives device i's context as an ``OptixPrimeFunctionality``
    view (row range, masks, digests, closest hit)."""

    def __init__(self, mesh: MeshS, devices=None, ndev: int | None = None, rands=None, seed: int = 1):
        L = _lib.lib()
        self.mesh, self.N = mesh, mesh.numtriangles
        if devices is None:
            devices = list(range(ndev if ndev is not None else L.daisy_device_count()))
        self.devices = [int(d) for d in devices]
        dev = np.ascontiguousarray(self.devices, np.int32)
        v = np.ascontiguousarray(mesh.vertices, np.float32)
        n = np.ascontiguousarray(mesh.normals, np.float32)
        t = np.ascontiguousarray(mesh.triangleIndices, np.int32)
        self._g = C.c_void_p()
        _lib.check(L.daisy_group_create(_lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(t), t.shape[0], _lib.iptr(dev), len(self.devices),
                                        C.byref(self._g)), "group_create")
        self.rands = np.ascontiguousarray(msvc_sample_pattern(seed, RAYS_PER_PATCH) if rands is None else rands, np.float32)
        _lib.check(L.daisy_group_set_samples(self._g, _lib.fptr(self.rands), self.rands.shape[0]), "group_set_samples")

    def close(self):
        if getattr(self, "_g", None):
            _lib.lib().daisy_group_destroy(self._g)
            self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device(self, i: int) -> "OptixPrimeFunctionality":
        view = OptixPrimeFunctionality.__new__(OptixPrimeFunctionality)
        view.mesh, view.N, view.rands = self.mesh, self.N, self.rands
        view._ctx = C.c_void_p(_lib.lib().daisy_group_ctx(self._g, i))
        view.rank, view.nranks = i, len(self.devices)
        view.close = lambda: None  # the group owns the context
        return view

    def cudaCalculateRadiosityMatrix(self):
        _lib.check(_lib.lib().daisy_group_formfactors_build(self._g, _lib.FF_DEVICE), "group_formfactors_build")
        return self

    def calculateRadiosityMatrix(self):
        _lib.check(_lib.lib().daisy_group_formfactors_build(self._g, _lib.FF_HOST), "group_formfactors_build")
        return self

    def update_geometry(self, vertices=None, normals=None) -> None:
        """:meth:`OptixPrimeFunctionality.updateGeometry` on every device."""
        v, n = _geometry_arrays(self.mesh, vertices, normals)
        _lib.check(_lib.lib().daisy_group_update_geometry(self._g, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0]), "group_update_geometry")
        self.mesh.vertices, self.mesh.normals = v, n

    def replace_mesh(self, mesh: MeshS, previous) -> None:
        """:meth:`OptixPrimeFunctionality.replaceMesh` on every device (the row blocks follow the new N)."""
        v, n, t, prev = _mesh_edit_arrays(mesh, previous)
        _lib.check(_lib.lib().daisy_group_replace_mesh(self._g, _lib.fptr(v), v.shape[0], _lib.fptr(n), n.shape[0], _lib.iptr(t), t.shape[0],
                                                       _lib.iptr(prev)), "group_replace_mesh")
        self.mesh, self.N = mesh, t.shape[0]

    def updateRadiosityMatrix(self, variant=_lib.FF_DEVICE):
        _lib.check(_lib.lib().daisy_group_formfactors_update(self._g, variant), "group_formfactors_update")
        return self

    def rows(self, row0=0, nrows=None) -> np.ndarray:
        nrows = self.N - row0 if nrows is None else nrows
        out = np.empty((nrows, self.N), np.float32)
        _lib.check(_lib.lib().daisy_group_formfactors_read_rows(self._g, row0, nrows, _lib.fptr(out)), "group_formfactors_read_rows")
        return out

    def to_csc(self):
        """(values, innerIndices, outerStarts) of the whole matrix, as :meth:`RadMat.to_csc` gives them on one GPU."""
        L = _lib.lib()
        nnz = C.c_int64()
        _lib.check(L.daisy_group_formfactors_to_csc(self._g, C.byref(nnz), None, None, None), "group_formfactors_to_csc")
        vals = np.empty(nnz.value, np.float32)
        inner = np.empty(nnz.value, np.int32)
        outer = np.empty(self.N + 1, np.int32)
        _lib.check(L.daisy_group_formfactors_to_csc(self._g, C.byref(nnz), _lib.fptr(vals), _lib.iptr(inner), _lib.iptr(outer)),
                   "group_formfactors_to_csc")
        return vals, inner, outer

    def loadRadiosityMatrixCSC(self, values, inner, outer):
        """:meth:`OptixPrimeFunctionality.loadRadiosityMatrixCSC` over the group: every device validates, then keeps its rows."""
        v, i, o = _csc_arrays(values, inner, outer, self.N)
        _lib.check(_lib.lib().daisy_group_formfactors_write_csc(self._g, v.size, _lib.fptr(v), _lib.iptr(i), _lib.iptr(o)),
                   "group_formfactors_write_csc")
        return self

    def stats(self):
        p, r, a, b = C.c_int64(), C.c_int64(), C.c_double(), C.c_double()
        _lib.check(_lib.lib().daisy_group_formfactors_stats(self._g, C.byref(p), C.byref(r), C.byref(a), C.byref(b)))
        return {"pairs": p.value, "rays": r.value, "lbvh_ms": a.value, "ff_ms": b.value}


class GroupSolver:
    """The Lightning family's solver over a :class:`DeviceGroup` (``daisy_group_solver_*``): same calls as the single-GPU
    solver, whole-scene ``K x N`` arrays in and out; a pass is one asynchronous kernel launch per device."""

    def __init__(self, group: DeviceGroup, K: int, E, M, mat_idx):
        self.group, self.K = group, K
        E = np.ascontiguousarray(E, np.float32)
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(mat_idx, np.int32)
        self._s = C.c_void_p()
        _lib.check(_lib.lib().daisy_group_solver_create(group._g, K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat), C.byref(self._s)),
                   "group_solver_create")

    def close(self):
        if getattr(self, "_s", None):
            _lib.lib().daisy_group_solver_destroy(self._s)
            self._s = None

    def reset(self):
        _lib.check(_lib.lib().daisy_group_solver_reset(self._s), "group_solver_reset")

    def step(self, want_sums: bool = True):
        if not want_sums:
            _lib.check(_lib.lib().daisy_group_solver_step(self._s, None), "group_solver_step")
            return None
        sums = np.zeros(self.K, np.float64)
        _lib.check(_lib.lib().daisy_group_solver_step(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))), "group_solver_step")
        return sums

    def band_sums(self):
        sums = np.zeros(self.K, np.float64)
        _lib.check(_lib.lib().daisy_group_solver_band_sums(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))), "group_solver_band_sums")
        return sums

    def converge(self, threshold: float, per_band: bool, max_passes: int = 0, on_device: bool = False) -> int:
        """``on_device=True``: the pass kernels apply the stop rule themselves and the passes follow each other without a host
        decision in between (``daisy_group_solver_converge_device``); same passes and bit-identical results."""
        passes = C.c_int()
        fn = _lib.lib().daisy_group_solver_converge_device if on_device else _lib.lib().daisy_group_solver_converge
        _lib.check(fn(self._s, float(threshold), int(per_band), max_passes, C.byref(passes)), "group_solver_converge")
        return passes.value

    @property
    def numpasses(self):
        return int(_lib.lib().daisy_group_solver_numpasses(self._s))

    def read(self):
        B = np.empty((self.K, self.group.N), np.float32)
        R = np.empty((self.K, self.group.N), np.float32)
        _lib.check(_lib.lib().daisy_group_solver_read(self._s, _lib.fptr(B), _lib.fptr(R)), "group_solver_read")
        return B, R

    def write(self, B, R):
        B = np.ascontiguousarray(B, np.float32)
        R = np.ascontiguousarray(R, np.float32)
        _lib.check(_lib.lib().daisy_group_solver_write(self._s, _lib.fptr(B), _lib.fptr(R)), "group_solver_write")

    def restart(self, B0=None):
        """:meth:`Lightning.restart` over every device; ``B0`` is K x N (whole scene) or ``None`` for the current B."""
        b = None
        if B0 is not None:
            b = np.ascontiguousarray(B0, np.float32)
            if b.shape != (self.K, self.group.N):
                raise ValueError("restart: B0 must be K x N, got %s" % (b.shape,))
        _lib.check(_lib.lib().daisy_group_solver_restart(self._s, None if b is None else _lib.fptr(b)), "group_solver_restart")

    def set_emission(self, E):
        E = np.ascontiguousarray(E, np.float32)
        if E.shape != (self.K, self.group.N):
            raise ValueError("set_emission: E must be K x N, got %s" % (E.shape,))
        _lib.check(_lib.lib().daisy_group_solver_set_emission(self._s, _lib.fptr(E)), "group_solver_set_emission")

    def set_materials(self, M, mat_idx):
        M, mat = _material_arrays(M, mat_idx, self.K, self.group.N)
        _lib.check(_lib.lib().daisy_group_solver_set_materials(self._s, _lib.fptr(M), M.shape[0], _lib.iptr(mat)), "group_solver_set_materials")


def remap_bands(B_old, previous, E_new) -> np.ndarray:
    """A warm start for the solver of an edited mesh (:meth:`OptixPrimeFunctionality.replaceMesh`): column t of the result is
    ``B_old[:, previous[t]]`` for a triangle that continues old triangle ``previous[t]``, and ``E_new[:, t]`` for a new one
    (``previous[t] == -1``).  K x N_new float32."""
    B_old = np.asarray(B_old, np.float32)
    E_new = np.asarray(E_new, np.float32)
    p = np.asarray(previous)
    if B_old.ndim != 2 or E_new.ndim != 2 or B_old.shape[0] != E_new.shape[0]:
        raise ValueError("remap_bands: B_old (K x N_old) and E_new (K x N_new) need the same band count")
    if p.ndim != 1 or p.shape[0] != E_new.shape[1]:
        raise ValueError("remap_bands: previous needs one entry per triangle of the new mesh")
    if p.size and not np.issubdtype(p.dtype, np.integer):
        raise ValueError("remap_bands: previous holds triangle indices (integers)")
    if p.size and (p.min() < -1 or p.max() >= B_old.shape[1]):
        raise ValueError("remap_bands: previous holds an index outside [-1, N_old)")
    out = np.array(E_new, np.float32, copy=True)
    kept = p >= 0
    out[:, kept] = B_old[:, p[kept]]
    return np.ascontiguousarray(out)


def _material_arrays(M, mat_idx, K: int, N: int):
    """Contiguous float32 nmat x K x K materials and int32 ids, checked for their shapes (the ids' range the library checks)."""
    M = np.ascontiguousarray(M, np.float32)
    mat = np.ascontiguousarray(mat_idx, np.int32).reshape(-1)
    if M.ndim != 3 or M.shape[1:] != (K, K) or mat.size != N:
        raise ValueError("set_materials: M must be nmat x K x K and mat_idx hold N ids")
    return M, mat


def _csc_arrays(values, inner, outer, n: int):
    """Contiguous float32 / int32 copies of CSC arrays, checked for their lengths (the values themselves the library checks)."""
    v = np.ascontiguousarray(values, np.float32).reshape(-1)
    i = np.ascontiguousarray(inner, np.int32).reshape(-1)
    o = np.ascontiguousarray(outer, np.int32).reshape(-1)
    if o.size != n + 1 or i.size != v.size:
        raise ValueError("CSC arrays: outer needs N + 1 entries and inner as many as values")
    return v, i, o


def _geometry_arrays(mesh: MeshS, vertices, normals):
    """The arrays of an update: the mesh's own where ``None``, float32 copies of the same shape otherwise."""
    v = np.array(mesh.vertices if vertices is None else vertices, np.float32, copy=True).reshape(-1, 3)
    n = np.array(mesh.normals if normals is None else normals, np.float32, copy=True).reshape(-1, 3)
    if v.shape != np.shape(mesh.vertices) or n.shape != np.shape(mesh.normals):
        raise ValueError("updateGeometry: the vertex and normal counts stay those of the mesh")
    return v, n


def _mesh_edit_arrays(mesh: MeshS, previous):
    """The arrays of a mesh replacement: contiguous float32 / int32 copies, ``previous`` checked for its length (one entry per
    new triangle) and for holding integers (the values themselves the library checks)."""
    v = np.ascontiguousarray(mesh.vertices, np.float32).reshape(-1, 3)
    n = np.ascontiguousarray(mesh.normals, np.float32).reshape(-1, 3)
    t = np.ascontiguousarray(mesh.triangleIndices, np.int32).reshape(-1, 6)
    p = np.asarray(previous)
    if p.ndim != 1 or p.shape[0] != t.shape[0]:
        raise ValueError("replaceMesh: previous needs one entry per triangle of the new mesh")
    if p.size and not np.issubdtype(p.dtype, np.integer):
        raise ValueError("replaceMesh: previous holds triangle indices (integers)")
    if p.size and (p.min() < np.iinfo(np.int32).min or p.max() > np.iinfo(np.int32).max):
        raise ValueError("replaceMesh: previous does not fit int32")
    return v, n, t, np.ascontiguousarray(p, np.int32)


def row_digest_host(F_rows: np.ndarray):
    """The digests of :meth:`RadMat.row_digest` from host rows (rows x N float32)."""
    bits = np.ascontiguousarray(F_rows, np.float32).view(np.uint32)
    w = (2 * np.arange(bits.shape[1], dtype=np.uint64) + np.uint64(1))
    with np.errstate(over="ignore"):
        ws = (bits.astype(np.uint64) * w[None, :]).sum(axis=1, dtype=np.uint64)
    return np.bitwise_xor.reduce(bits, axis=1), ws


def _dot32(a, b) -> np.float32:
    """glm::dot on vec3 in float32: (x*x' + y*y') + z*z'."""
    t = (np.asarray(a, np.float32) * np.asarray(b, np.float32)).astype(np.float32)
    return np.float32(np.float32(t[0] + t[1]) + t[2])


def _normalize32(v) -> np.ndarray:
    """glm::normalize in float32: v * (1 / sqrt(dot(v, v)))."""
    v = np.asarray(v, np.float32)
    return (v * (np.float32(1.0) / np.sqrt(_dot32(v, v), dtype=np.float32))).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------
def cie1931WavelengthToXYZFit(wavelength: float) -> np.ndarray:
    """``daisy_color::cie1931WavelengthToXYZFit`` (``color.h:14-45``), double math, float32 result."""
    wave = float(wavelength)
    t1 = (wave - 442.0) * (0.0624 if wave < 442.0 else 0.0374)
    t2 = (wave - 599.8) * (0.0264 if wave < 599.8 else 0.0323)
    t3 = (wave - 501.1) * (0.0490 if wave < 501.1 else 0.0382)
    x = 0.362 * math.exp(-0.5 * t1 * t1) + 1.056 * math.exp(-0.5 * t2 * t2) - 0.065 * math.exp(-0.5 * t3 * t3)
    t1 = (wave - 568.8) * (0.0213 if wave < 568.8 else 0.0247)
    t2 = (wave - 530.9) * (0.0613 if wave < 530.9 else 0.0322)
    y = 0.821 * math.exp(-0.5 * t1 * t1) + 0.286 * math.exp(-0.5 * t2 * t2)
    t1 = (wave - 437.0) * (0.0845 if wave < 437.0 else 0.0278)
    t2 = (wave - 459.0) * (0.0385 if wave < 459.0 else 0.0725)
    z = 1.217 * math.exp(-0.5 * t1 * t1) + 0.681 * math.exp(-0.5 * t2 * t2)
    return np.array([x, y, z], np.float32)


_XYZ2RGB = np.array([[3.240479, -1.537150, -0.498535], [-0.969256, 1.875991, 0.041556], [0.055648, -0.204043, 1.057311]], np.float32)


def serialize_mat(path: str, vals: np.ndarray, inner: np.ndarray, outer: np.ndarray, n: int) -> None:
    """``Lightning::SerializeMat`` byte layout (``Lightning.h:21-50``): rows, cols, nnz, outerSize, innerSize,
    values[nnz], outerIndex[outerSize], innerIndex[nnz]."""
    with open(path, "wb") as f:
        f.write(struct.pack("<5i", n, n, vals.size, n, n))
        f.write(np.ascontiguousarray(vals, np.float32).tobytes())
        f.write(np.ascontiguousarray(outer[:n], np.int32).tobytes())
        f.write(np.ascontiguousarray(inner, np.int32).tobytes())


def deserialize_mat(path: str):
    """``Lightning::DeserializeMat`` (``Lightning.h:51-74``) -> dense float32 matrix."""
    with open(path, "rb") as f:
        rows, cols, nnz, a, b = struct.unpack("<5i", f.read(20))
        vals = np.frombuffer(f.read(4 * nnz), np.float32)
        outer = np.frombuffer(f.read(4 * a), np.int32)
        inner = np.frombuffer(f.read(4 * nnz), np.int32)
    dense = np.zeros((rows, cols), np.float32)
    ends = np.append(outer[1:], nnz)
    for c in range(cols):
        s, e = outer[c], ends[c]
        dense[inner[s:e], c] = vals[s:e]
    return dense


def deserialize_csc(path: str):
    """``Lightning::DeserializeMat`` (``Lightning.h:51-74``) -> (values, innerIndices, outerStarts) as the file holds them,
    with the closing sentinel ``outer[N] = nnz`` appended (the file stores outerSize entries); no dense matrix is built."""
    with open(path, "rb") as f:
        rows, cols, nnz, a, b = struct.unpack("<5i", f.read(20))
        vals = np.frombuffer(f.read(4 * nnz), np.float32)
        outer = np.frombuffer(f.read(4 * a), np.int32)
        inner = np.frombuffer(f.read(4 * nnz), np.int32)
    if vals.size != nnz or outer.size != a or inner.size != nnz:
        raise ValueError("%s: truncated matrix file" % path)
    return vals, inner, np.append(outer, np.int32(nnz)).astype(np.int32)


class Lightning:
    """Reference ``Lightning`` base (``Lightning.h:7-97``): owns ``RadMat``; ``get_lightning`` is the factory."""

    numsamples = 0
    threshold = 1e-4
    per_band = 1

    @staticmethod
    def get_lightning(method: int, mesh: MeshS, optixP: OptixPrimeFunctionality, emissionval: float, wavelengthsvec=None,
                      cuda_enabled: bool = False, matfile: str | None = None, converge: bool = True) -> "Lightning":
        # Lightning.h:446-457.  BWLightning never receives cuda_on (:393,:449) => always the per-pair variant.
        if method == 0:
            return BWLightning(mesh, optixP, emissionval, matfile=matfile, converge=converge)
        if method == 1:
            return RGBLightning(mesh, optixP, emissionval, cuda_enabled, matfile, converge=converge)
        if method == 2:
            return SpectralLightning(mesh, optixP, emissionval, wavelengthsvec, cuda_enabled, matfile, converge=converge)
        raise ValueError("method must be 0 (BW), 1 (RGB) or 2 (Spectral)")

    # -- shared plumbing -------------------------------------------------------------------------------
    def _init(self, mesh, optixP, E, M, cuda_on, matfile, converge):
        self.mesh_, self.optixP = mesh, optixP
        self.cuda_on = cuda_on
        self.numpatches = mesh.numtriangles
        if matfile is None:
            self.initMat(mesh, optixP)
        else:
            self.initMatFromFile(mesh, optixP, matfile)
        self._create_solver(E, M)
        self.reset()
        if converge:
            self.converge_lightning()

    def _create_solver(self, E, M):
        """A solver on the context's current matrix for ``self.mesh_`` (emission E, materials M)."""
        E = np.ascontiguousarray(E, np.float32)
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(self.mesh_.materialIndexPerTriangle, np.int32)
        self.K = E.shape[0]
        self._s = C.c_void_p()
        _lib.check(_lib.lib().daisy_solver_create(self.optixP._ctx, self.K, _lib.fptr(E), _lib.fptr(M), M.shape[0], _lib.iptr(mat),
                                                  C.byref(self._s)), "solver_create")
        self.emission = E

    def _derive_inputs(self, emissionval):
        """(E, M) of ``self.mesh_`` by the flavour's own rule (set_sampled_emission / set_reflection*, Lightning.h:263-292)."""
        raise NotImplementedError

    def initMat(self, mesh, optixP):  # Lightning.h:75-83
        self.RadMat = optixP.cudaCalculateRadiosityMatrix() if self.cuda_on else optixP.calculateRadiosityMatrix()

    def initMatFromFile(self, mesh, optixP, matfile):  # Lightning.h:84-96
        if os.path.exists(matfile):
            self.RadMat = optixP.loadRadiosityMatrixCSC(*deserialize_csc(matfile))
        else:
            self.initMat(mesh, optixP)
            serialize_mat(matfile, *self.RadMat.to_csc(), mesh.numtriangles)

    def close(self):
        if getattr(self, "_s", None):
            _lib.lib().daisy_solver_destroy(self._s)
            self._s = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def numpasses(self) -> int:
        return int(_lib.lib().daisy_solver_numpasses(self._s))

    def band_sums(self) -> np.ndarray:
        out = np.zeros(self.K, np.float64)
        _lib.check(_lib.lib().daisy_solver_band_sums(self._s, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def read(self):
        """(lightningvalues, residualvector), each K x N band-major."""
        r0, r1 = self.optixP.row_range
        B = np.empty((self.K, r1 - r0), np.float32)
        R = np.empty((self.K, r1 - r0), np.float32)
        _lib.check(_lib.lib().daisy_solver_read(self._s, _lib.fptr(B), _lib.fptr(R)), "solver_read")
        return B, R

    @property
    def lightningvalues(self):
        return self.read()[0]

    @property
    def residualvector(self):
        return self.read()[1]

    def reset(self):
        _lib.check(_lib.lib().daisy_solver_reset(self._s), "solver_reset")
        self._after_update()

    def increment_lightpass(self):
        sums = np.zeros(self.K, np.float64)
        _lib.check(_lib.lib().daisy_solver_step(self._s, sums.ctypes.data_as(C.POINTER(C.c_double))), "solver_step")
        self._after_update()
        return sums

    def converge_lightning(self, max_passes: int = 0, on_device: bool = False):
        """``on_device=True``: the pass kernels apply the stop rule themselves and the passes follow each other without a host
        decision in between (``daisy_solver_converge_device``); same passes and bit-identical results."""
        passes = C.c_int()
        fn = _lib.lib().daisy_solver_converge_device if on_device else _lib.lib().daisy_solver_converge
        _lib.check(fn(self._s, float(self.threshold), int(self.per_band), max_passes, C.byref(passes)), "solver_converge")
        self._after_update()
        return passes.value

    # -- warm restart: the solve continues from the current (or a given) B after the matrix, emission or materials changed ----
    def restart(self, B0=None):
        """One pass that starts the iteration from ``B0`` (K x N of this context's rows) or, ``None``, from the current B:
        B = E + M F B0, residual = B - B0 (``daisy_solver_restart``).  Band sums then total |residual| until the next
        :meth:`reset`.  Returns those band sums."""
        b = None
        if B0 is not None:
            r0, r1 = self.optixP.row_range
            b = np.ascontiguousarray(B0, np.float32)
            if b.shape != (self.K, r1 - r0):
                raise ValueError("restart: B0 must be K x N (this context's rows), got %s" % (b.shape,))
        _lib.check(_lib.lib().daisy_solver_restart(self._s, None if b is None else _lib.fptr(b)), "solver_restart")
        self._after_update()
        return self.band_sums()

    def reconverge(self, max_passes: int = 0, on_device: bool = False):
        """Restart from the current B and converge: the passes of the new solve, restart pass included."""
        self.restart()
        return self.converge_lightning(max_passes, on_device)

    def set_emission_value(self, emissionval):
        """Re-derive E for a new emission value with the flavour's own rule; B and the residual are untouched until
        :meth:`restart` (or :meth:`reset`)."""
        E, _ = self._derive_inputs(emissionval)
        E = np.ascontiguousarray(E, np.float32)
        _lib.check(_lib.lib().daisy_solver_set_emission(self._s, _lib.fptr(E)), "solver_set_emission")
        self.emission, self.emission_value = E, emissionval

    def set_materials(self):
        """Re-derive M (and the material ids) from ``mesh.materials`` after a material changed; takes effect at the next pass."""
        _, M = self._derive_inputs(self.emission_value)
        M = np.ascontiguousarray(M, np.float32)
        mat = np.ascontiguousarray(self.mesh_.materialIndexPerTriangle, np.int32)
        _lib.check(_lib.lib().daisy_solver_set_materials(self._s, _lib.fptr(M), M.shape[0], _lib.iptr(mat)), "solver_set_materials")

    def after_mesh_edit(self, mesh, previous, B_before, converge: bool = True):
        """Follow ``optixP.replaceMesh(mesh, previous)`` + ``updateRadiosityMatrix()``: a new solver on the context's current
        matrix (no rebuild, no reload), restarted from ``B_before`` (the B read before the edit) remapped by
        :func:`remap_bands`; then converged unless ``converge=False``.  Returns the passes of the new solve."""
        self.close()
        self.mesh_, self.numpatches = mesh, mesh.numtriangles
        E, M = self._derive_inputs(self.emission_value)
        self._create_solver(E, M)
        self.restart(remap_bands(B_before, previous, self.emission))
        return self.converge_lightning() if converge else self.numpasses

    def _after_update(self):
        pass

    def get_color_of_patch(self, index: int) -> np.ndarray:
        raise NotImplementedError


class SpectralLightning(Lightning):
    """``SpectralLightning`` (``Lightning.h:99-295``): stop when the residual summed over all bands <= 200."""

    threshold, per_band = 200.0, 0

    def __init__(self, mesh, optixP, emissionval, wavelengthsvec, cuda_enabled=False, matfile=None, converge=True):
        self.numsamples = len(wavelengthsvec)
        self.xyz_per_wavelength = np.stack([cie1931WavelengthToXYZFit(w) for w in wavelengthsvec])  # :245-253
        self.emission_value = emissionval
        E, M = _mat.spectral_inputs(mesh.materials, mesh.materialIndexPerTriangle, emissionval)  # :263-292
        self._cache = None
        self._init(mesh, optixP, E, M, cuda_enabled, matfile, converge)

    def _derive_inputs(self, emissionval):
        return _mat.spectral_inputs(self.mesh_.materials, self.mesh_.materialIndexPerTriangle, emissionval)

    def _after_update(self):
        self._cache = None

    def update_color_cache(self):  # Lightning.h:168-183 (xyz starts from zero here; the reference leaves it uninitialised)
        B = self.lightningvalues
        xyz = np.zeros((B.shape[1], 3), np.float32)
        for j in range(self.numsamples):
            xyz += self.xyz_per_wavelength[j][None, :] * B[j][:, None]
        rgb = np.stack([
            _XYZ2RGB[0, 0] * xyz[:, 0] + _XYZ2RGB[0, 1] * xyz[:, 1] + _XYZ2RGB[0, 2] * xyz[:, 2],
            _XYZ2RGB[1, 0] * xyz[:, 0] + _XYZ2RGB[1, 1] * xyz[:, 1] + _XYZ2RGB[1, 2] * xyz[:, 2],
            _XYZ2RGB[2, 0] * xyz[:, 0] + _XYZ2RGB[2, 1] * xyz[:, 1] + _XYZ2RGB[2, 2] * xyz[:, 2]], axis=1).astype(np.float32)
        maxval = rgb.max(axis=1)
        scale = np.where(maxval > 1, maxval, np.float32(1))
        self._cache = (rgb / scale[:, None]).astype(np.float32)

    def get_color_of_patch(self, index):
        if self._cache is None:
            self.update_color_cache()
        return self._cache[index]


class RGBLightning(Lightning):
    """``RGBLightning`` (``Lightning.h:298-384``): stop when every channel's residual sum <= 1e-4."""

    threshold, per_band = 1e-4, 1

    def __init__(self, mesh, optixP, emissionval, cuda_enabled=False, matfile=None, converge=True):
        self.numsamples = 3
        self.emission_value = emissionval
        E, M = _mat.rgb_inputs(mesh.materials, mesh.materialIndexPerTriangle, emissionval)  # :359-382
        self._init(mesh, optixP, E, M, cuda_enabled, matfile, converge)

    def _derive_inputs(self, emissionval):
        return _mat.rgb_inputs(self.mesh_.materials, self.mesh_.materialIndexPerTriangle, emissionval)

    def get_color_of_patch(self, index):
        return self.lightningvalues[:, index].copy()


class BWLightning(Lightning):
    """``BWLightning`` (``Lightning.h:386-443``): residual = F residual, stop at sum <= 1e-4."""

    threshold, per_band = 1e-4, 1

    def __init__(self, mesh, optixP, emissionval, matfile=None, converge=True):
        self.numsamples = 1
        self.emission_value = emissionval
        E, M = _mat.bw_inputs(mesh.materials, mesh.materialIndexPerTriangle, emissionval)  # :434-442
        self._init(mesh, optixP, E, M, False, matfile, converge)

    def _derive_inputs(self, emissionval):
        return _mat.bw_inputs(self.mesh_.materials, self.mesh_.materialIndexPerTriangle, emissionval)

    def get_color_of_patch(self, index):
        v = self.lightningvalues[0, index]
        return np.array([v, v, v], np.float32)


# ---------------------------------------------------------------------------------------------------------------
# Camera ray cast + patch-colour interpolation: the step right after the solve and the only other optixQuery
# consumer (reference OptixPrimeFunctionality::traceScreen, .cpp:83-131; Camera.h:54-80; Drawer::interpolate,
# Drawer.cpp:161-186).  Rays are generated on the host as in the reference, traced by the closest-hit kernel.
class Camera:
    """``Camera`` of ``visual studio/Camera.h``: eye (0,0,10) looking at the origin, 45 (radian, as glm 0.9.8 reads
    it) field of view, viewport = window size; ``gen_rays_for_screen`` un-projects the near- and far-plane point of
    every (sub)pixel -- the far-plane POINT is what the reference passes as the ray direction."""

    def __init__(self, width: int, height: int, supersampling: int = 4):
        self.eye = np.array([0.0, 0.0, 10.0], np.float32)
        self.dir = np.zeros(3, np.float32)
        self.up = np.array([0.0, 1.0, 0.0], np.float32)
        self.pixwidth, self.pixheight, self.supersampling = width, height, supersampling
        self.viewport = np.array([0.0, 0.0, float(width), float(height)], np.float32)
        dim = int(math.sqrt(supersampling))
        step = np.float32(1.0 / (dim + 1))
        self.antialias_matrix = np.zeros(supersampling * 2, np.float32)  # Camera.h:87-100
        k = 0
        for x in range(1, dim + 1):
            for y in range(1, dim + 1):
                self.antialias_matrix[k], self.antialias_matrix[k + 1] = np.float32(x) * step, np.float32(y) * step
                k += 2

    def matrices(self):
        f32 = np.float32
        def nrm(v):  # glm::normalize = v * (1 / sqrt(dot)), dot = (x*x + y*y) + z*z
            t = (v * v).astype(f32)
            return (v * (f32(1) / np.sqrt(f32(f32(t[0] + t[1]) + t[2]), dtype=f32))).astype(f32)
        def crs(x, y):  # glm::cross
            return np.array([f32(x[1] * y[2]) - f32(y[1] * x[2]), f32(x[2] * y[0]) - f32(y[2] * x[0]), f32(x[0] * y[1]) - f32(y[0] * x[1])], f32)
        def dt(a, b):
            t = (a * b).astype(f32)
            return f32(f32(t[0] + t[1]) + t[2])
        f = nrm((self.dir - self.eye).astype(f32))                                          # glm::lookAt (RH)
        s = nrm(crs(f, self.up))
        u = crs(s, f)
        look = np.eye(4, dtype=f32)  # indexed [col][row] like glm
        look[0, 0], look[1, 0], look[2, 0] = s
        look[0, 1], look[1, 1], look[2, 1] = u
        look[0, 2], look[1, 2], look[2, 2] = -f
        look[3, 0], look[3, 1], look[3, 2] = -dt(s, self.eye), -dt(u, self.eye), dt(f, self.eye)
        aspect = f32(self.pixwidth) / f32(self.pixheight)
        t = f32(math.tan(f32(45.0) / f32(2.0)))                                              # glm::perspective (RH, -1..1)
        zn, zf = f32(0.1), f32(1000.0)
        proj = np.zeros((4, 4), f32)
        proj[0, 0] = f32(1) / (aspect * t)
        proj[1, 1] = f32(1) / t
        proj[2, 3] = -1
        proj[2, 2] = -(zf + zn) / (zf - zn)
        proj[3, 2] = -(f32(2) * zf * zn) / (zf - zn)
        return look, proj

    @staticmethod
    def _mat_mul(a, b):
        """glm mat4 * mat4 ([col][row] storage, float32, glm's association order)."""
        r = np.zeros((4, 4), np.float32)
        for c in range(4):
            r[c] = ((a[0] * b[c, 0] + a[1] * b[c, 1]) + a[2] * b[c, 2]) + a[3] * b[c, 3]
        return r

    @staticmethod
    def _mat_inverse(m):
        """glm::inverse(mat4) restated in float32 (glm/detail/func_matrix.inl:297-358)."""
        f = np.float32
        def co(a, b, c, d):
            return f(f(m[a[0], a[1]] * m[b[0], b[1]]) - f(m[c[0], c[1]] * m[d[0], d[1]]))
        C00 = co((2, 2), (3, 3), (3, 2), (2, 3)); C02 = co((1, 2), (3, 3), (3, 2), (1, 3)); C03 = co((1, 2), (2, 3), (2, 2), (1, 3))
        C04 = co((2, 1), (3, 3), (3, 1), (2, 3)); C06 = co((1, 1), (3, 3), (3, 1), (1, 3)); C07 = co((1, 1), (2, 3), (2, 1), (1, 3))
        C08 = co((2, 1), (3, 2), (3, 1), (2, 2)); C10 = co((1, 1), (3, 2), (3, 1), (1, 2)); C11 = co((1, 1), (2, 2), (2, 1), (1, 2))
        C12 = co((2, 0), (3, 3), (3, 0), (2, 3)); C14 = co((1, 0), (3, 3), (3, 0), (1, 3)); C15 = co((1, 0), (2, 3), (2, 0), (1, 3))
        C16 = co((2, 0), (3, 2), (3, 0), (2, 2)); C18 = co((1, 0), (3, 2), (3, 0), (1, 2)); C19 = co((1, 0), (2, 2), (2, 0), (1, 2))
        C20 = co((2, 0), (3, 1), (3, 0), (2, 1)); C22 = co((1, 0), (3, 1), (3, 0), (1, 1)); C23 = co((1, 0), (2, 1), (2, 0), (1, 1))
        v4 = lambda *x: np.array(x, np.float32)
        F0, F1, F2 = v4(C00, C00, C02, C03), v4(C04, C04, C06, C07), v4(C08, C08, C10, C11)
        F3, F4, F5 = v4(C12, C12, C14, C15), v4(C16, C16, C18, C19), v4(C20, C20, C22, C23)
        V0, V1 = v4(m[1, 0], m[0, 0], m[0, 0], m[0, 0]), v4(m[1, 1], m[0, 1], m[0, 1], m[0, 1])
        V2, V3 = v4(m[1, 2], m[0, 2], m[0, 2], m[0, 2]), v4(m[1, 3], m[0, 3], m[0, 3], m[0, 3])
        I0 = (V1 * F0 - V2 * F1) + V3 * F2
        I1 = (V0 * F0 - V2 * F3) + V3 * F4
        I2 = (V0 * F1 - V1 * F3) + V3 * F5
        I3 = (V0 * F2 - V1 * F4) + V2 * F5
        SA, SB = v4(1, -1, 1, -1), v4(-1, 1, -1, 1)
        inv = np.stack([I0 * SA, I1 * SB, I2 * SA, I3 * SB]).astype(np.float32)
        row0 = v4(inv[0, 0], inv[1, 0], inv[2, 0], inv[3, 0])
        d0 = m[0] * row0
        det = f(f(d0[0] + d0[1]) + f(d0[2] + d0[3]))
        return (inv * f(f(1) / det)).astype(np.float32)

    def gen_rays_for_screen(self, antialiasing: bool) -> np.ndarray:
        """(H*W*samples, 6) float32 in the reference's order ``((y*W + x)*samples + sample)`` (Camera.h:54-80); float32
        arithmetic in glm's operation order (lookAt, perspective, unProject = inverse(proj*model) * clip, / w)."""
        samples = self.supersampling if antialiasing else 1
        matrix = self.antialias_matrix if antialiasing else np.zeros(2, np.float32)
        look, proj = self.matrices()
        inv = self._mat_inverse(self._mat_mul(proj, look))
        W, H = self.pixwidth, self.pixheight
        ys, xs, ss = np.meshgrid(np.arange(H), np.arange(W), np.arange(samples), indexing="ij")
        x_ = (xs.astype(np.float32) + matrix[2 * ss]).astype(np.float32)
        y_ = (ys.astype(np.float32) + matrix[2 * ss + 1]).astype(np.float32)
        out = np.empty((H, W, samples, 6), np.float32)
        two, one = np.float32(2), np.float32(1)
        for depth, sl in ((0.0, slice(0, 3)), (1.0, slice(3, 6))):
            tx = ((x_ - self.viewport[0]) / self.viewport[2]) * two - one
            ty = ((y_ - self.viewport[1]) / self.viewport[3]) * two - one
            tz = np.float32(depth) * two - one
            tw = np.float32(1) * two - one
            obj = ((inv[0][None, :] * tx[..., None] + inv[1][None, :] * ty[..., None]) + (inv[2] * tz + inv[3] * tw)[None, :]).astype(np.float32)
            out[..., sl] = obj[..., :3] / obj[..., 3:4]
        return out.reshape(-1, 6)


def triangles_per_vertex(mesh: MeshS):
    """``MeshS::trianglesPerVertex`` (MeshS.cpp:107-109) as CSR (offsets, triangle ids)."""
    v = mesh.triangleIndices[:, :3].reshape(-1)
    t = np.repeat(np.arange(mesh.numtriangles, dtype=np.int64), 3)
    order = np.argsort(v, kind="stable")
    counts = np.bincount(v, minlength=mesh.vertices.shape[0])
    return np.concatenate([[0], np.cumsum(counts)]), t[order]


def traceScreen(optixP: OptixPrimeFunctionality, camera: Camera, patch_colors: np.ndarray, radiosityRendering: bool = True,
                antialiasing: bool = True, material_colors: np.ndarray | None = None, rays: np.ndarray | None = None,
                return_hits: bool = False):
    """``OptixPrimeFunctionality::traceScreen`` (.cpp:83-131): returns ``optixView`` as (H, W, 3) float32.
    ``patch_colors`` = ``lightning.get_color_of_patch`` for every patch (N,3); with ``radiosityRendering=False`` the frame
    shows ``material_colors[materialIndexPerTriangle]`` instead.  Closest hit, ``isFacingBack``, ``Drawer::interpolate``,
    the supersample average and the clamp all run in one kernel (``daisy_trace_screen``); ``return_hits=True`` also hands
    back the hit records (what the reference files into ``trianglesonScreen`` for picking)."""
    mesh = optixP.mesh
    samples = camera.supersampling if antialiasing else 1
    rays = np.ascontiguousarray(camera.gen_rays_for_screen(antialiasing) if rays is None else rays, np.float32)
    W, H = camera.pixwidth, camera.pixheight
    if rays.reshape(-1, 6).shape[0] != W * H * samples:
        raise ValueError("rays must hold width*height*samples origin/direction pairs")
    if radiosityRendering:
        rgb = np.ascontiguousarray(patch_colors, np.float32)
    else:
        rgb = np.ascontiguousarray(np.asarray(material_colors, np.float32)[mesh.materialIndexPerTriangle], np.float32)
    if rgb.shape != (mesh.numtriangles, 3):
        raise ValueError("one RGB colour per patch is needed")
    out = np.empty((H, W, 3), np.float32)
    hits = np.empty(W * H * samples, HIT_DTYPE) if return_hits else None
    eye = np.ascontiguousarray(camera.eye, np.float32)
    _lib.check(_lib.lib().daisy_trace_screen(optixP._ctx, W, H, samples, _lib.fptr(rays), _lib.fptr(eye), _lib.fptr(rgb),
                                             1 if radiosityRendering else 0, _lib.fptr(out),
                                             hits.ctypes.data if return_hits else None), "trace_screen")
    return (out, hits) if return_hits else out


def write_png(path: str, img: np.ndarray) -> None:
    """Headless stand-in for the reference's ``i`` key (``InputHandler`` -> ``ImageExporter::saveImage``): ``optixView`` as an
    8-bit RGB PNG, bottom row first like the OpenGL read-back (stdlib only: zlib + struct)."""
    import zlib
    a = (np.clip(np.asarray(img, np.float32), 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8)[::-1]
    h, w, _ = a.shape
    raw = b"".join(b"\x00" + a[y].tobytes() for y in range(h))

    def chunk(tag, data):
        c = struct.pack(">I", len(data)) + tag + data
        return c + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)) + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))
