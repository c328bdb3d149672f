/*
 * daisy_b200.h -- C-ABI of the B200-native form-factor + radiosity-gather path.
 *
 * Drop-in boundary for DaisyRiot's two data-parallel hot paths.  Plain pointers and sizes only; every
 * entry point is blocking (the reference is single-threaded and synchronous, main.cpp:97-113), returns 0 on
 * success or a negative DAISY_E_* code, and never throws.  daisy_last_error() gives the message of the last
 * failure on the calling thread.  Host arrays are copied on entry (the reference's OptiX model likewise
 * snapshots its host buffers at update(), OptixPrimeFunctionality.cpp:38-47); the caller keeps ownership.
 *
 * "VS/" = reference directory "visual studio/".  Layouts accepted verbatim from the reference:
 *   glm::vec3 = 3 packed floats; vertex::TriangleIndex = 6 int32 {v0,v1,v2,n0,n1,n2} (VS/Vertex.h:11-14);
 *   ray = 6 floats origin,direction (RTP_BUFFER_FORMAT_RAY_ORIGIN_DIRECTION, VS/OptixPrimeFunctionality.cpp:68);
 *   daisy_hit = optix_functionality::Hit (VS/optix_functionality.h:10-14); UV = 2 floats (VS/Defines.h:3-6);
 *   daisy_tripl = parallellism::Tripl {int,int,double} (VS/parallellism.cuh:30-33);
 *   band vectors = K contiguous float[N] (std::vector<Eigen::VectorXf>, VS/Lightning.h:107-109);
 *   material matrices = K x K column-major floats (Eigen::MatrixXf, VS/Material.h:17).
 */
#ifndef DAISY_B200_H
#define DAISY_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define DAISY_OK 0
#define DAISY_E_INVALID (-1) /* bad argument */
#define DAISY_E_CUDA (-2)    /* CUDA runtime error (message in daisy_last_error) */
#define DAISY_E_STATE (-3)   /* call out of order (e.g. solver before form factors) */
#define DAISY_E_NOMEM (-4)

#define DAISY_MAX_SAMPLES 64 /* visibility masks are 64-bit; the reference uses RAYS_PER_PATCH = 50 */
/* bands of a solver: kernels exist for 1, 3, 9, 16, 32 and 64 bands and K runs padded up to the next of these (inert zero
 * bands); K > 32 runs only on the tensor-core kernel (DAISY_GATHER=fp32 / ldg: daisy_solver_create returns DAISY_E_INVALID) */
#define DAISY_MAX_BANDS 64

typedef struct daisy_ctx daisy_ctx;       /* ~ OptixPrimeFunctionality (+ the RadMat it fills) */
typedef struct daisy_solver daisy_solver; /* ~ Lightning / SpectralLightning / RGBLightning / BWLightning */

typedef struct { float t; int32_t triangleId; float u, v; } daisy_hit;
typedef struct { int32_t m_row, m_col; double m_value; } daisy_tripl;

/* form-factor arithmetic variant */
#define DAISY_FF_DEVICE 0 /* cuda_on=true : calculateRow, double pi          (VS/parallellism.cu:91-207) */
#define DAISY_FF_HOST 1   /* cuda_on=false: per-pair loop, float pi + reciprocity (VS/OptixPrimeFunctionality.cpp:311-366) */

const char *daisy_last_error(void);
int daisy_version(void);
int daisy_device_count(void);

/* ---- context: mesh upload + LBVH build + sample pattern ------------------------------------------------
 * replaces OptixPrimeFunctionality::OptixPrimeFunctionality(MeshS&)         VS/OptixPrimeFunctionality.cpp:36-64
 * (Context::create, setTriangles(host idx, host vtx), model->update -> here: Morton LBVH on `device`). */
int daisy_ctx_create(const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                     int device, daisy_ctx **out);
void daisy_ctx_destroy(daisy_ctx *ctx);
/* the `rands` pattern (VS/OptixPrimeFunctionality.cpp:55-63); uv = S x {u,v}, 1 <= S <= 64.  The reference
 * draws it from rand() seeded by wall-clock time, so the drop-in takes it as an input. */
int daisy_ctx_set_samples(daisy_ctx *ctx, const float *uv, int S);
/* (the reference's pattern has u >= 0, v >= 0, u + v <= 1; a pattern with points outside the triangle is accepted and gives the
 * same closest-hit answers, but the form-factor kernel then culls nothing and walks the LBVH for every ray) */
/* diagnostic, host only (no device needed): the plane ids daisy_ctx_create assigns -- pid_out[t] >= 1 names a plane shared by
 * triangle t and at least one other triangle (exact for axis-aligned planes, fitted in double precision within 3e-7 x scene
 * extent otherwise), 0 = none.  The form-factor kernel skips triangles lying in the plane of a pair's own two patches. */
int daisy_plane_ids(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int32_t *pid_out);
/* diagnostic, host only: the planar face grids daisy_ctx_create builds (csrc/faces.cu) -- planes holding >= 32 triangles, at
 * most 64 of them, each with a uniform 2-D grid whose cells are empty / covered / mixed and list the triangles near them.  The
 * form-factor kernel resolves a visibility ray against a whole face with one plane crossing and one cell lookup.
 * stats6[6 f ..] = triangles, cells, empty, covered, mixed cells, list entries of face f (f < max_faces); pid_out (may be
 * NULL) = the plane ids after renumbering (face f = id f + 1). */
/* diagnostic, host only: one face's grid -- frame16 = plane (n, d), in-plane axes scaled to cell units with their offsets (cell
 * coordinate a = dot(X, ex.xyz) + ex.w, b likewise), nx, ny, triangle count, 0; state[q] (q = b * nx + a, `capacity` entries) =
 * 0 empty / 1 covered / 2 mixed, count[q] = triangles listed for the cell.  state / count may be NULL (frame only). */
int daisy_face_grid_dump(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int face, float *frame16, signed char *state, int32_t *count,
                         int64_t capacity);
int daisy_face_grid_stats(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int max_faces, int64_t *stats6, int32_t *nfaces_out, int32_t *pid_out);
/* multi-GPU (one process per GPU): this context builds and owns the row block `rank` of `nranks` equal blocks of
 * rows_per_rank = ceil(N/nranks) rounded up to a multiple of 256 when nranks > 1 (a 256-column TMA tile of the
 * residual never straddles two blocks), of 4 when nranks == 1 (default rank 0 of 1 = all rows).  Callers must not
 * re-derive the layout: daisy_ctx_row_range returns it.  Must be called before daisy_formfactors_alloc / _build /
 * _write_rows (DAISY_E_STATE afterwards: the allocation and any IPC mapping are sized from the row range). */
int daisy_ctx_set_partition(daisy_ctx *ctx, int rank, int nranks);
int daisy_ctx_row_range(daisy_ctx *ctx, int *row0, int *row1, int *rows_per_rank);
/* optional: run kernels on this cudaStream_t (default: the legacy default stream) */
int daisy_ctx_set_stream(daisy_ctx *ctx, void *cuda_stream);

/* ---- closest hit ----------------------------------------------------------------------------------------
 * replaces OptixPrimeFunctionality::optixQuery(int, vector<float3>&, vector<Hit>&)   VS/OptixPrimeFunctionality.cpp:66-81
 * RTP_QUERY_TYPE_CLOSEST, host ray buffer in, host hit buffer out; miss => t = -1, triangleId = -1. */
int daisy_query_closest(daisy_ctx *ctx, int n, const float *rays6, daisy_hit *hits);
/* same with device pointers (no copies) */
int daisy_query_closest_device(daisy_ctx *ctx, int n, const float *d_rays6, daisy_hit *d_hits);

/* ---- camera ray cast + shading (the step right after the solve; the only other optixQuery consumer) ---------------
 * replaces OptixPrimeFunctionality::traceScreen(Drawer::RenderContext)                 VS/OptixPrimeFunctionality.cpp:83-131
 *      with triangle_math::isFacingBack (VS/triangle_math.cpp:76-86) and Drawer::interpolate (VS/Drawer.cpp:161-186)
 * fused behind the closest-hit traversal.  rays6: width*height*samples rays in the order Camera::gen_rays_for_screen
 * emits them ((y*width + x)*samples + s, VS/Camera.h:54-80; "direction" = the un-projected far-plane point, exactly as
 * the reference passes it); eye3 = camera.eye; patch_rgb = N x 3, get_color_of_patch of every patch (interpolate = 1,
 * radiosityRendering) or the material rgbcolor of every patch (interpolate = 0).  out_rgb = optixView, height*width*3,
 * clamped to [0,1].  hits_out (may be NULL) = the width*height*samples hit records, for callers that rebuild
 * trianglesonScreen for picking. */
int daisy_trace_screen(daisy_ctx *ctx, int width, int height, int samples, const float *rays6, const float *eye3,
                       const float *patch_rgb, int interpolate, float *out_rgb, daisy_hit *hits_out);

/* ---- form factors -----------------------------------------------------------------------------------------
 * replaces parallellism::runCalculateRadiosityMatrix(SimpleMesh&)                    VS/parallellism.cu:4-89
 * dense unoccluded triplets of rows [row0,row0+nrows): out[(r-row0)*N + c] = {r, c, F_unoccluded(r->c)} */
int daisy_unoccluded_rows(daisy_ctx *ctx, int variant, int row0, int nrows, daisy_tripl *out);
/* replaces cudaCalculateRadiosityMatrix(SpMat&, MeshS&) (variant DEVICE)            VS/OptixPrimeFunctionality.cpp:6-34
 *      and calculateRadiosityMatrix(SpMat&, MeshS&)     (variant HOST)              VS/OptixPrimeFunctionality.cpp:311-366
 * i.e. runCalculateRadiosityMatrix + calculateAllVisibility (:169-242) fused: unoccluded 4x4 rule, S visibility
 * rays per mutually facing pair, RadMat(row,col) = visibility * F(row->col).  The matrix stays resident on the
 * device as dense FP32 rows [row0,row1) x N (leading dimension daisy_formfactors_ld). */
int daisy_formfactors_build(daisy_ctx *ctx, int variant);
int daisy_formfactors_ld(daisy_ctx *ctx, int64_t *ld_out);
/* copy rows to host: out[(r-row0)*N + c], rows must lie inside the context's row range */
int daisy_formfactors_read_rows(daisy_ctx *ctx, int row0, int nrows, float *out);
/* refill an Eigen::SparseMatrix<float> (column-major CSC, sorted inner indices, as setFromTriplets leaves it,
 * VS/OptixPrimeFunctionality.cpp:25).  Call with values==NULL to get nnz first.  Single-GPU contexts only.
 * Entry (r, c), c < N, is listed exactly when F[r][c] != 0.0f (+-0 are not, NaN, +-inf and denormals are), values bit for bit.
 * The conversion runs on the device and only the CSC arrays cross PCIe; DAISY_CSC_HOST=1 converts dense row read-backs on the
 * host instead (same arrays).  DAISY_E_INVALID when nnz > 2^31 - 1 (the count-only call still returns nnz). */
int daisy_formfactors_to_csc(daisy_ctx *ctx, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr);
/* load a dense matrix instead of building it (the reference's on-disk cache path, VS/Lightning.h:84-96) */
int daisy_formfactors_write_rows(daisy_ctx *ctx, int row0, int nrows, const float *in);
/* load F from a CSC matrix (Eigen::SparseMatrix<float> compressed, column-major, as DeserializeMat leaves it, VS/Lightning.h:51-74):
 * outer_ptr = N+1 column starts (outer_ptr[N] == nnz), inner_idx = row of each value, strictly ascending within a column.  Every
 * entry not listed becomes +0.0; listed values are stored bit for bit (explicit zeros and -0.0 included).  Partitioned contexts
 * take the whole matrix and keep the rows of their range.  Same effect on the context as daisy_formfactors_write_rows (F_version
 * moves, the build record is cleared, solvers rescan).  Invalid input: DAISY_E_INVALID and F unchanged.  Only the CSC arrays
 * cross PCIe; they stay resident on the device while validated and scattered when they fit in half its free memory, else they
 * go up in chunks twice (validation, then the scatter). */
int daisy_formfactors_write_csc(daisy_ctx *ctx, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr);
/* how the last daisy_formfactors_write_csc on this context staged the arrays: 1 = one upload kept resident, 2 = column chunks
 * uploaded twice (row indices for the validation, then values and rows for the scatter), 0 = none yet */
int daisy_formfactors_csc_uploads(daisy_ctx *ctx);
/* parity aid: visibility hit masks of rows [row0,row0+nrows): out[(r-row0)*N + c], bit i = sample i of the pair
 * (min(r,c) -> max(r,c)) saw its destination (the test at VS/OptixPrimeFunctionality.cpp:208); 0 if not traced. */
int daisy_visibility_masks(daisy_ctx *ctx, int variant, int row0, int nrows, uint64_t *out);
/* parity aid for matrices too large to read back: exact, order-free digests of rows [row0,row0+nrows) of the resident
 * matrix -- xor_out[r] = XOR over columns c of the float bit patterns, wsum_out[r] = SUM of bits * (2c+1) mod 2^64 */
int daisy_formfactors_row_digest(daisy_ctx *ctx, int row0, int nrows, uint32_t *xor_out, uint64_t *wsum_out);
/* what the last daisy_formfactors_build did: mutually facing pairs this context traced, how many of those have
 * their lower patch index inside this context's row range (summing that over all ranks counts every pair of the
 * matrix once), rays cast (= pairs_traced * S), and device milliseconds of the LBVH build and of the fused
 * form-factor/visibility kernel */
/* number of planar face grids this context built (csrc/faces.cu; 0 with DAISY_FF_FACES=0 or in a scene without large planar faces) */
int daisy_ctx_face_count(daisy_ctx *ctx);
int daisy_formfactors_stats(daisy_ctx *ctx, int64_t *pairs_traced, int64_t *pairs_owned, int64_t *rays, double *lbvh_ms,
                            double *ff_ms);

/* ---- geometry updates ---------------------------------------------------------------------------------------
 * daisy_ctx_update_geometry: new vertex positions (nv x 3) and/or normals (nn x 3) for the mesh given to daisy_ctx_create;
 * the triangle list stays, nv and nn must be the create-time counts (DAISY_E_INVALID otherwise), NULL keeps that array.
 * Everything derived from the geometry is rebuilt as daisy_ctx_create builds it (bounds, plane ids, face grids, LBVH,
 * patch records), so closest hit, daisy_trace_screen, daisy_visibility_masks and daisy_unoccluded_rows answer for the new
 * geometry at once.  F is left as it is until daisy_formfactors_update.
 * daisy_formfactors_update: F becomes, bit for bit, what daisy_formfactors_build(ctx, variant) gives on a fresh context with
 * the current geometry, samples and partition, but only the entries that can differ from the matrix F holds are traced and
 * stored: pairs with a changed patch (a position or normal differs bitwise), and pairs whose shaft meets a moved triangle in
 * its recorded or its current position.  The context records the variant, samples and geometry of its last build or update;
 * everything is traced when F holds no such matrix (no build yet, daisy_formfactors_write_rows since, another variant, other
 * samples) or the sample pattern has points outside the triangle.  Solvers on the context stay valid and rescan F (their B and
 * residual are untouched: reset them).  daisy_formfactors_stats describes the update's kernel run and the rebuild's LBVH.
 * Several processes (CUDA-IPC peers): every rank calls both with identical arrays, then the host barriers, as for the build.
 * daisy_formfactors_update_stats: the last update's triangles changed, tiles and facing pairs this context re-traced, and
 * device milliseconds of the tile classification. */
int daisy_ctx_update_geometry(daisy_ctx *ctx, const float *vertices, int nv, const float *normals, int nn);
/* daisy_ctx_replace_mesh: a new mesh with any counts (objects deleted, added, the vertex array renumbered).  previous[t] (ntri
 * entries) = index in the current mesh of the triangle that new triangle t continues (the same patch, possibly moved), or -1 for
 * a new triangle; each current index appears at most once; current triangles nobody continues are removed.  Invalid input
 * (what daisy_ctx_create rejects, previous out of range or with a duplicate): DAISY_E_INVALID, the context unchanged.
 * Everything daisy_ctx_create derives from the mesh is rebuilt, so N, daisy_ctx_row_range, daisy_formfactors_ld, closest hit,
 * daisy_trace_screen, daisy_visibility_masks and daisy_unoccluded_rows answer for the new mesh at once.  F is remapped at once
 * (its shape always matches N): entry (r, c) = the old entry (previous[r], previous[c]), +0.0 where r or c is new; nothing else
 * in F changes until daisy_formfactors_update, which re-traces only the pairs the edit can reach (pairs with a new or changed
 * patch, and pairs whose shaft meets a moved, new or removed triangle) and gives F bit for bit as a fresh build -- provided the
 * surviving triangles keep their relative order (previous increasing over its entries >= 0); otherwise that update traces
 * everything.  The old and the new matrix coexist during the remap: when both do not fit, DAISY_E_NOMEM and the context is
 * unchanged.  Solvers created on the context before the call return DAISY_E_STATE from every call but destroy: create new
 * ones.  A context partitioned across processes (daisy_ctx_set_partition with nranks > 1) cannot replace its mesh (the other
 * rows of its matrix live in the other processes): DAISY_E_STATE. */
int daisy_ctx_replace_mesh(daisy_ctx *ctx, const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                           const int32_t *previous);
int daisy_formfactors_update(daisy_ctx *ctx, int variant);
int daisy_formfactors_update_stats(daisy_ctx *ctx, int64_t *tris_changed, int64_t *tiles_retraced, int64_t *pairs_retraced, double *classify_ms);

/* multi-GPU build without redundant tracing: allocate (and zero) this rank's rows, publish a 64-byte CUDA IPC handle,
 * receive every rank's handle (nranks x 64 bytes, rank order), then daisy_formfactors_build computes each
 * upper-triangle tile on exactly one rank and stores the tile / its mirror straight into the owning ranks' matrices
 * over NVLink.  The host must barrier across ranks after the build before anyone reads the matrix. */
int daisy_formfactors_alloc(daisy_ctx *ctx);
int daisy_formfactors_ipc_handle(daisy_ctx *ctx, void *handle64);
int daisy_formfactors_set_peers(daisy_ctx *ctx, const void *handles, int nranks);
/* diagnostic: pairs of the last build whose shaft candidate list overflowed and were traced by per-ray LBVH walks */
int64_t daisy_formfactors_pairs_fallback(daisy_ctx *ctx);

/* ---- radiosity / fluorescence gather ------------------------------------------------------------------------
 * replaces the Lightning family (VS/Lightning.h): residual <- M (F residual); B += residual
 *   K=1, M=[1]            : BWLightning       (:386-443)
 *   K=3, M=diag(rho_rgb)  : RGBLightning      (:298-384)
 *   K=#wavelengths, full M: SpectralLightning (:99-295, hot loop :196-226)
 * E: K x N band-major emission (already scaled by emission_value, as set_sampled_emission does, :263-273).
 * M: nmat x K x K column-major; mat_idx: N material ids (MeshS::materialIndexPerTriangle).  1 <= K <= DAISY_MAX_BANDS. */
int daisy_solver_create(daisy_ctx *ctx, int K, const float *E, const float *M, int nmat, const int32_t *mat_idx,
                        daisy_solver **out);
void daisy_solver_destroy(daisy_solver *s);
int daisy_solver_reset(daisy_solver *s);                     /* reset(): residual = B = E             (:159-165) */
/* one pass (increment_lightpass / increment_light_fluorescent); band_sums[K] = sum over patches of the new
 * residual per band (the quantity check_convergence / .sum() test, :255-261), may be NULL */
int daisy_solver_step(daisy_solver *s, double *band_sums);
/* converge_lightning(): while (criterion(residual) > threshold) step.  per_band=0: sum over all bands > threshold
 * (spectral, threshold 200, :145-151); per_band=1: any band sum > threshold (RGB/BW, 1e-4, :336-340, :410-415). */
int daisy_solver_converge(daisy_solver *s, double threshold, int per_band, int max_passes, int *passes_out);
/* converge_lightning with the stop rule evaluated on the device: same arguments, pass count, B, residual and band sums (bit for
 * bit) as daisy_solver_converge, but the host does not wait between passes.  Single GPU, or a partitioned solver with the fused
 * exchange (every rank calls it with the same arguments); DAISY_E_STATE for a partition exchanged by the host.  The passes are
 * launched back to back in batches (on one GPU with programmatic dependent launch, whatever daisy_solver_set_chained says);
 * no per-pass events are recorded, so daisy_solver_last_step_ms keeps its value. */
int daisy_solver_converge_device(daisy_solver *s, double threshold, int per_band, int max_passes, int *passes_out);
int daisy_solver_numpasses(daisy_solver *s);
/* per-band sums of the current residual (what the convergence test looks at), K doubles */
int daisy_solver_band_sums(daisy_solver *s, double *band_sums);
/* lightningvalues and residualvector, K x N band-major (rows of this context's range; full N when single GPU) */
int daisy_solver_read(daisy_solver *s, float *B, float *residual);
/* overwrite the current residual and B from host (K x N band-major) -- used by the end-to-end benchmark */
int daisy_solver_write(daisy_solver *s, const float *B, const float *residual);
/* Warm restart (after the matrix, the emission or the materials changed): one pass that starts the iteration from B_old instead
 * of from E.  B_old = B0 (K x N band-major; a partitioned solver: this rank's K x (row1-row0) rows, as in write_slices), or the
 * solver's current B when B0 == NULL.  The pass streams F once with B_old as its input and, per row and band, forms
 *   y = M_p (F B_old)   (the arithmetic of an ordinary pass),   B_new = y + E,   r = B_new - B_old   (FP32, round to nearest)
 * and stores B = B_new, residual = r; the ordinary passes then continue (r <- M F r, B += r) towards the fixed point
 * B* = E + M F B* of a cold solve.  numpasses becomes 1.  r carries FP32 cancellation noise of about ulp(B) per entry, which
 * the passes contract like any residual.
 * From the restart to the next daisy_solver_reset / _write / _write_slices / _write_partitioned the solver is in restart mode:
 * every band sum (step, band_sums, converge, converge_device) is sum_p |r| -- the residual of a warm start has both signs, and
 * the reference's criteria applied to signed sums could stop while B is still off.  For a cold solve (E, M, F >= 0) that is the
 * same number.  Single GPU, or a partitioned solver with the fused exchange (every rank calls it); DAISY_E_STATE for a
 * partition exchanged by the host. */
int daisy_solver_restart(daisy_solver *s, const float *B0);
/* replace the emission (K x N, whole scene) or the material matrices (nmat x K x K; nmat may grow) and the N material ids: the
 * solver-side set_sampled_emission / set_reflectionvalues / set_reflectionmatrix (Lightning.h:263-292).  B and the residual
 * are untouched; the emission takes effect at the next reset or restart, the materials at the next pass.  Invalid input:
 * DAISY_E_INVALID and the solver unchanged. */
int daisy_solver_set_emission(daisy_solver *s, const float *E);
int daisy_solver_set_materials(daisy_solver *s, const float *M, int nmat, const int32_t *mat_idx);

/* ---- multi-GPU plumbing (one process per GPU; the host does the exchange with NCCL / torch.distributed) -----
 * With daisy_ctx_set_partition(rank, nranks) the residual lives in an exchange buffer of `nranks` equal blocks,
 * block g = [K x rows_per_rank floats][K doubles of partial band sums, padded to 16 B], so that one in-place
 * all-gather of `block_bytes` per rank completes a pass.
 *   daisy_solver_step_local : gather kernel over the local rows, writes block `rank` of the *next* buffer
 *   (host: all_gather in place on next_buffer)
 *   daisy_solver_step_finish: swap buffers, total the per-rank band sums */
int daisy_solver_step_local(daisy_solver *s);
int daisy_solver_exchange_info(daisy_solver *s, void **d_next_buffer, int64_t *block_bytes, int64_t *total_bytes);
int daisy_solver_step_finish(daisy_solver *s, double *band_sums);
/* timing of the last step: device milliseconds of the gather kernel (CUDA events on the context's stream) */
int daisy_solver_last_step_ms(daisy_solver *s, double *ms);
/* on != 0: passes issued without reading the band sums (daisy_solver_step(s, NULL), daisy_solver_step_local) are chained --
 * no per-pass events (daisy_solver_last_step_ms keeps its last value) and, on one GPU, programmatic dependent launch: the
 * next pass's grid moves onto SMs as the previous pass leaves them and streams its first F tiles meanwhile.  Results are
 * unchanged (the kernel waits for the previous pass before it reads or writes anything a pass writes). */
int daisy_solver_set_chained(daisy_solver *s, int on);
/* kernels one pass launches in this solver's configuration: 1 for K <= 9 (streaming, epilogue and exchange wait in one kernel),
 * 3 on the tensor-core path (K = 10-64: residual split, streaming kernel, epilogue), plus 1 with the fused exchange */
int daisy_solver_launches_per_pass(daisy_solver *s);
/* Tile skipping (K <= 9; DAISY_GATHER_SKIP=0 streams the whole matrix instead): a pass streams only the 64-row x 256-column tiles
 * of F that hold an entry other than +-0.  The solver scans F for them at daisy_solver_create and again before the first pass
 * after F changed through daisy_formfactors_build, daisy_formfactors_write_rows or daisy_group_formfactors_build of this
 * process.  A write into this context's rows made by another process through a CUDA-IPC mapping of F after the solver exists
 * is NOT seen: create the solver after the build's barrier (dist.py does).
 * daisy_solver_tile_map: dims2 = row blocks, column steps of the last scan (0, 0 on the dense plan); occ (may be NULL) = that
 * map, 1 = streamed, if capacity >= dims2[0] * dims2[1]; occupied = tiles streamed per pass; scan_ms = device time of the scan. */
int daisy_solver_tile_map(daisy_solver *s, int32_t *dims2, uint8_t *occ, int64_t capacity, int64_t *occupied, double *scan_ms);
/* diagnostic, host only: the plan a pass runs for an nrb x S tile map on `sms` SMs.  info5 = entries, CTAs, longest CTA range,
 * most pieces of one row block, pieces; list = column step of every entry (-1: the null entry of a row block without an
 * occupied tile), off = nrb + 1 entry offsets of the row blocks, pieces6 = {cta, row block, first entry, end entry, idx, np}
 * per piece in CTA order (a null entry's piece has first == end).  list / off / pieces6 may be NULL; capacity = int32 elements
 * each of them holds. */
int daisy_gather_plan_dump(const uint8_t *occ, int nrb, int S, int sms, int32_t *info5, int32_t *list, int32_t *off, int32_t *pieces6,
                           int64_t capacity);

/* Fused exchange (replaces the NCCL all-gather of the loop above when all ranks sit in one NVLink domain):
 *   daisy_solver_ipc_handles: 3 x 64-byte CUDA-IPC handles of this rank's two exchange buffers and its flag array
 *   daisy_solver_set_peers  : the handles of all ranks, rank-major (nranks x 192 bytes), gathered by the caller
 *   daisy_solver_step_fused : one pass; the epilogue kernel stores this rank's block (K x n floats + K band sums) into
 *                             every rank's next buffer over NVLink and raises per-rank flags; the next pass waits on
 *                             the flags on the device.  Same results as step_local / all-gather / step_finish. */
/* partitioned daisy_solver_write: B_local = K x (row1-row0), residual_full = K x N (whole vector on every rank) */
int daisy_solver_write_partitioned(daisy_solver *s, const float *B_local, const float *residual_full);
int daisy_solver_ipc_handles(daisy_solver *s, void *handles192);
int daisy_solver_set_peers(daisy_solver *s, const void *handles, int nranks);
int daisy_solver_step_fused(daisy_solver *s, double *band_sums);


/* upload only this rank's rows: B_local and residual_local are K x (row1-row0).  With more than one rank (fused exchange set
 * up) the residual slice and its band sums are handed to every rank over NVLink like the output of a pass, so the next
 * daisy_solver_step_fused finds the whole vector in place.  Single rank: same as daisy_solver_write. */
int daisy_solver_write_slices(daisy_solver *s, const float *B_local, const float *residual_local);

/* ---- several GPUs behind ONE host process ---------------------------------------------------------------------------------
 * The reference is a single process (main.cpp:97-113: MeshS -> OptixPrimeFunctionality -> Lightning::get_lightning ->
 * converge_lightning); daisy_group gives such a host all GPUs of the box: one context per device (row block g of the matrix
 * on device_ids[g], mesh and LBVH replicated), peer access enabled between all of them, peer pointers wired directly (no CUDA
 * IPC, no NCCL, no second process).  device_ids == NULL: devices 0 .. ndev-1.
 *   daisy_group_formfactors_build : every upper-triangle tile is traced by exactly one device and stored, with its mirror,
 *                                   into the owners' matrices over NVLink; the devices build concurrently
 *   daisy_group_solver_*          : the Lightning family over all devices; a pass is one asynchronous kernel launch per
 *                                   device, the exchange of the residual happens inside the kernels (fused exchange)
 * daisy_group_ctx(g, i) is device i's context for the per-context queries (row range, masks, digests, stats, closest hit). */
typedef struct daisy_group daisy_group;
typedef struct daisy_group_solver daisy_group_solver;
int daisy_group_create(const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                       const int *device_ids, int ndev, daisy_group **out);
void daisy_group_destroy(daisy_group *g);
int daisy_group_size(daisy_group *g);
daisy_ctx *daisy_group_ctx(daisy_group *g, int i);
int daisy_group_set_samples(daisy_group *g, const float *uv, int S);
int daisy_group_formfactors_build(daisy_group *g, int variant);
int daisy_group_formfactors_read_rows(daisy_group *g, int row0, int nrows, float *out);
int daisy_group_formfactors_write_rows(daisy_group *g, int row0, int nrows, const float *in);      /* the matrix-cache path, rows routed to their owners */
int daisy_group_formfactors_to_csc(daisy_group *g, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr);
/* daisy_formfactors_write_csc for the whole group: every device validates before any stores, each keeps its row block */
int daisy_group_formfactors_write_csc(daisy_group *g, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr);
/* unique mutually facing pairs of the whole matrix, rays cast, slowest device's LBVH / form-factor kernel milliseconds */
int daisy_group_formfactors_stats(daisy_group *g, int64_t *pairs, int64_t *rays, double *lbvh_ms, double *ff_ms);
/* daisy_ctx_update_geometry / daisy_formfactors_update on every device (each traces its share of the tiles the update reaches) */
int daisy_group_update_geometry(daisy_group *g, const float *vertices, int nv, const float *normals, int nn);
int daisy_group_formfactors_update(daisy_group *g, int variant);
/* daisy_ctx_replace_mesh on every device: the new row blocks are computed and every device's new matrix allocated first, then
 * each device remaps its block, reading the old rows from whichever device owned them over peer access */
int daisy_group_replace_mesh(daisy_group *g, const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                             const int32_t *previous);
int daisy_group_solver_create(daisy_group *g, int K, const float *E, const float *M, int nmat, const int32_t *mat_idx,
                              daisy_group_solver **out);
void daisy_group_solver_destroy(daisy_group_solver *gs);
int daisy_group_solver_reset(daisy_group_solver *gs);
int daisy_group_solver_step(daisy_group_solver *gs, double *band_sums);       /* band_sums may be NULL: nothing waits */
int daisy_group_solver_converge(daisy_group_solver *gs, double threshold, int per_band, int max_passes, int *passes_out);
/* daisy_solver_converge_device over every device (DAISY_E_STATE if the devices ran different pass counts) */
int daisy_group_solver_converge_device(daisy_group_solver *gs, double threshold, int per_band, int max_passes, int *passes_out);
int daisy_group_solver_numpasses(daisy_group_solver *gs);
int daisy_group_solver_band_sums(daisy_group_solver *gs, double *band_sums);
int daisy_group_solver_read(daisy_group_solver *gs, float *B, float *residual);   /* K x N band-major, whole scene */
int daisy_group_solver_write(daisy_group_solver *gs, const float *B, const float *residual);
/* daisy_solver_restart over every device (B0: K x N whole scene, or NULL), and the two setters on every device */
int daisy_group_solver_restart(daisy_group_solver *gs, const float *B0);
int daisy_group_solver_set_emission(daisy_group_solver *gs, const float *E);
int daisy_group_solver_set_materials(daisy_group_solver *gs, const float *M, int nmat, const int32_t *mat_idx);

#ifdef __cplusplus
}
#endif
#endif
