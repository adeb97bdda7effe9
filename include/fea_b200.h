/*
 * fea_b200.h -- C-ABI of libfea_b200.so: the B200-native replacement for the FEA
 * data-synthesis hot path of namanxkumar/fea-diffusion.
 *
 * The reference has no FFI; its boundary is the Python class
 * datagen.fea_analysis.FEAnalysis (reference datagen/fea_analysis.py:31-613) whose
 * arithmetic runs inside sfepy 2023.3 / scipy SuperLU / VTK.  Each entry point below
 * names the reference lines whose work it replaces.  All functions are extern "C",
 * take plain pointers and sizes, never throw, and return a fea_status (0 = OK);
 * fea_last_error(ctx) gives the message of the last failure on that context.
 *
 * Data model: a *batch* is a set of independent plate-condition samples
 * (one mesh + one constraint/force/material condition each) that are assembled and
 * solved together, lock-step, as one block-diagonal system.  Host arrays are the
 * concatenation over samples with offset tables (C-contiguous fp64/int32/uint8).
 * The caller owns every host buffer; the library owns device memory behind the
 * opaque handles.  One fea_ctx per (host thread, GPU); a ctx owns one CUDA stream.
 *
 * Units: vertex v of a sample has DOFs 2v (x) and 2v+1 (y) (sfepy field 'fu',
 * fea_analysis.py:66; SURVEY.md A-3).
 */
#ifndef FEA_B200_H
#define FEA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FEA_VERSION_MAJOR 0
#define FEA_VERSION_MINOR 3

typedef struct fea_ctx fea_ctx;
typedef struct fea_batch fea_batch;

/* return codes of every entry point */
enum fea_status {
  FEA_OK = 0,
  FEA_BAD_ARG = 1,
  FEA_CUDA_ERROR = 2,
  FEA_OUT_OF_MEMORY = 3,
  FEA_BAD_STATE = 4,      /* call order violated (e.g. solve before assemble) */
  FEA_MESH_ERROR = 5      /* vertex valence above the supported maximum, bad index */
};

/* per-sample solver outcome (fea_batch_download: status[]) */
enum fea_sample_status {
  FEA_SAMPLE_NOT_RUN = -1,
  FEA_SAMPLE_CONVERGED = 0,
  FEA_SAMPLE_MAX_ITER = 1,   /* not converged within max_iter */
  FEA_SAMPLE_BREAKDOWN = 2,  /* p^T A p <= 0 or non-finite: matrix not SPD (floating region, F4) */
  FEA_SAMPLE_EMPTY_ROW = 3,  /* an active vertex touches no stiffness cell: exactly singular
                                (the reference's SuperLU-NaN -> calculate() False path, A-18) */
  FEA_SAMPLE_STAGNATED = 4   /* no progress: the TRUE residual b - K x stopped falling (a mechanism the
                                classifier missed, an inconsistent system), or it stays above 10 rtol
                                although the recursive residual met rtol and the extended-precision
                                rounds could not close the gap (or are switched off, "refine_rounds" 0);
                                u is the best iterate, relres its TRUE residual */
};

/*
 * Concatenated description of n_samples plate-condition problems.
 * Replaces the state FEAnalysis.__init__ builds through sfepy
 * (fea_analysis.py:61-164): mesh, Dirichlet set, material cells, load.
 */
typedef struct fea_batch_desc {
  int32_t n_samples;
  int32_t nodes_per_cell;       /* 3 = P1 triangles, 4 = Q1 quads (uniform over the batch) */
  const int64_t* vtx_off;       /* [n_samples+1] vertex offsets */
  const int64_t* cell_off;      /* [n_samples+1] cell offsets */
  const int32_t* reg_off;       /* [n_samples+1] material-table offsets */
  const double*  xy;            /* [vtx_off[n]*2] vertex coordinates (fea_analysis.py:61) */
  const int32_t* conn;          /* [cell_off[n]*nodes_per_cell] sample-local vertex ids, as read
                                   from the mesh file; orientation is fixed on device (A-2) */
  const int8_t*  cell_region;   /* [cell_off[n]] sample-local material index, or -1 for cells that
                                   carry no stiffness (seam cells, F4; fea_analysis.py:235-252) */
  const double*  D;             /* [reg_off[n]*9] row-major 3x3 elasticity matrices,
                                   strain order (e11, e22, 2e12) (fea_analysis.py:257-266) */
  const uint8_t* fixed;         /* [vtx_off[n]] 1 = both DOFs of the vertex are Dirichlet-zero
                                   (EssentialBC 'u.all': 0, fea_analysis.py:362-369) */
  const double*  rhs;           /* [vtx_off[n]*2] full-DOF load of the final step (t = 1):
                                   N_regions * sum of point-load magnitudes (F2/F3,
                                   fea_analysis.py:313-359) */
} fea_batch_desc;

/*
 * The same n_samples problems described the way the reference's FEAnalysis constructor receives
 * them (fea_analysis.py:32-48): 1-based point tags, force magnitudes and the per-material
 * coordinate lists -- NOT derived arrays.  fea_batch_create_from_conditions runs the region
 * selection of FEAnalysis.__init__ on the device (fea_analysis.py:76-146, 182-194, 235-252):
 *   'vertex k' regions            tag - 1 (negative indices wrap like numpy's), :196-233
 *   _get_points_on_edge           |x1*y2 - x2*y1| < 1e-14 w.r.t. the infinite line through the two
 *                                 tagged vertices, evaluated without FMA contraction, :182-188;
 *                                 kind 'facet': only vertices of mesh edges with BOTH ends selected
 *                                 (SURVEY A-7)
 *   _get_points_in_list           np.isin(coors, list).all(axis=1): x AND y occur anywhere among the
 *                                 listed scalars (exact fp64 equality; hash set on the bit patterns,
 *                                 -0.0 == 0.0, NaN matches nothing), :190-194; kind 'cell': complete
 *                                 cells only (F4), a cell complete in several regions gets the sum of
 *                                 their D (A-18)
 *   edge-force magnitude          F / max(#region vertices, 1), :99-105
 *   load                          n_terms * sum of the per-vertex magnitudes (F2/F3)
 *   D                             plane strain from (E, nu), :263-265 (F1)
 * Several samples may share one mesh (the conditions of a plate): meshes are uploaded once.
 * Sample s has regions in this order: vertex forces, edge forces, vertex constraints, edge
 * constraints, material regions (n_regions[s] of them).
 */
typedef struct fea_conditions_desc {
  int32_t n_meshes;
  int32_t n_samples;
  int32_t nodes_per_cell;       /* 3 or 4, uniform */
  int32_t reserved;             /* 0 */
  const int64_t* mesh_vtx_off;  /* [n_meshes+1] */
  const int64_t* mesh_cell_off; /* [n_meshes+1] */
  const double*  xy;            /* [mesh_vtx_off[n_meshes]*2] */
  const int32_t* conn;          /* [mesh_cell_off[n_meshes]*nodes_per_cell] mesh-local vertex ids */
  const int32_t* sample_mesh;   /* [n_samples] mesh of each sample */
  const int32_t* vforce_off;    /* [n_samples+1] force_vertex_tags_magnitudes */
  const int32_t* vforce_tag;    /* [vforce_off[n]] 1-based point tag */
  const double*  vforce_mag;    /* [vforce_off[n]*2] (fx, fy) */
  const int32_t* eforce_off;    /* [n_samples+1] force_edges_tags_magnitudes */
  const int32_t* eforce_tag;    /* [eforce_off[n]*2] the two bounding point tags */
  const double*  eforce_mag;    /* [eforce_off[n]*2] total (fx, fy) of the edge */
  const int32_t* vfix_off;      /* [n_samples+1] constraints_vertex_tags */
  const int32_t* vfix_tag;      /* [vfix_off[n]] */
  const int32_t* efix_off;      /* [n_samples+1] constraints_edges_tags */
  const int32_t* efix_tag;      /* [efix_off[n]*2] */
  const int32_t* mat_off;       /* [n_samples+1] material regions (material_properties_to_vertices
                                   in dict order); a sample with none is the single-material problem */
  const double*  mat_E_nu;      /* [mat_off[n]*2] (E, nu) of each material region */
  const int64_t* mat_coord_off; /* [mat_off[n]+1] offsets, in points, into mat_coords */
  const double*  mat_coords;    /* [mat_coord_off[last]*2] the (x, y) lists */
  const double*  default_E_nu;  /* [n_samples*2] youngs_modulus, poisson_ratio of samples without a
                                   material table (may be NULL if every sample has one) */
} fea_conditions_desc;

typedef struct fea_batch_info {
  int64_t n_vertices;       /* total vertices */
  int64_t n_cells;
  int64_t n_active_dofs;    /* sum of reduced system sizes */
  int64_t nnz;              /* sum of reduced scalar CSR non-zeros (sfepy pattern, A-11) */
  int64_t block_rows;       /* padded 2x2 block rows of the lock-step system */
  int64_t sell_blocks;      /* stored 2x2 blocks incl. slice padding */
  int32_t n_flipped;        /* cells whose orientation was corrected (A-2) */
  int32_t max_row_blocks;   /* longest block row */
} fea_batch_info;

typedef struct fea_solve_stats {
  int32_t iterations;       /* PCG iterations of the slowest sample */
  int32_t n_converged;
  int32_t spmv_launches_timed;
  int32_t update_launches_timed;
  float   spmv_ms_avg;      /* CUDA-event average duration of the SpMV kernel launch */
  float   update_ms_avg;    /* same for the fused vector-update kernel */
  float   solve_ms;         /* whole solve (both paths), CUDA events on the ctx stream */
  int64_t kernel_launches;  /* kernels launched by this solve */
  /* on-chip path (one system per thread-block cluster, matrix in shared memory) */
  int32_t cluster_systems;     /* systems solved by k_pcg_cluster in this solve */
  int32_t cluster_count;       /* clusters launched (sum over the per-size kernels) */
  int64_t cluster_iterations;  /* sum of their iteration counts */
  float   cluster_ms;          /* CUDA-event duration of the group of per-size kernels */
  int32_t cluster_size;        /* CTAs per cluster (1..8) of the class that solved most systems */
  /* systems whose TRUE residual b - K x missed the tolerance after the recursive one had met it:
   * extended-precision refinement rounds (on-chip path) / restarts from the true residual (streaming) */
  int32_t refined_systems;
  int32_t pad_;
  /* where the on-chip path read its 2x2 blocks from: sum over its systems of iterations x blocks held in
   * tensor memory / in shared memory / streamed from L2 (32 bytes per block and iteration each) */
  int64_t cluster_block_reads_tmem;
  int64_t cluster_block_reads_smem;
  int64_t cluster_block_reads_l2;
} fea_solve_stats;

/* ---- library / context -------------------------------------------------- */
int  fea_version(int* major, int* minor);
int  fea_ctx_create(int device, fea_ctx** out);
/* same, with a CUDA stream priority (0 = default, negative = higher): several contexts on one
 * GPU let the tail of one batch overlap the bulk of the next; distinct priorities stagger them */
int  fea_ctx_create_prio(int device, int priority, fea_ctx** out);
int  fea_ctx_destroy(fea_ctx* ctx);
const char* fea_last_error(const fea_ctx* ctx);
/* pinned host memory for zero-staging uploads/downloads (optional) */
int  fea_host_alloc(fea_ctx* ctx, size_t bytes, void** out);
int  fea_host_free(fea_ctx* ctx, void* p);
int  fea_ctx_synchronize(fea_ctx* ctx);
/* Device staging for pipelined producers: fea_device_upload copies `bytes` from (pinned) host memory into a
 * buffer of fea_device_alloc on the context's stream and returns when the copy is done.  A producer thread with
 * a context of its own uploads the big arrays of the NEXT batch while the solving context is busy;
 * fea_conditions_desc.xy / conn / mat_coords may then point into that device buffer (every other field of the
 * descriptor stays in host memory). */
int  fea_device_alloc(fea_ctx* ctx, size_t bytes, void** out);
int  fea_device_free(fea_ctx* ctx, void* p);
int  fea_device_upload(fea_ctx* ctx, void* dev, const void* host, size_t bytes);
/* CUDA events on the context's stream, for timing regions that span several calls
 * (slot in [0, 8)); elapsed is valid once the later event has completed. */
int  fea_ctx_event_record(fea_ctx* ctx, int32_t slot);
int  fea_ctx_event_elapsed_ms(fea_ctx* ctx, int32_t slot_start, int32_t slot_stop, float* ms);
/* work submitted to ctx after this call starts only once everything submitted to `other` so far
 * has finished (same device): joins several contexts' streams for one event-timed region */
int  fea_ctx_wait_ctx(fea_ctx* ctx, fea_ctx* other);
/* integer options:
 *   "pcg_path"      0 = auto (systems of up to 16384 block rows are solved on chip by k_pcg_cluster,
 *                   larger ones by the streaming kernels), 1 = always the streaming kernels
 *   "cluster_min"   smallest thread-block cluster the on-chip path uses (1..8, default 1); a system
 *                   gets the smallest cluster whose CTAs hold its rows, 2048 per CTA
 *   "row_order"     order of the rows inside the solver: 0 = the input vertex numbering, 1 = Morton
 *                   code, 2 = strips, 3 = auto (default: keep a numbering that is already local,
 *                   sort by strips otherwise).  It decides how local the SpMV gathers are, never
 *                   what is exported (fea_batch_get_csr always follows sfepy's numbering)
 *   "refine_rounds" 0 = the true residual of a converged system is only checked and reported;
 *                   > 0 (default 1) = a system that misses the tolerance on its true residual is
 *                   finished by extended-precision refinement (on-chip path, up to 3 rounds) or
 *                   restarted from the true residual that many times (streaming path)
 *   "cluster_halo_cap"  test knob: the largest number of rows a CTA of the on-chip path accepts
 *                   from its cluster peers (default: whatever fits its shared memory); a system
 *                   above it is handed back to the streaming kernels
 * any other key fails with FEA_BAD_ARG */
int  fea_ctx_set_int(fea_ctx* ctx, const char* key, int64_t value);
/* number of kernels this context has launched so far (graph nodes included) */
int  fea_ctx_kernel_launches(fea_ctx* ctx, int64_t* out);

/* ---- batch life cycle ---------------------------------------------------
 * create   : H2D of the description; cell orientation fix (A-2); Dirichlet
 *            equation map (problem.set_bcs, fea_analysis.py:422; A-9).
 * assemble : element stiffness (dw_lin_elastic, fea_analysis.py:153-160,302-310; A-4/A-5),
 *            matrix graph (sfepy mesh_graph inside problem.solve, :437; A-11),
 *            value assembly with Dirichlet rows/cols dropped (A-10), 2x2 block-Jacobi scaling,
 *            load vector (dw_point_load, :338-344).
 * solve    : block-Jacobi-preconditioned fp64 CG of every sample (on chip, one sample per thread-block
 *            cluster, or lock-step streaming kernels for large systems); replaces
 *            Newton + ScipyDirect + SimpleTimeSteppingSolver (:371-375, 425-439):
 *            one solve at t = 1, load steps are t_k multiples of it (F5).
 *            Also produces per-sample (min,max) of both components (ranges.txt, A-17).
 * rasterize: displacement_x / displacement_y gray images of step 1
 *            (save_output_images, :526-613; custom_plotter.py:121-193; A-16).
 */
int  fea_batch_create(fea_ctx* ctx, const fea_batch_desc* desc, fea_batch** out);
/* The inputs of fea_batch_create / fea_batch_create_from_conditions / fea_batch_rasterize are read by
 * asynchronous copies on the context's stream: the caller must leave them untouched until the next
 * call that synchronises the context (fea_batch_download*, fea_ctx_synchronize, fea_solve_batch
 * returns synchronised). */
int  fea_batch_create_from_conditions(fea_ctx* ctx, const fea_conditions_desc* desc, fea_batch** out);
int  fea_batch_assemble(fea_batch* b);
int  fea_batch_solve(fea_batch* b, double rtol, int32_t max_iter);
/* affine[4*s..] = (ax, bx, ay, by): pixel = a*world + b; value_scale = t_1 (images are of
 * step 1); images are [n_samples][2][size][size] uint8, background 255. */
int  fea_batch_rasterize(fea_batch* b, int32_t size, const double* affine, double value_scale);
int  fea_batch_destroy(fea_batch* b);

/* ---- results (host buffers, may be NULL to skip) ------------------------- */
/* u [n_vertices*2] final-step displacement, zeros at fixed DOFs (A-15), NaN for EMPTY_ROW
 * samples; ranges [n_samples*4] = (min ux, max ux, min uy, max uy) of the final step;
 * iters/status [n_samples]; relres [n_samples] = sqrt(r.r / r0.r0) of the TRUE residual
 * r = S^T (b - K u) in the block-Jacobi-scaled norm (S = inverse transposed Cholesky factors of the
 * vertices' 2x2 diagonal blocks) for converged / stagnated samples. */
int  fea_batch_download(fea_batch* b, double* u, double* ranges, int32_t* iters,
                        double* relres, int32_t* status);
int  fea_batch_download_images(fea_batch* b, uint8_t* images);
/* Region images of every sample (regions_<Region>.png, fea_analysis.py:508-524) with the camera of
 * the preceding fea_batch_rasterize: sample s has field_off[s+1]-field_off[s] regions; flags holds,
 * sample after sample, one uint8 per (region, vertex) (1 = vertex in the region); images
 * [field_off[n]][size][size] uint8: the 0/1 flag interpolated over each triangle, black = 1. */
int  fea_batch_rasterize_flags(fea_batch* b, const int64_t* field_off, const uint8_t* flags,
                               uint8_t* images);
/* Final-step cell averages written into domain.<k>.vtk by the reference's post-process hook
 * (ev_cauchy_strain / ev_cauchy_stress 'el_avg', fea_analysis.py:397-416): strain [n_cells*3] =
 * (e11, e22, 2e12), stress [n_cells*3] = D * strain.  stress_region >= 0: material-table entry of
 * the sample used for EVERY cell (the hook evaluates the single material named 'm' over Omega);
 * -1: each cell's own D, zero for cells without stiffness.  Either pointer may be NULL. */
int  fea_batch_cell_strain_stress(fea_batch* b, int32_t stress_region, double* strain, double* stress);
/* Images of stress / strain components of every sample (outputs_{stress,strain}_{x,y}.png,
 * fea_analysis.py:539-558: cell scalars ("cauchy_stress"|"cauchy_strain", "c0"|"c1"), each normalised
 * to its own range), after fea_batch_rasterize, same camera and colour map.  field_ids[n_fields]:
 * 0 stress_x, 1 stress_y, 2 strain_x, 3 strain_y; stress_region as in fea_batch_cell_strain_stress;
 * images [n_fields][n_samples][size][size] are of value_scale * field (step 1); ranges
 * [n_fields][n_samples][2] = (min, max) of the FINAL step (ranges.txt lines are t_k multiples). */
int  fea_batch_rasterize_cell_components(fea_batch* b, int32_t stress_region, int32_t n_fields,
                                         const int32_t* field_ids, double value_scale, uint8_t* images,
                                         double* ranges);
int  fea_batch_get_info(fea_batch* b, fea_batch_info* out);
int  fea_batch_get_solve_stats(fea_batch* b, fea_solve_stats* out);
/* rounds [n_samples]: extended-precision refinement rounds each sample needed.  0 for ordinary
 * systems.  > 0 marks a system whose fp64 CG stalled above the tolerance (kappa ~ 1e7 and beyond: a
 * weakly held part): it was finished by iterative refinement with a double-double residual and solved
 * to rtol / 100, relres is that residual.  For such a system ANY fp64 solve -- the reference's SuperLU
 * included -- is only defined to about kappa * eps: one rounding of the matrix entries moves the
 * direct solve's own answer by ~1e-8 (tests/test_gpu_workload_parity.py measures it). */
int  fea_batch_get_refine_rounds(fea_batch* b, int32_t* rounds);
/* CUDA-event durations of the SpMV / update launch that opens each chunk of 32 PCG iterations
 * (launch t is iteration 32*t): at most cap entries are written, *n_out = number available. */
int  fea_batch_get_timed_launches(fea_batch* b, int32_t cap, float* spmv_ms, float* update_ms,
                                  int32_t* n_out);

/* ---- what the device set-up of fea_batch_create_from_conditions derived (any pointer may be NULL) --
 * fixed [n_vertices], cell_region [n_cells] (sample-local material-table index, -1 = no stiffness),
 * rhs [n_vertices*2]: the arrays fea_batch_desc would have carried, sample after sample;
 * region_count [total regions]: vertices of every region (an edge force is divided by
 * max(count, 1) in magnitudes.txt, fea_analysis.py:99-115);
 * region_flags: sample after sample, one uint8 per (region, vertex), regions in the order of
 * fea_conditions_desc (the vertex sets regions.vtk / regions_<Region>.png show, :377-381, 508-524). */
int  fea_batch_get_setup(fea_batch* b, uint8_t* fixed, int8_t* cell_region, double* rhs,
                         int32_t* region_count, uint8_t* region_flags);
/* material table: reg_off [n_samples+1] (capacity layout), n_used [n_samples] = terms + overlap
 * combinations in use, D [reg_off[n_samples]*9] */
int  fea_batch_get_materials(fea_batch* b, int32_t* reg_off, int32_t* n_used, double* D);
/* Region images of every sample from the DEVICE-resident flags (after fea_batch_rasterize):
 * sample s contributes its regions in order, then -- if with_plate_mask && with_plate_mask[s] --
 * one image of the constant field 1 (input.png, :472-506).  images [sum][size][size] uint8. */
int  fea_batch_rasterize_regions(fea_batch* b, const uint8_t* with_plate_mask, uint8_t* images);
/* Derived well-posedness check (SURVEY A-19), after fea_batch_assemble: floating_parts[s] = parts
 * of the stiffness mesh (cells connected through shared edges) with fewer than two fixed vertices,
 * empty_vertices[s] = active vertices touching no stiffness cell (the reference's SuperLU-NaN case). */
int  fea_batch_classify(fea_batch* b, int32_t* floating_parts, int32_t* empty_vertices);
/* Staged outputs: the read-back of one batch overlapped with the solve of the next (the batched form of the
 * reference's per-condition file writes, generate.py:126-157, for a pipelined generator).
 * fea_batch_stage_outputs (after fea_batch_rasterize, on the batch's own context) enqueues what is still
 * missing -- for a batch made by fea_batch_create_from_conditions the region images (as
 * fea_batch_rasterize_regions, with_plate_mask may be NULL) and the classifier -- into device buffers the batch
 * owns, records an event behind them and returns without synchronising.
 * fea_batch_fetch_outputs copies the results to host buffers (any may be NULL; pinned memory for real overlap)
 * on the stream of `copy_ctx` (NULL: the batch's own context) after that event and synchronises only that
 * stream; it may run on another host thread while the batch's context already works on the next batch.
 * region_images [fea_batch_staged_region_images][size][size]; the batch is destroyed by its own context's
 * thread after the fetch has returned. */
int  fea_batch_stage_outputs(fea_batch* b, const uint8_t* with_plate_mask);
int  fea_batch_staged_region_images(fea_batch* b, int64_t* n_images);
int  fea_batch_fetch_outputs(fea_batch* b, fea_ctx* copy_ctx, double* u, double* ranges, int32_t* iters,
                             double* relres, int32_t* status, uint8_t* images, uint8_t* region_images,
                             int32_t* floating_parts, int32_t* empty_vertices);

/* ---- inspection entry points used by the parity tests -------------------- */
/* per-sample reduced sizes: n_active_dofs[s], nnz[s] (scalar CSR) */
int  fea_batch_sample_sizes(fea_batch* b, int64_t* n_active_dofs, int64_t* nnz);
/* orientation-fixed connectivity (sample-local ids) and per-sample flip counts */
int  fea_batch_get_conn(fea_batch* b, int32_t* conn, int32_t* n_flipped);
/* element matrices [n_cells][2k][2k], local dof = 2*node + comp; zero for region -1 cells */
int  fea_batch_get_element_stiffness(fea_batch* b, double* ke);
/* reduced scalar CSR of one sample in sfepy's layout (A-11): indptr [n+1], indices [nnz],
 * data [nnz] = UNSCALED stiffness values; any pointer may be NULL */
int  fea_batch_get_csr(fea_batch* b, int32_t sample, int32_t* indptr, int32_t* indices,
                       double* data);
/* y = K x for one sample through the product SpMV kernel (x, y over active DOFs, unscaled) */
int  fea_batch_spmv(fea_batch* b, int32_t sample, const double* x, double* y);

/* ---- multigrid-preconditioned solve of a uniformly refined mesh ---------------------------
 * A batch whose only sample is a uniform red refinement of a coarser mesh may declare its hierarchy
 * (before fea_batch_assemble).  fea_batch_assemble then also builds the coarse levels -- Galerkin
 * operators P^T K P assembled cell by cell, block-Jacobi Chebyshev smoothers -- and fea_batch_solve
 * runs flexible CG preconditioned by one V-cycle per iteration, whose coarsest level is solved by the
 * block-Jacobi CG of fea_batch_solve to rtol 1e-4 (or exactly: fea_batch_set_coarse_solver).  Outputs keep their meaning: iterations are outer
 * iterations, relres is the TRUE residual in the block-Jacobi-scaled norm. */
typedef struct {
  int64_t n_vertices, n_cells, n_active_dofs, nnz;   /* nnz of the reduced scalar CSR */
  double lambda_max;   /* estimate of the largest eigenvalue of the block-Jacobi-scaled operator */
  double vcycle_ms;    /* V-cycle time spent on the level in the last solve, by fea_batch_solve or
                        * fea_batch_solve_load_cases (level 0: the coarse solves) */
} fea_mg_level;
/* The batch's only sample is its own mesh refined `levels` (1..8) times, in the vertex and cell numbering
 * of uniform red refinement: vertices of level l-1 keep their indices, the midpoint of each level-(l-1)
 * edge follows them, children of cell p are p, p+nc, p+2nc, p+3nc = (a,ab,ca), (ab,b,bc), (ca,bc,c),
 * (ab,bc,ca).  Checked on the device against the connectivity AS GIVEN (before the orientation fix) and
 * the coordinates (midpoint == 0.5*(a+b) bit for bit, children share the parent's cell_region):
 * FEA_MESH_ERROR if the mesh is not such a refinement; FEA_BAD_ARG for n_samples != 1,
 * nodes_per_cell != 3 or levels out of range; FEA_BAD_STATE after fea_batch_assemble.  A vertex that no cell
 * references is not a midpoint, so such a mesh is a MESH_ERROR too.  If fea_batch_assemble then fails to build
 * the coarse levels, the batch stays unassembled: a second fea_batch_assemble returns FEA_BAD_STATE. */
int  fea_batch_set_refinement(fea_batch* b, int32_t levels);
/* per level l = 0 (coarsest) .. levels: vertices, cells, active DOFs, nnz, lambda_max estimate,
 * V-cycle ms spent on the level in the last solve; *n_out = levels + 1 */
int  fea_batch_get_mg_levels(fea_batch* b, int32_t cap, fea_mg_level* out, int32_t* n_out);
/* reduced scalar CSR of level l's Galerkin operator, same layout and numbering rule as fea_batch_get_csr */
int  fea_batch_get_level_csr(fea_batch* b, int32_t level, int32_t* indptr, int32_t* indices, double* data);
/* z = M r: one V-cycle on an active-DOF vector of the finest level (unscaled, as fea_batch_spmv) */
int  fea_batch_mg_apply(fea_batch* b, const double* r, double* z);
/* K = n_cases load cases of the batch's one sample, solved together by the multigrid solve of
 * fea_batch_set_refinement / fea_batch_set_coarse_meshes / fea_batch_set_grid_hierarchy.  rhs
 * [n_cases][n_vertices*2]: full-DOF loads in the layout of fea_batch_desc.rhs (values at fixed DOFs are not read).  Outputs (any may be NULL), with the
 * meaning they have in fea_batch_download: u [n_cases][n_vertices*2], ranges [n_cases][4], iters, relres,
 * status [n_cases]; stats as fea_batch_get_solve_stats (iterations = the largest outer count).
 * Case k's outputs are bit for bit those fea_batch_solve gives a batch whose rhs is rhs[k], whatever other
 * cases share the call.  The batch's own results (fea_batch_download, images, strain/stress) are not touched.
 * The K cases share the hierarchy, every matrix read of the V-cycles and outer iterations (vectors of the
 * cases are interleaved per row), and their coarse systems are solved side by side in one batch of K copies
 * of level 0, built on the first call with that K and kept with the hierarchy.
 * FEA_BAD_STATE: no multigrid hierarchy, or not assembled.  FEA_BAD_ARG: n_cases outside 1..8, null rhs,
 * rtol < 0 or max_iter < 1.
 * A successful call keeps its K displacement fields (u as above), ranges and status on the device with the
 * hierarchy, replacing those of the previous successful call whatever its K; the three calls below read them. */
int  fea_batch_solve_load_cases(fea_batch* b, int32_t n_cases, const double* rhs, double rtol, int32_t max_iter,
                                double* u, double* ranges, int32_t* iters, double* relres, int32_t* status,
                                fea_solve_stats* stats);
/* Outputs of every case of the last successful fea_batch_solve_load_cases (K = its n_cases), case-major: case k is,
 * bit for bit, what the single-batch call gives a batch created with rhs[k] and solved by fea_batch_solve (a
 * BREAKDOWN case included: the outputs of its u).  The K cases share the mesh: one cover pass per image call and
 * one read of each cell's geometry and D serve them all.  FEA_BAD_STATE before a successful load-case call;
 * FEA_BAD_ARG for what the single-batch call rejects.
 * fea_batch_load_case_info: *n_cases = K, status [K] (may be NULL) = each kept case's status, *image_size (may be
 * NULL) = size of the camera the last fea_batch_load_case_images kept, 0 before one.  FEA_BAD_STATE (and
 * *n_cases = 0) before a successful load-case call.
 * images [K][2][size][size]: the displacement images of fea_batch_rasterize + fea_batch_download_images with the
 * same size, affine [4] and value_scale.  The call keeps its camera's owner map for the cell components below. */
int  fea_batch_load_case_info(fea_batch* b, int32_t* n_cases, int32_t* status, int32_t* image_size);
int  fea_batch_load_case_images(fea_batch* b, int32_t size, const double* affine, double value_scale, uint8_t* images);
/* strain, stress [K][n_cells*3] as fea_batch_cell_strain_stress; either may be NULL. */
int  fea_batch_load_case_strain_stress(fea_batch* b, int32_t stress_region, double* strain, double* stress);
/* images [n_fields][K][size][size] and ranges [n_fields][K][2] as fea_batch_rasterize_cell_components, with the
 * camera (size, affine) of the last fea_batch_load_case_images on the batch: FEA_BAD_STATE before one. */
int  fea_batch_load_case_cell_components(fea_batch* b, int32_t stress_region, int32_t n_fields, const int32_t* field_ids,
                                         double value_scale, uint8_t* images, double* ranges);

/* ---- multigrid-preconditioned solve of a mesh with coarser meshes of the same domain ------------
 * The batch's only sample (P1 triangles) is the finest level of a hierarchy whose coarser levels are the samples
 * of `coarse`, coarsest first (1..8 levels): meshes of the same domain, each with its own cell_region, D and
 * fixed mask (rhs is not read). Before fea_batch_assemble.  Accepted on batches from fea_batch_create and from
 * fea_batch_create_from_conditions.  Each vertex of level l is located in level l-1 on the device: the
 * lowest-index triangle that contains it (edge-inclusive), or, if it lies outside every triangle by at most
 * 1e-10 * the longest bounding-box side of level l-1, the nearest triangle with barycentric weights clamped to
 * [0, 1] and renormalised.  P_l interpolates linearly from those triangles; Dirichlet vertices have neither
 * rows nor columns.  Coarse operators are the coarse meshes' own stiffness matrices (rediscretised, not
 * Galerkin); smoothers, the coarsest solve, the outer flexible CG and every output are those of
 * fea_batch_set_refinement, and fea_batch_get_mg_levels / get_level_csr / mg_apply keep their meaning.
 * FEA_BAD_ARG: more than one sample, quads, 0 or more than 8 coarse meshes, a level without fewer vertices than
 * the next finer one, a null array.  FEA_BAD_STATE: after fea_batch_assemble, fea_batch_set_refinement or an
 * earlier successful fea_batch_set_coarse_meshes.  FEA_MESH_ERROR: a vertex of level l farther than the
 * tolerance from every triangle of level l-1 (the message names the level and the vertex), or a coarse
 * connectivity index out of range.  If fea_batch_assemble then fails to build the coarse levels, the batch
 * stays unassembled: a second fea_batch_assemble returns FEA_BAD_STATE. */
int  fea_batch_set_coarse_meshes(fea_batch* b, const fea_batch_desc* coarse);
/* Declare `levels` (1..8) coarse levels that fea_batch_assemble builds itself, for a single triangle mesh whose
 * coarser meshes the caller does not have: nested background grids over the mesh's bounding box (DESIGN.md
 * section 3.12).  With h = sqrt(2 * area / n_cells), coarse level levels-1 is a grid of spacing 2h and each
 * coarser level doubles it; the mesh's vertices are located in the finest grid's triangles by the rules of
 * fea_batch_set_coarse_meshes, and grid to grid P is the red refinement's (weights 1 and 1/2).  Grid vertices
 * that no active vertex of the next finer level reaches have no row.  Coarse operators are Galerkin,
 * K_(l-1) = P^T K_l P, so the grids need no material or constraint data.  Solves, load cases and every output
 * are those of fea_batch_set_coarse_meshes, and fea_batch_get_mg_levels / get_level_csr / get_level_transfer
 * read the grid levels.  FEA_BAD_ARG: more than one sample, quads, levels outside 1..8.  FEA_BAD_STATE: after
 * fea_batch_assemble or when the batch already has a hierarchy of any kind.  Accepted on batches from
 * fea_batch_create and from fea_batch_create_from_conditions.  If fea_batch_assemble fails to build the levels
 * (FEA_MESH_ERROR when a Galerkin row of a level would exceed 63 neighbours; the message names the level), the
 * batch stays unassembled: a second fea_batch_assemble returns FEA_BAD_STATE. */
int  fea_batch_set_grid_hierarchy(fea_batch* b, int32_t levels);
/* ---- coarsest-level solver of a multigrid batch ----------------------------------------------
 * FEA_COARSE_CG (the default): each V-cycle solves level 0 by the block-Jacobi CG of fea_batch_solve to rtol 1e-4.
 * FEA_COARSE_DIRECT: fea_batch_assemble also forms level 0's block-Jacobi-scaled operator Khat_0 = S^T K_0 S as a
 * dense matrix (its active block rows in the level's solver order), factorises it by Cholesky on the device and
 * replaces it with its full symmetric inverse; each V-cycle then applies that inverse to the restricted residuals of
 * all its load cases in one read (DESIGN.md section 3.13).  The coarse solve is exact, so the V-cycle is a fixed
 * symmetric operator.  The inverse takes n^2 * 8 bytes for n level-0 DOFs (188 MB at n = 4 844).
 * fea_batch_set_coarse_solver: after fea_batch_set_refinement, set_coarse_meshes or set_grid_hierarchy and before
 * fea_batch_assemble; the last call counts.  FEA_BAD_STATE without a hierarchy or after assemble; FEA_BAD_ARG for
 * another solver value.  With FEA_COARSE_DIRECT, fea_batch_assemble fails with FEA_MESH_ERROR (the message names the
 * number) when level 0 has more than 16 384 active DOFs, an empty row, or a Cholesky pivot at or below 1e-8 (a
 * floating or nearly floating level 0); the batch then stays unassembled: a second assemble returns FEA_BAD_STATE. */
enum { FEA_COARSE_CG = 0, FEA_COARSE_DIRECT = 1 };
typedef struct {
  int32_t solver;      /* FEA_COARSE_CG or FEA_COARSE_DIRECT */
  int32_t n;           /* DOFs of the dense inverse (level 0's active DOFs); 0 for CG */
  double factor_ms;    /* device time of the dense build, the factorisation and the inversion; 0 for CG */
  double min_pivot;    /* smallest Cholesky pivot of Khat_0, in (0, 1]; 0 for CG */
  int64_t bytes;       /* device memory the inverse keeps; 0 for CG */
} fea_coarse_info;
int  fea_batch_set_coarse_solver(fea_batch* b, int32_t solver);
/* FEA_BAD_STATE without a hierarchy or before fea_batch_assemble */
int  fea_batch_get_coarse_info(fea_batch* b, fea_coarse_info* out);
/* x = level 0's solver applied to r, one vector over level 0's active DOFs in the numbering of
 * fea_batch_get_level_csr(b, 0), both unscaled: the dense inverse, or the block-Jacobi CG to rtol 1e-4 that the
 * V-cycle runs.  An inspection call, like fea_batch_mg_apply.  FEA_BAD_ARG for null pointers; FEA_BAD_STATE without
 * a hierarchy or before fea_batch_assemble. */
int  fea_batch_coarse_solve(fea_batch* b, const double* r, double* x);

/* P_l (level l-1 -> level l) as CSR over active DOFs, unscaled: rows = active DOFs of level l, columns = active DOFs
 * of level l-1, same numbering rule as fea_batch_get_csr; level 1..levels; for either kind of hierarchy.  After
 * fea_batch_assemble; any pointer may be NULL (indptr [rows+1] alone gives nnz = indptr[rows]). */
int  fea_batch_get_level_transfer(fea_batch* b, int32_t level, int32_t* indptr, int32_t* indices, double* data);

/* ---- scalar-field images of one mesh ----------------------------------------
 * The point-scalar renders of FEAnalysis.save_input_image / save_region_images (reference
 * fea_analysis.py:472-524: the constant field "1" and the 0/1 region flags of regions.vtk) and the
 * cell-scalar renders of the stress/strain components (:541-549), same camera, coverage rule and
 * 'binary' colour map as fea_batch_rasterize (A-16).
 * fields [n_fields][n_v] (cell_fields = 0, interpolated) or [n_fields][n_cell] (cell_fields = 1,
 * constant per cell); clim [n_fields][2] = (min, max) mapped to white..black;
 * affine [4] as above; images [n_fields][size][size] uint8, background 255. */
int  fea_rasterize_fields(fea_ctx* ctx, const double* xy, int64_t n_v, const int32_t* conn,
                          int64_t n_cell, int32_t nodes_per_cell, const double* fields,
                          int32_t n_fields, int32_t cell_fields, const double* clim,
                          const double* affine, int32_t size, uint8_t* images);

/* ---- one-call convenience: create + assemble + solve (+ rasterize) + download + destroy.
 * This is the host-buffer end-to-end path (the "e2e" number of bench.py). */
int  fea_solve_batch(fea_ctx* ctx, const fea_batch_desc* desc, double rtol, int32_t max_iter,
                     int32_t image_size, const double* affine, double value_scale,
                     double* u, double* ranges, int32_t* iters, double* relres, int32_t* status,
                     uint8_t* images, fea_solve_stats* stats);

#ifdef __cplusplus
}
#endif
#endif /* FEA_B200_H */
