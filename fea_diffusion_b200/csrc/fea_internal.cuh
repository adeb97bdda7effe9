// Internal declarations shared by the translation units of libfea_b200.so.
// Layouts and kernels are described in DESIGN.md.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <map>
#include <string>
#include <vector>

#include "fea_b200.h"

namespace fea {

constexpr int kSlice = 32;      // block rows per SELL slice (= one warp)
constexpr int kCtaRows = 128;   // block rows per CTA in the solver kernels
constexpr int kMaxAdj = 64;     // supported vertex valence + 1
constexpr int kMaxSamplesPerBatch = 1 << 20;

constexpr int kChunk = 32;      // PCG iterations between host polls (even)
constexpr int kMaxTimed = 64;   // event-timed iterations per solve
constexpr int kPcgParamBytes = 512;  // device buffer for the solver's parameter block

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int sm_count = 148;
  // PCG driver state, owned by the context so that CUDA graphs survive across solves
  int32_t* h_flag = nullptr;           // pinned [8]: polled counters
  void* d_pcg_params = nullptr;        // device copy of the current solve's PcgPtrs
  std::map<int64_t, cudaGraphExec_t> pcg_graphs;  // key: grid size class * 2 + two_level
  std::vector<cudaEvent_t> events;     // 3 per timed launch
  cudaEvent_t ev_poll[2] = {nullptr, nullptr};
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
  cudaEvent_t ev_c0 = nullptr, ev_c1 = nullptr;  // around the cluster-path kernel
  int use_graphs = 1;                  // env FEA_NO_GRAPHS=1 disables
  int refine_rounds = 1;               // restarts from the true residual per solve (0 = check only)
  int pcg_path = 0;                    // 0 = auto (on-chip cluster kernel where systems fit), 1 = streaming only
  int cluster_capacity[9] = {-1, -1, -1, -1, -1, -1, -1, -1, -1};  // co-resident clusters of c CTAs (-1 = not queried)
  int row_order = 3;                   // solver row order: 0 = input numbering, 1 = Morton, 2 = strips, 3 = auto
  int cluster_min = 1;                 // smallest cluster size used (1..8)
  int cluster_halo_cap = 1 << 30;      // test knob: on-chip systems with a larger per-CTA halo go to the streaming path
  static constexpr int kAux = 8;       // one stream per cluster class (1..8) beside the main stream
  cudaStream_t aux[kAux] = {};         // cluster kernels of different classes run concurrently
  cudaEvent_t ev_fork = nullptr, ev_join[kAux] = {};
  int prio_lo = 0, prio_hi = 0;        // least / most urgent stream priority this context may use
  cudaStream_t prio_streams[9] = {};   // (cluster_prio knob) stream of class k at its chosen urgency, made on demand
  int prio_streams_key = 0;
  int cluster_prio = 0;                // tuning knob: decimal digit k (from the right) = urgency 1 (the device's least urgent level) .. 6 of class k, 0 = default rule
  int spmv_variant = 0;  // tuning knob (env FEA_SPMV_VARIANT), 0 = default
  int64_t launches = 0;  // kernels launched (bookkeeping for bench.py's gpu_launches)
};

// Per-system (sample) solver scalars, structure of arrays on device.
struct SysScalars {
  double* rz[2];     // r.z of the current / previous iterate (ping-pong by iteration parity)
  double* pq;        // p.Ap of the current iterate
  double* rz0;       // r0.z0
  double* tol2;      // rtol^2 * rz0
  int32_t* done;     // 0 = iterating, 1 = finished
  int32_t* iters;
  int32_t* cap;      // iteration budget of the current (re)start; < max_iter only after a reopen
  double* rz_mon;    // true r.r at the previous monitor pass (streaming path)
  int32_t* arrive;   // [2 ns] arrival counters of the in-kernel second reduction level (p.q / r.r)
  int32_t* rounds;   // extended-precision refinement rounds the system needed (0 for all but ill-conditioned ones)
  int32_t* status;
  double* psumA;     // per-system sums of the CTA partials (two-level mode, huge systems only)
  double* psumB;
  int32_t* n_done;   // single counter: finished systems
};

struct Mg;

struct Batch {
  Ctx* ctx = nullptr;
  int32_t ns = 0, npc = 3;
  int64_t NV = 0, NC = 0;
  int32_t NREG = 0;
  std::vector<int64_t> vtx_off, cell_off;
  std::vector<int32_t> reg_off;
  std::vector<void*> allocs;
  bool assembled = false, solved = false, rasterized = false;

  // inputs on device
  double* xy = nullptr;          // [NV*2]
  int32_t* conn = nullptr;       // [NC*npc] GLOBAL vertex ids, orientation-fixed
  int32_t* cell_dreg = nullptr;  // [NC] global index into D, or -1
  double* D = nullptr;           // [NREG*9]
  uint8_t* fixed = nullptr;      // [NV]
  double* rhs = nullptr;         // [NV*2]
  int64_t* d_vtx_off = nullptr;  // [ns+1]
  int64_t* d_cell_off = nullptr; // [ns+1]
  int32_t* d_reg_off = nullptr;  // [ns+1]
  int32_t* vsample = nullptr;    // [NV]
  int32_t* flips = nullptr;      // [ns]
  // equation map
  int32_t* vrank = nullptr;      // [NV] rank among active vertices of the sample, -1 if fixed
  int32_t* prank = nullptr;      // [NV] the same in the solver's spatial row order (k_spatial_rank)
  int32_t* n_active = nullptr;   // [ns] active vertices
  int64_t* row_base = nullptr;   // [ns+1] first (padded) block row of each sample
  int64_t NBR = 0;               // allocated block rows (upper bound, multiple of kCtaRows)
  int32_t* row_of_vertex = nullptr;  // [NV]
  int32_t* vertex_of_row = nullptr;  // [NBR]
  int32_t* sys_of_cta = nullptr;     // [NBR/kCtaRows]
  int32_t* cta_first = nullptr;      // [ns] first CTA of the system
  int32_t* cta_count = nullptr;      // [ns]
  int32_t max_cta_count = 0;         // host copy: most CTAs any one system owns
  int32_t* active_cta = nullptr;     // [NBR/kCtaRows] int4 work list: CTAs of unfinished systems
  int32_t* cl_order = nullptr;       // [ns] systems of the cluster path: class 0 then class 1
  int32_t cl_off[9] = {}, cl_cnt[9] = {};   // index = CTAs per cluster
  int32_t* cl_counter = nullptr;     // [24] device work-queue heads [1..8], restart count [0], scratch [9], handed back [10], [16..21] three 64-bit block-read counters
  // topology
  int32_t* inc_ptr = nullptr;    // [NV+1] vertex -> stiffness-cell incidence
  int32_t* inc = nullptr;        // entries: cell*4 + local node, ascending
  int32_t* adj_ptr = nullptr;    // [NV+1] vertex adjacency over active vertices (sorted)
  int32_t* adj = nullptr;
  int64_t n_adj = 0;
  int32_t* err_flag = nullptr;   // device error flag (valence overflow etc.)
  // element matrices
  double* ke = nullptr;          // [NC*(2*npc)^2]
  // scaled block-SELL matrix
  int32_t n_slices = 0;
  int32_t* slice_len = nullptr;  // [n_slices]
  int64_t* slice_ptr = nullptr;  // [n_slices+1] in block entries
  int64_t n_blocks = 0;
  double* val = nullptr;         // [n_blocks*4]  one 32-byte block (k00,k01,k10,k11) per entry
  int32_t* col = nullptr;        // [n_blocks]
  // Block scaling S (2x2 per vertex): Khat = S^T K S has IDENTITY diagonal blocks, so plain CG on Khat is
  // 2x2-block-Jacobi PCG on K at no cost per iteration.  With the Cholesky factor L of a vertex's diagonal
  // block, S = L^-T = [[i00, i10], [0, i11]]: dscale = (i00, i11), scoup = i10.
  double* dscale = nullptr;      // [NBR*2] (i00, i11)
  double* scoup = nullptr;       // [NBR] i10
  int32_t max_row_blocks = 0;
  // solver vectors: x, q [NBR*2]; rp [NBR*4] = one 32-byte record (r.x, r.y, p.x, p.y) per block
  // row, so that a neighbour's residual and search direction arrive with ONE 256-bit gather
  double *x = nullptr, *rp = nullptr, *q = nullptr;
  double *xlo = nullptr, *sb = nullptr;       // [NBR*2] low part of refined solutions; S b (extended-precision rounds)
  double *partA = nullptr, *partB = nullptr;  // [NBR/kCtaRows]
  SysScalars sc{};
  double* rz_last = nullptr;   // [ns] r.z at exit
  double* relres = nullptr;    // [ns]
  int32_t* empty = nullptr;    // [ns] 1 = an active vertex has no stiffness (A-18)
  // outputs
  double* u = nullptr;       // [NV*2]
  double* ranges = nullptr;  // [ns*4]
  int32_t img_size = 0;
  uint8_t* images = nullptr; // [ns*2*size*size]
  int32_t* owner = nullptr;  // [ns*size*size]
  double* affine = nullptr;  // [ns*4]
  fea_solve_stats stats{};
  std::vector<float> t_spmv, t_update;  // per timed launch (one per chunk)
  // ---- set-up derived on the device from tags / magnitudes / coordinate lists
  //      (fea_batch_create_from_conditions, k_conditions.cu) ----
  bool from_conditions = false;
  int64_t NR = 0;                  // regions of all samples
  std::vector<int32_t> sreg_off;   // [ns+1] first region of each sample
  std::vector<int64_t> flag_off;   // [ns+1] offset of each sample's flag block: (n_regions + 1) rows of n_v
                                   // bytes, the extra last row is all ones (the plate mask of input.png)
  uint8_t* rflags = nullptr;       // region vertex flags
  int32_t* rcount = nullptr;       // [NR] vertices per region
  int8_t* creg_local = nullptr;    // [NC] sample-local material-table index of each cell, -1 = none
  int32_t* n_reg_used = nullptr;   // [ns] material-table entries in use (terms + overlap combinations)
  // ---- outputs staged on the device for a reader on another stream (fea_batch_stage_outputs) ----
  std::vector<int64_t> stage_field_off;   // [ns+1] first region image of each sample
  uint8_t* stage_regions = nullptr;       // [stage_field_off[ns]][size][size]
  int32_t* stage_class = nullptr;         // [2*ns] floating parts, empty vertices
  cudaEvent_t ev_staged = nullptr;        // recorded behind the last kernel that writes an output
  // ---- multigrid hierarchy (fea_batch_set_refinement, k_mg.cu) ----
  int32_t* conn_given = nullptr;  // [NC*3] connectivity as given (single-sample triangle batches, until assemble)
  Mg* mg = nullptr;
};

// One level of the multigrid hierarchy of a uniformly refined single-sample batch (DESIGN.md section 3.9).
// Level 0 is the coarsest mesh, level `levels` the batch itself.  Vectors are in the level's scaled
// row space (Khat = S^T K S, rows in the level batch's solver order).
struct MgLevel {
  fea_batch* hb = nullptr;       // internal batch of a coarse level (nullptr for the finest: the batch itself)
  Batch* b = nullptr;            // the level's batch
  int64_t nv = 0, nc = 0;
  int32_t* conn = nullptr;       // [nc*3] as-given numbering (derived from the children for coarse levels)
  int32_t* creg = nullptr;       // [nc] cell region (the finest level: its cell_dreg)
  int8_t* creg8 = nullptr;       // [nc] the same as the int8 input of a coarse level batch
  int2* par = nullptr;           // [nv] levels >= 1: (v, -1) for a vertex of level l-1, else the edge's two ends
  int32_t* child_ptr = nullptr;  // [nv(l-1)+1] levels >= 1: vertex of level l-1 -> the midpoints of level l
  int32_t* child = nullptr;      //   that have it as an end, ascending
  double2 *x = nullptr, *bv = nullptr, *r = nullptr, *d[2] = {nullptr, nullptr};   // levels >= 1
  double lmax = 0.0;             // power-iteration estimate of the largest eigenvalue of Khat
  double inv_theta = 0.0, c1[2] = {0.0, 0.0}, c2[2] = {0.0, 0.0};   // Chebyshev coefficients
  double ms = 0.0;               // V-cycle time spent on the level in the last solve
};
struct Mg {
  int levels = 0;
  bool failed = false;           // building the hierarchy failed in fea_batch_assemble: the batch cannot be solved
  std::vector<MgLevel> lev;      // [levels + 1]
  double2 *r = nullptr, *p = nullptr, *q = nullptr;   // outer flexible CG, finest row space (x = Batch::x)
  double *partA = nullptr, *partB = nullptr;          // per-CTA partial sums
  double* sc = nullptr;          // device scalars (kSc* slots, k_mg.cu)
  double* h_sc = nullptr;        // pinned copy
  std::vector<cudaEvent_t> ev;   // 4 per level + 2 around the solve
};

}  // namespace fea

// the opaque handles of the C-ABI
struct fea_ctx {
  fea::Ctx c;
  cudaEvent_t ev_user[8] = {};
  cudaEvent_t ev_join = nullptr;
};
struct fea_batch {
  fea::Batch b;
  fea_ctx* owner = nullptr;
};

namespace fea {

// error bookkeeping shared by the API translation units (fea_api.cu)
int api_fail(fea_ctx* ctx, int code, const char* what, cudaError_t e = cudaSuccess);
void api_free_batch(fea_batch* hb);
// host-side part of batch creation that does not depend on how the set-up arrays were produced:
// sizes, offset tables, cluster classes.  Returns FEA_OK or a status (message set on ctx).
int api_batch_begin(fea_ctx* ctx, int32_t ns, int32_t npc, const int64_t* vtx_off, const int64_t* cell_off,
                    const int32_t* reg_off, fea_batch** out);
// allocations of the arrays launch_setup fills, offset-table uploads, launch_setup itself and the
// device-side ordering of the cluster queues; b.xy, b.D, b.fixed, b.rhs must be allocated and
// (stream-ordered) filled, conn_local / creg_local are consumed.
cudaError_t api_batch_finish(Batch& b, const int8_t* d_creg_local, const int32_t* d_conn_local);
// element stiffness (fill_ke: launch_element_stiffness, or the Galerkin product of a multigrid level),
// topology, block-SELL matrix and solver vectors of a created batch
int api_batch_assemble(fea_ctx* ctx, Batch& b, const std::function<cudaError_t(Batch&)>& fill_ke);

// multigrid path (k_mg.cu): return FEA_OK or a status with the message set on ctx
int mg_set_refinement(fea_ctx* ctx, Batch& b, int levels);   // derive and validate the hierarchy
int mg_assemble(fea_ctx* ctx, Batch& b);                     // coarse level batches, Galerkin operators, smoothers
int mg_solve(fea_ctx* ctx, Batch& b, double rtol, int max_iter);   // flexible CG preconditioned by V-cycles
int mg_apply(fea_ctx* ctx, Batch& b, const double* d_r, double* d_z);   // one V-cycle, active-DOF vectors
void mg_release(Batch& b);

template <class T>
inline cudaError_t dalloc(Batch& b, T** p, int64_t n) {
  *p = nullptr;
  if (n <= 0) n = 1;
  cudaError_t e = cudaMallocAsync((void**)p, sizeof(T) * (size_t)n, b.ctx->stream);
  if (e == cudaSuccess) b.allocs.push_back(*p);
  return e;
}

// ---- launchers implemented in the kernel translation units -----------------
// All return cudaError_t of the launch (cudaGetLastError).
cudaError_t launch_setup(Batch& b, const int8_t* d_cell_region_local, const int32_t* d_conn_local);
cudaError_t launch_cluster_order(Batch& b);                   // longest-job-first queues of the on-chip classes
cudaError_t launch_classify(Batch& b, int32_t* d_floating, int32_t* d_empty);   // A-19, needs the incidence lists
cudaError_t launch_topology_counts(Batch& b);                 // incidence + adjacency counts
cudaError_t launch_topology_fill(Batch& b);                   // adjacency fill
cudaError_t launch_element_stiffness(Batch& b);
cudaError_t launch_cell_strain_stress(Batch& b, int stress_region, double* d_strain, double* d_stress);
cudaError_t launch_sell_lengths(Batch& b);                    // slice_len + slice_ptr
cudaError_t launch_sell_fill(Batch& b);                       // dscale, val, col
cudaError_t launch_csr_export(Batch& b, int32_t s, int32_t* d_indptr, int32_t* d_indices,
                              double* d_data);
// whole lock-step PCG loop (init, chunks of kChunk iterations, polling); fills b.stats / timings
cudaError_t run_pcg(Batch& b, double rtol, int max_iter);
void pcg_release(Ctx& c);                                     // destroys the cached graphs
int pcg_cluster_class(int64_t n_vertices_of_sample, int min_cl);  // CTAs per cluster (1..8), 0: streaming
int pcg_cluster_capacity(Ctx& c, int cl);
int pcg_cluster_rows_per_cta();                               // block rows a CTA of the on-chip path holds                     // co-resident clusters (0 = unavailable)
struct PcgPtrs;
cudaError_t launch_pcg_cluster(Ctx& c, const PcgPtrs* dP, int n_systems, int cl, cudaStream_t st);
cudaError_t launch_finalize(Batch& b);                        // u, ranges, max-iter status
cudaError_t launch_plain_spmv(Batch& b, int32_t s, const double* d_x, double* d_y);
cudaError_t launch_raster(Batch& b, double value_scale);
cudaError_t launch_raster_flags(Batch& b, int64_t n_img, const int64_t* d_field_off, const int64_t* d_flag_off,
                                const uint8_t* d_flags, uint8_t* d_images);
cudaError_t launch_raster_cell_fields(Batch& b, int n_fields, const int32_t* d_ids, const double* d_strain,
                                      const double* d_stress, double scale, double* d_ranges, uint8_t* d_images);
// n_fields vertex-scalar images of one mesh; cell_off2 = device {0, n_cell}
cudaError_t launch_raster_fields(cudaStream_t st, int npc, int64_t n_v, int64_t n_cell, const int32_t* conn,
                                 const double* xy, const double* affine, const int64_t* cell_off2, int size,
                                 int32_t* owner, const double* fields, int n_fields, int cell_fields,
                                 const double* clim, uint8_t* images);

// scans (device-wide, deterministic)
cudaError_t exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* tmp,
                               cudaStream_t st);  // out[n] = total; tmp >= n/4096+2 ints
cudaError_t exclusive_scan_i32_to_i64(const int32_t* in, int64_t* out, int64_t n, int64_t mul,
                                      int64_t* tmp, cudaStream_t st);

}  // namespace fea

// ---- device helpers --------------------------------------------------------
#ifdef __CUDACC__
namespace fea {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// 32-byte aligned quadruple: a 2x2 block (k00,k01,k10,k11) or an (r.x, r.y, p.x, p.y) record;
// sm_100 moves it with one 256-bit load/store (LDG.E.256 / STG.E.256)
struct __align__(32) d4 {
  double x, y, z, w;
};
// streaming 32-byte load that does not allocate in L1 (matrix values, read once per kernel)
__device__ __forceinline__ d4 ld_stream_d4(const d4* p) {
  d4 v;
  asm("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}
// read-only 32-byte load through L1 (vector records gathered by several rows of a CTA)
__device__ __forceinline__ d4 ld_nc_d4(const d4* p) {
  d4 v;
  asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}
// L2 eviction policies: the matrix of a system larger than the L2 streams through it once per SpMV and
// must not push out the vector records that every row gathers (evict_first vs evict_last)
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ d4 ld_stream_d4_hint(const d4* p, uint64_t pol) {
  d4 v;
  asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ d4 ld_nc_d4_hint(const d4* p, uint64_t pol) {
  d4 v;
  asm("ld.global.nc.L2::cache_hint.v4.f64 {%0,%1,%2,%3}, [%4], %5;" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ int ld_stream_i32_hint(const int* p, uint64_t pol) {
  int v;
  asm("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ int ld_stream_i32(const int* p) {
  int v;
  asm("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
// binary search: largest s with off[s] <= i   (off has n+1 entries, off[0] = 0)
__device__ __forceinline__ int seg_of(const int64_t* off, int n, int64_t i) {
  int lo = 0, hi = n;
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (off[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}

}  // namespace fea
#endif
