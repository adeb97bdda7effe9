// C-ABI of libfea_b200.so (see include/fea_b200.h): context and batch life cycle, host<->device
// transfers, orchestration of the kernel stages, CUDA-graph driven lock-step PCG loop.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "fea_internal.cuh"

using namespace fea;

namespace {

#define CK(ctx, call)                                                        \
  do {                                                                       \
    cudaError_t e_ = (call);                                                 \
    if (e_ != cudaSuccess)                                                   \
      return api_fail(ctx, e_ == cudaErrorMemoryAllocation ? FEA_OUT_OF_MEMORY : FEA_CUDA_ERROR, #call, e_); \
  } while (0)

__global__ void k_gather_i32(const int32_t* __restrict__ src, const int64_t* __restrict__ idx, int n,
                             int32_t* __restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}

__global__ void k_localize_conn(int64_t NC, int npc, const int64_t* __restrict__ cell_off,
                                const int64_t* __restrict__ vtx_off, int ns, const int32_t* __restrict__ conn,
                                int32_t* __restrict__ out) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  const int s = seg_of(cell_off, ns, c);
  for (int a = 0; a < npc; ++a) out[c * npc + a] = (int32_t)(conn[c * npc + a] - vtx_off[s]);
}

}  // namespace

namespace fea {

int api_fail(fea_ctx* ctx, int code, const char* what, cudaError_t e) {
  if (ctx) {
    char buf[512];
    if (e != cudaSuccess)
      snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    else
      snprintf(buf, sizeof buf, "%s", what);
    ctx->c.err = buf;
  }
  if (e != cudaSuccess) cudaGetLastError();  // clear sticky-less errors
  return code;
}

void api_free_batch(fea_batch* hb) {
  if (!hb) return;
  Batch& b = hb->b;
  cudaSetDevice(b.ctx->device);
  mg_release(b);
  for (void* p : b.allocs) cudaFreeAsync(p, b.ctx->stream);
  b.allocs.clear();
  if (b.ev_staged) cudaEventDestroy(b.ev_staged);
  delete hb;
}

int api_batch_begin(fea_ctx* ctx, int32_t ns, int32_t npc, const int64_t* vtx_off, const int64_t* cell_off,
                    const int32_t* reg_off, fea_batch** out) {
  *out = nullptr;
  if (ns <= 0 || ns > kMaxSamplesPerBatch) return api_fail(ctx, FEA_BAD_ARG, "n_samples out of range");
  if (npc != 3 && npc != 4) return api_fail(ctx, FEA_BAD_ARG, "nodes_per_cell must be 3 or 4");
  if (vtx_off[0] != 0 || cell_off[0] != 0 || reg_off[0] != 0) return api_fail(ctx, FEA_BAD_ARG, "offset tables must start at 0");
  for (int s = 0; s < ns; ++s)
    if (vtx_off[s + 1] < vtx_off[s] || cell_off[s + 1] < cell_off[s] || reg_off[s + 1] < reg_off[s])
      return api_fail(ctx, FEA_BAD_ARG, "offset tables must be non-decreasing");
  if (vtx_off[ns] >= (1LL << 30) || cell_off[ns] >= (1LL << 29)) return api_fail(ctx, FEA_BAD_ARG, "batch too large for 32-bit indices");
  cudaError_t e0 = cudaSetDevice(ctx->c.device);
  if (e0 != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "cudaSetDevice", e0);
  fea_batch* hb = new (std::nothrow) fea_batch();
  if (!hb) return api_fail(ctx, FEA_OUT_OF_MEMORY, "host allocation");
  hb->owner = ctx;
  Batch& b = hb->b;
  b.ctx = &ctx->c;
  b.ns = ns;
  b.npc = npc;
  b.vtx_off.assign(vtx_off, vtx_off + ns + 1);
  b.cell_off.assign(cell_off, cell_off + ns + 1);
  b.reg_off.assign(reg_off, reg_off + ns + 1);
  b.NV = b.vtx_off[ns];
  b.NC = b.cell_off[ns];
  b.NREG = b.reg_off[ns];
  b.NBR = 0;
  for (int s = 0; s < ns; ++s) {
    const int64_t nv = b.vtx_off[s + 1] - b.vtx_off[s];
    const int64_t pad = (nv + kCtaRows - 1) / kCtaRows * kCtaRows;
    b.NBR += pad;
    b.max_cta_count = std::max<int32_t>(b.max_cta_count, (int32_t)(pad / kCtaRows));  // upper bound
  }
  // on-chip solver path: every system is assigned a cluster class by its own size alone (the queue
  // of a class is ordered on the device, launch_cluster_order)
  int32_t n = 0;
  for (int cls = 1; cls <= 8; ++cls) {
    b.cl_off[cls] = n;
    for (int s = 0; s < ns; ++s)
      if (pcg_cluster_class(b.vtx_off[s + 1] - b.vtx_off[s], ctx->c.cluster_min) == cls) ++n;
    b.cl_cnt[cls] = n - b.cl_off[cls];
  }
  *out = hb;
  return FEA_OK;
}

cudaError_t api_batch_finish(Batch& b, const int8_t* creg_local, const int32_t* conn_local) {
  cudaStream_t st = b.ctx->stream;
  const int ns = b.ns;
  cudaError_t e = cudaSuccess;
#define A(call) if (e == cudaSuccess) e = (call)
  A(dalloc(b, &b.conn, b.NC * b.npc));
  A(dalloc(b, &b.cell_dreg, b.NC));
  A(dalloc(b, &b.d_vtx_off, ns + 1));
  A(dalloc(b, &b.d_cell_off, ns + 1));
  A(dalloc(b, &b.d_reg_off, ns + 1));
  A(dalloc(b, &b.vsample, b.NV));
  A(dalloc(b, &b.flips, ns));
  A(dalloc(b, &b.vrank, b.NV));
  A(dalloc(b, &b.prank, b.NV));
  A(dalloc(b, &b.n_active, ns));
  A(dalloc(b, &b.row_base, ns + 1));
  A(dalloc(b, &b.row_of_vertex, b.NV));
  A(dalloc(b, &b.vertex_of_row, b.NBR));
  A(dalloc(b, &b.sys_of_cta, b.NBR / kCtaRows));
  A(dalloc(b, &b.cta_first, ns));
  A(dalloc(b, &b.cta_count, ns));
  A(dalloc(b, &b.err_flag, 4));
  A(dalloc(b, &b.empty, ns));
  A(dalloc(b, &b.cl_order, ns));
  A(dalloc(b, &b.cl_counter, 24));  // queue heads of the cluster classes, restart count, scratch
  A(cudaMemcpyAsync(b.d_vtx_off, b.vtx_off.data(), sizeof(int64_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(b.d_cell_off, b.cell_off.data(), sizeof(int64_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(b.d_reg_off, b.reg_off.data(), sizeof(int32_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  A(cudaMemsetAsync(b.flips, 0, sizeof(int32_t) * ns, st));
  A(cudaMemsetAsync(b.err_flag, 0, sizeof(int32_t) * 4, st));
  A(cudaMemsetAsync(b.empty, 0, sizeof(int32_t) * ns, st));
  A(cudaMemsetAsync(b.vertex_of_row, 0xFF, sizeof(int32_t) * std::max<int64_t>(1, b.NBR), st));
  A(launch_setup(b, creg_local, conn_local));
  A(launch_cluster_order(b));
#undef A
  b.ctx->launches += 7;
  return e;
}

int api_batch_assemble(fea_ctx* ctx, Batch& b, const std::function<cudaError_t(Batch&)>& fill_ke) {
  cudaStream_t st = ctx->c.stream;
  const int N = 2 * b.npc;
  CK(ctx, dalloc(b, &b.inc_ptr, b.NV + 1));
  CK(ctx, dalloc(b, &b.inc, b.NC * b.npc));
  CK(ctx, dalloc(b, &b.adj_ptr, b.NV + 1));
  CK(ctx, dalloc(b, &b.ke, b.NC * N * N));
  b.n_slices = (int32_t)(b.NBR / kSlice);
  CK(ctx, dalloc(b, &b.slice_len, b.n_slices));
  CK(ctx, dalloc(b, &b.slice_ptr, (int64_t)b.n_slices + 1));
  CK(ctx, fill_ke(b));
  CK(ctx, launch_topology_counts(b));
  CK(ctx, launch_sell_lengths(b));
  // one host round trip: totals and error flags
  int32_t h_adj = 0, h_err[3] = {0, 0, 0};
  int64_t h_blocks = 0;
  CK(ctx, cudaMemcpyAsync(&h_adj, b.adj_ptr + b.NV, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(&h_blocks, b.slice_ptr + b.n_slices, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(h_err, b.err_flag, 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  if (h_err[0] & 2) return api_fail(ctx, FEA_MESH_ERROR, "connectivity or cell_region index out of range");
  if (h_err[0] & 1) return api_fail(ctx, FEA_MESH_ERROR, "vertex valence exceeds the supported maximum (63)");
  if (h_err[2] & 4) return api_fail(ctx, FEA_MESH_ERROR, "more than 16 distinct overlap combinations of material regions in one sample");
  b.n_adj = h_adj;
  b.n_blocks = b.n_slices ? h_blocks : 0;
  b.max_row_blocks = h_err[1];
  CK(ctx, dalloc(b, &b.adj, b.n_adj));
  CK(ctx, launch_topology_fill(b));
  CK(ctx, dalloc(b, &b.val, b.n_blocks * 4));
  CK(ctx, dalloc(b, &b.col, b.n_blocks));
  CK(ctx, dalloc(b, &b.dscale, b.NBR * 2));
  CK(ctx, dalloc(b, &b.scoup, b.NBR));
  CK(ctx, dalloc(b, &b.x, b.NBR * 2));
  CK(ctx, dalloc(b, &b.rp, b.NBR * 4));
  CK(ctx, dalloc(b, &b.q, b.NBR * 2));
  CK(ctx, dalloc(b, &b.xlo, b.NBR * 2));
  CK(ctx, dalloc(b, &b.sb, b.NBR * 2));
  const int64_t ncta = b.NBR / kCtaRows;
  CK(ctx, dalloc(b, &b.active_cta, 4 * ncta));  // int4 entries
  CK(ctx, dalloc(b, &b.partA, ncta));
  CK(ctx, dalloc(b, &b.partB, ncta));
  CK(ctx, dalloc(b, &b.sc.rz[0], b.ns));
  CK(ctx, dalloc(b, &b.sc.rz[1], b.ns));
  CK(ctx, dalloc(b, &b.sc.pq, b.ns));
  CK(ctx, dalloc(b, &b.sc.rz0, b.ns));
  CK(ctx, dalloc(b, &b.sc.tol2, b.ns));
  CK(ctx, dalloc(b, &b.sc.done, b.ns));
  CK(ctx, dalloc(b, &b.sc.iters, b.ns));
  CK(ctx, dalloc(b, &b.sc.cap, b.ns));
  CK(ctx, dalloc(b, &b.sc.rz_mon, b.ns));
  CK(ctx, dalloc(b, &b.sc.rounds, b.ns));
  CK(ctx, dalloc(b, &b.sc.arrive, 2 * (int64_t)b.ns));
  CK(ctx, dalloc(b, &b.sc.status, b.ns));
  CK(ctx, dalloc(b, &b.sc.psumA, b.ns));
  CK(ctx, dalloc(b, &b.sc.psumB, b.ns));
  CK(ctx, dalloc(b, &b.sc.n_done, 1));
  CK(ctx, dalloc(b, &b.rz_last, b.ns));
  CK(ctx, dalloc(b, &b.relres, b.ns));
  CK(ctx, dalloc(b, &b.u, b.NV * 2));
  CK(ctx, dalloc(b, &b.ranges, (int64_t)b.ns * 4));
  CK(ctx, cudaMemsetAsync(b.sc.status, 0xFF, sizeof(int32_t) * b.ns, st));
  CK(ctx, cudaMemsetAsync(b.sc.iters, 0, sizeof(int32_t) * b.ns, st));
  CK(ctx, cudaMemsetAsync(b.relres, 0, sizeof(double) * b.ns, st));
  CK(ctx, launch_sell_fill(b));
  ctx->c.launches += 1 + 10 + 4 + 1 + 2;
  b.assembled = true;
  return FEA_OK;
}

}  // namespace fea

extern "C" {

int fea_version(int* major, int* minor) {
  if (major) *major = FEA_VERSION_MAJOR;
  if (minor) *minor = FEA_VERSION_MINOR;
  return FEA_OK;
}

int fea_ctx_create(int device, fea_ctx** out) { return fea_ctx_create_prio(device, 0, out); }

int fea_ctx_create_prio(int device, int priority, fea_ctx** out) {
  if (!out) return FEA_BAD_ARG;
  *out = nullptr;
  fea_ctx* ctx = new (std::nothrow) fea_ctx();
  if (!ctx) return FEA_OUT_OF_MEMORY;
  ctx->c.device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) { delete ctx; return FEA_CUDA_ERROR; }
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);  // lo = least urgent (numerically largest)
  priority = std::max(hi, std::min(lo, priority));
  // The main stream carries the kernel of the LARGEST cluster class of a solve, the auxiliary
  // streams the smaller ones.  Measured on B200 (400-system bench batch, new batch per solve):
  // large clusters first -> 56-58 ms per solve; equal priorities -> 47.5 ms with occasional 56 ms
  // outliers; small clusters first -> 47.8 +- 0.1 ms.  So the auxiliary streams get the more
  // urgent priorities, the smaller the cluster the more urgent.
  if ((e = cudaStreamCreateWithPriority(&ctx->c.stream, cudaStreamNonBlocking, priority)) != cudaSuccess) { delete ctx; return FEA_CUDA_ERROR; }
  cudaDeviceGetAttribute(&ctx->c.sm_count, cudaDevAttrMultiProcessorCount, device);
  if (const char* v = getenv("FEA_SPMV_VARIANT")) ctx->c.spmv_variant = atoi(v);
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  if (const char* v = getenv("FEA_NO_GRAPHS")) ctx->c.use_graphs = atoi(v) ? 0 : 1;
  if (const char* v = getenv("FEA_ROW_ORDER")) ctx->c.row_order = atoi(v);
  if (const char* v = getenv("FEA_CLUSTER_MIN")) ctx->c.cluster_min = std::max(1, std::min(8, atoi(v)));
  if (const char* v = getenv("FEA_PCG_PATH")) ctx->c.pcg_path = (strcmp(v, "stream") == 0 || atoi(v) == 1) ? 1 : 0;
  if (cudaHostAlloc((void**)&ctx->c.h_flag, 8 * sizeof(int32_t), cudaHostAllocDefault) != cudaSuccess ||
      cudaMalloc(&ctx->c.d_pcg_params, kPcgParamBytes) != cudaSuccess) {
    if (ctx->c.h_flag) cudaFreeHost(ctx->c.h_flag);
    cudaStreamDestroy(ctx->c.stream);
    delete ctx;
    cudaGetLastError();
    return FEA_CUDA_ERROR;
  }
  cudaEventCreateWithFlags(&ctx->c.ev_poll[0], cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->c.ev_poll[1], cudaEventDisableTiming);
  cudaEventCreate(&ctx->c.ev_t0);
  cudaEventCreate(&ctx->c.ev_t1);
  cudaEventCreateWithFlags(&ctx->c.ev_fork, cudaEventDisableTiming);
  for (int i = 0; i < Ctx::kAux; ++i) {   // (the device has fewer priority levels than classes: the smallest classes share the most urgent one)
    cudaStreamCreateWithPriority(&ctx->c.aux[i], cudaStreamNonBlocking, std::max(hi, priority - 1 - i));
    cudaEventCreateWithFlags(&ctx->c.ev_join[i], cudaEventDisableTiming);
  }
  ctx->c.prio_lo = priority;
  ctx->c.prio_hi = hi;
  cudaEventCreate(&ctx->c.ev_c0);
  cudaEventCreate(&ctx->c.ev_c1);
  for (auto& ev : ctx->ev_user) cudaEventCreate(&ev);
  cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  ctx->c.events.resize(3 * kMaxTimed);
  for (auto& ev : ctx->c.events) cudaEventCreate(&ev);
  *out = ctx;
  return FEA_OK;
}

int fea_ctx_destroy(fea_ctx* ctx) {
  if (!ctx) return FEA_OK;
  cudaSetDevice(ctx->c.device);
  cudaStreamSynchronize(ctx->c.stream);
  pcg_release(ctx->c);
  for (auto& ev : ctx->c.events) cudaEventDestroy(ev);
  cudaEventDestroy(ctx->c.ev_poll[0]);
  cudaEventDestroy(ctx->c.ev_poll[1]);
  cudaEventDestroy(ctx->c.ev_t0);
  cudaEventDestroy(ctx->c.ev_t1);
  cudaEventDestroy(ctx->c.ev_fork);
  for (int i = 0; i < Ctx::kAux; ++i) {
    cudaEventDestroy(ctx->c.ev_join[i]);
    if (ctx->c.aux[i]) cudaStreamDestroy(ctx->c.aux[i]);
  }
  for (auto& st : ctx->c.prio_streams)
    if (st) cudaStreamDestroy(st);
  cudaEventDestroy(ctx->c.ev_c0);
  cudaEventDestroy(ctx->c.ev_c1);
  for (auto& ev : ctx->ev_user) cudaEventDestroy(ev);
  cudaEventDestroy(ctx->ev_join);
  cudaFreeHost(ctx->c.h_flag);
  cudaFree(ctx->c.d_pcg_params);
  cudaStreamDestroy(ctx->c.stream);
  delete ctx;
  return FEA_OK;
}

const char* fea_last_error(const fea_ctx* ctx) { return ctx ? ctx->c.err.c_str() : "null context"; }

int fea_host_alloc(fea_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return FEA_BAD_ARG;
  cudaSetDevice(ctx->c.device);
  CK(ctx, cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
  return FEA_OK;
}
int fea_host_free(fea_ctx* ctx, void* p) {
  if (!ctx) return FEA_BAD_ARG;
  if (p) CK(ctx, cudaFreeHost(p));
  return FEA_OK;
}
// Device staging buffers: a producer thread with its own context uploads the big input arrays of the NEXT batch
// (coordinates, connectivity, material coordinate lists) while the solving context is busy; the batch is then
// created from device pointers (fea_conditions_desc.xy / conn / mat_coords) with device-to-device copies.
int fea_device_alloc(fea_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return FEA_BAD_ARG;
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaMalloc(out, bytes ? bytes : 1));
  return FEA_OK;
}
int fea_device_free(fea_ctx* ctx, void* p) {
  if (!ctx) return FEA_BAD_ARG;
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaFree(p));
  return FEA_OK;
}
int fea_device_upload(fea_ctx* ctx, void* dev, const void* host, size_t bytes) {
  if (!ctx || (bytes && (!dev || !host))) return FEA_BAD_ARG;
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->c.stream));
  CK(ctx, cudaStreamSynchronize(ctx->c.stream));
  return FEA_OK;
}

int fea_ctx_synchronize(fea_ctx* ctx) {
  if (!ctx) return FEA_BAD_ARG;
  CK(ctx, cudaStreamSynchronize(ctx->c.stream));
  return FEA_OK;
}

int fea_ctx_event_record(fea_ctx* ctx, int32_t slot) {
  if (!ctx || slot < 0 || slot >= 8) return FEA_BAD_ARG;
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaEventRecord(ctx->ev_user[slot], ctx->c.stream));
  return FEA_OK;
}
int fea_ctx_event_elapsed_ms(fea_ctx* ctx, int32_t a, int32_t b, float* ms) {
  if (!ctx || !ms || a < 0 || a >= 8 || b < 0 || b >= 8) return FEA_BAD_ARG;
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaEventSynchronize(ctx->ev_user[b]));
  CK(ctx, cudaEventElapsedTime(ms, ctx->ev_user[a], ctx->ev_user[b]));
  return FEA_OK;
}
int fea_ctx_wait_ctx(fea_ctx* ctx, fea_ctx* other) {
  if (!ctx || !other) return FEA_BAD_ARG;
  if (ctx == other) return FEA_OK;
  if (ctx->c.device != other->c.device) return api_fail(ctx, FEA_BAD_ARG, "contexts are on different devices");
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaEventRecord(other->ev_join, other->c.stream));
  CK(ctx, cudaStreamWaitEvent(ctx->c.stream, other->ev_join, 0));
  return FEA_OK;
}
int fea_ctx_set_int(fea_ctx* ctx, const char* key, int64_t value) {
  if (!ctx || !key) return FEA_BAD_ARG;
  if (strcmp(key, "pcg_path") == 0) ctx->c.pcg_path = value == 1 ? 1 : 0;
  else if (strcmp(key, "row_order") == 0) ctx->c.row_order = (value >= 1 && value <= 3) ? (int)value : 0;
  else if (strcmp(key, "cluster_halo_cap") == 0) ctx->c.cluster_halo_cap = value < 0 ? 0 : value > (1 << 30) ? (1 << 30) : (int)value;
  else if (strcmp(key, "cluster_prio") == 0) ctx->c.cluster_prio = (int)value;
  else if (strcmp(key, "cluster_min") == 0) ctx->c.cluster_min = value < 1 ? 1 : value > 8 ? 8 : (int)value;
  else if (strcmp(key, "refine_rounds") == 0) ctx->c.refine_rounds = value < 0 ? 0 : value > 8 ? 8 : (int)value;
  else if (strcmp(key, "spmv_variant") == 0) ctx->c.spmv_variant = (int)value;
  else if (strcmp(key, "use_graphs") == 0) ctx->c.use_graphs = value ? 1 : 0;
  else return api_fail(ctx, FEA_BAD_ARG, "unknown option key");
  return FEA_OK;
}
int fea_ctx_kernel_launches(fea_ctx* ctx, int64_t* out) {
  if (!ctx || !out) return FEA_BAD_ARG;
  *out = ctx->c.launches;
  return FEA_OK;
}

// ---------------------------------------------------------------------------
int fea_batch_create(fea_ctx* ctx, const fea_batch_desc* d, fea_batch** out) {
  if (!ctx || !d || !out) return FEA_BAD_ARG;
  *out = nullptr;
  if (!d->vtx_off || !d->cell_off || !d->reg_off || !d->xy || !d->conn || !d->cell_region || !d->D || !d->fixed || !d->rhs)
    return api_fail(ctx, FEA_BAD_ARG, "null array in fea_batch_desc");
  fea_batch* hb = nullptr;
  int rc = api_batch_begin(ctx, d->n_samples, d->nodes_per_cell, d->vtx_off, d->cell_off, d->reg_off, &hb);
  if (rc != FEA_OK) return rc;
  Batch& b = hb->b;
  cudaStream_t st = ctx->c.stream;
  int32_t* conn_local = nullptr;
  int8_t* creg_local = nullptr;
  cudaError_t e = cudaSuccess;
#define A(call) if (e == cudaSuccess) e = (call)
  A(dalloc(b, &b.xy, b.NV * 2));
  A(dalloc(b, &b.D, (int64_t)b.NREG * 9));
  A(dalloc(b, &b.fixed, b.NV));
  A(dalloc(b, &b.rhs, b.NV * 2));
  A(cudaMallocAsync((void**)&conn_local, sizeof(int32_t) * std::max<int64_t>(1, b.NC * b.npc), st));
  A(cudaMallocAsync((void**)&creg_local, std::max<int64_t>(1, b.NC), st));
  A(cudaMemcpyAsync(b.xy, d->xy, sizeof(double) * b.NV * 2, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(conn_local, d->conn, sizeof(int32_t) * b.NC * b.npc, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(creg_local, d->cell_region, b.NC, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(b.D, d->D, sizeof(double) * 9 * b.NREG, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(b.fixed, d->fixed, b.NV, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(b.rhs, d->rhs, sizeof(double) * b.NV * 2, cudaMemcpyHostToDevice, st));
  A(api_batch_finish(b, creg_local, conn_local));
  if (e == cudaSuccess && b.ns == 1 && b.npc == 3) {   // a possible uniform refinement (fea_batch_set_refinement)
    b.conn_given = conn_local;
    b.allocs.push_back(conn_local);
  } else if (conn_local) {
    cudaFreeAsync(conn_local, st);
  }
  if (creg_local) cudaFreeAsync(creg_local, st);
#undef A
  if (e != cudaSuccess) {
    rc = api_fail(ctx, e == cudaErrorMemoryAllocation ? FEA_OUT_OF_MEMORY : FEA_CUDA_ERROR, "fea_batch_create", e);
    api_free_batch(hb);
    return rc;
  }
  *out = hb;
  return FEA_OK;
}

int fea_batch_destroy(fea_batch* hb) {
  if (!hb) return FEA_OK;
  api_free_batch(hb);
  return FEA_OK;
}

int fea_batch_assemble(fea_batch* hb) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (b.assembled) return FEA_OK;
  if (b.mg && b.mg->failed) return api_fail(ctx, FEA_BAD_STATE, "building the multigrid hierarchy of this batch failed");
  CK(ctx, cudaSetDevice(ctx->c.device));
  int rc = api_batch_assemble(ctx, b, launch_element_stiffness);
  if (rc == FEA_OK && b.mg) {
    rc = mg_assemble(ctx, b);
    if (rc != FEA_OK) {   // terminal: no solve on a half-built hierarchy, no second build over it
      b.assembled = false;
      b.mg->failed = true;
    }
  }
  if (b.conn_given) {   // only fea_batch_set_refinement, which must precede assemble, reads it
    cudaFreeAsync(b.conn_given, ctx->c.stream);
    b.allocs.erase(std::find(b.allocs.begin(), b.allocs.end(), (void*)b.conn_given));
    b.conn_given = nullptr;
    if (b.mg) b.mg->lev[b.mg->levels].conn = nullptr;
  }
  return rc;
}

int fea_batch_solve(fea_batch* hb, double rtol, int32_t max_iter) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_solve before fea_batch_assemble");
  if (!(rtol >= 0.0) || max_iter < 1) return api_fail(ctx, FEA_BAD_ARG, "rtol must be >= 0 and max_iter >= 1");
  CK(ctx, cudaSetDevice(ctx->c.device));
  if (b.mg) {
    const int rc = mg_solve(ctx, b, rtol, max_iter);
    if (rc != FEA_OK) return rc;
  } else {
    CK(ctx, run_pcg(b, rtol, max_iter));
  }
  b.solved = true;
  return FEA_OK;
}

int fea_batch_rasterize(fea_batch* hb, int32_t size, const double* affine, double value_scale) {
  if (!hb || !affine) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.solved) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_rasterize before fea_batch_solve");
  if (size < 1 || size > 8192) return api_fail(ctx, FEA_BAD_ARG, "image size out of range");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (b.img_size != size) {
    const int64_t per = (int64_t)size * size;
    CK(ctx, dalloc(b, &b.images, (int64_t)b.ns * 2 * per));
    CK(ctx, dalloc(b, &b.owner, (int64_t)b.ns * per));
    if (!b.affine) CK(ctx, dalloc(b, &b.affine, (int64_t)b.ns * 4));
    b.img_size = size;
  }
  CK(ctx, cudaMemcpyAsync(b.affine, affine, sizeof(double) * 4 * b.ns, cudaMemcpyHostToDevice, st));
  CK(ctx, launch_raster(b, value_scale));
  ctx->c.launches += 3;
  b.rasterized = true;
  return FEA_OK;
}

int fea_batch_download(fea_batch* hb, double* u, double* ranges, int32_t* iters, double* relres, int32_t* status) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.solved) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_download before fea_batch_solve");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (u) CK(ctx, cudaMemcpyAsync(u, b.u, sizeof(double) * 2 * b.NV, cudaMemcpyDeviceToHost, st));
  if (ranges) CK(ctx, cudaMemcpyAsync(ranges, b.ranges, sizeof(double) * 4 * b.ns, cudaMemcpyDeviceToHost, st));
  if (iters) CK(ctx, cudaMemcpyAsync(iters, b.sc.iters, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  if (relres) CK(ctx, cudaMemcpyAsync(relres, b.relres, sizeof(double) * b.ns, cudaMemcpyDeviceToHost, st));
  if (status) CK(ctx, cudaMemcpyAsync(status, b.sc.status, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return FEA_OK;
}

int fea_batch_rasterize_flags(fea_batch* hb, const int64_t* field_off, const uint8_t* flags, uint8_t* images) {
  if (!hb || !field_off || !flags || !images) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.rasterized) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_rasterize_flags before fea_batch_rasterize");
  if (field_off[0] != 0) return api_fail(ctx, FEA_BAD_ARG, "field_off must start at 0");
  std::vector<int64_t> flag_off(b.ns + 1, 0);
  for (int s = 0; s < b.ns; ++s) {
    if (field_off[s + 1] < field_off[s]) return api_fail(ctx, FEA_BAD_ARG, "field_off must be non-decreasing");
    flag_off[s + 1] = flag_off[s] + (field_off[s + 1] - field_off[s]) * (b.vtx_off[s + 1] - b.vtx_off[s]);
  }
  const int64_t n_img = field_off[b.ns], n_flags = flag_off[b.ns];
  if (n_img == 0) return FEA_OK;
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  const size_t per = (size_t)b.img_size * b.img_size, tab = sizeof(int64_t) * (b.ns + 1);
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t o_fo = 0, o_go = up(tab), o_fl = o_go + up(tab), o_im = o_fl + up((size_t)n_flags), total = o_im + up(n_img * per);
  char* d = nullptr;
  CK(ctx, cudaMallocAsync((void**)&d, total, st));
  cudaError_t e = cudaMemcpyAsync(d + o_fo, field_off, tab, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + o_go, flag_off.data(), tab, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + o_fl, flags, (size_t)n_flags, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = launch_raster_flags(b, n_img, (const int64_t*)(d + o_fo), (const int64_t*)(d + o_go),
                                                (const uint8_t*)(d + o_fl), (uint8_t*)(d + o_im));
  if (e == cudaSuccess) e = cudaMemcpyAsync(images, d + o_im, n_img * per, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // flag_off (host vector) must outlive the copy
  cudaFreeAsync(d, st);
  ctx->c.launches += 1;
  if (e != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "fea_batch_rasterize_flags", e);
  return FEA_OK;
}

int fea_batch_cell_strain_stress(fea_batch* hb, int32_t stress_region, double* strain, double* stress) {
  if (!hb || (!strain && !stress)) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.solved) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_cell_strain_stress before fea_batch_solve");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  double* d = nullptr;
  const size_t n = (size_t)std::max<int64_t>(1, b.NC * 3);
  CK(ctx, cudaMallocAsync((void**)&d, sizeof(double) * 2 * n, st));
  cudaError_t e = launch_cell_strain_stress(b, stress_region, d, d + n);
  if (e == cudaSuccess && strain) e = cudaMemcpyAsync(strain, d, sizeof(double) * 3 * b.NC, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && stress) e = cudaMemcpyAsync(stress, d + n, sizeof(double) * 3 * b.NC, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFreeAsync(d, st);
  ctx->c.launches += 1;
  if (e != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "fea_batch_cell_strain_stress", e);
  return FEA_OK;
}

int fea_batch_rasterize_cell_components(fea_batch* hb, int32_t stress_region, int32_t n_fields, const int32_t* field_ids,
                                        double value_scale, uint8_t* images, double* ranges) {
  if (!hb || !field_ids || n_fields < 1 || n_fields > 4 || (!images && !ranges)) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.rasterized) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_rasterize_cell_components before fea_batch_rasterize");
  for (int f = 0; f < n_fields; ++f)
    if (field_ids[f] < 0 || field_ids[f] > 3) return api_fail(ctx, FEA_BAD_ARG, "field id must be 0..3");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  const size_t per = (size_t)b.img_size * b.img_size, nc3 = (size_t)std::max<int64_t>(1, b.NC * 3);
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t o_stress = up(sizeof(double) * nc3), o_ids = o_stress + up(sizeof(double) * nc3), o_rng = o_ids + 256,
               o_img = o_rng + up(sizeof(double) * 2 * n_fields * b.ns), total = o_img + up((size_t)n_fields * b.ns * per);
  char* d = nullptr;
  CK(ctx, cudaMallocAsync((void**)&d, total, st));
  int32_t ids[4] = {0, 0, 0, 0};
  for (int f = 0; f < n_fields; ++f) ids[f] = field_ids[f];
  cudaError_t e = cudaMemcpyAsync(d + o_ids, ids, sizeof(ids), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = launch_cell_strain_stress(b, stress_region, (double*)d, (double*)(d + o_stress));
  if (e == cudaSuccess)
    e = launch_raster_cell_fields(b, n_fields, (const int32_t*)(d + o_ids), (const double*)d, (const double*)(d + o_stress),
                                  value_scale, (double*)(d + o_rng), (uint8_t*)(d + o_img));
  if (e == cudaSuccess && images) e = cudaMemcpyAsync(images, d + o_img, (size_t)n_fields * b.ns * per, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && ranges) e = cudaMemcpyAsync(ranges, d + o_rng, sizeof(double) * 2 * n_fields * b.ns, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);   // ids (host array) must outlive the copy
  cudaFreeAsync(d, st);
  ctx->c.launches += 3;
  if (e != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "fea_batch_rasterize_cell_components", e);
  return FEA_OK;
}

int fea_batch_download_images(fea_batch* hb, uint8_t* images) {
  if (!hb || !images) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.rasterized) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_download_images before fea_batch_rasterize");
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaMemcpyAsync(images, b.images, (size_t)b.ns * 2 * b.img_size * b.img_size, cudaMemcpyDeviceToHost, ctx->c.stream));
  CK(ctx, cudaStreamSynchronize(ctx->c.stream));
  return FEA_OK;
}

int fea_batch_sample_sizes(fea_batch* hb, int64_t* n_active_dofs, int64_t* nnz) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_sample_sizes before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  std::vector<int32_t> na(b.ns), ap(b.ns + 1);
  int32_t* d_tmp = nullptr;
  CK(ctx, cudaMallocAsync((void**)&d_tmp, sizeof(int32_t) * (b.ns + 1), st));
  k_gather_i32<<<(b.ns + 1 + 255) / 256, 256, 0, st>>>(b.adj_ptr, b.d_vtx_off, b.ns + 1, d_tmp);
  CK(ctx, cudaMemcpyAsync(ap.data(), d_tmp, sizeof(int32_t) * (b.ns + 1), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(na.data(), b.n_active, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  cudaFreeAsync(d_tmp, st);
  for (int s = 0; s < b.ns; ++s) {
    if (n_active_dofs) n_active_dofs[s] = 2 * (int64_t)na[s];
    if (nnz) nnz[s] = 4 * (int64_t)(ap[s + 1] - ap[s]);
  }
  return FEA_OK;
}

int fea_batch_get_info(fea_batch* hb, fea_batch_info* out) {
  if (!hb || !out) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_info before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  std::vector<int32_t> na(b.ns), fl(b.ns);
  int64_t rows = 0;
  CK(ctx, cudaMemcpy(na.data(), b.n_active, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost));
  CK(ctx, cudaMemcpy(fl.data(), b.flips, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost));
  CK(ctx, cudaMemcpy(&rows, b.row_base + b.ns, sizeof(int64_t), cudaMemcpyDeviceToHost));
  out->n_vertices = b.NV;
  out->n_cells = b.NC;
  out->n_active_dofs = 0;
  out->n_flipped = 0;
  for (int s = 0; s < b.ns; ++s) {
    out->n_active_dofs += 2 * (int64_t)na[s];
    out->n_flipped += fl[s];
  }
  out->nnz = 4 * b.n_adj;
  out->block_rows = rows;
  out->sell_blocks = b.n_blocks;
  out->max_row_blocks = b.max_row_blocks;
  return FEA_OK;
}

int fea_batch_get_refine_rounds(fea_batch* hb, int32_t* rounds) {
  if (!hb || !rounds) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.solved) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_refine_rounds before fea_batch_solve");
  CK(ctx, cudaSetDevice(ctx->c.device));
  CK(ctx, cudaMemcpyAsync(rounds, b.sc.rounds, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, ctx->c.stream));
  CK(ctx, cudaStreamSynchronize(ctx->c.stream));
  return FEA_OK;
}

int fea_batch_get_solve_stats(fea_batch* hb, fea_solve_stats* out) {
  if (!hb || !out) return FEA_BAD_ARG;
  *out = hb->b.stats;
  return FEA_OK;
}

int fea_batch_get_timed_launches(fea_batch* hb, int32_t cap, float* spmv_ms, float* update_ms, int32_t* n_out) {
  if (!hb || !n_out || cap < 0) return FEA_BAD_ARG;
  const Batch& b = hb->b;
  const int n = (int)b.t_spmv.size();
  *n_out = n;
  for (int i = 0; i < n && i < cap; ++i) {
    if (spmv_ms) spmv_ms[i] = b.t_spmv[i];
    if (update_ms) update_ms[i] = b.t_update[i];
  }
  return FEA_OK;
}

int fea_batch_get_conn(fea_batch* hb, int32_t* conn, int32_t* n_flipped) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (conn && b.NC) {
    int32_t* tmp = nullptr;
    CK(ctx, cudaMallocAsync((void**)&tmp, sizeof(int32_t) * b.NC * b.npc, st));
    k_localize_conn<<<(unsigned)((b.NC + 255) / 256), 256, 0, st>>>(b.NC, b.npc, b.d_cell_off, b.d_vtx_off, b.ns, b.conn, tmp);
    CK(ctx, cudaMemcpyAsync(conn, tmp, sizeof(int32_t) * b.NC * b.npc, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    cudaFreeAsync(tmp, st);
  }
  if (n_flipped) {
    CK(ctx, cudaMemcpyAsync(n_flipped, b.flips, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
  }
  return FEA_OK;
}

int fea_batch_get_element_stiffness(fea_batch* hb, double* ke) {
  if (!hb || !ke) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "element stiffness requested before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  const int N = 2 * b.npc;
  CK(ctx, cudaMemcpyAsync(ke, b.ke, sizeof(double) * b.NC * N * N, cudaMemcpyDeviceToHost, ctx->c.stream));
  CK(ctx, cudaStreamSynchronize(ctx->c.stream));
  return FEA_OK;
}

int fea_batch_get_csr(fea_batch* hb, int32_t s, int32_t* indptr, int32_t* indices, double* data) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_csr before fea_batch_assemble");
  if (s < 0 || s >= b.ns) return api_fail(ctx, FEA_BAD_ARG, "sample index out of range");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  int32_t na = 0, a0 = 0, a1 = 0;
  CK(ctx, cudaMemcpyAsync(&na, b.n_active + s, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(&a0, b.adj_ptr + b.vtx_off[s], sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(&a1, b.adj_ptr + b.vtx_off[s + 1], sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  const int64_t n = 2 * (int64_t)na, nnz = 4 * (int64_t)(a1 - a0);
  int32_t *d_ip = nullptr, *d_ix = nullptr;
  double* d_dt = nullptr;
  if (indptr) {
    CK(ctx, cudaMallocAsync((void**)&d_ip, sizeof(int32_t) * (n + 1), st));
    CK(ctx, cudaMemsetAsync(d_ip, 0, sizeof(int32_t) * (n + 1), st));
  }
  if (indices) CK(ctx, cudaMallocAsync((void**)&d_ix, sizeof(int32_t) * std::max<int64_t>(1, nnz), st));
  if (data) CK(ctx, cudaMallocAsync((void**)&d_dt, sizeof(double) * std::max<int64_t>(1, nnz), st));
  CK(ctx, launch_csr_export(b, s, d_ip, d_ix, d_dt));
  if (indptr) CK(ctx, cudaMemcpyAsync(indptr, d_ip, sizeof(int32_t) * (n + 1), cudaMemcpyDeviceToHost, st));
  if (indices) CK(ctx, cudaMemcpyAsync(indices, d_ix, sizeof(int32_t) * nnz, cudaMemcpyDeviceToHost, st));
  if (data) CK(ctx, cudaMemcpyAsync(data, d_dt, sizeof(double) * nnz, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  if (d_ip) cudaFreeAsync(d_ip, st);
  if (d_ix) cudaFreeAsync(d_ix, st);
  if (d_dt) cudaFreeAsync(d_dt, st);
  return FEA_OK;
}

int fea_batch_spmv(fea_batch* hb, int32_t s, const double* x, double* y) {
  if (!hb || !x || !y) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_spmv before fea_batch_assemble");
  if (s < 0 || s >= b.ns) return api_fail(ctx, FEA_BAD_ARG, "sample index out of range");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  int32_t na = 0;
  CK(ctx, cudaMemcpyAsync(&na, b.n_active + s, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  const int64_t n = 2 * (int64_t)na;
  double *dx = nullptr, *dy = nullptr;
  CK(ctx, cudaMallocAsync((void**)&dx, sizeof(double) * std::max<int64_t>(1, n), st));
  CK(ctx, cudaMallocAsync((void**)&dy, sizeof(double) * std::max<int64_t>(1, n), st));
  CK(ctx, cudaMemcpyAsync(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  CK(ctx, launch_plain_spmv(b, s, dx, dy));
  CK(ctx, cudaMemcpyAsync(y, dy, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  cudaFreeAsync(dx, st);
  cudaFreeAsync(dy, st);
  b.solved = false;  // solver vectors were overwritten
  return FEA_OK;
}

int fea_rasterize_fields(fea_ctx* ctx, const double* xy, int64_t n_v, const int32_t* conn, int64_t n_cell,
                         int32_t nodes_per_cell, const double* fields, int32_t n_fields, int32_t cell_fields,
                         const double* clim, const double* affine, int32_t size, uint8_t* images) {
  if (!ctx) return FEA_BAD_ARG;
  if (!xy || !conn || !fields || !clim || !affine || !images) return api_fail(ctx, FEA_BAD_ARG, "null array");
  if (nodes_per_cell != 3 && nodes_per_cell != 4) return api_fail(ctx, FEA_BAD_ARG, "nodes_per_cell must be 3 or 4");
  if (n_v < 1 || n_cell < 0 || n_fields < 1 || size < 1 || size > 8192 || n_v >= (1LL << 30))
    return api_fail(ctx, FEA_BAD_ARG, "size out of range");
  for (int64_t i = 0; i < n_cell * nodes_per_cell; ++i)
    if (conn[i] < 0 || conn[i] >= n_v) return api_fail(ctx, FEA_MESH_ERROR, "connectivity index out of range");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  const int64_t per = (int64_t)size * size;
  const size_t b_xy = sizeof(double) * 2 * n_v, b_cn = sizeof(int32_t) * n_cell * nodes_per_cell,
               b_f = sizeof(double) * n_fields * (cell_fields ? std::max<int64_t>(n_cell, 1) : n_v), b_img = (size_t)n_fields * per;
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t o_xy = 0, o_cn = o_xy + up(b_xy), o_f = o_cn + up(b_cn), o_cl = o_f + up(b_f),
               o_af = o_cl + up(sizeof(double) * 2 * n_fields), o_co = o_af + 256, o_ow = o_co + 256,
               o_im = o_ow + up(sizeof(int32_t) * per), total = o_im + up(b_img);
  char* d = nullptr;
  CK(ctx, cudaMallocAsync((void**)&d, total, st));
  const int64_t h_off[2] = {0, n_cell};
  cudaError_t e = cudaMemcpyAsync(d + o_xy, xy, b_xy, cudaMemcpyHostToDevice, st);
#define A(call) if (e == cudaSuccess) e = (call)
  if (b_cn) A(cudaMemcpyAsync(d + o_cn, conn, b_cn, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(d + o_f, fields, b_f, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(d + o_cl, clim, sizeof(double) * 2 * n_fields, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(d + o_af, affine, sizeof(double) * 4, cudaMemcpyHostToDevice, st));
  A(cudaMemcpyAsync(d + o_co, h_off, sizeof(h_off), cudaMemcpyHostToDevice, st));
  A(launch_raster_fields(st, nodes_per_cell, n_v, n_cell, (const int32_t*)(d + o_cn), (const double*)(d + o_xy),
                         (const double*)(d + o_af), (const int64_t*)(d + o_co), size, (int32_t*)(d + o_ow),
                         (const double*)(d + o_f), n_fields, cell_fields ? 1 : 0, (const double*)(d + o_cl), (uint8_t*)(d + o_im)));
  A(cudaMemcpyAsync(images, d + o_im, b_img, cudaMemcpyDeviceToHost, st));
  A(cudaStreamSynchronize(st));
#undef A
  cudaFreeAsync(d, st);
  ctx->c.launches += 3;
  if (e != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "fea_rasterize_fields", e);
  return FEA_OK;
}

int fea_solve_batch(fea_ctx* ctx, const fea_batch_desc* desc, double rtol, int32_t max_iter, int32_t image_size,
                    const double* affine, double value_scale, double* u, double* ranges, int32_t* iters,
                    double* relres, int32_t* status, uint8_t* images, fea_solve_stats* stats) {
  fea_batch* hb = nullptr;
  int rc = fea_batch_create(ctx, desc, &hb);
  if (rc != FEA_OK) return rc;
  rc = fea_batch_assemble(hb);
  if (rc == FEA_OK) rc = fea_batch_solve(hb, rtol, max_iter);
  if (rc == FEA_OK && image_size > 0 && affine) rc = fea_batch_rasterize(hb, image_size, affine, value_scale);
  if (rc == FEA_OK) rc = fea_batch_download(hb, u, ranges, iters, relres, status);
  if (rc == FEA_OK && image_size > 0 && affine && images) rc = fea_batch_download_images(hb, images);
  if (rc == FEA_OK && stats) *stats = hb->b.stats;
  fea_batch_destroy(hb);
  return rc;
}

int fea_batch_set_refinement(fea_batch* hb, int32_t levels) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_set_refinement after fea_batch_assemble");
  if (b.mg) return api_fail(ctx, FEA_BAD_STATE, "the batch already declared its refinement");
  if (b.ns != 1 || b.npc != 3) return api_fail(ctx, FEA_BAD_ARG, "a refinement hierarchy needs one sample of triangles");
  if (levels < 1 || levels > 8) return api_fail(ctx, FEA_BAD_ARG, "levels must be 1..8");
  if (!b.conn_given) return api_fail(ctx, FEA_BAD_ARG, "a refinement hierarchy is declared on a batch made by fea_batch_create, before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  return mg_set_refinement(ctx, b, levels);
}

int fea_batch_get_mg_levels(fea_batch* hb, int32_t cap, fea_mg_level* out, int32_t* n_out) {
  if (!hb || !n_out || cap < 0 || (cap > 0 && !out)) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.mg) return api_fail(ctx, FEA_BAD_STATE, "the batch declared no refinement");
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_mg_levels before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  const int n = b.mg->levels + 1;
  *n_out = n;
  for (int l = 0; l < n && l < cap; ++l) {
    const MgLevel& L = b.mg->lev[l];
    int32_t na = 0;
    CK(ctx, cudaMemcpyAsync(&na, L.b->n_active, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->c.stream));
    CK(ctx, cudaStreamSynchronize(ctx->c.stream));
    out[l].n_vertices = L.nv;
    out[l].n_cells = L.nc;
    out[l].n_active_dofs = 2 * (int64_t)na;
    out[l].nnz = 4 * L.b->n_adj;
    out[l].lambda_max = L.lmax;
    out[l].vcycle_ms = L.ms;
  }
  return FEA_OK;
}

int fea_batch_get_level_csr(fea_batch* hb, int32_t level, int32_t* indptr, int32_t* indices, double* data) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.mg) return api_fail(ctx, FEA_BAD_STATE, "the batch declared no refinement");
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_level_csr before fea_batch_assemble");
  if (level < 0 || level > b.mg->levels) return api_fail(ctx, FEA_BAD_ARG, "level out of range");
  fea_batch* lb = b.mg->lev[level].hb ? b.mg->lev[level].hb : hb;
  return fea_batch_get_csr(lb, 0, indptr, indices, data);
}

int fea_batch_mg_apply(fea_batch* hb, const double* r, double* z) {
  if (!hb || !r || !z) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.mg) return api_fail(ctx, FEA_BAD_STATE, "the batch declared no refinement");
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_mg_apply before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  int32_t na = 0;
  CK(ctx, cudaMemcpyAsync(&na, b.n_active, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  const int64_t n = 2 * (int64_t)na;
  double* d = nullptr;
  CK(ctx, cudaMallocAsync((void**)&d, sizeof(double) * 2 * std::max<int64_t>(1, n), st));
  cudaError_t e = cudaMemcpyAsync(d, r, sizeof(double) * n, cudaMemcpyHostToDevice, st);
  int rc = e == cudaSuccess ? mg_apply(ctx, b, d, d + std::max<int64_t>(1, n)) : FEA_CUDA_ERROR;
  if (rc == FEA_OK) e = cudaMemcpyAsync(z, d + std::max<int64_t>(1, n), sizeof(double) * n, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFreeAsync(d, st);
  if (rc != FEA_OK) return rc;
  if (e != cudaSuccess) return api_fail(ctx, FEA_CUDA_ERROR, "fea_batch_mg_apply", e);
  return FEA_OK;
}

}  // extern "C"
