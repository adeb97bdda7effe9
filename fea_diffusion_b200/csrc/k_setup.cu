// Batch set-up kernels: device-wide scans, connectivity globalisation + orientation fix
// (SURVEY A-2), Dirichlet equation map (A-9; reference problem.set_bcs,
// datagen/fea_analysis.py:422), vertex->cell incidence and the sorted vertex adjacency that
// *is* sfepy's matrix graph at 2x2-block granularity (A-11).
#include <algorithm>

#include "fea_internal.cuh"

namespace fea {

// ===========================================================================
// device-wide exclusive scan: 3 passes, 4096 items per block, deterministic
// ===========================================================================
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;
constexpr int kScanTile = kScanThreads * kScanItems;

template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* total, T* smem /*>=33*/) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  T inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    T t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) smem[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    const int nw = blockDim.x >> 5;
    T w = lane < nw ? smem[lane] : T(0);
    T winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      T t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    if (lane < nw) smem[lane] = winc - w;
    if (lane == 31) smem[32] = winc;
  }
  __syncthreads();
  T res = smem[wid] + inc - v;
  *total = smem[32];
  __syncthreads();
  return res;
}

template <typename TO>
__global__ void scan_tile_sums(const int32_t* __restrict__ in, int64_t n, TO mul, TO* __restrict__ sums) {
  __shared__ TO sm[33];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  TO s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) s += (TO)in[base + i] * mul;
  TO tot;
  block_exclusive_scan<TO>(s, &tot, sm);
  if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

template <typename TO>
__global__ void scan_of_sums(TO* sums, int nb) {  // one block; sums[nb] = grand total
  __shared__ TO sm[33];
  TO carry = 0;
  for (int base = 0; base < nb; base += blockDim.x) {
    int i = base + threadIdx.x;
    TO v = i < nb ? sums[i] : TO(0);
    TO tot;
    TO ex = block_exclusive_scan<TO>(v, &tot, sm);
    if (i < nb) sums[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) sums[nb] = carry;
}

template <typename TO>
__global__ void scan_tile_final(const int32_t* __restrict__ in, TO* __restrict__ out, int64_t n, TO mul,
                                const TO* __restrict__ sums, int nb) {
  __shared__ TO sm[33];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  TO v[kScanItems];
  TO s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < n) ? (TO)in[base + i] * mul : TO(0);
    s += v[i];
  }
  TO tot;
  TO ex = block_exclusive_scan<TO>(s, &tot, sm) + sums[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = ex;
    ex += v[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = sums[nb];
}

template <typename TO>
static cudaError_t scan_impl(const int32_t* in, TO* out, int64_t n, TO mul, TO* tmp, cudaStream_t st) {
  int nb = (int)((n + kScanTile - 1) / kScanTile);
  if (nb == 0) nb = 1;
  scan_tile_sums<TO><<<nb, kScanThreads, 0, st>>>(in, n, mul, tmp);
  scan_of_sums<TO><<<1, 1024, 0, st>>>(tmp, nb);
  scan_tile_final<TO><<<nb, kScanThreads, 0, st>>>(in, out, n, mul, tmp, nb);
  return cudaGetLastError();
}

cudaError_t exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* tmp, cudaStream_t st) {
  return scan_impl<int32_t>(in, out, n, 1, tmp, st);
}
cudaError_t exclusive_scan_i32_to_i64(const int32_t* in, int64_t* out, int64_t n, int64_t mul,
                                      int64_t* tmp, cudaStream_t st) {
  return scan_impl<int64_t>(in, out, n, mul, (int64_t*)tmp, st);
}

// ===========================================================================
// set-up
// ===========================================================================
__global__ void k_vertex_sample(const int64_t* __restrict__ vtx_off, int ns, int64_t NV,
                                int32_t* __restrict__ vsample) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < NV) vsample[v] = seg_of(vtx_off, ns, v);
}

// conn_local -> global ids with orientation fix (A-2); region -> global D index.
template <int NPC>
__global__ void k_cells(const int64_t* __restrict__ cell_off, const int64_t* __restrict__ vtx_off,
                        const int32_t* __restrict__ reg_off, int ns, int64_t NC,
                        const double* __restrict__ xy, const int32_t* __restrict__ conn_local,
                        const int8_t* __restrict__ creg_local, int32_t* __restrict__ conn,
                        int32_t* __restrict__ cell_dreg, int32_t* __restrict__ flips,
                        int32_t* __restrict__ err_flag) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  const int s = seg_of(cell_off, ns, c);
  const int64_t voff = vtx_off[s];
  const int64_t nv = vtx_off[s + 1] - voff;
  int32_t g[NPC];
  double x[NPC], y[NPC];
  bool bad = false;
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
    int32_t l = conn_local[c * NPC + a];
    if (l < 0 || l >= nv) { bad = true; l = 0; }
    g[a] = (int32_t)(voff + l);
    x[a] = xy[2 * (int64_t)g[a]];
    y[a] = xy[2 * (int64_t)g[a] + 1];
  }
  if (bad) atomicOr(err_flag, 2);
  double a2 = 0.0;  // shoelace, same operation order as the oracle (no FMA)
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
    const int n = (a + 1) % NPC;
    a2 = __dadd_rn(a2, __dsub_rn(__dmul_rn(x[a], y[n]), __dmul_rn(x[n], y[a])));
  }
  if (a2 < 0.0) {
    if (NPC == 3) { int32_t t = g[1]; g[1] = g[2]; g[2] = t; }
    else { int32_t t = g[1]; g[1] = g[3]; g[3] = t; }
    atomicAdd(&flips[s], 1);
  }
#pragma unroll
  for (int a = 0; a < NPC; ++a) conn[c * NPC + a] = g[a];
  const int r = creg_local[c];
  const int nreg = reg_off[s + 1] - reg_off[s];
  if (r >= nreg) atomicOr(err_flag, 2);
  cell_dreg[c] = (r < 0 || r >= nreg) ? -1 : reg_off[s] + r;
}

// One CTA per sample: rank of every non-fixed vertex in ascending order (A-9).
__global__ void k_vrank(const int64_t* __restrict__ vtx_off, const uint8_t* __restrict__ fixed,
                        int32_t* __restrict__ vrank, int32_t* __restrict__ n_active) {
  __shared__ int sm[33];
  const int s = blockIdx.x;
  const int64_t v0 = vtx_off[s], v1 = vtx_off[s + 1];
  int carry = 0;
  for (int64_t base = v0; base < v1; base += blockDim.x * 4) {
    const int64_t i0 = base + (int64_t)threadIdx.x * 4;
    int a[4], cnt = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      a[k] = (i0 + k < v1) ? (fixed[i0 + k] ? 0 : 1) : 0;
      cnt += a[k];
    }
    int tot;
    int ex = block_exclusive_scan<int>(cnt, &tot, sm) + carry;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (i0 + k < v1) vrank[i0 + k] = a[k] ? ex : -1;
      ex += a[k];
    }
    carry += tot;
  }
  if (threadIdx.x == 0) n_active[s] = carry;
}

// Serial over samples (ns is small): padded block-row bases and CTA ranges.
__global__ void k_row_bases(const int32_t* __restrict__ n_active, int ns, int64_t* __restrict__ row_base,
                            int32_t* __restrict__ cta_first, int32_t* __restrict__ cta_count) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  int64_t r = 0;
  for (int s = 0; s < ns; ++s) {
    row_base[s] = r;
    const int64_t pad = ((int64_t)n_active[s] + kCtaRows - 1) / kCtaRows * kCtaRows;
    cta_first[s] = (int32_t)(r / kCtaRows);
    cta_count[s] = (int32_t)(pad / kCtaRows);
    r += pad;
  }
  row_base[ns] = r;
}

__global__ void k_cta_sys(const int64_t* __restrict__ row_base, int ns, int ncta, int32_t* __restrict__ sys_of_cta) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ncta) return;
  const int64_t row = (int64_t)i * kCtaRows;
  sys_of_cta[i] = row < row_base[ns] ? seg_of(row_base, ns, row) : -1;
}

__global__ void k_row_maps(const int32_t* __restrict__ vsample, const int32_t* __restrict__ vrank,
                           const int64_t* __restrict__ row_base, int64_t NV,
                           int32_t* __restrict__ row_of_vertex, int32_t* __restrict__ vertex_of_row) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV) return;
  const int rk = vrank[v];
  if (rk < 0) { row_of_vertex[v] = -1; return; }
  const int64_t row = row_base[vsample[v]] + rk;
  row_of_vertex[v] = (int32_t)row;
  vertex_of_row[row] = (int32_t)v;
}

// ---------------------------------------------------------------------------
// Solver row order.  The matrix graph exported to the caller follows sfepy's numbering (ascending
// DOF, A-9), but the ORDER OF THE ROWS inside the solver is free, and it decides how local the
// SpMV gathers are: with a contiguous row range per CTA (cluster path) or per 32-row slice, rows
// that are neighbours in the mesh should be neighbours in memory.  Mesh generators do not promise
// that (gmsh numbers boundary nodes first and interior nodes in insertion order; a random
// numbering makes the on-chip solver 2.4x slower), so every sample's active vertices are sorted by
// a spatial key computed from their coordinates: one CTA per sample, bitonic sort in shared memory.
//   mode 1: Morton (Z-order) code of the position in the sample's bounding box
//   mode 2: horizontal strips one mesh-size high, x inside a strip (a lattice-like row-major order)
//   mode 3: (default) keep the input numbering when it is already local -- at most 20 % of the
//           cells span more than 4 sqrt(n_v) vertex indices, as for row-by-row lattice numberings,
//           which beat any generic spatial order (consecutive rows have consecutive neighbours:
//           conflict-free gathers) -- and sort by strips otherwise
// prank[v] = rank of vertex v among the active vertices of its sample in that order (-1 if fixed).
// Samples with more than 16384 vertices keep the input order (prank = vrank).
// Measured on the bench batch (solve time): lattice input 48.2 ms in input order, 49.1 ms strips,
// 50.7 ms Morton; the same meshes randomly renumbered: 108 ms input order, 50.2 / 50.1 ms sorted.
// ---------------------------------------------------------------------------
constexpr int kSortThreads = 1024;
constexpr int kSortMax = 16384;

__device__ __forceinline__ uint32_t spread16(uint32_t v) {
  v &= 0xffffu;
  v = (v | (v << 8)) & 0x00ff00ffu;
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}

__global__ void __launch_bounds__(kSortThreads) k_spatial_rank(const int64_t* __restrict__ vtx_off,
                                                               const int64_t* __restrict__ cell_off,
                                                               const int32_t* __restrict__ conn, int npc,
                                                               const double* __restrict__ xy,
                                                               const int32_t* __restrict__ vrank, int mode,
                                                               int32_t* __restrict__ prank) {
  extern __shared__ unsigned long long keys[];
  __shared__ double red[4][kSortThreads / 32];
  __shared__ double box[4];
  __shared__ int far_cells;
  const int s = blockIdx.x;
  const int64_t v0 = vtx_off[s];
  const int nv = (int)(vtx_off[s + 1] - v0);
  bool keep = nv > kSortMax || nv == 0;
  if (!keep && mode == 3) {   // is the input numbering already local?
    if (threadIdx.x == 0) far_cells = 0;
    __syncthreads();
    const int64_t c0 = cell_off[s], c1 = cell_off[s + 1];
    const int limit = 4 * (int)sqrt((double)nv) + 16;
    int cnt = 0;
    for (int64_t c = c0 + threadIdx.x; c < c1; c += blockDim.x) {
      int lo = 0x7fffffff, hi = -1;
      for (int a = 0; a < npc; ++a) {
        const int v = conn[c * npc + a];
        lo = min(lo, v);
        hi = max(hi, v);
      }
      cnt += (hi - lo) > limit;
    }
    atomicAdd(&far_cells, cnt);
    __syncthreads();
    keep = 5 * (int64_t)far_cells <= (c1 - c0);
    mode = 2;
  }
  if (keep) {
    for (int i = threadIdx.x; i < nv; i += blockDim.x) prank[v0 + i] = vrank[v0 + i];
    return;
  }
  // bounding box of the sample
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double mnx = inf, mxx = -inf, mny = inf, mxy = -inf;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const double x = xy[2 * (v0 + i)], y = xy[2 * (v0 + i) + 1];
    mnx = fmin(mnx, x); mxx = fmax(mxx, x); mny = fmin(mny, y); mxy = fmax(mxy, y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fmin(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
    mxx = fmax(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    mny = fmin(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxy = fmax(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = mnx; red[1][threadIdx.x >> 5] = mxx;
    red[2][threadIdx.x >> 5] = mny; red[3][threadIdx.x >> 5] = mxy;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kSortThreads / 32; ++w) {
      red[0][0] = fmin(red[0][0], red[0][w]); red[1][0] = fmax(red[1][0], red[1][w]);
      red[2][0] = fmin(red[2][0], red[2][w]); red[3][0] = fmax(red[3][0], red[3][w]);
    }
    box[0] = red[0][0]; box[1] = red[1][0]; box[2] = red[2][0]; box[3] = red[3][0];
  }
  __syncthreads();
  const double x0 = box[0], y0 = box[2];
  const double w = fmax(box[1] - x0, 1e-300), hgt = fmax(box[3] - y0, 1e-300);
  const double ext = fmax(w, hgt);
  const double hmesh = sqrt(w * hgt / (double)nv);       // mesh size estimate (mode 2)
  int n2 = 1;
  while (n2 < nv) n2 <<= 1;
  for (int i = threadIdx.x; i < n2; i += blockDim.x) {
    unsigned long long k = ~0ull;
    if (i < nv && vrank[v0 + i] >= 0) {
      const double x = xy[2 * (v0 + i)] - x0, y = xy[2 * (v0 + i) + 1] - y0;
      uint32_t hi;
      if (mode == 1) {
        const uint32_t xq = (uint32_t)fmin(65535.0, x / ext * 65535.0), yq = (uint32_t)fmin(65535.0, y / ext * 65535.0);
        hi = spread16(xq) | (spread16(yq) << 1);
      } else {
        const uint32_t strip = (uint32_t)fmin(32767.0, y / hmesh);
        const uint32_t xq = (uint32_t)fmin(65535.0, x / w * 65535.0);
        hi = (strip << 16) | xq;
      }
      if (hi == 0xffffffffu) hi = 0xfffffffeu;            // the all-ones key marks fixed vertices
      k = ((unsigned long long)hi << 32) | (unsigned)i;
    }
    keys[i] = k;
  }
  __syncthreads();
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (n2 >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));        // index with bit `stride` cleared
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const unsigned long long a = keys[lo], b = keys[hi];
        if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const unsigned long long k = keys[i];
    if ((uint32_t)(k >> 32) != 0xffffffffu) prank[v0 + (int)(k & 0xffffffffu)] = i;
  }
  for (int i = threadIdx.x; i < nv; i += blockDim.x)
    if (vrank[v0 + i] < 0) prank[v0 + i] = -1;
}

// ---------------------------------------------------------------------------
// Queues of the on-chip solver classes (k_pcg_cluster): inside a class the systems are ordered
// longest-job-first by an estimate of the work, rows x iterations.  The iteration count of
// Jacobi-PCG on these plates falls with the number of constrained vertices (measured on 800 bench
// samples: iters ~ 2560 - 344 ln(n_fixed), R^2 0.44), and starting the long solves first shortens
// the tail of a batch by 15-20 %.  The order only decides WHEN a system is solved, never its bits.
// One CTA: 64-bit keys (class | inverted work | system) sorted by a bitonic network in global
// memory (L2 resident; a batch has at most 2^20 systems).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_cluster_order(int ns, int n2, const int64_t* __restrict__ vtx_off,
                                                        const int32_t* __restrict__ n_active, int rows_per_cta,
                                                        int min_cl, int max_cl, unsigned long long* __restrict__ keys,
                                                        int n_out, int32_t* __restrict__ cl_order) {
  for (int s = threadIdx.x; s < n2; s += blockDim.x) {
    unsigned long long k = ~0ull;
    if (s < ns) {
      const int64_t nv = vtx_off[s + 1] - vtx_off[s];
      const int64_t pad = (nv + kCtaRows - 1) / kCtaRows * kCtaRows;
      int64_t cl = pad > 0 ? (pad + rows_per_cta - 1) / rows_per_cta : 0;
      if (cl > 0 && cl < min_cl) cl = min_cl;
      if (cl >= 1 && cl <= max_cl) {
        const int na = n_active[s];
        const int64_t nfix = nv - na;
        const double it = fmax(100.0, 2560.0 - 344.0 * log((double)(nfix > 1 ? nfix : 1)));
        const double work = fmin(it * (double)na, 268435455.0);
        k = ((unsigned long long)cl << 60) | ((unsigned long long)(268435455u - (unsigned)work) << 32) | (unsigned)s;
      }
    }
    keys[s] = k;
  }
  __syncthreads();
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < (n2 >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const unsigned long long a = keys[lo], b = keys[hi];
        if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n_out; i += blockDim.x) cl_order[i] = (int32_t)(keys[i] & 0xffffffffu);
}

cudaError_t launch_cluster_order(Batch& b) {
  cudaStream_t st = b.ctx->stream;
  const int n_out = b.cl_off[8] + b.cl_cnt[8];
  if (n_out == 0) return cudaSuccess;
  int n2 = 2;
  while (n2 < b.ns) n2 <<= 1;
  Scratch scratch(st);
  unsigned long long* keys = nullptr;
  cudaError_t e = scratch.alloc(&keys, n2);
  if (e != cudaSuccess) return e;
  k_cluster_order<<<1, 1024, 0, st>>>(b.ns, n2, b.d_vtx_off, b.n_active, pcg_cluster_rows_per_cta(), b.ctx->cluster_min, 8,
                                      keys, n_out, b.cl_order);
  return cudaGetLastError();
}

cudaError_t launch_setup(Batch& b, const int8_t* d_creg_local, const int32_t* d_conn_local) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  if (b.NV) k_vertex_sample<<<(unsigned)((b.NV + T - 1) / T), T, 0, st>>>(b.d_vtx_off, b.ns, b.NV, b.vsample);
  if (b.NC) {
    unsigned g = (unsigned)((b.NC + T - 1) / T);
    if (b.npc == 3)
      k_cells<3><<<g, T, 0, st>>>(b.d_cell_off, b.d_vtx_off, b.d_reg_off, b.ns, b.NC, b.xy, d_conn_local,
                                  d_creg_local, b.conn, b.cell_dreg, b.flips, b.err_flag);
    else
      k_cells<4><<<g, T, 0, st>>>(b.d_cell_off, b.d_vtx_off, b.d_reg_off, b.ns, b.NC, b.xy, d_conn_local,
                                  d_creg_local, b.conn, b.cell_dreg, b.flips, b.err_flag);
  }
  k_vrank<<<b.ns, 256, 0, st>>>(b.d_vtx_off, b.fixed, b.vrank, b.n_active);
  k_row_bases<<<1, 32, 0, st>>>(b.n_active, b.ns, b.row_base, b.cta_first, b.cta_count);
  const int ncta = (int)(b.NBR / kCtaRows);
  if (ncta) k_cta_sys<<<(ncta + T - 1) / T, T, 0, st>>>(b.row_base, b.ns, ncta, b.sys_of_cta);
  const int32_t* rank_for_rows = b.vrank;
  if (b.ctx->row_order != 0 && b.prank) {
    // (function attributes are per device: set it on every call, it costs microseconds)
    cudaFuncSetAttribute(k_spatial_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, kSortMax * 8);
    int64_t nvmax = 0;
    for (int s = 0; s < b.ns; ++s) nvmax = std::max<int64_t>(nvmax, b.vtx_off[s + 1] - b.vtx_off[s]);
    int n2 = 1;
    while (n2 < nvmax && n2 < kSortMax) n2 <<= 1;
    k_spatial_rank<<<b.ns, kSortThreads, (size_t)n2 * 8, st>>>(b.d_vtx_off, b.d_cell_off, b.conn, b.npc, b.xy, b.vrank,
                                                               b.ctx->row_order, b.prank);
    rank_for_rows = b.prank;
  }
  if (b.NV)
    k_row_maps<<<(unsigned)((b.NV + T - 1) / T), T, 0, st>>>(b.vsample, rank_for_rows, b.row_base, b.NV,
                                                            b.row_of_vertex, b.vertex_of_row);
  return cudaGetLastError();
}

// ===========================================================================
// topology: incidence and adjacency
// ===========================================================================
template <int NPC>
__global__ void k_inc_count(const int32_t* __restrict__ conn, const int32_t* __restrict__ cell_dreg,
                            int64_t NC, int32_t* __restrict__ cnt) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC || cell_dreg[c] < 0) return;
#pragma unroll
  for (int a = 0; a < NPC; ++a) atomicAdd(&cnt[conn[c * NPC + a]], 1);
}

template <int NPC>
__global__ void k_inc_fill(const int32_t* __restrict__ conn, const int32_t* __restrict__ cell_dreg,
                           int64_t NC, const int32_t* __restrict__ inc_ptr, int32_t* __restrict__ cursor,
                           int32_t* __restrict__ inc) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC || cell_dreg[c] < 0) return;
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
    const int v = conn[c * NPC + a];
    const int pos = atomicAdd(&cursor[v], 1);
    inc[inc_ptr[v] + pos] = (int32_t)(c * 4 + a);
  }
}

// ascending order makes every later per-vertex summation order deterministic
__global__ void k_inc_sort(const int32_t* __restrict__ inc_ptr, int64_t NV, int32_t* __restrict__ inc) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV) return;
  const int b = inc_ptr[v], e = inc_ptr[v + 1];
  for (int i = b + 1; i < e; ++i) {
    const int key = inc[i];
    int j = i - 1;
    while (j >= b && inc[j] > key) { inc[j + 1] = inc[j]; --j; }
    inc[j + 1] = key;
  }
}

// Sorted unique list of ACTIVE vertices sharing a stiffness cell with v (v included).
template <int NPC>
__device__ __forceinline__ int gather_adjacency(int64_t v, const int32_t* __restrict__ inc_ptr,
                                                const int32_t* __restrict__ inc,
                                                const int32_t* __restrict__ conn,
                                                const int32_t* __restrict__ vrank, int* lst) {
  int n = 0;
  const int b = inc_ptr[v], e = inc_ptr[v + 1];
  for (int i = b; i < e; ++i) {
    const int64_t c = inc[i] >> 2;
#pragma unroll
    for (int a = 0; a < NPC; ++a) {
      const int w = conn[c * NPC + a];
      if (vrank[w] < 0) continue;
      int k = 0;
      while (k < n && lst[k] < w) ++k;
      if (k < n && lst[k] == w) continue;
      if (n == kMaxAdj) return -1;
      for (int m = n; m > k; --m) lst[m] = lst[m - 1];
      lst[k] = w;
      ++n;
    }
  }
  return n;
}

template <int NPC>
__global__ void k_adj_count(int64_t NV, const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                            const int32_t* __restrict__ conn, const int32_t* __restrict__ vrank,
                            int32_t* __restrict__ cnt, int32_t* __restrict__ max_len,
                            int32_t* __restrict__ err_flag) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int n = 0;
  if (v < NV && vrank[v] >= 0) {
    int lst[kMaxAdj];
    n = gather_adjacency<NPC>(v, inc_ptr, inc, conn, vrank, lst);
    if (n < 0) { atomicOr(err_flag, 1); n = 0; }
  }
  if (v < NV) cnt[v] = n;
  const int m = warp_max_i(n);
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(max_len, m);
}

template <int NPC>
__global__ void k_adj_fill(int64_t NV, const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                           const int32_t* __restrict__ conn, const int32_t* __restrict__ vrank,
                           const int32_t* __restrict__ adj_ptr, int32_t* __restrict__ adj) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV || vrank[v] < 0) return;
  int lst[kMaxAdj];
  const int n = gather_adjacency<NPC>(v, inc_ptr, inc, conn, vrank, lst);
  const int o = adj_ptr[v];
  for (int k = 0; k < n; ++k) adj[o + k] = lst[k];
}

// Phase 1: incidence (count, scan, fill, sort) and adjacency counts + scan.
// Uses b.adj_ptr as the count buffer before scanning in place is avoided via a temp.
cudaError_t launch_topology_counts(Batch& b) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const unsigned gv = (unsigned)((b.NV + T - 1) / T), gc = (unsigned)((b.NC + T - 1) / T);
  // scratch: cnt [NV+1], tmp for scans
  Scratch scratch(st);
  int32_t* cnt = nullptr;
  int32_t* tmp = nullptr;
  cudaError_t e;
  if ((e = scratch.alloc(&cnt, b.NV + 1)) != cudaSuccess) return e;
  if ((e = scratch.alloc(&tmp, b.NV / kScanTile + 4)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (b.NV + 1), st)) != cudaSuccess) return e;
  if (b.NC) {
    if (b.npc == 3) k_inc_count<3><<<gc, T, 0, st>>>(b.conn, b.cell_dreg, b.NC, cnt);
    else k_inc_count<4><<<gc, T, 0, st>>>(b.conn, b.cell_dreg, b.NC, cnt);
  }
  if ((e = exclusive_scan_i32(cnt, b.inc_ptr, b.NV, tmp, st)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (b.NV + 1), st)) != cudaSuccess) return e;
  if (b.NC) {
    if (b.npc == 3) k_inc_fill<3><<<gc, T, 0, st>>>(b.conn, b.cell_dreg, b.NC, b.inc_ptr, cnt, b.inc);
    else k_inc_fill<4><<<gc, T, 0, st>>>(b.conn, b.cell_dreg, b.NC, b.inc_ptr, cnt, b.inc);
  }
  if (b.NV) {
    k_inc_sort<<<gv, T, 0, st>>>(b.inc_ptr, b.NV, b.inc);
    int32_t* max_len = b.err_flag + 1;
    if (b.npc == 3)
      k_adj_count<3><<<gv, T, 0, st>>>(b.NV, b.inc_ptr, b.inc, b.conn, b.vrank, cnt, max_len, b.err_flag);
    else
      k_adj_count<4><<<gv, T, 0, st>>>(b.NV, b.inc_ptr, b.inc, b.conn, b.vrank, cnt, max_len, b.err_flag);
  }
  return exclusive_scan_i32(cnt, b.adj_ptr, b.NV, tmp, st);
}

cudaError_t launch_topology_fill(Batch& b) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const unsigned gv = (unsigned)((b.NV + T - 1) / T);
  if (b.NV) {
    if (b.npc == 3) k_adj_fill<3><<<gv, T, 0, st>>>(b.NV, b.inc_ptr, b.inc, b.conn, b.vrank, b.adj_ptr, b.adj);
    else k_adj_fill<4><<<gv, T, 0, st>>>(b.NV, b.inc_ptr, b.inc, b.conn, b.vrank, b.adj_ptr, b.adj);
  }
  return cudaGetLastError();
}

}  // namespace fea
