// K3/K4: value assembly straight into the solver's layout, with Dirichlet rows/columns
// dropped (SURVEY A-9/A-10) and symmetric Jacobi scaling folded in.
//
// Matrix layout ("block-SELL-32"): active vertices are block rows (2 DOFs each, both DOFs of a
// vertex are always eliminated together, reference datagen/fea_analysis.py:367).  32 block rows
// form a slice; a slice stores slice_len 2x2 blocks per row, column-major over the slice:
//   entry e = slice_ptr[slice] + j*32 + lane
//   val[e] = (k00, k01, k10, k11)   one 32-byte record per block
//   col[e] = block column (global block row id of the neighbour vertex)
// so a warp reads 1024 contiguous bytes with one 256-bit load instruction per lane.  Values are stored scaled:
//   Khat = S^T K S,  S = blockdiag(L_v^-T),  L_v = Cholesky factor of the vertex's 2x2 diagonal block
//   ->  CG on Khat == 2x2-block-Jacobi PCG on K (4.7 % fewer iterations than point Jacobi on the bench plates)
//   at no cost per iteration.
// Only OFF-diagonal blocks live in the SELL arrays: the scaled diagonal block of a vertex is the identity (up
// to one rounding, taken as exact), so it is not stored at all.
// Row sums run over the vertex's incident cells in ascending cell order: atomic-free,
// bitwise reproducible.
#include "fea_internal.cuh"

namespace fea {

__global__ void k_slice_len(int n_slices, const int32_t* __restrict__ vertex_of_row,
                            const int32_t* __restrict__ adj_ptr, int32_t* __restrict__ slice_len) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int slice = (int)(row >> 5);
  if (slice >= n_slices) return;
  const int v = vertex_of_row[row];
  int len = v >= 0 ? max(adj_ptr[v + 1] - adj_ptr[v] - 1, 0) : 0;  // off-diagonal blocks only
  len = warp_max_i(len);
  if ((threadIdx.x & 31) == 0) slice_len[slice] = len;
}

cudaError_t launch_sell_lengths(Batch& b) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  if (b.n_slices == 0) return cudaSuccess;
  k_slice_len<<<(unsigned)((b.NBR + T - 1) / T), T, 0, st>>>(b.n_slices, b.vertex_of_row, b.adj_ptr, b.slice_len);
  Scratch scratch(st);
  int64_t* tmp = nullptr;
  cudaError_t e = scratch.alloc(&tmp, b.n_slices / 4096 + 4);
  if (e != cudaSuccess) return e;
  return exclusive_scan_i32_to_i64(b.slice_len, b.slice_ptr, b.n_slices, 32, tmp, st);
}

// 2x2 block K[v][w] summed over the stiffness cells containing both, ascending cell order.
template <int NPC>
__device__ __forceinline__ void block_of_pair(int v, int w, const int32_t* __restrict__ inc_ptr,
                                              const int32_t* __restrict__ inc,
                                              const int32_t* __restrict__ conn,
                                              const double* __restrict__ ke, double k[4]) {
  constexpr int N = 2 * NPC;
  k[0] = k[1] = k[2] = k[3] = 0.0;
  const int b = inc_ptr[v], e = inc_ptr[v + 1];
  for (int i = b; i < e; ++i) {
    const int64_t c = inc[i] >> 2;
    const int a = inc[i] & 3;
#pragma unroll
    for (int bb = 0; bb < NPC; ++bb) {
      if (conn[c * NPC + bb] == w) {
        const double* K = ke + c * (N * N);   // both pairs are 16-byte aligned (even offsets)
        const double2 top = __ldg(reinterpret_cast<const double2*>(K + (2 * a) * N + 2 * bb));
        const double2 bot = __ldg(reinterpret_cast<const double2*>(K + (2 * a + 1) * N + 2 * bb));
        k[0] += top.x;
        k[1] += top.y;
        k[2] += bot.x;
        k[3] += bot.y;
      }
    }
  }
}

// The same sum with the corners of the (up to 8) cells around v already in registers: the search for w costs
// compares instead of loads (block_of_pair re-reads the connectivity of every incident cell for every neighbour:
// 7 x 6 x 3 loads per row on a triangle mesh).  Same cells, same order, same bits.
template <int NPC>
__device__ __forceinline__ void block_of_pair_cached(int w, int ik, const int (&cc)[8], const int (&ca)[8],
                                                     const int (&cv)[8][NPC], const double* __restrict__ ke, double k[4]) {
  constexpr int N = 2 * NPC;
  k[0] = k[1] = k[2] = k[3] = 0.0;
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    if (m < ik) {
#pragma unroll
      for (int bb = 0; bb < NPC; ++bb) {
        if (cv[m][bb] == w) {
          const double* K = ke + (int64_t)cc[m] * (N * N);
          const double2 top = __ldg(reinterpret_cast<const double2*>(K + (2 * ca[m]) * N + 2 * bb));
          const double2 bot = __ldg(reinterpret_cast<const double2*>(K + (2 * ca[m] + 1) * N + 2 * bb));
          k[0] += top.x;
          k[1] += top.y;
          k[2] += bot.x;
          k[3] += bot.y;
        }
      }
    }
  }
}

// S = L^-T of the Cholesky factor L of a vertex's diagonal block [[d0, dc], [dc, d1]]: (i00, i10, i11); false if
// the block is not positive definite (then all three are 0)
__device__ __forceinline__ bool block_scale(double d0, double d1, double dc, double& i00, double& i10, double& i11) {
  const double l00 = d0 > 0.0 ? sqrt(d0) : 0.0;
  const double l10 = d0 > 0.0 ? dc / l00 : 0.0;
  const double t = d1 - l10 * l10;
  if (d0 > 0.0 && d1 > 0.0 && t > 0.0) {
    const double l11 = sqrt(t);
    i00 = 1.0 / l00;
    i11 = 1.0 / l11;
    i10 = -l10 * i00 * i11;
    return true;
  }
  return false;
}

// Khat_vw = L_v^-1 K_vw L_w^-T with L_v^-1 = [[s0, 0], [sc, s1]] and L_w^-T = [[t0, tc], [0, t1]]
__device__ __forceinline__ d4 scaled_block(const double k[4], double s0, double s1, double sc, double t0, double t1, double tc) {
  const double a00 = s0 * k[0], a01 = s0 * k[1];
  const double a10 = fma(sc, k[0], s1 * k[2]), a11 = fma(sc, k[1], s1 * k[3]);
  d4 blk;
  blk.x = a00 * t0;
  blk.y = fma(a00, tc, a01 * t1);
  blk.z = a10 * t0;
  blk.w = fma(a10, tc, a11 * t1);
  return blk;
}

template <int NPC>
__global__ void k_diag_scale(int64_t NBR, const int32_t* __restrict__ vertex_of_row,
                             const int32_t* __restrict__ vsample, const int32_t* __restrict__ inc_ptr,
                             const int32_t* __restrict__ inc, const double* __restrict__ ke,
                             double* __restrict__ dscale, double* __restrict__ scoup, int32_t* __restrict__ empty) {
  constexpr int N = 2 * NPC;
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int v = vertex_of_row[row];
  double i00 = 0.0, i10 = 0.0, i11 = 0.0;
  if (v >= 0) {
    double d0 = 0.0, d1 = 0.0, dc = 0.0;   // diagonal block [[d0, dc], [dc, d1]] of the vertex
    const int b = inc_ptr[v], e = inc_ptr[v + 1];
    for (int i = b; i < e; ++i) {
      const int64_t c = inc[i] >> 2;
      const int a = inc[i] & 3;
      d0 += ke[c * (N * N) + (2 * a) * N + 2 * a];
      d1 += ke[c * (N * N) + (2 * a + 1) * N + 2 * a + 1];
      dc += ke[c * (N * N) + (2 * a) * N + 2 * a + 1];
    }
    // Cholesky factor L = [[l00, 0], [l10, l11]] of the block; S = L^-T
    if (!block_scale(d0, d1, dc, i00, i10, i11)) empty[vsample[v]] = 1;  // A-18: exactly singular
  }
  dscale[2 * row] = i00;
  dscale[2 * row + 1] = i11;
  scoup[row] = i10;
}

template <int NPC>
__global__ void k_sell_fill(int64_t NBR, const int32_t* __restrict__ vertex_of_row,
                            const int32_t* __restrict__ row_of_vertex, const int32_t* __restrict__ adj_ptr,
                            const int32_t* __restrict__ adj, const int32_t* __restrict__ inc_ptr,
                            const int32_t* __restrict__ inc, const int32_t* __restrict__ conn,
                            const double* __restrict__ ke, const double* __restrict__ dscale,
                            const double* __restrict__ scoup, const int32_t* __restrict__ slice_len, const int64_t* __restrict__ slice_ptr,
                            d4* __restrict__ val, int32_t* __restrict__ col) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = slice_len[slice];
  const int64_t base = slice_ptr[slice];
  const int v = vertex_of_row[row];
  int a0 = 0, n = 0;
  double s0 = 0.0, s1 = 0.0, sc = 0.0;   // L_v^-1 = [[s0, 0], [sc, s1]]
  if (v >= 0) {
    a0 = adj_ptr[v];
    n = adj_ptr[v + 1] - a0;
    s0 = dscale[2 * row];
    s1 = dscale[2 * row + 1];
    sc = scoup[row];
  }
  int j = 0;
  int ik = 0, cc[8], ca[8], cv[8][NPC];          // the cells around v (fast path: at most 8)
  if (v >= 0) {
    const int ib = inc_ptr[v];
    ik = inc_ptr[v + 1] - ib;
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const int ent = (ik <= 8 && m < ik) ? inc[ib + m] : 0;
      cc[m] = ent >> 2;
      ca[m] = ent & 3;
#pragma unroll
      for (int bb = 0; bb < NPC; ++bb) cv[m][bb] = (ik <= 8 && m < ik) ? conn[(int64_t)cc[m] * NPC + bb] : -1;
    }
  }
  for (int i = 0; i < n; ++i) {
    const int w = adj[a0 + i];
    double k[4];
    if (ik <= 8) block_of_pair_cached<NPC>(w, ik, cc, ca, cv, ke, k);
    else block_of_pair<NPC>(v, w, inc_ptr, inc, conn, ke, k);
    if (w == v) continue;                  // the scaled diagonal block is the identity (k_diag_scale)
    const int wr = row_of_vertex[w];
    const double t0 = dscale[2 * (int64_t)wr], t1 = dscale[2 * (int64_t)wr + 1], tc = scoup[wr];
    const int64_t e = base + (int64_t)j * 32;
    // Khat_vw = L_v^-1 K_vw L_w^-T,  L_w^-T = [[t0, tc], [0, t1]]
    val[e + lane] = scaled_block(k, s0, s1, sc, t0, t1, tc);
    col[e + lane] = wr;
    ++j;
  }
  for (; j < L; ++j) {  // slice padding: zero block pointing at the own row
    const int64_t e = base + (int64_t)j * 32;
    d4 zero;
    zero.x = zero.y = zero.z = zero.w = 0.0;
    val[e + lane] = zero;
    col[e + lane] = (int32_t)row;
  }
}

// ---------------------------------------------------------------------------
// Matrices given as an unscaled block-CSR over the vertices (multigrid grid levels, api_batch_assemble_csr):
// adj_ptr / adj are its pattern, blk [n_adj] its blocks.  Same scaling, same SELL layout, same padding.
// ---------------------------------------------------------------------------
__global__ void k_diag_scale_csr(int64_t NBR, const int32_t* __restrict__ vertex_of_row, const int32_t* __restrict__ vsample,
                                 const int32_t* __restrict__ adj_ptr, const int32_t* __restrict__ adj, const d4* __restrict__ blk,
                                 double* __restrict__ dscale, double* __restrict__ scoup, int32_t* __restrict__ empty) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int v = vertex_of_row[row];
  double i00 = 0.0, i10 = 0.0, i11 = 0.0;
  if (v >= 0) {
    double d0 = 0.0, d1 = 0.0, dc = 0.0;
    for (int i = adj_ptr[v]; i < adj_ptr[v + 1]; ++i)
      if (adj[i] == v) {
        d0 = blk[i].x;
        d1 = blk[i].w;
        dc = blk[i].y;
      }
    if (!block_scale(d0, d1, dc, i00, i10, i11)) empty[vsample[v]] = 1;
  }
  dscale[2 * row] = i00;
  dscale[2 * row + 1] = i11;
  scoup[row] = i10;
}

__global__ void k_sell_fill_csr(int64_t NBR, const int32_t* __restrict__ vertex_of_row, const int32_t* __restrict__ row_of_vertex,
                                const int32_t* __restrict__ adj_ptr, const int32_t* __restrict__ adj, const d4* __restrict__ blk,
                                const double* __restrict__ dscale, const double* __restrict__ scoup,
                                const int32_t* __restrict__ slice_len, const int64_t* __restrict__ slice_ptr, d4* __restrict__ val,
                                int32_t* __restrict__ col) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = slice_len[slice];
  const int64_t base = slice_ptr[slice];
  const int v = vertex_of_row[row];
  int j = 0;
  if (v >= 0) {
    const double s0 = dscale[2 * row], s1 = dscale[2 * row + 1], sc = scoup[row];
    for (int i = adj_ptr[v]; i < adj_ptr[v + 1]; ++i) {
      const int w = adj[i];
      if (w == v) continue;
      const d4 b = blk[i];
      const double k[4] = {b.x, b.y, b.z, b.w};
      const int wr = row_of_vertex[w];
      const int64_t e = base + (int64_t)j * 32;
      val[e + lane] = scaled_block(k, s0, s1, sc, dscale[2 * (int64_t)wr], dscale[2 * (int64_t)wr + 1], scoup[wr]);
      col[e + lane] = wr;
      ++j;
    }
  }
  for (; j < L; ++j) {
    const int64_t e = base + (int64_t)j * 32;
    d4 zero;
    zero.x = zero.y = zero.z = zero.w = 0.0;
    val[e + lane] = zero;
    col[e + lane] = (int32_t)row;
  }
}

cudaError_t launch_sell_fill_csr(Batch& b, const double* d_blocks) {
  const int T = 128;
  if (b.NBR == 0) return cudaSuccess;
  const unsigned g = (unsigned)((b.NBR + T - 1) / T);
  cudaStream_t st = b.ctx->stream;
  k_diag_scale_csr<<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.vsample, b.adj_ptr, b.adj, (const d4*)d_blocks, b.dscale, b.scoup,
                                    b.empty);
  k_sell_fill_csr<<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.row_of_vertex, b.adj_ptr, b.adj, (const d4*)d_blocks, b.dscale,
                                   b.scoup, b.slice_len, b.slice_ptr, (d4*)b.val, b.col);
  return cudaGetLastError();
}

// the element matrices of a triangle batch summed into blocks over its adjacency (the pattern of each active row)
__global__ void k_block_csr(int64_t NV, const int32_t* __restrict__ vrank, const int32_t* __restrict__ adj_ptr,
                            const int32_t* __restrict__ adj, const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                            const int32_t* __restrict__ conn, const double* __restrict__ ke, d4* __restrict__ out) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV || vrank[v] < 0) return;
  for (int i = adj_ptr[v]; i < adj_ptr[v + 1]; ++i) {
    double k[4];
    block_of_pair<3>((int)v, adj[i], inc_ptr, inc, conn, ke, k);
    d4 b;
    b.x = k[0];
    b.y = k[1];
    b.z = k[2];
    b.w = k[3];
    out[i] = b;
  }
}

cudaError_t launch_block_csr(Batch& b, double* d_blocks) {
  const int T = 128;
  if (b.NV == 0) return cudaSuccess;
  k_block_csr<<<(unsigned)((b.NV + T - 1) / T), T, 0, b.ctx->stream>>>(b.NV, b.vrank, b.adj_ptr, b.adj, b.inc_ptr, b.inc, b.conn,
                                                                        b.ke, (d4*)d_blocks);
  return cudaGetLastError();
}

cudaError_t launch_sell_fill(Batch& b) {
  cudaStream_t st = b.ctx->stream;
  const int T = 128;
  if (b.NBR == 0) return cudaSuccess;
  const unsigned g = (unsigned)((b.NBR + T - 1) / T);
  if (b.npc == 3) {
    k_diag_scale<3><<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.vsample, b.inc_ptr, b.inc, b.ke, b.dscale, b.scoup, b.empty);
    k_sell_fill<3><<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.row_of_vertex, b.adj_ptr, b.adj, b.inc_ptr, b.inc,
                                    b.conn, b.ke, b.dscale, b.scoup, b.slice_len, b.slice_ptr, (d4*)b.val, b.col);
  } else {
    k_diag_scale<4><<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.vsample, b.inc_ptr, b.inc, b.ke, b.dscale, b.scoup, b.empty);
    k_sell_fill<4><<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.row_of_vertex, b.adj_ptr, b.adj, b.inc_ptr, b.inc,
                                    b.conn, b.ke, b.dscale, b.scoup, b.slice_len, b.slice_ptr, (d4*)b.val, b.col);
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Scalar CSR export of one sample in sfepy's layout (A-11): active DOFs renumbered in
// ascending order, columns ascending, full 2x2 node blocks, explicit zeros kept.
// ---------------------------------------------------------------------------
template <int NPC>
__global__ void k_csr_export(int64_t v0, int64_t v1, const int32_t* __restrict__ vrank,
                             const int32_t* __restrict__ adj_ptr, const int32_t* __restrict__ adj,
                             const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                             const int32_t* __restrict__ conn, const double* __restrict__ ke,
                             int32_t n_act, int32_t* __restrict__ indptr, int32_t* __restrict__ indices,
                             double* __restrict__ data) {
  const int64_t v = v0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= v1) return;
  const int abase = adj_ptr[v0];
  if (v == v0 && indptr) indptr[2 * n_act] = 4 * (adj_ptr[v1] - abase);
  const int rk = vrank[v];
  if (rk < 0) return;
  const int A = adj_ptr[v] - abase, L = adj_ptr[v + 1] - adj_ptr[v];
  if (indptr) {
    indptr[2 * rk] = 4 * A;
    indptr[2 * rk + 1] = 4 * A + 2 * L;
  }
  for (int j = 0; j < L; ++j) {
    const int w = adj[adj_ptr[v] + j];
    const int cr = vrank[w];
    if (indices) {
      indices[4 * A + 2 * j] = 2 * cr;
      indices[4 * A + 2 * j + 1] = 2 * cr + 1;
      indices[4 * A + 2 * L + 2 * j] = 2 * cr;
      indices[4 * A + 2 * L + 2 * j + 1] = 2 * cr + 1;
    }
    if (data) {
      double k[4];
      block_of_pair<NPC>((int)v, w, inc_ptr, inc, conn, ke, k);
      data[4 * A + 2 * j] = k[0];
      data[4 * A + 2 * j + 1] = k[1];
      data[4 * A + 2 * L + 2 * j] = k[2];
      data[4 * A + 2 * L + 2 * j + 1] = k[3];
    }
  }
}

// The export of a batch assembled from a block-CSR, which keeps no unscaled matrix: K_vw = L_v Khat_vw L_w^T
// from the SELL values (L = S^-T; the diagonal block, Khat_vv = I, is L_v L_v^T), equal to the given blocks up
// to roundings.
__device__ __forceinline__ void l_of(const double* ds, const double* scp, int64_t r, double& l00, double& l10, double& l11) {
  l00 = 1.0 / ds[2 * r];
  l11 = 1.0 / ds[2 * r + 1];
  l10 = -scp[r] / (ds[2 * r] * ds[2 * r + 1]);
}
__global__ void k_csr_export_sell(int64_t v0, int64_t v1, const int32_t* __restrict__ vrank, const int32_t* __restrict__ adj_ptr,
                                  const int32_t* __restrict__ adj, const int32_t* __restrict__ row_of_vertex,
                                  const int64_t* __restrict__ slice_ptr, const d4* __restrict__ val, const double* __restrict__ ds,
                                  const double* __restrict__ scp, int32_t n_act, int32_t* __restrict__ indptr,
                                  int32_t* __restrict__ indices, double* __restrict__ data) {
  const int64_t v = v0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= v1) return;
  const int abase = adj_ptr[v0];
  if (v == v0 && indptr) indptr[2 * n_act] = 4 * (adj_ptr[v1] - abase);
  const int rk = vrank[v];
  if (rk < 0) return;
  const int A = adj_ptr[v] - abase, L = adj_ptr[v + 1] - adj_ptr[v];
  if (indptr) {
    indptr[2 * rk] = 4 * A;
    indptr[2 * rk + 1] = 4 * A + 2 * L;
  }
  const int64_t row = row_of_vertex[v];
  double a00, a10, a11;
  l_of(ds, scp, row, a00, a10, a11);
  int jo = 0;
  for (int j = 0; j < L; ++j) {
    const int w = adj[adj_ptr[v] + j];
    const int cr = vrank[w];
    if (indices) {
      indices[4 * A + 2 * j] = 2 * cr;
      indices[4 * A + 2 * j + 1] = 2 * cr + 1;
      indices[4 * A + 2 * L + 2 * j] = 2 * cr;
      indices[4 * A + 2 * L + 2 * j + 1] = 2 * cr + 1;
    }
    d4 h;   // Khat_vw
    int64_t wr = row;
    if (w == v) {
      h.x = 1.0; h.y = 0.0; h.z = 0.0; h.w = 1.0;
    } else {
      h = val[slice_ptr[row >> 5] + (int64_t)jo * 32 + (row & 31)];
      wr = row_of_vertex[w];
      ++jo;
    }
    if (data) {
      double b00, b10, b11;
      l_of(ds, scp, wr, b00, b10, b11);
      // M = L_v Khat, then K = M L_w^T with L_w^T = [[b00, b10], [0, b11]]
      const double m00 = a00 * h.x, m01 = a00 * h.y;
      const double m10 = a10 * h.x + a11 * h.z, m11 = a10 * h.y + a11 * h.w;
      data[4 * A + 2 * j] = m00 * b00;
      data[4 * A + 2 * j + 1] = m00 * b10 + m01 * b11;
      data[4 * A + 2 * L + 2 * j] = m10 * b00;
      data[4 * A + 2 * L + 2 * j + 1] = m10 * b10 + m11 * b11;
    }
  }
}

cudaError_t launch_csr_export(Batch& b, int32_t s, int32_t* d_indptr, int32_t* d_indices, double* d_data) {
  const int64_t v0 = b.vtx_off[s], v1 = b.vtx_off[s + 1];
  if (v1 == v0) return cudaSuccess;
  int32_t n_act = 0;
  cudaMemcpyAsync(&n_act, b.n_active + s, sizeof(int32_t), cudaMemcpyDeviceToHost, b.ctx->stream);
  cudaStreamSynchronize(b.ctx->stream);
  const int T = 128;
  const unsigned g = (unsigned)((v1 - v0 + T - 1) / T);
  if (b.from_csr)
    k_csr_export_sell<<<g, T, 0, b.ctx->stream>>>(v0, v1, b.vrank, b.adj_ptr, b.adj, b.row_of_vertex, b.slice_ptr, (const d4*)b.val,
                                                 b.dscale, b.scoup, n_act, d_indptr, d_indices, d_data);
  else if (b.npc == 3)
    k_csr_export<3><<<g, T, 0, b.ctx->stream>>>(v0, v1, b.vrank, b.adj_ptr, b.adj, b.inc_ptr, b.inc, b.conn, b.ke,
                                                n_act, d_indptr, d_indices, d_data);
  else
    k_csr_export<4><<<g, T, 0, b.ctx->stream>>>(v0, v1, b.vrank, b.adj_ptr, b.adj, b.inc_ptr, b.inc, b.conn, b.ke,
                                                n_act, d_indptr, d_indices, d_data);
  return cudaGetLastError();
}

}  // namespace fea
