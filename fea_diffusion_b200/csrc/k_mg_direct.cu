// Direct coarsest-level solve of the multigrid V-cycle (fea_batch_set_coarse_solver(b, FEA_COARSE_DIRECT);
// DESIGN.md section 3.13): the dense inverse of level 0's scaled operator Khat_0 = S^T K_0 S, built once at
// assemble time and applied to the K restricted residuals of a V-cycle by one matrix read.
//
//   layout    : Khat_0 over level 0's active block rows in the level batch's solver order (DOF 2r + c is
//               component c of block row r), row-major with a leading dimension N padded to kTile; the padding
//               is the identity, so the factor and the inverse of the padded matrix are blockdiag(., I).
//   build     : one thread per block row scatters its block-SELL row and the identity diagonal block.
//   Cholesky  : blocked, right-looking, tiles of kTile: per step k, one CTA factors the diagonal tile in shared
//               memory (recording its smallest pivot) and inverts it; the panel below is L_ik = A_ik L_kk^-T, a
//               product with that inverse; the trailing lower triangle takes A_ij -= L_ik L_jk^T.
//   inverse   : W = L^-1 in place by blocked forward substitution (step k: X_kj = L_kk^-1 B_kj, then
//               B_ij -= L_ik X_kj), then Khat_0^-1 = W^T W, each lower tile (i, j) a sum over the tile rows
//               m >= i, written to the kept buffer together with its mirror (i, j) -> (j, i).
//   products  : every tile product is one 64 x 64 tile of C per CTA of 64 threads, an 8 x 8 register tile of
//               plain DFMA per thread over inner chunks of kChunkK staged in shared memory.
//   apply     : y = S^T rhs per case (what k_pcg_init_vectors forms from the coarse batch's unscaled rhs), then
//               x^ = Khat_0^-1 y, one warp per DOF row with fixed lane striding and a fixed shuffle tree for every
//               case: a case's bits do not depend on K or on the other cases.
// Every sum has one fixed order and there are no atomics: two builds of the inverse are bit-identical.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <vector>

#include "fea_internal.cuh"

namespace fea {

namespace {

constexpr int kTile = 64;      // tile edge of the dense factorisation
constexpr int kChunkK = 16;    // inner-dimension chunk staged in shared memory per tile product step
constexpr int kProdT = 64;     // threads of a tile-product CTA: 8 x 8, each an 8 x 8 register tile

// ---------------------------------------------------------------------------------------------------------
// dense Khat_0 (zeroed before): identity diagonal blocks, block-SELL off-diagonal blocks; rows past n_rows are
// the identity padding
__global__ void k_mgd_build(int64_t n_rows, int64_t n_pad_rows, const int32_t* __restrict__ slice_len,
                            const int64_t* __restrict__ slice_ptr, const d4* __restrict__ val, const int32_t* __restrict__ col,
                            int64_t ld, double* __restrict__ A) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_pad_rows) return;
  double* a0 = A + (2 * r) * ld;
  double* a1 = a0 + ld;
  a0[2 * r] = 1.0;
  a1[2 * r + 1] = 1.0;
  if (r >= n_rows) return;
  const int64_t slice = r >> 5;
  const int lane = (int)(r & 31);
  const int L = slice_len[slice];
  const int64_t base = slice_ptr[slice] + lane;
  for (int j = 0; j < L; ++j) {
    const int c = col[base + (int64_t)j * 32];
    if (c == r) continue;   // slice padding: a zero block on the own row
    const d4 k = val[base + (int64_t)j * 32];
    a0[2 * c] = k.x;
    a0[2 * c + 1] = k.y;
    a1[2 * c] = k.z;
    a1[2 * c + 1] = k.w;
  }
}

// Cholesky factor of diagonal tile k in place (lower triangle; the upper one is left alone) and its inverse
// into linv[k] (full 64 x 64, zeros above the diagonal).  One thread per tile row.  piv[k], piv_at[k]: the smallest
// pivot (the value a square root is taken of) and its DOF, or, once a pivot is at or below `floor` or NaN, that
// first failing pivot (what follows it is NaN and says nothing).
__global__ void __launch_bounds__(kTile) k_mgd_potrf(double* __restrict__ A, int64_t ld, int k, double floor,
                                                     double* __restrict__ linv, double* __restrict__ piv,
                                                     int64_t* __restrict__ piv_at) {
  __shared__ double T[kTile][kTile + 1];
  const int i = threadIdx.x;
  double* tile = A + (int64_t)k * kTile * ld + (int64_t)k * kTile;
  for (int c = 0; c < kTile; ++c) T[c][i] = tile[(int64_t)c * ld + i];
  __syncthreads();
  double best = INFINITY;
  int best_at = 0;
  for (int j = 0; j < kTile; ++j) {
    const double d = T[j][j];
    if (i == 0 && best > floor && !(d >= best)) {
      best = d;
      best_at = j;
    }
    __syncthreads();
    const double l = sqrt(d);
    if (i == j) T[j][j] = l;
    if (i > j) T[i][j] = T[i][j] / l;
    __syncthreads();
    if (i > j)
      for (int c = j + 1; c <= i; ++c) T[i][c] = fma(-T[i][j], T[c][j], T[i][c]);
    __syncthreads();
  }
  for (int c = 0; c <= i; ++c) tile[(int64_t)i * ld + c] = T[i][c];
  if (i == 0) {
    piv[k] = best;
    piv_at[k] = (int64_t)k * kTile + best_at;
  }
  // column i of X = L_kk^-1 by forward substitution, X[r][i] (r >= i) kept at T[i][r + 1]: row i's strictly upper part
  // and its padding column, which the factor does not use, and which only thread i touches
  for (int r = i; r < kTile; ++r) {
    double s = r == i ? 1.0 : 0.0;
    for (int t = i; t < r; ++t) s = fma(-T[r][t], T[i][t + 1], s);
    T[i][r + 1] = s / T[r][r];
  }
  double* X = linv + (int64_t)k * kTile * kTile;
  for (int r = 0; r < kTile; ++r) X[r * kTile + i] = r < i ? 0.0 : T[i][r + 1];
}

// C = beta C + alpha sum_t a(r, t) b(t, c) on one kTile x kTile tile, t over kt tiles:
//   a(r, t) = TA ? A[t * lda + r] : A[r * lda + t],   b(t, c) = TB ? B[c * ldb + t] : B[t * ldb + c].
// beta is 0 or 1.  C may be one of the operands: every operand load precedes the last barrier before the store.
// Cmirror, if given, also receives the transpose; a diagonal tile (Cmirror == C) stores its lower half twice, so
// no element has two writers.
template <bool TA, bool TB>
__device__ __forceinline__ void tile_product(const double* A, int64_t lda, const double* B, int64_t ldb, int kt, double alpha,
                                             int beta, double* C, int64_t ldc, double* Cmirror = nullptr) {
  __shared__ double As[kChunkK][kTile + 1], Bs[kChunkK][kTile + 1];
  const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;
  double acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;
  const int nk = kt * (kTile / kChunkK);
  for (int s = 0; s < nk; ++s) {
    const int64_t t0 = (int64_t)s * kChunkK;
#pragma unroll 4   // (a full unroll keeps 32 loads in flight beside the 64 accumulators and spills)
    for (int q = 0; q < kChunkK * kTile / kProdT; ++q) {
      const int e = tid + q * kProdT;
      if (TA) {
        const int t = e >> 6, r = e & 63;
        As[t][r] = A[(t0 + t) * lda + r];
      } else {
        const int r = e >> 4, t = e & 15;
        As[t][r] = A[(int64_t)r * lda + t0 + t];
      }
      if (TB) {
        const int c = e >> 4, t = e & 15;
        Bs[t][c] = B[(int64_t)c * ldb + t0 + t];
      } else {
        const int t = e >> 6, c = e & 63;
        Bs[t][c] = B[(t0 + t) * ldb + c];
      }
    }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < kChunkK; ++t) {
      double av[8], bv[8];
#pragma unroll
      for (int a = 0; a < 8; ++a) av[a] = As[t][ty + 8 * a];
#pragma unroll
      for (int b = 0; b < 8; ++b) bv[b] = Bs[t][tx + 8 * b];
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 8; ++a) {
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int r = ty + 8 * a, c = tx + 8 * b;
      if (Cmirror == C && c > r) continue;
      double* p = C + (int64_t)r * ldc + c;
      const double v = beta ? fma(alpha, acc[a][b], *p) : alpha * acc[a][b];
      *p = v;
      if (Cmirror) Cmirror[(int64_t)c * ldc + r] = v;
    }
  }
}

__device__ __forceinline__ double* tile_at(double* A, int64_t ld, int i, int j) {
  return A + (int64_t)i * kTile * ld + (int64_t)j * kTile;
}

// panel of step k: L_ik = A_ik L_kk^-T, tile i = k + 1 + blockIdx.x
__global__ void __launch_bounds__(kProdT) k_mgd_panel(double* A, int64_t ld, int k, const double* __restrict__ linv) {
  const int i = k + 1 + blockIdx.x;
  double* C = tile_at(A, ld, i, k);
  tile_product<false, true>(C, ld, linv + (int64_t)k * kTile * kTile, kTile, 1, 1.0, 0, C, ld);
}

// trailing update of step k: A_ij -= L_ik L_jk^T for k < j <= i
__global__ void __launch_bounds__(kProdT) k_mgd_syrk(double* A, int64_t ld, int k) {
  const int i = k + 1 + blockIdx.x, j = k + 1 + blockIdx.y;
  if (j > i) return;
  tile_product<false, true>(tile_at(A, ld, i, k), ld, tile_at(A, ld, j, k), ld, 1, -1.0, 1, tile_at(A, ld, i, j), ld);
}

// forward substitution L W = I, step k.  Row: X_kj = L_kk^-1 B_kj for j < k (blockIdx.x = j), X_kk = L_kk^-1.
__global__ void __launch_bounds__(kProdT) k_mgd_trtri_row(double* A, int64_t ld, int k, const double* __restrict__ linv) {
  const int j = blockIdx.x;
  const double* Li = linv + (int64_t)k * kTile * kTile;
  double* C = tile_at(A, ld, k, j);
  if (j == k) {
    for (int e = threadIdx.x; e < kTile * kTile; e += kProdT) C[(int64_t)(e >> 6) * ld + (e & 63)] = Li[e];
    return;
  }
  tile_product<false, false>(Li, kTile, C, ld, 1, 1.0, 0, C, ld);
}
// B_ij -= L_ik X_kj for i > k, j < k (position (i, k) still holds L_ik)
__global__ void __launch_bounds__(kProdT) k_mgd_trtri_update(double* A, int64_t ld, int k) {
  const int i = k + 1 + blockIdx.x, j = blockIdx.y;
  tile_product<false, false>(tile_at(A, ld, i, k), ld, tile_at(A, ld, k, j), ld, 1, -1.0, 1, tile_at(A, ld, i, j), ld);
}
// then B_ik = -L_ik X_kk, in place, for i > k
__global__ void __launch_bounds__(kProdT) k_mgd_trtri_col(double* A, int64_t ld, int k) {
  const int i = k + 1 + blockIdx.x;
  double* C = tile_at(A, ld, i, k);
  tile_product<false, false>(C, ld, tile_at(A, ld, k, k), ld, 1, -1.0, 0, C, ld);
}

// Khat^-1 = W^T W: tile (i, j), j <= i, is sum_{m >= i} W_mi^T W_mj; stored at (i, j) and mirrored to (j, i)
__global__ void __launch_bounds__(kProdT) k_mgd_lauum(const double* __restrict__ W, int64_t ld, int T, double* __restrict__ M) {
  const int i = blockIdx.x, j = blockIdx.y;
  if (j > i) return;
  const double* Wi = W + (int64_t)i * kTile * ld;   // tile row m = i
  tile_product<true, false>(Wi + (int64_t)i * kTile, ld, Wi + (int64_t)j * kTile, ld, T - i, 1.0, 0, tile_at(M, ld, i, j), ld,
                            tile_at(M, ld, j, i));
}

// ---------------------------------------------------------------------------------------------------------
// apply.  y[q][2r + c] = (S^T rhs_q)[r] for the active rows r < n_rows; case q's vertex v is v + q * nv_stride
__global__ void k_mgd_rhs(int64_t n_rows, int K, const int32_t* __restrict__ vertex_of_row, const double* __restrict__ dscale,
                          const double* __restrict__ scoup, const double* __restrict__ rhs, int64_t nv_stride, int64_t ld,
                          double* __restrict__ y) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const int64_t v = vertex_of_row[r];
  for (int q = 0; q < K; ++q) {
    const double b0 = rhs[2 * (v + q * nv_stride)], b1 = rhs[2 * (v + q * nv_stride) + 1];
    y[q * ld + 2 * r] = dscale[2 * r] * b0;
    y[q * ld + 2 * r + 1] = fma(scoup[r], b0, dscale[2 * r + 1] * b1);
  }
}

// x^ = Khat^-1 y for K cases, one warp per DOF row i: lane l sums columns 2l + 64m, 2l + 64m + 1 in ascending m,
// then warp_sum.  DOF i = 2r + c lands in component c of x[r * row_stride + q * col_stride].
template <int K>
__global__ void __launch_bounds__(256) k_mgd_apply(int64_t n, const double* __restrict__ M, int64_t ld, const double* __restrict__ y,
                                                   double* __restrict__ x, int64_t row_stride, int64_t col_stride) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const double2* m = reinterpret_cast<const double2*>(M + i * ld);
  double acc[K];
#pragma unroll
  for (int q = 0; q < K; ++q) acc[q] = 0.0;
  for (int64_t c = lane; 2 * c < n; c += 32) {
    const double2 a = __ldcs(m + c);
#pragma unroll
    for (int q = 0; q < K; ++q) {
      const double2 b = __ldg(reinterpret_cast<const double2*>(y + q * ld) + c);
      acc[q] = fma(a.x, b.x, acc[q]);
      acc[q] = fma(a.y, b.y, acc[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < K; ++q) acc[q] = warp_sum(acc[q]);
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < K; ++q) x[2 * ((i >> 1) * row_stride + q * col_stride) + (i & 1)] = acc[q];
  }
}

// rhs by vertex of an active-DOF vector (unscaled, numbered by vrank): 0 at fixed vertices
__global__ void k_mgd_scatter(int64_t nv, const int32_t* __restrict__ vrank, const double* __restrict__ in, double* __restrict__ rhs) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  const int k = vrank[v];
  rhs[2 * v] = k >= 0 ? in[2 * (int64_t)k] : 0.0;
  rhs[2 * v + 1] = k >= 0 ? in[2 * (int64_t)k + 1] : 0.0;
}

}  // namespace

int mg_direct_factor(fea_ctx* ctx, Batch& b) {
  Mg& mg = *b.mg;
  const Batch& l0 = *mg.lev[0].b;
  cudaStream_t st = ctx->c.stream;
  int32_t na = 0, empty = 0;
  CK(ctx, cudaMemcpyAsync(&na, l0.n_active, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(&empty, l0.empty, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  const int64_t n = 2 * (int64_t)na;
  char msg[192];
  if (n > kMaxDirectDofs) {
    snprintf(msg, sizeof(msg), "level 0 has %lld active DOFs, more than the %lld of the direct coarse solver", (long long)n,
             (long long)kMaxDirectDofs);
    return api_fail(ctx, FEA_MESH_ERROR, msg);
  }
  if (empty) return api_fail(ctx, FEA_MESH_ERROR, "level 0 has an empty row: the direct coarse solver needs every row");
  const int T = (int)std::max<int64_t>(1, (n + kTile - 1) / kTile);
  const int64_t N = (int64_t)T * kTile;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  CK(ctx, cudaEventCreate(&ev[0]));
  CK(ctx, cudaEventCreate(&ev[1]));
  struct Events {
    cudaEvent_t* e;
    ~Events() {
      cudaEventDestroy(e[0]);
      cudaEventDestroy(e[1]);
    }
  } own{ev};
  CK(ctx, cudaMallocAsync((void**)&mg.coarse_inv, sizeof(double) * N * N, st));
  CK(ctx, cudaMallocAsync((void**)&mg.coarse_y, sizeof(double) * N * kMaxCases, st));
  CK(ctx, cudaMemsetAsync(mg.coarse_y, 0, sizeof(double) * N * kMaxCases, st));
  Scratch scratch(st);
  double *W = nullptr, *linv = nullptr, *piv = nullptr;
  int64_t* piv_at = nullptr;
  CK(ctx, scratch.alloc(&W, N * N));
  CK(ctx, scratch.alloc(&linv, (int64_t)T * kTile * kTile));
  CK(ctx, scratch.alloc(&piv, T));
  CK(ctx, scratch.alloc(&piv_at, T));
  CK(ctx, cudaEventRecord(ev[0], st));
  CK(ctx, cudaMemsetAsync(W, 0, sizeof(double) * N * N, st));
  k_mgd_build<<<(unsigned)((N / 2 + 127) / 128), 128, 0, st>>>(na, N / 2, l0.slice_len, l0.slice_ptr, (const d4*)l0.val, l0.col, N, W);
  for (int k = 0; k < T; ++k) {   // Cholesky
    k_mgd_potrf<<<1, kTile, 0, st>>>(W, N, k, kMinDirectPivot, linv, piv, piv_at);
    if (k + 1 < T) {
      k_mgd_panel<<<T - k - 1, kProdT, 0, st>>>(W, N, k, linv);
      k_mgd_syrk<<<dim3(T - k - 1, T - k - 1), kProdT, 0, st>>>(W, N, k);
    }
  }
  for (int k = 0; k < T; ++k) {   // W = L^-1
    k_mgd_trtri_row<<<k + 1, kProdT, 0, st>>>(W, N, k, linv);
    if (k + 1 < T) {
      if (k > 0) k_mgd_trtri_update<<<dim3(T - k - 1, k), kProdT, 0, st>>>(W, N, k);
      k_mgd_trtri_col<<<T - k - 1, kProdT, 0, st>>>(W, N, k);
    }
  }
  k_mgd_lauum<<<dim3(T, T), kProdT, 0, st>>>(W, N, T, mg.coarse_inv);
  CK(ctx, cudaGetLastError());
  CK(ctx, cudaEventRecord(ev[1], st));
  std::vector<double> hp(T);
  std::vector<int64_t> ha(T);
  CK(ctx, cudaMemcpyAsync(hp.data(), piv, sizeof(double) * T, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaMemcpyAsync(ha.data(), piv_at, sizeof(int64_t) * T, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  ctx->c.launches += 2 + 3 * (int64_t)T + 3 * (int64_t)T;
  float ms = 0.f;
  CK(ctx, cudaEventElapsedTime(&ms, ev[0], ev[1]));
  double best = INFINITY;
  int64_t at = 0;
  for (int k = 0; k < T; ++k)   // the rule of k_mgd_potrf across tiles: the smallest pivot, or the first failing one
    if (best > kMinDirectPivot && !(hp[k] >= best)) {
      best = hp[k];
      at = ha[k];
    }
  if (!(best > kMinDirectPivot)) {
    snprintf(msg, sizeof(msg), "level 0 is not positive definite enough for the direct coarse solver: Cholesky pivot %.6g "
             "at DOF %lld is at or below %g", best, (long long)at, kMinDirectPivot);
    return api_fail(ctx, FEA_MESH_ERROR, msg);
  }
  mg.coarse_n = n;
  mg.coarse_ld = N;
  mg.factor_ms = ms;
  mg.min_pivot = best;
  return FEA_OK;
}

cudaError_t mg_direct_apply(const Mg& mg, int K, const double* rhs, int64_t nv_stride, double* x, int64_t row_stride,
                            int64_t col_stride, cudaStream_t st) {
  const Batch& l0 = *mg.lev[0].b;
  const int64_t rows = mg.coarse_n / 2, N = mg.coarse_ld;
  if (!rows) return cudaSuccess;
  k_mgd_rhs<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(rows, K, l0.vertex_of_row, l0.dscale, l0.scoup, rhs, nv_stride, N,
                                                            mg.coarse_y);
  const unsigned g = (unsigned)((mg.coarse_n * 32 + 255) / 256);
  const double* M = mg.coarse_inv;
  double* y = mg.coarse_y;
  switch (K) {
    case 1: k_mgd_apply<1><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 2: k_mgd_apply<2><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 3: k_mgd_apply<3><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 4: k_mgd_apply<4><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 5: k_mgd_apply<5><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 6: k_mgd_apply<6><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 7: k_mgd_apply<7><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    case 8: k_mgd_apply<8><<<g, 256, 0, st>>>(mg.coarse_n, M, N, y, x, row_stride, col_stride); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

cudaError_t launch_active_to_vertices(cudaStream_t st, int64_t nv, const int32_t* vrank, const double* in, double* rhs) {
  if (nv) k_mgd_scatter<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(nv, vrank, in, rhs);
  return cudaGetLastError();
}

void mg_direct_release(Mg& mg, cudaStream_t st) {
  for (double* p : {mg.coarse_inv, mg.coarse_y})
    if (p) cudaFreeAsync(p, st);
  mg.coarse_inv = mg.coarse_y = nullptr;
}

}  // namespace fea
