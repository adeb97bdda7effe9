// K1: element stiffness integration -- replaces sfepy's dw_lin_elastic(m.D, v, u) with the
// order-2 integral (reference datagen/fea_analysis.py:71-73, 153-160, 302-310; SURVEY A-4/A-5).
//   P1 triangle: K_e = area * B^T D B (B constant over the cell).
//   Q1 quad    : bilinear basis on the [0,1]^2 reference cell, 2x2 Gauss-Legendre (unpinned, F11).
// Local DOF order: 2*node + component.  One thread per cell; 36 (64) doubles written per thread.
#include "fea_internal.cuh"

namespace fea {

// K[(2a+i), (2b+j)] += w * sum_{p,q} B[p][2a+i] * D[p][q] * B[q][2b+j]
// with B rows (e11, e22, 2e12): B[0][2a]=gx_a, B[1][2a+1]=gy_a, B[2][2a]=gy_a, B[2][2a+1]=gx_a.
template <int NPC>
__device__ __forceinline__ void accumulate_btdb(const double* gx, const double* gy, const double* D,
                                                double w, double* K) {
  constexpr int N = 2 * NPC;
  // DB[p][col] for col = 2b+j
  double DB[3][N];
#pragma unroll
  for (int b = 0; b < NPC; ++b) {
#pragma unroll
    for (int p = 0; p < 3; ++p) {
      DB[p][2 * b] = D[p * 3 + 0] * gx[b] + D[p * 3 + 2] * gy[b];
      DB[p][2 * b + 1] = D[p * 3 + 1] * gy[b] + D[p * 3 + 2] * gx[b];
    }
  }
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
#pragma unroll
    for (int c = 0; c < N; ++c) {
      K[(2 * a) * N + c] += w * (gx[a] * DB[0][c] + gy[a] * DB[2][c]);
      K[(2 * a + 1) * N + c] += w * (gy[a] * DB[1][c] + gx[a] * DB[2][c]);
    }
  }
}

__global__ void k_element_p1(int64_t NC, const double* __restrict__ xy, const int32_t* __restrict__ conn,
                             const int32_t* __restrict__ cell_dreg, const double* __restrict__ Dtab,
                             double* __restrict__ ke) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  double K[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) K[i] = 0.0;
  const int r = cell_dreg[c];
  if (r >= 0) {
    double x[3], y[3], D[9];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const int64_t v = conn[c * 3 + a];
      x[a] = xy[2 * v];
      y[a] = xy[2 * v + 1];
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) D[i] = Dtab[(int64_t)r * 9 + i];
    const double b0 = y[1] - y[2], b1 = y[2] - y[0], b2 = y[0] - y[1];
    const double c0 = x[2] - x[1], c1 = x[0] - x[2], c2 = x[1] - x[0];
    const double det = x[0] * b0 + x[1] * b1 + x[2] * b2;  // 2 * signed area
    const double inv = 1.0 / det;
    const double gx[3] = {b0 * inv, b1 * inv, b2 * inv};
    const double gy[3] = {c0 * inv, c1 * inv, c2 * inv};
    accumulate_btdb<3>(gx, gy, D, 0.5 * fabs(det), K);
  }
  // 288 B per cell = nine 32-byte sectors: 256-bit stores write whole sectors
  d4* out = reinterpret_cast<d4*>(ke + c * 36);
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    d4 v;
    v.x = K[4 * i];
    v.y = K[4 * i + 1];
    v.z = K[4 * i + 2];
    v.w = K[4 * i + 3];
    out[i] = v;
  }
}

__global__ void k_element_q1(int64_t NC, const double* __restrict__ xy, const int32_t* __restrict__ conn,
                             const int32_t* __restrict__ cell_dreg, const double* __restrict__ Dtab,
                             double* __restrict__ ke) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  double K[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) K[i] = 0.0;
  const int r = cell_dreg[c];
  if (r >= 0) {
    double x[4], y[4], D[9];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int64_t v = conn[c * 4 + a];
      x[a] = xy[2 * v];
      y[a] = xy[2 * v + 1];
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) D[i] = Dtab[(int64_t)r * 9 + i];
    const double g = 0.5 / sqrt(3.0);
    const double qx[4] = {0.5 - g, 0.5 + g, 0.5 + g, 0.5 - g};
    const double qy[4] = {0.5 - g, 0.5 - g, 0.5 + g, 0.5 + g};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double xi = qx[q], eta = qy[q];
      const double dxi[4] = {-(1.0 - eta), (1.0 - eta), eta, -eta};
      const double det_[4] = {-(1.0 - xi), -xi, xi, (1.0 - xi)};
      double J00 = 0, J01 = 0, J10 = 0, J11 = 0;  // J[i][j] = d x_j / d xi_i
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        J00 += dxi[a] * x[a];
        J01 += dxi[a] * y[a];
        J10 += det_[a] * x[a];
        J11 += det_[a] * y[a];
      }
      const double det = J00 * J11 - J01 * J10;
      const double inv = 1.0 / det;
      double gx[4], gy[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        gx[a] = (J11 * dxi[a] - J01 * det_[a]) * inv;
        gy[a] = (-J10 * dxi[a] + J00 * det_[a]) * inv;
      }
      accumulate_btdb<4>(gx, gy, D, 0.25 * fabs(det), K);
    }
  }
  d4* out = reinterpret_cast<d4*>(ke + c * 64);
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    d4 v;
    v.x = K[4 * i];
    v.y = K[4 * i + 1];
    v.z = K[4 * i + 2];
    v.w = K[4 * i + 3];
    out[i] = v;
  }
}

// Per-cell pieces of the strain / stress kernels below, shared so that the single-batch and the load-case kernel
// compute each cell the same way.
// gradients of the P1 shape functions of a triangle (constant over the cell)
__device__ __forceinline__ void p1_gradients(const double x[3], const double y[3], double gx[3], double gy[3]) {
  const double b0 = y[1] - y[2], b1 = y[2] - y[0], b2 = y[0] - y[1];
  const double c0 = x[2] - x[1], c1 = x[0] - x[2], c2 = x[1] - x[0];
  const double inv = 1.0 / (x[0] * b0 + x[1] * b1 + x[2] * b2);
  gx[0] = b0 * inv;
  gx[1] = b1 * inv;
  gx[2] = b2 * inv;
  gy[0] = c0 * inv;
  gy[1] = c1 * inv;
  gy[2] = c2 * inv;
}
// (e11, e22, 2e12) of a triangle from its shape-function gradients and nodal displacements
__device__ __forceinline__ void p1_strain(const double gx[3], const double gy[3], const double ux[3], const double uy[3],
                                          double e[3]) {
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    e[0] += gx[a] * ux[a];
    e[1] += gy[a] * uy[a];
    e[2] += gy[a] * ux[a] + gx[a] * uy[a];
  }
}
// the material-table entry whose D gives cell c's stress (-1: none)
__device__ __forceinline__ int stress_entry(int64_t c, int stress_region, const int64_t* __restrict__ cell_off,
                                            const int32_t* __restrict__ reg_off, int ns,
                                            const int32_t* __restrict__ cell_dreg) {
  int r = cell_dreg[c];
  if (stress_region >= 0) {
    const int s = seg_of(cell_off, ns, c);
    r = (stress_region < reg_off[s + 1] - reg_off[s]) ? reg_off[s] + stress_region : -1;
  }
  return r;
}
// strain e and D e of cell c (row c of the [n][3] outputs), D = entry r of Dtab (r < 0: zero stress)
__device__ __forceinline__ void store_strain_stress(int64_t c, const double e[3], int r, const double* Dtab, double* strain,
                                                    double* stress) {
#pragma unroll
  for (int p = 0; p < 3; ++p) {
    strain[c * 3 + p] = e[p];
    double sg = 0.0;
    if (r >= 0) sg = Dtab[(int64_t)r * 9 + p * 3] * e[0] + Dtab[(int64_t)r * 9 + p * 3 + 1] * e[1] + Dtab[(int64_t)r * 9 + p * 3 + 2] * e[2];
    stress[c * 3 + p] = sg;
  }
}

// Post-process of the reference's calculate_stress_strain hook (datagen/fea_analysis.py:397-416):
// ev_cauchy_strain / ev_cauchy_stress in 'el_avg' mode = cell averages of (e11, e22, 2e12) and of
// D * strain.  stress_region >= 0 uses that material-table entry of the sample for every cell
// (the hook evaluates one material named 'm' over Omega); -1 uses each cell's own D (0 for cells
// that carry no stiffness).  One thread per cell.
template <int NPC>
__global__ void k_cell_strain_stress(int64_t NC, const int64_t* __restrict__ cell_off, const int32_t* __restrict__ reg_off,
                                     int ns, const double* __restrict__ xy, const int32_t* __restrict__ conn,
                                     const int32_t* __restrict__ cell_dreg, const double* __restrict__ Dtab,
                                     const double* __restrict__ u, int stress_region,
                                     double* __restrict__ strain, double* __restrict__ stress) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  double x[NPC], y[NPC], ux[NPC], uy[NPC];
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
    const int64_t v = conn[c * NPC + a];
    x[a] = xy[2 * v];
    y[a] = xy[2 * v + 1];
    ux[a] = u[2 * v];
    uy[a] = u[2 * v + 1];
  }
  double e[3] = {0.0, 0.0, 0.0};
  if constexpr (NPC == 3) {
    double gx[3], gy[3];
    p1_gradients(x, y, gx, gy);
    p1_strain(gx, gy, ux, uy, e);
  } else {
    const double g = 0.5 / sqrt(3.0);
    const double qx[4] = {0.5 - g, 0.5 + g, 0.5 + g, 0.5 - g};
    const double qy[4] = {0.5 - g, 0.5 - g, 0.5 + g, 0.5 + g};
    double vol = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const double xi = qx[q], eta = qy[q];
      const double dxi[4] = {-(1.0 - eta), (1.0 - eta), eta, -eta};
      const double det_[4] = {-(1.0 - xi), -xi, xi, (1.0 - xi)};
      double J00 = 0, J01 = 0, J10 = 0, J11 = 0;
#pragma unroll
      for (int a = 0; a < NPC; ++a) {
        J00 += dxi[a] * x[a];
        J01 += dxi[a] * y[a];
        J10 += det_[a] * x[a];
        J11 += det_[a] * y[a];
      }
      const double det = J00 * J11 - J01 * J10;
      const double inv = 1.0 / det;
      const double w = 0.25 * fabs(det);
      vol += w;
#pragma unroll
      for (int a = 0; a < NPC; ++a) {
        const double gx = (J11 * dxi[a] - J01 * det_[a]) * inv;
        const double gy = (-J10 * dxi[a] + J00 * det_[a]) * inv;
        e[0] += w * gx * ux[a];
        e[1] += w * gy * uy[a];
        e[2] += w * (gy * ux[a] + gx * uy[a]);
      }
    }
    e[0] /= vol;
    e[1] /= vol;
    e[2] /= vol;
  }
  const int r = stress_entry(c, stress_region, cell_off, reg_off, ns, cell_dreg);
  store_strain_stress(c, e, r, Dtab, strain, stress);
}

// The load cases of one triangle mesh (fea_batch_load_case_strain_stress): one thread per cell reads the cell's
// geometry and D once and applies them to the n_cases displacements u [n_cases][u_stride], with the helpers of
// k_cell_strain_stress, so case k is bit for bit what that kernel gives a batch solved with load k.
__global__ void k_cell_strain_stress_cases(int64_t NC, int n_cases, const int64_t* __restrict__ cell_off,
                                           const int32_t* __restrict__ reg_off, const double* __restrict__ xy,
                                           const int32_t* __restrict__ conn, const int32_t* __restrict__ cell_dreg,
                                           const double* __restrict__ Dtab, const double* __restrict__ u, int64_t u_stride,
                                           int stress_region, double* __restrict__ strain, double* __restrict__ stress) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC) return;
  int64_t v[3];
  double x[3], y[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    v[a] = conn[c * 3 + a];
    x[a] = xy[2 * v[a]];
    y[a] = xy[2 * v[a] + 1];
  }
  double gx[3], gy[3];
  p1_gradients(x, y, gx, gy);
  const int r = stress_entry(c, stress_region, cell_off, reg_off, 1, cell_dreg);
  double D[9];
  if (r >= 0) {
#pragma unroll
    for (int i = 0; i < 9; ++i) D[i] = Dtab[(int64_t)r * 9 + i];
  }
  for (int k = 0; k < n_cases; ++k) {
    const double* uk = u + k * u_stride;
    double ux[3], uy[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      ux[a] = uk[2 * v[a]];
      uy[a] = uk[2 * v[a] + 1];
    }
    double e[3] = {0.0, 0.0, 0.0};
    p1_strain(gx, gy, ux, uy, e);
    store_strain_stress(k * NC + c, e, r >= 0 ? 0 : -1, D, strain, stress);   // D: entry r, read once
  }
}

cudaError_t launch_case_strain_stress(Batch& b, int n_cases, const double* u, int stress_region, double* d_strain,
                                      double* d_stress) {
  if (!b.NC) return cudaSuccess;
  const int T = 128;
  k_cell_strain_stress_cases<<<(unsigned)((b.NC + T - 1) / T), T, 0, b.ctx->stream>>>(
      b.NC, n_cases, b.d_cell_off, b.d_reg_off, b.xy, b.conn, b.cell_dreg, b.D, u, 2 * b.NV, stress_region, d_strain, d_stress);
  return cudaGetLastError();
}

cudaError_t launch_cell_strain_stress(Batch& b, int stress_region, double* d_strain, double* d_stress) {
  if (!b.NC) return cudaSuccess;
  const int T = 128;
  const unsigned g = (unsigned)((b.NC + T - 1) / T);
  if (b.npc == 3)
    k_cell_strain_stress<3><<<g, T, 0, b.ctx->stream>>>(b.NC, b.d_cell_off, b.d_reg_off, b.ns, b.xy, b.conn, b.cell_dreg, b.D,
                                                        b.u, stress_region, d_strain, d_stress);
  else
    k_cell_strain_stress<4><<<g, T, 0, b.ctx->stream>>>(b.NC, b.d_cell_off, b.d_reg_off, b.ns, b.xy, b.conn, b.cell_dreg, b.D,
                                                        b.u, stress_region, d_strain, d_stress);
  return cudaGetLastError();
}

cudaError_t launch_element_stiffness(Batch& b) {
  if (!b.NC) return cudaSuccess;
  const int T = 128;
  const unsigned g = (unsigned)((b.NC + T - 1) / T);
  if (b.npc == 3) k_element_p1<<<g, T, 0, b.ctx->stream>>>(b.NC, b.xy, b.conn, b.cell_dreg, b.D, b.ke);
  else k_element_q1<<<g, T, 0, b.ctx->stream>>>(b.NC, b.xy, b.conn, b.cell_dreg, b.D, b.ke);
  return cudaGetLastError();
}

}  // namespace fea
