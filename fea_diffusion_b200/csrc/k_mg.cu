// Multigrid-preconditioned flexible CG for a single sample that is a uniform red refinement of a coarser
// mesh (fea_batch_set_refinement; DESIGN.md section 3.9).
//
//   hierarchy : level l-1 is read off level l's children (cells p, p+nc, p+2nc, p+3nc of a parent p) and
//               checked against the input (structure, bit-exact midpoints, regions); a coarse level keeps
//               a prefix of the fine vertices.  Every coarse level is an internal Batch of its own.
//   operators : Galerkin K_c = P^T K_f P, summed cell by cell: the 6x6 matrix of parent p is the sum over its
//               four children of P_e^T M K_e M P_e (P_e: weights 0, 1/2, 1 of the child's vertices from the
//               parent's; M zeroes the DOFs fixed on the finer level).  k_sell_fill turns it into the
//               level's block-SELL matrix and 2x2 scaling, exactly as for element matrices.
//   transfers : in the scaled spaces, P^ = S_f^-1 P S_c and R^ = P^^T, so Khat_c = R^ Khat_f P^ exactly;
//               prolongation gathers from a vertex's two parents, restriction over a coarse vertex's
//               midpoint list.  No floating-point atomics anywhere.
//   smoother  : Chebyshev, three steps before and three after the coarse correction (symmetric V-cycle),
//               on Khat (identity diagonal blocks: block-Jacobi Chebyshev) over [lmax/30, 1.1 lmax], lmax
//               from 20 Lanczos steps per level at assemble time.
//   coarsest  : run_pcg on the level-0 batch to rtol 1e-4; the inexact coarse solve makes the outer
//               iteration flexible CG, beta = z+.(r+ - r) / (r.z) = -alpha z+.q / (r.z).  A batch that asks for
//               it (fea_batch_set_coarse_solver) applies a dense inverse of level 0 instead (k_mg_direct.cu;
//               DESIGN.md section 3.13), and its V-cycle is a fixed symmetric operator.
// Dot products: one partial per CTA, summed by one block in a fixed order (bitwise reproducible).
// A non-nested hierarchy (fea_batch_set_coarse_meshes, k_mg_nonnested.cu; DESIGN.md section 3.10) runs the same
// V-cycle and outer CG with rediscretised coarse operators and the k_mgn_* transfers (up to 3 weighted parents).
// A grid hierarchy (fea_batch_set_grid_hierarchy, k_mg_grid.cu; DESIGN.md section 3.12) uses the same transfers
// with nested background grids as coarse levels and Galerkin operators read from block-CSRs.
// Both solve K = 1..8 load cases at once (fea_batch_solve_load_cases; DESIGN.md section 3.11): the V-cycle and
// outer-CG kernels are templates on the number of columns they carry (a group of at most 4 cases), and
// fea_batch_solve is the case K = 1.
// The hierarchy (Mg) keeps what assemble builds: level batches, transfers, smoother coefficients, the coarse
// solver.  The vectors of a solve, a V-cycle or a Lanczos estimate belong to the call (a Scratch).
#include <cmath>
#include <cstdio>
#include <memory>
#include <type_traits>
#include <vector>

#include "fea_internal.cuh"

namespace fea {

namespace {

constexpr int kT = 128;            // threads per block of the row kernels (= kCtaRows: grids cover NBR exactly)
constexpr int kLanczos = 20;      // Lanczos steps of the lambda_max estimate
constexpr double kCoarseRtol = 1e-4;
constexpr int kCoarseMaxIter = 20000;
constexpr int kMaxRestarts = 4;    // outer restarts from the true residual before a solve counts as stagnated
constexpr unsigned long long kNoKey = ~0ull;

// device scalar slots
enum { kScRR = 0, kScRZ, kScBeta, kScAlpha, kScPQ, kScNrm, kScRZ0, kScTrue, kScCount };

struct MgOp {   // block-SELL matrix of one level (identity diagonal blocks not stored)
  const int32_t* slice_len;
  const int64_t* slice_ptr;
  const d4* val;
  const int32_t* col;
};
MgOp op_of(const Batch& b) { return MgOp{b.slice_len, b.slice_ptr, (const d4*)b.val, b.col}; }

// A kernel carries K columns (load cases; a group of at most 4, see each_group), interleaved per block row:
// column k of row r is v[r * K + k], so one gathered neighbour brings all K columns.  Every kernel below does,
// per column, exactly the arithmetic of
// K = 1 in the same order (the same fma chains, the same per-CTA partials): a column's bits do not depend on
// K or on the other columns.
// (Khat v)[row] of the K columns; row's lane in its slice = threadIdx.x & 31
template <int K>
__device__ __forceinline__ void khat_row(const MgOp& A, int64_t row, const double2* __restrict__ v, double2 (&out)[K]) {
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = A.slice_len[slice];
  const int64_t base = A.slice_ptr[slice];
  const d4* __restrict__ vt = A.val + base + lane;
  const int32_t* __restrict__ cp = A.col + base + lane;
  double a0[K], a1[K];
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const double2 own = v[row * K + q];
    a0[q] = own.x;
    a1[q] = own.y;
  }
  for (int j = 0; j < L; ++j) {
    const int c = ld_stream_i32(cp + j * 32);
    const d4 k = ld_stream_d4(vt + j * 32);
#pragma unroll
    for (int q = 0; q < K; ++q) {
      const double2 xj = __ldg(v + (int64_t)c * K + q);
      a0[q] = fma(k.x, xj.x, a0[q]);
      a0[q] = fma(k.y, xj.y, a0[q]);
      a1[q] = fma(k.z, xj.x, a1[q]);
      a1[q] = fma(k.w, xj.y, a1[q]);
    }
  }
#pragma unroll
  for (int q = 0; q < K; ++q) out[q] = make_double2(a0[q], a1[q]);
}

// deterministic block sums of K columns, written by thread 0 to part[q * gridDim.x + blockIdx.x]
template <int K>
__device__ __forceinline__ void block_partial(const double (&v)[K], double* __restrict__ part) {
  __shared__ double sm[K][kT / 32];
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const double s = warp_sum(v[q]);
    if ((threadIdx.x & 31) == 0) sm[q][threadIdx.x >> 5] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int q = 0; q < K; ++q) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < kT / 32; ++w) t += sm[q][w];
      part[(int64_t)q * gridDim.x + blockIdx.x] = t;
    }
  }
}
__device__ __forceinline__ void block_partial(double v, double* __restrict__ part) {
  const double a[1] = {v};
  block_partial<1>(a, part);
}
__device__ __forceinline__ bool on(unsigned mask, int q) { return (mask >> q) & 1u; }

__device__ __forceinline__ double dot2(double2 a, double2 b) { return fma(a.x, b.x, a.y * b.y); }

// scaled <-> unscaled per vertex: S = [[i00, i10], [0, i11]] (dscale = (i00, i11), scoup = i10)
__device__ __forceinline__ double2 mul_S(const double* ds, const double* sc, int64_t row, double2 v) {
  return make_double2(fma(sc[row], v.y, ds[2 * row] * v.x), ds[2 * row + 1] * v.y);
}
__device__ __forceinline__ double2 mul_St(const double* ds, const double* sc, int64_t row, double2 v) {
  return make_double2(ds[2 * row] * v.x, fma(sc[row], v.x, ds[2 * row + 1] * v.y));
}
__device__ __forceinline__ double2 solve_S(const double* ds, const double* sc, int64_t row, double2 v) {   // S^-1 v
  const double y = v.y / ds[2 * row + 1];
  return make_double2((v.x - sc[row] * y) / ds[2 * row], y);
}
__device__ __forceinline__ double2 solve_St(const double* ds, const double* sc, int64_t row, double2 v) {  // S^-T v
  const double x = v.x / ds[2 * row];
  return make_double2(x, (v.y - sc[row] * x) / ds[2 * row + 1]);
}

// ---------------------------------------------------------------------------------------------------------
// hierarchy: level l (fine) -> level l-1 (coarse), one thread per coarse cell
// flag[0]: error bits (1 structure / index / region, 2 a midpoint with two different edges, 4 a midpoint not
// at 0.5*(a+b), 8 vertex numbering not "coarse vertices, then midpoints"); flag[1]: largest coarse vertex id
__global__ void k_mg_derive(int64_t nc, int64_t nvf, const int32_t* __restrict__ conn_f, const int32_t* __restrict__ creg_f,
                            const double* __restrict__ xy, int32_t* __restrict__ conn_c, int32_t* __restrict__ creg_c,
                            int8_t* __restrict__ creg8_c, unsigned long long* __restrict__ key, int32_t* __restrict__ flag) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nc) return;
  const int32_t* c0 = conn_f + 3 * p;
  const int32_t* c1 = conn_f + 3 * (p + nc);
  const int32_t* c2 = conn_f + 3 * (p + 2 * nc);
  const int32_t* c3 = conn_f + 3 * (p + 3 * nc);
  const int a = c0[0], ab = c0[1], ca = c0[2], b = c1[1], bc = c1[2], c = c2[2];
  bool ok = c1[0] == ab && c2[0] == ca && c2[1] == bc && c3[0] == ab && c3[1] == bc && c3[2] == ca;
  const int r = creg_f[p];
  ok = ok && creg_f[p + nc] == r && creg_f[p + 2 * nc] == r && creg_f[p + 3 * nc] == r;
  ok = ok && a != b && b != c && c != a;
  const int v6[6] = {a, b, c, ab, bc, ca};
#pragma unroll
  for (int i = 0; i < 6; ++i) ok = ok && v6[i] >= 0 && v6[i] < nvf;
  if (!ok) {
    atomicOr(flag, 1);
    return;
  }
  conn_c[3 * p] = a;
  conn_c[3 * p + 1] = b;
  conn_c[3 * p + 2] = c;
  creg_c[p] = r;
  creg8_c[p] = (int8_t)r;
  atomicMax(flag + 1, max(a, max(b, c)));
  const int mids[3] = {ab, bc, ca}, e0[3] = {a, b, c}, e1[3] = {b, c, a};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int m = mids[i], u = min(e0[i], e1[i]), w = max(e0[i], e1[i]);
    const unsigned long long k = ((unsigned long long)(unsigned)u << 32) | (unsigned)w;
    const unsigned long long old = atomicCAS(key + m, kNoKey, k);
    if (old != kNoKey && old != k) atomicOr(flag, 2);
    if (!(xy[2 * (int64_t)m] == 0.5 * (xy[2 * (int64_t)u] + xy[2 * (int64_t)w]) &&
          xy[2 * (int64_t)m + 1] == 0.5 * (xy[2 * (int64_t)u + 1] + xy[2 * (int64_t)w + 1])))
      atomicOr(flag, 4);
  }
}

// vertices below n_c are the coarse level's, every other one is the midpoint of exactly one coarse edge;
// par[v] = (v, -1) or the edge; cnt[u] += 1 for both ends u of each midpoint
__global__ void k_mg_parents(int64_t nvf, int n_c, const unsigned long long* __restrict__ key, int2* __restrict__ par,
                             int32_t* __restrict__ cnt, int32_t* __restrict__ flag) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf) return;
  const unsigned long long k = key[v];
  if (v < n_c) {
    if (k != kNoKey) atomicOr(flag, 8);
    par[v] = make_int2((int)v, -1);
    return;
  }
  if (k == kNoKey) {
    atomicOr(flag, 8);
    par[v] = make_int2(0, -1);
    return;
  }
  const int u = (int)(k >> 32), w = (int)(k & 0xffffffffu);
  par[v] = make_int2(u, w);
  atomicAdd(cnt + u, 1);
  atomicAdd(cnt + w, 1);
}

__global__ void k_mg_child_fill(int64_t nvf, int n_c, const int2* __restrict__ par, const int32_t* __restrict__ ptr,
                                int32_t* __restrict__ cur, int32_t* __restrict__ child) {
  const int64_t v = n_c + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nvf) return;
  const int2 pr = par[v];
  if (pr.y < 0) return;   // not a midpoint (rejected before this kernel runs)
  child[ptr[pr.x] + atomicAdd(cur + pr.x, 1)] = (int)v;
  child[ptr[pr.y] + atomicAdd(cur + pr.y, 1)] = (int)v;
}

__global__ void k_mg_child_sort(int n_c, const int32_t* __restrict__ ptr, int32_t* __restrict__ child) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_c) return;
  const int b = ptr[v], e = ptr[v + 1];
  for (int i = b + 1; i < e; ++i) {   // insertion sort: a few entries per vertex
    const int t = child[i];
    int j = i - 1;
    while (j >= b && child[j] > t) {
      child[j + 1] = child[j];
      --j;
    }
    child[j + 1] = t;
  }
}

// Galerkin 6x6 matrices of level l-1 (orientation-fixed conn_c) from level l's (conn_f), one thread per coarse cell
__global__ void k_mg_galerkin(int64_t nc, const int32_t* __restrict__ conn_f, const double* __restrict__ ke_f,
                              const uint8_t* __restrict__ fixed_f, const int2* __restrict__ par_f,
                              const int32_t* __restrict__ conn_c, double* __restrict__ ke_c) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nc) return;
  const int C0 = conn_c[3 * p], C1 = conn_c[3 * p + 1], C2 = conn_c[3 * p + 2];
  double K[36];
#pragma unroll
  for (int i = 0; i < 36; ++i) K[i] = 0.0;
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    const int64_t cell = p + k * nc;
    double W[3][3];   // W[a][j]: weight of coarse node j in fine node a (0 at DOFs fixed on the fine level)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const int f = conn_f[3 * cell + a];
      const int2 pr = par_f[f];
      const double wx = fixed_f[f] ? 0.0 : (pr.y < 0 ? 1.0 : 0.5), wy = (fixed_f[f] || pr.y < 0) ? 0.0 : 0.5;
      W[a][0] = (C0 == pr.x ? wx : 0.0) + (C0 == pr.y ? wy : 0.0);
      W[a][1] = (C1 == pr.x ? wx : 0.0) + (C1 == pr.y ? wy : 0.0);
      W[a][2] = (C2 == pr.x ? wx : 0.0) + (C2 == pr.y ? wy : 0.0);
    }
    const double* Ke = ke_f + cell * 36;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int bb = 0; bb < 3; ++bb) {
        const double2 top = __ldg(reinterpret_cast<const double2*>(Ke + (2 * a) * 6 + 2 * bb));
        const double2 bot = __ldg(reinterpret_cast<const double2*>(Ke + (2 * a + 1) * 6 + 2 * bb));
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
          for (int j = 0; j < 3; ++j) {
            const double w = W[a][i] * W[bb][j];
            K[(2 * i) * 6 + 2 * j] = fma(w, top.x, K[(2 * i) * 6 + 2 * j]);
            K[(2 * i) * 6 + 2 * j + 1] = fma(w, top.y, K[(2 * i) * 6 + 2 * j + 1]);
            K[(2 * i + 1) * 6 + 2 * j] = fma(w, bot.x, K[(2 * i + 1) * 6 + 2 * j]);
            K[(2 * i + 1) * 6 + 2 * j + 1] = fma(w, bot.y, K[(2 * i + 1) * 6 + 2 * j + 1]);
          }
        }
      }
    }
  }
  double2* out = reinterpret_cast<double2*>(ke_c + p * 36);
#pragma unroll
  for (int i = 0; i < 18; ++i) out[i] = make_double2(K[2 * i], K[2 * i + 1]);
}

// ---------------------------------------------------------------------------------------------------------
// reductions: one block per case sums that case's partials in a fixed order, then updates its scalars (the
// kScCount slots from sc + case * kScCount; out, if given, advances by the same stride).  Cases outside
// `mask` are left alone; bit q of `first` is case q's first-iteration flag.
enum { kRedStore = 0, kRedDots = 1, kRedPQ = 2 };
__global__ void __launch_bounds__(1024) k_mg_reduce(const double* __restrict__ pa, const double* __restrict__ pb, int n,
                                                    double* __restrict__ sc, int mode, double* __restrict__ out,
                                                    unsigned first_bits, unsigned mask) {
  __shared__ double sa[32], sb[32];
  const int q = blockIdx.x;
  if (!on(mask, q)) return;
  pa += (int64_t)q * n;
  if (pb) pb += (int64_t)q * n;
  sc += q * kScCount;
  out += q * kScCount;
  const int first = on(first_bits, q);
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < n; i += 1024) {
    a += pa[i];
    if (pb) b += pb[i];
  }
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) {
    sa[threadIdx.x >> 5] = a;
    sb[threadIdx.x >> 5] = b;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double ta = 0.0, tb = 0.0;
  for (int w = 0; w < 32; ++w) {
    ta += sa[w];
    tb += sb[w];
  }
  if (mode == kRedStore) {
    *out = ta;
  } else if (mode == kRedDots) {   // ta = z.r, tb = z.q (q of the previous iteration)
    sc[kScBeta] = first ? 0.0 : -sc[kScAlpha] * tb / sc[kScRZ];
    sc[kScRZ] = ta;
  } else {                         // ta = p.q
    sc[kScPQ] = ta;
    sc[kScAlpha] = sc[kScRZ] / ta;
  }
}

// Lanczos estimate of lambda_max: v_0 random (partials of v.v), then per step
//   w = Khat v (partials of v.w -> alpha),  w -= alpha v + beta_prev v_prev (partials of w.w -> beta^2),
//   v_prev = v, v = w / beta
__global__ void __launch_bounds__(kT) k_mg_lz_init(const int32_t* __restrict__ vertex_of_row, double2* __restrict__ v,
                                                   double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int vx = vertex_of_row[row];
  double2 o = make_double2(0.0, 0.0);
  if (vx >= 0) {
    uint32_t h = (uint32_t)vx * 0x9E3779B9u + 0x7F4A7C15u;
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    o = make_double2((double)(h & 0xffff) / 32768.0 - 1.0, (double)(h >> 16) / 32768.0 - 1.0);
  }
  v[row] = o;
  block_partial(dot2(o, o), part);
}
__global__ void __launch_bounds__(kT) k_mg_lz_apply(MgOp A, const double2* __restrict__ v, double2* __restrict__ w,
                                                    double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double2 t[1];
  khat_row<1>(A, row, v, t);
  w[row] = t[0];
  block_partial(dot2(v[row], t[0]), part);
}
__global__ void __launch_bounds__(kT) k_mg_lz_orth(const double2* __restrict__ v, const double2* __restrict__ vp,
                                                   double2* __restrict__ w, const double* __restrict__ alpha,
                                                   const double* __restrict__ beta2_prev, double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double a = *alpha;
  const double2 vv = v[row];
  double2 t = w[row];
  t.x -= a * vv.x;
  t.y -= a * vv.y;
  if (beta2_prev) {   // not in the first step: v_prev is not a Lanczos vector yet
    const double bp = sqrt(*beta2_prev);
    const double2 pv = vp[row];
    t.x -= bp * pv.x;
    t.y -= bp * pv.y;
  }
  w[row] = t;
  block_partial(dot2(t, t), part);
}
__global__ void __launch_bounds__(kT) k_mg_lz_next(double2* __restrict__ v, double2* __restrict__ vp, const double2* __restrict__ w,
                                                   const double* __restrict__ norm2) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double s = *norm2 > 0.0 ? 1.0 / sqrt(*norm2) : 0.0;
  const double2 t = w[row];
  vp[row] = v[row];
  v[row] = make_double2(s * t.x, s * t.y);
}

// ---------------------------------------------------------------------------------------------------------
// V-cycle kernels of one level, K columns (state: x, r, d where d is not yet added to x)
// Chebyshev step: x += d_in; r -= Khat d_in; d_out = c1 d_in + c2 r.  The last step of the pre-smoother
// (d_out == nullptr) leaves the unscaled residual S^-T r in ru for the restriction instead.
template <int K>
__global__ void __launch_bounds__(kT) k_mg_cheb_step(MgOp A, const double2* __restrict__ din, double2* __restrict__ dout,
                                                     double2* __restrict__ x, double2* __restrict__ r, double c1, double c2,
                                                     const double* __restrict__ ds, const double* __restrict__ scp,
                                                     double2* __restrict__ ru) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double2 ad[K];
  khat_row<K>(A, row, din, ad);
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 d = din[i];
    double2 xv = x[i], rv = r[i];
    xv.x += d.x;
    xv.y += d.y;
    rv.x -= ad[q].x;
    rv.y -= ad[q].y;
    x[i] = xv;
    r[i] = rv;
    if (dout) dout[i] = make_double2(fma(c1, d.x, c2 * rv.x), fma(c1, d.y, c2 * rv.y));
    else ru[i] = ds[2 * row] > 0.0 ? solve_St(ds, scp, row, rv) : make_double2(0.0, 0.0);   // padding rows: 0
  }
}
// after the coarse correction: r = b - Khat x, d = r / theta
template <int K>
__global__ void __launch_bounds__(kT) k_mg_resid(MgOp A, const double2* __restrict__ x, const double2* __restrict__ b,
                                                 double2* __restrict__ r, double2* __restrict__ d, double inv_theta) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double2 ax[K];
  khat_row<K>(A, row, x, ax);
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 bv = b[i];
    const double2 rv = make_double2(bv.x - ax[q].x, bv.y - ax[q].y);
    r[i] = rv;
    d[i] = make_double2(rv.x * inv_theta, rv.y * inv_theta);
  }
}
template <int K>
__global__ void __launch_bounds__(kT) k_mg_add(double2* __restrict__ x, const double2* __restrict__ d) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 a = x[i], b = d[i];
    x[i] = make_double2(a.x + b.x, a.y + b.y);
  }
}
// entry of the finest level: r = b, d = b / theta, x = 0; a column outside `mask` (a finished case) enters
// with b = 0, so its coarse system is zero and it costs the coarse solve nothing
template <int K>
__global__ void __launch_bounds__(kT) k_mg_top_init(const double2* __restrict__ b, double2* __restrict__ x,
                                                    double2* __restrict__ r, double2* __restrict__ d, double inv_theta,
                                                    unsigned mask) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 bv = on(mask, q) ? b[i] : make_double2(0.0, 0.0);
    r[i] = bv;
    d[i] = make_double2(bv.x * inv_theta, bv.y * inv_theta);
    x[i] = make_double2(0.0, 0.0);
  }
}

struct Side {   // one level's maps and scaling
  const int32_t* vertex_of_row;
  const int32_t* row_of_vertex;
  const double* dscale;
  const double* scoup;
};
Side side_of(const Batch& b) { return Side{b.vertex_of_row, b.row_of_vertex, b.dscale, b.scoup}; }

// Where column k of a coarse-level vector lives.  A smoothed level interleaves: (row, k) at row * K + k.
// The coarsest level is a batch with one sample per case, each a copy of level 0: case k's row r is row
// r + k * rows_per_sample of that batch, and its vertex v is vertex v + k * n_vertices (the restriction writes
// the batch's rhs by vertex).
struct ColMap {
  int64_t row_stride, col_stride;
};

// restriction, one thread per coarse row: r_c = P^T S_f^-T r^_f at the coarse vertex (ru = S_f^-T r^_f).  Into a smoothed level:
// b = r = S_c^T r_c, d = b / theta, x = 0; into the coarsest level: its unscaled load vector rhs[vertex].
template <int K>
__global__ void __launch_bounds__(kT) k_mg_restrict(Side F, Side Cs, const double2* __restrict__ ru,
                                                    const int32_t* __restrict__ child_ptr, const int32_t* __restrict__ child,
                                                    double2* __restrict__ bc, double2* __restrict__ xc, double2* __restrict__ rc,
                                                    double2* __restrict__ dc, double inv_theta, double2* __restrict__ rhs0,
                                                    int64_t rhs0_stride) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int j = Cs.vertex_of_row[row];
  double2 acc[K];
#pragma unroll
  for (int q = 0; q < K; ++q) acc[q] = make_double2(0.0, 0.0);
  if (j >= 0) {
    const int fr = F.row_of_vertex[j];
    if (fr >= 0) {
#pragma unroll
      for (int q = 0; q < K; ++q) acc[q] = ru[(int64_t)fr * K + q];
    }
    for (int i = child_ptr[j]; i < child_ptr[j + 1]; ++i) {
      const int m = child[i];
      const int mr = F.row_of_vertex[m];
      if (mr < 0) continue;
#pragma unroll
      for (int q = 0; q < K; ++q) {
        const double2 t = ru[(int64_t)mr * K + q];
        acc[q].x = fma(0.5, t.x, acc[q].x);
        acc[q].y = fma(0.5, t.y, acc[q].y);
      }
    }
  }
  if (rhs0) {
    if (j >= 0) {
#pragma unroll
      for (int q = 0; q < K; ++q) rhs0[j + q * rhs0_stride] = acc[q];
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 h = j >= 0 ? mul_St(Cs.dscale, Cs.scoup, row, acc[q]) : make_double2(0.0, 0.0);
    bc[i] = h;
    rc[i] = h;
    dc[i] = make_double2(h.x * inv_theta, h.y * inv_theta);
    xc[i] = make_double2(0.0, 0.0);
  }
}

// prolongation-add, one thread per fine row: x^_f += S_f^-1 P S_c x^_c (Cs: the coarse level's maps and scaling;
// column k of its row r at xc[r * cm.row_stride + k * cm.col_stride])
template <int K>
__global__ void __launch_bounds__(kT) k_mg_prolong(Side F, Side Cs, const int2* __restrict__ par, const double2* __restrict__ xc,
                                                   ColMap cm, double2* __restrict__ xf) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int f = F.vertex_of_row[row];
  if (f < 0) return;
  const int2 pr = par[f];
  double2 e[K];
#pragma unroll
  for (int q = 0; q < K; ++q) e[q] = make_double2(0.0, 0.0);
  const int r0 = Cs.row_of_vertex[pr.x];
  const double w = pr.y < 0 ? 1.0 : 0.5;
  if (r0 >= 0) {
#pragma unroll
    for (int q = 0; q < K; ++q) {
      const double2 t = mul_S(Cs.dscale, Cs.scoup, r0, xc[r0 * cm.row_stride + q * cm.col_stride]);
      e[q] = make_double2(w * t.x, w * t.y);
    }
  }
  if (pr.y >= 0) {
    const int r1 = Cs.row_of_vertex[pr.y];
    if (r1 >= 0) {
#pragma unroll
      for (int q = 0; q < K; ++q) {
        const double2 t = mul_S(Cs.dscale, Cs.scoup, r1, xc[r1 * cm.row_stride + q * cm.col_stride]);
        e[q].x = fma(0.5, t.x, e[q].x);
        e[q].y = fma(0.5, t.y, e[q].y);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const double2 c = solve_S(F.dscale, F.scoup, row, e[q]);
    double2 xv = xf[row * K + q];
    xv.x += c.x;
    xv.y += c.y;
    xf[row * K + q] = xv;
  }
}

// non-nested hierarchies (k_mg_nonnested.cu): the same two transfers with up to 3 weighted parents per vertex.
// Restriction gathers over a coarse vertex's (fine vertex, weight) list, ascending in the fine vertex.
template <int K>
__global__ void __launch_bounds__(kT) k_mgn_restrict(Side F, Side Cs, const double2* __restrict__ ru,
                                                     const int32_t* __restrict__ child_ptr, const int32_t* __restrict__ child,
                                                     const double* __restrict__ child_w, double2* __restrict__ bc,
                                                     double2* __restrict__ xc, double2* __restrict__ rc, double2* __restrict__ dc,
                                                     double inv_theta, double2* __restrict__ rhs0, int64_t rhs0_stride) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int j = Cs.vertex_of_row[row];
  double2 acc[K];
#pragma unroll
  for (int q = 0; q < K; ++q) acc[q] = make_double2(0.0, 0.0);
  if (j >= 0) {
    for (int i = child_ptr[j]; i < child_ptr[j + 1]; ++i) {
      const int fr = F.row_of_vertex[child[i]];
      if (fr < 0) continue;
      const double w = child_w[i];
#pragma unroll
      for (int q = 0; q < K; ++q) {
        const double2 t = ru[(int64_t)fr * K + q];
        acc[q].x = fma(w, t.x, acc[q].x);
        acc[q].y = fma(w, t.y, acc[q].y);
      }
    }
  }
  if (rhs0) {
    if (j >= 0) {
#pragma unroll
      for (int q = 0; q < K; ++q) rhs0[j + q * rhs0_stride] = acc[q];
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const int64_t i = row * K + q;
    const double2 h = j >= 0 ? mul_St(Cs.dscale, Cs.scoup, row, acc[q]) : make_double2(0.0, 0.0);
    bc[i] = h;
    rc[i] = h;
    dc[i] = make_double2(h.x * inv_theta, h.y * inv_theta);
    xc[i] = make_double2(0.0, 0.0);
  }
}
template <int K>
__global__ void __launch_bounds__(kT) k_mgn_prolong(Side F, Side Cs, const int32_t* __restrict__ par3, const double* __restrict__ w3,
                                                    const double2* __restrict__ xc, ColMap cm, double2* __restrict__ xf) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int f = F.vertex_of_row[row];
  if (f < 0) return;
  double2 e[K];
#pragma unroll
  for (int q = 0; q < K; ++q) e[q] = make_double2(0.0, 0.0);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int p = par3[3 * (int64_t)f + k];
    if (p < 0) continue;
    const int r = Cs.row_of_vertex[p];
    if (r < 0) continue;   // a Dirichlet vertex of the coarse level: no column
    const double w = w3[3 * (int64_t)f + k];
#pragma unroll
    for (int q = 0; q < K; ++q) {
      const double2 t = mul_S(Cs.dscale, Cs.scoup, r, xc[r * cm.row_stride + q * cm.col_stride]);
      e[q].x = fma(w, t.x, e[q].x);
      e[q].y = fma(w, t.y, e[q].y);
    }
  }
#pragma unroll
  for (int q = 0; q < K; ++q) {
    const double2 c = solve_S(F.dscale, F.scoup, row, e[q]);
    double2 xv = xf[row * K + q];
    xv.x += c.x;
    xv.y += c.y;
    xf[row * K + q] = xv;
  }
}

// ---------------------------------------------------------------------------------------------------------
// outer flexible CG on the finest level, K cases; x, r, p and q change only in the columns of `mask` (the cases
// still iterating), so a finished case keeps its last iterate and its p and q
// r = S^T b (mode 0) or S^T b - Khat x (modes 1, 2); mode 0 also clears x, modes 0 and 2 (a restart) p and q.
// b of case k: the full-DOF load rhs + k * rhs_stride.  Partials of r.r.
template <int K>
__global__ void __launch_bounds__(kT) k_mg_fcg_residual(MgOp A, Side F, const double* __restrict__ rhs, int64_t rhs_stride,
                                                        double2* __restrict__ x, double2* __restrict__ r, double2* __restrict__ p,
                                                        double2* __restrict__ q, int mode, unsigned mask, double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int v = F.vertex_of_row[row];
  double2 bv[K];
#pragma unroll
  for (int c = 0; c < K; ++c) {
    bv[c] = make_double2(0.0, 0.0);
    const double* rc = rhs + c * rhs_stride;
    if (v >= 0) bv[c] = mul_St(F.dscale, F.scoup, row, make_double2(rc[2 * (int64_t)v], rc[2 * (int64_t)v + 1]));
  }
  if (mode) {
    double2 ax[K];
    khat_row<K>(A, row, x, ax);
#pragma unroll
    for (int c = 0; c < K; ++c) {
      bv[c].x -= ax[c].x;
      bv[c].y -= ax[c].y;
    }
  }
  double rr[K];
#pragma unroll
  for (int c = 0; c < K; ++c) {
    const int64_t i = row * K + c;
    if (on(mask, c)) {
      if (!mode) x[i] = make_double2(0.0, 0.0);
      if (mode != 1) {   // (re)start: p = q = 0
        p[i] = make_double2(0.0, 0.0);
        q[i] = make_double2(0.0, 0.0);
      }
      r[i] = bv[c];
    }
    rr[c] = dot2(bv[c], bv[c]);
  }
  block_partial<K>(rr, part);
}
template <int K>
__global__ void __launch_bounds__(kT) k_mg_fcg_dots(const double2* __restrict__ z, const double2* __restrict__ r,
                                                    const double2* __restrict__ q, double* __restrict__ pa, double* __restrict__ pb) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double zr[K], zq[K];
#pragma unroll
  for (int c = 0; c < K; ++c) {
    const int64_t i = row * K + c;
    const double2 zv = z[i];
    zr[c] = dot2(zv, r[i]);
    zq[c] = dot2(zv, q[i]);
  }
  block_partial<K>(zr, pa);
  __syncthreads();
  block_partial<K>(zq, pb);
}
template <int K>
__global__ void __launch_bounds__(kT) k_mg_fcg_dir(const double2* __restrict__ z, double2* __restrict__ p, const double* __restrict__ sc,
                                                   unsigned mask) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
#pragma unroll
  for (int c = 0; c < K; ++c) {
    if (!on(mask, c)) continue;
    const int64_t i = row * K + c;
    const double beta = sc[c * kScCount + kScBeta];
    const double2 zv = z[i], pv = p[i];
    p[i] = make_double2(fma(beta, pv.x, zv.x), fma(beta, pv.y, zv.y));
  }
}
template <int K>
__global__ void __launch_bounds__(kT) k_mg_fcg_spmv(MgOp A, const double2* __restrict__ p, double2* __restrict__ q,
                                                    unsigned mask, double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double2 qv[K];
  khat_row<K>(A, row, p, qv);
  double pq[K];
#pragma unroll
  for (int c = 0; c < K; ++c) {
    const int64_t i = row * K + c;
    if (on(mask, c)) q[i] = qv[c];
    pq[c] = dot2(p[i], qv[c]);
  }
  block_partial<K>(pq, part);
}
template <int K>
__global__ void __launch_bounds__(kT) k_mg_fcg_update(double2* __restrict__ x, double2* __restrict__ r, const double2* __restrict__ p,
                                                      const double2* __restrict__ q, const double* __restrict__ sc, unsigned mask,
                                                      double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  double rr[K];
#pragma unroll
  for (int c = 0; c < K; ++c) {
    const int64_t i = row * K + c;
    const double alpha = sc[c * kScCount + kScAlpha], pq = sc[c * kScCount + kScPQ];
    double2 rv = r[i];
    // p.q <= 0 or a non-finite step: breakdown (the host stops the case), x and r keep the last sound iterate
    if (on(mask, c) && pq > 0.0 && isfinite(pq) && isfinite(alpha)) {
      const double2 pv = p[i], qv = q[i];
      double2 xv = x[i];
      xv.x = fma(alpha, pv.x, xv.x);
      xv.y = fma(alpha, pv.y, xv.y);
      rv.x = fma(-alpha, qv.x, rv.x);
      rv.y = fma(-alpha, qv.y, rv.y);
      x[i] = xv;
      r[i] = rv;
    }
    rr[c] = dot2(rv, rv);
  }
  block_partial<K>(rr, part);
}
// what launch_finalize and fea_batch_download read, per case
struct CaseInts {
  int32_t v[kMaxCases];
};
__global__ void k_mg_finish(int n, int32_t* __restrict__ status, int32_t* __restrict__ iters, double* __restrict__ rz0,
                            double* __restrict__ rz_last, const double* __restrict__ sc, CaseInts st, CaseInts it) {
  const int c = threadIdx.x;
  if (blockIdx.x != 0 || c >= n) return;
  status[c] = st.v[c];
  iters[c] = it.v[c];
  rz0[c] = sc[c * kScCount + kScRZ0];
  rz_last[c] = sc[c * kScCount + kScTrue];
}
// column c of a K-column vector, contiguous (the layout launch_finalize_to reads)
__global__ void __launch_bounds__(kT) k_mg_column(const double2* __restrict__ v, int K, int c, double2* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  out[row] = v[row * K + c];
}

// active-DOF vector (unscaled) <-> scaled rows of the finest level
__global__ void __launch_bounds__(kT) k_mg_load(Side F, const int32_t* __restrict__ vrank, const double* __restrict__ in,
                                                double2* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int v = F.vertex_of_row[row];
  double2 o = make_double2(0.0, 0.0);
  if (v >= 0) {
    const int k = vrank[v];
    o = mul_St(F.dscale, F.scoup, row, make_double2(in[2 * (int64_t)k], in[2 * (int64_t)k + 1]));
  }
  out[row] = o;
}
__global__ void __launch_bounds__(kT) k_mg_store(Side F, const int32_t* __restrict__ vrank, const double2* __restrict__ in,
                                                 double* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int v = F.vertex_of_row[row];
  if (v < 0) return;
  const int k = vrank[v];
  const double2 o = mul_S(F.dscale, F.scoup, row, in[row]);
  out[2 * (int64_t)k] = o.x;
  out[2 * (int64_t)k + 1] = o.y;
}

unsigned grid_rows(const Batch& b) { return (unsigned)(b.NBR / kT); }

// the partials of n CTAs per case into the scalars sc of the cases in `mask` (slot: kRedStore's destination)
cudaError_t reduce(const Batch& fine, double* sc, int n_cases, const double* pa, const double* pb, int n, int mode,
                   int slot = 0, unsigned first = 0, unsigned mask = 1, double* out = nullptr) {
  k_mg_reduce<<<n_cases, 1024, 0, fine.ctx->stream>>>(pa, pb, n, sc, mode, out ? out : sc + slot, first, mask);
  return cudaGetLastError();
}

// largest eigenvalue of a symmetric tridiagonal matrix (diagonal a, off-diagonal b) by Sturm-count bisection
double tridiag_max(const std::vector<double>& a, const std::vector<double>& b) {
  const int m = (int)a.size();
  double lo = 0.0, hi = 0.0;
  for (int i = 0; i < m; ++i) {
    const double r = (i > 0 ? fabs(b[i - 1]) : 0.0) + (i + 1 < m ? fabs(b[i]) : 0.0);
    lo = i ? std::min(lo, a[i] - r) : a[i] - r;
    hi = i ? std::max(hi, a[i] + r) : a[i] + r;
  }
  for (int it = 0; it < 200 && hi - lo > 1e-14 * fabs(hi); ++it) {
    const double mid = 0.5 * (lo + hi);
    int below = 0;   // eigenvalues < mid
    double q = a[0] - mid;
    for (int i = 0; i < m; ++i) {
      if (i > 0) q = a[i] - mid - b[i - 1] * b[i - 1] / q;
      if (q == 0.0) q = -1e-300;
      below += q < 0.0;
    }
    if (below == m) hi = mid; else lo = mid;
  }
  return hi;
}

// largest eigenvalue of level L's Khat: the top Ritz value of kLanczos Lanczos steps.  v, vp, w [NBR] and
// part [NBR/kT] are sized to the finest level, sc holds kScCount + 2 kLanczos scalars.  15 power iterations,
// the cheaper alternative, stay at 2.03-2.07 on the C3 meshes where Lanczos finds 2.34-2.39 (true 2.36-2.42):
// the smoother would then amplify the top of the spectrum.
cudaError_t estimate_lmax(Batch& fine, MgLevel& L, double2* v, double2* vp, double2* w, double* part, double* sc) {
  cudaStream_t st = fine.ctx->stream;
  const Batch& b = *L.b;
  const unsigned g = grid_rows(b);
  if (!g) return cudaSuccess;
  double* lz = sc + kScCount;   // [2 kLanczos]: alpha_k, beta_k^2
  k_mg_lz_init<<<g, kT, 0, st>>>(b.vertex_of_row, w, part);
  cudaError_t e = reduce(fine, sc, 1, part, nullptr, (int)g, kRedStore, kScNrm);
  if (e == cudaSuccess) k_mg_lz_next<<<g, kT, 0, st>>>(v, vp, w, sc + kScNrm);
  for (int k = 0; k < kLanczos && e == cudaSuccess; ++k) {
    k_mg_lz_apply<<<g, kT, 0, st>>>(op_of(b), v, w, part);
    e = reduce(fine, sc, 1, part, nullptr, (int)g, kRedStore, 0, 0, 1, lz + 2 * k);
    k_mg_lz_orth<<<g, kT, 0, st>>>(v, vp, w, lz + 2 * k, k ? lz + 2 * k - 1 : nullptr, part);
    if (e == cudaSuccess) e = reduce(fine, sc, 1, part, nullptr, (int)g, kRedStore, 0, 0, 1, lz + 2 * k + 1);
    k_mg_lz_next<<<g, kT, 0, st>>>(v, vp, w, lz + 2 * k + 1);
  }
  std::vector<double> h(2 * kLanczos, 0.0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h.data(), lz, sizeof(double) * 2 * kLanczos, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  fine.ctx->launches += 3 + 5 * kLanczos;
  std::vector<double> al, be;
  for (int k = 0; k < kLanczos; ++k) {   // stop at a breakdown (an invariant subspace: its Ritz values are exact)
    al.push_back(h[2 * k]);
    if (!(h[2 * k + 1] > 0.0) || k == kLanczos - 1) break;
    be.push_back(sqrt(h[2 * k + 1]));
  }
  L.lmax = tridiag_max(al, be);
  // Chebyshev over [lmax/30, 1.1 lmax]: d_0 = r_0/theta, d_k = rho_k rho_(k-1) d_(k-1) + (2 rho_k / delta) r_k
  const double hi = 1.1 * L.lmax, lo = L.lmax / 30.0;
  const double theta = 0.5 * (hi + lo), delta = 0.5 * (hi - lo), sigma = theta / delta;
  double rho = 1.0 / sigma;
  L.inv_theta = 1.0 / theta;
  for (int k = 0; k < 2; ++k) {
    const double rn = 1.0 / (2.0 * sigma - rho);
    L.c1[k] = rn * rho;
    L.c2[k] = 2.0 * rn / delta;
    rho = rn;
  }
  return e;
}

// Column groups.  The kernels run on at most kGroup columns at once: K <= kGroup cases are one group, more are
// split into two groups of ceil(K/2) and floor(K/2).  A K-column vector over n block rows holds group (c0, G) at
// v + c0 * n, interleaved G columns per row.  Measured on a B200 (plate at h = 0.000625, 18 V-cycles): a
// single 8-column group ran the finest level 7.8x slower than one column, 4 columns 2.45x (DESIGN.md section
// 3.11).  A group's columns do the K = 1 arithmetic, so the split changes no bit.
constexpr int kGroup = 4;
constexpr int groups_of(int K) { return K > kGroup ? 2 : 1; }
template <int K, class F>
void each_group(F&& f) {
  constexpr int G0 = K <= kGroup ? K : (K + 1) / 2;
  f(std::integral_constant<int, G0>{}, 0);
  if constexpr (K > G0) f(std::integral_constant<int, K - G0>{}, G0);
}
template <class T>
T* at(T* v, int64_t n, int c0) { return v ? v + c0 * n : v; }

// The vectors of one call on K cases (make_work): a solve, a V-cycle of fea_batch_mg_apply (K = 1).  The
// coarsest systems are those of a batch: level 0's own for K = 1, K copies of level 0 for K > 1.
struct Vecs {
  double2 *x = nullptr, *bv = nullptr, *r = nullptr, *d[2] = {nullptr, nullptr};
};
struct Work {
  std::vector<Vecs> v;                    // [levels + 1]: V-cycle state of levels >= 1
  double2 *x = nullptr, *r = nullptr, *p = nullptr, *q = nullptr;   // outer flexible CG, K columns in groups (at)
  double *partA = nullptr, *partB = nullptr;                        // [K][CTAs]
  double* sc = nullptr;                   // [K][kScCount]
  const double* rhs = nullptr;            // full-DOF loads, case k at rhs + k * rhs_stride
  int64_t rhs_stride = 0;
  Batch* coarse = nullptr;                // coarsest batch: its sample k solves case k
  ColMap coarse_map{1, 0};                // case k's rows in coarse->x
  int64_t coarse_nv = 0;                  // vertices per sample of the coarsest batch
};

// level 0's solver on the K systems of `coarse`, whose rhs holds case k's load by vertex at vertex k * nv_stride:
// the dense inverse, all K cases in one read of it, into coarse.x at cm; or block-Jacobi CG of the whole batch
cudaError_t coarse_solve(const Mg& mg, Batch& coarse, int K, int64_t nv_stride, ColMap cm, cudaStream_t st) {
  if (mg.coarse_solver == FEA_COARSE_DIRECT)
    return mg_direct_apply(mg, K, coarse.rhs, nv_stride, coarse.x, cm.row_stride, cm.col_stride, st);
  return run_pcg(coarse, kCoarseRtol, kCoarseMaxIter);
}

// one V-cycle from level l down; level l's b, r, d[0], x are set up by the caller (restriction / top init)
template <int K>
cudaError_t vcycle(fea_ctx* ctx, Batch& fine, Work& w, int l) {
  Mg& mg = *fine.mg;
  Ctx& c = ctx->c;
  cudaStream_t st = c.stream;
  MgLevel& L = mg.lev[l];
  cudaEvent_t* ev = mg.ev.data() + 4 * l;
  cudaError_t e;
  if (l == 0) {   // coarsest: the restricted residuals are in the coarsest batch's rhs
    if ((e = cudaEventRecord(ev[0], st)) != cudaSuccess) return e;
    e = coarse_solve(mg, *w.coarse, K, w.coarse_nv, w.coarse_map, st);
    if (mg.coarse_solver == FEA_COARSE_DIRECT) c.launches += 2;
    if (e != cudaSuccess) return e;
    return cudaEventRecord(ev[1], st);
  }
  const Batch& b = *L.b;
  MgLevel& C = mg.lev[l - 1];
  Vecs& V = w.v[l];
  Vecs& Cv = w.v[l - 1];   // unused below level 1: the coarsest batch holds its own vectors
  const unsigned g = grid_rows(b), gc = grid_rows(*C.b);
  const int64_t n = b.NBR, nc = C.b->NBR;
  const MgOp A = op_of(b);
  double2* rhs0 = l == 1 ? (double2*)w.coarse->rhs : nullptr;
  cudaEventRecord(ev[0], st);
  each_group<K>([&](auto width, int c0) {
    constexpr int G = decltype(width)::value;
    double2 *d0 = at(V.d[0], n, c0), *d1 = at(V.d[1], n, c0), *x = at(V.x, n, c0), *r = at(V.r, n, c0);
    k_mg_cheb_step<G><<<g, kT, 0, st>>>(A, d0, d1, x, r, L.c1[0], L.c2[0], nullptr, nullptr, nullptr);
    k_mg_cheb_step<G><<<g, kT, 0, st>>>(A, d1, d0, x, r, L.c1[1], L.c2[1], nullptr, nullptr, nullptr);
    k_mg_cheb_step<G><<<g, kT, 0, st>>>(A, d0, nullptr, x, r, 0.0, 0.0, b.dscale, b.scoup, d1);
    double2* r0 = rhs0 ? rhs0 + c0 * w.coarse_nv : nullptr;
    if (gc && mg.nonnested)
      k_mgn_restrict<G><<<gc, kT, 0, st>>>(side_of(b), side_of(*C.b), d1, L.child_ptr, L.child, L.child_w, at(Cv.bv, nc, c0),
                                           at(Cv.x, nc, c0), at(Cv.r, nc, c0), at(Cv.d[0], nc, c0), C.inv_theta, r0,
                                           w.coarse_nv);
    else if (gc)
      k_mg_restrict<G><<<gc, kT, 0, st>>>(side_of(b), side_of(*C.b), d1, L.child_ptr, L.child, at(Cv.bv, nc, c0),
                                          at(Cv.x, nc, c0), at(Cv.r, nc, c0), at(Cv.d[0], nc, c0), C.inv_theta, r0,
                                          w.coarse_nv);
  });
  cudaEventRecord(ev[1], st);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = vcycle<K>(ctx, fine, w, l - 1)) != cudaSuccess) return e;
  cudaEventRecord(ev[2], st);
  each_group<K>([&](auto width, int c0) {
    constexpr int G = decltype(width)::value;
    double2 *d0 = at(V.d[0], n, c0), *d1 = at(V.d[1], n, c0), *x = at(V.x, n, c0), *r = at(V.r, n, c0);
    const double2* xc = l == 1 ? (const double2*)w.coarse->x + c0 * w.coarse_map.col_stride : at(Cv.x, nc, c0);
    const ColMap cm = l == 1 ? w.coarse_map : ColMap{G, 1};
    if (mg.nonnested)
      k_mgn_prolong<G><<<g, kT, 0, st>>>(side_of(b), side_of(*C.b), L.par3, L.w3, xc, cm, x);
    else
      k_mg_prolong<G><<<g, kT, 0, st>>>(side_of(b), side_of(*C.b), L.par, xc, cm, x);
    k_mg_resid<G><<<g, kT, 0, st>>>(A, x, at(V.bv, n, c0), r, d0, L.inv_theta);
    k_mg_cheb_step<G><<<g, kT, 0, st>>>(A, d0, d1, x, r, L.c1[0], L.c2[0], nullptr, nullptr, nullptr);
    k_mg_cheb_step<G><<<g, kT, 0, st>>>(A, d1, d0, x, r, L.c1[1], L.c2[1], nullptr, nullptr, nullptr);
    k_mg_add<G><<<g, kT, 0, st>>>(x, d0);
  });
  cudaEventRecord(ev[3], st);
  c.launches += 9 * groups_of(K);
  return cudaGetLastError();
}

// z = V(rhs) on the finest level for the cases in `mask` (the others get z = V(0)): the result is in v[levels].x
template <int K>
cudaError_t vcycle_top(fea_ctx* ctx, Batch& fine, Work& w, const double2* rhs, unsigned mask) {
  Mg& mg = *fine.mg;
  Vecs& V = w.v[mg.levels];
  V.bv = const_cast<double2*>(rhs);
  const int64_t n = fine.NBR;
  each_group<K>([&](auto width, int c0) {
    constexpr int G = decltype(width)::value;
    k_mg_top_init<G><<<grid_rows(fine), kT, 0, ctx->c.stream>>>(rhs + c0 * n, at(V.x, n, c0), at(V.r, n, c0), at(V.d[0], n, c0),
                                                                 mg.lev[mg.levels].inv_theta, mask >> c0);
  });
  ctx->c.launches += groups_of(K);
  return vcycle<K>(ctx, fine, w, mg.levels);
}

void accumulate_level_ms(Mg& mg) {
  for (int l = 0; l <= mg.levels; ++l) {
    float a = 0.f, b = 0.f;
    cudaEvent_t* ev = mg.ev.data() + 4 * l;
    cudaEventElapsedTime(&a, ev[0], ev[1]);
    if (l > 0) cudaEventElapsedTime(&b, ev[2], ev[3]);
    mg.lev[l].ms += (double)a + (double)b;
  }
}

// device outputs of a solve, per case: what fea_batch_download reads (status, iters, rz0, r.r at exit, u,
// ranges, relres); col [NBR] holds one case's x for the finalize kernels when K > 1
struct Out {
  int32_t *status, *iters;
  double *rz0, *rz_last, *u, *ranges, *relres;
  double2* col;
};

// Flexible CG preconditioned by one V-cycle per iteration, for K cases at once.  Per case, every decision is
// that of a single solve: its own status, iteration count, first-iteration flag, restarts from the true residual
// (kMaxRestarts) and breakdown test.  A finished case is frozen (x and r no longer change, and it enters the
// V-cycle with a zero right-hand side); the loop ends when every case has finished.  One host poll per outer
// iteration serves all cases.
template <int K>
int solve(fea_ctx* ctx, Batch& b, Work& w, double rtol, int max_iter, const Out& o, fea_solve_stats& stats) {
  Mg& mg = *b.mg;
  Ctx& c = ctx->c;
  cudaStream_t st = c.stream;
  const unsigned g = grid_rows(b);
  const int np = (int)g;
  const MgOp A = op_of(b);
  const Side F = side_of(b);
  double* h = mg.h_sc;
  cudaEvent_t ev0 = mg.ev[4 * (mg.levels + 1)], ev1 = mg.ev[4 * (mg.levels + 1) + 1];
  const unsigned all = (1u << K) - 1;
  stats = fea_solve_stats{};
  for (auto& L : mg.lev) L.ms = 0.0;
  const int64_t launches0 = c.launches;
  CK(ctx, cudaEventRecord(ev0, st));
  int32_t empty = 0;
  CK(ctx, cudaMemcpyAsync(&empty, b.empty, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  const int64_t n = b.NBR;
  auto residual = [&](int mode, unsigned mask, int slot) -> cudaError_t {
    each_group<K>([&](auto width, int c0) {
      constexpr int G = decltype(width)::value;
      k_mg_fcg_residual<G><<<g, kT, 0, st>>>(A, F, w.rhs + c0 * w.rhs_stride, w.rhs_stride, at(w.x, n, c0), at(w.r, n, c0),
                                             at(w.p, n, c0), at(w.q, n, c0), mode, mask >> c0, w.partA + c0 * np);
    });
    return reduce(b, w.sc, K, w.partA, nullptr, np, kRedStore, slot, 0, mask);
  };
  auto poll = [&]() -> cudaError_t {
    cudaError_t e = cudaMemcpyAsync(h, w.sc, sizeof(double) * K * kScCount, cudaMemcpyDeviceToHost, st);
    return e == cudaSuccess ? cudaStreamSynchronize(st) : e;
  };
  CK(ctx, residual(0, all, kScRZ0));
  CK(ctx, poll());
  CaseInts status, it;
  int restarts[K], first[K];
  double rr[K], tol2[K], rz0[K];
  for (int q = 0; q < K; ++q) {
    const double* hq = h + q * kScCount;
    rz0[q] = hq[kScRZ0];
    tol2[q] = rtol * rtol * rz0[q];
    rr[q] = rz0[q];
    status.v[q] = FEA_SAMPLE_NOT_RUN;
    it.v[q] = restarts[q] = 0;
    first[q] = 1;
    if (empty) status.v[q] = FEA_SAMPLE_EMPTY_ROW;
    else if (!(rz0[q] > 0.0)) status.v[q] = std::isfinite(rz0[q]) ? FEA_SAMPLE_CONVERGED : FEA_SAMPLE_BREAKDOWN;
    if (status.v[q] == FEA_SAMPLE_CONVERGED)
      CK(ctx, cudaMemcpyAsync(w.sc + q * kScCount + kScTrue, &rz0[q], sizeof(double), cudaMemcpyHostToDevice, st));
  }
  for (;;) {
    // recursive residuals that met the tolerance: decide on the TRUE residual
    unsigned check = 0;
    for (int q = 0; q < K; ++q)
      if (status.v[q] == FEA_SAMPLE_NOT_RUN && rr[q] <= tol2[q]) check |= 1u << q;
    if (check) {
      CK(ctx, residual(2, check, kScTrue));
      CK(ctx, poll());
      c.launches += 2;
      for (int q = 0; q < K; ++q) {
        if (!((check >> q) & 1u)) continue;
        rr[q] = h[q * kScCount + kScTrue];
        if (rr[q] <= tol2[q]) status.v[q] = FEA_SAMPLE_CONVERGED;
        else if (!std::isfinite(rr[q])) status.v[q] = FEA_SAMPLE_BREAKDOWN;
        else if (++restarts[q] > kMaxRestarts) status.v[q] = FEA_SAMPLE_STAGNATED;
        else first[q] = 1;   // restart from the true residual (p = q = 0)
      }
    }
    unsigned act = 0, first_bits = 0;
    for (int q = 0; q < K; ++q) {
      if (status.v[q] != FEA_SAMPLE_NOT_RUN) continue;
      if (it.v[q] >= max_iter) {
        status.v[q] = FEA_SAMPLE_MAX_ITER;
        continue;
      }
      act |= 1u << q;
      if (first[q]) first_bits |= 1u << q;
    }
    if (!act) break;
    CK(ctx, vcycle_top<K>(ctx, b, w, w.r, act));
    const double2* z = w.v[mg.levels].x;
    each_group<K>([&](auto width, int c0) {
      constexpr int G = decltype(width)::value;
      k_mg_fcg_dots<G><<<g, kT, 0, st>>>(at(z, n, c0), at(w.r, n, c0), at(w.q, n, c0), w.partA + c0 * np, w.partB + c0 * np);
    });
    CK(ctx, reduce(b, w.sc, K, w.partA, w.partB, np, kRedDots, 0, first_bits, act));
    each_group<K>([&](auto width, int c0) {
      constexpr int G = decltype(width)::value;
      k_mg_fcg_dir<G><<<g, kT, 0, st>>>(at(z, n, c0), at(w.p, n, c0), w.sc + c0 * kScCount, act >> c0);
      k_mg_fcg_spmv<G><<<g, kT, 0, st>>>(A, at(w.p, n, c0), at(w.q, n, c0), act >> c0, w.partA + c0 * np);
    });
    CK(ctx, reduce(b, w.sc, K, w.partA, nullptr, np, kRedPQ, 0, 0, act));
    each_group<K>([&](auto width, int c0) {
      constexpr int G = decltype(width)::value;
      k_mg_fcg_update<G><<<g, kT, 0, st>>>(at(w.x, n, c0), at(w.r, n, c0), at(w.p, n, c0), at(w.q, n, c0),
                                           w.sc + c0 * kScCount, act >> c0, w.partA + c0 * np);
    });
    CK(ctx, reduce(b, w.sc, K, w.partA, nullptr, np, kRedStore, kScRR, 0, act));
    CK(ctx, poll());   // one host poll per outer iteration (the coarse solve polls anyway)
    c.launches += 4 + 4 * groups_of(K);
    accumulate_level_ms(mg);
    unsigned broke = 0;
    for (int q = 0; q < K; ++q) {
      if (!((act >> q) & 1u)) continue;
      const double* hq = h + q * kScCount;
      if (!(hq[kScPQ] > 0.0) || !std::isfinite(hq[kScPQ]) || !std::isfinite(hq[kScAlpha]) || !std::isfinite(hq[kScRR])) {
        // not SPD on this Krylov space (or a non-finite step): k_mg_fcg_update left x and r alone, so u and
        // relres are those of the last sound iterate
        status.v[q] = FEA_SAMPLE_BREAKDOWN;
        broke |= 1u << q;
        continue;
      }
      ++it.v[q];
      first[q] = 0;
      rr[q] = hq[kScRR];
    }
    if (broke) CK(ctx, residual(1, broke, kScTrue));
  }
  unsigned unfinished = 0;
  for (int q = 0; q < K; ++q)
    if (status.v[q] == FEA_SAMPLE_MAX_ITER || status.v[q] == FEA_SAMPLE_STAGNATED) unfinished |= 1u << q;
  if (unfinished) CK(ctx, residual(1, unfinished, kScTrue));
  k_mg_finish<<<1, 32, 0, st>>>(K, o.status, o.iters, o.rz0, o.rz_last, w.sc, status, it);
  CK(ctx, cudaGetLastError());
  for (int q = 0; q < K; ++q) {
    const double* xq = (const double*)w.x;
    if (K > 1) {
      each_group<K>([&](auto width, int c0) {
        constexpr int G = decltype(width)::value;
        if (q >= c0 && q < c0 + G) k_mg_column<<<g, kT, 0, st>>>(at(w.x, n, c0), G, q - c0, o.col);
      });
      xq = (const double*)o.col;
    }
    CK(ctx, launch_finalize_to(b, xq, o.status + q, o.rz_last + q, o.rz0 + q, o.u + 2 * b.NV * q, o.ranges + 4 * q,
                               o.relres + q));
  }
  CK(ctx, cudaEventRecord(ev1, st));
  CK(ctx, cudaStreamSynchronize(st));
  for (int q = 0; q < K; ++q) {
    stats.iterations = std::max(stats.iterations, it.v[q]);
    stats.n_converged += status.v[q] == FEA_SAMPLE_CONVERGED;
    stats.refined_systems += restarts[q] > 0;
  }
  cudaEventElapsedTime(&stats.solve_ms, ev0, ev1);
  c.launches += 1 + groups_of(K) + 3 * K + (K > 1 ? K : 0) + 3;
  stats.kernel_launches = c.launches - launches0;
  return FEA_OK;
}

// cells of level 0 replicated per case: case k's cell c is cell c of level 0 with its vertices shifted by
// k * vertex_shift; creg (if given) gets level 0's region as the int8 input of api_batch_finish
__global__ void k_mg_replicate_cells(int64_t nc, int n_cases, const int32_t* __restrict__ conn0, const int32_t* __restrict__ creg0,
                                     int64_t vertex_shift, int32_t* __restrict__ conn, int8_t* __restrict__ creg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nc * n_cases) return;
  const int k = (int)(i / nc);
  const int64_t cell = i - k * nc;
#pragma unroll
  for (int a = 0; a < 3; ++a) conn[3 * i + a] = (int32_t)(conn0[3 * cell + a] + k * vertex_shift);
  if (creg) creg[i] = (int8_t)creg0[cell];
}

// The coarsest batch of a solve of K > 1 cases: K samples, each a copy of level 0 -- mesh, fixed mask, D and
// its matrices ke or block-CSR (copied, not recomputed; Galerkin or rediscretised alike) -- so that each of its systems is
// bit for bit level 0's.  Built once per K and kept in mg.coarse[K].
int coarse_for_cases(fea_ctx* ctx, Batch& b, int K) {
  Mg& mg = *b.mg;
  if (mg.coarse[K]) return FEA_OK;
  const Batch& c0 = *mg.lev[0].b;
  cudaStream_t st = ctx->c.stream;
  const int64_t nv = c0.NV, nc = c0.NC;
  const int32_t nr = c0.NREG;
  std::vector<int64_t> vo(K + 1), co(K + 1);
  std::vector<int32_t> ro(K + 1);
  for (int k = 0; k <= K; ++k) {
    vo[k] = k * nv;
    co[k] = k * nc;
    ro[k] = k * nr;
  }
  fea_batch* created = nullptr;
  int rc = api_batch_begin(ctx, K, 3, vo.data(), co.data(), ro.data(), &created);
  if (rc != FEA_OK) return rc;
  std::unique_ptr<fea_batch, decltype(&api_free_batch)> hb(created, api_free_batch);
  Batch& kb = hb->b;
  CK(ctx, dalloc(kb, &kb.xy, kb.NV * 2));
  CK(ctx, dalloc(kb, &kb.D, (int64_t)kb.NREG * 9));
  CK(ctx, dalloc(kb, &kb.fixed, kb.NV));
  CK(ctx, dalloc(kb, &kb.rhs, kb.NV * 2));
  for (int k = 0; k < K; ++k) {
    CK(ctx, cudaMemcpyAsync(kb.xy + 2 * nv * k, c0.xy, sizeof(double) * 2 * nv, cudaMemcpyDeviceToDevice, st));
    CK(ctx, cudaMemcpyAsync(kb.D + 9 * (int64_t)nr * k, c0.D, sizeof(double) * 9 * nr, cudaMemcpyDeviceToDevice, st));
    CK(ctx, cudaMemcpyAsync(kb.fixed + nv * k, c0.fixed, nv, cudaMemcpyDeviceToDevice, st));
  }
  CK(ctx, cudaMemsetAsync(kb.rhs, 0, sizeof(double) * 2 * kb.NV, st));
  const unsigned gcell = (unsigned)((std::max<int64_t>(kb.NC, 1) + 255) / 256);
  {
    Scratch scratch(st);
    int32_t* conn = nullptr;
    int8_t* creg = nullptr;
    CK(ctx, scratch.alloc(&conn, kb.NC * 3));
    CK(ctx, scratch.alloc(&creg, kb.NC));
    k_mg_replicate_cells<<<gcell, 256, 0, st>>>(nc, K, c0.conn, c0.cell_dreg, 0, conn, creg);
    CK(ctx, cudaGetLastError());
    if ((rc = api_batch_finish(ctx, kb, creg, conn)) != FEA_OK) return rc;
  }
  // level 0's cells are oriented already: take them exactly as they are, whatever the orientation test made of them
  k_mg_replicate_cells<<<gcell, 256, 0, st>>>(nc, K, c0.conn, c0.cell_dreg, nv, kb.conn, nullptr);
  CK(ctx, cudaGetLastError());
  if (mg.grid)   // a grid level 0 has no element matrices: its Galerkin block-CSR is copied instead
    rc = mg_grid_assemble_cases(ctx, mg.lev[0], kb, K);
  else
    rc = api_batch_assemble(ctx, kb, [&c0, K](Batch& x) -> cudaError_t {
      for (int k = 0; k < K; ++k) {
        const cudaError_t e = cudaMemcpyAsync(x.ke + 36 * c0.NC * k, c0.ke, sizeof(double) * 36 * c0.NC, cudaMemcpyDeviceToDevice,
                                              x.ctx->stream);
        if (e != cudaSuccess) return e;
      }
      return cudaSuccess;
    });
  if (rc != FEA_OK) return rc;
  int64_t rows = 0;   // block rows of one sample (every sample has level 0's)
  CK(ctx, cudaMemcpyAsync(&rows, kb.row_base + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  mg.case_rows = rows;
  ctx->c.launches += 2;
  mg.coarse[K] = hb.release();
  return FEA_OK;
}

// The Work of K (1..kMaxCases) cases, its vectors from `scratch` (one allocation each: DESIGN.md section 3.11).
// Only the scalars are cleared: the driver and the V-cycle write every row of a vector before they read it.
int make_work(fea_ctx* ctx, Batch& b, int K, Scratch& scratch, Work& w) {
  Mg& mg = *b.mg;
  if (K == 1) {
    w.coarse = mg.lev[0].b;
  } else {
    const int rc = coarse_for_cases(ctx, b, K);
    if (rc != FEA_OK) return rc;
    w.coarse = &mg.coarse[K]->b;
    w.coarse_map = ColMap{1, mg.case_rows};
  }
  w.coarse_nv = mg.lev[0].b->NV;
  w.v.resize(mg.levels + 1);
  for (int l = 1; l <= mg.levels; ++l) {
    const int64_t n = mg.lev[l].b->NBR * K;
    Vecs& V = w.v[l];
    CK(ctx, scratch.alloc(&V.x, n));
    CK(ctx, scratch.alloc(&V.r, n));
    CK(ctx, scratch.alloc(&V.d[0], n));
    CK(ctx, scratch.alloc(&V.d[1], n));
    if (l < mg.levels) CK(ctx, scratch.alloc(&V.bv, n));   // the finest level's b is the outer CG's r
  }
  const int64_t nbr = b.NBR, np = nbr / kT;
  CK(ctx, scratch.alloc(&w.x, nbr * K));
  CK(ctx, scratch.alloc(&w.r, nbr * K));
  CK(ctx, scratch.alloc(&w.p, nbr * K));
  CK(ctx, scratch.alloc(&w.q, nbr * K));
  CK(ctx, scratch.alloc(&w.partA, np * K));
  CK(ctx, scratch.alloc(&w.partB, np * K));
  CK(ctx, scratch.alloc(&w.sc, (int64_t)kScCount * K));
  CK(ctx, cudaMemsetAsync(w.sc, 0, sizeof(double) * kScCount * K, ctx->c.stream));
  return FEA_OK;
}

// solve<K> of K (1..kMaxCases) cases on a Work of the call: loads on the device, case k at rhs + k * rhs_stride
int solve_cases(fea_ctx* ctx, Batch& b, int K, const double* rhs, int64_t rhs_stride, double rtol, int max_iter, const Out& o,
                fea_solve_stats& stats) {
  Scratch scratch(ctx->c.stream);
  Work w;
  const int rc = make_work(ctx, b, K, scratch, w);
  if (rc != FEA_OK) return rc;
  w.rhs = rhs;
  w.rhs_stride = rhs_stride;
  switch (K) {
    case 1: return solve<1>(ctx, b, w, rtol, max_iter, o, stats);
    case 2: return solve<2>(ctx, b, w, rtol, max_iter, o, stats);
    case 3: return solve<3>(ctx, b, w, rtol, max_iter, o, stats);
    case 4: return solve<4>(ctx, b, w, rtol, max_iter, o, stats);
    case 5: return solve<5>(ctx, b, w, rtol, max_iter, o, stats);
    case 6: return solve<6>(ctx, b, w, rtol, max_iter, o, stats);
    case 7: return solve<7>(ctx, b, w, rtol, max_iter, o, stats);
    case 8: return solve<8>(ctx, b, w, rtol, max_iter, o, stats);
  }
  return FEA_BAD_ARG;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
int mg_set_refinement(fea_ctx* ctx, Batch& b, int levels) {
  cudaStream_t st = ctx->c.stream;
  int64_t nc = b.NC;
  for (int l = 0; l < levels; ++l) {
    if (nc % 4 != 0 || nc == 0) return api_fail(ctx, FEA_MESH_ERROR, "cell count is not that of a uniform refinement");
    nc /= 4;
  }
  std::unique_ptr<Mg> mg(new Mg());
  mg->levels = levels;
  mg->lev.resize(levels + 1);
  MgLevel& top = mg->lev[levels];
  top.b = &b;
  top.nv = b.NV;
  top.nc = b.NC;
  top.conn = b.conn_given;
  top.creg = b.cell_dreg;
  Scratch scratch(st);
  int32_t* flag = nullptr;
  unsigned long long* key = nullptr;
  int32_t* tmp = nullptr;
  CK(ctx, scratch.alloc(&flag, 2));
  CK(ctx, scratch.alloc(&key, b.NV));
  CK(ctx, scratch.alloc(&tmp, b.NV / 4096 + 4));
  for (int l = levels; l >= 1; --l) {
    MgLevel& F = mg->lev[l];
    MgLevel& C = mg->lev[l - 1];
    C.nc = F.nc / 4;
    CK(ctx, dalloc(b, &C.conn, C.nc * 3));
    CK(ctx, dalloc(b, &C.creg, C.nc));
    CK(ctx, dalloc(b, &C.creg8, C.nc));
    CK(ctx, dalloc(b, &F.par, F.nv));
    CK(ctx, cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), st));
    CK(ctx, cudaMemsetAsync(key, 0xFF, sizeof(unsigned long long) * F.nv, st));
    k_mg_derive<<<(unsigned)((C.nc + 255) / 256), 256, 0, st>>>(C.nc, F.nv, F.conn, F.creg, b.xy, C.conn, C.creg, C.creg8, key, flag);
    int32_t h[2] = {0, 0};
    CK(ctx, cudaMemcpyAsync(h, flag, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    if (h[0])
      return api_fail(ctx, FEA_MESH_ERROR, (h[0] & 1) ? "children of a cell are not those of a uniform red refinement"
                                           : (h[0] & 2) ? "a midpoint is shared by two different edges"
                                                        : "a midpoint is not at the middle of its edge (bit for bit)");
    C.nv = (int64_t)h[1] + 1;
    CK(ctx, dalloc(b, &F.child_ptr, C.nv + 1));
    CK(ctx, dalloc(b, &F.child, 2 * (F.nv - C.nv)));
    int32_t* cnt = nullptr;
    CK(ctx, scratch.alloc(&cnt, C.nv + 1));
    CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (C.nv + 1), st));
    k_mg_parents<<<(unsigned)((F.nv + 255) / 256), 256, 0, st>>>(F.nv, (int)C.nv, key, F.par, cnt, flag);
    // the midpoint lists are built from par: only once every vertex from n_c on is known to be a midpoint
    CK(ctx, cudaMemcpyAsync(h, flag, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    if (h[0]) return api_fail(ctx, FEA_MESH_ERROR, "vertices are not numbered coarse vertices first, then one midpoint per coarse edge");
    CK(ctx, exclusive_scan_i32(cnt, F.child_ptr, C.nv, tmp, st));
    CK(ctx, cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (C.nv + 1), st));
    if (F.nv > C.nv)
      k_mg_child_fill<<<(unsigned)((F.nv - C.nv + 255) / 256), 256, 0, st>>>(F.nv, (int)C.nv, F.par, F.child_ptr, cnt, F.child);
    k_mg_child_sort<<<(unsigned)((C.nv + 255) / 256), 256, 0, st>>>((int)C.nv, F.child_ptr, F.child);
    CK(ctx, cudaGetLastError());
    ctx->c.launches += 5;
  }
  b.mg = mg.release();
  return FEA_OK;
}

int mg_assemble(fea_ctx* ctx, Batch& b) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  // coarse level batches, finest-but-one first: each one's matrices are the Galerkin product of the next finer.
  // A non-nested hierarchy's coarse batches exist already (mg_set_coarse_meshes) and are rediscretised:
  // each level's operator is its own mesh's stiffness matrix.  A grid hierarchy builds its levels in k_mg_grid.cu.
  if (mg.grid) {
    const int rc = mg_grid_assemble(ctx, b);
    if (rc != FEA_OK) return rc;
  }
  for (int l = mg.levels - 1; l >= 0 && !mg.grid; --l) {
    MgLevel& C = mg.lev[l];
    if (mg.nonnested) {
      const int rc = fea_batch_assemble(C.hb);
      if (rc != FEA_OK) return rc;
      continue;
    }
    const MgLevel& F = mg.lev[l + 1];
    const int64_t vo[2] = {0, C.nv}, co[2] = {0, C.nc};
    const int32_t ro[2] = {0, b.NREG};
    int rc = api_batch_begin(ctx, 1, 3, vo, co, ro, &C.hb);
    if (rc != FEA_OK) return rc;
    Batch& cb = C.hb->b;
    C.b = &cb;
    CK(ctx, dalloc(cb, &cb.xy, cb.NV * 2));
    CK(ctx, dalloc(cb, &cb.D, (int64_t)cb.NREG * 9));
    CK(ctx, dalloc(cb, &cb.fixed, cb.NV));
    CK(ctx, dalloc(cb, &cb.rhs, cb.NV * 2));
    CK(ctx, cudaMemcpyAsync(cb.xy, b.xy, sizeof(double) * 2 * cb.NV, cudaMemcpyDeviceToDevice, st));   // a prefix of the finest
    CK(ctx, cudaMemcpyAsync(cb.D, b.D, sizeof(double) * 9 * cb.NREG, cudaMemcpyDeviceToDevice, st));
    CK(ctx, cudaMemcpyAsync(cb.fixed, b.fixed, cb.NV, cudaMemcpyDeviceToDevice, st));
    CK(ctx, cudaMemsetAsync(cb.rhs, 0, sizeof(double) * 2 * cb.NV, st));
    if ((rc = api_batch_finish(ctx, cb, C.creg8, C.conn)) != FEA_OK) return rc;
    const Batch& fb = *F.b;
    const int2* par = F.par;
    rc = api_batch_assemble(ctx, cb, [&fb, par](Batch& c) -> cudaError_t {
      if (c.NC) k_mg_galerkin<<<(unsigned)((c.NC + 127) / 128), 128, 0, c.ctx->stream>>>(c.NC, fb.conn, fb.ke, fb.fixed, par, c.conn, c.ke);
      return cudaGetLastError();
    });
    if (rc != FEA_OK) return rc;
    ctx->c.launches += 1;
  }
  if (!mg.h_sc) CK(ctx, cudaHostAlloc((void**)&mg.h_sc, sizeof(double) * kScCount * kMaxCases, cudaHostAllocDefault));
  if (mg.ev.empty()) {
    mg.ev.resize(4 * (mg.levels + 1) + 2);
    for (auto& ev : mg.ev) CK(ctx, cudaEventCreate(&ev));
  }
  {   // Lanczos vectors of every level, sized to the finest
    Scratch scratch(st);
    const int64_t nbr = b.NBR;
    double2 *v = nullptr, *vp = nullptr, *w = nullptr;
    double *part = nullptr, *sc = nullptr;
    CK(ctx, scratch.alloc(&v, nbr));
    CK(ctx, scratch.alloc(&vp, nbr));
    CK(ctx, scratch.alloc(&w, nbr));
    CK(ctx, scratch.alloc(&part, nbr / kT));
    CK(ctx, scratch.alloc(&sc, kScCount + 2 * kLanczos));
    for (int l = 0; l <= mg.levels; ++l) CK(ctx, estimate_lmax(b, mg.lev[l], v, vp, w, part, sc));
  }
  if (mg.coarse_solver == FEA_COARSE_DIRECT) return mg_direct_factor(ctx, b);
  return FEA_OK;
}

int mg_apply(fea_ctx* ctx, Batch& b, const double* d_r, double* d_z) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  const unsigned g = grid_rows(b);
  if (!g) return FEA_OK;
  for (auto& L : mg.lev) L.ms = 0.0;
  Scratch scratch(st);
  Work w;
  const int rc = make_work(ctx, b, 1, scratch, w);
  if (rc != FEA_OK) return rc;
  k_mg_load<<<g, kT, 0, st>>>(side_of(b), b.vrank, d_r, w.r);
  CK(ctx, vcycle_top<1>(ctx, b, w, w.r, 1u));
  k_mg_store<<<g, kT, 0, st>>>(side_of(b), b.vrank, w.v[mg.levels].x, d_z);
  ctx->c.launches += 2;
  CK(ctx, cudaGetLastError());
  CK(ctx, cudaStreamSynchronize(st));
  accumulate_level_ms(mg);
  return FEA_OK;
}

int mg_coarse_solve(fea_ctx* ctx, Batch& b, const double* d_r, double* d_x) {
  Mg& mg = *b.mg;
  Batch& l0 = *mg.lev[0].b;
  cudaStream_t st = ctx->c.stream;
  CK(ctx, launch_active_to_vertices(st, l0.NV, l0.vrank, d_r, l0.rhs));
  CK(ctx, coarse_solve(mg, l0, 1, l0.NV, ColMap{1, 0}, st));
  const unsigned g = grid_rows(l0);
  if (g) k_mg_store<<<g, kT, 0, st>>>(side_of(l0), l0.vrank, (const double2*)l0.x, d_x);
  ctx->c.launches += 3;
  CK(ctx, cudaGetLastError());
  CK(ctx, cudaStreamSynchronize(st));
  return FEA_OK;
}

int mg_solve(fea_ctx* ctx, Batch& b, double rtol, int max_iter) {
  b.t_spmv.clear();
  b.t_update.clear();
  const Out o{b.sc.status, b.sc.iters, b.sc.rz0, b.rz_last, b.u, b.ranges, b.relres, nullptr};
  return solve_cases(ctx, b, 1, b.rhs, 0, rtol, max_iter, o, b.stats);
}

int mg_solve_load_cases(fea_ctx* ctx, Batch& b, int K, const double* rhs, double rtol, int max_iter, double* u, double* ranges,
                        int32_t* iters, double* relres, int32_t* status, fea_solve_stats* stats) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  Scratch scratch(st);
  double* d_rhs = nullptr;
  CK(ctx, scratch.alloc(&d_rhs, 2 * b.NV * K));
  CK(ctx, cudaMemcpyAsync(d_rhs, rhs, sizeof(double) * 2 * b.NV * K, cudaMemcpyHostToDevice, st));
  Out o{};
  CK(ctx, scratch.alloc(&o.status, K));
  CK(ctx, scratch.alloc(&o.iters, K));
  CK(ctx, scratch.alloc(&o.rz0, K));
  CK(ctx, scratch.alloc(&o.rz_last, K));
  CK(ctx, scratch.alloc(&o.u, 2 * b.NV * K));
  CK(ctx, scratch.alloc(&o.ranges, 4 * K));
  CK(ctx, scratch.alloc(&o.relres, K));
  if (K > 1) CK(ctx, scratch.alloc(&o.col, b.NBR));
  fea_solve_stats s{};
  const int rc = solve_cases(ctx, b, K, d_rhs, 2 * b.NV, rtol, max_iter, o, s);
  if (rc != FEA_OK) return rc;
  // keep u, ranges and status of the cases for the fea_batch_load_case_* outputs, replacing the last call's
  mg.n_kept = 0;
  if (mg.kept_cap < K) {
    if (mg.case_u) CK(ctx, cudaFreeAsync(mg.case_u, st));
    mg.case_u = nullptr;
    mg.kept_cap = 0;
    CK(ctx, cudaMallocAsync((void**)&mg.case_u, sizeof(double) * 2 * b.NV * K, st));
    mg.kept_cap = K;
  }
  if (!mg.case_ranges) CK(ctx, cudaMallocAsync((void**)&mg.case_ranges, sizeof(double) * 4 * kMaxCases, st));
  if (!mg.case_status) CK(ctx, cudaMallocAsync((void**)&mg.case_status, sizeof(int32_t) * kMaxCases, st));
  CK(ctx, cudaMemcpyAsync(mg.case_u, o.u, sizeof(double) * 2 * b.NV * K, cudaMemcpyDeviceToDevice, st));
  CK(ctx, cudaMemcpyAsync(mg.case_ranges, o.ranges, sizeof(double) * 4 * K, cudaMemcpyDeviceToDevice, st));
  CK(ctx, cudaMemcpyAsync(mg.case_status, o.status, sizeof(int32_t) * K, cudaMemcpyDeviceToDevice, st));
  if (u) CK(ctx, cudaMemcpyAsync(u, o.u, sizeof(double) * 2 * b.NV * K, cudaMemcpyDeviceToHost, st));
  if (ranges) CK(ctx, cudaMemcpyAsync(ranges, o.ranges, sizeof(double) * 4 * K, cudaMemcpyDeviceToHost, st));
  if (iters) CK(ctx, cudaMemcpyAsync(iters, o.iters, sizeof(int32_t) * K, cudaMemcpyDeviceToHost, st));
  if (relres) CK(ctx, cudaMemcpyAsync(relres, o.relres, sizeof(double) * K, cudaMemcpyDeviceToHost, st));
  if (status) CK(ctx, cudaMemcpyAsync(status, o.status, sizeof(int32_t) * K, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  mg.n_kept = K;
  if (stats) *stats = s;
  return FEA_OK;
}

void mg_release(Batch& b) {
  if (!b.mg) return;
  Mg* mg = b.mg;
  for (auto& L : mg->lev)
    if (L.hb) api_free_batch(L.hb);
  for (fea_batch* cb : mg->coarse)
    if (cb) api_free_batch(cb);
  for (void* p : {(void*)mg->case_u, (void*)mg->case_ranges, (void*)mg->case_status, (void*)mg->case_owner})
    if (p) cudaFreeAsync(p, b.ctx->stream);
  mg_direct_release(*mg, b.ctx->stream);
  for (auto& ev : mg->ev) cudaEventDestroy(ev);
  if (mg->h_sc) cudaFreeHost(mg->h_sc);
  delete mg;
  b.mg = nullptr;
}

}  // namespace fea
