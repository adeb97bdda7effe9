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
//               iteration flexible CG, beta = z+.(r+ - r) / (r.z) = -alpha z+.q / (r.z).
// Dot products: one partial per CTA, summed by one block in a fixed order (bitwise reproducible).
#include <cmath>
#include <cstdio>
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

// (Khat v)[row]; row's lane in its slice = threadIdx.x & 31
__device__ __forceinline__ double2 khat_row(const MgOp& A, int64_t row, const double2* __restrict__ v) {
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = A.slice_len[slice];
  const int64_t base = A.slice_ptr[slice];
  const d4* __restrict__ vt = A.val + base + lane;
  const int32_t* __restrict__ cp = A.col + base + lane;
  const double2 own = v[row];
  double a0 = own.x, a1 = own.y;
  for (int j = 0; j < L; ++j) {
    const int c = ld_stream_i32(cp + j * 32);
    const d4 k = ld_stream_d4(vt + j * 32);
    const double2 xj = __ldg(v + c);
    a0 = fma(k.x, xj.x, a0);
    a0 = fma(k.y, xj.y, a0);
    a1 = fma(k.z, xj.x, a1);
    a1 = fma(k.w, xj.y, a1);
  }
  return make_double2(a0, a1);
}

// deterministic block sum, result written by thread 0 to part[blockIdx.x]
__device__ __forceinline__ void block_partial(double v, double* __restrict__ part) {
  __shared__ double sm[kT / 32];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kT / 32; ++w) t += sm[w];
    part[blockIdx.x] = t;
  }
}

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
// reductions: one block sums the partials in a fixed order, then updates the scalars
enum { kRedStore = 0, kRedDots = 1, kRedPQ = 2 };
__global__ void __launch_bounds__(1024) k_mg_reduce(const double* __restrict__ pa, const double* __restrict__ pb, int n,
                                                    double* __restrict__ sc, int mode, double* __restrict__ out, int first) {
  __shared__ double sa[32], sb[32];
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
  const double2 t = khat_row(A, row, v);
  w[row] = t;
  block_partial(dot2(v[row], t), part);
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
// V-cycle kernels of one level (state: x, r, d where d is not yet added to x)
// Chebyshev step: x += d_in; r -= Khat d_in; d_out = c1 d_in + c2 r.  The last step of the pre-smoother
// (d_out == nullptr) leaves the unscaled residual S^-T r in ru for the restriction instead.
__global__ void __launch_bounds__(kT) k_mg_cheb_step(MgOp A, const double2* __restrict__ din, double2* __restrict__ dout,
                                                     double2* __restrict__ x, double2* __restrict__ r, double c1, double c2,
                                                     const double* __restrict__ ds, const double* __restrict__ scp,
                                                     double2* __restrict__ ru) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 ad = khat_row(A, row, din);
  const double2 d = din[row];
  double2 xv = x[row], rv = r[row];
  xv.x += d.x;
  xv.y += d.y;
  rv.x -= ad.x;
  rv.y -= ad.y;
  x[row] = xv;
  r[row] = rv;
  if (dout) dout[row] = make_double2(fma(c1, d.x, c2 * rv.x), fma(c1, d.y, c2 * rv.y));
  else ru[row] = ds[2 * row] > 0.0 ? solve_St(ds, scp, row, rv) : make_double2(0.0, 0.0);   // padding rows: 0
}
// after the coarse correction: r = b - Khat x, d = r / theta
__global__ void __launch_bounds__(kT) k_mg_resid(MgOp A, const double2* __restrict__ x, const double2* __restrict__ b,
                                                 double2* __restrict__ r, double2* __restrict__ d, double inv_theta) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 ax = khat_row(A, row, x);
  const double2 bv = b[row];
  const double2 rv = make_double2(bv.x - ax.x, bv.y - ax.y);
  r[row] = rv;
  d[row] = make_double2(rv.x * inv_theta, rv.y * inv_theta);
}
__global__ void __launch_bounds__(kT) k_mg_add(double2* __restrict__ x, const double2* __restrict__ d) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 a = x[row], b = d[row];
  x[row] = make_double2(a.x + b.x, a.y + b.y);
}
// entry of the finest level: r = b, d = b / theta, x = 0
__global__ void __launch_bounds__(kT) k_mg_top_init(const double2* __restrict__ b, double2* __restrict__ x,
                                                    double2* __restrict__ r, double2* __restrict__ d, double inv_theta) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 bv = b[row];
  r[row] = bv;
  d[row] = make_double2(bv.x * inv_theta, bv.y * inv_theta);
  x[row] = make_double2(0.0, 0.0);
}

struct Side {   // one level's maps and scaling
  const int32_t* vertex_of_row;
  const int32_t* row_of_vertex;
  const double* dscale;
  const double* scoup;
};
Side side_of(const Batch& b) { return Side{b.vertex_of_row, b.row_of_vertex, b.dscale, b.scoup}; }

// restriction, one thread per coarse row: r_c = P^T S_f^-T r^_f at the coarse vertex (ru = S_f^-T r^_f).  Into a smoothed level:
// b = r = S_c^T r_c, d = b / theta, x = 0; into the coarsest level: its unscaled load vector rhs[vertex].
__global__ void __launch_bounds__(kT) k_mg_restrict(Side F, Side Cs, const double2* __restrict__ ru,
                                                    const int32_t* __restrict__ child_ptr, const int32_t* __restrict__ child,
                                                    double2* __restrict__ bc, double2* __restrict__ xc, double2* __restrict__ rc,
                                                    double2* __restrict__ dc, double inv_theta, double2* __restrict__ rhs0) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int j = Cs.vertex_of_row[row];
  double2 acc = make_double2(0.0, 0.0);
  if (j >= 0) {
    const int fr = F.row_of_vertex[j];
    if (fr >= 0) acc = ru[fr];
    for (int i = child_ptr[j]; i < child_ptr[j + 1]; ++i) {
      const int m = child[i];
      const int mr = F.row_of_vertex[m];
      if (mr < 0) continue;
      const double2 t = ru[mr];
      acc.x = fma(0.5, t.x, acc.x);
      acc.y = fma(0.5, t.y, acc.y);
    }
  }
  if (rhs0) {
    if (j >= 0) rhs0[j] = acc;
    return;
  }
  const double2 h = j >= 0 ? mul_St(Cs.dscale, Cs.scoup, row, acc) : make_double2(0.0, 0.0);
  bc[row] = h;
  rc[row] = h;
  dc[row] = make_double2(h.x * inv_theta, h.y * inv_theta);
  xc[row] = make_double2(0.0, 0.0);
}

// prolongation-add, one thread per fine row: x^_f += S_f^-1 P S_c x^_c
__global__ void __launch_bounds__(kT) k_mg_prolong(Side F, Side Cs, const int2* __restrict__ par, const double2* __restrict__ xc,
                                                   double2* __restrict__ xf) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int f = F.vertex_of_row[row];
  if (f < 0) return;
  const int2 pr = par[f];
  double2 e = make_double2(0.0, 0.0);
  const int r0 = Cs.row_of_vertex[pr.x];
  const double w = pr.y < 0 ? 1.0 : 0.5;
  if (r0 >= 0) {
    const double2 t = mul_S(Cs.dscale, Cs.scoup, r0, xc[r0]);
    e = make_double2(w * t.x, w * t.y);
  }
  if (pr.y >= 0) {
    const int r1 = Cs.row_of_vertex[pr.y];
    if (r1 >= 0) {
      const double2 t = mul_S(Cs.dscale, Cs.scoup, r1, xc[r1]);
      e.x = fma(0.5, t.x, e.x);
      e.y = fma(0.5, t.y, e.y);
    }
  }
  const double2 c = solve_S(F.dscale, F.scoup, row, e);
  double2 xv = xf[row];
  xv.x += c.x;
  xv.y += c.y;
  xf[row] = xv;
}

// ---------------------------------------------------------------------------------------------------------
// outer flexible CG on the finest level
// r = S^T b (true = 0) or S^T b - Khat x (true = 1); true = 0 also clears x, p, q.  Partials of r.r.
__global__ void __launch_bounds__(kT) k_mg_fcg_residual(MgOp A, Side F, const double* __restrict__ rhs, double2* __restrict__ x,
                                                        double2* __restrict__ r, double2* __restrict__ p, double2* __restrict__ q,
                                                        int true_res, double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int v = F.vertex_of_row[row];
  double2 bv = make_double2(0.0, 0.0);
  if (v >= 0) bv = mul_St(F.dscale, F.scoup, row, make_double2(rhs[2 * (int64_t)v], rhs[2 * (int64_t)v + 1]));
  if (true_res) {
    const double2 ax = khat_row(A, row, x);
    bv.x -= ax.x;
    bv.y -= ax.y;
  } else {
    x[row] = make_double2(0.0, 0.0);
  }
  if (!true_res || true_res == 2) {   // (re)start: p = q = 0
    p[row] = make_double2(0.0, 0.0);
    q[row] = make_double2(0.0, 0.0);
  }
  r[row] = bv;
  block_partial(dot2(bv, bv), part);
}
__global__ void __launch_bounds__(kT) k_mg_fcg_dots(const double2* __restrict__ z, const double2* __restrict__ r,
                                                    const double2* __restrict__ q, double* __restrict__ pa, double* __restrict__ pb) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 zv = z[row];
  block_partial(dot2(zv, r[row]), pa);
  __syncthreads();
  block_partial(dot2(zv, q[row]), pb);
}
__global__ void __launch_bounds__(kT) k_mg_fcg_dir(const double2* __restrict__ z, double2* __restrict__ p, const double* __restrict__ sc) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double beta = sc[kScBeta];
  const double2 zv = z[row], pv = p[row];
  p[row] = make_double2(fma(beta, pv.x, zv.x), fma(beta, pv.y, zv.y));
}
__global__ void __launch_bounds__(kT) k_mg_fcg_spmv(MgOp A, const double2* __restrict__ p, double2* __restrict__ q,
                                                    double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double2 qv = khat_row(A, row, p);
  q[row] = qv;
  block_partial(dot2(p[row], qv), part);
}
__global__ void __launch_bounds__(kT) k_mg_fcg_update(double2* __restrict__ x, double2* __restrict__ r, const double2* __restrict__ p,
                                                      const double2* __restrict__ q, const double* __restrict__ sc,
                                                      double* __restrict__ part) {
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const double alpha = sc[kScAlpha], pq = sc[kScPQ];
  double2 rv = r[row];
  // p.q <= 0 or a non-finite step: breakdown (the host stops), x and r keep the last sound iterate
  if (pq > 0.0 && isfinite(pq) && isfinite(alpha)) {
    const double2 pv = p[row], qv = q[row];
    double2 xv = x[row];
    xv.x = fma(alpha, pv.x, xv.x);
    xv.y = fma(alpha, pv.y, xv.y);
    rv.x = fma(-alpha, qv.x, rv.x);
    rv.y = fma(-alpha, qv.y, rv.y);
    x[row] = xv;
    r[row] = rv;
  }
  block_partial(dot2(rv, rv), part);
}
// what launch_finalize and fea_batch_download read
__global__ void k_mg_finish(SysScalars s, double* __restrict__ rz_last, const double* __restrict__ sc, int status, int iters) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  s.status[0] = status;
  s.iters[0] = iters;
  s.rz0[0] = sc[kScRZ0];
  rz_last[0] = sc[kScTrue];
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

cudaError_t reduce(Batch& fine, const double* pa, const double* pb, int n, int mode, int slot = 0, int first = 0,
                   double* out = nullptr) {
  k_mg_reduce<<<1, 1024, 0, fine.ctx->stream>>>(pa, pb, n, fine.mg->sc, mode, out ? out : fine.mg->sc + slot, first);
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

// largest eigenvalue of level L's Khat: the top Ritz value of kLanczos Lanczos steps (vectors borrowed from
// the outer CG).  15 power iterations, the cheaper alternative, stay at 2.03-2.07 on the C3 meshes where
// Lanczos finds 2.34-2.39 (true 2.36-2.42): the smoother would then amplify the top of the spectrum.
cudaError_t estimate_lmax(Batch& fine, MgLevel& L) {
  Mg& mg = *fine.mg;
  cudaStream_t st = fine.ctx->stream;
  const Batch& b = *L.b;
  const unsigned g = grid_rows(b);
  if (!g) return cudaSuccess;
  double2 *v = mg.p, *vp = mg.q, *w = mg.r;
  double* lz = mg.sc + kScCount;   // [2 kLanczos]: alpha_k, beta_k^2
  k_mg_lz_init<<<g, kT, 0, st>>>(b.vertex_of_row, w, mg.partA);
  cudaError_t e = reduce(fine, mg.partA, nullptr, (int)g, kRedStore, kScNrm);
  if (e == cudaSuccess) k_mg_lz_next<<<g, kT, 0, st>>>(v, vp, w, mg.sc + kScNrm);
  for (int k = 0; k < kLanczos && e == cudaSuccess; ++k) {
    k_mg_lz_apply<<<g, kT, 0, st>>>(op_of(b), v, w, mg.partA);
    e = reduce(fine, mg.partA, nullptr, (int)g, kRedStore, 0, 0, lz + 2 * k);
    k_mg_lz_orth<<<g, kT, 0, st>>>(v, vp, w, lz + 2 * k, k ? lz + 2 * k - 1 : nullptr, mg.partA);
    if (e == cudaSuccess) e = reduce(fine, mg.partA, nullptr, (int)g, kRedStore, 0, 0, lz + 2 * k + 1);
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

// one V-cycle from level l down; level l's b, r, d[0], x are set up by the caller (restriction / top init)
cudaError_t vcycle(fea_ctx* ctx, Batch& fine, int l) {
  Mg& mg = *fine.mg;
  Ctx& c = ctx->c;
  cudaStream_t st = c.stream;
  MgLevel& L = mg.lev[l];
  cudaEvent_t* ev = mg.ev.data() + 4 * l;
  cudaError_t e;
  if (l == 0) {   // coarsest: block-Jacobi CG of the level-0 batch on the restricted residual
    if ((e = cudaEventRecord(ev[0], st)) != cudaSuccess) return e;
    if ((e = run_pcg(*L.b, kCoarseRtol, kCoarseMaxIter)) != cudaSuccess) return e;
    return cudaEventRecord(ev[1], st);
  }
  const Batch& b = *L.b;
  MgLevel& C = mg.lev[l - 1];
  const unsigned g = grid_rows(b), gc = grid_rows(*C.b);
  const MgOp A = op_of(b);
  cudaEventRecord(ev[0], st);
  k_mg_cheb_step<<<g, kT, 0, st>>>(A, L.d[0], L.d[1], L.x, L.r, L.c1[0], L.c2[0], nullptr, nullptr, nullptr);
  k_mg_cheb_step<<<g, kT, 0, st>>>(A, L.d[1], L.d[0], L.x, L.r, L.c1[1], L.c2[1], nullptr, nullptr, nullptr);
  k_mg_cheb_step<<<g, kT, 0, st>>>(A, L.d[0], nullptr, L.x, L.r, 0.0, 0.0, b.dscale, b.scoup, L.d[1]);
  if (gc)
    k_mg_restrict<<<gc, kT, 0, st>>>(side_of(b), side_of(*C.b), L.d[1], L.child_ptr, L.child, C.bv, C.x, C.r, C.d[0],
                                     C.inv_theta, l == 1 ? (double2*)C.b->rhs : nullptr);
  cudaEventRecord(ev[1], st);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = vcycle(ctx, fine, l - 1)) != cudaSuccess) return e;
  cudaEventRecord(ev[2], st);
  k_mg_prolong<<<g, kT, 0, st>>>(side_of(b), side_of(*C.b), L.par, l == 1 ? (const double2*)C.b->x : C.x, L.x);
  k_mg_resid<<<g, kT, 0, st>>>(A, L.x, L.bv, L.r, L.d[0], L.inv_theta);
  k_mg_cheb_step<<<g, kT, 0, st>>>(A, L.d[0], L.d[1], L.x, L.r, L.c1[0], L.c2[0], nullptr, nullptr, nullptr);
  k_mg_cheb_step<<<g, kT, 0, st>>>(A, L.d[1], L.d[0], L.x, L.r, L.c1[1], L.c2[1], nullptr, nullptr, nullptr);
  k_mg_add<<<g, kT, 0, st>>>(L.x, L.d[0]);
  cudaEventRecord(ev[3], st);
  c.launches += 9;
  return cudaGetLastError();
}

// z = V(rhs) on the finest level: the result is in lev[levels].x
cudaError_t vcycle_top(fea_ctx* ctx, Batch& fine, const double2* rhs) {
  Mg& mg = *fine.mg;
  MgLevel& L = mg.lev[mg.levels];
  L.bv = const_cast<double2*>(rhs);
  k_mg_top_init<<<grid_rows(fine), kT, 0, ctx->c.stream>>>(rhs, L.x, L.r, L.d[0], L.inv_theta);
  ctx->c.launches += 1;
  return vcycle(ctx, fine, mg.levels);
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

#define MGCK(call)                                                                                              \
  do {                                                                                                          \
    cudaError_t e_ = (call);                                                                                    \
    if (e_ != cudaSuccess)                                                                                      \
      return api_fail(ctx, e_ == cudaErrorMemoryAllocation ? FEA_OUT_OF_MEMORY : FEA_CUDA_ERROR, #call, e_);    \
  } while (0)

}  // namespace

// ---------------------------------------------------------------------------------------------------------
int mg_set_refinement(fea_ctx* ctx, Batch& b, int levels) {
  cudaStream_t st = ctx->c.stream;
  int64_t nc = b.NC;
  for (int l = 0; l < levels; ++l) {
    if (nc % 4 != 0 || nc == 0) return api_fail(ctx, FEA_MESH_ERROR, "cell count is not that of a uniform refinement");
    nc /= 4;
  }
  Mg* mg = new Mg();
  mg->levels = levels;
  mg->lev.resize(levels + 1);
  MgLevel& top = mg->lev[levels];
  top.b = &b;
  top.nv = b.NV;
  top.nc = b.NC;
  top.conn = b.conn_given;
  top.creg = b.cell_dreg;
  int32_t* flag = nullptr;
  unsigned long long* key = nullptr;
  int32_t* tmp = nullptr;
  cudaError_t e = cudaSuccess;
  int rc = FEA_OK;
#define A(call) if (e == cudaSuccess) e = (call)
  A(cudaMallocAsync((void**)&flag, 2 * sizeof(int32_t), st));
  A(cudaMallocAsync((void**)&key, sizeof(unsigned long long) * std::max<int64_t>(1, b.NV), st));
  A(cudaMallocAsync((void**)&tmp, sizeof(int32_t) * (b.NV / 4096 + 4), st));
  for (int l = levels; l >= 1 && e == cudaSuccess && rc == FEA_OK; --l) {
    MgLevel& F = mg->lev[l];
    MgLevel& C = mg->lev[l - 1];
    C.nc = F.nc / 4;
    A(dalloc(b, &C.conn, C.nc * 3));
    A(dalloc(b, &C.creg, C.nc));
    A(dalloc(b, &C.creg8, C.nc));
    A(dalloc(b, &F.par, F.nv));
    A(cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), st));
    A(cudaMemsetAsync(key, 0xFF, sizeof(unsigned long long) * F.nv, st));
    if (e != cudaSuccess) break;
    k_mg_derive<<<(unsigned)((C.nc + 255) / 256), 256, 0, st>>>(C.nc, F.nv, F.conn, F.creg, b.xy, C.conn, C.creg, C.creg8, key, flag);
    int32_t h[2] = {0, 0};
    A(cudaMemcpyAsync(h, flag, sizeof(h), cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e != cudaSuccess) break;
    if (h[0]) {
      rc = api_fail(ctx, FEA_MESH_ERROR, (h[0] & 1) ? "children of a cell are not those of a uniform red refinement"
                                         : (h[0] & 2) ? "a midpoint is shared by two different edges"
                                                      : "a midpoint is not at the middle of its edge (bit for bit)");
      break;
    }
    C.nv = (int64_t)h[1] + 1;
    A(dalloc(b, &F.child_ptr, C.nv + 1));
    A(dalloc(b, &F.child, 2 * (F.nv - C.nv)));
    int32_t* cnt = nullptr;
    A(cudaMallocAsync((void**)&cnt, sizeof(int32_t) * (C.nv + 1), st));
    A(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (C.nv + 1), st));
    if (e != cudaSuccess) break;
    k_mg_parents<<<(unsigned)((F.nv + 255) / 256), 256, 0, st>>>(F.nv, (int)C.nv, key, F.par, cnt, flag);
    // the midpoint lists are built from par: only once every vertex from n_c on is known to be a midpoint
    A(cudaMemcpyAsync(h, flag, sizeof(h), cudaMemcpyDeviceToHost, st));
    A(cudaStreamSynchronize(st));
    if (e == cudaSuccess && h[0]) {
      cudaFreeAsync(cnt, st);
      rc = api_fail(ctx, FEA_MESH_ERROR, "vertices are not numbered coarse vertices first, then one midpoint per coarse edge");
      break;
    }
    A(exclusive_scan_i32(cnt, F.child_ptr, C.nv, tmp, st));
    A(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (C.nv + 1), st));
    if (F.nv > C.nv && e == cudaSuccess)
      k_mg_child_fill<<<(unsigned)((F.nv - C.nv + 255) / 256), 256, 0, st>>>(F.nv, (int)C.nv, F.par, F.child_ptr, cnt, F.child);
    if (e == cudaSuccess) k_mg_child_sort<<<(unsigned)((C.nv + 255) / 256), 256, 0, st>>>((int)C.nv, F.child_ptr, F.child);
    A(cudaGetLastError());
    if (cnt) cudaFreeAsync(cnt, st);
    ctx->c.launches += 5;
  }
#undef A
  if (flag) cudaFreeAsync(flag, st);
  if (key) cudaFreeAsync(key, st);
  if (tmp) cudaFreeAsync(tmp, st);
  if (e != cudaSuccess) rc = api_fail(ctx, e == cudaErrorMemoryAllocation ? FEA_OUT_OF_MEMORY : FEA_CUDA_ERROR, "fea_batch_set_refinement", e);
  if (rc != FEA_OK) {
    delete mg;
    return rc;
  }
  b.mg = mg;
  return FEA_OK;
}

int mg_assemble(fea_ctx* ctx, Batch& b) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  // coarse level batches, finest-but-one first: each one's matrices are the Galerkin product of the next finer
  for (int l = mg.levels - 1; l >= 0; --l) {
    MgLevel& C = mg.lev[l];
    const MgLevel& F = mg.lev[l + 1];
    const int64_t vo[2] = {0, C.nv}, co[2] = {0, C.nc};
    const int32_t ro[2] = {0, b.NREG};
    int rc = api_batch_begin(ctx, 1, 3, vo, co, ro, &C.hb);
    if (rc != FEA_OK) return rc;
    Batch& cb = C.hb->b;
    C.b = &cb;
    MGCK(dalloc(cb, &cb.xy, cb.NV * 2));
    MGCK(dalloc(cb, &cb.D, (int64_t)cb.NREG * 9));
    MGCK(dalloc(cb, &cb.fixed, cb.NV));
    MGCK(dalloc(cb, &cb.rhs, cb.NV * 2));
    MGCK(cudaMemcpyAsync(cb.xy, b.xy, sizeof(double) * 2 * cb.NV, cudaMemcpyDeviceToDevice, st));   // a prefix of the finest
    MGCK(cudaMemcpyAsync(cb.D, b.D, sizeof(double) * 9 * cb.NREG, cudaMemcpyDeviceToDevice, st));
    MGCK(cudaMemcpyAsync(cb.fixed, b.fixed, cb.NV, cudaMemcpyDeviceToDevice, st));
    MGCK(cudaMemsetAsync(cb.rhs, 0, sizeof(double) * 2 * cb.NV, st));
    MGCK(api_batch_finish(cb, C.creg8, C.conn));
    const Batch& fb = *F.b;
    const int2* par = F.par;
    rc = api_batch_assemble(ctx, cb, [&fb, par](Batch& c) -> cudaError_t {
      if (c.NC) k_mg_galerkin<<<(unsigned)((c.NC + 127) / 128), 128, 0, c.ctx->stream>>>(c.NC, fb.conn, fb.ke, fb.fixed, par, c.conn, c.ke);
      return cudaGetLastError();
    });
    if (rc != FEA_OK) return rc;
    ctx->c.launches += 1;
  }
  // vectors: outer CG on the finest level, V-cycle state on every smoothed level
  const int64_t nbr = b.NBR;
  MGCK(dalloc(b, &mg.r, nbr));
  MGCK(dalloc(b, &mg.p, nbr));
  MGCK(dalloc(b, &mg.q, nbr));
  MGCK(dalloc(b, &mg.partA, nbr / kT));
  MGCK(dalloc(b, &mg.partB, nbr / kT));
  MGCK(dalloc(b, &mg.sc, kScCount + 2 * kLanczos));
  MGCK(cudaMemsetAsync(mg.sc, 0, sizeof(double) * (kScCount + 2 * kLanczos), st));
  for (int l = 1; l <= mg.levels; ++l) {
    MgLevel& L = mg.lev[l];
    const int64_t n = L.b->NBR;
    double2** v[5] = {&L.x, &L.r, &L.d[0], &L.d[1], &L.bv};   // the finest level's b is the outer CG's r
    for (double2** p : v) {
      if (p == &L.bv && l == mg.levels) continue;
      MGCK(dalloc(b, p, n));
      MGCK(cudaMemsetAsync(*p, 0, sizeof(double2) * std::max<int64_t>(1, n), st));
    }
  }
  if (!mg.h_sc) MGCK(cudaHostAlloc((void**)&mg.h_sc, sizeof(double) * kScCount, cudaHostAllocDefault));
  if (mg.ev.empty()) {
    mg.ev.resize(4 * (mg.levels + 1) + 2);
    for (auto& ev : mg.ev) MGCK(cudaEventCreate(&ev));
  }
  for (int l = 0; l <= mg.levels; ++l) MGCK(estimate_lmax(b, mg.lev[l]));
  return FEA_OK;
}

int mg_apply(fea_ctx* ctx, Batch& b, const double* d_r, double* d_z) {
  Mg& mg = *b.mg;
  cudaStream_t st = ctx->c.stream;
  const unsigned g = grid_rows(b);
  if (!g) return FEA_OK;
  for (auto& L : mg.lev) L.ms = 0.0;
  k_mg_load<<<g, kT, 0, st>>>(side_of(b), b.vrank, d_r, mg.r);
  MGCK(vcycle_top(ctx, b, mg.r));
  k_mg_store<<<g, kT, 0, st>>>(side_of(b), b.vrank, mg.lev[mg.levels].x, d_z);
  ctx->c.launches += 2;
  MGCK(cudaGetLastError());
  MGCK(cudaStreamSynchronize(st));
  accumulate_level_ms(mg);
  return FEA_OK;
}

int mg_solve(fea_ctx* ctx, Batch& b, double rtol, int max_iter) {
  Mg& mg = *b.mg;
  Ctx& c = ctx->c;
  cudaStream_t st = c.stream;
  const unsigned g = grid_rows(b);
  const int np = (int)g;
  const MgOp A = op_of(b);
  const Side F = side_of(b);
  double2* x = (double2*)b.x;
  double* h = mg.h_sc;
  cudaEvent_t ev0 = mg.ev[4 * (mg.levels + 1)], ev1 = mg.ev[4 * (mg.levels + 1) + 1];
  b.stats = fea_solve_stats{};
  b.t_spmv.clear();
  b.t_update.clear();
  for (auto& L : mg.lev) L.ms = 0.0;
  const int64_t launches0 = c.launches;
  MGCK(cudaEventRecord(ev0, st));
  int32_t empty = 0;
  MGCK(cudaMemcpyAsync(&empty, b.empty, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  k_mg_fcg_residual<<<g, kT, 0, st>>>(A, F, b.rhs, x, mg.r, mg.p, mg.q, 0, mg.partA);
  MGCK(reduce(b, mg.partA, nullptr, np, kRedStore, kScRZ0));
  MGCK(cudaMemcpyAsync(h, mg.sc, sizeof(double) * kScCount, cudaMemcpyDeviceToHost, st));
  MGCK(cudaStreamSynchronize(st));
  const double rz0 = h[kScRZ0], tol2 = rtol * rtol * rz0;
  int status = FEA_SAMPLE_NOT_RUN, it = 0, restarts = 0, first = 1;
  double rr = rz0;
  if (empty) status = FEA_SAMPLE_EMPTY_ROW;
  else if (!(rz0 > 0.0)) status = std::isfinite(rz0) ? FEA_SAMPLE_CONVERGED : FEA_SAMPLE_BREAKDOWN;
  if (status == FEA_SAMPLE_CONVERGED) {
    MGCK(cudaMemcpyAsync(mg.sc + kScTrue, &rz0, sizeof(double), cudaMemcpyHostToDevice, st));
  }
  while (status == FEA_SAMPLE_NOT_RUN) {
    if (rr <= tol2) {   // recursive residual met the tolerance: decide on the TRUE residual
      k_mg_fcg_residual<<<g, kT, 0, st>>>(A, F, b.rhs, x, mg.r, mg.p, mg.q, 2, mg.partA);
      MGCK(reduce(b, mg.partA, nullptr, np, kRedStore, kScTrue));
      MGCK(cudaMemcpyAsync(h, mg.sc, sizeof(double) * kScCount, cudaMemcpyDeviceToHost, st));
      MGCK(cudaStreamSynchronize(st));
      c.launches += 2;
      rr = h[kScTrue];
      if (rr <= tol2) { status = FEA_SAMPLE_CONVERGED; break; }
      if (!std::isfinite(rr)) { status = FEA_SAMPLE_BREAKDOWN; break; }
      if (++restarts > kMaxRestarts) { status = FEA_SAMPLE_STAGNATED; break; }
      first = 1;   // restart from the true residual (p = q = 0)
    }
    if (it >= max_iter) { status = FEA_SAMPLE_MAX_ITER; break; }
    MGCK(vcycle_top(ctx, b, mg.r));
    const double2* z = mg.lev[mg.levels].x;
    k_mg_fcg_dots<<<g, kT, 0, st>>>(z, mg.r, mg.q, mg.partA, mg.partB);
    MGCK(reduce(b, mg.partA, mg.partB, np, kRedDots, 0, first));
    k_mg_fcg_dir<<<g, kT, 0, st>>>(z, mg.p, mg.sc);
    k_mg_fcg_spmv<<<g, kT, 0, st>>>(A, mg.p, mg.q, mg.partA);
    MGCK(reduce(b, mg.partA, nullptr, np, kRedPQ));
    k_mg_fcg_update<<<g, kT, 0, st>>>(x, mg.r, mg.p, mg.q, mg.sc, mg.partA);
    MGCK(reduce(b, mg.partA, nullptr, np, kRedStore, kScRR));
    MGCK(cudaMemcpyAsync(h, mg.sc, sizeof(double) * kScCount, cudaMemcpyDeviceToHost, st));
    MGCK(cudaStreamSynchronize(st));   // one host poll per outer iteration (the coarse solve polls anyway)
    c.launches += 8;
    accumulate_level_ms(mg);
    if (!(h[kScPQ] > 0.0) || !std::isfinite(h[kScPQ]) || !std::isfinite(h[kScAlpha]) || !std::isfinite(h[kScRR])) {
      // not SPD on this Krylov space (or a non-finite step): k_mg_fcg_update left x and r alone, so u and
      // relres are those of the last sound iterate
      status = FEA_SAMPLE_BREAKDOWN;
      k_mg_fcg_residual<<<g, kT, 0, st>>>(A, F, b.rhs, x, mg.r, mg.p, mg.q, 1, mg.partA);
      MGCK(reduce(b, mg.partA, nullptr, np, kRedStore, kScTrue));
      break;
    }
    ++it;
    first = 0;
    rr = h[kScRR];
  }
  if (status == FEA_SAMPLE_MAX_ITER || status == FEA_SAMPLE_STAGNATED) {
    k_mg_fcg_residual<<<g, kT, 0, st>>>(A, F, b.rhs, x, mg.r, mg.p, mg.q, 1, mg.partA);
    MGCK(reduce(b, mg.partA, nullptr, np, kRedStore, kScTrue));
  }
  k_mg_finish<<<1, 32, 0, st>>>(b.sc, b.rz_last, mg.sc, status, it);
  MGCK(cudaGetLastError());
  MGCK(launch_finalize(b));
  MGCK(cudaEventRecord(ev1, st));
  MGCK(cudaStreamSynchronize(st));
  b.stats.iterations = it;
  b.stats.n_converged = status == FEA_SAMPLE_CONVERGED ? 1 : 0;
  b.stats.refined_systems = restarts > 0 ? 1 : 0;
  cudaEventElapsedTime(&b.stats.solve_ms, ev0, ev1);
  c.launches += 8;
  b.stats.kernel_launches = c.launches - launches0;
  return FEA_OK;
}

void mg_release(Batch& b) {
  if (!b.mg) return;
  Mg* mg = b.mg;
  for (auto& L : mg->lev)
    if (L.hb) api_free_batch(L.hb);
  for (auto& ev : mg->ev) cudaEventDestroy(ev);
  if (mg->h_sc) cudaFreeHost(mg->h_sc);
  delete mg;
  b.mg = nullptr;
}

}  // namespace fea
