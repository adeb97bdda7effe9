// K6: rasterisation of the step-1 displacement components to the displacement_x / displacement_y
// gray images -- replaces custom_plotter.plot -> pyvista -> VTK off-screen rendering
// (reference datagen/fea_analysis.py:526-613, datagen/custom_plotter.py:121-193; SURVEY A-16).
//
// Semantics (identical to oracle/raster_oracle.py, operation for operation): a pixel is sampled
// at its centre; it belongs to the lowest-index triangle that contains the centre (edges
// inclusive); the scalar is interpolated barycentrically, normalised by the sample's own
// [min, max], and mapped through the 'binary' LUT: gray = 255 - min(floor(256 t), 255);
// background 255.  All coordinate arithmetic uses the *_rn intrinsics so that no FMA
// contraction can make coverage differ from the numpy oracle.
#include "fea_internal.cuh"

namespace fea {

__global__ void k_owner_init(int64_t n, int32_t* __restrict__ owner) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) owner[i] = 0x7fffffff;
}

struct Tri {
  double X[3], Y[3];
};

__device__ __forceinline__ void bary(const Tri& t, double qx, double qy, double w[3], double* area2) {
  const double ax = t.X[0], bx = t.X[1], cx = t.X[2];
  const double ay = t.Y[0], by = t.Y[1], cy = t.Y[2];
  double wa = __dsub_rn(__dmul_rn(__dsub_rn(bx, qx), __dsub_rn(cy, qy)), __dmul_rn(__dsub_rn(cx, qx), __dsub_rn(by, qy)));
  double wb = __dsub_rn(__dmul_rn(__dsub_rn(cx, qx), __dsub_rn(ay, qy)), __dmul_rn(__dsub_rn(ax, qx), __dsub_rn(cy, qy)));
  double wc = __dsub_rn(__dmul_rn(__dsub_rn(ax, qx), __dsub_rn(by, qy)), __dmul_rn(__dsub_rn(bx, qx), __dsub_rn(ay, qy)));
  double a2 = __dsub_rn(__dmul_rn(__dsub_rn(bx, ax), __dsub_rn(cy, ay)), __dmul_rn(__dsub_rn(cx, ax), __dsub_rn(by, ay)));
  const double sgn = a2 < 0.0 ? -1.0 : 1.0;
  w[0] = __dmul_rn(wa, sgn);
  w[1] = __dmul_rn(wb, sgn);
  w[2] = __dmul_rn(wc, sgn);
  *area2 = __dmul_rn(a2, sgn);
}

template <int NPC>
__device__ __forceinline__ void load_tri(int64_t cell, int sub, const int32_t* __restrict__ conn,
                                         const double* __restrict__ xy, const double* __restrict__ aff,
                                         Tri& t, int32_t vid[3]) {
  const int l0 = 0, l1 = (NPC == 3) ? 1 : (sub ? 2 : 1), l2 = (NPC == 3) ? 2 : (sub ? 3 : 2);
  const int ls[3] = {l0, l1, l2};
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int32_t v = conn[cell * NPC + ls[k]];
    vid[k] = v;
    t.X[k] = __dadd_rn(__dmul_rn(xy[2 * (int64_t)v], aff[0]), aff[1]);
    t.Y[k] = __dadd_rn(__dmul_rn(xy[2 * (int64_t)v + 1], aff[2]), aff[3]);
  }
}

template <int NPC>
__global__ void k_raster_cover(int64_t NT, const int64_t* __restrict__ cell_off, int ns,
                               const int32_t* __restrict__ conn, const double* __restrict__ xy,
                               const double* __restrict__ affine, int size, int32_t* __restrict__ owner) {
  constexpr int SUB = (NPC == 3) ? 1 : 2;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= NT) return;
  const int64_t cell = tid / SUB;
  const int sub = (int)(tid % SUB);
  const int s = seg_of(cell_off, ns, cell);
  const int32_t local = (int32_t)((cell - cell_off[s]) * SUB + sub);
  Tri t;
  int32_t vid[3];
  load_tri<NPC>(cell, sub, conn, xy, affine + 4 * s, t, vid);
  const double mnx = fmin(t.X[0], fmin(t.X[1], t.X[2])), mxx = fmax(t.X[0], fmax(t.X[1], t.X[2]));
  const double mny = fmin(t.Y[0], fmin(t.Y[1], t.Y[2])), mxy = fmax(t.Y[0], fmax(t.Y[1], t.Y[2]));
  const double fi0 = fmax(ceil(__dsub_rn(mnx, 0.5)), 0.0), fi1 = fmin(floor(__dsub_rn(mxx, 0.5)), (double)(size - 1));
  const double fj0 = fmax(ceil(__dsub_rn(mny, 0.5)), 0.0), fj1 = fmin(floor(__dsub_rn(mxy, 0.5)), (double)(size - 1));
  if (!(fi1 >= fi0 && fj1 >= fj0)) return;
  const int i0 = (int)fi0, i1 = (int)fi1, j0 = (int)fj0, j1 = (int)fj1;
  int32_t* own = owner + (int64_t)s * size * size;
  for (int j = j0; j <= j1; ++j) {
    for (int i = i0; i <= i1; ++i) {
      double w[3], a2;
      bary(t, (double)i + 0.5, (double)j + 0.5, w, &a2);
      if (w[0] >= 0.0 && w[1] >= 0.0 && w[2] >= 0.0 && a2 != 0.0) atomicMin(&own[j * size + i], local);
    }
  }
}

// Gray level of component c of a displacement u at a pixel of triangle vid (weights w / a2): value_scale * u
// interpolated, normalised by value_scale * (rng[2c], rng[2c+1]).  Every displacement image is shaded by this.
__device__ __forceinline__ uint8_t shade_displacement(const double w[3], double a2, const int32_t vid[3],
                                                      const double* __restrict__ u, int c, const double* __restrict__ rng4,
                                                      double value_scale) {
  const double s0 = __dmul_rn(value_scale, u[2 * (int64_t)vid[0] + c]);
  const double s1 = __dmul_rn(value_scale, u[2 * (int64_t)vid[1] + c]);
  const double s2 = __dmul_rn(value_scale, u[2 * (int64_t)vid[2] + c]);
  const double val = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(w[0], s0), __dmul_rn(w[1], s1)), __dmul_rn(w[2], s2)), a2);
  const double vmin = __dmul_rn(value_scale, rng4[2 * c]);
  const double vmax = __dmul_rn(value_scale, rng4[2 * c + 1]);
  const double rng = __dsub_rn(vmax, vmin);
  double tt = 0.0;
  if (rng > 0.0) tt = __ddiv_rn(__dsub_rn(val, vmin), rng);
  tt = fmin(fmax(tt, 0.0), 1.0);
  const double q = fmin(floor(__dmul_rn(256.0, tt)), 255.0);
  return (uint8_t)(255.0 - q);
}

template <int NPC>
__global__ void k_raster_shade(int ns, int size, const int64_t* __restrict__ cell_off,
                               const int32_t* __restrict__ conn, const double* __restrict__ xy,
                               const double* __restrict__ affine, const int32_t* __restrict__ owner,
                               const double* __restrict__ u, const double* __restrict__ ranges,
                               double value_scale, uint8_t* __restrict__ images) {
  constexpr int SUB = (NPC == 3) ? 1 : 2;
  const int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)size * size;
  if (pix >= per * ns) return;
  const int s = (int)(pix / per);
  const int64_t lp = pix - (int64_t)s * per;
  const int j = (int)(lp / size), i = (int)(lp - (int64_t)j * size);
  const int32_t o = owner[pix];
  uint8_t g0 = 255, g1 = 255;
  if (o != 0x7fffffff) {
    const int64_t cell = cell_off[s] + o / SUB;
    Tri t;
    int32_t vid[3];
    load_tri<NPC>(cell, o % SUB, conn, xy, affine + 4 * s, t, vid);
    double w[3], a2;
    bary(t, (double)i + 0.5, (double)j + 0.5, w, &a2);
    uint8_t g[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) g[c] = shade_displacement(w, a2, vid, u, c, ranges + 4 * s, value_scale);
    g0 = g[0];
    g1 = g[1];
  }
  images[((int64_t)s * 2 + 0) * per + lp] = g0;
  images[((int64_t)s * 2 + 1) * per + lp] = g1;
}

// Generic scalar fields of ONE mesh -- per vertex (region flags, the constant "1" field of
// input.png: reference fea_analysis.py:472-524) or per cell (cauchy_strain / cauchy_stress
// components, :541-549): field f is normalised by clim[f] and mapped like above.
template <int NPC>
__global__ void k_raster_shade_fields(int size, const int32_t* __restrict__ conn, const double* __restrict__ xy,
                                      const double* __restrict__ affine, const int32_t* __restrict__ owner,
                                      const double* __restrict__ fields, int64_t n_per_field, int n_fields,
                                      int cell_fields, const double* __restrict__ clim,
                                      uint8_t* __restrict__ images) {
  constexpr int SUB = (NPC == 3) ? 1 : 2;
  const int64_t lp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)size * size;
  if (lp >= per) return;
  const int j = (int)(lp / size), i = (int)(lp - (int64_t)j * size);
  const int32_t o = owner[lp];
  if (o == 0x7fffffff) {
    for (int f = 0; f < n_fields; ++f) images[(int64_t)f * per + lp] = 255;
    return;
  }
  Tri t;
  int32_t vid[3];
  load_tri<NPC>(o / SUB, o % SUB, conn, xy, affine, t, vid);
  double w[3], a2;
  bary(t, (double)i + 0.5, (double)j + 0.5, w, &a2);
  for (int f = 0; f < n_fields; ++f) {
    const double* __restrict__ fv = fields + (int64_t)f * n_per_field;
    const double val = cell_fields ? fv[o / SUB]
                                   : __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(w[0], fv[vid[0]]), __dmul_rn(w[1], fv[vid[1]])),
                                                         __dmul_rn(w[2], fv[vid[2]])), a2);
    const double vmin = clim[2 * f], rng = __dsub_rn(clim[2 * f + 1], vmin);
    double tt = 0.0;
    if (rng > 0.0) tt = __ddiv_rn(__dsub_rn(val, vmin), rng);
    tt = fmin(fmax(tt, 0.0), 1.0);
    images[(int64_t)f * per + lp] = (uint8_t)(255.0 - fmin(floor(__dmul_rn(256.0, tt)), 255.0));
  }
}

cudaError_t launch_raster_fields(cudaStream_t st, int npc, int64_t n_v, int64_t n_cell, const int32_t* conn,
                                 const double* xy, const double* affine, const int64_t* cell_off2, int size,
                                 int32_t* owner, const double* fields, int n_fields, int cell_fields,
                                 const double* clim, uint8_t* images) {
  const int T = 256;
  const int64_t per = (int64_t)size * size;
  k_owner_init<<<(unsigned)((per + T - 1) / T), T, 0, st>>>(per, owner);
  const int64_t NT = n_cell * (npc == 3 ? 1 : 2);
  if (NT) {
    const unsigned g = (unsigned)((NT + T - 1) / T);
    if (npc == 3) k_raster_cover<3><<<g, T, 0, st>>>(NT, cell_off2, 1, conn, xy, affine, size, owner);
    else k_raster_cover<4><<<g, T, 0, st>>>(NT, cell_off2, 1, conn, xy, affine, size, owner);
  }
  const unsigned gp = (unsigned)((per + T - 1) / T);
  if (npc == 3) k_raster_shade_fields<3><<<gp, T, 0, st>>>(size, conn, xy, affine, owner, fields, cell_fields ? n_cell : n_v, n_fields, cell_fields, clim, images);
  else k_raster_shade_fields<4><<<gp, T, 0, st>>>(size, conn, xy, affine, owner, fields, cell_fields ? n_cell : n_v, n_fields, cell_fields, clim, images);
  return cudaGetLastError();
}

// Region-flag images of every sample of a batch (regions_<Region>.png of the dataset tree,
// reference fea_analysis.py:508-524): 0/1 vertex flags interpolated over the owner triangle of each
// pixel (owner map of the preceding fea_batch_rasterize), clim (0, 1), same colour map.
// One thread per (sample, pixel): the owner triangle and its barycentric weights are found once and reused for
// every region image of the sample (a dozen or more); a triangle none of whose vertices is in the region -- almost
// all of them, regions are small -- is white without any arithmetic.
template <int NPC>
__global__ void k_raster_flags(int ns, int size, const int64_t* __restrict__ field_off,
                               const int64_t* __restrict__ flag_off, const int64_t* __restrict__ cell_off,
                               const int64_t* __restrict__ vtx_off, const int32_t* __restrict__ conn,
                               const double* __restrict__ xy, const double* __restrict__ affine,
                               const int32_t* __restrict__ owner, const uint8_t* __restrict__ flags,
                               uint8_t* __restrict__ images) {
  constexpr int SUB = (NPC == 3) ? 1 : 2;
  const int64_t per = (int64_t)size * size;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)ns * per) return;
  const int s = (int)(gid / per);
  const int64_t lp = gid - (int64_t)s * per;
  const int nf = (int)(field_off[s + 1] - field_off[s]);
  if (nf == 0) return;
  uint8_t* __restrict__ out = images + field_off[s] * per + lp;
  const int32_t o = owner[gid];
  if (o == 0x7fffffff) {
    for (int f = 0; f < nf; ++f) out[(int64_t)f * per] = 255;
    return;
  }
  const int j = (int)(lp / size), i = (int)(lp - (int64_t)j * size);
  const int64_t cell = cell_off[s] + o / SUB;
  Tri t;
  int32_t vid[3];
  load_tri<NPC>(cell, o % SUB, conn, xy, affine + 4 * s, t, vid);
  double w[3], a2;
  bary(t, (double)i + 0.5, (double)j + 0.5, w, &a2);
  const int64_t nv = vtx_off[s + 1] - vtx_off[s];
  const uint8_t* fl = flags + flag_off[s] - vtx_off[s];   // indexed by GLOBAL vertex id
  for (int f = 0; f < nf; ++f, fl += nv) {
    const uint8_t f0 = fl[vid[0]], f1 = fl[vid[1]], f2 = fl[vid[2]];
    uint8_t g = 255;
    if (f0 | f1 | f2) {
      const double v0 = f0 ? 1.0 : 0.0, v1 = f1 ? 1.0 : 0.0, v2 = f2 ? 1.0 : 0.0;
      double tt = __ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(w[0], v0), __dmul_rn(w[1], v1)), __dmul_rn(w[2], v2)), a2);
      tt = fmin(fmax(tt, 0.0), 1.0);
      g = (uint8_t)(255.0 - fmin(floor(__dmul_rn(256.0, tt)), 255.0));
    }
    out[(int64_t)f * per] = g;
  }
}

cudaError_t launch_raster_flags(Batch& b, int64_t n_img, const int64_t* d_field_off, const int64_t* d_flag_off,
                                const uint8_t* d_flags, uint8_t* d_images) {
  const int T = 256;
  const int64_t n = (int64_t)b.ns * b.img_size * b.img_size;
  if (n == 0 || n_img == 0) return cudaSuccess;
  const unsigned g = (unsigned)((n + T - 1) / T);
  if (b.npc == 3)
    k_raster_flags<3><<<g, T, 0, b.ctx->stream>>>(b.ns, b.img_size, d_field_off, d_flag_off, b.d_cell_off, b.d_vtx_off,
                                                  b.conn, b.xy, b.affine, b.owner, d_flags, d_images);
  else
    k_raster_flags<4><<<g, T, 0, b.ctx->stream>>>(b.ns, b.img_size, d_field_off, d_flag_off, b.d_cell_off, b.d_vtx_off,
                                                  b.conn, b.xy, b.affine, b.owner, d_flags, d_images);
  return cudaGetLastError();
}

// Per-cell scalar images of every sample of a batch: component x / y of the final-step cauchy stress /
// strain cell averages at step 1 (outputs_{stress,strain}_{x,y}.png, reference fea_analysis.py:539-558:
// fields ("cauchy_stress", "c0") ..., each normalised to its own (min, max)).  Field id: 0 stress_x,
// 1 stress_y, 2 strain_x, 3 strain_y.  One CTA per (field, sample) finds the range first.
__device__ __forceinline__ const double* cell_component(int id, const double* strain, const double* stress) {
  return (id < 2 ? stress : strain) + (id & 1);
}
__global__ void k_cell_field_ranges(int ns, const int32_t* __restrict__ ids, const int64_t* __restrict__ cell_off,
                                    const double* __restrict__ strain, const double* __restrict__ stress,
                                    double* __restrict__ ranges) {
  __shared__ double sm[2][8];
  const int f = blockIdx.x / ns, s = blockIdx.x - f * ns;
  const double* src = cell_component(ids[f], strain, stress);
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double mn = inf, mx = -inf;
  for (int64_t c = cell_off[s] + threadIdx.x; c < cell_off[s + 1]; c += blockDim.x) {
    const double v = src[3 * c];
    mn = fmin(mn, v);
    mx = fmax(mx, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = mn; sm[1][threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) { mn = fmin(mn, sm[0][i]); mx = fmax(mx, sm[1][i]); }
    ranges[2 * blockIdx.x] = mn;
    ranges[2 * blockIdx.x + 1] = mx;
  }
}
// Gray level of the cell value v: scale * v normalised by scale * (rng[0], rng[1]).  Every cell-component image
// is shaded by this.
__device__ __forceinline__ uint8_t shade_cell(double scale, double v, const double* __restrict__ rng2) {
  const double val = __dmul_rn(scale, v);
  const double vmin = __dmul_rn(scale, rng2[0]), vmax = __dmul_rn(scale, rng2[1]);
  const double rng = __dsub_rn(vmax, vmin);
  double tt = 0.0;
  if (rng > 0.0) tt = __ddiv_rn(__dsub_rn(val, vmin), rng);
  tt = fmin(fmax(tt, 0.0), 1.0);
  return (uint8_t)(255.0 - fmin(floor(__dmul_rn(256.0, tt)), 255.0));
}
template <int NPC>
__global__ void k_raster_cell_fields(int ns, int size, int n_fields, const int32_t* __restrict__ ids,
                                     const int64_t* __restrict__ cell_off, const int32_t* __restrict__ owner,
                                     const double* __restrict__ strain, const double* __restrict__ stress,
                                     const double* __restrict__ ranges, double scale, uint8_t* __restrict__ images) {
  constexpr int SUB = (NPC == 3) ? 1 : 2;
  const int64_t per = (int64_t)size * size;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)n_fields * ns * per) return;
  const int f = (int)(gid / (ns * per));
  const int64_t rem = gid - (int64_t)f * ns * per;
  const int s = (int)(rem / per);
  const int64_t lp = rem - (int64_t)s * per;
  const int32_t o = owner[(int64_t)s * per + lp];
  uint8_t g = 255;
  if (o != 0x7fffffff) {
    const int64_t cell = cell_off[s] + o / SUB;
    g = shade_cell(scale, cell_component(ids[f], strain, stress)[3 * cell], ranges + 2 * (f * ns + s));
  }
  images[gid] = g;
}

cudaError_t launch_raster_cell_fields(Batch& b, int n_fields, const int32_t* d_ids, const double* d_strain,
                                      const double* d_stress, double scale, double* d_ranges, uint8_t* d_images) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const int64_t n = (int64_t)n_fields * b.ns * b.img_size * b.img_size;
  if (n == 0) return cudaSuccess;
  k_cell_field_ranges<<<n_fields * b.ns, 256, 0, st>>>(b.ns, d_ids, b.d_cell_off, d_strain, d_stress, d_ranges);
  const unsigned g = (unsigned)((n + T - 1) / T);
  if (b.npc == 3)
    k_raster_cell_fields<3><<<g, T, 0, st>>>(b.ns, b.img_size, n_fields, d_ids, b.d_cell_off, b.owner, d_strain, d_stress, d_ranges, scale, d_images);
  else
    k_raster_cell_fields<4><<<g, T, 0, st>>>(b.ns, b.img_size, n_fields, d_ids, b.d_cell_off, b.owner, d_strain, d_stress, d_ranges, scale, d_images);
  return cudaGetLastError();
}

// ---- the load cases of one triangle mesh (fea_batch_load_case_images / _cell_components, DESIGN.md 3.11) ----
// The cases share the mesh, so one cover pass finds each pixel's owner triangle for all of them, and one thread
// per pixel computes that triangle's weights once and shades every case (and field) from them with the helpers
// of the single-batch kernels above: case k's pixels are, bit for bit, those of a batch solved with load k.
__global__ void k_raster_shade_cases(int n_cases, int size, const int32_t* __restrict__ conn, const double* __restrict__ xy,
                                     const double* __restrict__ affine, const int32_t* __restrict__ owner,
                                     const double* __restrict__ u, int64_t u_stride, const double* __restrict__ ranges,
                                     double value_scale, uint8_t* __restrict__ images) {
  const int64_t lp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)size * size;
  if (lp >= per) return;
  const int32_t o = owner[lp];
  if (o == 0x7fffffff) {
    for (int m = 0; m < 2 * n_cases; ++m) images[(int64_t)m * per + lp] = 255;
    return;
  }
  const int j = (int)(lp / size), i = (int)(lp - (int64_t)j * size);
  Tri t;
  int32_t vid[3];
  load_tri<3>(o, 0, conn, xy, affine, t, vid);
  double w[3], a2;
  bary(t, (double)i + 0.5, (double)j + 0.5, w, &a2);
  for (int k = 0; k < n_cases; ++k) {
#pragma unroll
    for (int c = 0; c < 2; ++c)
      images[(2 * (int64_t)k + c) * per + lp] = shade_displacement(w, a2, vid, u + k * u_stride, c, ranges + 4 * k, value_scale);
  }
}

__global__ void k_raster_cell_fields_cases(int n_cases, int size, int n_fields, const int32_t* __restrict__ ids, int64_t nc,
                                           const int32_t* __restrict__ owner, const double* __restrict__ strain,
                                           const double* __restrict__ stress, const double* __restrict__ ranges,
                                           double scale, uint8_t* __restrict__ images) {
  const int64_t lp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = (int64_t)size * size;
  if (lp >= per) return;
  const int32_t o = owner[lp];
  for (int f = 0; f < n_fields; ++f) {
    const double* src = cell_component(ids[f], strain, stress);
    for (int k = 0; k < n_cases; ++k) {
      uint8_t g = 255;
      if (o != 0x7fffffff) g = shade_cell(scale, src[3 * (k * nc + o)], ranges + 2 * (f * n_cases + k));
      images[((int64_t)f * n_cases + k) * per + lp] = g;
    }
  }
}

cudaError_t launch_case_owner(Batch& b, int size, const double* d_affine, int32_t* owner) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const int64_t per = (int64_t)size * size;
  k_owner_init<<<(unsigned)((per + T - 1) / T), T, 0, st>>>(per, owner);
  if (b.NC) k_raster_cover<3><<<(unsigned)((b.NC + T - 1) / T), T, 0, st>>>(b.NC, b.d_cell_off, 1, b.conn, b.xy, d_affine, size, owner);
  return cudaGetLastError();
}

cudaError_t launch_case_raster(Batch& b, int n_cases, int size, const double* d_affine, const int32_t* owner,
                               const double* u, const double* ranges, double value_scale, uint8_t* d_images) {
  const int T = 256;
  const int64_t per = (int64_t)size * size;
  k_raster_shade_cases<<<(unsigned)((per + T - 1) / T), T, 0, b.ctx->stream>>>(n_cases, size, b.conn, b.xy, d_affine, owner, u,
                                                                                 2 * b.NV, ranges, value_scale, d_images);
  return cudaGetLastError();
}

cudaError_t launch_case_cell_fields(Batch& b, int n_cases, int size, const int32_t* owner, int n_fields,
                                    const int32_t* d_ids, const int64_t* d_case_off, const double* d_strain,
                                    const double* d_stress, double scale, double* d_ranges, uint8_t* d_images) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const int64_t per = (int64_t)size * size;
  // case k is "sample" k of the case-major strain / stress arrays: each (field, case) range is reduced by the
  // single-batch kernel in the single batch's order
  k_cell_field_ranges<<<n_fields * n_cases, 256, 0, st>>>(n_cases, d_ids, d_case_off, d_strain, d_stress, d_ranges);
  k_raster_cell_fields_cases<<<(unsigned)((per + T - 1) / T), T, 0, st>>>(n_cases, size, n_fields, d_ids, b.NC, owner, d_strain,
                                                                          d_stress, d_ranges, scale, d_images);
  return cudaGetLastError();
}

cudaError_t launch_raster(Batch& b, double value_scale) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const int64_t npix = (int64_t)b.ns * b.img_size * b.img_size;
  if (npix == 0) return cudaSuccess;
  k_owner_init<<<(unsigned)((npix + T - 1) / T), T, 0, st>>>(npix, b.owner);
  const int64_t NT = b.NC * (b.npc == 3 ? 1 : 2);
  if (NT) {
    const unsigned g = (unsigned)((NT + T - 1) / T);
    if (b.npc == 3) k_raster_cover<3><<<g, T, 0, st>>>(NT, b.d_cell_off, b.ns, b.conn, b.xy, b.affine, b.img_size, b.owner);
    else k_raster_cover<4><<<g, T, 0, st>>>(NT, b.d_cell_off, b.ns, b.conn, b.xy, b.affine, b.img_size, b.owner);
  }
  const unsigned gp = (unsigned)((npix + T - 1) / T);
  if (b.npc == 3)
    k_raster_shade<3><<<gp, T, 0, st>>>(b.ns, b.img_size, b.d_cell_off, b.conn, b.xy, b.affine, b.owner, b.u, b.ranges,
                                        value_scale, b.images);
  else
    k_raster_shade<4><<<gp, T, 0, st>>>(b.ns, b.img_size, b.d_cell_off, b.conn, b.xy, b.affine, b.owner, b.u, b.ranges,
                                        value_scale, b.images);
  return cudaGetLastError();
}

}  // namespace fea
