// Device-side problem set-up: everything FEAnalysis.__init__ (reference
// datagen/fea_analysis.py:76-146, 182-194, 235-252) derives from the condition dict -- region vertex
// sets, Dirichlet mask, material cells, D matrices, load vector -- plus the derived well-posedness
// classifier (SURVEY A-19).  Entry point: fea_batch_create_from_conditions.
//
// Exactness rules (the selectors decide set membership, so they must reproduce numpy bit for bit):
//   * collinearity |x1*y2 - x2*y1| < 1e-14 uses __dmul_rn / __dsub_rn: no FMA contraction
//     (fea_analysis.py:182-188);
//   * np.isin(coors, list).all(axis=1) is exact fp64 equality of scalars: one hash set per material
//     region over the bit patterns of its listed x and y values (-0.0 folded into +0.0, NaN never
//     matches), probed with the x and the y of every vertex (fea_analysis.py:190-194, A-18);
//   * 'facet' regions keep only vertices of mesh edges with both ends selected, 'cell' regions own
//     complete cells only (A-7, F4); a cell complete in several regions gets the sum of their D as
//     an extra material-table entry, numbered in order of first occurrence by cell index (the
//     numbering host.ProblemSetup produces);
//   * loads are accumulated per vertex in the reference's order (vertex forces, then edge forces),
//     an edge force divided by max(#region vertices, 1) (fea_analysis.py:99-105), times the number
//     of LHS terms (F2).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>
#include <new>
#include <vector>

#include "fea_internal.cuh"

namespace fea {

constexpr int kMaxMat = 32;     // material regions per sample (cell membership is a 32-bit mask)
constexpr int kMaxCombo = 16;   // distinct overlap combinations (A-18) per sample
constexpr unsigned long long kEmptyKey = ~0ull;   // a NaN pattern: never a stored key

enum RegionKind : int32_t { kVForce = 0, kEForce = 1, kVFix = 2, kEFix = 3, kMaterial = 4, kPlateMask = 5 };

struct Region {            // one row of a sample's flag block
  int32_t sample;
  int32_t kind;
  int32_t i0, i1;          // sample-local vertex indices of the tags (numpy wrap-around applied), -1 = out of range
  double mx, my;           // force magnitude
  int64_t flag_off;        // first byte of the row in rflags
  int64_t tab_off;         // material: first slot of the hash set
  int32_t tab_mask;        // material: slots - 1
  int32_t mat_local;       // material: index inside the sample
};

struct SampleCond {
  int32_t reg0;            // first region (rows: vforce, eforce, vfix, efix, material, plate mask)
  int32_t n_vf, n_ef, n_vc, n_ec, n_mat;
  int32_t mesh;
  int32_t pad_;
  double E, nu;            // default material of a sample without a table
};

__device__ __forceinline__ uint32_t hash_bits(unsigned long long x) {
  x ^= x >> 33;
  x *= 0xff51afd7ed558ccdULL;
  x ^= x >> 33;
  x *= 0xc4ceb9fe1a85ec53ULL;
  x ^= x >> 33;
  return (uint32_t)x;
}
__device__ __forceinline__ bool canon_key(double v, unsigned long long* key) {
  if (v != v) return false;          // NaN equals nothing
  if (v == 0.0) v = 0.0;             // -0.0 == 0.0
  *key = (unsigned long long)__double_as_longlong(v);
  return true;
}

// ---- mesh replication: every sample gets its own copy of its plate's mesh ----------------------
__global__ void k_replicate_vertices(const SampleCond* __restrict__ sc, const int64_t* __restrict__ vtx_off,
                                     const int64_t* __restrict__ mesh_vtx_off, const double2* __restrict__ mesh_xy,
                                     double2* __restrict__ xy) {
  const int s = blockIdx.x;
  const int64_t nv = vtx_off[s + 1] - vtx_off[s];
  const int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  xy[vtx_off[s] + i] = mesh_xy[mesh_vtx_off[sc[s].mesh] + i];
}
__global__ void k_replicate_cells(const SampleCond* __restrict__ sc, const int64_t* __restrict__ cell_off, int npc,
                                  const int64_t* __restrict__ mesh_cell_off, const int32_t* __restrict__ mesh_conn,
                                  int32_t* __restrict__ conn_local) {
  const int s = blockIdx.x;
  const int64_t n = (cell_off[s + 1] - cell_off[s]) * npc;
  const int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (i >= n) return;
  conn_local[cell_off[s] * npc + i] = mesh_conn[mesh_cell_off[sc[s].mesh] * npc + i];
}

// ---- hash sets of the material coordinate lists -------------------------------------------------
__global__ void k_hash_insert(int64_t n_scalars, int n_mat_regions, const int64_t* __restrict__ coord_off,
                              const int32_t* __restrict__ mat_region, const Region* __restrict__ reg,
                              const double* __restrict__ coords, unsigned long long* __restrict__ tab) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_scalars) return;
  const int m = seg_of(coord_off, n_mat_regions, i >> 1);   // material region (global index) of point i/2
  unsigned long long key;
  if (!canon_key(coords[i], &key)) return;
  const Region& R = reg[mat_region[m]];
  uint32_t slot = hash_bits(key) & (uint32_t)R.tab_mask;
  for (;;) {
    const unsigned long long prev = atomicCAS(tab + R.tab_off + slot, kEmptyKey, key);
    if (prev == kEmptyKey || prev == key) return;
    slot = (slot + 1) & (uint32_t)R.tab_mask;
  }
}
__device__ __forceinline__ bool hash_contains(const unsigned long long* __restrict__ tab, const Region& R, double v) {
  unsigned long long key;
  if (!canon_key(v, &key)) return false;
  uint32_t slot = hash_bits(key) & (uint32_t)R.tab_mask;
  for (;;) {
    const unsigned long long k = tab[R.tab_off + slot];
    if (k == key) return true;
    if (k == kEmptyKey) return false;
    slot = (slot + 1) & (uint32_t)R.tab_mask;
  }
}

// ---- region selection, pass 1: candidate vertex sets --------------------------------------------
// grid.x = region row, grid.y = chunks of vertices.  Vertex-kind rows and the plate mask are final
// here; edge and material rows write their candidate set V0 and are finished by k_region_cells.
__global__ void k_region_vertices(const Region* __restrict__ reg, const int64_t* __restrict__ vtx_off,
                                  const double2* __restrict__ xy, const unsigned long long* __restrict__ tab,
                                  uint8_t* __restrict__ v0, uint8_t* __restrict__ flags) {
  const Region R = reg[blockIdx.x];
  const int64_t base = vtx_off[R.sample];
  const int64_t nv = vtx_off[R.sample + 1] - base;
  const int64_t v = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  uint8_t cand = 0, fin = 0;
  switch (R.kind) {
    case kVForce:
    case kVFix:
      fin = v == R.i0;
      break;
    case kPlateMask:
      fin = 1;
      break;
    case kEForce:
    case kEFix:
      if (R.i0 >= 0 && R.i1 >= 0) {   // fea_analysis.py:182-188, numpy operation order, no FMA
        const double2 p0 = xy[base + R.i0], p1 = xy[base + R.i1], p = xy[base + v];
        const double x1 = __dsub_rn(p1.x, p0.x), y1 = __dsub_rn(p1.y, p0.y);
        const double x2 = __dsub_rn(p.x, p0.x), y2 = __dsub_rn(p.y, p0.y);
        cand = fabs(__dsub_rn(__dmul_rn(x1, y2), __dmul_rn(x2, y1))) < 1e-14;
      }
      break;
    default: {                        // fea_analysis.py:190-194: x AND y among the listed scalars
      const double2 p = xy[base + v];
      cand = hash_contains(tab, R, p.x) && hash_contains(tab, R, p.y);
    }
  }
  v0[R.flag_off + v] = cand;
  flags[R.flag_off + v] = fin;
}

// ---- pass 2: facet / cell semantics (A-7) -------------------------------------------------------
template <int NPC>
__global__ void k_region_cells(const Region* __restrict__ reg, const int64_t* __restrict__ vtx_off,
                               const int64_t* __restrict__ cell_off, const int32_t* __restrict__ conn_local,
                               const uint8_t* __restrict__ v0, uint8_t* __restrict__ flags,
                               uint32_t* __restrict__ cell_member) {
  const Region R = reg[blockIdx.x];
  if (R.kind != kEForce && R.kind != kEFix && R.kind != kMaterial) return;
  const int64_t nv = vtx_off[R.sample + 1] - vtx_off[R.sample];
  const int64_t c0 = cell_off[R.sample], nc = cell_off[R.sample + 1] - c0;
  const int64_t c = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  int32_t v[NPC];
  bool in[NPC];
#pragma unroll
  for (int a = 0; a < NPC; ++a) {
    v[a] = conn_local[(c0 + c) * NPC + a];
    if (v[a] < 0 || v[a] >= nv) return;   // reported by k_cells
    in[a] = v0[R.flag_off + v[a]] != 0;
  }
  uint8_t* fl = flags + R.flag_off;
  if (R.kind == kMaterial) {
    bool all = true;
#pragma unroll
    for (int a = 0; a < NPC; ++a) all = all && in[a];
    if (all) {
      atomicOr(cell_member + c0 + c, 1u << R.mat_local);
#pragma unroll
      for (int a = 0; a < NPC; ++a) fl[v[a]] = 1;
    }
  } else {
#pragma unroll
    for (int a = 0; a < NPC; ++a) {
      const int n = (a + 1) % NPC;
      if (in[a] && in[n]) { fl[v[a]] = 1; fl[v[n]] = 1; }
    }
  }
}

// one CTA per region row: number of region vertices
__global__ void k_region_count(const Region* __restrict__ reg, const int64_t* __restrict__ vtx_off,
                               const uint8_t* __restrict__ flags, int32_t* __restrict__ rcount) {
  __shared__ int sm[32];
  const Region R = reg[blockIdx.x];
  const int64_t nv = vtx_off[R.sample + 1] - vtx_off[R.sample];
  int n = 0;
  for (int64_t v = threadIdx.x; v < nv; v += blockDim.x) n += flags[R.flag_off + v] != 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
    rcount[blockIdx.x] = t;
  }
}

// ---- Dirichlet mask and load vector (grid.x = sample, grid.y = vertex chunks) -------------------
__global__ void k_fixed_rhs(const SampleCond* __restrict__ sc, const Region* __restrict__ reg,
                            const int64_t* __restrict__ vtx_off, const uint8_t* __restrict__ flags,
                            const int32_t* __restrict__ rcount, uint8_t* __restrict__ fixed,
                            double2* __restrict__ rhs) {
  const SampleCond S = sc[blockIdx.x];
  const int64_t base = vtx_off[blockIdx.x];
  const int64_t nv = vtx_off[blockIdx.x + 1] - base;
  const int64_t v = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (v >= nv) return;
  double ax = 0.0, ay = 0.0;
  int r = S.reg0;
  for (int i = 0; i < S.n_vf; ++i, ++r) {           // dw_point_load on 'vertex k' (fea_analysis.py:76-91)
    if (v == reg[r].i0) {
      ax = __dadd_rn(ax, reg[r].mx);
      ay = __dadd_rn(ay, reg[r].my);
    }
  }
  for (int i = 0; i < S.n_ef; ++i, ++r) {           // edge force: F / max(#vertices, 1) at every region vertex (:93-115)
    if (flags[reg[r].flag_off + v]) {
      const double cnt = (double)max(rcount[r], 1);
      ax = __dadd_rn(ax, __ddiv_rn(reg[r].mx, cnt));
      ay = __dadd_rn(ay, __ddiv_rn(reg[r].my, cnt));
    }
  }
  uint8_t fx = 0;
  for (int i = 0; i < S.n_vc + S.n_ec; ++i, ++r) fx |= flags[reg[r].flag_off + v];   // EssentialBC 'u.all': 0 (:127-138)
  const double terms = (double)(S.n_mat > 0 ? S.n_mat : 1);   // one Equation per LHS term, each with ALL loads (F2)
  fixed[base + v] = fx ? 1 : 0;
  rhs[base + v] = make_double2(__dmul_rn(terms, ax), __dmul_rn(terms, ay));
}

// ---- material table index of every cell (grid.x = sample, grid.y = cell chunks) -----------------
__global__ void k_cell_region(const SampleCond* __restrict__ sc, const int64_t* __restrict__ cell_off,
                              const uint32_t* __restrict__ cell_member, uint32_t* __restrict__ combo_mask,
                              int32_t* __restrict__ combo_first, int8_t* __restrict__ creg, int32_t* __restrict__ err_flag) {
  const int s = blockIdx.x;
  const int64_t c0 = cell_off[s], nc = cell_off[s + 1] - c0;
  const int64_t c = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  int r;
  if (sc[s].n_mat == 0) {
    r = 0;                                     // single material over Omega
  } else {
    const uint32_t m = cell_member[c0 + c];
    const int n = __popc(m);
    if (n == 0) r = -1;                        // seam cell: no stiffness (F4)
    else if (n == 1) r = __ffs(m) - 1;
    else {                                     // complete in several regions (A-18): sum of their D
      int slot = -1;
      for (int i = 0; i < kMaxCombo && slot < 0; ++i) {
        const uint32_t prev = atomicCAS(combo_mask + s * kMaxCombo + i, 0u, m);
        if (prev == 0u || prev == m) slot = i;
      }
      if (slot < 0) { atomicOr(err_flag, 4); r = -1; }
      else {
        atomicMin(combo_first + s * kMaxCombo + slot, (int32_t)c);
        r = -2 - slot;
      }
    }
  }
  creg[c0 + c] = (int8_t)r;
}

__device__ __forceinline__ void plane_strain(double E, double nu, double* D) {
  // stiffness_from_youngpoisson(dim=2, ...), sfepy default plane='strain' (fea_analysis.py:263-265, F1),
  // operation order of host.stiffness_plane_strain, no contraction
  const double lam = __ddiv_rn(__dmul_rn(E, nu), __dmul_rn(__dadd_rn(1.0, nu), __dsub_rn(1.0, __dmul_rn(2.0, nu))));
  const double mu = __ddiv_rn(E, __dmul_rn(2.0, __dadd_rn(1.0, nu)));
  const double d = __dadd_rn(lam, __dmul_rn(2.0, mu));
  D[0] = d;   D[1] = lam; D[2] = 0.0;
  D[3] = lam; D[4] = d;   D[5] = 0.0;
  D[6] = 0.0; D[7] = 0.0; D[8] = mu;
}

// one thread per sample: D of every material term, overlap combinations numbered by first cell
__global__ void k_material_table(int ns, const SampleCond* __restrict__ sc, const int32_t* __restrict__ reg_off,
                                 const double* __restrict__ mat_E_nu, const int32_t* __restrict__ mat_first,
                                 const uint32_t* __restrict__ combo_mask, const int32_t* __restrict__ combo_first,
                                 int32_t* __restrict__ combo_id, double* __restrict__ D, int32_t* __restrict__ n_used) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ns) return;
  const SampleCond S = sc[s];
  double* Ds = D + (int64_t)reg_off[s] * 9;
  if (S.n_mat == 0) {
    plane_strain(S.E, S.nu, Ds);
    n_used[s] = 1;
    return;
  }
  for (int j = 0; j < S.n_mat; ++j) plane_strain(mat_E_nu[2 * (mat_first[s] + j)], mat_E_nu[2 * (mat_first[s] + j) + 1], Ds + 9 * j);
  int order[kMaxCombo], n = 0;
  for (int i = 0; i < kMaxCombo; ++i)
    if (combo_mask[s * kMaxCombo + i]) {
      int k = n++;
      while (k > 0 && combo_first[s * kMaxCombo + order[k - 1]] > combo_first[s * kMaxCombo + i]) { order[k] = order[k - 1]; --k; }
      order[k] = i;
    }
  for (int k = 0; k < n; ++k) {
    const int slot = order[k];
    combo_id[s * kMaxCombo + slot] = S.n_mat + k;
    double* Dc = Ds + 9 * (S.n_mat + k);
    uint32_t m = combo_mask[s * kMaxCombo + slot];
    bool first = true;
    while (m) {                                   // sum(Ds[r] for r in key), ascending region index
      const int r = __ffs(m) - 1;
      m &= m - 1;
      for (int e = 0; e < 9; ++e) Dc[e] = first ? Ds[9 * r + e] : __dadd_rn(Dc[e], Ds[9 * r + e]);
      first = false;
    }
  }
  n_used[s] = S.n_mat + n;
}

__global__ void k_cell_region_combos(const int64_t* __restrict__ cell_off, const int32_t* __restrict__ combo_id,
                                     int8_t* __restrict__ creg) {
  const int s = blockIdx.x;
  const int64_t c0 = cell_off[s], nc = cell_off[s + 1] - c0;
  const int64_t c = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const int r = creg[c0 + c];
  if (r <= -2) creg[c0 + c] = (int8_t)combo_id[s * kMaxCombo + (-2 - r)];
}

// ===========================================================================
// A-19 classifier: parts of the stiffness mesh (cells joined through shared edges) with fewer than
// two fixed vertices, and active vertices without any stiffness cell.  Lock-free union-find over
// the cells (roots are hooked with atomicCAS in a fixed pseudo-random order of the indices), so the
// partition -- and with it every count -- is independent of the execution order.
// ===========================================================================
// Which of two roots goes under the other is decided by a fixed pseudo-random order of the cell indices (a
// bijective hash), not by the indices themselves: cells are numbered along the mesh, and "larger index under
// smaller" with thousands of concurrent unions of neighbouring cells builds chains as long as a strip of the mesh
// (measured: 27 k cycles per union on a 9 k-cell plate), a random order keeps them logarithmic.
__device__ __forceinline__ uint32_t cc_prio(int x) {
  uint32_t h = (uint32_t)x * 0x9E3779B1u;
  h ^= h >> 15;
  h *= 0x85EBCA77u;
  h ^= h >> 13;
  return h;
}
__device__ __forceinline__ int cc_find(int32_t* parent, int x) {
  for (;;) {
    const int p = __ldcg(parent + x);
    if (p == x) return x;
    const int gp = __ldcg(parent + p);
    if (gp != p) parent[x] = gp;   // path halving (x is not a root and never becomes one again)
    x = p;
  }
}
__device__ __forceinline__ void cc_union(int32_t* parent, int a, int b) {
  for (;;) {
    a = cc_find(parent, a);
    b = cc_find(parent, b);
    if (a == b) return;
    if (cc_prio(a) < cc_prio(b)) { const int t = a; a = b; b = t; }
    const int old = atomicCAS(parent + a, a, b);
    if (old == a) return;
  }
}
__global__ void k_cc_init(int64_t NC, const int32_t* __restrict__ cell_dreg, int32_t* __restrict__ parent) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < NC) parent[c] = cell_dreg[c] >= 0 ? (int32_t)c : -1;
}
template <int NPC>
__global__ void k_cc_union(int64_t NC, const int32_t* __restrict__ conn, const int32_t* __restrict__ cell_dreg,
                           const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                           int32_t* __restrict__ parent) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t c = gid / NPC;
  const int a = (int)(gid - c * NPC);
  if (c >= NC || cell_dreg[c] < 0) return;
  const int va = conn[c * NPC + a], vb = conn[c * NPC + (a + 1) % NPC];
  for (int i = inc_ptr[va]; i < inc_ptr[va + 1]; ++i) {
    const int64_t c2 = inc[i] >> 2;
    if (c2 <= c) continue;                       // every pair once
    bool has = false;
#pragma unroll
    for (int k = 0; k < NPC; ++k) has = has || conn[c2 * NPC + k] == vb;
    if (has) cc_union(parent, (int)c, (int)c2);
  }
}
__global__ void k_cc_flatten(int64_t NC, int32_t* __restrict__ parent) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < NC && __ldcg(parent + c) >= 0) {
    const int r = cc_find(parent, (int)c);
    parent[c] = r;
  }
}
__global__ void k_cc_vertices(int64_t NV, const uint8_t* __restrict__ fixed, const int32_t* __restrict__ vsample,
                              const int32_t* __restrict__ inc_ptr, const int32_t* __restrict__ inc,
                              int32_t* __restrict__ parent, int32_t* __restrict__ nfix, int32_t* __restrict__ empty_cnt) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV) return;
  const int b = inc_ptr[v], e = inc_ptr[v + 1];
  if (!fixed[v]) {
    if (b == e) atomicAdd(empty_cnt + vsample[v], 1);
    return;
  }
  int roots[kMaxAdj], n = 0;                      // (part, vertex) pairs once each
  for (int i = b; i < e; ++i) {
    const int r = cc_find(parent, inc[i] >> 2);
    bool seen = false;
    for (int k = 0; k < n; ++k) seen = seen || roots[k] == r;
    if (!seen && n < kMaxAdj) { roots[n++] = r; atomicAdd(nfix + r, 1); }
  }
}
__global__ void k_cc_count(int64_t NC, int npc, const int32_t* __restrict__ conn, const int32_t* __restrict__ vsample,
                           const int32_t* __restrict__ parent, const int32_t* __restrict__ nfix,
                           int32_t* __restrict__ floating) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= NC || parent[c] != (int32_t)c) return;
  if (nfix[c] < 2) atomicAdd(floating + vsample[conn[c * npc]], 1);
}

// The same classifier for plate-sized samples: ONE CTA per sample, parent links and fixed-vertex counts of the
// sample's cells in shared memory (8 bytes per cell), so the pointer chasing of the union-find costs shared-memory
// instead of L2 latencies (measured on the 400-sample bench batch: 2.0 ms with the global-memory kernels above,
// which remain for samples too large for shared memory).  Counts are independent of the execution order.
__device__ __forceinline__ int cc_find_s(volatile int32_t* parent, int x) {
  for (;;) {
    const int p = parent[x];
    if (p == x) return x;
    const int gp = parent[p];
    if (gp != p) parent[x] = gp;
    x = p;
  }
}
template <int NPC>
__global__ void __launch_bounds__(1024) k_cc_sample(const int64_t* __restrict__ cell_off, const int64_t* __restrict__ vtx_off,
                                                    const int32_t* __restrict__ conn, const int32_t* __restrict__ cell_dreg,
                                                    const uint8_t* __restrict__ fixed, const int32_t* __restrict__ inc_ptr,
                                                    const int32_t* __restrict__ inc, int32_t* __restrict__ floating,
                                                    int32_t* __restrict__ empty_cnt) {
  extern __shared__ int32_t cc_sm[];
  const int s = blockIdx.x;
  const int64_t c0 = cell_off[s], v0 = vtx_off[s];
  const int nc = (int)(cell_off[s + 1] - c0), nv = (int)(vtx_off[s + 1] - v0);
  int32_t* parent = cc_sm;
  int32_t* nfix = cc_sm + nc;
  __shared__ int32_t tot[2];
#ifdef FEA_CC_PROFILE
  long long tp[6];
  tp[0] = clock64();
#define CC_T(i) do { __syncthreads(); tp[i] = clock64(); } while (0)
#else
#define CC_T(i) do { } while (0)
#endif
  if (threadIdx.x < 2) tot[threadIdx.x] = 0;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) {
    parent[c] = cell_dreg[c0 + c] >= 0 ? c : -1;
    nfix[c] = 0;
  }
  __syncthreads();
  CC_T(1);
  // Two stiffness cells share an edge iff they share two vertices.  One thread per (cell c, corner a): the other
  // cells around the corner's vertex v come from v's incidence list; a cell c2 > c that also holds one of the two
  // edge neighbours w of v in c shares the edge (v, w) with c, which is handled at its smaller end (v < w).  All
  // loads of a step are issued together (up to 8 incidence entries, then the corners of those cells): four
  // dependent round trips per thread.  (A thread per vertex with the cells' corners in local arrays diverges in
  // its pair loop and ran no faster than k_cc_union's search, 1.0 - 1.2 M cycles per 9 k-cell sample.)
  for (int base = 0; base < nc * NPC; base += blockDim.x) {
    // the lanes of a warp leave the union loops below at different times: without an explicit reconvergence point
    // they run the rest of this loop one lane at a time (measured with ncu: 20 x the warp instructions, 2 M cycles
    // per 9 k-cell sample instead of 0.1 M)
    __syncwarp();
    const int gid = base + threadIdx.x;
    const int c = gid / NPC, a = gid - c * NPC;
    if (gid < nc * NPC && parent[c] >= 0) {
      const int32_t* cc = conn + (c0 + c) * NPC;
      const int v = cc[a], nxt = cc[(a + 1) % NPC], prv = cc[(a + NPC - 1) % NPC];
      const int b = inc_ptr[v], e = inc_ptr[v + 1];
      for (int m0 = b; m0 < e; m0 += 8) {
        int ent[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) ent[m] = m0 + m < e ? inc[m0 + m] : -1;
        int oth[8][NPC - 1];
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const int64_t c2 = ent[m] >> 2;
          const bool use = ent[m] >= 0 && (int)(c2 - c0) > c;         // every pair once
#pragma unroll
          for (int q = 1; q < NPC; ++q) oth[m][q - 1] = use ? conn[c2 * NPC + ((ent[m] & 3) + q) % NPC] : -1;
        }
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          bool adj = false;
#pragma unroll
          for (int q = 0; q < NPC - 1; ++q)
            adj = adj || (oth[m][q] > v && (oth[m][q] == nxt || oth[m][q] == prv));
          if (adj) {
            int x = c, y = (int)((ent[m] >> 2) - c0);
            for (;;) {                                   // lock-free union (cc_prio decides which root stays)
              x = cc_find_s(parent, x);
              y = cc_find_s(parent, y);
              if (x == y) break;
              if (cc_prio(x) < cc_prio(y)) { const int t = x; x = y; y = t; }
              if (atomicCAS(parent + x, x, y) == x) break;
            }
          }
        }
      }
    }
  }
  __syncthreads();
  CC_T(2);
  for (int c = threadIdx.x; c < nc; c += blockDim.x)
    if (parent[c] >= 0) parent[c] = cc_find_s(parent, c);
  __syncthreads();
  CC_T(3);
  int n_empty = 0;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const int b = inc_ptr[v0 + v], e = inc_ptr[v0 + v + 1];
    if (!fixed[v0 + v]) {
      n_empty += b == e ? 1 : 0;
      continue;
    }
    int roots[kMaxAdj], n = 0;                      // (part, vertex) pairs once each
    for (int i = b; i < e; ++i) {
      const int r = parent[(int)((inc[i] >> 2) - c0)];
      bool seen = false;
      for (int k = 0; k < n; ++k) seen = seen || roots[k] == r;
      if (!seen && n < kMaxAdj) { roots[n++] = r; atomicAdd(nfix + r, 1); }
    }
  }
  __syncthreads();
  CC_T(4);
  int n_float = 0;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) n_float += (parent[c] == c && nfix[c] < 2) ? 1 : 0;
  if (n_float) atomicAdd(&tot[0], n_float);
  if (n_empty) atomicAdd(&tot[1], n_empty);
  __syncthreads();
  if (threadIdx.x == 0) {
    floating[s] = tot[0];
    empty_cnt[s] = tot[1];
  }
#ifdef FEA_CC_PROFILE
  CC_T(5);
  if (threadIdx.x == 0 && (s == 0 || s == 200))
    printf("[cc] sample %d nc %d nv %d: init %lld union %lld flatten %lld vertices %lld count %lld cycles\n", s, nc, nv,
           tp[1] - tp[0], tp[2] - tp[1], tp[3] - tp[2], tp[4] - tp[3], tp[5] - tp[4]);
#endif
}

__global__ void k_merge_err(const int32_t* __restrict__ src, int32_t* __restrict__ dst) { *dst = *src; }

cudaError_t launch_classify(Batch& b, int32_t* d_floating, int32_t* d_empty) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  {   // plate-sized samples: one CTA per sample, union-find in shared memory
    int64_t max_nc = 0;
    for (int s = 0; s < b.ns; ++s) max_nc = std::max(max_nc, b.cell_off[s + 1] - b.cell_off[s]);
    const size_t bytes = (size_t)max_nc * 8;
    if (b.ns > 0 && max_nc > 0 && bytes <= 200 * 1024) {
      cudaError_t e;
      if (b.npc == 3) {
        if ((e = cudaFuncSetAttribute(k_cc_sample<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)) != cudaSuccess) return e;
        k_cc_sample<3><<<b.ns, 1024, bytes, st>>>(b.d_cell_off, b.d_vtx_off, b.conn, b.cell_dreg, b.fixed, b.inc_ptr, b.inc, d_floating, d_empty);
      } else {
        if ((e = cudaFuncSetAttribute(k_cc_sample<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)) != cudaSuccess) return e;
        k_cc_sample<4><<<b.ns, 1024, bytes, st>>>(b.d_cell_off, b.d_vtx_off, b.conn, b.cell_dreg, b.fixed, b.inc_ptr, b.inc, d_floating, d_empty);
      }
      b.ctx->launches += 1;
      return cudaGetLastError();
    }
  }
  Scratch scratch(st);
  int32_t *parent = nullptr, *nfix = nullptr;
  cudaError_t e;
  if ((e = cudaMemsetAsync(d_floating, 0, sizeof(int32_t) * b.ns, st)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(d_empty, 0, sizeof(int32_t) * b.ns, st)) != cudaSuccess) return e;
  if ((e = scratch.alloc(&parent, b.NC)) != cudaSuccess) return e;
  if ((e = scratch.alloc(&nfix, b.NC)) != cudaSuccess) return e;
  if ((e = cudaMemsetAsync(nfix, 0, sizeof(int32_t) * std::max<int64_t>(1, b.NC), st)) != cudaSuccess) return e;
  if (b.NC) {
    const unsigned gc = (unsigned)((b.NC + T - 1) / T), ge = (unsigned)((b.NC * b.npc + T - 1) / T);
    k_cc_init<<<gc, T, 0, st>>>(b.NC, b.cell_dreg, parent);
    if (b.npc == 3) k_cc_union<3><<<ge, T, 0, st>>>(b.NC, b.conn, b.cell_dreg, b.inc_ptr, b.inc, parent);
    else k_cc_union<4><<<ge, T, 0, st>>>(b.NC, b.conn, b.cell_dreg, b.inc_ptr, b.inc, parent);
    k_cc_flatten<<<gc, T, 0, st>>>(b.NC, parent);
  }
  if (b.NV) k_cc_vertices<<<(unsigned)((b.NV + T - 1) / T), T, 0, st>>>(b.NV, b.fixed, b.vsample, b.inc_ptr, b.inc, parent, nfix, d_empty);
  if (b.NC) k_cc_count<<<(unsigned)((b.NC + T - 1) / T), T, 0, st>>>(b.NC, b.npc, b.conn, b.vsample, parent, nfix, d_floating);
  b.ctx->launches += 5;
  return cudaGetLastError();
}

}  // namespace fea

// ===========================================================================
// C-ABI
// ===========================================================================
using namespace fea;

namespace {

// tag (1-based point tag) -> sample-local vertex index with numpy's negative wrap-around
// ('vertex {tag-1}', coors[tag - 1]; fea_analysis.py:184-185, 198)
inline int32_t tag_index(int32_t tag, int64_t nv) {
  int64_t i = (int64_t)tag - 1;
  if (i < 0) i += nv;
  return (i < 0 || i >= nv) ? -1 : (int32_t)i;
}

}  // namespace

extern "C" {

int fea_batch_create_from_conditions(fea_ctx* ctx, const fea_conditions_desc* d, fea_batch** out) {
  if (!ctx || !d || !out) return FEA_BAD_ARG;
  *out = nullptr;
  const int ns = d->n_samples, nm = d->n_meshes, npc = d->nodes_per_cell;
  if (ns <= 0 || ns > kMaxSamplesPerBatch || nm <= 0) return api_fail(ctx, FEA_BAD_ARG, "n_samples / n_meshes out of range");
  if (!d->mesh_vtx_off || !d->mesh_cell_off || !d->xy || !d->conn || !d->sample_mesh || !d->vforce_off || !d->eforce_off ||
      !d->vfix_off || !d->efix_off || !d->mat_off || !d->mat_coord_off)
    return api_fail(ctx, FEA_BAD_ARG, "null array in fea_conditions_desc");
  if (d->mesh_vtx_off[0] != 0 || d->mesh_cell_off[0] != 0) return api_fail(ctx, FEA_BAD_ARG, "offset tables must start at 0");
  for (int m = 0; m < nm; ++m)
    if (d->mesh_vtx_off[m + 1] < d->mesh_vtx_off[m] || d->mesh_cell_off[m + 1] < d->mesh_cell_off[m])
      return api_fail(ctx, FEA_BAD_ARG, "offset tables must be non-decreasing");
  const int32_t* offs[5] = {d->vforce_off, d->eforce_off, d->vfix_off, d->efix_off, d->mat_off};
  for (const int32_t* o : offs) {
    if (o[0] != 0) return api_fail(ctx, FEA_BAD_ARG, "offset tables must start at 0");
    for (int s = 0; s < ns; ++s)
      if (o[s + 1] < o[s]) return api_fail(ctx, FEA_BAD_ARG, "offset tables must be non-decreasing");
  }
  if ((d->vforce_off[ns] && (!d->vforce_tag || !d->vforce_mag)) || (d->eforce_off[ns] && (!d->eforce_tag || !d->eforce_mag)) ||
      (d->vfix_off[ns] && !d->vfix_tag) || (d->efix_off[ns] && !d->efix_tag) || (d->mat_off[ns] && (!d->mat_E_nu || !d->mat_coords)))
    return api_fail(ctx, FEA_BAD_ARG, "null array in fea_conditions_desc");
  const int n_matreg = d->mat_off[ns];
  if (d->mat_coord_off[0] != 0) return api_fail(ctx, FEA_BAD_ARG, "offset tables must start at 0");
  for (int r = 0; r < n_matreg; ++r)
    if (d->mat_coord_off[r + 1] < d->mat_coord_off[r]) return api_fail(ctx, FEA_BAD_ARG, "offset tables must be non-decreasing");

  // ---- host tables: per-sample offsets, region rows, hash-set layout ---------------------------
  std::vector<int64_t> vtx_off(ns + 1, 0), cell_off(ns + 1, 0);
  std::vector<int32_t> reg_off(ns + 1, 0), mat_first(ns, 0);
  std::vector<SampleCond> sc(ns);
  std::vector<Region> reg;
  std::vector<int32_t> mat_region(std::max(n_matreg, 1), 0);   // global material region -> region row
  std::vector<int32_t> sreg_off(ns + 1, 0);
  std::vector<int64_t> flag_off(ns + 1, 0);
  int64_t flag_bytes = 0, tab_slots = 0;
  for (int s = 0; s < ns; ++s) {
    const int m = d->sample_mesh[s];
    if (m < 0 || m >= nm) return api_fail(ctx, FEA_BAD_ARG, "sample_mesh out of range");
    const int64_t nv = d->mesh_vtx_off[m + 1] - d->mesh_vtx_off[m], nc = d->mesh_cell_off[m + 1] - d->mesh_cell_off[m];
    vtx_off[s + 1] = vtx_off[s] + nv;
    cell_off[s + 1] = cell_off[s] + nc;
    SampleCond& S = sc[s];
    S.reg0 = (int32_t)reg.size();
    S.n_vf = d->vforce_off[s + 1] - d->vforce_off[s];
    S.n_ef = d->eforce_off[s + 1] - d->eforce_off[s];
    S.n_vc = d->vfix_off[s + 1] - d->vfix_off[s];
    S.n_ec = d->efix_off[s + 1] - d->efix_off[s];
    S.n_mat = d->mat_off[s + 1] - d->mat_off[s];
    S.mesh = m;
    S.pad_ = 0;
    S.E = S.nu = 0.0;
    if (S.n_mat > kMaxMat) return api_fail(ctx, FEA_BAD_ARG, "more than 32 material regions in one sample");
    if (S.n_mat == 0) {
      if (!d->default_E_nu) return api_fail(ctx, FEA_BAD_ARG, "default_E_nu is required for samples without a material table");
      S.E = d->default_E_nu[2 * s];
      S.nu = d->default_E_nu[2 * s + 1];
    }
    mat_first[s] = d->mat_off[s];
    reg_off[s + 1] = reg_off[s] + std::max(S.n_mat, 1) + (S.n_mat > 1 ? kMaxCombo : 0);
    sreg_off[s] = S.reg0;
    flag_off[s] = flag_bytes;
    auto row = [&](int kind) -> Region& {
      Region R{};
      R.sample = s;
      R.kind = kind;
      R.i0 = R.i1 = -1;
      R.flag_off = flag_bytes;
      flag_bytes += nv;
      reg.push_back(R);
      return reg.back();
    };
    for (int i = d->vforce_off[s]; i < d->vforce_off[s + 1]; ++i) {
      Region& R = row(kVForce);
      R.i0 = tag_index(d->vforce_tag[i], nv);
      R.mx = d->vforce_mag[2 * i];
      R.my = d->vforce_mag[2 * i + 1];
      if (R.i0 < 0) return api_fail(ctx, FEA_BAD_ARG, "force vertex tag out of range");
    }
    for (int i = d->eforce_off[s]; i < d->eforce_off[s + 1]; ++i) {
      Region& R = row(kEForce);
      R.i0 = tag_index(d->eforce_tag[2 * i], nv);
      R.i1 = tag_index(d->eforce_tag[2 * i + 1], nv);
      R.mx = d->eforce_mag[2 * i];
      R.my = d->eforce_mag[2 * i + 1];
      if (R.i0 < 0 || R.i1 < 0) return api_fail(ctx, FEA_BAD_ARG, "force edge tag out of range");
    }
    for (int i = d->vfix_off[s]; i < d->vfix_off[s + 1]; ++i) {
      Region& R = row(kVFix);
      R.i0 = tag_index(d->vfix_tag[i], nv);
      if (R.i0 < 0) return api_fail(ctx, FEA_BAD_ARG, "constraint vertex tag out of range");
    }
    for (int i = d->efix_off[s]; i < d->efix_off[s + 1]; ++i) {
      Region& R = row(kEFix);
      R.i0 = tag_index(d->efix_tag[2 * i], nv);
      R.i1 = tag_index(d->efix_tag[2 * i + 1], nv);
      if (R.i0 < 0 || R.i1 < 0) return api_fail(ctx, FEA_BAD_ARG, "constraint edge tag out of range");
    }
    for (int j = 0; j < S.n_mat; ++j) {
      const int g = d->mat_off[s] + j;
      mat_region[g] = (int32_t)reg.size();
      Region& R = row(kMaterial);
      R.mat_local = j;
      const int64_t pts = d->mat_coord_off[g + 1] - d->mat_coord_off[g];
      int64_t cap = 16;
      while (cap < 4 * pts) cap <<= 1;            // 2 scalars per point: load factor <= 0.5
      if (cap > (1LL << 30)) return api_fail(ctx, FEA_BAD_ARG, "material coordinate list too long");
      R.tab_off = tab_slots;
      R.tab_mask = (int32_t)(cap - 1);
      tab_slots += cap;
    }
    row(kPlateMask);
  }
  sreg_off[ns] = (int32_t)reg.size();
  flag_off[ns] = flag_bytes;
  const int64_t NRrows = (int64_t)reg.size();
  const int64_t n_scalars = 2 * d->mat_coord_off[n_matreg];
  const int64_t MV = d->mesh_vtx_off[nm], MC = d->mesh_cell_off[nm];

  fea_batch* created = nullptr;
  int rc = api_batch_begin(ctx, ns, npc, vtx_off.data(), cell_off.data(), reg_off.data(), &created);
  if (rc != FEA_OK) return rc;
  std::unique_ptr<fea_batch, decltype(&api_free_batch)> hb(created, api_free_batch);
  Batch& b = hb->b;
  b.from_conditions = true;
  b.NR = NRrows;
  b.sreg_off = sreg_off;
  b.flag_off = flag_off;
  cudaStream_t st = ctx->c.stream;
  const int T = 256;
  Scratch scratch(st);
  double2 *m_xy = nullptr;
  int32_t *m_conn = nullptr, *conn_local = nullptr, *d_mat_region = nullptr, *d_mat_first = nullptr, *combo_first = nullptr,
          *combo_id = nullptr, *d_regoff = nullptr;
  int64_t *m_vtx_off = nullptr, *m_cell_off = nullptr, *d_voff = nullptr, *d_coff = nullptr, *d_coord_off = nullptr;
  SampleCond* d_sc = nullptr;
  Region* d_reg = nullptr;
  double *d_E_nu = nullptr, *d_coords = nullptr;
  unsigned long long* tab = nullptr;
  uint8_t* v0 = nullptr;
  uint32_t *cell_member = nullptr, *combo_mask = nullptr;
  CK(ctx, dalloc(b, &b.xy, b.NV * 2));
  CK(ctx, dalloc(b, &b.D, (int64_t)b.NREG * 9));
  CK(ctx, dalloc(b, &b.fixed, b.NV));
  CK(ctx, dalloc(b, &b.rhs, b.NV * 2));
  CK(ctx, dalloc(b, &b.rflags, flag_bytes));
  CK(ctx, dalloc(b, &b.rcount, NRrows));
  CK(ctx, dalloc(b, &b.creg_local, b.NC));
  CK(ctx, dalloc(b, &b.n_reg_used, ns));
  CK(ctx, scratch.alloc(&m_xy, MV));
  CK(ctx, scratch.alloc(&m_conn, MC * npc));
  CK(ctx, scratch.alloc(&m_vtx_off, nm + 1));
  CK(ctx, scratch.alloc(&m_cell_off, nm + 1));
  CK(ctx, scratch.alloc(&d_voff, ns + 1));
  CK(ctx, scratch.alloc(&d_coff, ns + 1));
  CK(ctx, scratch.alloc(&conn_local, b.NC * npc));
  CK(ctx, scratch.alloc(&d_sc, ns));
  CK(ctx, scratch.alloc(&d_reg, NRrows));
  CK(ctx, scratch.alloc(&d_mat_region, n_matreg));
  CK(ctx, scratch.alloc(&d_mat_first, ns));
  CK(ctx, scratch.alloc(&d_regoff, ns + 1));
  CK(ctx, scratch.alloc(&d_coord_off, n_matreg + 1));
  CK(ctx, scratch.alloc(&d_E_nu, 2 * std::max(n_matreg, 1)));
  CK(ctx, scratch.alloc(&d_coords, n_scalars));
  CK(ctx, scratch.alloc(&tab, tab_slots));
  CK(ctx, scratch.alloc(&v0, flag_bytes));
  CK(ctx, scratch.alloc(&cell_member, b.NC));
  CK(ctx, scratch.alloc(&combo_mask, ns * kMaxCombo));
  CK(ctx, scratch.alloc(&combo_first, ns * kMaxCombo));
  CK(ctx, scratch.alloc(&combo_id, ns * kMaxCombo));
  // err_flag is allocated by api_batch_finish; the combination overflow is collected in a word of its own first
  int32_t* d_err = nullptr;
  CK(ctx, dalloc(b, &d_err, 1));
  CK(ctx, cudaMemsetAsync(d_err, 0, sizeof(int32_t), st));
  CK(ctx, cudaMemcpyAsync(m_xy, d->xy, sizeof(double) * 2 * MV, cudaMemcpyDefault, st));       // host or device (fea_device_upload)
  CK(ctx, cudaMemcpyAsync(m_conn, d->conn, sizeof(int32_t) * MC * npc, cudaMemcpyDefault, st));
  CK(ctx, cudaMemcpyAsync(m_vtx_off, d->mesh_vtx_off, sizeof(int64_t) * (nm + 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(m_cell_off, d->mesh_cell_off, sizeof(int64_t) * (nm + 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_voff, vtx_off.data(), sizeof(int64_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_coff, cell_off.data(), sizeof(int64_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_sc, sc.data(), sizeof(SampleCond) * ns, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_reg, reg.data(), sizeof(Region) * NRrows, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_mat_region, mat_region.data(), sizeof(int32_t) * std::max(n_matreg, 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_mat_first, mat_first.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_regoff, reg_off.data(), sizeof(int32_t) * (ns + 1), cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_coord_off, d->mat_coord_off, sizeof(int64_t) * (n_matreg + 1), cudaMemcpyHostToDevice, st));
  if (n_matreg) CK(ctx, cudaMemcpyAsync(d_E_nu, d->mat_E_nu, sizeof(double) * 2 * n_matreg, cudaMemcpyHostToDevice, st));
  if (n_scalars) CK(ctx, cudaMemcpyAsync(d_coords, d->mat_coords, sizeof(double) * n_scalars, cudaMemcpyDefault, st));
  CK(ctx, cudaMemsetAsync(tab, 0xFF, sizeof(unsigned long long) * std::max<int64_t>(tab_slots, 1), st));
  CK(ctx, cudaMemsetAsync(cell_member, 0, sizeof(uint32_t) * std::max<int64_t>(b.NC, 1), st));
  CK(ctx, cudaMemsetAsync(combo_mask, 0, sizeof(uint32_t) * ns * kMaxCombo, st));
  CK(ctx, cudaMemsetAsync(combo_first, 0x7F, sizeof(int32_t) * ns * kMaxCombo, st));
  CK(ctx, cudaMemsetAsync(combo_id, 0, sizeof(int32_t) * ns * kMaxCombo, st));
  CK(ctx, cudaMemsetAsync(b.D, 0, sizeof(double) * 9 * std::max<int64_t>(b.NREG, 1), st));
  int64_t nv_max = 0, nc_max = 0;
  for (int s = 0; s < ns; ++s) {
    nv_max = std::max(nv_max, vtx_off[s + 1] - vtx_off[s]);
    nc_max = std::max(nc_max, cell_off[s + 1] - cell_off[s]);
  }
  const unsigned gyv = (unsigned)std::max<int64_t>(1, (nv_max + T - 1) / T), gyc = (unsigned)std::max<int64_t>(1, (nc_max + T - 1) / T),
                 gyn = (unsigned)std::max<int64_t>(1, (nc_max * npc + T - 1) / T);
  if (gyv > 65535u || gyn > 65535u)
    return api_fail(ctx, FEA_CUDA_ERROR, "more than 16 M vertices or cell corners in one sample");
  k_replicate_vertices<<<dim3(ns, gyv), T, 0, st>>>(d_sc, d_voff, m_vtx_off, m_xy, (double2*)b.xy);
  k_replicate_cells<<<dim3(ns, gyn), T, 0, st>>>(d_sc, d_coff, npc, m_cell_off, m_conn, conn_local);
  if (n_scalars)
    k_hash_insert<<<(unsigned)((n_scalars + T - 1) / T), T, 0, st>>>(n_scalars, n_matreg, d_coord_off, d_mat_region, d_reg, d_coords, tab);
  k_region_vertices<<<dim3((unsigned)NRrows, gyv), T, 0, st>>>(d_reg, d_voff, (const double2*)b.xy, tab, v0, b.rflags);
  if (npc == 3) k_region_cells<3><<<dim3((unsigned)NRrows, gyc), T, 0, st>>>(d_reg, d_voff, d_coff, conn_local, v0, b.rflags, cell_member);
  else k_region_cells<4><<<dim3((unsigned)NRrows, gyc), T, 0, st>>>(d_reg, d_voff, d_coff, conn_local, v0, b.rflags, cell_member);
  k_region_count<<<(unsigned)NRrows, T, 0, st>>>(d_reg, d_voff, b.rflags, b.rcount);
  k_fixed_rhs<<<dim3(ns, gyv), T, 0, st>>>(d_sc, d_reg, d_voff, b.rflags, b.rcount, b.fixed, (double2*)b.rhs);
  k_cell_region<<<dim3(ns, gyc), T, 0, st>>>(d_sc, d_coff, cell_member, combo_mask, combo_first, b.creg_local, d_err);
  k_material_table<<<(ns + 127) / 128, 128, 0, st>>>(ns, d_sc, d_regoff, d_E_nu, d_mat_first, combo_mask, combo_first,
                                                    combo_id, b.D, b.n_reg_used);
  k_cell_region_combos<<<dim3(ns, gyc), T, 0, st>>>(d_coff, combo_id, b.creg_local);
  CK(ctx, cudaGetLastError());
  ctx->c.launches += 10;
  rc = api_batch_finish(ctx, b, b.creg_local, conn_local);
  if (rc != FEA_OK) return rc;
  // material-combination overflow found by k_cell_region -> bit 2 of the batch's error word (read by assemble)
  k_merge_err<<<1, 1, 0, st>>>(d_err, b.err_flag + 2);
  CK(ctx, cudaGetLastError());
  *out = hb.release();
  return FEA_OK;
}

int fea_batch_get_setup(fea_batch* hb, uint8_t* fixed, int8_t* cell_region, double* rhs, int32_t* region_count,
                        uint8_t* region_flags) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.from_conditions) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_get_setup needs a batch made by fea_batch_create_from_conditions");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (fixed) CK(ctx, cudaMemcpyAsync(fixed, b.fixed, (size_t)b.NV, cudaMemcpyDeviceToHost, st));
  if (cell_region) CK(ctx, cudaMemcpyAsync(cell_region, b.creg_local, (size_t)b.NC, cudaMemcpyDeviceToHost, st));
  if (rhs) CK(ctx, cudaMemcpyAsync(rhs, b.rhs, sizeof(double) * 2 * b.NV, cudaMemcpyDeviceToHost, st));
  std::vector<int32_t> cnt;
  if (region_count) {
    cnt.resize((size_t)b.NR);
    CK(ctx, cudaMemcpyAsync(cnt.data(), b.rcount, sizeof(int32_t) * b.NR, cudaMemcpyDeviceToHost, st));
  }
  if (region_flags) {   // every sample's block without its trailing plate-mask row
    size_t o = 0;
    for (int s = 0; s < b.ns; ++s) {
      const size_t nv = (size_t)(b.vtx_off[s + 1] - b.vtx_off[s]);
      const size_t bytes = (size_t)(b.sreg_off[s + 1] - b.sreg_off[s] - 1) * nv;
      if (bytes) CK(ctx, cudaMemcpyAsync(region_flags + o, b.rflags + b.flag_off[s], bytes, cudaMemcpyDeviceToHost, st));
      o += bytes;
    }
  }
  CK(ctx, cudaStreamSynchronize(st));
  if (region_count) {
    size_t o = 0;
    for (int s = 0; s < b.ns; ++s)
      for (int r = b.sreg_off[s]; r < b.sreg_off[s + 1] - 1; ++r) region_count[o++] = cnt[r];
  }
  return FEA_OK;
}

int fea_batch_get_materials(fea_batch* hb, int32_t* reg_off, int32_t* n_used, double* D) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (reg_off) memcpy(reg_off, b.reg_off.data(), sizeof(int32_t) * (b.ns + 1));
  if (n_used) {
    if (b.n_reg_used) CK(ctx, cudaMemcpyAsync(n_used, b.n_reg_used, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
    else for (int s = 0; s < b.ns; ++s) n_used[s] = b.reg_off[s + 1] - b.reg_off[s];
  }
  if (D && b.NREG) CK(ctx, cudaMemcpyAsync(D, b.D, sizeof(double) * 9 * b.NREG, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return FEA_OK;
}

int fea_batch_rasterize_regions(fea_batch* hb, const uint8_t* with_plate_mask, uint8_t* images) {
  if (!hb || !images) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.from_conditions) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_rasterize_regions needs a batch made by fea_batch_create_from_conditions");
  if (!b.rasterized) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_rasterize_regions before fea_batch_rasterize");
  std::vector<int64_t> field_off(b.ns + 1, 0);
  for (int s = 0; s < b.ns; ++s)
    field_off[s + 1] = field_off[s] + (b.sreg_off[s + 1] - b.sreg_off[s] - 1) + ((with_plate_mask && with_plate_mask[s]) ? 1 : 0);
  const int64_t n_img = field_off[b.ns];
  if (n_img == 0) return FEA_OK;
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  const size_t per = (size_t)b.img_size * b.img_size, tabb = sizeof(int64_t) * (b.ns + 1);
  Scratch scratch(st);
  int64_t *d_field_off = nullptr, *d_flag_off = nullptr;
  uint8_t* d_images = nullptr;
  CK(ctx, scratch.alloc(&d_field_off, b.ns + 1));
  CK(ctx, scratch.alloc(&d_flag_off, b.ns + 1));
  CK(ctx, scratch.alloc(&d_images, n_img * (int64_t)per));
  CK(ctx, cudaMemcpyAsync(d_field_off, field_off.data(), tabb, cudaMemcpyHostToDevice, st));
  CK(ctx, cudaMemcpyAsync(d_flag_off, b.flag_off.data(), tabb, cudaMemcpyHostToDevice, st));
  CK(ctx, launch_raster_flags(b, n_img, d_field_off, d_flag_off, b.rflags, d_images));
  ctx->c.launches += 1;
  CK(ctx, cudaMemcpyAsync(images, d_images, n_img * per, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));   // field_off (host vector) must outlive the copy
  return FEA_OK;
}

int fea_batch_classify(fea_batch* hb, int32_t* floating_parts, int32_t* empty_vertices) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.assembled) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_classify before fea_batch_assemble");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  Scratch scratch(st);
  int32_t* dv = nullptr;
  CK(ctx, scratch.alloc(&dv, 2 * (int64_t)b.ns));
  CK(ctx, launch_classify(b, dv, dv + b.ns));
  if (floating_parts) CK(ctx, cudaMemcpyAsync(floating_parts, dv, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  if (empty_vertices) CK(ctx, cudaMemcpyAsync(empty_vertices, dv + b.ns, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return FEA_OK;
}

// ---- staged outputs: everything a dataset writer reads, produced on the batch's stream and read back on
// another one.  The D2H copies of batch j (u, images, region images: ~60 MB for 400 plate-conditions) then run
// on a copy engine while the batch's own context already solves batch j + 1.
int fea_batch_stage_outputs(fea_batch* hb, const uint8_t* with_plate_mask) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = hb->owner;
  Batch& b = hb->b;
  if (!b.rasterized) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_stage_outputs before fea_batch_rasterize");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  if (!b.ev_staged) CK(ctx, cudaEventCreateWithFlags(&b.ev_staged, cudaEventDisableTiming));
  if (b.from_conditions && !b.stage_class) {   // committed to b last, so that a failed call is staged again in full
    std::vector<int64_t> field_off(b.ns + 1, 0);
    for (int s = 0; s < b.ns; ++s)
      field_off[s + 1] = field_off[s] + (b.sreg_off[s + 1] - b.sreg_off[s] - 1) + ((with_plate_mask && with_plate_mask[s]) ? 1 : 0);
    const int64_t n_img = field_off[b.ns];
    const size_t per = (size_t)b.img_size * b.img_size;
    int32_t* cls = nullptr;
    uint8_t* regions = nullptr;
    CK(ctx, dalloc(b, &cls, (int64_t)2 * b.ns));
    CK(ctx, launch_classify(b, cls, cls + b.ns));
    if (n_img > 0) {
      int64_t* tab = nullptr;
      CK(ctx, dalloc(b, &tab, (int64_t)2 * (b.ns + 1)));
      CK(ctx, dalloc(b, &regions, (int64_t)(n_img * per)));
      CK(ctx, cudaMemcpyAsync(tab, field_off.data(), sizeof(int64_t) * (b.ns + 1), cudaMemcpyHostToDevice, st));
      CK(ctx, cudaMemcpyAsync(tab + b.ns + 1, b.flag_off.data(), sizeof(int64_t) * (b.ns + 1), cudaMemcpyHostToDevice, st));
      CK(ctx, launch_raster_flags(b, n_img, tab, tab + b.ns + 1, b.rflags, regions));
      ctx->c.launches += 1;
    }
    b.stage_class = cls;
    b.stage_regions = regions;
    b.stage_field_off = std::move(field_off);
  }
  CK(ctx, cudaEventRecord(b.ev_staged, st));
  return FEA_OK;
}

int fea_batch_staged_region_images(fea_batch* hb, int64_t* n_images) {
  if (!hb || !n_images) return FEA_BAD_ARG;
  *n_images = hb->b.stage_field_off.empty() ? 0 : hb->b.stage_field_off[hb->b.ns];
  return FEA_OK;
}

int fea_batch_fetch_outputs(fea_batch* hb, fea_ctx* copy_ctx, double* u, double* ranges, int32_t* iters, double* relres,
                            int32_t* status, uint8_t* images, uint8_t* region_images, int32_t* floating_parts,
                            int32_t* empty_vertices) {
  if (!hb) return FEA_BAD_ARG;
  fea_ctx* ctx = copy_ctx ? copy_ctx : hb->owner;     // errors are reported on the calling thread's context
  const Batch& b = hb->b;
  if (!b.ev_staged) return api_fail(ctx, FEA_BAD_STATE, "fea_batch_fetch_outputs before fea_batch_stage_outputs");
  if ((region_images || floating_parts || empty_vertices) && !b.stage_class)
    return api_fail(ctx, FEA_BAD_STATE, "region images / classifier need a batch made by fea_batch_create_from_conditions");
  if (ctx->c.device != hb->owner->c.device) return api_fail(ctx, FEA_BAD_ARG, "copy context on another device");
  CK(ctx, cudaSetDevice(ctx->c.device));
  cudaStream_t st = ctx->c.stream;
  CK(ctx, cudaStreamWaitEvent(st, b.ev_staged, 0));
  const size_t per = (size_t)b.img_size * b.img_size;
  if (u) CK(ctx, cudaMemcpyAsync(u, b.u, sizeof(double) * 2 * b.NV, cudaMemcpyDeviceToHost, st));
  if (ranges) CK(ctx, cudaMemcpyAsync(ranges, b.ranges, sizeof(double) * 4 * b.ns, cudaMemcpyDeviceToHost, st));
  if (iters) CK(ctx, cudaMemcpyAsync(iters, b.sc.iters, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  if (relres) CK(ctx, cudaMemcpyAsync(relres, b.relres, sizeof(double) * b.ns, cudaMemcpyDeviceToHost, st));
  if (status) CK(ctx, cudaMemcpyAsync(status, b.sc.status, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  if (images) CK(ctx, cudaMemcpyAsync(images, b.images, (size_t)b.ns * 2 * per, cudaMemcpyDeviceToHost, st));
  if (region_images && b.stage_regions)
    CK(ctx, cudaMemcpyAsync(region_images, b.stage_regions, (size_t)b.stage_field_off[b.ns] * per, cudaMemcpyDeviceToHost, st));
  if (floating_parts) CK(ctx, cudaMemcpyAsync(floating_parts, b.stage_class, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  if (empty_vertices) CK(ctx, cudaMemcpyAsync(empty_vertices, b.stage_class + b.ns, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st));
  CK(ctx, cudaStreamSynchronize(st));
  return FEA_OK;
}

}  // extern "C"
