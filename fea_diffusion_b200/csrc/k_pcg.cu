// K5: lock-step Jacobi-preconditioned fp64 CG over all samples of a batch -- replaces
// Newton + ScipyDirect(SuperLU) + SimpleTimeSteppingSolver (reference
// datagen/fea_analysis.py:371-375, 425-439; SURVEY A-12..A-14, F5).
//
// The matrix is stored Jacobi-scaled (Khat = S K S), so preconditioned CG on K is plain CG
// on Khat:  two kernels per iteration, no host involvement:
//
//   spmv  : rz   = sum of the r.r partials the previous update left   -> convergence test
//           p    = r + beta * p_old      (beta = rz / rz_prev)
//           q    = Khat p                (block-SELL-32, one thread per 2x2 block row; p is formed
//                                         on the fly at the gathered columns, so there is no
//                                         separate p-update pass over HBM)
//           partA[cta] = p . q over the CTA's rows
//   update: pq   = sum of the p.q partials;  alpha = rz / pq
//           p = r + beta * p_old (same expression, same bits);  x += alpha p;  r -= alpha q
//           partB[cta] = r . r over the CTA's rows
//
// r and p live interleaved in one array of 32-byte records (r.x, r.y, p.x, p.y): the SpMV fetches
// a neighbour's residual and previous direction with ONE 256-bit gather that uses a whole 32-byte
// sector, and a 2x2 matrix block is one 256-bit load as well.  Only the update kernel writes the
// records (its own rows), so the SpMV reads them without any ping-pong buffer.
//
// Every CTA (128 block rows) belongs to exactly one system.  Dot products never use atomics or
// fences: a kernel leaves one partial per CTA and every warp of the *next* kernel re-adds the
// partials of its own system in a fixed order (a few dozen L2-resident doubles).  Results are
// therefore bitwise reproducible and independent of which other systems share the batch or the
// GPU.  Systems owning more than kDirectSumMax CTAs (the ~1M-DOF single solves) get their partials
// pre-summed by whichever of their CTAs finishes last (two-level mode, presum_if_last).  Finished
// systems cost one flag read per CTA.
#include <cstdio>
#include <cstdlib>

#include "fea_internal.cuh"
#include "pcg_params.cuh"

namespace fea {

#if defined(FEA_CLUSTER_PROFILE) || defined(FEA_CLUSTER_ACCOUNT)
void pcg_cluster_profile_dump();
#endif

constexpr int kT = kCtaRows;       // threads per CTA
constexpr int kDirectSumMax = 128;  // partials a consumer warp sums itself

// Deterministic CTA sum of one double per thread; result valid in thread 0.
__device__ __forceinline__ double cta_sum(double v, double* sm /*[kT/32]*/) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < kT / 32; ++w) t += sm[w];
  }
  return t;
}

// Two-level mode (systems owning more than kDirectSumMax CTAs): the CTA of the system that finishes LAST
// (arrival counter) pre-sums the system's partials for the next kernel, in the same fixed order whichever
// CTA that is -- partial i goes to thread i mod kT, then the CTA sum -- so the result has the same bits in
// every run.  Replaces a separate one-CTA-per-system kernel between the two solver kernels (two launches
// per iteration of a ~1 M-DOF solve).
__device__ __forceinline__ void presum_if_last(const double* __restrict__ part, int first, int n, int32_t* arrive,
                                               double* psum, double* sm /*[kT/32]*/) {
  __shared__ int last;
  if (threadIdx.x == 0) {
    __threadfence();                       // this CTA's partial is visible before it is counted
    last = atomicAdd(arrive, 1) == n - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();                         // the other CTAs' partials are visible after the count was read
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += kT) acc += __ldcg(part + first + i);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kT / 32; ++w) t += sm[w];
    *psum = t;
    *arrive = 0;                           // ready for the next kernel of this kind
  }
}

// Ordered sum of n partials, identical in every lane of every warp that calls it.
__device__ __forceinline__ double sum_partials(const double* __restrict__ part, int n) {
  double acc = 0.0;
  for (int i = threadIdx.x & 31; i < n; i += 32) acc += __ldg(part + i);
  return warp_sum(acc);
}


// Grid = any size >= P.n_active (the host picks a size class from a slightly stale count).
// 16 resident CTAs per SM (a 32-register budget): the SpMV of a single ~1 M-DOF system is latency-bound
// and needs full occupancy.
// HINT: L2 eviction policies on the loads (matrix evict_first, gathered records evict_last) for systems
// whose matrix does not fit the L2.
template <bool HINT>
__global__ void __launch_bounds__(kT, 16) k_pcg_spmv(const PcgPtrs* __restrict__ Pp, int parity) {
  __shared__ double sm[kT / 32];
  const PcgPtrs& P = *Pp;
  if ((int)blockIdx.x >= P.n_active) return;
  const int4 w = __ldg(P.active + blockIdx.x);
  const int cta = w.x, s = w.y, first = w.z;
  if (P.sc.done[s]) return;
  const bool leader = cta == first && threadIdx.x == 0;
  const double rz = P.two_level ? P.sc.psumB[s] : sum_partials(P.partB + first, w.w);
  {
    int st = -1;
    if (!isfinite(rz)) st = FEA_SAMPLE_BREAKDOWN;
    else if (rz <= P.sc.tol2[s]) st = FEA_SAMPLE_CONVERGED;
    else if (P.sc.iters[s] >= P.sc.cap[s]) st = P.sc.cap[s] < P.max_iter ? FEA_SAMPLE_STAGNATED : FEA_SAMPLE_MAX_ITER;
    if (st >= 0) {  // every CTA of the system takes the same decision; the leader records it
      if (leader) {
        P.sc.done[s] = 1;
        P.sc.status[s] = st;
        P.rz_last[s] = rz;
        atomicAdd(P.sc.n_done, 1);
      }
      return;
    }
  }
  const double beta = rz / P.sc.rz[parity ^ 1][s];
  if (leader) P.sc.rz[parity][s] = rz;
  const int64_t row = (int64_t)cta * kT + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = P.slice_len[slice];
  const int64_t base = P.slice_ptr[slice];
  const d4* __restrict__ vt = P.val + base + lane;
  const int32_t* __restrict__ cp = P.col + base + lane;
  const d4* __restrict__ rp = P.rp;
  const uint64_t pol_m = HINT ? l2_policy_evict_first() : 0, pol_v = HINT ? l2_policy_evict_last() : 0;
  // own row: p_i and the diagonal block [[1, a], [a, 1]]
  const d4 own = HINT ? ld_nc_d4_hint(rp + row, pol_v) : ld_nc_d4(rp + row);
  const double2 pn = make_double2(fma(beta, own.z, own.x), fma(beta, own.w, own.y));
  double a0 = pn.x, a1 = pn.y;   // the diagonal block of Khat is the identity
#pragma unroll 1
  for (int j = 0; j < L; ++j) {
    const int c = HINT ? ld_stream_i32_hint(cp + j * 32, pol_m) : ld_stream_i32(cp + j * 32);
    const d4 k = HINT ? ld_stream_d4_hint(vt + j * 32, pol_m) : ld_stream_d4(vt + j * 32);
    const d4 g = HINT ? ld_nc_d4_hint(rp + c, pol_v) : ld_nc_d4(rp + c);
    const double px = fma(beta, g.z, g.x);
    const double py = fma(beta, g.w, g.y);
    a0 = fma(k.x, px, a0);
    a0 = fma(k.y, py, a0);
    a1 = fma(k.z, px, a1);
    a1 = fma(k.w, py, a1);
  }
  P.q[row] = make_double2(a0, a1);
  const double part = cta_sum(fma(pn.x, a0, pn.y * a1), sm);
  if (threadIdx.x == 0) P.partA[cta] = part;
  if (P.two_level) presum_if_last(P.partA, first, w.w, P.sc.arrive + 2 * s, P.sc.psumA + s, sm);
}

__global__ void __launch_bounds__(kT) k_pcg_update(const PcgPtrs* __restrict__ Pp, int parity) {
  __shared__ double sm[kT / 32];
  const PcgPtrs& P = *Pp;
  if ((int)blockIdx.x >= P.n_active) return;
  const int4 w = __ldg(P.active + blockIdx.x);
  const int cta = w.x, s = w.y, first = w.z;
  if (P.sc.done[s]) return;
  const bool leader = cta == first && threadIdx.x == 0;
  const double pq = P.two_level ? P.sc.psumA[s] : sum_partials(P.partA + first, w.w);
  if (!(pq > 0.0 && isfinite(pq))) {  // not SPD on this Krylov space (floating region, F4)
    if (leader) {
      P.sc.done[s] = 1;
      P.sc.status[s] = FEA_SAMPLE_BREAKDOWN;
      atomicAdd(P.sc.n_done, 1);
    }
    return;
  }
  const double rz = P.sc.rz[parity][s];
  const double alpha = rz / pq;
  const double beta = rz / P.sc.rz[parity ^ 1][s];  // the value the SpMV of this iteration used
  const int64_t row = (int64_t)cta * kT + threadIdx.x;
  d4 rec = P.rp[row];
  const double2 qv = P.q[row];
  double2 xv = P.x[row];
  rec.z = fma(beta, rec.z, rec.x);   // p of this iteration, bit-identical to the SpMV's
  rec.w = fma(beta, rec.w, rec.y);
  xv.x = fma(alpha, rec.z, xv.x);
  xv.y = fma(alpha, rec.w, xv.y);
  rec.x = fma(-alpha, qv.x, rec.x);
  rec.y = fma(-alpha, qv.y, rec.y);
  P.x[row] = xv;
  P.rp[row] = rec;
  const double part = cta_sum(fma(rec.x, rec.x, rec.y * rec.y), sm);
  if (threadIdx.x == 0) {
    P.partB[cta] = part;
    if (leader) P.sc.iters[s] += 1;
  }
  if (P.two_level) presum_if_last(P.partB, first, w.w, P.sc.arrive + 2 * s + 1, P.sc.psumB + s, sm);
}

// Residual replacement.  The recursion r -= alpha q drifts away from b - K x by rounding (the gap
// grows with the iteration count: ~1e-9 relative after 12 k iterations of a 1.2 M-DOF system), so
// a system whose RECURSIVE residual met the tolerance is checked once more against the TRUE one:
//   r = S b - Khat x  (same block-SELL gather, on x),  p = 0,  partB = r.r partials.
// k_pcg_refine_scalars then either confirms convergence (rz_last = true r.r, which is what relres
// reports) or, when the true residual is more than 10x the tolerance, reopens the system: CG
// restarts from the current x with the true residual.
//
// monitor = 1: the same pass for systems that are still iterating, every kMonitorChunks chunks: r
// is replaced by the true residual, p is kept, and a system whose true residual has not even halved
// since the previous pass is stopped as STAGNATED (singular / inconsistent: it would iterate to
// max_iter otherwise).
__global__ void __launch_bounds__(kT) k_pcg_true_residual(const PcgPtrs* __restrict__ Pp,
                                                          const int32_t* __restrict__ vertex_of_row,
                                                          const double* __restrict__ rhs,
                                                          const double* __restrict__ dscale,
                                                          const double* __restrict__ scoup, int monitor) {
  __shared__ double sm[kT / 32];
  const PcgPtrs& P = *Pp;
  const int cta = blockIdx.x;
  const int s = P.sys_of_cta[cta];
  if (s < 0) return;
  const int st = P.sc.status[s];
  if (monitor) {
    if (P.sc.done[s]) return;
  } else if ((st != FEA_SAMPLE_CONVERGED && st != FEA_SAMPLE_STAGNATED) || P.sc.iters[s] == 0 || P.sc.cap[s] < 0) {
    return;
  }
  const int64_t row = (int64_t)cta * kT + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int64_t slice = row >> 5;
  const int L = P.slice_len[slice];
  const int64_t base = P.slice_ptr[slice];
  const d4* __restrict__ vt = P.val + base + lane;
  const int32_t* __restrict__ cp = P.col + base + lane;
  const double2* __restrict__ x = P.x;
  const double2 xi = x[row];
  double a0 = xi.x, a1 = xi.y;   // the diagonal block of Khat is the identity
  for (int j = 0; j < L; ++j) {
    const int c = ld_stream_i32(cp + j * 32);
    const d4 k = ld_stream_d4(vt + j * 32);
    const double2 xj = __ldg(x + c);
    a0 = fma(k.x, xj.x, a0);
    a0 = fma(k.y, xj.y, a0);
    a1 = fma(k.z, xj.x, a1);
    a1 = fma(k.w, xj.y, a1);
  }
  const int v = vertex_of_row[row];
  d4 rec;
  rec.x = rec.y = rec.z = rec.w = 0.0;
  if (monitor) rec = P.rp[row];   // keep p
  rec.x = rec.y = 0.0;
  if (v >= 0) {
    const double b0 = rhs[2 * (int64_t)v], b1 = rhs[2 * (int64_t)v + 1];     // S^T b = L^-1 b
    rec.x = dscale[2 * row] * b0 - a0;
    rec.y = fma(scoup[row], b0, dscale[2 * row + 1] * b1) - a1;
  }
  P.rp[row] = rec;
  const double part = cta_sum(fma(rec.x, rec.x, rec.y * rec.y), sm);
  if (threadIdx.x == 0) P.partB[cta] = part;
}

// one warp per system; reopened systems restart CG (beta = 0) from their current x
__global__ void k_pcg_refine_scalars(const PcgPtrs* __restrict__ Pp, int32_t* __restrict__ n_reopened, int allow_reopen,
                                     int monitor) {
  const PcgPtrs& P = *Pp;
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= P.ns) return;
  if (monitor) {
    if (P.sc.done[s]) return;
    const double total = sum_partials(P.partB + P.cta_first[s], P.cta_count[s]);
    if ((threadIdx.x & 31) != 0) return;
    P.sc.psumB[s] = total;
    if (!(total < 0.25 * P.sc.rz_mon[s]) || !isfinite(total)) {
      P.sc.status[s] = FEA_SAMPLE_STAGNATED;
      P.sc.done[s] = 1;
      P.rz_last[s] = total;
      atomicAdd(P.sc.n_done, 1);
    }
    P.sc.rz_mon[s] = total;
    return;
  }
  const int st = P.sc.status[s];
  if ((st != FEA_SAMPLE_CONVERGED && st != FEA_SAMPLE_STAGNATED) || P.sc.iters[s] == 0 || P.sc.cap[s] < 0) return;
  const double total = sum_partials(P.partB + P.cta_first[s], P.cta_count[s]);
  if ((threadIdx.x & 31) != 0) return;
  P.rz_last[s] = total;                       // what relres reports: the true residual
  if (st == FEA_SAMPLE_STAGNATED) return;
  // restart only when the gap is material (true residual more than 10x the tolerance): a restart
  // costs the Krylov space, and errors against a direct solve are already ~1e-10 at this level
  if (!(total > 100.0 * P.sc.tol2[s] && isfinite(total))) return;
  if (!allow_reopen || P.sc.iters[s] >= P.max_iter) {
    P.sc.status[s] = FEA_SAMPLE_STAGNATED;
    return;
  }
  {
    // a restart that cannot close the gap (attainable accuracy ~ eps * cond) must not run away
    const int it = P.sc.iters[s];
    const int cap = it + it / 4 + 100;
    P.sc.cap[s] = cap < P.max_iter ? cap : P.max_iter;
    P.sc.rz[0][s] = total;
    P.sc.rz[1][s] = __longlong_as_double(0x7ff0000000000000LL);  // +inf -> beta = 0
    P.sc.psumB[s] = total;
    P.sc.status[s] = FEA_SAMPLE_NOT_RUN;
    P.sc.done[s] = 0;
    atomicSub(P.sc.n_done, 1);
    atomicAdd(n_reopened, 1);
  }
}

// Work list of the CTAs whose system is still iterating, in CTA order (one CTA does the whole
// compaction: a batch has at most a few 10^4 solver CTAs).  Runs once per chunk of iterations;
// systems that finish inside a chunk cost one flag read per CTA until the next compaction.
__global__ void __launch_bounds__(1024) k_compact_active(PcgPtrs* __restrict__ Pp) {
  __shared__ int wsum[32];
  __shared__ int carry;
  const PcgPtrs& P = *Pp;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < P.ncta; base += 1024) {
    const int c = base + threadIdx.x;
    int s = -1;
    if (c < P.ncta) {
      s = P.sys_of_cta[c];
      if (s >= 0 && P.sc.done[s]) s = -1;
    }
    const unsigned m = __ballot_sync(0xffffffffu, s >= 0);
    if (lane == 0) wsum[wid] = __popc(m);
    __syncthreads();
    int off = carry;
    for (int i = 0; i < wid; ++i) off += wsum[i];
    if (s >= 0) P.active[off + __popc(m & ((1u << lane) - 1u))] = make_int4(c, s, P.cta_first[s], P.cta_count[s]);
    __syncthreads();
    if (threadIdx.x == 0) {
      int t = 0;
      for (int i = 0; i < 32; ++i) t += wsum[i];
      carry += t;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) Pp->n_active = carry;
}

__global__ void k_store_params(PcgPtrs P, PcgPtrs* __restrict__ dst) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *dst = P;
}

// r0 = S b, x0 = 0, p = 0; partB = r0.r0 partials.
__global__ void __launch_bounds__(kT) k_pcg_init_vectors(const PcgPtrs* __restrict__ Pp,
                                                         const int32_t* __restrict__ vertex_of_row,
                                                         const double* __restrict__ rhs,
                                                         const double* __restrict__ dscale,
                                                         const double* __restrict__ scoup) {
  __shared__ double sm[kT / 32];
  const PcgPtrs& P = *Pp;
  const int s = P.sys_of_cta[blockIdx.x];
  if (s < 0) return;
  const int64_t row = (int64_t)blockIdx.x * kT + threadIdx.x;
  const int v = vertex_of_row[row];
  double2 b = make_double2(0.0, 0.0);
  if (v >= 0) {   // S^T b = L^-1 b
    const double b0 = rhs[2 * (int64_t)v], b1 = rhs[2 * (int64_t)v + 1];
    b = make_double2(dscale[2 * row] * b0, fma(scoup[row], b0, dscale[2 * row + 1] * b1));
  }
  const double2 z = make_double2(0.0, 0.0);
  d4 rec;
  rec.x = b.x;
  rec.y = b.y;
  rec.z = rec.w = 0.0;
  P.x[row] = z;
  P.rp[row] = rec;
  P.q[row] = z;
  const_cast<double2*>(P.sb)[row] = b;   // kept for the extended-precision rounds of the on-chip path
  const double part = cta_sum(fma(b.x, b.x, b.y * b.y), sm);
  if (threadIdx.x == 0) P.partB[blockIdx.x] = part;
}

// one warp per system: r0.r0, tolerance, flags (also covers systems with no active vertex)
__global__ void k_pcg_init_scalars(const PcgPtrs* __restrict__ Pp, const int32_t* __restrict__ empty, double rtol) {
  const PcgPtrs& P = *Pp;
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= P.ns) return;
  const double total = sum_partials(P.partB + P.cta_first[s], P.cta_count[s]);
  if ((threadIdx.x & 31) != 0) return;
  P.sc.rz[0][s] = total;
  P.sc.rz[1][s] = __longlong_as_double(0x7ff0000000000000LL);  // +inf -> beta_0 = 0
  P.sc.rz0[s] = total;
  P.rz_last[s] = total;
  P.sc.tol2[s] = rtol * rtol * total;
  P.sc.pq[s] = 1.0;
  P.sc.psumA[s] = 1.0;
  P.sc.psumB[s] = total;
  P.sc.iters[s] = 0;
  P.sc.cap[s] = P.max_iter;
  P.sc.rz_mon[s] = __longlong_as_double(0x7ff0000000000000LL);
  P.sc.rounds[s] = 0;
  int st = FEA_SAMPLE_NOT_RUN, dn = 0;
  if (empty[s]) { st = FEA_SAMPLE_EMPTY_ROW; dn = 1; }
  else if (!(total > 0.0)) { st = isfinite(total) ? FEA_SAMPLE_CONVERGED : FEA_SAMPLE_BREAKDOWN; dn = 1; }
  P.sc.status[s] = st;
  P.sc.done[s] = dn;
  if (dn) atomicAdd(P.sc.n_done, 1);
}

static PcgPtrs make_ptrs(Batch& b, int max_iter) {
  PcgPtrs P;
  P.sys_of_cta = b.sys_of_cta;
  P.cta_first = b.cta_first;
  P.cta_count = b.cta_count;
  P.slice_len = b.slice_len;
  P.slice_ptr = b.slice_ptr;
  P.val = (const d4*)b.val;
  P.col = b.col;
  P.x = (double2*)b.x;
  P.rp = (d4*)b.rp;
  P.q = (double2*)b.q;
  P.partA = b.partA;
  P.partB = b.partB;
  P.sc = b.sc;
  P.rz_last = b.rz_last;
  P.active = (int4*)b.active_cta;
  P.n_active = 0;
  P.ncta = (int32_t)(b.NBR / kCtaRows);
  P.ns = b.ns;
  P.max_iter = max_iter;
  P.two_level = b.max_cta_count > kDirectSumMax ? 1 : 0;
  P.cl_order = b.cl_order;
  for (int k = 0; k < 9; ++k) {
    P.cl_off[k] = b.cl_off[k];
    P.cl_cnt[k] = b.cl_cnt[k];
  }
  P.cl_counter = b.cl_counter;
  P.cl_halo_cap = b.ctx->cluster_halo_cap;
  P.refine_dd = b.ctx->refine_rounds > 0 ? 1 : 0;
  P.xlo = (double2*)b.xlo;
  P.sb = (const double2*)b.sb;
  return P;
}

// one iteration = two kernels on a grid of g CTAs
static void launch_iteration(const PcgPtrs* dP, int g, int parity, cudaStream_t st, bool hint) {
  (hint ? k_pcg_spmv<true> : k_pcg_spmv<false>)<<<g, kT, 0, st>>>(dP, parity);
  k_pcg_update<<<g, kT, 0, st>>>(dP, parity);
}

// grid size classes: 148 * 2^(j/2), so a stale count costs at most ~41% idle CTAs
static int grid_class(int n_active, int ncta) {
  double g = 148.0;
  while ((int)g < n_active) g *= 1.4142135623730951;
  const int gi = (int)g;
  return gi < ncta ? gi : ncta;
}

static cudaError_t get_chunk_graph(Ctx& c, const PcgPtrs* dP, int g, bool hint, cudaGraphExec_t* out) {
  const int64_t key = 2 * (int64_t)g + (hint ? 1 : 0);   // the SpMV instantiation is baked into the kernel nodes
  auto it = c.pcg_graphs.find(key);
  if (it != c.pcg_graphs.end()) { *out = it->second; return cudaSuccess; }
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) return e;
  for (int i = 2; i < kChunk; ++i) launch_iteration(dP, g, i & 1, c.stream, hint);
  k_compact_active<<<1, 1024, 0, c.stream>>>((PcgPtrs*)dP);
  e = cudaStreamEndCapture(c.stream, &graph);
  if (e != cudaSuccess) return e;
  cudaGraphExec_t exec = nullptr;
  e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) return e;
  if (c.pcg_graphs.size() >= 256) {  // batches of many different sizes: start over
    for (auto& kv : c.pcg_graphs) cudaGraphExecDestroy(kv.second);
    c.pcg_graphs.clear();
  }
  c.pcg_graphs[key] = exec;
  *out = exec;
  return cudaSuccess;
}

// The whole lock-step solve.  Per chunk of kChunk iterations: two plain iterations (the first one
// bracketed by timing events), a cached graph of kChunk-2 iterations + work-list compaction, and
// an async read-back of (finished systems, active CTAs) that the host consumes one chunk late, so
// the stream never drains while systems are still iterating.
cudaError_t run_pcg(Batch& b, double rtol, int max_iter) {
  Ctx& c = *b.ctx;
  cudaStream_t st = c.stream;
  const int ncta = (int)(b.NBR / kCtaRows);
  PcgPtrs* dP = (PcgPtrs*)c.d_pcg_params;
  PcgPtrs P = make_ptrs(b, max_iter);
  int n_cluster = 0;
  P.cl_cnt[0] = 0;
  // the gather codes of a CTA's slices (2 B per block, up to 64 slices of 32 rows) must fit beside
  // the vectors in shared memory: meshes with extreme vertex valences use the streaming kernels
  const bool codes_fit = (int64_t)b.max_row_blocks * 64 * 32 * 2 <= 160 * 1024;
  for (int k = 1; k <= 8; ++k) {
    if (c.pcg_path != 0 || !codes_fit || (P.cl_cnt[k] && pcg_cluster_capacity(c, k) <= 0)) P.cl_cnt[k] = 0;
    n_cluster += P.cl_cnt[k];
  }
  const int per_iter = 2;
  // L2 eviction hints (matrix evict_first, gathered records evict_last) when the matrix does not fit the L2
  const bool hint = (int64_t)b.n_blocks * 36 > (int64_t)96 << 20;
  int64_t launches = 0;
  cudaError_t e;
  b.stats = fea_solve_stats{};
  b.t_spmv.clear();
  b.t_update.clear();
  if ((e = cudaEventRecord(c.ev_t0, st)) != cudaSuccess) return e;
  k_store_params<<<1, 32, 0, st>>>(P, dP);
  cudaMemsetAsync(b.sc.n_done, 0, sizeof(int32_t), st);
  cudaMemsetAsync(b.sc.arrive, 0, sizeof(int32_t) * 2 * b.ns, st);
  if (ncta) k_pcg_init_vectors<<<ncta, kT, 0, st>>>(dP, b.vertex_of_row, b.rhs, b.dscale, b.scoup);
  k_pcg_init_scalars<<<(b.ns + 3) / 4, 128, 0, st>>>(dP, b.empty, rtol);
  launches += 3;
  if (n_cluster > 0) {  // systems that fit on chip: one per cluster, pulled from a queue
    cudaMemsetAsync(b.cl_counter, 0, 24 * sizeof(int32_t), st);
    cudaEventRecord(c.ev_c0, st);
    // one persistent kernel per cluster class, largest clusters first; the largest class runs on the
    // main stream, every other one on an auxiliary stream of its own (more urgent the smaller its
    // clusters, fea_ctx_create), so that their clusters are co-scheduled and small clusters fill the
    // SMs that larger ones cannot use (GPC granularity)
    cudaEventRecord(c.ev_fork, st);
    bool used[Ctx::kAux] = {};
    int slot = 0;
    for (int k = 8; k >= 1; --k) {
      if (!P.cl_cnt[k]) continue;
      cudaStream_t ks = st;
      const int a = slot - 1;   // auxiliary stream of this class
      if (a >= 0 && c.aux[a]) {
        ks = c.aux[a];
        cudaStreamWaitEvent(ks, c.ev_fork, 0);
        used[a] = true;
      }
      if ((e = launch_pcg_cluster(c, dP, P.cl_cnt[k], k, ks)) != cudaSuccess) return e;
      launches += 1;
      ++slot;
    }
    for (int a = 0; a < Ctx::kAux; ++a) {
      if (!used[a]) continue;
      cudaEventRecord(c.ev_join[a], c.aux[a]);
      cudaStreamWaitEvent(st, c.ev_join[a], 0);
    }
    cudaEventRecord(c.ev_c1, st);
  }
  k_compact_active<<<1, 1024, 0, st>>>(dP);
  launches += 1;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  std::vector<int> done_after;  // finished systems observed after chunk k
  int timed = 0, k = 0, reopened_total = 0;
  const int max_chunks = (max_iter + kChunk - 1) / kChunk + 2;
  for (int round = 0; ncta && round <= c.refine_rounds + 1; ++round) {
    if (round > 0) {
      // residual replacement: check converged systems against their true residual, reopen failures
      int32_t* d_reopened = b.cl_counter + 9;
      cudaMemsetAsync(d_reopened, 0, sizeof(int32_t), st);
      k_pcg_true_residual<<<ncta, kT, 0, st>>>(dP, b.vertex_of_row, b.rhs, b.dscale, b.scoup, 0);
      k_pcg_refine_scalars<<<(b.ns + 3) / 4, 128, 0, st>>>(dP, d_reopened, round <= c.refine_rounds ? 1 : 0, 0);
      k_compact_active<<<1, 1024, 0, st>>>(dP);
      launches += 3;
      int32_t h_reopened = 0;
      if ((e = cudaMemcpyAsync(&h_reopened, d_reopened, sizeof(int32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
      if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
      reopened_total += h_reopened;
      if (h_reopened == 0) break;
    } else if (n_cluster >= b.ns) {
      // everything was solved AND verified against its true residual on chip -- unless a cluster
      // handed its system back (halo of a CTA too large for its shared memory)
      int32_t h_back = 0;
      if ((e = cudaMemcpyAsync(&h_back, b.cl_counter + 10, sizeof(int32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
      if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
      if (h_back == 0) break;
    }
    int n_active = ncta;  // stale upper bound of the work-list length
    const int k_end = k + max_chunks;
    const int k_first = k;  // polls of earlier rounds say "everything finished": never read them
    // monitor interval: 1024 iterations for plate-sized systems, longer for large ones whose
    // convergence curves have long plateaus (one chunk per 128 rows of the largest system)
    const int mon_chunks = b.max_cta_count > 32 ? b.max_cta_count : 32;
    for (; k < k_end; ++k) {
      const int g = grid_class(n_active, ncta);
      cudaGraphExec_t exec = nullptr;
      if ((e = get_chunk_graph(c, dP, g, hint, &exec)) != cudaSuccess) return e;
      const bool t = timed < kMaxTimed;
      if (t) cudaEventRecord(c.events[3 * timed], st);
      (hint ? k_pcg_spmv<true> : k_pcg_spmv<false>)<<<g, kT, 0, st>>>(dP, 0);
      if (t) cudaEventRecord(c.events[3 * timed + 1], st);
      k_pcg_update<<<g, kT, 0, st>>>(dP, 0);
      if (t) { cudaEventRecord(c.events[3 * timed + 2], st); ++timed; }
      launch_iteration(dP, g, 1, st, hint);
      if ((e = cudaGraphLaunch(exec, st)) != cudaSuccess) return e;
      launches += (int64_t)per_iter * kChunk + 1;
      if ((k - k_first + 1) % mon_chunks == 0) {   // periodic true-residual monitor (see k_pcg_true_residual)
        k_pcg_true_residual<<<ncta, kT, 0, st>>>(dP, b.vertex_of_row, b.rhs, b.dscale, b.scoup, 1);
        k_pcg_refine_scalars<<<(b.ns + 3) / 4, 128, 0, st>>>(dP, nullptr, 0, 1);
        launches += 2;
      }
      int32_t* hf = c.h_flag + 2 * (k & 1);
      cudaMemcpyAsync(hf, b.sc.n_done, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
      cudaMemcpyAsync(hf + 1, &dP->n_active, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
      cudaEventRecord(c.ev_poll[k & 1], st);
      if (k > k_first) {
        if ((e = cudaEventSynchronize(c.ev_poll[(k - 1) & 1])) != cudaSuccess) return e;
        const int32_t* hp = c.h_flag + 2 * ((k - 1) & 1);
        done_after.push_back(hp[0]);
        n_active = hp[1];
        if (hp[0] >= b.ns) { ++k; break; }
      }
    }
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;   // the polls lag one chunk
  }
  b.stats.refined_systems += reopened_total;
  if ((e = launch_finalize(b)) != cudaSuccess) return e;
  launches += 3;
  if ((e = cudaEventRecord(c.ev_t1, st)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  // statistics
  std::vector<int32_t> it(b.ns), stt(b.ns), order(n_cluster > 0 ? b.cl_off[8] + b.cl_cnt[8] : 0);
  int32_t h_restarts = 0;
  long long h_reads[3] = {0, 0, 0};
  if ((e = cudaMemcpyAsync(it.data(), b.sc.iters, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(stt.data(), b.sc.status, sizeof(int32_t) * b.ns, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  if (n_cluster > 0) {
    if ((e = cudaMemcpyAsync(order.data(), b.cl_order, sizeof(int32_t) * order.size(), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(&h_restarts, b.cl_counter, sizeof(int32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(h_reads, b.cl_counter + 16, sizeof(h_reads), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
  }
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
  int itmax = 0, nconv = 0;
  for (int s = 0; s < b.ns; ++s) {
    itmax = it[s] > itmax ? it[s] : itmax;
    nconv += stt[s] == FEA_SAMPLE_CONVERGED;
  }
  b.stats.iterations = itmax;
  b.stats.n_converged = nconv;
  if (n_cluster > 0) {
    int64_t tot = 0;
    int nclusters = 0;
    int best = 1;
    for (int k = 1; k <= 8; ++k) {
      if (P.cl_cnt[k] > P.cl_cnt[best]) best = k;
      for (int i = 0; i < P.cl_cnt[k]; ++i) tot += it[order[b.cl_off[k] + i]];
      const int capn = P.cl_cnt[k] ? pcg_cluster_capacity(c, k) : 0;
      if (P.cl_cnt[k]) nclusters += P.cl_cnt[k] < capn ? P.cl_cnt[k] : capn;
    }
    b.stats.cluster_systems = n_cluster;
    b.stats.cluster_size = best;   // the class that solved most systems
    b.stats.cluster_count = nclusters;
    b.stats.cluster_iterations = tot;
    cudaEventElapsedTime(&b.stats.cluster_ms, c.ev_c0, c.ev_c1);
    b.stats.refined_systems += h_restarts;
    b.stats.cluster_block_reads_tmem = h_reads[0];
    b.stats.cluster_block_reads_smem = h_reads[1];
    b.stats.cluster_block_reads_l2 = h_reads[2];
#if defined(FEA_CLUSTER_PROFILE) || defined(FEA_CLUSTER_ACCOUNT)
    pcg_cluster_profile_dump();
#endif
  }
  b.t_spmv.assign(timed, 0.f);
  b.t_update.assign(timed, 0.f);
  for (int t = 0; t < timed; ++t) {
    cudaEventElapsedTime(&b.t_spmv[t], c.events[3 * t], c.events[3 * t + 1]);
    cudaEventElapsedTime(&b.t_update[t], c.events[3 * t + 1], c.events[3 * t + 2]);
  }
  // average only over timed launches that ran with (nearly) every system still active
  // (a few systems may finish at once, e.g. loads that fall on constrained vertices)
  double sa = 0, su = 0;
  int na = 0;
  for (int t = 0; t < timed; ++t) {
    const bool all_active = (t == 0) || (t - 1 < (int)done_after.size() && done_after[t - 1] * 20 <= b.ns);
    if (!all_active) break;
    sa += b.t_spmv[t];
    su += b.t_update[t];
    ++na;
  }
  if (getenv("FEA_DEBUG")) {
    fprintf(stderr, "[fea] solve: chunks=%d timed=%d na=%d graphs=%zu done_after:", k, timed, na, c.pcg_graphs.size());
    for (size_t i = 0; i < done_after.size() && i < 24; ++i) fprintf(stderr, " %d", done_after[i]);
    fprintf(stderr, "\n");
  }
  b.stats.spmv_launches_timed = na;
  b.stats.update_launches_timed = na;
  b.stats.spmv_ms_avg = na ? (float)(sa / na) : 0.f;
  b.stats.update_ms_avg = na ? (float)(su / na) : 0.f;
  cudaEventElapsedTime(&b.stats.solve_ms, c.ev_t0, c.ev_t1);
  b.stats.kernel_launches = launches;
  c.launches += launches;
  return cudaSuccess;
}

void pcg_release(Ctx& c) {
  for (auto& kv : c.pcg_graphs) cudaGraphExecDestroy(kv.second);
  c.pcg_graphs.clear();
}

// ---------------------------------------------------------------------------
// finalisation: u = S xhat scattered to the full DOF numbering (zeros at fixed DOFs, A-15),
// per-sample (min, max) of both components (ranges.txt, A-17), relative residuals.
// ---------------------------------------------------------------------------
__global__ void k_unscale_scatter(int64_t NV, const int32_t* __restrict__ vsample,
                                  const int32_t* __restrict__ row_of_vertex, const double* __restrict__ dscale,
                                  const double* __restrict__ scoup,
                                  const double2* __restrict__ x, const int32_t* __restrict__ status,
                                  double2* __restrict__ u) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV) return;
  double2 o = make_double2(0.0, 0.0);
  if (status[vsample[v]] == FEA_SAMPLE_EMPTY_ROW) {
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    o = make_double2(nan, nan);
  } else {
    const int row = row_of_vertex[v];
    if (row >= 0) {
      const double2 xv = x[row];
      o = make_double2(fma(scoup[row], xv.y, dscale[2 * (int64_t)row] * xv.x), dscale[2 * (int64_t)row + 1] * xv.y);   // u = S xhat
    }
  }
  u[v] = o;
}

__global__ void k_minmax(const int64_t* __restrict__ vtx_off, const double2* __restrict__ u,
                         double* __restrict__ ranges) {
  __shared__ double sm[4][8];
  const int s = blockIdx.x;
  const int64_t v0 = vtx_off[s], v1 = vtx_off[s + 1];
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  double mnx = inf, mxx = -inf, mny = inf, mxy = -inf;
  for (int64_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
    const double2 w = u[v];
    mnx = fmin(mnx, w.x); mxx = fmax(mxx, w.x);
    mny = fmin(mny, w.y); mxy = fmax(mxy, w.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fmin(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
    mxx = fmax(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    mny = fmin(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxy = fmax(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { sm[0][w] = mnx; sm[1][w] = mxx; sm[2][w] = mny; sm[3][w] = mxy; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) {
      mnx = fmin(mnx, sm[0][i]); mxx = fmax(mxx, sm[1][i]);
      mny = fmin(mny, sm[2][i]); mxy = fmax(mxy, sm[3][i]);
    }
    ranges[4 * s + 0] = mnx; ranges[4 * s + 1] = mxx;
    ranges[4 * s + 2] = mny; ranges[4 * s + 3] = mxy;
  }
}

__global__ void k_relres(int ns, const double* __restrict__ rz_last, const double* __restrict__ rz0,
                         double* __restrict__ relres) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ns) return;
  relres[s] = rz0[s] > 0.0 ? sqrt(rz_last[s] / rz0[s]) : 0.0;
}

cudaError_t launch_finalize_to(Batch& b, const double* x, const int32_t* status, const double* rz_last, const double* rz0,
                               double* u, double* ranges, double* relres) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  if (b.NV)
    k_unscale_scatter<<<(unsigned)((b.NV + T - 1) / T), T, 0, st>>>(b.NV, b.vsample, b.row_of_vertex, b.dscale, b.scoup,
                                                                   (const double2*)x, status, (double2*)u);
  k_minmax<<<b.ns, 256, 0, st>>>(b.d_vtx_off, (const double2*)u, ranges);
  k_relres<<<(b.ns + T - 1) / T, T, 0, st>>>(b.ns, rz_last, rz0, relres);
  return cudaGetLastError();
}

cudaError_t launch_finalize(Batch& b) {
  return launch_finalize_to(b, b.x, b.sc.status, b.rz_last, b.sc.rz0, b.u, b.ranges, b.relres);
}

// ---------------------------------------------------------------------------
// Test hook: y = K x for one sample through k_pcg_spmv (beta = 0 path).
// ---------------------------------------------------------------------------
__global__ void k_spmv_load(int64_t NBR, const int32_t* __restrict__ vertex_of_row,
                            const int32_t* __restrict__ vrank, int64_t v0, int64_t v1,
                            const double* __restrict__ dscale, const double* __restrict__ scoup,
                            const double* __restrict__ xin, d4* __restrict__ rp) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int v = vertex_of_row[row];
  double2 o = make_double2(0.0, 0.0);
  if (v >= v0 && v < v1) {
    const int rk = vrank[v];
    const double s0 = dscale[2 * row], s1 = dscale[2 * row + 1];
    if (s0 > 0 && s1 > 0) {   // xhat = S^-1 x
      const double x1 = xin[2 * rk + 1] / s1;
      o = make_double2((xin[2 * rk] - scoup[row] * x1) / s0, x1);
    }
  }
  d4 rec;
  rec.x = o.x;
  rec.y = o.y;
  rec.z = rec.w = 0.0;
  rp[row] = rec;
}
__global__ void k_spmv_store(int64_t NBR, const int32_t* __restrict__ vertex_of_row,
                             const int32_t* __restrict__ vrank, int64_t v0, int64_t v1,
                             const double* __restrict__ dscale, const double* __restrict__ scoup,
                             const double2* __restrict__ q, double* __restrict__ yout) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= NBR) return;
  const int v = vertex_of_row[row];
  if (v >= v0 && v < v1) {
    const int rk = vrank[v];
    const double s0 = dscale[2 * row], s1 = dscale[2 * row + 1];
    const double2 qv = q[row];
    const double y0 = s0 > 0 ? qv.x / s0 : 0.0;                       // y = S^-T q
    yout[2 * rk] = y0;
    yout[2 * rk + 1] = s1 > 0 ? (qv.y - scoup[row] * y0) / s1 : 0.0;
  }
}
__global__ void k_spmv_scalars(int ns, SysScalars sc, const int32_t* __restrict__ cta_first,
                               const int32_t* __restrict__ cta_count, double* __restrict__ partB) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= ns) return;
  sc.rz[0][s] = 1.0;
  sc.rz[1][s] = __longlong_as_double(0x7ff0000000000000LL);  // beta = 0: p = r
  sc.done[s] = 0;
  sc.iters[s] = 0;
  sc.cap[s] = 1 << 30;
  sc.tol2[s] = 0.0;
  sc.psumB[s] = 1.0;
  for (int i = 0; i < cta_count[s]; ++i) partB[cta_first[s] + i] = 1.0;  // "not converged"
}

cudaError_t launch_plain_spmv(Batch& b, int32_t s, const double* d_x, double* d_y) {
  cudaStream_t st = b.ctx->stream;
  const int T = 256;
  const int ncta = (int)(b.NBR / kCtaRows);
  if (!ncta) return cudaSuccess;
  const unsigned g = (unsigned)((b.NBR + T - 1) / T);
  const int64_t v0 = b.vtx_off[s], v1 = b.vtx_off[s + 1];
  PcgPtrs* dP = (PcgPtrs*)b.ctx->d_pcg_params;
  k_store_params<<<1, 32, 0, st>>>(make_ptrs(b, 1 << 30), dP);
  k_spmv_scalars<<<(b.ns + T - 1) / T, T, 0, st>>>(b.ns, b.sc, b.cta_first, b.cta_count, b.partB);
  k_compact_active<<<1, 1024, 0, st>>>(dP);
  k_spmv_load<<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.vrank, v0, v1, b.dscale, b.scoup, d_x, (d4*)b.rp);
  cudaMemsetAsync(b.sc.arrive, 0, sizeof(int32_t) * 2 * b.ns, st);
  k_pcg_spmv<false><<<ncta, kT, 0, st>>>(dP, 0);
  k_spmv_store<<<g, T, 0, st>>>(b.NBR, b.vertex_of_row, b.vrank, v0, v1, b.dscale, b.scoup, (const double2*)b.q, d_y);
  return cudaGetLastError();
}

}  // namespace fea
