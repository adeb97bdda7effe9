// K5 (on-chip path): Jacobi-PCG of one system per thread-block cluster, matrix resident in shared
// memory -- replaces Newton + ScipyDirect(SuperLU) + SimpleTimeSteppingSolver (reference
// datagen/fea_analysis.py:371-375, 425-439) for the plate-sized systems of the data-synthesis loop.
//
// A default-density plate has 2.5-10 k vertices: its scaled block-SELL matrix is 0.5-2.3 MB and its
// CG vectors a few hundred KB.  A thread-block cluster of CL CTAs x 512 threads keeps ONE system on
// chip for its whole solve; CL (1..8) is the smallest cluster whose CTAs hold the system's rows
// (2048 per CTA), one persistent kernel per CL, launched on concurrent streams (run_pcg):
//
//   * every CTA owns a contiguous range of the system's 32-row slices; the gather codes of all its
//     slices and the 2x2 blocks of as many slices as fit are copied from HBM to shared memory ONCE,
//     the blocks of the other slices are streamed from L2 every iteration;
//   * x, r of a thread's (up to 4) block rows live in registers for the whole solve;
//   * the search direction p lives in the owner's shared memory.  The rows a CTA gathers from its
//     peers (its "halo", found once per system with a bitmap + prefix sum) have slots behind its own
//     rows, and their owners PUSH the new values into those slots every iteration (send list,
//     st.async): every gather of the SpMV is a plain ld.shared;
//   * dot products: every warp pushes its partial into a table in all CTAs (st.async); every warp
//     then adds its local copy in the same fixed order -- no atomics, bitwise reproducible,
//     independent of which cluster or SM runs the system;
//   * NO cluster barrier inside the iteration: the three hand-overs (halo of p, p.q partials, r.r
//     partials) complete on mbarrier transaction counts in the receiving CTA; a warp waits for the
//     halo only when it reaches a slice that reads it;
//   * a converged system is verified against its TRUE residual; if fp64 CG cannot reach the
//     tolerance (the floor eps |K| |x| of an ill-conditioned plate) it is finished by iterative
//     refinement with a double-double residual; every 1024 iterations the same pass monitors
//     progress and stops mechanisms.
//
// Clusters are persistent and pull systems from a queue (longest job first), so there is no
// lock-step and no tail of idle CTAs waiting for the slowest system of a batch.  HBM traffic is one
// read of the matrix and vectors per SOLVE instead of per iteration.
// Systems too large for a cluster (> 16 384 block rows), and systems whose halo does not fit beside
// the matrix (handed back by the kernel), use the streaming kernels of k_pcg.cu.
#include <cooperative_groups.h>

#include <cstdio>
#include <cstdlib>

#include "fea_internal.cuh"
#include "pcg_params.cuh"

namespace cg = cooperative_groups;

namespace fea {

#if defined(FEA_CLUSTER_PROFILE) || defined(FEA_CLUSTER_ACCOUNT)
__device__ unsigned long long g_cl_prof[16];
#endif
#ifdef FEA_CLUSTER_TRACE
// per system: start / end of its solve (ns, %globaltimer), SM of rank 0, cluster size and iterations -- the
// timeline of a batch (tools/cluster_timeline.py); dumped by pcg_cluster_profile_dump to $FEA_CLUSTER_TRACE_FILE
__device__ unsigned long long g_cl_trace[8192][4];
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#endif
#ifdef FEA_CLUSTER_DEBUG
#define DBG(...) do { if (rank == 0 && tid == 0) printf(__VA_ARGS__); } while (0)
#else
#define DBG(...) do { } while (0)
#endif
#ifdef FEA_CLUSTER_PROFILE
#define PROF_T(i) do { if (prof) { const long long t_ = clock64(); h->prof[i] += t_ - h->prof[9]; h->prof[9] = t_; } } while (0)
#else
#define PROF_T(i) do { } while (0)
#endif

constexpr int kClMax = 8;                   // largest cluster (portable maximum)
constexpr int kClT = 512;                   // threads per CTA (one CTA per SM)
constexpr int kClW = kClT / 32;             // warps per CTA
constexpr int kClRpt = 4;                   // block rows per thread
constexpr int kClU = 4;                     // gathers in flight per thread (resident slices)
constexpr int kClUs = 4;                    // blocks in flight per thread (slices streamed from L2)
static_assert(kClU % 4 == 0 && kClUs % 4 == 0, "gather codes are fetched four at a time");
constexpr int kMonitor = 1024;              // iterations between true-residual monitor passes
constexpr int kClSlices = kClT / 32 * kClRpt;  // local slices per CTA (64 with 512 threads)
constexpr int kClSmemBytes = 227 * 1024;    // dynamic shared memory per CTA: all an SM has
constexpr int kClWords = (kClMax * kClSlices + kClT - 1) / kClT * kClT;   // 32-row slices of the largest system = words of the halo bitmap (padded to whole threads)
static_assert(kClWords % kClT == 0 && kClSlices <= kClT && kClSlices * 32 <= 4096, "the halo scan handles kClWords / kClT bitmap words per thread");
constexpr int kClWpt = kClWords / kClT;     // bitmap words per thread (consecutive)
constexpr int kClTmpBytes = 2 * kClWords * 4 + 128;   // halo bitmap + its prefix sums (set-up only)
// Tensor memory as a matrix store.  The SM's 256 KB of TMEM is idle in fp64 code; tcgen05.ld.32x32b gives
// every thread of a warp a private strip of it (lane = thread, column = 32-bit word), which is exactly the
// shape of a block-SELL slice (one row per lane, one 2x2 block = 8 columns).  Measured (tools/tmem_bw.cu):
// 456 B/clk/SM into registers, and beside saturating ld.shared traffic both run at 120 B/clk/SM -- TMEM reads
// do not use the L1TEX data pipe that bounds this kernel, while blocks streamed from L2 do (at 61 B/clk/SM).
// A warp may only touch the 32 lanes of its quadrant (warp % 4); the warps of a quadrant split the columns.
constexpr int kTmCols = 512;                             // columns allocated per CTA: all of the SM's TMEM (a power of two)
constexpr int kTmWarpCols = kTmCols / (kClW / 4) / 8 * 8;  // columns of one warp's strip
constexpr int kTmWarpBlocks = kTmWarpCols / 8;             // 2x2 blocks per lane in that strip
static_assert(kClW % 4 == 0, "TMEM strips are per quadrant of four warps");

struct ClHeader {                 // start of the dynamic shared memory of every CTA
  // one hand-over per iteration: every warp pushes the record (p.q, q.q, r.q, r.r) of its rows to all CTAs;
  // two tables + two barriers used alternately, so that a warp that runs ahead can never write into the
  // table a slower warp is still summing, nor complete bytes on a phase that has not opened yet
  alignas(32) double partA[2][kClMax * kClW * 4];
  double partB[kClMax * kClW];    // r.r partials of the true-residual passes (check / monitor / refinement)
  double pad1_;                   // unused; without it ptxas allocates one more register in some k_pcg_cluster<CL>
  double rz_monitor;              // smallest true r.r any monitor pass has seen
  double tol2;                    // rtol^2 * r0.r0 of the current system (tightened by an extended-precision round)
  int32_t mon_strikes;            // consecutive monitor passes without a 4x gain on rz_monitor
  int32_t pad2_;
  uint64_t mbarA[2], mbarB, mbarP; // transaction barriers: iteration records (even / odd) / true-residual partials / halo of p
  int32_t it_limit;               // iteration budget of the current system (tightened after a restart)
  int32_t next_sys;               // (rank 0) queue entry the cluster works on next
  int32_t n_send;                 // entries of this CTA's send list
  int32_t off_pbuf, mat0;         // byte offsets of the p buffer and of the matrix area
  int32_t pad_;
  int32_t send_from[kClMax];      // (owner side) rows of this CTA that CTA c gathers
  int32_t seg_off[kClMax];        // (consumer side) first entry of this CTA's segment in owner o's send list
  int32_t fit[kClMax];            // the layout of CTA c fits into its shared memory
  int32_t wsum[kClW];             // block-scan scratch
  int32_t s_halo[kClSlices];      // the slice gathers rows of other CTAs (its warp waits for the halo first)
  int32_t s_off[kClSlices];       // byte offset of the slice's other blocks in the matrix area, -1 = global
  int32_t s_len[kClSlices];       // blocks per row of the slice
  int32_t s_aoff[kClSlices];      // entry offset of the slice's gather codes (groups of 4 per lane: [L/4][32][4] u16)
  int32_t s_nt[kClSlices];        // the first s_nt blocks of every row of the slice live in tensor memory
  int32_t s_tcol[kClSlices];      // their first column inside the warp's TMEM strip
  uint32_t tmem_base;             // address of the CTA's TMEM allocation
  int32_t pad3_;
  int64_t s_base[kClSlices];      // first entry of the slice in the global block-SELL arrays
#ifdef FEA_CLUSTER_PROFILE
  long long prof[10];
#endif
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ double2 ld_shared_f64x2(uint32_t addr) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ int ld_cluster_s32(uint32_t addr) {
  int v;
  asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void st_cluster_s32(uint32_t addr, int v) {
  asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// ---- tensor memory: 2x2 blocks of one row per lane (8 words per block) ---------------------------------
// Four (two) blocks of this lane's row and the matching four (two) gathered entries of p, in ONE asm
// statement: the registers of a tcgen05.ld are valid after tcgen05.wait::ld only, so the wait and the
// moves into 64-bit registers must not be separable from the load by the compiler's scheduler.  The
// shared-memory gathers are issued between the load and the wait, i.e. both are in flight together.
__device__ __forceinline__ void tmem_ld4_gather4(uint32_t taddr, const uint32_t (&ga)[4], d4 (&b)[4], double2 (&p)[4]) {
  asm volatile(
      "{\n\t"
      ".reg .b32 t<32>;\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15,t16,t17,t18,t19,t20,t21,t22,t23,t24,t25,t26,t27,t28,t29,t30,t31}, [%24];\n\t"
      "ld.shared.v2.f64 {%16,%17}, [%25];\n\t"
      "ld.shared.v2.f64 {%18,%19}, [%26];\n\t"
      "ld.shared.v2.f64 {%20,%21}, [%27];\n\t"
      "ld.shared.v2.f64 {%22,%23}, [%28];\n\t"
      "tcgen05.wait::ld.sync.aligned;\n\t"
      "mov.b64 %0, {t0,t1};\n\t mov.b64 %1, {t2,t3};\n\t mov.b64 %2, {t4,t5};\n\t mov.b64 %3, {t6,t7};\n\t"
      "mov.b64 %4, {t8,t9};\n\t mov.b64 %5, {t10,t11};\n\t mov.b64 %6, {t12,t13};\n\t mov.b64 %7, {t14,t15};\n\t"
      "mov.b64 %8, {t16,t17};\n\t mov.b64 %9, {t18,t19};\n\t mov.b64 %10, {t20,t21};\n\t mov.b64 %11, {t22,t23};\n\t"
      "mov.b64 %12, {t24,t25};\n\t mov.b64 %13, {t26,t27};\n\t mov.b64 %14, {t28,t29};\n\t mov.b64 %15, {t30,t31};\n\t"
      "}"
      : "=d"(b[0].x), "=d"(b[0].y), "=d"(b[0].z), "=d"(b[0].w), "=d"(b[1].x), "=d"(b[1].y), "=d"(b[1].z), "=d"(b[1].w),
        "=d"(b[2].x), "=d"(b[2].y), "=d"(b[2].z), "=d"(b[2].w), "=d"(b[3].x), "=d"(b[3].y), "=d"(b[3].z), "=d"(b[3].w),
        "=d"(p[0].x), "=d"(p[0].y), "=d"(p[1].x), "=d"(p[1].y), "=d"(p[2].x), "=d"(p[2].y), "=d"(p[3].x), "=d"(p[3].y)
      : "r"(taddr), "r"(ga[0]), "r"(ga[1]), "r"(ga[2]), "r"(ga[3]));
}
__device__ __forceinline__ void tmem_ld2_gather2(uint32_t taddr, uint32_t ga0, uint32_t ga1, d4 (&b)[4], double2 (&p)[4]) {
  asm volatile(
      "{\n\t"
      ".reg .b32 t<16>;\n\t"
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {t0,t1,t2,t3,t4,t5,t6,t7,t8,t9,t10,t11,t12,t13,t14,t15}, [%12];\n\t"
      "ld.shared.v2.f64 {%8,%9}, [%13];\n\t"
      "ld.shared.v2.f64 {%10,%11}, [%14];\n\t"
      "tcgen05.wait::ld.sync.aligned;\n\t"
      "mov.b64 %0, {t0,t1};\n\t mov.b64 %1, {t2,t3};\n\t mov.b64 %2, {t4,t5};\n\t mov.b64 %3, {t6,t7};\n\t"
      "mov.b64 %4, {t8,t9};\n\t mov.b64 %5, {t10,t11};\n\t mov.b64 %6, {t12,t13};\n\t mov.b64 %7, {t14,t15};\n\t"
      "}"
      : "=d"(b[0].x), "=d"(b[0].y), "=d"(b[0].z), "=d"(b[0].w), "=d"(b[1].x), "=d"(b[1].y), "=d"(b[1].z), "=d"(b[1].w),
        "=d"(p[0].x), "=d"(p[0].y), "=d"(p[1].x), "=d"(p[1].y)
      : "r"(taddr), "r"(ga0), "r"(ga1));
}
__device__ __forceinline__ void tmem_st_block(uint32_t taddr, const d4& b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr),
               "r"(__double2loint(b.x)), "r"(__double2hiint(b.x)), "r"(__double2loint(b.y)), "r"(__double2hiint(b.y)),
               "r"(__double2loint(b.z)), "r"(__double2hiint(b.z)), "r"(__double2loint(b.w)), "r"(__double2hiint(b.w))
               : "memory");
}

// ---- synchronisation inside an iteration: transaction barriers, no cluster barrier --------------
// Everything a CTA needs from its peers in an iteration -- the dot-product partials and the halo
// of the search direction -- is PUSHED into its shared memory with st.async, which adds the bytes
// it delivers to the transaction count of an mbarrier in the DESTINATION CTA.  A thread that sees
// the phase complete (try_wait, acquire at cluster scope) sees the data.  Compared with
// barrier.cluster this needs no release fence (cg::cluster_group::sync() compiles to MEMBAR.ALL.GPU
// + ERRBAR before the arrive: measured 7 % of the solve for the one barrier that published p) and
// no cluster-wide rendezvous.  Each barrier has one pending arrival per phase: thread 0 of the
// waiting CTA arrives with expect_tx(bytes) just before it waits; bytes that land earlier only make
// the transaction count transiently negative.  A phase cannot be overtaken: the pushes of iteration
// k+1 follow the sender's wait on the r.r partials of iteration k, which every warp of the cluster
// has pushed only after its last gather of iteration k.
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arm(uint32_t mbar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(mbar), "r"(parity) : "memory");
}
// all `bytes` of the phase have landed in this CTA (parity = phases of this barrier seen so far, mod 2)
__device__ __forceinline__ void await_tx(uint64_t* mbar, uint32_t bytes, uint32_t parity, int tid) {
  const uint32_t a = smem_u32(mbar);
  if (tid == 0) mbar_arm(a, bytes);
  mbar_wait(a, parity);
}

// Dot products over the cluster, push model: lane c < CL of every warp sends the warp's partial to
// slot [rank][warp] of CTA c's table; once all CL x 16 partials have landed every warp of every CTA
// adds the slots of its own copy in the same fixed order, so all of them hold the same bits and no
// intra-CTA broadcast is needed.
template <int CL>
__device__ __forceinline__ void push_partial(ClHeader* h, uint32_t field_off, uint32_t mbar_off, int rank, int warp, int lane, double v) {
  if (lane < CL) {
    const uint32_t base = mapa_u32(smem_u32(h), lane);   // the header of CTA `lane`
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f64 [%0], %1, [%2];" ::"r"(
                     base + field_off + 8u * (uint32_t)(rank * kClW + warp)),
                 "d"(v), "r"(base + mbar_off)
                 : "memory");
  }
}
// The iteration's record: lane c < CL of every warp sends (p.q, q.q, r.q, r.r) of the warp's rows to slot
// [rank][warp] of CTA c's table (two 16-byte st.async).  The sum: lane l adds component l & 3 of the records
// l >> 2, (l >> 2) + 8, ... (consecutive doubles across the lanes: conflict-free), three butterfly steps
// combine the lanes of a component, four broadcasts hand every lane all four totals -- the same order
// in every warp of every CTA, hence the same bits.
template <int CL>
__device__ __forceinline__ void push_record(ClHeader* h, int buf, int rank, int warp, int lane, double a, double b, double c, double d) {
  if (lane < CL) {
    const uint32_t base = mapa_u32(smem_u32(h), lane);   // the header of CTA `lane`
    const uint32_t dst = base + (uint32_t)offsetof(ClHeader, partA) + (uint32_t)buf * (uint32_t)sizeof(h->partA[0]) +
                         32u * (uint32_t)(rank * kClW + warp);
    const uint32_t bar = base + (uint32_t)offsetof(ClHeader, mbarA) + 8u * (uint32_t)buf;
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(dst), "d"(a), "d"(b), "r"(bar) : "memory");
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(dst + 16u), "d"(c), "d"(d), "r"(bar) : "memory");
  }
}
template <int CL>
__device__ __forceinline__ void sum_records(const double* t, int lane, double& a, double& b, double& c, double& d) {
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < (CL * kClW * 4 + 31) / 32; ++i)
    if (lane + 32 * i < CL * kClW * 4) acc += t[lane + 32 * i];
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  acc += __shfl_xor_sync(0xffffffffu, acc, 8);
  acc += __shfl_xor_sync(0xffffffffu, acc, 16);
  a = __shfl_sync(0xffffffffu, acc, 0);
  b = __shfl_sync(0xffffffffu, acc, 1);
  c = __shfl_sync(0xffffffffu, acc, 2);
  d = __shfl_sync(0xffffffffu, acc, 3);
}
template <int CL>
__device__ __forceinline__ double sum_table(const double* t, int lane) {
  double acc = 0.0;
#pragma unroll
  for (int i = 0; i < (CL * kClW + 31) / 32; ++i)
    if (lane + 32 * i < CL * kClW) acc += t[lane + 32 * i];
  return warp_sum(acc);
}

// ---- extended-precision refinement ------------------------------------------------------------
// fp64 CG cannot push the TRUE residual b - K x below ~eps * |K| * max_k |x_k| (the recursion
// r -= alpha q and the product K x both round at that level).  On plates with a weakly held part
// (kappa ~ 1e7 and beyond; the residual climbs by orders of magnitude before it falls) that floor is
// above the tolerance: the recursive residual converges, the true one stalls around 1e-7, and the
// displacement is off by more than the 1e-8 the reference's direct solve is matched to.  Such a
// system is finished by iterative refinement: x is kept as an unevaluated sum xhi + xlo, the true
// residual is formed in double-double arithmetic (error-free products and sums, ~1e-30), and the
// SAME fp64 CG solves K d = r for the correction, which only has to gain a few digits per round.
// The rounds run on the rows' owners through global memory (a few per 1000 systems; the vectors are
// L2 resident), out of line so that the registers of the iteration are untouched.
struct dd2 { double hi, lo; };
__device__ __forceinline__ dd2 two_sum(double a, double b) {
  const double s = __dadd_rn(a, b);
  const double bb = __dsub_rn(s, a);
  return dd2{s, __dadd_rn(__dsub_rn(a, __dsub_rn(s, bb)), __dsub_rn(b, bb))};
}
__device__ __forceinline__ dd2 quick_two_sum(double a, double b) {   // |a| >= |b|
  const double s = __dadd_rn(a, b);
  return dd2{s, __dsub_rn(b, __dsub_rn(s, a))};
}
__device__ __forceinline__ dd2 dd_add(dd2 a, double bh, double bl) {
  const dd2 s = two_sum(a.hi, bh);
  return quick_two_sum(s.hi, __dadd_rn(__dadd_rn(s.lo, a.lo), bl));
}
// acc -= k * (xh + xl), the product k * xh taken exactly (fma residual)
__device__ __forceinline__ dd2 dd_msub(dd2 acc, double k, double xh, double xl) {
  const double p = __dmul_rn(k, xh);
  const double e = __fma_rn(k, xl, __fma_rn(k, xh, -p));
  return dd_add(acc, -p, -e);
}
// x (hi, lo) += d for this thread's rows; first = the sum starts from d alone
__device__ __forceinline__ void dd_fold_rows(const PcgPtrs& P, int64_t my_row0, int n_own, int tid, const double2 (&d)[kClRpt], bool first) {
#pragma unroll
  for (int k = 0; k < kClRpt; ++k) {
    const int lr = tid + kClT * k;
    if (lr >= n_own) continue;
    double2 hi = d[k], lo = make_double2(0.0, 0.0);
    if (!first) {
      const double2 h0 = P.x[my_row0 + lr], l0 = P.xlo[my_row0 + lr];
      const dd2 a = dd_add(dd2{h0.x, l0.x}, d[k].x, 0.0), b = dd_add(dd2{h0.y, l0.y}, d[k].y, 0.0);
      hi = make_double2(a.hi, b.hi);
      lo = make_double2(a.lo, b.lo);
    }
    P.x[my_row0 + lr] = hi;
    P.xlo[my_row0 + lr] = lo;
  }
}
// r = S b - Khat (xhi + xlo) for this thread's rows, in double-double, rounded once; written into
// the (r.x, r.y) fields of the row records (the right-hand side of the correction solve);
// returns the thread's part of r.r
__device__ __noinline__ double dd_residual_rows(const PcgPtrs* Pp, int64_t my_row0, int n_own, int tid) {
  const PcgPtrs& P = *Pp;
  double part = 0.0;
#pragma unroll 1
  for (int k = 0; k < kClRpt; ++k) {
    const int lr = tid + kClT * k;
    if (lr >= n_own) continue;
    const int64_t row = my_row0 + lr;
    const int lane = (int)(row & 31);
    const int L = P.slice_len[row >> 5];
    const int64_t base = P.slice_ptr[row >> 5] + lane;
    const double2 b = P.sb[row], xh = __ldcg(P.x + row), xl = __ldcg(P.xlo + row);
    dd2 r0{b.x, 0.0}, r1{b.y, 0.0};
    r0 = dd_add(r0, -xh.x, -xl.x);            // the scaled diagonal block is the identity
    r1 = dd_add(r1, -xh.y, -xl.y);
#pragma unroll 1
    for (int j = 0; j < L; ++j) {
      const int c = P.col[base + (int64_t)j * 32];
      const d4 kv = P.val[base + (int64_t)j * 32];
      const double2 ch = __ldcg(P.x + c), cl = __ldcg(P.xlo + c);
      r0 = dd_msub(r0, kv.x, ch.x, cl.x);
      r0 = dd_msub(r0, kv.y, ch.y, cl.y);
      r1 = dd_msub(r1, kv.z, ch.x, cl.x);
      r1 = dd_msub(r1, kv.w, ch.y, cl.y);
    }
    d4 rec = P.rp[row];
    rec.x = __dadd_rn(r0.hi, r0.lo);
    rec.y = __dadd_rn(r1.hi, r1.lo);
    P.rp[row] = rec;
    part = fma(rec.x, rec.x, fma(rec.y, rec.y, part));
  }
  return part;
}
constexpr int kMaxRefine = 3;            // extended-precision rounds per system
constexpr double kRefineTighten = 1e-4;  // a refined system is solved to rtol / 100: what stalls fp64 CG also
                                         // amplifies the residual into the displacement (measured: 200x)

template <int CL>
__global__ void __launch_bounds__(kClT, 1) k_pcg_cluster(const PcgPtrs* __restrict__ Pp) {
  constexpr int kCl = CL;
  constexpr int kClass = CL;
  extern __shared__ __align__(128) unsigned char smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const PcgPtrs& P = *Pp;
  ClHeader* h = reinterpret_cast<ClHeader*>(smem);
  constexpr int kHdr = (sizeof(ClHeader) + 127) / 128 * 128;
  const int rank = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  const uint32_t smem_a = smem_u32(smem);
  uint32_t phase = 0;   // bits 0 / 3: parity of the next phase of the even / odd record barrier; bit 1: true-residual partials; bit 2: halo
#ifdef FEA_CLUSTER_ACCOUNT
  const long long acc_t0 = clock64();   // SM-cycle accounting: CTA lifetime / system set-up / iterations
#endif
  if (tid == 0) {
    mbar_init(smem_u32(&h->mbarA[0]), 1);
    mbar_init(smem_u32(&h->mbarA[1]), 1);
    mbar_init(smem_u32(&h->mbarB), 1);
    mbar_init(smem_u32(&h->mbarP), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // (the first cluster.sync() of the queue loop orders the initialisation before any push)
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&h->tmem_base)), "n"(kTmCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // this warp's TMEM strip: lanes of its quadrant, its share of the columns
  const uint32_t tm_strip = h->tmem_base + ((uint32_t)(warp & 3) * 32u << 16) + (uint32_t)(warp >> 2) * (uint32_t)kTmWarpCols;

  for (;;) {
    // ---- next system of the queue (rank 0 pulls, everyone reads it through DSMEM) --------------
    if (rank == 0 && tid == 0) h->next_sys = atomicAdd(P.cl_counter + kClass, 1);
    cluster.sync();
    const int qi = ld_cluster_s32(mapa_u32(smem_u32(&h->next_sys), 0));
    if (qi >= P.cl_cnt[kClass]) {   // uniform over the cluster
      cluster.sync();          // rank 0's shared memory must outlive everybody's read of next_sys
      break;
    }
    const int s = P.cl_order[P.cl_off[kClass] + qi];
    if (P.sc.done[s]) { cluster.sync(); continue; }   // empty / zero-load systems (init_scalars)
#ifdef FEA_CLUSTER_ACCOUNT
    const long long acc_t1 = clock64();
#endif
#ifdef FEA_CLUSTER_TRACE
    const unsigned long long tr_t0 = gtime();
#endif

    // ---- geometry of the system inside the cluster ----------------------------------------------
    const int64_t row0 = (int64_t)P.cta_first[s] * kCtaRows;       // first block row of the system
    const int n_sl = P.cta_count[s] * (kCtaRows / 32);             // 32-row slices of the system
    const int Sc = (n_sl + kCl - 1) / kCl;                         // slices per CTA (<= kClSlices)
    const int Rc = Sc * 32;                                        // rows per CTA
    const int my_sl = max(0, min(Sc, n_sl - rank * Sc));           // slices this CTA owns
    const int64_t my_row0 = row0 + (int64_t)rank * Rc;

    // ---- halo: which rows of other CTAs do my rows gather? ----------------------------------------
    // One bit per row of the system (word w = slice w of the system).  The marked rows, in row
    // order, become halo slots Rc, Rc+1, ... of this CTA's p buffer; their owners get a send list.
    uint32_t* bmp = reinterpret_cast<uint32_t*>(smem + kClSmemBytes - kClTmpBytes);
    int32_t* pre = reinterpret_cast<int32_t*>(bmp) + kClWords;     // [kClWords + 1] exclusive prefix of popc
    if (tid < kClSlices) {
      h->s_len[tid] = tid < my_sl ? P.slice_len[(my_row0 >> 5) + tid] : 0;
      h->s_base[tid] = tid < my_sl ? P.slice_ptr[(my_row0 >> 5) + tid] : 0;
    }
#pragma unroll
    for (int i = 0; i < kClWpt; ++i) bmp[tid * kClWpt + i] = 0;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kClRpt; ++k) {
      const int ls = warp + kClW * k;        // local slice handled by this warp
      if (ls >= my_sl) continue;
      const int L = h->s_len[ls];
      const int64_t base = h->s_base[ls];
      for (int j = 0; j < L; ++j) {
        const int c = ld_stream_i32(P.col + base + j * 32 + lane) - (int)row0;   // row inside the system
        if (c / Rc != rank) atomicOr(&bmp[c >> 5], 1u << (c & 31));
      }
    }
    __syncthreads();
    int H;                                   // halo rows of this CTA
    {
      int mine = 0;                          // marked rows in this thread's words
#pragma unroll
      for (int i = 0; i < kClWpt; ++i) mine += __popc(bmp[tid * kClWpt + i]);
      int incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (lane == 31) h->wsum[warp] = incl;
      __syncthreads();
      int woff = 0;
      H = 0;
#pragma unroll
      for (int w = 0; w < kClW; ++w) {
        const int t = h->wsum[w];
        woff += w < warp ? t : 0;
        H += t;
      }
      int run = woff + incl - mine;
#pragma unroll
      for (int i = 0; i < kClWpt; ++i) {
        pre[tid * kClWpt + i] = run;
        run += __popc(bmp[tid * kClWpt + i]);
      }
      if (tid == 0) pre[kClWords] = H;
      __syncthreads();
    }
    if (tid < kCl)   // tell every owner how many of its rows I gather (0 for myself)
      st_cluster_s32(mapa_u32(smem_u32(&h->send_from[rank]), tid),
                     pre[min((tid + 1) * Sc, kClWords)] - pre[min(tid * Sc, kClWords)]);
    cluster.sync();                                                // #1: send_from[] complete

    // ---- layout of the shared memory (depends on the halo and send-list sizes) -------------------
    //   header | send list [n_send] u32 | p: own rows [Rc] + halo [H] double2 |
    //   gather codes of all owned slices (u16 index into p) | 2x2 blocks of the resident slices
    if (tid < kCl) {
      int off = 0;
      for (int c = 0; c < rank; ++c) off += ld_cluster_s32(mapa_u32(smem_u32(&h->send_from[c]), tid));
      h->seg_off[tid] = off;
    }
    if (tid == 0) {
      int S = 0;
      for (int c = 0; c < kCl; ++c) S += h->send_from[c];
      h->n_send = S;
      int ent = 0;
      for (int i = 0; i < kClSlices; ++i) { h->s_aoff[i] = ent; ent += (h->s_len[i] + 3) / 4 * 128; }
      const int off_pbuf = kHdr + (4 * S + 127) / 128 * 128;
      const int mat0 = (off_pbuf + 16 * (Rc + H) + 127) / 128 * 128;
      int off = (ent * 2 + 127) / 128 * 128;
      const int fit = (mat0 + off <= kClSmemBytes - kClTmpBytes && Rc + H <= 0xffff && H <= P.cl_halo_cap) ? 1 : 0;
      h->off_pbuf = off_pbuf;
      h->mat0 = mat0;
      // resident slices: the first slices (round k = 0 of every warp) are resident.  (Measured against
      // giving whole warps resident slices, 48.5 ms, and a warp/round checkerboard, 49.9 ms: 47.2 ms.)
      // tensor memory first: every warp fills its strip with the leading blocks of its slices (slice i belongs to
      // warp i % kClW); what is left of a slice goes to shared memory while there is room, else it is streamed
      const int cap = kClSmemBytes - mat0;
      for (int w = 0; w < kClW; ++w) h->wsum[w] = 0;    // blocks per lane already placed in warp w's strip
      for (int i = 0; i < kClSlices; ++i) {
        // a slice that fits takes its blocks in pairs (an odd row length is padded with a zero block); a slice
        // that does not fit is split at a multiple of four blocks, the granularity of the gather codes
        const int L = h->s_len[i], used = h->wsum[i % kClW], rem = kTmWarpBlocks - used, Le = (L + 1) & ~1;
        const int nt = i >= my_sl ? 0 : (Le <= rem ? Le : (rem & ~3));
        h->s_nt[i] = nt;
        h->s_tcol[i] = used * 8;
        h->wsum[i % kClW] = used + nt;
        const int bytes = max(L - nt, 0) * 32 * 32;
        if (i < my_sl && off + bytes <= cap) { h->s_off[i] = off; off += bytes; }
        else h->s_off[i] = -1;
      }
      for (int c = 0; c < kCl; ++c) st_cluster_s32(mapa_u32(smem_u32(&h->fit[rank]), c), fit);
    }
    cluster.sync();                                                // #2: fit[] complete, layout visible
    {
      bool ok = true;
#pragma unroll
      for (int c = 0; c < kCl; ++c) ok = ok && h->fit[c] != 0;
      if (!ok) {   // (uniform) halo too large for the shared memory: left to the streaming kernels
        if (rank == 0 && tid == 0) atomicAdd(P.cl_counter + 10, 1);
        continue;
      }
    }
    const int off_pbuf = h->off_pbuf, mat0 = h->mat0;
    double2* pbuf = reinterpret_cast<double2*>(smem + off_pbuf);   // [Rc] published p + [H] halo
    const uint32_t pbuf_a = smem_u32(pbuf);
    uint16_t* sa_all = reinterpret_cast<uint16_t*>(smem + mat0);
    const uint32_t* sendl = reinterpret_cast<const uint32_t*>(smem + kHdr);

    // ---- gather codes: index into p (own row, or halo slot of a row owned by another CTA) --------
#pragma unroll
    for (int k = 0; k < kClRpt; ++k) {
      const int ls = warp + kClW * k;
      if (ls >= my_sl) continue;
      const int L = h->s_len[ls];
      const int64_t base = h->s_base[ls];
      uint16_t* sa = sa_all + h->s_aoff[ls];
      bool remote = false;
      for (int j = 0; j < L; ++j) {
        const int c = ld_stream_i32(P.col + base + j * 32 + lane) - (int)row0;
        const int cr = c / Rc;
        const int code = cr == rank ? c - cr * Rc
                                    : Rc + pre[c >> 5] + __popc(bmp[c >> 5] & ((1u << (c & 31)) - 1u));
        remote = remote || cr != rank;
        sa[((j >> 2) * 32 + lane) * 4 + (j & 3)] = (uint16_t)code;   // one 8-byte load fetches 4 codes of a lane
      }
      for (int j = L; j < (L + 3) / 4 * 4; ++j)                      // tail of the last group: the own row
        sa[((j >> 2) * 32 + lane) * 4 + (j & 3)] = (uint16_t)(ls * 32 + lane);
      remote = __any_sync(0xffffffffu, remote);
      if (lane == 0) h->s_halo[ls] = remote ? 1 : 0;
    }
    // ---- send lists: one entry per halo row, written into its owner's list -----------------------
    // entry = row inside the owner (12 bits) | consumer rank (3 bits) | consumer's p slot (>> 4 of
    // the byte offset in ITS shared memory: the layouts of the CTAs differ)
#pragma unroll
    for (int i = 0; i < kClWpt; ++i) {
      const int wd = tid * kClWpt + i;
      uint32_t bits = bmp[wd];
      if (bits) {
        const int o = wd / Sc;
        int slot = pre[wd];
        int pos = h->seg_off[o] + slot - pre[min(o * Sc, kClWords)];
        const int lr0 = (wd - o * Sc) * 32;
        const uint32_t dst = mapa_u32(smem_a + kHdr, o);
        while (bits) {
          const int b = __ffs(bits) - 1;
          bits &= bits - 1;
          const uint32_t e = (uint32_t)(lr0 + b) | ((uint32_t)rank << 12) | ((uint32_t)(off_pbuf / 16 + Rc + slot) << 15);
          st_cluster_s32(dst + 4u * (uint32_t)pos, (int)e);
          ++slot;
          ++pos;
        }
      }
    }
    cluster.sync();                                                // #3: send lists complete; bitmap dead
    const int n_send = h->n_send;

    // ---- 2x2 blocks of the resident slices --------------------------------------------------------
#pragma unroll
    for (int k = 0; k < kClRpt; ++k) {
      const int ls = warp + kClW * k;
      if (ls >= my_sl) continue;
      const int off = h->s_off[ls];
      const int L = h->s_len[ls], nt = h->s_nt[ls];
      const int64_t base = h->s_base[ls];
      const uint32_t tcol = tm_strip + (uint32_t)h->s_tcol[ls];
      for (int j = 0; j < nt; ++j) {                 // leading blocks: this lane's strip of tensor memory
        d4 blk;
        blk.x = blk.y = blk.z = blk.w = 0.0;         // (the pad block of an odd row length)
        if (j < L) blk = ld_stream_d4(P.val + base + j * 32 + lane);
        tmem_st_block(tcol + 8u * (uint32_t)j, blk);
      }
      if (off < 0 || nt >= L) continue;
      // values per slice: (L - nt) x 32 top halves (k00,k01) then (L - nt) x 32 bottom halves (k10,k11)
      // (16-byte lane stride: conflict-free 128-bit shared loads)
      double2* st = reinterpret_cast<double2*>(smem + mat0 + off);
      double2* sb = st + (L - nt) * 32;
      for (int j = nt; j < L; ++j) {
        const d4 blk = ld_stream_d4(P.val + base + j * 32 + lane);
        st[(j - nt) * 32 + lane] = make_double2(blk.x, blk.y);
        sb[(j - nt) * 32 + lane] = make_double2(blk.z, blk.w);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");

    // ---- vectors of the thread's rows in registers ----------------------------------------------
    double2 x[kClRpt], r[kClRpt];   // p lives in pbuf (its owner is the only writer)
    bool own[kClRpt];
#pragma unroll
    for (int k = 0; k < kClRpt; ++k) {
      const int lr = tid + kClT * k;
      own[k] = lr < my_sl * 32;
      x[k] = make_double2(0.0, 0.0);
      r[k] = x[k];
      if (own[k]) {
        const d4 rec = P.rp[my_row0 + lr];   // r0 = S b (k_pcg_init_vectors)
        r[k] = make_double2(rec.x, rec.y);
        pbuf[lr] = r[k];                     // first direction p = r
      }
    }
#ifdef FEA_CLUSTER_PROFILE
    const bool prof = rank == 0 && tid == 0;
    if (prof) {
      for (int i = 0; i < 9; ++i) h->prof[i] = 0;
      h->prof[9] = clock64();
    }
#endif
    double rz = P.sc.rz[0][s];
    if (tid == 0) {                           // loop constants that are needed once per iteration live in
      h->tol2 = P.sc.tol2[s];                 // shared memory: registers are the scarce resource here
      h->it_limit = P.max_iter;
      h->rz_monitor = inf;                    // smallest true r.r found by a monitor pass
      h->mon_strikes = 0;
    }
    __syncthreads();
    int iters = 0, status = FEA_SAMPLE_NOT_RUN;
#ifdef FEA_CLUSTER_ACCOUNT
    const long long acc_t2 = clock64();
#endif
    bool monitored = false;                   // the monitor pass of the current iteration count is done
    bool gap = false;                         // the recursive residual converged, the TRUE one did not (fp64 floor)
    int refine_round = 0;                     // extended-precision rounds done; > 0: the solution is (P.x, P.xlo)
    double rz_round = inf;                    // true r.r at the start of the current refinement round

    for (;;) {   // ---- refinement rounds: one pass for all but the ill-conditioned systems ----------------
    // CG with ONE hand-over per iteration.  After q = Khat p every warp pushes the record
    //   (p.q, q.q, r.q, r.r)  of its rows; with the four sums every thread knows
    //   alpha      = r.r / p.q
    //   |r_new|^2  = r.r - 2 alpha r.q + alpha^2 q.q      (r_new = r - alpha q, expanded)
    //   beta       = |r_new|^2 / r.r
    // before touching a vector, so x, r AND the next direction p = r_new + beta p are updated in one
    // pass.  r.r in the record is the exact norm of the current residual (nothing is accumulated from
    // iteration to iteration; the expansion only serves beta, where a relative error of
    // eps r.r / |r_new|^2 tilts the next direction by that much), and it is what convergence is
    // decided on -- one SpMV later than in the textbook loop (+1 SpMV per solve).
    //
    // mode 0 = iteration; mode 1 / 2 = "check" / "monitor": the published vector is x and the TRUE
    // residual S b - Khat x is measured (the recursion r -= alpha q drifts from it by rounding).  A
    // converged system is checked once; a material gap goes to the extended-precision rounds below.
    // The monitor pass runs every kMonitor iterations (2 kMonitor for the 5..8-CTA classes, whose
    // convergence curves have longer plateaus): p is parked in the global q rows meanwhile and CG
    // continues undisturbed; a system whose TRUE residual does not fall any more is not going to
    // converge (singular or inconsistent: a mechanism the classifier missed, F4) and is stopped as
    // STAGNATED instead of holding its cluster for max_iter iterations.
    int mode = 0;
    for (;;) {
      PROF_T(0);
      // S1: the CTA's published vector is complete (bar.sync) and its boundary rows are pushed into the
      // halo slots of the CTAs that gather them.  A warp waits for this CTA's own halo only when it reaches
      // a slice that gathers from it (the few slices along the CTA's borders) or at the end of its
      // SpMV: the flight time of the pushes is hidden behind the interior slices.
      __syncthreads();
      for (int i = tid; i < n_send; i += kClT) {
        const uint32_t e = sendl[i];
        const double2 v = pbuf[e & 0xfffu];
        const uint32_t base = mapa_u32(smem_a, (e >> 12) & 7u);
        asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(
                         base + 16u * (e >> 15)),
                     "d"(v.x), "d"(v.y), "r"(base + (uint32_t)offsetof(ClHeader, mbarP))
                     : "memory");
      }
      if (tid == 0) mbar_arm(smem_u32(&h->mbarP), 16u * (uint32_t)H);
      bool halo_here = false;
      PROF_T(1);
      double2 q[kClRpt];
#pragma unroll
      for (int k = 0; k < kClRpt; ++k) {
        const int ls = warp + kClW * k;
        double a0 = 0.0, a1 = 0.0;
        if (ls < my_sl) {
          const double2 pk = pbuf[tid + kClT * k];   // the diagonal block of Khat is the identity
          a0 = pk.x;
          a1 = pk.y;
          const int L = h->s_len[ls];
          const int off = h->s_off[ls];
          const uint2* sa = reinterpret_cast<const uint2*>(sa_all + h->s_aoff[ls]) + lane;   // 4 codes per load
          const uint32_t self = (uint32_t)(tid + kClT * k);
          if (!halo_here && h->s_halo[ls]) {
            mbar_wait(smem_u32(&h->mbarP), (phase >> 2) & 1u);
            halo_here = true;
          }
          const int nt = h->s_nt[ls];
          if (nt > 0) {   // leading blocks from tensor memory: their own datapath, not the L1TEX pipe
            const uint32_t tcol = tm_strip + (uint32_t)h->s_tcol[ls];
            d4 kv[4];
            double2 pj[4];
            int j = 0;
            // (the block loops of the three storage tiers are NOT unrolled: ptxas' own unrolling by two costs spills
            // and code -- 11 168 instead of 8 632 instructions per kernel -- and measured 27.7 against 26.4 ms per
            // 400-system batch; the (up to 4) slices of a warp stay unrolled, their products live in registers)
#pragma unroll 1
            for (; j + 4 <= nt; j += 4) {
              const uint2 cc = sa[(j >> 2) * 32];
              const uint32_t ga[4] = {pbuf_a + 16u * (cc.x & 0xffffu), pbuf_a + 16u * (cc.x >> 16), pbuf_a + 16u * (cc.y & 0xffffu), pbuf_a + 16u * (cc.y >> 16)};
              tmem_ld4_gather4(tcol + 8u * (uint32_t)j, ga, kv, pj);
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                a0 = fma(kv[u].x, pj[u].x, a0); a0 = fma(kv[u].y, pj[u].y, a0);
                a1 = fma(kv[u].z, pj[u].x, a1); a1 = fma(kv[u].w, pj[u].y, a1);
              }
            }
            if (j < nt) {   // a last pair
              const uint32_t cx = reinterpret_cast<const uint32_t*>(sa + (j >> 2) * 32)[0];
              tmem_ld2_gather2(tcol + 8u * (uint32_t)j, pbuf_a + 16u * (cx & 0xffffu), pbuf_a + 16u * (cx >> 16), kv, pj);
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                a0 = fma(kv[u].x, pj[u].x, a0); a0 = fma(kv[u].y, pj[u].y, a0);
                a1 = fma(kv[u].z, pj[u].x, a1); a1 = fma(kv[u].w, pj[u].y, a1);
              }
            }
          }
          // the other blocks [nt, L) of a split slice (nt is a multiple of four there)
          if (nt >= L) {
          } else if (off >= 0) {
            const double2* st = reinterpret_cast<const double2*>(smem + mat0 + off) + lane - nt * 32;
            const double2* sb = st + (L - nt) * 32;
#pragma unroll 1
            for (int j = nt; j < L; j += kClU) {   // kClU gathers in flight; the tail round is predicated
              uint32_t g[kClU];
              double2 pj[kClU];
#pragma unroll
              for (int u = 0; u < kClU; u += 4) {
                const uint2 cc = (u == 0 || j + u < L) ? sa[((j + u) >> 2) * 32] : make_uint2(self | (self << 16), self | (self << 16));
                g[u] = cc.x & 0xffffu; g[u + 1] = cc.x >> 16; g[u + 2] = cc.y & 0xffffu; g[u + 3] = cc.y >> 16;
              }
#pragma unroll
              for (int u = 0; u < kClU; ++u) pj[u] = ld_shared_f64x2(pbuf_a + 16u * g[u]);
#pragma unroll
              for (int u = 0; u < kClU; ++u) {
                if (j + u < L) {
                  const double2 kt = st[(j + u) * 32], kb = sb[(j + u) * 32];
                  a0 = fma(kt.x, pj[u].x, a0); a0 = fma(kt.y, pj[u].y, a0);
                  a1 = fma(kb.x, pj[u].x, a1); a1 = fma(kb.y, pj[u].y, a1);
                }
              }
            }
          } else {  // blocks that fit neither: streamed from global memory (L2 resident), 4 in flight
            const d4* vt = P.val + h->s_base[ls] + lane;
#pragma unroll 1
            for (int j = nt; j < L; j += kClUs) {
              d4 kv[kClUs];
#pragma unroll
              for (int u = 0; u < kClUs; ++u) {
                kv[u].x = kv[u].y = kv[u].z = kv[u].w = 0.0;
                if (j + u < L) kv[u] = ld_stream_d4(vt + (j + u) * 32);
              }
              uint32_t g[kClUs];
              double2 pj[kClUs];
#pragma unroll
              for (int u = 0; u < kClUs; u += 4) {
                const uint2 cc = (u == 0 || j + u < L) ? sa[((j + u) >> 2) * 32] : make_uint2(self | (self << 16), self | (self << 16));
                g[u] = cc.x & 0xffffu; g[u + 1] = cc.x >> 16; g[u + 2] = cc.y & 0xffffu; g[u + 3] = cc.y >> 16;
              }
#pragma unroll
              for (int u = 0; u < kClUs; ++u) pj[u] = ld_shared_f64x2(pbuf_a + 16u * g[u]);
#pragma unroll
              for (int u = 0; u < kClUs; ++u) {
                a0 = fma(kv[u].x, pj[u].x, a0); a0 = fma(kv[u].y, pj[u].y, a0);
                a1 = fma(kv[u].z, pj[u].x, a1); a1 = fma(kv[u].w, pj[u].y, a1);
              }
            }
          }
        }
        q[k] = make_double2(a0, a1);
      }
      if (!halo_here) mbar_wait(smem_u32(&h->mbarP), (phase >> 2) & 1u);   // every thread consumes every phase
      phase ^= 4u;
      if (mode == 0) {
        double s_pq = 0.0, s_qq = 0.0, s_rq = 0.0, s_rr = 0.0;
        double2 pown[kClRpt];   // this thread's rows of p: read once for the record, kept for the update
#pragma unroll
        for (int k = 0; k < kClRpt; ++k) {
          pown[k] = make_double2(0.0, 0.0);
          if (own[k]) {
            const double2 pk = pbuf[tid + kClT * k];
            pown[k] = pk;
            s_pq = fma(pk.x, q[k].x, fma(pk.y, q[k].y, s_pq));
            s_qq = fma(q[k].x, q[k].x, fma(q[k].y, q[k].y, s_qq));
            s_rq = fma(r[k].x, q[k].x, fma(r[k].y, q[k].y, s_rq));
            s_rr = fma(r[k].x, r[k].x, fma(r[k].y, r[k].y, s_rr));
          }
        }
        s_pq = warp_sum(s_pq); s_qq = warp_sum(s_qq); s_rq = warp_sum(s_rq); s_rr = warp_sum(s_rr);
        const int ab = iters & 1;
        push_record<CL>(h, ab, rank, warp, lane, s_pq, s_qq, s_rq, s_rr);
        PROF_T(2);
        await_tx(&h->mbarA[ab], 32u * CL * kClW, (phase >> (ab ? 3 : 0)) & 1u, tid);   // S2: the records have landed
        phase ^= ab ? 8u : 1u;
        PROF_T(3);
        double pq, qq, rq;
        sum_records<CL>(h->partA[ab], lane, pq, qq, rq, rz);     // rz = r.r of the current residual, exact
        const double ipq = 1.0 / pq;                             // (started before the exit tests: it is the longest
                                                                 //  scalar dependency of the iteration)
        PROF_T(4);
        bool check = false, monitor = false;
#ifdef FEA_CLUSTER_DEBUG
        if ((iters & 127) == 0 || (iters > 1020 && iters < 1030)) DBG("[cl] sys %d it %d rr/rr0 %.3e pq %.3e qq %.3e rq %.3e\n", s, iters, rz / P.sc.rz0[s], pq, qq, rq);
#endif
        if (!isfinite(rz)) { status = FEA_SAMPLE_BREAKDOWN; break; }
        if (rz <= *(volatile double*)&h->tol2) {
          status = FEA_SAMPLE_CONVERGED;
          if (iters == 0) break;
          check = true;
        } else if (iters >= *(volatile int32_t*)&h->it_limit) {
          status = FEA_SAMPLE_MAX_ITER;
          break;
        } else if (!monitored && iters > 0 && (iters & ((CL > 4 ? 2 * kMonitor : kMonitor) - 1)) == 0) {
          check = monitor = monitored = true;
        }
        if (check) {   // publish x instead of p (q of this round is dropped: one SpMV per pass)
#pragma unroll
          for (int k = 0; k < kClRpt; ++k) {
            if (own[k]) {
              if (monitor) P.q[my_row0 + tid + kClT * k] = pbuf[tid + kClT * k];
              pbuf[tid + kClT * k] = x[k];
            }
          }
          mode = monitor ? 2 : 1;
          continue;
        }
        if (!(pq > 0.0 && isfinite(pq))) { status = FEA_SAMPLE_BREAKDOWN; break; }
        // one division (fp64 division is ~150 cycles of dependent instructions that every warp repeats):
        //   alpha = rz / pq;  beta = |r - alpha q|^2 / rz = 1 + (rz qq / pq - 2 rq) / pq
        const double alpha = rz * ipq;
        const double b1 = fma(fma(rz * qq, ipq, -2.0 * rq), ipq, 1.0);
        const double beta = b1 > 0.0 ? b1 : 0.0;
#pragma unroll
        for (int k = 0; k < kClRpt; ++k) {
          if (own[k]) {
            double2 pk = pown[k];
            x[k].x = fma(alpha, pk.x, x[k].x);
            x[k].y = fma(alpha, pk.y, x[k].y);
            r[k].x = fma(-alpha, q[k].x, r[k].x);
            r[k].y = fma(-alpha, q[k].y, r[k].y);
            pk.x = fma(beta, pk.x, r[k].x);
            pk.y = fma(beta, pk.y, r[k].y);
            pbuf[tid + kClT * k] = pk;
          }
        }
        ++iters;
        monitored = false;
        PROF_T(5);
        continue;
      }
      // ---- check / monitor: q = Khat x; the TRUE residual S b - q is only measured, never put into the
      // recursion: once CG runs below the fp64 floor of the true residual (eps |K| |x|, see the
      // extended-precision rounds) a replaced r is orders of magnitude larger than the direction it is
      // combined with, and the iteration blows up (observed on the ill-conditioned bench plate)
      double part = 0.0;
#pragma unroll
      for (int k = 0; k < kClRpt; ++k) {
        if (own[k]) {
          const d4 rec = P.rp[my_row0 + tid + kClT * k];      // S b (the correction's right-hand side in a refinement round)
          const double t0 = rec.x - q[k].x, t1 = rec.y - q[k].y;
          part += fma(t0, t0, t1 * t1);
        }
      }
      part = warp_sum(part);
      push_partial<CL>(h, (uint32_t)offsetof(ClHeader, partB), (uint32_t)offsetof(ClHeader, mbarB), rank, warp, lane, part);
      await_tx(&h->mbarB, 8u * CL * kClW, (phase >> 1) & 1u, tid);  // S3: r.r partials have landed
      phase ^= 2u;
      const double rz_new = sum_table<CL>(h->partB, lane);
      if (mode == 1) rz = rz_new;                               // what relres reports: the TRUE residual
      DBG("[cl] sys %d it %d mode %d true rr/rr0 %.3e (tol2/rr0 %.3e)\n", s, iters, mode, rz_new / P.sc.rz0[s], h->tol2 / P.sc.rz0[s]);
      if (mode == 2) {
        // every gather of x is done (S3; the halo copies are refreshed by the next push): put p back
        // and continue CG undisturbed
#pragma unroll
        for (int k = 0; k < kClRpt; ++k)
          if (own[k]) pbuf[tid + kClT * k] = P.q[my_row0 + tid + kClT * k];
        // no progress = the true |r| has not even halved against the best value any pass has seen, for two
        // passes in a row (a slowly converging but well-posed system -- kappa ~ 1e7 -- gains about that much
        // per interval, and CG residuals are not monotone)
        const bool gained = rz_new < 0.25 * h->rz_monitor;
        const bool stuck = !gained && h->mon_strikes >= 1;
        __syncthreads();
        if (tid == 0) {
          h->mon_strikes = gained ? 0 : h->mon_strikes + 1;
          h->rz_monitor = fmin(h->rz_monitor, rz_new);
        }
        if (stuck || !isfinite(rz_new)) {
          status = FEA_SAMPLE_STAGNATED;
          rz = rz_new;
          break;
        }
        mode = 0;
        continue;
      }
      {
        const double tol2 = *(volatile double*)&h->tol2;
        if (!(rz_new > 100.0 * tol2 && isfinite(rz_new))) {     // true residual within 10x the tolerance
          if (isfinite(rz_new)) status = FEA_SAMPLE_CONVERGED;
          break;
        }
        // the recursion says converged, b - K x says no: the fp64 floor of this system is above the
        // tolerance.  Left to an extended-precision round (below) -- or reported, if those are off.
        gap = true;
        status = FEA_SAMPLE_STAGNATED;
        break;
      }
    }

      // ---- extended-precision round (see dd_residual_rows) --------------------------------------
      // entered when fp64 CG hit its floor (gap), and after every correction solve to fold the
      // correction in and verify the sum against its double-double residual
      // (a correction whose solve was stopped by the monitor or ran out of iterations is dropped)
      if (!(P.refine_dd && ((gap && refine_round == 0) || (refine_round > 0 && (gap || status == FEA_SAMPLE_CONVERGED)))))
        break;
      dd_fold_rows(P, my_row0, my_sl * 32, tid, x, refine_round == 0);
      __threadfence();
      cluster.sync();                                            // every CTA's part of xhi + xlo is visible
      {
        double part = warp_sum(dd_residual_rows(Pp, my_row0, my_sl * 32, tid));
        push_partial<CL>(h, (uint32_t)offsetof(ClHeader, partB), (uint32_t)offsetof(ClHeader, mbarB), rank, warp, lane, part);
        await_tx(&h->mbarB, 8u * CL * kClW, (phase >> 1) & 1u, tid);
        phase ^= 2u;
        rz = sum_table<CL>(h->partB, lane);                      // TRUE r.r of xhi + xlo, to ~1e-30
      }
      const double tol2_ref = kRefineTighten * P.sc.tol2[s];
      DBG("[cl] sys %d it %d round %d status %d dd rr/rr0 %.3e\n", s, iters, refine_round, status, rz / P.sc.rz0[s]);
      if (rz <= tol2_ref) { status = FEA_SAMPLE_CONVERGED; break; }
      if (refine_round >= kMaxRefine || !(rz < 0.25 * rz_round) || !isfinite(rz)) { status = FEA_SAMPLE_STAGNATED; break; }
      // correction solve: Khat d = r, from d = 0, to the (absolute) refined tolerance
      rz_round = rz;
      ++refine_round;
      if (rank == 0 && tid == 0) atomicAdd(P.cl_counter, 1);
#pragma unroll
      for (int k = 0; k < kClRpt; ++k) {
        x[k] = make_double2(0.0, 0.0);
        r[k] = x[k];
        if (own[k]) {
          const d4 rec = P.rp[my_row0 + tid + kClT * k];
          r[k] = make_double2(rec.x, rec.y);
          pbuf[tid + kClT * k] = r[k];                           // first direction p = r
        }
      }
      status = FEA_SAMPLE_NOT_RUN;
      gap = false;
      monitored = false;
      __syncthreads();                                           // everybody has read the old constants
      if (tid == 0) {
        h->tol2 = tol2_ref;
        h->it_limit = P.max_iter;
        h->rz_monitor = inf;
        h->mon_strikes = 0;
      }
      __syncthreads();
    }

    // ---- results ------------------------------------------------------------------------------
    if (refine_round == 0 && !(P.refine_dd && gap)) {            // otherwise P.x already holds the high part of the sum
#pragma unroll
      for (int k = 0; k < kClRpt; ++k)
        if (own[k]) P.x[my_row0 + tid + kClT * k] = x[k];
    }
#ifdef FEA_CLUSTER_PROFILE
    if (prof) {
      for (int i = 0; i < 8; ++i) atomicAdd(&g_cl_prof[i], (unsigned long long)h->prof[i]);
      atomicAdd(&g_cl_prof[8], (unsigned long long)iters);
    }
#endif
#ifdef FEA_CLUSTER_ACCOUNT
    if (tid == 0) {
      const long long t3 = clock64();
      atomicAdd(&g_cl_prof[10], (unsigned long long)(acc_t2 - acc_t1));
      atomicAdd(&g_cl_prof[11], (unsigned long long)(t3 - acc_t2));
      if (rank == 0) atomicAdd(&g_cl_prof[12], 1ull);
      if (rank == 0) atomicAdd(&g_cl_prof[14], (unsigned long long)iters * CL);
    }
#endif
    if (tid == 0) {   // where this CTA read its blocks from (bench: bytes through the shared-memory pipe / TMEM / L2)
      long long nb[3] = {0, 0, 0};
      for (int i = 0; i < my_sl; ++i) {
        const int L = h->s_len[i], nt = min(h->s_nt[i], L);
        nb[0] += 32 * nt;
        nb[h->s_off[i] >= 0 ? 1 : 2] += 32 * (L - nt);
      }
      unsigned long long* cnt = reinterpret_cast<unsigned long long*>(P.cl_counter + 16);
      for (int i = 0; i < 3; ++i)
        if (nb[i]) atomicAdd(cnt + i, (unsigned long long)(nb[i] * (long long)(iters + 1 + refine_round)));
    }
#ifdef FEA_CLUSTER_TRACE
    if (rank == 0 && tid == 0 && s < 8192) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      g_cl_trace[s][0] = tr_t0;
      g_cl_trace[s][1] = gtime();
      g_cl_trace[s][2] = ((unsigned long long)CL << 32) | smid;
      g_cl_trace[s][3] = (unsigned long long)iters;
    }
#endif
    if (rank == 0 && tid == 0) {
      P.sc.iters[s] = iters;
      P.sc.status[s] = status;
      P.sc.cap[s] = -1;     // verified against the true residual on chip: skip the streaming check
      P.sc.rounds[s] = refine_round;
      P.sc.done[s] = 1;
      P.rz_last[s] = rz;
      atomicAdd(P.sc.n_done, 1);
    }
  }
#ifdef FEA_CLUSTER_ACCOUNT
  if (tid == 0) atomicAdd(&g_cl_prof[13], (unsigned long long)(clock64() - acc_t0));
#endif
  // every CTA must give its tensor memory back: the next CTA on this SM allocates all of it
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(h->tmem_base), "n"(kTmCols) : "memory");
}

typedef void (*cluster_fn)(const PcgPtrs*);
static cluster_fn cluster_kernel(int cl) {
  switch (cl) {
    case 1: return k_pcg_cluster<1>;
    case 2: return k_pcg_cluster<2>;
    case 3: return k_pcg_cluster<3>;
    case 4: return k_pcg_cluster<4>;
    case 5: return k_pcg_cluster<5>;
    case 6: return k_pcg_cluster<6>;
    case 7: return k_pcg_cluster<7>;
    default: return k_pcg_cluster<8>;
  }
}

static void cluster_config(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* at, int cl, int nclusters, cudaStream_t st) {
  *cfg = cudaLaunchConfig_t{};
  cfg->gridDim = dim3(cl * nclusters);
  cfg->blockDim = dim3(kClT);
  cfg->dynamicSmemBytes = kClSmemBytes;
  cfg->stream = st;
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cl;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg->attrs = at;
  cfg->numAttrs = 1;
}

// Co-resident clusters of `cl` CTAs (0 = path unavailable on this device).  The occupancy API accounts for the
// GPC structure (B200: 74 / 45 / 33 clusters of 2 / 3 / 4 CTAs, i.e. 148 / 135 / 132 SMs -- the same numbers a probe
// kernel that timestamps its clusters' arrivals measures), so a persistent grid of this size has no pending CTAs.
int pcg_cluster_capacity(Ctx& c, int cl) {
  const int slot = cl;
  if (c.cluster_capacity[slot] >= 0) return c.cluster_capacity[slot];
  c.cluster_capacity[slot] = 0;
  if (cudaFuncSetAttribute(cluster_kernel(cl), cudaFuncAttributeMaxDynamicSharedMemorySize, kClSmemBytes) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute at[1];
  cluster_config(&cfg, at, cl, 256, nullptr);
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, cluster_kernel(cl), &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  c.cluster_capacity[slot] = n;
  return n;
}

#if defined(FEA_CLUSTER_TRACE) && !defined(FEA_CLUSTER_ACCOUNT)
#error "FEA_CLUSTER_TRACE needs FEA_CLUSTER_ACCOUNT (the dump hook)"
#endif
#if defined(FEA_CLUSTER_PROFILE) || defined(FEA_CLUSTER_ACCOUNT)
void pcg_cluster_profile_dump() {
#ifdef FEA_CLUSTER_TRACE
  if (const char* path = getenv("FEA_CLUSTER_TRACE_FILE")) {
    static unsigned long long tr[8192][4];
    cudaMemcpyFromSymbol(tr, g_cl_trace, sizeof(tr));
    if (FILE* f = fopen(path, "w")) {
      for (int i = 0; i < 8192; ++i)
        if (tr[i][1]) fprintf(f, "%d %llu %llu %llu %llu %llu\n", i, tr[i][0], tr[i][1], tr[i][2] >> 32, tr[i][2] & 0xffffffffull, tr[i][3]);
      fclose(f);
    }
    static unsigned long long zero[8192][4];
    cudaMemcpyToSymbol(g_cl_trace, zero, sizeof(zero));
  }
#endif
  unsigned long long h[16];
  cudaMemcpyFromSymbol(h, g_cl_prof, sizeof(h));
#ifdef FEA_CLUSTER_ACCOUNT
  fprintf(stderr, "[cluster account] systems %llu  set-up %.3f SM-Mcycles  iterating %.3f SM-Mcycles  CTA lifetime %.3f SM-Mcycles  "
                  "iterations x CTAs %llu  (cycles per iteration %.0f)\n",
          h[12], h[10] * 1e-6, h[11] * 1e-6, h[13] * 1e-6, h[14], h[14] ? (double)h[11] / (double)h[14] : 0.0);
#endif
  const char* names[8] = {"(loop back)", "bar.sync + halo push", "spmv + record push", "wait for records", "sum records", "update x r p", "-", "-"};
  const double it = (double)(h[8] ? h[8] : 1);
  for (int i = 0; i < 8; ++i) fprintf(stderr, "[cluster prof] %-20s %8.0f cycles/iter\n", names[i], h[i] / it);
  unsigned long long z[16] = {};
  cudaMemcpyToSymbol(g_cl_prof, z, sizeof(z));
}
#endif

// Cluster class of a system = CTAs per cluster, from its vertex count (an upper bound of its block
// rows): the smallest cluster (at least min_cl CTAs) whose CTAs hold the rows, 2048 per CTA.  Small
// clusters spend fewer SM-cycles in barriers per iteration and pack the GPU better; they stream a
// larger part of the matrix from L2.  0 = too large for 8 CTAs: streaming kernels.
int pcg_cluster_class(int64_t n_vertices_of_sample, int min_cl) {
  const int64_t pad = (n_vertices_of_sample + kCtaRows - 1) / kCtaRows * kCtaRows;
  if (pad <= 0) return 0;
  const int64_t rows_per_cta = (int64_t)kClSlices * 32;
  int64_t cl = (pad + rows_per_cta - 1) / rows_per_cta;
  if (cl < min_cl) cl = min_cl;
  return cl <= kClMax ? (int)cl : 0;
}

int pcg_cluster_rows_per_cta() { return kClSlices * 32; }

cudaError_t launch_pcg_cluster(Ctx& c, const PcgPtrs* dP, int n_systems, int cl, cudaStream_t st) {
  const int capn = pcg_cluster_capacity(c, cl);
  if (capn <= 0 || n_systems <= 0) return cudaSuccess;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute at[1];
  cluster_config(&cfg, at, cl, n_systems < capn ? n_systems : capn, st);
  return cudaLaunchKernelEx(&cfg, cluster_kernel(cl), dP);
}

}  // namespace fea
