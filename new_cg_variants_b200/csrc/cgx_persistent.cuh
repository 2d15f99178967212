// cgx_persistent.cuh -- latency-bound path: ONE cooperative launch runs every iteration,
// on one GPU or on every GPU of a row partition.
//
// Every matrix in predict_and_recompute/matrices (n <= 15 439) and the 64^3 Poisson tail are
// far below one GPU's worth of bandwidth work: with 2-4 launches per iteration the stream
// path is bounded by launch latency.  Here
//   * the grid (co-resident by cooperative launch) stays on the SMs for the whole solve;
//   * the STATE VECTORS LIVE IN SHARED MEMORY: CTA c owns the row chunks c, c+nb, c+2nb, ...
//     (T rows each) in both stages of an iteration, so x, r, r~, p, s, ... never leave the
//     SM; only the SpMV input (p | r~ | w~ | s~ [, r~]) is exported to global memory -- L2 --
//     for the neighbouring rows to read (double-buffered by iteration parity), and on a
//     partition its boundary planes go straight into the neighbours' ghost planes over NVLink;
//   * a sync point = one atomic arrive per CTA + a relaxed spin; the CTA that arrives last
//     adds the per-CTA partial dots in CTA order.  One GPU: every warp reads the partials
//     itself.  Partition: the last CTA stores the rank's record into every rank's window and
//     publishes the epoch; consumers add the records in rank order (bit-identical everywhere);
//   * alpha/beta and the other recurrences live in registers;
//   * the number of sync points per iteration is the variant's number of global
//     synchronisations: 3 for HS-CG, 2 for CG-CG / PR-CG / M-CG, ONE for GV-CG and the
//     pipe-PR family -- whose scalar exchange then travels while the SpMV stage runs
//     (the paper's communication-hiding claim, pipeprcg.c:154-173).
//
// The stage arithmetic is the stream path's ew_body / Op::row / sp_epilogue (called with
// an Args whose vector pointers address shared memory), so every per-row operation is
// identical; only the summation order of the dots differs, and stays deterministic.
//
// Ranks of a partition can also be emulated inside ONE cooperative launch (CTA range r*nb ..
// (r+1)*nb-1 acts as rank r): that is how the multi-GPU protocol of this kernel is tested on
// a single GPU without ever having two launches wait for each other.
#pragma once
#include <type_traits>

#include "cgx_kernels.cuh"

namespace cgx {

constexpr int kPersMaxGrid = 1024;
constexpr int kPersRed = 8;            // <= 4 recurrence sums + 4 instrumentation sums
constexpr int kPersMaxVec = 12;        // 10 state vectors + dinv + spare

struct PersOut { u64 epoch; u64 hepoch[kChan]; int err; int pad; };

template <class Op>
struct PersRank {
  Op A;
  Args g;                              // global pointers; g.d = this rank's Dist (world 1: unused)
  double* vecs[kPersMaxVec];           // global address of state vector v (cgx.cu V_* order), dinv at [10]
  double* exp_[2][2];                  // exported SpMV inputs [parity][rhs]
  u64* bar;                            // sync-point counter of this rank (zeroed by the host)
  double* part;                        // [2][nb][kPersRed]
  PersOut* out;
  u64 epoch0;
  u64 hepoch0[kChan];
};

struct PersLaunch {
  int k0, k1;                          // iterations k0 .. k1 (inclusive)
  int nb;                              // CTAs per rank
  int R;                               // row chunks per CTA
  unsigned vmask;                      // state vectors of the variant (bit v)
  int nslot;                           // shared-memory vector slots (popcount(vmask) [+1 for dinv])
  int slab_cap;                        // CSR: non-zeros of a CTA's rows kept in shared memory (0 = off; needs R == 1)
};

// A CTA's rows of a CSR matrix, resident in shared memory for the whole solve (values, columns,
// row offsets relative to the CTA's first non-zero).
struct CsrSlab { const double* val; const int* col; const int* ptr; };

__device__ __forceinline__ u64 ld_relaxed_gpu(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ u64 ld_relaxed_sys(const u64* p) {
  u64 v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// Bounded waits.  After the first time-out every later wait returns at once, so a lost
// peer costs one time-out, not one per iteration.
__device__ __forceinline__ void pers_wait_gpu(const u64* p, u64 target, int* err) {
  if (ld_relaxed_gpu(p) < target) {
    const u64 t0 = timer_ns();
    bool ok = false;
    while (!ok) {
#pragma unroll 1
      for (int spin = 0; spin < 64 && !ok; ++spin) ok = ld_relaxed_gpu(p) >= target;
      if (ok || *(volatile int*)err) break;
      if (timer_ns() - t0 > 10000000000ull) { atomicExch(err, 1); break; }
    }
  }
  fence_acq_rel_gpu();
}
__device__ __forceinline__ void pers_wait_sys(const u64* p, u64 target, int* err) {
  if (ld_relaxed_sys(p) < target) {
    const u64 t0 = timer_ns();
    bool ok = false;
    while (!ok) {
#pragma unroll 1
      for (int spin = 0; spin < 64 && !ok; ++spin) ok = ld_relaxed_sys(p) >= target;
      if (ok || *(volatile int*)err) break;
      if (timer_ns() - t0 > 10000000000ull) { atomicExch(err, 1); break; }
    }
  }
  fence_acq_rel_sys();
}

template <int VAR> struct PersPlan;      // stage kernels of each variant
template <> struct PersPlan<CGX_HS> { static constexpr int EW = EW_HS1, SP = SP_HS; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_CG> { static constexpr int EW = EW_CG, SP = SP_CG; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_GV> { static constexpr int EW = EW_GV, SP = SP_GV; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_PR> { static constexpr int EW = EW_PR, SP = SP_PR; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_M> { static constexpr int EW = EW_PR, SP = SP_PR; static constexpr bool MEUR = true; };
template <> struct PersPlan<CGX_PIPE_PR> { static constexpr int EW = EW_PIPE_R, SP = SP_PIPE_R; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_PIPE_PR_M> { static constexpr int EW = EW_PIPE_R, SP = SP_PIPE_R; static constexpr bool MEUR = true; };
template <> struct PersPlan<CGX_PIPE_P> { static constexpr int EW = EW_PIPE_N, SP = SP_PIPE_N; static constexpr bool MEUR = false; };
template <> struct PersPlan<CGX_PIPE_P_M> { static constexpr int EW = EW_PIPE_N, SP = SP_PIPE_N; static constexpr bool MEUR = true; };

// index (cgx.cu V_* order) of the state vector(s) the SpMV stage multiplies
template <int MODE> struct SpInV { static constexpr int v0 = 3, v1 = -1; };            // p
template <> struct SpInV<SP_CG> { static constexpr int v0 = 2, v1 = -1; };            // rt
template <> struct SpInV<SP_GV> { static constexpr int v0 = 7, v1 = -1; };            // wt
template <> struct SpInV<SP_PIPE_R> { static constexpr int v0 = 5, v1 = 2; };         // st, rt
template <> struct SpInV<SP_PIPE_N> { static constexpr int v0 = 5, v1 = -1; };        // st

__device__ __forceinline__ double*& args_vec(Args& g, int v) {
  switch (v) {
    case 0: return g.x; case 1: return g.r; case 2: return g.rt; case 3: return g.p; case 4: return g.s;
    case 5: return g.st; case 6: return g.w; case 7: return g.wt; case 8: return g.u; default: return g.t;
  }
}

// Row product inside the persistent kernel.  The stencil's neighbour pattern of a row does not
// change between iterations: it is decoded once (two integer divisions) into a 6-bit mask kept
// in shared memory; the sum keeps the canonical term order of StencilOp::row.
__device__ __forceinline__ unsigned stencil_mask(const StencilOp& A, int row) {
  const int plane = A.nx * A.ny;
  const int z = row / plane, rem = row - z * plane, yy = rem / A.nx, xx = rem - yy * A.nx;
  return (unsigned)((z > 0 || A.has_zlo) ? 1 : 0) | ((yy > 0) ? 2u : 0u) | ((xx > 0) ? 4u : 0u) |
         ((xx < A.nx - 1) ? 8u : 0u) | ((yy < A.ny - 1) ? 16u : 0u) | ((z < A.nz - 1 || A.has_zhi) ? 32u : 0u);
}
__device__ __forceinline__ unsigned stencil_mask(const CsrOp&, int) { return 0u; }

template <int NVX, class Ld>
__device__ __forceinline__ void pers_row(const StencilOp& A, int row, unsigned m, Ld ld, double (&y)[NVX]) {
  const int plane = A.nx * A.ny;
  double v[NVX];
#pragma unroll
  for (int c = 0; c < NVX; ++c) y[c] = 0.0;
#define CGX_PT(bit, j, coef)                                                               \
  {                                                                                        \
    const bool ex = (m & (bit)) != 0u;               /* absent neighbour: read the row itself, drop the term */ \
    ld(ex ? (j) : row, v);                                                                 \
    _Pragma("unroll") for (int c = 0; c < NVX; ++c) {                                      \
      const double t = add_(y[c], mul_((coef), v[c]));                                     \
      y[c] = ex ? t : y[c];                                                                \
    }                                                                                      \
  }
  CGX_PT(1u, row - plane, A.off)
  CGX_PT(2u, row - A.nx, A.off)
  CGX_PT(4u, row - 1, A.off)
  CGX_PT(~0u, row, A.diag)
  CGX_PT(8u, row + 1, A.off)
  CGX_PT(16u, row + A.nx, A.off)
  CGX_PT(32u, row + plane, A.off)
#undef CGX_PT
}
template <int NVX, class Ld>
__device__ __forceinline__ void pers_row(const CsrOp& A, int row, unsigned, Ld ld, double (&y)[NVX]) {
  A.template row<NVX>((i64)row, [&](i64 c, double (&v)[NVX]) { ld((int)c, v); }, y);
}
// same sum (stored order, separately rounded multiply and add) from the shared-memory slab
template <int NVX, class Ld>
__device__ __forceinline__ void pers_row_slab(const CsrSlab& S, int lrow, Ld ld, double (&y)[NVX]) {
#pragma unroll
  for (int c = 0; c < NVX; ++c) y[c] = 0.0;
  const int e = S.ptr[lrow + 1];
  for (int jj = S.ptr[lrow]; jj < e; ++jj) {
    const double a = S.val[jj];
    double v[NVX];
    ld(S.col[jj], v);
#pragma unroll
    for (int c = 0; c < NVX; ++c) y[c] = add_(y[c], mul_(a, v[c]));
  }
}
template <int NVX, class Ld>
__device__ __forceinline__ void pers_row_slab(const CsrSlab&, int, Ld, double (&)[NVX], const StencilOp&) {}

struct PersRec { u64 e; int kind; int k; int hist; };      // a published record still to be folded

// The whole solve of one rank, run by CTA `cta` (0 .. L.nb-1) of the rank's CTA range.  The
// static shared scratch is declared by the calling kernel, so that a kernel that can run several
// variants (persistent_batch_kernel) holds one copy of it, not one per inlined body:
// sh[kPersRed * 32], sh_acc[kPersRed], gg (the rank's global-memory Args), sh_last.
template <class Op, int VAR, int PM>
__device__ __forceinline__ void persistent_body(const PersRank<Op>& pr, const PersLaunch& L, const int cta,
                                                double* sh, double* sh_acc, Args& gg, int& sh_last) {
  using P = PersPlan<VAR>;
  constexpr int EW = P::EW, SP = P::SP;
  constexpr bool MEUR = P::MEUR;
  constexpr int NRE = EwTraits<EW>::NR, NRS = SpTraits<SP>::NR, NV = SpTraits<SP>::NV;
  constexpr bool SL = Op::kSlab;
  extern __shared__ __align__(16) double smem[];               // [nslot][R*T]

  const int T = blockDim.x, tid = threadIdx.x;
  const int nb = L.nb;
  const Op A = pr.A;
  if (tid == 0) gg = pr.g;
  __syncthreads();
  Args gl = gg;                                                // same, vectors in shared memory (per thread)
  {
    int slot = 0;
    for (int v = 0; v < 10; ++v)
      if (L.vmask & (1u << v)) { args_vec(gl, v) = smem + (size_t)slot * L.R * T; ++slot; }
    if (PM == 1) gl.dinv = smem + (size_t)slot * L.R * T;
    gl.d.world = 1;                                            // halo stores are done here, not in ew_body
  }
  const Args& g = gg;
  const i64 n = g.n;
  const int world = g.d.world, rank = g.d.rank;
  const bool dist = world > 1;
  int* err = &pr.out->err;
  u64* bar = pr.bar;
  const bool hist = g.hist_mask != 0;
  const bool has_xt = (g.hist_mask & 5u) != 0;
  const i64 pl = g.d.plane;
  WinHdr* mywin = dist ? g.d.win[rank] : nullptr;

  // ---- state -> shared memory ---------------------------------------------------------
  {
    int slot = 0;
    for (int v = 0; v < 10; ++v) {
      if (!(L.vmask & (1u << v))) continue;
      const double* src = pr.vecs[v];
      double* dst = smem + (size_t)slot * L.R * T;
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row < n) dst[j * T + tid] = src[row];
      }
      ++slot;
    }
    if (PM == 1) {
      double* dst = smem + (size_t)slot * L.R * T;
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row < n) dst[j * T + tid] = g.dinv[row];
      }
    }
  }
  unsigned char* smask = reinterpret_cast<unsigned char*>(smem + (size_t)L.nslot * L.R * T);
  for (int j = 0; j < L.R; ++j) {
    const i64 row = ((i64)j * nb + cta) * T + tid;
    if (row < n) smask[j * T + tid] = (unsigned char)stencil_mask(A, (int)row);
  }
  // CSR: this CTA's matrix rows -> shared memory (one coalesced sweep, once per launch)
  CsrSlab slab{nullptr, nullptr, nullptr};
  bool use_slab = false;
  if constexpr (!SL) {
    if (L.slab_cap > 0) {
      unsigned char* base = reinterpret_cast<unsigned char*>(smask) + (((size_t)L.R * T + 15) / 16) * 16;
      double* sval = reinterpret_cast<double*>(base);
      int* scol = reinterpret_cast<int*>(sval + L.slab_cap);
      int* sptr = scol + L.slab_cap;
      const i64 r0 = (i64)cta * T, r1 = min(n, r0 + T);
      if (r0 < n) {
        const int e0 = A.ptr[r0], cnt = A.ptr[r1] - e0;
        for (int e = tid; e < cnt; e += T) { sval[e] = A.val[e0 + e]; scol[e] = A.idx[e0 + e]; }
        for (int t = tid; t <= (int)(r1 - r0); t += T) sptr[t] = A.ptr[r0 + t] - e0;
      }
      slab = CsrSlab{sval, scol, sptr};
      use_slab = true;
    }
  }
  __syncthreads();

  Scal s;                                                      // the recurrences live in registers
  {
    const Scal* i0 = &g.sc[dist ? g.scpar : 0];
    s.a = i0->a; s.a1 = i0->a1; s.b = i0->b; s.nu = i0->nu; s.nu1 = i0->nu1; s.mu = i0->mu; s.eta = i0->eta;
    s.del = i0->del; s.gam = i0->gam; s.breakdown = i0->breakdown;
    s.stop_k = i0->stop_k; s.thr = i0->thr;
  }
  u64 nbar = 0, epoch = pr.epoch0;
  u64 hep[kChan];
#pragma unroll
  for (int c = 0; c < kChan; ++c) hep[c] = pr.hepoch0[c];
  int buf = 0;
  PersRec pend[3];
  int npend = 0;

  // does this CTA own rows of the first / last plane (it then reads ghost planes)?
  bool touch_lo = false, touch_hi = false;
  if (dist) {
    for (int j = 0; j < L.R; ++j) {
      const i64 r0 = ((i64)j * nb + cta) * T, r1 = min(n, r0 + T);
      if (r0 < n && r0 < pl) touch_lo = true;
      if (r0 < n && r1 > n - pl) touch_hi = true;
    }
  }
  // ---- sync point: every CTA of the rank has finished the stage; optionally the rank's
  //      record (NR sums) is formed and, on a partition, published with the halo epochs
  auto sync_point = [&](double (&red)[kPersRed], auto NRc, int kind, int k, bool rec_hist, int halo_n, int halo_ch) {
    constexpr int NR = decltype(NRc)::value;                   // sums in the record: 0 (barrier only) .. 8
    double* part = pr.part + (size_t)buf * kPersMaxGrid * kPersRed;
    double v[NR > 0 ? NR : 1];
    if constexpr (NR > 0) {
#pragma unroll
      for (int j = 0; j < NR; ++j) v[j] = red[j];
      block_sum<NR>(v, sh);                                    // totals of the CTA in warp 0
    }
    auto finish_local = [&](const double* acc) {               // one GPU: recurrences now
      if (kind != FK_NONE) apply_finalize(kind, MEUR, &s, acc, k);
      if constexpr (NR == kPersRed) {
        if (rec_hist && cta == 0 && tid == 0) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (g.hist_mask & (1u << j)) g.hist[(i64)j * g.hist_len + k] = sqrt(acc[4 + j]);
        }
      }
    };
    if (!dist && nb == 1) {                                    // a single CTA: shared memory only
      if constexpr (NR > 0) {
        if (tid == 0) {
#pragma unroll
          for (int j = 0; j < NR; ++j) sh_acc[j] = v[j];
        }
      }
      __syncthreads();
      if constexpr (NR > 0) {
        double acc[kPersRed] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int j = 0; j < NR; ++j) acc[j] = sh_acc[j];
        finish_local(acc);
      }
      return;
    }
    ++nbar;
    const u64 target = (u64)nb * nbar;
    u64 e = 0;
    if (NR > 0) e = ++epoch;
    if constexpr (NR == 0) __syncthreads();                    // (block_sum already synchronised the CTA)
    if (tid == 0) {
      if constexpr (NR > 0) {
#pragma unroll
        for (int j = 0; j < NR; ++j) __stcg(&part[(size_t)cta * kPersRed + j], v[j]);
      }
      if (dist) {
        fence_acq_rel_gpu();           // (records and ghost planes travel as self-validating LL words)
        const u64 t = atomicAdd(reinterpret_cast<unsigned long long*>(bar), 1ull);
        sh_last = (t == target - 1) ? 1 : 0;
      } else {                                                 // release-add, no round trip
        asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(bar), "l"(1ull) : "memory");
        pers_wait_gpu(bar, target, err);
      }
    }
    __syncthreads();
    if (dist) {
      if (sh_last && tid < 32) {                               // warp 0 of the last CTA: publish
        fence_acq_rel_gpu();
        if constexpr (NR > 0) {
          const int slot = (int)(e % kSlots);
          double tot[NR];
#pragma unroll
          for (int j = 0; j < NR; ++j) {
            double t = 0.0;
            for (int b = tid; b < nb; b += 32) t += __ldcg(&part[(size_t)b * kPersRed + j]);
            tot[j] = warp_sum(t);
          }
          if (tid < world && (g.d.mode != 3 || tid == rank)) {   // lane r -> rank r's window (LL words)
            u64* dst = g.d.win[tid]->ll[slot][rank];
#pragma unroll
            for (int j = 0; j < NR; ++j) ll_store(dst + 2 * j, tot[j], e);
          }
        }
      }
      if (tid == 0) pers_wait_gpu(bar, target, err);
      __syncthreads();
    }
    if constexpr (NR > 0) {
      if (dist) {
        pend[npend].e = e; pend[npend].kind = kind; pend[npend].k = k;
        pend[npend].hist = (rec_hist ? 1 : 0) | (NR << 8);
        ++npend;
      } else {                                                 // one GPU: every warp adds the partials itself
        double acc[kPersRed] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        const int lane = tid & 31;
#pragma unroll
        for (int j = 0; j < NR; ++j) {
          double t = 0.0;
          for (int b = lane; b < nb; b += 32) t += __ldcg(&part[(size_t)b * kPersRed + j]);
          acc[j] = warp_sum(t);
        }
        finish_local(acc);
      }
      buf ^= 1;
    }
  };
  using NR0 = std::integral_constant<int, 0>;
  using NR8 = std::integral_constant<int, kPersRed>;

  // ---- partition: fold the published records of all ranks into the scalars ---------------
  auto fold_pending = [&]() {
    if (!dist) return;
    for (int q = 0; q < npend; ++q) {
      const u64 e = pend[q].e;
      const int slot = (int)(e % kSlots);
      __syncthreads();
      if (tid < 32) {
        double tot[kPersRed];
        ll_totals<kPersRed>(mywin, slot, e, world, pend[q].hist >> 8, g.d.mode == 3 ? rank : -1, tot);
        if (tid == 0) {
#pragma unroll
          for (int j = 0; j < kPersRed; ++j) sh_acc[j] = tot[j];
        }
      }
      __syncthreads();
      double acc[kPersRed];
#pragma unroll
      for (int j = 0; j < kPersRed; ++j) acc[j] = sh_acc[j];
      if (pend[q].kind != FK_NONE) apply_finalize(pend[q].kind, MEUR, &s, acc, pend[q].k);
      if ((pend[q].hist & 1) && cta == 0 && tid == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (g.hist_mask & (1u << j)) g.hist[(i64)j * g.hist_len + pend[q].k] = sqrt(acc[4 + j]);
      }
    }
    npend = 0;
  };

  // ---- export the SpMV input(s) (and x when instrumenting) of the rows this CTA owns ------
  auto export_inputs = [&](int par) {
    const double* l0 = args_vec(gl, SpInV<SP>::v0);
    const double* l1 = NV == 2 ? args_vec(gl, SpInV<SP>::v1 < 0 ? 0 : SpInV<SP>::v1) : nullptr;
    double* e0 = pr.exp_[par][0];
    double* e1 = pr.exp_[par][1];
    if (dist) { ++hep[0]; if (NV == 2) ++hep[1]; if (hist) ++hep[2]; }
    const int hp0 = (int)(hep[0] & 1), hp1 = (int)(hep[1] & 1), hp2 = (int)(hep[2] & 1);
    for (int j = 0; j < L.R; ++j) {
      const i64 row = ((i64)j * nb + cta) * T + tid;
      if (row >= n) continue;
      const double a0 = l0[j * T + tid];
      e0[row] = a0;
      double a1 = 0.0, xv = 0.0;
      if (NV == 2) { a1 = l1[j * T + tid]; e1[row] = a1; }
      if (hist) { xv = gl.x[j * T + tid]; pr.vecs[0][row] = xv; }
      if (dist) {
        if (g.d.has_lo && row < pl) {
          ll_store(g.d.ghl_lo + ghl_off(g.d, 0, hp0, 1) + 2 * row, a0, hep[0]);
          if (NV == 2) ll_store(g.d.ghl_lo + ghl_off(g.d, 1, hp1, 1) + 2 * row, a1, hep[1]);
          if (hist) ll_store(g.d.ghl_lo + ghl_off(g.d, 2, hp2, 1) + 2 * row, xv, hep[2]);
        }
        if (g.d.has_hi && row >= n - pl) {
          const i64 o = row - (n - pl);
          ll_store(g.d.ghl_hi + ghl_off(g.d, 0, hp0, 0) + 2 * o, a0, hep[0]);
          if (NV == 2) ll_store(g.d.ghl_hi + ghl_off(g.d, 1, hp1, 0) + 2 * o, a1, hep[1]);
          if (hist) ll_store(g.d.ghl_hi + ghl_off(g.d, 2, hp2, 0) + 2 * o, xv, hep[2]);
        }
      }
    }
  };

  // x_true ghost planes (channel 3) were pushed by the stream kernels when the problem was
  // loaded: one flag wait for the whole launch
  if (dist && hist && has_xt) {
    if (tid == 0) {
      if (touch_lo && g.d.has_lo) pers_wait_sys(&mywin->hflag[3][g.xt_par][0], g.xt_epoch, err);
      if (touch_hi && g.d.has_hi) pers_wait_sys(&mywin->hflag[3][g.xt_par][1], g.xt_epoch, err);
    }
    __syncthreads();
  }

  for (int k = L.k0; k <= L.k1; ++k) {
    const int par = k & 1;
    double red[kPersRed];
    // ---- vector stage(s) ----------------------------------------------------------
    fold_pending();
#pragma unroll
    for (int j = 0; j < kPersRed; ++j) red[j] = 0.0;
    {
      double r4[kNRed] = {0.0, 0.0, 0.0, 0.0};
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row < n) ew_body<EW, PM, 1>(gl, (i64)j * T + tid, s.a, s.b, r4);
      }
#pragma unroll
      for (int j = 0; j < kNRed; ++j) red[j] = r4[j];
    }
    if constexpr (VAR == CGX_HS) {                 // hs_cg.py:120-122: beta needs nu first
      sync_point(red, std::integral_constant<int, NRE>{}, EwKind<EW>::FK, k, false, 0, 0);
      fold_pending();
      double r4[kNRed] = {0.0, 0.0, 0.0, 0.0};
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row < n) ew_body<EW_HS2, PM, 1>(gl, (i64)j * T + tid, s.a, s.b, r4);
      }
      export_inputs(par);
      sync_point(red, NR0{}, FK_NONE, k, false, hist ? 3 : 1, 0);
    } else {
      export_inputs(par);
      sync_point(red, std::integral_constant<int, NRE>{}, EwKind<EW>::FK, k, false, hist ? 3 : NV, 0);
    }
    // ---- SpMV stage with the fused epilogue (+ instrumentation) --------------------
#pragma unroll
    for (int j = 0; j < kPersRed; ++j) red[j] = 0.0;
    {
      const int hp0 = (int)(hep[0] & 1), hp1 = (int)(hep[1] & 1), hp2 = (int)(hep[2] & 1);
      VecIn in0{pr.exp_[par][0], nullptr, nullptr}, in1{pr.exp_[par][1], nullptr, nullptr};
      VecIn xin{pr.vecs[0], nullptr, nullptr}, xtin{g.xtrue, nullptr, nullptr};
      struct GhostLL { const u64* lo; const u64* hi; u64 ep; };
      GhostLL q0{nullptr, nullptr, 0}, q1{nullptr, nullptr, 0}, qx{nullptr, nullptr, 0}, qn{nullptr, nullptr, 0};
      if (dist) {
        q0 = GhostLL{g.d.ghl + ghl_off(g.d, 0, hp0, 0), g.d.ghl + ghl_off(g.d, 0, hp0, 1), hep[0]};
        q1 = GhostLL{g.d.ghl + ghl_off(g.d, 1, hp1, 0), g.d.ghl + ghl_off(g.d, 1, hp1, 1), hep[1]};
        qx = GhostLL{g.d.ghl + ghl_off(g.d, 2, hp2, 0), g.d.ghl + ghl_off(g.d, 2, hp2, 1), hep[2]};
        xtin.lo = g.d.ghost + ghost_off(g.d, 3, g.xt_par, 0); xtin.hi = g.d.ghost + ghost_off(g.d, 3, g.xt_par, 1);
      }
      // element c of an exported vector: rows of the CTA's own chunk come from shared memory
      // (same bits as the exported copy), the rest from L2, ghost planes from the window
      // (one generic load through a selected pointer: no branch.  Global lines may sit in L1
      // only since the last sync point, whose acquire fence invalidated it.)
      const int ni = (int)n, pli = (int)pl;
      auto ldv = [&](const VecIn& a, const GhostLL& q, const double* loc, int r0, int c) -> double {
        if constexpr (SL) {             // ghost planes: LL words polled element by element (or plain doubles)
          if (c < 0) return q.lo ? ll_load16_cold(q.lo, c + pli, q.ep, err) : __ldcg(a.lo + (c + pli));
          if (c >= ni) return q.hi ? ll_load16_cold(q.hi, c - ni, q.ep, err) : __ldcg(a.hi + (c - ni));
        }
        const unsigned d = (unsigned)(c - r0);
        const double* p = (loc != nullptr && d < (unsigned)T) ? loc + d : a.v + c;
        return *p;
      };
      const VecIn loc0{args_vec(gl, SpInV<SP>::v0), nullptr, nullptr};
      const double* sl0 = loc0.v;
      const double* sl1 = NV == 2 ? args_vec(gl, SpInV<SP>::v1 < 0 ? 0 : SpInV<SP>::v1) : nullptr;
      double r4[kNRed] = {0.0, 0.0, 0.0, 0.0};
      double hs[4] = {0.0, 0.0, 0.0, 0.0};
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row >= n) continue;
        const int li = j * T + tid;
        const int r0 = (j * nb + cta) * T;
        if (hist) {
          double y[NV + 2];
          auto ldh = [&](int c, double (&v)[NV + 2]) {
            v[0] = ldv(in0, q0, sl0 + j * T, r0, c);
            if constexpr (NV == 2) v[1] = ldv(in1, q1, sl1 + j * T, r0, c);
            const double xj = ldv(xin, qx, gl.x + j * T, r0, c);
            v[NV] = xj;
            v[NV + 1] = has_xt ? sub_(xj, ldv(xtin, qn, nullptr, r0, c)) : 0.0;
          };
          if (!SL && use_slab) pers_row_slab<NV + 2>(slab, tid, ldh, y);
          else pers_row<NV + 2>(A, (int)row, smask[li], ldh, y);
          double ysp[NV];
#pragma unroll
          for (int c = 0; c < NV; ++c) ysp[c] = y[c];
          sp_epilogue<SP, PM, NV>(gl, loc0, li, ysp, r4, nullptr);
          if (has_xt) {                            // callbacks/error_A_norm.py, error_2_norm.py
            const double e = sub_(gl.x[li], g.xtrue[row]);
            hs[0] = fma(e, y[NV + 1], hs[0]);
            hs[2] = fma(e, e, hs[2]);
          }
          const double res = sub_(g.b[row], y[NV]);  // callbacks/residual_2_norm.py
          hs[1] = fma(res, res, hs[1]);
          const double ri = gl.r[li];                // callbacks/updated_residual_2_norm.py
          hs[3] = fma(ri, ri, hs[3]);
        } else {
          double y[NV];
          auto ldp2 = [&](int c, double (&v)[NV]) {
            v[0] = ldv(in0, q0, sl0 + j * T, r0, c);
            if constexpr (NV == 2) v[1] = ldv(in1, q1, sl1 + j * T, r0, c);
          };
          if (!SL && use_slab) pers_row_slab<NV>(slab, tid, ldp2, y);
          else pers_row<NV>(A, (int)row, smask[li], ldp2, y);
          sp_epilogue<SP, PM, NV>(gl, loc0, li, y, r4, nullptr);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) { red[j] = r4[j]; red[4 + j] = hs[j]; }
    }
    if (hist) sync_point(red, NR8{}, SpTraits<SP>::FK, k, true, 0, 0);
    else if constexpr (NRS > 0) sync_point(red, std::integral_constant<int, NRS>{}, SpTraits<SP>::FK, k, false, 0, 0);
    // a tolerance was met in this iteration: every CTA formed the same stop_k from the same totals at a
    // sync point of this iteration and leaves here, after the last one, so none waits on a counter
    if (s.stop_k >= 0) break;
  }
  fold_pending();

  // ---- shared memory -> state; scalars and epoch counters back to the host's view ---------
  __syncthreads();
  {
    int slot = 0;
    for (int v = 0; v < 10; ++v) {
      if (!(L.vmask & (1u << v))) continue;
      double* dstv = pr.vecs[v];
      const double* src = smem + (size_t)slot * L.R * T;
      for (int j = 0; j < L.R; ++j) {
        const i64 row = ((i64)j * nb + cta) * T + tid;
        if (row < n) dstv[row] = src[j * T + tid];
      }
      ++slot;
    }
  }
  if (cta == 0 && tid == 0) {
    Scal* o = &g.sc[dist ? g.scpar : 0];           // (tmp[] is initialisation scratch: not kept live)
    o->a = s.a; o->a1 = s.a1; o->b = s.b; o->nu = s.nu; o->nu1 = s.nu1; o->mu = s.mu; o->eta = s.eta;
    o->del = s.del; o->gam = s.gam; o->breakdown = s.breakdown; o->stop_k = s.stop_k;
    pr.out->epoch = epoch;
    for (int c = 0; c < kChan; ++c) pr.out->hepoch[c] = hep[c];
  }
}

// One variant; CTA range r*nb .. (r+1)*nb-1 is rank r of ranks[] (one entry on a single GPU).
template <class Op, int VAR, int PM>
__global__ void __launch_bounds__(512) persistent_kernel(const PersRank<Op>* __restrict__ ranks,
                                                          const PersLaunch L) {
  __shared__ double sh[kPersRed * 32];
  __shared__ double sh_acc[kPersRed];
  __shared__ Args gg;
  __shared__ int sh_last;
  const int rk = blockIdx.x / L.nb;
  persistent_body<Op, VAR, PM>(ranks[rk], L, blockIdx.x - rk * L.nb, sh, sh_acc, gg, sh_last);
}

// A batch of independent single-GPU solves (cgx_batch_run): entry i owns CTAs cta0 .. cta0+L.nb-1
// and runs its own variant with its own sync counter, partials and PersOut.  Entries never wait
// for each other; one that has fewer iterations simply finishes first.  The grid is one
// cooperative launch, so every entry's CTAs are co-resident (separate launches would not be
// guaranteed to run side by side).  blockDim is common; the dynamic shared memory is the largest
// entry's.
template <class Op>
struct PersEntry {
  PersRank<Op> r;
  PersLaunch L;
  int variant;
  int cta0;                            // first CTA of the entry (entries in ascending order)
};

template <class Op, int PM>
__global__ void __launch_bounds__(512) persistent_batch_kernel(const PersEntry<Op>* __restrict__ entries, int count) {
  __shared__ double sh[kPersRed * 32];
  __shared__ double sh_acc[kPersRed];
  __shared__ Args gg;
  __shared__ int sh_last;
  int i = 0;
  while (i + 1 < count && (int)blockIdx.x >= entries[i + 1].cta0) ++i;
  const PersEntry<Op>& e = entries[i];
  const int cta = (int)blockIdx.x - e.cta0;
  switch (e.variant) {
#define CGX_PB(V) case V: persistent_body<Op, V, PM>(e.r, e.L, cta, sh, sh_acc, gg, sh_last); break;
    CGX_PB(CGX_HS) CGX_PB(CGX_CG) CGX_PB(CGX_GV) CGX_PB(CGX_PR) CGX_PB(CGX_M) CGX_PB(CGX_PIPE_PR)
    CGX_PB(CGX_PIPE_P) CGX_PB(CGX_PIPE_PR_M) CGX_PB(CGX_PIPE_P_M)
#undef CGX_PB
    default: break;
  }
}

}  // namespace cgx
