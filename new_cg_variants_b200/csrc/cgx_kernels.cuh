// cgx_kernels.cuh -- streaming-path kernels: operators, fused vector passes, fused
// SpMV passes, instrumentation.  One template per dependency stage; the variant is a
// compile-time tag.  Reference statements: SURVEY.md section 8 / the file:line cited at each
// body (paths relative to predict_and_recompute/numerical_experiments/cg_variants/).
#pragma once
#include "cgx_common.cuh"

namespace cgx {

// =====================================================================================
// Operators.  row<NV>(i, ld, y): y[c] = sum_j A_ij * v_c[j] for NV right-hand sides whose
// entries are produced by ld(j, vals).  Accumulation mirrors scipy's csr_matvec
// (sum = 0; sum += a*v, stored order, multiply and add rounded separately).
// =====================================================================================
struct CsrOp {
  static constexpr bool kSlab = false;
  const int* __restrict__ ptr;
  const int* __restrict__ idx;
  const double* __restrict__ val;
  i64 n;
  template <int NV, class Ld>
  __device__ __forceinline__ void row(i64 i, Ld ld, double (&y)[NV]) const {
#pragma unroll
    for (int c = 0; c < NV; ++c) y[c] = 0.0;
    const int e = __ldg(ptr + i + 1);
    for (int jj = __ldg(ptr + i); jj < e; ++jj) {
      const double a = __ldg(val + jj);
      double v[NV];
      ld((i64)__ldg(idx + jj), v);
#pragma unroll
      for (int c = 0; c < NV; ++c) y[c] = add_(y[c], mul_(a, v[c]));
    }
  }
};

// Matrix-free Dirichlet Poisson stencil, natural ordering.  Visits the neighbours in
// ascending column order (z-1, y-1, x-1, centre, x+1, y+1, z+1), i.e. exactly the order
// of the canonical CSR matrix, so the result is bit-identical to scipy on that matrix.
// In a multi-GPU run the operator is the z-slab [z_begin, z_begin + nz) of the global grid:
// has_zlo / has_zhi say that a plane exists below local z = 0 / above local z = nz-1; the
// loader is then called with j < 0 or j >= n for those neighbours (see VecIn).
struct StencilOp {
  static constexpr bool kSlab = true;
  int nx, ny, nz;
  double diag, off;
  i64 n;
  int has_zlo, has_zhi;
  template <int NV, class Ld>
  __device__ __forceinline__ void row(i64 i, Ld ld, double (&y)[NV]) const {
    const int plane = nx * ny;
    const int ii = (int)i;
    const int z = ii / plane;
    const int rem = ii - z * plane;
    const int yy = rem / nx;
    const int xx = rem - yy * nx;
    double v[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) y[c] = 0.0;
#define CGX_ST_TERM(cond, j, coef)                                         \
    if (cond) {                                                            \
      ld((i64)(j), v);                                                     \
      _Pragma("unroll") for (int c = 0; c < NV; ++c) y[c] = add_(y[c], mul_((coef), v[c])); \
    }
    CGX_ST_TERM(z > 0 || has_zlo, ii - plane, off)
    CGX_ST_TERM(yy > 0, ii - nx, off)
    CGX_ST_TERM(xx > 0, ii - 1, off)
    CGX_ST_TERM(true, ii, diag)
    CGX_ST_TERM(xx < nx - 1, ii + 1, off)
    CGX_ST_TERM(yy < ny - 1, ii + nx, off)
    CGX_ST_TERM(z < nz - 1 || has_zhi, ii + plane, off)
#undef CGX_ST_TERM
  }
};

// =====================================================================================
// Kernel argument block (plain pointers; unused ones are null).
// =====================================================================================
struct Args {
  double* x; double* r; double* rt; double* p; double* s; double* st;
  double* w; double* wt; double* u; double* t;
  const double* dinv; double dinv_s;
  const double* b; const double* xtrue;
  Scal* sc; double* partials; unsigned* ticket;
  double* hist; int hist_len; unsigned hist_mask;
  i64 n; int k;
  // ---- multi-GPU (d.world > 1), filled per launch by the host ----
  Dist d;
  int scpar;                 // which of sc[0], sc[1] holds the scalars this kernel starts from
  int npend;                 // reductions of earlier kernels still to be folded into them
  int pend_kind[3], pend_k[3];
  u64 pend_e[3];             // their epochs
  u64 sepoch;                // epoch of the reduction this kernel produces
  int hout_n, hout_ch, hout_par;   // halo planes this kernel produces: channels hout_ch ..
  u64 hout_epoch;
  int hin_ch, hin_par;             // halo planes this kernel consumes
  u64 hin_epoch;
  int xt_par;                      // ghost planes of x_true (channel 3), pushed when the problem is loaded
  u64 xt_epoch;
  int meur;                        // Meurant predictor (kernels that are not templated on it)
  int halo_ll;                     // the consumer is the TMA stencil kernel: boundary planes travel as LL words
  int* errflag;                    // device word set by a bounded in-kernel wait that expired
  unsigned long long l2pol;        // 0, or an L2 cache-policy word for the state-vector accesses (kL2EvictLast)
  double* gscr;                    // fused PR kernel on a partition: [plane] new p of the ghost plane above the slab
  int tol_on;                      // a tolerance is set: launches of iterations after sc->stop_k return at entry
  int dbg;                         // timing experiments (cgx_set_option "debug_skip"): 1 = no halo traffic, 2 = time stamps
  u64* dbg_t;                      // dbg & 2: CTA 0 writes %globaltimer at kernel start / after the scalar fold / at its end
};

// Every kernel of the iteration loop starts with this test (after griddepcontrol.wait where the kernel
// is launched with programmatic serialisation: stop_k is written by an earlier kernel).  stop_k was
// written before the launch, so every CTA takes the same branch.  On a partition the scalars live in
// sc[scpar]: every consumer of pending records persists its fold there, also after the stop (dist_fold),
// so the parity the host hands to a launch always holds the latest stop_k.  (One GPU: scpar = 0.)
// The vector passes of a partition do not take this test at entry: they fold first (dist_fold).
__device__ __forceinline__ bool after_stop(const Args& g) { return g.tol_on && past_stop(g.sc + g.scpar, g.k); }

// An SpMV input vector: the owned slab and (multi-GPU) the ghost planes below and above.
struct VecIn { const double* v; const double* lo; const double* hi; };
template <bool SLAB>
__device__ __forceinline__ double vload(const VecIn& a, i64 j, i64 n, i64 plane) {
  if constexpr (SLAB) {
    if (j < 0) return a.lo[j + plane];
    if (j >= n) return a.hi[j - n];
    return a.v[j];
  } else {
    // CSR row partition: columns >= n address the staging array of gathered ghost entries
    return (j < n ? a.v : a.lo - n)[j];
  }
}

// Stage tags
enum {
  EW_HS1 = 0,   // r -= a s ; nu = r.(M r)
  EW_HS2,       // x += a p ; p = M r + b p
  EW_CG,        // [deferred p,s] ; x,r ; rt = M r
  EW_GV,        // [deferred p,s,st,u] ; x,r,rt,w ; wt = M w ; nu,eta
  EW_PR,        // x,r,rt ; p ; nu = rt.r
  EW_PIPE_R,    // pipe family with recompute of w (pipe_pr, pipe_pr_m)
  EW_PIPE_N,    // pipe family without recompute (pipe_p, pipe_p_m)
  EW_CG_E       // EW_CG with r~ elided: identity / constant-diagonal Jacobi and the TMA stencil pass,
                // which then multiplies M r on the fly (r~ = M r is recomputed every iteration in CG-CG,
                // cg_cg.py:132, so the products are the same bits; 3 of 14 words per row less)
  , EW_GV_E     // EW_GV with w~ elided on the same grounds (w~ = M w, gv_cg.py:160): 2 of 21 words less
};
enum { SP_PLAIN = 0, SP_HS, SP_CG, SP_GV, SP_PR, SP_PIPE_R, SP_PIPE_N, SP_RESID, SP_CG_E, SP_GV_E };

template <int KID> struct EwTraits { static constexpr int NR = 0; };
template <> struct EwTraits<EW_HS1> { static constexpr int NR = 1; };
template <> struct EwTraits<EW_GV> { static constexpr int NR = 2; };
template <> struct EwTraits<EW_GV_E> { static constexpr int NR = 2; };
template <> struct EwTraits<EW_PR> { static constexpr int NR = 1; };
template <> struct EwTraits<EW_PIPE_R> { static constexpr int NR = 4; };
template <> struct EwTraits<EW_PIPE_N> { static constexpr int NR = 4; };

// Predicted nu and the beta it gives (pr_cg.py:149-150, pipe_pr_cg.py:174-175):
//   PR: nu' = nu - 2 a del + a^2 gam      M: nu' = -nu + a^2 gam      b = nu'/nu
__device__ __forceinline__ double predict_beta(bool meurant, double nu, double a, double del,
                                               double gam) {
  const double a2g = mul_(mul_(a, a), gam);
  const double nup = meurant ? add_(-nu, a2g) : add_(sub_(nu, mul_(mul_(2.0, a), del)), a2g);
  return div_(nup, nu);
}

// Scalar recurrences that close a fused reduction (run by one thread with the grid -- or,
// multi-GPU, the all-rank -- totals).  kind: FK_* of cgx_common.cuh.  The tolerance is tested where
// nu_k is assigned (note_stop; without a tolerance thr is NaN and nothing stops).
__device__ __forceinline__ void apply_finalize(int kind, bool meurant, Scal* sc, const double* acc, int k) {
  if (kind == FK_HS_NU) {                    // hs_cg.py:120-121
    const double nu1 = sc->nu;
    sc->nu1 = nu1; sc->nu = acc[0];
    sc->b = div_(acc[0], nu1);
    note_breakdown(sc, k, sc->a, sc->b);
    note_stop(sc, k);
  } else if (kind == FK_HS_MU) {             // hs_cg.py:124-125
    sc->mu = acc[0];
    sc->a1 = sc->a; sc->a = div_(sc->nu, acc[0]);
    note_breakdown(sc, k, sc->a, sc->b);
  } else if (kind == FK_CGGV) {              // cg_cg.py:134-136,139-140 ; gv_cg.py:162-164,169-170
    const double nu1 = sc->nu, a1 = sc->a, nu = acc[0], eta = acc[1];
    const double bb = div_(nu, nu1);
    const double mu = sub_(eta, mul_(div_(bb, a1), nu));
    sc->nu1 = nu1; sc->nu = nu; sc->eta = eta; sc->b = bb; sc->mu = mu;
    sc->a1 = a1; sc->a = div_(nu, mu);
    note_breakdown(sc, k, sc->a, bb);
    note_stop(sc, k);
  } else if (kind == FK_PR_NU) {             // pr_cg.py:157 (consumed by the SpMV pass)
    sc->nu1 = sc->nu; sc->nu = acc[0];
    note_stop(sc, k);
  } else if (kind == FK_PR_SP) {             // pr_cg.py:154-158 then :149-150
    const double mu = acc[0], del = acc[1], gam = acc[2], nu = sc->nu;
    sc->mu = mu; sc->del = del; sc->gam = gam;
    const double an = div_(nu, mu);
    sc->a1 = sc->a; sc->a = an;
    sc->b = predict_beta(meurant, nu, an, del, gam);
    note_breakdown(sc, k, an, sc->b);
  } else if (kind == FK_PIPE) {              // pipe_pr_cg.py:183-187 then :174-175
    const double mu = acc[0], del = acc[1], gam = acc[2], nu = acc[3];
    sc->nu1 = sc->nu; sc->nu = nu; sc->mu = mu; sc->del = del; sc->gam = gam;
    const double an = div_(nu, mu);
    sc->a1 = sc->a; sc->a = an;
    sc->b = predict_beta(meurant, nu, an, del, gam);
    note_breakdown(sc, k, an, sc->b);
    note_stop(sc, k);
  }
}

// ---- multi-GPU scalar exchange ------------------------------------------------------
// Producer side (ONE thread, after the grid total is known): store this rank's record of
// epoch g.sepoch into every rank's window, fence, then publish the epoch -- and the halo
// epoch of the planes this kernel wrote into the neighbours' ghosts.
__device__ __forceinline__ void st_relaxed_sys(u64* p, u64 v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void dist_publish_halo_flags(const Args& g) {
  for (int c = 0; c < g.hout_n; ++c) {
    const int ch = g.hout_ch + c;
    if (g.d.has_lo) st_relaxed_sys(&g.d.win[g.d.rank - 1]->hflag[ch][g.hout_par][1], g.hout_epoch);
    if (g.d.has_hi) st_relaxed_sys(&g.d.win[g.d.rank + 1]->hflag[ch][g.hout_par][0], g.hout_epoch);
  }
}
template <int NR>
__device__ __forceinline__ void dist_publish(const Args& g, const double* acc) {
  const int slot = (int)(g.sepoch % kSlots);
  if (NR > 0) {
    if (g.d.mode == 1 || g.d.mode == 3) {
      for (int r = 0; r < g.d.world; ++r) {
        if (g.d.mode == 3 && r != g.d.rank) continue;     // stub: the record stays local
        u64* dst = g.d.win[r]->ll[slot][g.d.rank];
#pragma unroll
        for (int j = 0; j < NR; ++j) ll_store(dst + 2 * j, acc[j], g.sepoch);
      }
    } else {
      volatile double* dst = g.d.nccl_in + (size_t)slot * kSumW;
#pragma unroll
      for (int j = 0; j < NR; ++j) dst[j] = acc[j];
    }
  }
  if (g.hout_n > 0 && !g.halo_ll) {   // plain ghost planes are bulk data: fence, then their epochs
    __threadfence_system();
    dist_publish_halo_flags(g);
  }
}

// Consumer side (warp 0 of a CTA): all-rank totals of epoch e, added in rank order.
// number of sums in a record of kind FK_* (a consumer must not poll words nobody stores)
__device__ __forceinline__ int fk_width(int kind) {
  switch (kind) {
    case FK_NONE: return 0;
    case FK_CGGV: return 2;
    case FK_PR_SP: return 3;
    case FK_PIPE: return 4;
    default: return 1;               // FK_HS_NU, FK_HS_MU, FK_PR_NU
  }
}
__device__ __forceinline__ void dist_totals(const Args& g, u64 e, int nr, double (&acc)[kNRed]) {
  const int slot = (int)(e % kSlots);
  if (g.d.mode == 1 || g.d.mode == 3) {
    ll_totals<kNRed>(g.d.win[g.d.rank], slot, e, g.d.world, nr, g.d.mode == 3 ? g.d.rank : -1, acc);
  } else {
#pragma unroll
    for (int j = 0; j < kNRed; ++j) acc[j] = __ldcv(g.d.nccl_out + (size_t)slot * kSumW + j);
  }
}

// Every CTA of a kernel that needs alpha/beta: fold the pending reductions into the scalars
// (redundantly, identical bits everywhere); CTA 0 persists the result in the other parity.
// dist_fold: the warp-0 part (call with threadIdx.x < 32); the caller synchronises the CTA (or
// its compute warps) before reading sh_ab[0..2].
// Tolerance stop: nu_k of a partition is known only here, in the first consumer of iteration k + 1 (HS:
// in EW_HS2 of iteration k); apply_finalize makes the test where it assigns nu.  A record of an
// iteration after stop_k was never published (its launch returned): it is skipped without a poll; the
// records are in order, so once one sets stop_k the rest are skipped.
// The fold is persisted also after the stop -- the parity the host flips to must hold the scalars -- and
// is then exactly what the flush of a run ending at stop_k persists.
// sh_ab[2] != 0: this launch belongs to an iteration after stop_k and must return without any work.
__device__ __forceinline__ void dist_fold(const Args& g, bool meurant, double* sh_ab) {
  const bool stamp = (g.dbg & 2) && blockIdx.x == 0 && threadIdx.x == 0;
  {
    // Peer-to-peer records: every word of every pending record is requested FIRST (lane l: value
    // l & 3 of rank l >> 2), then the persisted scalars are loaded, then the records are
    // validated, summed in rank order and folded -- one memory round trip for the whole fold
    // (the in-kernel time stamps showed 1.2-1.9 us per record when they were fetched in turn).
    const bool ll = g.d.mode == 1 || g.d.mode == 3;
    const int lane = threadIdx.x, r = lane >> 2, j = lane & 3;
    const int only = g.d.mode == 3 ? g.d.rank : -1;
    WinHdr* w = g.d.win[g.d.rank];
    LLReq rq[3];
    bool on[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      on[q] = ll && q < g.npend && r < g.d.world && j < fk_width(g.pend_kind[q]) && (only < 0 || r == only);
      rq[q].src = w->ll[(int)(g.pend_e[q] % kSlots)][r < kMaxWorld ? r : 0] + 2 * j;
      rq[q].lo = rq[q].hi = 0;
      if (on[q]) ll_issue(rq[q]);
    }
    Scal s = g.sc[g.scpar];
    if (stamp) g.dbg_t[4] = (u64)clock64();
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      if (q < g.npend && !(g.tol_on && past_stop(&s, g.pend_k[q]))) {
        double acc[kNRed];
        if (ll) {
          const double v = on[q] ? ll_finish(rq[q], g.pend_e[q], &w->error) : 0.0;
#pragma unroll
          for (int c = 0; c < kNRed; ++c) {
            double t = 0.0;
            for (int rr = 0; rr < g.d.world; ++rr) t += __shfl_sync(0xffffffffu, v, rr * 4 + c);
            acc[c] = (only >= 0) ? t * (double)g.d.world : t;
          }
        } else {
          dist_totals(g, g.pend_e[q], fk_width(g.pend_kind[q]), acc);
        }
        if (stamp) g.dbg_t[5 + 2 * q] = (u64)clock64();
        apply_finalize(g.pend_kind[q], meurant, &s, acc, g.pend_k[q]);
        if (stamp) g.dbg_t[6 + 2 * q] = (u64)clock64();
      }
    }
    if (threadIdx.x == 0) {
      sh_ab[0] = s.a; sh_ab[1] = s.b;
      sh_ab[2] = (g.tol_on && past_stop(&s, g.k)) ? 1.0 : 0.0;
      if (blockIdx.x == 0 && g.npend) {          // (tmp[] is initialisation scratch: not carried over)
        Scal* o = &g.sc[g.scpar ^ 1];
        o->a = s.a; o->a1 = s.a1; o->b = s.b; o->nu = s.nu; o->nu1 = s.nu1; o->mu = s.mu; o->eta = s.eta;
        o->del = s.del; o->gam = s.gam; o->breakdown = s.breakdown; o->stop_k = s.stop_k; o->thr = s.thr;
      }
    }
  }
  if (stamp) g.dbg_t[9] = (u64)clock64();
}
// (returns true when the launch belongs to an iteration after a tolerance stop: see dist_fold)
__device__ __forceinline__ bool dist_scalars(const Args& g, bool meurant, double& a, double& b) {
  __shared__ double sh_ab[3];
  if (threadIdx.x < 32) dist_fold(g, meurant, sh_ab);
  __syncthreads();
  a = sh_ab[0]; b = sh_ab[1];
  return sh_ab[2] != 0.0;
}

// The SpMV-input vector a vector pass produces: also store its first / last plane into the
// ghost planes of the rank below / above (peer memory; 16-byte stores, plane is even).
template <int W>
__device__ __forceinline__ void halo_store(const Args& g, int c, i64 i, const Pk<W>& v) {
  if (g.d.world > 1 && !(g.dbg & 1)) {
    const i64 pl = g.d.plane;
    if (g.halo_ll) {
      // LL words (value halves tagged with the halo epoch): no flag, no fence -- a system-scope
      // fence after bulk peer stores costs several microseconds per launch (tools/dist_probe.py)
      if (g.d.has_lo && i < pl) {
        u64* q = g.d.ghl_lo + ghl_off(g.d, g.hout_ch + c, g.hout_par, 1) + 2 * i;
#pragma unroll
        for (int l = 0; l < W; ++l) ll_store(q + 2 * l, v.v[l], g.hout_epoch);
      }
      if (g.d.has_hi && i >= g.n - pl) {
        u64* q = g.d.ghl_hi + ghl_off(g.d, g.hout_ch + c, g.hout_par, 0) + 2 * (i - (g.n - pl));
#pragma unroll
        for (int l = 0; l < W; ++l) ll_store(q + 2 * l, v.v[l], g.hout_epoch);
      }
      return;
    }
    if (g.d.has_lo && i < pl) stp<W>(g.d.ghost_lo + ghost_off(g.d, g.hout_ch + c, g.hout_par, 1), i, v);
    if (g.d.has_hi && i >= g.n - pl)
      stp<W>(g.d.ghost_hi + ghost_off(g.d, g.hout_ch + c, g.hout_par, 0), i - (g.n - pl), v);
  }
}
// Generic (non-TMA) consumers: one thread waits for the ghost planes of channels
// hin_ch .. hin_ch+nch-1 before the CTA reads them.
__device__ __forceinline__ void csr_wait_channel(const Args& g, int ch, int par, u64 epoch) {
  WinHdr* w = g.d.win[g.d.rank];
  for (int r = 0; r < g.d.world; ++r)
    if (g.d.src_mask & (1u << r)) wait_epoch(&w->gflag[ch][par][r], epoch, &w->error);
}
__device__ __forceinline__ void halo_wait_all(const Args& g, int nch) {
  if (g.d.world > 1) {
    if (threadIdx.x == 0 && g.d.csr) {
      for (int c = 0; c < nch; ++c) csr_wait_channel(g, g.hin_ch + c, g.hin_par, g.hin_epoch);
    } else if (threadIdx.x == 0) {
      WinHdr* w = g.d.win[g.d.rank];
      for (int c = 0; c < nch; ++c) {
        if (g.d.has_lo) wait_epoch(&w->hflag[g.hin_ch + c][g.hin_par][0], g.hin_epoch, &w->error);
        if (g.d.has_hi) wait_epoch(&w->hflag[g.hin_ch + c][g.hin_par][1], g.hin_epoch, &w->error);
      }
    }
    __syncthreads();
  }
}

// -------------------------------------------------------------------------------------
// Fused vector pass: one HBM sweep over the state vectors of stage KID.
// -------------------------------------------------------------------------------------
// PM: preconditioner mode -- 0 identity, 1 Jacobi vector g.dinv, 2 Jacobi scalar g.dinv_s
// (a constant diagonal, e.g. every Poisson stencil: same products, one HBM stream less).
template <int KID, int PM, int W>
__device__ __forceinline__ void ew_body(const Args& g, i64 i, double a, double b,
                                        double (&red)[kNRed]) {
  constexpr bool PREC = PM != 0;
  Pk<W> dv{};
  if constexpr (PM == 1) dv = ldp<W>(g.dinv, i, g.l2pol);
  const double ds = g.dinv_s;
  auto M = [&](double v, int l) { return PM == 1 ? mul_(dv.v[l], v) : (PM == 2 ? mul_(ds, v) : v); };

  if constexpr (KID == EW_HS1) {             // hs_cg.py:118-120
    Pk<W> r = ldp<W>(g.r, i, g.l2pol), s = ldp<W>(g.s, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      red[0] = fma(r.v[l], M(r.v[l], l), red[0]);
    }
    stp<W>(g.r, i, r, g.l2pol);
  } else if constexpr (KID == EW_HS2) {      // hs_cg.py:117,119,122
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      p.v[l] = axpy_(M(r.v[l], l), b, p.v[l]);
    }
    stp<W>(g.x, i, x, g.l2pol); stp<W>(g.p, i, p, g.l2pol);
    halo_store<W>(g, 0, i, p);
  } else if constexpr (KID == EW_CG) {       // cg_cg.py:137-138 (deferred), :130-132
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), rt = ldp<W>(g.rt, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol),
          s = ldp<W>(g.s, i, g.l2pol), w = ldp<W>(g.w, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      p.v[l] = axpy_(rt.v[l], b, p.v[l]);
      s.v[l] = axpy_(w.v[l], b, s.v[l]);
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      rt.v[l] = M(r.v[l], l);
    }
    stp<W>(g.p, i, p, g.l2pol); stp<W>(g.s, i, s, g.l2pol); stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol);
    stp<W>(g.rt, i, rt, g.l2pol);
    halo_store<W>(g, 0, i, rt);
  } else if constexpr (KID == EW_CG_E) {     // EW_CG without the r~ stream (PM 0 / 2 only)
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol), s = ldp<W>(g.s, i, g.l2pol), w = ldp<W>(g.w, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      p.v[l] = axpy_(M(r.v[l], l), b, p.v[l]);          // r~_{k-1} = M r_{k-1}, the bits EW_CG stored
      s.v[l] = axpy_(w.v[l], b, s.v[l]);
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
    }
    stp<W>(g.p, i, p, g.l2pol); stp<W>(g.s, i, s, g.l2pol); stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol);
    halo_store<W>(g, 0, i, r);                           // the stencil pass scales it
  } else if constexpr (KID == EW_GV_E) {     // EW_GV without the w~ stream (PM 0 / 2 only)
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), rt = ldp<W>(g.rt, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol),
          s = ldp<W>(g.s, i, g.l2pol), st = ldp<W>(g.st, i, g.l2pol), w = ldp<W>(g.w, i, g.l2pol), u = ldp<W>(g.u, i, g.l2pol), t = ldp<W>(g.t, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      p.v[l] = axpy_(rt.v[l], b, p.v[l]);
      s.v[l] = axpy_(w.v[l], b, s.v[l]);
      st.v[l] = axpy_(M(w.v[l], l), b, st.v[l]);        // w~_{k-1} = M w_{k-1}, the bits EW_GV stored
      u.v[l] = axpy_(t.v[l], b, u.v[l]);
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      rt.v[l] = axmy_(rt.v[l], a, st.v[l]);
      w.v[l] = axmy_(w.v[l], a, u.v[l]);
      red[0] = fma(r.v[l], rt.v[l], red[0]);
      red[1] = fma(w.v[l], rt.v[l], red[1]);
    }
    stp<W>(g.p, i, p, g.l2pol); stp<W>(g.s, i, s, g.l2pol); stp<W>(g.st, i, st, g.l2pol); stp<W>(g.u, i, u, g.l2pol);
    stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol); stp<W>(g.rt, i, rt, g.l2pol); stp<W>(g.w, i, w, g.l2pol);
    halo_store<W>(g, 0, i, w);                           // the stencil pass scales it
  } else if constexpr (KID == EW_GV) {       // gv_cg.py:165-168 (deferred), :151-154,160,162-163
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), rt = ldp<W>(g.rt, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol),
          s = ldp<W>(g.s, i, g.l2pol), st = ldp<W>(g.st, i, g.l2pol), w = ldp<W>(g.w, i, g.l2pol), wt = ldp<W>(g.wt, i, g.l2pol),
          u = ldp<W>(g.u, i, g.l2pol), t = ldp<W>(g.t, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      p.v[l] = axpy_(rt.v[l], b, p.v[l]);
      s.v[l] = axpy_(w.v[l], b, s.v[l]);
      st.v[l] = axpy_(wt.v[l], b, st.v[l]);
      u.v[l] = axpy_(t.v[l], b, u.v[l]);
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      rt.v[l] = axmy_(rt.v[l], a, st.v[l]);
      w.v[l] = axmy_(w.v[l], a, u.v[l]);
      wt.v[l] = M(w.v[l], l);
      red[0] = fma(r.v[l], rt.v[l], red[0]);
      red[1] = fma(w.v[l], rt.v[l], red[1]);
    }
    stp<W>(g.p, i, p, g.l2pol); stp<W>(g.s, i, s, g.l2pol); stp<W>(g.st, i, st, g.l2pol); stp<W>(g.u, i, u, g.l2pol);
    stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol); stp<W>(g.rt, i, rt, g.l2pol); stp<W>(g.w, i, w, g.l2pol);
    stp<W>(g.wt, i, wt, g.l2pol);
    halo_store<W>(g, 0, i, wt);
  } else if constexpr (KID == EW_PR) {       // pr_cg.py:146-148,151,157
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), rt = ldp<W>(g.rt, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol),
          s = ldp<W>(g.s, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      rt.v[l] = axmy_(rt.v[l], a, M(s.v[l], l));       // st_{k-1} = M s_{k-1} exactly
      p.v[l] = axpy_(rt.v[l], b, p.v[l]);
      red[0] = fma(rt.v[l], r.v[l], red[0]);
    }
    stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol); stp<W>(g.rt, i, rt, g.l2pol); stp<W>(g.p, i, p, g.l2pol);
    halo_store<W>(g, 0, i, p);
  } else {                                   // pipe_pr_cg.py:169-178,183-186
    constexpr bool RECOMP = (KID == EW_PIPE_R);
    Pk<W> x = ldp<W>(g.x, i, g.l2pol), r = ldp<W>(g.r, i, g.l2pol), rt = ldp<W>(g.rt, i, g.l2pol), p = ldp<W>(g.p, i, g.l2pol),
          s = ldp<W>(g.s, i, g.l2pol), st = ldp<W>(g.st, i, g.l2pol), w = ldp<W>(g.w, i, g.l2pol), u = ldp<W>(g.u, i, g.l2pol);
    Pk<W> wt;
    if constexpr (!RECOMP && PREC) wt = ldp<W>(g.wt, i, g.l2pol);
#pragma unroll
    for (int l = 0; l < W; ++l) {
      x.v[l] = axpy_(x.v[l], a, p.v[l]);
      r.v[l] = axmy_(r.v[l], a, s.v[l]);
      rt.v[l] = axmy_(rt.v[l], a, st.v[l]);
      // wt_{k-1}: = M w_{k-1} exactly when w is recomputed every iteration (or M = I),
      // otherwise its own recurrence.  ut_{k-1} = M u_{k-1} always.
      double wt_old;
      if constexpr (!RECOMP && PREC) wt_old = wt.v[l]; else wt_old = M(w.v[l], l);
      const double wn = axmy_(w.v[l], a, u.v[l]);
      const double wtn = axmy_(wt_old, a, M(u.v[l], l));
      p.v[l] = axpy_(rt.v[l], b, p.v[l]);
      s.v[l] = axpy_(wn, b, s.v[l]);
      st.v[l] = axpy_(wtn, b, st.v[l]);
      w.v[l] = wn;
      if constexpr (!RECOMP && PREC) wt.v[l] = wtn;
      red[0] = fma(p.v[l], s.v[l], red[0]);      // mu
      red[1] = fma(r.v[l], st.v[l], red[1]);     // delta
      red[2] = fma(st.v[l], s.v[l], red[2]);     // gamma
      red[3] = fma(rt.v[l], r.v[l], red[3]);     // nu (recomputed)
    }
    stp<W>(g.x, i, x, g.l2pol); stp<W>(g.r, i, r, g.l2pol); stp<W>(g.rt, i, rt, g.l2pol); stp<W>(g.p, i, p, g.l2pol);
    stp<W>(g.s, i, s, g.l2pol); stp<W>(g.st, i, st, g.l2pol);
    halo_store<W>(g, 0, i, st);
    if constexpr (RECOMP) halo_store<W>(g, 1, i, rt);
    if constexpr (!RECOMP) {
      stp<W>(g.w, i, w, g.l2pol);
      if constexpr (PREC) stp<W>(g.wt, i, wt, g.l2pol);
    }
  }
}

template <int KID> struct EwKind { static constexpr int FK = FK_NONE; };
template <> struct EwKind<EW_HS1> { static constexpr int FK = FK_HS_NU; };
template <> struct EwKind<EW_GV> { static constexpr int FK = FK_CGGV; };
template <> struct EwKind<EW_GV_E> { static constexpr int FK = FK_CGGV; };
template <> struct EwKind<EW_PR> { static constexpr int FK = FK_PR_NU; };
template <> struct EwKind<EW_PIPE_R> { static constexpr int FK = FK_PIPE; };
template <> struct EwKind<EW_PIPE_N> { static constexpr int FK = FK_PIPE; };

// L2 prefetch of the operands of element i of stage KID (partitioned runs: issued before the
// CTA folds the all-rank scalar records, so the HBM latency of the first sweep overlaps the
// exchange instead of following it).
template <int KID, int PM>
__device__ __forceinline__ void ew_prefetch(const Args& g, i64 i) {
  auto pf = [&](const double* p) { if (p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + i)); };
  if constexpr (PM == 1) pf(g.dinv);
  pf(g.r);
  if constexpr (KID == EW_HS1) { pf(g.s); }
  else if constexpr (KID == EW_HS2) { pf(g.x); pf(g.p); }
  else {
    pf(g.x); pf(g.p); pf(g.s);
    if constexpr (KID != EW_CG_E) pf(g.rt);
    if constexpr (KID == EW_CG || KID == EW_CG_E) pf(g.w);
    if constexpr (KID == EW_GV) { pf(g.st); pf(g.w); pf(g.wt); pf(g.u); pf(g.t); }
    if constexpr (KID == EW_GV_E) { pf(g.st); pf(g.w); pf(g.u); pf(g.t); }
    if constexpr (KID == EW_PIPE_R || KID == EW_PIPE_N) { pf(g.st); pf(g.w); pf(g.u); }
    if constexpr (KID == EW_PIPE_N && PM != 0) pf(g.wt);
  }
}

template <int KID, int PM, bool MEURANT>
__global__ void __launch_bounds__(kBlock) ew_kernel(const Args g) {
  const bool dist = g.d.world > 1;
  const i64 nv = g.n >> 1;
  const i64 stride = (i64)gridDim.x * kBlock;
  double a, b;
  const bool stamp = (g.dbg & 2) && blockIdx.x == 0 && threadIdx.x == 0;
  pdl_launch_dependents();
  pdl_wait();                          // nothing of the previous kernel's data is touched before this
  if (!dist && after_stop(g)) return;  // (a partition decides after its fold, below)
  if (stamp) g.dbg_t[0] = (u64)clock64();
  if (dist) {
    const i64 rot0 = (g.hout_n > 0 && g.d.has_hi) ? nv - (g.d.plane >> 1) : 0;
    i64 i0 = (i64)blockIdx.x * kBlock + threadIdx.x;
    const bool pf = i0 < nv;
    if (pf) { i0 += rot0; if (i0 >= nv) i0 -= nv; }
    // warps 1..7 prefetch while warp 0 folds the records (its own prefetch follows its loads, so
    // the few record loads are not queued behind the prefetch burst)
    if (pf && threadIdx.x >= 32) ew_prefetch<KID, PM>(g, 2 * i0);
    if (dist_scalars(g, MEURANT, a, b)) return;     // folded and persisted: nothing of this iteration runs
    if (pf && threadIdx.x < 32) ew_prefetch<KID, PM>(g, 2 * i0);
  } else { a = g.sc->a; b = g.sc->b; }
  if (stamp) g.dbg_t[1] = (u64)clock64();
  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};
  // Only the CTAs that stored boundary planes into a peer need a system-scope fence before
  // they take their ticket (a fence.sys in each of ~1200 CTAs costs tens of microseconds).
  bool peer = false;
  const i64 lo_end = g.d.has_lo ? g.d.plane : 0, hi_begin = g.d.has_hi ? g.n - g.d.plane : g.n;
  // Partitioned run: rotate the row order so that the boundary planes (last plane, then first
  // plane) are updated FIRST -- their halo copies then cross NVLink while the interior is
  // still being streamed, and the neighbour's SpMV pass finds them waiting.
  const i64 rot = (dist && g.hout_n > 0 && g.d.has_hi) ? nv - (g.d.plane >> 1) : 0;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < nv; i += stride) {
    i64 ph = i + rot;
    if (ph >= nv) ph -= nv;
    ew_body<KID, PM, 2>(g, 2 * ph, a, b, red);
    peer |= (2 * ph < lo_end) | (2 * ph + 2 > hi_begin);
  }
  if ((g.n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    ew_body<KID, PM, 1>(g, g.n - 1, a, b, red);
    peer = true;
  }
  const bool cta_peer = dist && g.hout_n > 0 && !g.halo_ll && __syncthreads_or(peer ? 1 : 0);
  if (stamp) g.dbg_t[2] = (u64)clock64();

  constexpr int NR = EwTraits<KID>::NR;
  if constexpr (NR > 0) {
    double v[NR];
#pragma unroll
    for (int j = 0; j < NR; ++j) v[j] = red[j];
    grid_sum_finalize<NR>(v, g.partials, g.ticket, [&](const double* acc) {
      if (dist) dist_publish<NR>(g, acc);
      else apply_finalize(EwKind<KID>::FK, MEURANT, g.sc, acc, g.k);
    }, cta_peer);
  } else {
    if (dist && g.hout_n > 0 && !g.halo_ll)
      grid_last_finalize(g.ticket, [&]() { dist_publish<0>(g, nullptr); }, cta_peer);
  }
}

// -------------------------------------------------------------------------------------
// Fused SpMV pass: one sweep over the matrix (or stencil) with the stage's epilogue.
// -------------------------------------------------------------------------------------
template <int MODE> struct SpTraits { static constexpr int NR = 0, FK = FK_NONE, NV = 1; };
template <> struct SpTraits<SP_HS> { static constexpr int NR = 1, FK = FK_HS_MU, NV = 1; };
template <> struct SpTraits<SP_CG> { static constexpr int NR = 2, FK = FK_CGGV, NV = 1; };
template <> struct SpTraits<SP_CG_E> { static constexpr int NR = 2, FK = FK_CGGV, NV = 1; };
template <> struct SpTraits<SP_PR> { static constexpr int NR = 3, FK = FK_PR_SP, NV = 1; };
template <> struct SpTraits<SP_PIPE_R> { static constexpr int NR = 0, FK = FK_NONE, NV = 2; };

// Close a fused SpMV pass: single GPU -> scalar recurrences now; multi-GPU -> publish the
// rank's record (the next vector pass folds all ranks' records).
template <int MODE, bool MEURANT>
__device__ __forceinline__ void spmv_close(const Args& g, double (&red)[kNRed]) {
  constexpr int NR = SpTraits<MODE>::NR;
  if constexpr (NR > 0) {
    const bool dist = g.d.world > 1;
    double v[NR];
#pragma unroll
    for (int j = 0; j < NR; ++j) v[j] = red[j];
    grid_sum_finalize<NR>(v, g.partials, g.ticket, [&](const double* acc) {
      if (dist) dist_publish<NR>(g, acc);
      else apply_finalize(SpTraits<MODE>::FK, MEURANT, g.sc, acc, g.k);
    }, false);
  }
}

// What a fused SpMV pass does with row i once y = (A in0)_i [, (A in1)_i] is known.
// in0 / in1: the SpMV input vector(s) of the stage (p | rt | wt | st [, rt]); for SP_PLAIN
// and SP_RESID any vector.  vout: output of SP_PLAIN / SP_RESID.
template <int MODE, int PM, int NV>
__device__ __forceinline__ void sp_epilogue(const Args& g, const VecIn& in0, i64 i, const double (&y)[NV],
                                            double (&red)[kNRed], double* vout) {
  if constexpr (MODE == SP_PIPE_R) {           // pipe_pr_cg.py:179-182: one matrix pass, 2 RHS
    g.u[i] = y[0];
    g.w[i] = y[NV - 1];
  } else if constexpr (MODE == SP_PLAIN) {     // y = A v
    vout[i] = y[0];
  } else if constexpr (MODE == SP_RESID) {     // r = b - A x0   (e.g. hs_cg.py:84)
    vout[i] = sub_(g.b[i], y[0]);
  } else if constexpr (MODE == SP_HS) {        // hs_cg.py:123-124
    g.s[i] = y[0];
    red[0] = fma(in0.v[i], y[0], red[0]);
  } else if constexpr (MODE == SP_CG_E || MODE == SP_GV_E) {      // TMA stencil kernel only (see cgx_stencil_tma.cuh)
    (void)y;
  } else if constexpr (MODE == SP_CG) {        // cg_cg.py:133-135
    g.w[i] = y[0];
    const double rti = in0.v[i];
    red[0] = fma(g.r[i], rti, red[0]);
    red[1] = fma(y[0], rti, red[1]);
  } else if constexpr (MODE == SP_GV) {        // gv_cg.py:161
    g.t[i] = y[0];
  } else if constexpr (MODE == SP_PR) {        // pr_cg.py:152-156
    g.s[i] = y[0];
    const double sti = PM == 1 ? mul_(g.dinv[i], y[0]) : (PM == 2 ? mul_(g.dinv_s, y[0]) : y[0]);
    red[0] = fma(in0.v[i], y[0], red[0]);
    red[1] = fma(g.r[i], sti, red[1]);
    red[2] = fma(sti, y[0], red[2]);
  } else {                                     // SP_PIPE_N: pipe_pr_cg.py:179-180
    g.u[i] = y[0];
  }
}

// Generic pass: one thread per row (matrix-free stencil without TMA, slabs included).
template <class Op, int MODE, int PM, bool MEURANT>
__global__ void __launch_bounds__(kBlock) spmv_kernel(const Op A, const Args g, const VecIn in0,
                                                     const VecIn in1, double* vout) {
  constexpr bool SL = Op::kSlab;
  constexpr int NV = SpTraits<MODE>::NV;
  if (after_stop(g)) return;
  halo_wait_all(g, NV);
  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};
  const i64 n = g.n, pl = g.d.plane;
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
    double y[NV];
    A.template row<NV>(i, [&](i64 j, double (&v)[NV]) {
      v[0] = vload<SL>(in0, j, n, pl);
      if constexpr (NV == 2) v[1] = vload<SL>(in1, j, n, pl);
    }, y);
    sp_epilogue<MODE, PM, NV>(g, in0, i, y, red, vout);
  }
  spmv_close<MODE, MEURANT>(g, red);
}

// CSR pass ("CSR-stream"): a CTA owns a block of consecutive rows holding at most kCsrCap
// non-zeros (host-built row_blocks).  The whole CTA streams that contiguous range of
// (value, column) pairs with coalesced loads, forms the products a_ij * v_j into shared memory,
// then thread t adds up row t's products IN STORED ORDER -- the matrix is read at full
// width whatever the row lengths (1 .. 81 in matrices/), and the row sums keep scipy's
// csr_matvec rounding exactly.  A row longer than kCsrCap is a block of its own, summed in
// order by one thread chunk after chunk.
constexpr int kCsrCap = 2048;
constexpr int kCsrRows = 223;          // rows per block at most: a loader thread per row extent (rows + 1 of them)

// Warp-specialised: 7 LOADER warps stream a block's (value, column) pairs with coalesced loads -- all of
// a thread's loads in flight at once, then all its gathers --, multiply and store the products into one
// slot of a ring in shared memory, together with the block's row extents and the operands of the fused
// epilogue (SpMV input at the row, r or b, Jacobi entry); 1 SUMMING warp adds up every row's products in
// stored order (lane l: rows l, l+32, ... of the block) and applies the epilogue, all from shared memory.
// Slots are handed over through full / empty mbarriers, so the (latency-bound, few-threads) row sums of
// block k overlap the streaming of blocks k+1, k+2 in the SAME CTA; there is no CTA-wide barrier.
// (History: the one-phase-at-a-time form reached 0.63-0.79 of the HBM peak on the banded model problem
// and 0.45 with two right-hand sides -- ncu: 61 % of the stall samples on the load -> gather chain, 27 % at
// the two barriers around the row sums, which a single warp's worth of threads executed.)
// A row longer than kCsrCap is a block of its own, handed over chunk by chunk.
// GHOST: this launch is a rank of a CSR row partition -- columns >= n address the staging array of gathered
// ghost entries (a pointer select per gather; compiled out for single-GPU runs).
constexpr int kCsrLoaders = kBlock - 32;                       // 224 loader threads
constexpr int kCsrUL = (kCsrCap + kCsrLoaders - 1) / kCsrLoaders;   // elements per loader thread per block
__host__ __device__ constexpr int csr_ring(int nv) { return nv == 2 ? 2 : 3; }
struct CsrSlotMeta { int r0, r1, cnt, last; };                 // rows, products in the slot, last chunk of its block
__host__ __device__ constexpr size_t csr_slot_doubles(int nv) { return (size_t)nv * kCsrCap + 3 * kBlock; }
__host__ __device__ constexpr size_t csr_stream_smem_bytes(int nv) {
  return (size_t)csr_ring(nv) * (csr_slot_doubles(nv) * sizeof(double) + (kBlock + 4) * sizeof(int) + sizeof(CsrSlotMeta));
}

template <int MODE, int PM, bool MEURANT, bool GHOST>
__global__ void __launch_bounds__(kBlock)
csr_stream_kernel(const CsrOp A, const int* __restrict__ row_blocks, const int* __restrict__ blk_e0, int nblocks, const Args g,
                                                           const VecIn in0, const VecIn in1, double* vout) {
  constexpr int NV = SpTraits<MODE>::NV;
  constexpr int S = csr_ring(NV);
  extern __shared__ __align__(16) unsigned char csr_smem[];
  double* sm_d = reinterpret_cast<double*>(csr_smem);                                   // [S][NV*cap + 3*kBlock]
  int* sm_rp = reinterpret_cast<int*>(sm_d + (size_t)S * csr_slot_doubles(NV));         // [S][kBlock + 4] row extents
  CsrSlotMeta* sm_meta = reinterpret_cast<CsrSlotMeta*>(sm_rp + S * (kBlock + 4));      // [S]
  __shared__ __align__(8) uint64_t full_bar[3], empty_bar[3];
  if (after_stop(g)) return;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], kCsrLoaders / 32); mbar_init(&empty_bar[s], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if constexpr (GHOST) halo_wait_all(g, NV);
  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};
  const int nloc = (int)g.n;
  auto ld0 = [&](int cj) { if constexpr (GHOST) return (cj < nloc ? in0.v : in0.lo - nloc)[cj]; else return in0.v[cj]; };
  auto ld1 = [&](int cj) { if constexpr (GHOST) return (cj < nloc ? in1.v : in1.lo - nloc)[cj]; else return in1.v[cj]; };
  constexpr bool kEpP = (MODE == SP_HS || MODE == SP_CG || MODE == SP_PR);
  constexpr bool kEpR = (MODE == SP_CG || MODE == SP_PR || MODE == SP_RESID);
  constexpr bool kEpD = (MODE == SP_PR && PM == 1);

  if (tid < kCsrLoaders) {
    // ------------------------------------------------------------------ loader warps
    // Work items = (row block, chunk) in launch order.  The (value, column) loads of item i+1 are issued
    // BEFORE item i is gathered / multiplied / handed over (two alternating register sets), so that each
    // loader thread keeps two blocks' worth of the matrix stream in flight.
    // Block metadata (rows and first non-zero of the block: row_blocks / blk_e0, host-built) is fetched TWO
    // blocks ahead, so that neither the stream loads nor the gathers ever wait on a pointer chase.
    struct Item { int blk, base, r0, r1, e0, total; bool ok; };
    auto load_meta = [&](int blk) {
      Item t{blk, 0, 0, 0, 0, 0, blk < nblocks};
      if (t.ok) {
        t.r0 = __ldg(row_blocks + blk); t.r1 = __ldg(row_blocks + blk + 1);
        t.e0 = __ldg(blk_e0 + blk); t.total = __ldg(blk_e0 + blk + 1) - t.e0;
      }
      return t;
    };
    Item ahead = load_meta((int)blockIdx.x + (int)gridDim.x);
    auto first_item = [&]() { return load_meta((int)blockIdx.x); };
    auto next_item = [&](const Item& c) {
      Item t = c;
      if (c.base + kCsrCap < c.total) { t.base = c.base + kCsrCap; return t; }
      t = ahead;
      ahead = load_meta(t.blk + (int)gridDim.x);
      return t;
    };
    struct Regs { double a[kCsrUL]; int col[kCsrUL]; };
    auto issue = [&](const Item& t, Regs& R) {
      const int cnt = min(kCsrCap, t.total - t.base);
#pragma unroll
      for (int u = 0; u < kCsrUL; ++u) {
        const int j = tid + u * kCsrLoaders;
        const bool ok = j < cnt;
        R.a[u] = ok ? __ldg(A.val + t.e0 + t.base + j) : 0.0;
        R.col[u] = ok ? __ldg(A.idx + t.e0 + t.base + j) : t.r0;
      }
    };
    uint32_t it = 0;
    auto process = [&](const Item& t, Regs& R) {
      const int cnt = min(kCsrCap, t.total - t.base);
      const int slot = it % S;
      double x0v[kCsrUL], x1v[kCsrUL];
#pragma unroll
      for (int u = 0; u < kCsrUL; ++u) {
        x0v[u] = ld0(R.col[u]);
        if constexpr (NV == 2) x1v[u] = ld1(R.col[u]); else x1v[u] = 0.0;
      }
      // row extent and epilogue operands of this thread's row of the block (first chunk only): fetched
      // with the gathers (same round trip)
      const int row = t.r0 + tid;
      const bool hasrow = t.base == 0 && row <= t.r1;
      int rp = 0;
      double pv = 0.0, rv = 0.0, dv = 0.0;
      if (hasrow) {
        rp = __ldg(A.ptr + row) - t.e0;
        if (row < t.r1) {
          if constexpr (kEpP) pv = in0.v[row];
          if constexpr (kEpR) rv = (MODE == SP_RESID) ? g.b[row] : g.r[row];
          if constexpr (kEpD) dv = g.dinv[row];
        }
      }
      if (it >= (uint32_t)S) mbar_wait(&empty_bar[slot], ((it / S) - 1) & 1u, g.errflag);
      double* prod = sm_d + (size_t)slot * csr_slot_doubles(NV);
      double* ep = prod + (size_t)NV * kCsrCap;                  // [3][kBlock]: pv, rv, dv
      int* rps = sm_rp + slot * (kBlock + 4);
#pragma unroll
      for (int u = 0; u < kCsrUL; ++u) {
        const int j = tid + u * kCsrLoaders;
        if (j < cnt) {
          prod[j] = mul_(R.a[u], x0v[u]);
          if constexpr (NV == 2) prod[kCsrCap + j] = mul_(R.a[u], x1v[u]);
        }
      }
      if (hasrow) { rps[tid] = rp; ep[tid] = pv; ep[kBlock + tid] = rv; ep[2 * kBlock + tid] = dv; }
      if (tid == 0) sm_meta[slot] = CsrSlotMeta{t.r0, t.r1, cnt, t.base + kCsrCap >= t.total ? 1 : 0};
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(&full_bar[slot]);
      ++it;
    };
    Regs RA, RB;
    Item ia = first_item(), ib;
    if (ia.ok) issue(ia, RA);
    while (ia.ok) {
      ib = next_item(ia);
      if (ib.ok) issue(ib, RB);
      process(ia, RA);
      if (!ib.ok) break;
      ia = next_item(ib);
      if (ia.ok) issue(ia, RA);
      process(ib, RB);
    }
  } else {
    // ------------------------------------------------------------------ summing warp
    const int lane = tid - kCsrLoaders;
    uint32_t it = 0;
    double ylong[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) ylong[c] = 0.0;
    for (int blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
      const int total = __ldg(blk_e0 + blk + 1) - __ldg(blk_e0 + blk);
      for (int base = 0; base == 0 || base < total; base += kCsrCap, ++it) {
        const int slot = it % S;
        mbar_wait(&full_bar[slot], (it / S) & 1u, g.errflag);
        const double* prod = sm_d + (size_t)slot * csr_slot_doubles(NV);
        const double* ep = prod + (size_t)NV * kCsrCap;
        const int* rps = sm_rp + slot * (kBlock + 4);
        const CsrSlotMeta m = sm_meta[slot];
        auto epilogue = [&](int row, int t, const double (&y)[NV]) {     // same statements as sp_epilogue
          const double pv = ep[t], rv = ep[kBlock + t], dv = ep[2 * kBlock + t];
          if constexpr (MODE == SP_PIPE_R) { g.u[row] = y[0]; g.w[row] = y[NV - 1]; }
          else if constexpr (MODE == SP_PLAIN) vout[row] = y[0];
          else if constexpr (MODE == SP_RESID) vout[row] = sub_(rv, y[0]);
          else if constexpr (MODE == SP_HS) { g.s[row] = y[0]; red[0] = fma(pv, y[0], red[0]); }
          else if constexpr (MODE == SP_CG) { g.w[row] = y[0]; red[0] = fma(rv, pv, red[0]); red[1] = fma(y[0], pv, red[1]); }
          else if constexpr (MODE == SP_GV) g.t[row] = y[0];
          else if constexpr (MODE == SP_PR) {
            g.s[row] = y[0];
            const double sti = PM == 1 ? mul_(dv, y[0]) : (PM == 2 ? mul_(g.dinv_s, y[0]) : y[0]);
            red[0] = fma(pv, y[0], red[0]);
            red[1] = fma(rv, sti, red[1]);
            red[2] = fma(sti, y[0], red[2]);
          } else g.u[row] = y[0];                                  // SP_PIPE_N
          (void)pv; (void)rv; (void)dv;
        };
        if (total <= kCsrCap) {
          for (int t = lane; t < m.r1 - m.r0; t += 32) {
            const int b0 = rps[t], b1 = rps[t + 1];
            double y[NV];
#pragma unroll
            for (int c = 0; c < NV; ++c) y[c] = 0.0;
            // products fetched eight at a time (independent shared-memory loads), then added in stored
            // order: the chain the hardware must serialise is the additions only
            int j = b0;
            for (; j + 8 <= b1; j += 8) {
              double t8[NV][8];
#pragma unroll
              for (int c = 0; c < NV; ++c)
#pragma unroll
                for (int q = 0; q < 8; ++q) t8[c][q] = prod[c * kCsrCap + j + q];
#pragma unroll
              for (int q = 0; q < 8; ++q)
#pragma unroll
                for (int c = 0; c < NV; ++c) y[c] = add_(y[c], t8[c][q]);
            }
            for (; j < b1; ++j) {
#pragma unroll
              for (int c = 0; c < NV; ++c) y[c] = add_(y[c], prod[c * kCsrCap + j]);
            }
            epilogue(m.r0 + t, t, y);
          }
        } else {                                                   // one long row, chunk by chunk, in order
          if (lane == 0) {
            for (int j = 0; j < m.cnt; ++j) {
#pragma unroll
              for (int c = 0; c < NV; ++c) ylong[c] = add_(ylong[c], prod[c * kCsrCap + j]);
            }
            if (m.last) {
              // (the operands of the first chunk's slot are gone: fetch them here, once per long row)
              double pv = 0.0, rv = 0.0, dv = 0.0;
              if constexpr (kEpP) pv = in0.v[m.r0];
              if constexpr (kEpR) rv = (MODE == SP_RESID) ? g.b[m.r0] : g.r[m.r0];
              if constexpr (kEpD) dv = g.dinv[m.r0];
              const int row = m.r0;
              if constexpr (MODE == SP_PIPE_R) { g.u[row] = ylong[0]; g.w[row] = ylong[NV - 1]; }
              else if constexpr (MODE == SP_PLAIN) vout[row] = ylong[0];
              else if constexpr (MODE == SP_RESID) vout[row] = sub_(rv, ylong[0]);
              else if constexpr (MODE == SP_HS) { g.s[row] = ylong[0]; red[0] = fma(pv, ylong[0], red[0]); }
              else if constexpr (MODE == SP_CG) { g.w[row] = ylong[0]; red[0] = fma(rv, pv, red[0]); red[1] = fma(ylong[0], pv, red[1]); }
              else if constexpr (MODE == SP_GV) g.t[row] = ylong[0];
              else if constexpr (MODE == SP_PR) {
                g.s[row] = ylong[0];
                const double sti = PM == 1 ? mul_(dv, ylong[0]) : (PM == 2 ? mul_(g.dinv_s, ylong[0]) : ylong[0]);
                red[0] = fma(pv, ylong[0], red[0]);
                red[1] = fma(rv, sti, red[1]);
                red[2] = fma(sti, ylong[0], red[2]);
              } else g.u[row] = ylong[0];
              (void)pv; (void)rv; (void)dv;
#pragma unroll
              for (int c = 0; c < NV; ++c) ylong[c] = 0.0;
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[slot]);
      }
    }
  }
  spmv_close<MODE, MEURANT>(g, red);
}

// -------------------------------------------------------------------------------------
// Instrumentation = the four standard callbacks in one matrix pass (callbacks/*.py):
//   e = x - x_true ; error_A_norm = sqrt(e.(A e)) ; residual_2_norm = ||b - A x|| ;
//   error_2_norm = ||e|| ; updated_residual_2_norm = ||r||.
// Excluded from the roofline traffic model (SURVEY.md section 8d).
// Multi-GPU: xin / xtin carry the ghost planes of x (channel hin_ch) and x_true
// (channel 3, exchanged once when the problem is loaded); the record is published and
// hist_consume_kernel writes the history entry.
// -------------------------------------------------------------------------------------
template <class Op, bool HAS_XTRUE>
__global__ void __launch_bounds__(kBlock) instrument_kernel(const Op A, const Args g, const VecIn xin,
                                                           const VecIn xtin) {
  constexpr bool SL = Op::kSlab;
  if (after_stop(g)) return;
  if (HAS_XTRUE && g.d.world > 1 && threadIdx.x == 0 && g.d.csr) {
    csr_wait_channel(g, 3, g.xt_par, g.xt_epoch);
  } else if (HAS_XTRUE && g.d.world > 1 && threadIdx.x == 0) {
    WinHdr* w = g.d.win[g.d.rank];
    if (g.d.has_lo) wait_epoch(&w->hflag[3][g.xt_par][0], g.xt_epoch, &w->error);
    if (g.d.has_hi) wait_epoch(&w->hflag[3][g.xt_par][1], g.xt_epoch, &w->error);
  }
  halo_wait_all(g, 1);
  double red[4] = {0.0, 0.0, 0.0, 0.0};
  const i64 n = g.n, pl = g.d.plane;
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
    double y[2] = {0.0, 0.0};
    if constexpr (HAS_XTRUE) {
      A.template row<2>(i, [&](i64 j, double (&v)[2]) {
        v[0] = vload<SL>(xin, j, n, pl); v[1] = sub_(v[0], vload<SL>(xtin, j, n, pl)); }, y);
      const double e = sub_(g.x[i], g.xtrue[i]);
      red[0] = fma(e, y[1], red[0]);
      red[2] = fma(e, e, red[2]);
    } else {
      double y1[1];
      A.template row<1>(i, [&](i64 j, double (&v)[1]) { v[0] = vload<SL>(xin, j, n, pl); }, y1);
      y[0] = y1[0];
    }
    const double res = sub_(g.b[i], y[0]);
    red[1] = fma(res, res, red[1]);
    const double ri = g.r[i];
    red[3] = fma(ri, ri, red[3]);
  }
  const bool dist = g.d.world > 1;
  grid_sum_finalize<4>(red, g.partials, g.ticket, [&](const double* acc) {
    if (dist) { dist_publish<4>(g, acc); return; }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (g.hist_mask & (1u << j)) g.hist[(i64)j * g.hist_len + g.k] = sqrt(acc[j]);
  });
}

// multi-GPU: fold all ranks' instrumentation records of epoch pend_e[0] into history entry k
static __global__ void hist_consume_kernel(const Args g) {
  if (after_stop(g)) return;           // (its record was never published)
  double acc[kNRed];
  dist_totals(g, g.pend_e[0], 4, acc);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (g.hist_mask & (1u << j)) g.hist[(i64)j * g.hist_len + g.k] = sqrt(acc[j]);
  }
}

// multi-GPU: fold the pending reductions into the persisted scalars (end of cgx_advance)
static __global__ void flush_scalars_kernel(const Args g) {
  double a, b;
  dist_scalars(g, g.meur != 0, a, b);
}

// multi-GPU: copy the first / last plane of v into the neighbours' ghost planes of channel
// hout_ch (initialisation SpMVs, instrumentation x, x_true) and publish the halo epoch.
static __global__ void __launch_bounds__(kBlock) halo_push_kernel(const Args g, const double* __restrict__ v) {
  if (after_stop(g)) return;
  const i64 pl = g.d.plane;
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < pl; i += stride) {
    if (g.d.has_lo) g.d.ghost_lo[ghost_off(g.d, g.hout_ch, g.hout_par, 1) + i] = v[i];
    if (g.d.has_hi) g.d.ghost_hi[ghost_off(g.d, g.hout_ch, g.hout_par, 0) + i] = v[g.n - pl + i];
  }
  grid_last_finalize(g.ticket, [&]() { dist_publish<0>(g, nullptr); });
}

// CSR row partition: gather the entries of v the other ranks need and store them into their staging
// arrays (channel hout_ch, parity hout_par), then publish the epoch to every destination.
static __global__ void __launch_bounds__(kBlock) csr_halo_push_kernel(const Args g, const double* __restrict__ v) {
  if (after_stop(g)) return;
  const int total = g.d.send_ptr[g.d.world];
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < total; i += stride) {
    int q = 0;
    while ((int)i >= g.d.send_ptr[q + 1]) ++q;
    double* dst = g.d.stage_of[q] + (size_t)(g.hout_ch * 2 + g.hout_par) * (size_t)g.d.nghost_of[q] + g.d.send_off[q] +
                  ((int)i - g.d.send_ptr[q]);
    *dst = v[g.d.send_idx[i]];
  }
  grid_last_finalize(g.ticket, [&]() {
    for (int q = 0; q < g.d.world; ++q)
      if (g.d.send_ptr[q + 1] > g.d.send_ptr[q]) st_relaxed_sys(&g.d.win[q]->gflag[g.hout_ch][g.hout_par][g.d.rank], g.hout_epoch);
  });
}

// -------------------------------------------------------------------------------------
// Small helpers used only by the (non-timed) initialisation.
// -------------------------------------------------------------------------------------
// stop != nullptr: a step of GV residual replacement at iteration k (nothing to do after the stop)
static __global__ void __launch_bounds__(kBlock) scale_kernel(const double* __restrict__ dinv,
                                                      const double* __restrict__ v,
                                                      double* __restrict__ out, i64 n,
                                                      const Scal* stop, int k) {
  if (stop && past_stop(stop, k)) return;
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride)
    out[i] = dinv ? mul_(dinv[i], v[i]) : v[i];
}

// sc->tmp[slot] = u . (dinv ? dinv*v : v)   (multi-GPU: the rank's partial)
static __global__ void __launch_bounds__(kBlock) dot_kernel(const double* __restrict__ u,
                                                    const double* __restrict__ v,
                                                    const double* __restrict__ dinv, i64 n,
                                                    Scal* sc, int slot, double* partials,
                                                    unsigned* ticket, const Scal* stop, int k) {
  if (stop && past_stop(stop, k)) return;
  double red[1] = {0.0};
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
    const double vi = dinv ? mul_(dinv[i], v[i]) : v[i];
    red[0] = fma(u[i], vi, red[0]);
  }
  grid_sum_finalize<1>(red, partials, ticket, [=](const double* acc) { sc->tmp[slot] = acc[0]; });
}

// capture of the scalars after iteration k: out[0][k] = a, out[1][k] = b
static __global__ void capture_scalars_kernel(const Scal* sc, double* out, int k, int len, int tol_on) {
  if (tol_on && past_stop(sc, k)) return;
  if (threadIdx.x == 0) { out[k] = sc->a; out[len + k] = sc->b; }
}
// GV residual replacement (gv_cg.py:156-158, then :162-170 with the new w): eta was re-formed from the
// replaced w (tmp[5]); nu, nu1, b are those of the vector pass
static __global__ void gv_refinalize_kernel(Scal* sc, int k, int tol_on) {
  if (threadIdx.x != 0 || (tol_on && past_stop(sc, k))) return;
  const double eta = sc->tmp[5];
  sc->eta = eta;
  sc->mu = sub_(eta, mul_(div_(sc->b, sc->a1), sc->nu));
  sc->a = div_(sc->nu, sc->mu);
  note_breakdown(sc, k, sc->a, sc->b);
}

// multi-GPU: publish the rank's eight initialisation partials (tmp[0..7]) as epoch sepoch
static __global__ void push_tmp_kernel(const Args g) {
  if (threadIdx.x != 0) return;
  const Scal* sc = g.sc + g.scpar;
  const int slot = (int)(g.sepoch % kSlots);
  if (g.d.mode == 1 || g.d.mode == 3) {
    for (int r = 0; r < g.d.world; ++r) {
      if (g.d.mode == 3 && r != g.d.rank) continue;
      u64* dst = g.d.win[r]->ll[slot][g.d.rank];
      for (int j = 0; j < kSumW; ++j) ll_store(dst + 2 * j, sc->tmp[j], g.sepoch);
    }
  } else {
    volatile double* dst = g.d.nccl_in + (size_t)slot * kSumW;
    for (int j = 0; j < kSumW; ++j) dst[j] = sc->tmp[j];
  }
}

// Initial scalars from the initialisation dots.  tmp: 0 nu, 1 mu, 2 eta, 3 delta, 4 gamma.
// variant_class: 0 HS, 1 CG/GV (mu := p.s), 2 PR/M/pipe (predict first beta).
// Multi-GPU (g.d.world > 1): tmp[] first becomes the all-rank total of epoch pend_e[0].
// tol > 0: the relative tolerance of cgx_set_tolerance (threshold tol^2 nu_0); 0: none.
static __global__ void init_scalars_kernel(const Args g, int variant_class, int meurant, double tol) {
  if (threadIdx.x != 0) return;
  Scal* sc = g.sc + g.scpar;
  if (g.d.world > 1) {
    const int slot = (int)(g.pend_e[0] % kSlots);
    double acc[kSumW];
    for (int j = 0; j < kSumW; ++j) acc[j] = 0.0;
    if (g.d.mode == 1) {
      WinHdr* w = g.d.win[g.d.rank];
      for (int r = 0; r < g.d.world; ++r)
        for (int j = 0; j < kSumW; ++j) acc[j] += ll_load(w->ll[slot][r], j, g.pend_e[0], &w->error);
    } else if (g.d.mode == 3) {
      WinHdr* w = g.d.win[g.d.rank];
      for (int j = 0; j < kSumW; ++j)
        acc[j] = ll_load(w->ll[slot][g.d.rank], j, g.pend_e[0], &w->error) * (double)g.d.world;
    } else {
      for (int j = 0; j < kSumW; ++j) acc[j] = __ldcv(g.d.nccl_out + (size_t)slot * kSumW + j);
    }
    for (int j = 0; j < kSumW; ++j) sc->tmp[j] = acc[j];
  }
  const double nu = sc->tmp[0], mu = sc->tmp[1];
  sc->nu = nu; sc->nu1 = nu; sc->mu = mu; sc->eta = sc->tmp[2];
  sc->del = sc->tmp[3]; sc->gam = sc->tmp[4];
  sc->a1 = 0.0;
  sc->a = div_(nu, mu);
  sc->b = 0.0;
  sc->breakdown = -1;
  sc->stop_k = -1;
  g.sc[g.scpar ^ 1].stop_k = -1;       // (a partition's other parity: no stale stop of an earlier run)
  sc->thr = tol > 0.0 ? mul_(mul_(tol, tol), nu) : nan("");
  if (variant_class == 2) sc->b = predict_beta(meurant != 0, nu, sc->a, sc->del, sc->gam);
  note_breakdown(sc, 0, sc->a, sc->b);
}

}  // namespace cgx
