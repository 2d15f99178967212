// cgx_launch.cuh -- launchers of the fused vector passes and fused SpMV passes (templates;
// instantiated per preconditioner mode in cgx_iter.cu, and for the plain modes in cgx.cu).
#pragma once
#include "cgx_host.h"

// which state vector a fused SpMV pass reads (second one for the 2-RHS pass)
template <int MODE> struct SpInput { static constexpr int v0 = -1, v1 = -1; };
template <> struct SpInput<SP_HS> { static constexpr int v0 = V_P, v1 = -1; };
template <> struct SpInput<SP_PR> { static constexpr int v0 = V_P, v1 = -1; };
template <> struct SpInput<SP_CG> { static constexpr int v0 = V_RT, v1 = -1; };
template <> struct SpInput<SP_CG_E> { static constexpr int v0 = V_R, v1 = -1; };
template <> struct SpInput<SP_GV_E> { static constexpr int v0 = V_W, v1 = -1; };
template <> struct SpInput<SP_GV> { static constexpr int v0 = V_WT, v1 = -1; };
template <> struct SpInput<SP_PIPE_R> { static constexpr int v0 = V_ST, v1 = V_RT; };
template <> struct SpInput<SP_PIPE_N> { static constexpr int v0 = V_ST, v1 = -1; };


// CSR pass through csr_bulk_kernel: the ring takes what `csr_bulk_ctas` resident CTAs per SM leave of the SM's
// shared memory (1 KB per CTA is the system's, ~2 KB static: barriers, slot metadata, reduction scratch).
template <int MODE, int PM, bool MEUR, bool GHOST>
static void launch_csr_bulk(cgx_ctx* c, const Args& g, const VecIn& in0, const VecIn& in1, double* vout) {
  constexpr int nv = SpTraits<MODE>::NV;
  const size_t slot = cb_slot_bytes(nv, cb_ops(MODE, PM));
  const size_t per_cta = (size_t)c->smem_per_sm / (size_t)c->csr_bulk_ctas - 1024 - 2560;
  int ring = c->csr_bulk_ring > 0 ? c->csr_bulk_ring : (int)(per_cta / slot);
  ring = std::max(3, std::min(ring, (int)kCbMaxRing));       // (the gather warps work three items deep)
  const size_t sm = (size_t)ring * slot + 128;
  // (summing warps <= ring: a warp may only wait for the NEXT phase of a slot's barriers)
  const int threads = kCbSum0 + 32 * std::max(1, std::min(std::min(c->csr_bulk_sum, (int)kCbMaxSum), ring));
  const int per_sm = ctx_occupancy(c, (const void*)csr_bulk_kernel<MODE, PM, MEUR, GHOST>, threads, sm);
  const int grid = std::max(1, std::min(c->n_rowblk_b, c->sm_count * per_sm));
  csr_bulk_kernel<MODE, PM, MEUR, GHOST><<<grid, threads, sm, c->stream>>>(c->csr, c->d_rowblk_b, c->d_rowblk_b_e0, c->n_rowblk_b, ring,
                                                                            g, in0, in1, vout);
}

// TMA-staged pass of the variable-coefficient stencil (cgx_varstencil.cuh): one resident wave of
// (column, z-chunk) work units, as for stencil_tma_kernel.  tm0 / tm1: the vector(s) the pass reads.
template <int MODE, int PM, bool MEUR>
static void launch_varstencil_tma(cgx_ctx* c, Args g, const CUtensorMap& tm0, const CUtensorMap& tm1) {
  constexpr int nv = NV_OF(MODE);
  const size_t sm = varstencil_smem_bytes(nv);
  const int per_sm = ctx_occupancy(c, (const void*)varstencil_tma_kernel<MODE, PM, MEUR>, kSThreads, sm);
  TmaGeom G = c->geom;
  const int cap = per_sm * c->sm_count, ncols = G.ntx * G.nty;
  G.nchunk = std::max(1, std::min(cap / std::max(1, ncols), G.nz / std::max(1, c->tma_min_planes)));
  const int grid = (int)std::min<i64>((i64)ncols * G.nchunk, cap);
  // (2-D: no cz map; the kernel never reads its third coefficient map then)
  const CUtensorMap& tcz = c->vsten.cz ? c->coef_tmap[2] : c->coef_tmap[0];
  launch_k(varstencil_tma_kernel<MODE, PM, MEUR>, grid, kSThreads, sm, c->stream, use_pdl(c),
           tm0, tm1, c->coef_tmap[0], c->coef_tmap[1], tcz, c->vsten, G, g);
}

// Fused SpMV pass of stage MODE (vin/vout only for SP_PLAIN / SP_RESID).
template <int MODE, int PM, bool MEUR>
static void launch_spmv(cgx_ctx* c, Args g, const double* vin, double* vout) {
  constexpr int v0 = SpInput<MODE>::v0, v1 = SpInput<MODE>::v1;
  constexpr int nv = (v1 >= 0) ? 2 : 1;
  Plan p;
  p.produce = SpTraits<MODE>::FK;
  p.hin_n = nv; p.hin_ch = 0;
  plan_apply(c, g, p);
  {
    ProfScope ps(c, PC_SP0 + (MODE == SP_CG_E ? (int)SP_CG : MODE == SP_GV_E ? (int)SP_GV : MODE));
    bool done = false;
    if constexpr (v0 >= 0) {
      if (c->op_kind == 2 && c->use_tma && c->tmap_ok[v0] && (v1 < 0 || c->tmap_ok[v1 < 0 ? 0 : v1])) {
        // grid = the CTAs that are actually co-resident (one wave): the kernel splits the work
        // evenly over gridDim.x, so a partial second wave would cost a full extra pass
        const int per_sm = ctx_occupancy(c, (const void*)stencil_tma_kernel<MODE, PM, MEUR>, kSThreads, tma_smem_bytes(nv));
        // (column, z-chunk) work units, all co-resident when the columns fit (cgx_stencil_tma.cuh)
        TmaGeom G = c->geom;
        const int cap = per_sm * c->sm_count, ncols = G.ntx * G.nty;
        G.nchunk = std::max(1, std::min(cap / std::max(1, ncols), G.nz / std::max(1, c->tma_min_planes)));
        const int tgrid = (int)std::min<i64>((i64)ncols * G.nchunk, cap);
        g.gscr = c->d_gscr;
        launch_k(stencil_tma_kernel<MODE, PM, MEUR>, tgrid, kSThreads, tma_smem_bytes(nv), c->stream, use_pdl(c),
                 c->tmap[v0], c->tmap[v1 < 0 ? v0 : v1], G, g);
        done = true;
      } else if constexpr (MODE != SP_CG_E && MODE != SP_GV_E) {
        if (c->op_kind == 3 && c->use_tma && c->coef_tmap_ok && c->tmap_ok[v0] && (v1 < 0 || c->tmap_ok[v1 < 0 ? 0 : v1])) {
          launch_varstencil_tma<MODE, PM, MEUR>(c, g, c->tmap[v0], c->tmap[v1 < 0 ? v0 : v1]);
          done = true;
        }
      }
    }
    if (!done) {
      const double* a0 = v0 >= 0 ? c->vec[v0 < 0 ? 0 : v0] : vin;
      const double* a1 = v1 >= 0 ? c->vec[v1 < 0 ? 0 : v1] : nullptr;
      const VecIn in0 = vec_in(c, a0, 0, g), in1 = vec_in(c, a1, 1, g);
      if (c->op_kind == 1) {
        // (the two-right-hand-side pass stays on csr_stream_kernel unless csr_bulk = 2: measured 138 vs 121 us per pass)
        if (!c->no_csr_stream && (c->csr_bulk >= 2 || (c->csr_bulk == 1 && nv == 1))) {
          if (csr_dist(c)) launch_csr_bulk<MODE, PM, MEUR, true>(c, g, in0, in1, vout);
          else launch_csr_bulk<MODE, PM, MEUR, false>(c, g, in0, in1, vout);
        } else if (!c->no_csr_stream) {
          const size_t sm = csr_stream_smem_bytes(nv);
          if (csr_dist(c)) {
            const int per_sm = ctx_occupancy(c, (const void*)csr_stream_kernel<MODE, PM, MEUR, true>, kBlock, sm);
            const int grid1 = std::max(1, std::min(c->n_rowblk, c->sm_count * per_sm));
            csr_stream_kernel<MODE, PM, MEUR, true><<<grid1, kBlock, sm, c->stream>>>(c->csr, c->d_rowblk, c->d_rowblk_e0, c->n_rowblk, g, in0, in1, vout);
          } else {
            const int per_sm = ctx_occupancy(c, (const void*)csr_stream_kernel<MODE, PM, MEUR, false>, kBlock, sm);
            const int grid1 = std::max(1, std::min(c->n_rowblk, c->sm_count * per_sm));
            csr_stream_kernel<MODE, PM, MEUR, false><<<grid1, kBlock, sm, c->stream>>>(c->csr, c->d_rowblk, c->d_rowblk_e0, c->n_rowblk, g, in0, in1, vout);
          }
        } else {
          spmv_kernel<CsrOp, MODE, PM, MEUR><<<grid_for(c, c->n), kBlock, 0, c->stream>>>(c->csr, g, in0, in1, vout);
        }
      } else if (c->op_kind == 3) {
        spmv_kernel<VarStencilOp, MODE, PM, MEUR><<<grid_for(c, c->n), kBlock, 0, c->stream>>>(c->vsten, g, in0, in1, vout);
      } else {
        spmv_kernel<StencilOp, MODE, PM, MEUR><<<grid_for(c, c->n), kBlock, 0, c->stream>>>(c->sten, g, in0, in1, vout);
      }
    }
    c->launches++;
  }
  plan_commit(c, g, p);
}

template <int KID, int PM, bool MEUR>
static void launch_ew(cgx_ctx* c, Args g) {
  Plan p;
  p.consume = true;
  p.produce = EwKind<KID>::FK;
  p.hout_ch = 0;
  p.hout_n = (KID == EW_HS1) ? 0 : (KID == EW_PIPE_R ? 2 : 1);
  if (csr_dist(c)) p.hout_n = 0;      // CSR row partition: the ghost entries are gathered by a stage of their own
  plan_apply(c, g, p);
  {
    // One resident wave: on a partition every CTA folds the all-rank records before it streams
    // (2-4 us); with 1184 CTAs at 3 resident per SM that prologue was paid by three successive
    // waves (+10 us per launch, found with the in-kernel clock stamps).  Grid-stride covers the rows.
    const int per_sm = ctx_occupancy(c, (const void*)ew_kernel<KID, PM, MEUR>, kBlock, 0);
    int grid = grid_for(c, (c->n + 1) / 2);
    // (one GPU: measured neutral to slightly negative for the long passes, -4 % per iteration
    // for HS-CG's two short ones -- tools/onewave_probe.py)
    if (c->dist.world > 1 || c->one_wave || KID == EW_HS1 || KID == EW_HS2) grid = std::min(grid, per_sm * c->sm_count);
    ProfScope ps(c, PC_EW0 + (KID == EW_CG_E ? (int)EW_CG : KID == EW_GV_E ? (int)EW_GV : KID));
    launch_k(ew_kernel<KID, PM, MEUR>, grid, kBlock, 0, c->stream, use_pdl(c), g);
    c->launches++;
  }
  plan_commit(c, g, p);
}
