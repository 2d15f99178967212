// cgx_stencil_fused.cuh -- PR-CG / M-CG: ONE launch per iteration on the matrix-free stencil.
//
// The two dependency stages of pr_cg.py:146-158 (vector updates, then s = A p with its dots)
// are separated only by the halo of p: s_i needs the NEW p at the six neighbours of i.  This
// kernel recomputes p on that halo instead of going through HBM:
//
//   plane step zz (a CTA owns a kTX x kTY column and marches in z, as cgx_stencil_tma.cuh):
//     stage 1   p_old, s_old, rt_old of plane zz -- tile + one-point xy halo -- arrive by three
//               bulk-tensor copies (TMA, one mbarrier); on the tile:   x += a p ; r -= a s ;
//               rt -= a M s ; p = rt + b p  (+ nu = rt.r), on the halo only rt and p; the new p
//               plane stays in shared memory (ring of 4 planes);
//     stage 2   s = A p for plane zz-1 from the ring planes zz-2, zz-1, zz  (+ mu, delta, gamma)
//
//   HBM words per row: read x, r, p, s, rt; write x, r, p, s, rt = 10 (two-kernel path: 12),
//   one launch, one fused reduction {mu, delta, gamma, nu} per iteration.
//
// p, s and rt are read on the halo while other CTAs write them, so they are ping-pong buffered
// (read `cur`, write `nxt`); x and r are touched by their owner only and stay in place.
//
// Warp-specialised: warp 8 is the TMA producer (one elected lane, per-stage full/empty
// mbarriers, runs up to kFStages planes ahead and across column changes); warps 0-7 compute.
// The only CTA-level synchronisation is one 256-thread named barrier per plane (the new p
// plane is exchanged between threads through shared memory).
//
// Arithmetic: every elementwise product/sum and every row sum is the same separately rounded
// operation, in the same order, as ew_kernel<EW_PR> followed by stencil_tma_kernel<SP_PR>, so the
// state vectors after an iteration are bit-identical to the two-kernel path given the same
// (a, b); only the summation order of the four dots differs (deterministic).
#pragma once
#include "cgx_stencil_tma.cuh"

namespace cgx {

constexpr int kFStages = 2;                       // TMA input stages (3 planes each)
constexpr int kFRing = 4;                         // planes of new p kept in shared memory
constexpr int kFConsumers = 256;                  // 8 compute warps: warp w <-> row w of the tile
constexpr int kFThreads = kFConsumers + 32;       // + 1 producer warp
constexpr int kFPairs = kTX / 64;                 // a lane owns the point pairs (2 lx, 2 lx + 1) + 64 j

__host__ __device__ constexpr size_t fused_smem_bytes() {
  return (size_t)(kFStages * 3 + kFRing) * kPlaneStride * sizeof(double) + 128;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ double2 lds2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ void sts2(double* p, double a, double b) { *reinterpret_cast<double2*>(p) = make_double2(a, b); }

// PM: 0 identity, 2 Jacobi with a constant diagonal (a Jacobi VECTOR would need dinv on the halo:
// those runs keep the two-kernel path).
// DIST: this launch is one rank of a z-slab partition (cgx_common.cuh "Row-partitioned ..."): alpha and
// beta come from folding all ranks' records of the previous launch; the three input vectors of
// the ghost planes z = -1 / z = nz were stored by the neighbours' previous launch into this
// rank's window as LL words (channels 0 p, 1 s, 2 rt) and are polled by the compute warps; this
// launch stores its own first / last plane of the new p, s, rt into the neighbours' windows when
// the unit that owns them has finished its march, and ends by publishing its record.
template <int PM, bool MEUR, bool DIST>
__global__ void __launch_bounds__(kFThreads, 2)
pr_fused_kernel(const __grid_constant__ CUtensorMap tm_p, const __grid_constant__ CUtensorMap tm_s,
                const __grid_constant__ CUtensorMap tm_rt, const TmaGeom G, const Args g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
  double* stage = smem;                                            // [kFStages][3][kPlaneStride]
  double* ring = smem + (size_t)kFStages * 3 * kPlaneStride;       // [kFRing][kPlaneStride]
  __shared__ __align__(8) uint64_t full_bar[kFStages], empty_bar[kFStages];

  const int tid = threadIdx.x;
  if (g.tol_on) {                      // stop_k is visible only after the wait: no prologue overlap then
    pdl_launch_dependents();
    pdl_wait();
    if (after_stop(g)) return;
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kFStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], kFConsumers / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();                          // the prologue above overlapped the previous kernel's tail

  double a, b;
  if constexpr (DIST) {
    // only the compute warps need the scalars: the producer warp starts its copies at once
    __shared__ double sh_ab[2];
    if (tid < kFConsumers) {
      if (tid < 32) dist_fold(g, MEUR, sh_ab);
      named_bar_sync(1, kFConsumers);
      a = sh_ab[0]; b = sh_ab[1];
    } else { a = b = 0.0; }
  } else { a = g.sc->a; b = g.sc->b; }
  const double ds = g.dinv_s;
  auto M = [&](double v) { return PM == 2 ? mul_(ds, v) : v; };

  const int zmin = G.has_zlo ? -1 : 0, zmax = G.has_zhi ? G.nz : G.nz - 1;
  // Work units = (column, z-chunk), chunk-major: unit u is column u % ncols of chunk u / ncols, so the
  // CTAs of one chunk march through the same planes at the same time and the tile halos that
  // neighbouring columns share are served by L2 instead of HBM.  The host launches one CTA per
  // unit when they are all co-resident.
  const int ncols = G.ntx * G.nty;
  const int nunits = ncols * G.nchunk;
  constexpr uint32_t kBytes = (uint32_t)(3 * kPlane * 8);

  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};     // mu, delta, gamma, nu

  if (tid >= kFConsumers) {
    // ------------------------------------------------------------------ producer warp
    if (tid == kFConsumers) {
      uint32_t li = 0;
      for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        const int col = unit % ncols, chunk = unit / ncols;
        const int z0 = (int)((i64)chunk * G.nz / G.nchunk), z1 = (int)((i64)(chunk + 1) * G.nz / G.nchunk);
        const int x0 = (col % G.ntx) * kTX, y0 = (col / G.ntx) * kTY;
        const int lo = G.march_y ? z0 : max(z0 - 1, zmin), hi = G.march_y ? z1 - 1 : min(z1, zmax);
        for (int zz = lo; zz <= hi; ++zz) {
          if (zz < 0 || zz >= G.nz) continue;               // ghost plane of a slab: LL words, no copy
          const int slot = li % kFStages;
          if (li >= kFStages) mbar_wait(&empty_bar[slot], ((li / kFStages) - 1) & 1u, G.err);
          double* dst = stage + (size_t)slot * 3 * kPlaneStride;
          mbar_arrive_expect_tx(&full_bar[slot], kBytes);
          const int ty0 = G.march_y ? zz * kTY : y0, tz = G.march_y ? 0 : zz;
          tma_load_3d(dst, &tm_p, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          tma_load_3d(dst + kPlaneStride, &tm_s, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          tma_load_3d(dst + 2 * kPlaneStride, &tm_rt, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          ++li;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ compute warps
    const int ly = tid >> 5, lx = tid & 31;
    uint32_t li = 0;
    bool first_seg = true;
    for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
      const int col = unit % ncols, chunk = unit / ncols;
      const int z0 = (int)((i64)chunk * G.nz / G.nchunk), z1 = (int)((i64)(chunk + 1) * G.nz / G.nchunk);
      const int x0 = (col % G.ntx) * kTX, y0 = (col / G.ntx) * kTY;
      const int lo = G.march_y ? z0 : max(z0 - 1, zmin), hi = G.march_y ? z1 - 1 : min(z1, zmax);
      // the previous unit's last stencil stage may still be reading the ring
      if (!first_seg) named_bar_sync(1, kFConsumers);
      first_seg = false;

      // x and r do not go through shared memory: they are fetched ONE PLANE AHEAD into registers.
      // Two register sets alternate (the plane loop is unrolled by two), so that no register copy
      // of a value still in flight is ever needed -- such a copy, scheduled before the plane
      // barrier, exposed the whole load latency in every step (ncu: 28 % of the stall samples).
      typedef double Set[kFPairs][2];
      // element index of this lane's first pair in plane z (int: n + 2 planes < 2^31, cgx_set_stencil)
      const int step_stride = G.march_y ? kTY * G.nx : G.nx * G.ny;
      const int idx0 = (G.march_y ? ly : y0 + ly) * G.nx + x0 + 2 * lx;
      const int ybase = G.march_y ? ly : y0 + ly, ystep = G.march_y ? kTY : 0;
      bool okx[kFPairs];
#pragma unroll
      for (int j = 0; j < kFPairs; ++j) okx[j] = (x0 + 2 * lx + 64 * j) < G.nx;
      // real planes of the march (a slab's ghost planes are handled outside the plane loop)
      const int rlo = DIST ? max(lo, 0) : lo, rhi = DIST ? min(hi, G.nz - 1) : hi;
      auto fetch_xr = [&](int z, Set& xs, Set& rs) {
        const bool oky = ybase + z * ystep < G.ny;
        const int ib = idx0 + z * step_stride;
#pragma unroll
        for (int j = 0; j < kFPairs; ++j) {
          // unconditional loads (a pair outside the grid reads element 0 and is never used): a
          // select on the loaded value would wait for the load right here
          const int i = (oky && okx[j]) ? ib + 64 * j : 0;
          const double2 xv = *reinterpret_cast<const double2*>(g.x + i);
          const double2 rv = *reinterpret_cast<const double2*>(g.r + i);
          xs[j][0] = xv.x; xs[j][1] = xv.y; rs[j][0] = rv.x; rs[j][1] = rv.y;
        }
      };

      // One plane step.  (xc, rc): x and r of plane zz, fetched during the previous step;
      // (xn, rn): receive plane zz+1; rnew: receives the new r of plane zz; rold: the new r of
      // plane zz-1 (written by the previous step), for the dots of the stencil stage.
      auto plane_step = [&](const int zz, Set& xc, Set& rc, Set& xn, Set& rn, Set& rnew, Set& rold) {
        if (zz <= rhi) {
          const bool fullp = zz >= z0 && zz < z1;          // a plane this CTA owns (else: only its new p)
          if (zz + 1 >= z0 && zz + 1 < z1) fetch_xr(zz + 1, xn, rn);
          const int slot = li % kFStages;
          mbar_wait(&full_bar[slot], (li / kFStages) & 1u, G.err);
          const double* sp = stage + (size_t)slot * 3 * kPlaneStride;
          const double* ss = sp + kPlaneStride;
          const double* srt = sp + 2 * kPlaneStride;
          double* pn = ring + (size_t)(zz & (kFRing - 1)) * kPlaneStride;
          const bool oky = ybase + zz * ystep < G.ny;
          const int ib = idx0 + zz * step_stride;
#pragma unroll
          for (int j = 0; j < kFPairs; ++j) {
            const int c = (ly + 1) * kPX + 2 * lx + 64 * j + 2;
            const double2 po = lds2(sp + c), so = lds2(ss + c), rto = lds2(srt + c);
            const double pov[2] = {po.x, po.y}, sov[2] = {so.x, so.y}, rtov[2] = {rto.x, rto.y};
            double xo[2], rtn[2], pnw[2];
            const bool ok = fullp && oky && okx[j];
#pragma unroll
            for (int l = 0; l < 2; ++l) {                   // pr_cg.py:146-148,151,157
              rtn[l] = axmy_(rtov[l], a, M(sov[l]));
              pnw[l] = axpy_(rtn[l], b, pov[l]);
            }
            sts2(pn + c, pnw[0], pnw[1]);
            if (ok) {
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                xo[l] = axpy_(xc[j][l], a, pov[l]);
                rnew[j][l] = axmy_(rc[j][l], a, sov[l]);
                red[3] = fma(rtn[l], rnew[j][l], red[3]);
              }
              const int i = ib + 64 * j;
              *reinterpret_cast<double2*>(g.x + i) = make_double2(xo[0], xo[1]);
              *reinterpret_cast<double2*>(g.r + i) = make_double2(rnew[j][0], rnew[j][1]);
              *reinterpret_cast<double2*>(g.rt + i) = make_double2(rtn[0], rtn[1]);
              *reinterpret_cast<double2*>(g.p + i) = make_double2(pnw[0], pnw[1]);
            }
          }
          if (fullp) {
            // the new p on the one-point xy halo of the tile (recomputed, never stored to HBM)
            if (tid < 2 * (kTX / 2)) {
              const int py = (tid >= kTX / 2) ? kPY - 1 : 0;
              const int c = py * kPX + 2 * (tid & (kTX / 2 - 1)) + 2;
              const double2 po = lds2(sp + c), so = lds2(ss + c), rto = lds2(srt + c);
              const double r0 = axmy_(rto.x, a, M(so.x)), r1 = axmy_(rto.y, a, M(so.y));
              sts2(pn + c, axpy_(r0, b, po.x), axpy_(r1, b, po.y));
            } else if (tid < kTX + 2 * kTY) {
              const int u = tid - kTX;
              const int c = ((u % kTY) + 1) * kPX + ((u >= kTY) ? kTX + 2 : 1);
              const double r0 = axmy_(srt[c], a, M(ss[c]));
              pn[c] = axpy_(r0, b, sp[c]);
            }
          }
          __syncwarp();
          if (lx == 0) mbar_arrive(&empty_bar[slot]);       // this warp is done with the input stage
          ++li;
        } else if constexpr (DIST) {
          if (hi >= G.nz) {                                 // drain step of the top unit: plane nz from the scratch
            double* pn = ring + (size_t)(G.nz & (kFRing - 1)) * kPlaneStride + (ly + 1) * kPX + 2 * lx + 2;
#pragma unroll
            for (int j = 0; j < kFPairs; ++j) {
              const int e = (ybase < G.ny && okx[j]) ? idx0 + 64 * j : 0;
              const double2 t = *reinterpret_cast<const double2*>(g.gscr + e);
              sts2(pn + 64 * j, t.x, t.y);
            }
          }
        }
        named_bar_sync(1, kFConsumers);                     // the new p plane zz is complete

        const int q = zz - 1;                               // stencil + dots for plane q
        if (q >= z0 && q < z1) {
          const double* pm = ring + (size_t)((q - 1) & (kFRing - 1)) * kPlaneStride;
          const double* pc = ring + (size_t)(q & (kFRing - 1)) * kPlaneStride;
          const double* pp = ring + (size_t)((q + 1) & (kFRing - 1)) * kPlaneStride;
          const bool has_zm = !G.march_y && ((q > 0) || G.has_zlo);
          const bool has_zp = !G.march_y && ((q < G.nz - 1) || G.has_zhi);
          const bool oky = ybase + q * ystep < G.ny;
          const int ib = idx0 + q * step_stride;
#pragma unroll
          for (int j = 0; j < kFPairs; ++j) {
            if (oky && okx[j]) {
              const int c = (ly + 1) * kPX + 2 * lx + 64 * j + 2;
              const double2 zm = lds2(pm + c), zp = lds2(pp + c);
              const double2 ym = lds2(pc + c - kPX), yp = lds2(pc + c + kPX), ct = lds2(pc + c);
              const double xm = pc[c - 1], xp = pc[c + 2];
              const double zmv[2] = {zm.x, zm.y}, zpv[2] = {zp.x, zp.y}, ymv[2] = {ym.x, ym.y}, ypv[2] = {yp.x, yp.y},
                           ctv[2] = {ct.x, ct.y}, xmv[2] = {xm, ct.x}, xpv[2] = {ct.y, xp};
              double y[2];
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                // canonical CSR order z-1, y-1, x-1, centre, x+1, y+1, z+1; xy neighbours outside
                // the domain are +0.0 (TMA fill -> p = 0): adding off * 0 never changes the sum;
                // absent z planes are stale shared memory and keep their select (cgx_stencil_tma.cuh)
                double acc = 0.0, t;
                t = add_(acc, mul_(G.off, zmv[l]));          acc = has_zm ? t : acc;
                acc = add_(acc, mul_(G.off, ymv[l]));
                acc = add_(acc, mul_(G.off, xmv[l]));
                acc = add_(acc, mul_(G.diag, ctv[l]));
                acc = add_(acc, mul_(G.off, xpv[l]));
                acc = add_(acc, mul_(G.off, ypv[l]));
                t = add_(acc, mul_(G.off, zpv[l]));          acc = has_zp ? t : acc;
                y[l] = acc;
                const double sti = M(acc);                   // pr_cg.py:152-156
                red[0] = fma(ctv[l], acc, red[0]);
                red[1] = fma(rold[j][l], sti, red[1]);
                red[2] = fma(sti, acc, red[2]);
              }
              *reinterpret_cast<double2*>(g.s + ib + 64 * j) = make_double2(y[0], y[1]);
            }
          }
        }
      };

      Set xa, ra, xb, rb, rna = {}, rnb = {};
      if (rlo >= z0) fetch_xr(rlo, xa, ra);
      if constexpr (DIST) {
        // Ghost planes of the slab, BEFORE the march: the new p at this lane's own points of plane
        // z = -1 / nz, from the LL words (p, s, rt = channels 0, 1, 2) the neighbour's previous launch
        // stored, into the scratch planes.  Nothing of this lives in the plane loop.
        int* err = &g.d.win[g.d.rank]->error;
        const size_t chs = ghl_off(g.d, 1, 0, 0);              // channel stride of the LL ghost planes
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
          if (side == 0 ? lo >= 0 : hi < G.nz) continue;
          const u64* gh = g.d.ghl + ghl_off(g.d, 0, g.hin_par, side);
#pragma unroll 1
          for (int j = 0; j < kFPairs; ++j) {
            if (!(ybase < G.ny && okx[j])) continue;
            const int e = idx0 + 64 * j;
            double pnw[2] = {0.0, 0.0};
            if (!(g.dbg & 1)) {
              LLReq rq[3][2];
#pragma unroll
              for (int v = 0; v < 3; ++v)
#pragma unroll
                for (int l = 0; l < 2; ++l) { rq[v][l].src = gh + v * chs + 2 * (size_t)(e + l); ll_issue(rq[v][l]); }
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                const double po = ll_finish(rq[0][l], g.hin_epoch, err), so = ll_finish(rq[1][l], g.hin_epoch, err),
                             rto = ll_finish(rq[2][l], g.hin_epoch, err);
                pnw[l] = axpy_(axmy_(rto, a, M(so)), b, po);
              }
            }
            // below: straight into the ring slot of plane -1 (this thread reads it back itself in the
            // stencil stage of plane 0, before plane 3 reuses the slot); above: parked in the scratch
            // plane until the drain step (the ring slot of plane nz is in use until then)
            if (side == 0) sts2(ring + (size_t)((-1) & (kFRing - 1)) * kPlaneStride + (ly + 1) * kPX + 2 * lx + 64 * j + 2, pnw[0], pnw[1]);
            else *reinterpret_cast<double2*>(g.gscr + e) = make_double2(pnw[0], pnw[1]);
          }
        }
      }
      for (int zz = rlo; zz <= rhi + 1; zz += 2) {
        plane_step(zz, xa, ra, xb, rb, rna, rnb);
        if (zz + 1 <= rhi + 1) plane_step(zz + 1, xb, rb, xa, ra, rnb, rna);
      }
      if constexpr (DIST) {
        // Boundary planes of the slab this unit computed, AFTER the march: the new p, s, rt go to the
        // neighbour's window as LL words; every thread re-reads what it stored itself.
        if (!(g.dbg & 1)) {
          const size_t chs = ghl_off(g.d, 1, 0, 0);
          const double* src[3] = {g.p, g.s, g.rt};
#pragma unroll 1
          for (int side = 0; side < 2; ++side) {
            if (side == 0 ? !(z0 == 0 && g.d.has_lo) : !(z1 == G.nz && g.d.has_hi)) continue;
            u64* dst = (side == 0 ? g.d.ghl_lo : g.d.ghl_hi) + ghl_off(g.d, 0, g.hout_par, side ^ 1);
            const int i0 = idx0 + (side == 0 ? 0 : (G.nz - 1) * step_stride);
#pragma unroll 1
            for (int j = 0; j < kFPairs; ++j) {
              if (!(ybase < G.ny && okx[j])) continue;
#pragma unroll
              for (int v = 0; v < 3; ++v) {
                const double2 t = *reinterpret_cast<const double2*>(src[v] + i0 + 64 * j);
                ll_store(dst + v * chs + 2 * (size_t)(idx0 + 64 * j), t.x, g.hout_epoch);
                ll_store(dst + v * chs + 2 * (size_t)(idx0 + 64 * j + 1), t.y, g.hout_epoch);
              }
            }
          }
        }
      }
    }
  }

  // {mu, delta, gamma, nu} -> a, b of the next iteration (pr_cg.py:154-158 then :149-150)
  grid_sum_finalize<4>(red, g.partials, g.ticket, [&](const double* acc) {
    if constexpr (DIST) dist_publish<4>(g, acc);
    else apply_finalize(FK_PIPE, MEUR, g.sc, acc, g.k);
  }, false);
}

// Partitioned runs, once per solve after the initialisation: the boundary planes of p, s, rt as LL
// words into the neighbours' windows (what every later launch does for the planes it computes).
static __global__ void __launch_bounds__(kBlock) fused_halo_init_kernel(const Args g) {
  const i64 pl = g.d.plane;
  const double* src[3] = {g.p, g.s, g.rt};
  const i64 stride = (i64)gridDim.x * kBlock;
  for (i64 i = (i64)blockIdx.x * kBlock + threadIdx.x; i < pl; i += stride) {
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      if (g.d.has_lo) ll_store(g.d.ghl_lo + ghl_off(g.d, v, g.hout_par, 1) + 2 * i, src[v][i], g.hout_epoch);
      if (g.d.has_hi) ll_store(g.d.ghl_hi + ghl_off(g.d, v, g.hout_par, 0) + 2 * i, src[v][g.n - pl + i], g.hout_epoch);
    }
  }
}

}  // namespace cgx
