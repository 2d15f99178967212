// cgx_stencil_tma.cuh -- TMA-staged matrix-free stencil SpMV with fused epilogues (sm_100a).
//
// One CTA owns a BX x BY column of the grid and marches through a chunk of z-planes.  Each
// plane (with its one-point x/y halo) is brought into shared memory by ONE bulk-tensor copy
// (cp.async.bulk.tensor.3d, SASS UTMALDG) that completes on an mbarrier; out-of-range
// coordinates are zero-filled by the TMA unit, which is exactly the Dirichlet boundary, so
// the load path has no boundary branches.  A ring of kRing planes keeps the copy of plane
// z+2 in flight while plane z is computed from planes z-1, z, z+1, so every input value
// is read from L2/HBM once per CTA column (+ halo) instead of seven times.
//
// The row sum is still evaluated in canonical-CSR term order with separately rounded
// multiply and add (absent neighbours are skipped by a select, not by adding a zero), so
// results stay bit-identical to scipy's `A @ v` on the equivalent CSR matrix.
#pragma once
#include <cuda.h>

#include "cgx_kernels.cuh"

namespace cgx {

constexpr int kTX = 128;              // tile extent in x (points)
constexpr int kTY = 8;                // tile extent in y
constexpr int kPX = kTX + 4;          // box extent incl. halo: starts at x0-2 (TMA needs 16-B aligned starts)
constexpr int kPY = kTY + 2;
constexpr int kPlane = kPX * kPY;     // doubles per staged plane
constexpr int kPlaneStride = ((kPlane * 8 + 127) / 128) * 128 / 8;   // 128-B aligned slots
constexpr int kRing = 4;
constexpr int kTmaThreads = 256;
constexpr int kPtsPerThread = kTX * kTY / kTmaThreads;               // 4

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2),
      "r"(smem_u32(bar))
      : "memory");
}

// Geometry of one launch.  zlo/zhi: does a plane exist below z=0 / above z=nz-1 of THIS
// slab (multi-GPU partition).  Those ghost planes live in the rank's window as LL words,
// stored by the neighbours' vector passes, and are copied into the ring slot by fill_ghost.
struct TmaGeom {
  int nx, ny, nz;
  int ntx, nty;                  // tiles in x, y
  int has_zlo, has_zhi;
  int march_y;                   // 2-D grid: the "planes" of the march are the y-tiles (8 rows each) of a
                                 // column of x-tiles, so consecutive tiles pipeline through the ring like
                                 // z-planes do (nz = number of y-tiles, nty = 1; no z neighbours)
  double diag, off;
  int nchunk;                    // z-chunks per column (kernels that take (column, chunk) work units)
  int* err;                      // device word set when a plane copy did not land within 1 s
};

#define NV_OF(MODE) ((MODE) == SP_PIPE_R ? 2 : 1)

// ---- warp-specialised march ------------------------------------------------------------------
// 8 compute warps (warp w <-> row w of the 128 x 8 tile, a lane owns the point pairs 2 lx + 64 j)
// + 1 producer warp.  The producer's elected lane issues the bulk-tensor copies of the planes a
// unit needs into a ring of kRingOf(NV) slots, each guarded by a full (transaction) and an empty
// (one arrival per compute warp) mbarrier, and runs ahead across unit changes; a compute warp waits
// only for the planes it reads and releases plane z-1 when it has computed plane z.  There is NO
// CTA-wide barrier in the march.
// Work units are (column, z-chunk), chunk-major, one CTA per unit when they are co-resident: all
// columns of a chunk then march in lockstep and the tile halos neighbouring columns share come from
// L2 (cgx_stencil_fused.cuh uses the same decomposition).
constexpr int kSConsumers = 256;
constexpr int kSThreads = kSConsumers + 32;
constexpr int kSPairs = kTX / 64;
__host__ __device__ constexpr int kRingOf(int nv) { return nv == 2 ? 4 : 8; }
__host__ __device__ constexpr size_t stencil_smem_bytes(int nv) {
  return (size_t)kRingOf(nv) * nv * kPlaneStride * sizeof(double) + 128;
}

// MODE: SP_* of cgx_kernels.cuh.  PM: 0 identity, 1 Jacobi vector, 2 Jacobi scalar.
template <int MODE, int PM, bool MEUR>
__global__ void __launch_bounds__(kSThreads, 2)
stencil_tma_kernel(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
                   const TmaGeom G, const Args g) {
  constexpr int NV = NV_OF(MODE);
  constexpr int R = kRingOf(NV);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* smem = reinterpret_cast<double*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
  __shared__ __align__(8) uint64_t full_bar[R], empty_bar[R];

  const int tid = threadIdx.x;
  if (g.tol_on) {                      // stop_k is visible only after the wait: no prologue overlap then
    pdl_launch_dependents();
    pdl_wait();
    if (after_stop(g)) return;
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < R; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], kSConsumers / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_launch_dependents();
  pdl_wait();                          // the prologue above overlapped the previous kernel's tail

  const int ncols = G.ntx * G.nty;
  const int nunits = ncols * G.nchunk;
  constexpr uint32_t kBytes = (uint32_t)(kPlane * 8 * NV);
  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};

  if (tid >= kSConsumers) {
    // ------------------------------------------------------------------ producer warp
    if (tid == kSConsumers) {
      uint32_t li = 0;
      for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        const int col = unit % ncols, chunk = unit / ncols;
        const int z0 = (int)((i64)chunk * G.nz / G.nchunk), z1 = (int)((i64)(chunk + 1) * G.nz / G.nchunk);
        const int x0 = (col % G.ntx) * kTX, y0 = (col / G.ntx) * kTY;
        const int lo = G.march_y ? z0 : max(z0 - 1, 0), hi = G.march_y ? z1 - 1 : min(z1, G.nz - 1);
        for (int zz = lo; zz <= hi; ++zz, ++li) {
          const int slot = li % R;
          if (li >= (uint32_t)R) mbar_wait(&empty_bar[slot], ((li / R) - 1) & 1u, G.err);
          double* dst = smem + (size_t)slot * NV * kPlaneStride;
          mbar_arrive_expect_tx(&full_bar[slot], kBytes);
          const int ty0 = G.march_y ? zz * kTY : y0, tz = G.march_y ? 0 : zz;
          tma_load_3d(dst, &tm0, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          if constexpr (NV == 2) tma_load_3d(dst + kPlaneStride, &tm1, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ compute warps
    const int ly = tid >> 5, lx = tid & 31;
    uint32_t li = 0;
    constexpr bool kNeedR = (MODE == SP_CG || MODE == SP_PR);
    constexpr bool kNeedD = (MODE == SP_PR && PM == 1);
    constexpr bool kScaleIn = (MODE == SP_CG_E || MODE == SP_GV_E) && PM == 2;   // tile holds r / w: operand is M r / M w
    for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
      const int col = unit % ncols, chunk = unit / ncols;
      const int z0 = (int)((i64)chunk * G.nz / G.nchunk), z1 = (int)((i64)(chunk + 1) * G.nz / G.nchunk);
      const int x0 = (col % G.ntx) * kTX, y0 = (col / G.ntx) * kTY;
      const int lo = G.march_y ? z0 : max(z0 - 1, 0), hi = G.march_y ? z1 - 1 : min(z1, G.nz - 1);
      const uint32_t Lbase = li;                            // load index of plane lo
      const int step_stride = G.march_y ? kTY * G.nx : G.nx * G.ny;
      const int idx0 = (G.march_y ? ly : y0 + ly) * G.nx + x0 + 2 * lx;
      const int ybase = G.march_y ? ly : y0 + ly, ystep = G.march_y ? kTY : 0;
      bool okx[kSPairs];
#pragma unroll
      for (int j = 0; j < kSPairs; ++j) okx[j] = (x0 + 2 * lx + 64 * j) < G.nx;

      // Slab of a partition: the planes below z = 0 / above z = nz-1 live in the rank's window as LL
      // words stored by the neighbours' vector passes.  Only the z-1 / z+1 TERMS of this lane's own
      // points need them: they are decoded once, before the march, into the scratch planes
      // (g.gscr[(side * 2 + v) * plane + e]) and read back by the same thread -- no ring slot, no
      // synchronisation, nothing of the polling inside the plane loop.
      const bool ghost_lo = !G.march_y && z0 == 0 && G.has_zlo, ghost_hi = !G.march_y && z1 == G.nz && G.has_zhi;
      if (ghost_lo || ghost_hi) {
        int* err = &g.d.win[g.d.rank]->error;
#pragma unroll 1
        for (int side = 0; side < 2; ++side) {
          if (side == 0 ? !ghost_lo : !ghost_hi) continue;
#pragma unroll 1
          for (int v = 0; v < NV; ++v) {
            const u64* gh = g.d.ghl + ghl_off(g.d, g.hin_ch + v, g.hin_par, side);
#pragma unroll 1
            for (int j = 0; j < kSPairs; ++j) {
              if (!(ybase < G.ny && okx[j])) continue;
              const int e = idx0 + 64 * j;
              double t0 = 0.0, t1 = 0.0;
              if (!(g.dbg & 1)) {
                LLReq q0, q1;
                q0.src = gh + 2 * (size_t)e; q1.src = gh + 2 * (size_t)(e + 1);
                ll_issue(q0); ll_issue(q1);
                t0 = ll_finish(q0, g.hin_epoch, err); t1 = ll_finish(q1, g.hin_epoch, err);
              }
              *reinterpret_cast<double2*>(g.gscr + (size_t)(side * 2 + v) * g.d.plane + e) = make_double2(t0, t1);
            }
          }
        }
      }

      // operands that do not go through shared memory (r for the fused dots, a Jacobi vector): one
      // plane ahead, two alternating register sets (no copies of values in flight)
      typedef double Set[kSPairs][2];
      auto fetch_direct = [&](int q, Set& rs, Set& dsv) {
        if constexpr (kNeedR || kNeedD) {
          const bool oky = ybase + q * ystep < G.ny;
          const int ib = idx0 + q * step_stride;
#pragma unroll
          for (int j = 0; j < kSPairs; ++j) {
            const int i = (oky && okx[j]) ? ib + 64 * j : 0;
            if constexpr (kNeedR) { const double2 t = *reinterpret_cast<const double2*>(g.r + i); rs[j][0] = t.x; rs[j][1] = t.y; }
            if constexpr (kNeedD) { const double2 t = *reinterpret_cast<const double2*>(g.dinv + i); dsv[j][0] = t.x; dsv[j][1] = t.y; }
          }
        }
      };
      int nwait = 0;                                        // planes lo .. lo + nwait - 1 have landed
      auto plane_step = [&](const int q, Set& rc, Set& dc, Set& rn, Set& dn) {
        if (q + 1 < z1) fetch_direct(q + 1, rn, dn);
        const int need = G.march_y ? q : min(q + 1, hi);
        while (lo + nwait <= need) {
          const uint32_t l = Lbase + (uint32_t)nwait;
          mbar_wait(&full_bar[l % R], (l / R) & 1u, G.err);
          ++nwait;
        }
        const double* pc = smem + (size_t)((Lbase + (uint32_t)(q - lo)) % R) * NV * kPlaneStride;
        const double* pm = smem + (size_t)((Lbase + (uint32_t)(q - 1 - lo)) % R) * NV * kPlaneStride;   // (never read when q-1 < lo)
        const double* pp = smem + (size_t)((Lbase + (uint32_t)(q + 1 - lo)) % R) * NV * kPlaneStride;
        const bool has_zm = !G.march_y && ((q > 0) || G.has_zlo);
        const bool has_zp = !G.march_y && ((q < G.nz - 1) || G.has_zhi);
        const bool zm_scr = ghost_lo && q == 0, zp_scr = ghost_hi && q == G.nz - 1;
        const bool oky = ybase + q * ystep < G.ny;
        const int ib = idx0 + q * step_stride;
#pragma unroll
        for (int j = 0; j < kSPairs; ++j) {
          if (oky && okx[j]) {
            const int c = (ly + 1) * kPX + 2 * lx + 64 * j + 2;
            double y[NV][2], ctr[NV][2], raw[NV][2];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              const double* qm = pm + v * kPlaneStride;
              const double* qc = pc + v * kPlaneStride;
              const double* qp = pp + v * kPlaneStride;
              const double* zmp = zm_scr ? g.gscr + (size_t)v * g.d.plane + idx0 + 64 * j : qm + c;
              const double* zpp = zp_scr ? g.gscr + (size_t)(2 + v) * g.d.plane + idx0 + 64 * j : qp + c;
              const double2 zm = *reinterpret_cast<const double2*>(zmp), zp = *reinterpret_cast<const double2*>(zpp);
              const double2 ym = *reinterpret_cast<const double2*>(qc + c - kPX), yp = *reinterpret_cast<const double2*>(qc + c + kPX),
                            ct = *reinterpret_cast<const double2*>(qc + c);
              const double xm = qc[c - 1], xp = qc[c + 2];
              auto in = [&](double t) { if constexpr (kScaleIn) return mul_(g.dinv_s, t); else return t; };
              const double zmv[2] = {in(zm.x), in(zm.y)}, zpv[2] = {in(zp.x), in(zp.y)}, ymv[2] = {in(ym.x), in(ym.y)},
                           ypv[2] = {in(yp.x), in(yp.y)}, ctv[2] = {in(ct.x), in(ct.y)};
              const double xmv[2] = {in(xm), ctv[0]}, xpv[2] = {ctv[1], in(xp)};
              raw[v][0] = ct.x; raw[v][1] = ct.y;
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                // canonical CSR order z-1, y-1, x-1, centre, x+1, y+1, z+1.  xy neighbours outside the
                // domain were zero-filled by the TMA unit: off * (+0.0) never changes a running sum that
                // started at +0.0, so the bits equal scipy's sum over the stored entries.  Absent
                // z-planes are not loaded at all (stale shared memory): those two terms keep a select.
                double acc = 0.0, t;
                t = add_(acc, mul_(G.off, zmv[l]));          acc = has_zm ? t : acc;
                acc = add_(acc, mul_(G.off, ymv[l]));
                acc = add_(acc, mul_(G.off, xmv[l]));
                acc = add_(acc, mul_(G.diag, ctv[l]));
                acc = add_(acc, mul_(G.off, xpv[l]));
                acc = add_(acc, mul_(G.off, ypv[l]));
                t = add_(acc, mul_(G.off, zpv[l]));          acc = has_zp ? t : acc;
                y[v][l] = acc;
                ctr[v][l] = ctv[l];
              }
            }
            const int i = ib + 64 * j;
            auto M = [&](double t, int l) {
              if constexpr (PM == 1) return mul_(dc[j][l], t);
              else if constexpr (PM == 2) return mul_(g.dinv_s, t);
              else return t;
            };
            auto st2 = [&](double* dst, const double (&t)[2]) { *reinterpret_cast<double2*>(dst + i) = make_double2(t[0], t[1]); };
            if constexpr (MODE == SP_HS) {                 // hs_cg.py:123-124
              st2(g.s, y[0]);
#pragma unroll
              for (int l = 0; l < 2; ++l) red[0] = fma(ctr[0][l], y[0][l], red[0]);
            } else if constexpr (MODE == SP_CG_E) {        // cg_cg.py:133-135 with r from the tile
              st2(g.w, y[0]);
#pragma unroll
              for (int l = 0; l < 2; ++l) { red[0] = fma(raw[0][l], ctr[0][l], red[0]); red[1] = fma(y[0][l], ctr[0][l], red[1]); }
            } else if constexpr (MODE == SP_CG) {          // cg_cg.py:133-135
              st2(g.w, y[0]);
#pragma unroll
              for (int l = 0; l < 2; ++l) { red[0] = fma(rc[j][l], ctr[0][l], red[0]); red[1] = fma(y[0][l], ctr[0][l], red[1]); }
            } else if constexpr (MODE == SP_GV || MODE == SP_GV_E) {          // gv_cg.py:161
              st2(g.t, y[0]);
            } else if constexpr (MODE == SP_PR) {          // pr_cg.py:152-156
              st2(g.s, y[0]);
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                const double sti = M(y[0][l], l);
                red[0] = fma(ctr[0][l], y[0][l], red[0]);
                red[1] = fma(rc[j][l], sti, red[1]);
                red[2] = fma(sti, y[0][l], red[2]);
              }
            } else if constexpr (MODE == SP_PIPE_R) {      // pipe_pr_cg.py:179-182
              st2(g.u, y[0]);
              st2(g.w, y[NV - 1]);
            } else {                                       // SP_PIPE_N
              st2(g.u, y[0]);
            }
          }
        }
        if (q - 1 >= lo) {                                  // plane q-1 is not needed any more
          __syncwarp();
          const uint32_t l = Lbase + (uint32_t)(q - 1 - lo);
          if (lx == 0) mbar_arrive(&empty_bar[l % R]);
        }
      };

      Set ra, da, rb, db;
      fetch_direct(z0, ra, da);
      int q = z0;
      for (; q + 1 < z1; q += 2) {
        plane_step(q, ra, da, rb, db);
        plane_step(q + 1, rb, db, ra, da);
      }
      if (q < z1) plane_step(q, ra, da, rb, db);
      // release what is still held (plane z1-1 and, when loaded, z1); planes never waited for must be
      // waited for first so that the slot's phase bookkeeping stays in step
      while (lo + nwait <= hi) {
        const uint32_t l = Lbase + (uint32_t)nwait;
        mbar_wait(&full_bar[l % R], (l / R) & 1u, G.err);
        ++nwait;
      }
      __syncwarp();
      for (int zz = max(lo, z1 - 1); zz <= hi; ++zz) {
        const uint32_t l = Lbase + (uint32_t)(zz - lo);
        if (lx == 0) mbar_arrive(&empty_bar[l % R]);
      }
      li = Lbase + (uint32_t)(hi - lo + 1);
    }
  }

  spmv_close<MODE, MEUR>(g, red);
}

}  // namespace cgx
