// cgx_varstencil.cuh -- matrix-free symmetric variable-coefficient 5/7-point stencil (sm_100a):
// the operator (generic SpMV and instrumentation kernels), its row inside the persistent kernel,
// and a TMA-staged SpMV pass with the fused epilogues of every SP_* stage.
//
// The operator is given by four words per row: diag[i] = A[i,i], cx[i] = A[i,i+1], cy[i] = A[i,i+nx],
// cz[i] = A[i,i+nx*ny]; the backward couplings are those of the neighbour (A[i,i-1] = cx[i-1], ...).
// A coupling that leaves the grid is 0 (checked on the host).  Every row sum visits the in-grid
// neighbours in canonical CSR order (z-1, y-1, x-1, centre, x+1, y+1, z+1) with separately rounded
// multiply and add, so the bits equal scipy's product with the CSR matrix of the full 5/7-point pattern.
// Single-GPU contexts only: there are no ghost planes.
#pragma once
#include "cgx_stencil_tma.cuh"
#include "cgx_persistent.cuh"

namespace cgx {

struct VarStencilOp {
  static constexpr bool kSlab = true;     // (row indices only; a single GPU never asks for a ghost plane)
  int nx, ny, nz;
  i64 n;
  const double* __restrict__ diag;
  const double* __restrict__ cx;
  const double* __restrict__ cy;
  const double* __restrict__ cz;          // null in 2-D
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
#define CGX_VT(cond, j, coef)                                              \
    if (cond) {                                                            \
      const double a_ = (coef);                                            \
      ld((i64)(j), v);                                                     \
      _Pragma("unroll") for (int c = 0; c < NV; ++c) y[c] = add_(y[c], mul_(a_, v[c])); \
    }
    CGX_VT(z > 0, ii - plane, __ldg(cz + ii - plane))
    CGX_VT(yy > 0, ii - nx, __ldg(cy + ii - nx))
    CGX_VT(xx > 0, ii - 1, __ldg(cx + ii - 1))
    CGX_VT(true, ii, __ldg(diag + ii))
    CGX_VT(xx < nx - 1, ii + 1, __ldg(cx + ii))
    CGX_VT(yy < ny - 1, ii + nx, __ldg(cy + ii))
    CGX_VT(z < nz - 1, ii + plane, __ldg(cz + ii))
#undef CGX_VT
  }
};

// ---- persistent kernel: the neighbour mask of StencilOp; the coefficients are read through L2 ----
__device__ __forceinline__ unsigned stencil_mask(const VarStencilOp& A, int row) {
  const int plane = A.nx * A.ny;
  const int z = row / plane, rem = row - z * plane, yy = rem / A.nx, xx = rem - yy * A.nx;
  return (unsigned)((z > 0) ? 1 : 0) | ((yy > 0) ? 2u : 0u) | ((xx > 0) ? 4u : 0u) |
         ((xx < A.nx - 1) ? 8u : 0u) | ((yy < A.ny - 1) ? 16u : 0u) | ((z < A.nz - 1) ? 32u : 0u);
}
template <int NVX, class Ld>
__device__ __forceinline__ void pers_row(const VarStencilOp& A, int row, unsigned m, Ld ld, double (&y)[NVX]) {
  const int plane = A.nx * A.ny;
  const double* cz = A.cz ? A.cz : A.diag;     // (2-D: no z term is ever taken; any valid row address will do)
  double v[NVX];
#pragma unroll
  for (int c = 0; c < NVX; ++c) y[c] = 0.0;
#define CGX_VPT(bit, j, cp, ci)                                                            \
  {                                                                                        \
    const bool ex = (m & (bit)) != 0u;               /* absent neighbour: read the row itself, drop the term */ \
    const double a_ = __ldg((cp) + (ex ? (ci) : row));                                     \
    ld(ex ? (j) : row, v);                                                                 \
    _Pragma("unroll") for (int c = 0; c < NVX; ++c) {                                      \
      const double t = add_(y[c], mul_(a_, v[c]));                                         \
      y[c] = ex ? t : y[c];                                                                \
    }                                                                                      \
  }
  CGX_VPT(1u, row - plane, cz, row - plane)
  CGX_VPT(2u, row - A.nx, A.cy, row - A.nx)
  CGX_VPT(4u, row - 1, A.cx, row - 1)
  CGX_VPT(~0u, row, A.diag, row)
  CGX_VPT(8u, row + 1, A.cx, row)
  CGX_VPT(16u, row + A.nx, A.cy, row)
  CGX_VPT(32u, row + plane, cz, row)
#undef CGX_VPT
}

// ---- TMA-staged pass ------------------------------------------------------------------------------
// The march of stencil_tma_kernel (cgx_stencil_tma.cuh: 8 compute warps + 1 producer warp, (column,
// z-chunk) work units, full / empty mbarrier per ring slot, no CTA-wide barrier), with a ring slot that
// carries, next to the NV vector planes, the cx, cy [, cz] boxes of the same plane and geometry.  Every
// coupling then sits where its neighbour's value sits: cx[i-1] in the x halo, cy[i-nx] in the y halo,
// cz[i-plane] in slot z-1.  Couplings outside the grid come zero-filled by the TMA unit; their term adds
// +0 * +0 to a sum that started at +0.0 and so cannot be -0.0, which leaves its bits unchanged.  diag is
// read directly, one plane ahead, like r and a Jacobi vector.
// Ring depth: 4 slots (z-1, z, z+1 and one copy in flight).  A 1-RHS slot is 4 planes (42.5 KB), a 2-RHS
// slot 5 (53 KB): one CTA per SM either way (170 / 212 KB).
constexpr int kVRing = 4;
constexpr int kVCoef = 3;                       // cx, cy, cz planes reserved per slot
__host__ __device__ constexpr size_t varstencil_smem_bytes(int nv) {
  return (size_t)kVRing * (nv + kVCoef) * kPlaneStride * sizeof(double) + 128;
}

// MODE: SP_HS, SP_CG, SP_GV, SP_PR, SP_PIPE_R, SP_PIPE_N.  PM: 0 identity, 1 Jacobi vector, 2 Jacobi scalar.
// tcz is read only when A.cz != null and the march is through z-planes (a 3-D grid).
template <int MODE, int PM, bool MEUR>
__global__ void __launch_bounds__(kSThreads, 1)
varstencil_tma_kernel(const __grid_constant__ CUtensorMap tm0, const __grid_constant__ CUtensorMap tm1,
                      const __grid_constant__ CUtensorMap tcx, const __grid_constant__ CUtensorMap tcy,
                      const __grid_constant__ CUtensorMap tcz, const VarStencilOp A, const TmaGeom G, const Args g) {
  constexpr int NV = NV_OF(MODE);
  constexpr int R = kVRing;
  constexpr int SW = (NV + kVCoef) * kPlaneStride;      // doubles per ring slot
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
  pdl_wait();

  const bool has_cz = A.cz != nullptr && !G.march_y;
  const int ncoef = has_cz ? 3 : 2;
  const int ncols = G.ntx * G.nty;
  const int nunits = ncols * G.nchunk;
  const uint32_t kBytes = (uint32_t)(kPlane * 8 * (NV + ncoef));
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
          double* dst = smem + (size_t)slot * SW;
          mbar_arrive_expect_tx(&full_bar[slot], kBytes);
          const int ty0 = G.march_y ? zz * kTY : y0, tz = G.march_y ? 0 : zz;
          tma_load_3d(dst, &tm0, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          if constexpr (NV == 2) tma_load_3d(dst + kPlaneStride, &tm1, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          tma_load_3d(dst + NV * kPlaneStride, &tcx, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          tma_load_3d(dst + (NV + 1) * kPlaneStride, &tcy, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
          if (has_cz) tma_load_3d(dst + (NV + 2) * kPlaneStride, &tcz, x0 - 2, ty0 - 1, tz, &full_bar[slot]);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ compute warps
    const int ly = tid >> 5, lx = tid & 31;
    uint32_t li = 0;
    constexpr bool kNeedR = (MODE == SP_CG || MODE == SP_PR);
    constexpr bool kNeedD = (MODE == SP_PR && PM == 1);
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

      // operands that do not go through shared memory (diag, r for the fused dots, a Jacobi vector): one
      // plane ahead, two alternating register sets
      typedef double Set[kSPairs][2];
      auto fetch_direct = [&](int q, Set& as, Set& rs, Set& dsv) {
        const bool oky = ybase + q * ystep < G.ny;
        const int ib = idx0 + q * step_stride;
#pragma unroll
        for (int j = 0; j < kSPairs; ++j) {
          const int i = (oky && okx[j]) ? ib + 64 * j : 0;
          { const double2 t = *reinterpret_cast<const double2*>(A.diag + i); as[j][0] = t.x; as[j][1] = t.y; }
          if constexpr (kNeedR) { const double2 t = *reinterpret_cast<const double2*>(g.r + i); rs[j][0] = t.x; rs[j][1] = t.y; }
          if constexpr (kNeedD) { const double2 t = *reinterpret_cast<const double2*>(g.dinv + i); dsv[j][0] = t.x; dsv[j][1] = t.y; }
        }
      };
      int nwait = 0;                                        // planes lo .. lo + nwait - 1 have landed
      auto plane_step = [&](const int q, Set& ac, Set& rc, Set& dc, Set& an, Set& rn, Set& dn) {
        if (q + 1 < z1) fetch_direct(q + 1, an, rn, dn);
        const int need = G.march_y ? q : min(q + 1, hi);
        while (lo + nwait <= need) {
          const uint32_t l = Lbase + (uint32_t)nwait;
          mbar_wait(&full_bar[l % R], (l / R) & 1u, G.err);
          ++nwait;
        }
        const double* pc = smem + (size_t)((Lbase + (uint32_t)(q - lo)) % R) * SW;
        const double* pm = smem + (size_t)((Lbase + (uint32_t)(q - 1 - lo)) % R) * SW;   // (never read when q-1 < lo)
        const double* pp = smem + (size_t)((Lbase + (uint32_t)(q + 1 - lo)) % R) * SW;
        const double* ccx = pc + NV * kPlaneStride;
        const double* ccy = pc + (NV + 1) * kPlaneStride;
        const double* ccz = pc + (NV + 2) * kPlaneStride;
        const double* mcz = pm + (NV + 2) * kPlaneStride;
        const bool has_zm = !G.march_y && q > 0;
        const bool has_zp = !G.march_y && q < G.nz - 1;
        const bool oky = ybase + q * ystep < G.ny;
        const int ib = idx0 + q * step_stride;
#pragma unroll
        for (int j = 0; j < kSPairs; ++j) {
          if (oky && okx[j]) {
            const int c = (ly + 1) * kPX + 2 * lx + 64 * j + 2;
            // couplings of the pair (points c, c+1 of the tile), each in canonical term order
            const double2 czm = has_zm ? *reinterpret_cast<const double2*>(mcz + c) : make_double2(0.0, 0.0);
            const double2 czp = has_zp ? *reinterpret_cast<const double2*>(ccz + c) : make_double2(0.0, 0.0);
            const double2 cym = *reinterpret_cast<const double2*>(ccy + c - kPX), cyp = *reinterpret_cast<const double2*>(ccy + c);
            const double2 cxc = *reinterpret_cast<const double2*>(ccx + c);
            const double cxm0 = ccx[c - 1];
            const double kzm[2] = {czm.x, czm.y}, kym[2] = {cym.x, cym.y}, kxm[2] = {cxm0, cxc.x};
            const double kxp[2] = {cxc.x, cxc.y}, kyp[2] = {cyp.x, cyp.y}, kzp[2] = {czp.x, czp.y};
            double y[NV][2], ctr[NV][2];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              const double* qm = pm + v * kPlaneStride;
              const double* qc = pc + v * kPlaneStride;
              const double* qp = pp + v * kPlaneStride;
              const double2 zm = *reinterpret_cast<const double2*>(qm + c), zp = *reinterpret_cast<const double2*>(qp + c);
              const double2 ym = *reinterpret_cast<const double2*>(qc + c - kPX), yp = *reinterpret_cast<const double2*>(qc + c + kPX),
                            ct = *reinterpret_cast<const double2*>(qc + c);
              const double xm = qc[c - 1], xp = qc[c + 2];
              const double zmv[2] = {zm.x, zm.y}, zpv[2] = {zp.x, zp.y}, ymv[2] = {ym.x, ym.y}, ypv[2] = {yp.x, yp.y},
                           ctv[2] = {ct.x, ct.y};
              const double xmv[2] = {xm, ct.x}, xpv[2] = {ct.y, xp};
#pragma unroll
              for (int l = 0; l < 2; ++l) {
                // absent z-planes are not loaded at all (stale shared memory): those two terms keep a select
                double acc = 0.0, t;
                t = add_(acc, mul_(kzm[l], zmv[l]));         acc = has_zm ? t : acc;
                acc = add_(acc, mul_(kym[l], ymv[l]));
                acc = add_(acc, mul_(kxm[l], xmv[l]));
                acc = add_(acc, mul_(ac[j][l], ctv[l]));
                acc = add_(acc, mul_(kxp[l], xpv[l]));
                acc = add_(acc, mul_(kyp[l], ypv[l]));
                t = add_(acc, mul_(kzp[l], zpv[l]));         acc = has_zp ? t : acc;
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
            } else if constexpr (MODE == SP_CG) {          // cg_cg.py:133-135
              st2(g.w, y[0]);
#pragma unroll
              for (int l = 0; l < 2; ++l) { red[0] = fma(rc[j][l], ctr[0][l], red[0]); red[1] = fma(y[0][l], ctr[0][l], red[1]); }
            } else if constexpr (MODE == SP_GV) {          // gv_cg.py:161
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
              static_assert(MODE == SP_PIPE_N, "varstencil_tma_kernel: no such stage");
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

      Set aa, ra, da, ab, rb, db;
      fetch_direct(z0, aa, ra, da);
      int q = z0;
      for (; q + 1 < z1; q += 2) {
        plane_step(q, aa, ra, da, ab, rb, db);
        plane_step(q + 1, ab, rb, db, aa, ra, da);
      }
      if (q < z1) plane_step(q, aa, ra, da, ab, rb, db);
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
