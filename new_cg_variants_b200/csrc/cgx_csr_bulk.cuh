// cgx_csr_bulk.cuh -- CSR pass with the matrix stream staged by bulk async copies (sm_100a).
//
// Same work decomposition and the same arithmetic as csr_stream_kernel (cgx_kernels.cuh): a work
// item is a block of consecutive rows holding at most kCbCap non-zeros (or one chunk of a longer
// row); every product a_ij * v_j is rounded on its own and a row's products are added in stored
// order, so the result equals scipy's csr_matvec bit for bit.  What changed is who moves the bytes:
//
//   producer warp   issues `cp.async.bulk` (SASS UBLKCP) copies of the item's values, columns, row
//                   extents and the epilogue operands of its rows (contiguous ranges of the SpMV
//                   input, r or b, the Jacobi diagonal) into one slot of a ring in shared memory; they
//                   complete on the slot's transaction mbarrier.  No register is held for a byte in
//                   flight, so the ring depth -- not the register file -- sets how much of the matrix
//                   stream a CTA keeps in flight.  Lane l owns the l-th block of a batch of 32 (metadata
//                   in its own registers, slot and phase computed by all lanes at once) and issues that
//                   block's copies when its turn comes: no shuffles, no divisions per item.
//   14 gather warps read the columns from the slot, gather v_j (L1/L2), multiply with the values
//                   and write the products over the values (in place; second right-hand side into
//                   an array of its own).  The gathers of items i+1 and i+2 are issued before the
//                   products of item i are written.
//   summing warps   (blockDim.x / 32 - 15 of them, items dealt round robin) lane l adds up the products of
//                   rows l, l+32, ... of the item in stored order and applies the stage's epilogue, all
//                   from shared memory, then frees the slot.  A row sum is one dependent chain of
//                   additions (8.2 cycles each on B200: tools/dadd_probe.cu), so what this stage needs is
//                   rows in flight.  The chunks of a row longer than an item are chained through shared
//                   memory.
//
// Measured on the way (banded model problem, 65 non-zeros per row; tools/csr_bench.py, csr_stamp_probe.py):
// the per-item cost of the CONTROL code is what bounds such a pipeline, not memory.  A single producer thread
// that recomputed slot = it % ring and shuffled the block metadata per item was busy 95 % of the time at
// ~1000-1650 cycles per 1120-element item (even with every copy, gather and sum switched off); a variant in
// which every warp was a complete pipeline of its own (352-element items) spent ~400 instructions per item
// per warp and was bound by instruction issue (163 us per pass against 108 us of csr_stream_kernel).
// cp.async.bulk itself sustains 7.0 TB/s from 1 KB copies upward once 64 KB per SM are in flight
// (tools/bulk_probe.cu).  Hence: items as large as the ring allows and a producer without per-item
// arithmetic.
//
// Bulk copies need 16-byte aligned addresses and sizes: a range is widened to the enclosing aligned
// range (at most 3 elements before and after), which is why the host pads every array the copies
// read by kCbPadBytes (cgx.cu).
#pragma once
#include "cgx_kernels.cuh"

namespace cgx {

constexpr int kCbCap = 1792;                         // non-zeros per work item (4 per gather thread)
constexpr int kCbRows = 159;                         // rows per block at most
constexpr int kCbGather = 448;                       // gather threads (14 warps)
constexpr int kCbProducer = kCbGather;               // first thread of the producer warp
constexpr int kCbSum0 = kCbGather + 32;              // first thread of the summing warps
constexpr int kCbMaxSum = 4;
constexpr int kCbMaxThreads = kCbSum0 + 32 * kCbMaxSum;
constexpr int kCbUL = kCbCap / kCbGather;
constexpr int kCbPadBytes = 64;                      // slack behind every array a bulk copy may read
constexpr int kCbMaxRing = 16;
static_assert(kCbCap % kCbGather == 0, "one gather batch per thread");

__host__ __device__ constexpr size_t cb_align(size_t b) { return (b + 127) / 128 * 128; }
__host__ __device__ constexpr size_t cb_val_bytes() { return cb_align((size_t)(kCbCap + 8) * 8); }
__host__ __device__ constexpr size_t cb_col_bytes() { return cb_align((size_t)(kCbCap + 8) * 4); }
__host__ __device__ constexpr size_t cb_ptr_bytes() { return cb_align((size_t)(kCbRows + 1 + 7) * 4); }
__host__ __device__ constexpr size_t cb_op_bytes() { return cb_align((size_t)(kCbRows + 3) * 8); }
// which epilogue operands a stage reads per row: bit 0 the SpMV input, bit 1 r (b for SP_RESID), bit 2 the Jacobi entry
__host__ __device__ constexpr int cb_ops(int mode, int pm) {
  return ((mode == SP_HS || mode == SP_CG || mode == SP_PR) ? 1 : 0) |
         ((mode == SP_CG || mode == SP_PR || mode == SP_RESID) ? 2 : 0) | ((mode == SP_PR && pm == 1) ? 4 : 0);
}
__host__ __device__ constexpr int cb_nops(int ops) { return (ops & 1) + ((ops >> 1) & 1) + ((ops >> 2) & 1); }
__host__ __device__ constexpr size_t cb_slot_bytes(int nv, int ops) {
  return cb_val_bytes() * nv + cb_col_bytes() + cb_ptr_bytes() + cb_op_bytes() * cb_nops(ops);
}

struct CbMeta {
  int cnt;        // products of the item (-1: no more items)
  int off;        // index of the first one in the slot's arrays
  int r0, nrows;  // rows of the block
  int poff;       // index of row r0's extent in the slot's extent array
  int pbase;      // extent of a row minus pbase = index of its first product in the slot
                  // (chunk of a long row: how many such chunks this CTA was handed before this one)
  int ooff;       // index of row r0 in the slot's operand arrays
  int flags;      // 1: chunk of a long row, 2: its last chunk
};

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// Bounded wait that also gives up as soon as ANY thread of the grid has given up (the error word): a role
// that sees `false` leaves its loop, so a broken pipeline ends within about a second instead of hanging.
// The bound is kept on the SM's cycle counter and consulted every 256th attempt only: these waits DO block
// (several per work item), and a %globaltimer read per attempt is far slower than the wake-up itself.
__device__ __forceinline__ bool cb_wait(uint64_t* bar, uint32_t parity, int* err) {
  if (mbar_try_wait(bar, parity)) return true;
  const long long t0 = clock64();
  for (uint32_t spins = 1; !mbar_try_wait(bar, parity); ++spins) {
    if ((spins & 255u) == 0 && (clock64() - t0 > 3000000000ll || *reinterpret_cast<volatile int*>(err) != 0)) {
      atomicExch(err, 1);
      return false;
    }
  }
  return true;
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int MODE, int PM, bool MEURANT, bool GHOST>
__global__ void __launch_bounds__(kCbMaxThreads, 1)
csr_bulk_kernel(const CsrOp A, const int* __restrict__ row_blocks, const int* __restrict__ blk_e0, int nblocks, int ring,
                const Args g, const VecIn in0, const VecIn in1, double* vout) {
  constexpr int NV = SpTraits<MODE>::NV;
  constexpr int OPS = cb_ops(MODE, PM);
  constexpr bool kEpP = OPS & 1, kEpR = (OPS & 2) != 0, kEpD = (OPS & 4) != 0;
  constexpr size_t kSlot = cb_slot_bytes(NV, OPS);
  extern __shared__ __align__(128) unsigned char cb_raw[];
  unsigned char* base = cb_raw + ((128u - (smem_u32(cb_raw) & 127u)) & 127u);
  __shared__ __align__(8) uint64_t full_bar[kCbMaxRing], prod_bar[kCbMaxRing], empty_bar[kCbMaxRing];
  __shared__ CbMeta meta[kCbMaxRing];
  __shared__ double sh_ylong[2];                     // running sum of a long row, handed from chunk to chunk
  __shared__ int sh_long_done;                       // chunks of long rows summed so far
  if (after_stop(g)) return;
  const int tid = threadIdx.x;
  const int R = ring;
  const int nsum = ((int)blockDim.x - kCbSum0) / 32;
  if (tid == 0) {
    sh_ylong[0] = sh_ylong[1] = 0.0; sh_long_done = 0;
    for (int s = 0; s < R; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&prod_bar[s], kCbGather / 32); mbar_init(&empty_bar[s], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  auto slot_val = [&](int s, int c) { return reinterpret_cast<double*>(base + (size_t)s * kSlot + (size_t)c * cb_val_bytes()); };
  auto slot_col = [&](int s) { return reinterpret_cast<int*>(base + (size_t)s * kSlot + (size_t)NV * cb_val_bytes()); };
  auto slot_ptr = [&](int s) { return reinterpret_cast<int*>(base + (size_t)s * kSlot + (size_t)NV * cb_val_bytes() + cb_col_bytes()); };
  auto slot_op = [&](int s, int q) {
    return reinterpret_cast<double*>(base + (size_t)s * kSlot + (size_t)NV * cb_val_bytes() + cb_col_bytes() + cb_ptr_bytes() +
                                     (size_t)q * cb_op_bytes());
  };
  double red[kNRed] = {0.0, 0.0, 0.0, 0.0};
  // timing experiment 2: CTA 0 records, per role, the cycles its first warp spent blocked and its total
  // (dbg_t[10..15]: producer total / blocked, gather total / blocked, summing total / blocked)
  const bool stamp = (g.dbg & 2) && blockIdx.x == 0;
  long long t_blocked = 0;
  const long long t_begin = stamp ? clock64() : 0;
  auto wait = [&](uint64_t* bar, uint32_t parity) {
    if (!stamp) return cb_wait(bar, parity, g.errflag);
    const long long t0 = clock64();
    const bool ok = cb_wait(bar, parity, g.errflag);
    t_blocked += clock64() - t0;
    return ok;
  };

  if (tid >= kCbProducer && tid < kCbSum0) {
    // ------------------------------------------------------------------ producer warp
    const int lane = tid & 31;
    const int G = (int)gridDim.x;
    uint32_t it = 0;                                       // items handed out so far (uniform)
    int nlong = 0;                                         // chunks of long rows handed out so far (uniform)
    bool alive = true;
    // the copies of one item into slot s (executed by ONE lane)
    auto copy_block = [&](int s, int R0, int R1, int E0, int total) {
      const int ea = E0 & ~3, na = (E0 - ea + total + 3) & ~3;
      const int pa = R0 & ~3, np = (R0 - pa + (R1 - R0) + 1 + 3) & ~3;
      const int oa = R0 & ~1, no = (R0 - oa + (R1 - R0) + 1) & ~1;
      const bool stream = na > 0 && !(g.dbg & 16);       // (timing experiment 16: the matrix stream is not copied)
      meta[s] = CbMeta{total, E0 - ea, R0, R1 - R0, R0 - pa, ea, R0 - oa, 0};
      uint64_t* bar = &full_bar[s];
      mbar_arrive_expect_tx(bar, (uint32_t)((stream ? na * 12 : 0) + np * 4 + no * 8 * cb_nops(OPS)));
      if (stream) {
        bulk_g2s(slot_val(s, 0), A.val + ea, (uint32_t)na * 8, bar);
        bulk_g2s(slot_col(s), A.idx + ea, (uint32_t)na * 4, bar);
      }
      bulk_g2s(slot_ptr(s), A.ptr + pa, (uint32_t)np * 4, bar);
      int q = 0;
      if constexpr (kEpP) bulk_g2s(slot_op(s, q++), in0.v + oa, (uint32_t)no * 8, bar);
      if constexpr (kEpR) bulk_g2s(slot_op(s, q++), (MODE == SP_RESID ? g.b : g.r) + oa, (uint32_t)no * 8, bar);
      if constexpr (kEpD) bulk_g2s(slot_op(s, q++), g.dinv + oa, (uint32_t)no * 8, bar);
    };
    for (int b0 = blockIdx.x; b0 < nblocks && alive; b0 += 32 * G) {
      const int blk = b0 + lane * G;
      int r0 = 0, r1 = 0, e0 = 0, e1 = 0;
      if (blk < nblocks) {
        r0 = __ldg(row_blocks + blk); r1 = __ldg(row_blocks + blk + 1);
        e0 = __ldg(blk_e0 + blk); e1 = __ldg(blk_e0 + blk + 1);
      }
      const int nb = min(32, (nblocks - b0 + G - 1) / G);  // blocks of this batch
      if (!__any_sync(0xffffffffu, e1 - e0 > kCbCap)) {
        // every block is one item: lane l's item number, slot and phase follow from l alone
        const uint32_t my = it + (uint32_t)lane, q = my / (uint32_t)R;
        const int s = (int)(my - q * (uint32_t)R);
        for (int l = 0; l < nb; ++l) {
          if (lane == l) {
            if (my >= (uint32_t)R) alive = wait(&empty_bar[s], (q - 1u) & 1u);
            if (alive) copy_block(s, r0, r1, e0, e1 - e0);
          }
          __syncwarp();                                    // one lane after the other, in item order
        }
        it += (uint32_t)nb;
        alive = __all_sync(0xffffffffu, alive);
      } else {
        // a batch with a row longer than an item (rare): one block after the other, metadata by shuffle
        for (int l = 0; l < nb && alive; ++l) {
          const int R0 = __shfl_sync(0xffffffffu, r0, l), R1 = __shfl_sync(0xffffffffu, r1, l);
          const int E0 = __shfl_sync(0xffffffffu, e0, l), E1 = __shfl_sync(0xffffffffu, e1, l);
          const int total = E1 - E0;
          if (lane == 0) {
            for (int cb = 0; (cb == 0 || cb < total) && alive; cb += kCbCap, ++it) {
              const int s = (int)(it % (uint32_t)R);
              if (it >= (uint32_t)R) alive = wait(&empty_bar[s], ((it / (uint32_t)R) - 1u) & 1u);
              if (!alive) break;
              if (total <= kCbCap) { copy_block(s, R0, R1, E0, total); continue; }
              const int cnt = min(kCbCap, total - cb);
              const int ea = (E0 + cb) & ~3, na = (E0 + cb - ea + cnt + 3) & ~3;
              meta[s] = CbMeta{cnt, E0 + cb - ea, R0, 1, 0, nlong++, 0, 1 | (cb + kCbCap >= total ? 2 : 0)};
              mbar_arrive_expect_tx(&full_bar[s], (uint32_t)na * 12);
              bulk_g2s(slot_val(s, 0), A.val + ea, (uint32_t)na * 8, &full_bar[s]);
              bulk_g2s(slot_col(s), A.idx + ea, (uint32_t)na * 4, &full_bar[s]);
            }
          }
          it = __shfl_sync(0xffffffffu, it, 0);
          nlong = __shfl_sync(0xffffffffu, nlong, 0);
          alive = __shfl_sync(0xffffffffu, (int)alive, 0) != 0;
        }
      }
    }
    if (lane == 0) {                                       // end markers: one for every summing warp
      for (int e = 0; e < nsum && alive; ++e, ++it) {
        const int s = (int)(it % (uint32_t)R);
        if (it >= (uint32_t)R) alive = wait(&empty_bar[s], ((it / (uint32_t)R) - 1u) & 1u);
        if (alive) {
          meta[s] = CbMeta{-1, 0, 0, 0, 0, 0, 0, 0};
          mbar_arrive(&full_bar[s]);
        }
      }
      if (stamp) { g.dbg_t[10] = (u64)(clock64() - t_begin); g.dbg_t[11] = (u64)t_blocked; }
    }
  } else if (tid < kCbGather) {
    // ------------------------------------------------------------------ gather warps
    if constexpr (GHOST) {
      if (tid == 0 && g.d.world > 1) {
        for (int c = 0; c < NV; ++c) csr_wait_channel(g, g.hin_ch + c, g.hin_par, g.hin_epoch);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kCbGather) : "memory");
    }
    const int nloc = (int)g.n;
    auto ld0 = [&](int cj) { if constexpr (GHOST) return (cj < nloc ? in0.v : in0.lo - nloc)[cj]; else return in0.v[cj]; };
    auto ld1 = [&](int cj) { if constexpr (GHOST) return (cj < nloc ? in1.v : in1.lo - nloc)[cj]; else return in1.v[cj]; };
    struct GSet { double x[NV][kCbUL]; int cnt, off; };
    struct Pos { int s; uint32_t par; };                   // slot and phase parity of an item
    auto next = [&](Pos p) { if (++p.s == R) { p.s = 0; p.par ^= 1u; } return p; };
    auto gissue = [&](Pos p, GSet& S) {                     // false: end marker
      const int s = p.s;
      if (!wait(&full_bar[s], p.par)) { S.cnt = -1; return false; }
      S.cnt = meta[s].cnt; S.off = meta[s].off;
      const int* col = slot_col(s) + S.off;
#pragma unroll
      for (int u = 0; u < kCbUL; ++u) {
        const int j = tid + u * kCbGather;
        const int cj = j < S.cnt ? col[j] : 0;
        if (g.dbg & 4) { S.x[0][u] = 1.0; if constexpr (NV == 2) S.x[NV - 1][u] = 1.0; continue; }   // (timing experiment: no gathers)
        S.x[0][u] = ld0(cj);
        if constexpr (NV == 2) S.x[NV - 1][u] = ld1(cj);
      }
      return S.cnt >= 0;
    };
    auto gfinish = [&](Pos p, const GSet& S) {
      const int s = p.s;
      double* v0 = slot_val(s, 0) + S.off;
      double* v1 = slot_val(s, NV - 1) + S.off;
#pragma unroll
      for (int u = 0; u < kCbUL; ++u) {
        const int j = tid + u * kCbGather;
        if (j < S.cnt) {
          const double a = v0[j];
          v0[j] = mul_(a, S.x[0][u]);
          if constexpr (NV == 2) v1[j] = mul_(a, S.x[NV - 1][u]);
        }
      }
      // (the proxy fence that orders the generic-proxy accesses to this slot before the producer's next
      // async-proxy copy into it is executed by the summing warp, after it has observed these writes
      // through prod_bar; timing experiment 128 adds one in every gather thread: no measurable difference)
      if (g.dbg & 128) fence_proxy_async_smem();
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(&prod_bar[s]);
    };
    // three items deep: the gathers of items k+1 and k+2 are in flight while the products of item k are
    // written (an L2 round trip under load is longer than one item's worth of work); needs ring >= 3
    GSet S0, S1, S2;
    Pos p0{0, 0u};
    bool m0 = gissue(p0, S0);
    Pos p1 = next(p0);
    bool m1 = m0 && gissue(p1, S1);
    while (m0) {
      Pos p2 = next(p1);
      const bool m2 = m1 && gissue(p2, S2);
      gfinish(p0, S0);
      if (!m1) break;
      p0 = next(p2);
      m0 = m2 && gissue(p0, S0);
      gfinish(p1, S1);
      if (!m2) break;
      p1 = next(p0);
      m1 = m0 && gissue(p1, S1);
      gfinish(p2, S2);
    }
    if (stamp && tid == 0) { g.dbg_t[12] = (u64)(clock64() - t_begin); g.dbg_t[13] = (u64)t_blocked; }
  } else if (tid >= kCbSum0) {
    // ------------------------------------------------------------------ summing warps
    const int lane = tid & 31, sw = (tid - kCbSum0) >> 5;
    auto epilogue = [&](int row, double pv, double rv, double dv, const double (&y)[NV]) {   // the statements of sp_epilogue
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
    constexpr int kStride = (int)(cb_val_bytes() / 8);          // second right-hand side's products
    int s = sw % R;
    uint32_t par = (uint32_t)(sw / R) & 1u;
    for (;; s += nsum) {
      while (s >= R) { s -= R; par ^= 1u; }
      if (!wait(&full_bar[s], par)) break;          // (the metadata; the products follow)
      const CbMeta m = meta[s];
      if (m.cnt < 0) break;
      if (!wait(&prod_bar[s], par)) break;
      const double* prod = slot_val(s, 0);
      if (!(m.flags & 1)) {
        const int* rps = slot_ptr(s) + m.poff;
        for (int t = lane; t < ((g.dbg & 32) ? 0 : m.nrows); t += 32) {
          const int b0 = rps[t] - m.pbase, b1 = (g.dbg & 8) ? b0 + 1 : rps[t + 1] - m.pbase;   // (timing experiment 8: no row sums)
          double y[NV];
#pragma unroll
          for (int c = 0; c < NV; ++c) y[c] = 0.0;
          // products fetched a batch (KB per right-hand side) at a time, one batch ahead of the additions
          // (two register sets); the additions run in stored order: the chain the hardware must serialise
          // is theirs alone
          constexpr int KB = NV == 2 ? 4 : 8;
          typedef double Batch[NV][KB];
          auto fetch = [&](Batch& B, int j) {
#pragma unroll
            for (int c = 0; c < NV; ++c)
#pragma unroll
              for (int q = 0; q < KB; ++q) B[c][q] = prod[c * kStride + j + q];
          };
          auto addup = [&](const Batch& B) {
#pragma unroll
            for (int q = 0; q < KB; ++q)
#pragma unroll
              for (int c = 0; c < NV; ++c) y[c] = add_(y[c], B[c][q]);
          };
          Batch BA, BB;
          int j = b0;
          if (j + KB <= b1) fetch(BA, j);
          while (j + KB <= b1) {
            if (j + 2 * KB <= b1) fetch(BB, j + KB);
            addup(BA);
            j += KB;
            if (j + KB > b1) break;
            if (j + 2 * KB <= b1) fetch(BA, j + KB);
            addup(BB);
            j += KB;
          }
          for (; j < b1; ++j) {
#pragma unroll
            for (int c = 0; c < NV; ++c) y[c] = add_(y[c], prod[c * kStride + j]);
          }
          double pv = 0.0, rv = 0.0, dv = 0.0;
          int q = 0;
          if constexpr (kEpP) pv = slot_op(s, q++)[m.ooff + t];
          if constexpr (kEpR) rv = slot_op(s, q++)[m.ooff + t];
          if constexpr (kEpD) dv = slot_op(s, q++)[m.ooff + t];
          epilogue(m.r0 + t, pv, rv, dv, y);
        }
      } else if (lane == 0) {
        // chunk of a long row: continue the running sum where the previous chunk (maybe another warp's) left it
        volatile int* done = &sh_long_done;
        volatile double* run = sh_ylong;
        const long long t0 = clock64();
        bool ok = true;
        for (uint32_t spins = 1; *done != m.pbase; ++spins) {
          if ((spins & 255u) == 0 && (clock64() - t0 > 3000000000ll || *reinterpret_cast<volatile int*>(g.errflag) != 0)) {
            atomicExch(g.errflag, 1); ok = false; break;
          }
        }
        double yl[NV];
#pragma unroll
        for (int c = 0; c < NV; ++c) yl[c] = run[c];
        for (int j = 0; j < m.cnt; ++j) {
#pragma unroll
          for (int c = 0; c < NV; ++c) yl[c] = add_(yl[c], prod[c * kStride + m.off + j]);
        }
        if (m.flags & 2) {
          double pv = 0.0, rv = 0.0, dv = 0.0;
          if constexpr (kEpP) pv = in0.v[m.r0];
          if constexpr (kEpR) rv = (MODE == SP_RESID) ? g.b[m.r0] : g.r[m.r0];
          if constexpr (kEpD) dv = g.dinv[m.r0];
          epilogue(m.r0, pv, rv, dv, yl);
#pragma unroll
          for (int c = 0; c < NV; ++c) yl[c] = 0.0;
        }
#pragma unroll
        for (int c = 0; c < NV; ++c) run[c] = yl[c];
        __threadfence_block();
        if (ok) *done = m.pbase + 1;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
    }
    if (stamp && tid == kCbSum0) { g.dbg_t[14] = (u64)(clock64() - t_begin); g.dbg_t[15] = (u64)t_blocked; }
  }
  spmv_close<MODE, MEURANT>(g, red);
}

}  // namespace cgx
