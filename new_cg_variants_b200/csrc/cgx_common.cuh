// cgx_common.cuh -- shared device-side definitions for libcgx_b200 (sm_100a only).
//
// Numerical contract (DESIGN.md section "Arithmetic"): every elementwise update and every
// matrix row sum is evaluated with separately rounded IEEE multiply/add in the operand
// order of the reference's numpy/scipy expressions (no FMA contraction: the __d*_rn
// intrinsics are never fused by nvcc), so those steps are bit-identical to the reference.
// Only the inner products differ from OpenBLAS: they are accumulated with FMA in a fixed,
// run-to-run deterministic order (per-thread strided partial -> warp butterfly -> block ->
// fixed-order cross-block sum by the last-arriving block).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cgx {

typedef long long i64;

constexpr int kBlock = 256;          // threads per CTA for streaming kernels
constexpr int kMaxGrid = 148 * 16;   // upper bound on CTAs of any reducing kernel
constexpr int kNRed = 4;             // at most four fused inner products per pass

// Device-resident scalar recurrences.  One instance per context; written only by the
// finalising thread of a reducing kernel (or by init_scalars), read by every CTA of the
// next kernel.  Kernel boundaries order the accesses.
struct Scal {
  double a;    // alpha_{k-1} when an iteration starts, alpha_k when it ends
  double a1;   // previous alpha
  double b;    // beta the next vector pass applies
  double nu, nu1, mu, eta, del, gam;
  double tmp[8];      // initialisation dot products
  int breakdown;      // -1, or first k with a non-finite alpha/beta
  int stop_k;         // -1, or first k >= 1 with nu_k <= thr (cgx_set_tolerance); the run ends after iteration stop_k
  double thr;         // tol^2 * nu_0, or NaN when no tolerance is set (no nu satisfies the test)
};

// ---- arithmetic that must mirror numpy's two-rounding elementwise expressions ---------
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double div_(double a, double b) { return __ddiv_rn(a, b); }
// x + a*p  and  r - a*s  exactly as numpy evaluates `x + a * p`, `r - a * s`
__device__ __forceinline__ double axpy_(double x, double a, double p) { return add_(x, mul_(a, p)); }
__device__ __forceinline__ double axmy_(double r, double a, double s) { return sub_(r, mul_(a, s)); }

// ---- 1- and 2-wide packs for 128-bit global accesses ----------------------------------
template <int W> struct Pk { double v[W]; };

// pol != 0: an L2 cache-policy word (createpolicy encoding, e.g. kL2EvictLast) -- partitioned runs whose
// per-GPU working set fits the 126 MB L2 ask the cache to keep the state vectors (global pointers only).
constexpr unsigned long long kL2EvictLast = 0x14F0000000000000ull;     // fractional 1.0, L2::evict_last
template <int W> __device__ __forceinline__ Pk<W> ldp(const double* __restrict__ p, i64 i, unsigned long long pol = 0) {
  Pk<W> o;
  if constexpr (W == 2) {
    double2 t;
    if (pol) asm volatile("ld.global.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(t.x), "=d"(t.y) : "l"(p + i), "l"(pol));
    else t = *reinterpret_cast<const double2*>(p + i);
    o.v[0] = t.x; o.v[1] = t.y;
  } else {
    o.v[0] = p[i];
  }
  return o;
}
template <int W> __device__ __forceinline__ void stp(double* __restrict__ p, i64 i, const Pk<W>& o, unsigned long long pol = 0) {
  if constexpr (W == 2) {
    if (pol) asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1,%2}, %3;" ::"l"(p + i), "d"(o.v[0]), "d"(o.v[1]), "l"(pol) : "memory");
    else *reinterpret_cast<double2*>(p + i) = make_double2(o.v[0], o.v[1]);
  } else {
    p[i] = o.v[0];
  }
}

// ---- programmatic dependent launch (the kernels of the iteration loop are launched with
//      cudaLaunchAttributeProgrammaticStreamSerialization): a kernel lets its successor start launching at
//      once and does not touch global memory before its predecessor has completed -- the successor's
//      launch latency and prologue (barrier init, index math) overlap the predecessor's tail.  Both are
//      no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- mbarrier helpers (producer / consumer pipelines inside a CTA) --------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t global_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait: a copy that never lands (bad descriptor) must fail loudly, not hang the GPU.
// The flag is checked by the host after every synchronisation (CGX_ERR_CUDA).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = global_ns();
  while (!mbar_try_wait(bar, parity)) {
    if (global_ns() - t0 > 1000000000ull) { atomicExch(err, 1); return; }
  }
}

// ---- deterministic reductions ---------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;   // butterfly: every lane holds the same bits
}

// Sum NR per-thread values over the CTA; result valid in thread 0.  `sh` holds
// NR * (blockDim.x / 32) doubles.
template <int NR>
__device__ __forceinline__ void block_sum(double (&v)[NR], double* sh) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int j = 0; j < NR; ++j) v[j] = warp_sum(v[j]);
  __syncthreads();   // protect `sh` against the previous use
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < NR; ++j) sh[j * nw + wid] = v[j];
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int j = 0; j < NR; ++j) {
      double t = (lane < nw) ? sh[j * nw + lane] : 0.0;
      v[j] = warp_sum(t);
    }
  }
}

// Grid-wide sum of NR values with a fixed summation order, finished by whichever CTA
// arrives last (ticket counter); `fin(acc)` runs in ONE thread with the totals.
// partials: [gridDim.x][NR].  The order in which CTAs arrive does not influence the bits.
// `sys`: the CTAs also stored into peer memory (halo planes); make those stores visible
// system-wide before the ticket so that the finishing CTA may publish them.
template <int NR, class Fin>
__device__ __forceinline__ void grid_sum_finalize(double (&v)[NR], double* __restrict__ partials,
                                                  unsigned* __restrict__ ticket, Fin fin,
                                                  bool sys = false) {
  __shared__ double sh[NR * 32];          // any CTA width up to 1024 threads
  __shared__ bool is_last;
  block_sum<NR>(v, sh);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int j = 0; j < NR; ++j) __stcg(&partials[(i64)blockIdx.x * NR + j], v[j]);
    if (sys) __threadfence_system(); else __threadfence();
    unsigned t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double acc[NR];
#pragma unroll
  for (int j = 0; j < NR; ++j) acc[j] = 0.0;
  for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
#pragma unroll
    for (int j = 0; j < NR; ++j) acc[j] += __ldcg(&partials[(i64)i * NR + j]);
  }
  block_sum<NR>(acc, sh);
  if (threadIdx.x == 0) {
    *ticket = 0u;
    fin(acc);
  }
}

// For kernels without a reduction that still have something to publish when the whole grid
// is done (halo epochs): `fin()` runs in one thread of the CTA that arrives last.
template <class Fin>
__device__ __forceinline__ void grid_last_finalize(unsigned* __restrict__ ticket, Fin fin, bool sys = true) {
  __shared__ bool is_last0;
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sys) __threadfence_system(); else __threadfence();
    unsigned t = atomicAdd(ticket, 1u);
    is_last0 = (t == gridDim.x - 1);
    if (is_last0) { *ticket = 0u; fin(); }
  }
}

__device__ __forceinline__ void note_breakdown(Scal* sc, int k, double a, double b) {
  if (sc->breakdown < 0 && !(isfinite(a) && isfinite(b))) sc->breakdown = k;
}
// Called wherever nu_k is assigned: the natural norm of the updated residual, r~_k . r_k, against
// tol^2 nu_0.  A NaN nu (or threshold) never satisfies the test.
__device__ __forceinline__ void note_stop(Scal* sc, int k) {
  if (sc->stop_k < 0 && k >= 1 && sc->nu <= sc->thr) sc->stop_k = k;
}
// A launch that belongs to iteration k after the one at which the tolerance was met does nothing.
__device__ __forceinline__ bool past_stop(const Scal* sc, int k) {
  const int s = sc->stop_k;
  return s >= 0 && k > s;
}

// =====================================================================================
// Row-partitioned multi-GPU runs (one rank per GPU, z-slabs of the stencil grid).
//
// Every rank owns a "window": a device allocation that its peers map (CUDA IPC between
// processes, plain pointers inside one process) and write into directly over NVLink.
//   * scalar exchange: the CTA that finishes a fused reduction stores the rank's partial
//     sums into slot (epoch % kSlots) of EVERY rank's window, then the epoch number into
//     the matching flag (release, system scope).  The next kernel that needs alpha/beta
//     waits for all ranks' flags, adds the partials in rank order (bit-identical on every
//     GPU) and evaluates the scalar recurrences redundantly -- a one-hop all-to-all
//     "allreduce" with no extra launch.  (mode 2 swaps this for ncclAllReduce on a side
//     stream; the flags are then not used.)
//   * halo exchange: the vector pass that produces the SpMV input also stores its first
//     and last plane into the neighbours' ghost planes (double-buffered by parity), and
//     its last CTA publishes the halo epoch; the stencil kernel waits for that epoch only
//     before it touches a ghost plane.
// A kernel never waits for something produced by the same stage of another rank, so the
// ranks may also be emulated as contexts sharing one stream on one GPU (tests).
// =====================================================================================
constexpr int kMaxWorld = 8;
constexpr int kSumW = 8;     // doubles per exchanged record
constexpr int kSlots = 8;    // ring depth of the scalar exchange (see DESIGN.md "Epochs")
constexpr int kChan = 4;     // halo channels: 0,1 SpMV inputs, 2 x (instrumentation), 3 x_true

typedef unsigned long long u64;

struct WinHdr {
  // scalar records, "LL" style: every 8-byte word carries half a double and the epoch tag
  // ((epoch32 << 32) | 32 data bits), so a record needs no separate flag and no fence: the
  // consumer polls the words themselves (aligned 8-byte stores are single-copy atomic, also
  // across NVLink).  [slot][producer rank][2 words per value]
  u64 ll[kSlots][kMaxWorld][2 * kSumW];
  u64 hflag[kChan][2][2];          // [channel][parity][side]; side 0 = plane below, 1 = above
  u64 gflag[kChan][2][kMaxWorld];  // general CSR partition: [channel][parity][source rank] ghost-entry epochs
  int error;                       // set when a bounded wait expired
  int pad;
};
constexpr size_t kWinHdrBytes = (sizeof(WinHdr) + 1023) / 1024 * 1024;   // ghost planes follow

enum { FK_NONE = 0, FK_HS_NU, FK_HS_MU, FK_CGGV, FK_PR_NU, FK_PR_SP, FK_PIPE, FK_INIT };

struct Dist {
  int world, rank, mode;           // mode: 1 peer-to-peer scalars, 2 NCCL scalars, 3 timing stub (local only)
  int saved_mode;
  int has_lo, has_hi;              // a neighbour slab exists below / above
  WinHdr* win[kMaxWorld];          // every rank's window header (win[rank] is local)
  double* ghost;                   // local ghost planes [kChan][2 parity][2 side][plane]
  double* ghost_lo;                // ghost planes of the rank below (peer mapped) or null
  double* ghost_hi;
  // persistent kernel: ghost planes as LL words (2 x u64 per value, tag = halo epoch):
  // [3 channels][2 parity][2 side][2 * plane]; no flags, no fences, element-wise arrival
  u64* ghl;
  u64* ghl_lo;
  u64* ghl_hi;
  double* nccl_in;                 // mode 2: [kSlots][kSumW] local partials / reduced totals
  double* nccl_out;
  i64 plane;                       // points per exchanged plane
  // ---- general CSR row partition (SURVEY.md section 8e "General CSR"): the ghost entries of an SpMV
  //      input are gathered by index lists.  Rank r's window holds a staging array
  //      [kChan][2 parity][nghost_of[r]] after the header; the column indices of the local matrix
  //      address it as n_local + j.  A source rank's entries form one contiguous segment of it.
  int csr;                         // 1: this partition is a CSR row partition (no slabs, no planes)
  int nghost;                      // ghost entries of this rank
  unsigned src_mask;               // ranks this rank receives ghost entries from
  int send_ptr[kMaxWorld + 1];     // this rank's send entries per destination rank (prefix sums)
  int send_off[kMaxWorld];         // where this rank's segment starts in the destination's staging array
  int nghost_of[kMaxWorld];        // staging length of every rank
  const int* send_idx;             // device: local row indices to send, concatenated per destination
  double* stage_of[kMaxWorld];     // every rank's staging array (peer mapped)
};

__device__ __forceinline__ u64 ld_acquire_sys(const u64* p) {
  u64 v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(u64* p, u64 v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ u64 timer_ns() {
  u64 t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait for *flag >= epoch.  A peer that never arrives must surface as an error
// (CGX_ERR_CUDA after the next synchronisation), not as a hung GPU.
// (the clock and the error flag are looked at once per 64 polls: reading %globaltimer in every
// spin would put a microsecond of granularity on each cross-GPU dependency)
__device__ __forceinline__ void wait_epoch(const u64* flag, u64 epoch, int* err) {
  if (ld_acquire_sys(flag) >= epoch) return;
  const u64 t0 = timer_ns();
  for (;;) {
#pragma unroll 1
    for (int spin = 0; spin < 64; ++spin)
      if (ld_acquire_sys(flag) >= epoch) return;
    if (*(volatile int*)err) return;
    if (timer_ns() - t0 > 10000000000ull) { atomicExch(err, 1); return; }
  }
}
__host__ __device__ __forceinline__ size_t ghl_off(const Dist& d, int ch, int par, int side) {
  return ((size_t)(ch * 2 + par) * 2 + side) * 2 * (size_t)d.plane;
}
__device__ __forceinline__ void ll_store(u64* dst, double v, u64 epoch) {
  const u64 b = (u64)__double_as_longlong(v), tag = (epoch & 0xffffffffull) << 32;
  // one 16-byte store (dst is 16-byte aligned); each 8-byte half validates itself
  asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"((b & 0xffffffffull) | tag),
               "l"((b >> 32) | tag) : "memory");
}
__device__ __forceinline__ u64 ll_poll(const u64* src, u64 tag32, int* err) {
  u64 w;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
  if ((w >> 32) == tag32) return w;
  const u64 t0 = timer_ns();
  for (;;) {
#pragma unroll 1
    for (int spin = 0; spin < 64; ++spin) {
      asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
      if ((w >> 32) == tag32) return w;
    }
    if (*(volatile int*)err) return w;
    if (timer_ns() - t0 > 10000000000ull) { atomicExch(err, 1); return w; }
  }
}
// value j of the record of `epoch` (bounded wait; see wait_epoch)
__device__ __forceinline__ double ll_load(const u64* rec, int j, u64 epoch, int* err) {
  const u64 tag = epoch & 0xffffffffull;
  const u64 lo = ll_poll(rec + 2 * j, tag, err), hi = ll_poll(rec + 2 * j + 1, tag, err);
  return __longlong_as_double((long long)((lo & 0xffffffffull) | (hi << 32)));
}
// both words of value j with ONE 16-byte load, re-polled until both carry the tag
__device__ __forceinline__ double ll_load16(const u64* rec, int j, u64 epoch, int* err) {
  const u64 tag = epoch & 0xffffffffull;
  const u64* src = rec + 2 * j;
  u64 lo, hi;
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(src) : "memory");
  if ((lo >> 32) != tag || (hi >> 32) != tag) {
    const u64 t0 = timer_ns();
    bool ok = false;
    while (!ok) {
#pragma unroll 1
      for (int spin = 0; spin < 64 && !ok; ++spin) {
        asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(src) : "memory");
        ok = (lo >> 32) == tag && (hi >> 32) == tag;
      }
      if (ok || *(volatile int*)err) break;
      if (timer_ns() - t0 > 10000000000ull) { atomicExch(err, 1); break; }
    }
  }
  return __longlong_as_double((long long)((lo & 0xffffffffull) | (hi << 32)));
}
// Split form of ll_load16: issue the 16-byte load now, validate (and re-poll) later, so that
// several records and other loads are in flight together.
struct LLReq { const u64* src; u64 lo, hi; };
__device__ __forceinline__ void ll_issue(LLReq& r) {
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(r.lo), "=l"(r.hi) : "l"(r.src) : "memory");
}
__device__ __forceinline__ double ll_finish(LLReq& r, u64 epoch, int* err) {
  const u64 tag = epoch & 0xffffffffull;
  if ((r.lo >> 32) != tag || (r.hi >> 32) != tag) {
    r.lo = ll_poll(r.src, tag, err);
    r.hi = ll_poll(r.src + 1, tag, err);
  }
  return __longlong_as_double((long long)((r.lo & 0xffffffffull) | (r.hi << 32)));
}
// Out-of-line variant for rarely taken paths (keeps the polling loop out of hot code).
static __device__ __noinline__ double ll_load16_cold(const u64* rec, int j, u64 epoch, int* err) {
  return ll_load16(rec, j, epoch, err);
}
// Warp-collective: all-rank totals of the record of `epoch` (NQ = 4 or 8 sums, the first `nr`
// are live).  Lane l fetches value (l & 3) [+4] of rank (l >> 2): every word of the record is
// in flight at once -- one L2 round trip instead of one per value -- and the sums are formed in
// rank order by shuffles, identically in every warp of every GPU.  only_rank >= 0: timing stub
// (that rank's record times the number of ranks).
template <int NQ>
__device__ __forceinline__ void ll_totals(WinHdr* w, int slot, u64 epoch, int world, int nr, int only_rank,
                                          double (&acc)[NQ]) {
  const int lane = threadIdx.x & 31, r = lane >> 2, j = lane & 3;
#pragma unroll
  for (int h = 0; h < NQ / 4; ++h) {
    const int jj = j + 4 * h;
    double v = 0.0;
    if (r < world && jj < nr && (only_rank < 0 || r == only_rank)) v = ll_load16(w->ll[slot][r], jj, epoch, &w->error);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      double t = 0.0;
      for (int rr = 0; rr < world; ++rr) t += __shfl_sync(0xffffffffu, v, rr * 4 + q);
      acc[4 * h + q] = (only_rank >= 0) ? t * (double)world : t;
    }
  }
}
__host__ __device__ __forceinline__ size_t ghost_off(const Dist& d, int ch, int par, int side) {
  return ((size_t)(ch * 2 + par) * 2 + side) * (size_t)d.plane;
}

}  // namespace cgx
