// cgx_host.h -- host-side declarations shared by the translation units of libcgx_b200.so
// (cgx.cu: context + C ABI; cgx_iter.cu: the stage launchers, one object per preconditioner
// mode; cgx_pers.cu: the persistent-kernel launchers, one object per operator kind;
// cgx_fused.cu: single-launch iterations).  The split exists only so that the many template
// instantiations compile in parallel.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/cgx.h"
#include "cgx_kernels.cuh"
#include "cgx_stencil_tma.cuh"
#include "cgx_csr_bulk.cuh"
#include "cgx_persistent.cuh"
#include "cgx_varstencil.cuh"

using namespace cgx;

int cgx_fail(int code, const char* fmt, ...);
#define fail cgx_fail

#define CU(call)                                                                        \
  do {                                                                                  \
    cudaError_t e_ = (call);                                                            \
    if (e_ != cudaSuccess)                                                              \
      return fail(CGX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                  \
  } while (0)

struct Nid { char b[128]; };        // ncclUniqueId (passed by value)
struct NcclApi {
  void* h = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Nid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
extern NcclApi g_nccl;

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
enum { V_X = 0, V_R, V_RT, V_P, V_S, V_ST, V_W, V_WT, V_U, V_T, V_COUNT };
extern const char* const kVecNames[];

struct cgx_ctx {
  int device = 0;
  int sm_count = 148;
  int smem_per_sm = 233472;         // cudaDevAttrMaxSharedMemoryPerMultiprocessor
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  // operator
  int op_kind = 0;  // 0 none, 1 csr, 2 stencil, 3 variable-coefficient stencil
  CsrOp csr{};
  StencilOp sten{};
  VarStencilOp vsten{};
  double* d_coef[4] = {};          // op_kind 3: diag, cx, cy, cz (cz null in 2-D)
  CUtensorMap coef_tmap[3];        // op_kind 3: cx, cy, cz (encoded by cgx_set_stencil_coef_host)
  bool coef_tmap_ok = false;
  int* d_ptr = nullptr;
  int* d_idx = nullptr;
  double* d_val = nullptr;
  std::vector<int> h_ptr;          // host copy of indptr (persistent kernel: shared-memory slab sizing)
  bool no_elide = false;           // cgx_set_option("cg_elide", 0)
  bool no_slab = false;            // cgx_set_option("csr_slab", 0)
  int* d_send_idx = nullptr;       // CSR row partition: local rows to send (Dist::send_idx)
  int* d_rowblk = nullptr;         // CSR-stream row blocks (cgx_kernels.cuh)
  int* d_rowblk_e0 = nullptr;      // first non-zero of every row block (= indptr[row_blocks[b]])
  int n_rowblk = 0;
  int* d_rowblk_b = nullptr;       // the same for the bulk-copy CSR kernel (kCbRows / kCbCap: cgx_csr_bulk.cuh)
  int* d_rowblk_b_e0 = nullptr;
  int n_rowblk_b = 0;
  int csr_bulk = 1;                // option "csr_bulk": 0 = csr_stream_kernel, 1 = csr_bulk_kernel (cgx_csr_bulk.cuh) for one right-hand side, 2 = for both
  int csr_bulk_ring = 0;           // option "csr_bulk_ring": slots per CTA (0 = what csr_bulk_ctas resident CTAs per SM allow)
  int csr_bulk_sum = 4;            // option "csr_bulk_sum": summing warps per CTA (1 .. kCbMaxSum)
  int csr_bulk_ctas = 1;           // option "csr_bulk_ctas": resident CTAs per SM the ring is sized for
  i64 n = 0, nnz = 0;
  // preconditioner: pm = 0 identity, 1 Jacobi vector, 2 Jacobi with a constant diagonal
  double* d_dinv = nullptr;
  double dinv_s = 1.0;
  int pm = 0;
  // TMA-staged stencil path
  bool use_tma = false;
  int dbg = 0;                     // option "debug_skip" (timing experiments only)
  u64* d_dbg_t = nullptr;          // 16 time stamps (dbg & 2)
  bool cg_elide = false;           // CG-CG: r~ / GV: w~ not stored (EW_*_E / SP_*_E)
  bool one_wave = false;           // option "ew_one_wave": single-GPU vector passes also launch one resident wave
  int tma_min_planes = 4;          // option "tma_min_planes": planes per CTA the stencil grid aims for at least
  bool halo_ll = false;            // multi-GPU: the fused SpMV passes are TMA kernels -> LL ghost planes
  bool no_tma = false;             // cgx_set_option("tma", 0): force the generic stencil kernel
  bool no_csr_stream = false;      // cgx_set_option("csr_stream", 0): one thread per row
  TmaGeom geom{};
  int tma_grid[2] = {0, 0};        // grid size for 1 / 2 right-hand sides
  CUtensorMap tmap[10];
  bool tmap_ok[10] = {};
  // problem
  double* d_b = nullptr;
  double* d_x0 = nullptr;
  double* d_xtrue = nullptr;
  bool own_problem = false, has_xtrue = false, problem_loaded = false;
  // state
  double* vec[V_COUNT] = {};
  Scal* d_sc = nullptr;            // [2]: multi-GPU runs alternate (Args::scpar)
  double* d_partials = nullptr;
  unsigned* d_ticket = nullptr;
  double* d_hist = nullptr;
  int hist_len = 0;
  unsigned hist_mask = 0;
  bool ran = false;
  i64 launches = 0;
  // per-kernel-class profiling
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;
  std::vector<int> prof_cls;
  size_t prof_used = 0;
  double prof_ms[32] = {};
  i64 prof_n[32] = {};
  // multi-GPU (dist.world > 1): window, peers, epochs (cgx_common.cuh "Row-partitioned ...")
  Dist dist{};
  unsigned char* d_win = nullptr;
  size_t win_bytes = 0;
  unsigned char* peer_base[kMaxWorld] = {};
  bool peer_ipc[kMaxWorld] = {};
  bool dist_ready = false;
  cudaStream_t own_stream = nullptr;      // c->stream may be a group's shared stream
  u64 epoch = 0;                           // last scalar-exchange epoch produced
  u64 hepoch[kChan] = {};                  // last halo epoch produced per channel
  u64 fepoch = 0;                          // fused PR kernel: epoch of the LL ghost planes of p, s, rt
  int scpar = 0;
  struct Pend { u64 e; int kind; int k; };
  std::vector<Pend> pend;
  // mode 2: NCCL allreduce of the records on a side stream
  void* nccl_comm = nullptr;
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_prod[kSlots] = {}, ev_red[kSlots] = {};
  double* d_nccl = nullptr;                // [2][kSlots][kSumW]: in, out
  // persistent path
  double* d_ppart = nullptr;               // [2][kPersMaxGrid][kPersRed]
  u64* d_pbar = nullptr;                   // sync-point counter
  PersOut* d_pout = nullptr;
  void* d_prank = nullptr;                 // PersRank<Op>[kMaxWorld] (rank 0 of a group holds all)
  void* d_pbatch = nullptr;                // PersEntry<Op>[] of the last cgx_batch_run this context led
  size_t pbatch_bytes = 0;
  double* d_exp[2][2] = {};                // exported SpMV inputs [parity][rhs]
  int pers_threshold = 1 << 19;            // AUTO: rows below which the persistent kernel runs
  int pers_threads = 0, pers_ctas = 0;     // 0 = choose (options "pers_threads", "pers_ctas")
  // current run
  // PR-CG / M-CG in one launch per iteration (cgx_stencil_fused.cuh): p, s, rt ping-pong between
  // vec[] (parity 0) and alt[] (parity 1)
  bool pr_fused = false, no_fused = false;
  int fpar = 0;
  double* alt[3] = {};                     // second buffers of p, s, rt
  double* d_gscr = nullptr;                // partitioned: [2][plane] scratch (new p of the ghost planes)
  CUtensorMap ftmap[2][3];
  int pdl_mode = 1;                        // option "pdl": 0 off, 1 single-GPU contexts (default), 2 always
  int l2_keep = -1;                        // option "l2_keep": -1 auto (partitioned runs whose state fits L2), 0 off, 1 on
  int fused_min_slab = 64;                 // partitioned runs: planes per rank from which the fused kernel is used
  int fused_min_planes = 8, fused_chunks = 0;   // options: planes per CTA at least / force the chunk count
  // capture of x_k / r_k / (a, b) after every iteration, GV residual replacement (include/cgx.h)
  unsigned capture = 0, capture_req = 0;
  double* d_cap[3] = {};                   // x [max_iter][n], r [max_iter][n], scalars [2][max_iter]
  std::vector<uint8_t> gv_replace;
  bool gv_manual = false;                  // option "gv_manual": w may be replaced by hand (cgx_gv_replace_now): no w~ elision
  int cur_stage = 0;                       // cgx_advance_stages: next stage of iteration cur_k + 1
  std::map<std::pair<const void*, size_t>, int> occ;   // ctx_occupancy cache (per device)
  int* d_tma_err = nullptr;                // set by a TMA wait that expired (mbar_wait)
  int variant = 0, max_iter = 0, cur_k = 0, path = CGX_PATH_STREAM;
  // relative tolerance (cgx_set_tolerance): requested, and in force for the current run
  double tol = 0.0, run_tol = 0.0;
  int stop_k = -1;                         // host copy of Scal::stop_k once the run has stopped
  int* h_stop = nullptr;                   // pinned: stop_k after chunk j of the stream loop, slot j & 1
  cudaEvent_t ev_stop[2] = {nullptr, nullptr};
  i64 launches_run = 0;
  double setup_ms = 0.0, loop_ms = 0.0;
};

inline int grid_for(const cgx_ctx* c, i64 work_items) {
  i64 g = (work_items + kBlock - 1) / kBlock;
  i64 cap = (i64)c->sm_count * 8;   // 8 resident CTAs of 256 threads per SM
  if (cap > kMaxGrid) cap = kMaxGrid;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// ---------------------------------------------------------------------------------------
// launch bookkeeping
// ---------------------------------------------------------------------------------------
// Optional per-kernel-class timing (cgx_set_profile): an event pair around every launch of
// the iteration loop, resolved after the stream has drained.  Off in timed runs.
enum { PC_EW0 = 0, PC_SP0 = 7, PC_INSTR = 15, PC_FUSED = 16, PC_COUNT = 17 };

struct ProfScope {
  cgx_ctx* c; int cls; size_t slot = 0; bool on;
  ProfScope(cgx_ctx* c_, int cls_) : c(c_), cls(cls_), on(c_->profile) {
    if (!on) return;
    if (c->prof_used + 2 > c->prof_events.size()) {
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); c->prof_events.push_back(e); }
    }
    slot = c->prof_used; c->prof_used += 2;
    c->prof_cls.push_back(cls);
    cudaEventRecord(c->prof_events[slot], c->stream);
  }
  ~ProfScope() { if (on) cudaEventRecord(c->prof_events[slot + 1], c->stream); }
};

Args make_args(cgx_ctx* c);

// What one launch does in the multi-GPU protocol (cgx_common.cuh "Row-partitioned ..."):
struct Plan {
  bool consume = false;      // needs alpha/beta: folds every pending reduction into the scalars
  int produce = FK_NONE;     // publishes a reduction record of this kind (FK_*; -1: instrumentation)
  int hout_n = 0, hout_ch = 0;   // writes boundary planes of `hout_n` SpMV inputs into the neighbours
  int hin_n = 0, hin_ch = 0;     // reads ghost planes
};
enum { FK_INSTR = 100 };

void plan_apply(cgx_ctx* c, Args& g, const Plan& p);
void plan_commit(cgx_ctx* c, const Args& g, const Plan& p);
VecIn vec_in(cgx_ctx* c, const double* v, int ch, const Args& g);

// Resident CTAs per SM of kernel `fn` on THIS context's device (the dynamic-shared-memory opt-in
// is a per-device attribute, so it is applied -- and the result cached -- per context).
int ctx_occupancy(cgx_ctx* c, const void* fn, int threads, size_t smem);

// Launch with programmatic stream serialisation when `pdl` (cgx_common.cuh "programmatic dependent launch").
template <class... KArgs, class... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// (measured on 8 GPUs, 256^3: 50.1 us/iteration with it, 48.5 without -- the early-resident CTAs of the next
// kernel do not pay off when every kernel starts by waiting for its peers; one GPU at the same slab size:
// 37.3 vs 41.0.  Hence: single-GPU contexts only, unless the option forces it with value 2.)
inline bool use_pdl(const cgx_ctx* c) { return c->pdl_mode == 2 || (c->pdl_mode == 1 && c->dist.world <= 1); }

inline size_t tma_smem_bytes(int nv) { return stencil_smem_bytes(nv); }

// Stream path with a tolerance: iterations issued between two looks at stop_k.  The host waits for chunk
// j - 2 before it enqueues chunk j, so the queue stays at least a chunk deep and the launches issued after
// the stop (all of which return at entry) are at most two chunks' worth.
constexpr int kTolChunk = 32;

// kernel launches ("stages") of one iteration without the instrumentation
// (a CSR row partition adds one stage: the gather-and-push of the SpMV input's ghost entries)
inline bool csr_dist(const cgx_ctx* c) { return c->dist.world > 1 && c->dist.csr; }
inline int core_stages(const cgx_ctx* c) { return c->pr_fused ? 1 : (c->variant == CGX_HS ? 3 : 2) + (csr_dist(c) ? 1 : 0); }
bool tma_encode_dims(double* ptr, i64 nx, i64 ny, i64 nz, CUtensorMap* out);
// cgx_fused.cu
int cgx_fused_prepare(cgx_ctx* c);              // second buffers + tensor maps; sets c->pr_fused
void cgx_launch_pr_fused(cgx_ctx* c, Args g);   // one whole PR-CG / M-CG iteration
void cgx_fused_push_initial_halo(cgx_ctx* c);   // partitioned runs: boundary planes of the initial p, s, rt
double* cgx_cur_vec(cgx_ctx* c, int v);         // the buffer that currently holds state vector v

void launch_halo_push(cgx_ctx* c, Args g, const double* v, int ch);
void launch_halo_push2(cgx_ctx* c, Args g, const double* v0, const double* v1, int ch);
void launch_instrument(cgx_ctx* c, Args g);
void launch_hist_consume(cgx_ctx* c, Args g);
void launch_capture(cgx_ctx* c, const Args& g);

struct VariantInfo {
  bool meurant, pipe, recompute;
  int cls;                 // init_scalars class
  unsigned need;           // bitmask of state vectors
};
VariantInfo variant_info(int v, bool prec);

// stage s of one iteration, per preconditioner mode (cgx_iter.cu compiled with -DCGX_PM=0|1|2)
void cgx_iter_stage_pm0(cgx_ctx* c, int s, const Args& g);
void cgx_iter_stage_pm1(cgx_ctx* c, int s, const Args& g);
void cgx_iter_stage_pm2(cgx_ctx* c, int s, const Args& g);

struct PersGeom { int T, nb, R, nslot, slab_cap; unsigned vmask; size_t smem; bool ok; };

// persistent path, per operator kind (cgx_pers.cu compiled with -DCGX_PERS_OP=1 CSR | 2 stencil | 3 variable-coefficient
// stencil and -DCGX_PERS_PM=0|1|2)
#define CGX_PERS_DECL(name) int name(cgx_ctx** cs, int count, const PersGeom& G, int k0, int k1)
CGX_PERS_DECL(cgx_pers_launch_csr_pm0); CGX_PERS_DECL(cgx_pers_launch_csr_pm1); CGX_PERS_DECL(cgx_pers_launch_csr_pm2);
CGX_PERS_DECL(cgx_pers_launch_sten_pm0); CGX_PERS_DECL(cgx_pers_launch_sten_pm1); CGX_PERS_DECL(cgx_pers_launch_sten_pm2);
CGX_PERS_DECL(cgx_pers_launch_var_pm0); CGX_PERS_DECL(cgx_pers_launch_var_pm1); CGX_PERS_DECL(cgx_pers_launch_var_pm2);
// batch of independent solves in one cooperative launch (cgx_batch_run); launch = false: co-residency check only
#define CGX_PERS_BATCH_DECL(name) int name(cgx_ctx** cs, int count, const int* variants, const PersGeom* G, const int* k1, bool launch)
CGX_PERS_BATCH_DECL(cgx_pers_batch_csr_pm0); CGX_PERS_BATCH_DECL(cgx_pers_batch_csr_pm1); CGX_PERS_BATCH_DECL(cgx_pers_batch_csr_pm2);
CGX_PERS_BATCH_DECL(cgx_pers_batch_sten_pm0); CGX_PERS_BATCH_DECL(cgx_pers_batch_sten_pm1); CGX_PERS_BATCH_DECL(cgx_pers_batch_sten_pm2);
