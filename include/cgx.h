/* cgx.h -- C ABI of libcgx_b200.so: the B200 (sm_100a) implementation of the
 * predict-and-recompute CG inner loop of tchen-research/new_cg_variants.
 *
 * The reference has NO native boundary (it is pure Python on numpy/scipy); this header is
 * the boundary a binding for it would use.  Each entry point names the reference
 * interface it replaces (paths relative to predict_and_recompute/ in the reference).
 *
 * Conventions
 *   - plain C, no C++/torch types; every function returns a cgx_status (0 = ok) except
 *     the two getters; no exception crosses the ABI; the message of the last error of the
 *     calling thread is available from cgx_last_error().
 *   - "_host" pointers are ordinary host memory (numpy buffers); the library copies
 *     them to/from the device.  "_dev" pointers are device pointers on the context's GPU
 *     owned by the caller (e.g. torch tensors).
 *   - a context is bound to one GPU and owns one stream; it is not re-entrant.  Distinct
 *     contexts may be driven from distinct host threads/processes (one per GPU).
 *   - all floating point is IEEE binary64; indices are int32 (scipy's CSR index type).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with CGX_ERR_CUDA.
 */
#ifndef CGX_H_
#define CGX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGX_VERSION 100

typedef enum {
  CGX_OK = 0,
  CGX_ERR_ARG = 1,        /* bad argument / call order */
  CGX_ERR_CUDA = 2,       /* CUDA runtime error (see cgx_last_error) */
  CGX_ERR_BREAKDOWN = 3,  /* a reduced scalar became non-finite at iteration
                             info.breakdown_iter; histories are valid before it and hold
                             what IEEE arithmetic produced after it (as the reference) */
  CGX_ERR_UNSUPPORTED = 4
} cgx_status;

/* Variant ids.  Reference functions (numerical_experiments/cg_variants/):
 *   HS        hs_pcg        hs_cg.py:70-131        Hestenes-Stiefel
 *   CG        cg_pcg        cg_cg.py:77-146        Chronopoulos-Gear
 *   GV        gv_pcg        gv_cg.py:89-176        Ghysels-Vanroose (w_replace = never)
 *   PR        pr_pcg        pr_cg.py:93-171        predict-and-recompute
 *   M         m_pcg         pr_cg.py:93-164,172    Meurant predictor
 *   PIPE_PR   pipe_pr_pcg   pipe_pr_cg.py:109-205  pipelined predict-and-recompute
 *   PIPE_P    pipe_p_pcg    pipe_pr_cg.py:195-199  pipelined predict (no recompute of w)
 *   PIPE_PR_M pipe_pr_m_pcg pipe_pr_cg.py:213-217
 *   PIPE_P_M  pipe_p_m_pcg  pipe_pr_cg.py:207-211
 * The un-preconditioned twins (hs_cg, ...) are the same ids with no Jacobi vector set. */
typedef enum {
  CGX_HS = 0, CGX_CG = 1, CGX_GV = 2, CGX_PR = 3, CGX_M = 4,
  CGX_PIPE_PR = 5, CGX_PIPE_P = 6, CGX_PIPE_PR_M = 7, CGX_PIPE_P_M = 8,
  CGX_NUM_VARIANTS = 9
} cgx_variant;

/* History rows = the four standard callbacks (numerical_experiments/callbacks/):
 *   error_A_norm.py:29-48, residual_2_norm.py:29-41, error_2_norm.py:29-48,
 *   updated_residual_2_norm.py:29-40.  Row r of the history buffer is
 *   hist[r*max_iter + k], k = 0 .. max_iter-1 (k = 0 is the initial state). */
enum {
  CGX_HIST_ERROR_A_NORM = 1u,
  CGX_HIST_RESIDUAL_2_NORM = 2u,
  CGX_HIST_ERROR_2_NORM = 4u,
  CGX_HIST_UPDATED_RESIDUAL_2_NORM = 8u,
  CGX_HIST_ALL = 15u
};
#define CGX_HIST_ROWS 4

/* Execution path. AUTO picks PERSISTENT for latency-bound sizes. */
typedef enum {
  CGX_PATH_AUTO = 0,
  CGX_PATH_STREAM = 1,     /* 2-3 fused kernels per iteration, bandwidth-tuned */
  CGX_PATH_PERSISTENT = 2  /* one cooperative-grid launch runs every iteration */
} cgx_path;

typedef struct {
  double loop_ms;          /* device time of the iteration loop (CUDA events) */
  double setup_ms;         /* device time of the initialisation kernels */
  double h2d_bytes;        /* bytes copied host->device by the call */
  double d2h_bytes;        /* bytes copied device->host by the call */
  int64_t kernel_launches; /* kernels of this library launched by the call */
  int32_t iterations;      /* loop trips executed (max_iter - 1, or stop_iter after a tolerance stop) */
  int32_t breakdown_iter;  /* -1, or first k at which a reduced scalar was non-finite */
  int32_t path;            /* cgx_path actually used */
  int32_t stop_iter;       /* -1, or the iteration k at which the tolerance was met (cgx_set_tolerance) */
} cgx_info;

typedef struct cgx_ctx cgx_ctx;

int cgx_version(void);
const char* cgx_last_error(void);
/* number of CUDA devices visible, or 0 (never fails). */
int cgx_device_count(void);

int cgx_ctx_create(int device, cgx_ctx** out);
int cgx_ctx_destroy(cgx_ctx* ctx);

/* ---- operator A.  Replaces the scipy CSR operand of every `A @ v` in the solvers
 *      (e.g. hs_cg.py:123, pr_cg.py:152, pipe_pr_cg.py:179,181): canonical CSR, fp64
 *      values, int32 indices.  Row sums are accumulated in stored order with separately
 *      rounded multiply and add, as scipy's csr_matvec does. */
int cgx_set_csr_host(cgx_ctx* ctx, int64_t n, int64_t nnz, const int32_t* indptr_host,
                     const int32_t* indices_host, const double* data_host);
/* Matrix-free Dirichlet Poisson stencil in natural ordering i = x + nx*(y + ny*z):
 * dim = 2 (5-point, nz must be 1) or 3 (7-point); `diag` on the diagonal, `off` on the
 * 2*dim neighbours.  Equivalent to the CSR matrix kron(I,T)+kron(T,I)[+...] scaled
 * (SURVEY.md section 8d; matrices/poisson_ca.mtx is the 16x16 instance). */
int cgx_set_stencil(cgx_ctx* ctx, int dim, int64_t nx, int64_t ny, int64_t nz, double diag,
                    double off);
/* Matrix-free symmetric variable-coefficient stencil, same ordering and grid shapes as
 * cgx_set_stencil (dim 2: nz == 1 and cz == NULL; dim 3: cz required).  Host arrays of n
 * doubles: diag[i] = A[i,i], cx[i] = A[i,i+1], cy[i] = A[i,i+nx], cz[i] = A[i,i+nx*ny]; the
 * backward couplings follow by symmetry (A[i,i-1] = cx[i-1], ...).  A coupling that leaves the
 * grid (cx at x = nx-1, cy at y = ny-1, cz at z = nz-1) must be 0.  Row sums visit the full
 * 5/7-point pattern in canonical CSR order, zero couplings inside the grid included, so every
 * product equals scipy's on the CSR matrix that stores that pattern.
 * CGX_ERR_ARG: bad shape, NULL array, non-finite value or non-zero coupling off the grid.
 * CGX_ERR_UNSUPPORTED: the grid exceeds int32 indexing, or ctx is a rank of a partition.
 * Not accepted by cgx_batch_run (CGX_ERR_UNSUPPORTED); "tma" = 0 forces the generic kernel. */
int cgx_set_stencil_coef_host(cgx_ctx* ctx, int dim, int64_t nx, int64_t ny, int64_t nz,
                              const double* diag, const double* cx, const double* cy,
                              const double* cz);

/* ---- preconditioner.  Replaces the callable `preconditioner(v)` of the *_pcg solvers
 *      (figure_gen.py:40-44): dinv_host == NULL -> identity, else z = dinv * v
 *      elementwise (Jacobi: dinv = 1/A.diagonal(), computed by the caller). */
int cgx_set_jacobi_host(cgx_ctx* ctx, const double* dinv_host, int64_t n);

/* ---- problem vectors: b, x0 and (optional, may be NULL) x_true of
 *      `solver(A, b, x0, max_iter, ..., x_true=...)` (figure_gen.py:31-34,59). */
int cgx_load_problem_host(cgx_ctx* ctx, const double* b_host, const double* x0_host,
                          const double* x_true_host, int64_t n);
int cgx_load_problem_dev(cgx_ctx* ctx, const double* b_dev, const double* x0_dev,
                         const double* x_true_dev, int64_t n);

/* ---- run `max_iter - 1` iterations of `variant` on the loaded problem, recording the
 *      history rows selected by hist_mask on the device.  Replaces the body of
 *      hs_pcg / cg_pcg / gv_pcg / pr_master_pcg / pipe_pr_master_pcg.  Asynchronous work
 *      is complete when the call returns. */
int cgx_run(cgx_ctx* ctx, int variant, int max_iter, unsigned hist_mask, int path,
            cgx_info* info);

/* ---- the same solve, resumable: cgx_begin initialises (k = 0) and cgx_advance runs the
 *      next `niter` iterations (clamped to max_iter - 1).  cgx_run == begin + advance(all).
 *      This is what lets arbitrary Python callbacks (the reference's
 *      `callback(**locals())` protocol, e.g. hs_cg.py:128-129) observe x_k, r_k and the
 *      scalars between iterations without a CPU solve. */
int cgx_begin(cgx_ctx* ctx, int variant, int max_iter, unsigned hist_mask, int path);
int cgx_advance(cgx_ctx* ctx, int niter);
int cgx_get_info(cgx_ctx* ctx, cgx_info* info);
/* out9 = a_k, a_{k-1}, b_k, nu_k, nu_{k-1}, mu_k, eta_k, delta_k, gamma_k */
int cgx_get_scalars(cgx_ctx* ctx, double* out9);

/* ---- tuning/testing switches.  "tma" = 0 forces the generic (non-TMA) stencil kernel and
 *      "csr_stream" = 0 the thread-per-row CSR kernel, so that two SpMV implementations can
 *      be compared bit for bit; "csr_bulk" selects the warp-specialised CSR kernel: 1 (default)
 *      = matrix stream staged by cp.async.bulk for passes with one right-hand side, 2 = for the
 *      two-right-hand-side pass too, 0 = the register-staged csr_stream_kernel everywhere
 *      ("csr_bulk_ring" / "csr_bulk_sum" / "csr_bulk_ctas": slots per CTA, summing warps per CTA,
 *      resident CTAs per SM the ring is sized for); "persistent_threshold" = rows below which CGX_PATH_AUTO
 *      takes the persistent kernel ("pers_threads" / "pers_ctas" override its CTA shape);
 *      "csr_slab" = 0 keeps the persistent kernel's matrix in L2 instead of shared memory;
 *      "cg_elide" = 0 makes CG-CG / GV stream r~ / w~ on the TMA stencil path instead of
 *      forming them on the fly; "tma_min_planes" = planes per CTA the stencil grid aims for;
 *      "stub_allreduce" = 1 replaces the multi-GPU scalar
 *      exchange by a local stand-in (timing experiment: exposed allreduce time). */
int cgx_set_option(cgx_ctx* ctx, const char* name, int value);
/* ---- stop at a relative tolerance (one GPU: stream path, persistent path, cgx_batch_run; a partition:
 *      z-slabs or a CSR row partition, stream path, and the persistent path on slabs).
 *      rtol = 0 (the default) switches it off: every run then does max_iter - 1 iterations.
 *      Otherwise 0 < rtol < 1 (anything else, NaN included, is CGX_ERR_ARG), and a run stops at
 *      stop_iter = the first k >= 1 with nu_k <= rtol^2 * nu_0, where nu_k = r~_k . r_k is the
 *      recomputed inner product every variant already forms (the M^-1 norm of the updated residual;
 *      ||r_k||^2 without a preconditioner; never the predicted nu' of PR / M / pipe-*).  Iteration
 *      stop_iter is completed with all its stages, nothing after it runs.
 *      Contract: x, the state vectors, cgx_get_scalars and history entries 0 .. stop_iter are bitwise
 *      those of the same run without a tolerance and with max_iter = stop_iter + 1; later history
 *      entries are zero.  A run whose tolerance is never met is bitwise the run without one.
 *      info.stop_iter reports the stop (-1: none) and info.iterations the trips executed; cgx_advance
 *      (and cgx_advance_stages) after the stop do nothing and return CGX_OK.  A breakdown is reported
 *      as before; a NaN nu never meets the tolerance.
 *      Takes effect at the next cgx_begin / cgx_run / cgx_solve_host / cgx_batch_run (per context).
 *      Partitions: the call is collective -- every rank sets the same rtol.  nu_k is then the all-rank
 *      total, the same bits on every rank, so every rank stops at the same stop_iter; the contract above
 *      holds per rank against the same partition (same world, path and options) run without a
 *      tolerance and with max_iter = stop_iter + 1 (not against one GPU, which a partition matches only
 *      to rounding).  Refused with CGX_ERR_UNSUPPORTED before anything is enqueued: ranks of one
 *      cgx_group_begin whose tolerances differ; a scalar exchange other than peer to peer (NCCL, or the
 *      stub_allreduce stand-in, under which the ranks' nu differ); and cgx_begin / cgx_run /
 *      cgx_solve_host on a single rank whose peers are contexts of this process (cgx_dist_attach_ctx:
 *      drive those with cgx_group_*).  Ranks attached through CUDA IPC run with cgx_begin as usual. */
int cgx_set_tolerance(cgx_ctx* ctx, double rtol);
/* timing experiments: 16 %globaltimer stamps written by the last vector pass under
 * cgx_set_option("debug_skip", 2): [0] kernel start, [1] scalars folded, [2] CTA 0 done (ns). */
int cgx_debug_times(cgx_ctx* ctx, uint64_t* out16);

/* ---- optional per-kernel-class device timing of the iteration loop (CUDA event pair
 *      around every launch; used by bench.py for the roofline of the dominant kernel,
 *      never during a timed run).  Classes 0 .. cgx_profile_class_count()-1. */
int cgx_set_profile(cgx_ctx* ctx, int on);
int cgx_get_profile(cgx_ctx* ctx, int cls, double* ms, int64_t* launches);
const char* cgx_profile_class_name(int cls);
int cgx_profile_class_count(void);

/* ---- results: x_k of the last iteration and the history rows (CGX_HIST_ROWS*max_iter
 *      doubles, rows not selected are zero).  Either pointer may be NULL. */
int cgx_fetch_host(cgx_ctx* ctx, double* x_host, double* hist_host);
int cgx_fetch_dev(cgx_ctx* ctx, double* x_dev, double* hist_dev);
/* one named state vector ("x","r","rt","p","s","st","w","wt","u","ut","t") for tests */
int cgx_fetch_vector_host(cgx_ctx* ctx, const char* name, double* out_host);

/* ---- on-device support for the remaining reference callbacks and for GV residual replacement
 *      (single-GPU contexts, stream path).
 *   cgx_set_capture: what to record after every iteration k = 0 .. max_iter-1, in device memory
 *      (one device-to-host copy at the end instead of one per iteration):
 *        CGX_CAPTURE_X / _R   x_k / r_k   -> callbacks/save_x.py, save_r.py, and the inputs of
 *                                            lanczos_recurrence.py:43-61 (r_k, r_k1) and
 *                                            updated_error_A_norm.py:43-45 (r_k)
 *        CGX_CAPTURE_SCALARS  (a, b) as the recurrences hold them after iteration k
 *                                            -> a_k1, a_k2, b_k1 of lanczos_recurrence.py:51-53
 *      Takes effect at the next cgx_begin / cgx_run (mask 0 switches it off).
 *   cgx_fetch_capture_host: which = 0 x [max_iter][n], 1 r [max_iter][n], 2 scalars [2][max_iter].
 *   cgx_set_gv_replace: gv_cg.py:156-158 -- flags[k] != 0 makes iteration k of GV-CG replace
 *      w_k by A r_k after the vector updates (then wt, t, eta follow from the new w as in the
 *      reference); flags == NULL clears the schedule.
 *   cgx_advance_stages / cgx_gv_replace_now: for a host-evaluated `w_replace` predicate that
 *      looks at vectors: run `nstages` kernel stages of the current iteration (GV: stage 0 = the
 *      vector pass that forms x_k, r_k, w_k; stage 1 = t = A wt; then the instrumentation), and
 *      replace w between them. */
enum { CGX_CAPTURE_X = 1u, CGX_CAPTURE_R = 2u, CGX_CAPTURE_SCALARS = 4u };
int cgx_set_capture(cgx_ctx* ctx, unsigned mask);
int cgx_fetch_capture_host(cgx_ctx* ctx, int which, double* out_host);
int cgx_set_gv_replace(cgx_ctx* ctx, const uint8_t* flags, int n);
int cgx_advance_stages(cgx_ctx* ctx, int nstages);
int cgx_gv_replace_now(cgx_ctx* ctx);

/* ---- the whole reference call in one: load + run + fetch with HOST buffers
 *      (this is what `trial = method(A,b,x0,max_iter,callbacks=...,x_true=...,
 *      preconditioner=...)`, figure_gen.py:59, maps to once A and dinv are set). */
int cgx_solve_host(cgx_ctx* ctx, int variant, const double* b_host, const double* x0_host,
                   const double* x_true_host, int64_t n, int max_iter, unsigned hist_mask,
                   int path, double* x_host, double* hist_host, cgx_info* info);

/* ---- row-partitioned multi-GPU runs (one rank per GPU; SURVEY.md section 8e).  The
 *      reference's distributed solvers (scaling_experiments_mpi4py/cg_variants/*.py,
 *      `f(comm, A, b, max_iter)`) partition the unknowns over MPI ranks and Allreduce every
 *      iteration; here rank `rank` of `world` owns the z-slab of nz_local planes of the
 *      nx x ny x (sum of nz_local) Dirichlet 7-point grid (2-D grids: ny = 1, planes = grid
 *      rows), neighbours exchange one boundary plane per SpMV input by peer-to-peer stores
 *      over NVLink, and the <= 4 fused scalars per iteration are summed in rank order on
 *      every GPU (bit-identical everywhere).
 *      Set-up order on each rank: cgx_set_stencil_slab -> exchange the 64-byte window
 *      handles (cgx_dist_ipc_handle / cgx_dist_attach_ipc between processes, or
 *      cgx_dist_attach_ctx inside one process) -> cgx_dist_commit -> a barrier of the
 *      caller's -> cgx_set_jacobi_host / cgx_load_problem_* with the LOCAL slices ->
 *      cgx_run / cgx_begin / cgx_advance as on one GPU (collective: every rank calls them
 *      with the same arguments).  Histories are the global ones on every rank. */
int cgx_set_stencil_slab(cgx_ctx* ctx, int64_t nx, int64_t ny, int64_t nz_local, int world,
                         int rank, double diag, double off);
/* General CSR row partition (SURVEY.md section 8e "General CSR"; the layout of the reference's PETSc
 * driver, ex2b.c:71, and what its mpi4py column blocks transpose to for a symmetric matrix): rank
 * `rank` owns n_local consecutive rows.  indices are LOCAL: a column owned by this rank is its local
 * row number (0 .. n_local-1), a column owned by another rank is n_local + j with j the position of
 * that global column in this rank's sorted ghost list (n_ghost entries; the entries of one source
 * rank are contiguous).  The stored order inside a row is unchanged, so row sums keep scipy's
 * rounding.  recv_count[r] = ghost entries owned by rank r; send_count[r] / send_idx = the local rows
 * rank r needs (concatenated per destination, in the order of r's ghost list); send_off[r] = where
 * this rank's segment starts in r's ghost list; nghost_of[r] = n_ghost of rank r.
 * Then the same set-up as for slabs: window handles -> cgx_dist_commit -> local problem vectors. */
int cgx_set_csr_part_host(cgx_ctx* ctx, int64_t n_local, int64_t n_ghost, int64_t nnz, const int32_t* indptr_host,
                          const int32_t* indices_host, const double* data_host, int world, int rank,
                          const int32_t* recv_count, const int32_t* send_count, const int32_t* send_idx_host,
                          const int32_t* send_off, const int32_t* nghost_of);
int cgx_dist_ipc_handle(cgx_ctx* ctx, void* handle64);
int cgx_dist_attach_ipc(cgx_ctx* ctx, int peer_rank, const void* handle64);
int cgx_dist_attach_ctx(cgx_ctx* ctx, int peer_rank, cgx_ctx* peer);
/* scalar exchange mode: 1 = one-hop peer-to-peer flag exchange fused into the producing
 * kernel; 2 = ncclAllReduce (the comm.Allreduce of e.g. mpi4py pr_cg.py:61-69) on a side
 * stream, overlapped with the SpMV for the pipelined variants (pipeprcg.c:154-173).
 * Mode 2 needs the path of libnccl.so.2 and the 128-byte id from cgx_dist_nccl_unique_id
 * (made on rank 0, broadcast by the caller). */
int cgx_dist_nccl_unique_id(const char* nccl_libpath, void* id128);
int cgx_dist_commit(cgx_ctx* ctx, int mode, const char* nccl_libpath, const void* nccl_id128);
/* The same partition driven from ONE host thread: ctxs[r] is rank r (all on one GPU --
 * the ranks then share a stream and run interleaved, which is how the protocol is tested
 * on a single GPU -- or one context per GPU).  b/x0/x_true are the GLOBAL vectors. */
int cgx_group_load_problem_host(cgx_ctx** ctxs, int count, const double* b_host,
                                const double* x0_host, const double* x_true_host,
                                int64_t n_total);
int cgx_group_begin(cgx_ctx** ctxs, int count, int variant, int max_iter, unsigned hist_mask,
                    int path);
int cgx_group_advance(cgx_ctx** ctxs, int count, int niter);

/* ---- independent solves side by side on one GPU (e.g. the nine variants of one case,
 *      figure_gen.py:50-60, or one matrix with several right-hand sides).  Runs ctxs[i] as
 *      cgx_run(ctxs[i], variants[i], max_iters[i], hist_mask, CGX_PATH_PERSISTENT, &infos[i])
 *      would, except that all entries share one cooperative launch: entry i gets its own CTA
 *      range, sized by the persistent geometry for a 1/count share of the SMs (so its dot
 *      products are summed in the order of a solo run with that CTA shape -- its results are
 *      bitwise those of cgx_run with "pers_threads" / "pers_ctas" set to that shape, not
 *      necessarily those of a default cgx_run).  Entries never wait for each other; one with a
 *      smaller max_iter finishes first.  Each context keeps its own operator, preconditioner and
 *      problem (b, x0, optional x_true), loaded beforehand; results are fetched per context as
 *      after cgx_run.  The CTA width is common to the batch: the contexts' "pers_threads" when
 *      set (they must agree), else chosen so that every entry fits; "pers_ctas" and "csr_slab"
 *      act per entry as in cgx_run.  infos[i].loop_ms is the duration of the SHARED launch.
 *      Returns CGX_ERR_BREAKDOWN if any entry broke down (infos[i].breakdown_iter tells which).
 *      CGX_ERR_ARG: count < 1, a NULL pointer, a bad variant or max_iter, a context listed twice.
 *      CGX_ERR_UNSUPPORTED, before anything is launched: entries on different devices, a rank of
 *      a partition, a variable-coefficient stencil (cgx_set_stencil_coef_host), mixed operator
 *      kinds (CSR / stencil) or preconditioner modes (none / Jacobi
 *      vector / constant diagonal), a capture, a GV replacement schedule or "gv_manual" set, an
 *      entry that does not fit its share of the SMs, or a grid that is not co-resident.  After a
 *      refusal every context still runs normally with cgx_run. */
int cgx_batch_run(cgx_ctx** ctxs, int count, const int* variants, const int* max_iters,
                  unsigned hist_mask, cgx_info* infos);

/* ---- single primitives, exposed for the unit tests of SURVEY.md section 7:
 *      y = A v (scipy `A @ v`) and the deterministic fp64 dot (numpy `u @ v`). */
int cgx_spmv_host(cgx_ctx* ctx, const double* v_host, double* y_host, int64_t n);
int cgx_dot_host(cgx_ctx* ctx, const double* u_host, const double* v_host, int64_t n,
                 double* out);

#ifdef __cplusplus
}
#endif
#endif /* CGX_H_ */
