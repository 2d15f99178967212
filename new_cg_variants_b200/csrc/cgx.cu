// cgx.cu -- host side of libcgx_b200.so: context, device memory, the native iteration
// loop and the C ABI of include/cgx.h.  No torch, no cuBLAS/cuSPARSE, no CPU fallback.
#include <dlfcn.h>

#include "cgx_launch.cuh"

// cuTensorMapEncodeTiled is resolved through the runtime so the library has no link-time
// dependency on libcuda (it must load on the GPU-less build box for the ABI tests).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
static thread_local std::string g_err;


int cgx_fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

// ---------------------------------------------------------------------------------------
// NCCL (mode 2 of the scalar exchange) -- resolved with dlopen from the library the caller
// names (torch's bundled libnccl.so.2); the .so itself does not link NCCL.
// ---------------------------------------------------------------------------------------
NcclApi g_nccl;
static int nccl_load(const char* path) {
  if (g_nccl.h) return CGX_OK;
  void* h = dlopen(path && *path ? path : "libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail(CGX_ERR_UNSUPPORTED, "cannot load NCCL (%s): %s", path ? path : "libnccl.so.2", dlerror());
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(h, "ncclCommInitRank");
  g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(h, "ncclAllReduce");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(h, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy)
    return fail(CGX_ERR_UNSUPPORTED, "NCCL symbols missing in %s", path ? path : "libnccl.so.2");
  g_nccl.h = h;
  return CGX_OK;
}

const char* const kVecNames[V_COUNT] = {"x", "r", "rt", "p", "s", "st", "w", "wt", "u", "t"};

static void free_op(cgx_ctx* c) {
  cudaFree(c->d_ptr); cudaFree(c->d_idx); cudaFree(c->d_val); cudaFree(c->d_rowblk); cudaFree(c->d_send_idx); cudaFree(c->d_rowblk_e0);
  cudaFree(c->d_rowblk_b); cudaFree(c->d_rowblk_b_e0);
  c->d_ptr = c->d_idx = c->d_rowblk = c->d_send_idx = c->d_rowblk_e0 = c->d_rowblk_b = c->d_rowblk_b_e0 = nullptr; c->d_val = nullptr;
  c->n_rowblk_b = 0;
  c->n_rowblk = 0;
  c->h_ptr.clear();
  c->op_kind = 0;
}
static void free_problem(cgx_ctx* c) {
  if (c->own_problem) { cudaFree(c->d_b); cudaFree(c->d_x0); cudaFree(c->d_xtrue); }
  c->d_b = c->d_x0 = c->d_xtrue = nullptr;
  c->own_problem = false; c->problem_loaded = false; c->has_xtrue = false;
}
static void free_state(cgx_ctx* c) {
  for (int i = 0; i < V_COUNT; ++i) { cudaFree(c->vec[i]); c->vec[i] = nullptr; }
  for (auto& q : c->alt) { cudaFree(q); q = nullptr; }
  cudaFree(c->d_gscr); c->d_gscr = nullptr;
  for (int w = 0; w < 3; ++w) { cudaFree(c->d_cap[w]); c->d_cap[w] = nullptr; }
  for (auto& pp : c->d_exp) for (auto& q : pp) { cudaFree(q); q = nullptr; }
  cudaFree(c->d_hist); c->d_hist = nullptr; c->hist_len = 0;
  c->ran = false;
}
static void reset_size(cgx_ctx* c, i64 n) {
  if (c->n != n) {
    free_state(c); free_problem(c);
    cudaFree(c->d_dinv); c->d_dinv = nullptr; c->pm = 0; c->dinv_s = 1.0;
    c->n = n;
  }
}

extern "C" int cgx_version(void) { return CGX_VERSION; }
extern "C" const char* cgx_last_error(void) { return g_err.c_str(); }
extern "C" int cgx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" int cgx_ctx_create(int device, cgx_ctx** out) {
  if (!out) return fail(CGX_ERR_ARG, "cgx_ctx_create: out is NULL");
  *out = nullptr;
  int count = 0;
  CU(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count)
    return fail(CGX_ERR_CUDA, "cgx_ctx_create: device %d not available (%d CUDA devices); "
                "this library has no CPU fallback", device, count);
  CU(cudaSetDevice(device));
  cgx_ctx* c = new cgx_ctx();
  c->device = device;
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  c->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  c->stream = c->own_stream;
  for (auto& e : c->ev) CU(cudaEventCreate(&e));
  CU(cudaMalloc(&c->d_sc, 2 * sizeof(Scal)));
  CU(cudaMemset(c->d_sc, 0, 2 * sizeof(Scal)));
  CU(cudaMalloc(&c->d_partials, sizeof(double) * kMaxGrid * kNRed));
  CU(cudaMalloc(&c->d_ticket, sizeof(unsigned)));
  CU(cudaMemset(c->d_ticket, 0, sizeof(unsigned)));
  CU(cudaMalloc(&c->d_ppart, sizeof(double) * 2 * kPersMaxGrid * kPersRed));
  CU(cudaMalloc(&c->d_pbar, sizeof(u64) * 2));
  CU(cudaMemset(c->d_pbar, 0, sizeof(u64) * 2));
  CU(cudaMalloc(&c->d_tma_err, sizeof(int)));
  CU(cudaMemset(c->d_tma_err, 0, sizeof(int)));
  CU(cudaMalloc(&c->d_dbg_t, sizeof(u64) * 16));
  CU(cudaMemset(c->d_dbg_t, 0, sizeof(u64) * 16));
  CU(cudaMalloc(&c->d_pout, sizeof(PersOut)));
  CU(cudaMemset(c->d_pout, 0, sizeof(PersOut)));
  CU(cudaMalloc(&c->d_prank, std::max(sizeof(PersRank<CsrOp>), sizeof(PersRank<StencilOp>)) * kMaxWorld));
  c->dist.world = 1;
  *out = c;
  return CGX_OK;
}

static void dist_release(cgx_ctx* c) {
  if (c->nccl_comm && g_nccl.CommDestroy) { g_nccl.CommDestroy(c->nccl_comm); c->nccl_comm = nullptr; }
  for (int r = 0; r < kMaxWorld; ++r) {
    if (c->peer_ipc[r] && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
    c->peer_base[r] = nullptr; c->peer_ipc[r] = false;
  }
  cudaFree(c->d_win); c->d_win = nullptr; c->win_bytes = 0;
  cudaFree(c->d_nccl); c->d_nccl = nullptr;
  if (c->comm_stream) { cudaStreamDestroy(c->comm_stream); c->comm_stream = nullptr; }
  for (int s = 0; s < kSlots; ++s) {
    if (c->ev_prod[s]) { cudaEventDestroy(c->ev_prod[s]); c->ev_prod[s] = nullptr; }
    if (c->ev_red[s]) { cudaEventDestroy(c->ev_red[s]); c->ev_red[s] = nullptr; }
  }
  c->dist = Dist{}; c->dist.world = 1;
  c->dist_ready = false;
}

extern "C" int cgx_ctx_destroy(cgx_ctx* c) {
  if (!c) return CGX_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->own_stream);
  dist_release(c);
  free_state(c); free_problem(c); free_op(c);
  cudaFree(c->d_dinv); cudaFree(c->d_sc); cudaFree(c->d_partials); cudaFree(c->d_ticket);
  cudaFree(c->d_ppart); cudaFree(c->d_pbar); cudaFree(c->d_pout); cudaFree(c->d_prank); cudaFree(c->d_pbatch); cudaFree(c->d_dbg_t); cudaFree(c->d_tma_err);
  for (auto& e : c->ev) cudaEventDestroy(e);
  for (auto& e : c->prof_events) cudaEventDestroy(e);
  for (auto& e : c->ev_stop) if (e) cudaEventDestroy(e);
  cudaFreeHost(c->h_stop);
  cudaStreamDestroy(c->own_stream);
  delete c;
  return CGX_OK;
}

// ---------------------------------------------------------------------------------------
// operator / preconditioner / problem
// ---------------------------------------------------------------------------------------
// CSR-stream row blocks: consecutive rows, at most kCsrRows of them and kCsrCap non-zeros
// (a single longer row is a block of its own).
static void build_row_blocks(const int32_t* ptr, i64 n, std::vector<int>& blk, int max_rows = kCsrRows, int cap = kCsrCap) {
  blk.clear();
  blk.push_back(0);
  i64 r = 0;
  while (r < n) {
    i64 e = r + 1;
    while (e < n && e - r < max_rows && (i64)ptr[e + 1] - ptr[r] <= cap) ++e;
    blk.push_back((int)e);
    r = e;
  }
}

static int upload_csr(cgx_ctx* c, i64 n, i64 nnz, const int32_t* indptr, const int32_t* indices, const double* data) {
  CU(cudaSetDevice(c->device));
  free_op(c);
  reset_size(c, n);
  c->nnz = nnz;
  std::vector<int> blk;
  build_row_blocks(indptr, n, blk);
  // (kCbPadBytes of slack: the bulk copies of csr_bulk_kernel read whole 16-byte units)
  CU(cudaMalloc(&c->d_ptr, sizeof(int) * (n + 1) + kCbPadBytes));
  CU(cudaMalloc(&c->d_idx, sizeof(int) * std::max<i64>(nnz, 1) + kCbPadBytes));
  CU(cudaMalloc(&c->d_val, sizeof(double) * std::max<i64>(nnz, 1) + kCbPadBytes));
  CU(cudaMalloc(&c->d_rowblk, sizeof(int) * blk.size()));
  CU(cudaMalloc(&c->d_rowblk_e0, sizeof(int) * blk.size()));
  std::vector<int> blk_e0(blk.size());
  for (size_t q = 0; q < blk.size(); ++q) blk_e0[q] = indptr[blk[q]];
  CU(cudaMemcpyAsync(c->d_rowblk_e0, blk_e0.data(), sizeof(int) * blk.size(), cudaMemcpyHostToDevice, c->stream));
  std::vector<int> blkb, blkb_e0;
  build_row_blocks(indptr, n, blkb, kCbRows, kCbCap);
  blkb_e0.resize(blkb.size());
  for (size_t q = 0; q < blkb.size(); ++q) blkb_e0[q] = indptr[blkb[q]];
  CU(cudaMalloc(&c->d_rowblk_b, sizeof(int) * blkb.size()));
  CU(cudaMalloc(&c->d_rowblk_b_e0, sizeof(int) * blkb.size()));
  CU(cudaMemcpyAsync(c->d_rowblk_b, blkb.data(), sizeof(int) * blkb.size(), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_rowblk_b_e0, blkb_e0.data(), sizeof(int) * blkb.size(), cudaMemcpyHostToDevice, c->stream));
  c->n_rowblk_b = (int)blkb.size() - 1;
  CU(cudaMemcpyAsync(c->d_ptr, indptr, sizeof(int) * (n + 1), cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->d_rowblk, blk.data(), sizeof(int) * blk.size(), cudaMemcpyHostToDevice, c->stream));
  if (nnz) {
    CU(cudaMemcpyAsync(c->d_idx, indices, sizeof(int) * nnz, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->d_val, data, sizeof(double) * nnz, cudaMemcpyHostToDevice, c->stream));
  }
  CU(cudaStreamSynchronize(c->stream));
  c->n_rowblk = (int)blk.size() - 1;
  c->h_ptr.assign(indptr, indptr + n + 1);
  c->csr = CsrOp{c->d_ptr, c->d_idx, c->d_val, n};
  c->op_kind = 1;
  return CGX_OK;
}

extern "C" int cgx_set_csr_host(cgx_ctx* c, int64_t n, int64_t nnz, const int32_t* indptr,
                                const int32_t* indices, const double* data) {
  if (!c || n <= 0 || nnz < 0 || !indptr || (nnz > 0 && (!indices || !data)))
    return fail(CGX_ERR_ARG, "cgx_set_csr_host: bad arguments");
  if (n >= (1ll << 31) || nnz >= (1ll << 31))
    return fail(CGX_ERR_UNSUPPORTED, "cgx_set_csr_host: int32 index range exceeded");
  if (indptr[0] != 0 || indptr[n] != nnz)
    return fail(CGX_ERR_ARG, "cgx_set_csr_host: indptr[0] != 0 or indptr[n] != nnz");
  if (c->dist.world > 1)
    return fail(CGX_ERR_UNSUPPORTED, "cgx_set_csr_host: this context is a rank of a partitioned run; "
                "use cgx_set_csr_part_host (row block + ghost lists)");
  return upload_csr(c, n, nnz, indptr, indices, data);
}

static void dist_release(cgx_ctx* c);
extern "C" int cgx_set_csr_part_host(cgx_ctx* c, int64_t n, int64_t n_ghost, int64_t nnz, const int32_t* indptr,
                                     const int32_t* indices, const double* data, int world, int rank,
                                     const int32_t* recv_count, const int32_t* send_count, const int32_t* send_idx,
                                     const int32_t* send_off, const int32_t* nghost_of) {
  if (!c || n <= 0 || nnz < 0 || n_ghost < 0 || !indptr || (nnz > 0 && (!indices || !data)) || world < 1 || world > kMaxWorld ||
      rank < 0 || rank >= world || (world > 1 && (!recv_count || !send_count || !send_off || !nghost_of)))
    return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: bad arguments (world <= %d)", kMaxWorld);
  if (n + n_ghost >= (1ll << 31) || nnz >= (1ll << 31))
    return fail(CGX_ERR_UNSUPPORTED, "cgx_set_csr_part_host: int32 index range exceeded");
  if (indptr[0] != 0 || indptr[n] != nnz) return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: indptr[0] != 0 or indptr[n] != nnz");
  for (i64 e = 0; e < nnz; ++e)
    if (indices[e] < 0 || indices[e] >= n + n_ghost) return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: column index out of range");
  CU(cudaSetDevice(c->device));
  dist_release(c);
  int rc = upload_csr(c, n, nnz, indptr, indices, data);
  if (rc || world == 1) return rc;
  Dist& d = c->dist;
  d.world = world; d.rank = rank; d.mode = 1; d.saved_mode = 1; d.csr = 1;
  d.has_lo = d.has_hi = 0; d.plane = 0;
  d.nghost = (int)n_ghost;
  d.src_mask = 0;
  i64 total_send = 0, total_recv = 0;
  d.send_ptr[0] = 0;
  for (int r = 0; r < world; ++r) {
    if (recv_count[r] < 0 || send_count[r] < 0 || (r == rank && (recv_count[r] || send_count[r])))
      return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: bad send/receive counts");
    if (recv_count[r] > 0) d.src_mask |= 1u << r;
    total_recv += recv_count[r];
    total_send += send_count[r];
    d.send_ptr[r + 1] = (int)total_send;
    d.send_off[r] = send_off[r];
    d.nghost_of[r] = nghost_of[r];
  }
  if (total_recv != n_ghost || nghost_of[rank] != n_ghost) return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: receive counts do not add up to n_ghost");
  if (total_send > 0) {
    if (!send_idx) return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: send_idx is NULL");
    for (i64 e = 0; e < total_send; ++e)
      if (send_idx[e] < 0 || send_idx[e] >= n) return fail(CGX_ERR_ARG, "cgx_set_csr_part_host: send index out of range");
    CU(cudaMalloc(&c->d_send_idx, sizeof(int) * total_send));
    CU(cudaMemcpy(c->d_send_idx, send_idx, sizeof(int) * total_send, cudaMemcpyHostToDevice));
  }
  d.send_idx = c->d_send_idx;
  c->win_bytes = kWinHdrBytes + sizeof(double) * (size_t)kChan * 2 * (size_t)std::max<i64>(n_ghost, 1);
  CU(cudaMalloc(&c->d_win, c->win_bytes));
  CU(cudaMemset(c->d_win, 0, c->win_bytes));
  CU(cudaDeviceSynchronize());
  c->peer_base[rank] = c->d_win;
  c->epoch = 0; c->scpar = 0; c->pend.clear();
  for (auto& h : c->hepoch) h = 0;
  c->fepoch = 0;
  return CGX_OK;
}

static int set_stencil(cgx_ctx* c, int dim, i64 nx, i64 ny, i64 nz, double diag, double off, int has_lo,
                       int has_hi) {
  if (!c || (dim != 2 && dim != 3) || nx < 1 || ny < 1 || nz < 1 || (dim == 2 && nz != 1))
    return fail(CGX_ERR_ARG, "cgx_set_stencil: bad arguments");
  const i64 n = nx * ny * nz;
  if (n + 2 * nx * ny >= (1ll << 31))
    return fail(CGX_ERR_UNSUPPORTED, "cgx_set_stencil: grid too large for int32 indexing");
  CU(cudaSetDevice(c->device));
  free_op(c);
  reset_size(c, n);
  c->sten = StencilOp{(int)nx, (int)ny, (int)nz, diag, off, n, has_lo, has_hi};
  c->nnz = 0;
  c->op_kind = 2;
  return CGX_OK;
}

extern "C" int cgx_set_stencil(cgx_ctx* c, int dim, int64_t nx, int64_t ny, int64_t nz,
                               double diag, double off) {
  if (c && c->dist.world > 1)
    return fail(CGX_ERR_ARG, "cgx_set_stencil: this context is a rank of a partitioned run; use cgx_set_stencil_slab");
  return set_stencil(c, dim, nx, ny, nz, diag, off, 0, 0);
}

extern "C" int cgx_set_jacobi_host(cgx_ctx* c, const double* dinv, int64_t n) {
  if (!c) return fail(CGX_ERR_ARG, "cgx_set_jacobi_host: ctx is NULL");
  CU(cudaSetDevice(c->device));
  if (!dinv) { cudaFree(c->d_dinv); c->d_dinv = nullptr; c->pm = 0; c->dinv_s = 1.0; return CGX_OK; }
  if (c->op_kind == 0 || n != c->n)
    return fail(CGX_ERR_ARG, "cgx_set_jacobi_host: set the operator first; n must match (%lld vs %lld)",
                (long long)n, (long long)c->n);
  if (!c->d_dinv) CU(cudaMalloc(&c->d_dinv, sizeof(double) * n + kCbPadBytes));
  CU(cudaMemcpyAsync(c->d_dinv, dinv, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  // constant diagonal (every Poisson stencil): the same products with one HBM stream less
  bool constant = true;
  for (i64 i = 1; i < n && constant; ++i) constant = (memcmp(&dinv[i], &dinv[0], sizeof(double)) == 0);
  c->pm = constant ? 2 : 1;
  c->dinv_s = dinv[0];
  return CGX_OK;
}

static const char* kClassNames[PC_COUNT] = {
    "ew_hs1", "ew_hs2", "ew_cg", "ew_gv", "ew_pr", "ew_pipe_r", "ew_pipe_n",
    "sp_plain", "sp_hs", "sp_cg", "sp_gv", "sp_pr", "sp_pipe_r", "sp_pipe_n", "sp_resid",
    "instrument", "pr_fused"};
static void prof_resolve(cgx_ctx* c) {
  for (size_t i = 0; i < c->prof_cls.size(); ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->prof_events[2 * i], c->prof_events[2 * i + 1]) == cudaSuccess) {
      c->prof_ms[c->prof_cls[i]] += ms; c->prof_n[c->prof_cls[i]]++;
    }
  }
  c->prof_cls.clear(); c->prof_used = 0;
}

Args make_args(cgx_ctx* c) {
  Args g{};
  g.x = c->vec[V_X]; g.r = c->vec[V_R]; g.rt = c->vec[V_RT]; g.p = c->vec[V_P];
  g.s = c->vec[V_S]; g.st = c->vec[V_ST]; g.w = c->vec[V_W]; g.wt = c->vec[V_WT];
  g.u = c->vec[V_U]; g.t = c->vec[V_T];
  g.dinv = c->d_dinv; g.dinv_s = c->dinv_s; g.b = c->d_b; g.xtrue = c->d_xtrue;
  g.sc = c->d_sc; g.partials = c->d_partials; g.ticket = c->d_ticket;
  g.hist = c->d_hist; g.hist_len = c->hist_len; g.hist_mask = c->hist_mask;
  g.n = c->n; g.k = c->cur_k;
  g.d = c->dist;
  g.halo_ll = c->halo_ll ? 1 : 0;
  g.errflag = c->d_tma_err;
  // L2 residency hint: measured at 2.1 M rows (one slab of 256^3 / 8) 2-6 % per iteration; auto = on when this
  // GPU's state vectors (<= 10 x n) fit well inside the 126 MB L2
  g.l2pol = (c->l2_keep == 1 || (c->l2_keep < 0 && c->n > 0 && (size_t)c->n * 8 * 6 < ((size_t)96 << 20))) ? kL2EvictLast : 0;
  g.dbg = c->dbg;
  g.dbg_t = c->d_dbg_t;
  g.tol_on = c->run_tol > 0.0 ? 1 : 0;
  return g;
}


// before the launch: fill the per-launch fields of g; mode 2: make the stream wait for the
// NCCL reductions this kernel folds
void plan_apply(cgx_ctx* c, Args& g, const Plan& p) {
  if (c->dist.world <= 1) return;
  g.d = c->dist;
  g.scpar = c->scpar;
  g.npend = 0;
  if (p.consume) {
    g.npend = (int)c->pend.size();
    for (int q = 0; q < g.npend; ++q) {
      g.pend_kind[q] = c->pend[q].kind; g.pend_k[q] = c->pend[q].k; g.pend_e[q] = c->pend[q].e;
      if (c->dist.mode == 2) cudaStreamWaitEvent(c->stream, c->ev_red[c->pend[q].e % kSlots], 0);
    }
  }
  if (p.produce != FK_NONE) g.sepoch = c->epoch + 1;
  g.hout_n = p.hout_n; g.hout_ch = p.hout_ch;
  if (p.hout_n) {
    g.hout_epoch = c->hepoch[p.hout_ch] + 1;
    g.hout_par = (int)(g.hout_epoch & 1);
  }
  g.hin_ch = p.hin_ch;
  if (p.hin_n) {
    g.hin_epoch = c->hepoch[p.hin_ch];
    g.hin_par = (int)(g.hin_epoch & 1);
  }
  g.xt_epoch = c->hepoch[3];
  g.xt_par = (int)(g.xt_epoch & 1);
}
// after the launch: advance the epochs; mode 2: enqueue the allreduce of the new record
void plan_commit(cgx_ctx* c, const Args& g, const Plan& p) {
  if (c->dist.world <= 1) return;
  if (p.consume && !c->pend.empty()) { c->scpar ^= 1; c->pend.clear(); }
  if (p.produce != FK_NONE) {
    c->epoch++;
    if (p.produce != FK_INSTR) c->pend.push_back({c->epoch, p.produce, g.k});
    if (c->dist.mode == 2) {
      const int slot = (int)(c->epoch % kSlots);
      cudaEventRecord(c->ev_prod[slot], c->stream);
      cudaStreamWaitEvent(c->comm_stream, c->ev_prod[slot], 0);
      g_nccl.AllReduce(c->dist.nccl_in + (size_t)slot * kSumW, c->dist.nccl_out + (size_t)slot * kSumW, kSumW,
                       /*ncclFloat64*/ 8, /*ncclSum*/ 0, c->nccl_comm, c->comm_stream);
      cudaEventRecord(c->ev_red[slot], c->comm_stream);
    }
  }
  for (int i = 0; i < p.hout_n; ++i) c->hepoch[p.hout_ch + i]++;
}

VecIn vec_in(cgx_ctx* c, const double* v, int ch, const Args& g) {
  VecIn a{v, nullptr, nullptr};
  if (c->dist.world > 1 && c->dist.csr) {
    if (c->dist.ghost) a.lo = c->dist.ghost + (size_t)(ch * 2 + g.hin_par) * (size_t)c->dist.nghost;
    return a;
  }
  if (c->dist.world > 1 && c->dist.ghost) {
    a.lo = c->dist.ghost + ghost_off(c->dist, ch, g.hin_par, 0);
    a.hi = c->dist.ghost + ghost_off(c->dist, ch, g.hin_par, 1);
  }
  return a;
}


int ctx_occupancy(cgx_ctx* c, const void* fn, int threads, size_t smem) {
  const size_t key = smem | ((size_t)threads << 40);          // (kernels launched with more than one CTA width)
  auto it = c->occ.find({fn, key});
  if (it != c->occ.end()) return it->second;
  int per_sm = 0;
  if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem) != cudaSuccess) { cudaGetLastError(); per_sm = 0; }
  if (per_sm < 1) per_sm = 1;
  c->occ[{fn, key}] = per_sm;
  return per_sm;
}


// multi-GPU: push the boundary planes of v into the neighbours' ghost planes of channel ch
void launch_halo_push(cgx_ctx* c, Args g, const double* v, int ch) { launch_halo_push2(c, g, v, nullptr, ch); }
// one or two vectors (channels ch, ch + 1) under ONE halo epoch -- the consumer of a 2-RHS pass waits for
// a single epoch (that of channel ch) on both channels
void launch_halo_push2(cgx_ctx* c, Args g, const double* v0, const double* v1, int ch) {
  if (c->dist.world <= 1) return;
  Plan p;
  p.hout_n = v1 ? 2 : 1; p.hout_ch = ch;
  plan_apply(c, g, p);
  g.halo_ll = 0;                      // plain ghost planes + halo epoch flags (generic consumers)
  const double* vs[2] = {v0, v1};
  for (int i = 0; i < p.hout_n; ++i) {
    g.hout_ch = ch + i;
    g.hout_n = 1;
    if (c->dist.csr) {
      const int total = c->dist.send_ptr[c->dist.world];
      if (total > 0) { csr_halo_push_kernel<<<grid_for(c, total), kBlock, 0, c->stream>>>(g, vs[i]); c->launches++; }
    } else {
      halo_push_kernel<<<grid_for(c, c->dist.plane), kBlock, 0, c->stream>>>(g, vs[i]);
      c->launches++;
    }
  }
  plan_commit(c, g, p);
}

// ---- TMA stencil path: descriptors and work decomposition -------------------------------
bool tma_encode_dims(double* ptr, i64 nx, i64 ny, i64 nz, CUtensorMap* out) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc || !ptr) return false;
  cuuint64_t gdim[3] = {(cuuint64_t)nx, (cuuint64_t)ny, (cuuint64_t)nz};
  cuuint64_t gstr[2] = {(cuuint64_t)nx * 8, (cuuint64_t)nx * ny * 8};
  cuuint32_t box[3] = {(cuuint32_t)kPX, (cuuint32_t)kPY, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, ptr, gdim, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static bool tma_prepare_geom(cgx_ctx* c) {
  if (c->op_kind != 2 || c->no_tma) return false;
  const StencilOp& S = c->sten;
  if (S.nx % 2 != 0 || S.nx < 2) return false;         // TMA needs 16-byte global strides
  if (S.ny < 4 && S.nz > 1) return false;              // 2-D grid viewed as nx x 1 x ny slabs: tiles would idle
  if (!get_encode_tiled()) return false;
  TmaGeom& G = c->geom;
  G.nx = S.nx; G.ny = S.ny; G.nz = S.nz;
  G.ntx = (S.nx + kTX - 1) / kTX; G.nty = (S.ny + kTY - 1) / kTY;
  G.has_zlo = S.has_zlo; G.has_zhi = S.has_zhi;
  G.diag = S.diag; G.off = S.off;
  G.err = c->d_tma_err;
  G.nchunk = 1;
  G.march_y = 0;
  if (S.nz == 1 && !S.has_zlo && !S.has_zhi && G.nty > 1) {   // 2-D: march down the y-tiles of a column
    G.march_y = 1;
    G.nz = G.nty;
    G.nty = 1;
  }
  // resident CTAs: shared memory bound (227 KB/SM), 8 x 256 threads at most
  int per_sm1 = std::min(8, (int)(227 * 1024 / (tma_smem_bytes(1) + 1024)));
  int per_sm2 = std::min(8, (int)(227 * 1024 / (tma_smem_bytes(2) + 1024)));
  const int cap1 = c->sm_count * per_sm1, cap2 = c->sm_count * per_sm2;
  // one CTA per resident slot; the kernel cuts the (column, plane) sequence evenly between
  // them (>= 4 planes per CTA when the problem is large enough to keep the z-halo small)
  const i64 total = (i64)(G.ntx * G.nty) * G.nz;
  const i64 mp = std::max(1, c->tma_min_planes);
  const i64 want = std::max<i64>(1, (total + mp - 1) / mp);
  c->tma_grid[0] = (int)std::min<i64>(want, cap1);
  c->tma_grid[1] = (int)std::min<i64>(want, cap2);
  return true;
}

static int setup_tma(cgx_ctx* c, unsigned need) {
  c->use_tma = false;
  c->halo_ll = false;
  for (auto& ok : c->tmap_ok) ok = false;
  if (!tma_prepare_geom(c)) return CGX_OK;
  const StencilOp& S = c->sten;
  for (int i = 0; i < V_COUNT; ++i)
    if ((need & (1u << i)) && c->vec[i]) c->tmap_ok[i] = tma_encode_dims(c->vec[i], S.nx, S.ny, S.nz, &c->tmap[i]);
  // every fused SpMV pass of the variant must take the TMA kernel for the LL ghost planes
  bool all_ok = true;
  for (int i = 0; i < V_COUNT; ++i)
    if ((need & (1u << i)) && c->vec[i] && !c->tmap_ok[i]) all_ok = false;
  c->halo_ll = c->dist.world > 1 && all_ok;
  if (c->halo_ll && !c->d_gscr) CU(cudaMalloc(&c->d_gscr, sizeof(double) * 4 * (size_t)c->dist.plane));   // [2 sides][2 rhs][plane]
  if (c->dist.world > 1 && !all_ok) {                 // mixed would mix the two ghost formats: all generic
    for (auto& ok : c->tmap_ok) ok = false;
    return CGX_OK;
  }
  c->use_tma = true;
  return CGX_OK;
}

void launch_instrument(cgx_ctx* c, Args g) {
  const int grid = grid_for(c, c->n);
  Plan p;
  p.produce = FK_INSTR;
  p.hin_n = 1; p.hin_ch = 2;
  plan_apply(c, g, p);
  {
    ProfScope ps(c, PC_INSTR);
    const VecIn xin = vec_in(c, c->vec[V_X], 2, g);
    VecIn xtin{c->d_xtrue, nullptr, nullptr};
    if (c->dist.world > 1 && c->dist.csr) {
      if (c->dist.ghost) xtin.lo = c->dist.ghost + (size_t)(3 * 2 + g.xt_par) * (size_t)c->dist.nghost;
    } else if (c->dist.world > 1 && c->dist.ghost) {
      xtin.lo = c->dist.ghost + ghost_off(c->dist, 3, g.xt_par, 0);
      xtin.hi = c->dist.ghost + ghost_off(c->dist, 3, g.xt_par, 1);
    }
    if (c->op_kind == 1) {
      if (c->has_xtrue) instrument_kernel<CsrOp, true><<<grid, kBlock, 0, c->stream>>>(c->csr, g, xin, xtin);
      else instrument_kernel<CsrOp, false><<<grid, kBlock, 0, c->stream>>>(c->csr, g, xin, xtin);
    } else {
      if (c->has_xtrue) instrument_kernel<StencilOp, true><<<grid, kBlock, 0, c->stream>>>(c->sten, g, xin, xtin);
      else instrument_kernel<StencilOp, false><<<grid, kBlock, 0, c->stream>>>(c->sten, g, xin, xtin);
    }
    c->launches++;
  }
  plan_commit(c, g, p);
}
// multi-GPU: the history entry of the instrumentation record just produced
void launch_hist_consume(cgx_ctx* c, Args g) {
  if (c->dist.world <= 1) return;
  g.d = c->dist;
  g.pend_e[0] = c->epoch;
  if (c->dist.mode == 2) cudaStreamWaitEvent(c->stream, c->ev_red[c->epoch % kSlots], 0);
  hist_consume_kernel<<<1, 32, 0, c->stream>>>(g);
  c->launches++;
}
// stop != nullptr: a step of iteration k, skipped on the device after a tolerance stop
static void launch_dot(cgx_ctx* c, const double* u, const double* v, const double* dinv, int slot,
                       const Scal* stop = nullptr, int k = 0) {
  dot_kernel<<<grid_for(c, c->n), kBlock, 0, c->stream>>>(u, v, dinv, c->n, c->d_sc + c->scpar, slot,
                                                          c->d_partials, c->d_ticket, stop, k);
  c->launches++;
}
static void launch_scale(cgx_ctx* c, const double* dinv, const double* v, double* out,
                         const Scal* stop = nullptr, int k = 0) {
  scale_kernel<<<grid_for(c, c->n), kBlock, 0, c->stream>>>(dinv, v, out, c->n, stop, k);
  c->launches++;
}

VariantInfo variant_info(int v, bool prec) {
  auto bit = [](int i) { return 1u << i; };
  const unsigned base = bit(V_X) | bit(V_R) | bit(V_RT) | bit(V_P) | bit(V_S);
  switch (v) {
    case CGX_HS: return {false, false, false, 0, base};
    case CGX_CG: return {false, false, false, 1, base | bit(V_W)};
    case CGX_GV: return {false, false, false, 1, base | bit(V_W) | bit(V_WT) | bit(V_ST) | bit(V_U) | bit(V_T)};
    case CGX_PR: return {false, false, false, 2, base};
    case CGX_M: return {true, false, false, 2, base};
    case CGX_PIPE_PR: return {false, true, true, 2, base | bit(V_ST) | bit(V_W) | bit(V_U)};
    case CGX_PIPE_PR_M: return {true, true, true, 2, base | bit(V_ST) | bit(V_W) | bit(V_U)};
    case CGX_PIPE_P: return {false, true, false, 2, base | bit(V_ST) | bit(V_W) | bit(V_U) | (prec ? bit(V_WT) : 0u)};
    case CGX_PIPE_P_M: return {true, true, false, 2, base | bit(V_ST) | bit(V_W) | bit(V_U) | (prec ? bit(V_WT) : 0u)};
  }
  return {false, false, false, -1, 0};
}

// ---------------------------------------------------------------------------------------
// The iteration as a list of stages.  A stage is one kernel launch; stage s of rank A only
// ever waits for stages < s of other ranks, so a group of ranks may be driven in lockstep
// from one host thread (cgx_group_*), or every rank from its own process.
// ---------------------------------------------------------------------------------------
static int iter_stage_count(const cgx_ctx* c) {
  int ns = core_stages(c);
  if (c->hist_mask || c->capture) ns += (c->dist.world > 1) ? 3 : 1;
  return ns;
}

void launch_capture(cgx_ctx* c, const Args& g) {
  const size_t bytes = sizeof(double) * c->n;
  if (c->capture & CGX_CAPTURE_X) cudaMemcpyAsync(c->d_cap[0] + (size_t)g.k * c->n, c->vec[V_X], bytes, cudaMemcpyDeviceToDevice, c->stream);
  if (c->capture & CGX_CAPTURE_R) cudaMemcpyAsync(c->d_cap[1] + (size_t)g.k * c->n, c->vec[V_R], bytes, cudaMemcpyDeviceToDevice, c->stream);
  if (c->capture & CGX_CAPTURE_SCALARS) {
    capture_scalars_kernel<<<1, 32, 0, c->stream>>>(c->d_sc, c->d_cap[2], g.k, c->hist_len, g.tol_on);
    c->launches++;
  }
}

// GV residual replacement at iteration g.k, between the vector pass and t = A wt
static void launch_gv_replace(cgx_ctx* c, Args g) {
  const Scal* stop = g.tol_on ? c->d_sc : nullptr;
  launch_spmv<SP_PLAIN, 0, false>(c, g, c->vec[V_R], c->vec[V_W]);          // w = A r        gv_cg.py:158
  launch_scale(c, c->d_dinv, c->vec[V_W], c->vec[V_WT], stop, g.k);         // wt = M w       :160
  launch_dot(c, c->vec[V_W], c->vec[V_RT], nullptr, 5, stop, g.k);          // eta = w . rt   :163
  gv_refinalize_kernel<<<1, 32, 0, c->stream>>>(c->d_sc, g.k, g.tol_on);    // mu, a          :169-170
  c->launches++;
}

static void iter_stage(cgx_ctx* c, int s, const Args& g) {
  if (c->pr_fused && s == 0) { cgx_launch_pr_fused(c, g); return; }
  if (c->pm == 2) cgx_iter_stage_pm2(c, s, g);
  else if (c->pm == 1) cgx_iter_stage_pm1(c, s, g);
  else cgx_iter_stage_pm0(c, s, g);
}

// multi-GPU: fold what is still pending into the persisted scalars (end of an advance)
static void launch_flush(cgx_ctx* c, Args g, bool meurant) {
  if (c->dist.world <= 1 || c->pend.empty()) return;
  Plan p; p.consume = true;
  plan_apply(c, g, p);
  g.meur = meurant ? 1 : 0;
  flush_scalars_kernel<<<1, 32, 0, c->stream>>>(g);
  c->launches++;
  plan_commit(c, g, p);
}

// Initial state: hs_cg.py:83-94, cg_cg.py:90-104, gv_cg.py:105-121, pr_cg.py:106-120,
// pipe_pr_cg.py:122-140.  Built from plain kernels; not part of the timed loop.  Returned
// as a list of steps (one launch or copy each) with the same length on every rank.
typedef std::vector<std::function<void()>> Steps;

static void build_init_steps(cgx_ctx* c, int variant, const VariantInfo& vi, Steps& st) {
  const size_t bytes = sizeof(double) * c->n;
  const double* dinv = c->d_dinv;
  double** v = c->vec;
  const bool dist = c->dist.world > 1;
  auto copy = [=](double* dst, const double* src) {
    return [=]() { cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream); };
  };
  auto spmv = [=, &st](int mode, const double* in, double* out) {     // y = A in  /  r = b - A in
    if (dist) st.push_back([=]() { launch_halo_push(c, make_args(c), in, 0); });
    st.push_back([=]() {
      Args g = make_args(c);
      if (mode == SP_RESID) launch_spmv<SP_RESID, 0, false>(c, g, in, out);
      else launch_spmv<SP_PLAIN, 0, false>(c, g, in, out);
    });
  };
  auto dot = [=, &st](const double* a, const double* b, const double* dv, int slot) {
    st.push_back([=]() { launch_dot(c, a, b, dv, slot); });
  };
  auto scale = [=, &st](const double* in, double* out) { st.push_back([=]() { launch_scale(c, dinv, in, out); }); };

  st.push_back(copy(v[V_X], c->d_x0));
  spmv(SP_RESID, v[V_X], v[V_R]);                                       // r = b - A x0
  scale(v[V_R], v[V_RT]);                                               // rt = M r
  st.push_back(copy(v[V_P], v[V_RT]));                                  // p = rt
  dot(v[V_R], v[V_RT], nullptr, 0);                                     // nu = r.rt
  if (variant == CGX_HS || variant == CGX_PR || variant == CGX_M || vi.pipe) {
    spmv(SP_PLAIN, v[V_P], v[V_S]);                                     // s = A p
    dot(v[V_P], v[V_S], nullptr, 1);                                    // mu = p.s
  }
  if (variant == CGX_CG || variant == CGX_GV) {
    spmv(SP_PLAIN, v[V_RT], v[V_W]);                                    // w = A rt
    st.push_back(copy(v[V_S], v[V_W]));                                 // s = A p = w
    dot(v[V_P], v[V_S], nullptr, 1);                                    // mu = p.s
    dot(v[V_W], v[V_RT], nullptr, 2);                                   // eta = w.rt
  }
  if (variant == CGX_GV) {
    scale(v[V_W], v[V_WT]);                                             // wt = M w
    st.push_back(copy(v[V_ST], v[V_WT]));
    spmv(SP_PLAIN, v[V_WT], v[V_T]);                                    // t = A wt
    st.push_back(copy(v[V_U], v[V_T]));                                 // u = A wt
  }
  if (vi.cls == 2) {
    dot(v[V_R], v[V_S], dinv, 3);                                       // delta = r.(M s)
    dot(v[V_S], v[V_S], dinv, 4);                                       // gamma = (M s).s
  }
  if (vi.pipe) {
    scale(v[V_S], v[V_ST]);                                             // st = M s
    st.push_back(copy(v[V_W], v[V_S]));                                 // w = s
    if (v[V_WT]) st.push_back(copy(v[V_WT], v[V_ST]));
    spmv(SP_PLAIN, v[V_ST], v[V_U]);                                    // u = A st
  }
  if (dist) {
    st.push_back([=]() {                                                // publish the rank's partial dots
      Args g = make_args(c);
      Plan p; p.produce = FK_INIT;
      plan_apply(c, g, p);
      push_tmp_kernel<<<1, 32, 0, c->stream>>>(g);
      c->launches++;
      // not a pending recurrence: init_scalars consumes it directly
      c->epoch++;
      if (c->dist.mode == 2) {
        const int slot = (int)(c->epoch % kSlots);
        cudaEventRecord(c->ev_prod[slot], c->stream);
        cudaStreamWaitEvent(c->comm_stream, c->ev_prod[slot], 0);
        g_nccl.AllReduce(c->dist.nccl_in + (size_t)slot * kSumW, c->dist.nccl_out + (size_t)slot * kSumW, kSumW, 8, 0,
                         c->nccl_comm, c->comm_stream);
        cudaEventRecord(c->ev_red[slot], c->comm_stream);
      }
    });
  }
  const int cls = vi.cls, meur = vi.meurant ? 1 : 0;
  const double tol = c->run_tol;
  st.push_back([=]() {
    Args g = make_args(c);
    g.scpar = c->scpar;
    if (dist) {
      g.pend_e[0] = c->epoch;
      if (c->dist.mode == 2) cudaStreamWaitEvent(c->stream, c->ev_red[c->epoch % kSlots], 0);
    }
    init_scalars_kernel<<<1, 32, 0, c->stream>>>(g, cls, meur, tol);
    c->launches++;
  });
}

// ---------------------------------------------------------------------------------------
// problem vectors
// ---------------------------------------------------------------------------------------
static int load_problem(cgx_ctx* c, const double* b, const double* x0, const double* xt, i64 n,
                        cudaMemcpyKind kind) {
  if (!c || !b || !x0) return fail(CGX_ERR_ARG, "cgx_load_problem: b and x0 are required");
  if (c->op_kind == 0 || n != c->n)
    return fail(CGX_ERR_ARG, "cgx_load_problem: set the operator first; n must match (%lld vs %lld)",
                (long long)n, (long long)c->n);
  CU(cudaSetDevice(c->device));
  if (!c->own_problem) {
    c->d_b = c->d_x0 = c->d_xtrue = nullptr;
    CU(cudaMalloc(&c->d_b, sizeof(double) * n + kCbPadBytes));
    CU(cudaMalloc(&c->d_x0, sizeof(double) * n));
    CU(cudaMalloc(&c->d_xtrue, sizeof(double) * n));
    c->own_problem = true;
  }
  CU(cudaMemcpyAsync(c->d_b, b, sizeof(double) * n, kind, c->stream));
  CU(cudaMemcpyAsync(c->d_x0, x0, sizeof(double) * n, kind, c->stream));
  if (xt) CU(cudaMemcpyAsync(c->d_xtrue, xt, sizeof(double) * n, kind, c->stream));
  c->has_xtrue = xt != nullptr;
  c->problem_loaded = true;
  // multi-GPU: the neighbours need the boundary planes of x_true for e = x - x_true
  if (c->dist.world > 1 && c->dist_ready) {
    if (xt) launch_halo_push(c, make_args(c), c->d_xtrue, 3);
    else c->hepoch[3]++;      // keep the epoch counters of all ranks in step
  }
  return CGX_OK;
}

extern "C" int cgx_load_problem_host(cgx_ctx* c, const double* b, const double* x0,
                                     const double* xt, int64_t n) {
  int rc = load_problem(c, b, x0, xt, n, cudaMemcpyHostToDevice);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream));   // pageable host buffers may be reused by the caller
  return CGX_OK;
}
extern "C" int cgx_load_problem_dev(cgx_ctx* c, const double* b, const double* x0,
                                    const double* xt, int64_t n) {
  return load_problem(c, b, x0, xt, n, cudaMemcpyDeviceToDevice);
}

// ---------------------------------------------------------------------------------------
// persistent path (cgx_persistent.cuh): one cooperative launch runs every iteration
// ---------------------------------------------------------------------------------------

// CTA shape for n rows per rank with `ranks_in_launch` ranks sharing one GPU's SMs
static PersGeom pers_geometry_T(const cgx_ctx* c, int variant, int ranks_in_launch, int T) {
  PersGeom G{};
  const VariantInfo vi = variant_info(variant, c->d_dinv != nullptr);
  G.vmask = vi.need;
  G.nslot = __builtin_popcount(vi.need) + (c->pm == 1 ? 1 : 0);
  const int sm_cap = std::max(1, c->sm_count / std::max(1, ranks_in_launch));
  T = std::min(512, std::max(32, (T + 31) / 32 * 32));
  const i64 chunks = (c->n + T - 1) / T;
  int cap = c->pers_ctas ? std::min(c->pers_ctas, 4 * sm_cap) : sm_cap;     // co-residency is checked at launch
  cap = std::max(1, std::min(cap, kPersMaxGrid / std::max(1, ranks_in_launch)));
  const i64 R = (chunks + cap - 1) / cap;
  G.T = T; G.R = (int)R; G.nb = (int)((chunks + R - 1) / R);
  G.smem = (size_t)G.nslot * R * T * sizeof(double) + (((size_t)R * T + 15) / 16) * 16;   // + row masks
  G.ok = G.smem <= 216 * 1024;
  // CSR: keep each CTA's rows of the matrix in shared memory when they fit (one chunk per CTA)
  G.slab_cap = 0;
  if (c->op_kind == 1 && R == 1 && !c->h_ptr.empty() && !c->no_slab) {
    i64 mx = 0;
    for (i64 r0 = 0; r0 < c->n; r0 += T) mx = std::max<i64>(mx, c->h_ptr[std::min<i64>(c->n, r0 + T)] - c->h_ptr[r0]);
    mx = (mx + 3) / 4 * 4;
    const size_t slab = (size_t)mx * 12 + ((size_t)(T + 1) * 4 + 15) / 16 * 16;
    if (mx > 0 && G.smem + slab <= 216 * 1024) { G.slab_cap = (int)mx; G.smem += slab; }
  }
  return G;
}
// CTA shape for n rows per rank with `ranks_in_launch` ranks sharing one GPU's SMs
static PersGeom pers_geometry(const cgx_ctx* c, int variant, int ranks_in_launch) {
  const int sm_cap = std::max(1, c->sm_count / std::max(1, ranks_in_launch));
  if (c->pers_threads) return pers_geometry_T(c, variant, ranks_in_launch, c->pers_threads);
  PersGeom G = pers_geometry_T(c, variant, ranks_in_launch, c->n <= (i64)sm_cap * 256 ? 256 : 512);
  if (c->op_kind == 1 && G.slab_cap == 0) {            // narrower CTAs so that the matrix slabs fit
    for (int T : {128, 64}) {
      PersGeom H = pers_geometry_T(c, variant, ranks_in_launch, T);
      if (H.ok && H.slab_cap > 0) return H;
    }
  }
  return G;
}

static int pers_launch(cgx_ctx** cs, int count, const PersGeom& G, int k0, int k1) {
  const cgx_ctx* c = cs[0];
  if (c->op_kind == 1) {
    if (c->pm == 2) return cgx_pers_launch_csr_pm2(cs, count, G, k0, k1);
    if (c->pm == 1) return cgx_pers_launch_csr_pm1(cs, count, G, k0, k1);
    return cgx_pers_launch_csr_pm0(cs, count, G, k0, k1);
  }
  if (c->pm == 2) return cgx_pers_launch_sten_pm2(cs, count, G, k0, k1);
  if (c->pm == 1) return cgx_pers_launch_sten_pm1(cs, count, G, k0, k1);
  return cgx_pers_launch_sten_pm0(cs, count, G, k0, k1);
}
// after the launch has drained: adopt the epoch counters the kernel advanced
static int pers_collect(cgx_ctx* c) {
  PersOut o;
  CU(cudaMemcpy(&o, c->d_pout, sizeof o, cudaMemcpyDeviceToHost));
  if (o.err) return fail(CGX_ERR_CUDA, "persistent kernel: a sync point or a peer wait timed out (rank %d)", c->dist.rank);
  c->epoch = o.epoch;
  for (int ch = 0; ch < kChan; ++ch) c->hepoch[ch] = o.hepoch[ch];
  return CGX_OK;
}

// ---------------------------------------------------------------------------------------
// begin / advance, for one context or a lockstep group of ranks
// ---------------------------------------------------------------------------------------
static int begin_prepare(cgx_ctx* c, int variant, int max_iter, unsigned hist_mask, int path, int ranks_in_launch) {
  if (!c) return fail(CGX_ERR_ARG, "cgx_begin: ctx is NULL");
  if (variant < 0 || variant >= CGX_NUM_VARIANTS) return fail(CGX_ERR_ARG, "cgx_begin: unknown variant %d", variant);
  if (max_iter < 1) return fail(CGX_ERR_ARG, "cgx_begin: max_iter must be >= 1");
  if (c->op_kind == 0 || !c->problem_loaded) return fail(CGX_ERR_ARG, "cgx_begin: operator and problem must be set first");
  if (path != CGX_PATH_AUTO && path != CGX_PATH_STREAM && path != CGX_PATH_PERSISTENT)
    return fail(CGX_ERR_ARG, "cgx_begin: unknown path %d", path);
  if (c->dist.world > 1 && !c->dist_ready)
    return fail(CGX_ERR_ARG, "cgx_begin: cgx_dist_commit has not been called on this rank");
  if (c->dist.world > 1 && c->tol > 0.0)
    return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: a tolerance stops single-GPU solves only (rank %d of a partition has one set)",
                c->dist.rank);
  CU(cudaSetDevice(c->device));
  if (c->tol > 0.0 && !c->h_stop) {
    CU(cudaHostAlloc(&c->h_stop, 2 * sizeof(int), cudaHostAllocDefault));
    for (int i = 0; i < 2; ++i) CU(cudaEventCreateWithFlags(&c->ev_stop[i], cudaEventDisableTiming));
  }
  c->run_tol = c->tol;
  c->stop_k = -1;
  const bool prec = c->d_dinv != nullptr;
  const VariantInfo vi = variant_info(variant, prec);
  hist_mask &= CGX_HIST_ALL;
  if (!c->has_xtrue) hist_mask &= ~(CGX_HIST_ERROR_A_NORM | CGX_HIST_ERROR_2_NORM);

  // state vectors (allocated on demand, kept across runs)
  for (int i = 0; i < V_COUNT; ++i)
    if ((vi.need & (1u << i)) && !c->vec[i]) CU(cudaMalloc(&c->vec[i], sizeof(double) * c->n + kCbPadBytes));
  if (c->hist_len != max_iter) {
    cudaFree(c->d_hist); c->d_hist = nullptr;
    CU(cudaMalloc(&c->d_hist, sizeof(double) * CGX_HIST_ROWS * (size_t)max_iter));
    c->hist_len = max_iter;
  }
  CU(cudaMemsetAsync(c->d_hist, 0, sizeof(double) * CGX_HIST_ROWS * (size_t)max_iter, c->stream));
  c->hist_mask = hist_mask;
  c->capture = c->capture_req;
  c->cur_stage = 0;
  const bool gv_sched = variant == CGX_GV && std::any_of(c->gv_replace.begin(), c->gv_replace.end(), [](uint8_t f) { return f != 0; });
  if (c->capture || gv_sched) {
    if (c->dist.world > 1) return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: capture / GV residual replacement run on single-GPU contexts");
    if (path == CGX_PATH_PERSISTENT) return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: capture / GV residual replacement need the stream path");
    path = CGX_PATH_STREAM;
    for (int w = 0; w < 3; ++w) { cudaFree(c->d_cap[w]); c->d_cap[w] = nullptr; }
    const size_t vec_bytes = sizeof(double) * (size_t)c->n * (size_t)max_iter;
    if ((c->capture & (CGX_CAPTURE_X | CGX_CAPTURE_R)) && vec_bytes > (size_t)48 << 30)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: capturing %d vectors of %lld rows exceeds 48 GB per buffer", max_iter, (long long)c->n);
    if (c->capture & CGX_CAPTURE_X) CU(cudaMalloc(&c->d_cap[0], vec_bytes));
    if (c->capture & CGX_CAPTURE_R) CU(cudaMalloc(&c->d_cap[1], vec_bytes));
    if (c->capture & CGX_CAPTURE_SCALARS) CU(cudaMalloc(&c->d_cap[2], sizeof(double) * 2 * (size_t)max_iter));
  }
  { int trc = setup_tma(c, vi.need); if (trc) return trc; }
  c->variant = variant; c->max_iter = max_iter; c->cur_k = 0;
  {
    const PersGeom G = pers_geometry(c, variant, ranks_in_launch);
    const bool mode_ok = c->dist.world <= 1 || c->dist.mode == 1 || c->dist.mode == 3;   // in-kernel exchange only
    // measured (profiles/r01d_overlap_*): on a partition the persistent kernel wins at 2 GPUs
    // (64^3: 10-25 vs 21-31 us/iteration) and loses at 8 (22-45 vs 17-29): its all-to-all record
    // exchange is on the critical path of a much shorter iteration
    const bool world_ok = c->dist.world <= 2 && !csr_dist(c);
    if (path == CGX_PATH_PERSISTENT && csr_dist(c))
      return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: CSR row partitions run the stream kernels");
    if (path == CGX_PATH_AUTO)
      path = (c->n < c->pers_threshold && G.ok && mode_ok && world_ok) ? CGX_PATH_PERSISTENT : CGX_PATH_STREAM;
    if (path == CGX_PATH_PERSISTENT && !G.ok)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: %lld rows x %d resident vectors do not fit the SMs' shared memory "
                  "(%zu B per CTA); use the stream path", (long long)c->n, G.nslot, G.smem);
    if (path == CGX_PATH_PERSISTENT && !mode_ok)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: the persistent path exchanges scalars peer to peer (mode 1), not through NCCL");
  }
  if (path == CGX_PATH_PERSISTENT)
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < (vi.pipe && vi.recompute ? 2 : 1); ++b)
        if (!c->d_exp[a][b]) CU(cudaMalloc(&c->d_exp[a][b], sizeof(double) * c->n + kCbPadBytes));
  c->path = path;
  c->cg_elide = (variant == CGX_CG || variant == CGX_GV) && path == CGX_PATH_STREAM && c->op_kind == 2 && c->use_tma &&
                c->tmap_ok[variant == CGX_CG ? V_R : V_W] &&
                c->pm != 1 && !c->no_elide && !(variant == CGX_GV && (gv_sched || c->gv_manual));
  c->launches_run = 0; c->loop_ms = 0.0;
  c->pend.clear();
  c->pr_fused = false; c->fpar = 0;
  for (int ch = 0; ch < 3; ++ch) c->hepoch[ch] = std::max(c->hepoch[ch], c->fepoch);   // (LL tags stay unique)
  if ((variant == CGX_PR || variant == CGX_M) && path == CGX_PATH_STREAM && !c->no_fused) {
    int frc = cgx_fused_prepare(c);
    if (frc) return frc;
  }
  return CGX_OK;
}

static int begin_finish(cgx_ctx* c, i64 launches0) {
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaGetLastError());
  float ms0 = 0.f;
  CU(cudaEventElapsedTime(&ms0, c->ev[0], c->ev[1]));
  c->setup_ms = ms0;
  if (c->profile) { c->prof_cls.clear(); c->prof_used = 0; }   // initialisation is not profiled
  c->launches_run = c->launches - launches0;
  c->ran = true;
  return CGX_OK;
}

static int check_device_flags(cgx_ctx* c, const char* who) {
  if (c->use_tma || c->op_kind == 1) {
    int flag = 0;
    CU(cudaMemcpy(&flag, c->d_tma_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) return fail(CGX_ERR_CUDA, "%s: an in-kernel pipeline wait (TMA plane copy / CSR product slot) did not complete within 1 s", who);
  }
  if (c->dist.world > 1 && c->d_win) {
    int err = 0;
    CU(cudaMemcpy(&err, c->d_win + offsetof(WinHdr, error), sizeof(int), cudaMemcpyDeviceToHost));
    if (err) return fail(CGX_ERR_CUDA, "%s: rank %d waited more than 10 s for a peer (halo or scalar exchange)",
                         who, c->dist.rank);
  }
  return CGX_OK;
}

// Lockstep driver: `count` contexts (ranks of one partitioned problem, or a single context).
static int group_begin(cgx_ctx** cs, int count, int variant, int max_iter, unsigned hist_mask, int path) {
  for (int i = 0; i < count; ++i)       // (before any rank has enqueued anything)
    if (cs[i] && cs[i]->dist.world > 1 && cs[i]->tol > 0.0)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_begin: a tolerance stops single-GPU solves only (rank %d of a partition has one set)",
                  cs[i]->dist.rank);
  bool same_device = count > 1;
  for (int i = 1; i < count; ++i) same_device = same_device && cs[i]->device == cs[0]->device;
  for (int i = 0; i < count; ++i) {
    int rc = begin_prepare(cs[i], variant, max_iter, hist_mask, path, same_device ? count : 1);
    if (rc) return rc;
  }
  std::vector<Steps> steps(count);
  std::vector<i64> l0(count);
  for (int i = 0; i < count; ++i) {
    cgx_ctx* c = cs[i];
    l0[i] = c->launches;
    const VariantInfo vi = variant_info(variant, c->d_dinv != nullptr);
    build_init_steps(c, variant, vi, steps[i]);
    CU(cudaSetDevice(c->device));
    CU(cudaEventRecord(c->ev[0], c->stream));
  }
  for (size_t s = 0; s < steps[0].size(); ++s)
    for (int i = 0; i < count; ++i) {
      if (count > 1) cudaSetDevice(cs[i]->device);
      steps[i][s]();
    }
  for (int i = 0; i < count; ++i) {
    if (count > 1) cudaSetDevice(cs[i]->device);
    cgx_fused_push_initial_halo(cs[i]);
  }
  // k = 0 entry of the histories (the reference's callbacks fire on the initial state)
  for (int i = 0; i < count; ++i) cs[i]->cur_k = 0;
  if (cs[0]->hist_mask || cs[0]->capture) {
    const int core = core_stages(cs[0]);
    for (int s = core; s < iter_stage_count(cs[0]); ++s)
      for (int i = 0; i < count; ++i) {
        if (count > 1) cudaSetDevice(cs[i]->device);
        Args g = make_args(cs[i]);
        g.k = 0;
        iter_stage(cs[i], s, g);
      }
  }
  for (int i = 0; i < count; ++i) {
    cudaSetDevice(cs[i]->device);
    CU(cudaEventRecord(cs[i]->ev[1], cs[i]->stream));
  }
  for (int i = 0; i < count; ++i) {
    int rc = begin_finish(cs[i], l0[i]);
    if (rc) return rc;
    rc = check_device_flags(cs[i], "cgx_begin");
    if (rc) return rc;
  }
  return CGX_OK;
}

// After the stream has drained: adopt the stop_k the device decided (runs with a tolerance only).
static int read_stop(cgx_ctx* c) {
  if (c->run_tol <= 0.0) return CGX_OK;
  int s = -1;
  CU(cudaMemcpy(&s, &c->d_sc[c->scpar].stop_k, sizeof(int), cudaMemcpyDeviceToHost));
  c->stop_k = s;
  // the fused PR kernel swaps the buffers of p, s, rt once per iteration it runs; the launches after the
  // stop returned at entry, so the current buffers are those of iteration stop_k (cgx_cur_vec)
  if (s >= 0 && c->pr_fused) c->fpar = s & 1;
  return CGX_OK;
}

static int group_advance(cgx_ctx** cs, int count, int niter) {
  for (int i = 0; i < count; ++i)
    if (!cs[i] || !cs[i]->ran) return fail(CGX_ERR_ARG, "cgx_advance: call cgx_begin first");
  if (niter < 0) return fail(CGX_ERR_ARG, "cgx_advance: niter must be >= 0");
  cgx_ctx* c0 = cs[0];
  if (c0->stop_k >= 0) return CGX_OK;   // the tolerance was met: nothing left to run
  const int last = std::min(c0->max_iter - 1, c0->cur_k + niter);
  std::vector<i64> l0(count);
  std::vector<Args> gs(count);
  for (int i = 0; i < count; ++i) {
    CU(cudaSetDevice(cs[i]->device));
    l0[i] = cs[i]->launches;
    gs[i] = make_args(cs[i]);
    CU(cudaEventRecord(cs[i]->ev[1], cs[i]->stream));
  }
  const bool ran_pers = c0->path == CGX_PATH_PERSISTENT && last > c0->cur_k;
  if (c0->path == CGX_PATH_PERSISTENT) {
    if (last > c0->cur_k) {
      bool same_device = count > 1;
      for (int i = 1; i < count; ++i) same_device = same_device && cs[i]->device == cs[0]->device;
      if (count > 1 && !same_device)
        return fail(CGX_ERR_UNSUPPORTED, "cgx_group_advance: persistent path: one process per GPU, or all ranks on one GPU");
      const PersGeom G = pers_geometry(c0, c0->variant, count);
      int rc = pers_launch(cs, count, G, c0->cur_k + 1, last);
      if (rc) return rc;
    }
  } else {
    const int ns = iter_stage_count(c0);
    if (c0->cur_stage != 0) return fail(CGX_ERR_ARG, "cgx_advance: an iteration is half done (cgx_advance_stages); finish it first");
    // with a tolerance (single contexts only): chunks of kTolChunk iterations, each followed by a copy of
    // stop_k into pinned slot j & 1; chunk j is enqueued once chunk j - 2 has completed and did not stop
    const bool poll = c0->run_tol > 0.0;
    const int first = c0->cur_k + 1;
    for (int k = first; k <= last; ++k) {
      const int j = (k - first) / kTolChunk;
      const bool chunk_start = (k - first) % kTolChunk == 0, chunk_end = (k - first) % kTolChunk == kTolChunk - 1 || k == last;
      if (poll && chunk_start && j >= 2) {
        CU(cudaEventSynchronize(c0->ev_stop[j & 1]));
        if (c0->h_stop[j & 1] >= 0) break;
      }
      for (int s = 0; s < ns; ++s)
        for (int i = 0; i < count; ++i) {
          if (count > 1) cudaSetDevice(cs[i]->device);
          gs[i].k = k;
          if (s == 1 && cs[i]->variant == CGX_GV && k < (int)cs[i]->gv_replace.size() && cs[i]->gv_replace[k])
            launch_gv_replace(cs[i], gs[i]);
          iter_stage(cs[i], s, gs[i]);
        }
      if (poll && chunk_end) {
        CU(cudaMemcpyAsync(&c0->h_stop[j & 1], &c0->d_sc[c0->scpar].stop_k, sizeof(int), cudaMemcpyDeviceToHost, c0->stream));
        CU(cudaEventRecord(c0->ev_stop[j & 1], c0->stream));
      }
    }
    for (int i = 0; i < count; ++i) {
      if (count > 1) cudaSetDevice(cs[i]->device);
      const VariantInfo vi = variant_info(cs[i]->variant, cs[i]->d_dinv != nullptr);
      launch_flush(cs[i], gs[i], vi.meurant);
    }
  }
  for (int i = 0; i < count; ++i) {
    cudaSetDevice(cs[i]->device);
    CU(cudaEventRecord(cs[i]->ev[2], cs[i]->stream));
  }
  for (int i = 0; i < count; ++i) {
    cgx_ctx* c = cs[i];
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    if (c->comm_stream) CU(cudaStreamSynchronize(c->comm_stream));
    CU(cudaGetLastError());
    float ms1 = 0.f;
    CU(cudaEventElapsedTime(&ms1, c->ev[1], c->ev[2]));
    c->loop_ms += ms1;
    if (c->profile) prof_resolve(c);
    int rc = check_device_flags(c, "cgx_advance");
    if (rc) return rc;
    if (ran_pers) { rc = pers_collect(c); if (rc) return rc; }
    c->launches_run += c->launches - l0[i];
    rc = read_stop(c);
    if (rc) return rc;
    c->cur_k = c->stop_k >= 0 ? c->stop_k : std::max(c->cur_k, last);
  }
  return CGX_OK;
}

extern "C" int cgx_begin(cgx_ctx* c, int variant, int max_iter, unsigned hist_mask, int path) {
  return group_begin(&c, 1, variant, max_iter, hist_mask, path);
}
extern "C" int cgx_advance(cgx_ctx* c, int niter) {
  if (!c) return fail(CGX_ERR_ARG, "cgx_advance: ctx is NULL");
  return group_advance(&c, 1, niter);
}

// Ranks emulated inside one process (all on one GPU -> they share rank 0's stream, or one
// context per GPU): same kernels, same protocol, launched stage by stage in rank order.
static int group_check(cgx_ctx** cs, int count) {
  if (!cs || count < 1 || count > kMaxWorld) return fail(CGX_ERR_ARG, "cgx_group: bad arguments");
  for (int i = 0; i < count; ++i)
    if (!cs[i] || cs[i]->dist.world != count || cs[i]->dist.rank != i)
      return fail(CGX_ERR_ARG, "cgx_group: contexts must be ranks 0..%d of one partition, in order", count - 1);
  return CGX_OK;
}
static void group_share_stream(cgx_ctx** cs, int count, bool on) {
  for (int i = 1; i < count; ++i)
    if (cs[i]->device == cs[0]->device) cs[i]->stream = on ? cs[0]->own_stream : cs[i]->own_stream;
}
extern "C" int cgx_group_begin(cgx_ctx** cs, int count, int variant, int max_iter, unsigned hist_mask, int path) {
  int rc = group_check(cs, count);
  if (rc) return rc;
  group_share_stream(cs, count, true);
  rc = group_begin(cs, count, variant, max_iter, hist_mask, path);
  group_share_stream(cs, count, false);
  return rc;
}
extern "C" int cgx_group_advance(cgx_ctx** cs, int count, int niter) {
  int rc = group_check(cs, count);
  if (rc) return rc;
  group_share_stream(cs, count, true);
  rc = group_advance(cs, count, niter);
  group_share_stream(cs, count, false);
  return rc;
}
extern "C" int cgx_group_load_problem_host(cgx_ctx** cs, int count, const double* b, const double* x0,
                                           const double* xt, int64_t n_total) {
  int rc = group_check(cs, count);
  if (rc) return rc;
  if (!b || !x0) return fail(CGX_ERR_ARG, "cgx_group_load_problem_host: b and x0 are required");
  i64 off = 0;
  group_share_stream(cs, count, true);
  for (int i = 0; i < count && !rc; ++i) {
    rc = load_problem(cs[i], b + off, x0 + off, xt ? xt + off : nullptr, cs[i]->n, cudaMemcpyHostToDevice);
    off += cs[i]->n;
  }
  for (int i = 0; i < count; ++i) { cudaSetDevice(cs[i]->device); cudaStreamSynchronize(cs[i]->stream); }
  group_share_stream(cs, count, false);
  if (!rc && off != n_total) return fail(CGX_ERR_ARG, "cgx_group_load_problem_host: slabs cover %lld rows, n = %lld",
                                         (long long)off, (long long)n_total);
  return rc;
}

// ---------------------------------------------------------------------------------------
// batch: independent single-GPU solves in ONE cooperative launch (include/cgx.h cgx_batch_run)
// ---------------------------------------------------------------------------------------
static int pers_batch(cgx_ctx** cs, int count, const int* variants, const PersGeom* G, const int* k1, bool launch) {
  const cgx_ctx* c = cs[0];
  if (c->op_kind == 1) {
    if (c->pm == 2) return cgx_pers_batch_csr_pm2(cs, count, variants, G, k1, launch);
    if (c->pm == 1) return cgx_pers_batch_csr_pm1(cs, count, variants, G, k1, launch);
    return cgx_pers_batch_csr_pm0(cs, count, variants, G, k1, launch);
  }
  if (c->pm == 2) return cgx_pers_batch_sten_pm2(cs, count, variants, G, k1, launch);
  if (c->pm == 1) return cgx_pers_batch_sten_pm1(cs, count, variants, G, k1, launch);
  return cgx_pers_batch_sten_pm0(cs, count, variants, G, k1, launch);
}

// The CTA width common to the batch: the contexts' "pers_threads" when set (they must agree);
// otherwise, among the widths pers_geometry would pick for the entries on their own, the one with
// which every entry fits, most CSR entries keep their matrix rows in shared memory, and CTAs are widest.
static int batch_geometry(cgx_ctx** cs, int count, const int* variants, std::vector<PersGeom>& G) {
  int T = 0;
  for (int i = 0; i < count; ++i) {
    if (!cs[i]->pers_threads) continue;
    if (T && cs[i]->pers_threads != T)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: the entries' pers_threads differ (%d, %d); one CTA width per launch",
                  T, cs[i]->pers_threads);
    T = cs[i]->pers_threads;
  }
  std::vector<int> cand;
  if (T) cand.push_back(T);
  else
    for (int i = 0; i < count; ++i) cand.push_back(pers_geometry(cs[i], variants[i], count).T);
  int best[3] = {-1, -1, -1};
  std::vector<PersGeom> H(count);
  for (int t : cand) {
    int ok = 0, slabs = 0;
    for (int i = 0; i < count; ++i) {
      H[i] = pers_geometry_T(cs[i], variants[i], count, t);
      ok += H[i].ok ? 1 : 0;
      slabs += H[i].slab_cap > 0 ? 1 : 0;
    }
    const int score[3] = {ok == count ? 1 : 0, slabs, H[0].T};
    if (std::lexicographical_compare(best, best + 3, score, score + 3)) {
      std::copy(score, score + 3, best);
      G = H;
    }
  }
  for (int i = 0; i < count; ++i)
    if (!G[i].ok)
      return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entry %d (%lld rows x %d resident vectors) does not fit the shared "
                  "memory of its 1/%d share of the SMs (%zu B per CTA)", i, (long long)cs[i]->n, G[i].nslot, count, G[i].smem);
  return CGX_OK;
}

static int batch_run(cgx_ctx** cs, int count, const int* variants, const int* max_iters, unsigned hist_mask, cgx_info* infos) {
  // ---- refusals: nothing has been enqueued yet -------------------------------------------
  for (int i = 0; i < count; ++i) {
    const cgx_ctx* c = cs[i];
    if (c->op_kind == 0 || !c->problem_loaded) return fail(CGX_ERR_ARG, "cgx_batch_run: entry %d has no operator or problem", i);
    for (int j = 0; j < i; ++j)
      if (cs[j] == c) return fail(CGX_ERR_ARG, "cgx_batch_run: entries %d and %d are the same context", j, i);
    if (c->device != cs[0]->device) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entries on different devices");
    if (c->dist.world > 1) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entry %d is a rank of a partition", i);
    if (c->op_kind != cs[0]->op_kind) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: CSR and stencil operators mixed");
    if (c->pm != cs[0]->pm) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: preconditioner modes mixed (%d, %d)", cs[0]->pm, c->pm);
    if (c->capture_req) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entry %d has a capture set (stream path only)", i);
    if (std::any_of(c->gv_replace.begin(), c->gv_replace.end(), [](uint8_t f) { return f != 0; }))
      return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entry %d has a GV replacement schedule (stream path only)", i);
    if (c->gv_manual) return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: entry %d has gv_manual set (stream path only)", i);
  }
  CU(cudaSetDevice(cs[0]->device));
  std::vector<PersGeom> G(count);
  int rc = batch_geometry(cs, count, variants, G);
  if (rc) return rc;
  // entries with max_iter == 1 have no loop to run (as cgx_run: no launch)
  std::vector<cgx_ctx*> lc;
  std::vector<int> lv, lk;
  std::vector<PersGeom> lg;
  for (int i = 0; i < count; ++i)
    if (max_iters[i] > 1) { lc.push_back(cs[i]); lv.push_back(variants[i]); lk.push_back(max_iters[i] - 1); lg.push_back(G[i]); }
  if (!lc.empty()) {
    rc = pers_batch(lc.data(), (int)lc.size(), lv.data(), lg.data(), lk.data(), false);
    if (rc) return rc;
  }

  // ---- initial state (k = 0) of every entry, on the shared stream ------------------------
  for (int i = 0; i < count; ++i) {
    cgx_ctx* c = cs[i];
    rc = begin_prepare(c, variants[i], max_iters[i], hist_mask, CGX_PATH_PERSISTENT, count);
    if (rc) return rc;
    const i64 l0 = c->launches;
    Steps steps;
    build_init_steps(c, variants[i], variant_info(variants[i], c->d_dinv != nullptr), steps);
    CU(cudaEventRecord(c->ev[0], c->stream));
    for (auto& st : steps) st();
    cgx_fused_push_initial_halo(c);
    c->cur_k = 0;
    if (c->hist_mask) {
      for (int s = core_stages(c); s < iter_stage_count(c); ++s) {
        Args g = make_args(c);
        g.k = 0;
        iter_stage(c, s, g);
      }
    }
    CU(cudaEventRecord(c->ev[1], c->stream));
    rc = begin_finish(c, l0);
    if (rc) return rc;
    rc = check_device_flags(c, "cgx_batch_run");
    if (rc) return rc;
  }

  // ---- the iterations of every entry: one launch -----------------------------------------
  std::vector<i64> l0(count);
  for (int i = 0; i < count; ++i) {
    l0[i] = cs[i]->launches;
    CU(cudaEventRecord(cs[i]->ev[1], cs[i]->stream));
  }
  if (!lc.empty()) {
    rc = pers_batch(lc.data(), (int)lc.size(), lv.data(), lg.data(), lk.data(), true);
    if (rc) return rc;
  }
  for (int i = 0; i < count; ++i) CU(cudaEventRecord(cs[i]->ev[2], cs[i]->stream));
  CU(cudaStreamSynchronize(cs[0]->stream));
  CU(cudaGetLastError());
  bool broke = false;
  for (int i = 0; i < count; ++i) {
    cgx_ctx* c = cs[i];
    float ms1 = 0.f;
    CU(cudaEventElapsedTime(&ms1, c->ev[1], c->ev[2]));
    c->loop_ms = ms1;
    rc = check_device_flags(c, "cgx_batch_run");
    if (rc) return rc;
    if (max_iters[i] > 1) { rc = pers_collect(c); if (rc) return rc; }
    c->launches_run += c->launches - l0[i];
    rc = read_stop(c);
    if (rc) return rc;
    c->cur_k = c->stop_k >= 0 ? c->stop_k : c->max_iter - 1;
    rc = cgx_get_info(c, &infos[i]);
    if (rc) return rc;
    broke = broke || infos[i].breakdown_iter >= 0;
  }
  return broke ? CGX_ERR_BREAKDOWN : CGX_OK;
}

extern "C" int cgx_batch_run(cgx_ctx** cs, int count, const int* variants, const int* max_iters, unsigned hist_mask,
                             cgx_info* infos) {
  if (!cs || count < 1 || !variants || !max_iters || !infos) return fail(CGX_ERR_ARG, "cgx_batch_run: bad arguments");
  for (int i = 0; i < count; ++i) {
    if (!cs[i]) return fail(CGX_ERR_ARG, "cgx_batch_run: ctxs[%d] is NULL", i);
    if (variants[i] < 0 || variants[i] >= CGX_NUM_VARIANTS) return fail(CGX_ERR_ARG, "cgx_batch_run: unknown variant %d", variants[i]);
    if (max_iters[i] < 1) return fail(CGX_ERR_ARG, "cgx_batch_run: max_iter must be >= 1 (entry %d)", i);
  }
  // every entry on the first context's stream, as the ranks of a group (group_share_stream)
  for (int i = 1; i < count; ++i)
    if (cs[i]->device == cs[0]->device) cs[i]->stream = cs[0]->own_stream;
  const int rc = batch_run(cs, count, variants, max_iters, hist_mask, infos);
  for (int i = 1; i < count; ++i) cs[i]->stream = cs[i]->own_stream;
  return rc;
}

extern "C" int cgx_get_info(cgx_ctx* c, cgx_info* info) {
  if (!c || !c->ran || !info) return fail(CGX_ERR_ARG, "cgx_get_info: bad arguments");
  CU(cudaSetDevice(c->device));
  Scal h;
  CU(cudaMemcpy(&h, c->d_sc + c->scpar, sizeof(Scal), cudaMemcpyDeviceToHost));
  info->setup_ms = c->setup_ms; info->loop_ms = c->loop_ms;
  info->h2d_bytes = 0; info->d2h_bytes = 0;
  info->kernel_launches = c->launches_run;
  info->iterations = c->cur_k;
  info->breakdown_iter = h.breakdown;
  info->path = c->path;
  info->stop_iter = c->stop_k;
  return CGX_OK;
}

extern "C" int cgx_set_option(cgx_ctx* c, const char* name, int value) {
  if (!c || !name) return fail(CGX_ERR_ARG, "cgx_set_option: bad arguments");
  if (!strcmp(name, "tma")) { c->no_tma = (value == 0); return CGX_OK; }
  if (!strcmp(name, "csr_stream")) { c->no_csr_stream = (value == 0); return CGX_OK; }
  if (!strcmp(name, "csr_bulk")) { c->csr_bulk = value; return CGX_OK; }
  if (!strcmp(name, "csr_bulk_ring")) { c->csr_bulk_ring = std::max(0, std::min(value, (int)kCbMaxRing)); return CGX_OK; }
  if (!strcmp(name, "csr_bulk_sum")) { c->csr_bulk_sum = value; return CGX_OK; }
  if (!strcmp(name, "csr_bulk_ctas")) { c->csr_bulk_ctas = std::max(1, std::min(value, 4)); return CGX_OK; }
  if (!strcmp(name, "csr_slab")) { c->no_slab = (value == 0); return CGX_OK; }
  if (!strcmp(name, "cg_elide")) { c->no_elide = (value == 0); return CGX_OK; }
  if (!strcmp(name, "pr_fused")) { c->no_fused = (value == 0); return CGX_OK; }
  if (!strcmp(name, "gv_manual")) { c->gv_manual = value != 0; return CGX_OK; }
  if (!strcmp(name, "fused_min_planes")) { c->fused_min_planes = std::max(1, value); return CGX_OK; }
  if (!strcmp(name, "pdl")) { c->pdl_mode = value; return CGX_OK; }
  if (!strcmp(name, "l2_keep")) { c->l2_keep = value; return CGX_OK; }
  if (!strcmp(name, "fused_min_slab")) { c->fused_min_slab = std::max(1, value); return CGX_OK; }
  if (!strcmp(name, "fused_chunks")) { c->fused_chunks = std::max(0, value); return CGX_OK; }
  if (!strcmp(name, "persistent_threshold")) { c->pers_threshold = value; return CGX_OK; }
  if (!strcmp(name, "pers_threads")) { c->pers_threads = value; return CGX_OK; }
  if (!strcmp(name, "pers_ctas")) { c->pers_ctas = value; return CGX_OK; }
  if (!strcmp(name, "debug_skip")) { c->dbg = value; return CGX_OK; }
  if (!strcmp(name, "tma_min_planes")) { c->tma_min_planes = value; return CGX_OK; }
  if (!strcmp(name, "ew_one_wave")) { c->one_wave = value != 0; return CGX_OK; }
  if (!strcmp(name, "stub_allreduce")) {
    // timing experiment (SURVEY.md section 8d "allreduce-hiding metric"): value != 0 replaces the
    // scalar exchange by a local stand-in; value == 0 restores the mode chosen at commit
    if (c->dist.world <= 1) return fail(CGX_ERR_ARG, "cgx_set_option: stub_allreduce needs a partitioned run");
    if (value) { if (c->dist.mode != 3) { c->dist.saved_mode = c->dist.mode; c->dist.mode = 3; } }
    else if (c->dist.mode == 3) c->dist.mode = c->dist.saved_mode;
    return CGX_OK;
  }
  return fail(CGX_ERR_ARG, "cgx_set_option: unknown option '%s'", name);
}

extern "C" int cgx_set_tolerance(cgx_ctx* c, double rtol) {
  if (!c) return fail(CGX_ERR_ARG, "cgx_set_tolerance: ctx is NULL");
  if (!(rtol == 0.0 || (rtol > 0.0 && rtol < 1.0)))
    return fail(CGX_ERR_ARG, "cgx_set_tolerance: rtol must be 0 (off) or in (0, 1), got %g", rtol);
  c->tol = rtol;
  return CGX_OK;
}

// timing experiments: the 16 %globaltimer stamps kernels wrote under option debug_skip & 2
extern "C" int cgx_debug_times(cgx_ctx* c, uint64_t* out16) {
  if (!c || !out16) return fail(CGX_ERR_ARG, "cgx_debug_times: bad arguments");
  CU(cudaSetDevice(c->device));
  CU(cudaMemcpy(out16, c->d_dbg_t, sizeof(u64) * 16, cudaMemcpyDeviceToHost));
  return CGX_OK;
}

extern "C" int cgx_set_profile(cgx_ctx* c, int on) {
  if (!c) return fail(CGX_ERR_ARG, "cgx_set_profile: ctx is NULL");
  c->profile = on != 0;
  for (int i = 0; i < PC_COUNT; ++i) { c->prof_ms[i] = 0.0; c->prof_n[i] = 0; }
  c->prof_cls.clear(); c->prof_used = 0;
  return CGX_OK;
}
extern "C" int cgx_get_profile(cgx_ctx* c, int cls, double* ms, int64_t* launches) {
  if (!c || cls < 0 || cls >= PC_COUNT) return fail(CGX_ERR_ARG, "cgx_get_profile: bad arguments");
  if (ms) *ms = c->prof_ms[cls];
  if (launches) *launches = c->prof_n[cls];
  return CGX_OK;
}
extern "C" const char* cgx_profile_class_name(int cls) {
  return (cls >= 0 && cls < PC_COUNT) ? kClassNames[cls] : "";
}
extern "C" int cgx_profile_class_count(void) { return PC_COUNT; }

// scalars of the recurrences after the last completed iteration:
// out[0..8] = a_k, a_{k-1}, b_k, nu_k, nu_{k-1}, mu_k, eta_k, delta_k, gamma_k
extern "C" int cgx_get_scalars(cgx_ctx* c, double* out9) {
  if (!c || !c->ran || !out9) return fail(CGX_ERR_ARG, "cgx_get_scalars: bad arguments");
  CU(cudaSetDevice(c->device));
  Scal h;
  CU(cudaMemcpy(&h, c->d_sc + c->scpar, sizeof(Scal), cudaMemcpyDeviceToHost));
  const double v[9] = {h.a, h.a1, h.b, h.nu, h.nu1, h.mu, h.eta, h.del, h.gam};
  memcpy(out9, v, sizeof v);
  return CGX_OK;
}

extern "C" int cgx_set_capture(cgx_ctx* c, unsigned mask) {
  if (!c || (mask & ~7u)) return fail(CGX_ERR_ARG, "cgx_set_capture: bad arguments");
  c->capture_req = mask;
  return CGX_OK;
}
extern "C" int cgx_fetch_capture_host(cgx_ctx* c, int which, double* out) {
  if (!c || !c->ran || !out || which < 0 || which > 2 || !c->d_cap[which] || !(c->capture & (1u << which)))
    return fail(CGX_ERR_ARG, "cgx_fetch_capture_host: nothing captured for selector %d", which);
  CU(cudaSetDevice(c->device));
  const size_t bytes = which == 2 ? sizeof(double) * 2 * (size_t)c->hist_len : sizeof(double) * (size_t)c->n * (size_t)c->hist_len;
  CU(cudaMemcpyAsync(out, c->d_cap[which], bytes, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return CGX_OK;
}
extern "C" int cgx_set_gv_replace(cgx_ctx* c, const uint8_t* flags, int n) {
  if (!c || n < 0) return fail(CGX_ERR_ARG, "cgx_set_gv_replace: bad arguments");
  c->gv_replace.clear();
  if (flags && n > 0) c->gv_replace.assign(flags, flags + n);
  return CGX_OK;
}
// Run `nstages` kernel stages, continuing inside iteration cur_k + 1 (single context, stream path).
extern "C" int cgx_advance_stages(cgx_ctx* c, int nstages) {
  if (!c || !c->ran || nstages < 0) return fail(CGX_ERR_ARG, "cgx_advance_stages: call cgx_begin first");
  if (c->path != CGX_PATH_STREAM || c->dist.world > 1)
    return fail(CGX_ERR_UNSUPPORTED, "cgx_advance_stages: single-GPU stream path only");
  if (c->stop_k >= 0) return CGX_OK;
  CU(cudaSetDevice(c->device));
  const int ns = iter_stage_count(c);
  Args g = make_args(c);
  const i64 l0 = c->launches;
  for (; nstages > 0 && c->cur_k + 1 <= c->max_iter - 1; --nstages) {
    g.k = c->cur_k + 1;
    iter_stage(c, c->cur_stage, g);
    if (++c->cur_stage == ns) { c->cur_stage = 0; c->cur_k++; }
  }
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaGetLastError());
  c->launches_run += c->launches - l0;
  int rc = read_stop(c);
  if (rc) return rc;
  if (c->stop_k >= 0 && c->stop_k > c->cur_k) c->stop_k = -1;      // iteration stop_k is not complete yet
  if (c->stop_k >= 0) { c->cur_k = c->stop_k; c->cur_stage = 0; }
  return check_device_flags(c, "cgx_advance_stages");
}
extern "C" int cgx_gv_replace_now(cgx_ctx* c) {
  if (!c || !c->ran || c->variant != CGX_GV || c->cur_stage != 1 || c->cg_elide)
    return fail(CGX_ERR_ARG, "cgx_gv_replace_now: only between the vector pass and the SpMV pass of a GV-CG iteration "
                "begun with option gv_manual = 1");
  CU(cudaSetDevice(c->device));
  Args g = make_args(c);
  g.k = c->cur_k + 1;
  launch_gv_replace(c, g);
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaGetLastError());
  return CGX_OK;
}

extern "C" int cgx_run(cgx_ctx* c, int variant, int max_iter, unsigned hist_mask, int path,
                       cgx_info* info) {
  int rc = cgx_begin(c, variant, max_iter, hist_mask, path);
  if (rc) return rc;
  rc = cgx_advance(c, max_iter - 1);
  if (rc) return rc;
  cgx_info tmp;
  rc = cgx_get_info(c, &tmp);
  if (rc) return rc;
  if (info) *info = tmp;
  return tmp.breakdown_iter >= 0 ? CGX_ERR_BREAKDOWN : CGX_OK;
}

static int fetch(cgx_ctx* c, double* x, double* hist, cudaMemcpyKind kind) {
  if (!c || !c->ran) return fail(CGX_ERR_ARG, "cgx_fetch: nothing has been run");
  CU(cudaSetDevice(c->device));
  if (x) CU(cudaMemcpyAsync(x, c->vec[V_X], sizeof(double) * c->n, kind, c->stream));
  if (hist) CU(cudaMemcpyAsync(hist, c->d_hist, sizeof(double) * CGX_HIST_ROWS * (size_t)c->hist_len, kind, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return CGX_OK;
}
extern "C" int cgx_fetch_host(cgx_ctx* c, double* x, double* hist) { return fetch(c, x, hist, cudaMemcpyDeviceToHost); }
extern "C" int cgx_fetch_dev(cgx_ctx* c, double* x, double* hist) { return fetch(c, x, hist, cudaMemcpyDeviceToDevice); }

extern "C" int cgx_fetch_vector_host(cgx_ctx* c, const char* name, double* out) {
  if (!c || !c->ran || !name || !out) return fail(CGX_ERR_ARG, "cgx_fetch_vector_host: bad arguments");
  for (int i = 0; i < V_COUNT; ++i)
    if (!strcmp(name, kVecNames[i])) {
      if (!c->vec[i]) return fail(CGX_ERR_ARG, "cgx_fetch_vector_host: vector '%s' is not part of the last variant's state", name);
      CU(cudaSetDevice(c->device));
      if (((i == V_RT && c->variant == CGX_CG) || (i == V_WT && c->variant == CGX_GV)) && c->cg_elide && c->cur_k > 0) {
        // r~ (CG-CG) / w~ (GV) was elided in the loop: it is M r / M w
        launch_scale(c, c->d_dinv, c->vec[i == V_RT ? V_R : V_W], c->vec[i]);
        CU(cudaStreamSynchronize(c->stream));
      }
      CU(cudaMemcpy(out, cgx_cur_vec(c, i), sizeof(double) * c->n, cudaMemcpyDeviceToHost));
      return CGX_OK;
    }
  return fail(CGX_ERR_ARG, "cgx_fetch_vector_host: unknown vector '%s'", name);
}

extern "C" int cgx_solve_host(cgx_ctx* c, int variant, const double* b, const double* x0,
                              const double* xt, int64_t n, int max_iter, unsigned hist_mask,
                              int path, double* x, double* hist, cgx_info* info) {
  int rc = load_problem(c, b, x0, xt, n, cudaMemcpyHostToDevice);
  if (rc) return rc;
  int rrc = cgx_run(c, variant, max_iter, hist_mask, path, info);
  if (rrc != CGX_OK && rrc != CGX_ERR_BREAKDOWN) return rrc;
  rc = cgx_fetch_host(c, x, hist);
  if (rc) return rc;
  if (info) {
    info->h2d_bytes = (double)sizeof(double) * n * (xt ? 3 : 2);
    info->d2h_bytes = (double)sizeof(double) * ((x ? n : 0) + (hist ? (i64)CGX_HIST_ROWS * max_iter : 0));
  }
  return rrc;
}

// ---------------------------------------------------------------------------------------
// multi-GPU set-up (include/cgx.h "row-partitioned runs")
// ---------------------------------------------------------------------------------------
extern "C" int cgx_set_stencil_slab(cgx_ctx* c, int64_t nx, int64_t ny, int64_t nz_local, int world, int rank,
                                    double diag, double off) {
  if (!c || world < 1 || world > kMaxWorld || rank < 0 || rank >= world)
    return fail(CGX_ERR_ARG, "cgx_set_stencil_slab: bad arguments (world <= %d)", kMaxWorld);
  if ((nx * ny) % 2 != 0 && world > 1)
    return fail(CGX_ERR_UNSUPPORTED, "cgx_set_stencil_slab: nx*ny must be even (16-byte halo stores)");
  CU(cudaSetDevice(c->device));
  dist_release(c);
  int rc = set_stencil(c, 3, nx, ny, nz_local, diag, off, rank > 0, rank < world - 1);
  if (rc) return rc;
  if (world == 1) return CGX_OK;
  Dist& d = c->dist;
  d.world = world; d.rank = rank; d.mode = 1; d.saved_mode = 1;
  d.has_lo = rank > 0; d.has_hi = rank < world - 1;
  d.plane = nx * ny;
  c->win_bytes = kWinHdrBytes + sizeof(double) * (size_t)kChan * 4 * (size_t)d.plane   // ghost planes (stream path)
                 + sizeof(u64) * 3 * 4 * 2 * (size_t)d.plane;                       // LL ghost planes (persistent path)
  CU(cudaMalloc(&c->d_win, c->win_bytes));
  CU(cudaMemset(c->d_win, 0, c->win_bytes));
  CU(cudaDeviceSynchronize());
  c->peer_base[rank] = c->d_win;
  c->epoch = 0; c->scpar = 0; c->pend.clear();
  for (auto& h : c->hepoch) h = 0;
  c->fepoch = 0;
  return CGX_OK;
}

extern "C" int cgx_dist_ipc_handle(cgx_ctx* c, void* handle64) {
  if (!c || !c->d_win || !handle64) return fail(CGX_ERR_ARG, "cgx_dist_ipc_handle: no window (cgx_set_stencil_slab first)");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
  CU(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, c->d_win));
  memcpy(handle64, &h, 64);
  return CGX_OK;
}
extern "C" int cgx_dist_attach_ipc(cgx_ctx* c, int peer, const void* handle64) {
  if (!c || !c->d_win || !handle64 || peer < 0 || peer >= c->dist.world || peer == c->dist.rank)
    return fail(CGX_ERR_ARG, "cgx_dist_attach_ipc: bad arguments");
  CU(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  c->peer_base[peer] = (unsigned char*)p;
  c->peer_ipc[peer] = true;
  return CGX_OK;
}
extern "C" int cgx_dist_attach_ctx(cgx_ctx* c, int peer, cgx_ctx* other) {
  if (!c || !other || !c->d_win || !other->d_win || peer < 0 || peer >= c->dist.world || peer == c->dist.rank ||
      other->dist.rank != peer || other->dist.world != c->dist.world)
    return fail(CGX_ERR_ARG, "cgx_dist_attach_ctx: bad arguments");
  if (other->device != c->device) {
    CU(cudaSetDevice(c->device));
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, c->device, other->device));
    if (!can) return fail(CGX_ERR_UNSUPPORTED, "cgx_dist_attach_ctx: device %d cannot access device %d", c->device, other->device);
    cudaError_t e = cudaDeviceEnablePeerAccess(other->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
      return fail(CGX_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
    cudaGetLastError();
  }
  c->peer_base[peer] = other->d_win;
  c->peer_ipc[peer] = false;
  return CGX_OK;
}
extern "C" int cgx_dist_nccl_unique_id(const char* libpath, void* id128) {
  if (!id128) return fail(CGX_ERR_ARG, "cgx_dist_nccl_unique_id: id is NULL");
  int rc = nccl_load(libpath);
  if (rc) return rc;
  int e = g_nccl.GetUniqueId(id128);
  if (e) return fail(CGX_ERR_CUDA, "ncclGetUniqueId: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(e) : "?");
  return CGX_OK;
}
// mode: 1 = peer-to-peer flag exchange of the fused scalars, 2 = ncclAllReduce on a side stream
extern "C" int cgx_dist_commit(cgx_ctx* c, int mode, const char* nccl_libpath, const void* nccl_id128) {
  if (!c || !c->d_win || (mode != 1 && mode != 2)) return fail(CGX_ERR_ARG, "cgx_dist_commit: bad arguments");
  CU(cudaSetDevice(c->device));
  Dist& d = c->dist;
  for (int r = 0; r < d.world; ++r) {
    if (!c->peer_base[r]) return fail(CGX_ERR_ARG, "cgx_dist_commit: rank %d's window is not attached", r);
    d.win[r] = reinterpret_cast<WinHdr*>(c->peer_base[r]);
  }
  d.ghost = reinterpret_cast<double*>(c->d_win + kWinHdrBytes);
  if (d.csr)
    for (int r = 0; r < d.world; ++r) d.stage_of[r] = reinterpret_cast<double*>(c->peer_base[r] + kWinHdrBytes);
  d.ghost_lo = d.has_lo ? reinterpret_cast<double*>(c->peer_base[d.rank - 1] + kWinHdrBytes) : nullptr;
  d.ghost_hi = d.has_hi ? reinterpret_cast<double*>(c->peer_base[d.rank + 1] + kWinHdrBytes) : nullptr;
  const size_t ll_at = kWinHdrBytes + sizeof(double) * (size_t)kChan * 4 * (size_t)d.plane;
  d.ghl = d.csr ? nullptr : reinterpret_cast<u64*>(c->d_win + ll_at);
  d.ghl_lo = d.has_lo ? reinterpret_cast<u64*>(c->peer_base[d.rank - 1] + ll_at) : nullptr;
  d.ghl_hi = d.has_hi ? reinterpret_cast<u64*>(c->peer_base[d.rank + 1] + ll_at) : nullptr;
  d.mode = mode; d.saved_mode = mode;
  if (mode == 2) {
    if (!nccl_id128) return fail(CGX_ERR_ARG, "cgx_dist_commit: mode 2 needs the NCCL unique id");
    int rc = nccl_load(nccl_libpath);
    if (rc) return rc;
    Nid id;
    memcpy(&id, nccl_id128, 128);
    int e = g_nccl.CommInitRank(&c->nccl_comm, d.world, id, d.rank);
    if (e) return fail(CGX_ERR_CUDA, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(e) : "?");
    CU(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
    for (int s = 0; s < kSlots; ++s) {
      CU(cudaEventCreateWithFlags(&c->ev_prod[s], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&c->ev_red[s], cudaEventDisableTiming));
    }
    CU(cudaMalloc(&c->d_nccl, sizeof(double) * 2 * kSlots * kSumW));
    CU(cudaMemset(c->d_nccl, 0, sizeof(double) * 2 * kSlots * kSumW));
    d.nccl_in = c->d_nccl;
    d.nccl_out = c->d_nccl + kSlots * kSumW;
  }
  CU(cudaDeviceSynchronize());
  c->dist_ready = true;
  return CGX_OK;
}

// ---------------------------------------------------------------------------------------
// primitives for unit tests
// ---------------------------------------------------------------------------------------
extern "C" int cgx_spmv_host(cgx_ctx* c, const double* v, double* y, int64_t n) {
  if (!c || !v || !y || c->op_kind == 0 || n != c->n) return fail(CGX_ERR_ARG, "cgx_spmv_host: bad arguments");
  if (c->dist.world > 1) return fail(CGX_ERR_UNSUPPORTED, "cgx_spmv_host: single-GPU primitive");
  CU(cudaSetDevice(c->device));
  double *dv = nullptr, *dy = nullptr;
  CU(cudaMalloc(&dv, sizeof(double) * n));
  CU(cudaMalloc(&dy, sizeof(double) * n));
  CU(cudaMemcpyAsync(dv, v, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  Args g{};
  g.n = n;
  g.d.world = 1;
  g.errflag = c->d_tma_err;
  CUtensorMap tm;
  if (c->op_kind == 2 && tma_prepare_geom(c) && tma_encode_dims(dv, c->sten.nx, c->sten.ny, c->sten.nz, &tm)) {
    // the TMA-staged stencil kernel in its plainest mode (SP_PIPE_N: u = A v, no epilogue)
    g.u = dy;
    const int per_sm = ctx_occupancy(c, (const void*)stencil_tma_kernel<SP_PIPE_N, 0, false>, kSThreads, tma_smem_bytes(1));
    TmaGeom G = c->geom;
    const int cap = per_sm * c->sm_count, ncols = G.ntx * G.nty;
    G.nchunk = std::max(1, std::min(cap / std::max(1, ncols), G.nz / std::max(1, c->tma_min_planes)));
    stencil_tma_kernel<SP_PIPE_N, 0, false><<<(int)std::min<i64>((i64)ncols * G.nchunk, cap), kSThreads, tma_smem_bytes(1), c->stream>>>(
        tm, tm, G, g);
    c->launches++;
  } else {
    launch_spmv<SP_PLAIN, 0, false>(c, g, dv, dy);
  }
  CU(cudaMemcpyAsync(y, dy, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaGetLastError());
  cudaFree(dv); cudaFree(dy);
  return CGX_OK;
}

extern "C" int cgx_dot_host(cgx_ctx* c, const double* u, const double* v, int64_t n, double* out) {
  if (!c || !u || !v || !out || n < 1) return fail(CGX_ERR_ARG, "cgx_dot_host: bad arguments");
  CU(cudaSetDevice(c->device));
  double *du = nullptr, *dv = nullptr;
  CU(cudaMalloc(&du, sizeof(double) * n));
  CU(cudaMalloc(&dv, sizeof(double) * n));
  CU(cudaMemcpyAsync(du, u, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(dv, v, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  const i64 keep = c->n;
  c->n = n;
  launch_dot(c, du, dv, nullptr, 7);
  c->n = keep;
  Scal h;
  CU(cudaMemcpyAsync(&h, c->d_sc + c->scpar, sizeof(Scal), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaGetLastError());
  *out = h.tmp[7];
  cudaFree(du); cudaFree(dv);
  return CGX_OK;
}
