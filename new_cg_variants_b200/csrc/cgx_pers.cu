// cgx_pers.cu -- launchers of the persistent cooperative kernels (cgx_persistent.cuh: one variant,
// or a batch of independent solves) for one operator kind and one preconditioner mode (compiled six times: -DCGX_PERS_OP=1 CSR | 2 matrix-free
// stencil, -DCGX_PERS_PM=0|1|2).
#include "cgx_host.h"

#ifndef CGX_PERS_OP
#error "compile with -DCGX_PERS_OP=1|2"
#endif

// the kernel's view of context c; its sync counter and PersOut are zeroed on `st`
template <class Op>
static int pers_fill_rank(cgx_ctx* c, cudaStream_t st, PersRank<Op>& r) {
  if constexpr (std::is_same<Op, CsrOp>::value) r.A = c->csr; else r.A = c->sten;
  Args g = make_args(c);
  Plan p;                                           // fills scpar / x_true epochs
  plan_apply(c, g, p);
  r.g = g;
  r.g.l2pol = 0;                                    // (the persistent kernel addresses shared memory)
  for (int v = 0; v < V_COUNT; ++v) r.vecs[v] = c->vec[v];
  r.vecs[10] = c->d_dinv; r.vecs[11] = nullptr;
  for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) r.exp_[a][b] = c->d_exp[a][b];
  r.bar = c->d_pbar; r.part = c->d_ppart; r.out = c->d_pout;
  r.epoch0 = c->epoch;
  for (int ch = 0; ch < kChan; ++ch) r.hepoch0[ch] = c->hepoch[ch];
  CU(cudaMemsetAsync(c->d_pbar, 0, sizeof(u64) * 2, st));
  CU(cudaMemsetAsync(c->d_pout, 0, sizeof(PersOut), st));
  return CGX_OK;
}

template <class Op, int PM>
static int pers_launch_pm(cgx_ctx** cs, int count, const PersGeom& G, int k0, int k1) {
  cgx_ctx* c0 = cs[0];
  std::vector<PersRank<Op>> h(count);
  for (int i = 0; i < count; ++i) {
    int rc = pers_fill_rank<Op>(cs[i], c0->stream, h[i]);
    if (rc) return rc;
  }
  CU(cudaMemcpyAsync(c0->d_prank, h.data(), sizeof(PersRank<Op>) * count, cudaMemcpyHostToDevice, c0->stream));
  CU(cudaStreamSynchronize(c0->stream));           // h is a host temporary
  PersLaunch L{};
  L.k0 = k0; L.k1 = k1; L.nb = G.nb; L.R = G.R; L.vmask = G.vmask; L.nslot = G.nslot; L.slab_cap = G.slab_cap;
  const PersRank<Op>* dr = static_cast<const PersRank<Op>*>(c0->d_prank);
  void* params[] = {(void*)&dr, (void*)&L};
  const void* fn = nullptr;
#define CGX_PV(V) case V: fn = (const void*)persistent_kernel<Op, V, PM>; break;
  switch (c0->variant) {
    CGX_PV(CGX_HS) CGX_PV(CGX_CG) CGX_PV(CGX_GV) CGX_PV(CGX_PR) CGX_PV(CGX_M) CGX_PV(CGX_PIPE_PR)
    CGX_PV(CGX_PIPE_P) CGX_PV(CGX_PIPE_PR_M) CGX_PV(CGX_PIPE_P_M)
  }
#undef CGX_PV
  if (!fn) return fail(CGX_ERR_ARG, "persistent path: unknown variant");
  CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G.smem));
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, G.T, G.smem));
  if ((i64)per_sm * c0->sm_count < (i64)G.nb * count)
    return fail(CGX_ERR_UNSUPPORTED, "persistent path: %d CTAs of %d threads / %zu B shared memory are not co-resident",
                G.nb * count, G.T, G.smem);
  CU(cudaLaunchCooperativeKernel(fn, dim3(G.nb * count), dim3(G.T), params, G.smem, c0->stream));
  c0->launches++;
  return CGX_OK;
}

// Batch of independent solves (cgx_batch_run): entry i = context cs[i] running variants[i] for
// iterations 1 .. k1[i] with CTA shape G[i], all in one cooperative launch on cs[0]'s stream.
// With `launch` false only the co-residency of the grid is checked (nothing is enqueued).
template <class Op, int PM>
static int pers_batch_pm(cgx_ctx** cs, int count, const int* variants, const PersGeom* G, const int* k1, bool launch) {
  cgx_ctx* c0 = cs[0];
  int ctas = 0, T = G[0].T;
  size_t smem = 0;
  for (int i = 0; i < count; ++i) {
    if (G[i].T != T) return fail(CGX_ERR_ARG, "cgx_batch_run: entries of one launch share the CTA width");
    ctas += G[i].nb;
    smem = std::max(smem, G[i].smem);
  }
  const void* fn = (const void*)persistent_batch_kernel<Op, PM>;
  CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, T, smem));
  if ((i64)per_sm * c0->sm_count < (i64)ctas)
    return fail(CGX_ERR_UNSUPPORTED, "cgx_batch_run: %d CTAs of %d threads / %zu B shared memory are not co-resident",
                ctas, T, smem);
  if (!launch) return CGX_OK;
  std::vector<PersEntry<Op>> h(count);
  int cta0 = 0;
  for (int i = 0; i < count; ++i) {
    PersEntry<Op>& e = h[i];
    int rc = pers_fill_rank<Op>(cs[i], c0->stream, e.r);
    if (rc) return rc;
    e.L = PersLaunch{};
    e.L.k0 = 1; e.L.k1 = k1[i]; e.L.nb = G[i].nb; e.L.R = G[i].R; e.L.vmask = G[i].vmask;
    e.L.nslot = G[i].nslot; e.L.slab_cap = G[i].slab_cap;
    e.variant = variants[i];
    e.cta0 = cta0;
    cta0 += G[i].nb;
  }
  const size_t bytes = sizeof(PersEntry<Op>) * count;
  if (c0->pbatch_bytes < bytes) {
    CU(cudaStreamSynchronize(c0->stream));         // (a previous batch may still read the old table)
    cudaFree(c0->d_pbatch);
    c0->d_pbatch = nullptr; c0->pbatch_bytes = 0;
    CU(cudaMalloc(&c0->d_pbatch, bytes));
    c0->pbatch_bytes = bytes;
  }
  CU(cudaMemcpyAsync(c0->d_pbatch, h.data(), bytes, cudaMemcpyHostToDevice, c0->stream));
  CU(cudaStreamSynchronize(c0->stream));           // h is a host temporary
  const PersEntry<Op>* de = static_cast<const PersEntry<Op>*>(c0->d_pbatch);
  int cnt = count;
  void* params[] = {(void*)&de, (void*)&cnt};
  CU(cudaLaunchCooperativeKernel(fn, dim3(ctas), dim3(T), params, smem, c0->stream));
  for (int i = 0; i < count; ++i) cs[i]->launches++;
  return CGX_OK;
}

#ifndef CGX_PERS_PM
#error "compile with -DCGX_PERS_PM=0|1|2"
#endif
#define CGX_CAT_(a, b, c) a##b##c
#define CGX_CAT(a, b, c) CGX_CAT_(a, b, c)
#if CGX_PERS_OP == 1
int CGX_CAT(cgx_pers_launch_csr, _pm, CGX_PERS_PM)(cgx_ctx** cs, int count, const PersGeom& G, int k0, int k1) {
  return pers_launch_pm<CsrOp, CGX_PERS_PM>(cs, count, G, k0, k1);
}
int CGX_CAT(cgx_pers_batch_csr, _pm, CGX_PERS_PM)(cgx_ctx** cs, int count, const int* variants, const PersGeom* G,
                                                  const int* k1, bool launch) {
  return pers_batch_pm<CsrOp, CGX_PERS_PM>(cs, count, variants, G, k1, launch);
}
#else
int CGX_CAT(cgx_pers_launch_sten, _pm, CGX_PERS_PM)(cgx_ctx** cs, int count, const PersGeom& G, int k0, int k1) {
  return pers_launch_pm<StencilOp, CGX_PERS_PM>(cs, count, G, k0, k1);
}
int CGX_CAT(cgx_pers_batch_sten, _pm, CGX_PERS_PM)(cgx_ctx** cs, int count, const int* variants, const PersGeom* G,
                                                   const int* k1, bool launch) {
  return pers_batch_pm<StencilOp, CGX_PERS_PM>(cs, count, variants, G, k1, launch);
}
#endif
