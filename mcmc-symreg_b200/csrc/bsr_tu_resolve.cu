// Resolve stage launches: rank test, ridge OLS, logR, accept, refit (one thread per chain).
#include <cstdio>
#include "bsr_handle.h"
#include "bsr_kernels.cuh"

static ResolveCtx make_rc(bsr_handle* h) {
  ResolveCtx rc;
  rc.n_total = (double)h->n_total; rc.n_local = (double)h->n; rc.ystats = h->ystats;
  rc.pivot_tol = h->cfg.precision == 1 ? 1e-13 : 3e-13;
  rc.sweep = h->sweep;
  rc.tape = h->tape_mode ? h->tape : nullptr; rc.tape_off = h->tape_off;
  rc.trace = (h->tape_pos < h->tape_steps) ? h->trace : nullptr;
  rc.steps = h->tape_steps; rc.step_base = h->tape_pos;
  rc.cached = (h->st.col[0] != nullptr && h->cfg.precision == 0 && h->cfg.K <= 5) ? 1 : 0;
  return rc;
}

template <int MODE>
static void launch_resolve(bsr_handle* h, cudaStream_t s, const ResolveCtx& rc, int init_only) {
  const int C = h->cfg.n_chains, P = 2 * h->cfg.K;
  const int cn = rc.cn;
  const double* sums = h->gram;
  const double* maxs = h->gram + (size_t)C * gram_n_sum(P);
  int KP = 1;
  while (KP < h->cfg.K) KP *= 2;                       // lanes per chain (a power of two, so chains do not straddle warps)
  const int threads = 32, cpb = threads / KP, blocks = (cn + cpb - 1) / cpb;
  const size_t smem = (size_t)cpb * ((gram_n_sum(P) + P) * sizeof(double) + h->cfg.K * sizeof(PropInfo));
  if (smem > 48 * 1024) {
    cudaFuncSetAttribute(k_resolve<MODE, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
  switch (h->cfg.K) {
    case 1: k_resolve<MODE, 1><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
    case 2: k_resolve<MODE, 2><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
    case 3: k_resolve<MODE, 3><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
    case 4: k_resolve<MODE, 4><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
    case 5: k_resolve<MODE, 5><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
    default: k_resolve<MODE, 0><<<blocks, threads, smem, s>>>(h->st, rc, sums, maxs, init_only, KP); break;
  }
}

int bsr_launch_resolve(bsr_handle* h, cudaStream_t s, int init_only, int c0, int cn) {
  ResolveCtx rc = make_rc(h);
  rc.c0 = c0; rc.cn = cn;
  const bool taped = !init_only && h->tape_mode && h->tape_pos < h->tape_steps;
  if (taped) launch_resolve<1>(h, s, rc, init_only);
  else launch_resolve<0>(h, s, rc, init_only);
  CK(cudaGetLastError());
  return 0;
}
