// Proposal stage launches: prior initialisation and Prop + auxProp (one thread per (chain, tree)).
#include <cstdio>
#include "bsr_handle.h"
#include "bsr_kernels.cuh"

int bsr_launch_init_chains(bsr_handle* h, cudaStream_t s) {
  const int total = h->cfg.n_chains * h->cfg.K;
  k_init_chains<0><<<(total + 63) / 64, 64, 0, s>>>(h->st, h->d_pt);
  CK(cudaGetLastError());
  return 0;
}

int bsr_launch_propose(bsr_handle* h, cudaStream_t s, int c0, int cn) {
  const int total = cn * h->cfg.K;
  ProposeCtx pc;
  pc.sweep = h->sweep;
  pc.tape = h->tape; pc.tape_off = h->tape_off; pc.steps = h->tape_steps; pc.step_base = h->tape_pos;
  pc.rec = h->rec; pc.rec_count = h->rec_count; pc.rec_steps = h->rec_steps; pc.rec_cap = h->rec_cap; pc.rec_base = h->rec_pos;
  pc.c0 = c0; pc.cn = cn;
  const bool taped = h->tape_mode && h->tape_pos < h->tape_steps;
  const int threads = 32, blocks = (total + threads - 1) / threads;
  if (taped) k_propose<1><<<blocks, threads, 0, s>>>(h->st, h->d_pt, pc);
  else if (h->rec != nullptr && h->rec_pos < h->rec_steps) k_propose<2><<<blocks, threads, 0, s>>>(h->st, h->d_pt, pc);
  else k_propose<0><<<blocks, threads, 0, s>>>(h->st, h->d_pt, pc);
  CK(cudaGetLastError());
  return 0;
}
