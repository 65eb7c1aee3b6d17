// Shared definitions for the BSR sampling kernels (sm_100a).
//
// Tree storage follows include/bsr_b200.h: one fixed-capacity slot of pre-order tokens per (chain, tree);
// slot i is the node with genList order i (reference codes/funcs.py:127-142).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/bsr_b200.h"

#define BSR_MAXN BSR_MAX_NODES
#define BSR_MAXK BSR_MAX_TREES

enum : int {
  OP_LEAF = 0, OP_INV = 1, OP_LT = 2, OP_NEG = 3, OP_SIN = 4, OP_COS = 5, OP_EXP = 6, OP_SQUARE = 7,
  OP_CUBIC = 8, OP_ADD = 9, OP_MUL = 10
};
enum : int { CH_NONE = 0, CH_EXPANSION = 1, CH_SHRINKAGE = 2 };
enum : int { MV_STAY = 0, MV_GROW, MV_PRUNE, MV_DETR, MV_TRANS, MV_ROP, MV_RFEAT };
#define BSR_N_MOVES 7
#ifndef BSR_N_SIZE_CLASSES
#define BSR_N_SIZE_CLASSES 1   // classes of the proposal sort besides the move: 4 = tree-size classes (measured slower), 2 = live tree with / without lt nodes
#endif
#define BSR_N_BINS (BSR_N_MOVES * BSR_N_SIZE_CLASSES)
// PropInfo.flags
enum : int { PF_CAPACITY = 1, PF_TAPE_DESYNC = 2, PF_SKIP = 4 };

__host__ __device__ __forceinline__ int tok_op(uint32_t t) { return (int)(t & 0xffu); }
__host__ __device__ __forceinline__ int tok_oi(uint32_t t) { return (int)((t >> 8) & 0xffu); }
__host__ __device__ __forceinline__ int tok_ft(uint32_t t) { return (int)(t >> 16); }
__host__ __device__ __forceinline__ uint32_t make_tok(int op, int oi, int ft) {
  return (uint32_t)op | ((uint32_t)oi << 8) | ((uint32_t)ft << 16);
}
__host__ __device__ __forceinline__ int op_arity(int op) { return op == OP_LEAF ? 0 : (op >= OP_ADD ? 2 : 1); }

// Prior / proposal constants, computed once on the host in float64 (so they match numpy) and passed by value.
struct PriorTables {
  int n_ops;
  int n_feature;
  int ops[BSR_MAX_OPS];
  double w[BSR_MAX_OPS];       // Op_weights
  double logw[BSR_MAX_OPS];    // log(Op_weights[i])
  double cdf[BSR_MAX_OPS];     // cumsum(Op_weights) for the categorical draw (np.random.choice)
  double psplit[BSR_MAXN + 1];   // 1 / (1+depth)^(-beta)              codes/funcs.py:79
  double logsplit[BSR_MAXN + 1]; // beta * log(1+depth)                codes/funcs.py:370
  double log1m[BSR_MAXN + 1];    // log(1 - psplit[depth])             codes/funcs.py:362-363
  double lognf;                  // log(n_feature)                     codes/funcs.py:364
  double beta;
};

// Everything logR needs from the proposal stage (codes/funcs.py:1189-1210), one per (chain, tree).
struct PropInfo {
  int move, change, flags, ndraws;
  double Q, Qinv, hratio, detjacob;
  double new_sigma, new_sa2, new_sb2;
  double ll_new, lp_new;       // fStruc of the proposed tree (with its new sigma_a, sigma_b): log p(T, M), log p(Theta | ...)
  double fs_old;               // prior term of the live tree as it enters log_strucratio (funcs.py:1241-1245 / 1287-1289)
  int m_new, m_old;
};
// prior term of the proposed tree as it enters log_strucratio: both parts of fStruc when the dimension changes, else the first
__host__ __device__ __forceinline__ double prop_fs_new(const PropInfo& pi) { return (pi.change != CH_NONE) ? (pi.ll_new + pi.lp_new) : pi.ll_new; }

// Device view of the chain state (all arrays live in HBM; SoA over chains).
struct ChainState {
  int C, K;
  // two tree buffers per (chain, tree); `which` selects the live one, the other receives the proposal
  uint32_t* tok[2];   // [C][K][MAXN]
  double* pa[2];      // [C][K][MAXN]
  double* pb[2];
  int* nn[2];         // [C][K]
  int* which;         // [C][K]
  int* report_which;  // [C][K]  buffer holding the tree BSR.fit would report in roots_ (quirk Q16)
  double* sigma;      // [C]
  double* sa;         // [C][K]
  double* sb;         // [C][K]
  double* sse;        // [C]   K-column, no-intercept SSE of the live state (ylogLike, funcs.py:1147-1162)
  double* beta;       // [C][K+1]
  double* err;        // [C][err_cap]
  int* nerr;          // [C]
  int* total;         // [C]  consecutive rejections (bsr_class.py:165,195,243)
  int* done;          // [C]
  long long* counters;  // [C][BSR_N_COUNTERS]
  PropInfo* pinfo;    // [C][K]
  // column cache (fp32 evaluation only): the values of every live tree on all local rows, double-buffered like the
  // trees (buffer `which` = live column, the other receives the proposal's column, accept = flip), plus the Gram
  // entries among the live columns.  Lets a sweep evaluate K trees instead of 2K.  col[0] == nullptr: disabled.
  float* col[2];      // [C][K][col_ld]
  long long col_ld;
  double* sg;         // [C][K(K+1)/2 + 3K]  G(live,live) upper, live'y, live sums, max|live|
  // what the proposal kernels need of a live tree besides its tokens, kept up to date by the window path (refit, accept):
  double* lfs;        // [C][K][2] fStruc of the live tree with its sigma_a, sigma_b: log p(T, M), log p(Theta | T, sigma_a, sigma_b)
  int* lcnt;          // [C][K] node count | lt nodes << 8 | terminals << 16 | detransform candidates << 24 (0: not computed)
  unsigned char* live_bad;   // [C][K] live column has values outside the fp32 range: the chain's sweeps run in fp64
  unsigned char* prop_bad;   // [C][K] same for the proposal of the current sweep
  // Philox key of every chain (bsr_init_chains: the handle's seed and the chain's global id) and the data set it fits
  uint64_t* key_seed; // [C]
  int64_t* key_id;    // [C]
  int* ds;            // [C]  index into the handle's data sets ([D][d][ld] X, [D][ld] y, [D][2] y statistics)
  int err_cap;
  int val;
  int plateau_rule;
};

// Speculative proposal windows (bsr_window.cuh): W consecutive proposals of every chain, generated from one live state.
#define BSR_MAXW 64

#define BSR_WIN_RING 8      // windows kept per chain at most: the current one and up to seven before it (record cache); WinState::R of them are
                            // allocated (bsr_tu_window.cu: ensure_window takes fewer when the slot arrays would not fit the device)

struct WinState {
  int W;                   // proposals per window (<= 64)
  int S;                   // row splits of the evaluation kernels
  int C;                   // chains of the handle
  int R;                   // ring depth in use, 2 .. BSR_WIN_RING
  // Every per-slot array holds R windows per chain (index = ring * C * W + c * W + i ...): a chain writes its
  // windows round-robin, so that the windows before the current one -- same live state as long as the chain accepted
  // nothing -- stay readable as an exact-match cache of records (bsr_window.cuh: k_wdedup).  chead[c]: ring index of the
  // chain's last window if it is still valid for the live state, else -1; cvalid[c]: how many consecutive windows ending
  // there are valid (<= R - 1); the current window goes to ring index (chead + 1) % R.
  uint32_t* tok;           // [RING][C][W][MAXN] proposed trees
  double* pa;
  double* pb;
  int* nn;                 // [RING][C][W]
  PropInfo* info;          // [RING][C][W]
  double* rec;             // [RING][C][S][W][K+4] partial sums of every proposal, one record per row split
  unsigned long long* bad; // [RING][C] bit i: proposal i left the fp32 range (its record comes from the double-range pass)
  unsigned long long* hash;// [RING][C][W] tree hash of every slot (0: slot not evaluated)
  signed char* chead;      // [C]
  unsigned char* cvalid;   // [C]
  unsigned char* rep;      // [C][W] first slot of the window that holds the same tree (itself if none): evaluated once; bit 7: the
                           //         record was taken from an earlier window (nothing interpreted)
  unsigned short* prevslot;// [C][W] for a slot with bit 7 set in rep: slot | (windows back - 1) << 6 of the window that holds its tree
  unsigned char* order;    // [C][W] the slots k_weval interprets, largest tree first; neval[c] of them
  int* neval;              // [C]
  long long* pos;          // [C] index of the chain's next proposal
  int* bucket;             // [BSR_N_BINS][C * W] slots sorted by (move, size class) (k_wclassify)
  // Cache of the live columns (fp32 evaluation mode; nullptr: disabled -- fp64 mode, or it would not fit the device): the fp32 values
  // of every live tree on all local rows, written by the first window that evaluates the tree and read by the following ones until
  // the tree is replaced.  A column with out-of-range vectors (value rule, bsr_window.cuh) is never cached: it is interpreted anew.
  float* lcol;             // [C][K][lcol_ld]
  long long lcol_ld;       // >= n, multiple of 4
  unsigned char* lcol_ok;  // [C][K] the cached column is the live tree's
  unsigned* lcol_wide;     // [C] bit j: live column j had an out-of-range vector in the current window (set by k_weval, reset by k_wclassify)
  int* bucket_count;       // [n_groups][32]
};
// ring index chain c writes its current window to
__device__ __forceinline__ int win_parity(const WinState& ws, int c) { const int p = ws.chead[c]; return p >= 0 ? ((p + 1) % ws.R) : 0; }
// the same WinState with its per-slot arrays rebased to ring index `par` (indexing by c * W + i etc. stays as it is)
__device__ __forceinline__ WinState win_half(const WinState& ws, int par, int K) {
  WinState v = ws;
  const size_t cw = (size_t)par * ws.C * ws.W;
  v.tok += cw * BSR_MAXN; v.pa += cw * BSR_MAXN; v.pb += cw * BSR_MAXN; v.nn += cw; v.info += cw; v.hash += cw;
  v.rec += cw * ws.S * (K + 4);
  v.bad += (size_t)par * ws.C;
  return v;
}
