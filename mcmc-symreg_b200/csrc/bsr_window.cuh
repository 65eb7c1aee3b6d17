// Speculative proposal windows: the production path of bsr_run.
//
// A chain's proposals form one linear sequence p = 0, 1, 2, ... (proposal p works on tree p % K; a sweep of
// codes/bsr_class.py:179 is K consecutive proposals).  A rejected newProp (codes/funcs.py:1298-1306) leaves the chain
// state untouched, and the acceptance rate of this sampler is of the order of 1 %, so a window of W <= 64 consecutive
// proposals is generated from the SAME live state, all W are evaluated and scored in parallel, and the window is then
// consumed in order up to and including its first accept (or a stop rule); the proposals behind an accept were
// generated from a stale state and are discarded -- the next window regenerates them from the new state.  Every
// random draw is a Philox function of (the chain's key, proposal index, purpose), so the chain is exactly the
// one the proposal-by-proposal pipeline (bsr_kernels.cuh) produces; only the order of the work changes:
//
//   k_wpropose  one thread per (chain, window slot): Prop + auxProp + fStruc     codes/funcs.py:1188-1210
//   k_weval     one block per chain: the K live columns are evaluated once per row tile into shared memory (fp64),
//               then each warp interprets one proposal at a time (allcal, codes/funcs.py:175-220) and accumulates
//               the K + 4 sums ylogLike / the refit need from it: proposal . live_j, proposal . y, |proposal|^2,
//               sum, max|.|  (codes/funcs.py:1147-1162).  No column ever goes to HBM.
//               a proposal whose fp32 column is not finite on the rows of a tile is interpreted there once more by its warp, with the
//               out-of-range 4-row vectors in double range (the value rule above live_tile)
//   k_wdedup    one 64-thread block per chain: which slots repeat a tree of this window or of the chain's earlier windows in the ring
//   k_wresolve  one or two warps per chain, one lane per proposal: rank test, ridge SSE, logR, accept draw in parallel, then
//               the in-order consumption, the accept bookkeeping and the stop rules  (codes/funcs.py:1226-1306,
//               codes/bsr_class.py:174-252)
#pragma once
#include "bsr_common.cuh"
#include "bsr_eval.cuh"
#include "bsr_propose.cuh"
#include "bsr_rng.cuh"
#include "bsr_solve.cuh"

#define BSR_MAX_PEERS 8
#ifndef BSR_WIDE_INLINE
#define BSR_WIDE_INLINE __forceinline__
#endif

#ifndef BSR_WEVAL_NV
#define BSR_WEVAL_NV 4   // row vectors (of 4 fp32 rows) per thread and token decode in k_weval (1: 599, 2 at 4 blocks/SM: 599,
                         // 3: 558, 4: 520, 8 at 2 blocks/SM: 617 us per 64-slot window at C2; level 0 of the operand
                         // stack in shared memory instead of local memory: 543)
#endif

struct WinCtx {
  long long p_target;      // chains stop consuming at this proposal index
  int c0, cn;              // chain range of this launch
  int* bucket;             // [BSR_N_BINS][bucket_stride] window slots (ci * W + i) of this launch sorted by bin
  int* bucket_count;       // [BSR_N_BINS]
  int bucket_stride;
  // draw recording (MODE 2) and trace rows, both indexed by proposal index - origin
  double* rec_draws; int* rec_count; int rec_steps, rec_cap; long long rec_origin;
  double* trace; int trace_steps; long long trace_origin;
  // value-level tape (MODE 1, reference fixtures): proposal p reads tape[tape_off[c * trace_steps + ti] .. tape_off[.. + 1]) with
  // ti = p - trace_origin (the tape and the trace rows share their indexing); nullptr: Philox
  const double* tape; const int64_t* tape_off;
  // proposed trees of the consumed proposals, by trace row (tests: bit-exact comparison with the reference's proposals)
  uint32_t* log_tok; double* log_pa; double* log_pb; int* log_nn;
  // data: D data sets of the same shape, X [D][d][ld], y [D][ld]; chain c reads data set st.ds[c], whose X starts at
  // ds * ds_stride (folded into the leaf offsets by stage_tokens) and whose y at ds * ld
  const float* X32; const double* X64; const double* y64;
  uint32_t n, ld, ds_stride;
  int precision;
  uint32_t rows_per_split;   // multiple of 4
  uint32_t TR;               // rows per shared-memory tile, multiple of 4
  int checked_m;             // node count from which k_weval's first pass tells finite from out-of-range vectors itself (K > 5 kernels)
  int dedup;                 // 0: every slot is interpreted; 1: repeated trees of a window once; 2: and trees of the chain's earlier windows (ring) not at all
  // resolve
  double n_total, n_local, sum_y, yy, pivot_tol;   // sum_y, yy: data set 0 (the kernels of one data set take them by value)
  const double* ystats;      // [D][2] sum(y), y'y of every data set
  // row-sharded handles: the records / out-of-range masks of this window on every rank (peer memory over NVLink,
  // index = rank); n_peers == 0: single device, ws.rec / ws.bad
  int n_peers;
  const double* peer_rec[BSR_MAX_PEERS];
  const unsigned long long* peer_bad[BSR_MAX_PEERS];
  // refit after (re)initialisation (k_wlive_bad, k_wlive_gram, k_wrefit): partial Grams of the live columns per split and rank
  const double* peer_lrec[BSR_MAX_PEERS];
  const int* abort_flag;     // set by k_wwait when a peer never signalled: the window is not resolved
  // rows of every data set ([D]; n is the largest, and the geometry is that of n), nullptr on a handle of one data set (its n rows, n_total
  // of them over all ranks).  Last member: the kernels of one data set address the members above exactly as they did without it.
  const uint32_t* ds_n;
};

// ---------------------------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------------------------
static __global__ void k_wprep(WinState ws, int C, long long p_start) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) ws.pos[c] = p_start;     // (the out-of-range masks are reset per window by k_wclassify; those of the earlier windows in the ring stay: record cache)
}
static __global__ void k_wcount(ChainState st, WinState ws, long long p_target, int* out) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  int v = (c < st.C && !st.done[c] && ws.pos[c] < p_target) ? 1 : 0;
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, v);
}

// Row-sharded windows: every rank evaluates its own rows, then k_wresolve on every rank sums the partial records of all
// ranks straight out of their memory (peer loads over NVLink, fixed rank order => identical decisions everywhere).
// The hand-over is one flag per (reader, writer) pair: after its evaluation kernels rank r stores the window's ticket
// into slot r of every peer's flag array (k_wsignal); k_wwait spins until all slots of the local array carry it.
struct PeerFlagPtrs { unsigned long long* p[BSR_MAX_PEERS]; };
static __global__ void k_wsignal(PeerFlagPtrs pf, int n_peers, int rank, unsigned long long ticket) {
  if ((int)threadIdx.x < n_peers) {
    __threadfence_system();
    volatile unsigned long long* f = pf.p[threadIdx.x] + rank;
    *f = ticket;
  }
}
// timeout_ns: measured on %globaltimer (nanoseconds of wall clock, independent of clocks and scheduling); on expiry the kernel
// records which rank was missing in *abort_flag and returns -- k_wresolve then leaves the window untouched and bsr_run reports
// the failure to its caller (no trap: the CUDA context stays usable, the caller can tear the group down in order).
static __global__ void k_wwait(const unsigned long long* flags, int n_peers, unsigned long long ticket, unsigned long long timeout_ns,
                               int* abort_flag) {
  if ((int)threadIdx.x < n_peers) {
    const volatile unsigned long long* f = flags + threadIdx.x;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while (*f < ticket) {
      __nanosleep(200);
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
      if (timeout_ns != 0ull && t1 - t0 > timeout_ns) { atomicCAS(abort_flag, 0, 1 + (int)threadIdx.x); break; }
      if (*reinterpret_cast<volatile int*>(abort_flag) != 0) break;
    }
  }
  __syncthreads();
  __threadfence_system();
}

// A tree, for the duplicate search, is its node count, (opcode, feature of a leaf) per token and the lt parameters as bit
// patterns; op_ind does not enter the evaluation.
__device__ __forceinline__ uint32_t dedup_key(uint32_t tk) { return tok_op(tk) == OP_LEAF ? (tk & 0xffff00ffu) : (tk & 0xffu); }
__device__ __forceinline__ unsigned long long dedup_mix(unsigned long long h, unsigned long long v) {
  h = (h ^ v) * 0xff51afd7ed558ccdull;
  return h ^ (h >> 32);
}
// Hash of a proposed tree: node count, (opcode, feature of a leaf) per token, lt parameters as bit patterns.  Never 0.
__device__ __noinline__ unsigned long long dedup_hash(const uint32_t* tok, const double* pa, const double* pb, int m) {
  unsigned long long h = dedup_mix(0x9e3779b97f4a7c15ull, (unsigned long long)m);
#pragma unroll 1
  for (int t = 0; t < m; ++t) {
    const uint32_t k = dedup_key(tok[t]);
    h = dedup_mix(h, k);
    if (k == (uint32_t)OP_LT) {
      h = dedup_mix(h, (unsigned long long)__double_as_longlong(pa[t]));
      h = dedup_mix(h, (unsigned long long)__double_as_longlong(pb[t]));
    }
  }
  return h | 1ull;
}

// ---------------------------------------------------------------------------------------------------------------
// proposals
// ---------------------------------------------------------------------------------------------------------------
// Pre-pass: the move each window slot is going to make (its first draw against the thresholds of the live tree), and
// a counting sort of the slots by (move, tree size class).  k_wpropose then runs homogeneous warps: Prop is seven
// different splice routines whose loops run over the tree, and a warp that mixes them executes all seven one after the
// other, each for as long as its largest tree takes.
static __global__ void k_wclassify(ChainState st, WinState ws, WinCtx wc) {
  const int gi = blockIdx.x * blockDim.x + threadIdx.x;
  const int W = ws.W;
  int mv = -1;
  int ci = 0, i = 0;
  if (gi < wc.cn * W) {
    ci = gi / W; i = gi % W;
    const int c = wc.c0 + ci;
    const long long p0 = ws.pos[c];
    if (!st.done[c] && p0 < wc.p_target) {
      const WinState wv = win_half(ws, win_parity(ws, c), st.K);
      if (i == 0) { wv.bad[c] = 0ull; if (ws.lcol_wide != nullptr) ws.lcol_wide[c] = 0u; }
      const long long p = p0 + i;
      if (p >= wc.p_target) { wv.info[(size_t)c * W + i].flags = PF_SKIP; wv.hash[(size_t)c * W + i] = 0ull; }
      else {
        const int K = st.K;
        const int g = c * K + (int)(p % K);
        // node / lt / terminal / detransform-candidate counts of the live tree: kept per tree by the refit and by every accept
        const int cnt = st.lcnt[g];
        const int m = cnt & 0xff, L = (cnt >> 8) & 0xff, T = (cnt >> 16) & 0xff, D = (cnt >> 24) & 0xff;
        const int Nt = m - T;
        double test;
        if (wc.tape != nullptr) {          // the proposal's first tape value is Prop's `test` draw (funcs.py:483)
          const long long ti = p - wc.trace_origin;
          test = 0.5;
          if (ti >= 0 && ti < wc.trace_steps) {
            const int64_t lo = wc.tape_off[(size_t)c * wc.trace_steps + ti], hi = wc.tape_off[(size_t)c * wc.trace_steps + ti + 1];
            if (lo < hi) test = wc.tape[lo];
          }
        } else {
          Draws<0> dr;
          dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)p, 1u);
          test = dr.u01();
        }
        mv = select_move(L, Nt, D, test) * BSR_N_SIZE_CLASSES + (BSR_N_SIZE_CLASSES == 4 ? (m <= 4 ? 0 : (m <= 8 ? 1 : (m <= 16 ? 2 : 3))) : (BSR_N_SIZE_CLASSES == 2 ? (L > 0 ? 1 : 0) : 0));
      }
    }
  }
  // append to the move's bucket: counted per block in shared memory, one global atomic per (block, move) -- seven counters
  // hit by every warp of the grid serialise in L2
  __shared__ int s_cnt[BSR_N_BINS], s_base[BSR_N_BINS];
  if (threadIdx.x < BSR_N_BINS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int my_off = 0;
#pragma unroll
  for (int q = 0; q < BSR_N_BINS; ++q) {
    const unsigned msk = __ballot_sync(FULL, mv == q);
    if (msk == 0u) continue;
    int base = 0;
    if (lane == __ffs(msk) - 1) base = atomicAdd(&s_cnt[q], __popc(msk));
    base = __shfl_sync(FULL, base, __ffs(msk) - 1);
    if (mv == q) my_off = base + __popc(msk & ((1u << lane) - 1u));
  }
  __syncthreads();
  if (threadIdx.x < BSR_N_BINS && s_cnt[threadIdx.x] > 0) s_base[threadIdx.x] = atomicAdd(wc.bucket_count + threadIdx.x, s_cnt[threadIdx.x]);
  __syncthreads();
  if (mv >= 0) wc.bucket[(size_t)mv * wc.bucket_stride + s_base[mv] + my_off] = ci * W + i;
}

#ifndef BSR_WPROP_MINB
#define BSR_WPROP_MINB 16   // 64 registers, 32 resident warps per SM (8 -> 12 -> 16: 276 -> 258 -> 246 us per window once the
                          // kernel was no longer instruction-cache bound)
#endif
template <int MODE>
__global__ void __launch_bounds__(64, BSR_WPROP_MINB) k_wpropose(ChainState st, WinState ws, const PriorTables* __restrict__ ptp, WinCtx wc,
                                                                const int* __restrict__ chain_pt) {
  // block -> (move, first slot of the move's bucket): the buckets are laid end to end in units of blocks, so the grid holds the
  // blocks that have work plus at most one partly filled block per move (a grid of moves x all slots launched six empty blocks
  // for every working one)
  int mv = 0, e = 0;
  {
    int b = blockIdx.x;
    bool found = false;
#pragma unroll
    for (int q = 0; q < BSR_N_BINS; ++q) {
      const int nb = (wc.bucket_count[q] + (int)blockDim.x - 1) / (int)blockDim.x;
      if (!found) { if (b < nb) { mv = q; found = true; } else b -= nb; }
    }
    if (!found) return;
    e = b * blockDim.x + threadIdx.x;
    if (e >= wc.bucket_count[mv]) return;
  }
  const int W = ws.W;
  const int gi = wc.bucket[(size_t)mv * wc.bucket_stride + e];
  const int c = wc.c0 + gi / W, i = gi % W;
  const size_t wi = (size_t)c * W + i;
  const long long p = ws.pos[c] + i;
  const int K = st.K;
  const int k = (int)(p % K);
  const int g = c * K + k;
  Draws<MODE> dr;
  dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)p, 1u);
  const long long ri = p - wc.rec_origin;
  const bool recording = MODE == 2 && wc.rec_draws != nullptr && ri >= 0 && ri < wc.rec_steps;
  if (recording) dr.init_record(wc.rec_draws + ((size_t)c * wc.rec_steps + ri) * wc.rec_cap, wc.rec_cap);
  if (MODE == 1) {
    // a slot behind an accept is proposed from a stale state and may run its (then foreign) tape segment dry or out of
    // range: Draws flags the desync, the slot is discarded and proposed again by the next window
    const long long ti = p - wc.trace_origin;
    if (ti >= 0 && ti < wc.trace_steps)
      dr.init_tape(wc.tape, (int)wc.tape_off[(size_t)c * wc.trace_steps + ti], (int)wc.tape_off[(size_t)c * wc.trace_steps + ti + 1]);
    else dr.init_tape(wc.tape, 0, 0);
  }
  const int w = st.which[g];
  const size_t slot = (size_t)g * BSR_MAXN, wslot = wi * BSR_MAXN;
  PropInfo info;
  const WinState wv = win_half(ws, win_parity(ws, c), K);
  propose_one<MODE>(ptp[chain_pt[c]], st.tok[w] + slot, st.pa[w] + slot, st.pb[w] + slot, st.nn[w][g], st.sa[g], st.sb[g], dr,
                    wv.tok + wslot, wv.pa + wslot, wv.pb + wslot, wv.nn + wi, info, st.lfs + 2 * (size_t)g);
  wv.info[wi] = info;
  // what the duplicate search (k_wdedup) compares: computed here, where the tree was just written (L1 / L2 hot)
  wv.hash[wi] = (info.flags & PF_CAPACITY) ? 0ull : dedup_hash(wv.tok + wslot, wv.pa + wslot, wv.pb + wslot, wv.nn[wi]);
  if (recording) wc.rec_count[(size_t)c * wc.rec_steps + ri] = dr.pos;
}

// ---------------------------------------------------------------------------------------------------------------
// evaluation
// ---------------------------------------------------------------------------------------------------------------
// Shared-memory layout of the evaluation kernels (T = evaluation type of in-range columns):
//   double2 live[TV][LS]            the K live columns and y on the rows of the current tile, as fp64, vector-major: row
//                                   vector q (R rows) owns LS = ((K+1) * R/2) | 1 double2 slots, slot j * R/2 + pl =
//                                   rows 2 pl, 2 pl + 1 of column j (column K = y).  The odd stride keeps the 16-byte
//                                   accesses of a quarter warp on distinct banks, and every slot of a vector is a
//                                   compile-time offset from one base address
//   double  acc[W][K+4]             running sums of every proposal over the tiles done so far
//   EvTok<T> ltok[K][MAXN], EvTok<T> ptok[NW][MAXN], int lm[K], the block's masks (out-of-range / non-finite proposals), work counter
struct WinSmem {
  size_t live, acc, ltok, ptok, lm, dd, bm, total;
};
template <typename T>
__host__ __device__ constexpr int win_live_stride(int K) { return ((K + 1) * (RowVec<T>::R / 2)) | 1; }
// multi: k_weval of several data sets, which keeps the chain's row count beside its data set (one int more; the geometry is
// chosen without it, see win_geometry)
template <typename T>
__host__ __device__ inline WinSmem win_smem_layout(int K, int W, int NW, uint32_t TR, bool multi = false) {
  WinSmem s;
  size_t o = 0;
  s.live = o; o += (size_t)(TR / RowVec<T>::R) * win_live_stride<T>(K) * sizeof(double2);
  s.acc = o; o += (size_t)W * (K + 4) * sizeof(double);
  o = (o + 15) / 16 * 16;
  s.ltok = o; o += (size_t)K * BSR_MAXN * sizeof(EvTok<T>);
  s.ptok = o; o += (size_t)NW * BSR_MAXN * sizeof(EvTok<T>);
  o = (o + 15) / 16 * 16;
  s.lm = o; o += (size_t)(K + (K & 1) + 8 + (multi ? 1 : 0)) * sizeof(int);   // + three 64-bit slot masks (second pass needed / its vectors already known / column not finite), + the work counter, + the data set (+ its rows)
  o = (o + 15) / 16 * 16;
  s.dd = o; o += 320;                                                   // results of the duplicate search (sizeof(DedupSmem))
  s.bm = o; if (sizeof(T) == 4 && K > 5) o += (size_t)W * 8 * sizeof(unsigned);   // per slot: which of the tile's <= 256 vectors are out of range (large trees, see k_weval)
  s.total = (o + 15) / 16 * 16;
  return s;
}

// xbase: offset of the chain's data set in X (ds * d * ld): the interpreters reach X through the leaf offsets alone
template <typename T>
__device__ __forceinline__ void stage_tokens(const uint32_t* tok, const double* pa, const double* pb, int m, uint32_t xbase, uint32_t ld,
                                             EvTok<T>* dst, int t0, int step) {
  for (int t = t0; t < m; t += step) {
    const uint32_t tk = tok[t];
    EvTok<T> e;
    e.op = tok_op(tk); e.off = xbase + (uint32_t)tok_ft(tk) * ld;
    e.a = (T)0; e.b = (T)0;
    if (e.op == OP_LT) { e.a = (T)pa[t]; e.b = (T)pb[t]; }      // one operator in ten: the other tokens cost one load, not three
    dst[t] = e;
  }
}

// The value rule of the fp32 evaluation mode.  A column is interpreted in fp32 (SFU transcendentals) in vectors of four
// consecutive rows (row index a multiple of 4); a vector with a non-finite fp32 value (overflow: exp beyond 88.7, powers
// of large values, and whatever inf turns into downstream) is interpreted again in double RANGE (OpMathWide: fp64 range and
// exact fp64 + * lt neg square cubic inv, fp32-accurate exp / sin / cos).  The rule is per vector, so the values of a column
// do not depend on row tiles, row splits, the rank that owns the rows, or on whether the tree is live or proposed: the Gram
// cache of the live columns (written from the accepted proposal's record) and the live values staged below stay consistent.
__device__ __forceinline__ bool vec_finite(const float (&v)[4]) {
  // 0 * v is NaN for v = inf / NaN and 0 otherwise (FMA pipe, the least loaded one)
  float c = v[0] * 0.0f;
  c = fmaf(v[1], 0.0f, c); c = fmaf(v[2], 0.0f, c); c = fmaf(v[3], 0.0f, c);
  return c == 0.0f;
}
// Double-range interpretation of two rows (element row0 of every column), from the tokens as staged for the fp32
// interpreter (opcode, column offset) and the lt parameters where they live in global memory (exact doubles).  Out of line:
// the path is rare (1 - 3 % of the proposals, and only their out-of-range vectors) and must not cost the fp32 loop registers.
static __device__ BSR_WIDE_INLINE double2 eval_tree_wide2(const EvTok<float>* tk, const double* __restrict__ pa, const double* __restrict__ pb, int m,
                                                       const double* __restrict__ X64, uint32_t row0) {
  double stk[BSR_STACK][2];
  double a0 = 0.0, a1 = 0.0;
  int sp = 0;
#pragma unroll 1
  for (int i = m - 1; i >= 0; --i) {
    const int o = tk[i].op;
    if (o == OP_LEAF) {
      if (i != m - 1) { stk[sp][0] = a0; stk[sp][1] = a1; ++sp; }
      const double2 x = __ldg(reinterpret_cast<const double2*>(X64 + (size_t)tk[i].off + row0));
      a0 = x.x; a1 = x.y;
    } else if (o >= OP_ADD) {
      --sp;
      if (o == OP_ADD) { a0 += stk[sp][0]; a1 += stk[sp][1]; }
      else { a0 *= stk[sp][0]; a1 *= stk[sp][1]; }
    } else {
      switch (o) {
        case OP_LT: { const double ca = pa[i], cb = pb[i]; a0 = ca * a0 + cb; a1 = ca * a1 + cb; } break;
        case OP_INV: a0 = OpMathWide::inv_guard(a0); a1 = OpMathWide::inv_guard(a1); break;
        case OP_NEG: a0 = -a0; a1 = -a1; break;
        case OP_SIN: a0 = OpMathWide::sin_(a0); a1 = OpMathWide::sin_(a1); break;
        case OP_COS: a0 = OpMathWide::cos_(a0); a1 = OpMathWide::cos_(a1); break;
        case OP_EXP: a0 = OpMathWide::exp_guard(a0); a1 = OpMathWide::exp_guard(a1); break;
        case OP_SQUARE: a0 = a0 * a0; a1 = a1 * a1; break;
        default: a0 = a0 * a0 * a0; a1 = a1 * a1 * a1; break;   // OP_CUBIC
      }
    }
  }
  return make_double2(a0, a1);
}

// The K live columns and y on rows [row_lo, row_lo + tile_rows) -> shared memory (fp64).  Block-cooperative; the
// caller synchronises before and after.  Rows >= n are written as zeros.  ds, n: the chain's data set (its y; the live tokens
// were staged with its X offset) and its row count.
// lcol (fp32 mode, k_weval only; nullptr otherwise): the cache of live columns (WinState::lcol ...).  A column whose flag is set is
// loaded instead of interpreted -- the same fp32 values; an interpreted one is written to the cache, k_wresolve sets its flag when the
// window is over (unless the tree was replaced or the column had an out-of-range vector: *wide_mask).
template <typename T>
__device__ __forceinline__ void live_tile(const ChainState& st, const WinCtx& wc, int c, int K, uint32_t ds, uint32_t n, const EvTok<T>* s_ltok, const int* s_lm,
                                          uint32_t row_lo, uint32_t tile_rows, double2* s_live, float* lcol = nullptr, long long lcol_ld = 0,
                                          const unsigned char* lcol_ok = nullptr, unsigned* wide_mask = nullptr) {
  constexpr int R = RowVec<T>::R, NP = R / 2;
  const int LS = win_live_stride<T>(K);
  const T* X = (sizeof(T) == 4) ? reinterpret_cast<const T*>(wc.X32) : reinterpret_cast<const T*>(wc.X64);
  const uint32_t tv = (tile_rows + R - 1) / R;
  for (int j = 0; j < K; ++j) {
    float* ccol = (sizeof(T) == 4 && lcol != nullptr) ? lcol + (size_t)(c * K + j) * (size_t)lcol_ld : nullptr;
    const bool cached = ccol != nullptr && lcol_ok[c * K + j] != 0;
    for (uint32_t q = threadIdx.x; q < tv; q += blockDim.x) {
      T v[R];
      if (cached) {
        const float4 f = *reinterpret_cast<const float4*>(ccol + row_lo + q * 4);
        const float fv[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = (T)fv[r < 4 ? r : 0];
      } else {
        eval_tree_rows<T, R>(s_ltok + j * BSR_MAXN, s_lm[j], X, row_lo + q * R, v);
        if (ccol != nullptr) *reinterpret_cast<float4*>(ccol + row_lo + q * 4) = make_float4((float)v[0], (float)v[1], (float)v[R > 2 ? 2 : 0], (float)v[R > 3 ? 3 : 0]);
      }
      double d[R];
#pragma unroll
      for (int r = 0; r < R; ++r) d[r] = (double)v[r];
      if (sizeof(T) == 4 && !cached) {
        float vf[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) vf[r] = (float)v[r < R ? r : 0];
        if (!vec_finite(vf)) {                     // this vector in double range (the value rule above)
          const int g = c * K + j;
          const int w = st.which[g];
          const size_t slot = (size_t)g * BSR_MAXN;
          if (wide_mask != nullptr) atomicOr(wide_mask + c, 1u << j);
#pragma unroll
          for (int pl = 0; pl < NP; ++pl) {
            const double2 x = eval_tree_wide2(reinterpret_cast<const EvTok<float>*>(s_ltok) + j * BSR_MAXN, st.pa[w] + slot, st.pb[w] + slot, s_lm[j],
                                              wc.X64, row_lo + q * R + 2 * pl);
            d[2 * pl] = x.x; d[2 * pl + 1] = x.y;
          }
        }
      }
#pragma unroll
      for (int pl = 0; pl < NP; ++pl) {
        const uint32_t r0 = row_lo + q * R + 2 * pl;
        double2 o;
        o.x = (r0 < n) ? d[2 * pl] : 0.0;
        o.y = (r0 + 1 < n) ? d[2 * pl + 1] : 0.0;
        s_live[q * LS + j * NP + pl] = o;
      }
    }
  }
  // every double2 slot of every vector is written (zeros on padding rows): the consumers multiply padded rows by a zero
  // proposal value, and 0 * (stale NaN bits) would be NaN
  const uint32_t tv2 = tv * NP;
  for (uint32_t q2 = threadIdx.x; q2 < tv2; q2 += blockDim.x) {
    const uint32_t r0 = row_lo + q2 * 2;
    const double2 yv = *reinterpret_cast<const double2*>(wc.y64 + (size_t)ds * wc.ld + r0);
    double2 d;
    d.x = (r0 < n) ? yv.x : 0.0;
    d.y = (r0 + 1 < n) ? yv.y : 0.0;
    s_live[(NP == 2 ? (q2 >> 1) : q2) * LS + K * NP + (NP == 2 ? (q2 & 1) : 0)] = d;
  }
}

// Duplicate proposals of a window.  All W proposals start from the same live state, and many moves land on the same tree
// (reassignFeature / reassignOperator drawing what is already there, grow staying a leaf, the same prune twice ...):
// at C2 a third of a window's proposals repeat an earlier one.  The record of a proposal (its sums against the live
// columns and y) depends on the tree alone, so a repeated tree is interpreted once and its record is shared -- the
// same bits the repeated interpretation would have produced.  A tree is its node count, (opcode, feature of a leaf)
// per token and the lt parameters as bit patterns; op_ind does not enter the evaluation.
// Exact comparison of two window slots with the same node count m (four tokens per load; lt parameters as bit patterns).
// The slots may lie in different ring entries of the slot arrays: (tok, pa, pb) A / B are the bases of the two slots.
__device__ __noinline__ bool dedup_same(const uint32_t* tokA, const double* paA, const double* pbA, const uint32_t* tokB, const double* paB,
                                        const double* pbB, int m) {
  for (int t0 = 0; t0 < m; t0 += 4) {
    const uint4 qa = *reinterpret_cast<const uint4*>(tokA + t0);
    const uint4 qb = *reinterpret_cast<const uint4*>(tokB + t0);
    const uint32_t ta[4] = {qa.x, qa.y, qa.z, qa.w}, tb[4] = {qb.x, qb.y, qb.z, qb.w};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + u;
      if (t < m) {
        const uint32_t ka = dedup_key(ta[u]);
        if (ka != dedup_key(tb[u])) return false;
        if (ka == (uint32_t)OP_LT) {
          if (__double_as_longlong(paA[t]) != __double_as_longlong(paB[t])) return false;
          if (__double_as_longlong(pbA[t]) != __double_as_longlong(pbB[t])) return false;
        }
      }
    }
  }
  return true;
}

// Duplicate search of a window, one 64-thread block per chain, thread i = slot i.  All W proposals start from one live state, so
// many are the same tree; and as long as the chain accepts nothing its earlier windows (up to R - 1 in the ring) were proposed from that state too.
// A record (the sums of a proposal against the live columns and y) depends on the tree and the live state alone, so
//   rep[i]      first slot i' <= i of this window with the same tree: slot i shares the record of i'
//   rep[i] | 80 the tree is not in this window before i but in an earlier window of the ring, prevslot[i] = slot | (windows back - 1) << 6: the record
//               is copied from there, nothing is interpreted
//   order[]     the neval slots that are left to interpret, largest tree first (the warps of a k_weval block take them from a
//               shared counter and end on the small ones, waiting less for each other)
// Hashes come from k_wpropose (0: slot skipped or over capacity); a hash match is confirmed token by token.  dedup: 0 every
// slot is interpreted, 1 duplicates within the window only, 2 also the earlier windows of the ring.  A kernel of its own because the search
// is a chain of dependent latencies on 64 threads: inside k_weval it held up 256 threads of 80 registers behind five barriers.
#define BSR_DD_TAB (2 * BSR_MAXW * BSR_WIN_RING)     // open-addressing table of the duplicate search (a power of two): <= 64 * BSR_WIN_RING keys
__device__ __forceinline__ int dd_probe(unsigned long long* key, unsigned long long h, bool insert) {
  int idx = (int)(h >> 17) & (BSR_DD_TAB - 1);
  for (;;) {
    const unsigned long long old = insert ? atomicCAS(&key[idx], 0ull, h) : key[idx];
    if (old == h || (insert && old == 0ull)) return idx;
    if (!insert && old == 0ull) return -1;
    idx = (idx + 1) & (BSR_DD_TAB - 1);
  }
}
static __global__ void __launch_bounds__(BSR_MAXW) k_wdedup(ChainState st, WinState ws, WinCtx wc) {
  __shared__ unsigned long long s_key[BSR_DD_TAB];
  __shared__ int s_in[BSR_DD_TAB], s_pv[BSR_DD_TAB];     // per key: first slot of this window, most recent (window, slot) before it
  __shared__ int s_hist[BSR_MAXN + 2];
  const int c = wc.c0 + blockIdx.x;
  if (st.done[c] || ws.pos[c] >= wc.p_target) return;
  const int K = st.K, W = ws.W, i = threadIdx.x;
  const int head = ws.chead[c];
  const int nprev = (head >= 0 && wc.dedup >= 2) ? (int)ws.cvalid[c] : 0;       // earlier windows proposed from this very live state
  const WinState wv = win_half(ws, head >= 0 ? ((head + 1) % ws.R) : 0, K);
  const size_t wi = (size_t)c * W + (i < W ? i : 0);
  unsigned long long h = 0ull, ph[BSR_WIN_RING - 1];
  int m = 0;
  bool ev = false;
  if (i < W) {
    h = wv.hash[wi];
    ev = h != 0ull;
    m = ev ? wv.nn[wi] : 0;
  }
#pragma unroll
  for (int d = 0; d < BSR_WIN_RING - 1; ++d)
    ph[d] = (i < W && d < nprev) ? win_half(ws, (head - d + ws.R) % ws.R, K).hash[wi] : 0ull;
  for (int e = i; e < BSR_DD_TAB; e += BSR_MAXW) { s_key[e] = 0ull; s_in[e] = 0x7fffffff; s_pv[e] = 0x7fffffff; }
  for (int e = i; e < BSR_MAXN + 2; e += BSR_MAXW) s_hist[e] = 0;
  __syncthreads();
  if (wc.dedup != 0) {
    if (ev) atomicMin(&s_in[dd_probe(s_key, h, true)], i);
#pragma unroll
    for (int d = 0; d < BSR_WIN_RING - 1; ++d)
      if (ph[d] != 0ull) atomicMin(&s_pv[dd_probe(s_key, ph[d], true)], d * BSR_MAXW + i);       // smallest = most recent window
  }
  __syncthreads();
  int rep = i, prev = 0;
  if (ev && wc.dedup != 0) {
    const uint32_t* tk = wv.tok + wi * BSR_MAXN; const double* ta = wv.pa + wi * BSR_MAXN; const double* tb = wv.pb + wi * BSR_MAXN;
    const int t = dd_probe(s_key, h, false);
    const int k = s_in[t];                               // first slot of this window with the hash (a hash that matches a
    if (k < i) {                                         // different tree: treated as no duplicate)
      const size_t wk = (size_t)c * W + k;
      if (wv.nn[wk] == m && dedup_same(wv.tok + wk * BSR_MAXN, wv.pa + wk * BSR_MAXN, wv.pb + wk * BSR_MAXN, tk, ta, tb, m)) rep = k;
    } else if (s_pv[t] != 0x7fffffff) {
      const int d = s_pv[t] / BSR_MAXW, kk = s_pv[t] % BSR_MAXW;
      const WinState pv = win_half(ws, (head - d + ws.R) % ws.R, K);
      const size_t pk = (size_t)c * W + kk;
      if (pv.nn[pk] == m && dedup_same(pv.tok + pk * BSR_MAXN, pv.pa + pk * BSR_MAXN, pv.pb + pk * BSR_MAXN, tk, ta, tb, m)) {
        rep = i | 0x80; prev = kk | (d << 6);
      }
    }
  }
  const int cost = (ev && rep == i) ? m : 0;       // 1 .. BSR_MAXN for a slot that is interpreted
  if (cost > 0) atomicAdd(&s_hist[cost], 1);
  const int E = __syncthreads_count(cost > 0);
  // order: largest tree first (counting sort by node count; slots of one size in arrival order -- the records do not depend on it)
  if (i == 0) {
    int run = 0;
    for (int q = BSR_MAXN; q >= 1; --q) { const int n = s_hist[q]; s_hist[q] = run; run += n; }
    ws.neval[c] = E;
  }
  __syncthreads();
  if (i < W) {
    ws.rep[wi] = (unsigned char)rep;
    ws.prevslot[wi] = (unsigned short)prev;
    if (cost > 0) ws.order[(size_t)c * W + atomicAdd(&s_hist[cost], 1)] = (unsigned char)i;
  }
}

// What k_weval keeps of the duplicate search in shared memory.
struct DedupSmem {
  unsigned short prev[BSR_MAXW];
  unsigned char rep[BSR_MAXW], order[BSR_MAXW], m[BSR_MAXW];   // m: node count, 0 for a slot that is skipped / over capacity
};
static_assert(sizeof(DedupSmem) == 320 && BSR_MAXW == 64, "win_smem_layout reserves sizeof(DedupSmem) bytes");
static_assert((BSR_DD_TAB & (BSR_DD_TAB - 1)) == 0 && BSR_WIN_RING <= 16, "table size must be a power of two; prevslot holds 4 bits of window distance");

// K + 4 running sums of one proposal column p against the live columns l_j and y.
template <int KC>
struct WAcc {
  double l[KC];      // p . l_j
  double y, pp, s;   // p . y, p . p, sum p
  double mx;         // max |p| over the values accumulated as doubles (fp64 mode, double-range vectors) ...
  float mxf;         // ... and over the fp32 values (one FMNMX per pair instead of a conversion and a 64-bit compare / select per vector)
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int j = 0; j < KC; ++j) l[j] = 0.0;
    y = pp = s = 0.0; mx = 0.0; mxf = 0.0f;
  }
  __device__ __forceinline__ void warp_reduce() {
#pragma unroll
    for (int j = 0; j < KC; ++j) l[j] = warp_sum(l[j]);
    y = warp_sum(y); pp = warp_sum(pp); s = warp_sum(s);
    const double m32 = (double)warp_max<float>(mxf);
    mx = warp_max<double>(mx);
    mx = mx > m32 ? mx : m32;
  }
  // The same sums with a third of the shuffles: a reduce-scatter.  The KC + 3 sums (padded to VP = 8 or 16) are halved over the
  // lanes round by round -- in the round with lane offset 16 the lower half-warp keeps the first VP / 2 sums and hands the others
  // to its partner, and so on -- until every lane holds one sum, which the remaining rounds finish.  Afterwards sum j (0 .. KC - 1:
  // p . l_j, KC: p . y, KC + 1: p . p, KC + 2: sum p) is complete in `l[0]` of the lanes owner(j) .. owner(j) + (32 / VP) - 1;
  // mx is complete in every lane.  (A warp_sum per value costs 5 x (2 SHFL + DADD) each: 9 % of k_weval's instructions at C2.)
  static constexpr int VP = (KC + 3 <= 8) ? 8 : ((KC + 3 <= 16) ? 16 : 32);
  static __device__ __forceinline__ int owner(int j) {
    return VP == 8 ? (((j >> 2) & 1) << 4 | ((j >> 1) & 1) << 3 | (j & 1) << 2)
                   : (VP == 16 ? (((j >> 3) & 1) << 4 | ((j >> 2) & 1) << 3 | ((j >> 1) & 1) << 2 | (j & 1) << 1) : j);
  }
  template <bool EX, bool MX_F32>
  __device__ __forceinline__ void warp_reduce_scatter_or_all(int lane) {
    if (EX) warp_reduce_scatter<MX_F32>(lane); else warp_reduce();
  }
  template <bool MX_F32>
  __device__ __forceinline__ void warp_reduce_scatter(int lane) {
    double v[VP];
#pragma unroll
    for (int j = 0; j < VP; ++j) v[j] = (j < KC) ? l[j] : (j == KC ? y : (j == KC + 1 ? pp : (j == KC + 2 ? s : 0.0)));
    int off = 16;
#pragma unroll
    for (int n = VP; n > 1; n >>= 1, off >>= 1) {
      const bool up = (lane & off) != 0;
#pragma unroll
      for (int k = 0; k < n / 2; ++k) {
        const double send = up ? v[k] : v[k + n / 2];
        const double keep = up ? v[k + n / 2] : v[k];
        v[k] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
#pragma unroll
    for (; off > 0; off >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
    l[0] = v[0];
    if (MX_F32) mx = (double)warp_max<float>(mxf);           // (the fp32 loop of k_weval accumulates fp32 values only)
    else mx = warp_max<double>(mx);
  }
};

// Accumulate one row vector of proposal values v (R rows of type T) against the live slots of the same rows.
// lv: first live slot of the vector (s_live + q * LS [+ plane offset]); LNP: planes per column in the layout (R/2 of
// the type the tile was laid out for).  TAIL: the vector may reach beyond row n (padding rows count as zeros).
template <typename T, int KC, int LNP, bool TAIL>
__device__ __forceinline__ void wacc_rows(WAcc<KC>& a, int K, const T* v, const double2* lv, uint32_t row0, uint32_t n) {
  constexpr int R = RowVec<T>::R, NP = R / 2;
  T av = (T)0;
#pragma unroll
  for (int pl = 0; pl < NP; ++pl) {
    double p0 = (double)v[2 * pl], p1 = (double)v[2 * pl + 1];
    T a0 = fabs(v[2 * pl]), a1 = fabs(v[2 * pl + 1]);
    if (TAIL) {                               // ragged tail: rows >= n are padding
      if (row0 + 2 * pl >= n) { p0 = 0.0; a0 = (T)0; }
      if (row0 + 2 * pl + 1 >= n) { p1 = 0.0; a1 = (T)0; }
    }
    // fmax drops a NaN operand: non-finite columns are recognised by their |p|^2 (NaN / inf), an inf survives here
    av = fmax(av, fmax(a0, a1));
    a.pp = fma(p0, p0, a.pp); a.pp = fma(p1, p1, a.pp);
    a.s += p0; a.s += p1;
#pragma unroll
    for (int j = 0; j < KC; ++j) {
      if (j < K) {
        const double2 l = lv[j * LNP + pl];
        a.l[j] = fma(p0, l.x, a.l[j]);
        a.l[j] = fma(p1, l.y, a.l[j]);
      }
    }
    const double2 yv = lv[K * LNP + pl];
    a.y = fma(p0, yv.x, a.y);
    a.y = fma(p1, yv.y, a.y);
  }
  if (sizeof(T) == 4) a.mxf = fmaxf(a.mxf, (float)av);
  else { const double avd = (double)av; a.mx = a.mx > avd ? a.mx : avd; }
}

// A warp's reduced sums of one proposal on one tile, added to the proposal's running record d[0 .. K + 3].  EXACT (compile-time K):
// after WAcc::warp_reduce_scatter, sum j sits in l[0] of the lanes owner(j) ..; else after warp_reduce, everything in every lane.
template <int KC, bool EXACT>
__device__ __forceinline__ void add_record(const WAcc<KC>& a, double* d, int K, int lane) {
  if (EXACT) {
    constexpr int LPV = 32 / WAcc<KC>::VP;      // lanes holding the same sum
    const int j = (WAcc<KC>::VP == 8) ? (((lane >> 4) & 1) << 2 | ((lane >> 3) & 1) << 1 | ((lane >> 2) & 1))
                                      : (WAcc<KC>::VP == 16 ? (((lane >> 4) & 1) << 3 | ((lane >> 3) & 1) << 2 | ((lane >> 2) & 1) << 1 | ((lane >> 1) & 1)) : lane);
    if ((lane & (LPV - 1)) == 0 && j < KC + 3) d[j] += a.l[0];
    if (lane == 1) d[K + 3] = d[K + 3] > a.mx ? d[K + 3] : a.mx;
  } else if (lane == 0) {
#pragma unroll
    for (int j = 0; j < KC; ++j) if (j < K) d[j] += a.l[j];
    d[K] += a.y; d[K + 1] += a.pp; d[K + 2] += a.s;
    d[K + 3] = d[K + 3] > a.mx ? d[K + 3] : a.mx;
  }
}

#ifndef BSR_CHECKED_M
#define BSR_CHECKED_M 12   // node count from which k_weval's first pass checks every vector for finiteness itself
#endif

// Second pass over the rows of a tile for a proposal whose fp32 column is not finite there, by the whole block (few proposals
// need it, and a warp left alone with it would hold up its block): the value rule vector by vector (vec_finite /
// eval_tree_wide2) -- out-of-range vectors in double range, the others stay the fp32 values they are.  The per-warp partials
// are summed in warp order into s_acc[i].  s_tok, s_part: the (now idle) per-warp token staging, 1 KB per warp (>= 8 warps).
// bm != nullptr: the first pass was the checked one (large tree): it kept the sums of the finite vectors and left the bitmap of the others.  Out of line:
// it must not cost the fp32 loop of k_weval a register.  Must be called by every thread of the block.
template <int KC>
static __device__ BSR_WIDE_INLINE void careful_tile(const uint32_t* __restrict__ tok, const double* __restrict__ pa, const double* __restrict__ pb, int m,
                                                 const float* __restrict__ X32, const double* __restrict__ X64, uint32_t xbase, uint32_t ld, uint32_t n, int K, int i,
                                                 uint32_t t_lo, uint32_t tile_rows, const double2* s_live, EvTok<float>* s_tok, double* s_part,
                                                 double* s_acc, unsigned long long* s_dead, const unsigned* bm) {
  const int RECN = K + 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  const uint32_t tv = (tile_rows + 3) / 4;
  const int LS = win_live_stride<float>(K);
  // scratch behind the partials (the idle per-warp token staging holds NW KB: tokens 1 KB, partials <= 1.25 KB, then these)
  int* s_cnt = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(s_tok) + 2304);               // [steps][NW] out-of-range vectors per warp and step
  unsigned short* s_list = reinterpret_cast<unsigned short*>(reinterpret_cast<unsigned char*>(s_tok) + 2560);   // [<= tv] their indices, ascending
  const int nsteps = (int)((tv + blockDim.x - 1) / blockDim.x);       // <= 8 (tile budget of win_geometry: tv <= 640)
  __syncthreads();
  stage_tokens<float>(tok, pa, pb, m, xbase, ld, s_tok, threadIdx.x, blockDim.x);
  __syncthreads();
  WAcc<KC> a;
  a.zero();
  // fp32 vectors: accumulated where they are finite, listed where they are not
  unsigned mybad = 0u;
  for (int k = 0; k < nsteps; ++k) {
    const uint32_t q = threadIdx.x + (uint32_t)k * blockDim.x;
    bool bad = false;
    if (q < tv) {
      if (bm != nullptr) bad = (bm[q >> 5] >> (q & 31)) & 1u;      // the first pass told the vectors apart already (and kept the finite ones' sums)
      else {
        const uint32_t row0 = t_lo + q * 4;
        float v[4];
        eval_tree_rows<float, 4>(s_tok, m, X32, row0, v);
        if (vec_finite(v)) wacc_rows<float, KC, 2, true>(a, K, v, s_live + q * LS, row0, n);
        else bad = true;
      }
    }
    const unsigned bal = __ballot_sync(0xffffffffu, bad);
    if (bad) mybad |= 1u << k;
    if (lane == 0) s_cnt[k * NW + warp] = __popc(bal);
  }
  __syncthreads();
  int nl = 0;
  for (int k = 0; k < nsteps; ++k) {
    const unsigned bal = __ballot_sync(0xffffffffu, (mybad >> k) & 1u);
    int base = 0;
    for (int e = 0; e < nsteps * NW; ++e) { const int n_e = s_cnt[e]; base += (e < k * NW + warp) ? n_e : 0; nl += (k == 0) ? n_e : 0; }
    if ((mybad >> k) & 1u) s_list[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned short)(threadIdx.x + k * blockDim.x);
  }
  __syncthreads();
  // the listed vectors in double range, two rows (one plane of the tile layout) per thread and step: every lane busy whatever the
  // share of out-of-range rows; the list is in ascending order, so the sums do not depend on timing
#pragma unroll 1
  for (int e = threadIdx.x; e < 2 * nl; e += blockDim.x) {
    const uint32_t q = s_list[e >> 1];
    const int pl = e & 1;
    const uint32_t row0 = t_lo + q * 4 + 2 * pl;
    const double2 x = eval_tree_wide2(s_tok, pa, pb, m, X64, row0);
    const double xv[2] = {x.x, x.y};
    wacc_rows<double, KC, 2, true>(a, K, xv, s_live + q * LS + pl, row0, n);
  }
  a.warp_reduce();
  if (lane == 0) {
    double* d = s_part + (size_t)warp * RECN;
#pragma unroll
    for (int j = 0; j < KC; ++j) if (j < K) d[j] = a.l[j];
    d[K] = a.y; d[K + 1] = a.pp; d[K + 2] = a.s; d[K + 3] = a.mx;
  }
  __syncthreads();
  if ((int)threadIdx.x < RECN) {
    double v = s_acc[(size_t)i * RECN + threadIdx.x];
    for (int w = 0; w < NW; ++w) {
      const double x = s_part[(size_t)w * RECN + threadIdx.x];
      v = ((int)threadIdx.x < K + 3) ? v + x : (v > x ? v : x);
    }
    s_acc[(size_t)i * RECN + threadIdx.x] = v;
    // not finite in double range either: the column's record is settled (reject), later tiles skip it
    if ((int)threadIdx.x == K + 1 && !(fabs(v) <= DBL_MAX)) atomicOr(s_dead, 1ull << i);
    if ((int)threadIdx.x == K + 3 && !(v <= DBL_MAX)) atomicOr(s_dead, 1ull << i);
  }
}

#ifndef BSR_WEVAL_THREADS
#define BSR_WEVAL_THREADS 256
#endif
#ifndef BSR_WEVAL_MINB3
#define BSR_WEVAL_MINB3 3   // resident blocks per SM asked of the compiler for K <= 3: 3 x 256 threads x 80 registers; 4 blocks
                            // (64 registers, 220 KB of shared memory, ~28 KB left for L1) measured slower: the interpreter's
                            // local-memory stack then misses L1 (hit rate 60 %, long-scoreboard stalls on top)
#endif
// MULTI: the handle holds several data sets and every chain reads its own (st.ds).  The instances of one data set (MULTI = false)
// have no data-set term at all: whatever the term is written as, ptxas allocates the 80-register tile loop differently for it, with
// more spills in some instances (DESIGN.md section 5), and a handle of one data set must not pay for that.
// The data sets of a MULTI handle may differ in row count (wc.ds_n): the chain's rows end at its own n, and a (chain, split) block
// whose split starts at or past it has nothing to do -- k_wresolve reads only the splits that hold rows of the chain's data set.
template <typename T, int KC, bool EXACT, bool MULTI>
__global__ void __launch_bounds__(BSR_WEVAL_THREADS, (KC <= 3 ? BSR_WEVAL_MINB3 : (KC <= 5 ? 3 : 2))) k_weval(ChainState st, WinState ws, WinCtx wc) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int c = wc.c0 + blockIdx.x;
  if (st.done[c] || ws.pos[c] >= wc.p_target) return;
  const uint32_t n_c = MULTI ? wc.ds_n[st.ds[c]] : wc.n;
  if (MULTI && blockIdx.y * wc.rows_per_split >= n_c) return;
  const int K = EXACT ? KC : st.K;
  constexpr int R = RowVec<T>::R;
  const int W = ws.W, RECN = K + 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  const WinSmem L = win_smem_layout<T>(K, W, NW, wc.TR, MULTI);
  double2* s_live = reinterpret_cast<double2*>(smem_raw + L.live);
  double* s_acc = reinterpret_cast<double*>(smem_raw + L.acc);
  EvTok<T>* s_ltok = reinterpret_cast<EvTok<T>*>(smem_raw + L.ltok);
  EvTok<T>* s_ptok = reinterpret_cast<EvTok<T>*>(smem_raw + L.ptok) + (size_t)warp * BSR_MAXN;
  int* s_lm = reinterpret_cast<int*>(smem_raw + L.lm);
  unsigned long long* s_flag = reinterpret_cast<unsigned long long*>(s_lm + K + (K & 1));   // 8-byte aligned: slots of this tile that need the second pass
  unsigned long long* s_dead = s_flag + 1;                                                  // slots whose column is not finite even in double range
  unsigned long long* s_pre = s_dead + 1;                                                   // slots of this tile whose out-of-range vectors the first pass listed (s_bm)
  int* s_next = reinterpret_cast<int*>(s_pre + 1);
  int* s_ds = s_next + 1;                                                                   // (MULTI) the chain's data set and its row count: read
  uint32_t* s_n = reinterpret_cast<uint32_t*>(s_ds + 1);                                    // where they are used, so that the tile loop holds no
                                                                                            // register for them
  unsigned* s_bm = reinterpret_cast<unsigned*>(smem_raw + L.bm);
  const T* X = (sizeof(T) == 4) ? reinterpret_cast<const T*>(wc.X32) : reinterpret_cast<const T*>(wc.X64);
  DedupSmem& dd = *reinterpret_cast<DedupSmem*>(smem_raw + L.dd);
  const unsigned char* s_rep = dd.rep;
  if (threadIdx.x == 0) { *s_flag = 0ull; *s_dead = 0ull; if (MULTI) { *s_ds = st.ds[c]; *s_n = n_c; } }
  const int head = ws.chead[c];                   // ring index of the chain's last window (still valid for the live state), or -1
  const int nprev = (head >= 0 && wc.dedup >= 2) ? (int)ws.cvalid[c] : 0;
  const WinState wv = win_half(ws, head >= 0 ? ((head + 1) % ws.R) : 0, K);     // this window's slots (win_parity)
  const int n_eval = ws.neval[c];                 // k_wdedup: slots left to interpret (block-uniform)
  if ((int)threadIdx.x < W) {
    const size_t wi = (size_t)c * W + threadIdx.x;
    dd.rep[threadIdx.x] = ws.rep[wi];
    dd.prev[threadIdx.x] = ws.prevslot[wi];
    dd.order[threadIdx.x] = ws.order[wi];
    dd.m[threadIdx.x] = (wv.hash[wi] != 0ull) ? (unsigned char)wv.nn[wi] : (unsigned char)0;
  }
  if (n_eval > 0) {
    const uint32_t xbase = MULTI ? (uint32_t)st.ds[c] * wc.ds_stride : 0u;
    for (int j = 0; j < K; ++j) {
      const int g = c * K + j;
      const int w = st.which[g];
      const int m = st.nn[w][g];
      if (threadIdx.x == 0) s_lm[j] = m;
      const size_t slot = (size_t)g * BSR_MAXN;
      stage_tokens<T>(st.tok[w] + slot, st.pa[w] + slot, st.pb[w] + slot, m, xbase, wc.ld, s_ltok + j * BSR_MAXN, threadIdx.x, blockDim.x);
    }
    for (int i = threadIdx.x; i < W * RECN; i += blockDim.x) s_acc[i] = 0.0;
  }
  const unsigned char* s_order = dd.order;

  const uint32_t r_lo = blockIdx.y * wc.rows_per_split;
  const uint32_t r_hi = min(n_c, r_lo + wc.rows_per_split);
  unsigned long long wide_mask = 0ull;             // slots that needed the second pass on some tile of this block (block-uniform)
  for (uint32_t t_lo = r_lo; t_lo < r_hi; t_lo += wc.TR) {
    const uint32_t tile_rows = min(wc.TR, r_hi - t_lo);
    __syncthreads();
    if (threadIdx.x == 0) { *s_next = 0; *s_flag = 0ull; *s_pre = 0ull; }
    if (n_eval == 0) continue;                     // every tree of this window has its record already (block-uniform)
    // (the cache of live columns and the checked first pass belong to the K > 5 kernels: the 80-register kernels of K <= 5 pay for the
    // extra paths in spills -- measured: C4 -3 %, C5 -7 % -- what the cache gives their 4-node trees)
    if (KC > 5) live_tile<T>(st, wc, c, K, MULTI ? (uint32_t)*s_ds : 0u, MULTI ? *s_n : wc.n, s_ltok, s_lm, t_lo, tile_rows, s_live, ws.lcol, ws.lcol_ld, ws.lcol_ok, ws.lcol_wide);
    else live_tile<T>(st, wc, c, K, MULTI ? (uint32_t)*s_ds : 0u, MULTI ? *s_n : wc.n, s_ltok, s_lm, t_lo, tile_rows, s_live);
    __syncthreads();
    const uint32_t tv = (tile_rows + R - 1) / R;
    const unsigned long long dead = *s_dead;      // columns found non-finite on an earlier tile: their record is settled (reject)
    // the warps of the block take the proposals of the window from a shared counter: trees differ in size, a static
    // assignment leaves warps waiting at the barrier below
#pragma unroll 1
    for (;;) {
      int i = 0;
      if (lane == 0) i = atomicAdd(s_next, 1);
      i = __shfl_sync(0xffffffffu, i, 0);
      if (i >= n_eval) break;
      i = s_order[i];                            // the slots to interpret, largest tree first (repeated trees share a record)
      if ((dead >> i) & 1ull) continue;
      const size_t wi = (size_t)c * W + i;
      const int m = dd.m[i];                     // (node count of the slot, staged with the results of the duplicate search)
      __syncwarp();
      stage_tokens<T>(wv.tok + wi * BSR_MAXN, wv.pa + wi * BSR_MAXN, wv.pb + wi * BSR_MAXN, m, MULTI ? (uint32_t)*s_ds * wc.ds_stride : 0u, wc.ld, s_ptok, lane,
                      32);
      __syncwarp();
      WAcc<KC> a;
      // NV interleaved row vectors per thread and token decode: vector u of lane l is vector q + 32 u of the tile
      constexpr int NV = (sizeof(T) == 4) ? BSR_WEVAL_NV : 1;
      constexpr int NP = R / 2;
      const int LS = win_live_stride<T>(K);
      const bool tail_tile = t_lo + tv * R > (MULTI ? *s_n : wc.n);      // only the last vector of the last tile can be ragged
      a.zero();
      // Large trees (fp32 mode): the pass tells finite from out-of-range vectors as it goes (4 FFMA per vector: nothing beside a
      // 12+-node tree, 5 % beside the average 4-node tree of C2) -- it keeps the sums of the finite vectors and leaves a bitmap of the
      // others, so that the block's second pass interprets those in double range and nothing else.  (K = 10 with 31-node trees, C3:
      // 29 % of the proposals have out-of-range vectors; without this they cost a discarded first pass and a second fp32 pass.)
      if (sizeof(T) == 4 && KC > 5 && m >= wc.checked_m && tv <= 256) {   // (K > 5: the kernels of 128 registers; the 80-register ones have no room for a second loop)
        unsigned anyb = 0u;
#pragma unroll 1
        for (uint32_t q0 = 0; q0 < tv; q0 += 32 * NV) {
          const uint32_t q = q0 + lane;
          T v[NV][R];
          uint32_t rowoff[NV];
#pragma unroll
          for (int u = 0; u < NV; ++u) rowoff[u] = (q + 32 * u < tv) ? t_lo + (q + 32 * u) * R : t_lo;
          eval_tree_rows_nv<T, R, NV>(s_ptok, m, X, rowoff, v);
#pragma unroll
          for (int u = 0; u < NV; ++u) {
            const bool valid = q + 32 * u < tv;
            float vf[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) vf[r] = (float)v[u][r < R ? r : 0];
            const bool fin = vec_finite(vf);
            if (valid && fin) wacc_rows<T, KC, NP, true>(a, K, v[u], s_live + (size_t)(q + 32 * u) * LS, rowoff[u], MULTI ? *s_n : wc.n);
            const unsigned bal = __ballot_sync(0xffffffffu, valid && !fin);
            if (lane == 0) s_bm[i * 8 + (q0 >> 5) + u] = bal;
            anyb |= bal;
          }
        }
        a.template warp_reduce_scatter_or_all<EXACT, sizeof(T) == 4>(lane);
        if (anyb != 0u && lane == 0) { atomicOr(s_flag, 1ull << i); atomicOr(s_pre, 1ull << i); }
        add_record<KC, EXACT>(a, s_acc + (size_t)i * RECN, K, lane);
        continue;
      }
#pragma unroll 1
      for (uint32_t q = lane; q < tv; q += 32 * NV) {
        T v[NV][R];
        uint32_t rowoff[NV];
        rowoff[0] = t_lo + q * R;
#pragma unroll
        for (int u = 1; u < NV; ++u) rowoff[u] = (q + 32 * u < tv) ? rowoff[0] + 32 * u * R : rowoff[0];
        eval_tree_rows_nv<T, R, NV>(s_ptok, m, X, rowoff, v);
        const double2* lv = s_live + q * LS;
#pragma unroll
        for (int u = 0; u < NV; ++u) {
          if (u == 0 || q + 32 * u < tv) {
            if (tail_tile && rowoff[u] + R > (MULTI ? *s_n : wc.n)) wacc_rows<T, KC, NP, true>(a, K, v[u], lv + 32 * u * LS, rowoff[u], MULTI ? *s_n : wc.n);
            else wacc_rows<T, KC, NP, false>(a, K, v[u], lv + 32 * u * LS, rowoff[u], wc.n);
          }
        }
      }
      // (EXACT: the sums end up one per lane group, see WAcc::warp_reduce_scatter; the generic-K kernel reduces every sum in every lane)
      bool nonfinite;
      if (EXACT) {
        a.template warp_reduce_scatter<sizeof(T) == 4>(lane);
        const unsigned nf = __ballot_sync(0xffffffffu, !(fabs(a.l[0]) <= DBL_MAX));
        nonfinite = ((nf >> WAcc<KC>::owner(KC + 1)) & 1u) || !(a.mx <= DBL_MAX);
      } else {
        a.warp_reduce();
        nonfinite = !(fabs(a.pp) <= DBL_MAX) || !(a.mx <= DBL_MAX);
      }
      if (sizeof(T) == 4 && nonfinite) {
        // the column is not finite on the rows of this tile: the block goes through them once more with the value rule applied vector
        // by vector, once every warp is through its proposals (the live values of the tile are still in shared memory then)
        if (lane == 0) atomicOr(s_flag, 1ull << i);
        continue;
      }
      add_record<KC, EXACT>(a, s_acc + (size_t)i * RECN, K, lane);
    }
    if (sizeof(T) == 4) {
      __syncthreads();
      const unsigned long long tmask = *s_flag, pre = *s_pre;      // block-uniform
      if (tmask != 0ull) {
        EvTok<float>* s_tok0 = reinterpret_cast<EvTok<float>*>(smem_raw + L.ptok);
        double* s_part = reinterpret_cast<double*>(smem_raw + L.ptok + 1024);
        for (unsigned long long rest = tmask; rest != 0ull; rest &= rest - 1ull) {
          const int i = __ffsll((long long)rest) - 1;
          const size_t wi = (size_t)c * W + i;
          careful_tile<KC>(wv.tok + wi * BSR_MAXN, wv.pa + wi * BSR_MAXN, wv.pb + wi * BSR_MAXN, wv.nn[wi], wc.X32, wc.X64,
                           MULTI ? (uint32_t)*s_ds * wc.ds_stride : 0u, wc.ld,
                           MULTI ? *s_n : wc.n, K, i, t_lo, tile_rows,
                           s_live, s_tok0, s_part, s_acc, s_dead, (KC > 5 && ((pre >> i) & 1ull)) ? s_bm + i * 8 : nullptr);
        }
        wide_mask |= tmask;
      }
    }
  }
  __syncthreads();
  // slots whose record comes from an out-of-range slot of an earlier window are out-of-range proposals too
  unsigned long long pbad[BSR_WIN_RING - 1];
#pragma unroll
  for (int d = 0; d < BSR_WIN_RING - 1; ++d)
    pbad[d] = (d < nprev && sizeof(T) == 4) ? ws.bad[(size_t)((head - d + ws.R) % ws.R) * ws.C + c] : 0ull;
  // records: element e of the window's W x RECN block, one thread each (coalesced); the out-of-range masks from per-slot ballots
  {
    const unsigned long long mask = wide_mask;
    double* out = wv.rec + ((size_t)c * ws.S + blockIdx.y) * W * RECN;
    const size_t ring_stride = (size_t)ws.C * ws.S * W * RECN;      // records of one ring index
    const double* rec0 = ws.rec + ((size_t)c * ws.S + blockIdx.y) * W * RECN;
    for (int e = threadIdx.x; e < W * RECN; e += blockDim.x) {
      const int i = e / RECN, q = e - i * RECN;
      if (dd.m[i] == 0) continue;
      const int r = s_rep[i] & 0x7f;                  // first slot of this window with the same tree
      if (s_rep[r] & 0x80) {                          // ... whose record an earlier window holds (this split's part of it)
        const int pr = dd.prev[r], ring = (head - (pr >> 6) + ws.R) % ws.R;
        out[e] = rec0[(size_t)ring * ring_stride + (pr & 63) * RECN + q];
      } else out[e] = s_acc[r * RECN + q];
    }
    if ((int)threadIdx.x < W && sizeof(T) == 4) {
      const int i = threadIdx.x;
      bool bad = false;
      if (dd.m[i] != 0) {
        const int r = s_rep[i] & 0x7f;
        bad = (s_rep[r] & 0x80) ? ((pbad[dd.prev[r] >> 6] >> (dd.prev[r] & 63)) & 1ull) : ((mask >> r) & 1ull);
      }
      const unsigned b0 = __ballot_sync(0xffffffffu, bad);
      if (lane == 0 && b0) atomicOr(wv.bad + c, (unsigned long long)b0 << (32 * warp));
    }
  }
}

// First step of the refit (fp32 evaluation only): which live columns leave the fp32 range on this rank's rows (bookkeeping: the
// flag an accepted out-of-range proposal would have set; the evaluation itself applies the value rule vector by vector whatever
// the flag says).  st.live_bad is zeroed by the host before.
static __global__ void __launch_bounds__(BSR_WEVAL_THREADS) k_wlive_bad(ChainState st, WinCtx wc, int S) {
  __shared__ EvTok<float> s_tok[BSR_MAXN];
  __shared__ int s_bad;
  const int c = wc.c0 + blockIdx.x;
  const int K = st.K;
  const uint32_t n = wc.ds_n != nullptr ? wc.ds_n[st.ds[c]] : wc.n;
  const uint32_t r_lo = blockIdx.y * wc.rows_per_split;
  const uint32_t r_hi = min(n, r_lo + wc.rows_per_split);
  const uint32_t xbase = (uint32_t)st.ds[c] * wc.ds_stride;
  for (int j = 0; j < K; ++j) {
    const int g = c * K + j;
    const int w = st.which[g];
    const int m = st.nn[w][g];
    const size_t slot = (size_t)g * BSR_MAXN;
    __syncthreads();
    if (threadIdx.x == 0) s_bad = 0;
    stage_tokens<float>(st.tok[w] + slot, st.pa[w] + slot, st.pb[w] + slot, m, xbase, wc.ld, s_tok, threadIdx.x, blockDim.x);
    __syncthreads();
    bool bad = false;
    for (uint32_t row0 = r_lo + threadIdx.x * 4; row0 < r_hi; row0 += blockDim.x * 4) {
      float v[4];
      eval_tree_rows<float, 4>(s_tok, m, wc.X32, row0, v);
#pragma unroll
      for (int r = 0; r < 4; ++r) bad = bad || (row0 + r < n && !(fabsf(v[r]) <= FLT_MAX));
    }
    if (bad) s_bad = 1;
    __syncthreads();
    if (threadIdx.x == 0 && s_bad) st.live_bad[g] = 1;
  }
}

// Per live tree: the counts the move selection needs and fStruc with the tree's sigma_a, sigma_b (codes/funcs.py:349-398,
// 457-480).  Runs at every refit; an accept updates the entries of its tree (k_wresolve).
__device__ __forceinline__ int live_counts(const uint32_t* tk, int m) {
  int L = 0, T = 0;
  for (int j = 0; j < m; ++j) { const int o = tok_op(tk[j]); L += (o == OP_LT); T += (o == OP_LEAF); }
  const int D = det_count(tk, m, m - T);
  return m | (L << 8) | (T << 16) | (D << 24);
}
static __global__ void k_wlive_prior(ChainState st, const PriorTables* __restrict__ ptp, const int* __restrict__ chain_pt) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= st.C * st.K) return;
  const int w = st.which[g];
  const int m = st.nn[w][g];
  const size_t slot = (size_t)g * BSR_MAXN;
  uint32_t tk[BSR_MAXN];
  for (int j = 0; j < m; ++j) tk[j] = st.tok[w][slot + j];
  st.lcnt[g] = live_counts(tk, m);
  double ll, lp;
  fstruc_tree(ptp[chain_pt[g / st.K]], tk, m, st.pa[w] + slot, st.pb[w] + slot, st.sa[g], st.sb[g], ll, lp);
  st.lfs[2 * (size_t)g] = ll; st.lfs[2 * (size_t)g + 1] = lp;
}

// Last step of the refit: the partial Grams of all splits (and ranks, in rank order) summed into the chain's live Gram, from
// which the K-column SSE of the live state (ylogLike, codes/funcs.py:1147-1162) and the intercept fit (codes/bsr_class.py:147-163)
// follow.  One thread per chain; runs once per (re)initialisation.
static __global__ void k_wrefit(ChainState st, WinCtx wc, int S, int c0, int cn) {
  const int ci = blockIdx.x * blockDim.x + threadIdx.x;
  if (ci >= cn) return;
  if (wc.abort_flag != nullptr && *wc.abort_flag != 0) return;
  const int c = c0 + ci;
  const int K = st.K;
  const int sgn = sg_size(K);
  double* sg = st.sg + (size_t)c * sgn;
  const int n_src = wc.n_peers > 0 ? wc.n_peers : 1;
  // several data sets: the chain's own rows and the splits that hold them; one data set: all rows of all ranks, every split
  const int ds = st.ds[c];
  const double n_rows = wc.ds_n != nullptr ? (double)wc.ds_n[ds] : wc.n_total;
  const int S_c = wc.ds_n != nullptr ? (int)((wc.ds_n[ds] + wc.rows_per_split - 1) / wc.rows_per_split) : S;
  for (int e = 0; e < sgn; ++e) {
    double v = 0.0;
    for (int pr = 0; pr < n_src; ++pr)
      for (int sp = 0; sp < S_c; ++sp) {
        const double x = wc.peer_lrec[pr][((size_t)c * S + sp) * sgn + e];
        v = (e < sgn - K) ? v + x : (v > x ? v : x);
      }
    sg[e] = v;
  }
  for (int j = 0; j < K; ++j) {     // a non-finite live column (even in double range): marked like a proposal's would be
    const double gjj = sg[gram_idx(K, j, j)];
    if (!(fabs(gjj) <= DBL_MAX) || !(sg[sgn - K + j] <= DBL_MAX)) sg[sgn - K + j] = INFINITY;
  }
  GramView gl{sg, sg + K * (K + 1) / 2 + 2 * K, K};
  int il[BSR_MAXK];
  double bl[BSR_LDA];
  for (int j = 0; j < K; ++j) il[j] = j;
  const double* ys = wc.ystats + 2 * (size_t)ds;
  st.sse[c] = ridge_sse<BSR_LDA, false>(gl, il, K, n_rows, ys[0], ys[1], bl);
  (void)ridge_sse<BSR_LDA, true>(gl, il, K, n_rows, ys[0], ys[1], bl);
  for (int j = 0; j <= K; ++j) st.beta[(size_t)c * (K + 1) + j] = bl[j];
}

template <typename T, int KC, bool EXACT>
__global__ void __launch_bounds__(BSR_WEVAL_THREADS) k_wlive_gram(ChainState st, WinState ws, WinCtx wc, double* lrec) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int c = wc.c0 + blockIdx.x;
  const int K = EXACT ? KC : st.K;
  constexpr int R = RowVec<T>::R, NP = R / 2;
  constexpr int NG = KC * (KC + 1) / 2;
  const int W = ws.W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  const WinSmem L = win_smem_layout<T>(K, W, NW, wc.TR);
  double2* s_live = reinterpret_cast<double2*>(smem_raw + L.live);
  double* s_red = reinterpret_cast<double*>(smem_raw + L.total);      // [NW][sgn], behind the layout k_weval uses
  EvTok<T>* s_ltok = reinterpret_cast<EvTok<T>*>(smem_raw + L.ltok);
  int* s_lm = reinterpret_cast<int*>(smem_raw + L.lm);
  const uint32_t ds = (uint32_t)st.ds[c];
  const uint32_t n = wc.ds_n != nullptr ? wc.ds_n[ds] : wc.n;
  for (int j = 0; j < K; ++j) {
    const int g = c * K + j;
    const int w = st.which[g];
    const int m = st.nn[w][g];
    if (threadIdx.x == 0) s_lm[j] = m;
    const size_t slot = (size_t)g * BSR_MAXN;
    stage_tokens<T>(st.tok[w] + slot, st.pa[w] + slot, st.pb[w] + slot, m, ds * wc.ds_stride, wc.ld, s_ltok + j * BSR_MAXN, threadIdx.x, blockDim.x);
  }
  double g_[NG], by[KC], cs[KC], mx[KC];
#pragma unroll
  for (int e = 0; e < NG; ++e) g_[e] = 0.0;
#pragma unroll
  for (int j = 0; j < KC; ++j) { by[j] = 0.0; cs[j] = 0.0; mx[j] = 0.0; }
  const int LS = win_live_stride<T>(K);
  const uint32_t r_lo = blockIdx.y * wc.rows_per_split;
  const uint32_t r_hi = min(n, r_lo + wc.rows_per_split);
  for (uint32_t t_lo = r_lo; t_lo < r_hi; t_lo += wc.TR) {
    const uint32_t tile_rows = min(wc.TR, r_hi - t_lo);
    __syncthreads();
    live_tile<T>(st, wc, c, K, ds, n, s_ltok, s_lm, t_lo, tile_rows, s_live);
    __syncthreads();
    const uint32_t tv = (tile_rows + R - 1) / R;
#pragma unroll 1
    for (uint32_t q = threadIdx.x; q < tv; q += blockDim.x) {
#pragma unroll
      for (int pl = 0; pl < NP; ++pl) {
        const double2 yv = s_live[q * LS + K * NP + pl];
        double2 l[KC];
#pragma unroll
        for (int j = 0; j < KC; ++j) l[j] = (j < K) ? s_live[q * LS + j * NP + pl] : make_double2(0.0, 0.0);
        int e = 0;
#pragma unroll
        for (int i = 0; i < KC; ++i) {
#pragma unroll
          for (int j = i; j < KC; ++j, ++e) { g_[e] = fma(l[i].x, l[j].x, g_[e]); g_[e] = fma(l[i].y, l[j].y, g_[e]); }
          by[i] = fma(l[i].x, yv.x, by[i]); by[i] = fma(l[i].y, yv.y, by[i]);
          cs[i] += l[i].x; cs[i] += l[i].y;
          // fmax drops a NaN operand; a non-finite column shows in its diagonal Gram entry
          mx[i] = fmax(mx[i], fmax(fabs(l[i].x), fabs(l[i].y)));
        }
      }
    }
  }
  // sg layout: G(i, j), i <= j < K row-major, then by, cs, mx
  const int sgn = sg_size(K);
  __syncthreads();
  {
    int e = 0, o = 0;
#pragma unroll
    for (int i = 0; i < KC; ++i)
#pragma unroll
      for (int j = i; j < KC; ++j, ++e) {
        const double v = warp_sum(g_[e]);
        if (i < K && j < K) { if (lane == 0) s_red[(size_t)warp * sgn + o] = v; ++o; }
      }
    const int kg = K * (K + 1) / 2;
#pragma unroll
    for (int i = 0; i < KC; ++i) {
      const double a = warp_sum(by[i]), b = warp_sum(cs[i]), m = warp_max<double>(mx[i]);
      if (i < K && lane == 0) { s_red[(size_t)warp * sgn + kg + i] = a; s_red[(size_t)warp * sgn + kg + K + i] = b; s_red[(size_t)warp * sgn + kg + 2 * K + i] = m; }
    }
  }
  __syncthreads();
  double* out = lrec + ((size_t)c * ws.S + blockIdx.y) * sgn;
  for (int e = threadIdx.x; e < sgn; e += blockDim.x) {
    double v = 0.0;
    for (int w = 0; w < NW; ++w) {
      const double x = s_red[(size_t)w * sgn + e];
      v = (e < sgn - K) ? v + x : (v > x ? v : x);
    }
    out[e] = v;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// resolve
// ---------------------------------------------------------------------------------------------------------------
// LPC = 32 (W <= 32) or 64 lanes per chain, lane i = window slot i.  Phase A (all lanes): the proposal's Gram against
// the live set is put together from the chain's live Gram cache (st.sg) and the proposal's K + 4 sums, then rank test,
// ridge SSE, logR and the accept draw exactly as resolve_chain (bsr_solve.cuh) computes them.  Phase B: in-order
// consumption from the ballots of the chain's lanes (two warps exchange theirs through shared memory when LPC = 64).
#ifndef BSR_WRES_MINB
#define BSR_WRES_MINB 4
#endif
// MULTI: as for k_weval -- the chain's sum(y), y'y come from its data set's entry of wc.ystats, else from wc.sum_y, wc.yy; its row
// count from wc.ds_n (else wc.n_total, wc.n_local: a handle of several data sets is never row-sharded, so the two are one number),
// and its records from the splits that hold its rows.  PRIORS: the chains differ in their stop rule (bsr_set_chain_priors), chain c's
// is chain_stop[c] = val (0: never) | plateau rule << 31; else every chain's is st.val, st.plateau_rule and chain_stop is not read (the
// instances of one prior are those of a handle without per-chain priors, register for register).
template <int KT, bool MULTI, bool PRIORS>
__global__ void __launch_bounds__(128, (KT > 0 ? BSR_WRES_MINB : 1)) k_wresolve(ChainState st, WinState ws, WinCtx wc,
                                                                               const int* __restrict__ chain_stop) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int LD = (KT > 0) ? KT + 1 : BSR_LDA;
  constexpr int PC = (KT > 0) ? KT + 1 : BSR_MAXK + 1;
  constexpr int NS = PC * (PC + 1) / 2 + 2 * PC;
  const int K = (KT > 0) ? KT : st.K;
  const int P1 = K + 1, RECN = K + 4, W = ws.W;
  const int LPC = (W > 32) ? 64 : 32;
  const int cpb = blockDim.x / LPC;                 // chains per block
  const int cl = threadIdx.x / LPC;                 // chain slot inside the block
  const int sl = threadIdx.x % LPC;                 // window slot of this thread
  const int lane = threadIdx.x & 31;
  const int half = sl >> 5;                         // which warp of the chain (LPC = 64)
  const int ci = blockIdx.x * cpb + cl;
  const int c = wc.c0 + (ci < wc.cn ? ci : 0);
  if (wc.abort_flag != nullptr && *wc.abort_flag != 0) return;   // a peer never delivered this window (k_wwait): leave the chains as they are
  bool live = ci < wc.cn && !st.done[c];
  const long long p0 = live ? ws.pos[c] : 0;
  live = live && p0 < wc.p_target;
  if (LPC == 32 && !live) return;                   // (with two warps per chain everybody must reach the barriers below)
  const int sgn = sg_size(K);
  double* s_sg = reinterpret_cast<double*>(smem_raw) + (size_t)cl * sgn;
  unsigned* s_bal = reinterpret_cast<unsigned*>(reinterpret_cast<double*>(smem_raw) + (size_t)cpb * sgn) + (size_t)cl * 8;
  if (live) for (int e = sl; e < sgn; e += LPC) s_sg[e] = st.sg[(size_t)c * sgn + e];
  if (LPC == 32) __syncwarp(); else __syncthreads();

  const size_t wi = (size_t)c * W + (sl < W ? sl : 0);
  const int wpar = (live && wc.n_peers == 0) ? win_parity(ws, c) : 0;
  const WinState wv = win_half(ws, wpar, K);                 // the ring entry of the slot arrays this window was written to
  PropInfo pi = wv.info[wi];
  const long long p = p0 + sl;
  const bool valid = live && sl < W && p < wc.p_target && !(pi.flags & PF_SKIP);
  const bool cap = valid && (pi.flags & PF_CAPACITY);
  const int k = (int)(p % K);
  unsigned long long badmask = 0ull;
  if (live) {
    if (wc.n_peers == 0) badmask = wv.bad[c];
    else {
#pragma unroll 1
      for (int r = 0; r < wc.n_peers; ++r) badmask |= wc.peer_bad[r][c];
    }
  }

  // ---- phase A ----
  double lsums[NS], lmaxs[PC];
  GramView gv{lsums, lmaxs, P1};
  const int ng = P1 * (P1 + 1) / 2;
  bool rank_rej = false, accepted = false;
  double logR = nan(""), sse_new = nan(""), u = nan("");
  RankDiag dg;
  dg.pivot_min = nan(""); dg.sv_ratio = -1.0; dg.path = 0;
  const double sigma = st.sigma[c];
  const double sse_old = st.sse[c];
  const uint32_t n_c = MULTI ? wc.ds_n[st.ds[c]] : 0u;     // (MULTI only)
  int msum = 0;
  for (int j = 0; j < K; ++j) msum += st.nn[st.which[c * K + j]][c * K + j];
  const int m_old_k = st.nn[st.which[c * K + k]][c * K + k];
  if (valid && !cap) {
    {
      int e = 0;
#pragma unroll
      for (int i = 0; i < K; ++i)
#pragma unroll
        for (int j = i; j < K; ++j) lsums[gram_idx(P1, i, j)] = s_sg[e++];
#pragma unroll
      for (int i = 0; i < K; ++i) {
        lsums[ng + i] = s_sg[e + i];
        lsums[ng + P1 + i] = s_sg[e + K + i];
        lmaxs[i] = s_sg[e + 2 * K + i];
      }
    }
    double r[PC + 3];
#pragma unroll
    for (int q = 0; q < RECN; ++q) r[q] = 0.0;
    const int n_src = wc.n_peers > 0 ? wc.n_peers : 1;
#pragma unroll 1
    for (int pr = 0; pr < n_src; ++pr) {
      const double* base = wc.n_peers > 0 ? wc.peer_rec[pr] : wv.rec;
#pragma unroll 1
      for (int s = 0; s < (MULTI ? (int)((n_c + wc.rows_per_split - 1) / wc.rows_per_split) : ws.S); ++s) {
        const double* src = base + (((size_t)c * ws.S + s) * W + sl) * RECN;
#pragma unroll
        for (int q = 0; q < RECN; ++q) {
          const double x = src[q];
          r[q] = (q < K + 3) ? r[q] + x : (r[q] > x ? r[q] : x);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < K; ++i) lsums[gram_idx(P1, i, K)] = r[i];
    lsums[gram_idx(P1, K, K)] = r[K + 1];
    lsums[ng + K] = r[K];
    lsums[ng + P1 + K] = r[K + 2];
    lmaxs[K] = r[K + 3];
    if (!(fabs(r[K + 1]) <= DBL_MAX) || !(r[K + 3] <= DBL_MAX)) lmaxs[K] = INFINITY;   // non-finite column

    int idx[BSR_MAXK];
    double beta[BSR_LDA];
    bool finite_cols = true;
    for (int j = 0; j < K; ++j) { idx[j] = (j == k) ? K : j; finite_cols = finite_cols && (gv.mx(idx[j]) <= DBL_MAX); }
    if (!finite_cols || rank_deficient<LD>(gv, idx, K, MULTI ? (double)n_c : wc.n_total, wc.pivot_tol, dg)) {
      rank_rej = true;                                                         // funcs.py:1226-1228: no accept draw
    } else {
      sse_new = MULTI ? ridge_sse<LD, false>(gv, idx, K, (double)n_c, wc.ystats[2 * (size_t)st.ds[c]], wc.ystats[2 * (size_t)st.ds[c] + 1], beta)
                      : ridge_sse<LD, false>(gv, idx, K, wc.n_total, wc.sum_y, wc.yy, beta);
      const double ns = pi.new_sigma;
      const double yll_new = -sse_new / (2 * ns * ns) - 0.5 * (MULTI ? (double)n_c : wc.n_total) * log(2 * 3.141592653589793 * ns * ns);
      const double yll_old = -sse_old / (2 * sigma * sigma) - 0.5 * (MULTI ? (double)n_c : wc.n_total) * log(2 * 3.141592653589793 * sigma * sigma);
      const double qr = pi.Qinv / pi.Q;
      logR = (yll_new - yll_old) + (pi.fs_old - prop_fs_new(pi)) + log(qr > 1e-5 ? qr : 1e-5);
      if (pi.change != CH_NONE)
        logR += log(pi.hratio > 1e-5 ? pi.hratio : 1e-5) + log(pi.detjacob > 1e-5 ? pi.detjacob : 1e-5);
      logR = logR + log_ig4_pdf(ns) - log_ig4_pdf(sigma);
      const double alpha = (0.0 < logR) ? 0.0 : logR;                          // python min(logR, 0): NaN stays NaN (Q14)
      if (wc.tape != nullptr) {            // the value behind the proposal's own draws (funcs.py:1299)
        const long long ti = p - wc.trace_origin;
        u = 0.5;
        if (ti >= 0 && ti < wc.trace_steps) {
          const int64_t lo = wc.tape_off[(size_t)c * wc.trace_steps + ti] + pi.ndraws, hi = wc.tape_off[(size_t)c * wc.trace_steps + ti + 1];
          if (lo < hi) u = wc.tape[lo];
        }
      } else {
        Draws<0> dr;
        dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)p, 2u);
        u = dr.u01();
      }
      accepted = !(log(u) >= alpha);                                           // funcs.py:1300
    }
  }

  // ---- phase B: consume the window in order ----
  const unsigned FULL = 0xffffffffu;
  unsigned long long valid_mask = __ballot_sync(FULL, valid);
  unsigned long long acc_mask = __ballot_sync(FULL, accepted);
  unsigned long long rank_mask = __ballot_sync(FULL, rank_rej);
  unsigned long long cap_mask = __ballot_sync(FULL, cap);
  if (LPC == 64) {   // the chain's two warps exchange their ballots
    if (lane == 0) {
      s_bal[half * 4 + 0] = (unsigned)valid_mask; s_bal[half * 4 + 1] = (unsigned)acc_mask;
      s_bal[half * 4 + 2] = (unsigned)rank_mask; s_bal[half * 4 + 3] = (unsigned)cap_mask;
    }
    __syncthreads();
    valid_mask = (unsigned long long)s_bal[0] | ((unsigned long long)s_bal[4] << 32);
    acc_mask = (unsigned long long)s_bal[1] | ((unsigned long long)s_bal[5] << 32);
    rank_mask = (unsigned long long)s_bal[2] | ((unsigned long long)s_bal[6] << 32);
    cap_mask = (unsigned long long)s_bal[3] | ((unsigned long long)s_bal[7] << 32);
    if (!live) return;
  }
  int total = st.total[c];
  const int stop_rule = PRIORS ? chain_stop[c] : 0;
  const int val = PRIORS ? (stop_rule & 0x7fffffff) : st.val;
  int n_cons = 0, a = -1;
  bool done = false;
  {
    // consumed = leading valid slots up to and including the first accept ...
    const unsigned long long inval = ~valid_mask;
    const int n_valid = inval ? (__ffsll((long long)inval) - 1) : 64;
    const unsigned long long first_acc = acc_mask & ((n_valid >= 64) ? ~0ull : ((1ull << n_valid) - 1ull));
    n_cons = first_acc ? __ffsll((long long)first_acc) : n_valid;
    if (first_acc) a = n_cons - 1;
    // ... or up to the sweep boundary at which `total` consecutive rejections reach val (bsr_class.py:174)
    if (val > 0) {
      const int k0 = (int)(p0 % K);
      int need = val - total;                         // rejections still missing
      if (need < 1) need = 1;
      int stop = need + ((K - (k0 + need) % K) % K);  // first slot count >= need that ends a sweep
      if (stop <= n_cons - (a >= 0 ? 1 : 0)) { n_cons = stop; a = -1; done = true; }
    }
    total += n_cons;
  }
  if (n_cons == 0) return;
  const unsigned long long cons = (n_cons >= 64) ? ~0ull : ((1ull << n_cons) - 1ull);
  const bool consumed = (cons >> sl) & 1ull;

  if (wc.trace != nullptr && consumed) {
    const long long ti = p - wc.trace_origin;
    if (ti >= 0 && ti < wc.trace_steps) {
      double* tr = wc.trace + ((size_t)c * wc.trace_steps + ti) * BSR_TRACE_DOUBLES;
      tr[BSR_TR_MOVE] = pi.move; tr[BSR_TR_CHANGE] = pi.change; tr[BSR_TR_Q] = pi.Q; tr[BSR_TR_QINV] = pi.Qinv;
      tr[BSR_TR_HRATIO] = pi.hratio; tr[BSR_TR_DETJACOB] = pi.detjacob; tr[BSR_TR_NEW_SIGMA] = pi.new_sigma;
      tr[BSR_TR_NEW_SA2] = pi.new_sa2; tr[BSR_TR_NEW_SB2] = pi.new_sb2; tr[BSR_TR_RANK_REJECT] = rank_rej;
      tr[BSR_TR_LOGR] = logR; tr[BSR_TR_ACCEPTED] = accepted; tr[BSR_TR_SSE_NEW] = sse_new; tr[BSR_TR_SSE_OLD] = sse_old;
      tr[BSR_TR_NDRAWS] = pi.ndraws + (cap || rank_rej ? 0 : 1); tr[BSR_TR_FLAGS] = pi.flags;
      tr[BSR_TR_U] = u; tr[BSR_TR_FS_NEW] = prop_fs_new(pi); tr[BSR_TR_FS_OLD] = pi.fs_old; tr[BSR_TR_M_NEW] = pi.m_new;
      tr[BSR_TR_PIVOT_MIN] = dg.pivot_min; tr[BSR_TR_SV_RATIO] = dg.sv_ratio; tr[BSR_TR_RANK_PATH] = dg.path;
      tr[BSR_TR_WIDE] = (double)((badmask >> sl) & 1ull);
      if (wc.log_tok != nullptr) {           // the proposed tree itself (tests compare it bit for bit with the reference's)
        const size_t lo = ((size_t)c * wc.trace_steps + ti) * BSR_MAXN, src = wi * BSR_MAXN;
        const int m = cap ? 0 : wv.nn[wi];
        wc.log_nn[(size_t)c * wc.trace_steps + ti] = m;
#pragma unroll 1
        for (int t = 0; t < m; ++t) { wc.log_tok[lo + t] = wv.tok[src + t]; wc.log_pa[lo + t] = wv.pa[src + t]; wc.log_pb[lo + t] = wv.pb[src + t]; }
      }
    }
  }

  // node-evaluation counters: summed per warp, added atomically (the chain may span two warps)
  long long ev_ref = (consumed && !cap) ? (long long)(pi.m_new + msum) : 0;          // n (m_new + m_old + sum_{i != j} m_i)
  long long ev_exec = (valid && !cap && ws.rep[(size_t)c * W + sl] == sl) ? (long long)pi.m_new * (((badmask >> sl) & 1ull) ? 2 : 1) : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ev_ref += __shfl_xor_sync(FULL, ev_ref, o);
    ev_exec += __shfl_xor_sync(FULL, ev_exec, o);
  }
  (void)m_old_k;
  long long* cnt = st.counters + (size_t)c * BSR_N_COUNTERS;
  if (lane == 0) {
    if (half == 0) ev_exec += msum;                 // the live columns, once per window
    atomicAdd(reinterpret_cast<unsigned long long*>(cnt + BSR_CNT_NODE_EVALS_REF), (unsigned long long)(ev_ref * (MULTI ? (long long)n_c : (long long)wc.n_local)));
    atomicAdd(reinterpret_cast<unsigned long long*>(cnt + BSR_CNT_NODE_EVALS_EXEC), (unsigned long long)(ev_exec * (MULTI ? (long long)n_c : (long long)wc.n_local)));
  }

  // everything else is written by the warp that holds the accepting slot (or by the chain's first warp)
  const int wwarp = (a >= 0) ? (a >> 5) : 0;
  if (half != wwarp) return;
  int plateau_done = 0;
  if (a >= 0) {
    const int ka = (int)((p0 + a) % K);
    const int g = c * K + ka;
    const int prev = st.which[g];
    const int nb = prev ^ 1;
    const size_t src = ((size_t)c * W + a) * BSR_MAXN, dst = (size_t)g * BSR_MAXN;
    const int m = wv.nn[(size_t)c * W + a];
    for (int t = lane; t < m; t += 32) {
      st.tok[nb][dst + t] = wv.tok[src + t];
      st.pa[nb][dst + t] = wv.pa[src + t];
      st.pb[nb][dst + t] = wv.pb[src + t];
    }
    if (sl == a) {
      st.nn[nb][g] = m;
      st.which[g] = nb;                          // the proposal becomes the live tree
      st.sigma[c] = pi.new_sigma;
      st.sa[g] = pi.new_sa2;                     // bsr_class.py:197-198 (on reject the old values stay)
      st.sb[g] = pi.new_sb2;
      st.sse[c] = sse_new;
      st.live_bad[g] = (unsigned char)((badmask >> a) & 1ull);
      st.lfs[2 * (size_t)g] = pi.ll_new; st.lfs[2 * (size_t)g + 1] = pi.lp_new;     // fStruc of the new live tree (its sigma_a, sigma_b are the proposal's)
      st.lcnt[g] = live_counts(wv.tok + src, m);
      int cur[BSR_MAXK];
      for (int j = 0; j < K; ++j) cur[j] = (j == ka) ? K : j;
      store_live_gram(gv, cur, K, st.sg + (size_t)c * sgn);
      // intercept refit + RMSE (bsr_class.py:211-233)
      double beta[BSR_LDA];
      const double sse_i = MULTI ? ridge_sse<LD, true>(gv, cur, K, (double)n_c, wc.ystats[2 * (size_t)st.ds[c]], wc.ystats[2 * (size_t)st.ds[c] + 1], beta)
                                 : ridge_sse<LD, true>(gv, cur, K, wc.n_total, wc.sum_y, wc.yy, beta);
      for (int j = 0; j <= K; ++j) st.beta[(size_t)c * (K + 1) + j] = beta[j];
      const double rmse = sqrt(sse_i / (MULTI ? (double)n_c : wc.n_total));
      int nerr = st.nerr[c];
      double* e = st.err + (size_t)c * st.err_cap;
      if (nerr < st.err_cap) e[nerr] = rmse;
      else {   // keep the newest err_cap entries
#pragma unroll 1
        for (int j = 1; j < st.err_cap; ++j) e[j - 1] = e[j];
        e[st.err_cap - 1] = rmse;
      }
      ++nerr;
      st.nerr[c] = nerr;
      // plateau rule (bsr_class.py:248-252): len(errList) > 100 and 1 - min(last10)/mean(last10) < 0.05
      if ((PRIORS ? stop_rule < 0 : st.plateau_rule != 0) && nerr > 100) {
        const int have = nerr < st.err_cap ? nerr : st.err_cap;
        const int k10 = have < 10 ? have : 10;
        double mn = DBL_MAX, sm = 0.0;
#pragma unroll 1
        for (int j = have - k10; j < have; ++j) { mn = fmin(mn, e[j]); sm += e[j]; }
        if (1.0 - mn / (sm / k10) < 0.05) plateau_done = 1;
      }
      for (int j = 0; j < K; ++j) st.report_which[c * K + j] = (j == ka) ? nb : st.which[c * K + j];
      if (plateau_done) st.report_which[g] = prev;   // ROOTS gets the pre-accept snapshot, BETAS the new Beta (Q16)
    }
    plateau_done = __shfl_sync(FULL, plateau_done, a & 31);
    total = 0;
  }
  if (lane == 0) {
    cnt[BSR_CNT_PROPOSALS] += n_cons;
    cnt[BSR_CNT_ACCEPTS] += (a >= 0) ? 1 : 0;
    cnt[BSR_CNT_RANK_REJECTS] += __popcll(rank_mask & cons);
    cnt[BSR_CNT_CAPACITY_REJECTS] += __popcll(cap_mask & cons);
    cnt[BSR_CNT_FP64_SWEEPS] += __popcll(badmask & cons & ~cap_mask);
    cnt[BSR_CNT_SWEEPS] += (p0 + n_cons) / K - p0 / K;
    if (a < 0) for (int j = 0; j < K; ++j) st.report_which[c * K + j] = st.which[c * K + j];
    st.total[c] = total;
    if (done || plateau_done) st.done[c] = 1;
    ws.pos[c] = p0 + n_cons;
    // cache of live columns: a column interpreted (and written) by this window's k_weval is the live tree's from now on -- unless it
    // had an out-of-range vector, or the tree was just replaced
    if (ws.lcol_ok != nullptr) {
      const unsigned widem = ws.lcol_wide[c];
      const bool computed = ws.neval[c] > 0;
      const int ka = (a >= 0) ? (int)((p0 + a) % K) : -1;
      for (int j = 0; j < K; ++j) {
        if (j == ka) ws.lcol_ok[c * K + j] = 0;
        else if (computed && !((widem >> j) & 1u)) ws.lcol_ok[c * K + j] = 1;
      }
    }
    // the window stays valid as a record cache for the next one unless the live state just changed (or the records live in the
    // exchange buffer of a row-sharded handle, which has its own double buffering)
    if (a >= 0 || wc.n_peers > 0) { ws.chead[c] = (signed char)-1; ws.cvalid[c] = 0; }
    else {
      const int nv = (ws.chead[c] >= 0) ? (int)ws.cvalid[c] + 1 : 1;
      ws.chead[c] = (signed char)wpar;
      ws.cvalid[c] = (unsigned char)(nv < ws.R - 1 ? nv : ws.R - 1);
    }
  }
}
