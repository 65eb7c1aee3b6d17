// __global__ kernels of the split (three-phase) sweep pipeline:
//   k_init_chains  prior initialisation                         codes/bsr_class.py:123-142
//   k_propose      Prop + auxProp + fStruc for K trees/chain    codes/funcs.py:1188-1210
//   k_eval         allcal of the 2K columns + Gram reductions   codes/funcs.py:1212-1224, 1147-1157
//   k_resolve      rank test, ylogLike, logR, accept, refit     codes/funcs.py:1226-1306, bsr_class.py:195-252
// (allcal / BSR.predict for arbitrary trees, k_eval_trees / k_predict_groups, are in bsr_misc_kernels.cuh)
#pragma once
#include "bsr_common.cuh"
#include "bsr_eval.cuh"
#include "bsr_propose.cuh"
#include "bsr_rng.cuh"
#include "bsr_solve.cuh"

struct ProposeCtx {
  int64_t sweep;
  const double* tape;
  const int64_t* tape_off;
  int steps, step_base;
  double* rec;        // [C][rec_steps][rec_cap] recorded draws (MODE 2)
  int* rec_count;     // [C][rec_steps]
  int rec_steps, rec_cap, rec_base;
  int c0, cn;         // chain range [c0, c0 + cn) handled by this launch
};

template <int MODE>
__global__ void k_init_chains(ChainState st, const PriorTables* __restrict__ ptp, const int* __restrict__ chain_pt) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= st.C * st.K) return;
  int c = g / st.K, k = g % st.K;
  const PriorTables& pt = ptp[chain_pt[c]];   // tables live in global memory: indexed divergently, and out-of-line callees take them by
                                              // reference; one per feature count, the chain's data set's
  Draws<MODE> dr;
  dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)k, 0u);
  size_t slot = (size_t)g * BSR_MAXN;
  double sa, sb;
  init_tree<MODE>(pt, dr, st.tok[0] + slot, st.pa[0] + slot, st.pb[0] + slot, st.nn[0] + g, sa, sb);
  st.sa[g] = sa; st.sb[g] = sb;
  st.which[g] = 0; st.report_which[g] = 0;
  st.nn[1][g] = 0;
  if (k == 0) {
    Draws<MODE> ds;
    ds.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)st.K, 0u);
    st.sigma[c] = ds.invgamma(1);                                             // bsr_class.py:123
  }
}

template <int MODE>
__global__ void k_propose(ChainState st, const PriorTables* __restrict__ ptp, ProposeCtx pc) {
  const PriorTables& pt = *ptp;
  int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= pc.cn * st.K) return;
  const int g = pc.c0 * st.K + gi;
  int c = g / st.K, k = g % st.K;
  if (st.done[c]) return;
  Draws<MODE> dr;
  dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)(pc.sweep * st.K + k), 1u);
  if (MODE == 1) {
    size_t s = (size_t)c * pc.steps + pc.step_base + k;
    dr.init_tape(pc.tape, (int)pc.tape_off[s], (int)pc.tape_off[s + 1]);
  }
  if (MODE == 2 && pc.rec != nullptr && pc.rec_base + k < pc.rec_steps)
    dr.init_record(pc.rec + ((size_t)c * pc.rec_steps + pc.rec_base + k) * pc.rec_cap, pc.rec_cap);
  const int w = st.which[g];
  const size_t slot = (size_t)g * BSR_MAXN;
  PropInfo info;
  propose_one<MODE>(pt, st.tok[w] + slot, st.pa[w] + slot, st.pb[w] + slot, st.nn[w][g], st.sa[g], st.sb[g], dr,
                    st.tok[w ^ 1] + slot, st.pa[w ^ 1] + slot, st.pb[w ^ 1] + slot, st.nn[w ^ 1] + g, info);
  st.pinfo[g] = info;
  if (MODE == 2 && pc.rec != nullptr && pc.rec_base + k < pc.rec_steps)
    pc.rec_count[(size_t)c * pc.rec_steps + pc.rec_base + k] = dr.pos;
}

struct EvalCtx {
  const float* X32; const float* y32;     // column-major [d][ld], [n]
  const double* X64; const double* y64;
  uint32_t n;        // rows on this device
  uint32_t ld;       // leading dimension (multiple of 4)
  double* sums;      // [C][n_sum]
  double* maxs;      // [C][P]
  int precision;     // 0: fp32 evaluation, fp64 re-evaluation when a column leaves the fp32 range; 1: fp64
  int init_only;     // evaluate the K live trees only
  int tpc;           // threads per chain: 32 (warp per chain) or blockDim.x (block per chain)
  int c0, cn;        // chain range [c0, c0 + cn) handled by this launch
  int fill_cache;    // evaluate everything and (re)fill the column cache (initial fit / data changed)
  int* need64;       // [C] set by the fp32 pass for chains that need the fp64 pass
  // row splits (block-per-chain mode only): blockIdx.y = split; each block reduces its rows into part[c][split], the
  // last block to finish a chain sums the partials in split order (deterministic) and finalises the record
  int n_splits;
  double* part;      // [C][n_splits][n_sum + P]
  int* split_cnt;    // [C] arrival counters (self-resetting)
};

// Shared-memory footprint: per chain group the pre-decoded tokens of the P trees (sized for double parameters so
// the fp64 re-evaluation can re-stage in place), per block the column staging vectors and the reduction scratch.
__host__ __device__ inline size_t eval_group_bytes(int P) {
  size_t b = (size_t)P * BSR_MAXN * sizeof(EvTok<double>) + (size_t)(P + (P & 1)) * sizeof(int) + (size_t)P * sizeof(void*);
  return (b + 15) / 16 * 16;
}
__host__ __device__ inline size_t eval_smem_bytes(int P, int threads, int tpc) {
  const int groups = threads / tpc;
  const size_t cv = (size_t)P * threads * 16;
  const size_t red = (tpc > 32) ? (size_t)(threads / 32) * (gram_n_sum(P) + P) * sizeof(double) + 16 : 0;   // + flag word
  return groups * eval_group_bytes(P) + cv + red + 64;
}

// Stage the P = 2K trees of chain c (K live trees, then the K proposals) as pre-decoded tokens of type T.
template <typename T>
__device__ __forceinline__ void stage_trees(const ChainState& st, int c, int K, int init_only, int lane, int tpc, uint32_t ld,
                                            EvTok<T>* s_tok, int* s_m) {
  const int P = 2 * K;
  for (int p = 0; p < P; ++p) {
    const int k = (p < K) ? p : p - K;
    const int g = c * K + k;
    const int w = st.which[g] ^ (p < K ? 0 : 1);
    int m = st.nn[w][g];
    if (p >= K && (init_only || (st.pinfo[g].flags & PF_CAPACITY))) m = 0;
    if (lane == 0) s_m[p] = m;
    const size_t slot = (size_t)g * BSR_MAXN;
    for (int j = lane; j < m; j += tpc) {
      const uint32_t t = st.tok[w][slot + j];
      EvTok<T> e;
      e.op = tok_op(t);
      e.off = (uint32_t)tok_ft(t) * ld;
      e.a = (T)st.pa[w][slot + j];
      e.b = (T)st.pb[w][slot + j];
      s_tok[p * BSR_MAXN + j] = e;
    }
  }
}

// Generic-K accumulation (K > 5): same interpreter, accumulators in local memory.
template <typename T>
__device__ __noinline__ void eval_chain_rows_generic(double* genG, double* genY, double* genS, double* genM, int P,
                                                     const EvTok<T>* s_tok, const int* s_m, typename RowVec<T>::V* my_cv, int cvs,
                                                     const T* __restrict__ X, const double* __restrict__ y, uint32_t n, uint32_t v0,
                                                     uint32_t v1, int lane, int tpc) {
  constexpr int R = RowVec<T>::R;
  typedef typename RowVec<T>::V V;
  for (uint32_t q = v0 + lane; q < v1; q += tpc) {
    const uint32_t row0 = q * R;
    for (int p = 0; p < P; ++p) {
      T v[R];
      const int m = s_m[p];
      if (m > 0) eval_tree_rows<T, R>(s_tok + p * BSR_MAXN, m, X, row0, v);
      else {
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = (T)0;
      }
      V pack;
#pragma unroll
      for (int r = 0; r < R; ++r) ((T*)&pack)[r] = v[r];
      my_cv[p * cvs] = pack;
    }
    for (int r = 0; r < R; ++r) {
      if (row0 + r >= n) continue;
      const double yr = __ldg(y + row0 + r);
      int k = 0;
      for (int i = 0; i < P; ++i) {
        const double vi = (double)((const T*)&my_cv[i * cvs])[r];
        for (int j = i; j < P; ++j) { genG[k] = fma(vi, (double)((const T*)&my_cv[j * cvs])[r], genG[k]); ++k; }
        genY[i] = fma(vi, yr, genY[i]);
        genS[i] += vi;
        genM[i] = fmax(genM[i], fabs(vi));
      }
    }
  }
}

// One evaluation pass in type T for the chain of this thread group; the record lands in out_rec[0 .. n_sum + P).
// Returns (to every thread of the group) the bit mask of columns with non-finite values.
// is_last: false for the blocks of a row-split chain that are not the last to finish (they are done).
// LOADALL: the columns were already written to the cache by k_trees; this pass only builds the Gram record.
template <typename T, int KT, int CM, bool LOADALL = false>
__device__ __forceinline__ unsigned eval_pass(const ChainState& st, const EvalCtx& ec, int c, int K, int lane, int tpc,
                                              unsigned char* gbase, unsigned char* cv_base, double* s_red, double* out_rec,
                                              const T* X, const double* y, bool& is_last) {
  typedef typename RowVec<T>::V V;
  const int P = 2 * K;
  const bool block_mode = tpc > 32;
  is_last = true;
  const int S = block_mode ? ec.n_splits : 1;
  const int split = block_mode ? (int)blockIdx.y : 0;
  const uint32_t n_vec = (ec.n + RowVec<T>::R - 1) / RowVec<T>::R;
  const uint32_t v_per = (n_vec + S - 1) / S;
  const uint32_t v0 = min(n_vec, (uint32_t)split * v_per), v1 = min(n_vec, v0 + v_per);
  EvTok<T>* s_tok = reinterpret_cast<EvTok<T>*>(gbase);
  int* s_m = reinterpret_cast<int*>(gbase + (size_t)P * BSR_MAXN * sizeof(EvTok<double>));
  V* my_cv = reinterpret_cast<V*>(cv_base) + threadIdx.x;
  const int cvs = blockDim.x;
  if (LOADALL) {
    if (lane < P) {
      const int k = (lane < K) ? lane : lane - K;
      const int g = c * K + k;
      int m = st.nn[st.which[g] ^ (lane < K ? 0 : 1)][g];
      if (lane >= K && (ec.init_only || (st.pinfo[g].flags & PF_CAPACITY))) m = 0;
      s_m[lane] = m;
    }
  } else {
    stage_trees<T>(st, c, K, ec.init_only, lane, tpc, ec.ld, s_tok, s_m);
  }
  if (block_mode) __syncthreads(); else __syncwarp();

  const int n_sum = gram_n_sum(P), nacc = n_sum + P;
  const int wlane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* dst = block_mode ? (s_red + (size_t)wid * nacc) : out_rec;
  if (KT > 0) {
    constexpr int PC = (KT > 0) ? 2 * KT : 2;
    GramAcc<T, PC> ga;
    ga.zero();
    T** s_cp = reinterpret_cast<T**>(gbase + (size_t)P * BSR_MAXN * sizeof(EvTok<double>) + (size_t)(P + (P & 1)) * sizeof(int));
    unsigned badmask = 0;
    if (CM != CM_PLAIN) {
      // per-slot cache columns (always fp32): the live / spare buffer of slot k is chosen by which[c][k]
      float** s_cpf = reinterpret_cast<float**>(s_cp);
      if (lane < K) {
        const int g = c * K + lane;
        const int w = st.which[g];
        s_cpf[lane] = st.col[w] + (size_t)g * st.col_ld;
        s_cpf[K + lane] = st.col[w ^ 1] + (size_t)g * st.col_ld;
      }
      if (CM == CM_MIXED)
        for (int k = 0; k < K; ++k)
          badmask |= (st.live_bad[c * K + k] ? (1u << k) : 0u) | (st.prop_bad[c * K + k] ? (1u << (K + k)) : 0u);
      if (block_mode) __syncthreads(); else __syncwarp();
    }
    eval_chain_rows<T, PC, CM, LOADALL>(ga, s_tok, s_m, my_cv, cvs, X, y, ec.n, v0, v1, lane, tpc, s_cp, badmask);
    warp_reduce_store<T, PC, CM>(ga, dst, wlane);
  } else {
    double genG[(2 * BSR_MAXK) * (2 * BSR_MAXK + 1) / 2], genY[2 * BSR_MAXK], genS[2 * BSR_MAXK], genM[2 * BSR_MAXK];
    for (int i = 0; i < P * (P + 1) / 2; ++i) genG[i] = 0.0;
    for (int i = 0; i < P; ++i) { genY[i] = 0.0; genS[i] = 0.0; genM[i] = 0.0; }
    eval_chain_rows_generic<T>(genG, genY, genS, genM, P, s_tok, s_m, my_cv, cvs, X, y, ec.n, v0, v1, lane, tpc);
    const int ng = P * (P + 1) / 2;
    for (int i = 0; i < nacc; ++i) {
      const double a = i < ng ? genG[i] : (i < ng + P ? genY[i - ng] : (i < ng + 2 * P ? genS[i - ng - P] : genM[i - ng - 2 * P]));
      const double v = (i < n_sum) ? warp_sum(a) : warp_max<double>(a);
      if (wlane == 0) dst[i] = v;
    }
  }
  unsigned bad = 0;
  const int p0 = (CM == CM_CACHED) ? K : 0;     // cached live columns are known to be in range
  if (block_mode) {
    __syncthreads();
    const int nw = blockDim.x >> 5;
    double* blk_rec = (S > 1) ? (ec.part + ((size_t)c * S + split) * nacc) : out_rec;
    for (int i = threadIdx.x; i < nacc; i += blockDim.x) {
      double v = 0.0;
      for (int w = 0; w < nw; ++w) {
        const double x = s_red[(size_t)w * nacc + i];
        v = (i < n_sum) ? v + x : fmax(v, x);
      }
      blk_rec[i] = v;
    }
    unsigned* s_flag = reinterpret_cast<unsigned*>(s_red + (size_t)nw * nacc);
    if (S > 1) {
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) *s_flag = (unsigned)atomicAdd(ec.split_cnt + c, 1);
      __syncthreads();
      if (*s_flag != (unsigned)(S - 1)) { is_last = false; return 0; }
      __threadfence();
      if (threadIdx.x == 0) ec.split_cnt[c] = 0;
      const double* pc = ec.part + (size_t)c * S * nacc;
      for (int i = threadIdx.x; i < nacc; i += blockDim.x) {
        double v = 0.0;
        for (int sp = 0; sp < S; ++sp) {
          const double x = __ldcg(pc + (size_t)sp * nacc + i);
          v = (i < n_sum) ? v + x : fmax(v, x);
        }
        out_rec[i] = v;
      }
    }
    __syncthreads();
    if (CM == CM_CACHED) sg_to_record(st.sg + (size_t)c * sg_size(K), out_rec, K, threadIdx.x, blockDim.x);
    __syncthreads();
    if (threadIdx.x == 0) *s_flag = mark_bad_columns(out_rec, out_rec + n_sum, P, p0);
    __syncthreads();
    bad = *s_flag;
  } else {
    if (CM == CM_CACHED) { __syncwarp(); sg_to_record(st.sg + (size_t)c * sg_size(K), out_rec, K, wlane, 32); __syncwarp(); }
    if (wlane == 0) bad = mark_bad_columns(out_rec, out_rec + n_sum, P, p0);
    bad = __shfl_sync(0xffffffffu, bad, 0);
  }
  return bad;
}

// Tree evaluation alone (allcal, codes/funcs.py:175-220): one warp per (chain, tree) interprets its tree on all local
// rows and writes the fp32 column into the column cache; no reductions, so the kernel is small and runs at high
// occupancy.  In steady state only the K proposals of a chain are evaluated (into the spare buffer of their slot); in
// fill mode (initial fit, data changed) the K live trees are evaluated too.  k_eval<..., LOADALL> then builds the
// Gram record from the cached columns.
static __global__ void __launch_bounds__(128) k_trees(ChainState st, EvalCtx ec) {
  __shared__ EvTok<float> s_tok[4][BSR_MAXN];
  const int K = st.K;
  const int per_chain = ec.fill_cache ? 2 * K : K;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * (blockDim.x >> 5) + wid;
  if (item >= ec.cn * per_chain) return;
  const int c = ec.c0 + item / per_chain;
  const int t = item % per_chain;
  const bool live = ec.fill_cache && t < K;
  const int k = live ? t : (ec.fill_cache ? t - K : t);
  if (!ec.init_only && st.done[c]) return;
  if (!live && ec.init_only) return;                      // no proposals exist yet
  const int g = c * K + k;
  const int w = st.which[g] ^ (live ? 0 : 1);
  if (!live && (st.pinfo[g].flags & PF_CAPACITY)) return;
  const int m = st.nn[w][g];
  const size_t slot = (size_t)g * BSR_MAXN;
  for (int j = lane; j < m; j += 32) {
    const uint32_t tk = st.tok[w][slot + j];
    EvTok<float> e;
    e.op = tok_op(tk); e.off = (uint32_t)tok_ft(tk) * ec.ld;
    e.a = (float)st.pa[w][slot + j]; e.b = (float)st.pb[w][slot + j];
    s_tok[wid][j] = e;
  }
  __syncwarp();
  float* dst = st.col[w] + (size_t)g * st.col_ld;
  const uint32_t n_vec = (ec.n + 3) / 4;
#pragma unroll 1
  for (uint32_t q = lane; q < n_vec; q += 32) {
    float v[4];
    eval_tree_rows<float, 4>(s_tok[wid], m, ec.X32, q * 4, v);
    *reinterpret_cast<float4*>(dst + q * 4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// allcal of the 2K columns of every chain + Gram reductions (codes/funcs.py:1212-1224, 1147-1157).
// PASS 0: the fp32 pass (column cache, SFU transcendentals).  A chain with an out-of-range column (live or proposed)
//         is flagged in need64 instead of being evaluated / trusted.
// PASS 1: the fp64 pass: all chains when precision == fp64, else only the chains flagged by PASS 0 (launched right
//         after it with fatter blocks, since few chains are flagged and their latency is what matters).
template <int KT, int PASS, int CM, bool LOADALL = false>
__global__ void __launch_bounds__(256) k_eval(ChainState st, EvalCtx ec) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = (KT > 0) ? KT : st.K;
  const int P = 2 * K;
  const int tpc = ec.tpc;
  const int groups = blockDim.x / tpc;
  const int grp = threadIdx.x / tpc;
  const int lane = threadIdx.x % tpc;       // index inside the chain group
  const int ci = blockIdx.x * groups + grp;
  if (ci >= ec.cn) return;                  // whole group exits together (a warp, or the block in block mode)
  const int c = ec.c0 + ci;
  if (!ec.init_only && st.done[c]) return;
  bool live_bad = false;
  if (ec.precision == 0 && !ec.fill_cache)
    for (int k = 0; k < K; ++k) live_bad = live_bad || st.live_bad[c * K + k];
  if (PASS == 1 && ec.precision == 0 && !ec.need64[c]) return;

  unsigned char* gbase = smem_raw + (size_t)grp * eval_group_bytes(P);
  unsigned char* cv_base = smem_raw + (size_t)groups * eval_group_bytes(P);
  double* s_red = reinterpret_cast<double*>(cv_base + (size_t)P * blockDim.x * 16);
  const int n_sum = gram_n_sum(P);
  double* out_s = ec.sums + (size_t)c * n_sum;
  double* out_m = ec.maxs + (size_t)c * P;
  // eval_pass writes [sums | maxs] contiguously into a scratch record behind the two arrays, then it is split
  double* rec = ec.sums + (size_t)st.C * n_sum + (size_t)st.C * P + (size_t)c * (n_sum + P);

  unsigned bad = 0;
  if (PASS == 0) {
    // chains with an out-of-range live column still run this pass: it tells which *proposal* columns are in range
    // (new diagonal); the record itself is then rebuilt by the fp64 pass
    bool is_last;
    bad = eval_pass<float, KT, CM, LOADALL>(st, ec, c, K, lane, tpc, gbase, cv_base, s_red, rec, ec.X32, ec.y64, is_last);
    if (!is_last) return;
    if (lane == 0) {
      for (int k = 0; k < K; ++k) {
        st.prop_bad[c * K + k] = (unsigned char)((bad >> (K + k)) & 1u);
        if (ec.fill_cache) st.live_bad[c * K + k] = (unsigned char)((bad >> k) & 1u);
      }
      if (bad || live_bad) ec.need64[c] = 1;
    }
    if (bad || live_bad) return;            // the fp64 pass will produce this chain's record
  } else {
    bool is_last;
    bad = eval_pass<double, KT, CM>(st, ec, c, K, lane, tpc, gbase, cv_base, s_red, rec, ec.X64, ec.y64, is_last);
    if (!is_last) return;
    if (lane == 0 && ec.precision == 0) {
      ec.need64[c] = 0;
      if (!ec.init_only) st.counters[(size_t)c * BSR_N_COUNTERS + BSR_CNT_FP64_SWEEPS] += 1;
    }
  }
  if (tpc > 32) __syncthreads(); else __syncwarp();
  for (int i = lane; i < n_sum + P; i += tpc) {
    const double v = rec[i];
    if (i < n_sum) out_s[i] = v; else out_m[i - n_sum] = v;
  }
}

// KP lanes per chain (KP = K rounded up to a power of two): lane j < K of a chain first runs the expensive,
// state-independent part of proposal j (rank test + ridge SSE against the unchanged live set) in parallel with its
// siblings, then lane 0 replays the reference's sequential accept logic for the chain.  The Gram records and
// PropInfo of the block's chains are first copied to shared memory with coalesced loads, so the serial code never
// waits on global memory.
template <int MODE, int KT>
__global__ void k_resolve(ChainState st, ResolveCtx rc, const double* sums, const double* maxs, int init_only, int KP) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = (KT > 0) ? KT : st.K;
  const int P = 2 * K, n_sum = gram_n_sum(P);
  const int cpb = blockDim.x / KP;                    // chains per block
  const int cb = blockIdx.x * cpb;                    // first chain (relative) of this block
  const int nb = min(cpb, rc.cn - cb);                // chains in this block
  if (nb <= 0) return;
  double* s_sums = reinterpret_cast<double*>(smem_raw);
  double* s_maxs = s_sums + (size_t)cpb * n_sum;
  PropInfo* s_pi = reinterpret_cast<PropInfo*>(s_maxs + (size_t)cpb * P);
  const size_t c_first = (size_t)(rc.c0 + cb);
  for (int i = threadIdx.x; i < nb * n_sum; i += blockDim.x) s_sums[i] = sums[c_first * n_sum + i];
  for (int i = threadIdx.x; i < nb * P; i += blockDim.x) s_maxs[i] = maxs[c_first * P + i];
  {
    const int words = nb * K * (int)(sizeof(PropInfo) / 4);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(st.pinfo + c_first * K);
    uint32_t* dst = reinterpret_cast<uint32_t*>(s_pi);
    for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int ci = threadIdx.x / KP, j = threadIdx.x % KP;
  const bool chain_ok = ci < nb;
  const int c = rc.c0 + cb + (chain_ok ? ci : 0);
  const double* my_sums = s_sums + (size_t)(chain_ok ? ci : 0) * n_sum;
  const double* my_maxs = s_maxs + (size_t)(chain_ok ? ci : 0) * P;
  const PropInfo* my_pi = s_pi + (size_t)(chain_ok ? ci : 0) * K;
  // ---- phase A: lane j precomputes proposal j ----
  bool my_rank = false;
  double my_sse = nan("");
  const bool active = chain_ok && !init_only && !st.done[c];
  if (active && j < K) precompute_slot<KT>(rc, K, j, my_sums, my_maxs, my_pi[j], my_rank, my_sse);
  // ---- gather the K results of every chain on its lane 0 ----
  const int lane = threadIdx.x & 31;
  const int base = (lane / KP) * KP;
  unsigned pre_rank = 0;
  double pre_sse[(KT > 0) ? KT : BSR_MAXK];
#pragma unroll
  for (int k = 0; k < ((KT > 0) ? KT : BSR_MAXK); ++k) {
    if (k < K) {
      const int r = __shfl_sync(0xffffffffu, (int)my_rank, base + k);
      pre_sse[k] = __shfl_sync(0xffffffffu, my_sse, base + k);
      pre_rank |= (unsigned)(r & 1) << k;
    }
  }
  // ---- phase B: sequential accept logic on lane 0 of each chain ----
  if (!chain_ok || j != 0) return;
  resolve_chain<MODE, KT>(st, rc, c, my_sums, my_maxs, my_pi, init_only != 0, !init_only, pre_rank, pre_sse);
}

