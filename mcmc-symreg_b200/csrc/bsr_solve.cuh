// Per-chain fp64 linear algebra on the sweep Gram: rank test, ridge OLS, SSE, log-likelihood, logR and the
// Metropolis-Hastings accept, one thread per chain.
//
//   rank test      np.linalg.matrix_rank(new_outputs) < K            codes/funcs.py:1226-1228
//   ylogLike       scale by max|.|, ridge 1e-6, SSE, Gaussian ll      codes/funcs.py:1147-1174
//   logR + accept  codes/funcs.py:1230-1306
//   accept path    intercept refit, Beta/scale, RMSE, stop rules      codes/bsr_class.py:195-252
//
// The sweep Gram holds all 2K columns (K live trees followed by the K proposals of this sweep), so the K
// proposals of a sweep are resolved sequentially here from one pass over the rows: proposal k only needs the
// live state of the other slots, which the 2K x 2K Gram contains for every accept pattern.
#pragma once
#include "bsr_common.cuh"
#include "bsr_eval.cuh"
#include "bsr_rng.cuh"

#define BSR_LDA (BSR_MAXK + 1)
// full unrolling (matrices in registers) only when LD is a small compile-time K+1; LD is in scope at every use
#define BSR_UNROLL_LD _Pragma("unroll (LD <= 6 ? 32 : 1)")

struct GramView {
  const double* sums;   // G upper triangle, col.y, col sums
  const double* maxs;   // max|col| (+inf marks a non-finite column)
  int P;
  __device__ __forceinline__ double g(int i, int j) const { return i <= j ? sums[gram_idx(P, i, j)] : sums[gram_idx(P, j, i)]; }
  __device__ __forceinline__ double by(int i) const { return sums[P * (P + 1) / 2 + i]; }
  __device__ __forceinline__ double cs(int i) const { return sums[P * (P + 1) / 2 + P + i]; }
  __device__ __forceinline__ double mx(int i) const { return maxs[i]; }
};

// All small-matrix routines are templated on LD (leading dimension = compile-time bound of every loop): for the
// compile-time-K instantiations (K <= 5) the loops unroll completely and the matrices live in registers; the
// generic instantiation (LD = BSR_LDA) keeps them in local memory.

// In-place Cholesky A = L L^T (lower) of the leading q x q block, returns false on a non-positive / NaN pivot.
template <int LD>
__device__ __forceinline__ bool chol(double (&A)[LD][LD], int q) {
BSR_UNROLL_LD
  for (int j = 0; j < LD; ++j) {
    if (j < q) {
      double s = A[j][j];
BSR_UNROLL_LD
      for (int p = 0; p < j; ++p) s -= A[j][p] * A[j][p];
      if (!(s > 0.0)) return false;
      double d = sqrt(s);
      A[j][j] = d;
      const double id = 1.0 / d;
BSR_UNROLL_LD
      for (int i = j + 1; i < LD; ++i) {
        if (i < q) {
          double t = A[i][j];
BSR_UNROLL_LD
          for (int p = 0; p < j; ++p) t -= A[i][p] * A[j][p];
          A[i][j] = t * id;
        }
      }
    }
  }
  return true;
}
template <int LD>
__device__ __forceinline__ void chol_solve(const double (&A)[LD][LD], int q, double (&x)[LD]) {
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) {
    if (i < q) {
      double t = x[i];
BSR_UNROLL_LD
      for (int p = 0; p < i; ++p) t -= A[i][p] * x[p];
      x[i] = t / A[i][i];
    }
  }
BSR_UNROLL_LD
  for (int i = LD - 1; i >= 0; --i) {
    if (i < q) {
      double t = x[i];
BSR_UNROLL_LD
      for (int p = i + 1; p < LD; ++p) if (p < q) t -= A[p][i] * x[p];
      x[i] = t / A[i][i];
    }
  }
}

// Scaled ridge OLS on columns idx[0..k) of the Gram (optionally with a leading ones column):
//   XX = [1?, cols] / scale, scale = max|XX|;  beta = (XX'XX + 1e-6 I)^-1 XX'y;  sse = |y - XX beta|^2
// (codes/funcs.py:1148-1162, codes/bsr_class.py:216-227).  beta_out (k [+1] entries) is divided by scale, i.e. it
// applies to the un-scaled columns.  SSE is evaluated as the exact quadratic form in fp64.
template <int LD, bool INTERCEPT>
__device__ __noinline__ double ridge_sse(const GramView& gv, const int* idx, int k, double n_rows, double sum_y, double yy,
                                            double* beta_out) {
  double A[LD][LD], Gs[LD][LD], b[LD], x[LD];
  constexpr int o = INTERCEPT ? 1 : 0;
  const int q = k + o;
  double scale = INTERCEPT ? 1.0 : 0.0;
BSR_UNROLL_LD
  for (int i = 0; i < LD - 1; ++i) if (i < k) scale = fmax(scale, gv.mx(idx[i]));
  if (!(scale > 0.0) || !(scale <= DBL_MAX)) {
    for (int i = 0; i < q; ++i) beta_out[i] = nan("");
    return nan("");
  }
  const double is = 1.0 / scale, is2 = is * is;
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) {
BSR_UNROLL_LD
    for (int j = 0; j < LD; ++j) Gs[i][j] = 0.0;
    b[i] = 0.0;
  }
  if (INTERCEPT) {
    Gs[0][0] = n_rows * is2; b[0] = sum_y * is;
BSR_UNROLL_LD
    for (int i = 0; i < LD - 1; ++i) if (i < k) { Gs[0][i + 1] = Gs[i + 1][0] = gv.cs(idx[i]) * is2; }
  }
BSR_UNROLL_LD
  for (int i = 0; i < LD - o; ++i) {
    if (i < k) {
      b[i + o] = gv.by(idx[i]) * is;
BSR_UNROLL_LD
      for (int j = 0; j <= i; ++j) { double v = gv.g(idx[i], idx[j]) * is2; Gs[i + o][j + o] = v; Gs[j + o][i + o] = v; }
    }
  }
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) {
BSR_UNROLL_LD
    for (int j = 0; j < LD; ++j) A[i][j] = Gs[i][j];
    A[i][i] += 1e-6;
    x[i] = b[i];
  }
  if (!chol<LD>(A, q)) {
    for (int i = 0; i < q; ++i) beta_out[i] = nan("");
    return nan("");
  }
  chol_solve<LD>(A, q, x);
  double lin = 0.0, quad = 0.0;
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) {
    if (i < q) {
      lin += x[i] * b[i];
      double t = 0.0;
BSR_UNROLL_LD
      for (int j = 0; j < LD; ++j) if (j < q) t += Gs[i][j] * x[j];
      quad += x[i] * t;
    }
  }
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) if (i < q) beta_out[i] = x[i] * is;
  double sse = yy - 2.0 * lin + quad;
  return sse < 0.0 ? 0.0 : sse;
}

// What the rank test saw (trace rows / census): the smallest pivot of the column-scaled Gram (sin^2 of the angle between a
// column and the span of the columns before it), sigma_min / sigma_max when the Jacobi pass ran (else -1), and the path taken.
enum : int { RP_NONFINITE = 1, RP_PIVOT = 2, RP_BOUND_FULL = 3, RP_JACOBI_FULL = 4, RP_JACOBI_DEFICIENT = 5 };
struct RankDiag {
  double pivot_min, sv_ratio;
  int path;
};

// Singular values of the data block from B = L^T D by one-sided Jacobi; only reached for strongly graded columns.
template <int LD>
__device__ __noinline__ bool jacobi_rank_deficient(const double (&Lm)[LD][LD], const double (&d)[LD], int k, double tol, double& ratio) {
  double B[LD][LD];
  for (int i = 0; i < k; ++i)
    for (int j = 0; j < k; ++j) B[i][j] = (j >= i) ? Lm[j][i] * d[j] : 0.0;
  for (int sweep = 0; sweep < 40; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < k - 1; ++p)
      for (int q = p + 1; q < k; ++q) {
        double al = 0.0, be = 0.0, ga = 0.0;
        for (int i = 0; i < k; ++i) { al += B[i][p] * B[i][p]; be += B[i][q] * B[i][q]; ga += B[i][p] * B[i][q]; }
        if (fabs(ga) <= 1e-15 * sqrt(al * be) || ga == 0.0) continue;
        rotated = true;
        double zeta = (be - al) / (2.0 * ga);
        double t = (zeta >= 0.0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int i = 0; i < k; ++i) {
          double bp = B[i][p], bq = B[i][q];
          B[i][p] = c * bp - s * bq;
          B[i][q] = s * bp + c * bq;
        }
      }
    if (!rotated) break;
  }
  double smax = 0.0, smin = DBL_MAX;
  for (int j = 0; j < k; ++j) {
    double s2 = 0.0;
    for (int i = 0; i < k; ++i) s2 += B[i][j] * B[i][j];
    double s = sqrt(s2);
    smax = fmax(smax, s); smin = fmin(smin, s);
  }
  ratio = smin / smax;
  return !(smin > smax * tol);
}

// np.linalg.matrix_rank(new_outputs) < K on the n x k block whose Gram is G[idx, idx].
// numpy: rank = #{ sigma_i > sigma_max * max(n, k) * eps } -- a criterion on the UNSCALED columns, so a block with one huge
// column (exp(exp(.)), 1/sin(.) near a zero) is rank deficient by it however independent its columns are.  Singular values
// are taken from R = L^T D where G = D C D (unit-diagonal C = L L^T): the Cholesky factor of the column-scaled Gram is
// accurate with respect to the column norms, so graded columns are handled.
// pivot_tol: smallest pivot (sin^2 of the angle between a column and the span of the columns before it) that the Gram can
// still tell from zero.  The Gram is the exact Gram of the evaluated columns up to the rounding of its fp64 sums, but the
// columns themselves carry the rounding of the evaluation type: two columns that are the same function computed along two
// operator sequences (x and 1/(1/x), (x^3)^3 and ((x^3)^2)*(x^3)) differ by a few ulp of that type per value, sin ~ 1e-7 in
// fp32.  numpy evaluates in float64 and calls them collinear (sigma_min / sigma_max ~ 1e-16 << max(n,k) eps); a pivot at or
// below the type's own noise (pivot_tol) is therefore rank deficient here.  Everything above it goes through numpy's
// criterion (the cheap bound below, else the Jacobi pass).  What cannot match: columns whose true angle lies between
// numpy's ~2e-13 and the type's noise -- numpy resolves them, fp32 values do not (measured rate: profiles/README.md r02).
template <int LD>
__device__ __noinline__ bool rank_deficient(const GramView& gv, const int* idx, int k, double n_total, double pivot_tol, RankDiag& dg) {
  double Lm[LD][LD], d[LD];
  double dmin = DBL_MAX, dmax = 0.0;
  bool bad = false;
  dg.pivot_min = 1.0; dg.sv_ratio = -1.0; dg.path = RP_NONFINITE;
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i) {
    d[i] = 1.0;
    if (i < k) {
      double gii = gv.g(idx[i], idx[i]);
      if (!(gii > 0.0) || !(gii <= DBL_MAX)) bad = true;   // zero or non-finite column
      d[i] = sqrt(gii);
      dmin = fmin(dmin, d[i]); dmax = fmax(dmax, d[i]);
    }
  }
  if (bad) return true;
BSR_UNROLL_LD
  for (int i = 0; i < LD; ++i)
BSR_UNROLL_LD
    for (int j = 0; j < LD; ++j) Lm[i][j] = (i < k && j <= i) ? gv.g(idx[i], idx[j]) / (d[i] * d[j]) : 0.0;
  // Cholesky with pivot threshold
  dg.path = RP_PIVOT;
BSR_UNROLL_LD
  for (int j = 0; j < LD; ++j) {
    if (j < k) {
      double s = Lm[j][j];
BSR_UNROLL_LD
      for (int p = 0; p < j; ++p) s -= Lm[j][p] * Lm[j][p];
      dg.pivot_min = fmin(dg.pivot_min, s);
      if (!(s > pivot_tol)) return true;
      double dj = sqrt(s);
      Lm[j][j] = dj;
BSR_UNROLL_LD
      for (int i = j + 1; i < LD; ++i) {
        if (i < k) {
          double t = Lm[i][j];
BSR_UNROLL_LD
          for (int p = 0; p < j; ++p) t -= Lm[i][p] * Lm[j][p];
          Lm[i][j] = t / dj;
        }
      }
    }
  }
  const double tol = fmax(n_total, (double)k) * 2.220446049250313e-16;
  // cheap sufficient condition: sigma_min >= dmin / sqrt(tr(C^-1)), sigma_max <= sqrt(k) dmax
  double tr = 0.0;   // tr(C^-1) = |L^-1|_F^2
BSR_UNROLL_LD
  for (int c = 0; c < LD; ++c) {
    if (c < k) {
      double col[LD];
BSR_UNROLL_LD
      for (int i = 0; i < LD; ++i) {
        col[i] = 0.0;
        if (i >= c && i < k) {
          double t = (i == c) ? 1.0 : 0.0;
BSR_UNROLL_LD
          for (int p = 0; p < i; ++p) if (p >= c) t -= Lm[i][p] * col[p];
          col[i] = t / Lm[i][i];
          tr += col[i] * col[i];
        }
      }
    }
  }
  dg.path = RP_BOUND_FULL;
  if (dmin / sqrt(tr) > 4.0 * tol * sqrt((double)k) * dmax) return false;
  const bool def = jacobi_rank_deficient<LD>(Lm, d, k, tol, dg.sv_ratio);
  dg.path = def ? RP_JACOBI_DEFICIENT : RP_JACOBI_FULL;
  return def;
}
template <int LD>
__device__ __forceinline__ bool rank_deficient(const GramView& gv, const int* idx, int k, double n_total, double pivot_tol) {
  RankDiag dg;
  return rank_deficient<LD>(gv, idx, k, n_total, pivot_tol, dg);
}

// Write the Gram entries among the columns idx[0..K) (the live set) to the state's Gram cache (layout: sg_size()).
__device__ __forceinline__ void store_live_gram(const GramView& gv, const int* idx, int K, double* sg) {
  int e = 0;
  for (int i = 0; i < K; ++i)
    for (int j = i; j < K; ++j) sg[e++] = gv.g(idx[i], idx[j]);
  for (int i = 0; i < K; ++i) sg[e++] = gv.by(idx[i]);
  for (int i = 0; i < K; ++i) sg[e++] = gv.cs(idx[i]);
  for (int i = 0; i < K; ++i) sg[e++] = gv.mx(idx[i]);
}

// Everything the resolve stage needs besides the chain state.
struct ResolveCtx {
  double n_total;      // global number of rows
  double n_local;      // rows on this rank (for the executed node-eval counter)
  const double* ystats; // sum(y), y'y over all rows: entry 0 of the handle's [D][2] (this pipeline runs on one data set)
  double pivot_tol;
  int64_t sweep;       // global sweep index (Philox counter)
  // tape / trace window (may be null)
  const double* tape;
  const int64_t* tape_off;   // [C*steps + 1]
  double* trace;             // [C][steps][BSR_TRACE_DOUBLES]
  int steps;                 // proposals per chain in the window
  int step_base;             // index of this sweep's first proposal inside the window
  int c0, cn;                // chain range [c0, c0 + cn) handled by this launch
  int cached;                // the fp32 pass reads live columns from the cache (executed node-eval accounting)
};

static __device__ __noinline__ double log_ig4_pdf(double x) { return -5.0 * log(x) - 1.0 / x - 1.791759469228055; }   // lgamma(4)=log 6

// Resolve the K proposals of one sweep for chain c, sequentially (bsr_class.py:179-252).
// Rank test + K-column ridge SSE of proposal k against the live state of the other slots, assuming no proposal of
// this sweep has been accepted yet.  This is the expensive, state-independent part of a proposal's decision, so the
// K proposals of a chain compute it on K lanes in parallel; the sequential accept logic then consumes the results
// for as long as the live set is indeed unchanged (an accept invalidates the remaining ones, which are recomputed).
template <int KT>
__device__ __forceinline__ void precompute_slot(const ResolveCtx& rc, int K, int k, const double* sums, const double* maxs,
                                                const PropInfo& pi, bool& rank_rej, double& sse_new) {
  constexpr int LD = (KT > 0) ? KT + 1 : BSR_LDA;
  GramView gv{sums, maxs, 2 * K};
  int idx[BSR_MAXK];
  double beta[BSR_LDA];
  rank_rej = false;
  sse_new = nan("");
  if (pi.flags & PF_CAPACITY) return;
  bool finite_cols = true;
  for (int j = 0; j < K; ++j) { idx[j] = (j == k) ? (K + k) : j; finite_cols = finite_cols && (gv.mx(idx[j]) <= DBL_MAX); }
  if (!finite_cols || rank_deficient<LD>(gv, idx, K, rc.n_total, rc.pivot_tol)) { rank_rej = true; return; }
  sse_new = ridge_sse<LD, false>(gv, idx, K, rc.n_total, rc.ystats[0], rc.ystats[1], beta);
}

// pinfo: the K PropInfo records of this chain (any address space).  pre_rank / pre_sse: results of precompute_slot
// for the K proposals (have_pre), valid until the first accept of the sweep.
template <int MODE, int KT>
__device__ void resolve_chain(const ChainState& st, const ResolveCtx& rc, int c, const double* sums, const double* maxs,
                              const PropInfo* pinfo, bool init_only, bool have_pre = false, unsigned pre_rank = 0,
                              const double* pre_sse = nullptr) {
  constexpr int LD = (KT > 0) ? KT + 1 : BSR_LDA;
  const int K = (KT > 0) ? KT : st.K, P = 2 * K;
  GramView gv{sums, maxs, P};
  int idx[BSR_MAXK];
  double beta[BSR_LDA];
  long long* cnt = st.counters + (size_t)c * BSR_N_COUNTERS;

  if (init_only) {   // initial fit of a fresh state (bsr_class.py:147-163) + the state's K-column SSE
    for (int j = 0; j < K; ++j) idx[j] = j;
    st.sse[c] = ridge_sse<LD, false>(gv, idx, K, rc.n_total, rc.ystats[0], rc.ystats[1], beta);
    (void)ridge_sse<LD, true>(gv, idx, K, rc.n_total, rc.ystats[0], rc.ystats[1], beta);
    for (int j = 0; j <= K; ++j) st.beta[(size_t)c * (K + 1) + j] = beta[j];
    if (st.sg != nullptr) store_live_gram(gv, idx, K, st.sg + (size_t)c * sg_size(K));
    return;
  }
  if (st.done[c]) return;

  int cur[BSR_MAXK];   // Gram column currently live for each slot
  int msize[BSR_MAXK];
  for (int j = 0; j < K; ++j) { cur[j] = j; msize[j] = st.nn[st.which[c * K + j]][c * K + j]; }
  double sigma = st.sigma[c];
  double sse_old = st.sse[c];
  int total = st.total[c];
  int nerr = st.nerr[c];
  bool done = false, any_accept = false;
  long long evals_exec = 0;
  bool live_evaluated = !rc.cached;
  if (rc.cached) for (int j = 0; j < K; ++j) live_evaluated = live_evaluated || st.live_bad[c * K + j];
  if (live_evaluated) for (int j = 0; j < K; ++j) evals_exec += msize[j];

#pragma unroll 1
  for (int k = 0; k < K && !done; ++k) {
    const PropInfo& pi = pinfo[k];
    double* tr = (rc.trace != nullptr && rc.step_base + k < rc.steps)
                     ? rc.trace + ((size_t)c * rc.steps + rc.step_base + k) * BSR_TRACE_DOUBLES : nullptr;
    cnt[BSR_CNT_PROPOSALS] += 1;
    ++total;
    // every live slot points at its own buffer again for the report (bsr_class.py:180-182)
    for (int j = 0; j < K; ++j) st.report_which[c * K + j] = st.which[c * K + j];
    bool accepted = false, rank_rej = false;
    double logR = nan(""), sse_new = nan(""), u = nan("");
    if (pi.flags & PF_CAPACITY) {
      cnt[BSR_CNT_CAPACITY_REJECTS] += 1;
    } else {
      evals_exec += pi.m_new;
      long long mo = 0;
      for (int j = 0; j < K; ++j) if (j != k) mo += msize[j];
      cnt[BSR_CNT_NODE_EVALS_REF] += (long long)rc.n_local * (pi.m_new + msize[k] + mo);
      for (int j = 0; j < K; ++j) idx[j] = (j == k) ? (K + k) : cur[j];
      bool deficient;
      if (have_pre && !any_accept) {                    // live set unchanged so far: use the lane-parallel results
        deficient = (pre_rank >> k) & 1u;
        sse_new = pre_sse[k];
      } else {
        bool finite_cols = true;
        for (int j = 0; j < K; ++j) finite_cols = finite_cols && (gv.mx(idx[j]) <= DBL_MAX);
        deficient = !finite_cols || rank_deficient<LD>(gv, idx, K, rc.n_total, rc.pivot_tol);
        if (!deficient) sse_new = ridge_sse<LD, false>(gv, idx, K, rc.n_total, rc.ystats[0], rc.ystats[1], beta);
      }
      if (deficient) {
        rank_rej = true;                                                     // funcs.py:1226-1228: no accept draw
        cnt[BSR_CNT_RANK_REJECTS] += 1;
        sse_new = nan("");
      } else {
        const double ns = pi.new_sigma;
        const double yll_new = -sse_new / (2 * ns * ns) - 0.5 * rc.n_total * log(2 * 3.141592653589793 * ns * ns);
        const double yll_old = -sse_old / (2 * sigma * sigma) - 0.5 * rc.n_total * log(2 * 3.141592653589793 * sigma * sigma);
        const double qr = pi.Qinv / pi.Q;
        logR = (yll_new - yll_old) + (pi.fs_old - prop_fs_new(pi)) + log(qr > 1e-5 ? qr : 1e-5);
        if (pi.change != CH_NONE)
          logR += log(pi.hratio > 1e-5 ? pi.hratio : 1e-5) + log(pi.detjacob > 1e-5 ? pi.detjacob : 1e-5);
        logR = logR + log_ig4_pdf(ns) - log_ig4_pdf(sigma);
        const double alpha = (0.0 < logR) ? 0.0 : logR;                        // python min(logR, 0): NaN stays NaN (Q14)
        if (MODE == 1) {
          int64_t lo = rc.tape_off[(size_t)c * rc.steps + rc.step_base + k] + pi.ndraws;
          int64_t hi = rc.tape_off[(size_t)c * rc.steps + rc.step_base + k + 1];
          u = (lo < hi) ? rc.tape[lo] : 0.5;
        } else {
          Draws<0> dr;
          dr.init_philox(st.key_seed[c], (uint64_t)st.key_id[c], (uint32_t)(rc.sweep * K + k), 2u);
          u = dr.u01();
        }
        accepted = !(log(u) >= alpha);                                       // funcs.py:1300
      }
    }
    if (tr != nullptr) {
      tr[BSR_TR_MOVE] = pi.move; tr[BSR_TR_CHANGE] = pi.change; tr[BSR_TR_Q] = pi.Q; tr[BSR_TR_QINV] = pi.Qinv;
      tr[BSR_TR_HRATIO] = pi.hratio; tr[BSR_TR_DETJACOB] = pi.detjacob; tr[BSR_TR_NEW_SIGMA] = pi.new_sigma;
      tr[BSR_TR_NEW_SA2] = pi.new_sa2; tr[BSR_TR_NEW_SB2] = pi.new_sb2; tr[BSR_TR_RANK_REJECT] = rank_rej;
      tr[BSR_TR_LOGR] = logR; tr[BSR_TR_ACCEPTED] = accepted; tr[BSR_TR_SSE_NEW] = sse_new; tr[BSR_TR_SSE_OLD] = sse_old;
      tr[BSR_TR_NDRAWS] = pi.ndraws + ((pi.flags & PF_CAPACITY) || rank_rej ? 0 : 1); tr[BSR_TR_FLAGS] = pi.flags;
      tr[BSR_TR_U] = u; tr[BSR_TR_FS_NEW] = prop_fs_new(pi); tr[BSR_TR_FS_OLD] = pi.fs_old; tr[BSR_TR_M_NEW] = pi.m_new;
    }
    if (accepted) {
      cnt[BSR_CNT_ACCEPTS] += 1;
      const int prev = st.which[c * K + k];
      st.which[c * K + k] = prev ^ 1;          // the proposal buffer becomes the live tree
      cur[k] = K + k;
      msize[k] = pi.m_new;
      sigma = pi.new_sigma;
      st.sa[c * K + k] = pi.new_sa2;           // bsr_class.py:197-198 (on reject the old values come back)
      st.sb[c * K + k] = pi.new_sb2;
      sse_old = sse_new;
      if (st.live_bad != nullptr) st.live_bad[c * K + k] = st.prop_bad[c * K + k];
      any_accept = true;
      // intercept refit + RMSE (bsr_class.py:211-233)
      double sse_i = ridge_sse<LD, true>(gv, cur, K, rc.n_total, rc.ystats[0], rc.ystats[1], beta);
      for (int j = 0; j <= K; ++j) st.beta[(size_t)c * (K + 1) + j] = beta[j];
      double rmse = sqrt(sse_i / rc.n_total);
      if (nerr < st.err_cap) st.err[(size_t)c * st.err_cap + nerr] = rmse;
      else {   // keep the newest err_cap entries
        double* e = st.err + (size_t)c * st.err_cap;
        for (int j = 1; j < st.err_cap; ++j) e[j - 1] = e[j];
        e[st.err_cap - 1] = rmse;
      }
      ++nerr;
      total = 0;
      // plateau rule (bsr_class.py:248-252): len(errList) > 100 and 1 - min(last10)/mean(last10) < 0.05
      if (st.plateau_rule && nerr > 100) {
        const double* e = st.err + (size_t)c * st.err_cap;
        int have = nerr < st.err_cap ? nerr : st.err_cap;
        int k10 = have < 10 ? have : 10;
        double mn = DBL_MAX, sm = 0.0;
        for (int j = have - k10; j < have; ++j) { mn = fmin(mn, e[j]); sm += e[j]; }
        if (1.0 - mn / (sm / k10) < 0.05) {
          done = true;
          st.report_which[c * K + k] = prev;   // ROOTS gets the pre-accept snapshot, BETAS the new Beta (Q16)
        }
      }
    }
  }
  if (!done) for (int j = 0; j < K; ++j) st.report_which[c * K + j] = st.which[c * K + j];
  if (any_accept && st.sg != nullptr) store_live_gram(gv, cur, K, st.sg + (size_t)c * sg_size(K));
  cnt[BSR_CNT_NODE_EVALS_EXEC] += evals_exec * (long long)rc.n_local;
  cnt[BSR_CNT_SWEEPS] += 1;
  st.sigma[c] = sigma;
  st.sse[c] = sse_old;
  st.total[c] = total;
  st.nerr[c] = nerr;
  if (st.val > 0 && total >= st.val) done = true;                             // bsr_class.py:174
  if (done) st.done[c] = 1;
}
