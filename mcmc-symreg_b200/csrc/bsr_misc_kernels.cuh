// Small utility kernels used by the host API (bsr_capi.cu): allcal for explicit trees, prediction, layout
// conversion, y statistics.
#pragma once
#include "bsr_common.cuh"
#include "bsr_eval.cuh"

// allcal for arbitrary trees: out[t][row] (float64), one block per tree.
template <typename T>
__global__ void k_eval_trees(const uint32_t* tok, const double* pa, const double* pb, const int* nn, const T* X, uint32_t n,
                             uint32_t ld, double* out) {
  constexpr int R = RowVec<T>::R;
  __shared__ EvTok<T> s_tok[BSR_MAXN];
  const int t = blockIdx.x;
  const int m = nn[t];
  for (int j = threadIdx.x; j < m; j += blockDim.x) {
    const uint32_t w = tok[(size_t)t * BSR_MAXN + j];
    EvTok<T> e;
    e.op = tok_op(w); e.off = (uint32_t)tok_ft(w) * ld;
    e.a = (T)pa[(size_t)t * BSR_MAXN + j]; e.b = (T)pb[(size_t)t * BSR_MAXN + j];
    s_tok[j] = e;
  }
  __syncthreads();
  const uint32_t n_vec = (n + R - 1) / R;
  for (uint32_t q = threadIdx.x; q < n_vec; q += blockDim.x) {
    T acc[R];
    eval_tree_rows<T, R>(s_tok, m, X, q * R, acc);
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (q * R + r < n) out[(size_t)t * n + q * R + r] = (double)acc[r];
  }
}

// The device tables of bsr_predict_groups (bsr_capi.cu).
// Models, packed as bsr_read_packed leaves them: tree t = m * K + k is the tokens tok[node_off[t] .. node_off[t + 1]) and the (a, b)
// pairs ab[lt_off[t] .. lt_off[t + 1]) of its lt nodes in node order; beta [M][K + 1].
// Test set s: n_rows[s] rows, column-major at X + col_off[s] * d with ld_s = col_off[s + 1] - col_off[s] (a multiple of 4).
// Task t (one block row) is model task_model[t] of group task_grp[t]; the tasks of group g are grp_off[g] .. grp_off[g + 1], in model
// order.  Group g predicts on set grp_set[g]; its model j writes its rows to out + grp_out[g] + j * n_rows, or, for a group that
// reduces (grp_scr[g] >= 0), to scr + grp_scr[g] + j * chunk, relative to the chunk's first row.  red_grp lists the reducing
// groups; used[g] is the smallest number of models a row of group g used.
struct GroupTables {
  const uint32_t* tok;
  const double* ab;
  const int64_t* node_off;
  const int64_t* lt_off;
  const double* beta;
  const double* X;
  const int64_t* col_off;
  const int64_t* n_rows;
  const int* task_model;
  const int* task_grp;
  const int* grp_set;
  const int64_t* grp_off;
  const int64_t* grp_out;
  const int64_t* grp_scr;
  const int* red_grp;
  double* out;
  double* scr;
  int* used;
  int K, d;
};

// BSR.predict (bsr_class.py:53-68) of many models, each on its own test set: rows [r0, r0 + chunk) of task blockIdx.x, blockIdx.y
// splits the rows.  The trees are staged from the packed layout (one warp per tree, the lt pairs located by a ballot over the node's
// lt flags) and evaluated in float64, two rows per thread: v = beta0 + beta_k * tree_k, accumulated over k in order.
__global__ void k_predict_groups(GroupTables p, int64_t r0, int64_t chunk) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EvTok<double>* s_tok = reinterpret_cast<EvTok<double>*>(smem_raw);
  __shared__ int s_nn[BSR_MAXK];
  const int64_t t = blockIdx.x;
  const int g = p.task_grp[t], m = p.task_model[t], s = p.grp_set[g];
  const int64_t n = p.n_rows[s];
  if (r0 >= n) return;
  const uint32_t rows = (uint32_t)min(chunk, n - r0);
  const uint32_t n_vec = (rows + 1) / 2;
  if (blockIdx.y * blockDim.x >= n_vec) return;               // whole block past this set's rows (before any barrier)
  const int K = p.K;
  const uint32_t ld = (uint32_t)(p.col_off[s + 1] - p.col_off[s]);
  const int lane = threadIdx.x & 31;
  for (int k = threadIdx.x >> 5; k < K; k += blockDim.x >> 5) {
    const int64_t tr = (int64_t)m * K + k;
    const int64_t n0 = p.node_off[tr];
    const int nk = (int)(p.node_off[tr + 1] - n0);
    int64_t lt = p.lt_off[tr];
    for (int i0 = 0; i0 < nk; i0 += 32) {                     // nk is warp-uniform: full-warp ballots
      const int i = i0 + lane;
      const uint32_t w = i < nk ? p.tok[n0 + i] : 0u;
      const bool is_lt = i < nk && tok_op(w) == OP_LT;
      const unsigned lts = __ballot_sync(0xffffffffu, is_lt);
      if (i < nk) {
        EvTok<double> e;
        e.op = tok_op(w); e.off = (uint32_t)tok_ft(w) * ld; e.a = 0.0; e.b = 0.0;
        if (is_lt) {
          const int64_t j = lt + __popc(lts & ((1u << lane) - 1u));
          e.a = p.ab[2 * j]; e.b = p.ab[2 * j + 1];
        }
        s_tok[k * BSR_MAXN + i] = e;
      }
      lt += __popc(lts);
    }
    if (lane == 0) s_nn[k] = nk;
  }
  __syncthreads();
  const double* X = p.X + (size_t)p.col_off[s] * p.d;
  const double* b = p.beta + (size_t)m * (K + 1);
  const int64_t j = t - p.grp_off[g];
  double* dst = p.grp_scr[g] >= 0 ? p.scr + p.grp_scr[g] + j * chunk : p.out + p.grp_out[g] + j * n + r0;
  for (uint32_t q = blockIdx.y * blockDim.x + threadIdx.x; q < n_vec; q += gridDim.y * blockDim.x) {
    double v[2] = {b[0], b[0]};
    for (int k = 0; k < K; ++k) {
      double acc[2];
      eval_tree_rows<double, 2>(s_tok + k * BSR_MAXN, s_nn[k], X, (uint32_t)r0 + q * 2, acc);
      v[0] += b[k + 1] * acc[0];
      v[1] += b[k + 1] * acc[1];
    }
    if (q * 2 < rows) dst[q * 2] = v[0];
    if (q * 2 + 1 < rows) dst[q * 2 + 1] = v[1];
  }
}

// Posterior-predictive mean, sample standard deviation and used count over the models of reducing group red_grp[blockIdx.x], rows
// [r0, r0 + chunk) of its set, row by row, models in index order (deterministic), two-pass; a model whose prediction at a row is not
// finite is left out of that row.  mean goes to out + grp_out[g], std n rows later.
__global__ void k_predict_groups_reduce(GroupTables p, int64_t r0, int64_t chunk) {
  const int g = p.red_grp[blockIdx.x];
  const int64_t n = p.n_rows[p.grp_set[g]];
  if (r0 >= n) return;
  const int64_t rows = min(chunk, n - r0);
  const int M = (int)(p.grp_off[g + 1] - p.grp_off[g]);
  const double* pred = p.scr + p.grp_scr[g];
  double* mean = p.out + p.grp_out[g] + r0;
  double* sd = mean + n;
  int lo = M;
  for (int64_t r = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.y * blockDim.x) {
    double s = 0.0;
    int cnt = 0;
    for (int m = 0; m < M; ++m) {
      const double v = pred[(size_t)m * chunk + r];
      if (fabs(v) <= DBL_MAX) { s += v; ++cnt; }
    }
    const double mu = cnt ? s / cnt : nan("");
    double q = 0.0;
    for (int m = 0; m < M; ++m) {
      const double v = pred[(size_t)m * chunk + r];
      if (fabs(v) <= DBL_MAX) q += (v - mu) * (v - mu);
    }
    mean[r] = mu;
    sd[r] = cnt > 1 ? sqrt(q / (cnt - 1)) : 0.0;
    lo = min(lo, cnt);
  }
  if (lo < M) atomicMin(p.used + g, lo);
}

template <typename TI, typename TO>
__global__ void k_convert(const TI* in, TO* out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (TO)in[i];
}

// row-major float64 -> column-major T for several data sets: data set b = blockIdx.y is rows row_off[b] .. row_off[b + 1] of the
// input and goes to out + col_off[b] * d with leading dimension ld = col_off[b + 1] - col_off[b], with zeros on the rows past its own
// (up to ld).
// A handle's data sets share one ld (col_off[b] = b * ld); the test sets of bsr_predict_groups each have their own.
template <typename TO>
__global__ void k_transpose_datasets_in(const double* in, const int64_t* row_off, const int64_t* col_off, TO* out, int d) {
  const int64_t r0 = row_off[blockIdx.y], n = row_off[blockIdx.y + 1] - r0;
  const int64_t ld = col_off[blockIdx.y + 1] - col_off[blockIdx.y];
  in += (size_t)r0 * d;
  out += (size_t)col_off[blockIdx.y] * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < ld * d; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = i / d;
    int col = (int)(i % d);
    out[(int64_t)col * ld + row] = row < n ? (TO)in[i] : (TO)0;
  }
}

// y statistics: sum(y), y'y in fp64 over the n_rows[b] rows of every data set b (one block each, deterministic order per launch
// geometry): y [D][ld] -> out2 [D][2]
__global__ void k_y_stats(const double* y, const uint32_t* n_rows, int64_t ld, double* out2) {
  __shared__ double s1[32], s2[32];
  const int64_t n = n_rows[blockIdx.x];
  y += (size_t)blockIdx.x * ld;
  out2 += 2 * (size_t)blockIdx.x;
  double a = 0.0, b = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { double v = y[i]; a += v; b = fma(v, v, b); }
  a = warp_sum(a); b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = a; s2[threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double x = 0.0, z = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { x += s1[w]; z += s2[w]; }
    out2[0] = x; out2[1] = z;
  }
}

__global__ void k_count_done(const int* done, int C, int* out) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  int v = (c < C) ? (done[c] != 0) : 0;
  unsigned b = __ballot_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && b) atomicAdd(out, __popc(b));
}
