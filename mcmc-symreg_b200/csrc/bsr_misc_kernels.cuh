// Small utility kernels used by the host API (bsr_capi.cu): allcal / predict for explicit trees, layout
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

// BSR.predict (bsr_class.py:53-68): out[row] = beta0 + sum_k beta_k * tree_k(X[row]), float64 evaluation.
__global__ void k_predict(const uint32_t* tok, const double* pa, const double* pb, const int* nn, int K, const double* beta,
                          const double* X, uint32_t n, uint32_t ld, double* out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EvTok<double>* s_tok = reinterpret_cast<EvTok<double>*>(smem_raw);
  for (int j = threadIdx.x; j < K * BSR_MAXN; j += blockDim.x) {
    int k = j / BSR_MAXN, i = j % BSR_MAXN;
    if (i < nn[k]) {
      EvTok<double> e;
      e.op = tok_op(tok[j]); e.off = (uint32_t)tok_ft(tok[j]) * ld; e.a = pa[j]; e.b = pb[j];
      s_tok[j] = e;
    }
  }
  __syncthreads();
  const uint32_t n_vec = (n + 1) / 2;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_vec; q += gridDim.x * blockDim.x) {
    double v[2] = {beta[0], beta[0]};
    for (int k = 0; k < K; ++k) {
      double acc[2];
      eval_tree_rows<double, 2>(s_tok + k * BSR_MAXN, nn[k], X, q * 2, acc);
      v[0] += beta[k + 1] * acc[0];
      v[1] += beta[k + 1] * acc[1];
    }
    if (q * 2 < n) out[q * 2] = v[0];
    if (q * 2 + 1 < n) out[q * 2 + 1] = v[1];
  }
}

// BSR.predict for M models at once (the restarts of one fit): blockIdx.y = model, pred[m][row] over rows [row0, row0 + rows).
__global__ void k_predict_many(const uint32_t* tok, const double* pa, const double* pb, const int* nn, int K, const double* beta,
                               const double* X, uint32_t ld, uint32_t row0, uint32_t rows, double* pred, uint32_t pred_ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EvTok<double>* s_tok = reinterpret_cast<EvTok<double>*>(smem_raw);
  const int m = blockIdx.y;
  const size_t base = (size_t)m * K * BSR_MAXN;
  for (int j = threadIdx.x; j < K * BSR_MAXN; j += blockDim.x) {
    const int k = j / BSR_MAXN, i = j % BSR_MAXN;
    if (i < nn[m * K + k]) {
      EvTok<double> e;
      const uint32_t t = tok[base + j];
      e.op = tok_op(t); e.off = (uint32_t)tok_ft(t) * ld; e.a = pa[base + j]; e.b = pb[base + j];
      s_tok[j] = e;
    }
  }
  __syncthreads();
  const double* b = beta + (size_t)m * (K + 1);
  const uint32_t n_vec = (rows + 1) / 2;
  for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n_vec; q += gridDim.x * blockDim.x) {
    double v[2] = {b[0], b[0]};
    for (int k = 0; k < K; ++k) {
      double acc[2];
      eval_tree_rows<double, 2>(s_tok + k * BSR_MAXN, nn[m * K + k], X, row0 + q * 2, acc);
      v[0] += b[k + 1] * acc[0];
      v[1] += b[k + 1] * acc[1];
    }
    if (q * 2 < rows) pred[(size_t)m * pred_ld + q * 2] = v[0];
    if (q * 2 + 1 < rows) pred[(size_t)m * pred_ld + q * 2 + 1] = v[1];
  }
}

// Posterior-predictive mean and standard deviation over the M models, row by row, models in index order (deterministic);
// a model whose prediction at a row is not finite is left out of that row.  used[row] = models that entered.
__global__ void k_predict_reduce(const double* pred, uint32_t pred_ld, int M, uint32_t rows, double* mean, double* sd, int* used) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double s = 0.0;
  int cnt = 0;
  for (int m = 0; m < M; ++m) {
    const double v = pred[(size_t)m * pred_ld + r];
    if (fabs(v) <= DBL_MAX) { s += v; ++cnt; }
  }
  const double mu = cnt ? s / cnt : nan("");
  double q = 0.0;
  for (int m = 0; m < M; ++m) {
    const double v = pred[(size_t)m * pred_ld + r];
    if (fabs(v) <= DBL_MAX) q += (v - mu) * (v - mu);
  }
  mean[r] = mu;
  sd[r] = cnt > 1 ? sqrt(q / (cnt - 1)) : 0.0;
  used[r] = cnt;
}

template <typename TI, typename TO>
__global__ void k_convert(const TI* in, TO* out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = (TO)in[i];
}

// row-major float64 (n x d) -> column-major T (d x ld)
template <typename TO>
__global__ void k_transpose_in(const double* in, TO* out, int64_t n, int d, int64_t ld) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * d; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = i / d;
    int col = (int)(i % d);
    out[(int64_t)col * ld + row] = (TO)in[i];
  }
}

// The same for the data sets of a handle: data set b = blockIdx.y is rows row_off[b] .. row_off[b + 1] of the input and goes to
// out + b * d * ld, with zeros on the rows past its own (up to ld)
template <typename TO>
__global__ void k_transpose_datasets_in(const double* in, const int64_t* row_off, TO* out, int d, int64_t ld) {
  const int64_t r0 = row_off[blockIdx.y], n = row_off[blockIdx.y + 1] - r0;
  in += (size_t)r0 * d;
  out += (size_t)blockIdx.y * d * ld;
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
