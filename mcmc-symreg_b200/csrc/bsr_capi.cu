// C-ABI of libbsr_b200.so (see include/bsr_b200.h): host-side handle, memory, launches.
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <algorithm>
#include <vector>

#include "bsr_handle.h"
#include "bsr_misc_kernels.cuh"
#include <cstdlib>
#include <cub/device/device_scan.cuh>

static thread_local std::string g_err;
int bsr_fail(const std::string& m) { g_err = m; return 1; }
static int fail(const std::string& m) { return bsr_fail(m); }

template <typename T>
static int dalloc(bsr_handle* h, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  CK(cudaMalloc(&q, bytes));
  if (zero) CK(cudaMemset(q, 0, bytes));
  h->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return 0;
}
static void dfree(bsr_handle* h, void* p) {
  if (!p) return;
  for (size_t i = 0; i < h->allocs.size(); ++i)
    if (h->allocs[i] == p) { h->allocs.erase(h->allocs.begin() + i); break; }
  cudaFree(p);
}

// One device buffer carved into 256-byte aligned sections (bsr_predict_groups).
struct Carve {
  size_t bytes = 0;
  template <typename T> size_t take(size_t count) {
    const size_t at = bytes;
    bytes += (count * sizeof(T) + 255) / 256 * 256;
    return at;
  }
};

extern "C" {

// What bsr_create refuses of an operator set and its weights (nullptr: nothing).
static const char* prior_error(int n_ops, const int32_t* ops, const double* w) {
  if (n_ops < 1 || n_ops > BSR_MAX_OPS) return "n_ops must be in [1, 16]";
  double wsum = 0;
  for (int i = 0; i < n_ops; ++i) {
    if (ops[i] < OP_INV || ops[i] > OP_MUL) return "unknown opcode";
    if (!(w[i] > 0)) return "operator weights must be positive";
    wsum += w[i];
  }
  if (fabs(wsum - 1.0) > 1e-8) return "operator weights must sum to 1";
  return nullptr;
}

// A prior as the handle keeps it: the entries past n_ops and the reserved fields zero, val <= 0 as 0, plateau_rule 0 / 1 -- so that
// two priors that sample alike compare equal field by field.
static bsr_prior canonical_prior(int n_ops, const int32_t* ops, const double* w, double beta, int32_t val, int32_t plateau_rule) {
  bsr_prior p;
  memset(&p, 0, sizeof p);
  p.n_ops = n_ops;
  for (int i = 0; i < n_ops; ++i) { p.ops[i] = ops[i]; p.op_weights[i] = w[i]; }
  p.beta = beta;
  p.val = val > 0 ? val : 0;
  p.plateau_rule = plateau_rule != 0;
  return p;
}
static bool same_prior(const bsr_prior& a, const bsr_prior& b) {
  if (a.n_ops != b.n_ops || a.beta != b.beta || a.val != b.val || a.plateau_rule != b.plateau_rule) return false;
  for (int i = 0; i < a.n_ops; ++i)
    if (a.ops[i] != b.ops[i] || a.op_weights[i] != b.op_weights[i]) return false;
  return true;
}

static int build_tables(bsr_handle* h);

// Commits h->priors / h->chain_prior: the stop rule of every chain (chain_stop, read by k_wresolve; st.val / st.plateau_rule, read
// by the proposal-by-proposal pipeline, when all chains share one prior) and, once there is data, the prior tables.
static int commit_priors(bsr_handle* h) {
  ChainState& st = h->st;
  h->several_priors = h->priors.size() > 1;
  if (!h->several_priors) { st.val = h->priors[0].val; st.plateau_rule = h->priors[0].plateau_rule; }
  std::vector<int> stop((size_t)st.C);
  for (int c = 0; c < st.C; ++c) {
    const bsr_prior& p = h->priors[(size_t)h->chain_prior[(size_t)c]];
    stop[(size_t)c] = (int)((uint32_t)p.val | (p.plateau_rule ? 0x80000000u : 0u));
  }
  CK(cudaMemcpy(h->chain_stop, stop.data(), stop.size() * sizeof(int), cudaMemcpyHostToDevice));
  return h->X32 ? build_tables(h) : 0;
}

const char* bsr_last_error(void) { return g_err.c_str(); }
int bsr_version(void) { return 100; }
int bsr_max_nodes(void) { return BSR_MAXN; }

int bsr_create(const bsr_config* cfg, bsr_handle** out) {
  if (!cfg || !out) return fail("bsr_create: null argument");
  if (cfg->K < 1 || cfg->K > BSR_MAXK) return fail("bsr_create: K must be in [1, 16]");
  if (cfg->n_chains < 1) return fail("bsr_create: n_chains must be >= 1");
  if (cfg->n_ops < 1 || cfg->n_ops > BSR_MAX_OPS) return fail("bsr_create: n_ops must be in [1, 16]");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("bsr_create: no CUDA device (this library has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail("bsr_create: bad device ordinal");
  CK(cudaSetDevice(cfg->device));
  if (const char* e = prior_error(cfg->n_ops, cfg->ops, cfg->op_weights)) return fail(std::string("bsr_create: ") + e);
  bsr_handle* h = new bsr_handle();
  h->cfg = *cfg;
  if (h->cfg.err_cap <= 0) h->cfg.err_cap = 512;
  const int C = cfg->n_chains, K = cfg->K;
  ChainState& st = h->st;
  memset(&st, 0, sizeof st);
  st.C = C; st.K = K; st.err_cap = h->cfg.err_cap; st.val = cfg->val; st.plateau_rule = cfg->plateau_rule;
  const size_t CK_ = (size_t)C * K;
  int rc = 0;
  for (int b = 0; b < 2 && !rc; ++b) {
    rc |= dalloc(h, &st.tok[b], CK_ * BSR_MAXN);
    rc |= dalloc(h, &st.pa[b], CK_ * BSR_MAXN);
    rc |= dalloc(h, &st.pb[b], CK_ * BSR_MAXN);
    rc |= dalloc(h, &st.nn[b], CK_);
  }
  rc |= dalloc(h, &st.which, CK_);
  rc |= dalloc(h, &st.report_which, CK_);
  rc |= dalloc(h, &st.sigma, (size_t)C);
  rc |= dalloc(h, &st.sa, CK_);
  rc |= dalloc(h, &st.sb, CK_);
  rc |= dalloc(h, &st.sse, (size_t)C);
  rc |= dalloc(h, &st.beta, (size_t)C * (K + 1));
  rc |= dalloc(h, &st.err, (size_t)C * st.err_cap);
  rc |= dalloc(h, &st.nerr, (size_t)C);
  rc |= dalloc(h, &st.total, (size_t)C);
  rc |= dalloc(h, &st.done, (size_t)C);
  rc |= dalloc(h, &st.counters, (size_t)C * BSR_N_COUNTERS);
  rc |= dalloc(h, &st.pinfo, CK_);
  rc |= dalloc(h, &st.lfs, 2 * CK_);
  rc |= dalloc(h, &st.lcnt, CK_);
  rc |= dalloc(h, &st.key_seed, (size_t)C);
  rc |= dalloc(h, &st.key_id, (size_t)C);
  rc |= dalloc(h, &st.ds, (size_t)C);
  rc |= dalloc(h, &h->chain_pt, (size_t)C);
  rc |= dalloc(h, &h->chain_stop, (size_t)C);
  const int P = 2 * K;
  rc |= dalloc(h, &h->gram, (size_t)2 * C * (gram_n_sum(P) + P));   // [sums | maxs | per-chain scratch records]
  rc |= dalloc(h, &h->need64, (size_t)C);
  rc |= dalloc(h, &h->split_cnt, (size_t)C);
  rc |= dalloc(h, &h->d_count, 2);      // [1]: abort flag of the peer-memory exchange (k_wwait)
  rc |= dalloc(h, &h->ystats, 2);
  rc |= dalloc(h, &h->ds_n, 1);
  h->priors.assign(1, canonical_prior(cfg->n_ops, cfg->ops, cfg->op_weights, cfg->beta, cfg->val, cfg->plateau_rule));
  h->chain_prior.assign((size_t)C, 0);
  if (rc || commit_priors(h)) { bsr_destroy(h); return 1; }
  for (int i = 0; i < 8; ++i) cudaEventCreate(&h->ev[i]);
  if (const char* e = getenv("BSR_SEQ_PIPELINE")) h->seq_pipeline = atoi(e) != 0;
  if (const char* e = getenv("BSR_WINDOW")) h->window = std::max(1, std::min(BSR_MAXW, atoi(e)));
  *out = h;
  return 0;
}

int bsr_destroy(bsr_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  for (void* p : h->allocs) cudaFree(p);
  if (h->part) cudaFree(h->part);
  if (h->gt_dev) cudaFree(h->gt_dev);
  if (h->gt_host) cudaFreeHost(h->gt_host);
  if (h->pk_head) cudaFree(h->pk_head);
  if (h->pk_body) cudaFree(h->pk_body);
  if (h->stage) cudaFree(h->stage);
  bsr_window_free(h);
  for (int i = 0; i < 8; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  for (auto st : h->gstreams) cudaStreamDestroy(st);
  for (auto ev : h->gevents) cudaEventDestroy(ev);
  if (h->fork_event) cudaEventDestroy(h->fork_event);
  delete h;
  return 0;
}

static PriorTables prior_tables(const bsr_prior& p, int n_feature) {
  PriorTables pt;
  memset(&pt, 0, sizeof pt);
  pt.n_ops = p.n_ops;
  pt.n_feature = n_feature;
  pt.beta = p.beta;
  double acc = 0;
  for (int i = 0; i < pt.n_ops; ++i) {
    pt.ops[i] = p.ops[i];
    pt.w[i] = p.op_weights[i];
    pt.logw[i] = log(pt.w[i]);
    acc += pt.w[i];
    pt.cdf[i] = acc;
  }
  for (int dpt = 0; dpt <= BSR_MAXN; ++dpt) {
    double ps = 1.0 / pow((double)(1 + dpt), -p.beta);   // codes/funcs.py:79
    pt.psplit[dpt] = ps;
    pt.logsplit[dpt] = log((double)(1 + dpt)) * p.beta;  // codes/funcs.py:370
    pt.log1m[dpt] = log(1.0 - ps);                       // codes/funcs.py:362-363 (-inf at depth 0)
  }
  pt.lognf = log((double)n_feature);
  return pt;
}

static int32_t chain_features(const bsr_handle* h, int c);

// One table per distinct (feature count, prior) pair that some chain uses -- never one per chain or per data set (a table is ~2 KB;
// a handle may hold 65535 data sets) -- and the table of every chain (chain_pt).  A handle of one feature count and one prior has one
// table, entry 0, and every chain reads it.
static int build_tables(bsr_handle* h) {
  const int C = h->st.C;
  std::vector<int64_t> key((size_t)C);     // feature count << 32 | prior
  for (int c = 0; c < C; ++c) key[(size_t)c] = ((int64_t)chain_features(h, c) << 32) | h->chain_prior[(size_t)c];
  std::vector<int64_t> keys(key);
  std::sort(keys.begin(), keys.end());
  keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
  std::vector<PriorTables> pt;
  for (int64_t k : keys) pt.push_back(prior_tables(h->priors[(size_t)(k & 0xffffffff)], (int)(k >> 32)));
  if ((int)pt.size() != h->n_pt) {
    dfree(h, h->d_pt);
    h->d_pt = nullptr; h->n_pt = 0;
    if (dalloc(h, &h->d_pt, pt.size())) return 1;
    h->n_pt = (int)pt.size();
  }
  CK(cudaMemcpy(h->d_pt, pt.data(), pt.size() * sizeof(PriorTables), cudaMemcpyHostToDevice));
  std::vector<int> idx((size_t)C);
  for (int c = 0; c < C; ++c) idx[(size_t)c] = (int)(std::lower_bound(keys.begin(), keys.end(), key[(size_t)c]) - keys.begin());
  CK(cudaMemcpy(h->chain_pt, idx.data(), idx.size() * sizeof(int), cudaMemcpyHostToDevice));
  return 0;
}

// feature count of chain c's data set
static int32_t chain_features(const bsr_handle* h, int c) {
  return h->chain_ds.empty() ? h->d : h->ds_d[(size_t)h->chain_ds[(size_t)c]];
}

static int setup_col_cache(bsr_handle* h) {
  ChainState& st = h->st;
  // the column cache only serves the proposal-by-proposal pipeline when it is the one bsr_run uses (BSR_SEQ_PIPELINE=1)
  const bool want = h->seq_pipeline && h->cfg.K <= 5 && h->cfg.precision == 0 && !h->cfg.row_sharded && !getenv("BSR_NO_COL_CACHE");
  if (st.live_bad != nullptr && st.col_ld == h->ld && (st.col[0] != nullptr) == want) return 0;   // same shape
  dfree(h, st.col[0]); dfree(h, st.col[1]); dfree(h, st.sg); dfree(h, st.live_bad); dfree(h, st.prop_bad);
  st.col[0] = st.col[1] = nullptr; st.sg = nullptr; st.live_bad = nullptr; st.prop_bad = nullptr; st.col_ld = 0;
  const size_t CKn = (size_t)st.C * st.K;
  if (dalloc(h, &st.live_bad, CKn) || dalloc(h, &st.prop_bad, CKn)) return 1;
  if (dalloc(h, &st.sg, (size_t)st.C * sg_size(st.K))) return 1;      // Gram of the live columns (window path, CM_CACHED)
  st.col_ld = h->ld;
  h->col_cache_wanted = false;
  if (!want) return 0;
  const size_t bytes = 2 * CKn * (size_t)h->ld * sizeof(float);
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  if (bytes > (size_t)(0.4 * (double)free_b)) return 0;   // recompute instead of caching
  if (dalloc(h, &st.col[0], CKn * (size_t)h->ld, false) || dalloc(h, &st.col[1], CKn * (size_t)h->ld, false)) return 1;
  h->col_cache_wanted = true;
  return 0;
}

static int finish_data(bsr_handle* h) {
  if (setup_col_cache(h)) return 1;
  if (h->initialised) h->needs_refit = true;
  // y statistics over the local rows of every data set; in row-sharded mode the caller replaces them with the global values
  k_y_stats<<<h->n_ds, 1024>>>(h->y64, h->ds_n, h->ld, h->ystats);
  double s[2];
  CK(cudaMemcpy(s, h->ystats, sizeof s, cudaMemcpyDeviceToHost));
  h->sum_y = s[0]; h->yy = s[1];
  return build_tables(h);
}

static void free_data(bsr_handle* h) {
  if (h->own_x32) { dfree(h, h->X32); dfree(h, h->y32); }
  dfree(h, h->X64); dfree(h, h->y64);
  h->X32 = nullptr; h->y32 = nullptr; h->X64 = nullptr; h->y64 = nullptr;
}

// Number of data sets, their row counts (nullptr: all of h->n rows), their feature counts and the data set of every chain (nullptr:
// all chains on data set 0), committed once the data of the D data sets is in place.  On failure the caller drops the data
// (free_data): no entry point then runs on chains that name data sets the handle does not hold.
static int set_chain_datasets(bsr_handle* h, int D, const int64_t* n_rows, const int32_t* n_features, const int32_t* chain_dataset) {
  if (D != h->n_ds) {
    double* ys = nullptr;
    uint32_t* dn = nullptr;
    if (dalloc(h, &ys, 2 * (size_t)D) || dalloc(h, &dn, (size_t)D)) { dfree(h, ys); return 1; }
    dfree(h, h->ystats); dfree(h, h->ds_n);
    h->ystats = ys; h->ds_n = dn;
    h->n_ds = D;
  }
  std::vector<uint32_t> dn((size_t)D, (uint32_t)h->n);
  if (n_rows) for (int b = 0; b < D; ++b) dn[(size_t)b] = (uint32_t)n_rows[b];
  CK(cudaMemcpy(h->ds_n, dn.data(), (size_t)D * sizeof(uint32_t), cudaMemcpyHostToDevice));
  if (chain_dataset) CK(cudaMemcpy(h->st.ds, chain_dataset, (size_t)h->st.C * sizeof(int), cudaMemcpyHostToDevice));
  else CK(cudaMemset(h->st.ds, 0, (size_t)h->st.C * sizeof(int)));
  h->ds_d.assign(n_features, n_features + D);
  if (chain_dataset) h->chain_ds.assign(chain_dataset, chain_dataset + h->st.C);
  else h->chain_ds.assign((size_t)h->st.C, 0);
  h->mixed = std::any_of(h->ds_d.begin(), h->ds_d.end(), [&](int32_t v) { return v != h->ds_d[0]; });
  return 0;
}

// Replacing the data under initialised chains when the old or the new data sets differ in feature count: no chain may end up with
// fewer features than its trees were grown on (a leaf would read a column of zeros).  n_features [D], chain_dataset [C].  (Handles of
// one feature count keep their behaviour: the caller answers for the trees there, as bsr_set_state leaves it to them.)
static int check_live_features(const bsr_handle* h, const char* fn, int D, const int32_t* n_features, const int32_t* chain_dataset) {
  if (!h->initialised || !h->X32 || h->chain_ds.empty()) return 0;
  if (!h->mixed && std::all_of(n_features, n_features + D, [&](int32_t v) { return v == n_features[0]; })) return 0;
  for (int c = 0; c < h->st.C; ++c) {
    const int32_t now = chain_features(h, c), next = n_features[chain_dataset[c]];
    if (next < now) {
      char msg[240];
      snprintf(msg, sizeof msg, "%s: chain %d has trees over %d features and would get a data set of %d features (load it into a new "
               "handle)", fn, c, (int)now, (int)next);
      return fail(msg);
    }
  }
  return 0;
}

// D data sets of n_rows[b] rows x n_features[b] features from host memory (X row-major, the data sets one after another; y likewise)
// into the handle's buffers: X [D][d][ld], y [D][ld] with ld the largest row count rounded up to 4 and d the largest feature count,
// zeros past a data set's own rows and columns.
static int upload_host(bsr_handle* h, int D, const double* X, const double* y, const int64_t* n_rows, const int32_t* n_features,
                       int64_t n_total) {
  // staged tables: first row of every data set in y, then the first column element of every data set in the handle's X (b * ld), then
  // the first element of every data set in X (each the totals at [D]), then the feature counts
  const size_t D1 = (size_t)D + 1;
  std::vector<int64_t> off(3 * D1, 0);
  int64_t n = 0;
  int32_t d = 0;
  for (int b = 0; b < D; ++b) {
    off[(size_t)b + 1] = off[(size_t)b] + n_rows[b];
    off[2 * D1 + b + 1] = off[2 * D1 + b] + n_rows[b] * n_features[b];
    n = std::max(n, n_rows[b]);
    d = std::max(d, n_features[b]);
  }
  const int64_t rows = off[(size_t)D];
  const bool same_shape = h->own_x32 && h->X32 != nullptr && h->n == n && h->d == d && h->n_ds == D;
  const size_t ld = (size_t)(n + 3) / 4 * 4;
  if (!same_shape) {
    CK(cudaDeviceSynchronize());
    free_data(h);
    h->n = n; h->d = d; h->ld = (int64_t)ld;
    h->own_x32 = true;
    if (dalloc(h, &h->X32, D * ld * d) || dalloc(h, &h->X64, D * ld * d) || dalloc(h, &h->y32, D * ld) || dalloc(h, &h->y64, D * ld)) return 1;
  }
  for (int b = 0; b <= D; ++b) off[D1 + b] = (int64_t)b * (int64_t)ld;
  // staging: X, then y, then the offsets, then the feature counts
  const size_t xs = (size_t)off[3 * D1 - 1];
  const size_t bytes = (xs + (size_t)rows) * sizeof(double) + off.size() * sizeof(int64_t) + (size_t)D * sizeof(int32_t);
  if (bytes > h->stage_bytes) {
    CK(cudaDeviceSynchronize());
    if (h->stage) cudaFree(h->stage);
    h->stage = nullptr; h->stage_bytes = 0;
    CK(cudaMalloc((void**)&h->stage, bytes));
    h->stage_bytes = bytes;
  }
  double* ystage = h->stage + xs;
  int64_t* d_off = reinterpret_cast<int64_t*>(ystage + rows);
  int32_t* d_nf = reinterpret_cast<int32_t*>(d_off + off.size());
  h->n_total = n_total > 0 ? n_total : n;
  // stream-ordered after any sweep still in flight on the default stream; the copies from pageable memory are synchronous
  CK(cudaMemcpy(h->stage, X, xs * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ystage, y, (size_t)rows * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_off, off.data(), off.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_nf, n_features, (size_t)D * sizeof(int32_t), cudaMemcpyHostToDevice));
  // one launch per buffer for all D data sets (blockIdx.y); y is the one-column case
  const dim3 blocks((unsigned)std::min<int64_t>(((int64_t)ld * d + 255) / 256, 148 * 16), (unsigned)D);
  k_transpose_datasets_in<float><<<blocks, 256>>>(h->stage, d_off, d_off + D1, d_off + 2 * D1, d_nf, h->X32, d);
  k_transpose_datasets_in<double><<<blocks, 256>>>(h->stage, d_off, d_off + D1, d_off + 2 * D1, d_nf, h->X64, d);
  k_transpose_datasets_in<float><<<blocks, 256>>>(ystage, d_off, d_off + D1, nullptr, nullptr, h->y32, 1);
  k_transpose_datasets_in<double><<<blocks, 256>>>(ystage, d_off, d_off + D1, nullptr, nullptr, h->y64, 1);
  CK(cudaGetLastError());
  return 0;
}

// The checks every host upload makes before it reads any data, then the upload.  n_rows, n_features: D row and feature counts (the
// caller checked them); chain_dataset: nullptr (all chains on data set 0) or C indices in [0, D).
static int set_data_host(bsr_handle* h, const char* fn, int D, const double* X, const double* y, const int64_t* n_rows,
                         const int32_t* n_features, int64_t n_total, const int32_t* chain_dataset) {
  const std::string f(fn);
  int64_t n = 0;
  int32_t d = 0;
  for (int b = 0; b < D; ++b) { n = std::max(n, n_rows[b]); d = std::max(d, n_features[b]); }
  if (d < 1 || d > 65535) return fail(f + ": need n >= 1 and 1 <= d <= 65535");
  if ((n + 3) / 4 * 4 * (int64_t)d * D >= (int64_t)1 << 32)
    return fail(f + ": n_datasets * d * n (the largest row count) must stay below 2^32 elements per device (shard the rows, or fit fewer data "
                "sets per handle)");
  const std::vector<int32_t> one_ds(chain_dataset ? 0 : (size_t)h->st.C, 0);
  if (!chain_dataset) chain_dataset = one_ds.data();
  if (check_live_features(h, fn, D, n_features, chain_dataset)) return 1;
  CK(cudaSetDevice(h->cfg.device));
  if (upload_host(h, D, X, y, n_rows, n_features, n_total) || set_chain_datasets(h, D, n_rows, n_features, chain_dataset)) {
    free_data(h);
    return 1;
  }
  return finish_data(h);
}

int bsr_set_data_host(bsr_handle* h, const double* X, const double* y, int64_t n, int32_t d, int64_t n_total) {
  if (!h || !X || !y) return fail("bsr_set_data_host: null argument");
  if (n < 1) return fail("bsr_set_data_host: need n >= 1 and 1 <= d <= 65535");
  return set_data_host(h, "bsr_set_data_host", 1, X, y, &n, &d, n_total, nullptr);
}

// the refusals of every call that loads several data sets
static int check_datasets(bsr_handle* h, const char* fn, int32_t n_datasets, const int32_t* chain_dataset) {
  const std::string f(fn);
  if (n_datasets < 1 || n_datasets > 65535) return fail(f + ": n_datasets must be in [1, 65535]");
  for (int c = 0; c < h->st.C; ++c)
    if (chain_dataset[c] < 0 || chain_dataset[c] >= n_datasets) {
      char msg[200];
      snprintf(msg, sizeof msg, "%s: chain_dataset[%d] = %d is outside [0, %d)", fn, c, (int)chain_dataset[c], (int)n_datasets);
      return fail(msg);
    }
  // (a row-sharded handle holds a slice of the rows of one data set: bsr_set_data_* with the global row count)
  if (h->cfg.row_sharded) return fail(f + ": not available on row-sharded handles (use bsr_set_data_host)");
  if (n_datasets > 1 && h->seq_pipeline)
    return fail(f + ": several data sets need the window path of bsr_run (this handle uses the proposal-by-proposal pipeline)");
  return 0;
}

int bsr_set_datasets_host(bsr_handle* h, int32_t n_datasets, const double* X, const double* y, int64_t n, int32_t d,
                          const int32_t* chain_dataset) {
  if (!h || !X || !y || !chain_dataset) return fail("bsr_set_datasets_host: null argument");
  if (check_datasets(h, "bsr_set_datasets_host", n_datasets, chain_dataset)) return 1;
  if (n < 1) return fail("bsr_set_datasets_host: need n >= 1 and 1 <= d <= 65535");
  const std::vector<int64_t> n_rows((size_t)n_datasets, n);
  const std::vector<int32_t> n_features((size_t)n_datasets, d);
  return set_data_host(h, "bsr_set_datasets_host", n_datasets, X, y, n_rows.data(), n_features.data(), 0, chain_dataset);
}

// Data sets of any row and feature counts: the refusals of bsr_set_datasets_mixed_host (include/bsr_b200.h), then the upload.
// n_features nullptr: every data set has d features (bsr_set_datasets_ragged_host).
static int set_datasets_mixed(bsr_handle* h, const char* fn, int32_t n_datasets, const double* X, const double* y, const int64_t* n_rows,
                              const int32_t* n_features, int32_t d, const int32_t* chain_dataset) {
  if (check_datasets(h, fn, n_datasets, chain_dataset)) return 1;
  for (int b = 0; b < n_datasets; ++b)
    if (n_rows[b] < 1) {
      char msg[160];
      snprintf(msg, sizeof msg, "%s: n_rows[%d] = %lld: every data set needs at least one row", fn, b, (long long)n_rows[b]);
      return fail(msg);
    }
  std::vector<int32_t> nf((size_t)n_datasets, d);
  if (n_features) {
    for (int b = 0; b < n_datasets; ++b)
      if (n_features[b] < 1 || n_features[b] > 65535) {
        char msg[160];
        snprintf(msg, sizeof msg, "%s: n_features[%d] = %d is outside 1 .. 65535", fn, b, (int)n_features[b]);
        return fail(msg);
      }
    nf.assign(n_features, n_features + n_datasets);
  }
  return set_data_host(h, fn, n_datasets, X, y, n_rows, nf.data(), 0, chain_dataset);
}

int bsr_set_datasets_ragged_host(bsr_handle* h, int32_t n_datasets, const double* X, const double* y, const int64_t* n_rows, int32_t d,
                                 const int32_t* chain_dataset) {
  if (!h || !X || !y || !n_rows || !chain_dataset) return fail("bsr_set_datasets_ragged_host: null argument");
  return set_datasets_mixed(h, "bsr_set_datasets_ragged_host", n_datasets, X, y, n_rows, nullptr, d, chain_dataset);
}

int bsr_set_datasets_mixed_host(bsr_handle* h, int32_t n_datasets, const double* X, const double* y, const int64_t* n_rows,
                                const int32_t* n_features, const int32_t* chain_dataset) {
  if (!h || !X || !y || !n_rows || !n_features || !chain_dataset) return fail("bsr_set_datasets_mixed_host: null argument");
  return set_datasets_mixed(h, "bsr_set_datasets_mixed_host", n_datasets, X, y, n_rows, n_features, 0, chain_dataset);
}

int bsr_set_data_device(bsr_handle* h, const float* X, const float* y, int64_t n, int32_t d, int64_t ld, int64_t n_total) {
  if (!h || !X || !y) return fail("bsr_set_data_device: null argument");
  if (n < 1 || d < 1 || d > 65535 || ld < n) return fail("bsr_set_data_device: bad shape");
  if (ld % 4 != 0 || ld < (n + 3) / 4 * 4 || ((uintptr_t)X & 15) || ((uintptr_t)y & 15))
    return fail("bsr_set_data_device: X and y must be 16-byte aligned, ld a multiple of 4 and >= n rounded up to 4 (rows are read as float4)");
  if (ld * (int64_t)d >= (int64_t)1 << 32) return fail("bsr_set_data_device: d * ld must stay below 2^32 elements per device (shard the rows)");
  const std::vector<int32_t> one_ds((size_t)h->st.C, 0);
  if (check_live_features(h, "bsr_set_data_device", 1, &d, one_ds.data())) return 1;
  CK(cudaSetDevice(h->cfg.device));
  free_data(h);
  h->n = n; h->d = d; h->ld = ld; h->n_total = n_total > 0 ? n_total : n;
  h->own_x32 = false;
  h->X32 = const_cast<float*>(X); h->y32 = const_cast<float*>(y);
  auto upload = [&]() -> int {
    if (dalloc(h, &h->X64, (size_t)ld * d) || dalloc(h, &h->y64, (size_t)ld)) return 1;
    int blocks = 148 * 16;
    k_convert<float, double><<<blocks, 256>>>(X, h->X64, ld * (int64_t)d);
    k_convert<float, double><<<blocks, 256>>>(y, h->y64, n);
    CK(cudaDeviceSynchronize());
    return 0;
  };
  if (upload() || set_chain_datasets(h, 1, nullptr, &d, nullptr)) {
    free_data(h);
    return 1;
  }
  return finish_data(h);
}

int bsr_set_chain_priors(bsr_handle* h, int32_t n_priors, const bsr_prior* priors, const int32_t* chain_prior) {
  if (!h || !priors || !chain_prior) return fail("bsr_set_chain_priors: null argument");
  if (n_priors < 1) return fail("bsr_set_chain_priors: n_priors must be >= 1");
  char msg[200];
  for (int b = 0; b < n_priors; ++b)
    if (const char* e = prior_error(priors[b].n_ops, priors[b].ops, priors[b].op_weights)) {
      snprintf(msg, sizeof msg, "bsr_set_chain_priors: priors[%d]: %s", b, e);
      return fail(msg);
    }
  const int C = h->st.C;
  for (int c = 0; c < C; ++c)
    if (chain_prior[c] < 0 || chain_prior[c] >= n_priors) {
      snprintf(msg, sizeof msg, "bsr_set_chain_priors: chain_prior[%d] = %d is outside [0, %d)", c, (int)chain_prior[c], (int)n_priors);
      return fail(msg);
    }
  if (h->cfg.row_sharded) return fail("bsr_set_chain_priors: not available on row-sharded handles");
  if (h->initialised)
    return fail("bsr_set_chain_priors: the chains are initialised (set the priors before bsr_init_chains* / bsr_set_state)");
  // the distinct priors the chains use, in order of first use
  std::vector<bsr_prior> uniq;
  std::vector<int32_t> slot((size_t)n_priors, -1), cp((size_t)C);
  for (int c = 0; c < C; ++c) {
    int32_t& s = slot[(size_t)chain_prior[c]];
    if (s < 0) {
      const bsr_prior& q = priors[chain_prior[c]];
      const bsr_prior p = canonical_prior(q.n_ops, q.ops, q.op_weights, q.beta, q.val, q.plateau_rule);
      s = (int32_t)(std::find_if(uniq.begin(), uniq.end(), [&](const bsr_prior& u) { return same_prior(u, p); }) - uniq.begin());
      if (s == (int32_t)uniq.size()) uniq.push_back(p);
    }
    cp[(size_t)c] = s;
  }
  if (uniq.size() > 1 && h->seq_pipeline)
    return fail("bsr_set_chain_priors: several priors need the window path of bsr_run (this handle uses the proposal-by-proposal pipeline)");
  CK(cudaSetDevice(h->cfg.device));
  h->priors = uniq;
  h->chain_prior = cp;
  return commit_priors(h);
}

// global sum(y), y'y for row-sharded runs (the caller all-reduces the local values): entry 0 of the data sets' statistics
int bsr_get_y_stats(bsr_handle* h, double* sum_y, double* yy) {
  if (!h || !sum_y || !yy) return fail("bsr_get_y_stats: null argument");
  CK(cudaSetDevice(h->cfg.device));
  double s[2];
  CK(cudaMemcpy(s, h->ystats, sizeof s, cudaMemcpyDeviceToHost));
  *sum_y = s[0]; *yy = s[1];
  return 0;
}
int bsr_set_y_stats(bsr_handle* h, double sum_y, double yy) {
  if (!h) return fail("bsr_set_y_stats: null handle");
  CK(cudaSetDevice(h->cfg.device));
  const double s[2] = {sum_y, yy};
  CK(cudaMemcpy(h->ystats, s, sizeof s, cudaMemcpyHostToDevice));
  h->sum_y = sum_y; h->yy = yy;
  return 0;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------------
// sweep phases
// ------------------------------------------------------------------------------------------------------------
static int launch_eval(bsr_handle* h, cudaStream_t s, int init_only) {
  return bsr_launch_eval(h, s, init_only, 0, h->cfg.n_chains);
}

extern "C" { static int initial_fit(bsr_handle* h); }
static int check_ready(bsr_handle* h) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));     // every entry point that launches work goes through here: handles on several devices may share a thread
  if (!h->X32) return fail("no data: call bsr_set_data_* first");
  if (!h->initialised) return fail("chains not initialised: call bsr_init_chains or bsr_set_state first");
  if (h->needs_refit) {          // the data changed under live chains: refit them (and refill the column cache) first
    if (h->cfg.row_sharded) return fail("row-sharded handles: re-initialise the chains after changing the data");
    h->needs_refit = false;
    if (initial_fit(h)) return 1;
  }
  return 0;
}

// the proposal-by-proposal pipeline and the phase API read one data set
static int check_one_dataset(bsr_handle* h, const char* fn) {
  if (h->n_ds > 1) return fail(std::string(fn) + ": not available on a handle with several data sets (bsr_set_datasets_host); use bsr_run");
  if (h->several_priors) return fail(std::string(fn) + ": not available on a handle with several priors (bsr_set_chain_priors); use bsr_run");
  return 0;
}

extern "C" {

int bsr_sweep_propose(bsr_handle* h, void* stream) {
  if (check_ready(h) || check_one_dataset(h, "bsr_sweep_propose")) return 1;
  if (h->tape_mode && h->tape_pos >= h->tape_steps)
    return fail("tape exhausted: call bsr_set_tape again (or with NULL to return to Philox)");
  return bsr_launch_propose(h, (cudaStream_t)stream, 0, h->cfg.n_chains);
}

int bsr_sweep_eval(bsr_handle* h, void* stream) {
  if (check_ready(h) || check_one_dataset(h, "bsr_sweep_eval")) return 1;
  return launch_eval(h, (cudaStream_t)stream, 0);
}

int bsr_sweep_resolve(bsr_handle* h, void* stream) {
  if (check_ready(h) || check_one_dataset(h, "bsr_sweep_resolve")) return 1;
  if (bsr_launch_resolve(h, (cudaStream_t)stream, 0, 0, h->cfg.n_chains)) return 1;
  h->sg_dirty = true;     // an accept here rewrites the live Gram from the sweep kernels' values: a later bsr_run refits first
  h->sweep += 1;
  if (h->tape_pos < h->tape_steps) h->tape_pos += h->cfg.K;
  if (h->rec != nullptr && h->rec_pos < h->rec_steps) h->rec_pos += h->cfg.K;
  return 0;
}

int bsr_gram_buffer(bsr_handle* h, void** device_ptr, int64_t* n_sum_per_chain, int64_t* n_max_per_chain) {
  if (!h) return fail("null handle");
  const int P = 2 * h->cfg.K;
  *device_ptr = h->gram; *n_sum_per_chain = gram_n_sum(P); *n_max_per_chain = P;
  return 0;
}

static int initial_fit(bsr_handle* h) {
  // initial OLS (bsr_class.py:147-163) and the live state's K-column SSE
  if (!h->seq_pipeline && !h->cfg.row_sharded) {
    // a handle that runs in windows: the fit comes from the window path's own evaluation of the live columns (the Gram a
    // proposal's record is later held against must be made of the same values), not from the sweep kernels
    if (bsr_window_refit(h, 0)) return 1;
    CK(cudaDeviceSynchronize());
    return 0;
  }
  h->sg_dirty = true;   // row-sharded windows: the first bsr_run refits through the peers once they are mapped
  if (launch_eval(h, 0, 1)) return 1;
  if (h->cfg.row_sharded) return 0;   // caller all-reduces, then calls bsr_finish_init
  if (bsr_launch_resolve(h, 0, 1, 0, h->cfg.n_chains)) return 1;
  CK(cudaDeviceSynchronize());
  return 0;
}

int bsr_finish_init(bsr_handle* h) {   // row-sharded mode: second half of the initial fit, after the all-reduce
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  if (bsr_launch_resolve(h, 0, 1, 0, h->cfg.n_chains)) return 1;
  CK(cudaDeviceSynchronize());
  return 0;
}

static int reset_run_state(bsr_handle* h) {
  ChainState& st = h->st;
  const int C = st.C, K = st.K;
  CK(cudaMemset(st.nerr, 0, sizeof(int) * C));
  CK(cudaMemset(st.total, 0, sizeof(int) * C));
  CK(cudaMemset(st.done, 0, sizeof(int) * C));
  CK(cudaMemset(st.counters, 0, sizeof(long long) * C * BSR_N_COUNTERS));
  CK(cudaMemset(st.err, 0, sizeof(double) * (size_t)C * st.err_cap));
  CK(cudaMemset(st.pinfo, 0, sizeof(PropInfo) * (size_t)C * K));
  CK(cudaMemset(h->need64, 0, sizeof(int) * C));
  if (st.live_bad) CK(cudaMemset(st.live_bad, 0, (size_t)C * K));
  if (st.prop_bad) CK(cudaMemset(st.prop_bad, 0, (size_t)C * K));
  h->sweep = 0;
  return 0;
}

// Philox keys of the chains: explicit (seeds, ids), or (seed, chain_offset + c)
static int upload_keys(bsr_handle* h, const uint64_t* seeds, const int64_t* ids) {
  CK(cudaMemcpy(h->st.key_seed, seeds, (size_t)h->st.C * sizeof(uint64_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->st.key_id, ids, (size_t)h->st.C * sizeof(int64_t), cudaMemcpyHostToDevice));
  return 0;
}
static void handle_keys(const bsr_handle* h, uint64_t seed, std::vector<uint64_t>& seeds, std::vector<int64_t>& ids) {
  seeds.assign((size_t)h->st.C, seed);
  ids.resize((size_t)h->st.C);
  for (int c = 0; c < h->st.C; ++c) ids[(size_t)c] = h->cfg.chain_offset + c;
}

int bsr_init_chains_keyed(bsr_handle* h, const uint64_t* seeds, const int64_t* ids) {
  if (!h || !seeds || !ids) return fail("bsr_init_chains_keyed: null argument");
  if (!h->X32) return fail("no data: call bsr_set_data_* first");
  CK(cudaSetDevice(h->cfg.device));
  if (upload_keys(h, seeds, ids)) return 1;
  if (reset_run_state(h)) return 1;
  if (bsr_launch_init_chains(h, 0)) return 1;
  h->initialised = true;
  h->needs_refit = false;
  return initial_fit(h);
}

int bsr_init_chains(bsr_handle* h, uint64_t seed) {
  if (!h) return fail("null handle");
  std::vector<uint64_t> seeds;
  std::vector<int64_t> ids;
  handle_keys(h, seed, seeds, ids);
  return bsr_init_chains_keyed(h, seeds.data(), ids.data());
}

int bsr_set_state(bsr_handle* h, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                  const double* sigma, const double* sa, const double* sb, uint64_t seed) {
  if (!h) return fail("null handle");
  if (!h->X32) return fail("no data: call bsr_set_data_* first");
  CK(cudaSetDevice(h->cfg.device));
  std::vector<uint64_t> seeds;
  std::vector<int64_t> ids;
  handle_keys(h, seed, seeds, ids);
  if (upload_keys(h, seeds.data(), ids.data()) || reset_run_state(h)) return 1;
  ChainState& st = h->st;
  const size_t CKn = (size_t)st.C * st.K;
  for (size_t g = 0; g < CKn; ++g)
    if (nn[g] < 2 || nn[g] > BSR_MAXN) return fail("bsr_set_state: tree size out of range [2, 64]");
  if (h->mixed)             // data sets of different feature counts: every leaf within its chain's own
    for (size_t g = 0; g < CKn; ++g) {
      const int32_t d = chain_features(h, (int)(g / st.K));
      for (int j = 0; j < nn[g]; ++j) {
        const uint32_t t = tok[g * BSR_MAXN + j];
        if (tok_op(t) == OP_LEAF && tok_ft(t) >= d) {
          char msg[200];
          snprintf(msg, sizeof msg, "bsr_set_state: tree %d of chain %d reads feature %d; the chain's data set has %d features",
                   (int)(g % st.K), (int)(g / st.K), tok_ft(t), (int)d);
          return fail(msg);
        }
      }
    }
  if (h->several_priors)     // chains of different priors: every operator within its chain's own set (op_ind indexes its weights)
    for (size_t g = 0; g < CKn; ++g) {
      const bsr_prior& p = h->priors[(size_t)h->chain_prior[g / st.K]];
      for (int j = 0; j < nn[g]; ++j) {
        const uint32_t t = tok[g * BSR_MAXN + j];
        const int op = tok_op(t), oi = tok_oi(t);
        if (op == OP_LEAF) continue;
        if (oi >= p.n_ops || std::find(p.ops, p.ops + p.n_ops, op) == p.ops + p.n_ops) {
          char msg[240];
          if (oi >= p.n_ops)
            snprintf(msg, sizeof msg, "bsr_set_state: tree %d of chain %d has op_ind %d; the chain's prior has %d operators",
                     (int)(g % st.K), (int)(g / st.K), oi, (int)p.n_ops);
          else
            snprintf(msg, sizeof msg, "bsr_set_state: tree %d of chain %d holds opcode %d, which is not in the chain's operator set",
                     (int)(g % st.K), (int)(g / st.K), op);
          return fail(msg);
        }
      }
    }
  CK(cudaMemcpy(st.tok[0], tok, CKn * BSR_MAXN * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(st.pa[0], pa, CKn * BSR_MAXN * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(st.pb[0], pb, CKn * BSR_MAXN * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(st.nn[0], nn, CKn * sizeof(int), cudaMemcpyHostToDevice));
  CK(cudaMemset(st.nn[1], 0, CKn * sizeof(int)));
  CK(cudaMemset(st.which, 0, CKn * sizeof(int)));
  CK(cudaMemset(st.report_which, 0, CKn * sizeof(int)));
  CK(cudaMemcpy(st.sigma, sigma, st.C * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(st.sa, sa, CKn * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(st.sb, sb, CKn * sizeof(double), cudaMemcpyHostToDevice));
  h->initialised = true;
  h->needs_refit = false;
  return initial_fit(h);
}

// Chains never interact, so bsr_run splits them into n_groups contiguous groups, each running its own
// propose -> eval -> resolve sequence on its own stream: the latency-bound, low-occupancy proposal / resolve kernels
// of one group overlap the throughput-bound evaluation kernel of the others.
static int ensure_streams(bsr_handle* h, int G) {
  while ((int)h->gstreams.size() < G) {
    cudaStream_t st; cudaEvent_t ev;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    h->gstreams.push_back(st); h->gevents.push_back(ev);
  }
  if (!h->fork_event) CK(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
  return 0;
}

int bsr_run(bsr_handle* h, int32_t n_sweeps, void* stream) {
  if (check_ready(h)) return 1;
  if (h->cfg.row_sharded && h->x_world < 1)
    return fail("bsr_run: a row-sharded handle runs either phase by phase (bsr_sweep_*) or, after bsr_peer_export / bsr_peer_import, in windows over peer memory");
  cudaStream_t s = (cudaStream_t)stream;
  const int C = h->cfg.n_chains;
  // production path: speculative windows (bsr_tu_window.cu), with Philox or a value-level tape; the proposal-by-proposal
  // pipeline below runs when asked for (bsr_set_pipeline / BSR_SEQ_PIPELINE) and under the phase API
  if (!h->seq_pipeline) return bsr_run_window(h, n_sweeps, s);
  const bool plain = h->profiling || h->tape_pos < h->tape_steps || (h->rec != nullptr && h->rec_pos < h->rec_steps);
  int G = plain ? 1 : h->n_groups;
  if (G > C) G = C;
  const int launches_per_sweep = h->cfg.precision == 0 ? 4 : 3;
  if (G <= 1) {
    for (int i = 0; i < n_sweeps; ++i) {
      if (h->profiling) {
        cudaEventRecord(h->ev[0], s);
        if (bsr_sweep_propose(h, stream)) return 1;
        cudaEventRecord(h->ev[1], s);
        cudaEventRecord(h->ev[4], s); cudaEventRecord(h->ev[5], s);     // overwritten by the split eval path
        h->prof_inner = true;
        if (bsr_sweep_eval(h, stream)) return 1;
        h->prof_inner = false;
        cudaEventRecord(h->ev[2], s);
        if (bsr_sweep_resolve(h, stream)) return 1;
        cudaEventRecord(h->ev[3], s);
        cudaEventSynchronize(h->ev[3]);
        for (int p = 0; p < 3; ++p) {
          float ms = 0;
          cudaEventElapsedTime(&ms, h->ev[p], h->ev[p + 1]);
          h->prof_ms[p] += ms;
        }
        { float ms = 0; cudaEventElapsedTime(&ms, h->ev[1], h->ev[4]); h->prof_ms[3] += ms;
          cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]); h->prof_ms[4] += ms; }
        for (int p = 0; p < 5; ++p) h->prof_launches[p] += 1;
      } else {
        if (bsr_sweep_propose(h, stream) || bsr_sweep_eval(h, stream) || bsr_sweep_resolve(h, stream)) return 1;
      }
      h->launches += launches_per_sweep;
    }
    return 0;
  }
  if (ensure_streams(h, G)) return 1;
  CK(cudaEventRecord(h->fork_event, s));
  for (int g = 0; g < G; ++g) CK(cudaStreamWaitEvent(h->gstreams[g], h->fork_event, 0));
  for (int i = 0; i < n_sweeps; ++i) {
    for (int g = 0; g < G; ++g) {
      const int c0 = (int)((int64_t)C * g / G), c1 = (int)((int64_t)C * (g + 1) / G);
      cudaStream_t gs = h->gstreams[g];
      if (bsr_launch_propose(h, gs, c0, c1 - c0) || bsr_launch_eval(h, gs, 0, c0, c1 - c0) ||
          bsr_launch_resolve(h, gs, 0, c0, c1 - c0)) return 1;
      h->launches += launches_per_sweep;
    }
    h->sweep += 1;
  }
  for (int g = 0; g < G; ++g) {
    CK(cudaEventRecord(h->gevents[g], h->gstreams[g]));
    CK(cudaStreamWaitEvent(s, h->gevents[g], 0));
  }
  return 0;
}

int bsr_get_launch_count(bsr_handle* h, int64_t* launches) { *launches = h->launches; return 0; }
// threads_eval: block size of the evaluation kernel (32..256); n_groups: chain groups pipelined on separate streams
// inside bsr_run (1 = everything on the caller's stream).  0 keeps the current value.
int bsr_set_launch_geometry(bsr_handle* h, int32_t threads_eval, int32_t n_groups) {
  if (!h) return fail("null handle");
  if (threads_eval >= 32 && threads_eval <= 256 && threads_eval % 32 == 0) h->threads_eval = threads_eval;
  if (n_groups >= 1 && n_groups <= 16) { h->n_groups = n_groups; h->win_groups = n_groups; }
  return 0;
}

int bsr_set_window(bsr_handle* h, int32_t window) {
  if (!h) return fail("null handle");
  if (window < 1 || window > BSR_MAXW) return fail("bsr_set_window: window must be in [1, 64]");
  h->window = window;
  return 0;
}

int bsr_set_pipeline(bsr_handle* h, int32_t sequential) {
  if (!h) return fail("null handle");
  if (sequential && check_one_dataset(h, "bsr_set_pipeline")) return 1;
  if (h->X32) return fail("bsr_set_pipeline: call before bsr_set_data_*");
  h->seq_pipeline = sequential != 0;
  return 0;
}

int bsr_count_done(bsr_handle* h, int32_t* n_done) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemset(h->d_count, 0, sizeof(int)));
  k_count_done<<<(h->cfg.n_chains + 255) / 256, 256>>>(h->st.done, h->cfg.n_chains, h->d_count);
  CK(cudaMemcpy(n_done, h->d_count, sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

static __global__ void k_max_int(const int* v, int n, int* out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int x = (i < n) ? v[i] : 0;
  x = __reduce_max_sync(0xffffffffu, x);
  if ((threadIdx.x & 31) == 0) atomicMax(out, x);
}

int bsr_reserve_err(bsr_handle* h, int32_t err_cap) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  ChainState& st = h->st;
  if (err_cap <= st.err_cap) return 0;
  CK(cudaDeviceSynchronize());
  double* grown = nullptr;
  const size_t C = (size_t)st.C;
  if (dalloc(h, &grown, C * (size_t)err_cap)) return 1;
  CK(cudaMemcpy2D(grown, (size_t)err_cap * sizeof(double), st.err, (size_t)st.err_cap * sizeof(double), (size_t)st.err_cap * sizeof(double), C,
                  cudaMemcpyDeviceToDevice));
  dfree(h, st.err);
  st.err = grown; st.err_cap = err_cap; h->cfg.err_cap = err_cap;
  return 0;
}

int bsr_get_err_cap(bsr_handle* h, int32_t* err_cap) {
  if (!h || !err_cap) return fail("null argument");
  *err_cap = h->st.err_cap;
  return 0;
}

int bsr_run_until_done(bsr_handle* h, int32_t max_sweeps, int32_t check_every, void* stream, int32_t* sweeps_done) {
  if (check_ready(h)) return 1;
  if (check_every < 1) check_every = 16;
  int done_sweeps = 0;
  const int C = h->cfg.n_chains;
  while (done_sweeps < max_sweeps) {
    int chunk = std::min(check_every, max_sweeps - done_sweeps);
    if (bsr_run(h, chunk, stream)) return 1;
    done_sweeps += chunk;
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    int nd = 0;
    if (bsr_count_done(h, &nd)) return 1;
    if (nd >= C) break;
    // the RMSE-at-accept trace is unbounded in the reference (errList, codes/bsr_class.py:233,270): grow it before a chunk could
    // overflow it (a chunk adds at most check_every * K entries to a chain)
    int mx = 0;
    CK(cudaMemset(h->d_count, 0, sizeof(int)));
    k_max_int<<<(C + 255) / 256, 256>>>(h->st.nerr, C, h->d_count);
    CK(cudaMemcpy(&mx, h->d_count, sizeof(int), cudaMemcpyDeviceToHost));
    if (mx + check_every * h->cfg.K >= h->st.err_cap && bsr_reserve_err(h, 2 * (mx + check_every * h->cfg.K))) return 1;
  }
  if (sweeps_done) *sweeps_done = done_sweeps;
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// tape / trace / record
// ------------------------------------------------------------------------------------------------------------
int bsr_set_tape(bsr_handle* h, const double* tape, const int64_t* offsets, int32_t steps) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  dfree(h, h->tape); dfree(h, h->tape_off); dfree(h, h->trace);
  dfree(h, h->log_tok); dfree(h, h->log_pa); dfree(h, h->log_pb); dfree(h, h->log_nn);
  h->log_tok = nullptr; h->log_pa = nullptr; h->log_pb = nullptr; h->log_nn = nullptr;
  h->tape = nullptr; h->tape_off = nullptr; h->trace = nullptr;
  h->tape_steps = 0; h->tape_pos = 0; h->tape_mode = false;
  if (steps <= 0) return 0;
  if (steps % h->cfg.K != 0) return fail("bsr_set_tape: steps must be a multiple of K");
  const size_t CS = (size_t)h->cfg.n_chains * steps;
  if (dalloc(h, &h->trace, CS * BSR_TRACE_DOUBLES)) return 1;
  h->tape_steps = steps;
  if (tape != nullptr) {
    if (!offsets) return fail("bsr_set_tape: offsets required");
    const int64_t total = offsets[CS];
    if (dalloc(h, &h->tape, (size_t)std::max<int64_t>(total, 1), false) || dalloc(h, &h->tape_off, CS + 1, false)) return 1;
    CK(cudaMemcpy(h->tape, tape, (size_t)total * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->tape_off, offsets, (CS + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    h->tape_mode = true;
  }
  return 0;
}

int bsr_get_trace(bsr_handle* h, double* trace) {
  if (!h || !h->trace) return fail("bsr_get_trace: no trace window (call bsr_set_tape first)");
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(trace, h->trace, (size_t)h->cfg.n_chains * h->tape_steps * BSR_TRACE_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int bsr_trace_trees(bsr_handle* h) {
  if (!h || !h->trace) return fail("bsr_trace_trees: no trace window (call bsr_set_tape first)");
  CK(cudaSetDevice(h->cfg.device));
  if (h->log_tok) return 0;
  const size_t CS = (size_t)h->cfg.n_chains * h->tape_steps;
  if (dalloc(h, &h->log_tok, CS * BSR_MAXN) || dalloc(h, &h->log_pa, CS * BSR_MAXN) || dalloc(h, &h->log_pb, CS * BSR_MAXN) ||
      dalloc(h, &h->log_nn, CS)) return 1;
  return 0;
}

int bsr_get_trace_trees(bsr_handle* h, uint32_t* tok, double* pa, double* pb, int32_t* nn) {
  if (!h || !h->log_tok) return fail("bsr_get_trace_trees: call bsr_trace_trees first");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  const size_t CS = (size_t)h->cfg.n_chains * h->tape_steps;
  CK(cudaMemcpy(tok, h->log_tok, CS * BSR_MAXN * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(pa, h->log_pa, CS * BSR_MAXN * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(pb, h->log_pb, CS * BSR_MAXN * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(nn, h->log_nn, CS * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int bsr_set_peer_timeout(bsr_handle* h, double seconds) {
  if (!h) return fail("null handle");
  h->peer_timeout_s = seconds;
  return 0;
}

int bsr_get_exchange_profile(bsr_handle* h, double* ms, int64_t* windows) {
  if (!h) return fail("null handle");
  *ms = h->prof_ms[5]; *windows = h->prof_launches[5];
  return 0;
}

int bsr_record_draws(bsr_handle* h, int32_t steps, int32_t capacity) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  dfree(h, h->rec); dfree(h, h->rec_count);
  h->rec = nullptr; h->rec_count = nullptr; h->rec_steps = 0; h->rec_cap = 0; h->rec_pos = 0;
  if (steps <= 0) return 0;
  if (steps % h->cfg.K != 0) return fail("bsr_record_draws: steps must be a multiple of K");
  const size_t CS = (size_t)h->cfg.n_chains * steps;
  if (dalloc(h, &h->rec, CS * capacity) || dalloc(h, &h->rec_count, CS)) return 1;
  h->rec_steps = steps; h->rec_cap = capacity;
  return 0;
}

int bsr_get_recorded_draws(bsr_handle* h, double* tape, int32_t* counts) {
  if (!h || !h->rec) return fail("bsr_get_recorded_draws: recording not enabled");
  CK(cudaDeviceSynchronize());
  const size_t CS = (size_t)h->cfg.n_chains * h->rec_steps;
  CK(cudaMemcpy(tape, h->rec, CS * h->rec_cap * sizeof(double), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(counts, h->rec_count, CS * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------------------
// Device-side gather of one tree buffer per (chain, tree) into a dense, zero-padded staging area, then one D2H copy
// per array: straight into the caller's arrays when they are page-locked (bsr_alloc_host), else through the handle's
// pinned staging buffer.  mode 0: roots_ (report_which), 1: live trees (which), 2: last proposals (which ^ 1).
static __global__ void k_gather_trees(ChainState st, int mode, uint32_t* tok, double* pa, double* pb, int* nn) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= st.C * st.K) return;
  const int w = (mode == 0) ? st.report_which[g] : (mode == 1 ? st.which[g] : (st.which[g] ^ 1));
  const int m = st.nn[w][g];
  const size_t slot = (size_t)g * BSR_MAXN;
  for (int j = lane; j < BSR_MAXN; j += 32) {
    const bool in = j < m;
    tok[slot + j] = in ? st.tok[w][slot + j] : 0u;
    pa[slot + j] = in ? st.pa[w][slot + j] : 0.0;
    pb[slot + j] = in ? st.pb[w][slot + j] : 0.0;
  }
  if (lane == 0) nn[g] = m;
}

static bool is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

static int gather_trees(bsr_handle* h, int mode, uint32_t* tok, double* pa, double* pb, int32_t* nn) {
  ChainState& st = h->st;
  const size_t CKn = (size_t)st.C * st.K, N = CKn * BSR_MAXN;
  const size_t bytes = N * (sizeof(uint32_t) + 2 * sizeof(double)) + CKn * sizeof(int);
  if (h->gt_bytes < bytes) {
    CK(cudaDeviceSynchronize());
    if (h->gt_dev) cudaFree(h->gt_dev);
    if (h->gt_host) cudaFreeHost(h->gt_host);
    h->gt_dev = nullptr; h->gt_host = nullptr; h->gt_bytes = 0;
    CK(cudaMalloc(&h->gt_dev, bytes));
    CK(cudaHostAlloc(&h->gt_host, bytes, cudaHostAllocDefault));
    h->gt_bytes = bytes;
  }
  unsigned char* d = (unsigned char*)h->gt_dev;
  double* d_pa = (double*)d; double* d_pb = d_pa + N;
  uint32_t* d_tok = (uint32_t*)(d_pb + N); int* d_nn = (int*)(d_tok + N);
  k_gather_trees<<<(unsigned)((CKn + 3) / 4), 128>>>(st, mode, d_tok, d_pa, d_pb, d_nn);
  CK(cudaGetLastError());
  unsigned char* hs = (unsigned char*)h->gt_host;
  double* h_pa = (double*)hs; double* h_pb = h_pa + N;
  uint32_t* h_tok = (uint32_t*)(h_pb + N); int* h_nn = (int*)(h_tok + N);
  const bool direct = is_pinned(tok) && is_pinned(pa) && is_pinned(pb) && is_pinned(nn);
  CK(cudaMemcpyAsync(direct ? (void*)pa : (void*)h_pa, d_pa, N * sizeof(double), cudaMemcpyDeviceToHost, 0));
  CK(cudaMemcpyAsync(direct ? (void*)pb : (void*)h_pb, d_pb, N * sizeof(double), cudaMemcpyDeviceToHost, 0));
  CK(cudaMemcpyAsync(direct ? (void*)tok : (void*)h_tok, d_tok, N * sizeof(uint32_t), cudaMemcpyDeviceToHost, 0));
  CK(cudaMemcpyAsync(direct ? (void*)nn : (void*)h_nn, d_nn, CKn * sizeof(int), cudaMemcpyDeviceToHost, 0));
  CK(cudaStreamSynchronize(0));
  if (!direct) {
    memcpy(pa, h_pa, N * sizeof(double)); memcpy(pb, h_pb, N * sizeof(double));
    memcpy(tok, h_tok, N * sizeof(uint32_t)); memcpy(nn, h_nn, CKn * sizeof(int));
  }
  return 0;
}

int bsr_get_trees(bsr_handle* h, int32_t current, uint32_t* tok, double* pa, double* pb, int32_t* nn) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  return gather_trees(h, current ? 1 : 0, tok, pa, pb, nn);
}

int bsr_get_proposals(bsr_handle* h, uint32_t* tok, double* pa, double* pb, int32_t* nn) {
  // valid right after bsr_sweep_propose (before resolve flips buffers): the non-live buffer holds the proposal
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  return gather_trees(h, 2, tok, pa, pb, nn);
}

// Packed results: only the node-count-long prefix of every tree slot leaves the device (a slot is 64 nodes x 20 bytes, a tree
// holds 3 - 31 of them), and the lt parameters only for lt nodes.  bsr_pack_trees counts, scans and packs on the device
// and returns the totals; bsr_read_packed copies exactly that much.
static __global__ void k_tree_counts(ChainState st, int mode, long long* cnt_nodes, long long* cnt_lt, int* nn) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= st.C * st.K) return;
  const int w = (mode == 0) ? st.report_which[g] : (mode == 1 ? st.which[g] : (st.which[g] ^ 1));
  const int m = st.nn[w][g];
  const uint32_t* tk = st.tok[w] + (size_t)g * BSR_MAXN;
  int L = 0;
  for (int j = 0; j < m; ++j) L += (tok_op(tk[j]) == OP_LT);
  cnt_nodes[g] = m; cnt_lt[g] = L; nn[g] = m;
}
static __global__ void k_pack_trees(ChainState st, int mode, const long long* off_nodes, const long long* off_lt, uint32_t* tok, double* ab) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (g >= st.C * st.K) return;
  const int w = (mode == 0) ? st.report_which[g] : (mode == 1 ? st.which[g] : (st.which[g] ^ 1));
  const int m = st.nn[w][g];
  const size_t slot = (size_t)g * BSR_MAXN;
  const long long o = off_nodes[g];
  long long ol = off_lt[g];
  for (int j0 = 0; j0 < m; j0 += 32) {
    const int j = j0 + lane;
    uint32_t t = 0u;
    bool lt = false;
    if (j < m) { t = st.tok[w][slot + j]; tok[o + j] = t; lt = tok_op(t) == OP_LT; }
    const unsigned msk = __ballot_sync(0xffffffffu, lt);
    if (lt) {
      const long long r = ol + __popc(msk & ((1u << lane) - 1u));
      ab[2 * r] = st.pa[w][slot + j]; ab[2 * r + 1] = st.pb[w][slot + j];
    }
    ol += __popc(msk);
  }
}

int bsr_pack_trees(bsr_handle* h, int32_t current, int64_t* n_nodes, int64_t* n_lt) {
  if (!h || !n_nodes || !n_lt) return fail("bsr_pack_trees: null argument");
  CK(cudaSetDevice(h->cfg.device));
  ChainState& st = h->st;
  const size_t CKn = (size_t)st.C * st.K;
  const int mode = current ? 1 : 0;
  // staging layout: cnt_nodes | cnt_lt | off_nodes | off_lt (long long [CKn + 1] each) | nn (int [CKn]) | scan scratch | tok | ab
  size_t scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (long long*)nullptr, (long long*)nullptr, (int)(CKn + 1));
  const size_t head = 4 * (CKn + 1) * sizeof(long long) + CKn * sizeof(int) + ((scan_bytes + 255) / 256 + 1) * 256;
  if (h->pk_head_bytes < head) {
    CK(cudaDeviceSynchronize());
    if (h->pk_head) cudaFree(h->pk_head);
    h->pk_head = nullptr; h->pk_head_bytes = 0;
    CK(cudaMalloc(&h->pk_head, head));
    CK(cudaMemset(h->pk_head, 0, head));
    h->pk_head_bytes = head;
  }
  long long* cnt_nodes = (long long*)h->pk_head; long long* cnt_lt = cnt_nodes + CKn + 1;
  long long* off_nodes = cnt_lt + CKn + 1; long long* off_lt = off_nodes + CKn + 1;
  int* nn = (int*)(off_lt + CKn + 1);
  void* scratch = (void*)(((uintptr_t)(nn + CKn) + 255) / 256 * 256);
  k_tree_counts<<<(unsigned)((CKn + 255) / 256), 256>>>(st, mode, cnt_nodes, cnt_lt, nn);
  CK(cudaGetLastError());
  CK(cub::DeviceScan::ExclusiveSum(scratch, scan_bytes, cnt_nodes, off_nodes, (int)(CKn + 1)));
  CK(cub::DeviceScan::ExclusiveSum(scratch, scan_bytes, cnt_lt, off_lt, (int)(CKn + 1)));
  long long tot[2];
  CK(cudaMemcpy(&tot[0], off_nodes + CKn, sizeof(long long), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&tot[1], off_lt + CKn, sizeof(long long), cudaMemcpyDeviceToHost));
  const size_t body = (size_t)tot[0] * sizeof(uint32_t) + 16 + (size_t)tot[1] * 2 * sizeof(double) + 16;
  if (h->pk_body_bytes < body) {
    if (h->pk_body) cudaFree(h->pk_body);
    h->pk_body = nullptr; h->pk_body_bytes = 0;
    CK(cudaMalloc(&h->pk_body, body + body / 4));
    h->pk_body_bytes = body + body / 4;
  }
  h->pk_nodes = tot[0]; h->pk_lt = tot[1];
  double* ab = (double*)h->pk_body;
  uint32_t* tok = (uint32_t*)(ab + 2 * (size_t)tot[1] + 2);
  k_pack_trees<<<(unsigned)((CKn + 3) / 4), 128>>>(st, mode, off_nodes, off_lt, tok, ab);
  CK(cudaGetLastError());
  *n_nodes = tot[0]; *n_lt = tot[1];
  return 0;
}

int bsr_read_packed(bsr_handle* h, int32_t* nn, uint32_t* tok, double* ab) {
  if (!h || !h->pk_head || !h->pk_body) return fail("bsr_read_packed: call bsr_pack_trees first");
  CK(cudaSetDevice(h->cfg.device));
  const size_t CKn = (size_t)h->st.C * h->st.K;
  const int* d_nn = (const int*)((long long*)h->pk_head + 4 * (CKn + 1));
  const double* d_ab = (const double*)h->pk_body;
  const uint32_t* d_tok = (const uint32_t*)(d_ab + 2 * (size_t)h->pk_lt + 2);
  CK(cudaMemcpyAsync(nn, d_nn, CKn * sizeof(int), cudaMemcpyDeviceToHost, 0));
  if (h->pk_nodes) CK(cudaMemcpyAsync(tok, d_tok, (size_t)h->pk_nodes * sizeof(uint32_t), cudaMemcpyDeviceToHost, 0));
  if (h->pk_lt) CK(cudaMemcpyAsync(ab, d_ab, (size_t)h->pk_lt * 2 * sizeof(double), cudaMemcpyDeviceToHost, 0));
  CK(cudaStreamSynchronize(0));
  return 0;
}

int bsr_alloc_host(size_t bytes, void** out) {
  if (!out) return fail("bsr_alloc_host: null argument");
  CK(cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault));
  return 0;
}
int bsr_free_host(void* p) {
  if (p) CK(cudaFreeHost(p));
  return 0;
}

int bsr_get_stats(bsr_handle* h, double* sigma, double* sa, double* sb, double* beta, double* sse, int64_t* counters,
                  int32_t* done, int32_t* nerr) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  ChainState& st = h->st;
  const size_t C = st.C, K = st.K;
  if (sigma) CK(cudaMemcpy(sigma, st.sigma, C * sizeof(double), cudaMemcpyDeviceToHost));
  if (sa) CK(cudaMemcpy(sa, st.sa, C * K * sizeof(double), cudaMemcpyDeviceToHost));
  if (sb) CK(cudaMemcpy(sb, st.sb, C * K * sizeof(double), cudaMemcpyDeviceToHost));
  if (beta) CK(cudaMemcpy(beta, st.beta, C * (K + 1) * sizeof(double), cudaMemcpyDeviceToHost));
  if (sse) CK(cudaMemcpy(sse, st.sse, C * sizeof(double), cudaMemcpyDeviceToHost));
  if (counters) CK(cudaMemcpy(counters, st.counters, C * BSR_N_COUNTERS * sizeof(long long), cudaMemcpyDeviceToHost));
  if (done) CK(cudaMemcpy(done, st.done, C * sizeof(int), cudaMemcpyDeviceToHost));
  if (nerr) CK(cudaMemcpy(nerr, st.nerr, C * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int bsr_get_err_trace(bsr_handle* h, double* err) {
  if (!h) return fail("null handle");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(err, h->st.err, (size_t)h->st.C * h->st.err_cap * sizeof(double), cudaMemcpyDeviceToHost));
  return 0;
}

int bsr_eval_trees(bsr_handle* h, int32_t n_trees, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                   int32_t precision, double* out) {
  if (!h || !h->X32) return fail("bsr_eval_trees: no data");
  if (check_one_dataset(h, "bsr_eval_trees")) return 1;
  CK(cudaSetDevice(h->cfg.device));
  uint32_t* d_tok; double *d_a, *d_b, *d_out; int* d_nn;
  const size_t TN = (size_t)n_trees * BSR_MAXN;
  CK(cudaMalloc((void**)&d_tok, TN * sizeof(uint32_t)));
  CK(cudaMalloc((void**)&d_a, TN * sizeof(double)));
  CK(cudaMalloc((void**)&d_b, TN * sizeof(double)));
  CK(cudaMalloc((void**)&d_nn, n_trees * sizeof(int)));
  CK(cudaMalloc((void**)&d_out, (size_t)n_trees * h->n * sizeof(double)));
  CK(cudaMemcpy(d_tok, tok, TN * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_a, pa, TN * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_b, pb, TN * sizeof(double), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_nn, nn, n_trees * sizeof(int), cudaMemcpyHostToDevice));
  if (precision == 1) k_eval_trees<double><<<n_trees, 128>>>(d_tok, d_a, d_b, d_nn, h->X64, (uint32_t)h->n, (uint32_t)h->ld, d_out);
  else k_eval_trees<float><<<n_trees, 128>>>(d_tok, d_a, d_b, d_nn, h->X32, (uint32_t)h->n, (uint32_t)h->ld, d_out);
  CK(cudaGetLastError());
  CK(cudaMemcpy(out, d_out, (size_t)n_trees * h->n * sizeof(double), cudaMemcpyDeviceToHost));
  cudaFree(d_tok); cudaFree(d_a); cudaFree(d_b); cudaFree(d_nn); cudaFree(d_out);
  return 0;
}

// The body of every prediction entry point: bsr_predict_groups (include/bsr_b200.h) and, through predict_dense, the dense ones;
// `name` heads the error messages.
static int predict_groups(const char* name, int32_t device, int32_t M, int32_t K, const int32_t* nn, const uint32_t* tok, int64_t n_tok,
                          const double* ab, int64_t n_lt, const double* beta, int32_t S, int32_t d, const double* X, const int64_t* set_off,
                          int32_t G, const int32_t* grp_set, const int64_t* grp_off, const int32_t* grp_models, const int32_t* grp_reduce,
                          double* out, int32_t* n_used) {
  const std::string f = std::string(name) + ": ";
  if (!nn || !tok || !ab || !beta || !X || !set_off || !grp_set || !grp_off || !grp_models || !grp_reduce || !out || !n_used)
    return fail(f + "null argument");
  if (M < 1 || K < 1 || K > BSR_MAXK || S < 1 || G < 1 || d < 1 || n_tok < 0 || n_lt < 0)
    return fail(f + "bad shape (need M, S, G, d >= 1, 1 <= K <= 16, n_tok, n_lt >= 0)");
  // models: every tree a well-formed pre-order token sequence of 1 .. 64 nodes reading features < d; the node counts cover tok and
  // the lt nodes cover ab exactly
  const size_t NT = (size_t)M * K;
  std::vector<int64_t> node_off(NT + 1, 0), lt_off(NT + 1, 0);
  for (size_t t = 0; t < NT; ++t) {
    if (nn[t] < 1 || nn[t] > BSR_MAXN) return fail(f + "tree size out of range (1 .. 64 nodes)");
    node_off[t + 1] = node_off[t] + nn[t];
    if (node_off[t + 1] > n_tok) return fail(f + "the node counts nn add up to more tokens than tok holds");
    int64_t lts = 0;
    int depth = 0;                                  // subtrees the right-to-left scan holds
    for (int64_t i = node_off[t + 1] - 1; i >= node_off[t]; --i) {
      const int op = tok_op(tok[i]);
      if (op > OP_MUL) return fail(f + "unknown opcode in tok");
      if (op == OP_LEAF && tok_ft(tok[i]) >= d) return fail(f + "a tree reads a feature the data does not have");
      const int ar = op_arity(op);
      if (depth < ar) return fail(f + "a token sequence is not a pre-order tree");
      depth += 1 - ar;
      lts += op == OP_LT;
    }
    if (depth != 1) return fail(f + "a token sequence is not a pre-order tree");
    lt_off[t + 1] = lt_off[t] + lts;
  }
  if (node_off[NT] != n_tok) return fail(f + "the node counts nn add up to fewer tokens than tok holds");
  if (lt_off[NT] != n_lt) return fail(f + "the lt nodes of tok and the (a, b) pairs of ab differ in number");
  // test sets: each its own ld (rows rounded up to 4, so every column starts 32-byte aligned)
  if (set_off[0] != 0) return fail(f + "set_off[0] must be 0");
  std::vector<int64_t> col_off((size_t)S + 1, 0), n_rows((size_t)S);
  int64_t max_n = 0;
  for (int s = 0; s < S; ++s) {
    const int64_t n = set_off[s + 1] - set_off[s];
    if (n < 0) return fail(f + "set_off decreases");
    if (n == 0) return fail(f + "test set " + std::to_string(s) + " has no rows");
    const int64_t ld = (n + 3) / 4 * 4;
    if (ld * (int64_t)d >= (int64_t)1 << 32) return fail(f + "a test set of d * n >= 2^32 elements");
    n_rows[(size_t)s] = n;
    col_off[(size_t)s + 1] = col_off[(size_t)s] + ld;
    max_n = std::max(max_n, n);
  }
  // groups and their tasks
  if (grp_off[0] != 0) return fail(f + "grp_off[0] must be 0");
  std::vector<int64_t> grp_out((size_t)G), grp_scr((size_t)G, -1);
  std::vector<int32_t> red_grp, used((size_t)G);
  int64_t out_total = 0, red_models = 0;
  for (int g = 0; g < G; ++g) {
    const int64_t cnt = grp_off[g + 1] - grp_off[g];
    if (cnt < 0) return fail(f + "grp_off decreases");
    if (cnt == 0) return fail(f + "group " + std::to_string(g) + " has no models");
    if (grp_set[g] < 0 || grp_set[g] >= S) return fail(f + "grp_set[" + std::to_string(g) + "] is outside [0, S)");
    if (grp_off[g + 1] > INT32_MAX) return fail(f + "more than 2^31 - 1 (group, model) tasks");
    const int64_t n = n_rows[(size_t)grp_set[g]];
    grp_out[(size_t)g] = out_total;
    out_total += (grp_reduce[g] ? 2 : cnt) * n;
    used[(size_t)g] = (int32_t)cnt;
    if (grp_reduce[g]) { red_grp.push_back(g); grp_scr[(size_t)g] = red_models; red_models += cnt; }
  }
  const int64_t T = grp_off[G];
  std::vector<int32_t> task_grp((size_t)T);
  for (int g = 0; g < G; ++g)
    for (int64_t t = grp_off[g]; t < grp_off[g + 1]; ++t) {
      if (grp_models[t] < 0 || grp_models[t] >= M) return fail(f + "grp_models[" + std::to_string(t) + "] is outside [0, M)");
      task_grp[(size_t)t] = g;
    }
  // rows in chunks so that the predictions of the reducing groups ([models][chunk]) stay near 256 MB; one chunk without them
  int64_t chunk = (max_n + 1) / 2 * 2;
  if (red_models) chunk = std::min(chunk, std::max<int64_t>(256, ((int64_t)32 << 20) / red_models) / 2 * 2);
  for (int64_t& o : grp_scr) if (o >= 0) o *= chunk;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(f + "no CUDA device (no CPU fallback)");
  // one device buffer: the uploaded sections first (one copy), then used and out (read back), the transposed sets and the scratch
  Carve c;
  const int64_t rows_total = set_off[S];
  const size_t o_X = c.take<double>((size_t)rows_total * d), o_tok = c.take<uint32_t>((size_t)n_tok), o_ab = c.take<double>(2 * (size_t)n_lt);
  const size_t o_beta = c.take<double>(NT + M), o_node = c.take<int64_t>(NT + 1), o_lt = c.take<int64_t>(NT + 1);
  const size_t o_soff = c.take<int64_t>((size_t)S + 1), o_col = c.take<int64_t>((size_t)S + 1), o_nrows = c.take<int64_t>((size_t)S);
  const size_t o_tmod = c.take<int32_t>((size_t)T), o_tgrp = c.take<int32_t>((size_t)T), o_gset = c.take<int32_t>((size_t)G);
  const size_t o_goff = c.take<int64_t>((size_t)G + 1), o_gout = c.take<int64_t>((size_t)G), o_gscr = c.take<int64_t>((size_t)G);
  const size_t o_red = c.take<int32_t>(red_grp.size()), o_used = c.take<int32_t>((size_t)G);
  const size_t up_bytes = c.bytes;
  const size_t o_out = c.take<double>((size_t)out_total), o_xc = c.take<double>((size_t)col_off[(size_t)S] * d);
  const size_t o_scr = c.take<double>((size_t)red_models * chunk);
  std::vector<unsigned char> up(up_bytes);
  auto put = [&](size_t at, const void* src, size_t bytes) { if (bytes) memcpy(up.data() + at, src, bytes); };
  put(o_X, X, (size_t)rows_total * d * sizeof(double));
  put(o_tok, tok, (size_t)n_tok * sizeof(uint32_t));
  put(o_ab, ab, 2 * (size_t)n_lt * sizeof(double));
  put(o_beta, beta, (NT + M) * sizeof(double));
  put(o_node, node_off.data(), (NT + 1) * sizeof(int64_t));
  put(o_lt, lt_off.data(), (NT + 1) * sizeof(int64_t));
  put(o_soff, set_off, ((size_t)S + 1) * sizeof(int64_t));
  put(o_col, col_off.data(), ((size_t)S + 1) * sizeof(int64_t));
  put(o_nrows, n_rows.data(), (size_t)S * sizeof(int64_t));
  put(o_tmod, grp_models, (size_t)T * sizeof(int32_t));
  put(o_tgrp, task_grp.data(), (size_t)T * sizeof(int32_t));
  put(o_gset, grp_set, (size_t)G * sizeof(int32_t));
  put(o_goff, grp_off, ((size_t)G + 1) * sizeof(int64_t));
  put(o_gout, grp_out.data(), (size_t)G * sizeof(int64_t));
  put(o_gscr, grp_scr.data(), (size_t)G * sizeof(int64_t));
  put(o_red, red_grp.data(), red_grp.size() * sizeof(int32_t));
  put(o_used, used.data(), (size_t)G * sizeof(int32_t));
  int prev = 0;
  cudaGetDevice(&prev);
  unsigned char* buf = nullptr;
  auto body = [&]() -> int {
    CK(cudaSetDevice(device));
    CK(cudaMalloc((void**)&buf, c.bytes));
    CK(cudaMemcpy(buf, up.data(), up_bytes, cudaMemcpyHostToDevice));
    GroupTables p;
    p.tok = (const uint32_t*)(buf + o_tok); p.ab = (const double*)(buf + o_ab);
    p.node_off = (const int64_t*)(buf + o_node); p.lt_off = (const int64_t*)(buf + o_lt); p.beta = (const double*)(buf + o_beta);
    p.X = (const double*)(buf + o_xc); p.col_off = (const int64_t*)(buf + o_col); p.n_rows = (const int64_t*)(buf + o_nrows);
    p.task_model = (const int*)(buf + o_tmod); p.task_grp = (const int*)(buf + o_tgrp); p.grp_set = (const int*)(buf + o_gset);
    p.grp_off = (const int64_t*)(buf + o_goff); p.grp_out = (const int64_t*)(buf + o_gout); p.grp_scr = (const int64_t*)(buf + o_gscr);
    p.red_grp = (const int*)(buf + o_red);
    p.out = (double*)(buf + o_out); p.scr = (double*)(buf + o_scr); p.used = (int*)(buf + o_used);
    p.K = K; p.d = d;
    // all test sets in one launch (blockIdx.y = set; 65535 sets per launch)
    const unsigned tx = (unsigned)std::min<int64_t>(((max_n + 3) / 4 * 4 * d + 255) / 256, 148 * 16);
    for (int s0 = 0; s0 < S; s0 += 65535)
      k_transpose_datasets_in<double><<<dim3(tx, (unsigned)std::min(65535, S - s0)), 256>>>(
          (const double*)(buf + o_X), (const int64_t*)(buf + o_soff) + s0, p.col_off + s0, nullptr, nullptr, (double*)(buf + o_xc), d);
    CK(cudaGetLastError());
    const size_t smem = (size_t)K * BSR_MAXN * sizeof(EvTok<double>);
    const unsigned by = (unsigned)std::max<int64_t>(1, std::min<int64_t>(((chunk + 1) / 2 + 127) / 128, 64));
    const unsigned ry = (unsigned)std::max<int64_t>(1, std::min<int64_t>((chunk + 127) / 128, 64));
    for (int64_t r0 = 0; r0 < max_n; r0 += chunk) {
      k_predict_groups<<<dim3((unsigned)T, by), 128, smem>>>(p, r0, chunk);
      CK(cudaGetLastError());
      if (!red_grp.empty()) {
        k_predict_groups_reduce<<<dim3((unsigned)red_grp.size(), ry), 128>>>(p, r0, chunk);
        CK(cudaGetLastError());
      }
    }
    CK(cudaMemcpy(n_used, buf + o_used, (size_t)G * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (out_total) CK(cudaMemcpy(out, buf + o_out, (size_t)out_total * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
  };
  const int rc = body();
  if (buf) cudaFree(buf);
  cudaSetDevice(prev);
  return rc;
}

int bsr_predict_groups(int32_t device, int32_t M, int32_t K, const int32_t* nn, const uint32_t* tok, int64_t n_tok, const double* ab,
                       int64_t n_lt, const double* beta, int32_t S, int32_t d, const double* X, const int64_t* set_off, int32_t G,
                       const int32_t* grp_set, const int64_t* grp_off, const int32_t* grp_models, const int32_t* grp_reduce, double* out,
                       int32_t* n_used) {
  return predict_groups("bsr_predict_groups", device, M, K, nn, tok, n_tok, ab, n_lt, beta, S, d, X, set_off, G, grp_set, grp_off,
                        grp_models, grp_reduce, out, n_used);
}

// M dense models ([M][K][BSR_MAXN] slots) on one test set: packed into the layout of bsr_predict_groups and predicted as one group
// of all M models.  nn is checked first, so the packing never reads past a tree's 64 slots.
static int predict_dense(const char* name, int32_t device, int32_t M, int32_t K, const uint32_t* tok, const double* pa, const double* pb,
                         const int32_t* nn, const double* beta, const double* X, int64_t n_test, int32_t d, int32_t reduce, double* out,
                         int32_t* n_used) {
  const std::string f = std::string(name) + ": ";
  if (!tok || !pa || !pb || !nn || !beta || !X || !out) return fail(f + "null argument");
  if (M < 1 || K < 1 || K > BSR_MAXK || n_test < 1 || d < 1) return fail(f + "bad shape");
  std::vector<uint32_t> ptok;
  std::vector<double> ab;
  for (size_t t = 0; t < (size_t)M * K; ++t) {
    if (nn[t] < 1 || nn[t] > BSR_MAXN) return fail(f + "tree size out of range (1 .. 64 nodes)");
    for (size_t i = t * BSR_MAXN; i < t * BSR_MAXN + nn[t]; ++i) {
      ptok.push_back(tok[i]);
      if (tok_op(tok[i]) == OP_LT) { ab.push_back(pa[i]); ab.push_back(pb[i]); }
    }
  }
  const double no_lt = 0.0;                         // a non-null ab when no tree has an lt node
  const int64_t set_off[2] = {0, n_test}, grp_off[2] = {0, M};
  std::vector<int32_t> models((size_t)M);
  for (int32_t m = 0; m < M; ++m) models[(size_t)m] = m;
  const int32_t grp_set = 0, grp_reduce = reduce != 0;
  int32_t used = 0;
  const int rc = predict_groups(name, device, M, K, nn, ptok.data(), (int64_t)ptok.size(), ab.empty() ? &no_lt : ab.data(),
                                (int64_t)ab.size() / 2, beta, 1, d, X, set_off, 1, &grp_set, grp_off, models.data(), &grp_reduce, out, &used);
  if (!rc && n_used) *n_used = used;
  return rc;
}

int bsr_predict_trees(int32_t device, int32_t K, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                      const double* beta, const double* X, int64_t n_test, int32_t d, double* out) {
  return predict_dense("bsr_predict_trees", device, 1, K, tok, pa, pb, nn, beta, X, n_test, d, 0, out, nullptr);
}

int bsr_predict_many(int32_t device, int32_t M, int32_t K, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                     const double* beta, const double* X, int64_t n_test, int32_t d, int32_t reduce, double* out, int32_t* n_used) {
  return predict_dense("bsr_predict_many", device, M, K, tok, pa, pb, nn, beta, X, n_test, d, reduce, out, n_used);
}

int bsr_predict(bsr_handle* h, int32_t chain, int32_t reported, const double* X, int64_t n_test, int32_t d, double* out) {
  if (!h) return fail("null handle");
  if (chain < 0 || chain >= h->st.C) return fail("bsr_predict: chain out of range");
  if (d != chain_features(h, chain)) return fail("bsr_predict: feature count differs from the training data");
  const int K = h->st.K, C = h->st.C;
  std::vector<uint32_t> tok((size_t)C * K * BSR_MAXN);
  std::vector<double> pa(tok.size()), pb(tok.size()), beta((size_t)C * (K + 1));
  std::vector<int32_t> nn((size_t)C * K);
  if (bsr_get_trees(h, reported ? 0 : 1, tok.data(), pa.data(), pb.data(), nn.data())) return 1;
  if (bsr_get_stats(h, nullptr, nullptr, nullptr, beta.data(), nullptr, nullptr, nullptr, nullptr)) return 1;
  const size_t o = (size_t)chain * K;
  return bsr_predict_trees(h->cfg.device, K, tok.data() + o * BSR_MAXN, pa.data() + o * BSR_MAXN, pb.data() + o * BSR_MAXN,
                           nn.data() + o, beta.data() + (size_t)chain * (K + 1), X, n_test, d, out);
}

int bsr_set_profiling(bsr_handle* h, int32_t enabled) {
  if (!h) return fail("null handle");
  h->profiling = enabled != 0;
  for (int i = 0; i < 6; ++i) { h->prof_ms[i] = 0; h->prof_launches[i] = 0; }
  return 0;
}
int bsr_get_profile(bsr_handle* h, double* ms, int64_t* launches) {
  if (!h) return fail("null handle");
  for (int i = 0; i < 5; ++i) { ms[i] = h->prof_ms[i]; launches[i] = h->prof_launches[i]; }
  return 0;
}

}  // extern "C"
