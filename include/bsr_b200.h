/*
 * bsr_b200.h -- C-ABI of libbsr_b200.so, the B200 (sm_100a) implementation of the BSR sampling hot path.
 *
 * The reference (ying531/MCMC-SymReg) is pure Python and has no FFI; the boundary it exposes for this
 * path is the estimator `BSR.fit / predict / model / complexity` (codes/bsr_class.py:26-278) and the
 * function-level API re-exported by codes/__init__.py:9-11.  Each entry point below names the reference
 * code it replaces.  Host code (mcmc-symreg_b200/*.py) binds these with ctypes; INTEGRATION.md shows the
 * stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success, non-zero on failure with a
 * message in bsr_last_error(); one host thread per handle; "host" pointers are ordinary host memory
 * (pinned or not), "device" pointers are CUDA device memory on the handle's device.  There is no CPU
 * fallback: without a CUDA device every compute entry point fails.
 *
 * Tree encoding (one slot per (chain, tree), fixed capacity BSR_MAX_NODES, pre-order = genList order,
 * codes/funcs.py:127-142):
 *     tok[i] = opcode | (op_ind << 8) | (feature << 16)
 *     opcode : 0 terminal, 1 inv, 2 lt ('ln' in the reference: a*x+b), 3 neg, 4 sin, 5 cos, 6 exp,
 *              7 square, 8 cubic, 9 '+', 10 '*'
 *     op_ind : index into bsr_config.ops the node was created with (reference Node.op_ind; stale after
 *              reassignOperator exactly like the reference, codes/funcs.py:812,829,879,900)
 *     pa[i], pb[i] : lt parameters (float64), meaningful where opcode == 2
 */
#ifndef BSR_B200_H
#define BSR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSR_MAX_NODES 64 /* node capacity per tree; a proposal that would exceed it is a counted reject */
#define BSR_MAX_OPS 16
#define BSR_MAX_TREES 16 /* K <= 16 */
#define BSR_N_COUNTERS 8
#define BSR_TRACE_DOUBLES 24

/* counters[chain][i] */
enum {
  BSR_CNT_PROPOSALS = 0,   /* newProp calls */
  BSR_CNT_ACCEPTS = 1,
  BSR_CNT_RANK_REJECTS = 2, /* rank-deficient or non-finite proposed block (codes/funcs.py:1226-1228) */
  BSR_CNT_CAPACITY_REJECTS = 3, /* tree would exceed BSR_MAX_NODES (documented deviation, DESIGN.md) */
  BSR_CNT_FP64_SWEEPS = 4, /* sweeps re-evaluated in fp64 because fp32 overflowed */
  BSR_CNT_NODE_EVALS_REF = 5, /* reference-equivalent node-row evaluations (SURVEY.md 8d) */
  BSR_CNT_NODE_EVALS_EXEC = 6, /* node-row evaluations actually executed (live columns once per window; a proposed tree that
                                   repeats an earlier slot of its window is interpreted once; out-of-range columns twice) */
  BSR_CNT_SWEEPS = 7
};

/* trace[chain][step][i] (tape/replay mode) */
enum {
  BSR_TR_MOVE = 0, BSR_TR_CHANGE = 1, BSR_TR_Q = 2, BSR_TR_QINV = 3, BSR_TR_HRATIO = 4, BSR_TR_DETJACOB = 5,
  BSR_TR_NEW_SIGMA = 6, BSR_TR_NEW_SA2 = 7, BSR_TR_NEW_SB2 = 8, BSR_TR_RANK_REJECT = 9, BSR_TR_LOGR = 10,
  BSR_TR_ACCEPTED = 11, BSR_TR_SSE_NEW = 12, BSR_TR_SSE_OLD = 13, BSR_TR_NDRAWS = 14, BSR_TR_FLAGS = 15,
  BSR_TR_U = 16 /* accept uniform */, BSR_TR_FS_NEW = 17, BSR_TR_FS_OLD = 18, BSR_TR_M_NEW = 19,
  /* what the rank test saw (window path): smallest pivot of the column-scaled Gram, sigma_min / sigma_max when the
   * Jacobi pass ran (else -1), path taken (1 non-finite / zero column, 2 pivot below the type's noise, 3 full rank by the
   * cheap bound, 4 / 5 Jacobi: full rank / deficient by numpy's criterion); 23: bit 0 = the proposal's column was
   * re-interpreted in double range */
  BSR_TR_PIVOT_MIN = 20, BSR_TR_SV_RATIO = 21, BSR_TR_RANK_PATH = 22, BSR_TR_WIDE = 23
};

typedef struct bsr_handle bsr_handle;

/* Replaces the constructor arguments of BSR (codes/bsr_class.py:27-35) and the constants hard-coded in
 * fit (ops / weights / types, codes/bsr_class.py:110-112). */
typedef struct bsr_config {
  int32_t K;              /* treeNum */
  int32_t n_chains;       /* chains resident on this device; the reference's itrNum restarts run in parallel */
  int64_t chain_offset;   /* global id of local chain 0: the RNG is keyed by global id, so results do not
                             depend on how chains are sharded over GPUs */
  int32_t n_ops;
  int32_t ops[BSR_MAX_OPS];        /* opcodes, reference order: inv, ln, neg, sin, cos, exp, square, cubic, +, * */
  double op_weights[BSR_MAX_OPS];  /* Op_weights */
  double beta;            /* split prior exponent (codes/funcs.py:79) */
  int32_t val;            /* stop a chain after `val` consecutive rejections (codes/bsr_class.py:174); <=0: never */
  int32_t plateau_rule;   /* 1: apply the RMSE plateau stop of codes/bsr_class.py:248-252 */
  int32_t precision;      /* 0: fp32 tree evaluation (+ fp64 re-evaluation on overflow), 1: fp64 evaluation */
  int32_t err_cap;        /* capacity of the per-chain RMSE-at-accept trace (train_err_) */
  int32_t device;         /* CUDA device ordinal */
  int32_t row_sharded;    /* 1: rows are sharded over ranks; the caller all-reduces bsr_gram_buffer between
                             bsr_sweep_eval and bsr_sweep_resolve */
  int32_t reserved[7];
} bsr_config;

const char* bsr_last_error(void);
int bsr_version(void);
int bsr_max_nodes(void);

/* BSR.__init__ (codes/bsr_class.py:27-35). */
int bsr_create(const bsr_config* cfg, bsr_handle** out);
int bsr_destroy(bsr_handle* h);

/* The (train_data, train_y) arguments of BSR.fit (codes/bsr_class.py:77-87).  X is row-major n x d float64
 * exactly as a numpy array / DataFrame.values; the library builds its own column-major fp32 (+fp64) copies.
 * n_total is the global row count when rows are sharded (n_total == n otherwise). */
int bsr_set_data_host(bsr_handle* h, const double* X_rowmajor, const double* y, int64_t n, int32_t d, int64_t n_total);
/* Same, from device memory: fp32 column-major X (leading dimension ld >= n) and fp32 y, used in place.
 * Both leave the handle with one data set, every chain on it. */
int bsr_set_data_device(bsr_handle* h, const float* X_colmajor, const float* y, int64_t n, int32_t d, int64_t ld,
                        int64_t n_total);
/* n_datasets data sets of the same shape in one handle: X row-major [n_datasets][n][d], y [n_datasets][n]; chain c fits data set
 * chain_dataset[c] (each in [0, n_datasets); n_datasets * d * n below 2^32 elements).  Chains never interact, so with chains keyed as
 * a handle of one data set would key them (bsr_init_chains_keyed), the chains of data set b end exactly -- bit for bit -- where that
 * handle's chains end, whenever both handles have the same window geometry (bsr_get_window_geometry).  They do for n < 16384 rows
 * (one row split, same tile); with more rows and few chains the split count depends on the chain count, and the results then agree
 * up to the fp64 summation order of the splits.  Several data sets run on the window path of bsr_run only: the proposal-by-proposal
 * pipeline (bsr_set_pipeline), the phase API (bsr_sweep_*), bsr_peer_export / bsr_peer_import and bsr_eval_trees refuse them.
 * Row-sharded handles (a slice of one data set, with its global row count) refuse this call; they use bsr_set_data_*.  A failed
 * call leaves the handle without data.  Lets one run fit a replication study, bootstrap refits or several targets on the same
 * features. */
int bsr_set_datasets_host(bsr_handle* h, int32_t n_datasets, const double* X_rowmajor, const double* y, int64_t n, int32_t d,
                          const int32_t* chain_dataset);
/* Same, for data sets of different row counts (the same d): data set b has n_rows[b] >= 1 rows, X_rowmajor holds the rows of the
 * data sets one after another (sum(n_rows) x d, row-major) and y their values (sum(n_rows)).  The handle keeps the layout of equal
 * row counts with n the largest row count (rows past a data set's own are zeros) and the window geometry of that n
 * (bsr_get_window_geometry); n_datasets * d * n (rounded up to 4) below 2^32 elements, checked before any data is read.  Every chain
 * works on its own data set's rows alone.  With rps the rows per split of the geometry, the chains of data set b end bit for bit where
 * the chains of a handle holding only data set b end (keyed alike) when n_rows[b] <= rps and that handle runs one split -- always below
 * 16384 rows; with n_rows[b] > rps the two agree up to the fp64 summation order of the splits.  The same refusals and the same failure
 * behaviour as bsr_set_datasets_host, which is the case of equal row counts.  Fits learning curves, cross-validation folds or groups
 * of different sizes in one run. */
int bsr_set_datasets_ragged_host(bsr_handle* h, int32_t n_datasets, const double* X_rowmajor, const double* y, const int64_t* n_rows,
                                 int32_t d, const int32_t* chain_dataset);
/* Same, for data sets of different row and feature counts: data set b is n_rows[b] >= 1 rows x n_features[b] features (1 .. 65535),
 * X_rowmajor holds the data sets one after another (data set b row-major, sum(n_rows[b] * n_features[b]) values) and y their values
 * (sum(n_rows)).  The handle keeps X as [n_datasets][d][ld] with d the largest feature count (columns past a data set's own are zeros
 * that no chain of it reads), so it holds n_datasets * d * ld values per precision -- ld the largest row count rounded up to 4 -- which
 * must stay below 2^32; a suite of mostly narrow data sets beside one wide one pays for the wide one's columns.  Every chain draws its
 * leaf features and charges its tree prior (log n_features per leaf) with its own data set's feature count: data set b is fitted as a
 * handle holding only data set b fits it, bit for bit under the row-split condition of bsr_set_datasets_ragged_host, which is the case
 * of one feature count.  The same refusals, checked before any data is read, and the same failure behaviour.  Further refusals once
 * the data sets differ in feature count: replacing the data so that an initialised chain gets fewer features than its trees were grown
 * on (here and in every other bsr_set_data*), and a bsr_set_state tree with a leaf feature >= its chain's feature count; bsr_predict
 * compares d with the chain's own feature count.  Fits a benchmark suite of problems with 1 to 9 inputs in one run. */
int bsr_set_datasets_mixed_host(bsr_handle* h, int32_t n_datasets, const double* X_rowmajor, const double* y, const int64_t* n_rows,
                                const int32_t* n_features, const int32_t* chain_dataset);

/* Prior initialisation of every chain: sigma ~ IG(1), per tree sigma_a, sigma_b ~ IG(1) and grow()
 * (codes/bsr_class.py:123-142, codes/funcs.py:74-119), then the initial intercept OLS (bsr_class.py:147-163). */
/* Every chain draws from Philox under its own key (seed, id): bsr_init_chains keys chain c with (seed, chain_offset + c),
 * bsr_init_chains_keyed with (seeds[c], ids[c]) (host arrays [n_chains] each). */
int bsr_init_chains(bsr_handle* h, uint64_t seed);
int bsr_init_chains_keyed(bsr_handle* h, const uint64_t* seeds, const int64_t* ids);
/* Load an explicit state instead (host arrays; tok/pa/pb are [n_chains][K][BSR_MAX_NODES], nn/sa/sb are
 * [n_chains][K], sigma is [n_chains]) and compute the initial fit; the chains are keyed as by bsr_init_chains(h, seed).
 * Used for replaying reference states. */
int bsr_set_state(bsr_handle* h, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                  const double* sigma, const double* sa, const double* sb, uint64_t seed);

/* The hot loop of BSR.fit (codes/bsr_class.py:174-255): n_sweeps sweeps of K newProp calls
 * (codes/funcs.py:1184-1306) for every chain that is not done.  Work is issued on `stream` (a cudaStream_t,
 * NULL = default stream); the call returns when it is complete (the number of windows a chain needs depends on its
 * accepts, so the driver reads back the count of unfinished chains).  In tape mode (bsr_set_tape) the same window
 * kernels consume the tape instead of Philox. */
int bsr_run(bsr_handle* h, int32_t n_sweeps, void* stream);
/* Launch geometry of bsr_run.  threads_eval: block size of the evaluation kernel (32..256).  n_groups: chains never
 * interact, so bsr_run can split them into n_groups contiguous groups that run their propose -> eval -> resolve
 * sequences on separate streams (results are identical for every n_groups).  0 keeps the current value. */
int bsr_set_launch_geometry(bsr_handle* h, int32_t threads_eval, int32_t n_groups);
int bsr_get_launch_count(bsr_handle* h, int64_t* launches);
/* bsr_run works in speculative windows: a rejected newProp (codes/funcs.py:1298-1306) leaves the chain untouched, so
 * `window` (1..64, default 64) consecutive proposals of a chain are generated from the same live state, evaluated and
 * scored in parallel, and consumed in order up to the first accept; the chain obtained is the same for every window
 * size (each draw is a Philox function of seed, chain id, proposal index).  bsr_run returns with the work complete. */
int bsr_set_window(bsr_handle* h, int32_t window);
/* Geometry the window kernels use for the current data (after bsr_set_data_*): geom[0] row splits of the evaluation kernels (one
 * partial record per split), geom[1] rows per split, geom[2] rows per shared-memory tile, geom[3] depth of the record ring (windows
 * kept per chain as an exact-match cache; 0 before the first run allocated it), geom[4] window.  Diagnostics / tests: the reference
 * has no counterpart (its allcal walks one tree over a DataFrame, codes/funcs.py:175-220). */
int bsr_get_window_geometry(bsr_handle* h, int64_t* geom5);
/* sequential != 0: bsr_run uses the proposal-by-proposal pipeline (bsr_sweep_propose / eval / resolve per sweep, with a
 * column cache) instead of speculative windows; for A/B measurements and tests.  Call before bsr_set_data_*. */
int bsr_set_pipeline(bsr_handle* h, int32_t sequential);
/* Runs until every chain hit its stop rule or max_sweeps; returns the number of sweeps done in *sweeps_done.  The RMSE-at-accept
 * trace (train_err_, the reference's unbounded errList, codes/bsr_class.py:233,270) is grown between chunks so that it never
 * truncates; under plain bsr_run a chain keeps its newest err_cap entries and nerr tells how many there were. */
int bsr_run_until_done(bsr_handle* h, int32_t max_sweeps, int32_t check_every, void* stream, int32_t* sweeps_done);
/* The three phases of one sweep, for callers that need to all-reduce the Gram partials in between
 * (row-sharded mode, SURVEY.md 8e).  bsr_run == n_sweeps x (propose, eval, resolve). */
int bsr_sweep_propose(bsr_handle* h, void* stream);
int bsr_sweep_eval(bsr_handle* h, void* stream);
int bsr_sweep_resolve(bsr_handle* h, void* stream);
/* Device buffer holding, per chain, the partial sums (to SUM-allreduce) followed by the partial max-abs values
 * (to MAX-allreduce): [n_chains][n_sum] doubles then [n_chains][n_max] doubles. */
int bsr_gram_buffer(bsr_handle* h, void** device_ptr, int64_t* n_sum_per_chain, int64_t* n_max_per_chain);
/* Row-sharded mode only (one data set).  sum(y), y'y are computed over the local rows by bsr_set_data_*; the caller all-reduces
 * them and writes the global values back.  bsr_init_chains / bsr_set_state then leave the initial Gram partials in
 * bsr_gram_buffer; after all-reducing them the caller completes the initial fit with bsr_finish_init. */
int bsr_get_y_stats(bsr_handle* h, double* sum_y, double* yy);
int bsr_set_y_stats(bsr_handle* h, double sum_y, double yy);
int bsr_finish_init(bsr_handle* h);

/* Row-sharded handles, second mode: speculative windows with the exchange fused into the resolve kernel.  Every rank
 * evaluates the window on its own rows; k_wresolve then reads the partial sums of ALL ranks straight from their memory
 * (CUDA IPC peer mappings, NVLink) in rank order, so every rank takes the same decisions with no collective call; the
 * hand-over is one flag per rank pair written / polled by two single-warp kernels.  Setup (once, after bsr_set_data_*):
 * each rank calls bsr_peer_export (64-byte cudaIpcMemHandle_t out), the host code all-gathers the handles, each rank
 * calls bsr_peer_import with all of them; from then on bsr_run works on the handle.  world <= 8, one node. */
int bsr_peer_export(bsr_handle* h, int32_t world, void* ipc_handle_out /* 64 bytes */);
int bsr_peer_import(bsr_handle* h, int32_t rank, int32_t world, const void* ipc_handles /* world x 64 bytes */);
/* Wall-clock limit (seconds, default 120; <= 0: none) a rank waits for the partial sums of one window from its peers.  On
 * expiry bsr_run fails with the missing rank in bsr_last_error() and the chains stay at the last resolved window; the CUDA
 * context remains usable. */
int bsr_set_peer_timeout(bsr_handle* h, double seconds);
/* Device time (ms, accumulated while bsr_set_profiling is on) between the end of a rank's evaluation kernels and the start
 * of its resolve kernel, i.e. k_wsignal + k_wwait: what the exchange costs a window; *windows = windows measured. */
int bsr_get_exchange_profile(bsr_handle* h, double* ms, int64_t* windows);

/* Value-level RNG tape (SURVEY.md 4.2): the next `steps` proposals of every chain consume draws from
 * tape[offsets[c*steps+s] .. offsets[c*steps+s+1]) instead of Philox, and record a trace.  steps must be a
 * multiple of K.  Pass tape == NULL to return to Philox (optionally still recording `steps` trace rows). */
int bsr_set_tape(bsr_handle* h, const double* tape, const int64_t* offsets, int32_t steps);
int bsr_get_trace(bsr_handle* h, double* trace /* [n_chains][steps][BSR_TRACE_DOUBLES] */);
/* Also keep the proposed tree of every traced proposal (after auxProp assigned its lt parameters, codes/funcs.py:1189-1210):
 * call after bsr_set_tape; bsr_get_trace_trees returns [n_chains][steps][BSR_MAX_NODES] tokens / parameters and
 * [n_chains][steps] node counts (0: capacity reject or proposal not consumed).  Window path (bsr_run) only. */
int bsr_trace_trees(bsr_handle* h);
int bsr_get_trace_trees(bsr_handle* h, uint32_t* tok, double* pa, double* pb, int32_t* nn);
/* Proposed trees of the last sweep (after the lt parameters were assigned), [n_chains][K][...]. */
int bsr_get_proposals(bsr_handle* h, uint32_t* tok, double* pa, double* pb, int32_t* nn);
/* Record the values Philox draws into a tape (for replay through the oracle): capacity doubles per proposal. */
int bsr_record_draws(bsr_handle* h, int32_t steps, int32_t capacity);
int bsr_get_recorded_draws(bsr_handle* h, double* tape /* [n_chains][steps][capacity] */, int32_t* counts);

/* Results.  roots: what BSR.fit stores in roots_ (codes/bsr_class.py:272, including the pre-accept
 * snapshot on a plateau break); current != 0 returns the live chain state instead. */
int bsr_get_trees(bsr_handle* h, int32_t current, uint32_t* tok, double* pa, double* pb, int32_t* nn);
/* The same trees without the padding of their slots: bsr_pack_trees gathers, on the device, the node-count-long token prefix
 * of every tree (tree after tree, in [chain][tree] order) and the (a, b) pairs of the lt nodes only (in node order), and
 * returns the totals; bsr_read_packed then copies nn [n_chains][K], tok [n_nodes] and ab [n_lt][2] to the host (straight
 * into page-locked arrays when they come from bsr_alloc_host).  A result read costs 4 bytes per node instead of 1280 per
 * tree. */
int bsr_pack_trees(bsr_handle* h, int32_t current, int64_t* n_nodes, int64_t* n_lt);
int bsr_read_packed(bsr_handle* h, int32_t* nn, uint32_t* tok, double* ab);
/* Page-locked host memory for result arrays: bsr_get_trees copies device -> host straight into arrays that were
 * allocated here (no staging copy); ordinary host memory works too. */
int bsr_alloc_host(size_t bytes, void** out);
int bsr_free_host(void* p);
/* sigma [C], sa/sb [C][K], beta [C][K+1] (intercept first, un-scaled: betas_, bsr_class.py:227), sse [C]
 * (K-column no-intercept SSE of the current state, codes/funcs.py:1147-1162), counters [C][BSR_N_COUNTERS],
 * done [C], nerr [C] (number of accepts recorded in the RMSE trace).  Any pointer may be NULL. */
int bsr_get_stats(bsr_handle* h, double* sigma, double* sa, double* sb, double* beta, double* sse,
                  int64_t* counters, int32_t* done, int32_t* nerr);
int bsr_get_err_trace(bsr_handle* h, double* err /* [n_chains][err_cap] */);
/* Grow the per-chain capacity of that trace (entries are kept); bsr_get_err_cap returns the current one. */
int bsr_reserve_err(bsr_handle* h, int32_t err_cap);
int bsr_get_err_cap(bsr_handle* h, int32_t* err_cap);
int bsr_count_done(bsr_handle* h, int32_t* n_done);

/* allcal (codes/funcs.py:175-220) for arbitrary trees on the current data: out is host [n_trees][n] float64.
 * precision as in bsr_config. */
int bsr_eval_trees(bsr_handle* h, int32_t n_trees, const uint32_t* tok, const double* pa, const double* pb,
                   const int32_t* nn, int32_t precision, double* out);
/* Prediction: BSR.predict (codes/bsr_class.py:53-68) of model m on row i, evaluated in float64 on `device` (all but bsr_predict
 * need no handle, so a fitted or un-pickled estimator predicts without chain state on the device):
 *   pred_m(X[i]) = beta_m[0] + sum_k beta_m[k+1] * tree_mk(X[i]),  k in order.
 * A reducing call returns instead, row by row, the posterior-predictive mean over its models and their sample standard deviation,
 * reduced on the device in model order; a model whose prediction at a row is not finite is left out of that row, and n_used
 * returns the smallest number of models any row used (the model count without reduce).  This extends codes/bsr_class.py:53-68,
 * which reads one restart (SURVEY.md 8f 1).  All four entry points run the same kernels, so a model predicts the same bits through
 * each.  Refused on the host, before the device reads anything: null pointers; K outside 1 .. BSR_MAX_TREES; a tree of 0 or more
 * than 64 nodes, with an unknown opcode, whose tokens are not a pre-order tree or with a leaf feature >= d; a test set without rows
 * or of ld * d >= 2^32 elements (ld = its rows rounded up to 4).  The model count has no limit of its own.  The caller's device is
 * restored and every device buffer freed on every path, failures included.  On the device a call holds its inputs and its whole
 * output (a non-reducing call [M][n_test] of them), plus, for the models of reducing groups, a [models][chunk] scratch: rows go in
 * chunks that keep it near 256 MB (at least 256 rows a chunk).
 *
 * bsr_predict: one chain of a handle; reported != 0 uses the roots_ snapshot, else the live state. */
int bsr_predict(bsr_handle* h, int32_t chain, int32_t reported, const double* X_rowmajor, int64_t n_test, int32_t d,
                double* out);

/* K explicit trees (host arrays [K][BSR_MAX_NODES], beta [K+1]): out [n_test]. */
int bsr_predict_trees(int32_t device, int32_t K, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                      const double* beta, const double* X_rowmajor, int64_t n_test, int32_t d, double* out);

/* M models at once -- the restarts of one fit (host arrays [M][K][BSR_MAX_NODES], nn [M][K], beta [M][K+1]).  reduce == 0: out is
 * [M][n_test]; reduce != 0: out is [2][n_test] (mean, then std).  n_used may be NULL. */
int bsr_predict_many(int32_t device, int32_t M, int32_t K, const uint32_t* tok, const double* pa, const double* pb, const int32_t* nn,
                     const double* beta, const double* X_rowmajor, int64_t n_test, int32_t d, int32_t reduce, double* out,
                     int32_t* n_used);

/* Many models on many test sets in one call -- the fits of BSR.fit_many, each on its own test set.
 * Models, in the packed layout of bsr_read_packed: nn [M][K] node counts; tok the n_tok tokens of tree after tree (tree m * K + k
 * holds nn[m][k]); ab [n_lt][2] the (a, b) pairs of the lt nodes in node order; beta [M][K+1].
 * Test sets: X_rowmajor holds the rows of S sets of d features one after another, set s is rows set_off[s] .. set_off[s+1].
 * Groups: group g evaluates the models grp_models[grp_off[g] .. grp_off[g+1]) on set grp_set[g].
 * out holds the groups' blocks in group order: [n_models_g][n_rows_s] predictions, or, when grp_reduce[g] != 0, [2][n_rows_s] (mean,
 * then std); n_used [G].  Also refused: node counts that do not cover tok, lt nodes that do not match n_lt, set_off or grp_off that
 * do not start at 0 or decrease, a group without models, a model index outside [0, M) or a set index outside [0, S). */
int bsr_predict_groups(int32_t device, int32_t M, int32_t K, const int32_t* nn, const uint32_t* tok, int64_t n_tok, const double* ab,
                       int64_t n_lt, const double* beta, int32_t S, int32_t d, const double* X_rowmajor, const int64_t* set_off,
                       int32_t G, const int32_t* grp_set, const int64_t* grp_off, const int32_t* grp_models, const int32_t* grp_reduce,
                       double* out, int32_t* n_used);

/* Timing helper for bench.py: accumulated device time (ms) and launch counts of the sweeps run while enabled, per
 * stage (0 propose, 1 evaluation stage as a whole, 2 resolve, 3 k_trees alone, 4 Gram kernel alone), measured with
 * CUDA events on the run's stream.  While enabled, bsr_run uses a single chain group and synchronises every sweep. */
int bsr_set_profiling(bsr_handle* h, int32_t enabled);
int bsr_get_profile(bsr_handle* h, double* ms /* [5] */, int64_t* launches /* [5] */);

#ifdef __cplusplus
}
#endif
#endif /* BSR_B200_H */
