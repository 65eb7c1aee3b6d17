// Host-side handle shared by the translation units of libbsr_b200.so (not part of the public ABI).
#pragma once
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "bsr_common.cuh"

struct bsr_handle {
  bsr_config cfg;
  // prior tables, one per distinct feature count of the data sets (ascending; one entry on a handle of one feature count), in
  // global memory: the kernels read them there.  chain_pt [C] (device): the table of every chain's data set.
  PriorTables* d_pt = nullptr;
  int n_pt = 0;
  int* chain_pt = nullptr;
  ChainState st;
  std::vector<void*> allocs;
  // data: n_ds data sets, X column-major [n_ds][d][ld], y [n_ds][ld]; data set b holds ds_n[b] rows (n: the largest, ld: n rounded
  // up to 4), zeros past them, and ds_d[b] features (d: the largest), zero columns past them that no chain of it reads
  float* X32 = nullptr; double* X64 = nullptr; float* y32 = nullptr; double* y64 = nullptr;
  int n_ds = 1;
  uint32_t* ds_n = nullptr;      // [n_ds] (device)
  std::vector<int32_t> ds_d;     // [n_ds] (host)
  std::vector<int32_t> chain_ds; // [C] (host copy of st.ds)
  bool mixed = false;            // the data sets differ in feature count
  bool own_x32 = false;
  double* stage = nullptr;       // device staging of the host data and its row offsets (bsr_set_data_host / bsr_set_datasets_*host)
  size_t stage_bytes = 0;
  void* gt_dev = nullptr; void* gt_host = nullptr; size_t gt_bytes = 0;   // gather staging of bsr_get_trees (device, pinned host)
  void* pk_head = nullptr; size_t pk_head_bytes = 0;   // packed results (bsr_pack_trees): counts / offsets / node counts / scan scratch
  void* pk_body = nullptr; size_t pk_body_bytes = 0;   //                                   lt parameter pairs, then tokens
  long long pk_nodes = 0, pk_lt = 0;
  int64_t n = 0, ld = 0, n_total = 0;
  int d = 0;
  bool y_stats_external = false;
  // sweep buffers
  double* gram = nullptr;   // [C][n_sum] then [C][P]
  int* need64 = nullptr;
  int* split_cnt = nullptr;      // [C] arrival counters of row-split eval launches
  double* part = nullptr;        // row-split partial records
  size_t part_cap = 0;
  int* d_count = nullptr;
  double* ystats = nullptr;      // [n_ds][2] sum(y), y'y of every data set (row-sharded handles: the global values, bsr_set_y_stats)
  double sum_y = 0, yy = 0;      // entry 0 of ystats on the host: the window kernels of one data set take it by value
  int64_t sweep = 0;
  bool initialised = false;
  bool col_cache_wanted = false;
  bool needs_refit = false;   // data changed under initialised chains: recompute the live fit + caches before the next sweep
  // tape / trace / record
  double* tape = nullptr; int64_t* tape_off = nullptr; double* trace = nullptr;
  int tape_steps = 0, tape_pos = 0; bool tape_mode = false;
  double* rec = nullptr; int* rec_count = nullptr; int rec_steps = 0, rec_cap = 0, rec_pos = 0;
  // profiling
  bool profiling = false;
  double prof_ms[6] = {0, 0, 0, 0, 0, 0};      // propose, eval (whole stage), resolve, k_trees / k_weval, Gram kernel / k_weval_fix, exchange (k_wsignal + k_wwait)
  long long prof_launches[6] = {0, 0, 0, 0, 0, 0};
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [4],[5]: after k_trees / after the Gram kernel; [6]: before the exchange
  bool prof_inner = false;                       // set while bsr_run profiles: bsr_launch_eval records ev[4], ev[5]
  int threads_eval = 128;
  // speculative-window path (bsr_tu_window.cu)
  WinState ws = WinState();
  size_t ws_rec_doubles = 0;
  int* h_count = nullptr;        // pinned [2]: number of chains that still have proposals to consume, abort flag of k_wwait
  double* lrec = nullptr;        // [C][S][sg_size(K)] partial Grams of the live columns (k_wlive_gram), single-device handles
  size_t lrec_doubles = 0;
  bool sg_dirty = true;          // the live Gram / SSE / intercept fit must be rebuilt by the next window (set by every initial fit)
  int* d_abort = nullptr;        // device flag: a peer never signalled (k_wwait timed out)
  double peer_timeout_s = 120.0; // wall-clock limit of one k_wwait (bsr_set_peer_timeout; <= 0: wait for ever)
  // proposed-tree log of the trace window (bsr_trace_trees)
  uint32_t* log_tok = nullptr; double* log_pa = nullptr; double* log_pb = nullptr; int* log_nn = nullptr;
  int window = 64;               // proposals per window (1..64)
  // row-sharded windows over peer memory (bsr_peer_export / bsr_peer_import)
  unsigned char* xbuf = nullptr; size_t xbuf_bytes = 0;    // local exchange buffer: records[2] | masks[2] | flags
  size_t x_rec_doubles = 0;                                // doubles per parity of the record area
  size_t x_lrec_doubles = 0;                               // doubles of the live-Gram partials behind the flags
  int x_world = 0, x_rank = 0;
  void* x_peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // peers' xbuf (own entry = xbuf)
  unsigned long long x_ticket = 0;
  bool seq_pipeline = false;     // BSR_SEQ_PIPELINE=1: bsr_run uses the proposal-by-proposal pipeline (A/B measurements)
  int n_groups = 4;   // chain groups pipelined on separate streams inside bsr_run (sequential pipeline)
  int win_groups = 2; // same for the window path: two groups let the scalar kernels of one fill the tail waves of the other's k_weval
                      // (measured at C2: 1 group 315, 2 groups 330, 4 groups 304 M proposals/s; profiles/README.md r02)
  std::vector<cudaStream_t> gstreams;
  std::vector<cudaEvent_t> gevents;
  cudaEvent_t fork_event = nullptr;
  long long launches = 0;   // kernel launches issued by bsr_run since the last bsr_set_profiling
};


// error plumbing (bsr_capi.cu)
int bsr_fail(const std::string& m);
#define CK(x)                                                                                        \
  do {                                                                                               \
    cudaError_t e_ = (x);                                                                            \
    if (e_ != cudaSuccess) {                                                                         \
      char buf_[512];                                                                                \
      snprintf(buf_, sizeof buf_, "%s:%d %s -> %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      return bsr_fail(buf_);                                                                         \
    }                                                                                                \
  } while (0)

// kernel launch wrappers, one translation unit each so they compile in parallel
struct ResolveCtx;
struct ProposeCtx;
// every launcher works on the chain range [c0, c0 + cn)
int bsr_launch_eval(bsr_handle* h, cudaStream_t s, int init_only, int c0, int cn);         // bsr_tu_eval.cu
int bsr_launch_resolve(bsr_handle* h, cudaStream_t s, int init_only, int c0, int cn);      // bsr_tu_resolve.cu
int bsr_launch_propose(bsr_handle* h, cudaStream_t s, int c0, int cn);                     // bsr_tu_propose.cu
int bsr_launch_init_chains(bsr_handle* h, cudaStream_t s);                                 // bsr_tu_propose.cu
int bsr_run_window(bsr_handle* h, int n_sweeps, cudaStream_t s);                           // bsr_tu_window.cu
int bsr_window_refit(bsr_handle* h, cudaStream_t s);                                       // bsr_tu_window.cu
void bsr_window_free(bsr_handle* h);
