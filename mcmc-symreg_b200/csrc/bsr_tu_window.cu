// Speculative-window driver of bsr_run (kernels: bsr_window.cuh): launches, buffers, completion loop.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "bsr_handle.h"
#include "bsr_window.cuh"

// BSR_WIN_TRACE=1: device timeline of the kernels of one bsr_run call (start / end of every launch relative to the first
// one, per chain group) on stderr -- a diagnostic for the stream-level overlap of the groups.
struct TraceRec { const char* label; int group; cudaEvent_t a, b; };
static std::vector<TraceRec> g_trace;
static bool g_trace_on = false;
static void trace_begin(const char* label, int group, cudaStream_t s) {
  if (!g_trace_on) return;
  TraceRec r; r.label = label; r.group = group;
  cudaEventCreate(&r.a); cudaEventCreate(&r.b);
  cudaEventRecord(r.a, s);
  g_trace.push_back(r);
}
static void trace_end(cudaStream_t s) { if (g_trace_on) cudaEventRecord(g_trace.back().b, s); }
static void trace_dump() {
  if (!g_trace_on || g_trace.empty()) return;
  cudaDeviceSynchronize();
  for (auto& r : g_trace) {
    float t0 = 0, t1 = 0;
    cudaError_t e0 = cudaEventElapsedTime(&t0, g_trace[0].a, r.a), e1 = cudaEventElapsedTime(&t1, g_trace[0].a, r.b);
    if (e0 != cudaSuccess || e1 != cudaSuccess) fprintf(stderr, "[trace] error %s / %s\n", cudaGetErrorString(e0), cudaGetErrorString(e1));
    fprintf(stderr, "[trace] g%d %-9s %9.1f -> %9.1f us (%7.1f)\n", r.group, r.label, t0 * 1e3, t1 * 1e3, (t1 - t0) * 1e3);
  }
  for (auto& r : g_trace) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_trace.clear();
}

static int win_alloc(void** p, size_t bytes, bool zero) {
  CK(cudaMalloc(p, bytes ? bytes : 16));
  if (zero) CK(cudaMemset(*p, 0, bytes ? bytes : 16));
  return 0;
}

void bsr_window_free(bsr_handle* h) {
  WinState& ws = h->ws;
  cudaFree(ws.tok); cudaFree(ws.pa); cudaFree(ws.pb); cudaFree(ws.nn); cudaFree(ws.info); cudaFree(ws.rec);
  cudaFree(ws.bad); cudaFree(ws.rep); cudaFree(ws.pos); cudaFree(ws.bucket); cudaFree(ws.bucket_count);
  cudaFree(ws.hash); cudaFree(ws.chead); cudaFree(ws.cvalid); cudaFree(ws.prevslot); cudaFree(ws.order); cudaFree(ws.neval);
  cudaFree(ws.lcol); cudaFree(ws.lcol_ok); cudaFree(ws.lcol_wide);
  ws = WinState();
  h->ws_rec_doubles = 0;
  if (h->lrec) { cudaFree(h->lrec); h->lrec = nullptr; }
  h->lrec_doubles = 0;
  if (h->h_count) { cudaFreeHost(h->h_count); h->h_count = nullptr; }
  for (int r = 0; r < 8; ++r) {
    if (h->x_peer[r] && h->x_peer[r] != (void*)h->xbuf) cudaIpcCloseMemHandle(h->x_peer[r]);
    h->x_peer[r] = nullptr;
  }
  if (h->xbuf) { cudaFree(h->xbuf); h->xbuf = nullptr; }
  h->x_world = 0;
}

// Geometry of the evaluation kernels for the current data: row splits and the shared-memory row tile.
//
// Tile: a warp covers a tile in steps of 4 row vectors x 32 lanes = 512 rows, so the tile is 1024 rows (two full steps) wherever the
// block's shared memory then still admits the resident blocks the register file admits (3 for K <= 5, 2 above), else the
// largest tile that does (K = 10: 972 rows).  Measured at C4 (K = 5, n = 5000): 852-row tiles 40.8 ms per window, 1024: 36.3,
// 1280: 46.6, 768: 42.7; at C3 (K = 10, n = 10 k): 1024 rows (one resident block) 332 ms, 768: 237, 896: 223, 960: 210; C5: 488 -> 460.
//
// Splits: with few chains the rows are split over blockIdx.y.  One block per (chain, split) runs for as long as its chain's trees
// take, and chains differ by a factor of five in distinct proposals x tree sizes, so the blocks must be many more than the GPU
// holds at once (3 x 148) for the tail to even out: about 28 waves, as long as a split keeps >= 8192 rows.  Measured at C5
// (256 chains x 12.5 M rows, 1024-row tiles): 3 splits 460 ms per window, 12: 309, 24: 281, 48: 268, 96: 262, 192: 260.
static int win_splits(int cn, int64_t n_rows) {
  const int want = (148 * 3 * 28 + cn - 1) / cn;
  const int max_s = (int)std::max<int64_t>(1, n_rows / 8192);
  return std::max(1, std::min(std::min(want, max_s), 4096));
}
static void win_geometry(bsr_handle* h, int cn, int* S, uint32_t* rows_per_split, uint32_t* TR) {
  const int K = h->cfg.K;
  const int64_t n = h->n;
  const bool sharded = h->cfg.row_sharded && h->x_world > 0;
  // (every rank of a row-sharded handle must use the same split count: derived from the global shape)
  int s = win_splits(cn, sharded ? std::max<int64_t>(1, h->n_total / std::max(1, h->x_world)) : n);
  if (const char* e = getenv("BSR_WIN_SPLITS")) s = std::max(1, atoi(e));
  const int resident = (K <= 5) ? 3 : 2;                          // blocks per SM the launch bounds of k_weval ask for
  const size_t limit = (size_t)233472 / resident - 1024;          // 228 KB of shared memory per SM, 1 KB reserved per block
  const int W = std::max(1, std::min(h->window, BSR_MAXW)), NW = BSR_WEVAL_THREADS / 32;
  int64_t tr = 1024;
  while (tr > 4 && (h->cfg.precision == 0 ? win_smem_layout<float>(K, W, NW, (uint32_t)tr).total : win_smem_layout<double>(K, W, NW, (uint32_t)tr).total) > limit) tr -= 4;
  if (const char* e = getenv("BSR_WIN_TILE")) tr = std::max(4, atoi(e) / 4 * 4);
  int64_t rps = (n + s - 1) / s;
  rps = (rps + 3) / 4 * 4;
  if (rps > tr) rps = (rps + tr - 1) / tr * tr;                  // whole tiles per split (the last split takes what is left)
  if (!sharded) s = (int)((n + rps - 1) / rps);
  tr = std::min<int64_t>(tr, rps);
  *S = s; *rows_per_split = (uint32_t)rps; *TR = (uint32_t)tr;
}

static int ensure_window(bsr_handle* h, int S) {
  WinState& ws = h->ws;
  const int C = h->cfg.n_chains, K = h->cfg.K;
  int W = h->window;
  if (W < 1) W = 1;
  if (W > BSR_MAXW) W = BSR_MAXW;
  if (ws.tok == nullptr || ws.W != W) {
    CK(cudaDeviceSynchronize());
    bsr_window_free(h);
    const size_t CW = (size_t)C * W;
    // the per-slot arrays hold R windows per chain (WinState: the earlier windows are the record cache of the current one): as many
    // as BSR_WIN_RING, fewer when they would take more than a third of the free device memory (65536 chains: 5.4 GB per window)
    // (a handle with the stop rule on runs its chains for val consecutive rejections -- ~140 proposals per chain at val = 100, accepts every
    // hundred proposals: earlier windows are rarely valid, and a 30-ms fit should not allocate 2.7 GB: two windows)
    int R = h->cfg.val > 0 ? 2 : BSR_WIN_RING;
    if (const char* e = getenv("BSR_WIN_RING_DEPTH")) R = std::max(2, std::min(BSR_WIN_RING, atoi(e)));
    {
      size_t free_b = 0, total_b = 0;
      CK(cudaMemGetInfo(&free_b, &total_b));
      const size_t per_ring = CW * (BSR_MAXN * (sizeof(uint32_t) + 2 * sizeof(double)) + sizeof(int) + sizeof(PropInfo) + sizeof(unsigned long long) +
                                    (size_t)(K + 4) * sizeof(double));
      while (R > 2 && (size_t)R * per_ring > free_b / 3) --R;
    }
    const size_t RG = (size_t)R;
    if (win_alloc((void**)&ws.tok, RG * CW * BSR_MAXN * sizeof(uint32_t), false) || win_alloc((void**)&ws.pa, RG * CW * BSR_MAXN * sizeof(double), false) ||
        win_alloc((void**)&ws.pb, RG * CW * BSR_MAXN * sizeof(double), false) || win_alloc((void**)&ws.nn, RG * CW * sizeof(int), true) ||
        win_alloc((void**)&ws.info, RG * CW * sizeof(PropInfo), true) || win_alloc((void**)&ws.bad, RG * (size_t)C * sizeof(unsigned long long), true) ||
        win_alloc((void**)&ws.hash, RG * CW * sizeof(unsigned long long), true) ||
        win_alloc((void**)&ws.chead, (size_t)C, false) || win_alloc((void**)&ws.cvalid, (size_t)C, true) || win_alloc((void**)&ws.prevslot, CW * sizeof(unsigned short), true) || win_alloc((void**)&ws.order, CW, true) ||
        win_alloc((void**)&ws.neval, (size_t)C * sizeof(int), true) ||
        win_alloc((void**)&ws.pos, (size_t)C * sizeof(long long), true) || win_alloc((void**)&ws.rep, CW, true) ||
        win_alloc((void**)&ws.bucket, (size_t)BSR_N_BINS * CW * sizeof(int), false) ||
        win_alloc((void**)&ws.bucket_count, (size_t)16 * 32 * sizeof(int), true))
      return 1;
    CK(cudaMemset(ws.chead, 0xFF, (size_t)C));
    ws.W = W; ws.C = C; ws.R = R;
    CK(cudaHostAlloc((void**)&h->h_count, 2 * sizeof(int), cudaHostAllocDefault));
    h->h_count[0] = h->h_count[1] = 0;
  }
  const size_t need = (size_t)ws.R * C * S * W * (K + 4);
  if (need > h->ws_rec_doubles || ws.S != S) {
    CK(cudaDeviceSynchronize());
    if (need > h->ws_rec_doubles) {
      cudaFree(ws.rec); ws.rec = nullptr;
      if (win_alloc((void**)&ws.rec, need * sizeof(double), true)) return 1;
      h->ws_rec_doubles = need;
    }
    CK(cudaMemset(ws.chead, 0xFF, (size_t)C));     // the record layout changed: nothing cached is valid
  }
  // cache of live columns (fp32 mode): C x K x ld floats, if a quarter of the free device memory holds it -- and only in the
  // one-split geometry (many chains or few rows): with few chains on many rows the blocks of a split share their rows of X in L2,
  // while every chain's cached columns are its own (a C5 slice of 4 M rows read 18 GB per window from HBM and was 4 % slower)
  const long long lcol_key = (S == 1 && K > 5) ? (long long)h->ld : -1;      // (K > 5: see k_weval)
  if (h->cfg.precision == 0 && ws.lcol_ld != lcol_key) {
    CK(cudaDeviceSynchronize());
    cudaFree(ws.lcol); cudaFree(ws.lcol_ok); cudaFree(ws.lcol_wide);
    ws.lcol = nullptr; ws.lcol_ok = nullptr; ws.lcol_wide = nullptr;
    ws.lcol_ld = lcol_key;
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const size_t bytes = (size_t)C * K * (size_t)h->ld * sizeof(float);
    if (S == 1 && K > 5 && !getenv("BSR_WIN_NO_LCOL") && bytes <= free_b / 4) {
      if (win_alloc((void**)&ws.lcol, bytes, false) || win_alloc((void**)&ws.lcol_ok, (size_t)C * K, true) ||
          win_alloc((void**)&ws.lcol_wide, (size_t)C * sizeof(unsigned), true))
        return 1;
    }
  }
  const size_t need_l = (size_t)C * S * sg_size(K);
  if (need_l > h->lrec_doubles) {
    CK(cudaDeviceSynchronize());
    if (h->lrec) cudaFree(h->lrec);
    h->lrec = nullptr;
    if (win_alloc((void**)&h->lrec, need_l * sizeof(double), true)) return 1;
    h->lrec_doubles = need_l;
  }
  ws.S = S;
  return 0;
}

template <typename T, int KC, bool EXACT, bool MULTI>
static int launch_weval_t(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc, int threads) {
  const size_t smem = win_smem_layout<T>(h->cfg.K, ws.W, threads / 32, wc.TR, MULTI).total;
  CK(cudaFuncSetAttribute(k_weval<T, KC, EXACT, MULTI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    // leave the rest of the unified L1 / shared-memory array to L1: the interpreter's operand stack (local memory) and
    // the leaf loads of X live there.  Ask for just enough shared memory for the blocks the register file admits.
    const int resident = (KC <= 3 ? BSR_WEVAL_MINB3 : (KC <= 5 ? 3 : 2));
    const size_t need = (size_t)resident * (smem + 1024);
    int pct = (int)((need * 100 + 228 * 1024 - 1) / (228 * 1024));
    if (const char* e = getenv("BSR_WEVAL_CARVEOUT")) pct = atoi(e);
    CK(cudaFuncSetAttribute(k_weval<T, KC, EXACT, MULTI>, cudaFuncAttributePreferredSharedMemoryCarveout, std::min(100, std::max(0, pct))));
  }
  k_weval<T, KC, EXACT, MULTI><<<dim3(wc.cn, ws.S), threads, smem, s>>>(h->st, ws, wc);
  CK(cudaGetLastError());
  return 0;
}
template <typename T, int KC, bool EXACT>
static int launch_wlive_t(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc, int threads, double* lrec) {
  const size_t smem = win_smem_layout<T>(h->cfg.K, ws.W, threads / 32, wc.TR).total + (size_t)(threads / 32) * sg_size(h->cfg.K) * sizeof(double);
  CK(cudaFuncSetAttribute(k_wlive_gram<T, KC, EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_wlive_gram<T, KC, EXACT><<<dim3(wc.cn, ws.S), threads, smem, s>>>(h->st, ws, wc, lrec);
  CK(cudaGetLastError());
  return 0;
}

#ifdef BSR_DEV_K3   // development builds only: one instantiation, for quick SASS inspection
#define BSR_WIN_DISPATCH(CALL_EXACT, CALL_GENERIC) return CALL_EXACT(3);
#else
#define BSR_WIN_DISPATCH(CALL_EXACT, CALL_GENERIC)  \
  switch (h->cfg.K) {                               \
    case 1: return CALL_EXACT(1);                   \
    case 2: return CALL_EXACT(2);                   \
    case 3: return CALL_EXACT(3);                   \
    case 4: return CALL_EXACT(4);                   \
    case 5: return CALL_EXACT(5);                   \
    case 10: return CALL_EXACT(10);                 \
    default: return CALL_GENERIC();                 \
  }
#endif

template <bool MULTI>
static int launch_weval_m(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc, int threads) {
  if (h->cfg.precision == 0) {
#define EX(KC) launch_weval_t<float, KC, true, MULTI>(h, ws, s, wc, threads)
#define GEN() launch_weval_t<float, BSR_MAXK, false, MULTI>(h, ws, s, wc, threads)
    BSR_WIN_DISPATCH(EX, GEN)
#undef EX
#undef GEN
  }
#define EX(KC) launch_weval_t<double, KC, true, MULTI>(h, ws, s, wc, threads)
#define GEN() launch_weval_t<double, BSR_MAXK, false, MULTI>(h, ws, s, wc, threads)
  BSR_WIN_DISPATCH(EX, GEN)
#undef EX
#undef GEN
}
// a handle of one data set runs the instances without a data-set term (k_weval)
static int launch_weval(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc, int threads) {
  return h->n_ds > 1 ? launch_weval_m<true>(h, ws, s, wc, threads) : launch_weval_m<false>(h, ws, s, wc, threads);
}
static int launch_wlive(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc, int threads, double* lrec) {
  if (h->cfg.precision == 0) {
#define EX(KC) launch_wlive_t<float, KC, true>(h, ws, s, wc, threads, lrec)
#define GEN() launch_wlive_t<float, BSR_MAXK, false>(h, ws, s, wc, threads, lrec)
    BSR_WIN_DISPATCH(EX, GEN)
#undef EX
#undef GEN
  }
#define EX(KC) launch_wlive_t<double, KC, true>(h, ws, s, wc, threads, lrec)
#define GEN() launch_wlive_t<double, BSR_MAXK, false>(h, ws, s, wc, threads, lrec)
  BSR_WIN_DISPATCH(EX, GEN)
#undef EX
#undef GEN
}
// group: index of the chain group (its own move counters); the buckets of a launch live at offset c0 * W of each
// move's array, so concurrent groups never overlap.
static int launch_wpropose(bsr_handle* h, const WinState& ws, cudaStream_t s, WinCtx& wc, int group) {
  const int W = ws.W;
  const int total = wc.cn * W;
  wc.bucket_stride = h->cfg.n_chains * W;
  wc.bucket = h->ws.bucket + (size_t)wc.c0 * W;
  wc.bucket_count = h->ws.bucket_count + group * 32;
  CK(cudaMemsetAsync(wc.bucket_count, 0, 32 * sizeof(int), s));
  k_wclassify<<<(total + 255) / 256, 256, 0, s>>>(h->st, ws, wc);
  const int threads = 64;
  const dim3 blocks((total + threads - 1) / threads + BSR_N_BINS);
  if (wc.tape != nullptr) k_wpropose<1><<<blocks, threads, 0, s>>>(h->st, ws, h->d_pt, wc, h->chain_pt);
  else if (wc.rec_draws != nullptr) k_wpropose<2><<<blocks, threads, 0, s>>>(h->st, ws, h->d_pt, wc, h->chain_pt);
  else k_wpropose<0><<<blocks, threads, 0, s>>>(h->st, ws, h->d_pt, wc, h->chain_pt);
  k_wdedup<<<wc.cn, BSR_MAXW, 0, s>>>(h->st, ws, wc);
  CK(cudaGetLastError());
  return 0;
}

template <bool MULTI>
static int launch_wresolve_m(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc) {
  const int K = h->cfg.K;
  const int threads = 128, lpc = ws.W > 32 ? 64 : 32, cpb = threads / lpc, blocks = (wc.cn + cpb - 1) / cpb;
  const size_t smem = (size_t)cpb * (sg_size(K) * sizeof(double) + 8 * sizeof(unsigned));
  switch (K) {
    case 1: k_wresolve<1, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
    case 2: k_wresolve<2, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
    case 3: k_wresolve<3, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
    case 4: k_wresolve<4, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
    case 5: k_wresolve<5, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
    case 10: k_wresolve<10, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;     // BASELINE configs[2]
    default: k_wresolve<0, MULTI><<<blocks, threads, smem, s>>>(h->st, ws, wc); break;
  }
  CK(cudaGetLastError());
  return 0;
}
static int launch_wresolve(bsr_handle* h, const WinState& ws, cudaStream_t s, const WinCtx& wc) {
  return h->n_ds > 1 ? launch_wresolve_m<true>(h, ws, s, wc) : launch_wresolve_m<false>(h, ws, s, wc);
}

static WinCtx make_wc(bsr_handle* h, long long p_start, long long p_target, uint32_t rps, uint32_t TR) {
  WinCtx wc;
  wc.p_target = p_target;
  wc.c0 = 0; wc.cn = h->cfg.n_chains;
  const bool recording = h->rec != nullptr && h->rec_pos < h->rec_steps;
  wc.rec_draws = recording ? h->rec : nullptr; wc.rec_count = h->rec_count; wc.rec_steps = h->rec_steps; wc.rec_cap = h->rec_cap;
  wc.rec_origin = p_start - h->rec_pos;
  const bool tracing = h->trace != nullptr && h->tape_pos < h->tape_steps;
  wc.trace = tracing ? h->trace : nullptr; wc.trace_steps = h->tape_steps; wc.trace_origin = p_start - h->tape_pos;
  const bool taped = h->tape_mode && h->tape_pos < h->tape_steps;
  wc.tape = taped ? h->tape : nullptr; wc.tape_off = h->tape_off;
  wc.log_tok = tracing ? h->log_tok : nullptr; wc.log_pa = h->log_pa; wc.log_pb = h->log_pb; wc.log_nn = h->log_nn;
  wc.X32 = h->X32; wc.X64 = h->X64; wc.y64 = h->y64;
  wc.n = (uint32_t)h->n; wc.ld = (uint32_t)h->ld; wc.ds_stride = (uint32_t)(h->d * h->ld); wc.precision = h->cfg.precision;
  wc.rows_per_split = rps; wc.TR = TR;
  // 2: repeated trees are interpreted once per window AND trees of the chain's earlier windows in the ring take their record from there;
  // 1: within the window only (BSR_WIN_NO_CACHE); 0: every slot is interpreted (BSR_WIN_NO_DEDUP) -- for A/B runs and tests
  wc.dedup = getenv("BSR_WIN_NO_DEDUP") ? 0 : (getenv("BSR_WIN_NO_CACHE") ? 1 : 2);
  wc.checked_m = getenv("BSR_WIN_NO_CHECKED") ? (1 << 30) : BSR_CHECKED_M;      // (A/B runs and tests)
  wc.n_total = (double)h->n_total; wc.n_local = (double)h->n; wc.sum_y = h->sum_y; wc.yy = h->yy; wc.ystats = h->ystats;
  wc.pivot_tol = h->cfg.precision == 1 ? 1e-13 : 3e-13;
  wc.n_peers = 0;
  for (int r = 0; r < BSR_MAX_PEERS; ++r) { wc.peer_rec[r] = nullptr; wc.peer_bad[r] = nullptr; wc.peer_lrec[r] = nullptr; }
  wc.peer_lrec[0] = h->lrec;
  wc.abort_flag = nullptr;
  wc.ds_n = h->n_ds > 1 ? h->ds_n : nullptr;
  return wc;
}

// Exchange-buffer layout of a row-sharded handle: records of the two window parities, their out-of-range masks, flags.
static double* x_rec(void* base, size_t rec_doubles, int parity) { return (double*)base + (size_t)parity * rec_doubles; }
static unsigned long long* x_bad(void* base, size_t rec_doubles, int C, int parity) {
  return (unsigned long long*)((double*)base + 2 * rec_doubles) + (size_t)parity * C;
}
static unsigned long long* x_flags(void* base, size_t rec_doubles, int C) {
  return (unsigned long long*)((double*)base + 2 * rec_doubles) + 2 * (size_t)C;
}
static double* x_lrec(void* base, size_t rec_doubles, int C) { return (double*)(x_flags(base, rec_doubles, C) + BSR_MAX_PEERS); }

// One window iteration of the chain range [c0, c0 + cn) on stream s.
static int window_iteration(bsr_handle* h, cudaStream_t s, WinCtx wc, int c0, int cn, bool profile, int group = 0) {
  wc.c0 = c0; wc.cn = cn;
  const int threads = BSR_WEVAL_THREADS;
  const int C = h->cfg.n_chains;
  WinState ws = h->ws;
  const bool peers = h->x_world > 1;
  int parity = 0;
  if (peers) {   // this window's records / masks live in the exchange buffer (double-buffered by window parity)
    ++h->x_ticket;
    parity = (int)(h->x_ticket & 1ull);
    ws.rec = x_rec(h->xbuf, h->x_rec_doubles, parity);
    ws.bad = x_bad(h->xbuf, h->x_rec_doubles, C, parity);
  }
  if (profile) cudaEventRecord(h->ev[0], s);
  trace_begin("propose", group, s);
  if (launch_wpropose(h, ws, s, wc, group)) return 1;
  trace_end(s);
  if (profile) cudaEventRecord(h->ev[1], s);
  trace_begin("eval", group, s);
  if (launch_weval(h, ws, s, wc, threads)) return 1;
  trace_end(s);
  if (profile) cudaEventRecord(h->ev[4], s);
  int nl = 5;
  if (profile) cudaEventRecord(h->ev[6], s);
  if (peers) {
    PeerFlagPtrs pf;
    wc.n_peers = h->x_world;
    for (int r = 0; r < h->x_world; ++r) {
      pf.p[r] = x_flags(h->x_peer[r], h->x_rec_doubles, C);
      wc.peer_rec[r] = x_rec(h->x_peer[r], h->x_rec_doubles, parity);
      wc.peer_bad[r] = x_bad(h->x_peer[r], h->x_rec_doubles, C, parity);
      wc.peer_lrec[r] = x_lrec(h->x_peer[r], h->x_rec_doubles, C);
    }
    wc.abort_flag = h->d_count + 1;
    const unsigned long long timeout_ns = h->peer_timeout_s > 0 ? (unsigned long long)(h->peer_timeout_s * 1e9) : 0ull;
    k_wsignal<<<1, 32, 0, s>>>(pf, h->x_world, h->x_rank, h->x_ticket);
    k_wwait<<<1, 32, 0, s>>>(x_flags(h->xbuf, h->x_rec_doubles, C), h->x_world, h->x_ticket, timeout_ns, h->d_count + 1);
    CK(cudaGetLastError());
    nl += 2;
  }
  if (profile) cudaEventRecord(h->ev[2], s);
  trace_begin("resolve", group, s);
  if (launch_wresolve(h, ws, s, wc)) return 1;
  trace_end(s);
  if (profile) {
    cudaEventRecord(h->ev[3], s);
    cudaEventSynchronize(h->ev[3]);
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->prof_ms[0] += ms;
    cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]); h->prof_ms[1] += ms;
    cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]); h->prof_ms[2] += ms;
    cudaEventElapsedTime(&ms, h->ev[1], h->ev[4]); h->prof_ms[3] += ms;
    cudaEventElapsedTime(&ms, h->ev[4], h->ev[6]); h->prof_ms[4] += ms;
    cudaEventElapsedTime(&ms, h->ev[6], h->ev[2]); h->prof_ms[5] += ms;      // k_wsignal + k_wwait: the exchange
    for (int p = 0; p < 6; ++p) h->prof_launches[p] += 1;
  }
  h->launches += nl;
  return 0;
}

static int ensure_group_streams(bsr_handle* h, int G) {
  while ((int)h->gstreams.size() < G) {
    cudaStream_t st; cudaEvent_t ev;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    h->gstreams.push_back(st); h->gevents.push_back(ev);
  }
  if (!h->fork_event) CK(cudaEventCreateWithFlags(&h->fork_event, cudaEventDisableTiming));
  return 0;
}

// Refit of every chain's live state with the window path's own evaluation: which live columns leave the fp32 range
// (k_wlive_bad), the partial Grams of the live columns (k_wlive_gram), then -- after the hand-over between the ranks of a
// row-sharded handle -- the live Gram, the K-column SSE and the intercept fit (k_wrefit).  Called by every initial fit
// (bsr_init_chains, bsr_set_state, data replaced under live chains) of a handle that runs in windows, and by the first
// bsr_run of a row-sharded handle once its peers are mapped.
int bsr_window_refit(bsr_handle* h, cudaStream_t s) {
  const int C = h->cfg.n_chains, K = h->cfg.K;
  int S; uint32_t rps, TR;
  win_geometry(h, C, &S, &rps, &TR);
  if (ensure_window(h, S)) return 1;
  const bool peers = h->x_world > 1;
  if (peers && h->x_lrec_doubles != (size_t)C * S * sg_size(K))
    return bsr_fail("bsr_run: data shape changed after bsr_peer_export: export and import again");
  WinCtx wc = make_wc(h, 0, 0, rps, TR);
  wc.c0 = 0; wc.cn = C;
  const int threads = BSR_WEVAL_THREADS;
  CK(cudaMemsetAsync(h->ws.chead, 0xFF, (size_t)C, s));   // the live state is being refitted: no window of the past is a record cache
  if (h->ws.lcol_ok) CK(cudaMemsetAsync(h->ws.lcol_ok, 0, (size_t)C * K, s));   // ... and no cached column is a live tree's
  k_wlive_prior<<<(C * K + 127) / 128, 128, 0, s>>>(h->st, h->d_pt, h->chain_pt);
  if (h->cfg.precision == 0) {
    CK(cudaMemsetAsync(h->st.live_bad, 0, (size_t)C * K, s));
    k_wlive_bad<<<dim3(C, S), threads, 0, s>>>(h->st, wc, S);
    CK(cudaGetLastError());
  }
  double* lrec = peers ? x_lrec(h->xbuf, h->x_rec_doubles, C) : h->lrec;
  if (launch_wlive(h, h->ws, s, wc, threads, lrec)) return 1;
  wc.peer_lrec[0] = lrec;
  if (peers) {
    ++h->x_ticket;
    PeerFlagPtrs pf;
    wc.n_peers = h->x_world;
    for (int r = 0; r < h->x_world; ++r) {
      pf.p[r] = x_flags(h->x_peer[r], h->x_rec_doubles, C);
      wc.peer_lrec[r] = x_lrec(h->x_peer[r], h->x_rec_doubles, C);
    }
    wc.abort_flag = h->d_count + 1;
    CK(cudaMemsetAsync(h->d_count + 1, 0, sizeof(int), s));
    const unsigned long long timeout_ns = h->peer_timeout_s > 0 ? (unsigned long long)(h->peer_timeout_s * 1e9) : 0ull;
    k_wsignal<<<1, 32, 0, s>>>(pf, h->x_world, h->x_rank, h->x_ticket);
    k_wwait<<<1, 32, 0, s>>>(x_flags(h->xbuf, h->x_rec_doubles, C), h->x_world, h->x_ticket, timeout_ns, h->d_count + 1);
  }
  k_wrefit<<<(C + 63) / 64, 64, 0, s>>>(h->st, wc, S, 0, C);
  CK(cudaGetLastError());
  h->launches += 4 + (peers ? 2 : 0);
  h->sg_dirty = false;
  return 0;
}

// n_sweeps sweeps for every live chain: windows are issued until every chain has consumed its n_sweeps * K proposals
// (or stopped).  The number of windows a chain needs depends on its accepts, so the loop reads back the number of
// unfinished chains between batches of launches; it returns with all work complete (the call synchronises).
int bsr_run_window(bsr_handle* h, int n_sweeps, cudaStream_t s) {
  const int C = h->cfg.n_chains, K = h->cfg.K;
  if (n_sweeps <= 0) return 0;
  g_trace_on = getenv("BSR_WIN_TRACE") != nullptr;
  int S; uint32_t rps, TR;
  win_geometry(h, C, &S, &rps, &TR);
  if (ensure_window(h, S)) return 1;
  const int W = h->ws.W;
  if (h->x_world > 1 && h->x_rec_doubles != (size_t)C * S * W * (K + 4))
    return bsr_fail("bsr_run: window size / data shape changed after bsr_peer_export: export and import again");
  const long long p_start = (long long)h->sweep * K, p_target = p_start + (long long)n_sweeps * K;
  WinCtx wc = make_wc(h, p_start, p_target, rps, TR);
  if (h->tape_mode && h->tape_pos < h->tape_steps && h->tape_pos + (long long)n_sweeps * K > h->tape_steps)
    return bsr_fail("bsr_run: the tape holds fewer proposals than this call would consume (bsr_set_tape)");
  k_wprep<<<(C + 255) / 256, 256, 0, s>>>(h->ws, C, p_start);
  CK(cudaGetLastError());
  CK(cudaMemsetAsync(h->d_count + 1, 0, sizeof(int), s));
  if (h->sg_dirty && bsr_window_refit(h, s)) return 1;   // first run after an initial fit on a row-sharded handle: refit through the peers
  int G = (h->profiling || h->x_world > 1) ? 1 : std::min(h->win_groups, std::max(1, C / 256));
  if (G > 1 && ensure_group_streams(h, G)) return 1;
  long long remaining_windows = ((long long)n_sweeps * K + W - 1) / W;
  int batch = (int)std::min<long long>(remaining_windows, 1 << 20);
  for (int guard = 0; guard < (1 << 24); ++guard) {
    if (G <= 1) {
      for (int it = 0; it < batch; ++it)
        if (window_iteration(h, s, wc, 0, C, h->profiling && guard == 0)) return 1;   // stage times: full windows only, not the stragglers' rounds
    } else {
      CK(cudaEventRecord(h->fork_event, s));
      for (int g = 0; g < G; ++g) CK(cudaStreamWaitEvent(h->gstreams[g], h->fork_event, 0));
      for (int it = 0; it < batch; ++it)
        for (int g = 0; g < G; ++g) {
          const int c0 = (int)((int64_t)C * g / G), c1 = (int)((int64_t)C * (g + 1) / G);
          if (window_iteration(h, h->gstreams[g], wc, c0, c1 - c0, false, g)) return 1;
        }
      for (int g = 0; g < G; ++g) {
        CK(cudaEventRecord(h->gevents[g], h->gstreams[g]));
        CK(cudaStreamWaitEvent(s, h->gevents[g], 0));
      }
    }
    CK(cudaMemsetAsync(h->d_count, 0, sizeof(int), s));
    k_wcount<<<(C + 255) / 256, 256, 0, s>>>(h->st, h->ws, p_target, h->d_count);
    CK(cudaMemcpyAsync(h->h_count, h->d_count, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (h->h_count[1] != 0) {
      char msg[200];
      snprintf(msg, sizeof msg, "bsr_run: rank %d never delivered its partial sums of a window within %.0f s (peer-memory exchange, "
               "bsr_set_peer_timeout); the chains were left at the last resolved window", h->h_count[1] - 1, h->peer_timeout_s);
      return bsr_fail(msg);
    }
    const int left = h->h_count[0];
    if (left == 0) break;
    // stragglers: every accept costs its chain at most one extra window
    batch = (left > C / 8) ? 2 : 1;
  }
  trace_dump();
  h->sweep += n_sweeps;
  const int adv = n_sweeps * K;
  if (h->tape_pos < h->tape_steps) h->tape_pos = std::min(h->tape_steps, h->tape_pos + adv);
  if (h->rec != nullptr && h->rec_pos < h->rec_steps) h->rec_pos = std::min(h->rec_steps, h->rec_pos + adv);
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// row-sharded windows over peer memory
// ---------------------------------------------------------------------------------------------------------------
extern "C" {

int bsr_get_window_geometry(bsr_handle* h, int64_t* geom5) {
  if (!h || !geom5) return bsr_fail("bsr_get_window_geometry: null argument");
  if (!h->X32) return bsr_fail("bsr_get_window_geometry: call bsr_set_data_* first");
  int S; uint32_t rps, TR;
  win_geometry(h, h->cfg.n_chains, &S, &rps, &TR);
  geom5[0] = S; geom5[1] = rps; geom5[2] = TR; geom5[3] = h->ws.R; geom5[4] = std::max(1, std::min(h->window, BSR_MAXW));
  return 0;
}

int bsr_peer_export(bsr_handle* h, int32_t world, void* ipc_handle_out) {
  if (!h || !ipc_handle_out) return bsr_fail("bsr_peer_export: null argument");
  if (h->n_ds > 1) return bsr_fail("bsr_peer_export: not available on a handle with several data sets (bsr_set_datasets_host)");
  if (!h->cfg.row_sharded) return bsr_fail("bsr_peer_export: the handle was not created with row_sharded = 1");
  if (!h->X32) return bsr_fail("bsr_peer_export: call bsr_set_data_* first (the exchange buffer is sized from the data)");
  if (world < 1 || world > BSR_MAX_PEERS) return bsr_fail("bsr_peer_export: world must be in [1, 8]");
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  h->x_world = world;             // the split count below depends on it
  int S; uint32_t rps, TR;
  win_geometry(h, h->cfg.n_chains, &S, &rps, &TR);
  if (ensure_window(h, S)) return 1;
  const int C = h->cfg.n_chains, K = h->cfg.K;
  h->x_rec_doubles = (size_t)C * S * h->ws.W * (K + 4);
  h->x_lrec_doubles = (size_t)C * S * sg_size(K);
  const size_t bytes = 2 * h->x_rec_doubles * sizeof(double) + 2 * (size_t)C * sizeof(unsigned long long) + BSR_MAX_PEERS * sizeof(unsigned long long) +
                       h->x_lrec_doubles * sizeof(double);
  if (h->xbuf) cudaFree(h->xbuf);
  h->xbuf = nullptr;
  CK(cudaMalloc((void**)&h->xbuf, bytes));
  CK(cudaMemset(h->xbuf, 0, bytes));
  h->xbuf_bytes = bytes;
  h->x_ticket = 0;
  cudaIpcMemHandle_t hdl;
  CK(cudaIpcGetMemHandle(&hdl, h->xbuf));
  memcpy(ipc_handle_out, &hdl, sizeof hdl);
  h->x_world = 0;                 // not usable before bsr_peer_import
  return 0;
}

int bsr_peer_import(bsr_handle* h, int32_t rank, int32_t world, const void* ipc_handles) {
  if (!h || !ipc_handles) return bsr_fail("bsr_peer_import: null argument");
  if (h->n_ds > 1) return bsr_fail("bsr_peer_import: not available on a handle with several data sets (bsr_set_datasets_host)");
  if (!h->xbuf) return bsr_fail("bsr_peer_import: call bsr_peer_export first");
  if (world < 1 || world > BSR_MAX_PEERS || rank < 0 || rank >= world) return bsr_fail("bsr_peer_import: bad rank / world");
  CK(cudaSetDevice(h->cfg.device));
  for (int r = 0; r < world; ++r) {
    if (r == rank) { h->x_peer[r] = h->xbuf; continue; }
    cudaIpcMemHandle_t hdl;
    memcpy(&hdl, (const unsigned char*)ipc_handles + (size_t)r * sizeof hdl, sizeof hdl);
    void* p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, hdl, cudaIpcMemLazyEnablePeerAccess));
    h->x_peer[r] = p;
  }
  h->x_world = world; h->x_rank = rank;
  return 0;
}

}  // extern "C"
