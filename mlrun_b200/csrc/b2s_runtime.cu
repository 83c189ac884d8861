// b2s_runtime.cu -- host runtime behind include/b200serve.h: plan lowering, device tables, launch
// configuration, pinned ring + dispatcher thread (event coalescing), CUDA-event timing.
#include <cuda_runtime.h>

#include <exception>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <limits>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/b200serve.h"
#include "b2s_internal.h"
#include "b2s_device.cuh"
#include "b2s_rowthread.cuh"
#include "b2s_trees3.cuh"
#include "b2s_dense.cuh"
#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost nothing unless a profiler is attached

using namespace b2s;

// ------------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
int b2s_int_fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CUDA_TRY(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail(B2S_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------------------------------ globals
struct Global {
  bool inited = false;
  int device = 0;
  cudaDeviceProp prop{};
  cudaStream_t stream = nullptr;  // library stream for run_device/run_host/time_device
  cudaStream_t copy_stream = nullptr;  // host->device copies of a chunked run_host (kernels + D2H stay on `stream`)
  int ring_slots = 4;
  int64_t max_batch = 65536;
  int64_t max_wait_us = 0;  // 0: a batch leaves as soon as the dispatcher is free (batches form while the previous one runs)
  std::atomic<int64_t> launches{0};
  std::mutex mu;
};
static Global G;

bool b2s_int_inited() { return G.inited; }
int b2s_int_device() { return G.device; }
int b2s_int_sm_count() { return G.prop.multiProcessorCount; }
cudaStream_t b2s_int_stream() { return G.stream; }
cudaStream_t b2s_int_copy_stream() { return G.copy_stream; }
void b2s_int_count_launches(int n) { G.launches.fetch_add(n, std::memory_order_relaxed); }

static int64_t cfg_get(const std::string& cfg, const char* key, int64_t dflt) {
  size_t pos = cfg.find(std::string(key) + "=");
  if (pos == std::string::npos) return dflt;
  return atoll(cfg.c_str() + pos + strlen(key) + 1);
}

// ------------------------------------------------------------------------------------------ plan
struct HostModel {
  int kind = MK_LINEAR;
  int n_scores = 1, link = 0;
  std::vector<int32_t> classes;
  // linear
  std::vector<double> W, b;
  // trees
  std::vector<int32_t> tree_offset, feature, left, right, tree_slot;
  std::vector<float> threshold;
  std::vector<double> leaf_value, tree_scale, init;
  std::vector<uint8_t> default_left;  // per node: a missing value (NaN) goes to the left child (empty: always right)
  bool nan_ok = false;                // the estimator routes NaN through its trees instead of refusing it
};

struct Slot {  // one in-flight batch of the coalescing ring
  char* h_in = nullptr;
  char* h_out = nullptr;     // out words then status words
  char* d_in = nullptr;
  char* d_out = nullptr;
  int32_t* d_status = nullptr;
  int64_t rows = 0;
  uint64_t batch_id = 0;
  int state = 0;  // 0 free/open, 1 sealed (queued for the dispatcher), 2 in flight, 3 done
  cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr, e3 = nullptr;
  std::chrono::steady_clock::time_point first_submit;
  b2s_stats stats{};
  int waiters = 0;      // tickets issued on this batch not yet collected
  std::shared_ptr<std::condition_variable> done_cv;  // the batch's own waiters (one wake-up per batch, not a herd over all tickets)
  bool wanted = false;  // a caller is blocked in b2s_wait on this (still open) batch: it leaves as soon as the dispatcher is free
  int err = 0;          // b2s_status of the batch (a failed copy / launch): every ticket of the batch gets it
  std::string err_msg;
};

// Ensemble-merge communicator: ONE device allocation per rank, exported over CUDA IPC and mapped by every peer:
//   [flags: 64 x uint32][CTA counter][timeout word][pad to kCommHeader = 512 B][merged rows, slot 0] .. [merged rows, slot 3]
// (round 2's first version started the rows at byte 256 = word 64: the first vote of a step overwrote the counter)
// merged rows = world x max_rows x out_cols 4-byte words; step e (epoch, 1-based) lands in slot e & 3.  Four slots let a
// caller wait for step e - 1 after launching step e (b2s_comm_wait_lag): see DESIGN.md section 7 for why that is safe.
constexpr size_t kCommHeader = 512;
constexpr uint32_t kCommSlots = 4;
struct b2s_comm_s {
  int rank = 0, world = 1, out_cols = 1;
  int64_t max_rows = 0;
  char* base = nullptr;            // this rank's allocation
  std::vector<char*> peer_base;    // [world] every rank's allocation as mapped here (peer_base[rank] == base)
  uint32_t epoch = 0;              // launches signalled so far
  int fused_lag = -1;              // b2s_comm_set_fused_wait: -1 off, 0 / 1: the launches wait in their own last CTA
  uint32_t fused_epoch = 0;        // highest step a launched kernel already waits for (0: none)
  size_t bytes = 0;
  bool connected = false;
  size_t buf_bytes() const { return (size_t)world * max_rows * out_cols * 4; }
  char* buf(int r, uint32_t e) const { return peer_base[r] + kCommHeader + (size_t)(e & (kCommSlots - 1u)) * buf_bytes(); }
  uint32_t* flags(int r) const { return reinterpret_cast<uint32_t*>(peer_base[r]); }
  uint32_t* counter() const { return reinterpret_cast<uint32_t*>(base) + 64; }
};

struct b2s_plan_s {
  int32_t n_in = 0;
  bool finalized = false;
  // builder state
  std::vector<float> fill;
  std::vector<std::vector<MapEntry>> maps;  // per column
  std::vector<int32_t> out_src, out_kind;
  std::vector<float> out_arg;
  std::vector<HostModel> models;
  int vote_kind = B2S_VOTE_NONE;
  std::vector<double> vote_w;
  // lowered
  int mode = MODE_STORE;
  int NS = 1;
  int out_cols = 0;
  int out_is_int = 0;
  KParams kp{};
  char* d_blob = nullptr;
  size_t blob_bytes = 0;
  int grid = 0, block = 0;
  int kernels_per_batch = 1;
  // row-thread kernel (constant-bank operands)
  bool rt_ok = false;
  int rt_cat_cols = 0;  // one-hot source columns of the row-thread plan
  int rt_NCH = 0, rt_NS = 0, rt_grid = 0, rt_smem = 0, rt_pitch = 0;
  std::vector<char> rt_blob;  // an RTParams<NCH, NS>
  // fused ensemble-merge targets (P2P)
  std::vector<void*> peers;
  int64_t peer_off = 0;
  struct b2s_comm_s* comm = nullptr;  // attached merge communicator (double-buffered targets + completion flags)
  // trees3 buffers between its three kernels: one scratch per stream the plan is launched on
  // (launches on one stream are ordered; the ring's stream, the library stream and caller streams may overlap)
  struct TreeScratch {
    double* pred = nullptr;    // partial sums, column-major (trees3_kernel -> t3_vote_kernel)
    int32_t* row_bad = nullptr;
    uint32_t* xt = nullptr;    // the batch transposed into tiles (t3_prep_kernel -> trees3_kernel)
    int64_t rows = 0;
  };
  std::map<cudaStream_t, TreeScratch> t3_scratch;
  std::mutex scratch_mu;
  // dense linear head on the tensor cores (b2s_dense.cu): > 8 scores over <= 128 plain numeric columns
  bool dense_ok = false;
  DenseParams dense{};
  int dense_smem = 0, dense_grid = 0;
  // round-2 tree kernel: parts resident in shared memory (b2s_trees3.cuh); scratch = partial sums, column-major
  bool t3_ok = false, t3_miss = false;
  int t3_D = 0, t3_grid = 0, t3_block = 0, t3_smem = 0, t3_cols = 0, t3_parts = 0;
  T3Params t3{};
  T3Prep t3_prep{};
  int t3_prep_smem = 0;
  char* d_t3_blob = nullptr;
  const int32_t* d_t3_col_score = nullptr;
  // host staging for run_host
  char* h_stage_in = nullptr;
  char* h_stage_out = nullptr;
  char* d_stage_in = nullptr;
  char* d_stage_out = nullptr;
  int32_t* d_stage_status = nullptr;
  int64_t stage_rows = 0;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> chunk_ev;  // 4 per chunk of a pipelined run_host: copied-in, kernel begin, kernel end, copied-out
  std::mutex host_mu;
  // coalescing ring
  std::vector<Slot> slots;
  int open_slot = -1;
  uint64_t next_batch = 1;
  std::map<uint64_t, int> batch_slot;  // live batches -> slot index
  std::deque<int> sealed;
  std::mutex mu;
  std::condition_variable cv_work, cv_done, cv_free;
  std::thread dispatcher;
  bool stop = false;
  bool dispatch_busy = false;  // a batch is on the ring's stream (run by the dispatcher thread or by a waiting caller)
  cudaStream_t ring_stream = nullptr;
  int64_t ring_cap = 0;
  // per-plan ring configuration (b2s_plan_set_ring; 0 / negative: the library defaults of b2s_init)
  std::atomic<int> spinners{0};  // waiters currently polling instead of sleeping (b2s_wait)
  int ring_cfg_slots = 0;
  int64_t ring_cfg_max_batch = 0;
  int ring_cfg_wait_us = -1;
  int wait_us() const { return ring_cfg_wait_us >= 0 ? ring_cfg_wait_us : G.max_wait_us; }
};

int b2s_int_plan_shape(b2s_plan_s* p, int* n_in, int* out_cols) {
  if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
  *n_in = p->n_in;
  *out_cols = p->out_cols;
  return B2S_OK;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct BlobBuilder {
  std::vector<char> data;
  template <typename T>
  size_t add(const std::vector<T>& v) {
    size_t off = align_up(data.size(), 16);
    data.resize(off + std::max<size_t>(v.size() * sizeof(T), 16));
    if (!v.empty()) memcpy(data.data() + off, v.data(), v.size() * sizeof(T));
    return off;
  }
};

template <int MODE, int NS>
static cudaError_t launch_rows(const KParams& kp, int grid, int block, cudaStream_t st) {
  static std::atomic<bool> attr_set{false};  // the dispatcher thread and callers may both get here first
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(rows_kernel<MODE, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)G.prop.sharedMemPerBlockOptin);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  rows_kernel<MODE, NS><<<grid, block, kp.sm_total, st>>>(kp);
  return cudaGetLastError();
}

static cudaError_t launch_plan(b2s_plan_s* p, const KParams& kp, int grid, int block, cudaStream_t st) {
  G.launches.fetch_add(1, std::memory_order_relaxed);
#define B2S_CASE(M, N) \
  if (p->mode == M && p->NS == N) return launch_rows<M, N>(kp, grid, block, st);
  B2S_CASE(MODE_LINEAR, 1) B2S_CASE(MODE_LINEAR, 2) B2S_CASE(MODE_LINEAR, 4) B2S_CASE(MODE_LINEAR, 8)
  B2S_CASE(MODE_LINEAR, 16) B2S_CASE(MODE_LINEAR, 32)
  B2S_CASE(MODE_TREES, 1) B2S_CASE(MODE_TREES, 4) B2S_CASE(MODE_TREES, 8) B2S_CASE(MODE_TREES, 16)
  B2S_CASE(MODE_STORE, 1)
#undef B2S_CASE
  return cudaErrorInvalidValue;
}

// cuTensorMapEncodeTiled, resolved at run time (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      sym = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(sym);
  }();
  return fn;
}
// rows viewed as a 2-D float32 tensor {n_in, n_rows}; boxes of 32 floats x tile_rows, 128-byte swizzle
static bool encode_rows_map(CUtensorMap* map, const void* rows, int64_t n_rows, int64_t stride, int n_in, int tile_rows) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)n_in, (cuuint64_t)n_rows};
  cuuint64_t gstride[1] = {(cuuint64_t)stride};
  cuuint32_t box[2] = {32u, (cuuint32_t)tile_rows};
  cuuint32_t estr[2] = {1u, 1u};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(rows), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct RTTables {  // what rt_build needs from finalize
  int n_in, n_out_cols, n_models, vote_kind, out_is_int, fast_epilogue, NS;
  const std::vector<float>* fill;
  const std::vector<uint32_t>* flags;
  const std::vector<double>* wnum;  // [n_in][NS]
  const std::vector<double>* bias;
  const std::vector<double>* vote_w;
  const std::vector<int32_t>* cat_off;
  const std::vector<float>* cat_val;
  const double* d_wcat;
  const double* d_vote_w;
  const ModelDesc* d_models;
  const int32_t* d_classes;
};

// threads per row: measured on B200 (profiles/r1_kernel_log.md): 2 beats 1 (more warps) and 4 (combine overhead)
constexpr int rt_tpr(int NCH) { return NCH >= 8 ? 2 : 1; }
constexpr int kRTTileRows = 128;  // rows per tile (the launch halves it for small batches)
constexpr int kRTStages = 2;      // depth of the tile ring

template <int NCH, int NS>
static void rt_build(b2s_plan_s* p, const RTTables& t) {
  using P = RTParams<NCH, NS>;
  p->rt_blob.assign(sizeof(P), 0);
  P& r = *reinterpret_cast<P*>(p->rt_blob.data());
  r.n_in = t.n_in;
  r.out_cols = t.n_out_cols;
  r.n_models = t.n_models;
  r.vote_kind = t.vote_kind;
  r.out_is_int = t.out_is_int;
  r.fast_epilogue = t.fast_epilogue;
  r.wcat = t.d_wcat;
  r.vote_w_g = t.d_vote_w;
  r.models = t.d_models;
  r.classes = t.d_classes;
  for (int c = 0; c < NCH * 4; ++c) {
    r.fill[c] = 0.0f;
    r.lim[c] = -1.0f;
    for (int k = 0; k < NS; ++k) r.w[c][k] = 0.0;
  }
  for (int c = 0; c < t.n_in; ++c) {
    const bool input = ((*t.flags)[c] & COL_COPIED) != 0;  // the column reaches the models as a number
    r.fill[c] = input ? (*t.fill)[c] : 0.0f;
    r.lim[c] = input ? std::numeric_limits<float>::infinity() : -1.0f;
    for (int k = 0; k < NS; ++k) r.w[c][k] = (*t.wnum)[(size_t)c * NS + k];
  }
  for (int k = 0; k < NS; ++k) {
    r.bias[k] = k < (int)t.bias->size() ? (*t.bias)[k] : 0.0;
    r.vote_w[k] = k < (int)t.vote_w->size() ? (*t.vote_w)[k] : 0.0;
  }
  int ncc = 0;
  for (int c = 0; c < t.n_in; ++c)
    if ((*t.cat_off)[c + 1] > (*t.cat_off)[c]) {
      r.cat_col[ncc] = c;
      r.cat_base[ncc] = (*t.cat_off)[c];
      r.cat_cnt[ncc] = (*t.cat_off)[c + 1] - (*t.cat_off)[c];
      r.cat_fill[ncc] = (*t.fill)[c];
      for (int q = 0; q < kRTCatsInline; ++q)
        r.cat_inl[ncc][q] = q < r.cat_cnt[ncc] ? (*t.cat_val)[r.cat_base[ncc] + q] : std::numeric_limits<float>::quiet_NaN();
      {  // consecutive small integers (the usual integer codes): the index is a conversion, not a search
        const float f0 = (*t.cat_val)[r.cat_base[ncc]];
        bool dense = f0 == std::floor(f0) && std::fabs(f0) < 8388608.0f;
        for (int q = 0; dense && q < r.cat_cnt[ncc]; ++q) dense = (*t.cat_val)[r.cat_base[ncc] + q] == f0 + (float)q;
        r.cat_dense[ncc] = dense ? 1 : 0;
        r.cat_first[ncc] = dense ? (int)f0 : 0;
      }
      ++ncc;
    }
  r.n_cat_cols = ncc;
  r.n_cat = (int)t.cat_val->size();
  r.cats_fast = 1;
  for (int cc = 0; cc < ncc; ++cc) {
    r.cats_fast = r.cats_fast && r.cat_dense[cc];
    r.catf[cc].first = r.cat_first[cc];
    r.catf[cc].cnt = r.cat_cnt[cc];
    r.catf[cc].woff_b = r.cat_base[cc] * NS * 8;
    r.catf[cc].fill = r.cat_fill[cc];
  }
  r.zero_woff_b = r.n_cat * NS * 8;
  {
    int last_live = -1;  // last chunk that holds a model-input column
    for (int c = 0; c < t.n_in; ++c)
      if (((*t.flags)[c] & COL_COPIED) != 0) last_live = c >> 2;
    r.dead_tail = last_live < 0 ? 0 : std::max(0, NCH - 1 - last_live);
  }
  for (int i = 0; i < r.n_cat; ++i) r.cat_val[i] = (*t.cat_val)[i];
}

// the tensor-map loader needs rows of >= 128 bytes that fill the plan's chunks exactly
static bool rt_tmap_ok(const b2s_plan_s* p) { return p->rt_NCH >= 8 && p->n_in == p->rt_NCH * 4 && tensor_map_encoder() != nullptr; }

struct LaunchCtx {             // per-launch context (launches of one plan may be issued from several threads at once)
  const KParams* k = nullptr;  // merge targets / completion signal of this launch
  bool host_rows = false;      // the rows live in mapped host memory (zero-copy small batches): plain cp.async loads
};

template <int NCH, int NS>
static cudaError_t rt_launch_t(b2s_plan_s* p, const void* rows, int64_t stride, int64_t n_rows, void* out, int32_t* status,
                               int vec_ok, cudaStream_t st, bool query, int* occ, const B2SGather* gather, const LaunchCtx* lc) {
  using P = RTParams<NCH, NS>;
  constexpr int TPR = rt_tpr(NCH);
  constexpr int LMT = NCH >= 8 ? 2 : 1;  // the tensor-map variants exist for rows of >= 128 bytes
  static std::atomic<bool> attr_set{false};  // the dispatcher thread and callers may both get here first
  if (!attr_set) {
    const int cap = (int)G.prop.sharedMemPerBlockOptin;
    cudaError_t e = cudaFuncSetAttribute(rowthread_kernel<NCH, NS, TPR, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(rowthread_kernel<NCH, NS, TPR, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e == cudaSuccess && NCH >= 8)
      e = cudaFuncSetAttribute(rowthread_kernel<NCH, NS, TPR, LMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  const bool tmap_ok = rt_tmap_ok(p);
  if (query) {  // occupancy of the variant an aligned launch takes
    if (tmap_ok)
      return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, rowthread_kernel<NCH, NS, TPR, LMT>, kRTTileRows * TPR, p->rt_smem);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, rowthread_kernel<NCH, NS, TPR, 0>, kRTTileRows * TPR, p->rt_smem);
  }
  P r = *reinterpret_cast<const P*>(p->rt_blob.data());
  r.rows = (const char*)rows;
  r.row_stride = stride;
  r.n_rows = n_rows;
  r.out = (float*)out;
  r.status = status;
  r.vec_ok = vec_ok;
  const KParams* lk = lc ? lc->k : nullptr;
  r.n_peers = lk ? lk->n_peers : (int)p->peers.size();
  r.peer_off = lk ? lk->peer_off : p->peer_off;
  for (int g = 0; g < r.n_peers; ++g) r.peers[g] = lk ? lk->peers[g] : (float*)p->peers[g];
  r.sig = lk ? lk->sig : MergeSig{};
  r.pitch = p->rt_pitch;
  r.stages = kRTStages;
  // tile loader: 2 TMA tensor-map boxes, 1 one TMA bulk copy per row, 0 cp.async (LDGSTS) for unaligned or host-resident rows
  int mode = vec_ok ? 2 : 0;
  if (lc && lc->host_rows) mode = 0;
  if (mode == 2 && !tmap_ok) mode = 1;
  if (gather) {  // rows come from the online table: one bulk copy per row, source found by key inside the kernel
    mode = 1;
    r.g_keys = gather->d_keys;
    r.g_slots = reinterpret_cast<const TableSlot*>(gather->d_slots);
    r.g_mask = gather->mask;
    r.g_values = gather->d_values;
    r.g_missing_row = gather->missing_row;
    // the table's impute policy (None / NaN / Inf -> value, feature_vector.py:1046-1052) runs before the plan's own
    // Imputer; on a column the plan reads as a number both fold into the kernel's one compare/select
    if (gather->any_impute)
      for (int c = 0; c < p->n_in; ++c) {
        const float f = gather->h_impute[c];
        if (f == f && r.lim[c] == std::numeric_limits<float>::infinity()) {
          r.lim[c] = std::numeric_limits<float>::max();
          r.fill[c] = f;
        }
      }
  }
  int tr = kRTTileRows;
  while (tr > 32 && (n_rows + tr - 1) / tr < (int64_t)G.prop.multiProcessorCount) tr /= 2;
  alignas(64) CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  if (mode == 2 && !encode_rows_map(&tmap, rows, n_rows, stride, p->n_in, tr)) mode = 1;
  r.tile_rows = tr;
  const int64_t tiles = (n_rows + tr - 1) / tr;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(p->rt_grid, tiles));
  r.use_bulk = mode;
  // single-barrier tile loop: measured better with 4 score columns (0.0506 vs 0.0512 ms, r2o) and worse with one
  // (0.0481 vs 0.0454 ms, r2q / r2o): it follows the number of score columns
  r.one_sync = NS >= 4 ? 1 : 0;
  for (int cc = 0; cc < r.n_cat_cols; ++cc) {  // tile-relative position of each categorical column
    const int col = r.cat_col[cc], ch = col >> 2;
    r.cat_off[cc] = mode == 2 ? (ch >> 3) * (tr * 32) + (col & 3) : col;
    r.cat_sw[cc] = mode == 2 ? (ch & 7) << 2 : 0;
    r.catf[cc].off_b = r.cat_off[cc] * 4;
    r.catf[cc].sw_b = r.cat_sw[cc] * 4;
  }
  if (mode == 2)
    rowthread_kernel<NCH, NS, TPR, LMT><<<grid, tr * TPR, p->rt_smem, st>>>(r, tmap);
  else if (mode == 1)
    rowthread_kernel<NCH, NS, TPR, 1><<<grid, tr * TPR, p->rt_smem, st>>>(r, tmap);
  else
    rowthread_kernel<NCH, NS, TPR, 0><<<grid, tr * TPR, p->rt_smem, st>>>(r, tmap);
  return cudaGetLastError();
}

#define RT_DISPATCH(FN, ...)                                                              \
  do {                                                                                    \
    const int nch_ = p->rt_NCH, ns_ = p->rt_NS;                                           \
    if (nch_ == 4 && ns_ == 1) return FN<4, 1>(__VA_ARGS__);                              \
    if (nch_ == 4 && ns_ == 2) return FN<4, 2>(__VA_ARGS__);                              \
    if (nch_ == 4 && ns_ == 4) return FN<4, 4>(__VA_ARGS__);                              \
    if (nch_ == 4 && ns_ == 8) return FN<4, 8>(__VA_ARGS__);                              \
    if (nch_ == 8 && ns_ == 1) return FN<8, 1>(__VA_ARGS__);                              \
    if (nch_ == 8 && ns_ == 2) return FN<8, 2>(__VA_ARGS__);                              \
    if (nch_ == 8 && ns_ == 4) return FN<8, 4>(__VA_ARGS__);                              \
    if (nch_ == 8 && ns_ == 8) return FN<8, 8>(__VA_ARGS__);                              \
    if (nch_ == 16 && ns_ == 1) return FN<16, 1>(__VA_ARGS__);                            \
    if (nch_ == 16 && ns_ == 2) return FN<16, 2>(__VA_ARGS__);                            \
    if (nch_ == 16 && ns_ == 4) return FN<16, 4>(__VA_ARGS__);                            \
    if (nch_ == 16 && ns_ == 8) return FN<16, 8>(__VA_ARGS__);                            \
    if (nch_ == 32 && ns_ == 1) return FN<32, 1>(__VA_ARGS__);                            \
    if (nch_ == 32 && ns_ == 2) return FN<32, 2>(__VA_ARGS__);                            \
    if (nch_ == 32 && ns_ == 4) return FN<32, 4>(__VA_ARGS__);                            \
    if (nch_ == 32 && ns_ == 8) return FN<32, 8>(__VA_ARGS__);                            \
  } while (0)

static cudaError_t rt_launch(b2s_plan_s* p, const void* rows, int64_t stride, int64_t n_rows, void* out, int32_t* status,
                             int vec_ok, cudaStream_t st, bool query = false, int* occ = nullptr, const B2SGather* gather = nullptr,
                             const LaunchCtx* lc = nullptr) {
  RT_DISPATCH(rt_launch_t, p, rows, stride, n_rows, out, status, vec_ok, st, query, occ, gather, lc);
  return cudaErrorInvalidValue;
}
static void rt_build_any(b2s_plan_s* p, const RTTables& t) {
  RT_DISPATCH(rt_build, p, t);
}

// ------------------------------------------------------------------------------------------ C-ABI: library
extern "C" int b2s_version(void) { return B2S_VERSION; }
extern "C" const char* b2s_last_error(void) { return g_err.c_str(); }

extern "C" int b2s_init(int device_ordinal, const char* cfg) {
  try {  // no C++ exception crosses the C boundary
    std::lock_guard<std::mutex> lk(G.mu);
    if (G.inited) return B2S_OK;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
      return fail(B2S_ERR_NO_DEVICE, "no CUDA device (%s); this engine has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device_ordinal < 0 || device_ordinal >= n) return fail(B2S_ERR_INVALID, "device ordinal %d out of range", device_ordinal);
    CUDA_TRY(cudaSetDevice(device_ordinal));
    CUDA_TRY(cudaGetDeviceProperties(&G.prop, device_ordinal));
    CUDA_TRY(cudaStreamCreateWithFlags(&G.stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&G.copy_stream, cudaStreamNonBlocking));
    G.device = device_ordinal;
    std::string c = cfg ? cfg : "";
    G.ring_slots = (int)cfg_get(c, "ring_slots", 4);
    G.max_batch = cfg_get(c, "max_batch", 65536);
    G.max_wait_us = cfg_get(c, "max_wait_us", 0);
    if (G.ring_slots < 2) G.ring_slots = 2;
    G.inited = true;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_shutdown(void) {
  try {  // no C++ exception crosses the C boundary
    std::lock_guard<std::mutex> lk(G.mu);
    if (!G.inited) return B2S_OK;
    cudaStreamDestroy(G.stream);
    cudaStreamDestroy(G.copy_stream);
    G.stream = G.copy_stream = nullptr;
    G.inited = false;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_device_info(b2s_devinfo* out) {
  try {  // no C++ exception crosses the C boundary
    if (!G.inited) return fail(B2S_ERR_STATE, "b2s_init was not called");
    if (!out) return fail(B2S_ERR_INVALID, "null out");
    memset(out, 0, sizeof(*out));
    out->ordinal = G.device;
    out->sm_count = G.prop.multiProcessorCount;
    out->cc_major = G.prop.major;
    out->cc_minor = G.prop.minor;
    out->total_mem = (int64_t)G.prop.totalGlobalMem;
    out->l2_bytes = G.prop.l2CacheSize;
    out->smem_per_block_optin = (int64_t)G.prop.sharedMemPerBlockOptin;
    strncpy(out->name, G.prop.name, sizeof(out->name) - 1);
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int64_t b2s_launch_count(void) { return G.launches.load(); }

// ------------------------------------------------------------------------------------------ C-ABI: plan building
extern "C" int b2s_plan_create(int32_t n_in_cols, b2s_plan_t* out) {
  try {  // no C++ exception crosses the C boundary
    if (!out || n_in_cols <= 0 || n_in_cols > 65536) return fail(B2S_ERR_INVALID, "bad n_in_cols %d", n_in_cols);
    auto* p = new b2s_plan_s();
    p->n_in = n_in_cols;
    p->fill.assign(n_in_cols, std::numeric_limits<float>::quiet_NaN());
    p->maps.resize(n_in_cols);
    *out = p;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int check_build(b2s_plan_t p) {
  if (!p) return fail(B2S_ERR_INVALID, "null plan");
  if (p->finalized) return fail(B2S_ERR_STATE, "plan already finalized");
  return B2S_OK;
}

extern "C" int b2s_plan_set_impute(b2s_plan_t p, const int32_t* cols, const float* fills, int32_t n) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    for (int i = 0; i < n; ++i) {
      if (cols[i] < 0 || cols[i] >= p->n_in) return fail(B2S_ERR_INVALID, "impute column %d out of range", cols[i]);
      p->fill[cols[i]] = fills[i];
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_add_value_map(b2s_plan_t p, int32_t col, const float* keys, const float* vals, int32_t n) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (col < 0 || col >= p->n_in) return fail(B2S_ERR_INVALID, "map column %d out of range", col);
    for (int i = 0; i < n; ++i) p->maps[col].push_back(MapEntry{keys[i], 0.f, vals[i], (i == 0 ? 256 : 0) | 0});
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_add_range_map(b2s_plan_t p, int32_t col, const float* lo, const float* hi, const float* vals, int32_t n) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (col < 0 || col >= p->n_in) return fail(B2S_ERR_INVALID, "map column %d out of range", col);
    for (int i = 0; i < n; ++i) p->maps[col].push_back(MapEntry{lo[i], hi[i], vals[i], (i == 0 ? 256 : 0) | 1});
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_set_output_schema(b2s_plan_t p, const int32_t* src_col, const int32_t* kind, const float* arg, int32_t n_out) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (n_out <= 0) return fail(B2S_ERR_INVALID, "empty output schema");
    if (!p->models.empty()) return fail(B2S_ERR_STATE, "set the output schema before adding models");
    p->out_src.assign(src_col, src_col + n_out);
    p->out_kind.assign(kind, kind + n_out);
    p->out_arg.assign(arg, arg + n_out);
    for (int j = 0; j < n_out; ++j) {
      if (src_col[j] < 0 || src_col[j] >= p->n_in) return fail(B2S_ERR_INVALID, "schema source column %d out of range", src_col[j]);
      if (kind[j] != B2S_OUT_COPY && kind[j] != B2S_OUT_ONEHOT) return fail(B2S_ERR_INVALID, "schema kind %d unknown", kind[j]);
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int n_out_of(b2s_plan_t p) { return p->out_src.empty() ? p->n_in : (int)p->out_src.size(); }

static int check_link(int link, int n_scores, int n_classes) {
  if (link < 0 || link > 3) return fail(B2S_ERR_INVALID, "unknown link %d", link);
  if (n_scores < 1 || n_scores > kMaxScores) return fail(B2S_ERR_UNSUPPORTED, "n_scores %d not in [1,%d]", n_scores, kMaxScores);
  if ((link == B2S_LINK_BINARY_GT || link == B2S_LINK_BINARY_GE) && n_classes != 0 && n_classes != 2)
    return fail(B2S_ERR_INVALID, "binary link needs 2 classes");
  if (link == B2S_LINK_ARGMAX && n_classes != 0 && n_classes != n_scores) return fail(B2S_ERR_INVALID, "argmax link needs n_scores classes");
  return B2S_OK;
}

extern "C" int b2s_plan_add_linear_model(b2s_plan_t p, const double* W, const double* b, int32_t n_scores, int32_t link,
                                         const int32_t* classes, int32_t n_classes) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (int rc = check_link(link, n_scores, classes ? n_classes : 0)) return rc;
    if ((int)p->models.size() >= kMaxModels) return fail(B2S_ERR_UNSUPPORTED, "more than %d models in one plan", kMaxModels);
    HostModel m;
    m.kind = MK_LINEAR;
    m.n_scores = n_scores;
    m.link = link;
    const int no = n_out_of(p);
    m.W.assign(W, W + (size_t)n_scores * no);
    m.b.assign(b, b + n_scores);
    if (classes) m.classes.assign(classes, classes + n_classes);
    p->models.push_back(std::move(m));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// float32 t' with  x < t  <=>  x <= t'  for every float32 x: the next float below t (nothing is below -inf: a NaN
// threshold sends every value right, which is what "x < -inf" does)
static float threshold_for_less_than(float t) {
  if (std::isnan(t)) return t;
  if (t == -std::numeric_limits<float>::infinity()) return std::numeric_limits<float>::quiet_NaN();
  return std::nextafterf(t, -std::numeric_limits<float>::infinity());
}

extern "C" int b2s_plan_add_tree_model_ex(b2s_plan_t p, int32_t n_trees, const int32_t* tree_offset, const int32_t* feature,
                                          const float* threshold, const int32_t* left, const int32_t* right,
                                          const double* leaf_value, const int32_t* tree_slot, const double* tree_scale,
                                          const double* init, int32_t n_scores, int32_t link, const int32_t* classes,
                                          int32_t n_classes, int32_t cmp_mode, const uint8_t* default_left, int32_t nan_mode) {
  try {
    if (cmp_mode != B2S_CMP_LE && cmp_mode != B2S_CMP_LT) return fail(B2S_ERR_INVALID, "unknown cmp_mode %d", cmp_mode);
    if (nan_mode != B2S_NAN_ERROR && nan_mode != B2S_NAN_DEFAULT_CHILD) return fail(B2S_ERR_INVALID, "unknown nan_mode %d", nan_mode);  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (int rc = check_link(link, n_scores, classes ? n_classes : 0)) return rc;
    if (n_scores > 16) return fail(B2S_ERR_UNSUPPORTED, "tree models support at most 16 scores");
    if ((int)p->models.size() >= kMaxModels) return fail(B2S_ERR_UNSUPPORTED, "more than %d models in one plan", kMaxModels);
    if (n_trees < 1) return fail(B2S_ERR_INVALID, "n_trees < 1");
    HostModel m;
    m.kind = MK_TREES;
    m.n_scores = n_scores;
    m.link = link;
    const int nn = tree_offset[n_trees];
    const int no = n_out_of(p);
    m.tree_offset.assign(tree_offset, tree_offset + n_trees + 1);
    m.feature.assign(feature, feature + nn);
    m.threshold.assign(threshold, threshold + nn);
    if (cmp_mode == B2S_CMP_LT)  // xgboost: left when x < t.  Stored as the equivalent "x <= t'" (every kernel tests <=)
      for (int i = 0; i < nn; ++i)
        if (feature[i] >= 0) m.threshold[i] = threshold_for_less_than(m.threshold[i]);
    if (default_left) m.default_left.assign(default_left, default_left + nn);
    m.nan_ok = nan_mode == B2S_NAN_DEFAULT_CHILD;
    m.left.assign(left, left + nn);
    m.right.assign(right, right + nn);
    m.leaf_value.assign(leaf_value, leaf_value + nn);
    m.tree_slot.assign(tree_slot, tree_slot + n_trees);
    m.tree_scale.assign(tree_scale, tree_scale + n_trees);
    m.init.assign(init, init + n_scores);
    if (classes) m.classes.assign(classes, classes + n_classes);
    for (int t = 0; t < n_trees; ++t) {
      if (tree_slot[t] < 0 || tree_slot[t] >= n_scores) return fail(B2S_ERR_INVALID, "tree %d slot out of range", t);
      const int lo = tree_offset[t], hi = tree_offset[t + 1];
      if (hi <= lo) return fail(B2S_ERR_INVALID, "tree %d is empty", t);
      for (int i = lo; i < hi; ++i) {
        if (feature[i] >= no) return fail(B2S_ERR_INVALID, "tree %d node %d feature %d >= n_out %d", t, i - lo, feature[i], no);
        if (feature[i] >= 0) {
          // children are tree-relative and must point forward (no cycles => the walk terminates)
          if (left[i] <= i - lo || right[i] <= i - lo || left[i] >= hi - lo || right[i] >= hi - lo)
            return fail(B2S_ERR_INVALID, "tree %d node %d has bad children", t, i - lo);
        }
      }
    }
    p->models.push_back(std::move(m));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_add_tree_model(b2s_plan_t p, int32_t n_trees, const int32_t* tree_offset, const int32_t* feature,
                                       const float* threshold, const int32_t* left, const int32_t* right,
                                       const double* leaf_value, const int32_t* tree_slot, const double* tree_scale,
                                       const double* init, int32_t n_scores, int32_t link, const int32_t* classes,
                                       int32_t n_classes) {
  return b2s_plan_add_tree_model_ex(p, n_trees, tree_offset, feature, threshold, left, right, leaf_value, tree_slot, tree_scale,
                                    init, n_scores, link, classes, n_classes, B2S_CMP_LE, nullptr, B2S_NAN_ERROR);
}

extern "C" int b2s_plan_set_vote(b2s_plan_t p, int32_t vote_kind, const double* weights, int32_t n_weights) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (vote_kind < 0 || vote_kind > 2) return fail(B2S_ERR_INVALID, "unknown vote kind %d", vote_kind);
    p->vote_kind = vote_kind;
    p->vote_w.assign(weights, weights + (weights ? n_weights : 0));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ trees3 plan
// order-preserving int32 key of a float32 (see t3_key in b2s_trees3.cuh): thresholds in the NaN-routing layout
static int32_t host_key(float x) {
  if (x == 0.0f) x = 0.0f;  // -0 -> +0
  int32_t b;
  memcpy(&b, &x, 4);
  return b ^ ((b >> 31) & 0x7fffffff);
}

// Lower a MODE_TREES plan to parts (b2s_trees3.cuh).  Leaves p->t3_ok false when the plan does not qualify (it then runs
// on the generic rows_kernel<TREES>); returns an error only for CUDA failures.
static int t3_build(b2s_plan_s* p, const KParams& k, bool any_fill) {
  const int n_in = p->n_in, M = (int)p->models.size();
  const int sms = G.prop.multiProcessorCount;
  const int smem_cap = (int)G.prop.sharedMemPerBlockOptin;
  constexpr int TR = kT3TR;
  // ---- depth, NaN mode, linear columns
  int D = 2, n_lin_cols = 0;
  bool all_nan_ok = true, any_trees = false;
  for (auto& m : p->models) {
    if (m.kind != MK_TREES) {
      n_lin_cols += m.n_scores;
      all_nan_ok = false;
      continue;
    }
    any_trees = true;
    all_nan_ok = all_nan_ok && m.nan_ok;
    const int nt = (int)m.tree_slot.size();
    for (int t = 0; t < nt; ++t) {
      const int base = m.tree_offset[t];
      std::vector<std::pair<int, int>> stack{{0, 0}};
      while (!stack.empty()) {
        auto [node, d] = stack.back();
        stack.pop_back();
        D = std::max(D, d);
        if (D > kT3MaxDepth) return B2S_OK;
        if (m.feature[base + node] >= 0) {
          stack.push_back({m.left[base + node], d + 1});
          stack.push_back({m.right[base + node], d + 1});
        }
      }
    }
  }
  if (!any_trees || n_lin_cols > kT3MaxLin) return B2S_OK;
  const bool miss = all_nan_ok;
  const int NN = 1 << D;
  const int n_in4 = (int)align_up(n_in, 4);
  const int xt_words = n_in4 * TR;
  // ---- shared-memory budget: tables | fill | partial sums | transposed tile(s) | landing tile | flags | barrier
  int pitch = n_in4 + 4;
  if (((pitch / 4) & 1) == 0) pitch += 4;
  const size_t land_bytes = std::max((size_t)TR * pitch * 4, (size_t)TR * n_in4 * 4);
  const int kMaxW = kT3MaxWalk;  // walking warps: (kMaxW + kT3Service) * 32 <= 1024 threads
  const size_t lin_bytes = (size_t)n_lin_cols * n_in * 8;
  // walking kernel: tables | two partial-sum buffers | two tiles (filled by TMA bulk copies) | four mbarriers
  auto fixed_bytes = [&](int w) {
    return 2 * (size_t)std::max(w, kT3MaxLin) * TR * 8 + 2 * (size_t)xt_words * 4 + 128 /* tile alignment */ + 64;
  };
  auto capacity = [&](int w) {  // trees one CTA can hold with w walking warps (0: the plan does not fit at all)
    const size_t fixed = fixed_bytes(w);
    if (fixed + std::max(lin_bytes, 2 * (size_t)NN * 16) > (size_t)smem_cap) return 0;
    return (int)(((size_t)smem_cap - fixed) / ((size_t)NN * 16));
  };
  // ---- walking warps per CTA: the partial-sum buffers grow with them, so they decide how many trees a CTA holds and with
  // that the number of parts; cost = shared-memory wavefronts per row: 8 per part for the transpose, (2 + 3 D) per tree
  // walk of 32 rows, whole iterations of U trees per warp
  std::vector<int> group_sizes;
  for (auto& m : p->models)
    if (m.kind == MK_TREES)
      for (int slot = 0; slot < m.n_scores; ++slot) {
        int n = 0;
        for (int32_t sl : m.tree_slot) n += sl == slot ? 1 : 0;
        if (n) group_sizes.push_back(n);
      }
  int W = 0;
  {
    double best = 1e300;
    for (int w = 16; w <= kMaxW; ++w) {
      const int cap = capacity(w);
      if (cap < 1) continue;
      double cost = n_lin_cols > 0 ? 2.0 : 0.0;
      int n_parts = n_lin_cols > 0 ? 1 : 0;
      for (int n : group_sizes) {
        const int n_chunks = (n + cap - 1) / cap, per = (n + n_chunks - 1) / n_chunks;
        for (int c0 = 0; c0 < n; c0 += per) {
          const int nt = std::min(per, n - c0), tpw = (nt + w - 1) / w, iters = (tpw + kT3U - 1) / kT3U;
          cost += 0.5 + (double)iters * kT3U * w * (2.0 + 3.0 * D) / 32.0;
          ++n_parts;
        }
      }
      if (n_parts > sms) continue;
      if (cost < best - 1e-9 || (std::fabs(cost - best) <= 1e-9 && w > W)) {
        best = cost;
        W = w;
      }
    }
  }
  if (W == 0) return B2S_OK;
  const int cap_trees = capacity(W);
  // ---- parts: per (tree model, score slot) the trees of that slot, split evenly when they exceed a CTA's capacity
  struct HostPart {
    int model, slot, n_trees = 0, n_cols = 1, col0 = 0;
    std::vector<uint2> nodes;
    std::vector<double> leaves;
    double cost = 0.0;
  };
  std::vector<HostPart> parts;
  std::vector<int32_t> col_score;
  {
    int so = 0;
    for (int mi = 0; mi < M; ++mi) {
      auto& m = p->models[mi];
      if (m.kind == MK_TREES) {
        const int nt = (int)m.tree_slot.size();
        for (int slot = 0; slot < m.n_scores; ++slot) {
          std::vector<int> mine;
          for (int t = 0; t < nt; ++t)
            if (m.tree_slot[t] == slot) mine.push_back(t);
          if (mine.empty()) continue;
          const int n_chunks = ((int)mine.size() + cap_trees - 1) / cap_trees;
          const int per = ((int)mine.size() + n_chunks - 1) / n_chunks;
          for (int c0 = 0; c0 < (int)mine.size(); c0 += per) {
            HostPart hp;
            hp.model = mi;
            hp.slot = slot;
            hp.n_trees = std::min(per, (int)mine.size() - c0);
            hp.nodes.assign((size_t)hp.n_trees * NN, make_uint2(0u, 0u));
            hp.leaves.assign((size_t)hp.n_trees * NN, 0.0);
            for (int q = 0; q < hp.n_trees; ++q) {
              const int t = mine[c0 + q];
              const int base = m.tree_offset[t];
              struct It { int heap, d, src; };  // heap: 1-based index in the complete tree
              std::vector<It> stack{{1, 0, 0}};
              while (!stack.empty()) {
                const It it = stack.back();
                stack.pop_back();
                const bool leaf = m.feature[base + it.src] < 0;
                if (it.d == D) {
                  hp.leaves[(size_t)q * NN + (it.heap - NN)] = m.tree_scale[t] * m.leaf_value[base + it.src];
                  continue;
                }
                uint2 nd;
                if (leaf) {  // pad: every value goes left, and both children carry the leaf anyway
                  const float inf = std::numeric_limits<float>::infinity();
                  nd.x = 0;
                  if (miss) nd.y = (uint32_t)0x7fffffff; else memcpy(&nd.y, &inf, 4);  // key(x) + 0 > INT_MAX never holds
                  stack.push_back({2 * it.heap, it.d + 1, it.src});
                  stack.push_back({2 * it.heap + 1, it.d + 1, it.src});
                } else {
                  const float thr = m.threshold[base + it.src];
                  const bool dl = !m.default_left.empty() && m.default_left[base + it.src] != 0;
                  nd.x = (uint32_t)(m.feature[base + it.src] * TR * 4) | ((miss && dl) ? 0x80000000u : 0u);
                  if (miss) {
                    // the walk tests key(x) + d > key(t) + d with d = 1 for "missing goes left": NaN's key INT_MAX wraps
                    // to INT_MIN.  NaN threshold ("x < -inf" of an xgboost model): every value goes right
                    const uint32_t d = dl ? 1u : 0u;
                    nd.y = (std::isnan(thr) ? 0x80000000u : (uint32_t)host_key(thr)) + d;
                  } else {
                    memcpy(&nd.y, &thr, 4);
                  }
                  stack.push_back({2 * it.heap, it.d + 1, m.left[base + it.src]});
                  stack.push_back({2 * it.heap + 1, it.d + 1, m.right[base + it.src]});
                }
                hp.nodes[(size_t)q * NN + it.heap] = nd;
              }
            }
            hp.cost = 0.5 + hp.n_trees * (2.0 + 3.0 * D) / 32.0 * 2.0;  // shared-memory wavefronts per row (the walks)
            hp.col0 = (int)col_score.size();
            col_score.push_back(so + slot);
            parts.push_back(std::move(hp));
          }
        }
      }
      so += m.n_scores;
    }
    if (n_lin_cols > 0) {  // one part for all the linear scorers: weights [col][n_in] (identity schema: n_out == n_in)
      HostPart hp;
      hp.model = -1;
      hp.slot = 0;
      hp.n_trees = 0;
      hp.n_cols = n_lin_cols;
      hp.col0 = (int)col_score.size();
      int so2 = 0;
      for (int mi = 0; mi < M; ++mi) {
        auto& m = p->models[mi];
        if (m.kind == MK_LINEAR)
          for (int kk = 0; kk < m.n_scores; ++kk) {
            for (int j = 0; j < n_in; ++j) hp.leaves.push_back(m.W[(size_t)kk * n_in + j]);
            col_score.push_back(so2 + kk);
          }
        so2 += m.n_scores;
      }
      // measured (r2i, router of 4 linear + 4 tree models over 64 columns): the linear part's tiles cost about a fifth of a
      // 100-tree part's; erring high only hands it a few CTAs more
      hp.cost = 8.0 + n_in * (n_lin_cols + 4) / 16.0;
      parts.push_back(std::move(hp));
    }
  }
  const int P = (int)parts.size();
  if (P == 0 || P > sms) return B2S_OK;
  // ---- CTAs per part, proportional to cost (largest-remainder rounding, at least one each)
  std::vector<int> n_ctas(P, 1);
  {
    double total = 0.0;
    for (auto& hp : parts) total += hp.cost;
    int left = sms - P;
    std::vector<double> want(P);
    for (int i = 0; i < P; ++i) want[i] = std::max(0.0, parts[i].cost / total * sms - 1.0);
    for (int i = 0; i < P; ++i) {
      const int take = std::min(left, (int)want[i]);
      n_ctas[i] += take;
      left -= take;
      want[i] -= (int)want[i];
    }
    while (left > 0) {
      int best = 0;
      for (int i = 1; i < P; ++i)
        if (want[i] > want[best]) best = i;
      ++n_ctas[best];
      want[best] = -1.0;
      --left;
      bool any = false;
      for (int i = 0; i < P; ++i) any |= want[i] >= 0.0;
      if (!any)
        for (int i = 0; i < P; ++i) want[i] = parts[i].cost;
    }
  }
  // ---- one blob: nodes / leaves of every part, the part table, the column -> score map
  BlobBuilder tb;
  std::vector<size_t> o_nodes(P), o_leaves(P);
  for (int i = 0; i < P; ++i) {
    o_nodes[i] = tb.add(parts[i].nodes);
    o_leaves[i] = tb.add(parts[i].leaves);
  }
  const size_t o_cols = tb.add(col_score);
  const size_t o_parts = align_up(tb.data.size(), 16);
  tb.data.resize(o_parts + sizeof(T3Part) * P);
  CUDA_TRY(cudaMalloc(&p->d_t3_blob, tb.data.size()));
  std::vector<T3Part> dev(P);
  int cta0 = 0;
  for (int i = 0; i < P; ++i) {
    T3Part& d = dev[i];
    d.nodes = parts[i].n_trees ? (const uint2*)(p->d_t3_blob + o_nodes[i]) : nullptr;
    d.leaves = (const double*)(p->d_t3_blob + o_leaves[i]);
    d.n_trees = parts[i].n_trees;
    d.n_cols = parts[i].n_cols;
    d.col0 = parts[i].col0;
    d.cta0 = cta0;
    d.n_ctas = n_ctas[i];
    cta0 += n_ctas[i];
  }
  memcpy(tb.data.data() + o_parts, dev.data(), sizeof(T3Part) * P);
  CUDA_TRY(cudaMemcpy(p->d_t3_blob, tb.data.data(), tb.data.size(), cudaMemcpyHostToDevice));
  p->d_t3_col_score = (const int32_t*)(p->d_t3_blob + o_cols);

  T3Params& t = p->t3;
  memset(&t, 0, sizeof(t));
  t.parts = (const T3Part*)(p->d_t3_blob + o_parts);
  t.n_in = n_in;
  t.n_parts = P;
  t.warps = W;
  t.xt_words = xt_words;
  size_t off = 0;
  auto take = [&](size_t bytes, size_t al) {
    off = align_up(off, al);
    const size_t o = off;
    off += bytes;
    return (int32_t)o;
  };
  int max_trees = 0;
  for (auto& hp : parts) max_trees = std::max(max_trees, hp.n_trees);
  take(std::max((size_t)max_trees * NN * 8, lin_bytes), 16);  // nodes (or the linear weights) at offset 0
  t.sm_leaf = take((size_t)max_trees * NN * 8, 16);
  t.part_words = std::max(W, kT3MaxLin) * TR;
  t.sm_part = take(2 * (size_t)t.part_words * 8, 16);
  t.sm_xt = take(2 * (size_t)xt_words * 4, 128);
  t.sm_bar = take(64, 16);
  if (n_lin_cols > 0) {
    // feature slices of the linear part: as many walking warps as fit -- either behind the weights, in the room the tree
    // parts use for their tables, or (small tree tables) in the per-warp partial-sum buffers
    const size_t w_end = align_up(lin_bytes, 16);
    const size_t per_slice = (size_t)n_lin_cols * TR * 8;
    const int cap_a = (size_t)t.sm_part > w_end ? (int)(((size_t)t.sm_part - w_end) / (2 * per_slice)) : 0;
    const int cap_b = std::max(W, kT3MaxLin) / n_lin_cols;
    const bool alias = cap_a >= cap_b;
    t.lin_slices = std::max(1, std::min({W, n_in, alias ? cap_a : cap_b}));
    t.lin_part_words = alias ? t.lin_slices * n_lin_cols * TR : t.part_words;
    t.sm_lin_part = alias ? (int32_t)w_end : t.sm_part;
  }
  if (off > (size_t)smem_cap) {  // cannot happen with the budget above; stay on the safe side
    cudaFree(p->d_t3_blob);
    p->d_t3_blob = nullptr;
    return B2S_OK;
  }
  // ---- the prepare kernel: transposed tile | landing tile (TMA boxes or padded rows) | fill | flags | mbarrier
  T3Prep& pr = p->t3_prep;
  memset(&pr, 0, sizeof(pr));
  pr.fill = k.fill;
  pr.n_in = n_in;
  pr.n_in4 = n_in4;
  pr.pitch = pitch;
  pr.any_fill = any_fill ? 1 : 0;
  {
    size_t po = 0;
    auto ptake = [&](size_t bytes, size_t al) {
      po = align_up(po, al);
      const size_t o = po;
      po += bytes;
      return (int32_t)o;
    };
    pr.sm_xt = ptake((size_t)xt_words * 4, 16);
    pr.sm_land = ptake(land_bytes, 1024);
    pr.sm_fill = ptake((size_t)n_in4 * 4, 16);
    pr.sm_bad = ptake((size_t)TR * 4, 16);
    pr.sm_bar = ptake(16, 16);
    p->t3_prep_smem = (int)align_up(po, 16);
    if (p->t3_prep_smem > smem_cap) {
      cudaFree(p->d_t3_blob);
      p->d_t3_blob = nullptr;
      return B2S_OK;
    }
  }
  p->t3_smem = (int)align_up(off, 16);
  p->t3_D = D;
  p->t3_miss = miss;
  p->t3_block = (W + kT3Service) * 32;
  p->t3_grid = cta0;
  p->t3_cols = (int)col_score.size();
  p->t3_parts = P;
  p->t3_ok = true;
  p->kernels_per_batch = 3;
  return B2S_OK;
}

// ------------------------------------------------------------------------------------------ finalize
static int pow2_at_least(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

extern "C" int b2s_plan_finalize(b2s_plan_t p) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_build(p)) return rc;
    if (!G.inited) return fail(B2S_ERR_STATE, "b2s_init was not called");
    const int n_in = p->n_in;
    if (p->out_src.empty()) {
      p->out_src.resize(n_in);
      p->out_kind.assign(n_in, B2S_OUT_COPY);
      p->out_arg.assign(n_in, 0.f);
      for (int j = 0; j < n_in; ++j) p->out_src[j] = j;
    }
    const int n_out = (int)p->out_src.size();
    bool identity_schema = n_out == n_in;  // no schema given, or one that copies every column in place
    for (int j = 0; identity_schema && j < n_out; ++j) identity_schema = p->out_kind[j] == B2S_OUT_COPY && p->out_src[j] == j;
    const int M = (int)p->models.size();
    if (p->vote_kind != B2S_VOTE_NONE) {
      if (M == 0) return fail(B2S_ERR_INVALID, "vote without models");
      if ((int)p->vote_w.size() != M) return fail(B2S_ERR_INVALID, "vote weights (%d) != models (%d)", (int)p->vote_w.size(), M);
    }
    bool any_tree = false, any_class = false, any_reg = false;
    int total_scores = 0, max_scores = 1;
    for (auto& m : p->models) {
      any_tree |= (m.kind == MK_TREES);
      (m.link == B2S_LINK_IDENTITY ? any_reg : any_class) = true;
      total_scores += m.n_scores;
      max_scores = std::max(max_scores, m.n_scores);
    }
    if (any_class && any_reg) return fail(B2S_ERR_UNSUPPORTED, "classifiers and regressors cannot share one plan output");
    if (p->vote_kind == B2S_VOTE_MAJORITY && !any_class && M) {
      // regression outputs voted as labels: allowed (VotingEnsemble casts to int, routers.py:778-780)
    }
    p->mode = M == 0 ? MODE_STORE : (any_tree ? MODE_TREES : MODE_LINEAR);
    p->out_is_int = (M > 0 && (any_class || p->vote_kind == B2S_VOTE_MAJORITY)) ? 1 : 0;
    if (p->vote_kind == B2S_VOTE_MEAN) p->out_is_int = 0;
    p->out_cols = M == 0 ? n_out : (p->vote_kind == B2S_VOTE_NONE ? M : 1);

    bool any_fill = false, any_map = false;
    for (int c = 0; c < n_in; ++c) {
      any_fill |= !std::isnan(p->fill[c]);
      any_map |= !p->maps[c].empty();
    }
    const bool need_expand = !identity_schema || any_fill || any_map;

    // ---- tables
    std::vector<uint32_t> flags(n_in, 0);
    std::vector<int32_t> map_off(n_in + 1, 0);
    std::vector<MapEntry> maps;
    for (int c = 0; c < n_in; ++c) {
      map_off[c] = (int)maps.size();
      for (auto& e : p->maps[c]) maps.push_back(e);
      if (!p->maps[c].empty()) flags[c] |= COL_HAS_MAP;
    }
    map_off[n_in] = (int)maps.size();
    for (int j = 0; j < n_out; ++j)
      if (p->out_kind[j] == B2S_OUT_COPY) flags[p->out_src[j]] |= COL_COPIED;

    int NS = 1;
    std::vector<int32_t> cat_off(n_in + 1, 0);
    std::vector<float> cat_val;
    std::vector<double> wnum, wcat, bias, wgen, leaf, tree_scale;
    std::vector<ModelDesc> descs(std::max(M, 1));
    std::vector<int32_t> classes, tree_root, tree_slot;
    std::vector<TreeNode> nodes;

    if (p->mode == MODE_LINEAR) {
      NS = pow2_at_least(total_scores);
      if (NS > kMaxScores) return fail(B2S_ERR_UNSUPPORTED, "total scores %d > %d", total_scores, kMaxScores);
      // categories per input column, in schema order
      std::vector<std::vector<int>> col_cats(n_in);
      for (int j = 0; j < n_out; ++j)
        if (p->out_kind[j] == B2S_OUT_ONEHOT) col_cats[p->out_src[j]].push_back(j);
      for (int c = 0; c < n_in; ++c) {
        cat_off[c] = (int)cat_val.size();
        for (int j : col_cats[c]) cat_val.push_back(p->out_arg[j]);
        if (!col_cats[c].empty()) flags[c] |= COL_HAS_CAT;
      }
      cat_off[n_in] = (int)cat_val.size();
      wnum.assign((size_t)n_in * NS, 0.0);
      wcat.assign(std::max<size_t>(cat_val.size(), 1) * NS, 0.0);
      bias.assign(NS, 0.0);
      int so = 0;
      for (int mi = 0; mi < M; ++mi) {
        auto& m = p->models[mi];
        for (int k = 0; k < m.n_scores; ++k) {
          bias[so + k] = m.b[k];
          std::vector<int> seen(n_in, 0);
          for (int j = 0; j < n_out; ++j) {
            const int c = p->out_src[j];
            const double w = m.W[(size_t)k * n_out + j];
            if (p->out_kind[j] == B2S_OUT_COPY) {
              wnum[(size_t)c * NS + so + k] += w;
            } else {
              const int idx = cat_off[c] + seen[c]++;
              wcat[(size_t)idx * NS + so + k] = w;
            }
          }
        }
        so += m.n_scores;
      }
    } else if (p->mode == MODE_TREES) {
      NS = max_scores <= 1 ? 1 : (max_scores <= 4 ? 4 : (max_scores <= 8 ? 8 : 16));
      bias.assign(std::max(total_scores, 1), 0.0);
    }
    {
      int so = 0, co = 0;
      for (int mi = 0; mi < M; ++mi) {
        auto& m = p->models[mi];
        ModelDesc d{};
        d.kind = m.kind;
        d.score_off = so;
        d.n_scores = m.n_scores;
        d.link = m.link;
        d.class_off = co;
        d.n_classes = (int)m.classes.size();
        for (int32_t c : m.classes) classes.push_back(c);
        co += (int)m.classes.size();
        if (p->mode == MODE_TREES) {
          if (m.kind == MK_TREES) {
            d.tree_begin = (int)tree_root.size();
            const int nt = (int)m.tree_slot.size();
            for (int t = 0; t < nt; ++t) {
              const int base = (int)nodes.size();
              tree_root.push_back(base);
              tree_slot.push_back(m.tree_slot[t]);
              tree_scale.push_back(m.tree_scale[t]);
              for (int i = m.tree_offset[t]; i < m.tree_offset[t + 1]; ++i) {
                TreeNode nd;
                nd.feature = m.feature[i];
                nd.threshold = m.threshold[i];
                nd.left = nd.feature >= 0 ? base + m.left[i] : 0;
                nd.right = nd.feature >= 0 ? base + m.right[i] : 0;
                nodes.push_back(nd);
                leaf.push_back(m.leaf_value[i]);
              }
            }
            d.tree_end = (int)tree_root.size();
            for (int k = 0; k < m.n_scores; ++k) bias[so + k] = m.init[k];
          } else {
            d.w_off = (int)wgen.size();
            for (double w : m.W) wgen.push_back(w);
            for (int k = 0; k < m.n_scores; ++k) bias[so + k] = m.b[k];
          }
        }
        descs[mi] = d;
        so += m.n_scores;
      }
    }
    if (bias.empty()) bias.assign(1, 0.0);

    std::vector<uint8_t> chunk_kind((n_in + 3) / 4, 1);
    for (int ch = 0; ch < (int)chunk_kind.size(); ++ch) {
      bool fast = (ch * 4 + 3 < n_in);
      for (int u = 0; fast && u < 4; ++u) fast = (flags[ch * 4 + u] == COL_COPIED);
      chunk_kind[ch] = fast ? 0 : 1;
    }
    // ---- dense head (tcgen05): linear scorers with more than 8 scores in total over plain numeric columns.  The float64
    // coefficients become three tf32 terms wh + wm + wl (11 significant bits each, 33 in total); W^T rows padded to 16 / 32
    std::vector<float> dense_wh, dense_wm, dense_wl;
    int dense_pad = 0;
    {
      const char* denv = getenv("B2S_DENSE");  // 1 (default) | 0: stay on the fp64 row kernels (A/B runs)
      int n_cat_cols = 0;
      for (int c = 0; c < n_in; ++c) n_cat_cols += (cat_off[c + 1] > cat_off[c]) ? 1 : 0;
      bool all_copied = true;
      for (int c = 0; c < n_in; ++c) all_copied = all_copied && (flags[c] & COL_COPIED);
      if ((!denv || atoi(denv) != 0) && p->mode == MODE_LINEAR && total_scores > 8 && total_scores <= 32 && identity_schema &&
          !any_map && n_cat_cols == 0 && all_copied && (n_in % 32) == 0 && n_in <= kDenseMaxIn) {
        dense_pad = total_scores <= 16 ? 16 : 32;
        dense_wh.assign((size_t)dense_pad * n_in, 0.0f);
        dense_wm.assign((size_t)dense_pad * n_in, 0.0f);
        dense_wl.assign((size_t)dense_pad * n_in, 0.0f);
        auto tf32 = [](double x) {  // the leading 11 significant bits of the float32 nearest to x
          float f = (float)x;
          if (!std::isfinite(f)) return f;
          uint32_t b;
          memcpy(&b, &f, 4);
          b &= 0xffffe000u;
          memcpy(&f, &b, 4);
          return f;
        };
        for (int kk = 0; kk < total_scores; ++kk)
          for (int c = 0; c < n_in; ++c) {
            const double w = wnum[(size_t)c * NS + kk];
            const float hi = tf32(w);
            const double r1 = w - (double)hi;  // exact in float64
            const float mid = tf32(r1);
            dense_wh[(size_t)kk * n_in + c] = hi;
            dense_wm[(size_t)kk * n_in + c] = mid;
            dense_wl[(size_t)kk * n_in + c] = tf32(r1 - (double)mid);
          }
      }
    }
    // ---- upload one blob
    BlobBuilder bb;
    const size_t o_dwh = bb.add(dense_wh), o_dwm = bb.add(dense_wm), o_dwl = bb.add(dense_wl);
    const size_t o_fill = bb.add(p->fill), o_flags = bb.add(flags), o_mapoff = bb.add(map_off), o_maps = bb.add(maps),
                 o_osrc = bb.add(p->out_src), o_okind = bb.add(p->out_kind), o_oarg = bb.add(p->out_arg),
                 o_catoff = bb.add(cat_off), o_catval = bb.add(cat_val), o_wnum = bb.add(wnum), o_wcat = bb.add(wcat),
                 o_bias = bb.add(bias), o_models = bb.add(descs), o_classes = bb.add(classes),
                 o_votew = bb.add(p->vote_w), o_wgen = bb.add(wgen), o_nodes = bb.add(nodes), o_leaf = bb.add(leaf),
                 o_troot = bb.add(tree_root), o_tslot = bb.add(tree_slot), o_tscale = bb.add(tree_scale),
                 o_chunk = bb.add(chunk_kind);
    CUDA_TRY(cudaSetDevice(G.device));
    CUDA_TRY(cudaMalloc(&p->d_blob, bb.data.size()));
    CUDA_TRY(cudaMemcpy(p->d_blob, bb.data.data(), bb.data.size(), cudaMemcpyHostToDevice));
    p->blob_bytes = bb.data.size();
    char* B = p->d_blob;

    KParams& k = p->kp;
    memset(&k, 0, sizeof(k));
    k.n_in = n_in;
    k.n_out = n_out;
    k.out_cols = p->out_cols;
    k.n_models = M;
    k.n_scores = total_scores;
    k.vote_kind = p->vote_kind;
    k.out_is_int = p->out_is_int;
    k.need_expand = need_expand ? 1 : 0;
    k.models_pow2 = pow2_at_least(std::max(M, 1));
    k.n_cat = (int)cat_val.size();
    k.n_maps = (int)maps.size();
    k.fill = (const float*)(B + o_fill);
    k.col_flags = (const uint32_t*)(B + o_flags);
    k.map_off = (const int32_t*)(B + o_mapoff);
    k.maps = (const MapEntry*)(B + o_maps);
    k.out_src = (const int32_t*)(B + o_osrc);
    k.out_kind = (const int32_t*)(B + o_okind);
    k.out_arg = (const float*)(B + o_oarg);
    k.cat_off = (const int32_t*)(B + o_catoff);
    k.cat_val = (const float*)(B + o_catval);
    k.wnum = (const double*)(B + o_wnum);
    k.wcat = (const double*)(B + o_wcat);
    k.bias = (const double*)(B + o_bias);
    k.models = (const ModelDesc*)(B + o_models);
    k.classes = (const int32_t*)(B + o_classes);
    k.vote_w = (const double*)(B + o_votew);
    k.wgen = (const double*)(B + o_wgen);
    k.nodes = (const TreeNode*)(B + o_nodes);
    k.leaf = (const double*)(B + o_leaf);
    k.tree_root = (const int32_t*)(B + o_troot);
    k.tree_slot = (const int32_t*)(B + o_tslot);
    k.tree_scale = (const double*)(B + o_tscale);
    k.chunk_kind = (const uint8_t*)(B + o_chunk);
    if (dense_pad > 0 && tensor_map_encoder() != nullptr) {
      DenseParams& d = p->dense;
      memset(&d, 0, sizeof(d));
      d.wh = (const float*)(B + o_dwh);
      d.wm = (const float*)(B + o_dwm);
      d.wl = (const float*)(B + o_dwl);
      d.fill = k.fill;
      d.bias = k.bias;
      d.n_in = n_in;
      d.n_scores = total_scores;
      d.n_pad = dense_pad;
      d.tmem_cols = dense_tmem_cols(n_in, dense_pad);
      d.exact = (getenv("B2S_DENSE_EXACT") && atoi(getenv("B2S_DENSE_EXACT")) != 0) ? 1 : 0;
      d.any_fill = any_fill ? 1 : 0;
      for (int kk = 0; kk < 32; ++kk) {
        d.biasf[kk] = kk < total_scores ? (float)bias[kk] : 0.0f;
        d.votewf[kk] = 0.0f;
        d.labels[kk] = kk;
      }
      {
        bool simple = true;  // every model: one identity score
        for (auto& m : p->models) simple = simple && m.link == B2S_LINK_IDENTITY && m.n_scores == 1;
        d.epi = DENSE_EPI_GENERIC;
        if (simple && p->vote_kind == B2S_VOTE_NONE) d.epi = DENSE_EPI_SCORES;
        if (simple && p->vote_kind == B2S_VOTE_MEAN) {
          d.epi = DENSE_EPI_MEAN;
          for (int mi = 0; mi < M; ++mi) d.votewf[mi] = (float)p->vote_w[mi];
        }
        if (M == 1 && p->models[0].link == B2S_LINK_ARGMAX && p->vote_kind == B2S_VOTE_NONE) {
          d.epi = DENSE_EPI_ARGMAX;
          const auto& cls = p->models[0].classes;
          for (int kk = 0; kk < total_scores && kk < 32; ++kk) d.labels[kk] = cls.empty() ? kk : cls[kk];
        }
      }
      p->dense_smem = dense_smem_bytes(n_in, dense_pad);
      if (p->dense_smem <= (int)G.prop.sharedMemPerBlockOptin) {
        p->dense_grid = G.prop.multiProcessorCount;  // persistent: one CTA per SM (its shared memory and TMEM see to that)
        p->dense_ok = true;
      }
    }

    // ---- launch geometry + shared-memory carve-up
    // pitch (words): rows 16B aligned and (pitch/4) odd -> conflict-free LDS.128 for one-thread-per-row
    const int n_in4 = (int)align_up(n_in, 4);
    int pitch = n_in4 + 4;
    if (((pitch / 4) & 1) == 0) pitch += 4;
    int exp_pitch = n_out | 1;
    const int smem_cap = (int)G.prop.sharedMemPerBlockOptin;
    const int sms = G.prop.multiProcessorCount;
    int block, tile_rows, stages, blocks_per_sm;
    int tpr = 1;
    if (p->mode == MODE_LINEAR) {
      tpr = NS <= 8 ? 4 : (NS == 16 ? 2 : 1);
      const int nch = (n_in + 3) / 4;
      while (tpr > 1 && nch < tpr * 2) tpr /= 2;
      tile_rows = 128;
      block = tile_rows * tpr;
      stages = 3;
      blocks_per_sm = 2;
    } else if (p->mode == MODE_TREES) {
      block = 256;
      tile_rows = block / k.models_pow2;
      stages = 2;
      blocks_per_sm = 2;
    } else {
      block = 256;
      tile_rows = 128;
      stages = 2;
      blocks_per_sm = 2;
    }
    auto carve = [&](int tr, int st) {
      size_t off = 0;
      auto take = [&](size_t bytes) {
        size_t o = align_up(off, 16);
        off = o + bytes;
        return (int32_t)o;
      };
      k.sm_fill = take((size_t)n_in * 4);
      k.sm_flags = take((size_t)n_in * 4);
      k.sm_mapoff = take((size_t)(n_in + 1) * 4);
      k.sm_catoff = take((size_t)(n_in + 1) * 4);
      k.sm_catval = take(std::max<size_t>(cat_val.size(), 1) * 4);
      k.sm_wnum = take(p->mode == MODE_LINEAR ? (size_t)n_in * NS * 8 : 16);
      k.sm_wcat = take(p->mode == MODE_LINEAR ? std::max<size_t>(cat_val.size(), 1) * NS * 8 : 16);
      k.sm_outsrc = take((size_t)n_out * 4);
      k.sm_outkind = take((size_t)n_out * 4);
      k.sm_outarg = take((size_t)n_out * 4);
      k.sm_pred = take(p->mode == MODE_TREES ? (size_t)tr * k.models_pow2 * 8 : 16);
      k.sm_chunk = take((size_t)(n_in + 3) / 4 + 16);
      k.sm_part = take((p->mode == MODE_LINEAR && tpr > 1) ? (size_t)tr * tpr * NS * 8 : 16);
      k.sm_pst = take((p->mode == MODE_LINEAR && tpr > 1) ? (size_t)tr * tpr * 4 : 16);
      k.sm_exp = take((p->mode != MODE_LINEAR && need_expand) ? (size_t)tr * exp_pitch * 4 : 16);
      k.sm_tiles = take((size_t)st * tr * pitch * 4);
      return (int)align_up(off, 16);
    };
    int total = carve(tile_rows, stages);
    // shrink until `blocks_per_sm` blocks fit (then until one fits)
    while (total * blocks_per_sm > smem_cap * 1 && (stages > 2 || blocks_per_sm > 1)) {
      if (stages > 2) --stages; else --blocks_per_sm;
      total = carve(tile_rows, stages);
    }
    while (total > smem_cap && stages > 1) total = carve(tile_rows, --stages);
    while (total > smem_cap && tile_rows > 8 && p->mode != MODE_LINEAR) {
      tile_rows /= 2;
      total = carve(tile_rows, stages);
    }
    if (total > smem_cap) {
      if (p->mode == MODE_LINEAR) {
        // wide rows: fewer rows per tile (threads beyond tile_rows idle in the compute phase)
        while (total > smem_cap && tile_rows > 8) {
          tile_rows /= 2;
          total = carve(tile_rows, stages);
        }
      }
      if (total > smem_cap) return fail(B2S_ERR_UNSUPPORTED, "plan needs %d B shared memory > %d B", total, smem_cap);
    }
    if (p->mode == MODE_TREES) block = std::max(32, tile_rows * k.models_pow2);
    if (p->mode == MODE_LINEAR) block = tile_rows * tpr;
    k.tpr = tpr;
    k.sm_total = total;
    k.tile_rows = tile_rows;
    k.pitch = pitch;
    k.exp_pitch = exp_pitch;
    k.stages = stages;
    p->NS = NS;
    p->block = block;
    int occ = std::max(1, std::min(blocks_per_sm, smem_cap / std::max(total, 1)));
    p->grid = sms * occ;

    {
      int n_cat_cols = 0;
      for (int c = 0; c < n_in; ++c) n_cat_cols += (cat_off[c + 1] > cat_off[c]) ? 1 : 0;
      if (p->mode == MODE_LINEAR && !any_map && n_in <= 128 && NS <= 8 && n_cat_cols <= kRTMaxCatCols &&
          (int)cat_val.size() <= kRTMaxCats) {
        const int nch = (n_in + 3) / 4;
        p->rt_NCH = nch <= 4 ? 4 : (nch <= 8 ? 8 : (nch <= 16 ? 16 : 32));
        p->rt_NS = NS;
        p->rt_cat_cols = n_cat_cols;
        bool simple = true;
        for (auto& m : p->models) simple = simple && m.link == B2S_LINK_IDENTITY && m.n_scores == 1;
        RTTables t{n_in, p->out_cols, M, p->vote_kind, p->out_is_int, (simple && p->vote_kind != B2S_VOTE_MAJORITY) ? 1 : 0, NS,
                   &p->fill, &flags, &wnum, &bias, &p->vote_w, &cat_off, &cat_val, k.wcat, k.vote_w, k.models, k.classes};
        rt_build_any(p, t);
        int rpitch = p->rt_NCH * 4 + 4;
        if (((rpitch / 4) & 1) == 0) rpitch += 4;
        p->rt_pitch = rpitch;
        {
          const size_t fixed = 1024 + 64 + align_up((size_t)(cat_val.size() + 1) * NS * 8, 16);
          const size_t part = (size_t)(rt_tpr(p->rt_NCH) - 1) * 128 * NS * 8;
          // padded tiles + one partial-sum buffer (LDGSTS / per-row bulk), or swizzled tiles + two (tensor map)
          const size_t padded = fixed + part + (size_t)kRTStages * kRTTileRows * rpitch * 4;
          const size_t swizzled = fixed + 2 * part + (size_t)kRTStages * kRTTileRows * p->rt_NCH * 16;
          p->rt_smem = (int)std::max(padded, swizzled);
        }
        int occ = 0;
        if (p->rt_smem <= smem_cap && rt_launch(p, nullptr, 0, 0, nullptr, nullptr, 0, nullptr, true, &occ) == cudaSuccess && occ >= 1) {
          p->rt_ok = true;
          p->rt_grid = sms * occ;
        } else {
          cudaGetLastError();
        }
      }
    }
    // ---- round-2 tree path: parts resident in shared memory (b2s_trees3.cuh).  Covers tree ensembles (any number of
    // score slots per model), ensembles mixing tree and linear scorers, an Imputer in front, and NaN routing.  The plans it
    // declines (deeper than kT3MaxDepth, more parts than SMs, rows too wide for a part, a schema or MapValues in front) run
    // on rows_kernel<TREES>.
    if (p->mode == MODE_TREES && identity_schema && !any_map) {
      if (int rc = t3_build(p, k, any_fill)) return rc;
    }
    for (int i = 0; i < 4; ++i) CUDA_TRY(cudaEventCreate(&p->ev[i]));
    p->finalized = true;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// which kernel family a finalized plan launches (so that a silent fallback cannot hide in a benchmark)
extern "C" const char* b2s_plan_kernel(b2s_plan_t p) {
  if (!p || !p->finalized) return "";
  static thread_local char buf[200];
  const bool tmap = rt_tmap_ok(p);
  if (p->dense_ok) snprintf(buf, sizeof(buf), "dense_head_kernel<N=%d> (tcgen05.mma kind::tf32, %s, TMEM accumulator groups; %d scores over %d columns)", p->dense.n_pad, p->dense.exact ? "exact 3-term input split" : "2-term input split", p->dense.n_scores, p->dense.n_in);
  else if (p->t3_ok) snprintf(buf, sizeof(buf), "t3_prep_kernel + trees3_kernel<D=%d,%s> + t3_vote_kernel (%d parts resident in shared memory, %d walking warps)", p->t3_D, p->t3_miss ? "NaN routing" : "floats", p->t3_parts, p->t3.warps);
  else if (p->rt_ok) snprintf(buf, sizeof(buf), "rowthread_kernel<NCH=%d,NS=%d,TPR=%d,%s>", p->rt_NCH, p->rt_NS, rt_tpr(p->rt_NCH), tmap ? "TMA tensor-map loads" : "TMA bulk loads");
  else snprintf(buf, sizeof(buf), "rows_kernel<%s,NS=%d>", p->mode == MODE_LINEAR ? "LINEAR" : (p->mode == MODE_TREES ? "TREES" : "STORE"), p->NS);
  return buf;
}

extern "C" int b2s_plan_out_info(b2s_plan_t p, int32_t* out_cols, int32_t* out_is_int) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (out_cols) *out_cols = p->out_cols;
    if (out_is_int) *out_is_int = p->out_is_int;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ execution
struct NvtxRange {  // one range per plan launch, named after the kernel family (nsys / ncu --nvtx timelines)
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

static int launch_on(b2s_plan_t p, const void* d_rows, int64_t n_rows, int64_t stride, void* d_out, int32_t* d_status,
                     cudaStream_t st, bool host_rows = false) {
  if (n_rows == 0) return B2S_OK;
  NvtxRange nvtx(p->dense_ok ? "b2s:dense_head" : p->t3_ok ? "b2s:trees3 (prep+walk+vote)"
                 : p->rt_ok ? "b2s:rowthread" : p->mode == MODE_STORE ? "b2s:rows_store" : "b2s:rows_kernel");
  KParams k = p->kp;
  k.rows = (const char*)d_rows;
  k.row_stride = stride;
  k.n_rows = n_rows;
  k.out = (float*)d_out;
  k.status = d_status;
  k.vec_ok = ((p->n_in % 4) == 0 && (stride % 16) == 0 && ((uintptr_t)d_rows % 16) == 0) ? 1 : 0;
  k.n_peers = (int)p->peers.size();
  k.peer_off = p->peer_off;
  for (int g = 0; g < k.n_peers; ++g) k.peers[g] = (float*)p->peers[g];
  k.sig = MergeSig{};
  if (p->comm) {
    // one more step of the attached communicator: this launch's votes go to slot (epoch & 3) of every rank's merged
    // rows, at this rank's row block; the launch's last CTA then publishes the epoch in every rank's flag array
    b2s_comm_s* c = p->comm;
    if (n_rows > c->max_rows) return fail(B2S_ERR_INVALID, "shard of %lld rows exceeds the communicator's %lld", (long long)n_rows, (long long)c->max_rows);
    if (p->mode == MODE_STORE) return fail(B2S_ERR_UNSUPPORTED, "transform-only plans have no vote to merge");
    const uint32_t e = ++c->epoch;
    k.n_peers = c->world;
    k.peer_off = (int64_t)c->rank * c->max_rows;
    k.sig.n = c->world;
    k.sig.rank = c->rank;
    k.sig.epoch = e;
    k.sig.counter = c->counter();
    for (int g = 0; g < c->world; ++g) {
      const int r = (c->rank + 1 + g) % c->world;  // start at the right-hand neighbour: the ranks write to different targets
      k.peers[g] = (float*)c->buf(r, e);
      k.sig.flags[g] = c->flags(r);
    }
    if (c->fused_lag >= 0 && e > (uint32_t)c->fused_lag) {
      static const long long fused_timeout_ns = (getenv("B2S_COMM_TIMEOUT_MS") ? atoll(getenv("B2S_COMM_TIMEOUT_MS")) : 10000ll) * 1000000ll;
      k.sig.wait_epoch = e - (uint32_t)c->fused_lag;
      k.sig.wait_flags = c->flags(c->rank);
      k.sig.timeout_flag = reinterpret_cast<uint32_t*>(c->base) + 65;
      k.sig.timeout_ns = fused_timeout_ns;
      c->fused_epoch = k.sig.wait_epoch;
    }
  }
  if (p->t3_ok) {
    const int C = p->t3_cols;
    const int64_t n_tiles = (n_rows + kT3TR - 1) / kT3TR;
    b2s_plan_s::TreeScratch sc;
    {
      std::lock_guard<std::mutex> lk(p->scratch_mu);
      b2s_plan_s::TreeScratch& mine = p->t3_scratch[st];
      if (n_rows > mine.rows) {  // cudaFree waits for the work that still reads the old buffers
        if (mine.pred) cudaFree(mine.pred);
        if (mine.row_bad) cudaFree(mine.row_bad);
        if (mine.xt) cudaFree(mine.xt);
        mine = b2s_plan_s::TreeScratch{};
        const int64_t cap = std::max<int64_t>(align_up((size_t)n_rows, 64), 65536);
        CUDA_TRY(cudaMalloc(&mine.pred, (size_t)cap * C * 8));
        CUDA_TRY(cudaMalloc(&mine.row_bad, (size_t)cap * 4));
        CUDA_TRY(cudaMalloc(&mine.xt, (size_t)(cap / kT3TR) * p->t3.xt_words * 4));
        mine.rows = cap;
      }
      sc = mine;
    }
    T3Prep pr = p->t3_prep;
    pr.rows = (const char*)d_rows;
    pr.row_stride = stride;
    pr.n_rows = n_rows;
    pr.xt = sc.xt;
    pr.row_bad = sc.row_bad;
    pr.vec_ok = k.vec_ok;
    alignas(64) CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    pr.use_tmap = (!host_rows && pr.vec_ok && (p->n_in % 32) == 0 && encode_rows_map(&tmap, d_rows, n_rows, stride, p->n_in, kT3TR)) ? 1 : 0;
    const int resident = std::max(1, (int)G.prop.sharedMemPerMultiprocessor / std::max(p->t3_prep_smem + 1024, 1));
    const int pgrid = (int)std::max<int64_t>(1, std::min<int64_t>(n_tiles, (int64_t)G.prop.multiProcessorCount * std::min(resident, 4)));
    G.launches.fetch_add(3, std::memory_order_relaxed);
    cudaError_t e3 = t3_launch_prep(pr, tmap, p->t3_miss, pgrid, p->t3_prep_smem, (int)G.prop.sharedMemPerBlockOptin, st);
    if (e3 != cudaSuccess) return fail(B2S_ERR_CUDA, "tree prepare kernel launch failed: %s", cudaGetErrorString(e3));
    T3Params t = p->t3;
    t.xt = sc.xt;
    t.n_rows = n_rows;
    t.partial = sc.pred;
    t.col_stride = sc.rows;
    e3 = t3_launch_walk(t, p->t3_D, p->t3_miss, p->t3_grid, p->t3_block, p->t3_smem, (int)G.prop.sharedMemPerBlockOptin, st);
    if (e3 != cudaSuccess) return fail(B2S_ERR_CUDA, "tree kernel launch failed: %s", cudaGetErrorString(e3));
    const int vgrid = (int)std::max<int64_t>(1, std::min<int64_t>(4 * G.prop.multiProcessorCount, (n_rows + 255) / 256));
    e3 = t3_launch_vote(k, sc.pred, sc.rows, p->d_t3_col_score, C, sc.row_bad, vgrid, st);
    if (e3 != cudaSuccess) return fail(B2S_ERR_CUDA, "vote kernel launch failed: %s", cudaGetErrorString(e3));
    return B2S_OK;
  }
  if (p->dense_ok && !host_rows && k.vec_ok) {
    alignas(64) CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    if (encode_rows_map(&tmap, d_rows, n_rows, stride, p->n_in, kDenseTileRows)) {
      DenseParams d = p->dense;
      d.n_rows = n_rows;
      const int64_t tiles = (n_rows + kDenseTileRows - 1) / kDenseTileRows;
      const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(p->dense_grid, tiles));
      G.launches.fetch_add(1, std::memory_order_relaxed);
      cudaError_t e = dense_launch(d, k, tmap, grid, p->dense_smem, (int)G.prop.sharedMemPerBlockOptin, st);
      if (e != cudaSuccess) return fail(B2S_ERR_CUDA, "dense head kernel launch failed: %s", cudaGetErrorString(e));
      return B2S_OK;
    }
  }
  if (p->rt_ok) {
    G.launches.fetch_add(1, std::memory_order_relaxed);
    LaunchCtx lc;
    lc.k = &k;
    lc.host_rows = host_rows;
    cudaError_t e = rt_launch(p, d_rows, stride, n_rows, d_out, d_status, k.vec_ok, st, false, nullptr, nullptr, &lc);
    if (e != cudaSuccess) return fail(B2S_ERR_CUDA, "row-thread kernel launch failed: %s", cudaGetErrorString(e));
    return B2S_OK;
  }
  // small batches: shrink the tile so that every SM gets work (latency path); the shared-memory
  // carve-up was sized for the largest tile, so any smaller power-of-two tile fits
  int block = p->block;
  if (p->mode != MODE_STORE) {
    const int per_row = p->block / k.tile_rows;
    while (k.tile_rows > 32 && (n_rows + k.tile_rows - 1) / k.tile_rows < (int64_t)G.prop.multiProcessorCount) k.tile_rows /= 2;
    block = k.tile_rows * per_row;
  }
  const int64_t tiles = (n_rows + k.tile_rows - 1) / k.tile_rows;
  const int grid = (int)std::min<int64_t>(p->grid, tiles);
  cudaError_t e = launch_plan(p, k, grid, block, st);
  if (e != cudaSuccess) return fail(B2S_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return B2S_OK;
}

extern "C" int b2s_run_device(b2s_plan_t p, const void* d_rows, int64_t n_rows, int64_t row_stride_bytes, void* d_out,
                              int32_t* d_status, void* stream) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (n_rows < 0 || row_stride_bytes < (int64_t)p->n_in * 4) return fail(B2S_ERR_INVALID, "bad n_rows/stride");
    return launch_on(p, d_rows, n_rows, row_stride_bytes, d_out, d_status, stream ? (cudaStream_t)stream : G.stream);
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

int b2s_int_launch_gathered(b2s_plan_s* p, const B2SGather& g, long long n, void* d_out, int* d_status, cudaStream_t st) {
  if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
  if (g.n_feat != p->n_in) return fail(B2S_ERR_INVALID, "the table has %d features, the plan takes %d", g.n_feat, p->n_in);
  static const int fused = getenv("B2S_ENRICH_FUSED") ? atoi(getenv("B2S_ENRICH_FUSED")) : 1;
  // the gather loader lives in the row-thread kernel (linear models, rows of whole 16-byte chunks); with a table impute
  // policy, one-hot sources would need the policy applied before the category search: those plans gather first
  if (!fused || !p->rt_ok || p->t3_ok || (p->n_in % 4) != 0) return fail(B2S_ERR_UNSUPPORTED, "plan is not fusable with the gather");
  if (g.any_impute && p->rt_cat_cols > 0) return fail(B2S_ERR_UNSUPPORTED, "one-hot columns under a table impute policy gather first");
  if (n <= 0) return B2S_OK;
  G.launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = rt_launch(p, nullptr, (int64_t)p->n_in * 4, n, d_out, d_status, 1, st, false, nullptr, &g);
  if (e != cudaSuccess) return fail(B2S_ERR_CUDA, "row-thread (gather) kernel launch failed: %s", cudaGetErrorString(e));
  return B2S_OK;
}

static int ensure_stage(b2s_plan_t p, int64_t n_rows) {
  if (n_rows <= p->stage_rows) return B2S_OK;
  // free first, and forget the old buffers before anything can fail: a failed allocation below must leave the plan
  // with no staging area (stage_rows = 0) rather than with dangling pointers a later call would copy into / free twice
  if (p->h_stage_in) cudaFreeHost(p->h_stage_in);
  if (p->h_stage_out) cudaFreeHost(p->h_stage_out);
  if (p->d_stage_in) cudaFree(p->d_stage_in);
  if (p->d_stage_out) cudaFree(p->d_stage_out);
  if (p->d_stage_status) cudaFree(p->d_stage_status);
  p->h_stage_in = nullptr;
  p->h_stage_out = nullptr;
  p->d_stage_in = nullptr;
  p->d_stage_out = nullptr;
  p->d_stage_status = nullptr;
  p->stage_rows = 0;
  const int64_t cap = std::max<int64_t>(n_rows, 4096);
  CUDA_TRY(cudaMallocHost(&p->h_stage_in, (size_t)cap * p->n_in * 4));
  CUDA_TRY(cudaMallocHost(&p->h_stage_out, (size_t)cap * (p->out_cols + 1) * 4));
  CUDA_TRY(cudaMalloc(&p->d_stage_in, (size_t)cap * p->n_in * 4));
  CUDA_TRY(cudaMalloc(&p->d_stage_out, (size_t)cap * p->out_cols * 4));
  CUDA_TRY(cudaMalloc(&p->d_stage_status, (size_t)cap * 4));
  p->stage_rows = cap;
  return B2S_OK;
}

static void pack_rows(char* dst, const void* rows, int64_t n_rows, int64_t stride, int64_t row_bytes) {
  if (stride == row_bytes) {
    memcpy(dst, rows, (size_t)n_rows * row_bytes);
  } else {
    const char* s = (const char*)rows;
    for (int64_t r = 0; r < n_rows; ++r) memcpy(dst + r * row_bytes, s + r * stride, (size_t)row_bytes);
  }
}

extern "C" int b2s_run_host(b2s_plan_t p, const void* rows, int64_t n_rows, int64_t row_stride_bytes, void* out,
                            int64_t out_bytes, int32_t* row_status, b2s_stats* stats) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    const int64_t row_bytes = (int64_t)p->n_in * 4;
    if (n_rows < 0 || row_stride_bytes < row_bytes) return fail(B2S_ERR_INVALID, "bad n_rows/stride");
    if (out_bytes < n_rows * p->out_cols * 4) return fail(B2S_ERR_INVALID, "out buffer too small");
    if (n_rows == 0) return B2S_OK;
    std::lock_guard<std::mutex> lk(p->host_mu);
    CUDA_TRY(cudaSetDevice(G.device));
    if (int rc = ensure_stage(p, n_rows)) return rc;
    cudaStream_t st = G.stream;
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, rows) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
                        row_stride_bytes == row_bytes;
    cudaGetLastError();
    const void* src = rows;
    if (!pinned) {
      pack_rows(p->h_stage_in, rows, n_rows, row_stride_bytes, row_bytes);
      src = p->h_stage_in;
    }
    const size_t out_sz = (size_t)n_rows * p->out_cols * 4;
    // Large pinned batches run as a pipeline of chunks: chunk c+1 crosses PCIe while chunk c is computed, copied back and
    // post-processed on the host, so the call costs about one H2D of the batch.  (Not with merge targets: their row offset
    // is per launch.)
    static const int64_t pipe_rows = getenv("B2S_HOST_CHUNK") ? atoll(getenv("B2S_HOST_CHUNK")) : 65536;  // measured: 16Ki 162, 32Ki 184, 64Ki 189 M events/s (one piece: 169)
    if (pinned && pipe_rows > 0 && n_rows >= 2 * pipe_rows && p->peers.empty()) {
      // whole tiles per chunk keep every chunk's base 16-byte (and tensor-map) aligned
      const int64_t chunk = (int64_t)align_up((size_t)std::max<int64_t>(pipe_rows, (n_rows + 63) / 64), 1024);
      const int n_chunks = (int)((n_rows + chunk - 1) / chunk);
      while ((int)p->chunk_ev.size() < 4 * n_chunks) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreate(&e));
        p->chunk_ev.push_back(e);
      }
      cudaStream_t cs = G.copy_stream;
      int32_t* h_status = (int32_t*)(p->h_stage_out + out_sz);
      const size_t out_row = (size_t)p->out_cols * 4;
      CUDA_TRY(cudaEventRecord(p->ev[0], cs));
      for (int c = 0; c < n_chunks; ++c) {
        const int64_t r0 = (int64_t)c * chunk, nr = std::min<int64_t>(chunk, n_rows - r0);
        cudaEvent_t* ce = &p->chunk_ev[4 * c];
        CUDA_TRY(cudaMemcpyAsync(p->d_stage_in + r0 * row_bytes, (const char*)src + r0 * row_bytes, (size_t)nr * row_bytes,
                                 cudaMemcpyHostToDevice, cs));
        CUDA_TRY(cudaEventRecord(ce[0], cs));
        CUDA_TRY(cudaStreamWaitEvent(st, ce[0], 0));
        CUDA_TRY(cudaEventRecord(ce[1], st));
        if (int rc = launch_on(p, p->d_stage_in + r0 * row_bytes, nr, row_bytes, p->d_stage_out + r0 * out_row,
                               p->d_stage_status + r0, st)) {
          cudaStreamSynchronize(cs);
          cudaStreamSynchronize(st);
          return rc;
        }
        CUDA_TRY(cudaEventRecord(ce[2], st));
        CUDA_TRY(cudaMemcpyAsync(p->h_stage_out + r0 * out_row, p->d_stage_out + r0 * out_row, (size_t)nr * out_row,
                                 cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(h_status + r0, p->d_stage_status + r0, (size_t)nr * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaEventRecord(ce[3], st));
      }
      int bad = 0;
      for (int c = 0; c < n_chunks; ++c) {  // hand each chunk to the caller as it lands
        const int64_t r0 = (int64_t)c * chunk, nr = std::min<int64_t>(chunk, n_rows - r0);
        CUDA_TRY(cudaEventSynchronize(p->chunk_ev[4 * c + 3]));
        memcpy((char*)out + r0 * out_row, p->h_stage_out + r0 * out_row, (size_t)nr * out_row);
        for (int64_t r = r0; r < r0 + nr; ++r) bad += (h_status[r] & B2S_ROW_NONFINITE_INPUT) ? 1 : 0;
        if (row_status) memcpy(row_status + r0, h_status + r0, (size_t)nr * 4);
      }
      CUDA_TRY(cudaStreamSynchronize(cs));
      if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rows = n_rows;
        cudaEventElapsedTime(&stats->h2d_ms, p->ev[0], p->chunk_ev[4 * (n_chunks - 1)]);
        for (int c = 0; c < n_chunks; ++c) {  // the phases of different chunks overlap: these are sums over chunks
          float k = 0.f, d = 0.f;
          cudaEventElapsedTime(&k, p->chunk_ev[4 * c + 1], p->chunk_ev[4 * c + 2]);
          cudaEventElapsedTime(&d, p->chunk_ev[4 * c + 2], p->chunk_ev[4 * c + 3]);
          stats->kernel_ms += k;
          stats->d2h_ms += d;
        }
        stats->kernels = p->kernels_per_batch * n_chunks;
        stats->nonfinite_rows = bad;
      }
      return B2S_OK;
    }
    // Not pipelined: the kernels write votes and status words straight into pinned host memory (posted PCIe writes of a few
    // bytes per row: no D2H copy, one synchronisation).  A tiny batch is also READ from pinned host memory by the kernels
    // (no H2D copy: the latency path of a small serving batch); larger ones cross PCIe on the copy engine first, which is
    // where the bandwidth is.  Not with merge targets: those kernels write to the targets.
    static const int64_t zc_in_bytes = getenv("B2S_ZEROCOPY_IN_BYTES") ? atoll(getenv("B2S_ZEROCOPY_IN_BYTES")) : 65536;
    static const int zc_out = getenv("B2S_ZEROCOPY_OUT") ? atoi(getenv("B2S_ZEROCOPY_OUT")) : 1;
    const bool merging = !p->peers.empty() || p->comm;
    if (zc_out && !merging) {
      const bool zc_in = n_rows * row_bytes <= zc_in_bytes;
      const void* d_src = p->d_stage_in;
      if (stats) CUDA_TRY(cudaEventRecord(p->ev[0], st));
      if (zc_in) d_src = pinned ? attr.devicePointer : (const void*)p->h_stage_in;
      else CUDA_TRY(cudaMemcpyAsync(p->d_stage_in, src, (size_t)n_rows * row_bytes, cudaMemcpyHostToDevice, st));
      if (stats) CUDA_TRY(cudaEventRecord(p->ev[1], st));
      if (int rc = launch_on(p, d_src, n_rows, row_bytes, p->h_stage_out, (int32_t*)(p->h_stage_out + out_sz), st, zc_in)) return rc;
      if (stats) CUDA_TRY(cudaEventRecord(p->ev[2], st));
      CUDA_TRY(cudaStreamSynchronize(st));
      memcpy(out, p->h_stage_out, out_sz);
      const int32_t* hs = (const int32_t*)(p->h_stage_out + out_sz);
      int bad = 0;
      for (int64_t r = 0; r < n_rows; ++r) bad += (hs[r] & B2S_ROW_NONFINITE_INPUT) ? 1 : 0;
      if (row_status) memcpy(row_status, hs, (size_t)n_rows * 4);
      if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rows = n_rows;
        cudaEventElapsedTime(&stats->h2d_ms, p->ev[0], p->ev[1]);
        cudaEventElapsedTime(&stats->kernel_ms, p->ev[1], p->ev[2]);  // includes the PCIe writes of the results
        stats->kernels = p->kernels_per_batch;
        stats->nonfinite_rows = bad;
      }
      return B2S_OK;
    }
    CUDA_TRY(cudaEventRecord(p->ev[0], st));
    CUDA_TRY(cudaMemcpyAsync(p->d_stage_in, src, (size_t)n_rows * row_bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(p->ev[1], st));
    if (int rc = launch_on(p, p->d_stage_in, n_rows, row_bytes, p->d_stage_out, p->d_stage_status, st)) return rc;
    CUDA_TRY(cudaEventRecord(p->ev[2], st));
    CUDA_TRY(cudaMemcpyAsync(p->h_stage_out, p->d_stage_out, out_sz, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(p->h_stage_out + out_sz, p->d_stage_status, (size_t)n_rows * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(p->ev[3], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memcpy(out, p->h_stage_out, out_sz);
    const int32_t* hs = (const int32_t*)(p->h_stage_out + out_sz);
    int bad = 0;
    for (int64_t r = 0; r < n_rows; ++r) bad += (hs[r] & B2S_ROW_NONFINITE_INPUT) ? 1 : 0;
    if (row_status) memcpy(row_status, hs, (size_t)n_rows * 4);
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->rows = n_rows;
      cudaEventElapsedTime(&stats->h2d_ms, p->ev[0], p->ev[1]);
      cudaEventElapsedTime(&stats->kernel_ms, p->ev[1], p->ev[2]);
      cudaEventElapsedTime(&stats->d2h_ms, p->ev[2], p->ev[3]);
      stats->kernels = p->kernels_per_batch;
      stats->nonfinite_rows = bad;
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_time_device(b2s_plan_t p, const void* const* d_rows, int32_t n_bufs, int64_t n_rows,
                               int64_t row_stride_bytes, void* d_out, int32_t n_iters, float* total_ms) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (n_bufs < 1 || n_iters < 1 || !total_ms) return fail(B2S_ERR_INVALID, "bad arguments");
    cudaStream_t st = G.stream;
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaEventRecord(p->ev[0], st));
    for (int i = 0; i < n_iters; ++i)
      if (int rc = launch_on(p, d_rows[i % n_bufs], n_rows, row_stride_bytes, d_out, nullptr, st)) return rc;
    CUDA_TRY(cudaEventRecord(p->ev[1], st));
    CUDA_TRY(cudaEventSynchronize(p->ev[1]));
    CUDA_TRY(cudaEventElapsedTime(total_ms, p->ev[0], p->ev[1]));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ coalescing ring
// One coalesced batch on the ring's stream: pinned slot -> (H2D) -> kernels -> (D2H) -> pinned slot, then the host waits for it.
// Runs WITHOUT the plan's lock, either on the dispatcher thread or on a caller blocked in b2s_wait (see there); `dispatch_busy`
// keeps it to one batch at a time.
struct BatchResult {
  b2s_stats stats{};
  int err = 0;
  std::string err_msg;
};

constexpr int kRingGraceUs = 50;

static BatchResult ring_run_batch(b2s_plan_s* p, Slot& s) {
  BatchResult res;
  const int64_t rows = s.rows;
  const float queue_us =
      std::chrono::duration<float, std::micro>(std::chrono::steady_clock::now() - s.first_submit).count();
  cudaStream_t st = p->ring_stream;
  const int64_t row_bytes = (int64_t)p->n_in * 4;
  const size_t out_sz = (size_t)rows * p->out_cols * 4;
  // every step is checked: a batch whose copy or launch failed is reported to all of its tickets (b2s_wait returns
  // the error and copies nothing) instead of handing out whatever an earlier batch left in the pinned slot
  int& err = res.err;
  std::string& err_msg = res.err_msg;
  auto step = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess && !err) {
      err = B2S_ERR_CUDA;
      err_msg = std::string("coalesced batch: ") + what + ": " + cudaGetErrorString(e);
    }
  };
  static const int64_t zc_in_bytes = getenv("B2S_ZEROCOPY_IN_BYTES") ? atoll(getenv("B2S_ZEROCOPY_IN_BYTES")) : 65536;
  static const int zc_out = getenv("B2S_ZEROCOPY_OUT") ? atoi(getenv("B2S_ZEROCOPY_OUT")) : 1;
  const bool zero_out = zc_out && p->peers.empty() && !p->comm;  // results go straight into the slot's pinned result area
  const bool zero_in = zero_out && rows * row_bytes <= zc_in_bytes;  // a tiny batch is read from the pinned slot as well
  step(cudaEventRecord(s.e0, st), "event record");
  if (!zero_in) step(cudaMemcpyAsync(s.d_in, s.h_in, (size_t)rows * row_bytes, cudaMemcpyHostToDevice, st), "H2D copy");
  step(cudaEventRecord(s.e1, st), "event record");
  if (!err) {
    int32_t* h_status = (int32_t*)(s.h_out + (size_t)p->ring_cap * p->out_cols * 4);
    const int rc = zero_out ? launch_on(p, zero_in ? s.h_in : s.d_in, rows, row_bytes, s.h_out, h_status, st, zero_in)
                            : launch_on(p, s.d_in, rows, row_bytes, s.d_out, s.d_status, st);
    if (rc) {
      err = rc;
      err_msg = std::string("coalesced batch: ") + g_err;
    }
  }
  step(cudaEventRecord(s.e2, st), "event record");
  if (!err && !zero_out) {
    step(cudaMemcpyAsync(s.h_out, s.d_out, out_sz, cudaMemcpyDeviceToHost, st), "D2H copy");
    step(cudaMemcpyAsync(s.h_out + (size_t)p->ring_cap * p->out_cols * 4, s.d_status, (size_t)rows * 4, cudaMemcpyDeviceToHost, st), "D2H copy");
  }
  step(cudaEventRecord(s.e3, st), "event record");
  step(cudaEventSynchronize(s.e3), "execution");
  b2s_stats& stt = res.stats;
  stt.rows = rows;
  if (!err) {
    cudaEventElapsedTime(&stt.h2d_ms, s.e0, s.e1);
    cudaEventElapsedTime(&stt.kernel_ms, s.e1, s.e2);
    cudaEventElapsedTime(&stt.d2h_ms, s.e2, s.e3);
  } else {
    cudaGetLastError();  // the error is reported through the tickets
  }
  stt.queue_us = queue_us;
  stt.kernels = p->kernels_per_batch;
  return res;
}

// with the lock held: publish the batch to its tickets and pass the stream on
static void ring_finish_batch(b2s_plan_s* p, Slot& s, const BatchResult& res) {
  s.stats = res.stats;
  s.err = res.err;
  s.err_msg = res.err_msg;
  s.state = 3;
  p->dispatch_busy = false;
  if (s.done_cv) s.done_cv->notify_all();
  // the batch that collected rows meanwhile: one of the callers blocked on it runs it (b2s_wait); the dispatcher thread
  // covers batches nobody is blocked on
  if (p->open_slot >= 0 && p->slots[p->open_slot].wanted && p->slots[p->open_slot].done_cv) p->slots[p->open_slot].done_cv->notify_one();
  p->cv_work.notify_one();
}

static void dispatcher_main(b2s_plan_s* p) {
  cudaSetDevice(G.device);
  std::unique_lock<std::mutex> lk(p->mu);
  for (;;) {
    // wake up when a batch is sealed, when the open batch is due, or on stop
    if (p->dispatch_busy) {  // a caller blocked in b2s_wait is running a batch on the ring's stream
      if (p->stop) return;
      p->cv_work.wait(lk);
      continue;
    }
    if (p->sealed.empty()) {
      if (p->stop) return;
      if (p->open_slot >= 0 && p->slots[p->open_slot].rows > 0) {
        // The open batch leaves when its oldest row has waited max_wait_us (0: at once -- this thread is free, so batches
        // form while the previous one runs) -- but only while another slot is free to take the submits that follow: the
        // last free slot keeps collecting rows (until it is full, a caller blocks on it, or b2s_flush), so that a caller
        // that submits many tickets before it collects any fills a batch instead of exhausting the ring.
        int spare = p->slots[p->open_slot].wanted ? 1 : 0;  // a caller blocked on this batch: holding it back gains nothing
        for (int i = 0; i < (int)p->slots.size(); ++i)
          spare += (i != p->open_slot && p->slots[i].state == 0 && p->slots[i].rows == 0 && p->slots[i].waiters == 0) ? 1 : 0;
        if (spare == 0) {
          p->cv_work.wait(lk);  // a slot is collected, the batch fills up, a waiter or a flush seals it
          continue;
        }
        // max_wait_us = 0: a caller that blocks on the batch runs it itself (b2s_wait); this thread takes what nobody has
        // claimed after a short grace period (callers that submit now and collect later)
        const auto hold = std::chrono::microseconds(p->wait_us() > 0 ? p->wait_us() : kRingGraceUs);
        auto deadline = p->slots[p->open_slot].first_submit + hold;
        if (std::chrono::steady_clock::now() >= deadline || p->cv_work.wait_until(lk, deadline) == std::cv_status::timeout) {
          if (!p->dispatch_busy && p->sealed.empty() && p->open_slot >= 0 && p->slots[p->open_slot].rows > 0 &&
              std::chrono::steady_clock::now() >= p->slots[p->open_slot].first_submit + hold) {
            p->slots[p->open_slot].state = 1;
            p->sealed.push_back(p->open_slot);
            p->open_slot = -1;
          }
        }
      } else {
        p->cv_work.wait(lk);  // nothing to run (blocked callers run their own batches: no reason to poll here)
      }
      continue;
    }
    const int si = p->sealed.front();
    p->sealed.pop_front();
    Slot& s = p->slots[si];
    s.state = 2;
    p->dispatch_busy = true;
    lk.unlock();
    BatchResult res = ring_run_batch(p, s);
    lk.lock();
    ring_finish_batch(p, s, res);
  }
}

static void ring_free_slot(Slot& s) {
  if (s.h_in) cudaFreeHost(s.h_in);
  if (s.h_out) cudaFreeHost(s.h_out);
  if (s.d_in) cudaFree(s.d_in);
  if (s.d_out) cudaFree(s.d_out);
  if (s.d_status) cudaFree(s.d_status);
  for (cudaEvent_t e : {s.e0, s.e1, s.e2, s.e3})
    if (e) cudaEventDestroy(e);
  s = Slot{};
}

static int ring_start(b2s_plan_s* p) {
  if (!p->slots.empty()) return B2S_OK;
  CUDA_TRY(cudaSetDevice(G.device));
  // built aside and committed only when everything (buffers, events, stream, dispatcher) exists: a failure leaves the
  // plan without a ring, so the next submit retries instead of queueing rows nobody will ever dispatch
  const int64_t cap = p->ring_cfg_max_batch > 0 ? p->ring_cfg_max_batch : G.max_batch;
  const int n_slots = p->ring_cfg_slots > 0 ? p->ring_cfg_slots : G.ring_slots;
  std::vector<Slot> slots(n_slots);
  cudaStream_t stream = nullptr;
  const int64_t row_bytes = (int64_t)p->n_in * 4;
  cudaError_t e = cudaSuccess;
  auto ok = [&](cudaError_t r) { return e == cudaSuccess && (e = r) == cudaSuccess; };
  for (auto& s : slots) {
    s.done_cv = std::make_shared<std::condition_variable>();
    if (!(ok(cudaMallocHost(&s.h_in, (size_t)cap * row_bytes)) && ok(cudaMallocHost(&s.h_out, (size_t)cap * (p->out_cols + 1) * 4)) &&
          ok(cudaMalloc(&s.d_in, (size_t)cap * row_bytes)) && ok(cudaMalloc(&s.d_out, (size_t)cap * p->out_cols * 4)) &&
          ok(cudaMalloc(&s.d_status, (size_t)cap * 4)) && ok(cudaEventCreate(&s.e0)) && ok(cudaEventCreate(&s.e1)) &&
          ok(cudaEventCreate(&s.e2)) && ok(cudaEventCreate(&s.e3))))
      break;
  }
  if (e == cudaSuccess) ok(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  if (e != cudaSuccess) {
    for (auto& s : slots) ring_free_slot(s);
    cudaGetLastError();
    return fail(B2S_ERR_CUDA, "coalescing ring of %d x %lld rows: %s", n_slots, (long long)cap, cudaGetErrorString(e));
  }
  p->ring_cap = cap;
  p->slots = std::move(slots);
  p->ring_stream = stream;
  p->stop = false;
  try {
    p->dispatcher = std::thread(dispatcher_main, p);
  } catch (const std::exception& ex) {
    for (auto& s : p->slots) ring_free_slot(s);
    p->slots.clear();
    cudaStreamDestroy(p->ring_stream);
    p->ring_stream = nullptr;
    return fail(B2S_ERR_STATE, "coalescing ring: cannot start the dispatcher thread: %s", ex.what());
  }
  return B2S_OK;
}

// ticket = batch_id << 24 | row offset inside the batch (max_batch <= 2^24 rows)
extern "C" int b2s_submit(b2s_plan_t p, const void* rows, int64_t n_rows, int64_t row_stride_bytes, uint64_t* ticket) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    const int64_t row_bytes = (int64_t)p->n_in * 4;
    if (n_rows <= 0 || row_stride_bytes < row_bytes || !ticket) return fail(B2S_ERR_INVALID, "bad submit arguments");
    std::unique_lock<std::mutex> lk(p->mu);
    if (int rc = ring_start(p)) return rc;
    if (n_rows > p->ring_cap || p->ring_cap > (1 << 24)) return fail(B2S_ERR_INVALID, "submit of %lld rows exceeds max_batch %lld", (long long)n_rows, (long long)p->ring_cap);
    for (;;) {
      if (p->open_slot >= 0 && p->slots[p->open_slot].rows + n_rows > p->ring_cap) {
        p->slots[p->open_slot].state = 1;
        p->sealed.push_back(p->open_slot);
        p->open_slot = -1;
        p->cv_work.notify_one();
      }
      if (p->open_slot < 0) {
        for (int i = 0; i < (int)p->slots.size(); ++i)
          if (p->slots[i].state == 0 && p->slots[i].rows == 0 && p->slots[i].waiters == 0) {
            p->open_slot = i;
            p->slots[i].batch_id = p->next_batch++;
            p->batch_slot[p->slots[i].batch_id] = i;
            break;
          }
        if (p->open_slot < 0) {
          p->cv_free.wait(lk);  // every slot is in flight or waiting to be collected
          continue;
        }
      }
      break;
    }
    Slot& s = p->slots[p->open_slot];
    if (s.rows == 0) s.first_submit = std::chrono::steady_clock::now();
    const int64_t off = s.rows;
    pack_rows(s.h_in + off * row_bytes, rows, n_rows, row_stride_bytes, row_bytes);
    s.rows += n_rows;
    s.waiters += 1;
    *ticket = (s.batch_id << 24) | (uint64_t)off;
    if (s.rows >= p->ring_cap) {
      s.state = 1;
      p->sealed.push_back(p->open_slot);
      p->open_slot = -1;
    }
    p->cv_work.notify_one();
    // remember how many rows this ticket covers (low 24 bits hold the offset; the count travels in a side map)
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_flush(b2s_plan_t p) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    std::unique_lock<std::mutex> lk(p->mu);
    if (p->open_slot >= 0 && p->slots[p->open_slot].rows > 0) {
      p->slots[p->open_slot].state = 1;
      p->sealed.push_back(p->open_slot);
      p->open_slot = -1;
      p->cv_work.notify_one();
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_set_ring(b2s_plan_t p, int32_t ring_slots, int64_t max_batch, int32_t max_wait_us) {
  try {  // no C++ exception crosses the C boundary
    if (!p) return fail(B2S_ERR_INVALID, "null plan");
    std::unique_lock<std::mutex> lk(p->mu);
    if (!p->slots.empty()) return fail(B2S_ERR_STATE, "the coalescing ring of this plan is already running");
    if (ring_slots < 0 || ring_slots > 64 || max_batch < 0 || max_batch > (1 << 24) || max_wait_us > 10000000)
      return fail(B2S_ERR_INVALID, "ring configuration out of range");
    p->ring_cfg_slots = ring_slots;
    p->ring_cfg_max_batch = max_batch;
    p->ring_cfg_wait_us = max_wait_us;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_wait(b2s_plan_t p, uint64_t ticket, void* out, int64_t out_bytes, int32_t* row_status, b2s_stats* stats) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    const uint64_t batch = ticket >> 24;
    const int64_t off = (int64_t)(ticket & ((1u << 24) - 1));
    const int64_t n_rows = out_bytes / ((int64_t)p->out_cols * 4);
    std::unique_lock<std::mutex> lk(p->mu);
    auto it = p->batch_slot.find(batch);
    if (it == p->batch_slot.end()) return fail(B2S_ERR_INVALID, "unknown ticket");
    Slot& s = p->slots[it->second];
    // Who runs the batch?  With max_wait_us = 0 the caller that blocks on it does, right here, as soon as the ring's stream is
    // free (no hand-off to another thread and back: that costs more than a small batch takes on the device, and under many
    // request threads the dispatcher thread would queue for a core behind them).  While a batch is in flight the rows of other
    // callers keep joining the open one (that is what coalesces concurrent request threads); whoever finishes a batch wakes one
    // caller of the next.  The dispatcher thread covers sealed batches and batches nobody is blocked on.
    const int idx = it->second;
    auto done = [&] { return s.state == 3 && s.batch_id == batch; };
    auto claim = [&] {  // with the lock held: may this thread run the ticket's batch now?
      if (p->dispatch_busy || p->stop) return false;
      if (s.state == 0 && p->open_slot == idx && s.rows > 0 && p->sealed.empty() && p->wait_us() == 0) {
        p->open_slot = -1;
        return true;
      }
      if (s.state == 1 && !p->sealed.empty() && p->sealed.front() == idx) {
        p->sealed.pop_front();
        return true;
      }
      return false;
    };
    bool spun = false;
    while (!done()) {
      if (claim()) {
        s.state = 2;
        p->dispatch_busy = true;
        lk.unlock();
        cudaSetDevice(G.device);
        BatchResult res = ring_run_batch(p, s);
        lk.lock();
        ring_finish_batch(p, s, res);
        continue;
      }
      if (s.state == 0 && p->open_slot == idx && !s.wanted) {  // a caller is blocked on this batch: it must not be held back
        s.wanted = true;
        p->cv_work.notify_one();
      }
      // a short spin before sleeping (only a couple of callers at a time: a crowd of spinners would fight for the lock)
      if (!spun) {
        spun = true;
        if (p->spinners.fetch_add(1, std::memory_order_relaxed) < 2) {
          for (int spin = 0; spin < 400 && !done(); ++spin) {
            lk.unlock();
            for (int i = 0; i < 40; ++i) __builtin_ia32_pause();
            lk.lock();
            if (!p->dispatch_busy && (s.state == 0 || s.state == 1)) break;  // the stream is free: try to claim the batch
          }
        }
        p->spinners.fetch_sub(1, std::memory_order_relaxed);
        continue;
      }
      s.done_cv->wait(lk);  // woken when the batch is done, or to take the stream over
    }
    // the batch is done: whatever this call returns, the ticket is spent and the last one recycles the slot
    int rc = B2S_OK;
    if (s.err) {
      rc = fail(s.err, "%s", s.err_msg.c_str());
    } else if (off + n_rows > s.rows) {
      rc = fail(B2S_ERR_INVALID, "ticket range exceeds its batch");
    } else {
      // the slot cannot be recycled while this ticket is outstanding (waiters > 0): copy without the lock, so that the
      // tickets of a batch are collected side by side
      const b2s_stats batch_stats = s.stats;
      lk.unlock();
      memcpy(out, s.h_out + (size_t)off * p->out_cols * 4, (size_t)n_rows * p->out_cols * 4);
      const int32_t* hs = (const int32_t*)(s.h_out + (size_t)p->ring_cap * p->out_cols * 4) + off;
      if (row_status) memcpy(row_status, hs, (size_t)n_rows * 4);
      if (stats) {
        *stats = batch_stats;
        int bad = 0;
        for (int64_t r = 0; r < n_rows; ++r) bad += (hs[r] & B2S_ROW_NONFINITE_INPUT) ? 1 : 0;
        stats->nonfinite_rows = bad;
      }
      lk.lock();
    }
    if (--s.waiters == 0) {  // last collector frees the slot
      p->batch_slot.erase(it);
      s.rows = 0;
      s.state = 0;
      s.wanted = false;
      s.err = 0;
      s.err_msg.clear();
      p->cv_free.notify_all();
      p->cv_work.notify_one();  // the dispatcher may have been holding the open batch for want of a spare slot
    }
    return rc;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// Throughput / latency of the coalescing ring itself, driven by native producer threads (no Python in the loop): every
// thread emits `rows_per_submit` rows and awaits them, like a request thread of the reference emits one event and blocks
// in await_result (serving/states.py:1283-1287), for `seconds`.
extern "C" int b2s_ring_bench(b2s_plan_t p, const void* rows, int64_t n_src_rows, int64_t row_stride_bytes, int32_t n_threads,
                              int32_t rows_per_submit, double seconds, int64_t* events, double* p50_us, double* p99_us) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (n_threads < 1 || n_threads > 1024 || rows_per_submit < 1 || rows_per_submit > n_src_rows || seconds <= 0 || !events)
      return fail(B2S_ERR_INVALID, "bad ring bench arguments");
    std::vector<std::thread> threads;
    std::vector<int64_t> done(n_threads, 0);
    std::vector<std::vector<float>> lat(n_threads);
    std::vector<int> rcs(n_threads, 0);
    std::vector<std::string> msgs(n_threads);
    const auto t_end = std::chrono::steady_clock::now() + std::chrono::duration_cast<std::chrono::steady_clock::duration>(
                                                               std::chrono::duration<double>(seconds));
    const size_t out_bytes = (size_t)rows_per_submit * p->out_cols * 4;
    for (int t = 0; t < n_threads; ++t) {
      threads.emplace_back([&, t] {
        std::vector<char> out(out_bytes);
        std::vector<int32_t> status(rows_per_submit);
        int64_t off = ((int64_t)t * 7919) % (n_src_rows - rows_per_submit + 1);
        while (std::chrono::steady_clock::now() < t_end) {
          const auto t0 = std::chrono::steady_clock::now();
          uint64_t ticket = 0;
          int rc = b2s_submit(p, (const char*)rows + off * row_stride_bytes, rows_per_submit, row_stride_bytes, &ticket);
          if (!rc) rc = b2s_wait(p, ticket, out.data(), (int64_t)out_bytes, status.data(), nullptr);
          if (rc) {
            rcs[t] = rc;
            msgs[t] = g_err;
            return;
          }
          if (lat[t].size() < (1u << 20))
            lat[t].push_back(std::chrono::duration<float, std::micro>(std::chrono::steady_clock::now() - t0).count());
          done[t] += rows_per_submit;
          off = (off + rows_per_submit * 13) % (n_src_rows - rows_per_submit + 1);
        }
      });
    }
    for (auto& th : threads) th.join();
    for (int t = 0; t < n_threads; ++t)
      if (rcs[t]) return fail(rcs[t], "ring bench producer %d: %s", t, msgs[t].c_str());
    int64_t total = 0;
    std::vector<float> all;
    for (int t = 0; t < n_threads; ++t) {
      total += done[t];
      all.insert(all.end(), lat[t].begin(), lat[t].end());
    }
    *events = total;
    std::sort(all.begin(), all.end());
    if (p50_us) *p50_us = all.empty() ? 0.0 : all[all.size() / 2];
    if (p99_us) *p99_us = all.empty() ? 0.0 : all[(size_t)((all.size() - 1) * 0.99)];
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_destroy(b2s_plan_t p) {
  try {  // no C++ exception crosses the C boundary
    if (!p) return B2S_OK;
    if (p->dispatcher.joinable()) {
      {
        std::lock_guard<std::mutex> lk(p->mu);
        p->stop = true;
        p->cv_work.notify_all();
      }
      p->dispatcher.join();
    }
    for (auto& s : p->slots) ring_free_slot(s);
    if (p->ring_stream) cudaStreamDestroy(p->ring_stream);
    if (p->h_stage_in) cudaFreeHost(p->h_stage_in);
    if (p->h_stage_out) cudaFreeHost(p->h_stage_out);
    if (p->d_stage_in) cudaFree(p->d_stage_in);
    if (p->d_stage_out) cudaFree(p->d_stage_out);
    if (p->d_stage_status) cudaFree(p->d_stage_status);
    for (int i = 0; i < 4; ++i)
      if (p->ev[i]) cudaEventDestroy(p->ev[i]);
    for (cudaEvent_t e : p->chunk_ev) cudaEventDestroy(e);
    if (p->d_blob) cudaFree(p->d_blob);
    if (p->d_t3_blob) cudaFree(p->d_t3_blob);
    for (auto& kv : p->t3_scratch)
      if (kv.second.pred) { cudaFree(kv.second.pred); cudaFree(kv.second.row_bad); if (kv.second.xt) cudaFree(kv.second.xt); }
    delete p;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ multi-GPU merge
extern "C" int b2s_plan_set_merge_targets(b2s_plan_t p, void* const* peer_out, int32_t n_peers, int64_t row_offset) {
  try {  // no C++ exception crosses the C boundary
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (n_peers < 0 || n_peers > 8 || row_offset < 0) return fail(B2S_ERR_INVALID, "bad merge targets");
    if (p->mode == MODE_STORE && n_peers > 0) return fail(B2S_ERR_UNSUPPORTED, "transform-only plans have no vote to merge");
    p->peers.assign(peer_out, peer_out + n_peers);
    p->peer_off = row_offset;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_ipc_export(void* dptr, void* handle64) {
  try {  // no C++ exception crosses the C boundary
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CUDA_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), dptr));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_ipc_open(const void* handle64, void** dptr_out) {
  try {  // no C++ exception crosses the C boundary
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    CUDA_TRY(cudaIpcOpenMemHandle(dptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_ipc_close(void* dptr) {
  try {  // no C++ exception crosses the C boundary
    CUDA_TRY(cudaIpcCloseMemHandle(dptr));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ ensemble-merge communicator
__global__ void merge_wait_kernel(const uint32_t* flags, int n, uint32_t epoch, uint32_t* timeout_flag, long long max_ns) {
  // one lane per source rank: acquire its flag until it shows `epoch` (or later)
  if ((int)threadIdx.x < n) {
    long long t0 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
      if ((int32_t)(v - epoch) >= 0) break;
      long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > max_ns) {  // a peer died: give up instead of hanging the GPU; the host reports it
        atomicExch(timeout_flag, 1u + threadIdx.x);
        break;
      }
      __nanosleep(200);
    }
  }
}

extern "C" int b2s_comm_create(int32_t rank, int32_t world, int64_t max_rows_per_rank, int32_t out_cols, b2s_comm_t* out) {
  try {  // no C++ exception crosses the C boundary
    if (!G.inited) return fail(B2S_ERR_STATE, "b2s_init was not called");
    if (!out || world < 1 || world > 8 || rank < 0 || rank >= world || max_rows_per_rank < 1 || out_cols < 1)
      return fail(B2S_ERR_INVALID, "bad communicator arguments (at most 8 ranks)");
    std::unique_ptr<b2s_comm_s> c(new b2s_comm_s);
    c->rank = rank;
    c->world = world;
    c->out_cols = out_cols;
    c->max_rows = (max_rows_per_rank + 3) / 4 * 4;  // row blocks start 16-byte aligned
    c->bytes = kCommHeader + kCommSlots * c->buf_bytes();
    CUDA_TRY(cudaSetDevice(G.device));
    CUDA_TRY(cudaMalloc(&c->base, c->bytes));
    CUDA_TRY(cudaMemset(c->base, 0, 512 < c->bytes ? 512 : c->bytes));
    c->peer_base.assign(world, nullptr);
    c->peer_base[rank] = c->base;
    if (world == 1) c->connected = true;
    *out = c.release();
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_comm_handle(b2s_comm_t c, void* handle64) {
  try {
    if (!c || !handle64) return fail(B2S_ERR_INVALID, "null communicator");
    CUDA_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), c->base));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_comm_connect(b2s_comm_t c, const void* all_handles) {
  try {
    if (!c || !all_handles) return fail(B2S_ERR_INVALID, "null communicator");
    if (c->connected) return B2S_OK;
    for (int r = 0; r < c->world; ++r) {
      if (r == c->rank) continue;
      cudaIpcMemHandle_t h;
      memcpy(&h, (const char*)all_handles + (size_t)r * 64, 64);
      void* ptr = nullptr;
      CUDA_TRY(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer_base[r] = (char*)ptr;
    }
    c->connected = true;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_plan_attach_comm(b2s_plan_t p, b2s_comm_t c) {
  try {
    if (!p || !p->finalized) return fail(B2S_ERR_STATE, "plan not finalized");
    if (c) {
      if (!c->connected) return fail(B2S_ERR_STATE, "communicator is not connected");
      if (c->out_cols != p->out_cols) return fail(B2S_ERR_INVALID, "communicator rows have %d words, the plan writes %d", c->out_cols, p->out_cols);
      if (p->mode == MODE_STORE) return fail(B2S_ERR_UNSUPPORTED, "transform-only plans have no vote to merge");
    }
    p->comm = c;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int comm_wait_epoch(b2s_comm_t c, void* stream, uint32_t e, const void** d_merged, uint32_t* epoch_out);

extern "C" int b2s_comm_wait(b2s_comm_t c, void* stream, const void** d_merged, uint32_t* epoch_out) {
  try {
    if (!c || !c->connected) return fail(B2S_ERR_STATE, "communicator is not connected");
    if (c->epoch == 0) return fail(B2S_ERR_STATE, "no step has been launched on this communicator");
    return comm_wait_epoch(c, stream, c->epoch, d_merged, epoch_out);
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// Pipelined steps: wait for the step launched `lag` launches ago (lag 0 = b2s_comm_wait, lag 1 = the previous step, so that
// the peers' stores and flags of step e travel while step e + 1 is being scored).  When fewer than lag + 1 steps have been
// launched there is nothing to wait for: *d_merged = NULL, *epoch_out = 0.
extern "C" int b2s_comm_wait_lag(b2s_comm_t c, void* stream, int32_t lag, const void** d_merged, uint32_t* epoch_out) {
  try {
    if (!c || !c->connected) return fail(B2S_ERR_STATE, "communicator is not connected");
    if (lag < 0 || lag > 1) return fail(B2S_ERR_INVALID, "lag must be 0 or 1 (four response slots)");
    if (c->epoch <= (uint32_t)lag) {
      if (d_merged) *d_merged = nullptr;
      if (epoch_out) *epoch_out = 0;
      return B2S_OK;
    }
    return comm_wait_epoch(c, stream, c->epoch - (uint32_t)lag, d_merged, epoch_out);
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int comm_wait_epoch(b2s_comm_t c, void* stream, uint32_t e, const void** d_merged, uint32_t* epoch_out) {
  {
    cudaStream_t st = stream ? (cudaStream_t)stream : G.stream;
    if (c->fused_epoch && (int32_t)(c->fused_epoch - e) >= 0) {  // the last launch's own last CTA waits for this step already
      if (d_merged) *d_merged = c->buf(c->rank, e);
      if (epoch_out) *epoch_out = e;
      return B2S_OK;
    }
    uint32_t* timeout_flag = reinterpret_cast<uint32_t*>(c->base) + 65;
    // how long a rank may lag behind before the step is declared dead (B2S_COMM_TIMEOUT_MS, default 10 s)
    static const long long timeout_ns = (getenv("B2S_COMM_TIMEOUT_MS") ? atoll(getenv("B2S_COMM_TIMEOUT_MS")) : 10000ll) * 1000000ll;
    // A one-warp polling kernel.  The cheap form is the fused wait (b2s_comm_set_fused_wait), which launches nothing.
    merge_wait_kernel<<<1, 32, 0, st>>>(c->flags(c->rank), c->world, e, timeout_flag, timeout_ns);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(B2S_ERR_CUDA, "merge wait launch failed: %s", cudaGetErrorString(err));
    G.launches.fetch_add(1, std::memory_order_relaxed);
    if (d_merged) *d_merged = c->buf(c->rank, e);
    if (epoch_out) *epoch_out = e;
    return B2S_OK;
  }
}

// Fused wait: lag = 0 / 1 makes every launch of an attached plan end by waiting (in its last CTA) for the flags of its own
// step / of the previous step; b2s_comm_wait / b2s_comm_wait_lag then launch nothing for steps that are covered.  lag = -1: off.
extern "C" int b2s_comm_set_fused_wait(b2s_comm_t c, int32_t lag) {
  try {
    if (!c) return fail(B2S_ERR_INVALID, "null communicator");
    if (lag < -1 || lag > 1) return fail(B2S_ERR_INVALID, "fused wait lag must be -1 (off), 0 or 1");
    c->fused_lag = lag;
    c->fused_epoch = 0;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_comm_check(b2s_comm_t c) {
  try {  // after a stream synchronisation: did a wait give up on a peer?
    if (!c) return fail(B2S_ERR_INVALID, "null communicator");
    uint32_t v = 0;
    CUDA_TRY(cudaMemcpy(&v, reinterpret_cast<uint32_t*>(c->base) + 65, 4, cudaMemcpyDeviceToHost));
    if (v) return fail(B2S_ERR_TIMEOUT, "ensemble-merge: rank %u did not signal its shard in time (B2S_COMM_TIMEOUT_MS)", v - 1);
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_comm_destroy(b2s_comm_t c) {
  try {
    if (!c) return B2S_OK;
    for (int r = 0; r < c->world; ++r)
      if (r != c->rank && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
    if (c->base) cudaFree(c->base);
    delete c;
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

// ------------------------------------------------------------------------------------------ memory helpers
extern "C" void* b2s_alloc_pinned(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) {
    fail(B2S_ERR_CUDA, "cudaMallocHost(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}
extern "C" int b2s_free_pinned(void* p) {
  try {  // no C++ exception crosses the C boundary
    CUDA_TRY(cudaFreeHost(p));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" void* b2s_device_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    fail(B2S_ERR_CUDA, "cudaMalloc(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}
extern "C" int b2s_device_free(void* p) {
  try {  // no C++ exception crosses the C boundary
    CUDA_TRY(cudaFree(p));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_memcpy_h2d(void* d, const void* h, size_t bytes) {
  try {  // no C++ exception crosses the C boundary
    // on the library stream and awaited: cudaMemcpy from pageable memory may return while the DMA is still in flight, and the
    // (non-blocking) library stream that launches the kernels is not ordered behind the legacy stream -- a kernel launched
    // right after the call read the tail of the previous batch (found by the 2-GPU test of ShardedGraphServer, r2n)
    cudaStream_t st = G.inited ? G.stream : (cudaStream_t)0;
    CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_memcpy_d2h(void* h, const void* d, size_t bytes) {
  try {  // no C++ exception crosses the C boundary
    cudaStream_t st = G.inited ? G.stream : (cudaStream_t)0;  // ordered behind the kernels of the library stream
    CUDA_TRY(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
extern "C" int b2s_device_sync(void) {
  try {  // no C++ exception crosses the C boundary
    CUDA_TRY(cudaDeviceSynchronize());
    return B2S_OK;
  } catch (const std::exception& e) {
    return fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
