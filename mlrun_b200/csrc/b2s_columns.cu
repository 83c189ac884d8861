// b2s_columns.cu -- C-ABI of the columnar feature-set transform plan (see include/b200serve.h, "columnar ingest").
#include <cuda_runtime.h>

#include <exception>

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/b200serve.h"
#include "b2s_columns.cuh"
#include "b2s_internal.h"

using namespace b2s;

#define COL_TRY(expr)                                                                                       \
  do {                                                                                                      \
    cudaError_t _e = (expr);                                                                                \
    if (_e != cudaSuccess)                                                                                  \
      return b2s_int_fail(B2S_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct b2s_cols_s {
  int32_t n_in = 0;
  bool finalized = false;
  std::vector<ColOp> ops;
  std::vector<double> tab;
  std::vector<uint8_t> out_words;  // per output slot: 1, or 2 for the first slot of an 8-byte column (its second slot holds 0)
  std::vector<uint8_t> in_used;    // per input slot: 0 unused, 1 4-byte, 2 first slot of an 8-byte column
  int32_t n_counters = 0;
  // device
  ColOp* d_ops = nullptr;
  double* d_tab = nullptr;
  int grid = 0;
  // host-call staging
  std::mutex mu;
  char *d_in = nullptr, *d_out = nullptr;
  unsigned long long* d_cnt = nullptr;
  int64_t cap_rows = 0;
  int64_t res_rows = 0, res_stride = 0;  // what d_out holds after the last host run (b2s_cols_stats_begin reads it there)
  unsigned long long res_gen = 0;        // host runs so far (the statistics calls check that the result is still theirs)
  ColStatsWS* stats_ws = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> chunk_ev;  // one per row range of a pipelined host run
};

static int check_src(b2s_cols_t c, int32_t src, int32_t kind) {
  if (!c) return b2s_int_fail(B2S_ERR_INVALID, "null plan");
  if (c->finalized) return b2s_int_fail(B2S_ERR_STATE, "plan already finalized");
  const int words = kind == B2S_COL_I64 ? 2 : 1;
  if (src < 0 || src + words > c->n_in) return b2s_int_fail(B2S_ERR_INVALID, "input slot %d out of range", src);
  if (kind != B2S_COL_F32 && kind != B2S_COL_I32 && kind != B2S_COL_I64) return b2s_int_fail(B2S_ERR_INVALID, "bad column kind %d", kind);
  c->in_used[src] = (uint8_t)words;
  return B2S_OK;
}

static int32_t new_out(b2s_cols_t c, int words) {
  const int32_t s = (int32_t)c->out_words.size();
  c->out_words.push_back((uint8_t)words);
  if (words == 2) c->out_words.push_back(0);
  return s;
}

static void set_check(b2s_cols_t c, ColOp& op, int32_t check, double cmin, double cmax, int32_t* counter) {
  op.check = check & 3;
  op.cmin = cmin;
  op.cmax = cmax;
  op.counter = -1;
  if (op.check) op.counter = c->n_counters++;
  if (counter) *counter = op.counter;
}

extern "C" int b2s_cols_create(int32_t n_in_slots, b2s_cols_t* out) {
  try {  // no C++ exception crosses the C boundary
    if (!out || n_in_slots <= 0 || n_in_slots > 65536) return b2s_int_fail(B2S_ERR_INVALID, "bad n_in_slots");
    auto* c = new b2s_cols_s();
    c->n_in = n_in_slots;
    c->in_used.assign(n_in_slots, 0);
    *out = c;
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_add_copy(b2s_cols_t c, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, int32_t keep,
                                 int32_t check, double cmin, double cmax, int32_t* out_slot, int32_t* check_counter) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_src(c, src_slot, kind)) return rc;
    if (kind == B2S_COL_I64 && (check || has_fill)) return b2s_int_fail(B2S_ERR_UNSUPPORTED, "8-byte columns are copied verbatim");
    if (!keep && !(check & 3)) return b2s_int_fail(B2S_ERR_INVALID, "a dropped column without a check is no op at all");
    ColOp op{};
    op.src = src_slot;
    op.src_int = kind == B2S_COL_I32;
    op.has_fill = (kind == B2S_COL_F32 && has_fill) ? 1 : 0;
    op.fill = fill;
    op.miss = -1;
    set_check(c, op, check, cmin, cmax, check_counter);
    if (!keep) {
      op.kind = CK_CHECK;
      op.dst = -1;
    } else if (kind == B2S_COL_I64) {
      op.kind = CK_COPY64;
      op.dst = new_out(c, 2);
    } else {
      op.kind = (kind == B2S_COL_F32 && (op.has_fill || op.check)) ? CK_F32 : CK_COPY32;
      op.dst = new_out(c, 1);
    }
    if (out_slot) *out_slot = op.dst;
    c->ops.push_back(op);
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int add_map(b2s_cols_t c, int kind_op, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* a,
                   const double* b, const double* v, int32_t n, int32_t check, double cmin, double cmax, int32_t* out_slot,
                   int32_t* miss_counter, int32_t* check_counter) {
  if (int rc = check_src(c, src_slot, kind)) return rc;
  if (kind == B2S_COL_I64) return b2s_int_fail(B2S_ERR_UNSUPPORTED, "maps take 4-byte columns");
  if (n <= 0 || n > 4096 || !a || !v || (kind_op == CK_RANGE && !b)) return b2s_int_fail(B2S_ERR_INVALID, "bad map table");
  ColOp op{};
  op.kind = kind_op;
  op.src = src_slot;
  op.src_int = kind == B2S_COL_I32;
  op.has_fill = (kind == B2S_COL_F32 && has_fill) ? 1 : 0;
  op.fill = fill;
  op.n = n;
  op.tab = (int32_t)c->tab.size();
  c->tab.insert(c->tab.end(), a, a + n);
  if (kind_op == CK_RANGE) c->tab.insert(c->tab.end(), b, b + n);
  c->tab.insert(c->tab.end(), v, v + n);
  op.miss = c->n_counters++;
  if (miss_counter) *miss_counter = op.miss;
  set_check(c, op, check, cmin, cmax, check_counter);
  op.dst = new_out(c, 1);
  if (out_slot) *out_slot = op.dst;
  c->ops.push_back(op);
  return B2S_OK;
}

extern "C" int b2s_cols_add_range_map(b2s_cols_t c, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* lo,
                                      const double* hi, const double* vals, int32_t n, int32_t check, double cmin, double cmax,
                                      int32_t* out_slot, int32_t* miss_counter, int32_t* check_counter) {
  try {  // no C++ exception crosses the C boundary
    return add_map(c, CK_RANGE, src_slot, kind, has_fill, fill, lo, hi, vals, n, check, cmin, cmax, out_slot, miss_counter, check_counter);
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_add_value_map(b2s_cols_t c, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* keys,
                                      const double* vals, int32_t n, int32_t check, double cmin, double cmax, int32_t* out_slot,
                                      int32_t* miss_counter, int32_t* check_counter) {
  try {  // no C++ exception crosses the C boundary
    return add_map(c, CK_VALUE, src_slot, kind, has_fill, fill, keys, nullptr, vals, n, check, cmin, cmax, out_slot, miss_counter, check_counter);
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_add_onehot(b2s_cols_t c, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* cats,
                                   int32_t n, int32_t* first_out_slot, int32_t* miss_counter) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_src(c, src_slot, kind)) return rc;
    if (kind == B2S_COL_I64) return b2s_int_fail(B2S_ERR_UNSUPPORTED, "one-hot takes 4-byte columns");
    if (n <= 0 || n > 4096 || !cats) return b2s_int_fail(B2S_ERR_INVALID, "bad category list");
    ColOp op{};
    op.kind = CK_ONEHOT;
    op.src = src_slot;
    op.src_int = kind == B2S_COL_I32;
    op.has_fill = (kind == B2S_COL_F32 && has_fill) ? 1 : 0;
    op.fill = fill;
    op.n = n;
    op.tab = (int32_t)c->tab.size();
    c->tab.insert(c->tab.end(), cats, cats + n);
    op.miss = c->n_counters++;
    op.counter = -1;
    if (miss_counter) *miss_counter = op.miss;
    op.dst = new_out(c, 1);
    for (int q = 1; q < n; ++q) new_out(c, 1);
    if (first_out_slot) *first_out_slot = op.dst;
    c->ops.push_back(op);
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_add_date_part(b2s_cols_t c, int32_t src_slot, int32_t part, int32_t* out_slot, int32_t* nat_counter) {
  try {  // no C++ exception crosses the C boundary
    if (int rc = check_src(c, src_slot, B2S_COL_I64)) return rc;
    if (part < 0 || part > DP_LAST) return b2s_int_fail(B2S_ERR_UNSUPPORTED, "date part %d is not computed on the device", part);
    ColOp op{};
    op.kind = CK_DATE;
    op.src = src_slot;
    op.part = part;
    op.miss = c->n_counters++;
    op.counter = -1;
    if (nat_counter) *nat_counter = op.miss;
    op.dst = new_out(c, 1);
    if (out_slot) *out_slot = op.dst;
    c->ops.push_back(op);
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_finalize(b2s_cols_t c) {
  try {  // no C++ exception crosses the C boundary
    if (!c) return b2s_int_fail(B2S_ERR_INVALID, "null plan");
    if (c->finalized) return B2S_OK;
    if (c->ops.empty()) return b2s_int_fail(B2S_ERR_INVALID, "plan has no column ops");
    if (!b2s_int_inited()) return b2s_int_fail(B2S_ERR_STATE, "b2s_init was not called (no CUDA device: there is no CPU fallback)");
    COL_TRY(cudaSetDevice(b2s_int_device()));
    COL_TRY(cudaMalloc(&c->d_ops, c->ops.size() * sizeof(ColOp)));
    COL_TRY(cudaMemcpy(c->d_ops, c->ops.data(), c->ops.size() * sizeof(ColOp), cudaMemcpyHostToDevice));
    COL_TRY(cudaMalloc(&c->d_tab, std::max<size_t>(c->tab.size(), 1) * sizeof(double)));
    if (!c->tab.empty()) COL_TRY(cudaMemcpy(c->d_tab, c->tab.data(), c->tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    COL_TRY(cudaMalloc(&c->d_cnt, std::max(c->n_counters, 1) * sizeof(unsigned long long)));
    int occ = 0;
    COL_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, columns_kernel, kColThreads, 0));
    c->grid = b2s_int_sm_count() * std::max(occ, 1);
    for (int i = 0; i < 4; ++i) COL_TRY(cudaEventCreate(&c->ev[i]));
    c->finalized = true;
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_info(b2s_cols_t c, int32_t* n_out_slots, int32_t* n_counters) {
  try {  // no C++ exception crosses the C boundary
    if (!c) return b2s_int_fail(B2S_ERR_INVALID, "null plan");
    if (n_out_slots) *n_out_slots = (int32_t)c->out_words.size();
    if (n_counters) *n_counters = c->n_counters;
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

static int launch_cols(b2s_cols_t c, const void* d_in, int64_t in_stride, int64_t n_rows, void* d_out, int64_t out_stride,
                       unsigned long long* d_counters, cudaStream_t st, int64_t row_begin = 0) {
  ColParams p{};
  p.row_begin = row_begin;
  p.in = (const char*)d_in;
  p.in_stride = in_stride;
  p.out = (char*)d_out;
  p.out_stride = out_stride;
  p.n_rows = n_rows;
  p.ops = c->d_ops;
  p.n_ops = (int32_t)c->ops.size();
  p.tab = c->d_tab;
  p.counters = d_counters;
  const int64_t items = ((n_rows + kColChunk - 1) / kColChunk) * p.n_ops;
  static const int grid_mode = getenv("B2S_COL_GRID") ? atoi(getenv("B2S_COL_GRID")) : 8;  // k x (SMs x resident CTAs); -1: one CTA per item.
  // Items differ in cost (a one-hot item writes n chunks) and a purely persistent grid with static striding leaves SMs idle
  // at the end: 8 waves of CTAs let the hardware scheduler balance them (measured: x1 0.270 ms, x8 0.245 ms, x64 0.268 ms)
  const int64_t want = grid_mode < 0 ? items : (int64_t)c->grid * std::max(grid_mode, 1);
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, items));
  b2s_int_count_launches(1);
  columns_kernel<<<grid, kColThreads, 0, st>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return b2s_int_fail(B2S_ERR_CUDA, "columns kernel launch failed: %s", cudaGetErrorString(e));
  return B2S_OK;
}

extern "C" int b2s_cols_run_device(b2s_cols_t c, const void* d_in, int64_t in_slot_stride, int64_t n_rows, void* d_out,
                                   int64_t out_slot_stride, uint64_t* d_counters, void* stream) {
  try {  // no C++ exception crosses the C boundary
    if (!c || !c->finalized) return b2s_int_fail(B2S_ERR_STATE, "plan not finalized");
    if (n_rows < 0 || in_slot_stride < n_rows * 4 || out_slot_stride < n_rows * 4 || (in_slot_stride & 7) || (out_slot_stride & 7))
      return b2s_int_fail(B2S_ERR_INVALID, "slot strides must hold n_rows words and be multiples of 8 bytes");
    if (n_rows == 0) return B2S_OK;
    if (c->n_counters && !d_counters) return b2s_int_fail(B2S_ERR_INVALID, "the plan has %d counters: pass a device array", c->n_counters);
    COL_TRY(cudaSetDevice(b2s_int_device()));
    return launch_cols(c, d_in, in_slot_stride, n_rows, d_out, out_slot_stride, (unsigned long long*)d_counters,
                       stream ? (cudaStream_t)stream : b2s_int_stream());
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_time_device(b2s_cols_t c, const void* const* d_in, int32_t n_bufs, int64_t in_slot_stride, int64_t n_rows,
                                    void* d_out, int64_t out_slot_stride, uint64_t* d_counters, int32_t n_iters, float* total_ms) {
  try {  // no C++ exception crosses the C boundary
    if (!c || !c->finalized) return b2s_int_fail(B2S_ERR_STATE, "plan not finalized");
    if (!d_in || n_bufs <= 0 || n_iters <= 0 || !total_ms) return b2s_int_fail(B2S_ERR_INVALID, "bad arguments");
    COL_TRY(cudaSetDevice(b2s_int_device()));
    cudaStream_t st = b2s_int_stream();
    std::lock_guard<std::mutex> lk(c->mu);
    COL_TRY(cudaEventRecord(c->ev[0], st));
    for (int i = 0; i < n_iters; ++i)
      if (int rc = launch_cols(c, d_in[i % n_bufs], in_slot_stride, n_rows, d_out, out_slot_stride, (unsigned long long*)d_counters, st)) return rc;
    COL_TRY(cudaEventRecord(c->ev[1], st));
    COL_TRY(cudaStreamSynchronize(st));
    COL_TRY(cudaEventElapsedTime(total_ms, c->ev[0], c->ev[1]));
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_run_host(b2s_cols_t c, const void* const* h_in_slots, int64_t n_rows, void* const* h_out_slots,
                                 uint64_t* counters, b2s_stats* stats) {
  try {  // no C++ exception crosses the C boundary
    if (!c || !c->finalized) return b2s_int_fail(B2S_ERR_STATE, "plan not finalized");
    if (n_rows < 0 || !h_in_slots || !h_out_slots) return b2s_int_fail(B2S_ERR_INVALID, "bad arguments");
    if (c->n_counters && !counters) return b2s_int_fail(B2S_ERR_INVALID, "the plan has %d counters: pass an array", c->n_counters);
    for (int i = 0; i < c->n_counters; ++i) counters[i] = 0;
    if (n_rows == 0) return B2S_OK;
    std::lock_guard<std::mutex> lk(c->mu);
    COL_TRY(cudaSetDevice(b2s_int_device()));
    const int64_t stride = ((n_rows * 4 + 255) / 256) * 256;
    c->res_rows = 0;
    ++c->res_gen;
    const size_t n_out = c->out_words.size();
    if (n_rows > c->cap_rows) {
      if (c->d_in) { cudaFree(c->d_in); cudaFree(c->d_out); c->d_in = c->d_out = nullptr; }
      c->cap_rows = 0;
      COL_TRY(cudaMalloc(&c->d_in, (size_t)stride * c->n_in));
      COL_TRY(cudaMalloc(&c->d_out, (size_t)stride * n_out));
      c->cap_rows = n_rows;
    }
    cudaStream_t st = b2s_int_stream();
    // Large frames run as a pipeline of row ranges: the columns of range r + 1 cross PCIe on the copy stream while range r
    // is transformed and its result columns travel back (the two PCIe directions overlap), so a frame costs about
    // max(H2D, D2H) instead of their sum.  Needs pinned column buffers on both sides to overlap at all (pageable copies
    // are staged synchronously by the driver) -- see mlrun_b200.feature_store.columnar.
    static const int64_t pipe_rows = getenv("B2S_COLS_CHUNK") ? atoll(getenv("B2S_COLS_CHUNK")) : 65536;
    if (pipe_rows > 0 && n_rows >= 2 * pipe_rows) {
      const int64_t chunk = (pipe_rows + kColChunk - 1) / kColChunk * kColChunk;
      const int n_chunks = (int)((n_rows + chunk - 1) / chunk);
      cudaStream_t cs = b2s_int_copy_stream();
      while ((int)c->chunk_ev.size() < n_chunks) {
        cudaEvent_t e;
        COL_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->chunk_ev.push_back(e);
      }
      for (int s = 0; s < c->n_in; ++s)
        if (c->in_used[s] && !h_in_slots[s]) return b2s_int_fail(B2S_ERR_INVALID, "input slot %d is read by the plan but its pointer is NULL", s);
      for (size_t s = 0; s < n_out; ++s)
        if (c->out_words[s] && !h_out_slots[s]) return b2s_int_fail(B2S_ERR_INVALID, "output slot %zu has no destination", s);
      if (c->n_counters) COL_TRY(cudaMemsetAsync(c->d_cnt, 0, c->n_counters * sizeof(unsigned long long), st));
      COL_TRY(cudaEventRecord(c->ev[0], st));
      COL_TRY(cudaStreamWaitEvent(cs, c->ev[0], 0));  // whatever ran on the library stream before is done with d_in
      // Columns that sit at a constant pitch in host memory (views of one pinned block: columnar.pinned_columns, the
      // ColumnBatch of the results) cross PCIe as ONE 2-D copy per row range and run of columns instead of one copy per
      // column: ~570 copies of 256 KB per range become a handful (copy-engine set-up and driver calls were 2/3 of the time).
      struct Run { int s0, count; size_t w, hpitch, dpitch; };
      auto find_runs = [&](int n_slots, auto words_of, auto host_of) {
        std::vector<Run> runs;
        static const int two_d = getenv("B2S_COLS_2D") ? atoi(getenv("B2S_COLS_2D")) : 1;
        int s = 0;
        while (s < n_slots) {
          const int wd = words_of(s);
          if (!wd) { ++s; continue; }
          Run r{s, 1, 4u * (size_t)wd, 0, (size_t)wd * (size_t)stride};
          int prev = s, t = s + wd;
          while (two_d && t < n_slots && words_of(t) == wd) {
            const ptrdiff_t d = (const char*)host_of(t) - (const char*)host_of(prev);
            if (d < (ptrdiff_t)(chunk * r.w) || d > (ptrdiff_t)0x7fffffff || r.dpitch > (size_t)0x7fffffff ||  // (pitch limit of 2-D copies)
                (r.count > 1 && (size_t)d != r.hpitch))
              break;
            r.hpitch = (size_t)d;
            ++r.count;
            prev = t;
            t += wd;
          }
          if (r.count == 1) r.hpitch = r.dpitch;
          runs.push_back(r);
          s = prev + wd;
        }
        return runs;
      };
      const std::vector<Run> in_runs = find_runs(c->n_in, [&](int s) { return (int)c->in_used[s]; }, [&](int s) { return h_in_slots[s]; });
      const std::vector<Run> out_runs = find_runs((int)n_out, [&](int s) { return (int)c->out_words[s]; }, [&](int s) { return (const void*)h_out_slots[s]; });
      for (int k = 0; k < n_chunks; ++k) {
        const int64_t r0 = (int64_t)k * chunk, nr = std::min<int64_t>(chunk, n_rows - r0);
        for (const Run& r : in_runs) {
          char* dst = c->d_in + (size_t)r.s0 * stride + (size_t)r0 * r.w;
          const char* src = (const char*)h_in_slots[r.s0] + (size_t)r0 * r.w;
          if (r.count == 1) COL_TRY(cudaMemcpyAsync(dst, src, (size_t)nr * r.w, cudaMemcpyHostToDevice, cs));
          else COL_TRY(cudaMemcpy2DAsync(dst, r.dpitch, src, r.hpitch, (size_t)nr * r.w, (size_t)r.count, cudaMemcpyHostToDevice, cs));
        }
        COL_TRY(cudaEventRecord(c->chunk_ev[k], cs));
        COL_TRY(cudaStreamWaitEvent(st, c->chunk_ev[k], 0));
        if (int rc = launch_cols(c, c->d_in, stride, nr, c->d_out, stride, c->d_cnt, st, r0)) {
          cudaStreamSynchronize(cs);
          cudaStreamSynchronize(st);
          return rc;
        }
        for (const Run& r : out_runs) {
          char* dst = (char*)h_out_slots[r.s0] + (size_t)r0 * r.w;
          const char* src = c->d_out + (size_t)r.s0 * stride + (size_t)r0 * r.w;
          if (r.count == 1) COL_TRY(cudaMemcpyAsync(dst, src, (size_t)nr * r.w, cudaMemcpyDeviceToHost, st));
          else COL_TRY(cudaMemcpy2DAsync(dst, r.hpitch, src, r.dpitch, (size_t)nr * r.w, (size_t)r.count, cudaMemcpyDeviceToHost, st));
        }
      }
      if (c->n_counters) COL_TRY(cudaMemcpyAsync(counters, c->d_cnt, c->n_counters * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
      COL_TRY(cudaEventRecord(c->ev[3], st));
      COL_TRY(cudaStreamSynchronize(st));
      COL_TRY(cudaStreamSynchronize(cs));
      c->res_rows = n_rows;
      c->res_stride = stride;
      if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rows = n_rows;
        cudaEventElapsedTime(&stats->kernel_ms, c->ev[0], c->ev[3]);  // the whole pipelined span
        stats->kernels = n_chunks;
      }
      return B2S_OK;
    }
    COL_TRY(cudaEventRecord(c->ev[0], st));
    for (int s = 0; s < c->n_in; ++s) {
      if (!c->in_used[s]) continue;
      if (!h_in_slots[s]) return b2s_int_fail(B2S_ERR_INVALID, "input slot %d is read by the plan but its pointer is NULL", s);
      COL_TRY(cudaMemcpyAsync(c->d_in + (size_t)s * stride, h_in_slots[s], (size_t)n_rows * 4 * c->in_used[s], cudaMemcpyHostToDevice, st));
    }
    if (c->n_counters) COL_TRY(cudaMemsetAsync(c->d_cnt, 0, c->n_counters * sizeof(unsigned long long), st));
    COL_TRY(cudaEventRecord(c->ev[1], st));
    if (int rc = launch_cols(c, c->d_in, stride, n_rows, c->d_out, stride, c->d_cnt, st)) return rc;
    COL_TRY(cudaEventRecord(c->ev[2], st));
    for (size_t s = 0; s < n_out; ++s) {
      if (!c->out_words[s]) continue;  // second half of an 8-byte column
      if (!h_out_slots[s]) return b2s_int_fail(B2S_ERR_INVALID, "output slot %zu has no destination", s);
      COL_TRY(cudaMemcpyAsync(h_out_slots[s], c->d_out + s * (size_t)stride, (size_t)n_rows * 4 * c->out_words[s], cudaMemcpyDeviceToHost, st));
    }
    if (c->n_counters) COL_TRY(cudaMemcpyAsync(counters, c->d_cnt, c->n_counters * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    COL_TRY(cudaEventRecord(c->ev[3], st));
    COL_TRY(cudaStreamSynchronize(st));
    c->res_rows = n_rows;
    c->res_stride = stride;
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->rows = n_rows;
      cudaEventElapsedTime(&stats->h2d_ms, c->ev[0], c->ev[1]);
      cudaEventElapsedTime(&stats->kernel_ms, c->ev[1], c->ev[2]);
      cudaEventElapsedTime(&stats->d2h_ms, c->ev[2], c->ev[3]);
      stats->kernels = 1;
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

std::mutex& b2s_int_cols_mutex(b2s_cols_s* c) { return c->mu; }

int b2s_int_cols_result(b2s_cols_s* c, const char** d_out, long long* stride, long long* rows, int* n_out_slots,
                        unsigned long long* generation) {
  if (!c || !c->finalized) return b2s_int_fail(B2S_ERR_STATE, "plan not finalized");
  *generation = c->res_gen;
  if (!c->res_rows) return b2s_int_fail(B2S_ERR_STATE, "the plan holds no result: run it with b2s_cols_run_host first (or pass d_out)");
  *d_out = c->d_out;
  *stride = c->res_stride;
  *rows = c->res_rows;
  *n_out_slots = (int)c->out_words.size();
  return B2S_OK;
}

ColStatsWS*& b2s_int_cols_stats_ws(b2s_cols_s* c) { return c->stats_ws; }

extern "C" int b2s_cols_destroy(b2s_cols_t c) {
  try {  // no C++ exception crosses the C boundary
    if (!c) return B2S_OK;
    if (c->d_ops) cudaFree(c->d_ops);
    if (c->d_tab) cudaFree(c->d_tab);
    if (c->d_cnt) cudaFree(c->d_cnt);
    if (c->d_in) cudaFree(c->d_in);
    if (c->d_out) cudaFree(c->d_out);
    for (auto& e : c->ev)
      if (e) cudaEventDestroy(e);
    for (auto& e : c->chunk_ev) cudaEventDestroy(e);
    b2s_int_colstats_free(c->stats_ws);
    delete c;
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
