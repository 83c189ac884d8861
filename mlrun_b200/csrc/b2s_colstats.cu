// b2s_colstats.cu -- C-ABI of the feature-set statistics over a columns plan's result (see include/b200serve.h,
// "feature-set statistics", and b2s_colstats.cuh for the passes).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <exception>
#include <mutex>
#include <vector>

#include "../../include/b200serve.h"
#include "b2s_colstats.cuh"
#include "b2s_internal.h"

using namespace b2s;

#define ST_TRY(expr)                                                                                        \
  do {                                                                                                      \
    cudaError_t _e = (expr);                                                                                \
    if (_e != cudaSuccess)                                                                                  \
      return b2s_int_fail(B2S_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

namespace {

constexpr int kUnroll = 4;   // 16-byte loads in flight per thread
constexpr int kVec = 4;      // rows per load group

// the warp's lanes add 1 to h[bin] (bin < 0: nothing).  A warp whose lanes all hit one bin (a constant or sorted stretch, a
// low-cardinality column) adds 32 with one atomic instead of 32 serialised ones; otherwise every lane adds its own.
// (__match_any_sync merging of every group was measured slower: it bounded the passes at 6-12 % of HBM bandwidth.)
__device__ __forceinline__ void agg_inc(unsigned int* h, int bin) {
  const int b0 = __shfl_sync(0xffffffffu, bin, 0);
  if (__all_sync(0xffffffffu, bin == b0)) {
    if (b0 >= 0 && (threadIdx.x & 31) == 0) atomicAdd(&h[b0], 32u);
  } else if (bin >= 0) {
    atomicAdd(&h[bin], 1u);
  }
}

struct Val {
  double x;
  unsigned long long key;
  unsigned long long raw;
  bool missing;
};

__device__ __forceinline__ Val decode32(int kind, uint32_t bits) {
  Val v;
  if (kind == SK_F32) {
    const float f = __uint_as_float(bits);
    v.missing = f != f;
    v.x = (double)f;
    v.key = (bits & 0x80000000u) ? (unsigned long long)(~bits) : (unsigned long long)(bits | 0x80000000u);
    v.raw = bits;
  } else {
    const int32_t i = (int32_t)bits;
    v.missing = kind == SK_I32_NAT && i < 0;
    v.x = (double)i;
    v.key = (unsigned long long)(bits ^ 0x80000000u);
    v.raw = (unsigned long long)(long long)i;
  }
  return v;
}

__device__ __forceinline__ Val decode64(long long i) {
  Val v;
  v.missing = i == (long long)INT64_MIN;
  v.x = (double)i;
  v.key = (unsigned long long)i ^ 0x8000000000000000ull;
  v.raw = (unsigned long long)i;
  return v;
}

// np.histogram's uniform-bin index (numpy/lib/_histograms_impl.py, the `uniform_bins` branch) in the bin dtype, with
// rounded operations only: f = ((x - first) / den) * n, truncated, then the +-1 correction against the edges
__device__ __forceinline__ int bin_f32(float x, float first, float den, const float* e) {
  const float f = __fmul_rn(__fdiv_rn(__fsub_rn(x, first), den), (float)kStBins);
  int i = (int)f;
  if (i >= kStBins) i = kStBins - 1;
  if (i < 0) i = 0;
  if (x < e[i]) --i;
  if (i != kStBins - 1 && x >= e[i + 1]) ++i;
  return i;
}

__device__ __forceinline__ int bin_f64(double x, double first, double den, const double* e) {
  const double f = __dmul_rn(__ddiv_rn(__dsub_rn(x, first), den), (double)kStBins);
  int i = (int)f;
  if (i >= kStBins) i = kStBins - 1;
  if (i < 0) i = 0;
  if (x < e[i]) --i;
  if (i != kStBins - 1 && x >= e[i + 1]) ++i;
  return i;
}

__global__ void __launch_bounds__(kStThreads) colstats_pass_kernel(const __grid_constant__ StatParams P) {
  extern __shared__ unsigned int s_dig[];  // [active slots][kStRadix]
  __shared__ unsigned int s_hist[kStBins];
  __shared__ float s_ef[kStBins + 1];
  __shared__ double s_ed[kStBins + 1];
  __shared__ unsigned long long s_pref[kStRanks];
  __shared__ int s_slot_of[kStRanks];  // rank -> position of its histogram in s_dig (-1: not counted in this pass)
  __shared__ int s_n_slots;
  __shared__ double s_red[kStThreads / 32];
  __shared__ unsigned long long s_cnt[4], s_kmax, s_kmin_inv;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t n_items = (int64_t)P.n_list * P.n_chunks;
  for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int col = P.list[item / P.n_chunks];
    const int64_t chunk = item % P.n_chunks;
    const StatCol& c = P.cols[col];
    const int kind = c.kind;
    const int64_t row0 = chunk * kStChunk;
    const int rows = (int)(P.n_rows - row0 < kStChunk ? P.n_rows - row0 : kStChunk);
    int shift, width;
    st_digit(c.key_bits, P.pass, shift, width);
    const unsigned long long hi_mask = (shift + width >= 64) ? 0ull : (~0ull << (shift + width));
    const bool do_hist = P.pass == 1 && c.hist;
    const bool do_m2 = P.pass == 1 && c.centre;
    if (tid == 0) {
      int n = 0;
      if (P.pass == 0) {
        s_slot_of[0] = n++;
        for (int r = 1; r < kStRanks; ++r) s_slot_of[r] = -1;
      } else {
        const StatSel& s = P.sel[col];
        for (int r = 0; r < kStRanks; ++r) {
          s_pref[r] = s.prefix[r];
          s_slot_of[r] = (s.rank[r] >= 0 && s.src[r] == r) ? n++ : -1;
        }
      }
      s_n_slots = n;
      s_cnt[0] = s_cnt[1] = s_cnt[2] = s_cnt[3] = 0;
      s_kmax = s_kmin_inv = 0;
    }
    if (do_hist && tid <= kStBins) {
      s_ed[tid] = c.edges[tid];
      s_ef[tid] = (float)c.edges[tid];
    }
    if (tid < kStBins) s_hist[tid] = 0;
    __syncthreads();
    const int n_slots = s_n_slots;
    for (int i = tid; i < n_slots * kStRadix; i += kStThreads) s_dig[i] = 0;
    __syncthreads();

    const float ff = (float)c.h_first, fd = (float)c.h_den;
    const double mean = c.mean;
    unsigned long long cnt = 0, miss = 0, ones = 0, flags = 0, kmax = 0, kmin_inv = 0;
    double acc = 0.0;
    auto visit = [&](const Val& v, bool valid) {
      const bool ok = valid && !v.missing;
      int dbin = -1, hbin = -1;
      if (P.pass == 0) {
        if (valid) {
          if (v.missing) {
            ++miss;
          } else {
            ++cnt;
            acc += v.x;
            kmax = max(kmax, v.key);
            kmin_inv = max(kmin_inv, ~v.key);
            if (kind == SK_F32 && isinf(v.x)) flags |= v.x > 0 ? 1ull : 2ull;
            if (kind == SK_BOOL && v.raw == 1) ++ones;
          }
        }
        if (ok) dbin = (int)(v.key >> shift);
      } else {
        if (ok) {
          if (do_m2) {
            const double d = v.x - mean;
            acc += d * d;
          }
          if (do_hist) hbin = c.hist == 1 ? bin_f32((float)v.x, ff, fd, s_ef) : bin_f64(v.x, c.h_first, c.h_den, s_ed);
          for (int r = 0; r < kStRanks; ++r)
            if (s_slot_of[r] >= 0 && (v.key & hi_mask) == s_pref[r])
              dbin = s_slot_of[r] * kStRadix + (int)((v.key >> shift) & ((1ull << width) - 1));
        }
      }
      if (n_slots) agg_inc(s_dig, dbin);
      if (do_hist) agg_inc(s_hist, hbin);
    };

    if (kind == SK_DT) {
      const long long* s = reinterpret_cast<const long long*>(P.base + (int64_t)c.slot * P.stride) + row0;
      const bool vec = (reinterpret_cast<uintptr_t>(s) & 15) == 0;
      for (int base = 0; base < rows; base += kStThreads * kVec * kUnroll) {
        long long w[kUnroll][kVec];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          const int r = base + (u * kStThreads + tid) * kVec;
          if (vec && r + kVec <= rows) {
            const longlong2 a = reinterpret_cast<const longlong2*>(s + r)[0];
            const longlong2 b = reinterpret_cast<const longlong2*>(s + r)[1];
            w[u][0] = a.x; w[u][1] = a.y; w[u][2] = b.x; w[u][3] = b.y;
          } else {
#pragma unroll
            for (int k = 0; k < kVec; ++k) w[u][k] = r + k < rows ? s[r + k] : 0;
          }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
#pragma unroll
          for (int k = 0; k < kVec; ++k) visit(decode64(w[u][k]), base + (u * kStThreads + tid) * kVec + k < rows);
      }
    } else {
      const uint32_t* s = kind == SK_ROW ? nullptr : reinterpret_cast<const uint32_t*>(P.base + (int64_t)c.slot * P.stride) + row0;
      const bool vec = (reinterpret_cast<uintptr_t>(s) & 15) == 0;
      for (int base = 0; base < rows; base += kStThreads * kVec * kUnroll) {
        uint32_t w[kUnroll][kVec];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
          const int r = base + (u * kStThreads + tid) * kVec;
          if (kind == SK_ROW) {
#pragma unroll
            for (int k = 0; k < kVec; ++k) w[u][k] = (uint32_t)(row0 + r + k);
          } else if (vec && r + kVec <= rows) {
            const uint4 a = reinterpret_cast<const uint4*>(s + r)[0];
            w[u][0] = a.x; w[u][1] = a.y; w[u][2] = a.z; w[u][3] = a.w;
          } else {
#pragma unroll
            for (int k = 0; k < kVec; ++k) w[u][k] = r + k < rows ? s[r + k] : 0u;
          }
        }
        const int dk = kind == SK_ROW ? SK_I32 : kind;
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
#pragma unroll
          for (int k = 0; k < kVec; ++k) visit(decode32(dk, w[u][k]), base + (u * kStThreads + tid) * kVec + k < rows);
      }
    }

    // item totals: integers through atomics, the fp64 sum in a fixed order (warps, then warp 0's lanes)
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s_red[warp] = acc;
    if (P.pass == 0) {
      for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        miss += __shfl_xor_sync(0xffffffffu, miss, o);
        ones += __shfl_xor_sync(0xffffffffu, ones, o);
        flags |= __shfl_xor_sync(0xffffffffu, flags, o);
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
        kmin_inv = max(kmin_inv, __shfl_xor_sync(0xffffffffu, kmin_inv, o));
      }
      if (lane == 0) {
        atomicAdd(&s_cnt[0], cnt);
        atomicAdd(&s_cnt[1], miss);
        atomicAdd(&s_cnt[2], ones);
        atomicOr(&s_cnt[3], flags);
        atomicMax(&s_kmax, kmax);
        atomicMax(&s_kmin_inv, kmin_inv);
      }
    }
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int k = 0; k < kStThreads / 32; ++k) t += s_red[k];
      P.part[(int64_t)col * P.n_chunks + chunk] = t;
      if (P.pass == 0) {
        StatAcc& a = P.acc[col];
        if (s_cnt[0]) atomicAdd(&a.count, s_cnt[0]);
        if (s_cnt[1]) atomicAdd(&a.missing, s_cnt[1]);
        if (s_cnt[2]) atomicAdd(&a.ones, s_cnt[2]);
        if (s_cnt[3]) atomicOr(&a.flags, s_cnt[3]);
        if (s_cnt[0]) {
          atomicMax(&a.kmax, s_kmax);
          atomicMax(&a.kmin_inv, s_kmin_inv);
        }
        if (chunk == 0) {
          Val v;
          if (kind == SK_DT) v = decode64(*reinterpret_cast<const long long*>(P.base + (int64_t)c.slot * P.stride));
          else if (kind == SK_ROW) v = decode32(SK_I32, 0u);
          else v = decode32(kind, *reinterpret_cast<const uint32_t*>(P.base + (int64_t)c.slot * P.stride));
          a.first = v.raw;
          a.first_missing = v.missing ? 1ull : 0ull;
        }
      }
    }
    if (do_hist && tid < kStBins && s_hist[tid]) atomicAdd(&P.acc[col].hist[tid], (unsigned long long)s_hist[tid]);
    for (int r = 0; r < kStRanks; ++r) {
      const int sl = s_slot_of[r];
      if (sl < 0) continue;
      unsigned int* g = P.digits + ((int64_t)col * kStRanks + r) * kStRadix;
      for (int b = tid; b < kStRadix; b += kStThreads) {
        const unsigned int v = s_dig[sl * kStRadix + b];
        if (v) atomicAdd(&g[b], v);
      }
    }
    __syncthreads();
  }
}

// fp64 partial sums of the pass, added in chunk order: one thread per column
__global__ void colstats_combine_kernel(const __grid_constant__ StatParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n_list) return;
  const int col = P.list[i];
  double t = 0.0;
  for (int64_t k = 0; k < P.n_chunks; ++k) t += P.part[(int64_t)col * P.n_chunks + k];
  if (P.pass == 0) P.acc[col].sum = t;
  else P.acc[col].m2 = t;
}

// one block per column, one warp per rank: find the digit bucket holding the rank in the histogram of its prefix
__global__ void __launch_bounds__(32 * kStRanks) colstats_select_kernel(const __grid_constant__ StatParams P) {
  const int col = P.list[blockIdx.x];
  const int r = threadIdx.x >> 5, lane = threadIdx.x & 31;
  StatSel& s = P.sel[col];
  const long long rank = s.rank[r];
  int shift, width;
  st_digit(P.cols[col].key_bits, P.pass, shift, width);
  if (rank >= 0) {
    const unsigned int* h = P.digits + ((int64_t)col * kStRanks + s.src[r]) * kStRadix;
    const int per = kStRadix / 32, b0 = lane * per, nb = 1 << width;
    unsigned long long mine = 0;
    for (int b = b0; b < b0 + per && b < nb; ++b) mine += h[b];
    unsigned long long incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const unsigned long long excl = incl - mine;
    if ((unsigned long long)rank >= excl && (unsigned long long)rank < incl) {
      unsigned long long before = excl;
      int b = b0;
      for (; b < b0 + per; ++b) {
        if ((unsigned long long)rank < before + h[b]) break;
        before += h[b];
      }
      s.rank[r] = rank - (long long)before;
      s.prefix[r] |= (unsigned long long)b << shift;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // ranks whose prefixes agree share one histogram in the next pass
    for (int q = 0; q < kStRanks; ++q) {
      s.src[q] = q;
      if (s.rank[q] < 0) continue;
      for (int t = 0; t < q; ++t)
        if (s.rank[t] >= 0 && s.prefix[t] == s.prefix[q]) {
          s.src[q] = s.src[t];
          break;
        }
    }
  }
}

int digit_passes(int key_bits) { return (key_bits + kStDigit - 1) / kStDigit; }

}  // namespace

// the statistics workspace of one columns plan (between b2s_cols_stats_begin and b2s_cols_stats_finish)
struct ColStatsWS {
  int32_t n_cols = 0, cap_cols = 0;
  int64_t n_rows = 0, n_chunks = 0, cap_parts = 0;
  const char* base = nullptr;
  int64_t stride = 0;
  std::vector<StatCol> cols;
  StatCol* d_cols = nullptr;
  StatAcc* d_acc = nullptr;
  StatSel* d_sel = nullptr;
  int32_t* d_list = nullptr;  // [n_cols] per pass slot: pass p's list at d_list + p * n_cols
  unsigned int* d_digits = nullptr;
  double* d_part = nullptr;
  cudaEvent_t ev[8] = {};
  float pass_ms[6] = {};
  int64_t pass_bytes[6] = {};
  int32_t n_passes = 0, launches = 0;
  bool begun = false;
  bool resident = false;              // describing the plan's own result: finish checks it is still the one begin saw
  unsigned long long generation = 0;
};

void b2s_int_colstats_free(ColStatsWS* w) {
  if (!w) return;
  cudaFree(w->d_cols);
  cudaFree(w->d_acc);
  cudaFree(w->d_sel);
  cudaFree(w->d_list);
  cudaFree(w->d_digits);
  cudaFree(w->d_part);
  for (auto& e : w->ev)
    if (e) cudaEventDestroy(e);
  delete w;
}

static int ws_reserve(ColStatsWS* w, int32_t n_cols, int64_t n_chunks) {
  if (!w->ev[0])
    for (auto& e : w->ev) ST_TRY(cudaEventCreate(&e));
  if (n_cols > w->cap_cols) {
    cudaFree(w->d_cols); cudaFree(w->d_acc); cudaFree(w->d_sel); cudaFree(w->d_list); cudaFree(w->d_digits);
    w->d_cols = nullptr; w->d_acc = nullptr; w->d_sel = nullptr; w->d_list = nullptr; w->d_digits = nullptr;
    w->cap_cols = 0;
    ST_TRY(cudaMalloc(&w->d_cols, sizeof(StatCol) * n_cols));
    ST_TRY(cudaMalloc(&w->d_acc, sizeof(StatAcc) * n_cols));
    ST_TRY(cudaMalloc(&w->d_sel, sizeof(StatSel) * n_cols));
    ST_TRY(cudaMalloc(&w->d_list, sizeof(int32_t) * n_cols * 6));
    ST_TRY(cudaMalloc(&w->d_digits, sizeof(unsigned int) * (size_t)n_cols * kStRanks * kStRadix));
    w->cap_cols = n_cols;
  }
  if ((int64_t)n_cols * n_chunks > w->cap_parts) {
    cudaFree(w->d_part);
    w->d_part = nullptr;
    w->cap_parts = 0;
    ST_TRY(cudaMalloc(&w->d_part, sizeof(double) * n_cols * n_chunks));
    w->cap_parts = (int64_t)n_cols * n_chunks;
  }
  return B2S_OK;
}

static int launch_pass(ColStatsWS* w, int pass, const int32_t* d_list, int n_list, int n_slots, cudaStream_t st) {
  StatParams p{};
  p.base = w->base;
  p.stride = w->stride;
  p.n_rows = w->n_rows;
  p.n_chunks = w->n_chunks;
  p.cols = w->d_cols;
  p.acc = w->d_acc;
  p.sel = w->d_sel;
  p.list = d_list;
  p.n_list = n_list;
  p.pass = pass;
  p.digits = w->d_digits;
  p.part = w->d_part;
  const size_t smem = (size_t)n_slots * kStRadix * sizeof(unsigned int);
  // the opt-in above 48 KB is a property of the current device's context: set it for the launch that needs it
  ST_TRY(cudaFuncSetAttribute(colstats_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  ST_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, colstats_pass_kernel, kStThreads, smem));
  const int64_t items = (int64_t)n_list * w->n_chunks;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(items, (int64_t)b2s_int_sm_count() * std::max(occ, 1) * 4));
  ST_TRY(cudaMemsetAsync(w->d_digits, 0, sizeof(unsigned int) * (size_t)w->n_cols * kStRanks * kStRadix, st));
  colstats_pass_kernel<<<grid, kStThreads, smem, st>>>(p);
  ST_TRY(cudaGetLastError());
  const bool sums = pass <= 1;
  if (sums) {
    colstats_combine_kernel<<<(n_list + 127) / 128, 128, 0, st>>>(p);
    ST_TRY(cudaGetLastError());
  }
  w->launches += sums ? 2 : 1;
  b2s_int_count_launches(sums ? 2 : 1);
  return B2S_OK;
}

static int launch_select(ColStatsWS* w, int pass, const int32_t* d_list, int n_list, cudaStream_t st) {
  StatParams p{};
  p.cols = w->d_cols;
  p.sel = w->d_sel;
  p.list = d_list;
  p.n_list = n_list;
  p.pass = pass;
  p.digits = w->d_digits;
  colstats_select_kernel<<<n_list, 32 * kStRanks, 0, st>>>(p);
  ST_TRY(cudaGetLastError());
  w->launches += 1;
  b2s_int_count_launches(1);
  return B2S_OK;
}

// order-preserving key -> the value's bits as b2s_colsum reports them (float32 bits for B2S_STAT_F32, else the integer)
static int64_t stat_value(int kind, unsigned long long key) {
  if (kind == SK_F32) {
    const uint32_t k = (uint32_t)key;
    return (int64_t)(uint32_t)((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
  }
  if (kind == SK_DT) return (int64_t)(key ^ 0x8000000000000000ull);
  return (int64_t)(int32_t)((uint32_t)key ^ 0x80000000u);
}

static int64_t bytes_per_row(int kind) { return kind == SK_ROW ? 0 : (kind == SK_DT ? 8 : 4); }

extern "C" int b2s_cols_stats_begin(b2s_cols_t plan, const void* d_out, int64_t out_slot_stride, int64_t n_rows,
                                    const int32_t* kinds, const int32_t* slots, int32_t n_cols, b2s_colsum* summary,
                                    b2s_stats* stats) {
  try {  // no C++ exception crosses the C boundary
    if (!plan || n_cols <= 0 || !kinds || !slots || !summary) return b2s_int_fail(B2S_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> lk(b2s_int_cols_mutex(plan));  // no host run of the plan interleaves with this call
    const char* base = (const char*)d_out;
    long long stride = out_slot_stride, rows = n_rows;
    int n_out = 0;
    unsigned long long gen = 0;
    if (!base) {
      if (int rc = b2s_int_cols_result(plan, &base, &stride, &rows, &n_out, &gen)) return rc;
      if (n_rows != rows) return b2s_int_fail(B2S_ERR_INVALID, "the plan's resident result holds %lld rows, not %lld", (long long)rows, (long long)n_rows);
    } else if (n_rows < 0 || (stride & 15) || stride < n_rows * 4) {
      return b2s_int_fail(B2S_ERR_INVALID, "slot stride must hold n_rows words and be a multiple of 16 bytes");
    }
    if (rows <= 0) return b2s_int_fail(B2S_ERR_INVALID, "no rows to describe");
    if (rows >= ((int64_t)1 << 31)) return b2s_int_fail(B2S_ERR_UNSUPPORTED, "frames of 2^31 rows or more");
    std::vector<StatCol> cols(n_cols);
    for (int i = 0; i < n_cols; ++i) {
      StatCol& c = cols[i];
      memset(&c, 0, sizeof(c));
      c.kind = kinds[i];
      c.slot = slots[i];
      if (c.kind < SK_F32 || c.kind > SK_ROW) return b2s_int_fail(B2S_ERR_INVALID, "column %d: bad stats kind %d", i, c.kind);
      const int words = c.kind == SK_DT ? 2 : 1;
      if (c.kind != SK_ROW && (c.slot < 0 || (n_out && c.slot + words > n_out)))
        return b2s_int_fail(B2S_ERR_INVALID, "column %d: result slot %d out of range", i, c.slot);
      c.key_bits = c.kind == SK_DT ? 64 : 32;
    }
    ColStatsWS*& w = b2s_int_cols_stats_ws(plan);
    if (!w) w = new ColStatsWS();
    ST_TRY(cudaSetDevice(b2s_int_device()));
    w->begun = false;
    w->resident = d_out == nullptr;
    w->generation = gen;
    const int64_t n_chunks = (rows + kStChunk - 1) / kStChunk;
    if (int rc = ws_reserve(w, n_cols, n_chunks)) return rc;
    w->cols = cols;
    w->n_cols = n_cols;
    w->n_rows = rows;
    w->n_chunks = n_chunks;
    w->base = base;
    w->stride = stride;
    w->launches = 0;
    w->n_passes = 0;
    cudaStream_t st = b2s_int_stream();
    std::vector<int32_t> all(n_cols);
    for (int i = 0; i < n_cols; ++i) all[i] = i;
    ST_TRY(cudaMemcpyAsync(w->d_cols, cols.data(), sizeof(StatCol) * n_cols, cudaMemcpyHostToDevice, st));
    ST_TRY(cudaMemcpyAsync(w->d_list, all.data(), sizeof(int32_t) * n_cols, cudaMemcpyHostToDevice, st));
    ST_TRY(cudaMemsetAsync(w->d_acc, 0, sizeof(StatAcc) * n_cols, st));
    ST_TRY(cudaEventRecord(w->ev[0], st));
    if (int rc = launch_pass(w, 0, w->d_list, n_cols, 1, st)) return rc;
    ST_TRY(cudaEventRecord(w->ev[1], st));
    std::vector<StatAcc> acc(n_cols);
    ST_TRY(cudaMemcpyAsync(acc.data(), w->d_acc, sizeof(StatAcc) * n_cols, cudaMemcpyDeviceToHost, st));
    ST_TRY(cudaStreamSynchronize(st));
    ST_TRY(cudaEventElapsedTime(&w->pass_ms[0], w->ev[0], w->ev[1]));
    int64_t bytes = 0;
    for (const StatCol& c : cols) bytes += bytes_per_row(c.kind) * rows;
    w->pass_bytes[0] = bytes;
    w->n_passes = 1;
    for (int i = 0; i < n_cols; ++i) {
      const StatAcc& a = acc[i];
      b2s_colsum& s = summary[i];
      memset(&s, 0, sizeof(s));
      s.count = (int64_t)a.count;
      s.missing = (int64_t)a.missing;
      s.ones = (int64_t)a.ones;
      s.pos_inf = (a.flags & 1) ? 1 : 0;
      s.neg_inf = (a.flags & 2) ? 1 : 0;
      s.sum = a.sum;
      s.first_bits = (int64_t)a.first;
      s.first_missing = (int32_t)a.first_missing;
      if (a.count) {
        s.min_bits = stat_value(cols[i].kind, ~a.kmin_inv);
        s.max_bits = stat_value(cols[i].kind, a.kmax);
      }
    }
    w->begun = true;
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->rows = rows;
      stats->kernel_ms = w->pass_ms[0];
      stats->kernels = w->launches;
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_stats_finish(b2s_cols_t plan, const double* means, const int32_t* hist_kind, const double* hist,
                                     const int64_t* ranks, double* m2, int64_t* hist_counts, int64_t* order_values,
                                     b2s_stats* stats) {
  try {  // no C++ exception crosses the C boundary
    if (!plan || !means || !hist_kind || !hist || !ranks || !m2 || !hist_counts || !order_values)
      return b2s_int_fail(B2S_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> lk(b2s_int_cols_mutex(plan));
    ColStatsWS* w = b2s_int_cols_stats_ws(plan);
    if (!w || !w->begun) return b2s_int_fail(B2S_ERR_STATE, "b2s_cols_stats_begin was not called");
    if (w->resident) {
      const char* base = nullptr;
      long long stride = 0, rows = 0;
      int n_out = 0;
      unsigned long long gen = 0;
      const int rc = b2s_int_cols_result(plan, &base, &stride, &rows, &n_out, &gen);
      if (rc || gen != w->generation || base != w->base || stride != w->stride || rows != w->n_rows) {
        w->begun = false;
        return b2s_int_fail(B2S_ERR_STATE, "the plan was run again after b2s_cols_stats_begin: its result is not the one described");
      }
    }
    ST_TRY(cudaSetDevice(b2s_int_device()));
    const int n = w->n_cols;
    std::vector<int32_t> lists[6];  // columns read by pass p (1..5); lists[0]: columns with ranks (select after pass 0)
    std::vector<StatSel> sel(n);
    for (int i = 0; i < n; ++i) {
      StatCol& c = w->cols[i];
      c.centre = std::isfinite(means[i]) ? 1 : 0;
      c.mean = c.centre ? means[i] : 0.0;
      c.hist = hist_kind[i];
      if (c.hist < 0 || c.hist > 2 || (c.hist && c.kind == SK_DT)) return b2s_int_fail(B2S_ERR_INVALID, "column %d: bad histogram kind", i);
      c.h_first = hist[i * 23];
      c.h_den = hist[i * 23 + 1];
      for (int e = 0; e <= kStBins; ++e) c.edges[e] = hist[i * 23 + 2 + e];
      StatSel& s = sel[i];
      bool any = false;
      for (int r = 0; r < kStRanks; ++r) {
        const long long k = ranks[i * kStRanks + r];
        if (k >= 0 && k >= (long long)w->n_rows) return b2s_int_fail(B2S_ERR_INVALID, "column %d: rank %lld out of range", i, k);
        s.rank[r] = k < 0 ? -1 : k;
        s.prefix[r] = 0;
        s.src[r] = 0;
        any |= k >= 0;
      }
      if (any) lists[0].push_back(i);
      if (any || c.centre || c.hist) lists[1].push_back(i);
      if (any)
        for (int p = 2; p < digit_passes(c.key_bits); ++p) lists[p].push_back(i);
    }
    cudaStream_t st = b2s_int_stream();
    ST_TRY(cudaMemcpyAsync(w->d_cols, w->cols.data(), sizeof(StatCol) * n, cudaMemcpyHostToDevice, st));
    ST_TRY(cudaMemcpyAsync(w->d_sel, sel.data(), sizeof(StatSel) * n, cudaMemcpyHostToDevice, st));
    for (int p = 0; p < 6; ++p)
      if (!lists[p].empty())
        ST_TRY(cudaMemcpyAsync(w->d_list + p * n, lists[p].data(), sizeof(int32_t) * lists[p].size(), cudaMemcpyHostToDevice, st));
    ST_TRY(cudaEventRecord(w->ev[0], st));
    // pass 0's digit histograms are still in the workspace: the first select needs no pass
    if (!lists[0].empty())
      if (int rc = launch_select(w, 0, w->d_list, (int)lists[0].size(), st)) return rc;
    ST_TRY(cudaEventRecord(w->ev[1], st));
    int from[6] = {}, prev_ev = 1;
    for (int p = 1; p < 6; ++p) {
      w->pass_ms[p] = 0.f;
      w->pass_bytes[p] = 0;
      if (lists[p].empty()) continue;
      const int32_t* dl = w->d_list + p * n;
      if (int rc = launch_pass(w, p, dl, (int)lists[p].size(), kStRanks, st)) return rc;
      if (int rc = launch_select(w, p, dl, (int)lists[p].size(), st)) return rc;  // columns without ranks return at once
      ST_TRY(cudaEventRecord(w->ev[p + 1], st));
      from[p] = prev_ev;
      prev_ev = p + 1;
      for (int i : lists[p]) w->pass_bytes[p] += bytes_per_row(w->cols[i].kind) * w->n_rows;
    }
    std::vector<StatAcc> acc(n);
    ST_TRY(cudaMemcpyAsync(acc.data(), w->d_acc, sizeof(StatAcc) * n, cudaMemcpyDeviceToHost, st));
    ST_TRY(cudaMemcpyAsync(sel.data(), w->d_sel, sizeof(StatSel) * n, cudaMemcpyDeviceToHost, st));
    ST_TRY(cudaStreamSynchronize(st));
    // per-pass kernel time (a pass's select counted with it); the select after pass 0 is in the total only
    float t = 0.f;
    w->n_passes = 1;
    for (int p = 1; p < 6; ++p) {
      if (lists[p].empty()) continue;
      ST_TRY(cudaEventElapsedTime(&w->pass_ms[p], w->ev[from[p]], w->ev[p + 1]));
      w->n_passes = p + 1;
    }
    ST_TRY(cudaEventElapsedTime(&t, w->ev[0], w->ev[prev_ev]));
    for (int i = 0; i < n; ++i) {
      m2[i] = acc[i].m2;
      for (int b = 0; b < kStBins; ++b) hist_counts[i * kStBins + b] = (int64_t)acc[i].hist[b];
      for (int r = 0; r < kStRanks; ++r)
        order_values[i * kStRanks + r] = sel[i].rank[r] < 0 ? 0 : stat_value(w->cols[i].kind, sel[i].prefix[r]);
    }
    w->begun = false;
    if (stats) {
      memset(stats, 0, sizeof(*stats));
      stats->rows = w->n_rows;
      stats->kernel_ms = t;
      stats->kernels = w->launches;
    }
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}

extern "C" int b2s_cols_stats_timing(b2s_cols_t plan, float* pass_ms, int64_t* pass_bytes, int32_t* n_passes, int32_t* launches) {
  try {  // no C++ exception crosses the C boundary
    if (!plan || !pass_ms || !pass_bytes || !n_passes) return b2s_int_fail(B2S_ERR_INVALID, "bad arguments");
    std::lock_guard<std::mutex> lk(b2s_int_cols_mutex(plan));
    ColStatsWS* w = b2s_int_cols_stats_ws(plan);
    if (!w) return b2s_int_fail(B2S_ERR_STATE, "no statistics were computed on this plan");
    for (int p = 0; p < 6; ++p) {
      pass_ms[p] = w->pass_ms[p];
      pass_bytes[p] = w->pass_bytes[p];
    }
    *n_passes = w->n_passes;
    if (launches) *launches = w->launches;
    return B2S_OK;
  } catch (const std::exception& e) {
    return b2s_int_fail(B2S_ERR_INVALID, "%s: %s", __func__, e.what());
  }
}
