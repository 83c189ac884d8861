// b2s_colstats.cuh -- feature-set statistics over the columns plan's result slots (sm_100a), the device side of
// `ingest(..., infer_options=InferOptions.Stats | Histogram)`.
//
// The reference profiles the ingested frame with get_df_stats (mlrun/data_types/infer.py:104-149): pandas
// `describe(include="all")` per column plus a 20-bin np.histogram.  Here the result columns are still resident in HBM
// after the transform, so the statistics are a few streaming passes over them:
//   pass 0  count / missing / fp64 sum / min / max (as order-preserving keys) / +-inf flags / ones (bool) / row 0, and the
//           histogram of the first 11-bit radix digit of every non-missing key;
//   pass 1  the centred sum of squares (two-pass, as pandas), the 20 histogram bins (numpy's uniform-bin arithmetic with
//           explicitly rounded operations: no FMA contraction can move a value to another bin), the next digit;
//   pass 2+ the remaining digits (32-bit keys: 11/11/10 bits; 64-bit datetime keys: 11 x 5 + 9).
// Exact order statistics come from radix select: for each requested rank (up to kStRanks per column) a tiny kernel scans
// the digit histogram after every pass and narrows the rank's key prefix; ranks that share a prefix share a histogram.
// Work items are (column, chunk of kStChunk rows); every integer result is accumulated with atomics (order-independent)
// and the fp64 sums are written per item and added in item order by one thread per column: results are deterministic.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace b2s {

enum StatKind : int32_t {
  SK_F32 = 0,      // float32 slot, NaN is missing
  SK_I32 = 1,      // int32 slot
  SK_I32_NAT = 2,  // int32 date part, -1 marks NaT (missing)
  SK_BOOL = 3,     // int32 0/1 slot
  SK_DT = 4,       // int64 nanoseconds over two slots, NaT (INT64_MIN) is missing
  SK_ROW = 5,      // virtual: the row number (no memory read)
};

constexpr int kStRanks = 6;        // order statistics per column: floor / ceil neighbours of the three quantiles
constexpr int kStBins = 20;        // np.histogram bins (get_df_stats' default_num_bins)
constexpr int kStDigit = 11;
constexpr int kStRadix = 1 << kStDigit;
constexpr int kStThreads = 256;
constexpr int kStChunk = 65536;    // rows per work item

struct StatCol {
  int32_t kind;
  int32_t slot;       // first result slot (unused for SK_ROW)
  int32_t hist;       // 0: no histogram, 1: float32 bins, 2: float64 bins
  int32_t key_bits;   // 32 or 64
  int32_t centre;     // pass 1 adds (x - mean)^2
  int32_t pad_;
  double mean;
  double h_first, h_den;       // np.histogram's first_edge and last_edge - first_edge, in the bin dtype
  double edges[kStBins + 1];   // np.linspace(first_edge, last_edge, 21) in the bin dtype
};

// per column, accumulated with atomics (integers) or combined in item order (doubles)
struct StatAcc {
  unsigned long long count, missing, ones, flags;  // flags: 1 +inf, 2 -inf
  unsigned long long kmax, kmin_inv;               // max key, max of ~key
  unsigned long long first;                        // raw bits of row 0 (sign-extended for int32 kinds)
  unsigned long long first_missing;
  double sum, m2;
  unsigned long long hist[kStBins];
};

// radix-select state of one (column, rank)
struct StatSel {
  long long rank[kStRanks];            // remaining rank inside the current prefix; -1: inactive
  unsigned long long prefix[kStRanks]; // key bits decided so far
  int32_t src[kStRanks];               // slot whose digit histogram serves this rank (shared prefixes)
};

struct StatParams {
  const char* base;          // result slots: slot s at base + s * stride
  int64_t stride;
  int64_t n_rows;
  int64_t n_chunks;
  const StatCol* cols;
  StatAcc* acc;
  StatSel* sel;
  const int32_t* list;       // columns of this pass
  int32_t n_list;
  int32_t pass;
  unsigned int* digits;      // [n_cols][kStRanks][kStRadix]
  double* part;              // [n_cols][n_chunks] fp64 partial sums of this pass
};

__device__ __forceinline__ void st_digit(int key_bits, int pass, int& shift, int& width) {
  const int hi = key_bits - kStDigit * pass;  // bits not yet decided
  shift = hi > kStDigit ? hi - kStDigit : 0;
  width = hi - shift;
}

}  // namespace b2s
