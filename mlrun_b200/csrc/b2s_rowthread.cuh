// b2s_rowthread.cuh -- linear path: row slices per thread, every table operand in the constant bank.
//
//   HBM rows --cp.async 16 B (LDGSTS), STAGES-deep ring--> shared-memory tile, pitch = 16 mod 128 bytes
//   TPR threads share one event row: thread (q, r) -- q = tid / tile_rows, so a warp is uniform in q --
//   owns the 16-byte chunks [q*NCH/TPR, (q+1)*NCH/TPR) of row r, read with conflict-free LDS.128.
//   The column loop is fully unrolled and its per-column operands (Imputer fill, copy mask, the NS fp64
//   weights) are constant-bank operands: the plan's tables travel as a __grid_constant__ kernel
//   parameter, so the inner loop has no table loads and no cross-lane traffic:
//        FSETP+FSEL (NaN -> fill)   LOP3 (drop non-copied columns)   F2F   NS x DFMA     per value
//   one-hot columns: "onehot(x) . w" is the gather w[cat_base + index_of(x)] -- the value is re-read from
//   the tile, the category index comes from compares against constant-bank categories, the weights
//   from shared memory (a zero row stands for "no category matched"); the row is never expanded.
//   The TPR partial sums of a row are combined in shared memory in a fixed order (deterministic fp64);
//   bias, link, vote and the coalesced 4-byte store are done by the row's q = 0 thread.  A non-finite
//   model input surfaces as a non-finite score (NaN/Inf survive fma even with a zero weight), which is
//   what the per-row status tests.
#pragma once
#include <cuda.h>  // CUtensorMap (type only; the encoder is resolved at run time by the host)
#include <type_traits>

#include "b2s_device.cuh"
#include "b2s_hash.cuh"

namespace b2s {

constexpr int kRTMaxCatCols = 16;
constexpr int kRTCatsInline = 4;   // categories compared as constant operands
constexpr int kRTMaxCats = 256;

template <int NCH, int NS>
struct RTParams {
  const char* rows;
  int64_t row_stride;
  int64_t n_rows;
  float* out;
  int32_t* status;
  int32_t n_in, out_cols, n_models, vote_kind, out_is_int, fast_epilogue, tile_rows, pitch, stages, vec_ok;
  int32_t n_cat_cols, n_cat;
  int32_t one_sync;  // single-barrier tile loop (tensor-map loader, TPR > 1)
  int32_t use_bulk;  // tile rows are fetched with cp.async.bulk (TMA, 1-D) + mbarrier instead of LDGSTS
  float* peers[8];   // ensemble-merge targets (see KParams)
  int64_t peer_off;
  int32_t n_peers;
  MergeSig sig;      // completion signal of the merge (b2s_device.cuh)
  const double* wcat;       // [n_cat][NS] (global; copied to shared memory, plus a zero row)
  const double* vote_w_g;   // generic epilogue
  const ModelDesc* models;
  const int32_t* classes;
  double w[NCH * 4][NS];    // constant-bank operands
  // Imputer + "column is not a model input" in one compare/select:  x = !(|x| <= lim[c]) ? fill[c] : x
  //   model input, imputed:      lim = +Inf, fill = the Imputer value (only NaN fails the compare)
  //   model input, not imputed:  lim = +Inf, fill = NaN
  //   one-hot source / dropped:  lim = -1,   fill = +0   (every value is replaced, so Inf * 0 cannot appear)
  float fill[NCH * 4];
  float lim[NCH * 4];
  double bias[NS];
  double vote_w[NS];
  int32_t cat_col[kRTMaxCatCols];   // input column of each categorical column
  int32_t cat_off[kRTMaxCatCols];   // where the column's word sits in a tile row (Row::at2; per launch)
  int32_t cat_sw[kRTMaxCatCols];
  int32_t cat_base[kRTMaxCatCols];  // first category (index into cat_val / wcat)
  int32_t cat_cnt[kRTMaxCatCols];
  float cat_fill[kRTMaxCatCols];
  float cat_inl[kRTMaxCatCols][kRTCatsInline];  // first categories, NaN padded (never match)
  int32_t cat_first[kRTMaxCatCols];  // dense columns: the categories are the integers first, first+1, ...
  int32_t cat_dense[kRTMaxCatCols];
  float cat_val[kRTMaxCats];
  // fused enrichment (per-row bulk loader only): tile rows are fetched from an online table by entity key instead of
  // from `rows` (b2s_table.cu).  Kept at the end: the offsets of everything above are those of the plain kernels.
  // fast one-hot path (every categorical column has consecutive integer codes): the constants of a column packed so that
  // two 16-byte constant loads fetch them; byte offsets, so that the address of a weight row is one shift-add
  struct CatFast {
    int32_t off_b;    // byte offset of the column's word in a tile row (per launch, like cat_off)
    int32_t sw_b;     // swizzle term in bytes (tensor-map tiles), 0 otherwise
    int32_t first;    // first category code
    int32_t cnt;      // number of categories
    int32_t woff_b;   // byte offset of the first category's weight row in s_wcat
    float fill;       // Imputer value of the column (NaN: not imputed)
    int32_t pad[2];
  };
  CatFast catf[kRTMaxCatCols];
  int32_t cats_fast;   // 1: catf describes every categorical column
  int32_t zero_woff_b; // byte offset of the all-zero weight row ("no category matched")
  int32_t dead_tail;   // trailing 16-byte chunks without a model-input column (one-hot sources at the end of the row):
                       // the dot products run over the live chunks only (0, 2 or 4 chunks skipped; see rt_row_slices)
  int32_t pad_fast;
  const long long* g_keys;     // [n_rows]; null = rows come from `rows`
  const TableSlot* g_slots;
  uint64_t g_mask;
  const float* g_values;       // [n_keys + 1][n_in]; row n_keys is all NaN and stands for an unknown key
  long long g_missing_row;
};

// how a thread finds the 16-byte chunks of its row inside the shared-memory tile
struct RowPadded {  // LDGSTS / per-row bulk copies: rows `pitch` words apart (pitch = 16 mod 128 bytes)
  const float* xr;
  __device__ __forceinline__ float4 chunk(int ch) const { return *reinterpret_cast<const float4*>(xr + ch * 4); }
  __device__ __forceinline__ float at2(int off, int) const { return xr[off]; }
  __device__ __forceinline__ float at_b(int off_b, int) const { return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(xr) + off_b); }
};
struct RowSwizzled {  // 2-D TMA boxes of 32 floats x TR rows, SWIZZLE_128B: chunk j of row r sits at j ^ (r & 7)
  const float* box0;  // row r of box 0
  int box_words;      // TR * 32
  int r7s;            // (r & 7) << 2, in floats
  __device__ __forceinline__ float4 chunk(int ch) const {
    return *reinterpret_cast<const float4*>(box0 + (ch >> 3) * box_words + (((ch & 7) << 2) ^ r7s));
  }
  // off = (ch >> 3) * box_words + (col & 3), sw = (ch & 7) << 2 with ch = col >> 2 (set per launch by the host)
  __device__ __forceinline__ float at2(int off, int sw) const { return box0[off + (sw ^ r7s)]; }
  __device__ __forceinline__ float at_b(int off_b, int sw_b) const {
    return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(box0) + off_b + (sw_b ^ (r7s << 2)));
  }
};

// dot products of the chunks [CH0, CH1) of a row with all NS weight columns (the weights, fills and limits
// are constant-bank / uniform-register operands)
template <int NCH, int NS, int CH0, int CH1, typename Row>
__device__ __forceinline__ void rt_slice(const RTParams<NCH, NS>& p, const Row& xr, double (&acc)[NS]) {
  constexpr int BATCH = 4;  // chunks converted before their DFMAs are issued (ILP)
#pragma unroll
  for (int b = CH0; b < CH1; b += BATCH) {
    double xd[BATCH * 4];
#pragma unroll
    for (int cb = 0; cb < BATCH; ++cb) {
      const int ch = b + cb;
      if (ch < CH1) {
        const float4 v = xr.chunk(ch);
        const float xs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = ch * 4 + u;
          float x = xs[u];
          x = !(fabsf(x) <= p.lim[c]) ? p.fill[c] : x;  // Imputer / non-input -> +0 (see RTParams)
          xd[cb * 4 + u] = (double)x;
        }
      }
    }
#pragma unroll
    for (int cb = 0; cb < BATCH; ++cb) {
      const int ch = b + cb;
      if (ch < CH1) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = ch * 4 + u;
#pragma unroll
          for (int k = 0; k < NS; ++k) acc[k] = fma(p.w[c][k], xd[cb * 4 + u], acc[k]);
        }
      }
    }
  }
}

// category search for a column whose categories are not consecutive integers (kept out of line: rare)
template <int NCH, int NS>
__device__ __noinline__ int rt_cat_search(const RTParams<NCH, NS>& p, int cc, float x) {
  const int b0 = p.cat_base[cc], cnt = p.cat_cnt[cc];
  int j = p.n_cat;
  if (cnt <= kRTCatsInline) {
#pragma unroll
    for (int qq = kRTCatsInline - 1; qq >= 0; --qq) j = (x == p.cat_inl[cc][qq]) ? b0 + qq : j;
  } else {
    for (int qq = cnt - 1; qq >= 0; --qq) j = (x == p.cat_val[b0 + qq]) ? b0 + qq : j;
  }
  return j;
}

// one-hot columns Q0, Q0+TPR, ... of one row: "onehot(x) . w" is a gather from the shared-memory weight rows.
// Fully unrolled with literal column slots (the caller's branch on the slice index is warp-uniform), so every
// table entry is a constant-bank operand and the address arithmetic stays in the uniform datapath.
template <int NCH, int NS, int Q0, int TPR, typename Row>
__device__ __forceinline__ void rt_cats(const RTParams<NCH, NS>& p, const Row& xr, const double* __restrict__ s_wcat,
                                        double (&acc)[NS]) {
  constexpr int ITERS = (kRTMaxCatCols - Q0 + TPR - 1) / TPR;
  if (p.cats_fast) {  // integer codes first .. first + cnt - 1 in every column: no search, no per-column branch
    const char* wb = reinterpret_cast<const char*>(s_wcat);
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
      const int cc = Q0 + it * TPR;
      if (cc >= p.n_cat_cols) break;
      const typename RTParams<NCH, NS>::CatFast cf = p.catf[cc];
      float x = xr.at_b(cf.off_b, cf.sw_b);
      x = (x != x) ? cf.fill : x;
      const int v = __float2int_rz(x);  // saturating; NaN -> 0 and fails the equality below
      const unsigned jj = (unsigned)(v - cf.first);
      const bool miss = ((float)v != x) | (jj >= (unsigned)cf.cnt);
      const int a = miss ? p.zero_woff_b : cf.woff_b + (int)jj * (NS * 8);
      if constexpr (NS % 2 == 0) {  // weight rows are 16-byte aligned: LDS.128
#pragma unroll
        for (int k = 0; k < NS; k += 2) {
          const double2 w2 = *reinterpret_cast<const double2*>(wb + a + k * 8);
          acc[k] += w2.x;
          acc[k + 1] += w2.y;
        }
      } else {
        const double* wc = reinterpret_cast<const double*>(wb + a);
#pragma unroll
        for (int k = 0; k < NS; ++k) acc[k] += wc[k];
      }
    }
    return;
  }
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int cc = Q0 + it * TPR;
    if (cc >= p.n_cat_cols) break;
    float x = xr.at2(p.cat_off[cc], p.cat_sw[cc]);
    x = (x != x) ? p.cat_fill[cc] : x;
    int j;
    if (p.cat_dense[cc]) {  // integer codes first, first+1, ...: the index is a conversion
      const int v = __float2int_rz(x);  // saturating; NaN -> 0 and fails the equality below
      const unsigned jj = (unsigned)(v - p.cat_first[cc]);
      j = ((float)v == x && jj < (unsigned)p.cat_cnt[cc]) ? p.cat_base[cc] + (int)jj : p.n_cat;  // n_cat: the zero row
    } else {
      j = rt_cat_search(p, cc, x);
    }
    const double* wc = s_wcat + (size_t)j * NS;
#pragma unroll
    for (int k = 0; k < NS; ++k) acc[k] += wc[k];
  }
}

// slice q of a row: the dot products over its share of the LIVE leading chunks + its share of the one-hot columns.
// The slice index is warp-uniform; each case has compile-time column indices (constant operands); the row's one-hot
// columns are dealt round-robin to its threads.
template <int NCH, int NS, int TPR, int LIVE, typename Row>
__device__ __forceinline__ void rt_row_slices(const RTParams<NCH, NS>& p, int q, const Row& xr, const double* __restrict__ s_wcat,
                                              double (&acc)[NS]) {
  static_assert(LIVE % TPR == 0, "live chunks must split evenly over the row's threads");
  constexpr int CPT = LIVE / TPR;
  if (TPR == 1 || q == 0) {
    rt_slice<NCH, NS, 0, CPT>(p, xr, acc);
    rt_cats<NCH, NS, 0, TPR>(p, xr, s_wcat, acc);
  } else if (q == 1) {
    rt_slice<NCH, NS, (TPR > 1 ? CPT : 0), (TPR > 1 ? 2 * CPT : 0)>(p, xr, acc);
    rt_cats<NCH, NS, (TPR > 1 ? 1 : 0), TPR>(p, xr, s_wcat, acc);
  } else if (q == 2) {
    rt_slice<NCH, NS, (TPR > 2 ? 2 * CPT : 0), (TPR > 2 ? 3 * CPT : 0)>(p, xr, acc);
    rt_cats<NCH, NS, (TPR > 2 ? 2 : 0), TPR>(p, xr, s_wcat, acc);
  } else {
    rt_slice<NCH, NS, (TPR > 3 ? 3 * CPT : 0), (TPR > 3 ? 4 * CPT : 0)>(p, xr, acc);
    rt_cats<NCH, NS, (TPR > 3 ? 3 : 0), TPR>(p, xr, s_wcat, acc);
  }
}

// ---- TMA (bulk async copy) + mbarrier helpers: one 1-D bulk copy per event row lands in the padded tile
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(a), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}

__device__ __forceinline__ void tensor_load_2d(void* smem_dst, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          (uint32_t)__cvta_generic_to_shared(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"((uint32_t)__cvta_generic_to_shared(bar))
      : "memory");
}

// classifier links / majority vote / integer outputs: the generic per-row epilogue (out of line)
template <int NCH, int NS>
__device__ __noinline__ void rt_generic_epilogue(const RTParams<NCH, NS>& p, const double* sl, int64_t row, uint32_t st) {
  double pred[kMaxModels];
  for (int m = 0; m < p.n_models; ++m) {
    const ModelDesc md = p.models[m];
    pred[m] = apply_link(md, sl + md.score_off, p.classes);
  }
  KParams kp;  // vote_and_store only reads these fields
  kp.out = p.out;
  kp.out_cols = p.out_cols;
  kp.n_models = p.n_models;
  kp.vote_kind = p.vote_kind;
  kp.out_is_int = p.out_is_int;
  kp.vote_w = p.vote_w_g;
  kp.status = p.status;
  kp.n_peers = p.n_peers;
  kp.peer_off = p.peer_off;
  for (int g = 0; g < p.n_peers; ++g) kp.peers[g] = p.peers[g];
  vote_and_store(kp, pred, row, st);
}

// LM: how tiles reach shared memory -- 0 LDGSTS (cp.async), 1 one TMA bulk copy per row, 2 TMA tensor-map boxes (swizzled)
template <int NCH, int NS, int TPR, int LM>
__global__ void __launch_bounds__(128 * TPR, TPR == 2 ? 3 : 4)
    rowthread_kernel(const __grid_constant__ RTParams<NCH, NS> p, const __grid_constant__ CUtensorMap tmap) {
  static_assert(NCH % TPR == 0, "chunks must split evenly over the row's threads");
  constexpr int CPT = NCH / TPR;  // chunks per thread
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem);  // 4 mbarriers (bulk variant); 64 bytes reserved
  double* s_wcat = reinterpret_cast<double*>(smem + 64);
  const size_t wcat_bytes = 64 + (((size_t)(p.n_cat + 1) * NS * 8 + 15) / 16) * 16;
  // With the tensor-map loader and TPR > 1 the tile loop has ONE barrier per tile (between the partial sums
  // and their combination): that barrier also proves the tile's stage is drained, so the next load into it is
  // issued right there, and the partial sums are double-buffered instead of fenced by a second barrier.
  const bool one_sync = (LM == 2) && TPR > 1 && p.one_sync;
  constexpr size_t part_words = (size_t)(TPR - 1) * 128 * NS;
  double* s_part = reinterpret_cast<double*>(smem + wcat_bytes);  // [one_sync ? 2 : 1][(TPR-1)][128][NS]
  float* s_tiles = reinterpret_cast<float*>(smem + wcat_bytes + (one_sync ? 2 : 1) * part_words * 8);
  if (LM == 2) {  // swizzled TMA boxes need a 1024-byte aligned base (the host reserved the slack)
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(s_tiles);
    s_tiles += ((1024u - (a & 1023u)) & 1023u) >> 2;
  }

  const int tid = threadIdx.x;
  const int TR = p.tile_rows;
  const int S = p.stages;
  const int tile_words = (LM == 2) ? TR * NCH * 4 : TR * p.pitch;
  const int64_t n_tiles = (p.n_rows + TR - 1) / TR;
  const int q = tid / TR;      // slice of the row (warp-uniform: TR is a multiple of 32)
  const int r = tid - q * TR;  // row inside the tile

  // (row, chunk) walk of the tile loader without per-iteration division
  const int cprv = p.vec_ok ? (p.n_in >> 2) : p.n_in;  // units per row: 16-byte chunks or 4-byte words
  const int r0 = tid / cprv, c0 = tid - r0 * cprv;
  const int dr = (int)blockDim.x / cprv, dc = (int)blockDim.x - dr * cprv;
  auto issue = [&](float* tile, int64_t row0) {
    int64_t left = p.n_rows - row0;
    const int rows = left < TR ? (left < 0 ? 0 : (int)left) : TR;
    const char* base = p.rows + row0 * p.row_stride;
    int rr = r0, cc = c0;
    if (p.vec_ok) {
      while (rr < rows) {
        cp_async16(tile + rr * p.pitch + cc * 4, base + (int64_t)rr * p.row_stride + cc * 16);
        rr += dr;
        cc += dc;
        if (cc >= cprv) {
          cc -= cprv;
          ++rr;
        }
      }
    } else {
      while (rr < rows) {
        cp_async4(tile + rr * p.pitch + cc, base + (int64_t)rr * p.row_stride + cc * 4);
        rr += dr;
        cc += dc;
        if (cc >= cprv) {
          cc -= cprv;
          ++rr;
        }
      }
    }
  };

  // bulk (TMA) variant: one mbarrier per stage; row `tid` of the tile is fetched by thread `tid`
  constexpr bool bulk = LM != 0;
  const uint32_t row_bytes = (uint32_t)p.n_in * 4u;
  uint32_t unknown_bits = 0;  // bit s: the key of this thread's row in stage s is not in the table (gather loader)
  // Gather loader, software pipelined.  key -> slot -> row are three dependent DRAM reads (random over a table far larger
  // than the TLB reach); done back to back they stall the thread -- which also computes -- for ~2 us per tile.  The loader
  // is called for this CTA's tiles in order (T_j = blockIdx + j * grid), so every hop runs one call ahead of its consumer:
  // call j finishes the slot probe started in call j - 1 and issues the row copy of T_j, starts the probe of T_{j+1}
  // (its key was loaded in call j - 1) and loads the key of T_{j+2}.  Each load has a whole tile of compute to land.
  long long gk_cur = 0, gk_nxt = 0;  // keys of T_j and T_{j+1} (thread tid: row tid of the tile)
  longlong2 g_slot = make_longlong2(0, -1);
  uint64_t g_hash = 0;
  int64_t g_tile_nxt = 0;
  auto g_key = [&](int64_t tile) -> long long {
    const int64_t row = tile * TR + tid;
    return row < p.n_rows ? __ldg(p.g_keys + row) : 0;
  };
  auto g_probe_start = [&](long long key) {
    g_hash = mix64((uint64_t)key) & p.g_mask;
    g_slot = __ldg(reinterpret_cast<const longlong2*>(p.g_slots) + g_hash);
  };
  auto g_probe_finish = [&](long long key) -> long long {  // the first slot decides for most keys (load factor <= 0.5)
    uint64_t h = g_hash;
    longlong2 sl = g_slot;
    for (;;) {
      if (sl.y < 0) return -1;
      if (sl.x == key) return sl.y;
      h = (h + 1) & p.g_mask;
      sl = __ldg(reinterpret_cast<const longlong2*>(p.g_slots) + h);
    }
  };
  if (LM == 1 && p.g_keys && tid < TR) {
    gk_cur = g_key(blockIdx.x);
    gk_nxt = g_key((int64_t)blockIdx.x + gridDim.x);
    g_probe_start(gk_cur);
    g_tile_nxt = (int64_t)blockIdx.x + 2 * (int64_t)gridDim.x;
  }
  auto issue_bulk = [&](int st, int64_t row0) {
    int64_t left = p.n_rows - row0;
    const int rows = left < TR ? (left < 0 ? 0 : (int)left) : TR;
    if (LM == 2) {
      // one thread, NCH/8 box copies of (32 floats x TR rows); rows past the end are zero-filled by the TMA unit
      if (tid == 0) {
        if (rows > 0) {
          mbar_expect_tx(&s_bar[st], (uint32_t)(NCH / 8) * (uint32_t)TR * 128u);
#pragma unroll
          for (int b = 0; b < NCH / 8; ++b)
            tensor_load_2d(s_tiles + st * tile_words + b * TR * 32, &tmap, b * 32, (int)row0, &s_bar[st]);
        } else {
          mbar_expect_tx(&s_bar[st], 0);
        }
      }
    } else {
      if (tid == 0) mbar_expect_tx(&s_bar[st], (uint32_t)rows * row_bytes);
      if (p.g_keys) {
        if (tid < TR) {  // thread tid is also the q = 0 thread of tile row tid: it keeps the "unknown key" flag for the epilogue
          const long long hit = g_probe_finish(gk_cur);
          if (tid < rows) {
            unknown_bits = (unknown_bits & ~(1u << st)) | ((hit < 0 ? 1u : 0u) << st);
            bulk_load(s_tiles + st * tile_words + tid * p.pitch,
                      reinterpret_cast<const char*>(p.g_values + (hit < 0 ? p.g_missing_row : hit) * p.n_in), row_bytes, &s_bar[st]);
          }
          gk_cur = gk_nxt;
          g_probe_start(gk_cur);        // consumed by the next call
          gk_nxt = g_key(g_tile_nxt);   // consumed by the call after that
          g_tile_nxt += gridDim.x;
        }
      } else if (tid < rows) {
        bulk_load(s_tiles + st * tile_words + tid * p.pitch, p.rows + (row0 + tid) * p.row_stride, row_bytes, &s_bar[st]);
      }
    }
  };
  if (bulk) {
    if (tid == 0) {
      for (int s = 0; s < S; ++s) mbar_init(&s_bar[s], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  for (int s = 0; s < (one_sync ? S : S - 1); ++s) {
    const int64_t t = (int64_t)blockIdx.x + (int64_t)s * gridDim.x;
    if (bulk) {
      issue_bulk(s, t * TR);
    } else {
      if (t < n_tiles) issue(s_tiles + s * tile_words, t * TR);
      cp_async_commit();
    }
  }
  uint32_t phase_bits = 0;  // bit s: parity to wait for on stage s
  for (int i = tid; i < p.n_cat * NS; i += blockDim.x) s_wcat[i] = p.wcat[i];
  for (int i = tid; i < NS; i += blockDim.x) s_wcat[p.n_cat * NS + i] = 0.0;
  if (one_sync) __syncthreads();  // the weight rows are read before the loop's first barrier

  int stage = 0;
  uint32_t iter = 0;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    if (bulk) {
      mbar_wait(&s_bar[stage], (phase_bits >> stage) & 1u);
      phase_bits ^= (1u << stage);
    } else if (S == 2) cp_async_wait<0>();
    else if (S == 3) cp_async_wait<1>();
    else cp_async_wait<2>();
    if (!one_sync) {
      __syncthreads();  // tile visible to everybody; everybody is done with the previous tile and s_part
      const int64_t tn = t + (int64_t)(S - 1) * gridDim.x;
      int sn = stage + S - 1;
      if (sn >= S) sn -= S;
      if (bulk) {
        issue_bulk(sn, tn * TR);  // rows = 0 past the end: the barrier completes on the arrive alone
      } else {
        if (tn < n_tiles) issue(s_tiles + sn * tile_words, tn * TR);
        cp_async_commit();
      }
    }
    const float* tile = s_tiles + stage * tile_words;
    const int64_t row0 = t * TR;                                                       // uniform
    const int live_rows = (int)(p.n_rows - row0 < (int64_t)TR ? p.n_rows - row0 : (int64_t)TR);  // uniform: rows of this tile
    const bool any_live = r < live_rows;  // rows past the end were zero-filled (TMA) or are skipped
    using Row = typename std::conditional<LM == 2, RowSwizzled, RowPadded>::type;
    Row xr;
    if constexpr (LM == 2) {
      xr.box0 = tile + r * 32;
      xr.box_words = TR * 32;
      xr.r7s = (r & 7) << 2;
    } else {
      xr.xr = tile + r * p.pitch;
    }
    double acc[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) acc[k] = 0.0;
    if (any_live) {
      // trailing chunks without a model input are not multiplied at all: the live chunks are split evenly over the row's
      // threads (a uniform branch picks the fully unrolled version for 0, 2 or 4 skipped chunks)
      if constexpr (LM == 2 && NCH >= 8 && (TPR == 1 || TPR == 2)) {  // (the tensor-map variants only: build time)
        if (p.dead_tail >= 4) rt_row_slices<NCH, NS, TPR, NCH - 4>(p, q, xr, s_wcat, acc);
        else if (p.dead_tail >= 2) rt_row_slices<NCH, NS, TPR, NCH - 2>(p, q, xr, s_wcat, acc);
        else rt_row_slices<NCH, NS, TPR, NCH>(p, q, xr, s_wcat, acc);
      } else {
        rt_row_slices<NCH, NS, TPR, NCH>(p, q, xr, s_wcat, acc);
      }
    }
    if (TPR > 1) {  // combine the row's slices in a fixed order (deterministic fp64 sum)
      double* s_part_cur = s_part + (one_sync ? (size_t)(iter & 1) * part_words : 0);
      if (q > 0) {
        double* part = s_part_cur + ((size_t)(q - 1) * 128 + r) * NS;
#pragma unroll
        for (int k = 0; k < NS; ++k) part[k] = acc[k];
      }
      __syncthreads();
      if (one_sync) issue_bulk(stage, (t + (int64_t)S * gridDim.x) * TR);  // every read of this stage is behind the barrier
      if (q == 0) {
#pragma unroll
        for (int qq = 1; qq < TPR; ++qq) {
          const double* o = s_part_cur + ((size_t)(qq - 1) * 128 + r) * NS;
#pragma unroll
          for (int k = 0; k < NS; ++k) acc[k] += o[k];
        }
      }
    }
    const int64_t row = row0 + r;
    if (q == 0 && r < live_rows) {
      uint32_t st = 0;
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        acc[k] += p.bias[k];
        st |= (fabs(acc[k]) <= 1.7976931348623157e308) ? 0u : 1u;
      }
      if (LM == 1) st |= ((unknown_bits >> stage) & 1u) << 2;  // B2S_ROW_UNKNOWN_KEY
      if (p.fast_epilogue) {
        if (p.vote_kind == 1) {  // VotingEnsemble._mean_vote: sum_m w[m] * pred[m], model order
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < NS; ++k) s = __dadd_rn(s, __dmul_rn(acc[k], p.vote_w[k]));
          store_word(p, row, 0, __float_as_uint((float)s));
        } else {
#pragma unroll
          for (int k = 0; k < NS; ++k)
            if (k < p.n_models) store_word(p, row, k, __float_as_uint((float)acc[k]));
        }
        if (p.status) p.status[row] = (int32_t)st;
      } else {
        double sl[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) sl[k] = acc[k];
        rt_generic_epilogue(p, sl, row, st);
      }
    }
    ++stage;
    ++iter;
    if (stage == S) stage = 0;
  }
  cp_async_wait<0>();
  merge_signal(p.sig);
}

}  // namespace b2s
