// b2s_trees3.cuh -- tree-ensemble scorer, round 2 (sm_100a): "parts" resident in shared memory.
//
// What bounds a root->leaf walk (measured on B200, profiles/r2/trees_lab_r2a*.{txt,csv}): with the model in shared memory
// and the event tile transposed (xt[feature][row], lanes = 32 consecutive rows walking the same tree) every LDS is
// conflict free, and the kernel runs exactly at the LSU limit of one 128-byte shared-memory wavefront per cycle and
// SM -- issue slots are 35-40 % busy.  So the design minimises *wavefronts per visit* and keeps the LSU queue full:
//   * 8-byte heap nodes {x offset, threshold}: one LDS.64 (2 wavefronts, same as 2 x LDS.32, one instruction fewer);
//   * the top two levels of every tree are read once per tree with warp-uniform loads (one broadcast wavefront each)
//     and kept in registers for the warp's RPT row blocks: levels 0-1 cost only their x gathers;
//   * node addresses are carried as absolute shared-window addresses, a' = 2a + ((right ? 8 : 0) - tree_base): a visit is
//     LDS.64, IADD, LDS, FSETP, SEL, IADD3;
//   * nothing but walks runs on the LSU of the walking kernel: the transpose is a kernel of its own (below), tiles arrive
//     by TMA bulk copies, and the only synchronisation is two mbarriers per tile buffer (no CTA-wide barrier).
//   (Rounds of this file that transposed inside the walking CTA -- in phases, then with producer warps -- lost 35-40 % of
//   the LSU cycles to barrier stalls and to loads of the producers queueing behind the walkers': profiles/r2/.)
//
// Three launches per batch:
//   t3_prep_kernel   rows (row-major, HBM) -> TMA boxes / cp.async -> transpose in shared memory (+ Imputer, + the non-finite
//                    test -> row flags, + order-preserving integer keys when NaN routing is on) -> xt tiles in HBM,
//                    [tile][feature][64 rows].  HBM bound, once per batch whatever the number of parts.
//   trees3_kernel    a *part* is what one CTA keeps resident: the trees of one (model, score slot) -- split further when they
//                    do not fit -- re-packed on the host as complete heap-ordered depth-D trees (early leaves are padded: +inf
//                    threshold, both children carry the leaf), or ALL linear models of the ensemble (fp64 weights).  Parts own
//                    CTAs in proportion to their cost; a CTA streams the tiles rank, rank + n_ctas, ... : one 1-D bulk copy per
//                    tile into a two-deep ring; warp g walks the trees g, g + W, ... for the tile's 64 rows; per-warp partial
//                    sums are combined in a fixed order by two service warps -> partial[column][row] (fp64, coalesced).
//   t3_vote_kernel   adds each model's columns to its init scores in column order, applies the link and the VotingEnsemble
//                    reduce (serving/routers.py:708-741), stores the votes (to every merge target when sharded).
// Multi-class GradientBoosting (n_classes x n_estimators trees) and ensembles mixing linear and tree scorers (BASELINE
// configs[3]) run on this path too.
//
// Missing values (xgboost / LightGBM / scikit-learn >= 1.3 trees route NaN to a per-node default child): with MISS the
// tiles hold order-preserving int32 keys (NaN = INT_MAX), a node's x offset carries its default direction d in bit 31 and
// its threshold key is stored as key + d; the walk tests key(x) + d > key(t) + d, and INT_MAX + 1 wraps to INT_MIN exactly
// when a missing value must go left.  `x < t` (xgboost) is `x <= prev(t)`: thresholds are converted when the model is
// added, not in the kernel.
#pragma once
#include "b2s_device.cuh"

namespace b2s {

constexpr int kT3RPT = 2;            // row blocks (of 32 rows) per warp: the tile is 64 rows
constexpr int kT3TR = 32 * kT3RPT;   // rows per tile
constexpr int kT3U = 2;              // trees in flight per warp (x RPT rows = 4 independent walks per thread)
constexpr int kT3MaxLin = 8;         // score columns of the linear part
constexpr int kT3MaxDepth = 8;
constexpr int kT3Service = 2;        // service warps of the walking kernel: combine the partial sums, issue the tile copies
constexpr int kT3MaxWalk = 28;       // walking warps at most
constexpr int kT3PrepThreads = 256;

struct T3Part {           // one per part, in global memory
  const uint2* nodes;     // trees: [n_trees][1 << D] heap nodes (slot 0 unused) {x byte offset in the tile, threshold bits}
  const double* leaves;   // trees: [n_trees][1 << D] tree_scale * leaf value;  linear part: weights [n_cols][n_in]
  int32_t n_trees;        // 0: the linear part
  int32_t n_cols;         // columns of `partial` this part writes (trees: 1)
  int32_t col0;
  int32_t cta0, n_ctas;   // the CTAs [cta0, cta0 + n_ctas) of the grid work on this part
};

struct T3Prep {           // t3_prep_kernel
  const char* rows;
  int64_t row_stride;
  int64_t n_rows;
  uint32_t* xt;           // [n_tiles][n_in4][TR] words
  int32_t* row_bad;       // [n_rows]
  const float* fill;      // [n_in] Imputer values (NaN: column not imputed)
  int32_t n_in, n_in4, use_tmap, vec_ok, pitch, any_fill;
  int32_t sm_xt, sm_land, sm_fill, sm_bad, sm_bar;  // byte offsets into dynamic shared memory
};

struct T3Params {         // trees3_kernel
  const uint32_t* xt;     // the prepared tiles
  int64_t n_rows;
  double* partial;        // [n_cols_total][col_stride]
  int64_t col_stride;
  const T3Part* parts;
  int32_t n_in, n_parts, warps;  // warps: walking warps (the CTA has kT3Service more)
  int32_t xt_words;              // words of one tile (n_in rounded up to 4, times TR); two tiles are resident
  int32_t part_words;            // doubles of one partial-sum buffer; two are resident
  int32_t sm_leaf, sm_part, sm_xt, sm_bar;  // byte offsets into dynamic shared memory
  // the linear part: walking warp s < lin_slices takes the feature slice s of every score column; its partial sums live where
  // the tree parts keep their tables (two buffers of lin_part_words doubles at sm_lin_part)
  int32_t lin_slices, lin_part_words, sm_lin_part;
};

// launchers (b2s_trees3.cu: the kernels are compiled in their own translation unit)
cudaError_t t3_launch_prep(const T3Prep& pr, const CUtensorMap& tmap, bool miss, int grid, int smem, int smem_optin, cudaStream_t st);
cudaError_t t3_launch_walk(const T3Params& t, int depth, bool miss, int grid, int block, int smem, int smem_optin, cudaStream_t st);
cudaError_t t3_launch_vote(const KParams& k, const double* partial, int64_t col_stride, const int32_t* col_score, int n_cols,
                           const int32_t* row_bad, int grid, cudaStream_t st);

#ifdef B2S_T3_KERNELS
// explicit shared-window loads (32-bit addresses: no generic->shared conversion in the address arithmetic)
__device__ __forceinline__ uint2 t3_lds64(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ uint4 t3_lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
template <int OFF>
__device__ __forceinline__ uint32_t t3_lds32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF));
  return v;
}
__device__ __forceinline__ double t3_ldsd(uint32_t a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void t3_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}

// order-preserving int32 key of a float (monotone for every non-NaN value; -0 and +0 share a key)
__device__ __forceinline__ int32_t t3_key(float x) {
  const int32_t b = __float_as_int(x + 0.0f);  // -0 -> +0
  return b ^ ((b >> 31) & 0x7fffffff);
}

template <bool MISS>
__device__ __forceinline__ uint32_t t3_xoff(uint32_t foff) { return MISS ? (foff & 0x7fffffffu) : foff; }
template <bool MISS>
__device__ __forceinline__ bool t3_right(uint32_t x, uint2 nd) {
  // floats: sklearn's rule "left when x <= threshold"; keys: the same order on integers, shifted by the node's default bit
  return MISS ? ((int32_t)(x + (nd.x >> 31)) > (int32_t)nd.y) : !(__uint_as_float(x) <= __uint_as_float(nd.y));
}

// ------------------------------------------------------------------------------------------ prepare: transpose once per batch
template <bool MISS>
__global__ void __launch_bounds__(kT3PrepThreads) t3_prep_kernel(const __grid_constant__ T3Prep p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) unsigned char smem_prep[];
  unsigned char* const smem = smem_prep;
  constexpr int TR = kT3TR;
  const int tid = threadIdx.x, nthr = kT3PrepThreads;
  uint32_t* s_xt = reinterpret_cast<uint32_t*>(smem + p.sm_xt);
  float* s_land = reinterpret_cast<float*>(smem + p.sm_land);  // 1024-byte aligned (TMA swizzle atom)
  float* s_fill = reinterpret_cast<float*>(smem + p.sm_fill);
  int* s_bad = reinterpret_cast<int*>(smem + p.sm_bad);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + p.sm_bar);
  for (int i = tid; i < p.n_in; i += nthr) s_fill[i] = p.fill[i];
  if (tid < TR) s_bad[tid] = 0;
  const bool tma = p.use_tmap != 0;
  if (tma && tid == 0) {
    mbar_init(s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t tma_phase = 0;
  const int64_t n_tiles = (p.n_rows + TR - 1) / TR;
  const int cprv = p.vec_ok ? (p.n_in >> 2) : p.n_in;
  auto issue = [&](int64_t row0) {
    if (tma) {  // one thread: n_in / 32 box copies of (32 floats x TR rows); rows past the end arrive as zeros
      if (tid == 0) {
        const int boxes = p.n_in >> 5;
        mbar_expect_tx(s_bar, (uint32_t)boxes * (uint32_t)TR * 128u);
        for (int b = 0; b < boxes; ++b) tensor_load_2d(s_land + b * TR * 32, &tmap, b * 32, (int)row0, s_bar);
      }
      return;
    }
    const int64_t left = p.n_rows - row0;
    const int rows = left < TR ? (left < 0 ? 0 : (int)left) : TR;
    const char* base = p.rows + row0 * p.row_stride;
    for (int i = tid; i < rows * cprv; i += nthr) {
      const int rr = i / cprv, cc = i - rr * cprv;
      if (p.vec_ok)
        cp_async16(s_land + rr * p.pitch + cc * 4, base + (int64_t)rr * p.row_stride + cc * 16);
      else
        cp_async4(s_land + rr * p.pitch + cc, base + (int64_t)rr * p.row_stride + cc * 4);
    }
  };
  if ((int64_t)blockIdx.x < n_tiles) issue((int64_t)blockIdx.x * TR);
  cp_async_commit();
  const int tile_words = p.n_in4 * TR;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t row0 = t * TR;
    if (tma) {
      mbar_wait(s_bar, tma_phase);
      tma_phase ^= 1u;
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();  // landing tile visible; the previous tile has been written out (s_xt, s_bad are free)
    const int64_t left = p.n_rows - row0;
    const int rows = left < TR ? (int)left : TR;
    // ---- transpose: lanes take consecutive rows, LDS.128 (swizzled / padded) and STS are conflict free
    if (p.vec_ok) {
      constexpr int PU = 4;  // chunks in flight per thread
      const int n_chunks = (p.n_in >> 2) * TR;
      for (int i0 = tid; i0 < n_chunks; i0 += nthr * PU) {
        float4 v[PU];
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          const int i = i0 + u * nthr;
          const int c = i / TR, rr = i - c * TR;
          v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (i < n_chunks && rr < rows)
            v[u] = tma ? *reinterpret_cast<const float4*>(s_land + (c >> 3) * (TR * 32) + rr * 32 + (((c & 7) ^ (rr & 7)) << 2))
                       : *reinterpret_cast<const float4*>(s_land + rr * p.pitch + c * 4);
        }
#pragma unroll
        for (int u = 0; u < PU; ++u) {
          const int i = i0 + u * nthr;
          if (i >= n_chunks) break;
          const int c = i / TR, rr = i - c * TR;
          float xs[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
          bool bad = false;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x = xs[e];
            if (p.any_fill) {
              const float f = s_fill[c * 4 + e];
              x = (x != x) ? f : x;  // Imputer._impute (feature_store/steps.py:397-406); f is NaN where nothing is imputed
            }
            // what scikit-learn's check_array refuses: Inf always, NaN unless every model routes missing values
            bad |= MISS ? (fabsf(x) == __int_as_float(0x7f800000)) : !is_finite_f(x);
            s_xt[(size_t)(c * 4 + e) * TR + rr] = MISS ? (uint32_t)((x != x) ? 0x7fffffff : t3_key(x)) : __float_as_uint(x);
          }
          if (bad) atomicOr(&s_bad[rr], 1);
        }
      }
    } else {
      for (int i = tid; i < p.n_in4 * TR; i += nthr) {
        const int f = i / TR, rr = i - f * TR;
        float x = (rr < rows && f < p.n_in) ? s_land[rr * p.pitch + f] : 0.0f;
        if (p.any_fill && f < p.n_in) {
          const float fv = s_fill[f];
          x = (x != x) ? fv : x;
        }
        const bool bad = MISS ? (fabsf(x) == __int_as_float(0x7f800000)) : !is_finite_f(x);
        s_xt[i] = MISS ? (uint32_t)((x != x) ? 0x7fffffff : t3_key(x)) : __float_as_uint(x);
        if (bad) atomicOr(&s_bad[rr], 1);
      }
    }
    __syncthreads();  // transposed tile complete; landing tile free
    {
      const int64_t tn = t + gridDim.x;
      if (tn < n_tiles) issue(tn * TR);  // lands while this tile is written out
      cp_async_commit();
    }
    uint4* dst = reinterpret_cast<uint4*>(p.xt + (size_t)t * tile_words);
    const uint4* src = reinterpret_cast<const uint4*>(s_xt);
    for (int i = tid; i < tile_words / 4; i += nthr) dst[i] = src[i];  // coalesced 16-byte stores, 32 KB per tile
    if (tid < TR) {
      if (row0 + tid < p.n_rows) p.row_bad[row0 + tid] = s_bad[tid];
      s_bad[tid] = 0;
    }
  }
  cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------ walk
template <int D, bool MISS>
__global__ void __launch_bounds__(1024) trees3_kernel(const __grid_constant__ T3Params p) {
  extern __shared__ __align__(1024) unsigned char smem3[];
  unsigned char* const smem = smem3;
  constexpr int NN = 1 << D;  // node slots per tree (1-based heap) == leaves per tree
  constexpr int TR = kT3TR, RPT = kT3RPT, U = kT3U;
  const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
  const int W = p.warps;                   // walking warps; the last kT3Service warps serve them
  const int n_all = (W + kT3Service) * 32;

  int pi = 0;
  while (pi + 1 < p.n_parts && (int)blockIdx.x >= p.parts[pi].cta0 + p.parts[pi].n_ctas) ++pi;
  const T3Part part = p.parts[pi];
  const int cta = (int)blockIdx.x - part.cta0;
  const int64_t n_tiles = (p.n_rows + TR - 1) / TR;
  if ((int64_t)cta >= n_tiles) return;  // small batch: this CTA has no tile (decided before the tables are loaded)
  const int K = (int)((n_tiles - cta + part.n_ctas - 1) / part.n_ctas);  // tiles of this CTA: cta, cta + n_ctas, ...
  const int NT = part.n_trees;
  const bool is_lin = NT == 0;
  const int ncols = part.n_cols;

  unsigned char* s_nodes = smem;
  double* s_leaf = reinterpret_cast<double*>(smem + p.sm_leaf);
  double* s_part = reinterpret_cast<double*>(smem + p.sm_part);  // [2][W x TR] one partial sum per walking warp and row
  double* s_lin = reinterpret_cast<double*>(smem + p.sm_lin_part);  // [2][lin_slices x n_cols x TR] (the linear part)
  uint32_t* s_xt = reinterpret_cast<uint32_t*>(smem + p.sm_xt);  // [2][n_in][TR] tiles (128-byte aligned)
  uint64_t* s_full = reinterpret_cast<uint64_t*>(smem + p.sm_bar);  // [2] tile landed (TMA transaction bytes)
  uint64_t* s_done = s_full + 2;                                    // [2] every walking warp is through with the tile
  uint64_t* s_pfree = s_full + 4;                                   // [2] the tile's partial sums have been combined
  const uint32_t tile_bytes = (uint32_t)p.xt_words * 4u;

  // ---- the part's tables -> shared memory (once per CTA, all warps)
  if (!is_lin) {
    uint2* sn = reinterpret_cast<uint2*>(s_nodes);
    for (int i = tid; i < NT * NN; i += n_all) {
      sn[i] = part.nodes[i];
      s_leaf[i] = part.leaves[i];
    }
  } else {
    double* sw = reinterpret_cast<double*>(s_nodes);
    for (int i = tid; i < ncols * p.n_in; i += n_all) sw[i] = part.leaves[i];
  }
  if (tid == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(&s_full[b], 1);
      mbar_init(&s_done[b], W);
      mbar_init(&s_pfree[b], kT3Service * 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();  // tables and barriers are ready (the only CTA-wide barrier of the kernel)

  auto tile_src = [&](int k) { return p.xt + ((size_t)cta + (size_t)k * part.n_ctas) * p.xt_words; };

  if (g >= W) {
    // =========================================================================================== service warps
    // lane = row of the tile.  Tile k: wait until every walking warp is done with it; refill its buffer with tile k + 2 at once
    // (the copy's latency is what the walkers could stall on); then add the warps' partial sums in warp order and store them.
    const int sid = tid - W * 32;  // 0 .. 63 == TR - 1
    auto refill = [&](int k, int buf) {
      mbar_expect_tx(&s_full[buf], tile_bytes);
      bulk_load(s_xt + (size_t)buf * p.xt_words, tile_src(k), tile_bytes, &s_full[buf]);
      if (k + 2 < K)  // and pull the tile after the next into L2 meanwhile
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(tile_src(k + 2)), "r"(tile_bytes) : "memory");
    };
    if (sid == 0)
      for (int k = 0; k < 2 && k < K; ++k) refill(k, k);
    const int n_sum = is_lin ? p.lin_slices : W;  // tree parts: one partial per warp; the linear part: one per feature slice
    for (int k = 0; k < K; ++k) {
      const int buf = k & 1;
      const int64_t row0 = ((int64_t)cta + (int64_t)k * part.n_ctas) * TR;
      mbar_wait(&s_done[buf], (uint32_t)(k >> 1) & 1u);
      if (sid == 0 && k + 2 < K) refill(k + 2, buf);
      const double* sp = is_lin ? s_lin + (size_t)buf * p.lin_part_words : s_part + (size_t)buf * p.part_words;
      for (int sc = 0; sc < ncols; ++sc) {
        // eight partials are requested before their adds (the LSU queue is full of the walkers' loads); warp order is kept
        double sum = 0.0;
        for (int q0 = 0; q0 < n_sum; q0 += 8) {
          double v[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = q0 + q < n_sum ? sp[((q0 + q) * ncols + sc) * TR + sid] : 0.0;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q0 + q < n_sum) sum = __dadd_rn(sum, v[q]);
        }
        if (row0 + sid < p.n_rows) p.partial[(int64_t)(part.col0 + sc) * p.col_stride + row0 + sid] = sum;
      }
      t3_mbar_arrive(&s_pfree[buf]);  // the walkers of tile k + 2 may overwrite this buffer's partial sums
    }
    return;
  }

  // ============================================================================================= walking warps
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
  const uint32_t leaf0 = (uint32_t)p.sm_leaf - (uint32_t)(NN * 8);  // leaf address = node address + leaf0
  const int TPW = (NT + W - 1) / W;                                 // trees per warp
  for (int k = 0; k < K; ++k) {
    const int buf = k & 1;
    const uint32_t xls = sbase + (uint32_t)p.sm_xt + (uint32_t)(buf * p.xt_words + lane) * 4u;  // this lane's column of the tile
    mbar_wait(&s_full[buf], (uint32_t)(k >> 1) & 1u);
    double acc[RPT];
#pragma unroll
    for (int j = 0; j < RPT; ++j) acc[j] = 0.0;
    if (!is_lin) {
      // ---- warp g takes the trees g, g + W, ...; lane = row (+ 32 j)
      for (int i = 0; i < TPW; i += U) {
        uint32_t tba[U], cl[U], cr[U], a[U][RPT];
        bool valid[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int tr = g + (i + u) * W;
          valid[u] = (i + u) < TPW && tr < NT;
          tba[u] = sbase + (uint32_t)((valid[u] ? tr : 0) * (NN * 8));
          cl[u] = 0u - tba[u];
          cr[u] = 8u - tba[u];
        }
        uint2 nd[U][RPT];
        uint32_t x[U][RPT];
        {  // levels 0 and 1: nodes 1..3 of the tree, one warp-uniform LDS.64 + LDS.128 for all RPT row blocks
          uint2 n1[U], n2[U], n3[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            n1[u] = t3_lds64(tba[u] + 8);
            const uint4 q = t3_lds128(tba[u] + 16);
            n2[u] = make_uint2(q.x, q.y);
            n3[u] = make_uint2(q.z, q.w);
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            x[u][0] = t3_lds32<0>(xls + t3_xoff<MISS>(n1[u].x));
            if (RPT > 1) x[u][1] = t3_lds32<128>(xls + t3_xoff<MISS>(n1[u].x));
          }
          bool r0[U][RPT];
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
              r0[u][j] = t3_right<MISS>(x[u][j], n1[u]);
              nd[u][j].x = r0[u][j] ? n3[u].x : n2[u].x;
              nd[u][j].y = r0[u][j] ? n3[u].y : n2[u].y;
            }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            x[u][0] = t3_lds32<0>(xls + t3_xoff<MISS>(nd[u][0].x));
            if (RPT > 1) x[u][1] = t3_lds32<128>(xls + t3_xoff<MISS>(nd[u][1].x));
          }
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
              const bool r1 = t3_right<MISS>(x[u][j], nd[u][j]);
              a[u][j] = tba[u] + 32u + (r0[u][j] ? 16u : 0u) + (r1 ? 8u : 0u);
            }
        }
#pragma unroll
        for (int d = 2; d < D; ++d) {
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < RPT; ++j) nd[u][j] = t3_lds64(a[u][j]);
#pragma unroll
          for (int u = 0; u < U; ++u) {
            x[u][0] = t3_lds32<0>(xls + t3_xoff<MISS>(nd[u][0].x));
            if (RPT > 1) x[u][1] = t3_lds32<128>(xls + t3_xoff<MISS>(nd[u][1].x));
          }
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int j = 0; j < RPT; ++j) a[u][j] = a[u][j] + a[u][j] + (t3_right<MISS>(x[u][j], nd[u][j]) ? cr[u] : cl[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int j = 0; j < RPT; ++j) {
            const double v = t3_ldsd(a[u][j] + leaf0);
            if (valid[u]) acc[j] = __dadd_rn(acc[j], v);
          }
      }
    }
    // the partial-sum buffer of this parity is free once tile k - 2 has been combined (long ago: that is one walk back)
    if (k >= 2) mbar_wait(&s_pfree[buf], (uint32_t)((k - 2) >> 1) & 1u);
    if (!is_lin) {
      double* sp = s_part + (size_t)buf * p.part_words;
#pragma unroll
      for (int j = 0; j < RPT; ++j) sp[g * TR + j * 32 + lane] = acc[j];
    } else if (g < p.lin_slices) {
      // ---- the linear part: warp s adds the features of slice s into every score column for the tile's rows (fp64 products of
      // float32 inputs are exact; each value is converted once); the service warps add the slices in order
      const double* sw = reinterpret_cast<const double*>(s_nodes);
      const uint32_t* xt = s_xt + (size_t)buf * p.xt_words;
      const int fps = (p.n_in + p.lin_slices - 1) / p.lin_slices;
      const int f0 = g * fps, f1 = min(p.n_in, f0 + fps);
      double a[RPT][kT3MaxLin];
#pragma unroll
      for (int j = 0; j < RPT; ++j)
#pragma unroll
        for (int c = 0; c < kT3MaxLin; ++c) a[j][c] = 0.0;
      for (int f = f0; f < f1; ++f) {
        double xv[RPT];
#pragma unroll
        for (int j = 0; j < RPT; ++j) xv[j] = (double)__uint_as_float(xt[(size_t)f * TR + j * 32 + lane]);
#pragma unroll
        for (int c = 0; c < kT3MaxLin; ++c)
          if (c < ncols) {
            const double wv = sw[(size_t)c * p.n_in + f];
#pragma unroll
            for (int j = 0; j < RPT; ++j) a[j][c] = fma(wv, xv[j], a[j][c]);
          }
      }
      double* sp = s_lin + (size_t)buf * p.lin_part_words;
#pragma unroll
      for (int c = 0; c < kT3MaxLin; ++c)
        if (c < ncols) {
#pragma unroll
          for (int j = 0; j < RPT; ++j) sp[((size_t)g * ncols + c) * TR + j * 32 + lane] = a[j][c];
        }
    }
    __syncwarp();
    if (lane == 0) t3_mbar_arrive(&s_done[buf]);  // release: the stores above are visible to whoever completes the wait
  }
}

// Per row: scores = init + the model's columns of `partial` in column order, link, then the VotingEnsemble reduce.
__global__ void __launch_bounds__(256) t3_vote_kernel(KParams kp, const double* __restrict__ partial, int64_t col_stride,
                                                      const int32_t* __restrict__ col_score, int n_cols,
                                                      const int32_t* __restrict__ row_bad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < kp.n_rows; row += stride) {
    double sc[kMaxScores];
    for (int k = 0; k < kp.n_scores; ++k) sc[k] = kp.bias[k];
    for (int c = 0; c < n_cols; ++c) {
      const int k = col_score[c];
      sc[k] = __dadd_rn(sc[k], partial[(int64_t)c * col_stride + row]);
    }
    double pred[kMaxModels];
    for (int m = 0; m < kp.n_models; ++m) {
      const ModelDesc md = kp.models[m];
      pred[m] = apply_link(md, sc + md.score_off, kp.classes);
    }
    vote_and_store(kp, pred, row, row_bad[row] ? 1u : 0u);
  }
  merge_signal(kp.sig);
}
#endif  // B2S_T3_KERNELS

}  // namespace b2s
