/*
 * b200serve.h -- C-ABI of the B200 serving-graph engine (libb200serve.so).
 *
 * The reference (mlrun/mlrun) has no FFI on this path: its hot path is pure Python.  This header is
 * the boundary a maintainer binds (ctypes/cffi) to replace the per-event Python step loop with a batched
 * device plan.  Every entry point names the reference code it replaces (paths relative to the
 * reference root).  Plain pointers and sizes only; no Python / torch types cross it.
 *
 * Conventions
 *   - every call returns 0 on success or a negative b2s_status; the message is thread-local in
 *     b2s_last_error();
 *   - the caller owns host buffers (the library copies on submit); the library owns device memory;
 *   - a "row" is one event's feature vector: n_in_cols 4-byte words (float32, or int32 where the
 *     plan says so), rows `row_stride_bytes` apart;
 *   - outputs are `out_cols` 4-byte words per row (float32 for regression / transform outputs, int32
 *     for class labels), plus an int32 status word per row (0 = ok) so that the Python layer can turn
 *     a bad row into that event's 400 response (mlrun/serving/server.py:278-288) without failing the
 *     whole batch.
 */
#ifndef B200SERVE_H
#define B200SERVE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2S_VERSION 100 /* 0.1.0 */

typedef enum b2s_status {
  B2S_OK = 0,
  B2S_ERR_INVALID = -1,   /* bad argument / plan not finalised / schema mismatch */
  B2S_ERR_CUDA = -2,      /* a CUDA runtime call failed (message has the CUDA error string) */
  B2S_ERR_NO_DEVICE = -3, /* no usable GPU: there is NO CPU fallback */
  B2S_ERR_STATE = -4,     /* call sequence error (not initialised, already finalised ...) */
  B2S_ERR_TIMEOUT = -5,
  B2S_ERR_UNSUPPORTED = -6
} b2s_status;

/* per-row status bits written next to each output row */
#define B2S_ROW_OK 0
#define B2S_ROW_NONFINITE_INPUT 1 /* NaN/Inf reached a model input: scikit-learn's predict raises
                                     ValueError there (called from pkl_model_server.py:58) */
#define B2S_ROW_BAD_LABEL 2       /* majority vote saw a negative label (serving/routers.py:717-725
                                     assumes labels 0..max) */
#define B2S_ROW_UNKNOWN_KEY 4     /* b2s_table_enrich_host: the entity key is not in the online table (the reference's
                                     OnlineVectorService.get returns None for it) */

typedef struct b2s_plan_s* b2s_plan_t;

/* output-schema column kinds (b2s_plan_set_output_schema) */
#define B2S_OUT_COPY 0   /* out = value of source column */
#define B2S_OUT_ONEHOT 1 /* out = (value == arg) ? 1 : 0 -- OneHotEncoder._encode, feature_store/steps.py:453-471 */

/* model link functions (what the estimator's predict() does after the raw score) */
#define B2S_LINK_IDENTITY 0   /* regression: out = score[0]                                   */
#define B2S_LINK_BINARY_GT 1  /* classes[score[0] >  0]  (sklearn LogisticRegression.predict) */
#define B2S_LINK_BINARY_GE 2  /* classes[score[0] >= 0]  (sklearn GradientBoostingClassifier) */
#define B2S_LINK_ARGMAX 3     /* classes[argmax_k score[k]], first max wins (np.argmax)       */

/* ensemble vote (VotingEnsemble._apply_logic, serving/routers.py:789-810) */
#define B2S_VOTE_NONE 0     /* emit every model's prediction: out_cols = n_models                 */
#define B2S_VOTE_MEAN 1     /* _mean_vote :732-741   -- sum_m w[m] * pred[m]  (fp64)             */
#define B2S_VOTE_MAJORITY 2 /* _majority_vote :708-730 -- argmax_c sum_m w[m]*[pred[m]==c], first max */

typedef struct b2s_stats {
  int64_t rows;          /* rows in the batch this call rode in                                  */
  float h2d_ms;          /* CUDA-event time of the host->device copy                             */
  float kernel_ms;       /* CUDA-event time of the plan's kernels (b2s_run_host pipelines large  */
  float d2h_ms;          /* pinned batches in chunks: kernel/d2h are then sums over the chunks)   */
  float queue_us;        /* submit -> batch sealed (coalescing wait)                             */
  int32_t kernels;       /* kernel launches in the batch                                         */
  int32_t nonfinite_rows;/* rows flagged B2S_ROW_NONFINITE_INPUT                                 */
} b2s_stats;

typedef struct b2s_devinfo {
  int32_t ordinal, sm_count, cc_major, cc_minor;
  int64_t total_mem, l2_bytes, smem_per_block_optin;
  char name[128];
} b2s_devinfo;

/* ---- library / device ---------------------------------------------------------------------- */
int b2s_version(void);
const char* b2s_last_error(void);
/* Replaces: nothing in the reference (device bring-up).  cfg is "key=value;..." or NULL:
 *   ring_slots (4), max_batch (65536 rows), max_wait_us (0: a coalesced batch leaves as soon as the dispatcher is free, so
 *   batches form while the previous one runs; > 0: the oldest row may wait that long for company).  Idempotent per process. */
int b2s_init(int device_ordinal, const char* cfg);
int b2s_shutdown(void);
int b2s_device_info(b2s_devinfo* out);
/* number of kernels this library has launched since b2s_init (for bench.py's gpu_launches) */
int64_t b2s_launch_count(void);

/* ---- plan construction ---------------------------------------------------------------------
 * A plan is the lowered form of a run of recognised graph steps.  It replaces, for those steps, the
 * reference's per-event loop  FlowStep.run (serving/states.py:1292-1323)  ->  TaskStep.run (:564-599)
 * -> step handler, and the storey Map chain built by _init_async_objects (:1622-1710). */
int b2s_plan_create(int32_t n_in_cols, b2s_plan_t* out);
int b2s_plan_destroy(b2s_plan_t plan);

/* Imputer._impute (feature_store/steps.py:397-406): NaN in column cols[i] -> fills[i]. */
int b2s_plan_set_impute(b2s_plan_t plan, const int32_t* cols, const float* fills, int32_t n);
/* MapValues._map_value exact-match branch (steps.py:200-201): v == keys[i] -> vals[i], else unchanged.
 * Maps are applied after the imputer, in the order they are added. */
int b2s_plan_add_value_map(b2s_plan_t plan, int32_t col, const float* keys, const float* vals, int32_t n);
/* MapValues._map_value range branch (steps.py:193-198): first i with lo[i] <= v < hi[i] -> vals[i]. */
int b2s_plan_add_range_map(b2s_plan_t plan, int32_t col, const float* lo, const float* hi, const float* vals, int32_t n);
/* Output schema after OneHotEncoder._do_storey (steps.py:473-478) / DropFeatures (:721-729):
 * out column j reads source column src_col[j] with kind[j] (B2S_OUT_*) and arg[j]. Default: identity. */
int b2s_plan_set_output_schema(b2s_plan_t plan, const int32_t* src_col, const int32_t* kind, const float* arg, int32_t n_out);

/* Linear scorer = what sklearn's linear estimators compute inside PickleModelServer.predict
 * (frameworks/_ml_common/pkl_model_server.py:52-60): score[k] = b[k] + sum_j W[k][j] * x_out[j] in fp64.
 * W is row-major (n_scores x n_out_cols).  classes: label per class index for the classifier links (may be NULL). */
int b2s_plan_add_linear_model(b2s_plan_t plan, const double* W, const double* b, int32_t n_scores, int32_t link,
                              const int32_t* classes, int32_t n_classes);
/* Tree-ensemble scorer (sklearn GradientBoosting* / RandomForest* / DecisionTree* behind the same
 * predict call).  Trees are concatenated SoA: node i of tree t lives at tree_offset[t] + i.
 *   feature[i] < 0 marks a leaf whose value is leaf_value[i]; otherwise go left when
 *   x[feature[i]] <= threshold[i] (sklearn: float32 x vs float64 threshold; thresholds are passed
 *   already rounded toward -inf to float32, which gives the identical decision).
 *   score[tree_slot[t]] += tree_scale[t] * leaf_value;  score[k] starts at init[k]. */
int b2s_plan_add_tree_model(b2s_plan_t plan, int32_t n_trees, const int32_t* tree_offset /* n_trees+1 */,
                            const int32_t* feature, const float* threshold, const int32_t* left,
                            const int32_t* right, const double* leaf_value, const int32_t* tree_slot,
                            const double* tree_scale, const double* init, int32_t n_scores, int32_t link,
                            const int32_t* classes, int32_t n_classes);
/* The same with the tree semantics of the other libraries behind the reference's model servers (XGBoostModelServer is
 * PickleModelServer, frameworks/xgboost/__init__.py:30; LGBMModelServer.predict, frameworks/lgbm/model_server.py:142-159):
 *   cmp_mode       B2S_CMP_LE: left when x <= threshold (scikit-learn, LightGBM);  B2S_CMP_LT: left when x < threshold (xgboost);
 *   default_left   per node (may be NULL = all 0): where a missing value (NaN) goes -- xgboost's "missing" child,
 *                  LightGBM's default_left, scikit-learn's tree_.missing_go_to_left;
 *   nan_mode       B2S_NAN_ERROR: a NaN input flags the row B2S_ROW_NONFINITE_INPUT (estimators whose predict refuses NaN);
 *                  B2S_NAN_DEFAULT_CHILD: NaN follows default_left.  It is honoured when every model of the plan routes
 *                  missing values and the plan runs on the shared-memory tree kernel (b2s_plan_kernel says so); in any
 *                  other plan a NaN row is still flagged -- an error, never a silently different answer.
 * Inf is flagged in both modes (what check_array / DMatrix refuse). */
#define B2S_CMP_LE 0
#define B2S_CMP_LT 1
#define B2S_NAN_ERROR 0
#define B2S_NAN_DEFAULT_CHILD 1
int b2s_plan_add_tree_model_ex(b2s_plan_t plan, int32_t n_trees, const int32_t* tree_offset /* n_trees+1 */,
                               const int32_t* feature, const float* threshold, const int32_t* left, const int32_t* right,
                               const double* leaf_value, const int32_t* tree_slot, const double* tree_scale,
                               const double* init, int32_t n_scores, int32_t link, const int32_t* classes, int32_t n_classes,
                               int32_t cmp_mode, const uint8_t* default_left, int32_t nan_mode);
/* VotingEnsemble reduce over the plan's models (weights in model order; fp64). */
int b2s_plan_set_vote(b2s_plan_t plan, int32_t vote_kind, const double* weights, int32_t n_weights);
/* Upload tables to HBM, pick kernels, size staging buffers.  After this the plan is immutable. */
int b2s_plan_finalize(b2s_plan_t plan);
/* name + template parameters of the kernel family the plan launches (diagnostics / bench provenance) */
const char* b2s_plan_kernel(b2s_plan_t plan);
/* out_cols 4-byte words per output row; out_is_int != 0 when they are int32 labels */
int b2s_plan_out_info(b2s_plan_t plan, int32_t* out_cols, int32_t* out_is_int);

/* ---- execution -------------------------------------------------------------------------------
 * Replaces GraphServer.run -> graph.run (serving/server.py:252-293) for a batch of events. */

/* Device-resident path: rows and outputs already in HBM (roofline runs, CUDA-graph capture, callers that
 * keep tensors on the GPU).  Asynchronous on `stream` (a cudaStream_t, NULL = the library's stream).
 * d_status may be NULL. */
int b2s_run_device(b2s_plan_t plan, const void* d_rows, int64_t n_rows, int64_t row_stride_bytes, void* d_out,
                   int32_t* d_status, void* stream);
/* Synchronous host call: pinned staging -> H2D -> kernels -> D2H -> out.  row_status / stats may be NULL.
 * Batches of at most B2S_ZEROCOPY_ROWS (8192) rows skip both copies: the kernels read the rows from (and write the votes
 * to) pinned host memory over PCIe themselves -- one launch and one synchronisation, the latency path of a serving batch;
 * pinned batches of 128 Ki rows and more are pipelined in chunks (copy of chunk c + 1 under the kernels of chunk c). */
int b2s_run_host(b2s_plan_t plan, const void* rows, int64_t n_rows, int64_t row_stride_bytes, void* out,
                 int64_t out_bytes, int32_t* row_status, b2s_stats* stats);
/* Coalescing path (thread-safe, many producers): rows are copied into a pinned ring slot; a dispatcher
 * thread seals a batch when it holds max_batch rows or the oldest row waited max_wait_us (0: as soon as the dispatcher is
 * free -- batches form while the previous one runs), and runs it on its own stream (small batches zero-copy, like b2s_run_host).  b2s_wait blocks until the ticket's batch completed and copies
 * that ticket's rows out.  This is the replacement of storey's SyncEmitSource.emit / await_result hand-off
 * (serving/states.py:1283-1287).  A ring slot is recycled when every ticket of its batch was collected, and the ring
 * has `ring_slots` (b2s_init cfg, default 4) batches: a producer that keeps submitting without collecting its tickets
 * eventually blocks in b2s_submit -- emit and await per request, as the reference's callers do. */
int b2s_submit(b2s_plan_t plan, const void* rows, int64_t n_rows, int64_t row_stride_bytes, uint64_t* ticket);
int b2s_wait(b2s_plan_t plan, uint64_t ticket, void* out, int64_t out_bytes, int32_t* row_status, b2s_stats* stats);
/* force the open batch out now (drain callback, serving/server.py:353-384) */
int b2s_flush(b2s_plan_t plan);
/* Per-plan ring configuration, before the plan's first b2s_submit: batches in flight, rows per batch and how long the
 * oldest row may wait for company (0 / 0 / negative keep the b2s_init defaults).  This is where a serving function's
 * `spec.parameters["b200"] = {"max_batch": .., "max_wait_us": .., "ring_slots": ..}` lands (runtimes/nuclio/serving.py:
 * 668-724 hands spec.parameters to the GraphServer). */
int b2s_plan_set_ring(b2s_plan_t plan, int32_t ring_slots, int64_t max_batch, int32_t max_wait_us);
/* The ring measured by itself: n_threads native producers, each emitting rows_per_submit rows of `rows` and awaiting them
 * (emit / await_result of one request), for `seconds`.  events = rows served; p50 / p99 of the submit -> wait round trip. */
int b2s_ring_bench(b2s_plan_t plan, const void* rows, int64_t n_src_rows, int64_t row_stride_bytes, int32_t n_threads,
                   int32_t rows_per_submit, double seconds, int64_t* events, double* p50_us, double* p99_us);

/* ---- multi-GPU: fused ensemble-merge ----------------------------------------------------------------
 * One process per GPU, events sharded by rows (they are independent: VotingEnsemble reduces across models,
 * serving/routers.py:797-810).  The only exchange is the merge of every shard's votes into the full
 * response.  Instead of a separate all-gather, a plan can be given the output buffers of all ranks
 * (peer-mapped over NVLink with the IPC calls below); its kernels then store each output row into every
 * target at row `row_offset + row` straight from the epilogue.  n_peers = 0 restores local output. */
int b2s_plan_set_merge_targets(b2s_plan_t plan, void* const* peer_out, int32_t n_peers, int64_t row_offset);
int b2s_ipc_export(void* dptr, void* handle64 /* 64 bytes out */);
int b2s_ipc_open(const void* handle64, void** dptr_out);
int b2s_ipc_close(void* dptr);

/* The same exchange as a product object: a communicator owns, per rank, ONE device allocation -- completion flags and the
 * merged response rows in four slots -- that every peer maps over CUDA IPC.  Bootstrap needs any out-of-band channel
 * that can all-gather 64 bytes per rank (torch.distributed, MPI, a file, a socket ...):
 *     b2s_comm_create(rank, world, max_rows_per_rank, out_cols, &c);  b2s_comm_handle(c, mine);
 *     <all-gather the 64-byte handles>;  b2s_comm_connect(c, all);  b2s_plan_attach_comm(plan, c);
 * Every b2s_run_device / b2s_run_host / ring batch of an attached plan is then one STEP (epoch e = 1, 2, ...) of the
 * ensemble-merge (serving/routers.py:414-455 fans the event out to the routes, :789-810 reduces them; here the rows are
 * sharded and the votes merged): the kernels store this rank's votes into slot e & 3 of EVERY rank's merged rows at row
 * block `rank`, and the launch's last CTA publishes e in every rank's flag array (st.release.sys).  b2s_comm_wait enqueues
 * a one-warp kernel that acquires all `world` flags of THIS rank at the current epoch, so work enqueued behind it (a D2H copy,
 * the next kernel) reads a complete response; *d_merged is that response, (world x max_rows_per_rank x out_cols) words, rank
 * r's rows at r * max_rows_per_rank.  Every launch must be followed by a wait on the same stream: b2s_comm_wait (step e,
 * lockstep) or b2s_comm_wait_lag(.., 1, ..) (step e - 1: the votes and flags of step e cross NVLink while step e + 1 is being
 * scored; the response of a step is then available one launch later, and a final b2s_comm_wait drains the last step).
 * Four slots make both safe: before a rank launches step e + 4 (which overwrites slot e & 3 everywhere) it has passed its
 * wait for step e + 2 at the latest, i.e. it has seen every peer's flag of step e + 2 -- and a peer's launch of step e + 2
 * sits behind that peer's wait for (and use of) step e in the peer's own stream.  A peer that never
 * signals makes the wait give up after B2S_COMM_TIMEOUT_MS (default 10 s; b2s_comm_check reports B2S_ERR_TIMEOUT) instead of hanging the GPU. */
typedef struct b2s_comm_s* b2s_comm_t;
int b2s_comm_create(int32_t rank, int32_t world, int64_t max_rows_per_rank, int32_t out_cols, b2s_comm_t* out);
int b2s_comm_handle(b2s_comm_t comm, void* handle64 /* 64 bytes out */);
int b2s_comm_connect(b2s_comm_t comm, const void* all_handles /* world x 64 bytes, in rank order */);
int b2s_plan_attach_comm(b2s_plan_t plan, b2s_comm_t comm /* NULL detaches */);
int b2s_comm_wait(b2s_comm_t comm, void* stream, const void** d_merged, uint32_t* epoch);
/* lag 0 or 1; with fewer than lag + 1 steps launched there is nothing to wait for: *d_merged = NULL, *epoch = 0 */
int b2s_comm_wait_lag(b2s_comm_t comm, void* stream, int32_t lag, const void** d_merged, uint32_t* epoch);
/* Fused wait: lag 0 / 1 makes every launch of an attached plan end by acquiring -- in the launch's last CTA, after it has
 * published its own flag -- this rank's flags of its own step / of the previous step (same timeout as the wait kernel);
 * b2s_comm_wait / b2s_comm_wait_lag then enqueue nothing for a step that is covered.  Saves the wait kernel and its two launch
 * boundaries per step (4.9 us of a 50 us step at 1 Mi events, 2 GPUs).  lag -1 = off (default). */
int b2s_comm_set_fused_wait(b2s_comm_t comm, int32_t lag);
int b2s_comm_check(b2s_comm_t comm);
int b2s_comm_destroy(b2s_comm_t comm);

/* pinned host memory for zero-extra-copy submits and for bench.py's e2e leg */
void* b2s_alloc_pinned(size_t bytes);
int b2s_free_pinned(void* p);
/* plain device memory helpers so that ctypes callers need no other CUDA binding */
void* b2s_device_alloc(size_t bytes);
int b2s_device_free(void* p);
int b2s_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes);
int b2s_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes);
int b2s_device_sync(void);
/* time n_iters back-to-back b2s_run_device launches with CUDA events on the library stream (ms total);
 * used by bench.py so that the timed region contains only the plan's kernels.  d_rows[i % n_bufs]. */
int b2s_time_device(b2s_plan_t plan, const void* const* d_rows, int32_t n_bufs, int64_t n_rows,
                    int64_t row_stride_bytes, void* d_out, int32_t n_iters, float* total_ms);

/* ---- columnar ingest: feature-set transforms over DataFrame-shaped data -------------------------------
 * Replaces the row-at-a-time walk of a feature-set graph by the storey engine
 * (feature_store/ingestion.py:38-127 init_featureset_graph; datastore/sources.py:886-895 DataframeSource emits one
 * dict per row; datastore/targets.py:1856-1868 ReduceToDataFrame re-assembles them).  Data is columnar on both
 * sides, like the DataFrame it comes from: an input/output "slot" is n_rows 4-byte words (float32 / int32); an
 * 8-byte column (datetime64[ns] as int64) takes two adjacent slots.  The plan is a list of column ops; every op
 * reads one input column and writes 0..n output columns; output slots are numbered in the order ops are added.
 * Float sources take an optional Imputer fill first (Imputer._impute, feature_store/steps.py:397-406).
 * `check` bits (1: min, 2: max) attach MinMaxValidator.check (mlrun/features.py:292-321) to the op's result:
 * violating rows are counted (the reference's FeaturesetValidator only prints them, steps.py:117-128). */
typedef struct b2s_cols_s* b2s_cols_t;
#define B2S_COL_F32 0
#define B2S_COL_I32 1
#define B2S_COL_I64 2
/* date parts of DateExtractor._do_storey (steps.py:593-602: getattr(pd.Timestamp(ts), part)) computed on the device */
#define B2S_DATE_YEAR 0
#define B2S_DATE_MONTH 1
#define B2S_DATE_DAY 2
#define B2S_DATE_HOUR 3
#define B2S_DATE_MINUTE 4
#define B2S_DATE_SECOND 5
#define B2S_DATE_DAY_OF_WEEK 6 /* Monday = 0 */
#define B2S_DATE_DAY_OF_YEAR 7
#define B2S_DATE_QUARTER 8
#define B2S_DATE_IS_LEAP_YEAR 9     /* the is_* parts give 0 / 1 */
#define B2S_DATE_DAYS_IN_MONTH 10
#define B2S_DATE_IS_MONTH_START 11
#define B2S_DATE_IS_MONTH_END 12
#define B2S_DATE_IS_QUARTER_START 13
#define B2S_DATE_IS_QUARTER_END 14
#define B2S_DATE_IS_YEAR_START 15
#define B2S_DATE_IS_YEAR_END 16
#define B2S_DATE_WEEK 17             /* ISO 8601 week (pd.Timestamp.week / weekofyear) */

int b2s_cols_create(int32_t n_in_slots, b2s_cols_t* out);
int b2s_cols_destroy(b2s_cols_t plan);
/* pass a column through (keep != 0) and/or validate it; keep == 0 is a column DropFeatures removed
 * (steps.py:721-729) that a validator placed before the drop still sees. */
int b2s_cols_add_copy(b2s_cols_t plan, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, int32_t keep,
                      int32_t check, double cmin, double cmax, int32_t* out_slot, int32_t* check_counter);
/* MapValues._map_value (steps.py:189-201): first i with lo[i] <= v < hi[i] -> vals[i]; no hit: v passes through
 * and counters[miss_counter] counts the row.  The output slot holds float32. */
int b2s_cols_add_range_map(b2s_cols_t plan, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* lo,
                           const double* hi, const double* vals, int32_t n, int32_t check, double cmin, double cmax,
                           int32_t* out_slot, int32_t* miss_counter, int32_t* check_counter);
/* MapValues exact-match branch (steps.py:200-201): v == keys[i] -> vals[i]. */
int b2s_cols_add_value_map(b2s_cols_t plan, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* keys,
                           const double* vals, int32_t n, int32_t check, double cmin, double cmax, int32_t* out_slot,
                           int32_t* miss_counter, int32_t* check_counter);
/* OneHotEncoder._encode (steps.py:453-470): n int32 0/1 output slots, in category order; a value matching no
 * category gives all zeros and is counted (the reference logs a warning). */
int b2s_cols_add_onehot(b2s_cols_t plan, int32_t src_slot, int32_t kind, int32_t has_fill, float fill, const double* cats,
                        int32_t n, int32_t* first_out_slot, int32_t* miss_counter);
/* DateExtractor: src_slot is an 8-byte nanosecond timestamp; the int32 output is -1 for NaT (counted). */
int b2s_cols_add_date_part(b2s_cols_t plan, int32_t src_slot, int32_t part, int32_t* out_slot, int32_t* nat_counter);
int b2s_cols_finalize(b2s_cols_t plan);
int b2s_cols_info(b2s_cols_t plan, int32_t* n_out_slots, int32_t* n_counters);
/* Device-resident run: slot s of the input starts at d_in + s * in_slot_stride (bytes, multiple of 8, >= 4 * n_rows);
 * d_counters (n_counters uint64, zeroed by the caller) accumulates.  Asynchronous on `stream`. */
int b2s_cols_run_device(b2s_cols_t plan, const void* d_in, int64_t in_slot_stride, int64_t n_rows, void* d_out,
                        int64_t out_slot_stride, uint64_t* d_counters, void* stream);
/* Host run: one pointer per input slot the plan reads (an 8-byte column: pointer at its first slot), one per output
 * slot (NULL at the second slot of an 8-byte column): H2D per column -> kernel -> D2H per column. */
int b2s_cols_run_host(b2s_cols_t plan, const void* const* h_in_slots, int64_t n_rows, void* const* h_out_slots,
                      uint64_t* counters, b2s_stats* stats);
/* n_iters back-to-back device runs over rotating inputs, CUDA-event timed (bench.py) */
int b2s_cols_time_device(b2s_cols_t plan, const void* const* d_in, int32_t n_bufs, int64_t in_slot_stride, int64_t n_rows,
                         void* d_out, int64_t out_slot_stride, uint64_t* d_counters, int32_t n_iters, float* total_ms);

/* ---- feature-set statistics: ingest(..., infer_options=Stats | Histogram) on the device -------------------------------
 * get_df_stats (data_types/infer.py:104-149), called on the ingested frame by _infer_from_static_df
 * (feature_store/api.py:1162-1196): pandas describe(include="all") plus a 20-bin np.histogram per column.  The columns of a
 * plan's result are described where they are: the plan's resident result of its last b2s_cols_run_host (d_out NULL), or a
 * caller's device buffer in the b2s_cols_run_device layout.  Two calls, because the host needs the first summary to choose
 * what the second pass computes (histogram edges from min / max, target ranks from the count):
 *   begin   one pass: per column count, missing, fp64 sum, min, max, +-inf, ones (bool), row 0 -> summary[n_cols];
 *   finish  the centred sum of squares around means[i] (NaN: none), the 20 histogram counts with the host's edges, and up to
 *           B2S_STAT_RANKS exact order statistics per column (radix select over the same data; ranks[i][r] < 0: none).
 * Stats kinds say how a slot is read and what is missing.  The calls run on the library stream and block until their results
 * are on the host.  A b2s_cols_run_host of the plan between begin and finish replaces the result: finish then fails with
 * B2S_ERR_STATE (call begin again). */
#define B2S_STAT_F32 0      /* float32 slot; NaN is missing                                   */
#define B2S_STAT_I32 1      /* int32 slot                                                     */
#define B2S_STAT_I32_NAT 2  /* int32 date part; -1 marks NaT (missing)                        */
#define B2S_STAT_BOOL 3     /* int32 0 / 1 slot                                               */
#define B2S_STAT_DT 4       /* int64 nanoseconds over two slots; NaT (INT64_MIN) is missing   */
#define B2S_STAT_ROW 5      /* the row number (no slot is read)                               */
#define B2S_STAT_RANKS 6
#define B2S_STAT_BINS 20
typedef struct b2s_colsum {
  int64_t count;          /* non-missing values                                                         */
  int64_t missing;
  int64_t ones;           /* B2S_STAT_BOOL: values equal to 1                                            */
  int32_t pos_inf, neg_inf;
  double sum;             /* fp64, added in a fixed order                                               */
  int64_t min_bits;       /* min / max of the non-missing values: float32 bits for B2S_STAT_F32, else the */
  int64_t max_bits;       /*   integer value (count > 0 only)                                           */
  int64_t first_bits;     /* row 0, in the same encoding                                                */
  int32_t first_missing;
  int32_t pad_;
} b2s_colsum;
int b2s_cols_stats_begin(b2s_cols_t plan, const void* d_out, int64_t out_slot_stride, int64_t n_rows, const int32_t* kinds,
                         const int32_t* slots, int32_t n_cols, b2s_colsum* summary, b2s_stats* stats);
/* hist_kind[i]: 0 none, 1 float32 bins, 2 float64 bins (np.histogram's bin dtype); hist[i] = 23 doubles: first_edge,
 * last_edge - first_edge, then the 21 edges, all exact values of the bin dtype.  Outputs: m2[n_cols],
 * hist_counts[n_cols][B2S_STAT_BINS], order_values[n_cols][B2S_STAT_RANKS] (the encoding of b2s_colsum.min_bits). */
int b2s_cols_stats_finish(b2s_cols_t plan, const double* means, const int32_t* hist_kind, const double* hist,
                          const int64_t* ranks, double* m2, int64_t* hist_counts, int64_t* order_values, b2s_stats* stats);
/* CUDA-event time and bytes read of each pass of the last begin / finish pair (pass 0 is begin's), kernel launches */
int b2s_cols_stats_timing(b2s_cols_t plan, float* pass_ms, int64_t* pass_bytes, int32_t* n_passes, int32_t* launches);

/* ---- body codec (host code): the step on either side of the path for HTTP / stream triggers ------------
 * GraphServer.run json-decodes the request body (serving/server.py:262-277) and _process_response json.dumps
 * the result (:298-308).  b2s_json_parse_inputs finds the top-level "inputs" member of a V2 body and converts
 * its numbers straight into float32 rows (row-major; a flat list is one scalar per event): the same values as
 * np.asarray(json.loads(body)["inputs"], dtype=float32) (null counts as NaN).  [value_begin, value_end) is the
 * member's text, so the caller can decode the small remainder of the body (id, model, operation) as usual.
 * B2S_ERR_UNSUPPORTED: not such a body (strings / dicts / ragged rows) -- the caller falls back to json.loads. */
int b2s_json_parse_inputs(const char* body, int64_t len, float* out, int64_t out_cap, int64_t* n_rows, int64_t* n_cols,
                          int64_t* value_begin, int64_t* value_end);
/* text of a result matrix exactly as json.dumps prints it: float32 values widened to double and printed with
 * Python's repr (vals = float32*), or int32 labels (is_int); flat != 0 prints [v0, v1, ...] for n_cols == 1. */
int b2s_json_format_outputs(const void* vals, int32_t is_int, int64_t n_rows, int64_t n_cols, int32_t flat, char* out,
                            int64_t out_cap, int64_t* out_len);

/* ---- online feature table: real-time enrichment on the device -----------------------------------------
 * EnrichmentModelRouter / EnrichmentVotingEnsemble.preprocess (serving/routers.py:1189-1196, 1335-1342) turn entity
 * keys into feature vectors with OnlineVectorService.get (feature_store/feature_vector.py:975-1067): one online-store
 * read per key, then None / NaN / Inf -> the impute policy's value (:1046-1052).  A b2s_table keeps the online table
 * in HBM (64-bit keys -> rows of n_features float32) and resolves a batch of keys in one launch, writing the rows in
 * the layout b2s_run_device reads.  impute[c] = NaN keeps column c as stored; rows of unknown keys are NaN (then
 * imputed) and reported in found[] (the reference returns None for them). */
typedef struct b2s_table_s* b2s_table_t;
int b2s_table_create(const int64_t* keys, int64_t n_keys, const float* values, int32_t n_features, const float* impute,
                     b2s_table_t* out);
int b2s_table_destroy(b2s_table_t table);
int b2s_table_info(b2s_table_t table, int64_t* n_keys, int32_t* n_features, int64_t* capacity);
int b2s_table_lookup_device(b2s_table_t table, const int64_t* d_keys, int64_t n, float* d_rows, int64_t row_stride_bytes,
                            int32_t* d_found, void* stream);
int b2s_table_lookup_host(b2s_table_t table, const int64_t* keys, int64_t n, float* rows, int32_t* found, b2s_stats* stats);
/* Enrichment + predict for a batch of HOST keys in one call (EnrichmentVotingEnsemble.do_event over a batch: preprocess
 * :1335-1342, then the ensemble): keys -> H2D -> gather -> the scoring plan -> D2H of the plan's outputs and status words,
 * nothing else crosses PCIe (one fused launch when b2s_table_enrich_device covers the plan).  row_status (may be NULL) carries the plan's B2S_ROW_* bits plus B2S_ROW_UNKNOWN_KEY.
 * Pinned caller buffers are used directly; pageable ones are staged through the table's pinned block. */
/* The same for device-resident keys, as ONE launch: the scoring kernel's tile loader finds each key in the table and
 * fetches the row from there (one TMA bulk copy per row), so the gathered rows never travel to HBM and back; the table's
 * impute policy folds into the kernel's Imputer operands.  B2S_ERR_UNSUPPORTED for plans the loader does not cover (tree
 * ensembles, MapValues, one-hot sources under an impute policy): use b2s_table_lookup_device + b2s_run_device then. */
int b2s_table_enrich_device(b2s_table_t table, b2s_plan_t plan, const int64_t* d_keys, int64_t n, void* d_out,
                            int32_t* d_status, void* stream);
int b2s_table_enrich_host(b2s_table_t table, b2s_plan_t plan, const int64_t* keys, int64_t n, void* out, int64_t out_bytes,
                          int32_t* row_status, b2s_stats* stats);
int b2s_table_time_device(b2s_table_t table, const int64_t* const* d_keys, int32_t n_bufs, int64_t n, float* d_rows,
                          int64_t row_stride_bytes, int32_t* d_found, int32_t n_iters, float* total_ms);
/* 64-bit FNV-1a of each string of a packed buffer (string i = bytes[offsets[i] .. offsets[i+1])): the key of a
 * string-valued entity.  Host code. */
int b2s_hash_strings(const char* bytes, const int64_t* offsets, int64_t n, int64_t* keys_out);

#ifdef __cplusplus
}
#endif
#endif /* B200SERVE_H */
