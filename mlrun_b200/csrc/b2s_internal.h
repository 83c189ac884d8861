// b2s_internal.h -- what the translation units of libb200serve.so share (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>

#include <mutex>

#define B2S_HIDDEN __attribute__((visibility("hidden")))

B2S_HIDDEN int b2s_int_fail(int code, const char* fmt, ...);  // sets b2s_last_error(), returns code
B2S_HIDDEN bool b2s_int_inited();
B2S_HIDDEN int b2s_int_device();
B2S_HIDDEN int b2s_int_sm_count();
B2S_HIDDEN cudaStream_t b2s_int_stream();                      // the library stream
B2S_HIDDEN cudaStream_t b2s_int_copy_stream();                 // the library's copy stream (pipelined host runs)
B2S_HIDDEN void b2s_int_count_launches(int n);
struct b2s_plan_s;
B2S_HIDDEN int b2s_int_plan_shape(b2s_plan_s* plan, int* n_in, int* out_cols);  // B2S_ERR_STATE unless finalized

// the columns plan as the statistics unit sees it (b2s_columns.cu): its mutex (held by b2s_cols_run_host, and by the
// statistics calls around everything below), the device-resident result of its last b2s_cols_run_host (slot s at
// *d_out + s * *stride; *generation counts the host runs, so a caller can tell that the result was replaced), and the
// statistics workspace it owns (freed with the plan by b2s_int_colstats_free).  The last two need the mutex held.
struct b2s_cols_s;
struct ColStatsWS;
B2S_HIDDEN std::mutex& b2s_int_cols_mutex(b2s_cols_s* c);
B2S_HIDDEN int b2s_int_cols_result(b2s_cols_s* c, const char** d_out, long long* stride, long long* rows, int* n_out_slots,
                                   unsigned long long* generation);
B2S_HIDDEN ColStatsWS*& b2s_int_cols_stats_ws(b2s_cols_s* c);
B2S_HIDDEN void b2s_int_colstats_free(ColStatsWS* ws);

// the online table as the scoring kernel's gather loader sees it (b2s_table.cu fills it in)
struct B2SGather {
  const long long* d_keys;   // [n]
  const void* d_slots;       // b2s::TableSlot[mask + 1]
  unsigned long long mask;
  const float* d_values;     // [n_keys + 1][n_feat], last row NaN
  long long missing_row;     // n_keys
  const float* h_impute;     // [n_feat] host copy; NaN = keep the stored value
  int any_impute;
  int n_feat;
};
// keys -> (gather inside the scoring kernel) -> outputs + status (B2S_ROW_UNKNOWN_KEY included), one launch.
// B2S_ERR_UNSUPPORTED when this plan / table pair cannot be fused (the caller then gathers first).
B2S_HIDDEN int b2s_int_launch_gathered(b2s_plan_s* plan, const B2SGather& g, long long n, void* d_out, int* d_status, cudaStream_t st);
