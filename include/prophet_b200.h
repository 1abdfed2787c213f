/*
 * prophet_b200.h -- C ABI of the B200-native batched Prophet fitter / scorer.
 *
 * Drop-in boundary for the per-series hot path of mageky/time-series-spark:
 *
 *   pb200_fit_*      replaces  model_time_series_udf            src/jobs/prophet_modeler.py:41-85
 *                    (floor/cap prep :56-60, Prophet(...).fit(pdf) :65-66) run once per
 *                    (series_id, dim_id) group by groupby().apply()  src/jobs/prophet_modeler.py:139-141
 *   pb200_predict_*  replaces  forecast_time_series_udf         src/jobs/prophet_scorer.py:35-102
 *                    (make_future_dataframe :64-66, floor/cap :67-68, predict :70,
 *                    int truncation :73, floor clamp :76-84) run once per model row by
 *                    groupby().apply()                          src/jobs/prophet_scorer.py:159-161
 *
 * All series of a shard go through ONE call.  Plain pointers and sizes only; no
 * torch / Arrow types.  "d_" = device (HBM) pointer, "h_" = host pointer.
 * Every function returns 0 on success or a negative PB200_E_* code; per-series
 * solver outcomes are reported in the status array, never as a call failure
 * (the reference turns a per-series RuntimeError into "no output row",
 * prophet_modeler.py:81-85 / prophet_scorer.py:99-102).
 *
 * There is NO CPU fallback behind this ABI: every entry point launches sm_100a
 * kernels and fails with PB200_E_CUDA if no device is usable.
 */
#ifndef PROPHET_B200_H
#define PROPHET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB200_ABI_VERSION 1

#if defined(__GNUC__)
#define PB200_API __attribute__((visibility("default")))
#else
#define PB200_API
#endif

/* call-level error codes */
#define PB200_OK            0
#define PB200_E_ARG        -1   /* bad argument (null pointer, negative size, unsupported option) */
#define PB200_E_CUDA       -2   /* CUDA runtime error; see pb200_last_error() */
#define PB200_E_WORKSPACE  -3   /* workspace too small */
#define PB200_E_UNSUPPORTED -4  /* series too long / option outside the compiled kernels */

/* per-series status (status[] output of fit).  >= 0 : Stan L-BFGS TerminationCondition
 * (stan/optimization/bfgs.hpp), a model row is produced;  < 0 : no model row. */
/* pb200_options.algorithm */
#define PB200_ALG_LBFGS_NEWTON 0  /* optimizing(LBFGS); except RuntimeError: optimizing(Newton)  -- fbprophet 0.5 Prophet.fit */
#define PB200_ALG_LBFGS        1  /* L-BFGS only: a line-search failure is final (status PB200_ST_LSFAIL, row dropped) */
#define PB200_ALG_NEWTON       2  /* Newton only (tests; later fbprophet versions use it for short histories) */

#define PB200_ST_SUCCESS      0   /* only transient; never final */
#define PB200_ST_ABSX        10
#define PB200_ST_ABSF        20
#define PB200_ST_RELF        21
#define PB200_ST_ABSGRAD     30
#define PB200_ST_RELGRAD     31
#define PB200_ST_MAXIT       40
#define PB200_ST_CONST_LINEAR 50  /* fbprophet "nothing to fit" shortcut: params = init, sigma_obs = 1e-9 */
#define PB200_ST_NEWTON      60   /* model from fbprophet 0.5's Newton retry after an L-BFGS line-search failure */
#define PB200_ST_LSFAIL      -1   /* line search failed (PyStan raises RuntimeError -> fbprophet Newton retry) */
#define PB200_ST_INIT_ERROR  -2   /* objective not finite at the initial point */
#define PB200_ST_TOO_FEW     -3   /* < 2 rows  (fbprophet ValueError) */
#define PB200_ST_CAP_LE_FLOOR -4  /* cap <= floor (fbprophet ValueError) */
#define PB200_ST_BAD_INPUT   -5   /* unsorted timestamps / non-finite y / zero time span */

/* y element type */
#define PB200_Y_I32 0
#define PB200_Y_F32 1
#define PB200_Y_F64 2

/* growth */
#define PB200_GROWTH_LINEAR   0
#define PB200_GROWTH_LOGISTIC 1

/* seasonality switch: PB200_SEAS_AUTO follows Prophet.set_auto_seasonalities,
 * 0 disables, > 0 forces the default Fourier order of that seasonality on
 * (yearly 10, weekly 3, daily 4).  Other orders are not compiled in. */
#define PB200_SEAS_AUTO (-1)

/* Options = Prophet.__init__ arguments the reference fixes at
 * prophet_modeler.py:65 plus fbprophet 0.5 / PyStan 2.19.1.1 defaults. */
typedef struct pb200_options {
    int32_t abi_version;            /* PB200_ABI_VERSION */
    int32_t growth;                 /* PB200_GROWTH_LOGISTIC (reference default) */
    int32_t multiplicative;         /* 1 = seasonality_mode='multiplicative' (reference default) */
    int32_t n_changepoints;         /* 25 */
    double  changepoint_range;      /* 0.8 */
    double  changepoint_prior_scale;/* 0.05 */
    double  seasonality_prior_scale;/* 10.0 */
    int32_t yearly;                 /* PB200_SEAS_AUTO | 0 | 1 */
    int32_t weekly;
    int32_t daily;
    int32_t max_iter;               /* 10000 (fbprophet passes iter=1e4) */
    int32_t history_size;           /* 5 */
    double  init_alpha;             /* 1e-3 */
    double  tol_obj;                /* 1e-12 */
    double  tol_rel_obj;            /* 1e4  (x machine epsilon) */
    double  tol_grad;               /* 1e-8 */
    double  tol_rel_grad;           /* 1e7  (x machine epsilon) */
    double  tol_param;              /* 1e-8 */
    double  interval_width;         /* 0.8 */
    int32_t uncertainty_samples;    /* 1000; 0 = skip yhat_lower / yhat_upper */
    int32_t algorithm;              /* PB200_ALG_*: 0 = fbprophet 0.5's fit(): Stan L-BFGS, Newton retry after a line-search failure */
} pb200_options;

/* Fills *o with the reference's defaults. */
PB200_API void pb200_default_options(pb200_options* o);

/* Layout of one fitted-model record (the arrays fit writes and predict reads).
 * smax = max(1, n_changepoints); kmax = 2*(10+3+4) = 34 or fewer when
 * seasonalities are forced off; params row = [k, m, sigma_obs, delta[smax], beta[kmax]]. */
typedef struct pb200_layout {
    int32_t smax;
    int32_t kmax;
    int32_t pstride;      /* doubles per params row = 3 + smax + kmax */
    int32_t meta_i32_stride; /* 8  : T, S, n_changepoints_real, seasonality mask (1 yearly|2 weekly|4 daily), status, iters, n_evals, reserved */
    int32_t meta_i64_stride; /* 2  : start_ns, t_scale_ns */
    int32_t meta_f64_stride; /* 4  : y_scale, floor, cap, neg_log_posterior */
} pb200_layout;

PB200_API int pb200_get_layout(const pb200_options* o, pb200_layout* out);

typedef struct pb200_ctx pb200_ctx;   /* owns a stream, device workspace and pinned staging */

/* Creates a context on CUDA device `device`.  Fails (NULL) when no GPU is present. */
PB200_API pb200_ctx* pb200_create(int device);
PB200_API void pb200_destroy(pb200_ctx* ctx);
PB200_API const char* pb200_last_error(void);
/* cudaStream_t the context launches on (as void*), for event timing by the caller. */
PB200_API void* pb200_stream(pb200_ctx* ctx);
/* number of kernel launches issued by this context so far */
PB200_API int64_t pb200_launch_count(pb200_ctx* ctx);
/* Diagnostics: how many series of the context's LAST fit went to each fit-kernel variant.
 * counts[v*8 + mask], summed over the CTA-width classes; v = 0 feature planes, 1 regular-grid rotation,
 * 2 week-period seasonal table, 3 day-period seasonal table; mask = bit0 yearly | bit1 weekly |
 * bit2 daily.  Synchronises the context's stream. */
/* Diagnostics (host arithmetic, no GPU needed): points per lane the seasonal-table kernel variants give a
 * series of T points whose table period is P grid steps -- the smallest chunk >= ceil(T / 32) for which the 64
 * residual bins the 32 lanes update in one loop step are pairwise distinct (what makes those updates race-free
 * and deterministic) -- or -1 if there is none within the slack the planes workspace allows. */
PB200_API int32_t pb200_tab_chunk(int32_t T, int32_t P);
#define PB200_N_VARIANT_COUNTS 32
PB200_API int pb200_last_fit_variant_counts(pb200_ctx* ctx, int32_t* h_counts);

/*
 * Batched fit: all series of a shard in one call.
 *
 * Input is the reference's (series_id, dim_id, ds, y) frame after grouping
 * (prophet_modeler.py:102-116,139-141) packed as a ragged batch: rows of series
 * i are [offsets[i], offsets[i+1]) of ds / y, sorted by ds ascending (the sort
 * fbprophet's setup_dataframe does), null y rows removed (fbprophet drops them).
 *   d_ds      int64 ns since epoch           [n_rows]
 *   d_y       y values, element type y_dtype [n_rows]
 *   h_offsets int64                          [n_series + 1]  (host copy; the
 *             device copy is made by the call)
 *   floor, cap_multiplier  config model.floor / model.cap_multiplier
 *             (prophet_modeler.py:56-60); cap_i = max(y_i) * cap_multiplier in double.
 *   d_cap     optional explicit per-series cap [n_series] (NULL = use cap_multiplier)
 * Outputs (device, caller-owned, sized per pb200_get_layout):
 *   d_params   double [n_series * pstride]
 *   d_tchange  double [n_series * smax]
 *   d_meta_i32 int32  [n_series * 8]
 *   d_meta_i64 int64  [n_series * 2]
 *   d_meta_f64 double [n_series * 4]
 * Stream-ordered on the context stream; returns after enqueueing.
 */
PB200_API int pb200_fit_device(pb200_ctx* ctx, const pb200_options* opts,
                     const int64_t* d_ds, const void* d_y, int32_t y_dtype,
                     const int64_t* h_offsets, int64_t n_series,
                     double floor, double cap_multiplier, const double* d_cap,
                     double* d_params, double* d_tchange,
                     int32_t* d_meta_i32, int64_t* d_meta_i64, double* d_meta_f64);

/* Same with HOST buffers in and out (pinned or pageable); the call stages
 * through the context's device workspace, copies results back and synchronises. */
PB200_API int pb200_fit_host(pb200_ctx* ctx, const pb200_options* opts,
                   const int64_t* h_ds, const void* h_y, int32_t y_dtype,
                   const int64_t* h_offsets, int64_t n_series,
                   double floor, double cap_multiplier, const double* h_cap,
                   double* h_params, double* h_tchange,
                   int32_t* h_meta_i32, int64_t* h_meta_i64, double* h_meta_f64);

/*
 * Parity-test hook: evaluates the Prophet MAP objective (-log posterior up to constants,
 * the function Stan's L-BFGS minimises) and its gradient at caller-supplied points, through
 * the same kernel code the fit uses.  h_theta / h_grad rows have stride pstride and hold
 * Stan's unconstrained order: k, m, delta[S_i], log(sigma_obs), beta[K_i] packed from 0.
 * h_f[i] = objective, h_meta_i32 as in fit (status PB200_ST_INIT_ERROR when not finite).
 */
PB200_API int pb200_objective_host(pb200_ctx* ctx, const pb200_options* opts,
                   const int64_t* h_ds, const void* h_y, int32_t y_dtype,
                   const int64_t* h_offsets, int64_t n_series,
                   double floor, double cap_multiplier, const double* h_theta,
                   double* h_f, double* h_grad, int32_t* h_meta_i32);

/*
 * Parity-test hook: pb200_fit_host that also records the optimiser's trajectory.  For every accepted
 * L-BFGS iteration it <= trace_cap of series i, h_trace[(i * trace_cap + it - 1) * 4 ...] =
 * (it, f_k, alpha_k, objective evaluations so far) -- the record oracle/prophet_oracle.py::stan_lbfgs(trace=...)
 * produces, so that the two can be compared step by step (a wrong line-search or update constant that still
 * converges shows up in the first rows).  Rows never written stay 0.
 */
PB200_API int pb200_fit_trace_host(pb200_ctx* ctx, const pb200_options* opts,
                   const int64_t* h_ds, const void* h_y, int32_t y_dtype,
                   const int64_t* h_offsets, int64_t n_series,
                   double floor, double cap_multiplier,
                   double* h_params, double* h_tchange,
                   int32_t* h_meta_i32, int64_t* h_meta_i64, double* h_meta_f64,
                   double* h_trace, int32_t trace_cap);

/*
 * Batched predict over `horizon` future timestamps per model.
 *   d_future_ds int64 ns [n_models * horizon]  (make_future_dataframe output,
 *               prophet_scorer.py:64-66; built by pb200_make_future_device or the caller)
 *   d_floor / d_cap  per-model doubles as the scorer reads them back from the
 *               float32 model-table columns (prophet_scorer.py:46-47,67-68)
 * Outputs [n_models * horizon]:
 *   d_yhat        double  trend*(1+multiplicative)+additive
 *   d_yhat_lower / d_yhat_upper  double, MC interval (NULL or uncertainty_samples=0 to skip)
 *   d_yhat_int    int32   (int)yhat, then < floor -> floor   (prophet_scorer.py:73-84)
 * Models whose meta status < 0 produce no forecast: their rows are filled with
 * NaN / INT32_MIN and the caller drops them (empty frame in the reference).
 */
PB200_API int pb200_predict_device(pb200_ctx* ctx, const pb200_options* opts,
                         const double* d_params, const double* d_tchange,
                         const int32_t* d_meta_i32, const int64_t* d_meta_i64,
                         const double* d_meta_f64, int64_t n_models,
                         const int64_t* d_future_ds, int32_t horizon,
                         const double* d_floor, const double* d_cap, uint64_t seed,
                         double* d_yhat, double* d_yhat_lower, double* d_yhat_upper,
                         int32_t* d_yhat_int);

PB200_API int pb200_predict_host(pb200_ctx* ctx, const pb200_options* opts,
                       const double* h_params, const double* h_tchange,
                       const int32_t* h_meta_i32, const int64_t* h_meta_i64,
                       const double* h_meta_f64, int64_t n_models,
                       const int64_t* h_future_ds, int32_t horizon,
                       const double* h_floor, const double* h_cap, uint64_t seed,
                       double* h_yhat, double* h_yhat_lower, double* h_yhat_upper,
                       int32_t* h_yhat_int);

/* future_ds[i*horizon + j] = last_ds[i] + (j+1)*freq_ns  -- make_future_dataframe
 * (include_history=False) for a fixed-width pandas frequency. */
PB200_API int pb200_make_future_device(pb200_ctx* ctx, const int64_t* d_last_ds, int64_t n_models,
                             int32_t horizon, int64_t freq_ns, int64_t* d_future_ds);

PB200_API int pb200_synchronize(pb200_ctx* ctx);

/*
 * Forecast CSV rows formatted on the device: the row formatting of convert_forecasts + write_forecasts
 * (src/jobs/prophet_scorer.py:131-150 -- extract_date per row :107-108, created_timestamp :134, Spark's CSV writer
 * :147-150) for the standard frame
 *     "created_timestamp",series_id,dim_id,"forecast_date","forecast_timestamp",forecast_quantity
 * Two passes: row lengths, then -- given the exclusive scan of the lengths as byte offsets -- the bytes
 * (d_out holds the sum of the lengths).  ds in [1970-01-01, 10000-01-01); created_timestamp at most 64 bytes.
 * pb200_forecast_csv_row_host runs the same row formatter on the host for ONE row (tests; returns the row's
 * length, out must hold 160 bytes).
 */
PB200_API int pb200_forecast_csv_lengths_device(pb200_ctx* ctx, const int32_t* d_series_id, const int32_t* d_dim_id,
                                                const int32_t* d_quantity, int64_t n_rows, int32_t created_len,
                                                int64_t* d_row_len);
PB200_API int pb200_forecast_csv_rows_device(pb200_ctx* ctx, const int32_t* d_series_id, const int32_t* d_dim_id,
                                             const int64_t* d_ds_ns, const int32_t* d_quantity, int64_t n_rows,
                                             const char* h_created, int32_t created_len, const int64_t* d_row_off,
                                             uint8_t* d_out);
PB200_API int32_t pb200_forecast_csv_row_host(int32_t series_id, int32_t dim_id, int64_t ds_ns, int32_t quantity,
                                              const char* created, int32_t created_len, char* out);

/*
 * The modeler's input CSV parsed on the device: header-less lines "dim_id,timestamp,quantity" (reference
 * src/jobs/prophet_modeler.py:12-17,102-116) of files concatenated into one byte buffer d_text, every file ending in
 * '\n'.  d_text is 16-byte aligned and readable up to n_bytes rounded up to 16 (the bytes past n_bytes are ignored).
 * Accepted grammar, everything else is refused:
 *     dim_id     -?[0-9]{1,10} within int32
 *     timestamp  YYYY-MM-DD[ T]HH:MM:SS with an optional '.' and 1..9 fraction digits; year 1900..2199, a valid
 *                calendar date, hour < 24, minute < 60, second < 60
 *     quantity   -?[0-9]{1,10} within int32, or empty (null: quantity 0, valid 0)
 *     line end   "\n" or "\r\n"
 * Passes, in order on the context's stream:
 *   count  d_tile_count[t] = newlines in bytes [t*PB200_INPUT_CSV_TILE, (t+1)*PB200_INPUT_CSV_TILE)
 *          (ceil(n_bytes / PB200_INPUT_CSV_TILE) tiles);
 *   index  given d_tile_off = exclusive scan of the tile counts, d_row_end[r] = offset one past row r's '\n'
 *          (n_rows = sum of the tile counts);
 *   parse  row r starts at d_row_end[r-1] (0 for r = 0); it belongs to the last file f with d_file_start[f] <= that
 *          offset (d_file_start ascending) and gets series_id d_file_sid[f].  Writes the four columns and the
 *          quantity valid mask; d_refused[0] = rows refused, d_refused[1] = index of the first refused row or -1.
 *          A refused row's column values are unspecified.
 * pb200_input_csv_row_host runs the same row parser on the host for ONE line of len bytes (its line end included):
 * 1 accepted, 0 refused, -1 bad argument.
 */
#define PB200_INPUT_CSV_TILE 4096
PB200_API int pb200_input_csv_count_device(pb200_ctx* ctx, const uint8_t* d_text, int64_t n_bytes, int64_t* d_tile_count);
PB200_API int pb200_input_csv_index_device(pb200_ctx* ctx, const uint8_t* d_text, int64_t n_bytes,
                                           const int64_t* d_tile_off, int64_t* d_row_end);
PB200_API int pb200_input_csv_parse_device(pb200_ctx* ctx, const uint8_t* d_text, const int64_t* d_row_end, int64_t n_rows,
                                           const int64_t* d_file_start, const int32_t* d_file_sid, int32_t n_files,
                                           int32_t* d_series_id, int32_t* d_dim_id, int64_t* d_ds_ns, int32_t* d_quantity,
                                           uint8_t* d_quantity_valid, int64_t* d_refused);
PB200_API int32_t pb200_input_csv_row_host(const char* line, int64_t len, int32_t* dim_id, int64_t* ds_ns,
                                           int32_t* quantity, int32_t* quantity_valid);

#ifdef __cplusplus
}
#endif
#endif /* PROPHET_B200_H */
