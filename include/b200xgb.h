/*
 * b200xgb.h -- C ABI of libb200xgb.so: a B200-native (sm_100a) gradient-boosted-tree trainer / predictor.
 *
 * DROP-IN BOUNDARY.  The SageMaker XGBoost container (aws/sagemaker-xgboost-container) never calls C directly:
 * it imports the `xgboost` Python package, which binds libxgboost's C API (include/xgboost/c_api.h of
 * xgboost==3.0.5, docker/3.0-5/base/Dockerfile.cpu:33) with ctypes.  The entry points below are the subset of
 * that C API the container's hot path reaches, with the same names, argument meaning, ownership and error
 * convention, so the same ctypes binding works against this library (see INTEGRATION.md).  Each declaration
 * cites the reference call site (file:line under /root/reference/src/sagemaker_xgboost_container) that
 * reaches it through the Python package.
 *
 * Conventions (identical to libxgboost):
 *   - every function returns 0 on success, -1 on failure; XGBGetLastError() returns the thread-local message;
 *   - handles are opaque; out-pointers (strings, float arrays, shapes) are owned by the handle / a thread-local
 *     buffer and stay valid until the next call on the same handle from the same thread;
 *   - all buffers passed in are HOST memory; the library copies them to the GPU.  There is NO CPU fallback:
 *     without a CUDA device every call that needs one fails with an error.
 */
#ifndef B200XGB_H_
#define B200XGB_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define XGB_DLL __attribute__((visibility("default")))
#else
#define XGB_DLL
#endif

typedef void* DMatrixHandle;
typedef void* BoosterHandle;
typedef uint64_t bst_ulong;

XGB_DLL const char* XGBGetLastError(void);
/* fills major/minor/patch of the xgboost API level this library mirrors (3.0.5) */
XGB_DLL void XGBoostVersion(int* major, int* minor, int* patch);
/* JSON describing the build: {"USE_CUDA": true, "arch": "sm_100a", ...} */
XGB_DLL int XGBuildInfo(const char** out);

/* ---- DMatrix: data_utils.py:309-313,361,384,453 ; encoder.py:52,76,87,98 ; serve_utils.py:137,205 ---------- */
/* dense row-major float matrix, `missing` marks absent values (NaN is always missing) */
/* upstream's Python package passes ndarray inputs as `__array_interface__` JSON ({"data":[ptr,ro],"shape":[n,m],"typestr":"<f4"}),
 * config {"missing": NaN, "nthread": 0}; data_utils.py:384 (Parquet -> numpy), encoder.py:52 (CSV payload) reach it */
XGB_DLL int XGDMatrixCreateFromDense(const char* data, const char* config, DMatrixHandle* out);
/* labels / weights / base_margin from an array interface (DMatrix(label=...), data_utils.py:384) */
XGB_DLL int XGDMatrixSetInfoFromInterface(DMatrixHandle handle, const char* field, const char* data);
/* {"uri": "<path>?format=csv&label_column=0[&weight_column=1][&delimiter=,]" | "<path>?format=libsvm"}: data_utils.py:309-313,361;
 * a directory means every regular file in it (data_utils.py:520-545); CSV text is parsed on the device */
XGB_DLL int XGDMatrixCreateFromURI(const char* config, DMatrixHandle* out);
XGB_DLL int XGDMatrixCreateFromMat(const float* data, bst_ulong nrow, bst_ulong ncol, float missing, DMatrixHandle* out);
/* CSR; num_col = 0 means "infer from the indices" (libsvm loader: indices kept as-is, data_utils.py:348-365) */
XGB_DLL int XGDMatrixCreateFromCSREx(const size_t* indptr, const unsigned* indices, const float* data, size_t nindptr,
                             size_t nelem, size_t num_col, DMatrixHandle* out);
/* device-resident input (what the reference's GPU path feeds through cupy/cudf, distributed_gpu/dask_data_utils.py:71-78):
 * `data` is a JSON __cuda_array_interface__ {"data":[ptr,ro],"shape":[n,F],"typestr":"<f4"[,"strides":null]},
 * config JSON {"missing": NaN} */
XGB_DLL int XGDMatrixCreateFromCudaArrayInterface(const char* data, const char* config, DMatrixHandle* out);
XGB_DLL int XGDMatrixFree(DMatrixHandle handle);
XGB_DLL int XGDMatrixNumRow(DMatrixHandle handle, bst_ulong* out);                                   /* train.py:339-342 */
XGB_DLL int XGDMatrixNumCol(DMatrixHandle handle, bst_ulong* out);
/* field: "label" | "weight" | "base_margin" */
XGB_DLL int XGDMatrixSetFloatInfo(DMatrixHandle handle, const char* field, const float* array, bst_ulong len);
XGB_DLL int XGDMatrixGetFloatInfo(DMatrixHandle handle, const char* field, bst_ulong* out_len, const float** out_dptr); /* train.py:394-396 get_label */
XGB_DLL int XGDMatrixSliceDMatrix(DMatrixHandle handle, const int* idxset, bst_ulong len, DMatrixHandle* out);          /* train.py:410-411 */
/* field: "feature_name" | "feature_type" */
XGB_DLL int XGDMatrixSetStrFeatureInfo(DMatrixHandle handle, const char* field, const char** features, bst_ulong size);
XGB_DLL int XGDMatrixGetStrFeatureInfo(DMatrixHandle handle, const char* field, bst_ulong* size, const char*** out_features);

/* ---- Booster: train.py:367-376,432-442 (xgb.train) ; checkpointing.py:74 ------------------------------------ */
XGB_DLL int XGBoosterCreate(const DMatrixHandle dmats[], bst_ulong len, BoosterHandle* out);
XGB_DLL int XGBoosterFree(BoosterHandle handle);
XGB_DLL int XGBoosterSetParam(BoosterHandle handle, const char* name, const char* value);
/* one boosting round of the configured objective on dtrain (the hot path) */
XGB_DLL int XGBoosterUpdateOneIter(BoosterHandle handle, int iter, DMatrixHandle dtrain);
/* custom objective: not implemented on the device path, returns -1 */
XGB_DLL int XGBoosterBoostOneIter(BoosterHandle handle, DMatrixHandle dtrain, float* grad, float* hess, bst_ulong len);
/* "[iter]\t<name>-<metric>:<value>..." -- callback.py:85 EvaluationMonitor parses this */
XGB_DLL int XGBoosterEvalOneIter(BoosterHandle handle, int iter, DMatrixHandle dmats[], const char* evnames[], bst_ulong len,
                         const char** out_result);
/* config JSON: {"type": 0 value | 1 margin | 6 leaf, "training": bool, "iteration_begin": int,
 *               "iteration_end": int, "strict_shape": bool}
 * serve_utils.py:244-250, serving.py:98, handler_service.py:73, train.py:445 */
XGB_DLL int XGBoosterPredictFromDMatrix(BoosterHandle handle, DMatrixHandle dmat, const char* config,
                                bst_ulong const** out_shape, bst_ulong* out_dim, float const** out_result);
/* file name extension picks the format: .json -> JSON text, anything else (incl. none) -> UBJSON  (train.py:480) */
XGB_DLL int XGBoosterSaveModel(BoosterHandle handle, const char* fname);
XGB_DLL int XGBoosterLoadModel(BoosterHandle handle, const char* fname);                              /* serve_utils.py:184-185 */
/* config JSON: {"format": "ubj" | "json"} */
XGB_DLL int XGBoosterSaveModelToBuffer(BoosterHandle handle, const char* config, bst_ulong* out_len, const char** out_dptr);
XGB_DLL int XGBoosterLoadModelFromBuffer(BoosterHandle handle, const void* buf, bst_ulong len);
/* model + configuration, used for pickling (serve_utils.py:180-182 pickle.load of a Booster) */
XGB_DLL int XGBoosterSerializeToBuffer(BoosterHandle handle, bst_ulong* out_len, const char** out_dptr);
XGB_DLL int XGBoosterUnserializeFromBuffer(BoosterHandle handle, const void* buf, bst_ulong len);
XGB_DLL int XGBoosterSaveJsonConfig(BoosterHandle handle, bst_ulong* out_len, const char** out_str);  /* serve.py:85-88 */
XGB_DLL int XGBoosterLoadJsonConfig(BoosterHandle handle, const char* config);
XGB_DLL int XGBoosterGetNumFeature(BoosterHandle handle, bst_ulong* out);
XGB_DLL int XGBoosterBoostedRounds(BoosterHandle handle, int* out);
XGB_DLL int XGBoosterSlice(BoosterHandle handle, int begin_layer, int end_layer, int step, BoosterHandle* out); /* EarlyStopping save_best */
XGB_DLL int XGBoosterGetAttr(BoosterHandle handle, const char* key, const char** out, int* success);  /* best_iteration */
XGB_DLL int XGBoosterSetAttr(BoosterHandle handle, const char* key, const char* value);               /* value NULL deletes */
XGB_DLL int XGBoosterGetAttrNames(BoosterHandle handle, bst_ulong* out_len, const char*** out);
XGB_DLL int XGBoosterSetStrFeatureInfo(BoosterHandle handle, const char* field, const char** features, bst_ulong size);
XGB_DLL int XGBoosterGetStrFeatureInfo(BoosterHandle handle, const char* field, bst_ulong* len, const char*** out_features);

/* ---- collective: distributed.py:119-136,219-220,238-243 (xgboost.collective) --------------------------------- */
/* config JSON: {"nccl_unique_id": "<hex, 128 bytes>", "rank": r, "world_size": w}; the id comes from
 * XGCommunicatorGetUniqueId on rank 0 and is shipped by the Python-side bootstrap (tracker / torch.distributed). */
XGB_DLL int XGCommunicatorInit(const char* config);
/* broadcast of a host buffer from `root` (distributed.py:119-136 via xgboost.collective.broadcast) */
XGB_DLL int XGCommunicatorBroadcast(void* send_receive_buffer, size_t size, int root);
XGB_DLL int XGCommunicatorFinalize(void);
XGB_DLL int XGCommunicatorGetRank(void);
XGB_DLL int XGCommunicatorGetWorldSize(void);
XGB_DLL int XGCommunicatorGetUniqueId(const char** out_hex);

/* ---- build-specific introspection (no libxgboost counterpart; used by tests/ and bench.py) -------------------- */
/* cuts as an explicit artefact shared with the oracle: ptrs[F+1], vals[ptrs[F]], mins[F] */
XGB_DLL int XGB200DMatrixGetCuts(DMatrixHandle handle, int max_bin, bst_ulong* n_ptrs, const int** ptrs, bst_ulong* n_vals,
                         const float** vals, const float** mins, int* has_missing);
XGB_DLL int XGB200DMatrixSetCuts(DMatrixHandle handle, const int* ptrs, bst_ulong n_ptrs, const float* vals, const float* mins);
/* Serving input path (SURVEY.md 8f-1): a CSV request body parsed on the device into the DMatrix.  Replaces the Python
 * split + np.array(...).astype(float) of encoder.csv_to_dmatrix (encoder.py:35-52, reached from serve_utils.py:121-131).
 * `text` is the stripped payload ('\n' between rows, `delimiter` between fields, empty field = NaN).  *status: 0 = parsed,
 * 1 = rows of different lengths, 2 = a field the exact device fast path cannot decide (caller parses on the host);
 * *out is NULL unless *status == 0. */
XGB_DLL int XGB200DMatrixCreateFromCSV(const char* text, bst_ulong len, char delimiter, int* status, DMatrixHandle* out);
/* Training loaders to the device (SURVEY.md 8f-2): the text of a CSV channel ("<dir>?format=csv&label_column=0[&weight_column=1]",
 * data_utils.py:289-318) parsed on the GPU; label_column / weight_column (-1 = none) become the "label" / "weight" float
 * info, the other columns the feature matrix.  Same status convention as XGB200DMatrixCreateFromCSV. */
XGB_DLL int XGB200DMatrixCreateFromCSVEx(const char* text, bst_ulong len, char delimiter, int label_column, int weight_column,
                             int* status, DMatrixHandle* out);
/* 1 when the per-level histogram all-reduce runs as the NVLink peer-memory kernel (nvlink.cu), 0 when it goes through NCCL */
/* A libsvm request body ("label idx:val ..." lines, already stripped) parsed on the device into a dense matrix.
 * whitespace_mode 0 / absent NaN = serve_utils._get_sparse_matrix_from_libsvm + xgb.DMatrix(csr) (algorithm_mode/serve_utils.py:94-118,
 * 132-137: tokens split on ' ', entries a line does not list are missing); whitespace_mode 1 / absent 0 = encoder.libsvm_to_dmatrix
 * (encoder.py:54-86: split on any whitespace, dense zeros).  Indices shift to 0-based when the smallest one is >= 1, as both do.
 * *status: 0 ok; 2 = the body holds something the Python routes treat specially (non-digit index, literal outside the exact
 * fast path, repeated index in a line, trailing empty lines ...): take the host route; 3 = no entry at all (ditto). */
XGB_DLL int XGB200DMatrixCreateFromLibsvmText(const char* text, bst_ulong len, int whitespace_mode, float absent, int* status, DMatrixHandle* out);
XGB_DLL int XGB200CommPeerReduceActive(void);
/* Columnar training input without a dense float32 matrix on the host (Parquet through pyarrow, pandas frames): `ncols` host
 * buffers of `nrow` items each, col_types[c] in {0 f32, 1 f64, 2 i32, 3 i64, 4 u8, 5 i8, 6 i16, 7 u16, 8 u32, 9 u64, 10 bool};
 * the buffers cross PCIe as they are and are converted (round to nearest, like numpy's astype(float32)) and transposed into
 * the row-major matrix on the device (ingest.cu).  label_column / weight_column (-1 = none) become the label / weight info.
 * Replaces the host copies of data_utils.get_parquet_dmatrix (data_utils.py:368-390: read_table -> to_pandas -> to_numpy ->
 * data[:, 1:]) in front of XGDMatrixCreateFromMat. */
XGB_DLL int XGB200DMatrixCreateFromColumns(const void* const* cols, const int* col_types, int ncols, bst_ulong nrow, int label_column,
                                   int weight_column, DMatrixHandle* out);
/* the float32 feature matrix as the engine holds it (row-major n x F, NaN = missing), for bit-exact checks of the input paths */
XGB_DLL int XGB200DMatrixGetRaw(DMatrixHandle handle, float* out_row_major);
/* binned feature blocks back on the host in plain row-major n x F order (for bit-exact checks of the binning kernel) */
XGB_DLL int XGB200DMatrixGetBins(DMatrixHandle handle, int max_bin, uint8_t* out_row_major);
/* flat tree arrays of the model; any pointer may be NULL. tree_offset has num_trees+1 entries. */
XGB_DLL int XGB200BoosterModelShape(BoosterHandle handle, bst_ulong* num_trees, bst_ulong* num_nodes, float* base_score, int* num_class);
XGB_DLL int XGB200BoosterExportModel(BoosterHandle handle, int64_t* tree_offset, int32_t* tree_info, int32_t* left, int32_t* right,
                             int32_t* parent, int32_t* split_index, int32_t* split_bin, uint8_t* default_left,
                             float* split_cond, float* base_weight, float* loss_chg, float* sum_hess);
/* root histogram of `dmat` for host gradient pairs (n x 2 floats): out_hist is int64 [F][256][2] fixed point,
 * scales[4] = {sg, sh, 1/sg, 1/sh}; the kernel is launched `repeats` times and its mean device time returned. */
XGB_DLL int XGB200BuildRootHistogram(BoosterHandle handle, DMatrixHandle dmat, const float* gpair, int repeats,
                             int64_t* out_hist, float* scales, float* out_ms);
/* same with a kernel choice and an optional row subset: mode 0 = production choice (TMA-staged root kernel), 1 = gather
 * kernel, 2 = G-only TMA root kernel (constant-hessian fast path: the H plane of out_hist stays zero).  With row_ids
 * (n_ids entries, ascending or not) the histogram covers that subset and gpair is given by POSITION (gpair[i] belongs to
 * row row_ids[i]) -- the deeper tree levels' access pattern.  out_kernel: name of the kernel variant that ran. */
XGB_DLL int XGB200BuildHistogramEx(BoosterHandle handle, DMatrixHandle dmat, const float* gpair, int repeats, int mode,
                             const unsigned* row_ids, bst_ulong n_ids, int64_t* out_hist, float* scales, float* out_ms,
                             const char** out_kernel);
/* mean device time (CUDA events) of the predictor kernel alone over `repeats` launches on `dmat` */
XGB_DLL int XGB200BoosterPredictKernelMs(BoosterHandle handle, DMatrixHandle dmat, int repeats, float* out_ms);
/* The predictor's launch plan as JSON: {"route": "tiled" | "thread_per_row", "kernel": ..., "pitch": floats per staged row,
 * "absent_features": bool (the matrix is narrower than the model), "node_budget": bytes, "smem_limit": bytes,
 * "chunks": [{"tree_lo", "tree_hi", "rows", "threads", "head", "smem"}, ...]}, chunks in tree order covering
 * [tree_begin, tree_end) on the tiled route.  XGB200PredictPlan is host code only (no device needed): node_counts holds the
 * node slots of trees tree_begin .. tree_end-1.  XGB200BoosterPredictPlan reports the plan XGBoosterPredictFromDMatrix runs
 * on `dmat` for the iteration range [iteration_begin, iteration_end) (0, 0 = all rounds), from the model's device slot sizes.
 * *out_json is a thread-local buffer (the handle's, for the Booster form), valid until the next string-returning call. */
XGB_DLL int XGB200PredictPlan(int data_features, int model_features, const int64_t* node_counts, int tree_begin, int tree_end,
                              int children_adjacent, const char** out_json);
XGB_DLL int XGB200BoosterPredictPlan(BoosterHandle handle, DMatrixHandle dmat, int iteration_begin, int iteration_end,
                                     const char** out_json);
/* raw margins of the prediction cache the trainer keeps for `dmat` (n x num_class), brought up to date first */
XGB_DLL int XGB200BoosterGetCachedMargin(BoosterHandle handle, DMatrixHandle dmat, float* out);
/* CUDA-event stopwatch on the engine's stream: Start records an event, Stop records another, waits, returns ms */
XGB_DLL int XGB200TimerStart(void);
XGB_DLL int XGB200TimerStop(float* out_ms);
/* per-kernel profile of the tree builder: enable, run rounds, then read
 * {"hist_ms":..,"hist_launches":..,"hist_rows":..,"root_hist_ms":..,"root_hist_launches":..,"root_hist_rows":..,"launches":..} */
XGB_DLL int XGB200BoosterSetProfile(BoosterHandle handle, int enable);
XGB_DLL int XGB200BoosterGetProfile(BoosterHandle handle, const char** out_json);
/* number of CUDA kernels this library has launched so far in this process */
XGB_DLL int XGB200LaunchCount(long long* out);
/* wait for all device work queued by this library */
XGB_DLL int XGB200Synchronize(void);
/* Host-only converter: a pre-JSON binary model (Booster.save_model of xgboost < 2, optionally behind the "CONFIG-offset:"
 * prefix of a pickled 1.x Booster) -> the UBJSON model document XGBoosterLoadModelFromBuffer reads.  The loaders call the
 * same code internally (legacy_io.cc); exported so that old model archives can be migrated, and checked, without a GPU.
 * Replaces: libxgboost's LearnerIO::LoadModel legacy branch behind serve_utils.get_loaded_booster
 * (algorithm_mode/serve_utils.py:171-197; fixtures test/resources/models/{saved_booster,pickled_model}).
 * *out is a thread-local buffer, valid until the next call of this function on the same thread. */
XGB_DLL int XGB200LegacyModelToUBJ(const void* buf, bst_ulong len, bst_ulong* out_len, const char** out);

#ifdef __cplusplus
}
#endif
#endif /* B200XGB_H_ */
