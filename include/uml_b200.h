/*
 * uml_b200.h - C ABI of the B200-native batch-prediction engine for UnionML's predict hot path.
 *
 * The reference (unionai-oss/unionml) is pure Python and has no FFI of its own; the single call this library stands
 * behind is the plugin boundary
 *
 *     predictions = self._predictor(model_object, features)      unionml/model.py:606 and unionml/model.py:642
 *
 * whose canonical body is `[float(x) for x in estimator.predict(features)]` (README.md:87-92), i.e. scikit-learn's
 * LinearClassifierMixin.predict (sklearn/linear_model/_base.py:366-427):  X @ coef_.T + intercept_ -> argmax -> take.
 * Each entry point below names the reference interface it replaces.  Plain pointers and sizes only - no torch,
 * numpy or CUDA types cross this boundary (streams and device pointers travel as void* / raw addresses).
 *
 * Conventions: every function returns a uml_status (0 = ok); uml_last_error() gives the text for the last failure on
 * that engine; handles are created/destroyed by the caller; `features`/`coef` buffers are borrowed for the duration of
 * the call only and never written (model.py:608-612 hands the same objects to callbacks afterwards).
 * One engine = one CUDA device = one process rank (one process per GPU; multi-GPU plumbing is torch.distributed/NCCL
 * above this ABI).  The CUDA context is created lazily by uml_engine_create, never at library load (uvicorn workers
 * fork, cli.py:289).  Calls on one engine must be serialised by the caller (the reference's /predict is
 * single-threaded per worker, fastapi.py:51-64).
 */
#ifndef UML_B200_H
#define UML_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UML_B200_ABI_VERSION 2

#if defined(__GNUC__)
#define UML_API __attribute__((visibility("default")))
#else
#define UML_API
#endif

typedef struct uml_engine uml_engine; /* device + stream + scratch                                   */
typedef struct uml_model uml_model;   /* linear classifier: coef_/intercept_ staged on the device     */
typedef struct uml_mlp uml_mlp;       /* 2-layer MLP classifier (PytorchModel of the torch quickstart) */
typedef struct uml_batch uml_batch;   /* a feature batch resident in HBM as fp32 row-major            */

typedef enum uml_status {
  UML_OK = 0,
  UML_ERR_INVALID = 1,     /* bad argument (NULL handle, negative size, ...)                                       */
  UML_ERR_CUDA = 2,        /* CUDA runtime/driver failure; text in uml_last_error                                  */
  UML_ERR_NONFINITE = 3,   /* NaN/Inf in the features: sklearn raises ValueError (utils/validation.py:107)         */
  UML_ERR_SHAPE = 4,       /* feature count differs from the model's n_features_in_ (utils/validation.py:2868)     */
  UML_ERR_NOMEM = 5,
  UML_ERR_UNSUPPORTED = 6, /* layout/dtype combination the engine does not take (caller should make it contiguous) */
  UML_ERR_NO_DEVICE = 7    /* no CUDA device: the product path fails loudly, there is no CPU fallback              */
} uml_status;

typedef enum uml_dtype { UML_F32 = 0, UML_F64 = 1, UML_I64 = 2, UML_I32 = 3, UML_U8 = 4 } uml_dtype;

/* uml_stage_rows flags */
#define UML_STAGE_KEEP_F64 1u  /* keep a float64 copy when the fp32 staging is lossy, so exact mode can re-score from it */
#define UML_STAGE_SKIP_FINITE_CHECK 2u

/* uml_*_predict modes */
#define UML_PREDICT_FAST 0   /* fp32 scores, argmax; no guarantee on near-ties                                     */
#define UML_PREDICT_EXACT 1  /* labels equal the argmax of the exactly-rounded float64 scores (sklearn's f64 path) */

typedef struct uml_stats {
  int64_t n_rows;
  int64_t n_flagged;    /* rows whose fp32 top-2 margin was inside the proven fp32 error bound -> re-scored in fp64   */
  int64_t n_ambiguous;  /* of those, rows whose fp64 margin is inside the fp64 bound (true ties / sub-1e-13 gaps)      */
  int64_t n_nonfinite;  /* rows containing NaN/Inf (call fails with UML_ERR_NONFINITE when > 0)                        */
  double kernel_ms;     /* CUDA-event time of the scoring kernel(s) of this call                                      */
  double recheck_ms;    /* CUDA-event time of the fp64 re-score kernel                                                */
  double total_ms;      /* CUDA-event time of the whole call on the engine stream (incl. copies when host buffers)    */
  int64_t h2d_bytes;
  int64_t d2h_bytes;
  int32_t kernel_launches; /* kernels of this library launched by the call                                            */
  int32_t path;            /* 1 = TMA fp32 tile kernel, 2 = generic fp64 kernel, 3 = MLP CUDA-core kernel, 5 = MLP tensor-core
                              (tcgen05) kernel, 4 = small-batch fp64
                              kernel of the online path (<= 64 rows: zero-copy request buffer, one kernel replayed as a CUDA graph)                 */
} uml_stats;

typedef struct uml_device_info {
  int32_t device_id, sm_count, cc_major, cc_minor;
  int64_t total_mem_bytes, l2_bytes;
  int32_t sm_clock_khz, mem_clock_khz;
  char name[64];
} uml_device_info;

/* ---- engine -------------------------------------------------------------------------------------------------- */
UML_API int uml_abi_version(void);
/* lazy per-process device binding; replaces nothing in the reference (it is CPU-only) - cf. fastapi.py:22-34 startup */
UML_API int uml_engine_create(uml_engine** out, int device_id);
UML_API void uml_engine_destroy(uml_engine* e);
UML_API const char* uml_last_error(const uml_engine* e); /* e may be NULL: last error of a failed uml_engine_create          */
UML_API int uml_engine_info(const uml_engine* e, uml_device_info* out);
/* run on the caller's stream (a cudaStream_t passed as void*), e.g. torch.cuda.current_stream().cuda_stream; NULL
 * restores the engine's own non-blocking stream */
UML_API int uml_engine_set_stream(uml_engine* e, void* cuda_stream);
UML_API int uml_engine_synchronize(uml_engine* e);
/* pinned host memory for feature frames / label vectors (what `bench.py` e2e and the serving path stage through) */
UML_API int uml_host_alloc(uml_engine* e, void** out, int64_t bytes);
UML_API int uml_host_free(uml_engine* e, void* p);
/* plain device memory (label vectors for callers that do not bring their own allocator) */
UML_API int uml_device_alloc(uml_engine* e, void** out, int64_t bytes);
UML_API int uml_device_free(uml_engine* e, void* p);

/* ---- model: where W, b come from - joblib.load(file)["model_obj"].coef_/intercept_ (model.py:1498-1500) -------- */
/* coef: n_classes x n_features row-major (sklearn coef_; a binary model passes its single row with n_classes = 1 and
 * gets the `scores > 0` rule of _base.py:416); intercept: n_classes; dtype UML_F32 or UML_F64. */
UML_API int uml_linear_load(uml_engine* e, uml_model** out, const void* coef, const void* intercept, int n_classes,
                    int n_features, int dtype);
UML_API void uml_model_free(uml_model* m);
/* optional per-feature affine folded in front of the dot product: x' = (x - shift) * scale  (StandardScaler of
 * docs/tutorials/mnist.md:116-124; a @dataset.feature_transformer affine).  NULL pointers = identity. */
UML_API int uml_linear_set_affine(uml_engine* e, uml_model* m, const double* shift, const double* scale);

/* ---- batch: Dataset.get_features output (dataset.py:350-359) staged once into HBM ---------------------------- */
/* host rows -> device fp32 row-major (transpose / down-cast on the GPU).  Strides are in bytes; a pandas block is
 * feature-major (col_stride < row_stride is NOT required: either order is taken).  Checks finiteness like
 * check_array (validation.py:107) unless UML_STAGE_SKIP_FINITE_CHECK. */
UML_API int uml_stage_rows(uml_engine* e, uml_batch** out, const void* host_ptr, int64_t n_rows, int n_features,
                   int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, uint32_t flags);
/* wrap rows that already live in HBM (fp32, row-major, leading dimension ld floats, ld % 4 == 0, 16-byte aligned) */
UML_API int uml_batch_from_device(uml_engine* e, uml_batch** out, const void* dev_ptr, int64_t n_rows, int n_features,
                          int64_t ld);
UML_API int uml_batch_info(const uml_batch* b, int64_t* n_rows, int* n_features, int64_t* ld, const void** dev_ptr,
                   int* lossless);
UML_API void uml_batch_free(uml_batch* b);

/* ---- predict: replaces estimator.predict(features) of the canonical predictor (README.md:92) ----------------- */
/* labels_out receives the argmax *index* per row (int32); the caller applies classes_.take (_base.py:423).
 * labels_on_device != 0: labels_out is a device pointer and the call is asynchronous on the engine stream unless
 * stats != NULL (reading the counters synchronises). */
UML_API int uml_linear_predict(uml_engine* e, const uml_model* m, const uml_batch* b, int32_t* labels_out,
                       int labels_on_device, int mode, uml_stats* stats);
/* fused compute + collective: every rank's kernel epilogue stores its labels straight into all peers' label vectors
 * over NVLink (peer_labels[0] = base of THIS rank's full-length vector, peer_labels[1..] = the other ranks' vectors,
 * already mapped for peer access; this rank's rows land at row_offset in each).  label_bytes = 4: int32 vectors;
 * label_bytes = 1 (n_classes <= 256): uint8 vectors - a 128-row tile leaves as one 128-byte store per peer.
 * Replaces kernel + ncclAllGather; the caller still needs one cross-rank barrier before reading peers' rows. */
UML_API int uml_linear_predict_peers(uml_engine* e, const uml_model* m, const uml_batch* b, void* const* peer_labels,
                             int n_peers, int64_t row_offset, int label_bytes, int mode, uml_stats* stats);
/* label post-processing on the device (labels_dev: int32 or uint8 class indices in device memory):
 * uml_labels_take        - classes_.take(indices) (sklearn/linear_model/_base.py:423) + the float conversion of the
 *                          canonical predictor (README.md:92): out_host[i] = classes_host[label[i]] as float64;
 * uml_labels_count_equal - rows whose predicted class value equals targets_host[i]: the numerator of the reference
 *                          evaluator's accuracy_score (README.md:94-100). */
UML_API int uml_labels_take(uml_engine* e, const void* labels_dev, int label_bytes, int64_t n, const double* classes_host,
                    int n_classes, double* out_host);
UML_API int uml_labels_count_equal(uml_engine* e, const void* labels_dev, int label_bytes, int64_t n,
                           const double* classes_host, int n_classes, const double* targets_host, int64_t* count_out);
/* second half of the two-step exchange: copy `bytes` of this rank's label slice (device memory) into each dst[i]
 * (peer-mapped vectors, or one NVLS multicast alias that reaches every rank) on the engine stream.  Used after a
 * uml_linear_predict_peers that targeted only the local vector, when a thin copy kernel beats in-epilogue stores. */
UML_API int uml_labels_push(uml_engine* e, const void* src, void* const* dst, int n_dst, int64_t bytes);
/* end to end from HOST rows to HOST labels in one call (the /predict and Model.predict(features=...) shape): chunked
 * H2D, staging kernel, scoring kernel and label D2H pipelined on two streams; never holds more than a few chunks in
 * HBM.  host_ptr/labels_out may be pageable or pinned (uml_host_alloc); large pageable sources are gathered into pinned
 * bounce buffers by a few host threads.  In exact mode rows inside the fp32 error bound are re-scored in float64 from
 * the caller's own values (float64 / int64 / int32 features that do not survive the fp32 down-cast included).  Batches
 * of <= 64 rows (the /predict shape, fastapi.py:50-64) take a one-kernel float64 route replayed as a CUDA graph. */
UML_API int uml_linear_predict_host(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows, int n_features,
                            int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                            int mode, int64_t chunk_rows, uml_stats* stats);

/* the same call returning `classes_[idx]` as float64 per row (sklearn/linear_model/_base.py:423 + the float conversion
 * of the canonical predictor, README.md:92) - the take runs on the device per chunk and the values travel back instead
 * of the indices.  classes_host: n_classes float64 values (a binary model passes its 2 classes). */
UML_API int uml_linear_predict_host_values(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows,
                                   int n_features, int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype,
                                   const double* classes_host, int n_classes, double* values_out, int mode,
                                   int64_t chunk_rows, uml_stats* stats);
/* asynchronous form of uml_linear_predict_host: _begin returns at once and the pipeline runs on a library thread;
 * uml_async_poll reports how long a prefix of labels_out is final (the caller may read it - the Python predictor fills
 * the List[float] of the predictor contract from it while the rest of the batch is still in flight); uml_async_finish
 * joins and returns the call's status (UML_ERR_NONFINITE ...) and stats.  One asynchronous call per engine; no other
 * call on the engine until _finish.  host_ptr / labels_out must stay valid until then. */
UML_API int uml_linear_predict_host_begin(uml_engine* e, const uml_model* m, const void* host_ptr, int64_t n_rows,
                                  int n_features, int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype,
                                  int32_t* labels_out, int mode, int64_t chunk_rows);
UML_API int uml_async_poll(uml_engine* e, int64_t* rows_done, int* finished);
UML_API int uml_async_finish(uml_engine* e, uml_stats* stats);
/* class probabilities of a resident batch: LogisticRegression.predict_proba (sklearn/linear_model/_logistic.py) =
 * softmax of decision_function (sigmoid for the binary layout: columns [1 - p, p]).  fp32 scores and exp;
 * proba_out: n_rows x n_classes row-major fp32 (n_classes = 2 for a binary model), host or device memory. */
UML_API int uml_linear_predict_proba(uml_engine* e, const uml_model* m, const uml_batch* b, float* proba_out,
                             int proba_on_device);

/* ---- 2-layer MLP predictor (tests/integration/pytorch_app/quickstart.py:14-24,68-70) -------------------------- */
/* w1: hidden x in, b1: hidden, w2: out x hidden, b2: out (torch nn.Linear layout, fp32).  Labels = argmax of
 * softmax(W2 relu(W1 x + b1) + b2) = argmax of the logits. */
UML_API int uml_mlp_load(uml_engine* e, uml_mlp** out, const float* w1, const float* b1, const float* w2, const float* b2,
                 int n_in, int n_hidden, int n_out);
UML_API void uml_mlp_free(uml_mlp* m);
UML_API int uml_mlp_predict(uml_engine* e, const uml_mlp* m, const uml_batch* b, int32_t* labels_out, int labels_on_device,
                    int mode, uml_stats* stats);

/* the MLP predictor from HOST rows through the same chunk pipeline as uml_linear_predict_host (pinned bounce buffers,
 * GPU transpose / down-cast to fp32 - the reference predictor casts features to float32 -, scoring kernel, fp64
 * re-score): labels_out[i] = the argmax class index of row i, what `module(features).argmax(1)` yields
 * (quickstart.py:68-70).  _begin is the asynchronous form (uml_async_poll / uml_async_finish as for the linear call). */
UML_API int uml_mlp_predict_host(uml_engine* e, const uml_mlp* m, const void* host_ptr, int64_t n_rows, int n_features,
                         int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out, int mode,
                         int64_t chunk_rows, uml_stats* stats);
UML_API int uml_mlp_predict_host_begin(uml_engine* e, const uml_mlp* m, const void* host_ptr, int64_t n_rows, int n_features,
                               int64_t row_stride_bytes, int64_t col_stride_bytes, int src_dtype, int32_t* labels_out,
                               int mode, int64_t chunk_rows);
/* fused compute + collective for the MLP predictor: same contract as uml_linear_predict_peers (labels of this rank's
 * rows are stored into every entry of peer_labels at row_offset from the kernel epilogue; int32 or uint8 vectors).
 * Batches whose features are tf32 values (integer / pixel domains) run layer 1 on the tensor cores (tcgen05, stats
 * path 5); other batches take the CUDA-core kernel (path 3) and a thin scatter kernel. */
UML_API int uml_mlp_predict_peers(uml_engine* e, const uml_mlp* m, const uml_batch* b, void* const* peer_labels, int n_peers,
                          int64_t row_offset, int label_bytes, int mode, uml_stats* stats);
/* class probabilities of the MLP: what PytorchModel.forward returns (quickstart.py:14-24), softmax of the logits, fp32
 * (m = max z, e_c = exp(z_c - m), p_c = e_c / sum e).  The kernel is chosen as for uml_mlp_predict: tensor cores for
 * batches of tf32 values (stats path 5), CUDA cores for other batches (path 3), an fp64 kernel for shapes neither
 * takes (path 2).  Rows the fast kernels cannot score (features that are not tf32 values on path 5, NaN/Inf) are
 * recomputed in fp64 (stats n_flagged).  A row with NaN/Inf returns UML_ERR_NONFINITE, wrapped device rows included.
 * proba_out: n_rows x n_out row-major fp32, host or (proba_on_device != 0) device memory, 16-byte aligned on the device
 * (UML_ERR_UNSUPPORTED otherwise).  stats may be NULL; the call is synchronous either way. */
UML_API int uml_mlp_predict_proba(uml_engine* e, const uml_mlp* m, const uml_batch* b, float* proba_out,
                                  int proba_on_device, uml_stats* stats);

#ifdef __cplusplus
}
#endif
#endif /* UML_B200_H */
