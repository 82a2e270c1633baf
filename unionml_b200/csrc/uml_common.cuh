// Shared declarations for the uml_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/uml_b200.h"

namespace uml {

// ---------------------------------------------------------------------------------------------------------------
// Tile geometry of the TMA fp32 scoring kernel (see DESIGN.md "linear_argmax_tma")
// ---------------------------------------------------------------------------------------------------------------
constexpr int kTileRows = 128;                            // rows per stage = TMA box height
constexpr int kChunkF = 32;                               // features per stage = TMA box width (128 B -> SWIZZLE_128B)
constexpr int kStageBytes = kTileRows * kChunkF * 4;      // 16 KiB
constexpr int kConsumerWarps = 8;                         // 2 per SM sub-partition
constexpr int kThreads = (kConsumerWarps + 1) * 32;       // + 1 TMA producer warp
constexpr int kRowsPerLane = kTileRows / 32;              // R = 4 rows per thread
constexpr int kMaxClassesTma = 16;                        // classes handled in registers by the TMA kernel
constexpr int kMaxSmemBytes = 227 * 1024;

struct LinearDeviceModel {
  // fp32 operands of the tile kernel: wt[f][cp] (feature-major, classes padded to cp = 4*ceil((C+1)/4), column C holds
  // wmax_f = max_c |w_cf| for the error bound), bias[cp] (column C = max_c |b_c|)
  const float* wt;
  const float* bias;
  // fp64 operands of the re-score / generic kernel: w64[F][w64_stride] (feature-major, classes contiguous and zero
  // padded; see linear_w64_stride), b64[C]
  const double* w64;
  const double* b64;
  int w64_stride;
  int n_classes;   // C after binary expansion (>= 2)
  int n_features;  // F
  int cp;          // padded class columns in wt
  int f_pad;       // rows of wt = 32 * ceil(F / 32), zero padded
};

// doubles per feature of the fp64 weight table: a lane reads the classes of ITS feature as 16-byte pairs, so the row
// length in 16-byte units must be odd for the eight lanes of a quarter-warp to land in eight different bank groups of
// shared memory (C = 10 -> 10 doubles = 80 bytes, C = 16 -> 18, C = 2 -> 2); rounds of 16 classes stay 16-byte aligned
__host__ __device__ inline int linear_w64_stride(int n_classes) {
  int pairs = (n_classes + 1) / 2;
  if (pairs % 2 == 0) pairs += 1;
  return 2 * pairs;
}

struct FlagList {
  int* count;        // number of flagged rows appended so far; the re-score kernel's last block resets it to 0
  int32_t* rows;     // flagged row indices
  int capacity;
  unsigned long long* counters;  // [0] = n_ambiguous, [1] = n_nonfinite, [2] = n_flagged, [3] = re-score blocks done
};

// The caller's own values for the rows of a launch: the raw source chunk as it was copied to the device (any dtype,
// either memory order).  The fp64 re-score reads the flagged rows from here, so labels follow the float64 (or int64)
// features the caller passed even when their fp32 copy is lossy (sklearn scores the float64 frame, _base.py:366-396).
struct SrcView {
  const void* base;      // nullptr: no view (re-score from x64 or from the fp32 rows)
  int dtype;             // uml_dtype of the elements
  long long row_stride;  // in elements
  long long col_stride;  // in elements
};

struct LinearLaunch {
  const float* x;       // device fp32 row-major
  const double* x64;    // optional fp64 copy of the same rows (lossy staging), else nullptr
  SrcView src;          // optional raw source view of the same rows (predict_host), wins over x64
  int64_t ld;           // floats per row
  int64_t ld64;
  int64_t n_rows;
  int32_t* labels;      // local label vector (device)
  // fused all-gather epilogue: labels are also stored to peers[i] + row_offset for i < n_peers
  void* peers[8];
  int n_peers;
  int wire_u8;  // 1: peer vectors are uint8 (one byte per label), 0: int32
  int64_t row_offset;
};

// launch `kern<<<grid, block, smem, stream>>>(p)` as a programmatic dependent of the previous kernel on the stream: its
// blocks may become resident while that kernel drains (the kernel itself waits with griddepcontrol.wait), which hides
// the launch latency between a scoring kernel and its fp64 re-score.  UML_B200_NO_PDL=1 falls back to a plain launch.
template <typename Params>
inline cudaError_t launch_dependent(void (*kern)(Params), int grid, int block, size_t smem, cudaStream_t stream, const Params& p) {
  static const bool no_pdl = getenv("UML_B200_NO_PDL") != nullptr;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(static_cast<unsigned>(block));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = no_pdl ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kern, p);
}

// scoring kernels (linear_kernels.cu)
// *rescore_kernel_needed: exact mode with the inline re-score switched off -> the caller launches launch_rescore_f64
cudaError_t launch_linear_tma(const CUtensorMap& xmap, const LinearDeviceModel& m, const LinearLaunch& l, bool exact,
                              const FlagList& flags, int sm_count, cudaStream_t stream, std::string* err,
                              bool* rescore_kernel_needed);
bool linear_tma_supported(const LinearDeviceModel& m, std::string* why);
cudaError_t launch_rescore_f64(const LinearDeviceModel& m, const LinearLaunch& l, const FlagList& flags, bool all_rows,
                               int sm_count, cudaStream_t stream);
// small-batch kernel of the online path (/predict, B <= 64): warp per row, fp64 straight from the raw source view
struct SmallResult {  // one per row, written by the kernel, copied back in one piece
  int32_t label;
  int32_t status;  // bit 0: NaN/Inf in the row, bit 1: fp64 margin inside the fp64 rounding bound (true tie)
};
cudaError_t launch_linear_small(const LinearDeviceModel& m, const SrcView& src, int n_rows, SmallResult* out,
                                cudaStream_t stream);
// class probabilities (LogisticRegression.predict_proba, sklearn/linear_model/_logistic.py): softmax of the scores
// (sigmoid for the binary layout), fp32 scores and exp; proba[n_rows][n_classes] row-major fp32
cudaError_t launch_linear_proba(const LinearDeviceModel& m, const float* x, int64_t ld, int64_t n_rows, float* proba,
                                int sm_count, cudaStream_t stream);

// 2-layer MLP (mlp_kernels.cu, mlp_tc_kernels.cu)
struct MlpHostModel {  // the caller's fp32 weights, torch nn.Linear layout
  std::vector<float> w1, b1, w2, b2;  // w1 [H][F], b1 [H], w2 [C][H], b2 [C]
};
struct MlpDeviceModel {
  const float* w1t;  // [f_pad][H + 4], column H = max_n |w1_nf|
  const float* b1;   // [H + 4], entry H = max_n |b1_n|
  const float* w2t;  // [H][cp], column C = max_c |w2_cn|
  const float* b2;   // [cp], entry C = max_c |b2_c|
  const double* rs_pack;  // fp64 operands of the re-score as one shared-memory image (mlp_rescore.cuh: mlp_rs_build_pack)
  int n_in, n_hidden, n_classes;
  int cp, f_pad;
  double w2_abs_row_sum_max;  // max_c sum_n |w2_cn|
  // tensor-core kernel: W1 split into tf32 hi | lo rows, pre-swizzled per 32-feature chunk (nullptr: not built)
  const float* w1_tiles;
  const MlpHostModel* host;
};
// where the labels of an MLP launch go (same contract as LinearLaunch's label fields)
struct MlpTcLaunch {
  int32_t* labels;  // local int32 vector or nullptr
  void* peers[8];
  int n_peers;
  int wire_u8;
  long long row_offset;
  long long n_rows;
  const float* x;  // the batch rows (the in-kernel fp64 re-score of the tensor-core kernel reads flagged rows again)
  long long ld;
};
bool mlp_tma_supported(const MlpDeviceModel& m, std::string* why);
// proba != nullptr: the softmax epilogue (n_rows x n_classes fp32 into proba, 16-byte aligned) instead of labels; rows
// with a non-finite A1 are appended to flags for launch_mlp_proba_f64
cudaError_t launch_mlp_tma(const CUtensorMap& xmap, const MlpDeviceModel& m, const float* x, int64_t n_rows,
                           int32_t* labels, bool exact, const FlagList& flags, int sm_count, cudaStream_t stream,
                           float* proba = nullptr);
cudaError_t launch_mlp_rescore_f64(const MlpDeviceModel& m, const float* x, int64_t ld, int64_t n_rows,
                                   const MlpTcLaunch& out, const FlagList& flags, bool all_rows, int sm_count,
                                   cudaStream_t stream);
bool mlp_tc_supported(const MlpDeviceModel& m, std::string* why);
std::vector<float> mlp_tc_build_w1_tiles(const float* w1, int H, int F, int f_pad);
cudaError_t launch_mlp_tc(const CUtensorMap& xmap, const MlpDeviceModel& m, const MlpTcLaunch& l, bool exact,
                          const FlagList& flags, int sm_count, cudaStream_t stream, bool* rescore_kernel_needed);
// class probabilities (uml_mlp_predict_proba): the tensor-core kernel with the softmax epilogue; rows whose features
// are not tf32 values or whose A1 is not finite are appended to flags.  launch_mlp_proba_f64 recomputes the flagged
// rows (all_rows = false) or every row (shapes neither tile kernel takes) in fp64 and rounds once to fp32.
cudaError_t launch_mlp_tc_proba(const CUtensorMap& xmap, const MlpDeviceModel& m, const MlpTcLaunch& l, float* proba,
                                const FlagList& flags, int sm_count, cudaStream_t stream);
cudaError_t launch_mlp_proba_f64(const MlpDeviceModel& m, const float* x, int64_t ld, int64_t n_rows, float* proba,
                                 const FlagList& flags, bool all_rows, int sm_count, cudaStream_t stream);
bool mlp_proba_staged_store();  // store scheme of the probability epilogues (mlp_proba.cuh: warp_store_proba)
// int32 labels (device) -> every target vector of a fused exchange (int32 or uint8 wire), for kernels without peer stores
cudaError_t launch_labels_scatter(const int32_t* labels, int64_t n, void* const* peers, int n_peers, int wire_u8,
                                  int64_t row_offset, int sm_count, cudaStream_t stream);

// staging kernels (stage_kernels.cu)
struct StageResult {  // device-side counters
  unsigned long long nonfinite;
  unsigned long long lossy;
  unsigned long long not_tf32;  // fp32 values with any of the low 13 mantissa bits set (tensor-core path needs none)
};
cudaError_t launch_stage_convert(const void* src, int src_dtype, bool feature_major, int64_t src_pitch_elems,
                                 int64_t rows, int n_features, float* dst, int64_t ld, double* dst64, int64_t ld64,
                                 StageResult* result, bool check_finite, cudaStream_t stream);

}  // namespace uml
