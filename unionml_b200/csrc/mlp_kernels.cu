// Scoring kernels for the 2-layer MLP predictor  argmax(softmax(W2 relu(W1 x + b1) + b2)) = argmax of the logits.
//
// Replaces PytorchModel.forward + .argmax(1) of the reference's torch quickstart
// (/root/reference/tests/integration/pytorch_app/quickstart.py:14-24, 68-70; hyperparameters 64 -> 32 -> 10 at :80).
//
//  * mlp_argmax_tma_kernel<H, C, EXACT>: the same persistent TMA + mbarrier ring (128-row x 32-feature boxes) as the
//    linear kernel; consumer warps work in pairs on a box (64 rows each, 2 rows x H hidden accumulators per lane).  Layer 1 runs per
//    landed box (W1^T rows are warp-uniform broadcast LDS.128 from shared memory), then ReLU, layer 2 and the argmax are
//    fused in registers.  EXACT mode carries two bound accumulators (A1 over layer 1, A2 over layer 2) and re-scores
//    rows whose logit margin is inside the propagated fp32 error bound in fp64.
//  * mlp_rescore_f64_kernel: warp per row, lane per hidden unit, fp64; flagged rows of EXACT mode, or every row for
//    shapes the tile kernel is not instantiated for.
//  * PROBA (uml_mlp_predict_proba): the tile kernel's epilogue stores the fp32 softmax of the logits (mlp_proba.cuh)
//    and flags rows with a non-finite A1; mlp_proba_f64_kernel recomputes those rows, or every row for other shapes,
//    in fp64.
//
// This is CUDA-core fp32 (FFMA): 4 736 flop/row puts the HBM roofline (25 G rows/s) above the FFMA peak, so this kernel
// is FMA-pipe bound (~0.66 ms per 10M rows at 1.9 GHz).  It serves batches whose features are NOT tf32 values (general
// floats); tf32-representable batches (integer / pixel domains) take the tensor-core kernel in mlp_tc_kernels.cu.
#include <algorithm>
#include <cstdlib>

#include "uml_common.cuh"
#include "tma_ring.cuh"
#include "mlp_rescore.cuh"
#include "mlp_proba.cuh"

#ifndef UML_MLP_UNROLL_Q
#define UML_MLP_UNROLL_Q 8  // feature-quad unroll of the layer-1 loop (same-box A/B, EXACT: 1 -> 1.120, 2 -> 1.056, 4 -> 1.023, 8 -> 1.015 ms)
#endif
#define UML_PRAGMA_(x) _Pragma(#x)
#define UML_UNROLL(n) UML_PRAGMA_(unroll n)

namespace uml {

// 8 consumer warps work as 4 PAIRS: a pair shares one 128-row x 32-feature box, warp 2p takes rows 0..63 and warp 2p+1
// rows 64..127 (2 rows per lane x 32 hidden accumulators = 64 registers, inside the 168-register cap of a 9-warp CTA)
// and two warps per SM sub-partition hide each other's LDS / barrier latency.  A stage is released by both warps.
constexpr int kMlpPairs = 4;
constexpr int kMlpConsumerWarps = 2 * kMlpPairs;
constexpr int kMlpThreads = (kMlpConsumerWarps + 1) * 32;
constexpr int kMlpTileRows = kTileRows;                      // 128 rows x 32 features, same boxes as the linear kernel
constexpr int kMlpStageBytes = kStageBytes;                  // 16 KiB
constexpr int kMlpRowsPerLane = 2;                           // rows per lane within a warp's 64-row half

struct MlpKernelParams {
  const float* w1t;  // [f_pad][H + 4]   column H = max_n |w1_nf|
  const float* b1;   // [H + 4]          entry  H = max_n |b1_n|
  const float* w2t;  // [H][CP]          column C = max_c |w2_cn|
  const float* b2;   // [CP]             entry  C = max_c |b2_c|
  int32_t* labels;
  long long n_rows;
  long long num_tiles;
  int f_pad;
  int kc;
  int num_stages;
  float e1_scale;  // (F+4) 2^-24 (1+slack) * max_c sum_n |w2_cn|   -> layer-1 error as it reaches a logit
  float e2_scale;  // (H+4) 2^-24 (1+slack)                          -> layer-2 accumulation error
  int* flag_count;
  int32_t* flag_rows;
  int flag_cap;
  float* proba;  // PROBA kernels: n_rows x C fp32, 16-byte aligned
};

template <int H, int C, bool EXACT, bool PROBA = false, bool STAGED = false>
__global__ void __launch_bounds__(kMlpThreads, 1)
mlp_argmax_tma_kernel(const __grid_constant__ CUtensorMap xmap, const MlpKernelParams p) {
  constexpr int HP = H + 4;
  constexpr int CP = (C + 1 + 3) / 4 * 4;
  constexpr int NC2 = C + (EXACT ? 1 : 0);
  constexpr int NW2 = (NC2 + 3) / 4;
  constexpr int R = kMlpRowsPerLane;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int S = p.num_stages;
  float* w1_s = reinterpret_cast<float*>(smem + static_cast<size_t>(S) * kMlpStageBytes);
  float* b1_s = w1_s + p.f_pad * HP;
  float* w2_s = b1_s + HP;
  float* b2_s = w2_s + H * CP;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(b2_s + CP);
  uint64_t* empty_bar = full_bar + S;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  {
    const float4* src = reinterpret_cast<const float4*>(p.w1t);
    float4* dst = reinterpret_cast<float4*>(w1_s);
    for (int i = threadIdx.x; i < p.f_pad * HP / 4; i += kMlpThreads) dst[i] = __ldg(src + i);
    for (int i = threadIdx.x; i < H * CP; i += kMlpThreads) w2_s[i] = __ldg(p.w2t + i);
    if (threadIdx.x < HP) b1_s[threadIdx.x] = __ldg(p.b1 + threadIdx.x);
    if (threadIdx.x < CP) b2_s[threadIdx.x] = __ldg(p.b2 + threadIdx.x);
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);  // both warps of the pair that read the stage
    }
    fence_barrier_init();
  }
  __syncthreads();

  pdl_launch_dependents();  // see linear_kernels.cu: the re-score kernel may be scheduled while this grid drains
  const long long G = gridDim.x;
  const long long num_tiles = p.num_tiles;
  const int KC = p.kc;

  if (warp == kMlpConsumerWarps) {
    if (elect_one_sync()) {
      tma_prefetch_desc(&xmap);
      const uint64_t policy = make_evict_first_policy();
      int stage = 0;
      uint32_t phase = 0;
      for (long long first = blockIdx.x; first < num_tiles; first += G * kMlpPairs) {
        const int nv = static_cast<int>(min(static_cast<long long>(kMlpPairs), (num_tiles - first + G - 1) / G));
        for (int k = 0; k < KC; ++k) {
          for (int w = 0; w < nv; ++w) {
            mbar_wait(&empty_bar[stage], phase ^ 1u);
            mbar_arrive_expect_tx(&full_bar[stage], kMlpStageBytes);
            tma_load_2d(smem + static_cast<size_t>(stage) * kMlpStageBytes, &xmap, &full_bar[stage], k * kChunkF,
                        static_cast<int>((first + w * G) * kMlpTileRows), policy);
            if (++stage == S) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else {
    const int pair = warp >> 1;
    const int half = warp & 1;
    const uint32_t lanebase = static_cast<uint32_t>(half * 64 + lane) * 128u + static_cast<uint32_t>(lane & 7) * 16u;
    uint32_t seq_base = 0;
    for (long long first = blockIdx.x; first < num_tiles; first += G * kMlpPairs) {
      const int nv = static_cast<int>(min(static_cast<long long>(kMlpPairs), (num_tiles - first + G - 1) / G));
      if (pair < nv) {
        const long long tile = first + pair * G;
        uint64_t h2[R][H / 2];  // hidden accumulators as fp32x2 pairs (units 2i, 2i+1)
        float a1[R];
#pragma unroll
        for (int j = 0; j < R; ++j) {
#pragma unroll
          for (int n = 0; n < H / 2; ++n) h2[j][n] = pack2(b1_s[2 * n], b1_s[2 * n + 1]);
          a1[j] = b1_s[H];
        }
        for (int k = 0; k < KC; ++k) {
          const uint32_t seq = seq_base + static_cast<uint32_t>(k * nv + pair);
          const uint32_t stage = seq % static_cast<uint32_t>(S);
          const uint32_t phase = (seq / static_cast<uint32_t>(S)) & 1u;
          mbar_wait(&empty_bar[stage], phase ^ 1u);  // previous occupant released (see linear_kernels.cu)
          mbar_wait(&full_bar[stage], phase);
          const uint8_t* xs = smem + static_cast<size_t>(stage) * kMlpStageBytes;
          const float* wk = w1_s + k * kChunkF * HP;
          UML_UNROLL(UML_MLP_UNROLL_Q)
          for (int q = 0; q < kChunkF / 4; ++q) {
            float4 xv[R];
            const uint32_t off = lanebase ^ static_cast<uint32_t>(q * 16);
#pragma unroll
            for (int j = 0; j < R; ++j) xv[j] = *reinterpret_cast<const float4*>(xs + off + j * 32 * 128);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float* wrow = wk + (q * 4 + e) * HP;
              float x[R];
#pragma unroll
              for (int j = 0; j < R; ++j) x[j] = e == 0 ? xv[j].x : e == 1 ? xv[j].y : e == 2 ? xv[j].z : xv[j].w;
#pragma unroll
              for (int m = 0; m < H / 4; ++m) {
                const float4 t = *reinterpret_cast<const float4*>(wrow + m * 4);
                const uint64_t w01 = pack2(t.x, t.y), w23 = pack2(t.z, t.w);
#pragma unroll
                for (int j = 0; j < R; ++j) {
                  const uint64_t xx = pack2(x[j], x[j]);
                  h2[j][m * 2 + 0] = fma2(xx, w01, h2[j][m * 2 + 0]);
                  h2[j][m * 2 + 1] = fma2(xx, w23, h2[j][m * 2 + 1]);
                }
              }
              if (EXACT || PROBA) {
                const float wmax = wrow[H];
#pragma unroll
                for (int j = 0; j < R; ++j) a1[j] = fmaf(fabsf(x[j]), wmax, a1[j]);
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty_bar[stage]);
        }

        // ---- ReLU, layer 2 (hidden unit outermost: each W2^T row is loaded once for the lane's 4 rows) ----
        constexpr int NZ2 = (NC2 + 1) / 2;  // logit accumulators as pairs (a padding lane multiplies a zero weight)
        uint64_t z2[R][NZ2];
#pragma unroll
        for (int j = 0; j < R; ++j)
#pragma unroll
          for (int c = 0; c < NZ2; ++c) z2[j][c] = pack2(b2_s[2 * c], 2 * c + 1 < CP ? b2_s[2 * c + 1] : 0.f);
#pragma unroll
        for (int n2 = 0; n2 < H / 2; ++n2) {
          float hv[R][2];
#pragma unroll
          for (int j = 0; j < R; ++j) {
            unpack2(h2[j][n2], hv[j][0], hv[j][1]);
            hv[j][0] = fmaxf(hv[j][0], 0.f);
            hv[j][1] = fmaxf(hv[j][1], 0.f);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int n = 2 * n2 + u;
            uint64_t w2p[NW2 * 2];
#pragma unroll
            for (int m = 0; m < NW2; ++m) {
              const float4 t = *reinterpret_cast<const float4*>(w2_s + n * CP + m * 4);
              w2p[m * 2 + 0] = pack2(t.x, t.y);
              w2p[m * 2 + 1] = pack2(t.z, t.w);
            }
#pragma unroll
            for (int j = 0; j < R; ++j) {
              const uint64_t hh = pack2(hv[j][u], hv[j][u]);
#pragma unroll
              for (int c = 0; c < NZ2; ++c) z2[j][c] = fma2(hh, w2p[c], z2[j][c]);
            }
          }
        }
        float z[R][2 * NZ2];
#pragma unroll
        for (int j = 0; j < R; ++j)
#pragma unroll
          for (int c = 0; c < NZ2; ++c) unpack2(z2[j][c], z[j][2 * c], z[j][2 * c + 1]);
        if constexpr (PROBA) {
          // ---- softmax, the warp's 32 rows out per j; a non-finite A1 (NaN/Inf feature) goes to the fp64 kernel ----
          float* strip = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(empty_bar + S) + 15u) & ~static_cast<uintptr_t>(15)) +
                         warp * 32 * C;
#pragma unroll
          for (int j = 0; j < R; ++j) {
            const long long row0 = tile * kMlpTileRows + half * 64 + 32 * j;
            float pr[C];
#pragma unroll
            for (int c = 0; c < C; ++c) pr[c] = z[j][c];
            softmax_f32<C>(pr);
            warp_store_proba<C, STAGED>(pr, p.proba, row0, p.n_rows, lane, strip);
            flag_list_append(row0 + lane < p.n_rows && !(a1[j] < INFINITY), row0 + lane, p.flag_count, p.flag_rows,
                             p.flag_cap, lane);
          }
        }
        // ---- argmax (first maximum wins), margin guard, label store ----
#pragma unroll
        for (int j = 0; j < R && !PROBA; ++j) {
          const long long row = tile * kMlpTileRows + half * 64 + lane + 32 * j;
          float best = z[j][0];
          float second = -INFINITY;
          int idx = 0;
#pragma unroll
          for (int c = 1; c < C; ++c) {
            if (z[j][c] > best) {
              second = best;
              best = z[j][c];
              idx = c;
            } else {
              second = fmaxf(second, z[j][c]);
            }
          }
          const bool in_range = row < p.n_rows;
          if (in_range) p.labels[row] = idx;
          if (EXACT) {
            // |z_c - true| <= E1 * sum_n |w2_cn| + (H+4) u A2, E1 = (F+4) u A1 (ReLU is 1-Lipschitz)
            const float err = p.e1_scale * a1[j] + p.e2_scale * z[j][C];
            const bool certain = (best - second) > 2.0f * err;
            const bool flagged = in_range && !certain;
            const unsigned mask = __ballot_sync(0xffffffffu, flagged);
            if (mask != 0u) {
              int base = 0;
              if (lane == 0) base = atomicAdd(p.flag_count, __popc(mask));
              base = __shfl_sync(0xffffffffu, base, 0);
              if (flagged) {
                const int pos = base + __popc(mask & ((1u << lane) - 1u));
                if (pos < p.flag_cap) p.flag_rows[pos] = static_cast<int32_t>(row);
              }
            }
          }
        }
      }
      seq_base += static_cast<uint32_t>(KC * nv);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// fp64 re-score / generic kernel: warp per row, lane per hidden unit
// ---------------------------------------------------------------------------------------------------------------
struct MlpRescoreParams {
  const float* x;
  long long ld;
  long long n_rows;
  const double* pack;  // the shared-memory image of the fp64 operands (mlp_rs_build_pack)
  int F, H, C;
  const int* flag_count;
  const int32_t* flag_rows;
  int flag_cap;
  int all_rows;
  int32_t* labels;
  void* peers[8];
  int n_peers;
  int wire_u8;
  long long row_offset;
  unsigned long long* counters;
};

constexpr int kMlpRsRows = 4;  // rows per warp pass (mlp_rescore.cuh: shared-memory wavefronts per row fall 3 -> 1)

// Shared-memory version (mlp_rescore.cuh): the fp64 image of the model (W1 [F][H], W2 [C][H+1], biases, bound vectors;
// built on the host at load) is copied once per block; a warp scores four rows per pass - their features and hidden
// activations interleaved in the warp's own strip, so every W element it reads from shared memory is used four times.
// Layer 1: lane per hidden unit.  Layer 2: lane per class (no warp reductions), then one butterfly per row for arg-max
// and runner-up.
__global__ void __launch_bounds__(256) mlp_rescore_f64_kernel(const MlpRescoreParams p) {
  extern __shared__ __align__(16) double rs_smem[];
  constexpr int R = kMlpRsRows;
  // (weights are staged first: they do not depend on the scoring kernel; the flag list does - see the wait below)
  MlpRsView view = mlp_rs_stage(rs_smem, p.pack, p.F, p.H, p.C);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* xs = rs_smem + mlp_rs_weight_doubles(p.F, p.H, p.C) + warp * mlp_rs_strip_doubles(p.F, p.H, R);
  double* hv = xs + p.F * R;
  __syncthreads();
  mlp_rs_finish_stage(view);

  pdl_wait_for_predecessor();  // from here on: the flag list and labels of the scoring kernel this launch depends on
  const long long warp_global = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long warps_total = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const long long n = p.all_rows ? p.n_rows : static_cast<long long>(min(*p.flag_count, p.flag_cap));
  if (!p.all_rows && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&p.counters[2], static_cast<unsigned long long>(n));
  // warp w takes entries [w*R, w*R + R) of the list, then strides by all warps: a short list spreads over many warps
  for (long long i = warp_global * R; i < n; i += warps_total * R) {
    long long row[R];
    const float* xr[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long long j = i + r < n ? i + r : i;  // unused slots repeat the first row (result ignored)
      row[r] = p.all_rows ? j : static_cast<long long>(p.flag_rows[j]);
      xr[r] = p.x + row[r] * p.ld;
    }
    MlpRowResult res[R];
    mlp_rs_rows<R>(view, xr, xs, hv, lane, res);
    if (lane < R && i + lane < n) {
      // lane r publishes row r (R <= 4 lanes, one per row)
      long long my_row = row[0];
      MlpRowResult mine = res[0];
#pragma unroll
      for (int r = 1; r < R; ++r) {
        if (lane == r) {
          my_row = row[r];
          mine = res[r];
        }
      }
      if (p.labels) p.labels[my_row] = mine.idx;
      for (int q = 0; q < p.n_peers; ++q) {
        if (p.wire_u8) static_cast<uint8_t*>(p.peers[q])[p.row_offset + my_row] = static_cast<uint8_t>(mine.idx);
        else static_cast<int32_t*>(p.peers[q])[p.row_offset + my_row] = mine.idx;
      }
      if (mine.bad) atomicAdd(&p.counters[1], 1ull);
      if (mine.ambiguous) atomicAdd(&p.counters[0], 1ull);
    }
  }
  // hand the flag list back empty (see rescore_f64_kernel in linear_kernels.cu)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long ticket = atomicAdd(&p.counters[3], 1ull);
    if (ticket == static_cast<unsigned long long>(gridDim.x) - 1ull) {
      *const_cast<int*>(p.flag_count) = 0;
      p.counters[3] = 0ull;
      __threadfence();
    }
  }
}

// fp64 softmax of flagged rows (all_rows = 0) or of every row: the re-score kernel's block layout and shared-memory
// image, mlp_rs_proba_rows instead of the arg-max
struct MlpProbaF64Params {
  const float* x;
  long long ld;
  long long n_rows;
  const double* pack;
  int F, H, C;
  const int* flag_count;
  const int32_t* flag_rows;
  int flag_cap;
  int all_rows;
  float* proba;
  unsigned long long* counters;
};

__global__ void __launch_bounds__(256) mlp_proba_f64_kernel(const MlpProbaF64Params p) {
  extern __shared__ __align__(16) double rs_smem[];
  constexpr int R = kMlpRsRows;
  MlpRsView view = mlp_rs_stage(rs_smem, p.pack, p.F, p.H, p.C);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* xs = rs_smem + mlp_rs_weight_doubles(p.F, p.H, p.C) + warp * mlp_rs_proba_strip_doubles(p.F, p.H, p.C, R);
  double* hv = xs + (p.F > p.C ? p.F : p.C) * R;
  __syncthreads();
  mlp_rs_finish_stage(view);

  pdl_wait_for_predecessor();  // the flag list and the probabilities of the scoring kernel this launch depends on
  const long long warp_global = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long warps_total = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const long long n = p.all_rows ? p.n_rows : static_cast<long long>(min(*p.flag_count, p.flag_cap));
  if (!p.all_rows && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&p.counters[2], static_cast<unsigned long long>(n));
  for (long long i = warp_global * R; i < n; i += warps_total * R) {
    const float* xr[R];
    float* out[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long long j = i + r < n ? i + r : i;  // unused slots repeat the first row and store nothing
      const long long row = p.all_rows ? j : static_cast<long long>(p.flag_rows[j]);
      xr[r] = p.x + row * p.ld;
      out[r] = i + r < n ? p.proba + row * p.C : nullptr;
    }
    bool bad[R];
    mlp_rs_proba_rows<R>(view, xr, xs, hv, lane, out, bad);
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (lane == 0 && bad[r] && i + r < n) atomicAdd(&p.counters[1], 1ull);
  }
  // hand the flag list back empty (see rescore_f64_kernel in linear_kernels.cu)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned long long ticket = atomicAdd(&p.counters[3], 1ull);
    if (ticket == static_cast<unsigned long long>(gridDim.x) - 1ull) {
      *const_cast<int*>(p.flag_count) = 0;
      p.counters[3] = 0ull;
      __threadfence();
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static size_t mlp_fixed_smem(const MlpDeviceModel& m, bool proba = false) {
  return 1024 + (static_cast<size_t>(m.f_pad) * (m.n_hidden + 4) + (m.n_hidden + 4) + static_cast<size_t>(m.n_hidden) * m.cp + m.cp) * 4 +
         2 * 64 * 8 + (proba ? 16 + static_cast<size_t>(kMlpConsumerWarps) * 32 * m.n_classes * 4 : 0);  // + output strips
}

bool mlp_tma_supported(const MlpDeviceModel& m, std::string* why) {
  const bool shape_ok = (m.n_hidden == 32 || m.n_hidden == 16) && (m.n_classes == 10 || m.n_classes == 2 || m.n_classes == 3);
  if (!shape_ok) {
    if (why) *why = "tile kernel instantiated for hidden in {16, 32} and classes in {2, 3, 10}";
    return false;
  }
  if (mlp_fixed_smem(m) + kMlpPairs * static_cast<size_t>(kMlpStageBytes) > static_cast<size_t>(kMaxSmemBytes)) {
    if (why) *why = "W1^T does not fit in shared memory next to a 4-stage ring";
    return false;
  }
  return true;
}

template <int H, int C, bool EXACT, bool PROBA = false, bool STAGED = false>
static cudaError_t mlp_launch_one(const CUtensorMap& xmap, const MlpKernelParams& p, int grid, size_t smem,
                                  cudaStream_t stream) {
  auto kern = mlp_argmax_tma_kernel<H, C, EXACT, PROBA, STAGED>;
  static size_t configured = 0;
  if (smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  kern<<<grid, kMlpThreads, smem, stream>>>(xmap, p);
  return cudaGetLastError();
}

template <bool EXACT>
static cudaError_t mlp_dispatch(int H, int C, const CUtensorMap& xmap, const MlpKernelParams& p, int grid, size_t smem,
                                cudaStream_t stream) {
#define UML_MLP_CASE(HH, CC) \
  if (H == HH && C == CC) return mlp_launch_one<HH, CC, EXACT>(xmap, p, grid, smem, stream);
  UML_MLP_CASE(32, 10) UML_MLP_CASE(32, 2) UML_MLP_CASE(32, 3) UML_MLP_CASE(16, 10) UML_MLP_CASE(16, 2) UML_MLP_CASE(16, 3)
#undef UML_MLP_CASE
  return cudaErrorInvalidValue;
}

template <bool STAGED>
static cudaError_t mlp_dispatch_proba(int H, int C, const CUtensorMap& xmap, const MlpKernelParams& p, int grid,
                                      size_t smem, cudaStream_t stream) {
#define UML_MLP_CASE(HH, CC) \
  if (H == HH && C == CC) return mlp_launch_one<HH, CC, false, true, STAGED>(xmap, p, grid, smem, stream);
  UML_MLP_CASE(32, 10) UML_MLP_CASE(32, 2) UML_MLP_CASE(32, 3) UML_MLP_CASE(16, 10) UML_MLP_CASE(16, 2) UML_MLP_CASE(16, 3)
#undef UML_MLP_CASE
  return cudaErrorInvalidValue;
}

// proba != nullptr: the PROBA kernel (softmax epilogue into proba, non-finite rows to the flag list); labels unused
cudaError_t launch_mlp_tma(const CUtensorMap& xmap, const MlpDeviceModel& m, const float* x, int64_t n_rows,
                           int32_t* labels, bool exact, const FlagList& flags, int sm_count, cudaStream_t stream,
                           float* proba) {
  (void)x;
  if (n_rows <= 0) return cudaSuccess;
  MlpKernelParams p{};
  p.w1t = m.w1t;
  p.b1 = m.b1;
  p.w2t = m.w2t;
  p.b2 = m.b2;
  p.labels = labels;
  p.n_rows = n_rows;
  p.num_tiles = (n_rows + kMlpTileRows - 1) / kMlpTileRows;
  p.f_pad = m.f_pad;
  p.kc = m.f_pad / kChunkF;
  const size_t fixed = mlp_fixed_smem(m, proba != nullptr);
  int stages = static_cast<int>((static_cast<size_t>(kMaxSmemBytes) - fixed) / kMlpStageBytes);
  stages = std::min(stages, 64);
  if (const char* env = getenv("UML_B200_STAGES")) stages = std::max(kMlpPairs, std::min(stages, atoi(env)));
  p.num_stages = stages;
  const double u = 5.9604644775390625e-08;
  const double F = m.n_in, H = m.n_hidden;
  p.e1_scale = static_cast<float>((F + 4.0) * u * (1.0 + F * 4.76837158203125e-07) * 1.0001 * m.w2_abs_row_sum_max);
  p.e2_scale = static_cast<float>((H + 4.0) * u * 1.0001);
  p.flag_count = flags.count;
  p.flag_rows = flags.rows;
  p.flag_cap = flags.capacity;
  p.proba = proba;
  const size_t smem = fixed + static_cast<size_t>(stages) * kMlpStageBytes;
  const long long slots = (p.num_tiles + kMlpPairs - 1) / kMlpPairs;
  const int grid = static_cast<int>(std::min<long long>(sm_count, std::max<long long>(1, slots)));
  if (proba)
    return mlp_proba_staged_store() ? mlp_dispatch_proba<true>(m.n_hidden, m.n_classes, xmap, p, grid, smem, stream)
                                    : mlp_dispatch_proba<false>(m.n_hidden, m.n_classes, xmap, p, grid, smem, stream);
  return exact ? mlp_dispatch<true>(m.n_hidden, m.n_classes, xmap, p, grid, smem, stream)
               : mlp_dispatch<false>(m.n_hidden, m.n_classes, xmap, p, grid, smem, stream);
}

cudaError_t launch_mlp_rescore_f64(const MlpDeviceModel& m, const float* x, int64_t ld, int64_t n_rows,
                                   const MlpTcLaunch& out, const FlagList& flags, bool all_rows, int sm_count,
                                   cudaStream_t stream) {
  if (n_rows <= 0) return cudaSuccess;
  MlpRescoreParams p{};
  p.x = x;
  p.ld = ld;
  p.n_rows = n_rows;
  p.pack = m.rs_pack;
  p.F = m.n_in;
  p.H = m.n_hidden;
  p.C = m.n_classes;
  p.flag_count = flags.count;
  p.flag_rows = flags.rows;
  p.flag_cap = flags.capacity;
  p.all_rows = all_rows ? 1 : 0;
  p.labels = out.labels;
  p.n_peers = out.n_peers;
  p.wire_u8 = out.wire_u8;
  for (int i = 0; i < 8; ++i) p.peers[i] = i < out.n_peers ? out.peers[i] : nullptr;
  p.row_offset = out.row_offset;
  p.counters = flags.counters;
  // shared memory: W1 + padded W2 + biases + the two bound vectors + one strip (x, hidden values) per warp
  const size_t smem = (mlp_rs_weight_doubles(m.n_in, m.n_hidden, m.n_classes) + 8 * mlp_rs_strip_doubles(m.n_in, m.n_hidden, kMlpRsRows)) * sizeof(double);
  if (smem > static_cast<size_t>(kMaxSmemBytes)) return cudaErrorInvalidValue;  // uml_mlp_load bounds F * H
  static size_t configured = 0;
  if (smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(mlp_rescore_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mlp_rescore_f64_kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  long long blocks = static_cast<long long>(sm_count) * per_sm;  // persistent: every resident warp loops over rows
  if (all_rows) blocks = std::min<long long>(blocks, (n_rows + 8 * kMlpRsRows - 1) / (8 * kMlpRsRows));
  cudaError_t lerr = launch_dependent(mlp_rescore_f64_kernel, static_cast<int>(std::max<long long>(1, blocks)), 256, smem, stream, p);
  if (lerr != cudaSuccess) return lerr;
  return cudaGetLastError();
}

cudaError_t launch_mlp_proba_f64(const MlpDeviceModel& m, const float* x, int64_t ld, int64_t n_rows, float* proba,
                                 const FlagList& flags, bool all_rows, int sm_count, cudaStream_t stream) {
  if (n_rows <= 0) return cudaSuccess;
  MlpProbaF64Params p{};
  p.x = x;
  p.ld = ld;
  p.n_rows = n_rows;
  p.pack = m.rs_pack;
  p.F = m.n_in;
  p.H = m.n_hidden;
  p.C = m.n_classes;
  p.flag_count = flags.count;
  p.flag_rows = flags.rows;
  p.flag_cap = flags.capacity;
  p.all_rows = all_rows ? 1 : 0;
  p.proba = proba;
  p.counters = flags.counters;
  const size_t smem = (mlp_rs_weight_doubles(m.n_in, m.n_hidden, m.n_classes) +
                       8 * mlp_rs_proba_strip_doubles(m.n_in, m.n_hidden, m.n_classes, kMlpRsRows)) * sizeof(double);
  if (smem > static_cast<size_t>(kMaxSmemBytes)) return cudaErrorInvalidValue;
  static size_t configured = 0;
  if (smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(mlp_proba_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mlp_proba_f64_kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  long long blocks = static_cast<long long>(sm_count) * per_sm;
  if (all_rows) blocks = std::min<long long>(blocks, (n_rows + 8 * kMlpRsRows - 1) / (8 * kMlpRsRows));
  cudaError_t lerr = launch_dependent(mlp_proba_f64_kernel, static_cast<int>(std::max<long long>(1, blocks)), 256, smem, stream, p);
  if (lerr != cudaSuccess) return lerr;
  return cudaGetLastError();
}

}  // namespace uml
