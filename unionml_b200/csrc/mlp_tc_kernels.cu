// Tensor-core scoring kernel for the 2-layer MLP predictor (cfg 5): layer 1 on tcgen05 (kind::tf32), accumulators in TMEM.
//
// Replaces PytorchModel.forward + .argmax(1) of the reference's torch quickstart
// (/root/reference/tests/integration/pytorch_app/quickstart.py:14-24, 68-70; hyperparameters 64 -> 32 -> 10 at :80).
//
// Why tensor cores here and not in the linear kernel: layer 1 is a real [rows x F] . [F x H] contraction (4 096 of the
// 4 736 flop per row); on CUDA cores it needs 1 408 FFMA2 per row and caps the kernel at 0.37 of the HBM roofline.
//
// Exactness with 10-bit tf32 mantissas.  The MMA multiplies tf32 x tf32 exactly and accumulates in fp32, so the only
// approximation is what the operands lose when they become tf32:
//   * X: this kernel is dispatched for batches whose features ARE tf32 values (low 13 mantissa bits zero - integer /
//     pixel domains such as the reference's digits and MNIST frames; the staging pass records it).  Every row is
//     re-checked here (scan warps OR the low bits): a row that is not tf32-exact gets A1 = +inf and is therefore
//     flagged for the fp64 re-score, so the answer is right for any input - only slower.
//   * W1: split on the host as w = hi + lo + r with hi, lo tf32 (round to nearest) and |r| <= 2^-22 |w|; B holds
//     [hi | lo] as 2H columns, so ONE MMA per K step yields main = x.hi and small = x.lo in separate TMEM columns
//     (the small terms never lose bits against the large accumulator), summed in fp32 in the epilogue.
// EXACT mode bounds the error per row, |h_n - h_n_true| <= E1 = (32 n_mma + 12) 2^-24 A1 with
// A1 = max|b1| + sum_f |x_f| max_n |w1_nf| (n_mma = F_pad / 8 accumulating MMA steps; the per-step term covers a
// truncating 9-addend aligner with no guard bits, DESIGN.md 3.3), propagates it through layer 2 exactly like the
// CUDA-core kernel, and re-scores rows whose logit margin is inside the bound in fp64 (mlp_rescore_f64_kernel).
//
// Roles (14 warps, one CTA per SM, persistent over 128-row tiles):
//   warp 12 : TMA producer - 128 x 32 fp32 boxes of X (16 KiB, SWIZZLE_128B) into an S-stage ring
//   warp 13 : MMA issuer   - one lane; per box 4 x tcgen05.mma (M128, N=2H, K8) from the box (A, K-major SW128) and
//             the resident W1 tile (B); tcgen05.commit frees the ring stage / publishes the accumulator
//   warps 0-3 : scan        - thread per row: A1 bound + tf32-exactness of the row from the same box (LDS.128)
//   warps 4-11: epilogue    - two sets of four warps taking alternate tiles (the first ncu capture showed one set
//             80 % busy and everything else waiting on it): tcgen05.ld the row's 2H accumulators, + b1, ReLU, layer 2
//             from constant-bank operands, argmax (first maximum wins), margin guard, label store (+ peer stores)
//
// PROBA kernels (uml_mlp_predict_proba) share the producer, MMA and scan roles; their epilogue turns the same C logits
// into an fp32 softmax and stores C floats per row (mlp_proba.cuh).  There is no margin guard; rows the MMA cannot
// score (features that are not tf32 values, or a non-finite A1) go to the flag list and mlp_proba_f64_kernel
// recomputes them.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "uml_common.cuh"
#include "tcgen05.cuh"
#include "mlp_rescore.cuh"
#include "mlp_proba.cuh"

#ifndef UML_MLP_QUEUE_DEFAULT
// 0: the queue variant lost the same-box A/B (profiles/r02_ab.json: 10M rows 0.640 vs 0.577 ms per step) - the scoring
// kernel is issue-bound (68 % issue slots), so the 58 000 fp64 rows it takes in slow the pipeline by more than the
// separate re-score kernel costs.  (The linear tile kernel, with 0.02 % flagged rows, wins with its queue.)
#define UML_MLP_QUEUE_DEFAULT 0
#endif

#ifndef UML_MLP_PROBA_STAGED_DEFAULT
#define UML_MLP_PROBA_STAGED_DEFAULT 0
#endif

namespace uml {

constexpr int kTcThreads = 448;
constexpr int kTcProducerWarp = 12;
constexpr int kTcMmaWarp = 13;
// QUEUE kernels: rows flagged by the epilogue warps are re-scored in fp64 by four more warps of the same launch while
// the tensor-core pipeline keeps streaming (fp64 units and these issue slots are otherwise idle)
constexpr int kTcRescoreWarps = 4;
constexpr int kTcFirstRescoreWarp = 14;
constexpr int kTcThreadsQueue = kTcThreads + 32 * kTcRescoreWarps;
constexpr int kTcEpilogueWarps = 8;
constexpr int kTcQueueCap = 1024;       // power of two
constexpr int kTcQueueHeadroom = 512;   // a warp publishes only while this many slots are free (8 warps x 32 rows at once)
constexpr int kTcAccStages = 4;    // TMEM accumulator stages (tiles in flight between MMA and epilogue)
constexpr int kTcSlots = 24;       // A1 hand-off slots (scan -> epilogue); > the scan warps' maximum lead over the epilogue
constexpr int kTcMaxFpad = 128;    // features (padded to 32) the resident W1 tile is sized for

template <int H, int C>
struct MlpTcParams {
  static constexpr int CP = (C + 1 + 3) / 4 * 4;
  float w2[H][CP];          // [n][c], column C = max_c |w2_cn| (EXACT bound), rest zero
  float b1[H];
  float b2[CP];             // entry C = max_c |b2_c|
  float w1max[kTcMaxFpad];  // max_n |w1_nf| per feature (zero padded)
  float b1max;
  float e1_scale, e2_scale;
  const float* w1_tiles;    // [KC][2H rows][32 floats], rows 128-byte swizzled exactly as the UMMA descriptor reads them
  int32_t* labels;
  void* peers[8];
  int n_peers;
  int wire_u8;
  long long row_offset;
  long long n_rows;
  long long num_tiles;
  int kc;
  int num_stages;
  int* flag_count;
  int32_t* flag_rows;
  int flag_cap;
  // QUEUE kernels: what the in-kernel fp64 re-score needs
  const float* x;
  long long ld;
  int n_in;
  const double* rs_pack;  // shared-memory image of the fp64 operands (mlp_rs_build_pack)
  unsigned long long* counters;  // [0] ambiguous, [1] nonfinite, [2] re-scored rows
  float* proba;  // PROBA kernels: n_rows x C fp32, 16-byte aligned
};

template <int H, int C>
__device__ __forceinline__ void tc_store_final_label(const MlpTcParams<H, C>& p, long long row, int idx) {
  if (p.labels) p.labels[row] = idx;
  for (int i = 0; i < p.n_peers; ++i) {
    if (p.wire_u8) static_cast<uint8_t*>(p.peers[i])[p.row_offset + row] = static_cast<uint8_t>(idx);
    else static_cast<int32_t*>(p.peers[i])[p.row_offset + row] = idx;
  }
}

template <int H, int C, bool EXACT, bool QUEUE, bool PROBA = false, bool STAGED = false>
__global__ void __launch_bounds__(kTcThreadsQueue, 1)
mlp_argmax_tc_kernel(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ MlpTcParams<H, C> p) {
  constexpr int N = 2 * H;  // accumulator columns per tile: [main | small]
  constexpr int TMEM_COLS = kTcAccStages * N;
  static_assert(TMEM_COLS == 128 || TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM columns must be a power of two");
  static_assert(N % 16 == 0 && N <= 256, "UMMA M=128 needs N % 16 == 0");
  constexpr int CP = MlpTcParams<H, C>::CP;
  constexpr uint32_t IDESC = umma_idesc_tf32(128, N);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int S = p.num_stages;
  const int KC = p.kc;
  uint8_t* ring = smem;                                                  // S x 16 KiB
  uint8_t* btile = ring + static_cast<size_t>(S) * kStageBytes;          // KC x (N x 128 B), 1 KiB aligned
  float* a1_s = reinterpret_cast<float*>(btile + static_cast<size_t>(KC) * N * 128);  // [kTcSlots][128]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(a1_s + kTcSlots * kTileRows);
  uint64_t* empty_bar = full_bar + S;
  uint64_t* dfull_bar = empty_bar + S;
  uint64_t* dempty_bar = dfull_bar + kTcAccStages;
  uint64_t* a1_bar = dempty_bar + kTcAccStages;
  uint32_t* tmem_base_s = reinterpret_cast<uint32_t*>(a1_bar + kTcSlots);
  // QUEUE kernels: flagged-row queue (slot = row + 1, 0 = empty; ctl: 0 tail reserved, 1 head claimed, 2 epilogue
  // warps done, 3 slots consumed), then the fp64 weights and one strip per epilogue / re-score warp
  int* q_slots = reinterpret_cast<int*>(tmem_base_s + 4);
  int* q_ctl = q_slots + kTcQueueCap;
  double* rs_area = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(q_ctl + 4) + 15u) & ~static_cast<uintptr_t>(15));  // 16-byte copies

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // W1 tile (already in the swizzled layout) -> shared memory, once per CTA
  {
    const float4* src = reinterpret_cast<const float4*>(p.w1_tiles);
    float4* dst = reinterpret_cast<float4*>(btile);
    const int n4 = KC * N * 32 / 4;
    for (int i = threadIdx.x; i < n4; i += blockDim.x) dst[i] = __ldg(src + i);
  }
  MlpRsView rs_view{};
  if constexpr (EXACT && QUEUE) {
    for (int i = threadIdx.x; i < kTcQueueCap + 4; i += blockDim.x) q_slots[i] = 0;
    rs_view = mlp_rs_stage(rs_area, p.rs_pack, p.n_in, H, C);
    __syncthreads();
    mlp_rs_finish_stage(rs_view);
  }
  double* rs_strips = rs_area + mlp_rs_weight_doubles(p.n_in, H, C);
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1 + 4);  // tcgen05.commit + the four scan warps
    }
    for (int a = 0; a < kTcAccStages; ++a) {
      mbar_init(&dfull_bar[a], 1);
      mbar_init(&dempty_bar[a], 4);  // the four epilogue warps
    }
    for (int s = 0; s < kTcSlots; ++s) mbar_init(&a1_bar[s], kTileRows);  // every scan thread arrives for its own row
    fence_barrier_init();
  }
  if (warp == kTcMmaWarp) tmem_alloc<TMEM_COLS>(tmem_base_s);
  fence_proxy_async_smem();  // the W1 tile was written with st.shared; UMMA reads it through the async proxy
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_s;

  pdl_launch_dependents();  // the fp64 re-score behind this launch may stage its weights while this grid runs
  const long long G = gridDim.x;
  const long long num_tiles = p.num_tiles;

  if (warp == kTcProducerWarp) {
    // ===================== TMA producer =====================
    if (elect_one_sync()) {
      tma_prefetch_desc(&xmap);
      const uint64_t policy = make_evict_first_policy();
      int stage = 0;
      uint32_t phase = 0;
      for (long long tile = blockIdx.x; tile < num_tiles; tile += G) {
        for (int k = 0; k < KC; ++k) {
          mbar_wait_relaxed(&empty_bar[stage], phase ^ 1u);
          mbar_arrive_expect_tx(&full_bar[stage], kStageBytes);
          tma_load_2d(ring + static_cast<size_t>(stage) * kStageBytes, &xmap, &full_bar[stage], k * kChunkF,
                      static_cast<int>(tile * kTileRows), policy);
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == kTcMmaWarp) {
    // ===================== MMA issuer (one lane) =====================
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0;
      for (long long tile = blockIdx.x; tile < num_tiles; tile += G, ++it) {
        const uint32_t acc = it % kTcAccStages;
        const uint32_t acc_phase = (it / kTcAccStages) & 1u;
        const uint32_t d_tmem = tmem_base + acc * N;
        for (int k = 0; k < KC; ++k) {
          mbar_wait_relaxed(&full_bar[stage], phase);
          if (k == 0) mbar_wait_relaxed(&dempty_bar[acc], acc_phase ^ 1u);  // epilogue has drained this accumulator
          tcgen05_fence_after();
          const uint32_t a_base = smem_u32(ring + static_cast<size_t>(stage) * kStageBytes);
          const uint32_t b_base = smem_u32(btile + static_cast<size_t>(k) * N * 128);
#pragma unroll
          for (int j = 0; j < kChunkF / 8; ++j) {  // K = 8 tf32 (32 bytes) per MMA
            umma_tf32_ss(d_tmem, umma_desc_k_sw128(a_base + j * 32), umma_desc_k_sw128(b_base + j * 32), IDESC,
                         (k | j) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);               // ring stage free once these MMAs have read it
          if (k == KC - 1) umma_commit(&dfull_bar[acc]);  // accumulator complete
          if (++stage == S) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp < 4) {
    // ===================== scan warps: thread per row, A1 bound + tf32 exactness =====================
    const int row = threadIdx.x;  // 0..127
    const uint32_t rowbase = static_cast<uint32_t>(row) * 128u;
    const uint32_t sw = static_cast<uint32_t>(row & 7) * 16u;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < num_tiles; tile += G, ++it) {
      float a1 = 0.f;
      uint32_t lowbits = 0u;
      for (int k = 0; k < KC; ++k) {
        mbar_wait_relaxed(&full_bar[stage], phase);
        const uint8_t* xs = ring + static_cast<size_t>(stage) * kStageBytes;
#pragma unroll
        for (int q = 0; q < kChunkF / 4; ++q) {
          const float4 v = *reinterpret_cast<const float4*>(xs + rowbase + ((static_cast<uint32_t>(q) * 16u) ^ sw));
          if (EXACT || PROBA) {
            const float* wm = p.w1max + k * kChunkF + q * 4;
            a1 = fmaf(fabsf(v.x), wm[0], a1);
            a1 = fmaf(fabsf(v.y), wm[1], a1);
            a1 = fmaf(fabsf(v.z), wm[2], a1);
            a1 = fmaf(fabsf(v.w), wm[3], a1);
          }
          lowbits |= __float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
        if (++stage == S) {
          stage = 0;
          phase ^= 1u;
        }
      }
      // a row whose features are not tf32 values was scored from truncated inputs: A1 = +inf sends it to the fp64 re-score
      const uint32_t slot = it % kTcSlots;
      a1_s[slot * kTileRows + row] = (lowbits & 0x1fffu) ? INFINITY : (a1 + p.b1max);
      mbar_arrive(&a1_bar[slot]);  // release: this thread's A1 is visible to whoever completes the wait
    }
  } else if (warp < 4 + kTcEpilogueWarps) {
    // ===================== epilogue warps 4..11: TMEM lane = row; set 0 (warps 4-7) even tiles, set 1 odd tiles ====
    const int wq = warp & 3;  // a warp may only touch TMEM lanes 32 * (warp % 4) .. + 31
    const int set = (warp - 4) >> 2;
    const int row_in_tile = wq * 32 + lane;
    uint32_t it = static_cast<uint32_t>(set);
    for (long long tile = blockIdx.x + set * G; tile < num_tiles; tile += 2 * G, it += 2) {
      const uint32_t acc = it % kTcAccStages;
      const uint32_t acc_phase = (it / kTcAccStages) & 1u;
      const uint32_t slot = it % kTcSlots;
      const uint32_t slot_phase = (it / kTcSlots) & 1u;
      mbar_wait_bounded(&dfull_bar[acc], acc_phase);
      mbar_wait_bounded(&a1_bar[slot], slot_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(wq * 32) << 16) + acc * N;
      uint32_t vmain[H], vsmall[H];
      if constexpr (H == 32) {
        tmem_ld_32x32b_x32(taddr, vmain);
        tmem_ld_32x32b_x32(taddr + H, vsmall);
      } else {
        tmem_ld_32x32b_x16(taddr, vmain);
        tmem_ld_32x32b_x16(taddr + H, vsmall);
      }
      tmem_ld_wait();
      const float a1 = a1_s[slot * kTileRows + row_in_tile];
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&dempty_bar[acc]);  // accumulator (and A1 slot) read: the MMA warp may reuse it

      // ---- + b1, ReLU, layer 2 (weights are constant-bank operands of the FMAs), argmax ----
      constexpr int NZ = C + (EXACT ? 1 : 0);
      float z[NZ];
#pragma unroll
      for (int c = 0; c < NZ; ++c) z[c] = p.b2[c];
#pragma unroll
      for (int n = 0; n < H; ++n) {
        const float h = (__uint_as_float(vsmall[n]) + __uint_as_float(vmain[n])) + p.b1[n];
        const float hv = fmaxf(h, 0.f);
#pragma unroll
        for (int c = 0; c < NZ; ++c) z[c] = fmaf(hv, p.w2[n][c], z[c]);
      }
      const long long row = tile * kTileRows + row_in_tile;
      if constexpr (PROBA) {
        // softmax, the warp's 32 rows out; rows the MMA could not score (A1 = +inf / NaN) are recomputed in fp64
        softmax_f32<C>(z);
        float* strip = reinterpret_cast<float*>(rs_area) + (warp - 4) * 32 * C;
        warp_store_proba<C, STAGED>(z, p.proba, tile * kTileRows + wq * 32, p.n_rows, lane, strip);
        flag_list_append(row < p.n_rows && !(a1 < INFINITY), row, p.flag_count, p.flag_rows, p.flag_cap, lane);
        continue;
      }
      float best = z[0];
      float second = -INFINITY;
      int idx = 0;
#pragma unroll
      for (int c = 1; c < C; ++c) {
        if (z[c] > best) {
          second = best;
          best = z[c];
          idx = c;
        } else {
          second = fmaxf(second, z[c]);
        }
      }
      const bool in_range = row < p.n_rows;
      if (in_range) {
        if (p.labels) p.labels[row] = idx;
        if (!p.wire_u8)
          for (int i = 0; i < p.n_peers; ++i) static_cast<int32_t*>(p.peers[i])[p.row_offset + row] = idx;
      }
      if (p.wire_u8 && p.n_peers > 0) {
        // byte labels: lanes 0..7 gather 4 consecutive rows each -> the warp's 32 labels leave as eight 4-byte words
        uint32_t word = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) word |= (static_cast<uint32_t>(__shfl_sync(0xffffffffu, idx, (4 * lane + t) & 31)) & 0xffu) << (8 * t);
        const long long row4 = tile * kTileRows + wq * 32 + 4 * lane;
        const long long at = p.row_offset + row4;
        if (lane < 8) {
          if (row4 + 3 < p.n_rows && (at & 3) == 0) {
            for (int i = 0; i < p.n_peers; ++i) *reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(p.peers[i]) + at) = word;
          } else {
            for (int t = 0; t < 4; ++t)
              if (row4 + t < p.n_rows)
                for (int i = 0; i < p.n_peers; ++i)
                  static_cast<uint8_t*>(p.peers[i])[at + t] = static_cast<uint8_t>((word >> (8 * t)) & 0xffu);
          }
        }
      }
      if (EXACT) {
        // |z_c - true| <= E1 * max_c sum_n |w2_cn| + (H+4) u A2   (ReLU is 1-Lipschitz); NaN/Inf -> comparison false
        const float err = p.e1_scale * a1 + p.e2_scale * z[C];
        const bool certain = (best - second) > 2.0f * err;
        const bool flagged = in_range && !certain;
        const unsigned mask = __ballot_sync(0xffffffffu, flagged);
        if (mask != 0u) {
          if constexpr (QUEUE) {
            // hand the flagged rows to the re-score warps of this launch; the labels stored above are provisional
            __threadfence();
            const int total = __popc(mask);
            int base = -1;
            if (lane == 0) {
              const int tail = atomicAdd(&q_ctl[0], 0);
              const int consumed = atomicAdd(&q_ctl[3], 0);
              if (tail - consumed <= kTcQueueCap - kTcQueueHeadroom) base = atomicAdd(&q_ctl[0], total);
            }
            base = __shfl_sync(0xffffffffu, base, 0);
            if (base >= 0) {
              if (flagged) {
                const int slot = (base + __popc(mask & ((1u << lane) - 1u))) & (kTcQueueCap - 1);
                while (atomicAdd(&q_slots[slot], 0) != 0) {  // only if the slot's previous ticket is claimed but not read yet
                }
                atomicExch(&q_slots[slot], static_cast<int>(row) + 1);
              }
            } else {
              // queue backed up (most rows near-ties): this warp re-scores its own rows in fp64
              double* xs = rs_strips + (warp - 4) * mlp_rs_strip_doubles(p.n_in, H);
              unsigned m2 = mask;
              while (m2 != 0u) {
                const int l = __ffs(static_cast<int>(m2)) - 1;
                m2 &= m2 - 1u;
                const long long frow = tile * kTileRows + wq * 32 + l;
                const MlpRowResult r = mlp_rs_row(rs_view, p.x + frow * p.ld, xs, xs + p.n_in, lane);
                if (lane == 0) {
                  tc_store_final_label(p, frow, r.idx);
                  if (r.bad) atomicAdd(&p.counters[1], 1ull);
                  if (r.ambiguous) atomicAdd(&p.counters[0], 1ull);
                }
              }
              if (lane == 0) atomicAdd(&p.counters[2], static_cast<unsigned long long>(total));
            }
          } else {
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
    if constexpr (EXACT && QUEUE) {
      __syncwarp();
      if (lane == 0) {
        __threadfence_block();
        atomicAdd(&q_ctl[2], 1);  // this epilogue warp has published everything it will ever publish
      }
    }
  } else {
    // ===================== re-score warps 14..17 (QUEUE kernels): fp64 rows from the queue =====================
    if constexpr (EXACT && QUEUE) {
      double* xs = rs_strips + (kTcEpilogueWarps + (warp - kTcFirstRescoreWarp)) * mlp_rs_strip_doubles(p.n_in, H);
      int n_done = 0;
      for (;;) {
        // claim the next ticket, then wait until its slot is published (lane 0 polls and broadcasts: the lanes of a
        // warp need not run in lockstep)
        int t = 0;
        if (lane == 0) t = atomicAdd(&q_ctl[1], 1);
        t = __shfl_sync(0xffffffffu, t, 0);
        int v = 0;
        for (;;) {
          int state = 0;  // 1: nothing will ever be published for this ticket
          if (lane == 0) {
            v = atomicAdd(&q_slots[t & (kTcQueueCap - 1)], 0);
            if (v == 0 && atomicAdd(&q_ctl[2], 0) == kTcEpilogueWarps) {
              __threadfence_block();
              if (t >= atomicAdd(&q_ctl[0], 0)) state = 1;
            }
          }
          v = __shfl_sync(0xffffffffu, v, 0);
          state = __shfl_sync(0xffffffffu, state, 0);
          if (v != 0 || state == 1) break;
          __nanosleep(200);
        }
        if (v == 0) break;
        if (lane == 0) {
          atomicExch(&q_slots[t & (kTcQueueCap - 1)], 0);
          atomicAdd(&q_ctl[3], 1);
        }
        const long long frow = static_cast<long long>(v) - 1;
        const MlpRowResult r = mlp_rs_row(rs_view, p.x + frow * p.ld, xs, xs + p.n_in, lane);
        if (lane == 0) {
          tc_store_final_label(p, frow, r.idx);
          if (r.bad) atomicAdd(&p.counters[1], 1ull);
          if (r.ambiguous) atomicAdd(&p.counters[0], 1ull);
        }
        ++n_done;
      }
      if (lane == 0 && n_done > 0) atomicAdd(&p.counters[2], static_cast<unsigned long long>(n_done));
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == kTcMmaWarp) {
    tcgen05_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static float tf32_round(float v) {  // round to nearest tf32 (10 mantissa bits), ties away from zero
  uint32_t b;
  memcpy(&b, &v, 4);
  if ((b & 0x7f800000u) == 0x7f800000u) return v;  // Inf / NaN
  b = (b + 0x1000u) & 0xffffe000u;
  float r;
  memcpy(&r, &b, 4);
  return r;
}

// B operand of layer 1: per 32-feature chunk, 2H rows ([hi rows | lo rows]) of 32 floats, each row's 16-byte chunks
// XOR-swizzled by (row & 7) - the SWIZZLE_128B K-major layout the UMMA descriptor (and TMA) use
std::vector<float> mlp_tc_build_w1_tiles(const float* w1 /*[H][F]*/, int H, int F, int f_pad) {
  const int KC = f_pad / kChunkF, N = 2 * H;
  std::vector<float> tiles(static_cast<size_t>(KC) * N * 32, 0.f);
  for (int kc = 0; kc < KC; ++kc)
    for (int n = 0; n < N; ++n)
      for (int j = 0; j < 32; ++j) {
        const int f = kc * 32 + j;
        float v = 0.f;
        if (f < F) {
          const float w = w1[static_cast<size_t>(n % H) * F + f];
          const float hi = tf32_round(w);
          v = n < H ? hi : tf32_round(w - hi);  // w - hi is exact in fp32
        }
        const size_t off = (static_cast<size_t>(kc) * N + n) * 32 + static_cast<size_t>(((j / 4) ^ (n & 7)) * 4 + (j % 4));
        tiles[off] = v;
      }
  return tiles;
}

static size_t mlp_tc_fixed_smem(const MlpDeviceModel& m, bool queue, bool proba = false) {
  const size_t kc = m.f_pad / kChunkF;
  size_t bytes = 1024 + kc * (2 * m.n_hidden) * 128 + static_cast<size_t>(kTcSlots) * kTileRows * 4 +
                 (2 * 64 + 2 * kTcAccStages + kTcSlots) * 8 + 16;
  if (proba)  // (queue control words, unused) + one 32-row output strip per epilogue warp
    bytes += (kTcQueueCap + 4) * 4 + 16 + static_cast<size_t>(kTcEpilogueWarps) * 32 * m.n_classes * 4;
  if (queue)  // flagged-row queue + fp64 weights + one strip per epilogue / re-score warp
    bytes += (kTcQueueCap + 4) * 4 + 16 +
             (mlp_rs_weight_doubles(m.n_in, m.n_hidden, m.n_classes) +
              (kTcEpilogueWarps + kTcRescoreWarps) * mlp_rs_strip_doubles(m.n_in, m.n_hidden)) * 8;
  return bytes;
}

bool mlp_tc_queue_rescore() {
  // UML_B200_MLP_RESCORE_MODE=queue: rows flagged by the epilogue go through a shared-memory queue to four fp64
  // re-score warps of the same launch; =kernel: flag list + mlp_rescore_f64_kernel behind the scoring kernel
  static const int mode = [] {
    const char* env = getenv("UML_B200_MLP_RESCORE_MODE");
    if (env && env[0] == 'q') return 1;
    if (env && env[0] == 'k') return 0;
    return UML_MLP_QUEUE_DEFAULT;
  }();
  return mode == 1;
}

bool mlp_tc_supported(const MlpDeviceModel& m, std::string* why) {
  const bool shape_ok = (m.n_hidden == 32 || m.n_hidden == 16) && (m.n_classes == 10 || m.n_classes == 2 || m.n_classes == 3);
  if (!shape_ok) {
    if (why) *why = "tensor-core kernel instantiated for hidden in {16, 32} and classes in {2, 3, 10}";
    return false;
  }
  if (m.f_pad > kTcMaxFpad || m.w1_tiles == nullptr) {
    if (why) *why = "more than 128 features: the resident W1 tile is sized for F_pad <= 128";
    return false;
  }
  return mlp_tc_fixed_smem(m, true) + 6 * static_cast<size_t>(kStageBytes) <= static_cast<size_t>(kMaxSmemBytes);
}

template <int H, int C, bool EXACT, bool QUEUE, bool PROBA = false, bool STAGED = false>
static cudaError_t mlp_tc_launch_one(const CUtensorMap& xmap, const MlpDeviceModel& m, const MlpTcLaunch& l,
                                     const FlagList& flags, int sm_count, cudaStream_t stream, float* proba = nullptr) {
  using Params = MlpTcParams<H, C>;
  static_assert(sizeof(Params) < 4000, "kernel parameters must stay below the 4 KiB limit");
  Params p;
  memset(&p, 0, sizeof(p));
  const MlpHostModel& hm = *m.host;
  for (int n = 0; n < H; ++n) {
    p.b1[n] = hm.b1[n];
    for (int c = 0; c < C; ++c) p.w2[n][c] = hm.w2[static_cast<size_t>(c) * H + n];
    float wmax = 0.f;
    for (int c = 0; c < C; ++c) wmax = fmaxf(wmax, fabsf(hm.w2[static_cast<size_t>(c) * H + n]));
    p.w2[n][C] = wmax;
  }
  float b2max = 0.f, b1max = 0.f;
  for (int c = 0; c < C; ++c) {
    p.b2[c] = hm.b2[c];
    b2max = fmaxf(b2max, fabsf(hm.b2[c]));
  }
  p.b2[C] = b2max;
  for (int n = 0; n < H; ++n) b1max = fmaxf(b1max, fabsf(hm.b1[n]));
  p.b1max = b1max;
  for (int f = 0; f < m.n_in; ++f) {
    float wmax = 0.f;
    for (int n = 0; n < H; ++n) wmax = fmaxf(wmax, fabsf(hm.w1[static_cast<size_t>(n) * m.n_in + f]));
    p.w1max[f] = wmax;
  }
  const double u = 5.9604644775390625e-08;  // 2^-24
  const double F = m.n_in, n_mma = m.f_pad / 8.0;
  // layer-1 error as it reaches a logit: per accumulating MMA step <= 32 u (running |.| sum) - a truncating 9-addend
  // aligner without guard bits gives (9 * 2 + 2) u = 20 u -, + 4 u for the W1 split remainder, + 8 u for the small
  // accumulator and the two fp32 adds of the epilogue; A1 itself is an fp32 sum of F terms (factor 1 + F 2^-21)
  p.e1_scale = static_cast<float>((32.0 * n_mma + 12.0) * u * (1.0 + F * 4.76837158203125e-07) * 1.0001 * m.w2_abs_row_sum_max);
  p.e2_scale = static_cast<float>((H + 4.0) * u * 1.0001);
  p.w1_tiles = m.w1_tiles;
  p.labels = l.labels;
  p.n_peers = l.n_peers;
  p.wire_u8 = l.wire_u8;
  for (int i = 0; i < 8; ++i) p.peers[i] = i < l.n_peers ? l.peers[i] : nullptr;
  p.row_offset = l.row_offset;
  p.n_rows = l.n_rows;
  p.num_tiles = (l.n_rows + kTileRows - 1) / kTileRows;
  p.kc = m.f_pad / kChunkF;
  p.x = l.x;
  p.ld = l.ld;
  p.n_in = m.n_in;
  p.rs_pack = m.rs_pack;
  p.counters = flags.counters;
  p.proba = proba;
  const size_t fixed = mlp_tc_fixed_smem(m, QUEUE, PROBA);
  int stages = static_cast<int>((static_cast<size_t>(kMaxSmemBytes) - fixed) / kStageBytes);
  stages = std::min(stages, 64);
  if (const char* env = getenv("UML_B200_STAGES")) stages = std::max(4, std::min(stages, atoi(env)));
  // the A1 hand-off has kTcSlots slots: the scan warps lead the epilogue by at most S / KC + 1 + kTcAccStages tiles
  stages = std::min(stages, (kTcSlots - 2 - kTcAccStages) * p.kc);
  p.num_stages = stages;
  p.flag_count = flags.count;
  p.flag_rows = flags.rows;
  p.flag_cap = flags.capacity;
  const size_t smem = fixed + static_cast<size_t>(stages) * kStageBytes;
  auto kern = mlp_argmax_tc_kernel<H, C, EXACT, QUEUE, PROBA, STAGED>;
  static size_t configured = 0;
  if (smem > configured) {
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (err != cudaSuccess) return err;
    configured = smem;
  }
  const int grid = static_cast<int>(std::min<long long>(sm_count, std::max<long long>(1, p.num_tiles)));
  kern<<<grid, QUEUE ? kTcThreadsQueue : kTcThreads, smem, stream>>>(xmap, p);
  return cudaGetLastError();
}

cudaError_t launch_mlp_tc(const CUtensorMap& xmap, const MlpDeviceModel& m, const MlpTcLaunch& l, bool exact,
                          const FlagList& flags, int sm_count, cudaStream_t stream, bool* rescore_kernel_needed) {
  const bool queue = exact && mlp_tc_queue_rescore();
  if (rescore_kernel_needed) *rescore_kernel_needed = exact && !queue;
  if (l.n_rows <= 0) return cudaSuccess;
#define UML_TC_CASE(HH, CC)                                                                                      \
  if (m.n_hidden == HH && m.n_classes == CC) {                                                                   \
    if (!exact) return mlp_tc_launch_one<HH, CC, false, false>(xmap, m, l, flags, sm_count, stream);             \
    return queue ? mlp_tc_launch_one<HH, CC, true, true>(xmap, m, l, flags, sm_count, stream)                    \
                 : mlp_tc_launch_one<HH, CC, true, false>(xmap, m, l, flags, sm_count, stream);                  \
  }
  UML_TC_CASE(32, 10) UML_TC_CASE(32, 2) UML_TC_CASE(32, 3) UML_TC_CASE(16, 10) UML_TC_CASE(16, 2) UML_TC_CASE(16, 3)
#undef UML_TC_CASE
  return cudaErrorInvalidValue;
}

bool mlp_proba_staged_store() {
  // UML_B200_MLP_PROBA_STORE=staged: probabilities leave through a shared-memory strip as coalesced 16-byte stores;
  // =direct: every lane stores its own row (DESIGN.md 3.6 has the same-box A/B behind the default)
  static const int mode = [] {
    const char* env = getenv("UML_B200_MLP_PROBA_STORE");
    if (env && env[0] == 's') return 1;
    if (env && env[0] == 'd') return 0;
    return UML_MLP_PROBA_STAGED_DEFAULT;
  }();
  return mode == 1;
}

cudaError_t launch_mlp_tc_proba(const CUtensorMap& xmap, const MlpDeviceModel& m, const MlpTcLaunch& l, float* proba,
                                const FlagList& flags, int sm_count, cudaStream_t stream) {
  if (l.n_rows <= 0) return cudaSuccess;
  const bool staged = mlp_proba_staged_store();
#define UML_TC_CASE(HH, CC)                                                                                        \
  if (m.n_hidden == HH && m.n_classes == CC)                                                                       \
    return staged ? mlp_tc_launch_one<HH, CC, false, false, true, true>(xmap, m, l, flags, sm_count, stream, proba) \
                  : mlp_tc_launch_one<HH, CC, false, false, true, false>(xmap, m, l, flags, sm_count, stream, proba);
  UML_TC_CASE(32, 10) UML_TC_CASE(32, 2) UML_TC_CASE(32, 3) UML_TC_CASE(16, 10) UML_TC_CASE(16, 2) UML_TC_CASE(16, 3)
#undef UML_TC_CASE
  return cudaErrorInvalidValue;
}

}  // namespace uml
