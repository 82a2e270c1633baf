// Probability epilogue of the MLP scoring kernels (uml_mlp_predict_proba): fp32 softmax of a row's C logits in torch's
// form and the store of a warp's 32 consecutive rows (128 * C contiguous bytes of the row-major output).
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace uml {

// softmax in place, as torch computes it: m = max z, e_c = exp(z_c - m), p_c = e_c / sum e (accurate expf: the
// probabilities are compared against the fp64 forward at ~1e-7)
template <int C>
__device__ __forceinline__ void softmax_f32(float (&z)[C]) {
  float m = z[0];
#pragma unroll
  for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    z[c] = expf(z[c] - m);
    s += z[c];
  }
#pragma unroll
  for (int c = 0; c < C; ++c) z[c] = z[c] / s;
}

// Warp-wide: lane l holds row row0 + l (row0 % 32 == 0; rows >= n_rows are not stored).  out is 16-byte aligned, so
// the warp's block out + row0 * C is too.
//   STAGED = false: each lane stores its own C floats (8-byte stores when C is even);
//   STAGED = true : the rows go through the warp's strip (32 * C floats of shared memory, 16-byte aligned) and leave
//                   as coalesced 16-byte stores.
template <int C, bool STAGED>
__device__ __forceinline__ void warp_store_proba(const float (&p)[C], float* __restrict__ out, long long row0,
                                                 long long n_rows, int lane, float* strip) {
  const long long row = row0 + lane;
  if constexpr (!STAGED) {
    if (row < n_rows) {
      float* o = out + row * C;
      if constexpr (C % 2 == 0) {
#pragma unroll
        for (int c = 0; c < C; c += 2) *reinterpret_cast<float2*>(o + c) = make_float2(p[c], p[c + 1]);
      } else {
#pragma unroll
        for (int c = 0; c < C; ++c) o[c] = p[c];
      }
    }
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) strip[lane * C + c] = p[c];
    __syncwarp();
    const long long left = n_rows - row0;
    const int total = (left >= 32 ? 32 : static_cast<int>(left > 0 ? left : 0)) * C;
    float* o = out + row0 * C;
    const int n4 = total / 4;
    for (int i = lane; i < n4; i += 32) reinterpret_cast<float4*>(o)[i] = reinterpret_cast<const float4*>(strip)[i];
    for (int i = 4 * n4 + lane; i < total; i += 32) o[i] = strip[i];
    __syncwarp();  // the strip is rewritten by the warp's next rows
  }
}

// Warp-wide: append the rows with `flagged` set to the flag list (the fp64 kernel behind the scoring kernel recomputes
// them).  Order within the list is irrelevant.
__device__ __forceinline__ void flag_list_append(bool flagged, long long row, int* count, int32_t* rows, int cap, int lane) {
  const unsigned mask = __ballot_sync(0xffffffffu, flagged);
  if (mask == 0u) return;
  int base = 0;
  if (lane == 0) base = atomicAdd(count, __popc(mask));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (flagged) {
    const int pos = base + __popc(mask & ((1u << lane) - 1u));
    if (pos < cap) rows[pos] = static_cast<int32_t>(row);
  }
}

}  // namespace uml
