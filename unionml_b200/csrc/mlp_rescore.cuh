// float64 re-score of rows of the 2-layer MLP by one warp, with every operand in shared memory.  Shared by the
// stand-alone re-score kernel (mlp_kernels.cu) and the re-score warps inside the tensor-core kernel (mlp_tc_kernels.cu).
//
// The kernel is bound by shared-memory bandwidth, not by fp64 math: W1 is F x H doubles and a warp that scores ONE row
// reads all of it (2 wavefronts per feature) for 1 fma per lane and feature.  mlp_rs_rows<R> therefore scores R rows
// per pass: each W1 / W2 element read from shared memory is used R times, the rows' features and hidden activations
// sit interleaved ([f][R]) so one broadcast 16-byte load carries two rows' values.  R = 4: 1 wavefront per row and
// feature instead of 3.
#pragma once

#include <vector>

#include "rescore_util.cuh"
#include "tma_ring.cuh"

namespace uml {

// fp64 operands of one block: an image built ONCE on the host at model load (mlp_rs_build_pack) and copied verbatim
// into shared memory - W1 [F][H], W2 [C][H + 1] (padded rows: lane-per-class reads are conflict free), biases, the two
// bound vectors w1m[f] = max_n |w1_nf|, w2m[n] = max_c |w2_cn| and three scalars.
struct MlpRsView {
  const double* w1s;
  const double* w2s;
  const double* b1s;
  const double* b2s;
  const double* w1m;
  const double* w2m;
  double b1max, b2max, w2sum;
  int F, H, C;
};

__host__ __device__ inline size_t mlp_rs_weight_doubles(int F, int H, int C) {
  const size_t n = static_cast<size_t>(F) * H + static_cast<size_t>(C) * (H + 1) + H + C + F + H + 3;
  return (n + 1) & ~static_cast<size_t>(1);  // even: 16-byte copies, and the strips behind it stay 16-byte aligned
}
// a warp's strip: features and hidden activations of the R rows of one pass
__host__ __device__ inline size_t mlp_rs_strip_doubles(int F, int H, int R = 1) { return (static_cast<size_t>(F) + H) * R; }

// host: the shared-memory image from the caller's (fp32) weights; w1 is [H][F], w2 is [C][H] as torch holds them
inline std::vector<double> mlp_rs_build_pack(const float* w1, const float* b1, const float* w2, const float* b2, int F,
                                             int H, int C) {
  std::vector<double> pack(mlp_rs_weight_doubles(F, H, C), 0.0);
  const int HP = H + 1;
  double* w1s = pack.data();
  double* w2s = w1s + static_cast<size_t>(F) * H;
  double* b1s = w2s + static_cast<size_t>(C) * HP;
  double* b2s = b1s + H;
  double* w1m = b2s + C;
  double* w2m = w1m + F;
  double* scal = w2m + H;
  for (int f = 0; f < F; ++f) {
    double m = 0.0;
    for (int n = 0; n < H; ++n) {
      const double v = static_cast<double>(w1[static_cast<size_t>(n) * F + f]);
      w1s[static_cast<size_t>(f) * H + n] = v;  // feature-major: lane n reads consecutive doubles
      m = v < 0 ? (-v > m ? -v : m) : (v > m ? v : m);
    }
    w1m[f] = m;
  }
  double b1max = 0.0, b2max = 0.0, w2sum = 0.0;
  for (int n = 0; n < H; ++n) {
    b1s[n] = static_cast<double>(b1[n]);
    const double a = b1s[n] < 0 ? -b1s[n] : b1s[n];
    b1max = a > b1max ? a : b1max;
    double m = 0.0;
    for (int c = 0; c < C; ++c) {
      const double v = static_cast<double>(w2[static_cast<size_t>(c) * H + n]);
      w2s[static_cast<size_t>(c) * HP + n] = v;
      const double av = v < 0 ? -v : v;
      m = av > m ? av : m;
    }
    w2m[n] = m;
    w2sum += m;  // sum_n max_c |w2_cn|: how far a hidden-layer error can move any logit
  }
  for (int c = 0; c < C; ++c) {
    b2s[c] = static_cast<double>(b2[c]);
    const double a = b2s[c] < 0 ? -b2s[c] : b2s[c];
    b2max = a > b2max ? a : b2max;
  }
  scal[0] = b1max;
  scal[1] = b2max;
  scal[2] = w2sum;
  return pack;
}

// all threads of the block: copy the image from global memory (16-byte loads); returns the view.  After a block-wide
// barrier every thread calls mlp_rs_finish_stage (the three scalars, broadcast reads) before scoring rows.
__device__ inline MlpRsView mlp_rs_stage(double* smem, const double* pack, int F, int H, int C) {
  const int n2 = static_cast<int>(mlp_rs_weight_doubles(F, H, C) / 2);
  const double2* src = reinterpret_cast<const double2*>(pack);
  double2* dst = reinterpret_cast<double2*>(smem);
  for (int i = threadIdx.x; i < n2; i += blockDim.x) dst[i] = src[i];
  MlpRsView v;
  v.w1s = smem;
  v.w2s = v.w1s + F * H;
  v.b1s = v.w2s + C * (H + 1);
  v.b2s = v.b1s + H;
  v.w1m = v.b2s + C;
  v.w2m = v.w1m + F;
  v.F = F;
  v.H = H;
  v.C = C;
  v.b1max = v.b2max = v.w2sum = 0.0;
  return v;
}

__device__ inline void mlp_rs_finish_stage(MlpRsView& v) {
  const double* scal = v.w2m + v.H;
  v.b1max = scal[0];
  v.b2max = scal[1];
  v.w2sum = scal[2];
}

struct MlpRowResult {
  int idx;
  bool bad;        // NaN/Inf in the row
  bool ambiguous;  // fp64 logit margin inside the fp64 rounding bound (a true tie; first index wins)
};

// Layer 1 of R rows on one warp: features -> xs ([f][R] doubles), ReLU'd hidden values -> hv ([n][R]).  xr[r] = row
// r's fp32 features in global memory (callers pass a valid row for unused slots and ignore that result).  Returns per
// row: NaN/Inf in the features, a hidden unit's own fp64 rounding bound (herr) and the bound on every logit's absolute
// sum (amax).
template <int R>
__device__ __forceinline__ void mlp_rs_hidden(const MlpRsView& v, const float* const (&xr)[R], double* xs, double* hv, int lane,
                                              bool (&bad)[R], double (&herr)[R], double (&amax)[R]) {
  static_assert(R == 1 || R == 2 || R == 4, "rows per pass");
  const double u = 1.1102230246251565e-16;  // 2^-53
  const int F = v.F, H = v.H;
  double a1[R];  // sum_f |x_f| max_n |w1_nf|: bounds every hidden unit's absolute sum (one chain instead of H)
#pragma unroll
  for (int r = 0; r < R; ++r) {
    bad[r] = false;
    a1[r] = 0.0;
  }
  for (int f = lane; f < F; f += 32) {
    float xf[R];
#pragma unroll
    for (int r = 0; r < R; ++r) xf[r] = xr[r][f];  // R independent coalesced loads in flight
    const double wm = v.w1m[f];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      bad[r] |= !isfinite(xf[r]);
      const double xd = static_cast<double>(xf[r]);
      xs[f * R + r] = xd;
      a1[r] = fma(fabs(xd), wm, a1[r]);
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    bad[r] = __any_sync(0xffffffffu, bad[r]);
    a1[r] = warp_sum(a1[r]) + v.b1max;
    herr[r] = (F + 6.0) * u * a1[r];  // any hidden unit's own fp64 rounding error (one chain of F fmas + the bias add)
  }
  __syncwarp();  // the strip writes above are read by other lanes below
  // ---- hidden layer: lane per unit, one chain per row over the features (R independent chains) ----
  double a2[R];  // sum_n h_n max_c |w2_cn|: bounds every logit's absolute sum
#pragma unroll
  for (int r = 0; r < R; ++r) a2[r] = 0.0;
  for (int hn = lane; hn < H; hn += 32) {
    double s[R];
#pragma unroll
    for (int r = 0; r < R; ++r) s[r] = 0.0;
    const double* wcol = v.w1s + hn;
#pragma unroll 4
    for (int f = 0; f < F; ++f) {
      const double w = wcol[f * H];
      if constexpr (R == 1) {
        s[0] = fma(xs[f], w, s[0]);
      } else {
#pragma unroll
        for (int r = 0; r < R; r += 2) {
          const double2 x2 = *reinterpret_cast<const double2*>(xs + f * R + r);  // broadcast 16-byte load: two rows
          s[r] = fma(x2.x, w, s[r]);
          s[r + 1] = fma(x2.y, w, s[r + 1]);
        }
      }
    }
    const double b = v.b1s[hn], wm = v.w2m[hn];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const double h = fmax(s[r] + b, 0.0);
      hv[hn * R + r] = h;
      a2[r] = fma(h, wm, a2[r]);
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) amax[r] = warp_sum(a2[r]) + herr[r] * v.w2sum + v.b2max;
  __syncwarp();
}

// One warp, R rows per pass: arg-max and runner-up of the fp64 logits.  xs / hv = the warp's strip, F x R and H x R
// doubles, 16-byte aligned.
template <int R>
__device__ __forceinline__ void mlp_rs_rows(const MlpRsView& v, const float* const (&xr)[R], double* xs, double* hv, int lane,
                                            MlpRowResult (&out)[R]) {
  const double u = 1.1102230246251565e-16;  // 2^-53
  const int H = v.H, C = v.C, HP = v.H + 1;
  bool bad[R];
  double herr[R], amax[R];
  mlp_rs_hidden<R>(v, xr, xs, hv, lane, bad, herr, amax);
  // ---- output layer: lane per class, one chain per row over the hidden units ----
  Top2 top[R];
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + lane;
    double s[R];
#pragma unroll
    for (int r = 0; r < R; ++r) s[r] = 0.0;
    if (c < C) {
      const double* w2c = v.w2s + c * HP;
#pragma unroll 4
      for (int nn = 0; nn < H; ++nn) {
        const double w = w2c[nn];
        if constexpr (R == 1) {
          s[0] = fma(hv[nn], w, s[0]);
        } else {
#pragma unroll
          for (int r = 0; r < R; r += 2) {
            const double2 h2 = *reinterpret_cast<const double2*>(hv + nn * R + r);
            s[r] = fma(h2.x, w, s[r]);
            s[r + 1] = fma(h2.y, w, s[r + 1]);
          }
        }
      }
    }
    const double b = c < C ? v.b2s[c] : 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      Top2 t;
      t.best = c < C ? s[r] + b : -INFINITY;
      t.second = -INFINITY;
      t.idx = c;
      top2_butterfly(t, 1);
      if (c0 == 0) {
        top[r] = t;
      } else if (t.best > top[r].best) {
        top[r].second = fmax(top[r].best, t.second);
        top[r].best = t.best;
        top[r].idx = t.idx;
      } else {
        top[r].second = fmax(top[r].second, t.best);
      }
    }
  }
  __syncwarp();  // the strip may be reused by the caller's next pass
#pragma unroll
  for (int r = 0; r < R; ++r) {
    out[r].idx = top[r].idx >= C ? 0 : top[r].idx;  // idx >= C only with NaN scores, which are reported through `bad`
    out[r].bad = bad[r];
    // fp64 error of a logit: the hidden units' own errors carried through W2, plus the output layer's chain
    const double err = herr[r] * v.w2sum + (static_cast<double>(H) + 16.0) * u * amax[r];
    out[r].ambiguous = !((top[r].best - top[r].second) > 2.0 * err);
  }
}

// doubles of a warp's strip for mlp_rs_proba_rows: the logits reuse the feature area once layer 1 is done with it
__host__ __device__ inline size_t mlp_rs_proba_strip_doubles(int F, int H, int C, int R) {
  return (static_cast<size_t>(F > C ? F : C) + H) * R;
}

// One warp, R rows per pass: softmax of the fp64 logits, rounded once to fp32 into out[r][0..C) (out[r] == nullptr:
// unused slot).  xs: max(F, C) x R doubles, hv: H x R, 16-byte aligned.  bad[r]: NaN/Inf in row r's features.
template <int R>
__device__ __forceinline__ void mlp_rs_proba_rows(const MlpRsView& v, const float* const (&xr)[R], double* xs, double* hv,
                                                  int lane, float* const (&out)[R], bool (&bad)[R]) {
  const int H = v.H, C = v.C, HP = v.H + 1;
  double herr[R], amax[R];
  mlp_rs_hidden<R>(v, xr, xs, hv, lane, bad, herr, amax);
  // ---- output layer: lane per class, logits -> xs ([c][R]) ----
  for (int c = lane; c < C; c += 32) {
    double s[R];
#pragma unroll
    for (int r = 0; r < R; ++r) s[r] = 0.0;
    const double* w2c = v.w2s + c * HP;
#pragma unroll 4
    for (int nn = 0; nn < H; ++nn) {
      const double w = w2c[nn];
#pragma unroll
      for (int r = 0; r < R; ++r) s[r] = fma(hv[nn * R + r], w, s[r]);
    }
#pragma unroll
    for (int r = 0; r < R; ++r) xs[c * R + r] = s[r] + v.b2s[c];
  }
  __syncwarp();
  // ---- softmax per row: max, sum of exp, one division ----
#pragma unroll
  for (int r = 0; r < R; ++r) {
    double m = -INFINITY;
    for (int c = lane; c < C; c += 32) m = fmax(m, xs[c * R + r]);
    m = warp_max(m, 1);
    double sum = 0.0;
    for (int c = lane; c < C; c += 32) sum += exp(xs[c * R + r] - m);
    sum = warp_sum(sum);
    if (out[r] != nullptr)
      for (int c = lane; c < C; c += 32) out[r][c] = static_cast<float>(exp(xs[c * R + r] - m) / sum);
  }
  __syncwarp();  // the strip may be reused by the caller's next pass
}

// one row (the re-score warps inside the tensor-core kernel take rows one at a time from their queue)
__device__ __forceinline__ MlpRowResult mlp_rs_row(const MlpRsView& v, const float* __restrict__ xr, double* xs, double* hv,
                                                  int lane) {
  const float* const rows[1] = {xr};
  MlpRowResult out[1];
  mlp_rs_rows<1>(v, rows, xs, hv, lane, out);
  return out[0];
}

}  // namespace uml
