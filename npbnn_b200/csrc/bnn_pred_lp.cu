// Opt-in reduced-precision posterior prediction (option "predict_tf32", north star: "opt-in TF32 ... tensor-core tiles",
// stated tolerance): the forward pass of get_posterior_cat_prob / RunPredict (BNN_lib.py:245-256, 376-392) for the
// 64 -> 64 -> 32 -> 16 padded family with the contractions on the TF32 tensor cores (mma.sync m16n8k8, FP32
// accumulators) in the error-compensated 3xTF32 form
//     a b ~= a_hi b_hi + a_hi b_lo + a_lo b_hi,     x_hi = tf32(x), x_lo = tf32(x - x_hi)
// (products exact to 2^-22 relative), activations and softmax in FP32, and the per-row class probabilities summed
// over the posterior samples in FP64.  Class probabilities agree with the FP64 kernel to ~1e-6 absolute
// (tests/test_gpu_api.py::test_predict_tf32_mode); the Metropolis-Hastings path NEVER uses this kernel: an accept
// decision compares log-posteriors whose difference is O(1) on a value of O(1e6).
//
// Layout and fragment mapping are the FP64 kernel's (bnn_common.cuh: K index permuted inside each group of 8 columns, so
// that the accumulator fragment of one layer IS the A fragment of the next).  A warp owns a 16-row tile whose X
// fragments (hi / lo) stay in registers for all samples; the packed weight sets are converted once per call, in place, to
// (hi, lo) float pairs -- 8 bytes per weight, like the double they replace -- and streamed through two shared-memory
// buffers by cp.async.
#include "bnn_common.cuh"
#include "bnn_kernels.h"

namespace {

constexpr int LP_WARPS = 10;          // 190-200 registers per thread: ten warps fill the register file of an SM
constexpr int KP0 = 64, N1 = 64, N2 = 32, N3 = 16;
constexpr int W1_OFF = 0, B1_OFF = N1 * KP0, W2_OFF = B1_OFF + N1, B2_OFF = W2_OFF + N2 * N1, W3_OFF = B2_OFF + N2,
              B3_OFF = W3_OFF + N3 * N2, PBF = B3_OFF + N3;

__device__ __forceinline__ uint32_t to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ void split_tf32(float v, uint32_t& hi, uint32_t& lo) {
  hi = to_tf32(v);
  lo = to_tf32(v - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// one k-group of an [16 x 8k] x [8k x 8] product in 3xTF32: (ah, al) A fragments, W row pointer to (hi, lo) float pairs
// One k-group of a layer for all NT output tiles.  PASSES = 3: error-compensated (products to 2^-22), PASSES = 1: plain TF32
// (10-bit mantissas, products to 2^-11).  The three products of an accumulator are issued NT instructions apart (pass by
// pass over the tiles), never back to back: a dependent mma.sync waits ~30 clk for its accumulator.
//   wr: W row (n0 + gq) of the layer as (hi, lo) float pairs, already offset by the swizzled column of this k-group
template <int PASSES, int NT>
__device__ __forceinline__ void mma_kgroup(float (&acc)[NT][4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                           const float2* wr, int row_stride8) {
  float4 w[NT];                                   // (W[n][2t].hi, W[n][2t+1].hi, W[n][2t].lo, W[n][2t+1].lo)
#pragma unroll
  for (int j = 0; j < NT; ++j) w[j] = *reinterpret_cast<const float4*>(wr + j * row_stride8);
  if (PASSES == 3) {
#pragma unroll
    for (int j = 0; j < NT; ++j) mma_tf32(acc[j], al, __float_as_uint(w[j].x), __float_as_uint(w[j].y));   // small terms first
#pragma unroll
    for (int j = 0; j < NT; ++j) mma_tf32(acc[j], ah, __float_as_uint(w[j].z), __float_as_uint(w[j].w));
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) mma_tf32(acc[j], ah, __float_as_uint(w[j].x), __float_as_uint(w[j].y));
}
template <int ACT>
__device__ __forceinline__ float act_f32(float z, float alpha) {
  if (ACT == BNN_ACT_RELU) return z < 0.f ? 0.f : z;
  if (ACT == BNN_ACT_LEAKY) return z < 0.f ? alpha * z : z;
  if (ACT == BNN_ACT_SWISH) return __fdividef(z, 1.0f + __expf(-z));
  return 1.0f - __fdividef(2.0f, __expf(2.0f * z) + 1.0f);
}

// packed weight sets (doubles) -> (tf32 hi, tf32 lo) float pairs, in place (the scratch copy bnn_predict packs per call):
// once per call instead of once per CTA and tile round; biases keep the full FP32 value in .x
__global__ void k_split_w_tf32(double* wp, long long n_pairs) {
  // one thread per PAIR of consecutive packed entries (columns 2t', 2t'+1 of a row, or two biases): the pair becomes
  // (hi0, hi1, lo0, lo1), so that the B operands of an MMA (b0, b1) sit in adjacent registers after one 16-byte load
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  const int e = (int)((2 * i) % PBF);
  const double2 d = reinterpret_cast<const double2*>(wp)[i];
  const float v0 = (float)d.x, v1 = (float)d.y;
  uint32_t h0, l0, h1, l1;
  split_tf32(v0, h0, l0);
  split_tf32(v1, h1, l1);
  const bool is_bias = (e >= B1_OFF && e < W2_OFF) || (e >= B2_OFF && e < W3_OFF) || e >= B3_OFF;
  // biases keep the full FP32 values in (.x, .y)
  reinterpret_cast<float4*>(wp)[i] = is_bias ? make_float4(v0, v1, 0.f, 0.f)
                                             : make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
}

template <int ACT, int PASSES>
__global__ void __launch_bounds__(LP_WARPS * 32, 1) k_pred_tf32x3(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* wbuf = reinterpret_cast<double*>(smem_raw);          // [2][PBF] (hi, lo) float pairs, 8 bytes per weight
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gq = lane >> 2, t = lane & 3;
  const int K = p.g.K;
  const long long total_warps = (long long)gridDim.x * LP_WARPS;
  const long long n_rounds = (p.n_tiles16 + total_warps - 1) / total_warps;

  auto stage_async = [&](int buf, int c) {                      // raw packed set c -> buffer (16-byte cp.async)
    const double* src = p.wp + (long long)c * PBF;
    double* dst = wbuf + (size_t)buf * PBF;
    for (int i = threadIdx.x * 2; i < PBF; i += blockDim.x * 2) {
      const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + i);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + i) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  for (long long it = 0; it < n_rounds; ++it) {
    const long long wt = (it * gridDim.x + blockIdx.x) * LP_WARPS + warp;
    const bool have_tile = wt < p.n_tiles16;
    // X fragments of this warp's tile, hi / lo, for the whole sample loop
    uint32_t xh[KP0 / 8][4], xl[KP0 / 8][4];
    if (have_tile) {
      const double* xr0 = p.x + (wt * 16 + gq) * (long long)KP0;
      const double* xr1 = xr0 + 8 * KP0;
      const int sw = (gq & 1) * 8;
#pragma unroll
      for (int kg = 0; kg < KP0 / 8; ++kg) {
        const int col = (8 * kg + 2 * t) ^ sw;
        const double2 lo2 = __ldg(reinterpret_cast<const double2*>(xr0 + col));
        const double2 hi2 = __ldg(reinterpret_cast<const double2*>(xr1 + col));
        split_tf32((float)lo2.x, xh[kg][0], xl[kg][0]);          // a0 = A[g][2t]
        split_tf32((float)hi2.x, xh[kg][1], xl[kg][1]);          // a1 = A[g+8][2t]
        split_tf32((float)lo2.y, xh[kg][2], xl[kg][2]);          // a2 = A[g][2t+1]
        split_tf32((float)hi2.y, xh[kg][3], xl[kg][3]);          // a3 = A[g+8][2t+1]
      }
    }
    double pacc[2][N3 / 4];
    int pvote[2][N3 / 4];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int i = 0; i < N3 / 4; ++i) { pacc[h][i] = 0.0; pvote[h][i] = 0; }

    // Every CTA walks the samples in the same cyclic order but starts at its own offset: 148 CTAs reading the SAME 54 KB
    // at the same time queue up on the few L2 slices that hold it (measured: 5.9 us per sample and round whatever the
    // number of MMAs); rotated, the reads spread over the whole L2.  A tile is summed by one warp in a fixed order either way.
    const int c_off = (int)(((long long)blockIdx.x * p.C) / gridDim.x);
    auto set_of = [&](int i) { const int s = i + c_off; return s >= p.C ? s - p.C : s; };
    __syncthreads();                                            // the previous round is done with both buffers
    stage_async(0, set_of(0));
    for (int ci = 0; ci < p.C; ++ci) {
      const int c = set_of(ci);
      const int buf = ci & 1;
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();                                          // set c has landed; nobody reads buffer buf ^ 1 any more
      if (ci + 1 < p.C) stage_async(buf ^ 1, set_of(ci + 1));
      if (have_tile) {
        const float2* W = reinterpret_cast<const float2*>(wbuf + (size_t)buf * PBF);
        const float a1 = (ACT == BNN_ACT_LEAKY && p.alpha) ? (float)p.alpha[c * 3 + 0] : 0.f;
        const float a2 = (ACT == BNN_ACT_LEAKY && p.alpha) ? (float)p.alpha[c * 3 + 1] : 0.f;
        // ---- layer 1
        float acc1[N1 / 8][4];
#pragma unroll
        for (int j = 0; j < N1 / 8; ++j) {
          const float b0 = W[B1_OFF + 8 * j + 2 * t].x, b1 = W[B1_OFF + 8 * j + 2 * t].y;
          acc1[j][0] = b0; acc1[j][1] = b1; acc1[j][2] = b0; acc1[j][3] = b1;
        }
        {
          const float2* wr = W + W1_OFF + gq * KP0;
          const int sw = (gq & 1) * 8;
#pragma unroll
          for (int kg = 0; kg < KP0 / 8; ++kg) {
            const int col = (8 * kg + 2 * t) ^ sw;
            mma_kgroup<PASSES, N1 / 8>(acc1, xh[kg], xl[kg], wr + col, 8 * KP0);
          }
        }
        // ---- layer 2 (A = activated acc1, split into hi / lo)
        float acc2[N2 / 8][4];
#pragma unroll
        for (int j = 0; j < N2 / 8; ++j) {
          const float b0 = W[B2_OFF + 8 * j + 2 * t].x, b1 = W[B2_OFF + 8 * j + 2 * t].y;
          acc2[j][0] = b0; acc2[j][1] = b1; acc2[j][2] = b0; acc2[j][3] = b1;
        }
        {
          const float2* wr = W + W2_OFF + gq * N1;
          const int sw = (gq & 1) * 8;
#pragma unroll
          for (int kg = 0; kg < N1 / 8; ++kg) {
            uint32_t ah[4], al[4];
            split_tf32(act_f32<ACT>(acc1[kg][0], a1), ah[0], al[0]);
            split_tf32(act_f32<ACT>(acc1[kg][2], a1), ah[1], al[1]);
            split_tf32(act_f32<ACT>(acc1[kg][1], a1), ah[2], al[2]);
            split_tf32(act_f32<ACT>(acc1[kg][3], a1), ah[3], al[3]);
            const int col = (8 * kg + 2 * t) ^ sw;
            mma_kgroup<PASSES, N2 / 8>(acc2, ah, al, wr + col, 8 * N1);
          }
        }
        // ---- layer 3
        float acc3[N3 / 8][4];
#pragma unroll
        for (int j = 0; j < N3 / 8; ++j) {
          const float b0 = W[B3_OFF + 8 * j + 2 * t].x, b1 = W[B3_OFF + 8 * j + 2 * t].y;
          acc3[j][0] = b0; acc3[j][1] = b1; acc3[j][2] = b0; acc3[j][3] = b1;
        }
        {
          const float2* wr = W + W3_OFF + gq * N2;
          const int sw = (gq & 1) * 8;
#pragma unroll
          for (int kg = 0; kg < N2 / 8; ++kg) {
            uint32_t ah[4], al[4];
            split_tf32(act_f32<ACT>(acc2[kg][0], a2), ah[0], al[0]);
            split_tf32(act_f32<ACT>(acc2[kg][2], a2), ah[1], al[1]);
            split_tf32(act_f32<ACT>(acc2[kg][1], a2), ah[2], al[2]);
            split_tf32(act_f32<ACT>(acc2[kg][3], a2), ah[3], al[3]);
            const int col = (8 * kg + 2 * t) ^ sw;
            mma_kgroup<PASSES, N3 / 8>(acc3, ah, al, wr + col, 8 * N2);
          }
        }
        // ---- softmax per row (rows gq and gq + 8; the 4 lanes of a quad hold the 16 columns), FP32
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float m = -INFINITY;
          int arg = 0x7fffffff;
#pragma unroll
          for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int col = 8 * j + 2 * t + e;
              const float v = acc3[j][2 * h + e];
              const bool take = col < K && v > m;
              m = take ? v : m;
              arg = take ? col : arg;
            }
#pragma unroll
          for (int o = 1; o <= 2; o <<= 1) {
            const float om = __shfl_xor_sync(0xffffffffu, m, o);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
            const bool take = om > m || (om == m && oa < arg);
            m = take ? om : m;
            arg = take ? oa : arg;
          }
          float ex[N3 / 4], S = 0.f;
#pragma unroll
          for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int col = 8 * j + 2 * t + e;
              ex[2 * j + e] = col < K ? __expf(acc3[j][2 * h + e] - m) : 0.f;
              S += ex[2 * j + e];
            }
          S += __shfl_xor_sync(0xffffffffu, S, 1);
          S += __shfl_xor_sync(0xffffffffu, S, 2);
          const float inv = 1.0f / S;
#pragma unroll
          for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int col = 8 * j + 2 * t + e;
              pacc[h][2 * j + e] += (double)(ex[2 * j + e] * inv);
              if (col == arg) pvote[h][2 * j + e] += 1;
            }
        }
      }
    }
    if (have_tile) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const long long row = wt * 16 + gq + 8 * h;
#pragma unroll
        for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int col = 8 * j + 2 * t + e;
            if (row < p.n_total && col < K) {
              if (p.mean_out) p.mean_out[row * K + col] = pacc[h][2 * j + e] / p.inv_sets;
              if (p.votes_out) p.votes_out[row * K + col] = (double)pvote[h][2 * j + e] / p.inv_sets;
            }
          }
      }
    }
  }
}

template <int ACT, int PASSES>
cudaError_t launch_lp(const FwdParams& p, int n_sms, cudaStream_t st) {
  auto kern = k_pred_tf32x3<ACT, PASSES>;
  const size_t bytes = 2 * (size_t)PBF * sizeof(double);
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, (int)bytes)) return e;
  {
    const long long n_pairs = (long long)p.C * PBF / 2;
    k_split_w_tf32<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(const_cast<double*>(p.wp), n_pairs);
  }
  const long long ctas = (p.n_tiles16 + LP_WARPS - 1) / LP_WARPS;
  const int grid = (int)(ctas < n_sms ? ctas : n_sms);          // one CTA per SM (231 registers x 256 threads)
  kern<<<grid, LP_WARPS * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

}  // namespace

// true when the reduced-precision prediction kernel covers this problem: the 64-64-32-16 padded family, categorical
// likelihood, summaries only (no dense tensor, no resampling)
bool bnn_pred_tf32_fits(const FwdParams& p) {
  return bnn_fwd3_family(p.g) == 1 && p.g.lik == BNN_LIK_CATEGORICAL && p.g.PB == PBF && !p.dense_out && !p.samp_u &&
         !p.samp_philox && !p.samp_counts && !p.samp_dense && (p.mean_out || p.votes_out);
}

cudaError_t bnn_launch_pred_tf32(const FwdParams& p, int n_sms, int passes, cudaStream_t st, const char** which) {
  static const char* const names[2][4] = {{"k_pred_tf32x3<relu>", "k_pred_tf32x3<leaky>", "k_pred_tf32x3<swish>", "k_pred_tf32x3<tanh>"},
                                          {"k_pred_tf32x1<relu>", "k_pred_tf32x1<leaky>", "k_pred_tf32x1<swish>", "k_pred_tf32x1<tanh>"}};
  if (which) *which = names[passes == 1][p.g.act];
  return bnn_with_act(p.g.act, [&](auto a) {
    constexpr int ACT = decltype(a)::value;
    return passes == 1 ? launch_lp<ACT, 1>(p, n_sms, st) : launch_lp<ACT, 3>(p, n_sms, st);
  });
}
