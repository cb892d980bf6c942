// Opt-in reduced-precision posterior prediction (option "predict_tf32", north star: "opt-in TF32 ... tensor-core tiles",
// stated tolerance): the forward pass of get_posterior_cat_prob / get_pdp (BNN_lib.py:245-256, 376-392), summaries and
// resampling, with the contractions on the TF32 tensor cores (mma.sync m16n8k8, FP32 accumulators) in the
// error-compensated 3xTF32 form
//     a b ~= a_hi b_hi + a_hi b_lo + a_lo b_hi,     x_hi = tf32(x), x_lo = tf32(x - x_hi)
// (products exact to 2^-22 relative), activations and softmax in FP32, and the per-row class probabilities summed
// over the posterior samples in FP64.  Class probabilities agree with the FP64 kernel to ~1e-6 absolute
// (tests/test_gpu_api.py::test_predict_tf32_mode); the Metropolis-Hastings path NEVER uses this kernel: an accept
// decision compares log-posteriors whose difference is O(1) on a value of O(1e6).
//
// k_pred_tf32x3 below serves the 64 -> 64 -> 32 -> 16 padded categorical family, k_pred_tf32_generic (further down)
// every other dense network.
//
// Layout and fragment mapping are the FP64 kernel's (bnn_common.cuh: K index permuted inside each group of 8 columns, so
// that the accumulator fragment of one layer IS the A fragment of the next).  A warp owns a 16-row tile whose X
// fragments (hi / lo) stay in registers for all samples; the packed weight sets are converted once per call, in place, to
// (hi, lo) float pairs -- 8 bytes per weight, like the double they replace -- and streamed through two shared-memory
// buffers by cp.async.
#include "bnn_common.cuh"
#include "bnn_generic_body.cuh"
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
// once per call instead of once per CTA and tile round; biases keep the full FP32 value in .x.  The layer offsets come
// from the geometry, so one converter serves the family-A kernel and the generic one (every w_off / b_off / PB is a
// multiple of 8, so a pair never straddles a matrix, a bias vector or a weight set).
__global__ void k_split_w_tf32(double* wp, long long n_pairs, const __grid_constant__ NetGeom g) {
  // one thread per PAIR of consecutive packed entries (columns 2t', 2t'+1 of a row, or two biases): the pair becomes
  // (hi0, hi1, lo0, lo1), so that the B operands of an MMA (b0, b1) sit in adjacent registers after one 16-byte load
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pairs) return;
  const int e = (int)((2 * i) % g.PB);
  const double2 d = reinterpret_cast<const double2*>(wp)[i];
  const float v0 = (float)d.x, v1 = (float)d.y;
  uint32_t h0, l0, h1, l1;
  split_tf32(v0, h0, l0);
  split_tf32(v1, h1, l1);
  bool is_bias = false;
  for (int l = 0; l < g.L; ++l) is_bias |= (e >= g.l[l].b_off && e < g.l[l].b_off + g.l[l].out_pad);
  // biases keep the full FP32 values in (.x, .y)
  reinterpret_cast<float4*>(wp)[i] = is_bias ? make_float4(v0, v1, 0.f, 0.f)
                                             : make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
}

cudaError_t launch_split_w(const FwdParams& p, cudaStream_t st) {
  const long long n_pairs = (long long)p.C * p.g.PB / 2;
  k_split_w_tf32<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(const_cast<double*>(p.wp), n_pairs, p.g);
  return cudaGetLastError();
}

// SAMP: posterior-predictive resampling (samp_u / samp_philox) instead of the mean / argmax summaries
template <int ACT, int PASSES, bool SAMP>
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
          if (SAMP) {
            // sample_from_categorical: the first class whose running sum reaches u, class 0 when none does.  The columns
            // of a row are spread over the 4 lanes of a quad (8j + 2t + e): each lane forms the running sums of its own
            // columns on top of the quad-exclusive prefix of the 8-column block and the totals of the blocks before it.
            const long long row = wt * 16 + gq + 8 * h;
            const bool live = row < p.n_total;
            const double u = !live ? 2.0
                             : p.samp_u ? p.samp_u[row * p.C + c]
                                        : bnn_samp_uniform(p.samp_seed, p.samp_row0 + row, p.samp_set0 + c);
            double base = 0.0;
            int drawn = 0x7fffffff;
#pragma unroll
            for (int j = 0; j < N3 / 8; ++j) {
              const int c0 = 8 * j + 2 * t;
              const double p0 = (double)(ex[2 * j] * inv), p1 = (double)(ex[2 * j + 1] * inv);   // 0 beyond K
              double incl = p0 + p1;
              const double up1 = __shfl_up_sync(0xffffffffu, incl, 1, 4);
              if (t >= 1) incl += up1;
              const double up2 = __shfl_up_sync(0xffffffffu, incl, 2, 4);
              if (t >= 2) incl += up2;
              const double cum0 = base + incl - (p0 + p1) + p0, cum1 = cum0 + p1;
              if (c0 + 1 < K && cum1 - u >= 0.0 && c0 + 1 < drawn) drawn = c0 + 1;
              if (c0 < K && cum0 - u >= 0.0 && c0 < drawn) drawn = c0;
              base += __shfl_sync(0xffffffffu, incl, 3, 4);
            }
            drawn = min(drawn, __shfl_xor_sync(0xffffffffu, drawn, 1));
            drawn = min(drawn, __shfl_xor_sync(0xffffffffu, drawn, 2));
            if (drawn == 0x7fffffff) drawn = 0;
            if (live) {
#pragma unroll
              for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
                for (int e = 0; e < 2; ++e)
                  if (8 * j + 2 * t + e == drawn) pvote[h][2 * j + e] += 1;
              if (t == 0 && p.samp_dense) p.samp_dense[row * p.C + c] = (double)drawn;
            }
            if (p.samp_counts) {
              // one atomic per distinct class among the rows of this half tile (lanes t == 0 speak for their row)
              const unsigned grp = __match_any_sync(0xffffffffu, (live && t == 0) ? drawn : 64 + lane);
              if (live && t == 0 && lane == __ffs(grp) - 1) atomicAdd(&p.samp_counts[c * K + drawn], __popc(grp));
            }
          } else {
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

template <int ACT, int PASSES, bool SAMP>
cudaError_t launch_lp(const FwdParams& p, int n_sms, cudaStream_t st) {
  auto kern = k_pred_tf32x3<ACT, PASSES, SAMP>;
  const size_t bytes = 2 * (size_t)PBF * sizeof(double);
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, (int)bytes)) return e;
  if (cudaError_t e = launch_split_w(p, st)) return e;
  const long long ctas = (p.n_tiles16 + LP_WARPS - 1) / LP_WARPS;
  const int grid = (int)(ctas < n_sms ? ctas : n_sms);          // one CTA per SM (231 registers x 256 threads)
  kern<<<grid, LP_WARPS * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

// ============================================================================================================
// Generic networks: every dense network bnn_set_net accepts (1-8 layers, any padded widths, up to 32 outputs, every
// likelihood).  The layer chain of k_fwd_generic (bnn_generic_body.cuh) in reduced precision: a warp owns a 16-row
// tile and runs every weight set over it in set order; each layer is computed in blocks of up to 4 n-tiles (32
// columns) with the 3xTF32 (or plain TF32) k-groups of mma_kgroup; hidden activations are evaluated in FP32 and
// staged as floats in per-warp shared memory -- half the bytes of the FP64 kernel's staging, so every network that
// fits k_fwd_generic fits here -- and split into (hi, lo) when they are read as the next layer's A fragments.
// Layer 1 reads X (FP64, swizzled rows) through L1.  The per-row epilogue runs in FP32 and adds to FP64 sums.
// ============================================================================================================
constexpr int LPG_WARPS = 4;          // at most 128 registers: four CTAs (16 warps) per SM

// staging row stride (floats): max_w brought to 8 mod 32, so that the 8-byte fragment loads / stores of a half warp
// (rows gq = 0..3 x columns 2t) fall on 16 distinct bank pairs
__host__ __device__ inline int lpg_stride(const NetGeom& g) { return g.max_w + (40 - g.max_w % 32) % 32; }
__host__ __device__ inline int lpg_pred_width(const NetGeom& g) { return g.lik == BNN_LIK_CATEGORICAL ? g.K : g.O; }
// per warp: FP64 sums [16][PW], vote ints [16][PW], two hidden-layer buffers [16][HS] and the output rows [16][ZS]
__host__ __device__ inline size_t lpg_warp_bytes(const NetGeom& g) {
  const int ZS = g.l[g.L - 1].out_pad + 1;
  return 16 * (size_t)lpg_pred_width(g) * (sizeof(double) + sizeof(int)) + (32 * (size_t)lpg_stride(g) + 16 * ZS) * sizeof(float);
}

// One block of NT output tiles of one layer over the warp's 16 rows: accumulators start at the bias, k-groups in
// ascending order, then the FP32 activation and the staging store (hidden layer) or the plain store (output layer).
//   X0: A is layer 1's input, read from X (rows xr0 / xr1 offset by 2t; FP64, swizzled like the layer's W rows);
//   otherwise A is the staged previous layer (rows a0 / a1 offset by 2t, not swizzled)
template <int ACT, int PASSES, int NT, bool X0>
__device__ __forceinline__ void lpg_block(const double* xr0, const double* xr1, const float* a0, const float* a1, int sw,
                                          int nkg, const float2* wrow, int stride, const float2* bias, bool last,
                                          float alpha, float* d0, float* d1) {
  float acc[NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const float2 b = bias[8 * j];
    acc[j][0] = b.x; acc[j][1] = b.y; acc[j][2] = b.x; acc[j][3] = b.y;
  }
  // (unrolled twice: deeper unrolling needs more than the 128 registers of four CTAs per SM and spills)
#pragma unroll 2
  for (int kg = 0; kg < nkg; ++kg) {
    const int off = (kg ^ sw) << 3;
    float2 r0, r1;                                              // rows gq / gq + 8, columns 2t / 2t + 1 of the k-group
    if (X0) {
      const double2 v0 = __ldg(reinterpret_cast<const double2*>(xr0 + off));
      const double2 v1 = __ldg(reinterpret_cast<const double2*>(xr1 + off));
      r0 = make_float2((float)v0.x, (float)v0.y);
      r1 = make_float2((float)v1.x, (float)v1.y);
    } else {
      r0 = *reinterpret_cast<const float2*>(a0 + 8 * kg);
      r1 = *reinterpret_cast<const float2*>(a1 + 8 * kg);
    }
    uint32_t ah[4], al[4];
    split_tf32(r0.x, ah[0], al[0]);                             // a0 = A[g][2t]
    split_tf32(r1.x, ah[1], al[1]);                             // a1 = A[g+8][2t]
    split_tf32(r0.y, ah[2], al[2]);                             // a2 = A[g][2t+1]
    split_tf32(r1.y, ah[3], al[3]);                             // a3 = A[g+8][2t+1]
    mma_kgroup<PASSES, NT>(acc, ah, al, wrow + off, 8 * stride);
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    if (!last) {
      *reinterpret_cast<float2*>(d0 + 8 * j) = make_float2(act_f32<ACT>(acc[j][0], alpha), act_f32<ACT>(acc[j][1], alpha));
      *reinterpret_cast<float2*>(d1 + 8 * j) = make_float2(act_f32<ACT>(acc[j][2], alpha), act_f32<ACT>(acc[j][3], alpha));
    } else {
      d0[8 * j] = acc[j][0]; d0[8 * j + 1] = acc[j][1];
      d1[8 * j] = acc[j][2]; d1[8 * j + 1] = acc[j][3];
    }
  }
}

// All layers of one weight set over one warp tile; leaves the output layer's pre-transform values in zs [16][ZS].
template <int ACT, int PASSES>
__device__ __forceinline__ void lpg_layers(const NetGeom& g, const double* xr0, const double* xr1, const float2* W,
                                           const double* alpha_c, float* h0, float* h1, int HS, float* zs, int ZS,
                                           int lane) {
  const int gq = lane >> 2, t = lane & 3;
  const float* src = h1;
  float* dst = h0;
#pragma unroll 1
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom& lg = g.l[l];
    const bool last = (l == g.L - 1);
    const float alpha = alpha_c ? (float)alpha_c[l] : 0.f;
    const int sw = (gq & 1) & (lg.swz >> 3);
    const int nkg = lg.in_pad >> 3, stride = lg.stride, out_pad = lg.out_pad;
    const float* a0 = src + gq * HS + 2 * t;
    const float* a1 = a0 + 8 * HS;
    float* d0 = last ? zs + gq * ZS + 2 * t : dst + gq * HS + 2 * t;
    float* d1 = last ? d0 + 8 * ZS : d0 + 8 * HS;
#pragma unroll 1
    for (int n0 = 0; n0 < out_pad; n0 += 32) {
      const float2* wrow = W + lg.w_off + (long long)(n0 + gq) * stride + 2 * t;
      const float2* bias = W + lg.b_off + n0 + 2 * t;
#define LPG_BLOCK(NT)                                                                                                   \
  do {                                                                                                                  \
    if (l == 0)                                                                                                         \
      lpg_block<ACT, PASSES, NT, true>(xr0, xr1, a0, a1, sw, nkg, wrow, stride, bias, last, alpha, d0 + n0, d1 + n0);   \
    else                                                                                                                \
      lpg_block<ACT, PASSES, NT, false>(xr0, xr1, a0, a1, sw, nkg, wrow, stride, bias, last, alpha, d0 + n0, d1 + n0);  \
  } while (0)
      switch (min(4, (out_pad - n0) >> 3)) {
        case 1: LPG_BLOCK(1); break;
        case 2: LPG_BLOCK(2); break;
        case 3: LPG_BLOCK(3); break;
        default: LPG_BLOCK(4); break;
      }
#undef LPG_BLOCK
    }
    __syncwarp();
    src = dst;
    dst = (dst == h0) ? h1 : h0;
  }
}

// Prediction epilogue of one (warp tile, weight set) in FP32 on the staged outputs, lane r < 16 owning row r; the same
// rules as bnn_epilogue's prediction branch (bnn_generic_body.cuh): first maximum wins the vote, the draw is the first
// class whose running sum reaches u (class 0 when none does), the sigma head's second half goes through softplus.
__device__ __forceinline__ void lpg_epilogue(const FwdParams& p, int c, long long wt, int lane, float* zs, int ZS,
                                             double* pacc, int* pvote) {
  const NetGeom& g = p.g;
  const long long row = wt * 16 + (lane & 15);
  const bool active = lane < 16 && row < p.n_total;
  float* z = zs + (lane & 15) * ZS;
  const bool sampling = p.samp_u || p.samp_philox;
  if (g.lik == BNN_LIK_CATEGORICAL) {
    const int K = g.K;
    int arg = 0;
    if (active) {
      float m = z[0];
      for (int k = 1; k < K; ++k)
        if (z[k] > m) { m = z[k]; arg = k; }
      float S = 0.f;
      for (int k = 0; k < K; ++k) { const float e = __expf(z[k] - m); z[k] = e; S += e; }   // the row is this lane's scratch
      const float inv = __fdividef(1.0f, S);
      double* pa = pacc + lane * K;
      const double u = p.samp_u ? p.samp_u[row * p.C + c]
                                : (p.samp_philox ? bnn_samp_uniform(p.samp_seed, p.samp_row0 + row, p.samp_set0 + c) : 0.0);
      double cum = 0.0;
      int drawn = -1;
      for (int k = 0; k < K; ++k) {
        const double pk = (double)(z[k] * inv);
        if (p.mean_out) pa[k] += pk;
        cum += pk;
        if (drawn < 0 && cum - u >= 0.0) drawn = k;
      }
      if (sampling) {
        arg = drawn < 0 ? 0 : drawn;
        if (p.samp_dense) p.samp_dense[row * p.C + c] = (double)arg;
      }
      pvote[lane * K + arg] += 1;
    }
    if (sampling && p.samp_counts) {
      // one atomic per distinct class among the 16 rows of the warp tile
      const unsigned grp = __match_any_sync(FULL_MASK, active ? arg : 64 + lane);
      if (active && lane == __ffs(grp) - 1) atomicAdd(&p.samp_counts[c * K + arg], __popc(grp));
    }
    return;
  }
  if (active) {
    const bool head = (g.lik == BNN_LIK_GAUSSIAN_HEAD);
    const int O = g.O, K = g.K;
    double* pa = pacc + lane * O;
    for (int j = 0; j < O; ++j) {
      float v = z[j];
      if (head && j >= K) v = fmaxf(v, 0.f) + log1pf(__expf(-fabsf(v)));       // softplus (np.logaddexp(0, z))
      pa[j] += (double)v;
    }
  }
}

// The warp count is blockDim.x / 32 (lpg_warps): every (tile, set) is computed by one warp with the same instruction
// sequence, and a tile's sets are summed in set order, so results do not depend on the launch geometry.
template <int ACT, int PASSES>
__global__ void __launch_bounds__(LPG_WARPS * 32, 4) k_pred_tf32_generic(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // the summaries are scaled by the reciprocal of the set count, formed once here: a division per stored value would
  // bring the FP64 division's out-of-line slow path into the tile loop, and the registers live across it to the stack
  const double rcp_sets = 1.0 / p.inv_sets;
  const NetGeom& g = p.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  const int gq = lane >> 2, t = lane & 3;
  const int PW = lpg_pred_width(g), HS = lpg_stride(g), ZS = g.l[g.L - 1].out_pad + 1;
  double* pacc = reinterpret_cast<double*>(smem_raw) + warp * 16 * PW;
  int* pvote = reinterpret_cast<int*>(reinterpret_cast<double*>(smem_raw) + n_warps * 16 * PW) + warp * 16 * PW;
  float* h0 = reinterpret_cast<float*>(smem_raw + (size_t)n_warps * 16 * PW * (sizeof(double) + sizeof(int))) +
              warp * (32 * HS + 16 * ZS);
  float* h1 = h0 + 16 * HS;
  float* zs = h1 + 16 * HS;
  const long long total_warps = (long long)gridDim.x * n_warps;
  for (long long wt = (long long)blockIdx.x * n_warps + warp; wt < p.n_tiles16; wt += total_warps) {
    for (int i = lane; i < 16 * PW; i += 32) { pacc[i] = 0.0; pvote[i] = 0; }
    __syncwarp();
    const double* xr0 = p.x + (wt * 16 + gq) * (long long)g.F_pad + 2 * t;
    const double* xr1 = xr0 + 8LL * g.F_pad;
    for (int c = 0; c < p.C; ++c) {
      lpg_layers<ACT, PASSES>(g, xr0, xr1, reinterpret_cast<const float2*>(p.wp + (long long)c * g.PB),
                              (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha + (long long)c * g.L : nullptr, h0, h1, HS, zs,
                              ZS, lane);
      lpg_epilogue(p, c, wt, lane, zs, ZS, pacc, pvote);
      __syncwarp();
    }
    for (int i = lane; i < 16 * PW; i += 32) {
      const long long row = wt * 16 + i / PW;
      if (row < p.n_total) {
        if (p.mean_out) p.mean_out[row * PW + (i % PW)] = pacc[i] * rcp_sets;
        if (p.votes_out) p.votes_out[row * PW + (i % PW)] = (double)pvote[i] * rcp_sets;
      }
    }
  }
}

// most warps per CTA (4, 2, 1) whose shared memory fits; 0 when none does
int lpg_warps(const NetGeom& g) {
  for (int w = LPG_WARPS; w >= 1; w >>= 1)
    if (w * lpg_warp_bytes(g) <= (size_t)BNN_MAX_DYN_SMEM) return w;
  return 0;
}

template <int ACT, int PASSES>
cudaError_t launch_lpg(const FwdParams& p, int n_sms, cudaStream_t st) {
  auto kern = k_pred_tf32_generic<ACT, PASSES>;
  const int warps = lpg_warps(p.g);
  if (!warps) return cudaErrorInvalidConfiguration;         // (cannot happen: k_fwd_generic's staging is larger)
  const size_t bytes = warps * lpg_warp_bytes(p.g);
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, BNN_MAX_DYN_SMEM)) return e;
  if (cudaError_t e = launch_split_w(p, st)) return e;
  int per_sm = 0;
  if (cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, bytes)) return e;
  const long long ctas = (p.n_tiles16 + warps - 1) / warps, max_grid = (long long)n_sms * (per_sm > 0 ? per_sm : 1);
  kern<<<(unsigned)(ctas < max_grid ? ctas : max_grid), warps * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

}  // namespace

// A prediction call the reduced-precision kernels take: summaries or resampling of any dense network.  The dense
// [S, N, K] tensor (RunPredict, mcmc._y, get_posterior_est) stays on the FP64 kernels, and so does the one class of
// shapes where 3xTF32 measured slower than the FP64 kernel it replaces (DESIGN.md section 4,
// profiles/r03_predict_tf32_generic.json): Gaussian and count outputs padded to k_fwd3's 32-32-16 width family, where
// config 2 took 0.117 s against 0.113 s at 1M rows x 1,024 samples (plain TF32 was faster there and is not excluded).
bool bnn_pred_tf32_fits(const FwdParams& p, int passes) {
  if (p.sp.prog || p.dense_out || !(p.mean_out || p.votes_out)) return false;
  const bool identity_out = p.g.lik == BNN_LIK_GAUSSIAN || bnn_lik_is_count(p.g.lik);
  return !(passes == 3 && identity_out && bnn_fwd3_family(p.g) == 2);
}

cudaError_t bnn_launch_pred_tf32(const FwdParams& p, int n_sms, int passes, cudaStream_t st, const char** which) {
  static const char* const names[2][2][4] = {
      {{"k_pred_tf32x3<relu>", "k_pred_tf32x3<leaky>", "k_pred_tf32x3<swish>", "k_pred_tf32x3<tanh>"},
       {"k_pred_tf32x1<relu>", "k_pred_tf32x1<leaky>", "k_pred_tf32x1<swish>", "k_pred_tf32x1<tanh>"}},
      {{"k_pred_tf32x3_generic<relu>", "k_pred_tf32x3_generic<leaky>", "k_pred_tf32x3_generic<swish>", "k_pred_tf32x3_generic<tanh>"},
       {"k_pred_tf32x1_generic<relu>", "k_pred_tf32x1_generic<leaky>", "k_pred_tf32x1_generic<swish>", "k_pred_tf32x1_generic<tanh>"}}};
  // the 64-64-32-16 categorical family keeps its activations in registers (k_pred_tf32x3); every other network runs
  // the generic kernel
  const bool fam_a = bnn_fwd3_family(p.g) == 1 && p.g.lik == BNN_LIK_CATEGORICAL && p.g.PB == PBF;
  const bool samp = p.samp_u || p.samp_philox;
  if (which) *which = names[!fam_a][passes == 1][p.g.act];
  return bnn_with_act(p.g.act, [&](auto a) {
    constexpr int ACT = decltype(a)::value;
    if (!fam_a) return passes == 1 ? launch_lpg<ACT, 1>(p, n_sms, st) : launch_lpg<ACT, 3>(p, n_sms, st);
    if (samp) return passes == 1 ? launch_lp<ACT, 1, true>(p, n_sms, st) : launch_lp<ACT, 3, true>(p, n_sms, st);
    return passes == 1 ? launch_lp<ACT, 1, false>(p, n_sms, st) : launch_lp<ACT, 3, false>(p, n_sms, st);
  });
}
