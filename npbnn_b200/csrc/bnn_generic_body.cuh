// Per-(warp tile, weight set) body of the generic forward kernel: layer chain on FP64 tensor-core MMAs with the hidden
// activations staged in per-warp shared memory, and the likelihood / prediction epilogue on the staged outputs.
// Shared by k_fwd_generic (bnn_forward.cu) and the persistent small-data chain loop (k_chain_loop, bnn_chainloop.cu).
#pragma once
#include "bnn_common.cuh"

#define FULL_MASK 0xffffffffu

// The generic path evaluates its exponentials with the 256-entry table (+ fourth-order term: one more FMA, same 3e-16
// accuracy): 2 KB of shared memory instead of 16 KB, which is what lets k_chain_loop keep the config-1 feature matrix
// resident next to it.  k_fwd_generic uses the same table so that both run the identical arithmetic.
constexpr int GEN_TB = 8;
constexpr int GEN_TAB_SIZE = 1 << GEN_TB;

#ifndef BNN_HAVE_LOGSQRT2PI
#define BNN_HAVE_LOGSQRT2PI
static constexpr double kLogSqrt2Pi = 0.91893853320467274178;
#endif

__device__ __forceinline__ double warp16_sum(double v) {
  // lanes 0..15 hold values; fixed xor tree => deterministic
  v += __shfl_xor_sync(FULL_MASK, v, 8);
  v += __shfl_xor_sync(FULL_MASK, v, 4);
  v += __shfl_xor_sync(FULL_MASK, v, 2);
  v += __shfl_xor_sync(FULL_MASK, v, 1);
  return v;
}

__device__ __forceinline__ double softplus_ref(double z) {
  // np.logaddexp(0, z) (BNN_lib.py:170-172)
  return fmax(z, 0.0) + log1p(exp(-fabs(z)));
}

// Per-warp epilogue on the staged outputs of one (warp tile, weight set).
//   zs  : [16][ZS] pre-transform outputs of the last layer (row-major, per warp)
//   lane r < 16 owns row r of the tile.
// Likelihood mode (PREDICT=false): writes part[(c*NF+slot)*n_tiles16 + wt] and bumps the CTA counters.
// Prediction mode: accumulates transformed outputs into pacc/pvote (per warp, [16][K_out]) and
// optionally writes the dense tensor.
// R32 (likelihood mode only): the warp owns 32 rows = warp tiles wt and wt + 1, lane r owns row r; the xor
// trees of warp16_sum stay inside each half-warp, so lanes 0 and 16 hold the two warp-tile sums.
template <bool PREDICT, bool R32 = false, int TB = BNN_EXP_TAB_BITS>
__device__ __forceinline__ void bnn_epilogue(const FwdParams& p, int c, long long wt, int lane, const double* zs,
                                             int ZS, const double* tab, int* cnt_smem, double* pacc, int* pvote,
                                             const int* lab16 = nullptr, const double* tgt16 = nullptr) {
  const NetGeom& g = p.g;
  const int rl = R32 ? lane : (lane & 15);
  const long long row = wt * 16 + rl;
  const bool active = (R32 || lane < 16) && row < p.n_total;
  const bool is_train = active && row < p.n_train;
  const bool is_test = active && !is_train;
  const double* z = zs + rl * ZS;
  const long long nt = p.n_tiles16;
  // lane that stores the warp-tile partial sums, and the tile it stores them for
  const bool writer = (lane == 0) || (R32 && lane == 16 && wt + 1 < nt);
  const long long wts = wt + (R32 ? (lane >> 4) : 0);

  if (g.lik == BNN_LIK_CATEGORICAL) {
    const int K = g.K;
    double m = -INFINITY;
    int arg = 0;
    double S = 0.0, ll = 0.0;
    if (active) {
      m = z[0];
      for (int k = 1; k < K; ++k) {
        double v = z[k];
        if (v > m) { m = v; arg = k; }   // first maximum wins, as np.argmax
      }
      if (!PREDICT && is_train) {
        for (int k = 0; k < K; ++k) S += bnn_exp_neg<TB>(z[k] - m, tab);
      }
    }
    if (!PREDICT) {
      int y = 0;
      if (active) {
        y = lab16 ? lab16[rl] : p.labels[row];
        bool ok = (arg == y);
        if (is_train) {
          double d = z[y] - m;
          // log(softmax) of the reference is -inf once exp(d) underflows to 0 (BNN_lib.py:121,168)
          ll = (d < -745.1332191019412) ? -INFINITY : d - log(S);
          if (p.class_w) ll *= p.class_w[y];
          if (p.inst_w) ll *= p.inst_w[row];
          int* cc = cnt_smem + c * bnn_n_counts(K);
          if (ok) atomicAdd(&cc[2 + y], 1);
          atomicAdd(&cc[2 + K + arg], 1);
          if (ok) atomicAdd(&cc[0], 1);
        } else if (ok) {
          atomicAdd(&cnt_smem[c * bnn_n_counts(K) + 1], 1);
        }
      }
      double s = warp16_sum(is_train ? ll : 0.0);
      if (writer) p.part[((long long)c * p.NF) * nt + wts] = s;
    } else {
      if (active) {
        double* zw = const_cast<double*>(z);     // the staged row is private to this lane: reuse as scratch
        for (int k = 0; k < K; ++k) { double e = bnn_exp_neg<TB>(z[k] - m, tab); zw[k] = e; S += e; }
        double inv = 1.0 / S;
        double* pa = pacc + (lane & 15) * K;
        // sample_from_categorical: first class whose running sum (np.cumsum order) reaches u; none => class 0
        const bool sampling = p.samp_u || p.samp_philox;
        const double u = p.samp_u ? p.samp_u[row * p.C + c] : (p.samp_philox ? bnn_samp_uniform(p.samp_seed, p.samp_row0 + row, p.samp_set0 + c) : 0.0);
        double cum = 0.0;
        int drawn = -1;
        for (int k = 0; k < K; ++k) {
          double pk = zw[k] * inv;
          pa[k] += pk;
          cum += pk;
          if (drawn < 0 && cum - u >= 0.0) drawn = k;
          if (p.dense_out) p.dense_out[((long long)c * p.n_total + row) * K + k] = pk;
        }
        if (sampling) {
          arg = drawn < 0 ? 0 : drawn;
          if (p.samp_dense) p.samp_dense[row * p.C + c] = (double)arg;
        }
        pvote[(lane & 15) * K + arg] += 1;
      }
      if ((p.samp_u || p.samp_philox) && p.samp_counts) {
        // one atomic per distinct class among the 16 rows of the warp tile
        const unsigned grp = __match_any_sync(FULL_MASK, active ? arg : 64 + lane);
        if (active && lane == __ffs(grp) - 1) atomicAdd(&p.samp_counts[c * K + arg], __popc(grp));
      }
    }
    return;
  }

  // Gaussian and count likelihoods: K modelled outputs, targets [n_total, K]
  const int K = g.K;
  const bool head = (g.lik == BNN_LIK_GAUSSIAN_HEAD);
  const bool count = bnn_lik_is_count(g.lik);
  if (!PREDICT) {
    double ll = 0.0;
    for (int j = 0; j < K; ++j) {
      double r = 0.0;
      if (active) {
        double t = tgt16 ? tgt16[rl * K + j] : p.targets[row * K + j];
        r = z[j] - t;
        if (count) {
          // (r is the residual of the count mean; test rows need it for the test MSE, the likelihood is train only)
          const double lr = bnn_count_loglik(g.lik, z[j], z[K + j], t, p.lgk1[row * K + j], &r);
          if (is_train) ll += lr;
        } else if (head && is_train) {
          double s = softplus_ref(z[K + j]);
          double u = (t - z[j]) / s;
          ll += -0.5 * u * u - kLogSqrt2Pi - log(s);
        }
      }
      double sr = warp16_sum(is_train ? r : 0.0);
      double sr2 = warp16_sum(is_train ? r * r : 0.0);
      double st2 = warp16_sum(is_test ? r * r : 0.0);
      if (writer) {
        p.part[((long long)c * p.NF + 1 + j) * nt + wts] = sr;
        p.part[((long long)c * p.NF + 1 + K + j) * nt + wts] = sr2;
        p.part[((long long)c * p.NF + 1 + 2 * K + j) * nt + wts] = st2;
      }
    }
    double s = warp16_sum(ll);
    if (writer) p.part[((long long)c * p.NF) * nt + wts] = s;
  } else {
    if (active) {
      const int O = g.O;
      double* pa = pacc + (lane & 15) * O;
      for (int j = 0; j < O; ++j) {
        double v = z[j];
        if (head && j >= K) v = softplus_ref(v);
        pa[j] += v;
        if (p.dense_out) p.dense_out[((long long)c * p.n_total + row) * O + j] = v;
      }
    }
  }
}

// number of output columns per row in prediction mode
__device__ __forceinline__ int bnn_pred_width(const NetGeom& g) { return g.lik == BNN_LIK_CATEGORICAL ? g.K : g.O; }

template <bool PREDICT>
__device__ __forceinline__ void bnn_pred_flush(const FwdParams& p, long long wt, int lane, double* pacc, int* pvote) {
  if (!PREDICT) return;
  const int W = bnn_pred_width(p.g);
  for (int i = lane; i < 16 * W; i += 32) {
    long long row = wt * 16 + i / W;
    if (row < p.n_total) {
      if (p.mean_out) p.mean_out[row * W + (i % W)] = pacc[i] / p.inv_sets;
      if (p.votes_out) p.votes_out[row * W + (i % W)] = (double)pvote[i] / p.inv_sets;
    }
  }
}

// 16-byte operand load: NC = read-only path (ld.global.nc; X and weight sets that no thread of the launch writes),
// otherwise a plain generic load (shared memory, or global data written earlier in the same launch)
template <bool NC>
__device__ __forceinline__ double2 gen_ld2(const double* p) {
  if (NC) return __ldg(reinterpret_cast<const double2*>(p));
  return *reinterpret_cast<const double2*>(p);
}

// One block of NT output tiles (8 columns each) of one layer over the warp's 16 rows: accumulators start at the
// bias, k-groups in ascending order (the summation order every caller shares), then activation + staging store for
// the next layer (or the plain store of the last layer's outputs).  Everything loop-invariant is in registers and
// the n-tile loop is unrolled at compile time: the k-loop is loads + DMMAs only.
//   arow0 / arow1 : A rows gq and gq + 8, already offset by 2t;  wrow : W row (n0 + gq), offset by 2t;
//   sx : 1 if this lane's rows are swizzled (k-group kg lives at column group kg ^ 1)
template <int ACT, bool ANC, bool WNC, int NT>
__device__ __forceinline__ void gen_layer_block(const double* arow0, const double* arow1, const double* wrow, int stride,
                                                int nkg, int sx, const double* bias, bool last, double alpha,
                                                double* dst0, double* dst1, int dsx, double* z0, double* z1,
                                                const double* tab) {
  // A lone warp is bound by the latency of the dependent DMMA chain (~280 clk per k-group measured), not by the pipe
  // (64 clk per m16n8k8): narrow blocks split the k-groups round-robin over NCH independent accumulator sets, summed
  // at the end in a fixed order (set 0 carries the bias).
  constexpr int NCH = (NT == 1) ? 4 : (NT == 2 ? 2 : 1);
  double accs[NCH][NT][4];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const double2 bb = *reinterpret_cast<const double2*>(bias + 8 * j);
    accs[0][j][0] = bb.x; accs[0][j][1] = bb.y; accs[0][j][2] = bb.x; accs[0][j][3] = bb.y;
#pragma unroll
    for (int q = 1; q < NCH; ++q) accs[q][j][0] = accs[q][j][1] = accs[q][j][2] = accs[q][j][3] = 0.0;
  }
  const int stride8 = 8 * stride;
  auto kgroup = [&](int kg, double (&a)[NT][4]) {
    const int off = (kg ^ sx) << 3;
    const double2 a_lo = gen_ld2<ANC>(arow0 + off);
    const double2 a_hi = gen_ld2<ANC>(arow1 + off);
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      const double2 bb = gen_ld2<WNC>(wrow + j * stride8 + off);
      dmma16x8x8(a[j], a_lo.x, a_hi.x, a_lo.y, a_hi.y, bb.x, bb.y);
    }
  };
  int kg = 0;
  for (; kg + NCH <= nkg; kg += NCH) {
#pragma unroll
    for (int q = 0; q < NCH; ++q) kgroup(kg + q, accs[q]);
  }
#pragma unroll
  for (int q = 0; q < NCH - 1; ++q)
    if (kg + q < nkg) kgroup(kg + q, accs[q]);
  double (&acc)[NT][4] = accs[0];
  if (NCH == 2) {
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] += accs[NCH - 1][j][e];
  } else if (NCH == 4) {
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = (accs[0][j][e] + accs[1][j][e]) + (accs[2][j][e] + accs[NCH - 1][j][e]);
  }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    if (!last) {
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][e] = bnn_act<ACT, GEN_TB>(acc[j][e], alpha, tab);
      const int o = ((j ^ dsx) << 3);
      *reinterpret_cast<double2*>(dst0 + o) = make_double2(acc[j][0], acc[j][1]);
      *reinterpret_cast<double2*>(dst1 + o) = make_double2(acc[j][2], acc[j][3]);
    } else {
      z0[8 * j] = acc[j][0]; z0[8 * j + 1] = acc[j][1];
      z1[8 * j] = acc[j][2]; z1[8 * j + 1] = acc[j][3];
    }
  }
}

// All layers of one weight set over one 16-row warp tile; leaves the last layer's pre-transform outputs in zs [16][ZS].
//   xrow0 / xrow1 : rows gq and gq + 8 of the tile in the swizzled-row layout (stride F_pad); W : packed weight set;
//   alpha_c : this set's activation slopes (leaky) or null; h0 / h1 : per-warp staging [16][max_w] each
template <int ACT, bool XNC, bool WNC>
__device__ __forceinline__ void fwd_generic_layers(const NetGeom& g, const double* xrow0, const double* xrow1,
                                                   const double* W, const double* alpha_c, double* h0, double* h1,
                                                   double* zs, int ZS, const double* tab, int lane) {
  const int gq = lane >> 2, t = lane & 3;
  const double* src = nullptr;
  double* dst = h0;
#pragma unroll 1
  for (int l = 0; l < g.L; ++l) {
    const LayerGeom lg = g.l[l];
    const bool last = (l == g.L - 1);
    const double alpha = alpha_c ? alpha_c[l] : 0.0;
    const int sx = (gq & 1) & (lg.swz >> 3);
    const int nkg = lg.in_pad >> 3;
    // destination geometry = next layer's A operand
    const int dstride = last ? ZS : g.l[l + 1].stride;
    const int dsx = last ? 0 : ((gq & 1) & (g.l[l + 1].swz >> 3));
    const double* arow0 = (l == 0) ? xrow0 + 2 * t : src + gq * lg.stride + 2 * t;
    const double* arow1 = (l == 0) ? xrow1 + 2 * t : src + (gq + 8) * lg.stride + 2 * t;
#pragma unroll 1
    for (int n0 = 0; n0 < lg.out_pad; n0 += 32) {
      const int ntile = min(4, (lg.out_pad - n0) >> 3);
      const double* wrow = W + lg.w_off + (long long)(n0 + gq) * lg.stride + 2 * t;
      const double* bias = W + lg.b_off + n0 + 2 * t;
      // staging stores: column n0 + 8j + 2t of rows gq / gq + 8, k-group j of the block swizzled like the consumer reads it
      double* dst0 = dst + gq * dstride + n0 + 2 * t;
      double* dst1 = dst + (gq + 8) * dstride + n0 + 2 * t;
      double* z0 = zs + gq * ZS + n0 + 2 * t;
      double* z1 = zs + (gq + 8) * ZS + n0 + 2 * t;
      // (X in shared memory loads like the staged activations: one instantiation serves every layer, which keeps the
      // executed code of k_chain_loop inside the instruction cache)
#define GEN_BLOCK(NT)                                                                                                     \
  do {                                                                                                                    \
    if (XNC && l == 0)                                                                                                    \
      gen_layer_block<ACT, true, WNC, NT>(arow0, arow1, wrow, lg.stride, nkg, sx, bias, last, alpha, dst0, dst1, dsx, z0,  \
                                          z1, tab);                                                                       \
    else                                                                                                                  \
      gen_layer_block<ACT, false, WNC, NT>(arow0, arow1, wrow, lg.stride, nkg, sx, bias, last, alpha, dst0, dst1, dsx, z0, \
                                           z1, tab);                                                                      \
  } while (0)
      switch (ntile) {
        case 1: GEN_BLOCK(1); break;
        case 2: GEN_BLOCK(2); break;
        case 3: GEN_BLOCK(3); break;
        default: GEN_BLOCK(4); break;
      }
#undef GEN_BLOCK
    }
    __syncwarp();
    src = dst;
    dst = (dst == h0) ? h1 : h0;
  }
}
