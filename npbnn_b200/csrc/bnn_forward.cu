// K1 / K3: chain-batched forward pass fused with likelihood, accuracy counters or posterior summaries.
//
// Replaces (reference file:line): RunHiddenLayer / MatrixMultiplicationD / ActFun.eval
// (BNN_lib.py:184-193, 154-162, 83-87), SoftMax / RegressTransform(Error) (BNN_lib.py:166-182),
// calc_likelihood* (BNN_lib.py:100-143), CalcAccuracy / CalcLabelAccuracy / CalcLabelFreq
// (BNN_lib.py:195-233) as called from MCMC.mh_step (BNN_env.py:449-518), and the RunPredict loops of
// get_posterior_cat_prob / get_posterior_est / get_pdp (BNN_lib.py:376-392, 731-737, BNN_pdp.py:63-73).
//
// Work decomposition: a warp owns 16 rows of X ("warp tile") and runs every weight set of the pass
// over them, so X is read from HBM exactly once per pass.  Each layer is a chain of FP64 tensor-core
// MMAs (m16n8k8, bnn_common.cuh) whose accumulators are the next layer's A operand.
//   k_fwd3        3-layer nets with compile-time padded widths: X warp tile in shared memory (bulk
//                 async copy), weight sets streamed through a 2-deep shared-memory ring by bulk async
//                 copies + mbarriers, hidden activations never leave registers.
//   k_fwd_generic any depth/width: hidden activations staged in per-warp shared memory, weights read
//                 through L1/L2.
#include <mutex>
#include <set>
#include <utility>
#include "bnn_kernels.h"
#include "bnn_generic_body.cuh"

// =============================================================================================
// generic kernel
// =============================================================================================
constexpr int GEN_WARPS = 4;

template <int ACT, bool PREDICT>
__global__ void __launch_bounds__(GEN_WARPS * 32) k_fwd_generic(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const NetGeom& g = p.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gq = lane >> 2;
  const int ZS = g.l[g.L - 1].out_pad + 1;        // the last layer may be padded beyond round_up(O, 8) (k_fwd3 width families)
  const int PW = bnn_pred_width(g);

  double* tab = reinterpret_cast<double*>(smem_raw);
  double* hbase = tab + GEN_TAB_SIZE;
  const int per_warp = 2 * 16 * g.max_w + 16 * ZS + (PREDICT ? 16 * PW : 0);
  double* h0 = hbase + warp * per_warp;
  double* h1 = h0 + 16 * g.max_w;
  double* zs = h1 + 16 * g.max_w;
  double* pacc = zs + 16 * ZS;
  int* ibase = reinterpret_cast<int*>(hbase + GEN_WARPS * per_warp);
  int* pvote = ibase + warp * (PREDICT ? 16 * PW : 0);
  int* cnt = ibase;   // likelihood mode: [C][2+2K]
  const int n_cnt = PREDICT ? 0 : bnn_smem_counts(g, p.C);

  for (int i = threadIdx.x; i < GEN_TAB_SIZE; i += blockDim.x) tab[i] = p.exp_tab_small[i];
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) cnt[i] = 0;
  __syncthreads();

  // likelihood mode: when there are fewer row tiles than the GPU has room for, the weight sets are split over
  // gridDim.y as well (every (tile, set) still has exactly one owner); prediction accumulates over sets per tile
  const int c_beg = PREDICT ? 0 : (int)((long long)p.C * blockIdx.y / gridDim.y);
  const int c_end = PREDICT ? p.C : (int)((long long)p.C * (blockIdx.y + 1) / gridDim.y);
  const long long total_warps = (long long)gridDim.x * GEN_WARPS;
  for (long long wt = (long long)blockIdx.x * GEN_WARPS + warp; wt < p.n_tiles16; wt += total_warps) {
    if (PREDICT) {
      for (int i = lane; i < 16 * PW; i += 32) { pacc[i] = 0.0; pvote[i] = 0; }
      __syncwarp();
    }
    const double* xrow0 = p.x + (wt * 16 + gq) * (long long)g.F_pad;
    const double* xrow1 = xrow0 + 8LL * g.F_pad;
    for (int c = c_beg; c < c_end; ++c) {
      fwd_generic_layers<ACT, true, true>(g, xrow0, xrow1, p.wp + (long long)c * g.PB,
                                    (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha + (long long)c * g.L : nullptr, h0, h1, zs, ZS,
                                    tab, lane);
      bnn_epilogue<PREDICT, false, GEN_TB>(p, c, wt, lane, zs, ZS, tab, cnt, pacc, pvote);
      __syncwarp();
    }
    bnn_pred_flush<PREDICT>(p, wt, lane, pacc, pvote);
  }
  if (n_cnt) {
    __syncthreads();
    for (int i = threadIdx.x; i < n_cnt; i += blockDim.x)
      if (cnt[i]) atomicAdd(&p.counts[i], cnt[i]);
  }
}

// =============================================================================================
// specialised 3-layer kernel (compile-time padded widths KP0 -> N1 -> N2 -> N3), categorical likelihood
// =============================================================================================
template <int KP0, int N1, int N2, int N3>
struct Fwd3Geom {
  static constexpr int SW0 = (KP0 % 16 == 0) ? 8 : 0;
  static constexpr int SW1 = (N1 % 16 == 0) ? 8 : 0;
  static constexpr int SW2 = (N2 % 16 == 0) ? 8 : 0;
  static constexpr int W1_OFF = 0, B1_OFF = N1 * KP0;
  static constexpr int W2_OFF = B1_OFF + N1, B2_OFF = W2_OFF + N2 * N1;
  static constexpr int W3_OFF = B2_OFF + N2, B3_OFF = W3_OFF + N3 * N2;
  static constexpr int PB = B3_OFF + N3;
};

template <int ACT, bool FAST = false, int TB = BNN_EXP_TAB_BITS>
__device__ __forceinline__ void act_tile(double (&a)[4], double alpha, const double* tab) {
#pragma unroll
  for (int e = 0; e < 4; ++e) a[e] = FAST ? bnn_act_fast<ACT>(a[e], alpha, tab) : bnn_act<ACT, TB>(a[e], alpha, tab);
}

// Does any pre-activation of this warp's fragments need the guarded evaluation (|z| beyond the exponential's range,
// inf, NaN)?  One vote per layer: the common case then runs a straight-line copy of the layer without the clamp /
// NaN fix-up instructions (6 integer instructions per element on the 16-lane ALU pipe, which the activation chains
// of three warps otherwise keep as busy as the FP64 pipe).
template <int ACT, int NT>
__device__ __forceinline__ bool frag_needs_care(const double (&acc)[NT][4]) {
  if (ACT == BNN_ACT_RELU || ACT == BNN_ACT_LEAKY) return false;
  int worst = 0;
#pragma unroll
  for (int j = 0; j < NT; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) worst = max(worst, __double2hiint(acc[j][e]) & 0x7fffffff);
  return __any_sync(FULL_MASK, worst >= (ACT == BNN_ACT_SWISH ? 0x40862000 : 0x40762000));
}

// ---------------------------------------------------------------------------------------------
// Epilogues on the accumulator fragments of the last layer.  The 4 lanes of a quad hold one row pair
// (rows g and g+8), columns 8j+2t+{0,1}; row statistics are combined with two xor-shuffles and all exps
// of a thread are independent (ILP).
// ---------------------------------------------------------------------------------------------
template <int N3>
struct RowStats {
  double m[2], S[2], zy[2];
  int arg[2];
  double ev[2][N3 / 4];
};

// stage 1: row maximum and arg-max (first maximum wins, as np.argmax)
template <int N3>
__device__ __forceinline__ void qs_max(const double (&acc)[N3 / 8][4], int K, int t, RowStats<N3>& r) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    double m = -INFINITY;
    int arg = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = 8 * j + 2 * t + e;
        const double v = acc[j][2 * h + e];
        const bool take = col < K && v > m;      // columns ascend within a thread
        m = take ? v : m;
        arg = take ? col : arg;
      }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      const double om = __shfl_xor_sync(FULL_MASK, m, o);
      const int oa = __shfl_xor_sync(FULL_MASK, arg, o);
      const bool take = om > m || (om == m && oa < arg);
      m = take ? om : m;
      arg = take ? oa : arg;
    }
    r.m[h] = m;
    r.arg[h] = (arg == 0x7fffffff) ? 0 : arg;
  }
}

// stage 2: exp(z - max) of this thread's columns of row h, local sums
template <int N3, int H, bool NEED_ZY, int TB = BNN_EXP_TAB_BITS>
__device__ __forceinline__ void qs_exp(const double (&acc)[N3 / 8][4], int K, int t, const int (&y)[2],
                                       const double* tab, RowStats<N3>& r) {
  double S = 0.0, zy = 0.0;
#pragma unroll
  for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = 8 * j + 2 * t + e;
      const double v = acc[j][2 * H + e];
      // padded columns: argument -1000 => exp flushes to exactly 0 (no branch around the evaluation)
      const double ex = bnn_exp_neg<TB>((col < K) ? v - r.m[H] : -1000.0, tab);
      r.ev[H][2 * j + e] = ex;
      S += ex;
      if (NEED_ZY) zy = (col == y[H]) ? v : zy;
    }
  r.S[H] = S;
  r.zy[H] = zy;
}

// stage 3: quad reductions of the sums
template <int N3, bool NEED_ZY>
__device__ __forceinline__ void qs_reduce(RowStats<N3>& r) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    r.S[h] += __shfl_xor_sync(FULL_MASK, r.S[h], 1);
    r.S[h] += __shfl_xor_sync(FULL_MASK, r.S[h], 2);
    if (NEED_ZY) {
      r.zy[h] += __shfl_xor_sync(FULL_MASK, r.zy[h], 1);
      r.zy[h] += __shfl_xor_sync(FULL_MASK, r.zy[h], 2);
    }
  }
}

template <int N3, bool NEED_ZY, int TB = BNN_EXP_TAB_BITS>
__device__ __forceinline__ void quad_softmax_stats(const double (&acc)[N3 / 8][4], int K, int t, const int (&y)[2],
                                                   const double* tab, RowStats<N3>& r) {
  qs_max<N3>(acc, K, t, r);
  qs_exp<N3, 0, NEED_ZY, TB>(acc, K, t, y, tab, r);
  qs_exp<N3, 1, NEED_ZY, TB>(acc, K, t, y, tab, r);
  qs_reduce<N3, NEED_ZY>(r);
}

// Likelihood + accuracy counters of one (warp tile, weight set), in two parts so that the kernel can place
// the arithmetic (part 1: softmax statistics and log-likelihood, branch-free, latency-bound FP64 chains and
// shuffles) in the same basic block as the first MMAs of the NEXT weight set -- ptxas then interleaves the
// two -- and the side effects (part 2: counters and the partial-sum store) at the end of that block.
//   * without class / instance weights  sum_r log softmax = sum_r (z_y - max) - log(prod_r S_r): ONE log per
//     warp tile (the product of 16 sums of at most 32 terms each stays below 2^80)
//   * counters: ballots for n_correct, full-mask match.any groups for the per-class counters: at most one
//     shared-memory atomic per distinct class and warp tile instead of three per row
struct LikRow {
  double ll;          // warp-tile log-likelihood (all lanes)
  int my_y, my_arg;   // lane t == 0 speaks for row g, lane t == 1 for row g + 8
  bool ok, train, role;
};

// stage 4: per-row roles, warp-tile reduction and the logarithm
template <int N3, bool WEIGHTED>
__device__ __forceinline__ LikRow quad_lik_finish(const FwdParams& p, long long wt, int lane, const RowStats<N3>& r,
                                                  const int (&y)[2], const double (&wgt)[2], bool valid) {
  const int gq = lane >> 2, t = lane & 3;
  LikRow o;
  const int h = t & 1;
  const long long row = wt * 16 + gq + 8 * h;
  o.role = valid && t < 2 && row < p.n_total;
  o.train = o.role && row < p.n_train;
  o.my_y = h ? y[1] : y[0];
  o.my_arg = h ? r.arg[1] : r.arg[0];
  const double my_S = h ? r.S[1] : r.S[0];
  const double d = (h ? r.zy[1] : r.zy[0]) - (h ? r.m[1] : r.m[0]);
  o.ok = o.role && o.my_arg == o.my_y;
  // log(softmax) of the reference is -inf once exp(d) underflows to 0 (BNN_lib.py:121,168)
  const bool neg_inf = o.train && d < -745.1332191019412;
  double ll;
  if (!WEIGHTED) {
    double sd = o.train ? d : 0.0, ps = o.train ? my_S : 1.0;
#pragma unroll
    for (int s = 1; s <= 16; s <<= 1) {        // fixed xor tree => deterministic
      sd += __shfl_xor_sync(FULL_MASK, sd, s);
      ps *= __shfl_xor_sync(FULL_MASK, ps, s);
    }
    ll = sd - bnn_log_ge1(ps);
  } else {
    ll = o.train ? (d - bnn_log_ge1(my_S)) * (h ? wgt[1] : wgt[0]) : 0.0;
#pragma unroll
    for (int s = 1; s <= 16; s <<= 1) ll += __shfl_xor_sync(FULL_MASK, ll, s);
  }
  o.ll = __any_sync(FULL_MASK, neg_inf) ? -INFINITY : ll;
  return o;
}

template <int N3>
__device__ __forceinline__ void quad_lik_commit(const FwdParams& p, int c, long long wt, int lane, int* cnt,
                                                const LikRow& o, bool valid) {
  static_assert(N3 < 32, "one lane per class plus one for the totals");
  const int K = p.g.K;
  int* cc = cnt + c * bnn_n_counts(K);
  // Counters without data-dependent control flow: one ballot per class and table (independent VOTEs that pipeline),
  // lane k keeps the count of class k, then ONE predicated shared-memory atomic per table with distinct addresses per
  // lane.  (Measured: the counters cost nothing -- a build without them runs in the same 17.3 ms.)
  const unsigned ok_train = __ballot_sync(FULL_MASK, o.ok && o.train);
  const unsigned ok_test = __ballot_sync(FULL_MASK, o.ok && !o.train);
  int n_y = 0, n_arg = 0;
#pragma unroll
  for (int k = 0; k < N3; ++k) {
    const unsigned by = __ballot_sync(FULL_MASK, o.ok && o.train && o.my_y == k);
    const unsigned ba = __ballot_sync(FULL_MASK, o.train && o.my_arg == k);
    if (lane == k) { n_y = __popc(by); n_arg = __popc(ba); }
  }
  if (lane == N3) { n_y = __popc(ok_train); n_arg = __popc(ok_test); }
  // lanes 0..K-1: class tables; lane N3: the two totals (cc[0], cc[1])
  const bool tab = lane < K;
  const int i_y = tab ? 2 + lane : 0, i_arg = tab ? 2 + K + lane : 1;
  if ((tab || lane == N3) && n_y) atomicAdd(&cc[i_y], n_y);
  if ((tab || lane == N3) && n_arg) atomicAdd(&cc[i_arg], n_arg);
  if (valid && lane == 0) p.part[((long long)c * p.NF) * p.n_tiles16 + wt] = o.ll;
}

// Posterior summaries: softmax probabilities accumulated per (row, class) in registers over the weight sets.
template <int N3>
__device__ __forceinline__ void quad_epilogue_pred(const FwdParams& p, int c, long long wt, int lane,
                                                   const double (&acc)[N3 / 8][4], const double* tab,
                                                   double (&pacc)[2][N3 / 4], int (&pvote)[2][N3 / 4]) {
  const int K = p.g.K;
  const int gq = lane >> 2, t = lane & 3;
  const int y[2] = {-1, -1};
  RowStats<N3> r;
  quad_softmax_stats<N3, false>(acc, K, t, y, tab, r);
  if (p.samp_philox) {
    // Posterior-predictive resampling (sample_from_categorical, BNN_lib.py:682-713) with in-kernel uniforms: the class of
    // (row, set) is the first one whose cumulative probability reaches u (none: class 0).  The classes of a row are
    // spread over the 4 lanes of a quad (columns 8j + 2t + e): each lane forms the cumulative sums of its own columns on
    // top of the quad-exclusive prefix of the 8-column block and the totals of the blocks before it.
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long row = wt * 16 + gq + 8 * h;
      const bool live = row < p.n_total;
      const double inv = 1.0 / r.S[h];
      const double u = live ? bnn_samp_uniform(p.samp_seed, p.samp_row0 + row, p.samp_set0 + c) : 2.0;
      double base = 0.0;
      int drawn = 0x7fffffff;
#pragma unroll
      for (int j = 0; j < N3 / 8; ++j) {
        const int c0 = 8 * j + 2 * t;
        const double p0 = (c0 < K) ? r.ev[h][2 * j] * inv : 0.0, p1 = (c0 + 1 < K) ? r.ev[h][2 * j + 1] * inv : 0.0;
        double incl = p0 + p1;                                    // inclusive scan over t (lanes of the quad)
        const double up1 = __shfl_up_sync(FULL_MASK, incl, 1, 4);
        if (t >= 1) incl += up1;
        const double up2 = __shfl_up_sync(FULL_MASK, incl, 2, 4);
        if (t >= 2) incl += up2;
        const double excl = base + incl - (p0 + p1);
        const double cum0 = excl + p0, cum1 = cum0 + p1;
        if (c0 + 1 < K && cum1 - u >= 0.0 && c0 + 1 < drawn) drawn = c0 + 1;
        if (c0 < K && cum0 - u >= 0.0 && c0 < drawn) drawn = c0;
        base += __shfl_sync(FULL_MASK, incl, 3, 4);               // total of this 8-column block
      }
      drawn = min(drawn, __shfl_xor_sync(FULL_MASK, drawn, 1));
      drawn = min(drawn, __shfl_xor_sync(FULL_MASK, drawn, 2));
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
        const unsigned grp = __match_any_sync(FULL_MASK, (live && t == 0) ? drawn : 64 + lane);
        if (live && t == 0 && lane == __ffs(grp) - 1) atomicAdd(&p.samp_counts[c * K + drawn], __popc(grp));
      }
    }
    return;
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const long long row = wt * 16 + gq + 8 * h;
    if (row < p.n_total) {
      const double inv = 1.0 / r.S[h];
#pragma unroll
      for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int col = 8 * j + 2 * t + e;
          if (col < K) {
            const double pk = r.ev[h][2 * j + e] * inv;
            pacc[h][2 * j + e] += pk;
            if (p.dense_out) p.dense_out[((long long)c * p.n_total + row) * K + col] = pk;
            if (col == r.arg[h]) pvote[h][2 * j + e] += 1;
          }
        }
    }
  }
}

// Gaussian likelihoods (calc_likelihood_regression / _error, BNN_lib.py:123-143) on the last layer's accumulator
// fragment (N3 = 8: thread (g, t) holds rows g and g + 8, columns 2t and 2t + 1).  Per (warp tile, weight set) and
// modelled output j the kernel leaves sum r, sum r^2 over the training rows and sum r^2 over the test rows
// (r = prediction - target), from which finalize_loglik forms the log-likelihood (fixed or empirical sigma) and the
// MSE statistics; with the sigma head (columns K..2K-1 through softplus) the per-row log-density is summed here.
template <int N3>
__device__ __forceinline__ void quad_gauss_lik(const FwdParams& p, int c, long long wt, int lane,
                                               const double (&acc)[N3 / 8][4], const double* tab) {
  static_assert(N3 == 8, "Gaussian outputs fit one 8-column tile");
  const int K = p.g.K;
  const bool head = (p.g.lik == BNN_LIK_GAUSSIAN_HEAD);
  const int gq = lane >> 2, t = lane & 3;
  const long long nt = p.n_tiles16;
  double ll = 0.0, sr[2] = {0.0, 0.0}, sr2[2] = {0.0, 0.0}, st2[2] = {0.0, 0.0};
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int col = 2 * t + e;
    const int scol = (col + K) & 7;                                // column of this output's sigma parameter (head)
    const int src = (gq << 2) | (scol >> 1);
    const double s00 = __shfl_sync(FULL_MASK, acc[0][0], src), s01 = __shfl_sync(FULL_MASK, acc[0][1], src);
    const double s10 = __shfl_sync(FULL_MASK, acc[0][2], src), s11 = __shfl_sync(FULL_MASK, acc[0][3], src);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long row = wt * 16 + gq + 8 * h;
      const bool active = row < p.n_total && col < K;
      const bool train = active && row < p.n_train;
      double r = 0.0;
      if (active) {
        const double tv = p.targets[row * K + col];
        const double mu = acc[0][2 * h + e];
        r = mu - tv;
        if (head && train) {
          const double zs = (scol & 1) ? (h ? s11 : s01) : (h ? s10 : s00);
          if (fabs(zs) < 700.0) {
            const double sd = bnn_softplus_fast(zs, tab);
            const double u = (tv - mu) * bnn_rcp(sd);
            ll += -0.5 * u * u - kLogSqrt2Pi - bnn_log_ge1(sd);
          } else {                                                   // out of the table routine's range, inf, NaN: libm
            const double sd = softplus_ref(zs);
            const double u = (tv - mu) / sd;
            ll += -0.5 * u * u - kLogSqrt2Pi - log(sd);
          }
        }
      }
      sr[e] += train ? r : 0.0;
      sr2[e] += train ? r * r : 0.0;
      st2[e] += (active && !train) ? r * r : 0.0;
    }
  }
#pragma unroll
  for (int o = 4; o <= 16; o <<= 1)                                 // rows: fixed xor tree over g => deterministic
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      sr[e] += __shfl_xor_sync(FULL_MASK, sr[e], o);
      sr2[e] += __shfl_xor_sync(FULL_MASK, sr2[e], o);
      st2[e] += __shfl_xor_sync(FULL_MASK, st2[e], o);
    }
#pragma unroll
  for (int o = 1; o <= 16; o <<= 1) ll += __shfl_xor_sync(FULL_MASK, ll, o);
  if (gq == 0) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = 2 * t + e;
      if (col < K) {
        p.part[((long long)c * p.NF + 1 + col) * nt + wt] = sr[e];
        p.part[((long long)c * p.NF + 1 + K + col) * nt + wt] = sr2[e];
        p.part[((long long)c * p.NF + 1 + 2 * K + col) * nt + wt] = st2[e];
      }
    }
  }
  if (lane == 0) p.part[((long long)c * p.NF) * nt + wt] = ll;
}

// Count likelihoods (BNN_LIK_POISSON / NEGBIN / NEGBIN10, BNN_lik.py:5-66) on the same fragment: per row and modelled
// column j the log-pmf of bnn_count_loglik (the dispersion output K + j fetched from the lane that holds it, as the
// sigma head does), summed over the training rows; sum r, sum r^2 (train) and sum r^2 (test) of r = mean - k for the
// companion MSE.  Same xor trees and slots as quad_gauss_lik, so finalize_loglik and the accept step read them alike.
template <int N3>
__device__ __forceinline__ void quad_count_lik(const FwdParams& p, int c, long long wt, int lane,
                                               const double (&acc)[N3 / 8][4]) {
  static_assert(N3 == 8, "count outputs fit one 8-column tile");
  const int K = p.g.K, lik = p.g.lik;
  const int gq = lane >> 2, t = lane & 3;
  const long long nt = p.n_tiles16;
  double ll = 0.0, sr[2] = {0.0, 0.0}, sr2[2] = {0.0, 0.0}, st2[2] = {0.0, 0.0};
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int col = 2 * t + e;
    const int dcol = (col + K) & 7;                                // column of this output's dispersion (NEGBIN*)
    const int src = (gq << 2) | (dcol >> 1);
    const double d00 = __shfl_sync(FULL_MASK, acc[0][0], src), d01 = __shfl_sync(FULL_MASK, acc[0][1], src);
    const double d10 = __shfl_sync(FULL_MASK, acc[0][2], src), d11 = __shfl_sync(FULL_MASK, acc[0][3], src);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long row = wt * 16 + gq + 8 * h;
      const bool active = row < p.n_total && col < K;
      const bool train = active && row < p.n_train;
      double r = 0.0;
      if (active) {
        const double zd = (dcol & 1) ? (h ? d11 : d01) : (h ? d10 : d00);
        const double lr = bnn_count_loglik(lik, acc[0][2 * h + e], zd, p.targets[row * K + col], p.lgk1[row * K + col], &r);
        if (train) ll += lr;
      }
      sr[e] += train ? r : 0.0;
      sr2[e] += train ? r * r : 0.0;
      st2[e] += (active && !train) ? r * r : 0.0;
    }
  }
#pragma unroll
  for (int o = 4; o <= 16; o <<= 1)                                 // rows: fixed xor tree over g => deterministic
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      sr[e] += __shfl_xor_sync(FULL_MASK, sr[e], o);
      sr2[e] += __shfl_xor_sync(FULL_MASK, sr2[e], o);
      st2[e] += __shfl_xor_sync(FULL_MASK, st2[e], o);
    }
#pragma unroll
  for (int o = 1; o <= 16; o <<= 1) ll += __shfl_xor_sync(FULL_MASK, ll, o);
  if (gq == 0) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = 2 * t + e;
      if (col < K) {
        p.part[((long long)c * p.NF + 1 + col) * nt + wt] = sr[e];
        p.part[((long long)c * p.NF + 1 + K + col) * nt + wt] = sr2[e];
        p.part[((long long)c * p.NF + 1 + 2 * K + col) * nt + wt] = st2[e];
      }
    }
  }
  if (lane == 0) p.part[((long long)c * p.NF) * nt + wt] = ll;
}

// prediction mode: transformed outputs (identity, softplus on the sigma head) accumulated over the weight sets
template <int N3>
__device__ __forceinline__ void quad_gauss_pred(const FwdParams& p, int c, long long wt, int lane,
                                                const double (&acc)[N3 / 8][4], double (&pacc)[2][N3 / 4], const double* tab) {
  static_assert(N3 == 8, "Gaussian outputs fit one 8-column tile");
  const int K = p.g.K, O = p.g.O;
  const bool head = (p.g.lik == BNN_LIK_GAUSSIAN_HEAD);
  const int gq = lane >> 2, t = lane & 3;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const long long row = wt * 16 + gq + 8 * h;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = 2 * t + e;
      if (row < p.n_total && col < O) {
        double v = acc[0][2 * h + e];
        if (head && col >= K) v = (fabs(v) < 700.0) ? bnn_softplus_fast(v, tab) : softplus_ref(v);
        pacc[h][e] += v;
        if (p.dense_out) p.dense_out[((long long)c * p.n_total + row) * O + col] = v;
      }
    }
  }
}

// MODE: 0 likelihood, 1 likelihood with class / instance weights, 2 posterior prediction
enum { FWD3_LIK = 0, FWD3_LIK_W = 1, FWD3_PRED = 2 };
// LIKK: 0 categorical (softmax epilogue, software-pipelined into the next weight set), 1 Gaussian (plain or sigma head),
// 2 count likelihoods (likelihood modes only: their prediction is the Gaussian instantiation's identity output)
enum { FWD3_CAT = 0, FWD3_GAUSS = 1, FWD3_COUNT = 2 };

template <int ACT, int KP0, int N1, int N2, int N3, int NWARPS, int MODE, int LIKK = FWD3_CAT>
__global__ void __launch_bounds__(NWARPS * 32, 1) k_fwd3(const __grid_constant__ FwdParams p) {
  using G3 = Fwd3Geom<KP0, N1, N2, N3>;
  constexpr bool PREDICT = (MODE == FWD3_PRED);
  constexpr bool CAT = (LIKK == FWD3_CAT);
  constexpr bool DEFER = !PREDICT && CAT;        // categorical likelihood: epilogue pipelined into the next set's layer 1
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const NetGeom& g = p.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gq = lane >> 2, t = lane & 3;

  // ---- shared memory carve-up
  // Weight ring, two slots per part: part 0 = first-layer matrix + bias (W1_D doubles), part 1 = the rest of the
  // packed weight set (W23_D doubles).  The parts are released separately: the first layer is 61 % of a use, so its
  // slot is free (and its refill under way) long before the warp is done with the use.
  constexpr int W1_D = G3::W2_OFF, W23_D = G3::PB - G3::W2_OFF;
  double* w1buf = reinterpret_cast<double*>(smem_raw);                  // [2][W1_D]
  double* w23buf = w1buf + 2 * W1_D;                                    // [2][W23_D]
  double* xs = w23buf + 2 * W23_D + warp * 16 * KP0;                    // [NWARPS][16*KP0] X warp tiles
  double* tab = w23buf + 2 * W23_D + NWARPS * 16 * KP0;                 // exp table
  uint64_t* bars = reinterpret_cast<uint64_t*>(tab + BNN_EXP_TAB_SIZE);
  uint64_t* full1 = bars;           // [2]
  uint64_t* full23 = bars + 2;      // [2]
  uint64_t* xbar = bars + 4 + warp; // [NWARPS]
  int* rel = reinterpret_cast<int*>(bars + 4 + NWARPS);   // [4] warps that released slot b of part 0 / part 1
  int* cnt = reinterpret_cast<int*>(bars + 6 + NWARPS);
  const int n_cnt = DEFER ? p.C * bnn_n_counts(g.K) : 0;
  const int PW = CAT ? g.K : g.O;                 // columns of a prediction row

  for (int i = threadIdx.x; i < BNN_EXP_TAB_SIZE; i += blockDim.x) tab[i] = p.exp_tab[i];
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) cnt[i] = 0;
  if (threadIdx.x == 0) {
    rel[0] = rel[1] = rel[2] = rel[3] = 0;
    mbar_init(&full1[0], 1); mbar_init(&full1[1], 1);
    mbar_init(&full23[0], 1); mbar_init(&full23[1], 1);
    for (int w = 0; w < NWARPS; ++w) mbar_init(&bars[4 + w], 1);
    mbar_fence_init();
  }
  __syncthreads();

  // Work decomposition.  n_full rounds in which every warp of the grid owns one 16-row tile and runs all C
  // weight sets over it; the remaining tiles (fewer than one per warp) form `groups` CTA-sized tile groups
  // whose (group, weight set) pairs are dealt out evenly over the CTAs, so that the last round costs
  // ceil(groups*C/grid) weight sets per CTA instead of C (c4: 7 instead of 32, 36 rounds -> 35.2).  A CTA's
  // share is a contiguous range of pairs, i.e. at most two segments (tile group, [lo, hi)).  Every (tile,
  // weight set) is still computed by exactly one warp with the same instruction sequence, so results do not
  // depend on the decomposition.  Prediction accumulates over weight sets in registers: no split there.
  const long long total_warps = (long long)gridDim.x * NWARPS;
  const long long n_full = p.n_tiles16 / total_warps;
  const long long tail_base = n_full * total_warps;
  const long long rem = p.n_tiles16 - tail_base;
  int seg_tg[2] = {0, 0}, seg_lo[2] = {0, 0}, seg_hi[2] = {0, 0};
  if (rem > 0) {
    const long long groups = (rem + NWARPS - 1) / NWARPS;
    if (PREDICT) {
      if ((long long)blockIdx.x < groups) { seg_tg[0] = blockIdx.x; seg_hi[0] = p.C; }
    } else {
      const long long pairs = groups * p.C;
      const long long per_cta = (pairs + gridDim.x - 1) / gridDim.x;
      const long long s0 = (long long)blockIdx.x * per_cta;
      const long long s1 = (s0 + per_cta < pairs) ? s0 + per_cta : pairs;
      if (s0 < s1) {
        seg_tg[0] = (int)(s0 / p.C);
        seg_lo[0] = (int)(s0 % p.C);
        const long long n0 = ((s1 - s0) < (long long)(p.C - seg_lo[0])) ? (s1 - s0) : (long long)(p.C - seg_lo[0]);
        seg_hi[0] = seg_lo[0] + (int)n0;
        if (s1 - s0 > n0) { seg_tg[1] = seg_tg[0] + 1; seg_hi[1] = (int)(s1 - s0 - n0); }
      }
    }
  }
  const long long q_seg0 = n_full * p.C;                         // first weight-set use of segment 0
  const long long q_seg1 = q_seg0 + (seg_hi[0] - seg_lo[0]);     // ... of segment 1
  const long long total_q = q_seg1 + (seg_hi[1] - seg_lo[1]);    // weight-set uses, identical for every warp of the CTA
  const long long n_iter = n_full + (seg_hi[0] > seg_lo[0] ? 1 : 0) + (seg_hi[1] > seg_lo[1] ? 1 : 0);
  auto set_of = [&](long long qq) -> long long {                 // weight set consumed by use qq of this CTA
    return qq < q_seg0 ? qq % p.C : (qq < q_seg1 ? seg_lo[0] + (qq - q_seg0) : seg_lo[1] + (qq - q_seg1));
  };
  constexpr uint32_t W1_BYTES = W1_D * sizeof(double), W23_BYTES = W23_D * sizeof(double);
  constexpr uint32_t X_BYTES = 16 * KP0 * sizeof(double);
  static_assert(W1_BYTES % 16 == 0 && W23_BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");

  auto load_part = [&](int part, long long qq) {
    const int b = (int)(qq & 1);
    const double* src = p.wp + set_of(qq) * G3::PB;
    if (part == 0) {
      mbar_arrive_expect_tx(&full1[b], W1_BYTES);
      bulk_g2s(w1buf + b * W1_D, src, W1_BYTES, &full1[b]);
    } else {
      mbar_arrive_expect_tx(&full23[b], W23_BYTES);
      bulk_g2s(w23buf + b * W23_D, src + W1_D, W23_BYTES, &full23[b]);
    }
  };
  if (threadIdx.x == 0) {
    for (int q = 0; q < 2 && q < total_q; ++q) { load_part(0, q); load_part(1, q); }
  }

  // A slot is released by every warp when it is done with use qq of that part; the warp whose release is the last
  // one issues the bulk copy of use qq+2 into the slot itself, so a refill starts the moment the slot is free (a fixed
  // producer thread would start it only when its own warp next reaches the top of the weight-set loop, and would make
  // that warp wait for the slowest one before every use: 17.01 -> 16.68 ms at c4).  The warp schedulers prefer the
  // younger warps (measured ring waits per warp: 0.3 / 2 / 4.5 % of the run for warps 0-3 / 4-7 / 8-11), so the
  // slowest warp is rarely warp 0.
  auto release_part = [&](int part, long long qq) {
    if (lane == 0) {
      int* r = &rel[2 * part + (int)(qq & 1)];
      __threadfence_block();                       // this warp's reads of the slot happen before the release
      const int old = atomicAdd(r, 1);
      if (old == NWARPS - 1) {                     // last warp out refills the slot
        *r = 0;
        if (qq + 2 < total_q) {
          __threadfence_block();
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          load_part(part, qq + 2);
        }
      }
    }
  };
  long long q = 0;
  uint32_t x_uses = 0;               // X tiles this warp has loaded (parity of its mbarrier)
  bool x_prefetched = false;         // the X tile of this iteration was requested during the previous one
  auto tile_of = [&](long long i) -> long long {             // 16-row tile of this warp in iteration i
    const int s2 = (int)(i - n_full);
    return s2 < 0 ? i * total_warps + (long long)blockIdx.x * NWARPS + warp
                  : tail_base + (long long)(s2 == 0 ? seg_tg[0] : seg_tg[1]) * NWARPS + warp;
  };
  // Likelihood modes: the epilogue of a (tile, weight set) is software-pipelined into layer 1 of the NEXT weight set
  // this warp runs -- also across a tile boundary, so that a tile's last set is not finished in a phase of its own
  // (that phase is 1/32 of a tile at 32 sets per GPU, but a quarter at 4 and everything for a single chain).
  // acc3 / ep_* describe the pending epilogue: last-layer accumulators, tile, weight set, labels (and weights).
  double acc3[N3 / 8][4];
  bool prev_valid = false;
  long long ep_wt = 0;
  int ep_c = 0;
  int ep_y[2] = {0, 0};
  double ep_wgt[2] = {1.0, 1.0};
#pragma unroll
  for (int j = 0; j < N3 / 8; ++j) acc3[j][0] = acc3[j][1] = acc3[j][2] = acc3[j][3] = 0.0;
  for (long long it = 0; it < n_iter; ++it) {
    const int sg = (int)(it - n_full);                       // tail segment (>= 0) or full round (< 0)
    const long long wt = tile_of(it);
    const int c_lo = sg < 0 ? 0 : (sg == 0 ? seg_lo[0] : seg_lo[1]);
    const int c_hi = sg < 0 ? p.C : (sg == 0 ? seg_hi[0] : seg_hi[1]);
    const bool have_tile = wt < p.n_tiles16;
    int y[2] = {0, 0};
    double wgt[2] = {1.0, 1.0};
    double pacc[2][N3 / 4];
    int pvote[2][N3 / 4];
    if (have_tile) {
      if (lane == 0 && !x_prefetched) {
        // order this warp's earlier generic-proxy reads of xs before the async-proxy overwrite
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive_expect_tx(xbar, X_BYTES);
        bulk_g2s(xs, p.x + wt * 16 * KP0, X_BYTES, xbar);
      }
      x_prefetched = false;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const long long row = wt * 16 + gq + 8 * h;
        if (DEFER && row < p.n_total) {
          y[h] = p.labels[row];
          if (MODE == FWD3_LIK_W) {
            if (p.class_w) wgt[h] *= p.class_w[y[h]];
            if (p.inst_w && row < p.n_train) wgt[h] *= p.inst_w[row];
          }
        }
#pragma unroll
        for (int i = 0; i < N3 / 4; ++i) { pacc[h][i] = 0.0; pvote[h][i] = 0; }
      }
      mbar_wait(xbar, x_uses & 1);
      ++x_uses;
    }
    for (int c = c_lo; c < c_hi; ++c, ++q) {
      const int b = (int)(q & 1);
      __syncwarp();
      mbar_wait(&full1[b], (uint32_t)((q >> 1) & 1));
      if (have_tile) {
        const double* W = w1buf + b * W1_D;                          // part 0; layers 2 / 3 index W23 with the same offsets
        const double* W23 = w23buf + b * W23_D - G3::W2_OFF;
        const double a1 = (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha[c * 3 + 0] : 0.0;
        const double a2 = (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha[c * 3 + 1] : 0.0;
        // ---------------- layer 1: [16 x KP0] x [KP0 x N1]
        double acc1[N1 / 8][4];
#pragma unroll
        for (int j = 0; j < N1 / 8; ++j) {
          const double2 bb = *reinterpret_cast<const double2*>(W + G3::B1_OFF + 8 * j + 2 * t);
          acc1[j][0] = bb.x; acc1[j][1] = bb.y; acc1[j][2] = bb.x; acc1[j][3] = bb.y;
        }
        {
          const double* xr0 = xs + gq * KP0;
          const double* xr1 = xs + (gq + 8) * KP0;
          const double* wr = W + G3::W1_OFF + gq * KP0;
          const int sw = (gq & 1) * G3::SW0;
          // Software pipeline over weight sets: the epilogue of the PREVIOUS set (softmax statistics, log-
          // likelihood: latency-bound FP64 chains and shuffles) is cut into four stages that are placed
          // between the MMA groups of the first two k-groups of this set's layer 1, whose DMMAs leave the
          // FP64 issue slots free.
          RowStats<N3> rs;
          LikRow lr;
          const int K = g.K;
#pragma unroll
          for (int kg = 0; kg < 2; ++kg) {
            const int col = (8 * kg + 2 * t) ^ sw;
            const double2 alo = *reinterpret_cast<const double2*>(xr0 + col);
            const double2 ahi = *reinterpret_cast<const double2*>(xr1 + col);
            if (DEFER) {
              if (kg == 0) qs_max<N3>(acc3, K, t, rs);
              else qs_exp<N3, 1, true>(acc3, K, t, ep_y, tab, rs);
            }
#pragma unroll
            for (int j = 0; j < N1 / 16; ++j) {
              const double2 bb = *reinterpret_cast<const double2*>(wr + j * 8 * KP0 + col);
              dmma16x8x8(acc1[j], alo.x, ahi.x, alo.y, ahi.y, bb.x, bb.y);
            }
            if (DEFER) {
              if (kg == 0) qs_exp<N3, 0, true>(acc3, K, t, ep_y, tab, rs);
              else {
                qs_reduce<N3, true>(rs);
                lr = quad_lik_finish<N3, MODE == FWD3_LIK_W>(p, ep_wt, lane, rs, ep_y, ep_wgt, prev_valid);
              }
            }
#pragma unroll
            for (int j = N1 / 16; j < N1 / 8; ++j) {
              const double2 bb = *reinterpret_cast<const double2*>(wr + j * 8 * KP0 + col);
              dmma16x8x8(acc1[j], alo.x, ahi.x, alo.y, ahi.y, bb.x, bb.y);
            }
          }
          if (DEFER) quad_lik_commit<N3>(p, ep_c, ep_wt, lane, cnt, lr, prev_valid);
#pragma unroll 2
          for (int kg = 2; kg < KP0 / 8 - 2; ++kg) {
            const int col = (8 * kg + 2 * t) ^ sw;
            const double2 alo = *reinterpret_cast<const double2*>(xr0 + col);
            const double2 ahi = *reinterpret_cast<const double2*>(xr1 + col);
#pragma unroll
            for (int j = 0; j < N1 / 8; ++j) {
              const double2 bb = *reinterpret_cast<const double2*>(wr + j * 8 * KP0 + col);
              dmma16x8x8(acc1[j], alo.x, ahi.x, alo.y, ahi.y, bb.x, bb.y);
            }
          }
          // last two k-groups tile by tile: acc1[0] is complete first, so its activation (below, same basic
          // block) overlaps with the MMAs that finish the other tiles
          {
            const int c0 = (8 * (KP0 / 8 - 2) + 2 * t) ^ sw, c1 = (8 * (KP0 / 8 - 1) + 2 * t) ^ sw;
            const double2 alo0 = *reinterpret_cast<const double2*>(xr0 + c0), ahi0 = *reinterpret_cast<const double2*>(xr1 + c0);
            const double2 alo1 = *reinterpret_cast<const double2*>(xr0 + c1), ahi1 = *reinterpret_cast<const double2*>(xr1 + c1);
#pragma unroll
            for (int j = 0; j < N1 / 8; ++j) {
              const double2 b0 = *reinterpret_cast<const double2*>(wr + j * 8 * KP0 + c0);
              const double2 b1 = *reinterpret_cast<const double2*>(wr + j * 8 * KP0 + c1);
              dmma16x8x8(acc1[j], alo0.x, ahi0.x, alo0.y, ahi0.y, b0.x, b0.y);
              dmma16x8x8(acc1[j], alo1.x, ahi1.x, alo1.y, ahi1.y, b1.x, b1.y);
            }
          }
        }
        // the first-layer weights of this use are no longer needed by this warp; layers 2 / 3 need part 1
        __syncwarp();
        release_part(0, q);
        mbar_wait(&full23[b], (uint32_t)((q >> 1) & 1));
        // X is read by layer 1 only: after layer 1 of the tile's LAST weight set the buffer is free, and the next
        // tile's X (one bulk copy, ~2 us from HBM) arrives under layers 2 / 3 and the epilogue instead of stalling
        // the start of the next tile -- 0.4 % of a 32-set tile, but 3 % at 4 sets per GPU and 12 % for a single chain.
        if (c == c_hi - 1 && it + 1 < n_iter) {
          const long long wt_next = tile_of(it + 1);
          if (wt_next < p.n_tiles16) {
            __syncwarp();                                      // every lane's reads of xs are done
            if (lane == 0) {
              asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
              mbar_arrive_expect_tx(xbar, X_BYTES);
              bulk_g2s(xs, p.x + wt_next * 16 * KP0, X_BYTES, xbar);
            }
            x_prefetched = true;
          }
        }
        // ---------------- layer 2: [16 x N1] x [N1 x N2]   (A operand = activated acc1, no data movement).
        // The activation of k-group kg+1 is independent of the MMAs of k-group kg, so its FP64 chains fill
        // the issue slots between the DMMAs instead of running as a separate latency-bound phase.
        // Two straight-line copies per layer: one warp vote decides whether any pre-activation needs the guarded
        // evaluation (frag_needs_care); the common copy carries no clamp / NaN fix-up instructions.
        double acc2[N2 / 8][4];
#pragma unroll
        for (int j = 0; j < N2 / 8; ++j) {
          const double2 bb = *reinterpret_cast<const double2*>(W23 + G3::B2_OFF + 8 * j + 2 * t);
          acc2[j][0] = bb.x; acc2[j][1] = bb.y; acc2[j][2] = bb.x; acc2[j][3] = bb.y;
        }
        auto layer2 = [&](auto fast_tag) {
          constexpr bool FAST = decltype(fast_tag)::value;
          const double* wr = W23 + G3::W2_OFF + gq * N1;
          const int sw = (gq & 1) * G3::SW1;
          act_tile<ACT, FAST>(acc1[0], a1, tab);
#pragma unroll
          for (int kg = 0; kg < N1 / 8 - 2; ++kg) {
            act_tile<ACT, FAST>(acc1[kg + 1], a1, tab);
            const int col = (8 * kg + 2 * t) ^ sw;
#pragma unroll
            for (int j = 0; j < N2 / 8; ++j) {
              const double2 bb = *reinterpret_cast<const double2*>(wr + j * 8 * N1 + col);
              dmma16x8x8(acc2[j], acc1[kg][0], acc1[kg][2], acc1[kg][1], acc1[kg][3], bb.x, bb.y);
            }
          }
          {
            constexpr int k0 = N1 / 8 - 2, k1 = N1 / 8 - 1;
            act_tile<ACT, FAST>(acc1[k1], a1, tab);
            const int c0 = (8 * k0 + 2 * t) ^ sw, c1 = (8 * k1 + 2 * t) ^ sw;
#pragma unroll
            for (int j = 0; j < N2 / 8; ++j) {
              const double2 b0 = *reinterpret_cast<const double2*>(wr + j * 8 * N1 + c0);
              const double2 b1 = *reinterpret_cast<const double2*>(wr + j * 8 * N1 + c1);
              dmma16x8x8(acc2[j], acc1[k0][0], acc1[k0][2], acc1[k0][1], acc1[k0][3], b0.x, b0.y);
              dmma16x8x8(acc2[j], acc1[k1][0], acc1[k1][2], acc1[k1][1], acc1[k1][3], b1.x, b1.y);
            }
          }
        };
        if (frag_needs_care<ACT, N1 / 8>(acc1)) layer2(std::false_type{});
        else layer2(std::true_type{});
        // ---------------- layer 3: [16 x N2] x [N2 x N3]
#pragma unroll
        for (int j = 0; j < N3 / 8; ++j) {
          const double2 bb = *reinterpret_cast<const double2*>(W23 + G3::B3_OFF + 8 * j + 2 * t);
          acc3[j][0] = bb.x; acc3[j][1] = bb.y; acc3[j][2] = bb.x; acc3[j][3] = bb.y;
        }
        auto layer3 = [&](auto fast_tag) {
          constexpr bool FAST = decltype(fast_tag)::value;
          const double* wr = W23 + G3::W3_OFF + gq * N2;
          const int sw = (gq & 1) * G3::SW2;
          act_tile<ACT, FAST>(acc2[0], a2, tab);
#pragma unroll
          for (int kg = 0; kg < N2 / 8; ++kg) {
            if (kg + 1 < N2 / 8) act_tile<ACT, FAST>(acc2[kg + 1], a2, tab);
            const int col = (8 * kg + 2 * t) ^ sw;
#pragma unroll
            for (int j = 0; j < N3 / 8; ++j) {
              const double2 bb = *reinterpret_cast<const double2*>(wr + j * 8 * N2 + col);
              dmma16x8x8(acc3[j], acc2[kg][0], acc2[kg][2], acc2[kg][1], acc2[kg][3], bb.x, bb.y);
            }
          }
        };
        if (frag_needs_care<ACT, N2 / 8>(acc2)) layer3(std::false_type{});
        else layer3(std::true_type{});
        // weights of this use are no longer needed by this warp
        __syncwarp();
        release_part(1, q);
        if (DEFER) {
          prev_valid = true;
          ep_wt = wt; ep_c = c;
          ep_y[0] = y[0]; ep_y[1] = y[1];
          if (MODE == FWD3_LIK_W) { ep_wgt[0] = wgt[0]; ep_wgt[1] = wgt[1]; }
        }
        if constexpr (CAT) {
          if (PREDICT) quad_epilogue_pred<N3>(p, c, wt, lane, acc3, tab, pacc, pvote);
        } else if constexpr (LIKK == FWD3_COUNT) {
          static_assert(!PREDICT, "count prediction runs the FWD3_GAUSS instantiation");
          quad_count_lik<N3>(p, c, wt, lane, acc3);
        } else {
          if (PREDICT) quad_gauss_pred<N3>(p, c, wt, lane, acc3, pacc, tab);
          else quad_gauss_lik<N3>(p, c, wt, lane, acc3, tab);
        }
      } else {
        // (a warp without a tile waits for both parts before releasing them, so that its releases cannot run ahead)
        mbar_wait(&full23[b], (uint32_t)((q >> 1) & 1));
        release_part(0, q);
        release_part(1, q);
      }
    }
    if (have_tile) {
      if (PREDICT) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const long long row = wt * 16 + gq + 8 * h;
#pragma unroll
          for (int j = 0; j < N3 / 8; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int col = 8 * j + 2 * t + e;
              if (row < p.n_total && col < PW) {
                if (p.mean_out) p.mean_out[row * PW + col] = pacc[h][2 * j + e] / p.inv_sets;
                if (CAT && p.votes_out) p.votes_out[row * PW + col] = (double)pvote[h][2 * j + e] / p.inv_sets;
              }
            }
        }
      }
    }
  }
  // drain the software pipeline: the epilogue of the last (tile, weight set) this warp ran
  if (DEFER && prev_valid) {
    RowStats<N3> rs;
    quad_softmax_stats<N3, true>(acc3, g.K, t, ep_y, tab, rs);
    const LikRow lr = quad_lik_finish<N3, MODE == FWD3_LIK_W>(p, ep_wt, lane, rs, ep_y, ep_wgt, true);
    quad_lik_commit<N3>(p, ep_c, ep_wt, lane, cnt, lr, true);
  }
  if (n_cnt) {
    __syncthreads();
    for (int i = threadIdx.x; i < n_cnt; i += blockDim.x)
      if (cnt[i]) atomicAdd(&p.counts[i], cnt[i]);
  }
}

// =============================================================================================
// host-side launchers
// =============================================================================================
cudaError_t bnn_prepare_kernel(const void* fn, int max_dyn_smem, bool nonportable_cluster) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;      // (kernel, device) pairs already prepared
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  if (done.count({fn, dev})) return cudaSuccess;
  e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn_smem);
  if (e == cudaSuccess && nonportable_cluster) e = cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e == cudaSuccess) done.insert({fn, dev});
  return e;
}

template <int KP0, int N1, int N2, int N3, int NWARPS, int MODE, int LIKK>
static size_t fwd3_smem_bytes(const FwdParams& p) {
  constexpr bool DEFER = (MODE != FWD3_PRED) && (LIKK == FWD3_CAT);
  using G3 = Fwd3Geom<KP0, N1, N2, N3>;
  size_t d = 2 * (size_t)G3::PB + (size_t)NWARPS * 16 * KP0 + BNN_EXP_TAB_SIZE;
  size_t bytes = d * sizeof(double) + (6 + NWARPS) * sizeof(uint64_t);     // barriers + the ring's release counters
  return bytes + (DEFER ? bnn_smem_counts(p.g, p.C) : 0) * sizeof(int);
}

template <int ACT, int KP0, int N1, int N2, int N3, int NWARPS, int MODE, int LIKK>
static cudaError_t launch_fwd3(const FwdParams& p, int n_sms, cudaStream_t st) {
  auto kern = k_fwd3<ACT, KP0, N1, N2, N3, NWARPS, MODE, LIKK>;
  size_t smem = fwd3_smem_bytes<KP0, N1, N2, N3, NWARPS, MODE, LIKK>(p);
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, BNN_MAX_DYN_SMEM)) return e;
  if (smem > BNN_MAX_DYN_SMEM) return cudaErrorInvalidConfiguration;
  long long ctas = (p.n_tiles16 + NWARPS - 1) / NWARPS;
  if (MODE != FWD3_PRED) ctas *= p.C;          // likelihood modes deal (tile group, weight set) pairs out over the CTAs
  int grid = (int)(ctas < n_sms ? ctas : n_sms);
  kern<<<grid, NWARPS * 32, smem, st>>>(p);
  return cudaGetLastError();
}

// k_fwd3 instantiations: two padded width families x four activations x {categorical (N3 = 16: likelihood, weighted
// likelihood, prediction), Gaussian / sigma head (N3 = 8: likelihood, prediction), count (N3 = 8: likelihood)}
//   family A   64 -> 64 -> 32 -> N3   12 warps per SM (BASELINE config 4 / 5 is its swish / categorical member)
//   family B   32 -> 32 -> 16 -> N3   16 warps per SM
template <int ACT, int KP0, int N1, int N2, int NWARPS>
static cudaError_t launch_fwd3_family(const FwdParams& p, bool predict, int n_sms, cudaStream_t st) {
  if (p.g.lik == BNN_LIK_CATEGORICAL) {
    if (predict) return launch_fwd3<ACT, KP0, N1, N2, 16, NWARPS, FWD3_PRED, FWD3_CAT>(p, n_sms, st);
    if (p.class_w || p.inst_w) return launch_fwd3<ACT, KP0, N1, N2, 16, NWARPS, FWD3_LIK_W, FWD3_CAT>(p, n_sms, st);
    return launch_fwd3<ACT, KP0, N1, N2, 16, NWARPS, FWD3_LIK, FWD3_CAT>(p, n_sms, st);
  }
  if (predict) return launch_fwd3<ACT, KP0, N1, N2, 8, NWARPS, FWD3_PRED, FWD3_GAUSS>(p, n_sms, st);
  if (bnn_lik_is_count(p.g.lik)) return launch_fwd3<ACT, KP0, N1, N2, 8, NWARPS, FWD3_LIK, FWD3_COUNT>(p, n_sms, st);
  return launch_fwd3<ACT, KP0, N1, N2, 8, NWARPS, FWD3_LIK, FWD3_GAUSS>(p, n_sms, st);
}

template <int KP0, int N1, int N2, int NWARPS>
static cudaError_t launch_fwd3_act(const FwdParams& p, bool predict, int n_sms, cudaStream_t st) {
  return bnn_with_act(p.g.act, [&](auto a) {
    return launch_fwd3_family<decltype(a)::value, KP0, N1, N2, NWARPS>(p, predict, n_sms, st);
  });
}

// which k_fwd3 family the padded geometry matches exactly: 1 = A, 2 = B, 0 = none
int bnn_fwd3_family(const NetGeom& g) {
  if (g.L != 3) return 0;
  const int n3 = (g.lik == BNN_LIK_CATEGORICAL) ? 16 : 8;
  if (g.l[2].out_pad != n3) return 0;
  if (g.F_pad == 64 && g.l[0].out_pad == 64 && g.l[1].out_pad == 32) return 1;
  if (g.F_pad == 32 && g.l[0].out_pad == 32 && g.l[1].out_pad == 16) return 2;
  return 0;
}

template <int ACT, bool PREDICT>
static cudaError_t launch_generic_t(const FwdParams& p, int n_sms, cudaStream_t st) {
  auto kern = k_fwd_generic<ACT, PREDICT>;
  const int ZS = p.g.l[p.g.L - 1].out_pad + 1;
  const int PW = (p.g.lik == BNN_LIK_CATEGORICAL) ? p.g.K : p.g.O;
  size_t per_warp = 2 * 16 * (size_t)p.g.max_w + 16 * ZS + (PREDICT ? 16 * PW : 0);
  size_t bytes = (GEN_TAB_SIZE + GEN_WARPS * per_warp) * sizeof(double);
  size_t ints = PREDICT ? (size_t)GEN_WARPS * 16 * PW : bnn_smem_counts(p.g, p.C);
  bytes += ints * sizeof(int);
  if (bytes > BNN_MAX_DYN_SMEM) return cudaErrorInvalidConfiguration;
  if (bytes > 48 * 1024)
    if (cudaError_t e = bnn_prepare_kernel((const void*)kern, BNN_MAX_DYN_SMEM)) return e;
  long long ctas = (p.n_tiles16 + GEN_WARPS - 1) / GEN_WARPS;
  // resident CTAs per SM limited by shared memory; cap the grid at a few waves of resident CTAs
  long long max_grid = (long long)n_sms * 8;
  int grid = (int)(ctas < max_grid ? ctas : max_grid);
  int ny = 1;
  if (!PREDICT && p.C > 1 && grid < n_sms * 4) {
    const int want = (n_sms * 4 + grid - 1) / grid;
    ny = want < p.C ? want : p.C;
  }
  kern<<<dim3(grid, ny), GEN_WARPS * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

template <bool PREDICT>
static cudaError_t launch_generic(const FwdParams& p, int n_sms, cudaStream_t st) {
  return bnn_with_act(p.g.act, [&](auto a) { return launch_generic_t<decltype(a)::value, PREDICT>(p, n_sms, st); });
}

// Dispatch: specialised kernel when the padded shape is one of the compiled instantiations.
// force_generic != 0 disables the specialised path (used by the tests to cross-check both kernels).
cudaError_t bnn_launch_forward(const FwdParams& p, bool predict, int n_sms, int force_generic, cudaStream_t st,
                               const char** which) {
  const NetGeom& g = p.g;
  if (p.sp.prog && !predict) return bnn_launch_sparse(p, n_sms, st, which);
  if (!force_generic && !p.samp_u) {
    static const char* const names[2][4] = {
        {"k_fwd3<relu,64,64,32>", "k_fwd3<leaky,64,64,32>", "k_fwd3<swish,64,64,32,16>", "k_fwd3<tanh,64,64,32>"},
        {"k_fwd3<relu,32,32,16>", "k_fwd3<leaky,32,32,16>", "k_fwd3<swish,32,32,16>", "k_fwd3<tanh,32,32,16>"}};
    const int fam = bnn_fwd3_family(g);
    if (fam) {
      if (which) *which = names[fam - 1][g.act];
      return fam == 1 ? launch_fwd3_act<64, 64, 32, 12>(p, predict, n_sms, st)
                      : launch_fwd3_act<32, 32, 16, 16>(p, predict, n_sms, st);
    }
  }
  if (which) *which = "k_fwd_generic";
  return predict ? launch_generic<true>(p, n_sms, st) : launch_generic<false>(p, n_sms, st);
}
