// Device-side body of the Metropolis-Hastings update (accept / adapt / propose / prior / pack) and the deterministic
// reduction of the forward partials, shared by k_mh_update (bnn_mcmc.cu, one launch per step) and the persistent
// small-data chain loop (k_chain_loop, bnn_chainloop.cu).
//
// COH = true: the data another CTA of the same launch produced (tile partials, proposal counters) is read with
// ld.global.cg / plain loads instead of the read-only path, which is only valid for data that no thread of the
// launch writes.
#pragma once
#include "bnn_common.cuh"
#include "bnn_kernels.h"

#ifndef BNN_HAVE_LOGSQRT2PI
#define BNN_HAVE_LOGSQRT2PI
static constexpr double kLogSqrt2Pi = 0.91893853320467274178;
#endif
static constexpr double kLogPi = 1.14472988584940017414;
static constexpr double kLog2 = 0.69314718055994530942;
#define UPD_THREADS 1024      // upper bound (launch bounds); small networks launch 256 (upd_threads)

__device__ __forceinline__ int layer_of(const NetGeom& g, int i) {
  int l = 0;
#pragma unroll 1
  for (int k = 1; k < g.L; ++k)
    if (i >= g.l[k].c_off) l = k;
  return l;
}


// ------------------------------------------------------------------------------------------------
// Thread team of the block-wide steps below: every thread of the CTA (k_mh_update and the other one-CTA-per-chain
// kernels: TEAM = false), or the first UPD_TEAM_THREADS threads of a larger CTA synchronising on named barrier 1
// (the leader CTA of k_chain_loop: TEAM = true; the other warps of the CTA are parked at the cluster barrier).
// ------------------------------------------------------------------------------------------------
#define UPD_TEAM_THREADS 256
template <bool TEAM>
__device__ __forceinline__ int upd_nthreads() { return TEAM ? UPD_TEAM_THREADS : (int)blockDim.x; }
template <bool TEAM>
__device__ __forceinline__ void upd_sync() {
  if (TEAM) asm volatile("bar.sync 1, %0;" ::"n"(UPD_TEAM_THREADS) : "memory");
  else __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// deterministic block reductions (fixed order: per-thread strided sum -> xor tree -> warps in order)
// ------------------------------------------------------------------------------------------------
template <bool TEAM = false>
__device__ __forceinline__ double block_sum_fixed(double v, double* sh) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  upd_sync<TEAM>();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  upd_sync<TEAM>();
  double s = 0.0;
  for (int w = 0; w < (upd_nthreads<TEAM>() >> 5); ++w) s += sh[w];
  return s;
}

// Sum of src[tid], src[tid + B], src[tid + 2B], ... in exactly that order, with the loads of eight terms issued
// before the first add: the plain loop is one L2 round trip per term (62,500 partials per chain at 1M rows).
template <bool COH>
__device__ __forceinline__ double ld_part(const double* p) {
  // COH: written by other CTAs of this launch -- plain (generic) load, valid for global and (distributed) shared memory
  if (COH) return *reinterpret_cast<const volatile double*>(p);
  return __ldg(p);
}
template <bool COH = false>
__device__ __forceinline__ double strided_sum_ordered(const double* src, long long nt) {
  const long long B = upd_nthreads<COH>();
  long long i = threadIdx.x;
  double v = 0.0;
  for (; i + 7 * B < nt; i += 8 * B) {
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = ld_part<COH>(src + i + k * B);
#pragma unroll
    for (int k = 0; k < 8; ++k) v += a[k];
  }
  for (; i < nt; i += B) v += ld_part<COH>(src + i);
  return v;
}

// The update body is latency-bound straight-line code that runs once per MH iteration, far larger than the 32 KB
// instruction cache when every libm call is inlined at its call site (7.7k instructions for k_mh_update): the
// double-precision routines it uses are kept as single out-of-line copies.
static __device__ __noinline__ double upd_log(double x) { return log(x); }
static __device__ __noinline__ double upd_div(double a, double b) { return a / b; }
static __device__ __noinline__ double upd_gauss(double ws, double u1, double u2) {      // Box-Muller: ws sqrt(-2 log u1) cos(2 pi u2)
  double s, co;
  sincospi(2.0 * u2, &s, &co);
  return ws * sqrt(-2.0 * log(u1)) * co;
}

__device__ __forceinline__ double logpdf_prior(double w, int kind, double scale, double log_scale) {
  // closed forms of scipy.stats.{norm,cauchy,laplace}.logpdf(w, 0, scale) (BNN_env.py:139-150)
  double x = upd_div(w, scale);
  if (kind == BNN_PRIOR_CAUCHY) return -kLogPi - log1p(x * x) - log_scale;
  if (kind == BNN_PRIOR_LAPLACE) return -kLog2 - fabs(x) - log_scale;
  return -0.5 * x * x - kLogSqrt2Pi - log_scale;
}

// Reduce the per-warp-tile partials of one chain (part: [NF, nt]) and turn them into the log-likelihood.
//   red : shared [1 + 3*BNN_MAX_OUT] receives the reduced slots; sig_out [K] the sigma that was used
// Four slots share one pair of block barriers (a Gaussian likelihood has 1 + 3K of them); per slot the order of the
// additions is the one of block_sum_fixed: thread-strided terms, xor tree, warps in order.
template <bool COH = false>
__device__ double finalize_loglik(const NetGeom& g, const double* part, int NF, long long nt, long long n_train,
                                  double lik_temp, int sigma_mode, const double* __restrict__ sigma_in, double* red,
                                  double* sig_out) {
  __shared__ double sh4[4][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int s0 = 0; s0 < NF; s0 += 4) {
    const int ns = (NF - s0 < 4) ? NF - s0 : 4;
    double v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v[j] = 0.0;
      if (j < ns) {
        v[j] = strided_sum_ordered<COH>(part + (long long)(s0 + j) * nt, nt);
        for (int o = 16; o > 0; o >>= 1) v[j] += __shfl_xor_sync(0xffffffffu, v[j], o);
      }
    }
    upd_sync<COH>();                                   // (the previous group's sh4 has been read)
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (j < ns) sh4[j][warp] = v[j];
    }
    upd_sync<COH>();
    if ((int)threadIdx.x < ns) {
      double s = 0.0;
      for (int w = 0; w < (upd_nthreads<COH>() >> 5); ++w) s += sh4[threadIdx.x][w];
      red[s0 + threadIdx.x] = s;
    }
  }
  upd_sync<COH>();
  double ll = red[0];
  if (g.lik == BNN_LIK_GAUSSIAN) {
    // calc_likelihood_regression (BNN_lib.py:123-131) from sum r, sum r^2:
    //   sum_i logN(y_i; mu_i, s) = -SSR/(2 s^2) - N log s - N log sqrt(2 pi)
    ll = 0.0;
    const double N = (double)n_train;
    for (int j = 0; j < g.K; ++j) {
      double sr = red[1 + j], ssr = red[1 + g.K + j];
      double s;
      if (sigma_mode == BNN_SIGMA_EMPIRICAL) {
        double mu = sr / N;                       // np.std(y' - labels, axis=0) (BNN_env.py:475-476)
        s = sqrt(fmax(ssr / N - mu * mu, 0.0));
      } else {
        s = sigma_in ? sigma_in[j] : 1.0;
      }
      if (threadIdx.x == 0) sig_out[j] = s;
      ll += -upd_div(ssr, 2.0 * s * s) - N * upd_log(s) - N * kLogSqrt2Pi;
    }
  }
  upd_sync<COH>();
  // the count likelihoods of BNN_lik.py take lik_temp and ignore it
  return bnn_lik_is_count(g.lik) ? ll : lik_temp * ll;
}

struct Draw { int ix, iy; double dz; };
// k-th proposal of layer l of chain c at iteration it
__device__ __forceinline__ Draw philox_draw(uint64_t seed, int c, int it, int l, int k, int rows, int cols, double ws) {
  uint2 key = make_uint2((uint32_t)seed ^ (uint32_t)c, (uint32_t)(seed >> 32));
  uint4 a = philox4x32(make_uint4((uint32_t)it, (uint32_t)k, (uint32_t)l, 0u), key);
  uint4 b = philox4x32(make_uint4((uint32_t)it, (uint32_t)k, (uint32_t)l, 1u), key);
  Draw d;
  d.ix = (int)__umulhi(a.x, (uint32_t)rows);
  d.iy = (int)__umulhi(a.y, (uint32_t)cols);
  double u1 = 1.0 - u53(a.z, a.w);            // (0,1]
  double u2 = u53(b.x, b.y);
  d.dz = upd_gauss(ws, u1, u2);
  return d;
}

// Context of the persistent loop (k_chain_loop); value-initialised (all null / false) for k_mh_update.
//   part_c / counts_c : this chain's tile partials [NF, n_tiles16] and proposal counters [2 + 2K] in the leader CTA's
//                       shared memory (the other CTAs of the cluster write them through distributed shared memory)
//   w_sm              : [2P] current | proposed canonical weights, resident in shared memory between the calls of a
//                       launch (loaded when `first`, written back to d.w_cur / d.w_prop when `last`)
//   owner_sm          : [P] last-write-wins scratch, all -1 between calls
//   wpk_sm            : [PB] the packed proposal as the forward body of this CTA reads it (padding pre-zeroed); the
//                       global copy d.wp_prop is written as well
//   first / last      : first / last call of the launch: the chain's scalar state (sf / si) is loaded from and stored
//                       to global memory only then
struct UpdLoop {
  const double* part_c;
  int* counts_c;
  double* w_sm;
  int* owner_sm;
  double* wpk_sm;
  int* didx_sm;               // [2][UPD_DRAW_CAP] draw cache (entry index), one buffer per iteration parity -- k_mh_update
  double* ddz_sm;             // [2][UPD_DRAW_CAP] draw cache (increment)      keeps a single one in static shared memory
  int* pk_sm;                 // [P] per canonical entry: layer << 24 | offset in the packed set (filled when `first`)
  bool first, last;
};

#define UPD_DRAW_CAP 1024     // draws of one proposal kept in shared memory (index + increment): 12 KB

// ------------------------------------------------------------------------------------------------
// one CTA (or thread team, see upd_sync) per chain: [accept previous proposal] + [adapt, propose, prior, pack]
// ------------------------------------------------------------------------------------------------
// (Loops are kept rolled -- #pragma unroll 1: this is latency-bound code that runs once per iteration, and unrolled it is
// several times the 32 KB instruction cache.)
template <bool COH>
__device__ void mh_update_body(const ChainDev& d, const int c, int accept_mode, int propose_mode, int step,
                               const UpdLoop lp_ctx) {
  __shared__ double red[1 + 3 * BNN_MAX_OUT];
  __shared__ double sig[BNN_MAX_OUT];
  __shared__ double sh[32];
  __shared__ int s_flag;
  __shared__ int s_prop[BNN_MAX_LAYERS], s_cnt[BNN_MAX_LAYERS], s_off[BNN_MAX_LAYERS];
  // on-device generator (free-running chains): indicator moves decided by thread 0, flip probabilities for the block
  __shared__ int s_ind_move, s_fi_move;
  __shared__ double s_ind_p, s_fi_p;
  // the draws of this proposal (entry index, increment), generated once and used by the three owner passes
  int* didx_base;
  double* ddz_base;
  if constexpr (!COH) {
    __shared__ int st_didx[UPD_DRAW_CAP];
    __shared__ double st_ddz[UPD_DRAW_CAP];
    didx_base = st_didx; ddz_base = st_ddz;
  } else {
    didx_base = lp_ctx.didx_sm; ddz_base = lp_ctx.ddz_sm;
  }
  // Pre-proposal of the persistent loop (propose_mode 3, see below): what iteration s_pp_it will need and does not
  // depend on the pending accept decision -- layer choice, counts, accept uniform, indicator moves, the scalar Philox
  // blocks and (s_pp_draws) the proposal's draws in draw-cache buffer s_pp_it & 1
  __shared__ int s_pp_it, s_pp_draws;
  __shared__ int s_prop_n[BNN_MAX_LAYERS], s_cnt_n[BNN_MAX_LAYERS], s_off_n[BNN_MAX_LAYERS];
  __shared__ int s_ind_move_n, s_fi_move_n;
  __shared__ double s_ind_p_n, s_fi_p_n, s_logu_n;
  __shared__ uint4 s_px[BNN_MAX_LAYERS + 5], s_px_n[BNN_MAX_LAYERS + 5];
  const NetGeom& g = d.g;
  const int tid = threadIdx.x;
  const int NT = upd_nthreads<COH>();
  // The chain's scalar state is staged in shared memory for the whole launch: the accept / adapt / propose logic is
  // a serial chain of ~100 reads and writes by one thread, each of which would otherwise be an L2 round trip.
  __shared__ double ssf[BNN_F_STRIDE];
  __shared__ int ssi[BNN_I_STRIDE];
  double* const gsf = d.sf + (long long)c * BNN_F_STRIDE;
  int* const gsi = d.si + (long long)c * BNN_I_STRIDE;
  const bool resident = COH && lp_ctx.w_sm != nullptr;            // persistent loop: state stays in shared memory
  const bool load_state = !resident || lp_ctx.first, store_state = !resident || lp_ctx.last;
  double* wc = d.w_cur + (long long)c * g.P;
  double* wn = d.w_prop + (long long)c * g.P;
  int* owner = d.owner + (long long)c * g.P;
  if (load_state) {
    if (tid == 0) { s_pp_it = -1; s_pp_draws = 0; }          // nothing pre-proposed yet (visible after the barrier below)
#pragma unroll 1
    for (int i = tid; i < BNN_F_STRIDE; i += NT) ssf[i] = gsf[i];
#pragma unroll 1
    for (int i = tid; i < BNN_I_STRIDE; i += NT) ssi[i] = gsi[i];
    if (resident) {
#pragma unroll 1
      for (int i = tid; i < g.P; i += NT) {
        lp_ctx.w_sm[i] = wc[i];
        lp_ctx.w_sm[g.P + i] = wn[i];
        lp_ctx.owner_sm[i] = -1;
        const int l = layer_of(g, i);
        const LayerGeom& lg = g.l[l];
        const int cols = lg.in + lg.bias;
        lp_ctx.pk_sm[i] = (l << 24) | bnn_packed_index(lg, (i - lg.c_off) / cols, (i - lg.c_off) % cols);
      }
    }
    upd_sync<COH>();
  }
  if (resident) { wc = lp_ctx.w_sm; wn = lp_ctx.w_sm + g.P; owner = lp_ctx.owner_sm; }
  double* sf = ssf;
  int* si = ssi;
  auto write_back = [&]() {
    upd_sync<COH>();
    if (!store_state) return;
#pragma unroll 1
    for (int i = tid; i < BNN_F_STRIDE; i += NT) gsf[i] = ssf[i];
#pragma unroll 1
    for (int i = tid; i < BNN_I_STRIDE; i += NT) gsi[i] = ssi[i];
    if (resident) {
      double* gwc = d.w_cur + (long long)c * g.P;
      double* gwn = d.w_prop + (long long)c * g.P;
#pragma unroll 1
      for (int i = tid; i < g.P; i += NT) { gwc[i] = wc[i]; gwn[i] = wn[i]; }
    }
  };
  const int NC = bnn_n_counts(g.K);
  const int P0 = g.l[0].out * (g.l[0].in + g.l[0].bias);      // size of the first weight matrix (indicator shape)
  // The free-running generator's scalar draws of iteration it_x (layer choice, accept uniform, indicator / slope
  // moves) are independent Philox blocks: the lanes of warp 0 evaluate them side by side, thread 0 consumes them.
  //   slot l < L: layer uniforms | L: accept uniform | L+1: weight indicators | L+2: feature indicators | L+3, L+4: slopes
  auto scalar_blocks = [&](int it_x, uint4* px) {
    if (tid < g.L + 5) {
      const uint2 key = make_uint2((uint32_t)d.cfg.seed ^ (uint32_t)(d.cfg.chain_offset + c), (uint32_t)(d.cfg.seed >> 32));
      const int q = tid - g.L;
      uint4 ctr;
      if (q < 0) ctr = make_uint4((uint32_t)it_x, 0xFFFFFFFFu, (uint32_t)tid, 2u);
      else if (q == 0) ctr = make_uint4((uint32_t)it_x, 0xFFFFFFFEu, 0u, 3u);
      else if (q == 1) ctr = make_uint4((uint32_t)it_x, 0xFFFFFFFCu, 0u, 5u);
      else if (q == 2) ctr = make_uint4((uint32_t)it_x, 0xFFFFFFFBu, 0u, 6u);
      else ctr = make_uint4((uint32_t)it_x, 0xFFFFFFFDu, (uint32_t)(q - 3), 4u);
      px[tid] = philox4x32(ctr, key);
    }
    __syncwarp();
  };
  // thread 0: which layers iteration it_x proposes, how many entries, the indicator moves and log u, from the blocks
  // px and the CURRENT adaptation state (freq_layer_update, update_n, update_f)
  auto select_layers = [&](int it_x, const uint4* px, int* prop, int* cnt, int* off_out, int& ind_move, double& ind_p,
                           int& fi_move, double& fi_p, double& log_u) {
    // rr = rs.random(L); rr[argmin] = 0; layer proposed iff rr < freq_layer_update (BNN_env.py:446-451)
    double rr[BNN_MAX_LAYERS];
    int amin = 0, off = 0;
#pragma unroll 1
    for (int l = 0; l < g.L; ++l) {
      const uint4 r = px[l];
      rr[l] = u53(r.x, r.y);
      if (rr[l] < rr[amin]) amin = l;
    }
    rr[amin] = 0.0;
    // weight indicators (BNN_env.py:449-460): the first layer is proposed only if rr[0] >= freq_indicator, otherwise
    // its indicators move: UpdateBinomial(ind, update_f[3], shape) flips each entry with probability u * update_f[3]
    ind_move = 0;
    if (d.cfg.use_indicators && rr[0] < d.cfg.freq_indicator) {
      const uint4 r = px[g.L + 1];
      ind_move = 1;
      ind_p = u53(r.x, r.y) * ssf[BNN_F_UPDATE_F + 3];
    }
    // feature indicators (BNN_env.py:423-431): past adapt_stop, with probability 0.2, flips with probability u * 0.5
    fi_move = 0;
    if (d.cfg.use_feature_indicators && it_x > d.cfg.adapt_stop) {
      const uint4 r = px[g.L + 2];
      if (u53(r.x, r.y) < 0.2) { fi_move = 1; fi_p = u53(r.z, r.w) * 0.5; }
    }
#pragma unroll 1
    for (int l = 0; l < g.L; ++l) {
      prop[l] = rr[l] < ssf[BNN_F_FREQ_LAYER + l] && !(l == 0 && ind_move);
      cnt[l] = prop[l] ? ssi[BNN_I_UPDATE_N + l] : 0;
      off_out[l] = off;
      off += cnt[l];
    }
    const uint4 r = px[g.L];
    log_u = upd_log(u53(r.x, r.y));
  };
  // k-th draw of layer l at iteration it_x: canonical entry index and increment (device generator)
  auto philox_entry = [&](int it_x, int l, int k, int& idx, double& dz) {
    const LayerGeom& lg = g.l[l];
    const int cols = lg.in + lg.bias;
    const Draw dr = philox_draw(d.cfg.seed, d.cfg.chain_offset + c, it_x, l, k, lg.out, cols, ssf[BNN_F_UPDATE_WS + l]);
    idx = lg.c_off + dr.ix * cols + dr.iy;
    dz = dr.dz;
  };
  auto layer_of_j = [&](const int* off, const int* cnt, int j) {
    int l = 0;
#pragma unroll 1
    for (int q = 1; q < g.L; ++q) if (j >= off[q] && cnt[q] > 0) l = q;
    return l;
  };

  // ------------------------------------------------------------------ pre-proposal (persistent loop only)
  // Called by the leader's team while the other CTAs of the cluster are still in the forward pass of the current
  // proposal: everything iteration it + 1 needs that does not depend on the pending accept decision.  Skipped (and
  // recomputed on the critical path) when iteration it + 1 adapts the proposal sizes or the draws are injected.
  if (propose_mode == 3) {
    if constexpr (COH) {
      const int itn = ssi[BNN_I_ITERATION] + 1;
      const bool can = !d.inj_proposed && !(itn % d.cfg.adapt_freq == 0 && itn < d.cfg.adapt_stop);
      if (can) scalar_blocks(itn, s_px_n);
      if (tid == 0) {
        s_pp_it = -1;
        s_pp_draws = 0;
        if (can) {
          select_layers(itn, s_px_n, s_prop_n, s_cnt_n, s_off_n, s_ind_move_n, s_ind_p_n, s_fi_move_n, s_fi_p_n, s_logu_n);
          s_pp_it = itn;
        }
      }
      upd_sync<COH>();
      if (can) {
        const int nd = s_off_n[g.L - 1] + s_cnt_n[g.L - 1];
        if (nd <= UPD_DRAW_CAP) {
          int* di = didx_base + (itn & 1) * UPD_DRAW_CAP;
          double* dd = ddz_base + (itn & 1) * UPD_DRAW_CAP;
#pragma unroll 1
          for (int j = tid; j < nd; j += NT) {
            const int l = layer_of_j(s_off_n, s_cnt_n, j);
            philox_entry(itn, l, j - s_off_n[l], di[j], dd[j]);
          }
          if (tid == 0) s_pp_draws = 1;
        }
      }
      upd_sync<COH>();
    }
    return;
  }

  // ------------------------------------------------------------------ accept / reject
  if (accept_mode) {
    const bool smode_is_empirical = (accept_mode != 2) && d.cfg.sigma_mode == BNN_SIGMA_EMPIRICAL;
    // the initial likelihood of MCMC.__init__ always uses the stored error_prm (ones), even with
    // empirical_error=True (BNN_env.py:313-319); the empirical std only enters in mh_step (:475-476)
    const int smode = (accept_mode == 2) ? BNN_SIGMA_FIXED : d.cfg.sigma_mode;
    const double* sg_in = (g.lik == BNN_LIK_GAUSSIAN && smode == BNN_SIGMA_FIXED) ? sf + BNN_F_SIGMA : nullptr;
    const double* part_chain = lp_ctx.part_c ? lp_ctx.part_c : d.part + (long long)c * d.NF * d.n_tiles16;
    double ll = finalize_loglik<COH>(g, part_chain, d.NF, d.n_tiles16, d.n_train, d.cfg.lik_temp, smode, sg_in, red, sig);
    if (d.cfg.sample_from_prior) ll = 0.0;
    if (tid == 0) {
      double lp = sf[BNN_F_LOGPRIOR_PROP];
      double post = ll + lp;
      sf[BNN_F_LOGLIK_PROP] = ll;
      // accept iff (logPost' - logPost) * T + hastings >= log u   (BNN_env.py:493-494); NaN compares false
      int acc = (accept_mode == 2) ? 1 : (((post - sf[BNN_F_LOGPOST]) * sf[BNN_F_TEMPERATURE] + 0.0 >= sf[BNN_F_LOG_U]) ? 1 : 0);
      s_flag = acc;
      if (acc) {
        sf[BNN_F_LOGLIK] = ll; sf[BNN_F_LOGPRIOR] = lp; sf[BNN_F_LOGPOST] = post;
        // ActFun.reset_accepted_prm (BNN_env.py:502-503)
#pragma unroll 1
        for (int l = 0; l < g.L; ++l) sf[BNN_F_ALPHA + l] = sf[BNN_F_ALPHA_PROP + l];
      }
      if (accept_mode == 1) {
        si[BNN_I_LAST_ACCEPTED] = acc;
        si[BNN_I_N_ACCEPTED] += acc;
        // acceptance window (BNN_env.py:523-529): mean over the stored outcomes + the new one, then keep 100
        int len = si[BNN_I_RING_LEN], head = si[BNN_I_RING_HEAD], sum = si[BNN_I_RING_SUM];
        sf[BNN_F_ACC_RATE] = (double)(sum + acc) / (double)(len + 1);
        if (len < 100) {
          si[BNN_I_RING + (head + len) % 100] = acc;
          si[BNN_I_RING_LEN] = len + 1;
          si[BNN_I_RING_SUM] = sum + acc;
        } else {
          si[BNN_I_RING_SUM] = sum + acc - si[BNN_I_RING + head];
          si[BNN_I_RING + head] = acc;
          si[BNN_I_RING_HEAD] = (head + 1) % 100;
        }
        si[BNN_I_ITERATION] += 1;
      }
    }
    upd_sync<COH>();
    if (s_flag) {
#pragma unroll 1
      for (int i = tid; i < g.P; i += NT) wc[i] = wn[i];
      // reset_indicators / _feature_indicators on accept (BNN_env.py:497-499)
      if (d.ind_cur)
#pragma unroll 1
        for (int i = tid; i < P0; i += NT) d.ind_cur[(long long)c * P0 + i] = d.ind_prop[(long long)c * P0 + i];
      if (d.fi_cur)
#pragma unroll 1
        for (int i = tid; i < g.F; i += NT) d.fi_cur[(long long)c * g.F + i] = d.fi_prop[(long long)c * g.F + i];
      if (g.lik == BNN_LIK_CATEGORICAL) {
        // (COH: the counters were accumulated by other CTAs of this launch -- volatile generic loads)
        const volatile int* cp = lp_ctx.counts_c ? lp_ctx.counts_c : d.counts_prop + (long long)c * NC;
        if (tid < 2) si[BNN_I_N_CORRECT + tid] = cp[tid];
#pragma unroll 1
        for (int i = tid; i < g.K; i += NT) {
          si[BNN_I_CLASS_CORRECT + i] = cp[2 + i];
          si[BNN_I_PRED_HIST + i] = cp[2 + g.K + i];
        }
      } else {
#pragma unroll 1
        for (int i = tid; i < g.K; i += NT) {
          sf[BNN_F_SUM_R + i] = red[1 + i];
          sf[BNN_F_SUM_R2 + i] = red[1 + g.K + i];
          sf[BNN_F_SUM_R2_TEST + i] = red[1 + 2 * g.K + i];
          // reset_error_prm on accept, regression mode only (BNN_env.py:500-501)
          if (g.lik == BNN_LIK_GAUSSIAN && smode_is_empirical) sf[BNN_F_SIGMA + i] = sig[i];
        }
      }
    }
    upd_sync<COH>();
  }
  if (!propose_mode) { write_back(); return; }

  // ------------------------------------------------------------------ adaptation + which layers
  const int it = si[BNN_I_ITERATION];
  // pre-proposed during the previous forward pass (persistent loop)?  s_pp_it was written before the team's last barrier
  const bool use_pp = COH && resident && propose_mode == 1 && !d.inj_proposed && s_pp_it == it;
  const bool pp_draws = use_pp && s_pp_draws;
  if (propose_mode == 1 && !d.inj_proposed) {
    if (use_pp) { if (tid < g.L + 5) s_px[tid] = s_px_n[tid]; __syncwarp(); }
    else scalar_blocks(it, s_px);
  }
  if (tid == 0) {
    if (propose_mode == 1) {
      // BNN_env.py:392-413
      if (it % d.cfg.adapt_freq == 0 && it < d.cfg.adapt_stop) {
        double ar = sf[BNN_F_ACC_RATE];
        if (ar < d.cfg.adapt_f) {
#pragma unroll 1
          for (int l = 0; l < g.L; ++l) {
            sf[BNN_F_FREQ_LAYER + l] *= 0.8;
            sf[BNN_F_UPDATE_F + l] *= 0.85;
            int n = (int)((double)si[BNN_I_MAX_N + l] * sf[BNN_F_UPDATE_F + l]);
            si[BNN_I_UPDATE_N + l] = n < 1 ? 1 : n;
            sf[BNN_F_UPDATE_WS + l] *= 0.9;
          }
        }
        int tot = 0;
#pragma unroll 1
        for (int l = 0; l < g.L; ++l) tot += si[BNN_I_UPDATE_N + l];
        if (ar > d.cfg.adapt_fM && tot < g.P) {
#pragma unroll 1
          for (int l = 0; l < g.L; ++l) {
            sf[BNN_F_UPDATE_F + l] = exp(upd_log(sf[BNN_F_UPDATE_F + l]) * 0.85);
            int n = (int)((double)si[BNN_I_MAX_N + l] * sf[BNN_F_UPDATE_F + l]);
            si[BNN_I_UPDATE_N + l] = n < 1 ? 1 : n;
            sf[BNN_F_UPDATE_WS + l] *= 1.2;
          }
        }
      }
      if (d.inj_proposed) {
        int off = 0;
        const long long base = ((long long)step * d.C + c) * g.L;
#pragma unroll 1
        for (int l = 0; l < g.L; ++l) {
          s_prop[l] = d.inj_proposed[base + l];
          s_cnt[l] = s_prop[l] ? d.inj_count[base + l] : 0;
          s_off[l] = off;
          off += s_cnt[l];
        }
        sf[BNN_F_LOG_U] = d.inj_logu[(long long)step * d.C + c];
      } else {
        if (use_pp) {
#pragma unroll 1
          for (int l = 0; l < g.L; ++l) { s_prop[l] = s_prop_n[l]; s_cnt[l] = s_cnt_n[l]; s_off[l] = s_off_n[l]; }
          s_ind_move = s_ind_move_n; s_ind_p = s_ind_p_n; s_fi_move = s_fi_move_n; s_fi_p = s_fi_p_n;
          sf[BNN_F_LOG_U] = s_logu_n;
        } else {
          double log_u;
          select_layers(it, s_px, s_prop, s_cnt, s_off, s_ind_move, s_ind_p, s_fi_move, s_fi_p, log_u);
          sf[BNN_F_LOG_U] = log_u;
        }
      }
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) si[BNN_I_PROPOSED + l] = s_prop[l];
      // trainable activation parameters (BNN_env.py:416-421): UpdateNormal1D(_acc_prm, d=0.05, n=1, Mb=1, mb=0) with
      // the injected draw, both reflections over every entry (BNN_mcmc.py:46-56), Exp(10) term into additional_prob.
      // additional_prob itself: the injected value of this step, else the chain's device value, else 0
      double addp = d.inj_add_prob ? d.inj_add_prob[(long long)step * d.C + c] : (d.add_prob ? d.add_prob[c] : 0.0);
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) sf[BNN_F_ALPHA_PROP + l] = sf[BNN_F_ALPHA + l];
      if (d.cfg.n_act_prm > 0 && (d.inj_alpha_ix || !d.inj_proposed)) {
        int ix;
        double adz;
        if (d.inj_alpha_ix) {
          ix = d.inj_alpha_ix[(long long)step * d.C + c];
          adz = d.inj_alpha_dz[(long long)step * d.C + c];
        } else {                                          // rs.integers(0, n, 1), rs.normal(0, 0.05, 1) on the device
          const uint4 r = s_px[g.L + 3];
          ix = (int)__umulhi(r.x, (uint32_t)d.cfg.n_act_prm);
          const uint4 r2 = s_px[g.L + 4];
          adz = upd_gauss(0.05, 1.0 - u53(r2.x, r2.y), u53(r.y, r.z));
        }
        sf[BNN_F_ALPHA_PROP + ix] = sf[BNN_F_ALPHA + ix] + adz;
        double sum = 0.0;
#pragma unroll 1
        for (int l = 0; l < d.cfg.n_act_prm; ++l) {
          double z = sf[BNN_F_ALPHA_PROP + l];
          if (z > 1.0) z = 1.0 - (z - 1.0);
          if (z < 0.0) z = 0.0 + (0.0 - z);
          sf[BNN_F_ALPHA_PROP + l] = z;
          sum += z;
        }
        addp += 2.302585092994046 * (-sum) * 10.0;
      }
      sf[BNN_F_ADD_PROB] = addp;
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) d.alpha_fwd[(long long)c * g.L + l] = sf[BNN_F_ALPHA_PROP + l];
    } else {
      s_ind_move = 0; s_fi_move = 0;
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) { s_prop[l] = 0; s_cnt[l] = 0; s_off[l] = 0; }
      // initial state (MCMC.__init__, BNN_env.py:313-320): stored parameters, init_additional_prob
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) sf[BNN_F_ALPHA_PROP + l] = sf[BNN_F_ALPHA + l];
      sf[BNN_F_ADD_PROB] = d.cfg.init_additional_prob;
    }
  }
  // zero the proposal's counters (the forward kernel accumulates into them)
  if (g.lik == BNN_LIK_CATEGORICAL)
#pragma unroll 1
    for (int i = tid; i < NC; i += NT) (lp_ctx.counts_c ? lp_ctx.counts_c : d.counts_prop + (long long)c * NC)[i] = 0;
#pragma unroll 1
  for (int i = tid; i < g.P; i += NT) wn[i] = wc[i];
  // indicator proposals: UpdateBinomial = |ind - flip| with the injected flips (BNN_mcmc.py:98-99), else unchanged
  const double* ind_p = nullptr;
  const double* fi_p = nullptr;
  upd_sync<COH>();                                   // s_ind_move / s_fi_move and their probabilities are visible
  const bool gen_moves = propose_mode == 1 && !d.inj_proposed;          // free-running chains draw the flips here
  const uint2 fkey = make_uint2((uint32_t)d.cfg.seed ^ (uint32_t)(d.cfg.chain_offset + c), (uint32_t)(d.cfg.seed >> 32));
  if (d.ind_cur) {
    const long long sc = (long long)step * d.C + c;
    const bool mv = propose_mode == 1 && d.inj_ind_move && d.inj_ind_move[sc];
    double* dst = d.ind_prop + (long long)c * P0;
#pragma unroll 1
    for (int i = tid; i < P0; i += NT) {
      double v = d.ind_cur[(long long)c * P0 + i];
      bool flip = mv && d.inj_ind_flip[sc * P0 + i];
      if (gen_moves && s_ind_move) {
        const uint4 r = philox4x32(make_uint4((uint32_t)it, (uint32_t)i, 0u, 7u), fkey);
        flip = u53(r.x, r.y) < s_ind_p;
      }
      if (flip) v = fabs(v - 1.0);
      dst[i] = v;
    }
    ind_p = dst;
  }
  if (d.fi_cur) {
    const long long sc = (long long)step * d.C + c;
    const bool mv = propose_mode == 1 && d.inj_fi_move && d.inj_fi_move[sc];
    double* dst = d.fi_prop + (long long)c * g.F;
#pragma unroll 1
    for (int i = tid; i < g.F; i += NT) {
      double v = d.fi_cur[(long long)c * g.F + i];
      bool flip = mv && d.inj_fi_flip[sc * g.F + i];
      if (gen_moves && s_fi_move) {
        const uint4 r = philox4x32(make_uint4((uint32_t)it, (uint32_t)i, 0u, 8u), fkey);
        flip = u53(r.x, r.y) < s_fi_p;
      }
      if (flip) v = fabs(v - 1.0);
      dst[i] = v;
    }
    fi_p = dst;
  }
  if (d.ind_cur || d.fi_cur) upd_sync<COH>();

  // ------------------------------------------------------------------ UpdateNormal (BNN_mcmc.py:57-69)
  // z[Ix,Iy] = z[Ix,Iy] + N(0, d): fancy assignment => for duplicate (ix,iy) the LAST draw wins and
  // increments are not accumulated.  owner[idx] = largest draw index touching idx (per layer: the layers' entry
  // ranges are disjoint).  The draws are generated once into shared memory when they fit (UPD_DRAW_CAP).
  const long long inj_base = ((long long)step * d.C + c) * d.inj_cap;
  const int n_draws = s_off[g.L - 1] + s_cnt[g.L - 1];
  const bool cached = n_draws <= UPD_DRAW_CAP;
  // draw cache of this iteration (persistent loop: one buffer per iteration parity, so that the pre-proposal of the
  // next iteration never writes the buffer in use)
  int* s_didx = didx_base + (COH ? (it & 1) * UPD_DRAW_CAP : 0);
  double* s_ddz = ddz_base + (COH ? (it & 1) * UPD_DRAW_CAP : 0);
  auto make_draw = [&](int l, int k, int& idx, double& dz) {
    if (d.inj_proposed) {
      const LayerGeom& lg = g.l[l];
      const int cols = lg.in + lg.bias;
      idx = lg.c_off + d.inj_ix[inj_base + s_off[l] + k] * cols + d.inj_iy[inj_base + s_off[l] + k];
      dz = d.inj_dz[inj_base + s_off[l] + k];
    } else {
      philox_entry(it, l, k, idx, dz);
    }
  };
  // one flat loop over the draws of all layers (s_off are prefix sums of s_cnt): the draws of the small layers are
  // generated by other threads at the same time instead of in a loop of their own
  if (cached) {
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll 1
      for (int j = tid; j < n_draws; j += NT) {
        int idx;
        double dz;
        const int k = j - s_off[layer_of_j(s_off, s_cnt, j)];
        if (pass == 0 && !pp_draws) {
          make_draw(layer_of_j(s_off, s_cnt, j), k, idx, dz);
          s_didx[j] = idx; s_ddz[j] = dz;
        } else {
          idx = s_didx[j]; dz = s_ddz[j];
        }
        if (pass == 0) atomicMax(&owner[idx], k);
        else if (pass == 1) { if (owner[idx] == k) wn[idx] = wc[idx] + dz; }
        else owner[idx] = -1;
      }
      upd_sync<COH>();
    }
  } else {
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
#pragma unroll 1
      for (int l = 0; l < g.L; ++l) {
        if (!s_prop[l]) continue;
#pragma unroll 1
        for (int k = tid; k < s_cnt[l]; k += NT) {
          int idx;
          double dz;
          make_draw(l, k, idx, dz);
          if (pass == 0) atomicMax(&owner[idx], k);
          else if (pass == 1) { if (owner[idx] == k) wn[idx] = wc[idx] + dz; }
          else owner[idx] = -1;
        }
      }
      upd_sync<COH>();
    }
  }

  // ------------------------------------------------------------------ reflect, mask, prior, pack
  const double hi = d.cfg.w_bound, lo = -d.cfg.w_bound;
  double lp = 0.0;
  double* wpk = d.wp_prop + (long long)c * g.PB;
#pragma unroll 1
  for (int i = tid; i < g.P; i += NT) {
    // layer and packed position of the entry: from the table of the persistent loop, else computed
    int l, pi;
    if (resident) { const int v = lp_ctx.pk_sm[i]; l = v >> 24; pi = v & 0xffffff; }
    else {
      l = layer_of(g, i);
      const LayerGeom& lq = g.l[l];
      const int cols = lq.in + lq.bias;
      pi = bnn_packed_index(lq, (i - lq.c_off) / cols, (i - lq.c_off) % cols);
    }
    double z = wn[i];
    if (propose_mode == 1) {
      if (s_prop[l]) {                 // single reflection at the bounds (BNN_mcmc.py:66-67)
        if (z > hi) z = hi - (z - hi);
        if (z < lo) z = lo + (lo - z);
      }
      if (d.mask) z *= d.mask[i];      // w' *= mask for every layer (BNN_env.py:461-462)
      wn[i] = z;
    }
    if (d.cfg.prior != BNN_PRIOR_UNIFORM) {
      const long long e = (long long)c * g.P + i;
      lp += logpdf_prior(z, d.cfg.prior, d.ps_entry ? d.ps_entry[e] : d.ps.s[l], d.ps_entry ? d.pls_entry[e] : d.ps.ls[l]);
    }
    // the forward pass sees w0' * indicators' (BNN_env.py:463-466; the prior above does not), and a feature whose
    // indicator is 0 is replaced by its mean: its weight column leaves the contraction and enters the bias below
    if (l == 0 && ind_p) z *= ind_p[i];
    if (l == 0 && fi_p) {
      const LayerGeom& l0 = g.l[0];
      const int cc = (i - l0.c_off) % (l0.in + l0.bias);
      if (!(l0.bias && cc == 0) && fi_p[cc - l0.bias] == 0.0) z = 0.0;
    }
    wpk[pi] = z;
    if (lp_ctx.wpk_sm) lp_ctx.wpk_sm[pi] = z;
  }
  double s = block_sum_fixed<COH>(lp, sh);
  if (ind_p && d.cfg.use_indicators) {
    // + sum(ind) log(pi1) + (size - sum(ind)) log(1 - pi1)   (BNN_env.py:191-193)
    double n1 = 0.0;
#pragma unroll 1
    for (int i = tid; i < P0; i += NT) n1 += ind_p[i];
    n1 = block_sum_fixed<COH>(n1, sh);
    s += n1 * upd_log(d.cfg.prior_ind1) + ((double)P0 - n1) * upd_log(1.0 - d.cfg.prior_ind1);
  }
  if (fi_p) {
    // data_transform (BNN_env.py:14-17): x'[:, j] = mean_j where the feature indicator is 0, i.e. every first-layer
    // node gets the constant  sum_j mean_j * w0'[r, j] * ind'[r, j]  on top of its bias
    upd_sync<COH>();
    const LayerGeom& l0 = g.l[0];
    const int cols0 = l0.in + l0.bias;
#pragma unroll 1
    for (int r = tid; r < l0.out; r += NT) {
      double adj = 0.0;
#pragma unroll 1
      for (int j = 0; j < l0.in; ++j)
        if (fi_p[j] == 0.0) {
          const int e = r * cols0 + l0.bias + j;
          adj += d.feat_mean[j] * wn[e] * (ind_p ? ind_p[e] : 1.0);
        }
      const double b = l0.bias ? wn[r * cols0] * (ind_p ? ind_p[r * cols0] : 1.0) : 0.0;
      wpk[l0.b_off + r] = b + adj;
      if (lp_ctx.wpk_sm) lp_ctx.wpk_sm[l0.b_off + r] = b + adj;
    }
  }
  if (tid == 0) sf[BNN_F_LOGPRIOR_PROP] = s + sf[BNN_F_ADD_PROB];     // calc_prior(...) + additional_prob (BNN_env.py:481)
  write_back();
}
