// K2: proposal generation, log-prior, Metropolis-Hastings accept/reject and state commit, plus the
// small layout kernels (X / weight packing) and the deterministic reduction of the forward partials.
//
// Replaces (reference file:line): UpdateNormal (BNN_mcmc.py:57-69), the proposal / mask / prior /
// accept / adaptation / acceptance-window parts of MCMC.mh_step (BNN_env.py:392-413, 446-466, 481,
// 492-530) and npBNN.calc_prior (BNN_env.py:180-194).
#include "bnn_common.cuh"
#include "bnn_kernels.h"

#include "bnn_mh_body.cuh"


// ------------------------------------------------------------------------------------------------
// layout kernels
// ------------------------------------------------------------------------------------------------
// canonical X [n, F] -> swizzled, padded rows [n_pad16, F_pad]; optional column override (PDP)
__global__ void k_pack_x(const double* __restrict__ x, double* __restrict__ xs, long long n, long long n_pad, int F,
                         int F_pad, int swz, const int* __restrict__ ov_cols, const double* __restrict__ ov_vals,
                         int n_ov) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = n_pad * F_pad;
  if (i >= total) return;
  long long r = i / F_pad;
  int c = (int)(i % F_pad);
  double v = 0.0;
  if (r < n && c < F) {
    v = x[r * F + c];
    for (int k = 0; k < n_ov; ++k)
      if (ov_cols[k] == c) v = ov_vals[k];
  }
  xs[r * F_pad + (c ^ ((int)(r & 1) * swz))] = v;
}

// canonical weight sets [n_sets, P] -> packed [n_sets, PB] (padding entries are pre-zeroed, never written); one thread
// per entry of all sets (a 1-D grid: a set count in gridDim.y would stop at 65,535)
__global__ void k_pack_w(const __grid_constant__ NetGeom g, const double* __restrict__ w, double* __restrict__ wp,
                         long long n_entries) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries) return;
  const long long set = e / g.P;
  const int i = (int)(e - set * g.P);
  int l = layer_of(g, i);
  const LayerGeom& lg = g.l[l];
  int cols = lg.in + lg.bias;
  int r = (i - lg.c_off) / cols, cc = (i - lg.c_off) % cols;
  wp[set * g.PB + bnn_packed_index(lg, r, cc)] = w[e];
}


// stateless scoring: loglik / sums for bnn_forward_lik
__global__ void __launch_bounds__(UPD_THREADS) k_finalize_lik(const __grid_constant__ NetGeom g, const double* part,
                                                               int NF, long long nt, long long n_train,
                                                               double lik_temp, int sigma_mode, const double* sigma,
                                                               double* loglik, double* sums, int set0) {
  __shared__ double red[1 + 3 * BNN_MAX_OUT];
  __shared__ double sig[BNN_MAX_OUT];
  const int c = blockIdx.x;
  const double* sg = sigma ? sigma + (long long)(set0 + c) * g.K : nullptr;
  double ll = finalize_loglik(g, part + (long long)c * NF * nt, NF, nt, n_train, lik_temp, sigma_mode, sg, red, sig);
  if (threadIdx.x == 0) loglik[set0 + c] = ll;
  if (sums && g.lik != BNN_LIK_CATEGORICAL)
    for (int i = threadIdx.x; i < 3 * g.K; i += blockDim.x) sums[(long long)(set0 + c) * 3 * g.K + i] = red[1 + i];
}

// ps_entry / pls_entry: per-entry scales and their logs (hyper-priors: npBNN._prior_scale holds a vector per input
// node or a matrix per weight after sample_prior_scale, BNN_env.py:196-219), set `entry_stride` doubles apart
// (0: the same scales for every set); null: one scale per layer.
__global__ void __launch_bounds__(UPD_THREADS) k_log_prior(const __grid_constant__ NetGeom g, const double* w, int prior,
                                                            PriorScales ps, const double* ps_entry,
                                                            const double* pls_entry, int entry_stride, double* out) {
  __shared__ double sh[32];
  const int c = blockIdx.x;
  double v = 0.0;
  if (prior != BNN_PRIOR_UNIFORM)
    for (int i = threadIdx.x; i < g.P; i += blockDim.x) {
      int l = layer_of(g, i);
      const long long e = (long long)c * entry_stride + i;
      v += logpdf_prior(w[(long long)c * g.P + i], prior, ps_entry ? ps_entry[e] : ps.s[l], ps_entry ? pls_entry[e] : ps.ls[l]);
    }
  double s = block_sum_fixed(v, sh);
  if (threadIdx.x == 0) out[c] = s;
}

// MCMC.gibbs_step (BNN_env.py:534-538) after new prior scales: logPrior = calc_prior(), logPost = logLik + logPrior
// of the CURRENT weights of every chain.
__global__ void __launch_bounds__(UPD_THREADS) k_prior_refresh(const __grid_constant__ ChainDev d) {
  __shared__ double sh[32];
  const int c = blockIdx.x;
  const NetGeom& g = d.g;
  double v = 0.0;
  if (d.cfg.prior != BNN_PRIOR_UNIFORM)
    for (int i = threadIdx.x; i < g.P; i += blockDim.x) {
      int l = layer_of(g, i);
      const long long e = (long long)c * g.P + i;
      v += logpdf_prior(d.w_cur[e], d.cfg.prior, d.ps_entry ? d.ps_entry[e] : d.ps.s[l], d.ps_entry ? d.pls_entry[e] : d.ps.ls[l]);
    }
  double s = block_sum_fixed(v, sh);
  if (d.ind_cur && d.cfg.use_indicators) {
    // calc_prior's indicator term (BNN_env.py:191-193), as in k_mh_update: gibbs_step recomputes the whole log-prior
    const int P0 = g.l[0].out * (g.l[0].in + g.l[0].bias);
    const double* ind = d.ind_cur + (long long)c * P0;
    double n1 = 0.0;
    for (int i = threadIdx.x; i < P0; i += (int)blockDim.x) n1 += ind[i];
    n1 = block_sum_fixed(n1, sh);
    s += n1 * log(d.cfg.prior_ind1) + ((double)P0 - n1) * log(1.0 - d.cfg.prior_ind1);
  }
  if (threadIdx.x == 0) {
    double* sf = d.sf + (long long)c * BNN_F_STRIDE;
    sf[BNN_F_LOGPRIOR] = s;
    sf[BNN_F_LOGPOST] = sf[BNN_F_LOGLIK] + s;
  }
}

// one CTA per chain: [accept previous proposal] + [adapt, propose, prior, pack] (body: bnn_mh_body.cuh)
__global__ void __launch_bounds__(UPD_THREADS) k_mh_update(const __grid_constant__ ChainDev d, int accept_mode,
                                                            int propose_mode, int step) {
  mh_update_body<false>(d, blockIdx.x, accept_mode, propose_mode, step, UpdLoop{});
}


// ------------------------------------------------------------------------------------------------
// launch wrappers (called from bnn_capi.cu)
// ------------------------------------------------------------------------------------------------
// threads per CTA of the one-CTA-per-chain kernels: the per-entry loops want the full 1024 at c4 size (6,474 entries,
// 62,500 partials), while at a few hundred entries the block-wide synchronisations of 32 warps cost more than they save
// (a function of the network only, so that sharded and unsharded runs of the same chains reduce in the same order)
static inline int upd_threads(const NetGeom& g) { return g.P > 2048 ? 1024 : 256; }

cudaError_t bnn_launch_pack_x(const double* x, double* xs, long long n, long long n_pad, int F, int F_pad, int swz,
                              const int* ov_cols, const double* ov_vals, int n_ov, cudaStream_t st) {
  long long total = n_pad * F_pad;
  if (total == 0) return cudaSuccess;
  k_pack_x<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(x, xs, n, n_pad, F, F_pad, swz, ov_cols, ov_vals, n_ov);
  return cudaGetLastError();
}
cudaError_t bnn_launch_pack_w(const NetGeom& g, const double* w, double* wp, int n_sets, cudaStream_t st) {
  const long long n = (long long)n_sets * g.P;
  k_pack_w<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g, w, wp, n);
  return cudaGetLastError();
}
cudaError_t bnn_launch_finalize_lik(const NetGeom& g, const double* part, int NF, long long nt, long long n_train,
                                    double lik_temp, int sigma_mode, const double* sigma, double* loglik, double* sums,
                                    int set0, int n_sets, cudaStream_t st) {
  k_finalize_lik<<<n_sets, upd_threads(g), 0, st>>>(g, part, NF, nt, n_train, lik_temp, sigma_mode, sigma, loglik, sums, set0);
  return cudaGetLastError();
}
cudaError_t bnn_launch_log_prior(const NetGeom& g, const double* w, int n_sets, int prior, const PriorScales& ps,
                                 const double* ps_entry, const double* pls_entry, int entry_stride, double* out,
                                 cudaStream_t st) {
  k_log_prior<<<n_sets, upd_threads(g), 0, st>>>(g, w, prior, ps, ps_entry, pls_entry, entry_stride, out);
  return cudaGetLastError();
}
cudaError_t bnn_launch_prior_refresh(const ChainDev& d, cudaStream_t st) {
  k_prior_refresh<<<d.C, upd_threads(d.g), 0, st>>>(d);
  return cudaGetLastError();
}
// ------------------------------------------------------------------------------------------------
// row sharding (SURVEY.md 8e-2): the rows of X are split over the ranks, every rank runs the same chains.
// After the forward pass each rank reduces its per-tile partials to one vector per chain (k_rowshard_local, same
// fixed order as finalize_loglik); the vectors are summed over the ranks (one all-reduce of C * (NF + 2 + 2K)
// doubles); k_rowshard_commit stores the sums where k_mh_update expects partials of a single tile, so the accept
// step runs unchanged and every rank takes the same decision.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(UPD_THREADS) k_rowshard_local(const double* __restrict__ part, int NF, long long nt,
                                                                 const int* __restrict__ counts, int NC,
                                                                 double* __restrict__ out) {
  __shared__ double sh[32];
  const int c = blockIdx.x;
  for (int slot = 0; slot < NF; ++slot) {
    const double* src = part + ((long long)c * NF + slot) * nt;
    const double v = strided_sum_ordered(src, nt);
    const double s = block_sum_fixed(v, sh);
    if (threadIdx.x == 0) out[(long long)c * (NF + NC) + slot] = s;
  }
  for (int i = threadIdx.x; i < NC; i += blockDim.x)
    out[(long long)c * (NF + NC) + NF + i] = counts ? (double)counts[(long long)c * NC + i] : 0.0;
}
__global__ void k_rowshard_commit(const double* __restrict__ in, int NF, int NC, double* __restrict__ part_red,
                                  int* __restrict__ counts) {
  const int c = blockIdx.x;
  for (int i = threadIdx.x; i < NF; i += blockDim.x) part_red[(long long)c * NF + i] = in[(long long)c * (NF + NC) + i];
  if (counts)
    for (int i = threadIdx.x; i < NC; i += blockDim.x)
      counts[(long long)c * NC + i] = (int)llrint(in[(long long)c * (NF + NC) + NF + i]);    // exact: integer-valued sums
}
cudaError_t bnn_launch_rowshard_local(const NetGeom& g, const double* part, int NF, long long nt, const int* counts, int NC,
                                      double* out, int n_chains, cudaStream_t st) {
  k_rowshard_local<<<n_chains, upd_threads(g), 0, st>>>(part, NF, nt, counts, NC, out);
  return cudaGetLastError();
}
cudaError_t bnn_launch_rowshard_commit(const double* in, int NF, int NC, double* part_red, int* counts, int n_chains,
                                       cudaStream_t st) {
  k_rowshard_commit<<<n_chains, 64, 0, st>>>(in, NF, NC, part_red, counts);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// First level of the partial-sum reduction.  The forward kernels leave one partial per (chain, slot, 16-row tile):
// 62,500 per chain at 1M rows, which k_mh_update -- one CTA per chain -- used to fold alone (18.5 MB through 32 SMs,
// 40 us per step, 2-3 % of a step at 4 chains per GPU).  Here C * NF * n_slices CTAs fold fixed slices of the tile
// axis in a fixed order (thread-strided terms, then the fixed block tree), so k_mh_update reads n_slices values per
// chain.  The slice boundaries depend on the tile count only: the result does not depend on how the forward kernel
// dealt its tiles out, nor on the number of chains in the pass.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_reduce_part(const double* __restrict__ part, long long nt, int n_slices,
                                                      double* __restrict__ out) {
  __shared__ double sh[32];
  const int slice = blockIdx.x;
  const long long cs = blockIdx.y;                       // chain * NF + slot
  const long long per = (nt + n_slices - 1) / n_slices;
  const long long a = slice * per;
  long long b = a + per;
  if (b > nt) b = nt;
  const double v = (a < b) ? strided_sum_ordered(part + cs * nt + a, b - a) : 0.0;
  const double s = block_sum_fixed(v, sh);
  if (threadIdx.x == 0) out[cs * n_slices + slice] = s;
}

int bnn_part_slices(long long nt) {
  if (nt < 4096) return 0;                               // small data sets: k_mh_update reads the tile partials itself
  long long s = nt / 1024;
  return (int)(s > 64 ? 64 : s);
}

cudaError_t bnn_launch_reduce_part(const double* part, long long nt, int n_slices, int n_rows, double* out, cudaStream_t st) {
  dim3 grid((unsigned)n_slices, (unsigned)n_rows);
  k_reduce_part<<<grid, 256, 0, st>>>(part, nt, n_slices, out);
  return cudaGetLastError();
}

cudaError_t bnn_launch_mh_update(const ChainDev& d, int accept_mode, int propose_mode, int step, cudaStream_t st) {
  k_mh_update<<<d.C, upd_threads(d.g), 0, st>>>(d, accept_mode, propose_mode, step);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// FP64 peak probe (same loop as tools/peak_fp64.cu, m16n8k8): 8 independent accumulators per warp
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dmma_peak(double* out, int iters) {
  double c[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = c[i][2] = c[i][3] = 0.0;
  const double a0 = 1.0 + threadIdx.x * 1e-6, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3;
  const double b0 = 1e-9 + threadIdx.x * 1e-12, b1 = b0 * 2;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) dmma16x8x8(c[i], a0, a1, a2, a3, b0, b1);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1] + c[i][2] + c[i][3];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// Labels index the class-probability row, the class weights and the per-class counters inside the forward epilogues
// (prediction[sample_id, labels], BNN_lib.py:104): a label outside [0, K) is an IndexError in the reference and would be
// an out-of-bounds access here, so bnn_set_data rejects it.
__global__ void k_check_labels(const int* __restrict__ labels, long long n_train, long long n_total, int K, int* flag) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  int bad = 0;
  for (; i < n_total; i += stride) {
    const int y = labels[i];
    bad |= (y < 0) || (y >= K);      // test labels feed the same counters (argmax == label), same range
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

cudaError_t bnn_launch_check_labels(const int* labels, long long n_train, long long n_total, int K, int* flag, cudaStream_t st) {
  long long blocks = (n_total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_check_labels<<<(int)blocks, 256, 0, st>>>(labels, n_train, n_total, K, flag);
  return cudaGetLastError();
}

// gammaln(k + 1) of the count likelihoods (BNN_lik.py:5-66) depends on the labels only
__global__ void k_lgamma1(const double* __restrict__ k, double* __restrict__ out, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = lgamma(k[i] + 1.0);
}

cudaError_t bnn_launch_lgamma1(const double* k, double* out, long long n, cudaStream_t st) {
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  k_lgamma1<<<(int)blocks, 256, 0, st>>>(k, out, n);
  return cudaGetLastError();
}

cudaError_t bnn_measure_dmma_peak(int n_sms, double* tflops) {
  const int grid = n_sms * 2, threads = 256, iters = 2048;
  double* out = nullptr;
  cudaError_t e = cudaMalloc(&out, sizeof(double) * grid * threads);
  if (e != cudaSuccess) return e;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int w = 0; w < 3; ++w) k_dmma_peak<<<grid, threads>>>(out, iters);
  double best = 1e30;
  for (int r = 0; r < 5; ++r) {
    cudaEventRecord(e0);
    k_dmma_peak<<<grid, threads>>>(out, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  e = cudaGetLastError();
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  if (e != cudaSuccess) return e;
  const double flops = 2.0 * 16 * 8 * 8 * (double)iters * 4 * 8 * (grid * threads / 32);
  *tflops = flops / (best * 1e-3) / 1e12;
  return cudaSuccess;
}
