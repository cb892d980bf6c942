// Internal interface between the kernel translation units and the C-ABI layer (bnn_capi.cu).
#pragma once
#include <type_traits>
#include <vector>
#include "bnn_common.cuh"

// Most dynamic shared memory a block of sm_100 may opt in to (227 KB).
constexpr int BNN_MAX_DYN_SMEM = 232448;

// Lets kernel `fn` use up to max_dyn_smem bytes of dynamic shared memory (and non-portable cluster sizes, if asked) on
// the current device.  Function attributes belong to a device's context, so they are set once per (kernel, device);
// safe when several host threads launch at once.
cudaError_t bnn_prepare_kernel(const void* fn, int max_dyn_smem, bool nonportable_cluster = false);

// f(std::integral_constant<int, ACT>{}) for the run-time activation `act`: where launchers pick a kernel's ACT.
template <typename F>
inline auto bnn_with_act(int act, F&& f) {
  switch (act) {
    case BNN_ACT_RELU: return f(std::integral_constant<int, BNN_ACT_RELU>{});
    case BNN_ACT_LEAKY: return f(std::integral_constant<int, BNN_ACT_LEAKY>{});
    case BNN_ACT_SWISH: return f(std::integral_constant<int, BNN_ACT_SWISH>{});
    default: return f(std::integral_constant<int, BNN_ACT_TANH>{});
  }
}

struct PriorScales {
  double s[BNN_MAX_LAYERS];    // npBNN._prior_scale
  double ls[BNN_MAX_LAYERS];   // log of it
};

// Device-resident state of C chains (DESIGN.md section 3).
struct ChainDev {
  NetGeom g;
  bnn_sampler_config cfg;
  PriorScales ps;
  int C;
  long long n_train, n_tiles16;
  double* w_cur;        // [C, P] canonical current weights
  double* w_prop;       // [C, P] canonical proposal
  double* wp_prop;      // [C, PB] packed proposal (input of the forward kernel)
  const double* mask;   // [P] or null
  const double* ps_entry;   // [C, P] per-entry prior scales (hyper-priors, BNN_env.py:196-219) or null
  const double* pls_entry;  // [C, P] their logarithms
  int* owner;           // [C, P] scratch for last-write-wins, all -1 between launches
  double* sf;           // [C, BNN_F_STRIDE]
  int* si;              // [C, BNN_I_STRIDE]
  const double* part;   // forward partials [C, NF, n_tiles16]
  int NF;
  int* counts_prop;     // [C, bnn_n_counts(K)]
  // injected draws of the current bnn_mh_steps call (device copies) or null
  const int* inj_proposed;
  const int* inj_count;
  const int* inj_ix;
  const int* inj_iy;
  const double* inj_dz;
  const double* inj_logu;
  int inj_cap;
  const int* inj_alpha_ix;    // [n_steps, C] or null
  const double* inj_alpha_dz;
  const double* inj_add_prob; // [n_steps, C] or null
  double* alpha_fwd;          // [C, L] slopes the forward kernel reads (= the proposal's)
  // indicators (null = absent): current / proposed weight indicators [C, P0], feature indicators [C, F]
  double* ind_cur;
  double* ind_prop;
  double* fi_cur;
  double* fi_prop;
  const double* feat_mean;    // [F]
  const int* inj_ind_move;    // [n_steps, C] or null
  const uint8_t* inj_ind_flip;
  const int* inj_fi_move;
  const uint8_t* inj_fi_flip;
  // additional_prob of every chain when no injection carries one ([C], bnn_chains_set_additional_prob) or null (0).
  // Appended, so that the offsets of the fields above stay those of the kernels that do not read it.
  const double* add_prob;
};

cudaError_t bnn_launch_forward(const FwdParams& p, bool predict, int n_sms, int force_generic, cudaStream_t st,
                               const char** which);
// Block-masked networks (bnn_sparse.cu).  bnn_sparse_build writes the dataflow program of `mask` and its FwdParams::sp
// (device pointers null) to *out; false: the dense kernels run instead (the block cover is not thin enough, or the
// program does not fit the kernels' shared memory).  bnn_launch_sparse runs the program in p.sp; *which = its kernel.
struct SparseProgram {
  std::vector<int> prog, widx;    // program ints, weight-index stream
  SparseParams sp;
};
bool bnn_sparse_build(const NetGeom& g, const double* mask, SparseProgram* out);
cudaError_t bnn_launch_sparse(const FwdParams& p, int n_sms, cudaStream_t st, const char** which);
// Prediction mode of the same program (mean / votes / dense / resampling outputs of FwdParams): thread = row, the sets
// of the launch summed in order 0 ... C-1.  bnn_sparse_predict_fits: the program fits the prediction kernel's shared
// memory.  bnn_launch_mask_violations: *flag = 1 if an entry that `mask` [P] drops is nonzero in a canonical set of w.
bool bnn_sparse_predict_fits(const FwdParams& p);
cudaError_t bnn_launch_sparse_predict(const FwdParams& p, int n_sms, cudaStream_t st, const char** which);
cudaError_t bnn_launch_mask_violations(const double* w, int n_sets, int P, const double* mask, int* flag, int n_sms,
                                       cudaStream_t st);
// opt-in reduced-precision posterior prediction (bnn_pred_lp.cu): 3xTF32 (passes = 3) or TF32 (passes = 1) tensor-core
// contractions, FP32 activations / softmax / softplus, FP64 accumulation over the samples in set order.  Summaries
// (mean / votes) and resampling of every dense network: k_pred_tf32x3 for the 64-64-32-16 categorical family,
// k_pred_tf32_generic for the others.  bnn_pred_tf32_fits: the call is one of those (no dense tensor, no block-sparse
// program) and not of the shape class measured slower than FP64 at that pass count.  The launcher converts the packed
// weight sets in p.wp to (hi, lo) TF32 pairs in place.
bool bnn_pred_tf32_fits(const FwdParams& p, int passes);
cudaError_t bnn_launch_pred_tf32(const FwdParams& p, int n_sms, int passes, cudaStream_t st, const char** which);
// Dynamic shared memory of a k_fwd_generic CTA of `warps` warps running C sets (likelihood) or posterior prediction, and
// the most warps (4, 2, 1) whose CTA fits BNN_MAX_DYN_SMEM: 0 when none does (the network is too wide for the kernel)
size_t bnn_generic_smem_bytes(const NetGeom& g, int C, bool predict, int warps);
int bnn_generic_warps(const NetGeom& g, int C, bool predict);
// k_fwd3 width family the padded geometry matches exactly: 1 = 64->64->32, 2 = 32->32->16, 0 = none (generic kernel)
int bnn_fwd3_family(const NetGeom& g);
// kernels bnn_launch_forward enqueues for these parameters (the int8 first layer adds the slicing of W1)
int bnn_forward_launches(const FwdParams& p, bool predict, int force_generic);
// 64 -> 64 -> 32 family: out[k] = largest |x| of feature k over the n staged rows (NaN if one is not finite),
// out[64 + k] = its nonzero entries, out[128 + k] = its nonzero entries of at least 2^-6 out[k]; then the rows divided by wmul [64] as the base-256 digits and row scales the
// likelihood kernel k_fwd3i reads (FwdParams::x_i8 / x_i8_scale), sized for bnn_i8_blocks(n_tiles16) blocks of 128 rows
inline long long bnn_i8_blocks(long long n_tiles16) { return (n_tiles16 + 7) / 8; }
cudaError_t bnn_launch_feature_stats(const double* xs, long long n, int swz, double* out, cudaStream_t st);
cudaError_t bnn_launch_slice_x(const double* xs, long long n_pad16, int swz, const double* wmul, int8_t* x_i8,
                               double* x_i8_scale, cudaStream_t st);
cudaError_t bnn_launch_pack_x(const double* x, double* xs, long long n, long long n_pad, int F, int F_pad, int swz,
                              const int* ov_cols, const double* ov_vals, int n_ov, cudaStream_t st);
// *flag |= 1 if a training label is outside [0, K) or a test label is negative (the reference raises IndexError there)
cudaError_t bnn_launch_check_labels(const int* labels, long long n_train, long long n_total, int K, int* flag, cudaStream_t st);
// out[i] = lgamma(k[i] + 1): the label-only term of the count likelihoods, once per data set
cudaError_t bnn_launch_lgamma1(const double* k, double* out, long long n, cudaStream_t st);
cudaError_t bnn_launch_pack_w(const NetGeom& g, const double* w, double* wp, int n_sets, cudaStream_t st);
cudaError_t bnn_launch_finalize_lik(const NetGeom& g, const double* part, int NF, long long nt, long long n_train,
                                    double lik_temp, int sigma_mode, const double* sigma, double* loglik, double* sums,
                                    int set0, int n_sets, cudaStream_t st);
cudaError_t bnn_launch_log_prior(const NetGeom& g, const double* w, int n_sets, int prior, const PriorScales& ps,
                                 const double* ps_entry, const double* pls_entry, int entry_stride, double* out,
                                 cudaStream_t st);
cudaError_t bnn_launch_prior_refresh(const ChainDev& d, cudaStream_t st);
// first-level reduction of the per-tile partials: part [n_rows, nt] -> out [n_rows, n_slices]; bnn_part_slices(nt) = 0
// means "not worth a launch" (k_mh_update reads the tile partials directly)
int bnn_part_slices(long long nt);
cudaError_t bnn_launch_reduce_part(const double* part, long long nt, int n_slices, int n_rows, double* out, cudaStream_t st);
cudaError_t bnn_launch_mh_update(const ChainDev& d, int accept_mode, int propose_mode, int step, cudaStream_t st);
// persistent small-data MH loop (bnn_chainloop.cu): n_steps iterations of every chain in one launch, one thread-block
// cluster per chain; cudaErrorNotSupported when the problem does not fit (bnn_chain_loop_fits)
bool bnn_chain_loop_fits(const NetGeom& g, int NF, long long nt, int C, int n_sms, int max_cluster, int mode);
cudaError_t bnn_launch_chain_loop(const ChainDev& d, const FwdParams& p, int n_steps, int n_sms, int max_cluster, int mode,
                                  cudaStream_t st, int* cluster_out);
cudaError_t bnn_launch_rowshard_local(const NetGeom& g, const double* part, int NF, long long nt, const int* counts, int NC,
                                      double* out, int n_chains, cudaStream_t st);
cudaError_t bnn_launch_rowshard_commit(const double* in, int NF, int NC, double* part_red, int* counts, int n_chains,
                                       cudaStream_t st);
// FP64 tensor-pipe peak (back-to-back DMMA, no memory traffic): the roofline denominator of the forward kernel
cudaError_t bnn_measure_dmma_peak(int n_sms, double* tflops);
