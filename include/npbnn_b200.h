/* npbnn_b200 -- C ABI of the B200-native npBNN Metropolis-Hastings hot path.
 *
 * The reference (dsilvestro/npBNN) is pure Python and has no FFI layer; its boundary is the
 * Python call surface of np_bnn/__init__.py:6-25.  The entry points below are what a ctypes
 * binding inside the reference would call in place of its numpy code (INTEGRATION.md shows
 * the stub).  Each entry point names the reference code it replaces (file:line into the
 * reference tree).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; bnn_last_error() gives the text
 *   - `*_dev` pointers are CUDA device pointers (e.g. torch.Tensor.data_ptr()); `*_host`
 *     pointers are host pointers (pinned memory gives asynchronous copies)
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream)
 *   - no ownership transfer: the context owns only its internal workspace
 *   - weights use the reference's canonical layout: layer l is a row-major
 *     [out_l, in_l + has_bias_l] float64 matrix, bias in column 0 (BNN_lib.py:154-162);
 *     a weight set is the concatenation of its layers (`n_params` doubles)
 */
#ifndef NPBNN_B200_H
#define NPBNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNN_ABI_VERSION 2
#define BNN_MAX_LAYERS 8
#define BNN_MAX_OUT 32          /* max width of the output layer (classes, or 2*O for the sigma head) */

/* activation of the hidden layers: relu_f / leaky_relu_f / swish_f / tanh_f, BNN_lib.py:50-66 */
enum { BNN_ACT_RELU = 0, BNN_ACT_LEAKY = 1, BNN_ACT_SWISH = 2, BNN_ACT_TANH = 3 };
/* output transform + likelihood:
 *   CATEGORICAL   SoftMax (BNN_lib.py:166-168) + calc_likelihood (BNN_lib.py:100-121)
 *   GAUSSIAN      RegressTransform (BNN_lib.py:174) + calc_likelihood_regression (BNN_lib.py:123-131)
 *   GAUSSIAN_HEAD RegressTransformError (BNN_lib.py:177-182) + calc_likelihood_regression_error (:134-143)
 * count data (estimation_mode="custom", RegressTransform outputs z, counts k; lik_temp is not applied, as there):
 *   POISSON       poi_likelihood (BNN_lik.py:5-14): sum xlogy(k, exp(z0)) - gammaln(k+1) - exp(z0); K = 1 modelled
 *                 column (output column 0), any output width
 *   NEGBIN        negbin_likelihood / negbin_likelihood2d (BNN_lik.py:16-50): per modelled column j < K = O/2,
 *                 nbinom.logpmf(k_j; n, p) with mean = exp(z_j), p = 1/(1+exp(-z_{K+j})), n = p mean/(1-p); even O
 *   NEGBIN10      negbin_likelihood_base10 (BNN_lik.py:52-66): NEGBIN with 10** in place of exp
 * For the count kinds the residual sums (sums_dev, BNN_F_SUM_R*) are of r = mean - k (mean = exp(z0), 10**z0):
 * poi_acc / negbin_acc / negbin2d_acc / negbin_acc_base10 = sum r^2 / (N K). */
enum { BNN_LIK_CATEGORICAL = 0, BNN_LIK_GAUSSIAN = 1, BNN_LIK_GAUSSIAN_HEAD = 2,
       BNN_LIK_POISSON = 3, BNN_LIK_NEGBIN = 4, BNN_LIK_NEGBIN10 = 5 };
/* npBNN prior_f, BNN_env.py:135-150 */
enum { BNN_PRIOR_UNIFORM = 0, BNN_PRIOR_NORMAL = 1, BNN_PRIOR_CAUCHY = 2, BNN_PRIOR_LAPLACE = 3 };
/* error parameter of the Gaussian likelihood: fixed sigma[O] per chain, or the population std of the
 * residuals recomputed for every proposal (empirical_error, BNN_env.py:475-476) */
enum { BNN_SIGMA_FIXED = 0, BNN_SIGMA_EMPIRICAL = 1 };
/* posterior summary of bnn_predict: argmax vote share / mean (get_posterior_cat_prob modes 0 / 1,
 * BNN_lib.py:382-392) */
enum { BNN_SUMMARY_VOTES = 1, BNN_SUMMARY_MEAN = 2, BNN_SUMMARY_DENSE = 4 };

typedef struct bnn_ctx bnn_ctx;

/* Network shape: what init_weight_prm (BNN_mcmc.py:9-25) and ActFun (BNN_lib.py:68-94) fix. */
typedef struct {
  int32_t n_layers;                    /* hidden layers + 1 */
  int32_t n_features;
  int32_t out_dim[BNN_MAX_LAYERS];     /* rows of each weight matrix */
  int32_t has_bias[BNN_MAX_LAYERS];    /* 1 if column 0 of that matrix is a bias */
  int32_t act;                         /* BNN_ACT_* */
  int32_t lik;                         /* BNN_LIK_* */
} bnn_net_spec;

/* Sampler configuration shared by all chains of a context: the constructor arguments of MCMC
 * (BNN_env.py:274-281) and the prior fields of npBNN (BNN_env.py:85-154). */
typedef struct {
  int32_t prior;                       /* BNN_PRIOR_* */
  int32_t sigma_mode;                  /* BNN_SIGMA_* (Gaussian likelihood only) */
  int32_t sample_from_prior;           /* MCMC(sample_from_prior=) : likelihood forced to 0 */
  int32_t adapt_freq;                  /* MCMC(adapt_freq=) */
  int32_t adapt_stop;                  /* MCMC(adapt_stop=), already resolved (int(0.05 n_iter) default) */
  int32_t use_mask;                    /* mask_dev given to bnn_chains_init */
  double adapt_f, adapt_fM;            /* MCMC(adapt_f=, adapt_fM=) */
  double lik_temp;                     /* MCMC(likelihood_tempering=) */
  double w_bound;                      /* npBNN._w_bound (inf = no reflection) */
  double prior_scale[BNN_MAX_LAYERS];  /* npBNN._prior_scale (one scalar per layer) */
  uint64_t seed;                       /* Philox key for free-running proposals */
  int32_t n_act_prm;                   /* ActFun(trainable=True): number of activation parameters (len(_acc_prm)); 0 = fixed */
  int32_t chain_offset;                /* global index of this context's first chain: the Philox key is seed ^ (chain_offset + c),
                                        * so chain blocks on different ranks (MC3 sharding) draw different streams from one seed */
  double init_additional_prob;         /* MCMC(init_additional_prob=): added to the initial log-prior (BNN_env.py:320) */
  /* indicators (appended; zero = absent).  Weight indicators: npBNN(freq_indicator > 0): a 0/1 matrix of the shape of
   * the first weight matrix multiplies it in the forward pass only, and calc_prior adds
   * sum(ind) log(prior_ind1) + (size - sum(ind)) log(1 - prior_ind1) (BNN_env.py:191-193,458-466).  Feature
   * indicators: npBNN(feature_indicators=True): features whose indicator is 0 are replaced by their training mean
   * (data_transform_obj, BNN_env.py:9-17,423-431; means given by bnn_set_feature_means).  Both start as all ones. */
  double prior_ind1;
  int32_t use_indicators;
  int32_t use_feature_indicators;
  /* npBNN(freq_indicator=): probability threshold of the weight-indicator move (BNN_env.py:449-460).  Only read by the
   * on-device generator (free-running chains); with injected draws the host decides the move (bnn_injection.ind_move). */
  double freq_indicator;
} bnn_sampler_config;

/* Random draws of `n_steps` MH iterations for every chain, recorded from (or generated like) the
 * reference's generator calls in BNN_env.py:446-453,493 and BNN_mcmc.py:62-65.  All host pointers.
 *   proposed [n_steps, C, L]        1 if the layer is proposed in that step
 *   count    [n_steps, C, L]        number of (ix, iy, dz) triples of that layer (= update_n)
 *   ix, iy   [n_steps, C, cap]      row / column indices, layers concatenated in order
 *   dz       [n_steps, C, cap]      the normal increments (already scaled by update_ws)
 *   log_u    [n_steps, C]           log of the accept uniform
 * With trainable activation parameters (n_act_prm > 0) alpha_ix / alpha_dz are required: the proposal
 * prm' = reflect_[0,1](prm + dz e_ix) enters the forward pass (genReLU slopes) and the log-prior through
 * additional_prob = log(10) * (-sum(prm')) * 10 (BNN_env.py:416-421); it is committed on accept. */
typedef struct {
  int32_t n_steps;
  int32_t cap;
  const int32_t* proposed;
  const int32_t* count;
  const int32_t* ix;
  const int32_t* iy;
  const double* dz;
  const double* log_u;
  /* optional draws of the branches that precede the layer proposals in mh_step (BNN_env.py:416-444); NULL = absent */
  const int32_t* alpha_ix;   /* [n_steps, C] index drawn by UpdateNormal1D(_acc_prm, d=0.05, n=1, Mb=1, mb=0) (BNN_mcmc.py:46-56) */
  const double* alpha_dz;    /* [n_steps, C] its normal increment */
  const double* add_prob;    /* [n_steps, C] the additional_prob argument of mh_step */
  /* indicator moves (appended; NULL = none in this call).  UpdateBinomial (BNN_mcmc.py:98-99) is
   * |ind - binomial(1, u * update_f, shape)|: the host draws the 0/1 flip matrices with the reference's generator, the
   * device applies them to the chain's current indicators.  ind_move[s, c] = 1: step s of chain c flips the weight
   * indicators (its layer 0 is then not proposed, BNN_env.py:449-460); fi_move likewise for the feature indicators. */
  const int32_t* ind_move;   /* [n_steps, C] */
  const uint8_t* ind_flip;   /* [n_steps, C, size of the first weight matrix] */
  const int32_t* fi_move;    /* [n_steps, C] */
  const uint8_t* fi_flip;    /* [n_steps, C, n_features] */
} bnn_injection;

/* ---- per-chain state export (bnn_chains_read): slot indices ------------------------------------ */
enum {
  BNN_F_LOGLIK = 0, BNN_F_LOGPRIOR = 1, BNN_F_LOGPOST = 2, BNN_F_TEMPERATURE = 3, BNN_F_ACC_RATE = 4,
  BNN_F_LOGLIK_PROP = 5, BNN_F_LOGPRIOR_PROP = 6, BNN_F_LOG_U = 7,
  BNN_F_ADD_PROB = 8,            /* additional_prob of the current proposal (part of BNN_F_LOGPRIOR_PROP) */
  BNN_F_UPDATE_F = 16,           /* [BNN_MAX_LAYERS] */
  BNN_F_UPDATE_WS = 24,          /* [BNN_MAX_LAYERS] */
  BNN_F_FREQ_LAYER = 32,         /* [BNN_MAX_LAYERS] */
  BNN_F_ALPHA = 40,              /* [BNN_MAX_LAYERS] genReLU slopes = accepted activation parameters (_acc_prm) */
  BNN_F_SIGMA = 48,              /* [BNN_MAX_OUT] current error_prm */
  BNN_F_SUM_R = 80,              /* [BNN_MAX_OUT] current sum of residuals (train) */
  BNN_F_SUM_R2 = 112,            /* [BNN_MAX_OUT] current sum of squared residuals (train) */
  BNN_F_SUM_R2_TEST = 144,       /* [BNN_MAX_OUT] current sum of squared residuals (test) */
  BNN_F_ALPHA_PROP = 176,        /* [BNN_MAX_LAYERS] proposed activation parameters (_prm) */
  BNN_F_STRIDE = 192
};
enum {
  BNN_I_ITERATION = 0, BNN_I_LAST_ACCEPTED = 1, BNN_I_N_ACCEPTED = 2, BNN_I_RING_LEN = 3, BNN_I_RING_HEAD = 4,
  BNN_I_RING_SUM = 5,
  BNN_I_UPDATE_N = 8,            /* [BNN_MAX_LAYERS] */
  BNN_I_MAX_N = 16,              /* [BNN_MAX_LAYERS] */
  BNN_I_PROPOSED = 24,           /* [BNN_MAX_LAYERS] layers proposed in the last step */
  BNN_I_N_CORRECT = 32, BNN_I_N_CORRECT_TEST = 33,
  BNN_I_CLASS_CORRECT = 34,      /* [BNN_MAX_OUT] */
  BNN_I_PRED_HIST = 66,          /* [BNN_MAX_OUT] */
  BNN_I_RING = 98,               /* [100] last outcomes */
  BNN_I_STRIDE = 200
};

const char* bnn_last_error(void);
int bnn_abi_version(void);

int bnn_ctx_create(bnn_ctx** ctx, int device);
int bnn_ctx_destroy(bnn_ctx* ctx);

/* Fix the network shape.  Replaces the shape bookkeeping of npBNN.__init__ (BNN_env.py:79-124). */
int bnn_set_net(bnn_ctx* ctx, const bnn_net_spec* spec);
int64_t bnn_n_params(const bnn_ctx* ctx);

/* Stage the data set once (npBNN._data/_labels/_test_data/_test_labels, BNN_env.py:35-49; the
 * reference re-copies X every step, BNN_env.py:388).  x_dev is [n_train + n_test, F] row-major,
 * training rows first.  labels_dev (int32 [n]) for CATEGORICAL, targets_dev (f64 [n, K]) for the
 * Gaussian and count likelihoods (K modelled columns: O, O/2 with the sigma head or NEGBIN*, 1 for POISSON).
 * inst_w_dev [n_train] and class_w_dev [K] may be NULL (calc_likelihood's instance_weight / class_weight,
 * BNN_lib.py:100-121); the count likelihoods refuse both (BNN_lik.py ignores them). */
int bnn_set_data(bnn_ctx* ctx, const double* x_dev, int64_t n_train, int64_t n_test,
                 const int32_t* labels_dev, const double* targets_dev,
                 const double* inst_w_dev, const double* class_w_dev, void* stream);

/* Score n_sets weight sets against the staged data in one pass over X.
 * Replaces, per weight set: RunPredict (BNN_lib.py:245-256) + likelihood_f (BNN_lib.py:100-143) +
 * CalcAccuracy / CalcLabelAccuracy / CalcLabelFreq (BNN_lib.py:195-233) on train and test rows.
 *   w_dev      [n_sets, n_params] canonical weights
 *   alpha_dev  [n_sets, n_layers] genReLU slopes or NULL
 *   sigma_dev  [n_sets, O] error_prm or NULL (= 1); ignored when sigma_mode == BNN_SIGMA_EMPIRICAL
 *   loglik_dev [n_sets]
 *   sums_dev   [n_sets, 3, O]  sum r, sum r^2 (train), sum r^2 (test)   (Gaussian; may be NULL)
 *   counts_dev [n_sets, 2 + 2K] n_correct, n_correct_test, class_correct[K], pred_hist[K] (may be NULL) */
int bnn_forward_lik(bnn_ctx* ctx, const double* w_dev, int32_t n_sets, const double* alpha_dev,
                    const double* sigma_dev, int32_t sigma_mode, double lik_temp,
                    double* loglik_dev, double* sums_dev, int32_t* counts_dev, void* stream);
/* Same call with host buffers: copies w_host to the device, runs, copies loglik back and synchronises. */
int bnn_forward_lik_host(bnn_ctx* ctx, const double* w_host, int32_t n_sets, const double* alpha_host,
                         const double* sigma_host, int32_t sigma_mode, double lik_temp,
                         double* loglik_host, double* sums_host, int32_t* counts_host, void* stream);

/* Log-prior of n_sets weight sets: npBNN.calc_prior (BNN_env.py:180-194) without indicators. */
int bnn_log_prior(bnn_ctx* ctx, const double* w_dev, int32_t n_sets, int32_t prior,
                  const double* prior_scale /* host [n_layers] */, double* logprior_dev, void* stream);

/* The same with one scale per weight entry (host [n_params], canonical layout): calc_prior after
 * npBNN.sample_prior_scale has replaced the per-layer scalars by a vector per input node or a matrix per weight
 * (hyper_p = 2, 3; BNN_env.py:180-194,196-219).  Scales must be positive and finite. */
int bnn_log_prior_entries(bnn_ctx* ctx, const double* w_dev, int32_t n_sets, int32_t prior,
                          const double* entry_scale_host, double* logprior_dev, void* stream);

/* Create n_chains chains resident on the device.  Replaces MCMC.__init__ (BNN_env.py:274-379) for
 * every chain: initial forward, likelihood, prior and accuracy counters are computed here.
 *   w0_host     [C, n_params]
 *   mask_host   [n_params] 0/1 (npBNN._mask, BNN_env.py:259-267) or NULL
 *   temperature [C]; update_f, update_ws [C, n_layers]; alpha [C, n_layers] or NULL; sigma0 [C, O] or NULL */
int bnn_chains_init(bnn_ctx* ctx, int32_t n_chains, const bnn_sampler_config* cfg, const double* w0_host,
                    const double* mask_host, const double* temperature, const double* update_f,
                    const double* update_ws, const double* alpha, const double* sigma0, void* stream);

/* Run n_steps MH iterations of every chain without leaving the device.  One iteration replaces
 * MCMC.mh_step (BNN_env.py:381-532) with update_function = UpdateNormal (BNN_mcmc.py:57-69).
 * inj == NULL: free-running Philox proposals; otherwise the recorded draws are replayed. */
int bnn_mh_steps(bnn_ctx* ctx, int32_t n_steps, const bnn_injection* inj, void* stream);

/* Export chain state (synchronises the stream).  Any pointer may be NULL.
 *   f64_host [C, BNN_F_STRIDE], i32_host [C, BNN_I_STRIDE], w_host [C, n_params] */
int bnn_chains_read(bnn_ctx* ctx, double* f64_host, int32_t* i32_host, double* w_host, void* stream);
/* Asynchronous export for the logger (SURVEY.md 8f-4; replaces the synchronous reads behind
 * postLogger.log_sample / log_weights, BNN_env.py:600-658, when the chains free-run on the device):
 * bnn_chains_snapshot copies the state of every chain (same three arrays as bnn_chains_read) into ring slot
 * `slot` (0..63) in stream order -- device-to-device on `stream`, then device-to-host into pinned memory on the
 * context's own copy stream -- and returns without waiting, so the caller can queue the next bnn_mh_steps at once.
 * bnn_snapshot_ready: 1 when the host copy of the slot is complete, 0 when not yet, -1 when the slot is empty.
 * bnn_snapshot_read waits for the slot, copies it out and frees the slot.  Any output pointer may be NULL. */
int bnn_chains_snapshot(bnn_ctx* ctx, int32_t slot, void* stream);
int bnn_snapshot_ready(bnn_ctx* ctx, int32_t slot);
int bnn_snapshot_read(bnn_ctx* ctx, int32_t slot, double* f64_host, int32_t* i32_host, double* w_host);
/* The indicators the same snapshot holds for chains that carry them (layouts of bnn_chains_read_indicators; either may
 * be NULL): waits for the slot and copies them out without freeing it, so call it before bnn_snapshot_read.  A snapshot
 * is one iteration's state, indicators included, however many steps were queued behind it. */
int bnn_snapshot_read_indicators(bnn_ctx* ctx, int32_t slot, double* ind_host, double* fi_host);
/* Training means of the features (host [n_features]) for the feature-indicator transform; call before
 * bnn_chains_init with cfg.use_feature_indicators. */
int bnn_set_feature_means(bnn_ctx* ctx, const double* mean_host, void* stream);
/* Current indicators of every chain: ind_host [C, size of the first weight matrix], fi_host [C, n_features]
 * (doubles 0/1; either may be NULL; synchronises). */
int bnn_chains_read_indicators(bnn_ctx* ctx, double* ind_host, double* fi_host, void* stream);
/* The counterpart: set the current indicators of every chain (same layouts, values 0 or 1; either may be NULL;
 * synchronises) and score the chains' current weights under them as bnn_chains_init scores w0 -- logLik, logPrior with
 * the indicator term, logPost and the accuracy counters of the initial state.  So it starts chains from indicators that
 * are not all ones (npBNN._indicators / _feature_indicators set before MCMC.__init__), and it is the indicator step of
 * restoring a saved chain, which ends with bnn_chains_write of the saved state.  Drops the captured graphs of
 * bnn_mh_steps.  Row-sharded chains stop before the accept step, as bnn_chains_init does. */
int bnn_chains_write_indicators(bnn_ctx* ctx, const double* ind_host, const double* fi_host, void* stream);
/* Write the state arrays back (same layout as bnn_chains_read; synchronises the stream): the host edits what it
 * read -- MCMC.reset_update_n / reset_update_f / reset_update_ws (BNN_env.py:540-547), the iteration count after
 * a Gibbs step.  Any pointer may be NULL. */
int bnn_chains_write(bnn_ctx* ctx, const double* f64_host, const int32_t* i32_host, void* stream);
/* New prior scales for the chains, one per weight entry (host [C, n_params]; NULL: back to the per-layer scalars
 * given at bnn_chains_init), then logPrior = calc_prior(), logPost = logLik + logPrior of every chain's current
 * weights: the device half of MCMC.gibbs_step (BNN_env.py:534-538) once the host has drawn the scales
 * (npBNN.sample_prior_scale, BNN_env.py:196-219; GibbsSampleNormStdGamma*, BNN_mcmc.py:124-141).  The proposals of
 * the following bnn_mh_steps are scored with these scales. */
int bnn_chains_set_prior_scales(bnn_ctx* ctx, const double* entry_scale_host, void* stream);
/* The additional_prob argument of mh_step (BNN_env.py:381,481) for chains whose proposals are drawn on the device
 * (host [C], finite; synchronises the stream).  Every following proposal of chain c adds per_chain_host[c] to its
 * log-prior, with the Exp(10) term of trainable activation parameters on top, until the next call.  Injected steps read
 * it too: a bnn_injection that carries add_prob takes precedence for its steps, one without add_prob (NULL) uses this
 * value, as free-running steps do.  The value lives in a buffer of the context whose address is
 * fixed from the first call after bnn_chains_init on, so a change reaches the captured graphs of bnn_mh_steps (the
 * copy runs in stream order before their next replay).  NULL, and never calling this, mean 0 for every chain.
 * bnn_chains_init clears it. */
int bnn_chains_set_additional_prob(bnn_ctx* ctx, const double* per_chain_host, void* stream);
/* Device pointers to the live chain state (same layout as bnn_chains_read; e.g. the log-posteriors for
 * the MC3 all-gather are f64_dev[c * BNN_F_STRIDE + BNN_F_LOGPOST]).  Any pointer may be NULL. */
int bnn_chains_state_dev(bnn_ctx* ctx, double** f64_dev, int32_t** i32_dev, double** w_dev);
/* Copy one f64 state slot of every chain (e.g. BNN_F_LOGPOST) into out_dev [C] on the stream: the send
 * buffer of the MC3 all-gather that replaces the pickling of whole chains in BNN_mc3.py:96. */
int bnn_chains_gather(bnn_ctx* ctx, int32_t slot, double* out_dev, void* stream);
/* Temperature update after an MC3 swap (BNN_mc3.py:98-112; reset_temperature, BNN_env.py:549-550). */
int bnn_chains_set_temperature(bnn_ctx* ctx, const double* temperature_host, void* stream);

/* Posterior prediction for n_sets weight sets over rows of x_dev [n, F] (not the staged data):
 * replaces the loop `for i in range(S): RunPredict(...)` of get_posterior_cat_prob (BNN_lib.py:376-397),
 * get_posterior_est (BNN_lib.py:731-737) and get_pdp (BNN_pdp.py:63-73).
 *   override_cols [n_override] / override_vals [n_override]: PDP column overwrite (BNN_pdp.py:65), host, may be NULL
 *   mean_dev [n, K] mean of the transformed outputs; votes_dev [n, K] argmax vote share;
 *   dense_dev [n_sets, n, K] every prediction (only for small problems); any may be NULL */
int bnn_predict(bnn_ctx* ctx, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                const double* alpha_dev, const int32_t* override_cols, const double* override_vals,
                int32_t n_override, double* mean_dev, double* votes_dev, double* dense_dev, void* stream);

/* Zero pattern of the weight sets the prediction calls below will score: mask_host [n_params] in the canonical layout,
 * 0 where every weight set is exactly zero (e.g. the union over the posterior samples of w != 0 of a block-masked
 * network, create_mask / apply_mask), NULL clears it.  While a pattern is set and option "sparse" is 1, bnn_predict,
 * bnn_predict_sample and bnn_predict_sample_philox(_at) run the block-sparse kernels on the program of the pattern
 * (bnn_last_kernel: "k_fwd_sparse<pairs,predict>" or "k_fwd_sparse<predict>"): same outputs as the dense kernels up to
 * the order of the sums, each row's sums over the sets in set order.  Each call first checks on the device that every
 * weight set is zero outside the pattern and runs the dense kernels when one is not; that check reads one flag back, so
 * with a pattern set these calls wait on the host for the stream's work up to the check (without one they stay
 * asynchronous).  The program is built per pattern and padded layout and kept while the pattern does not change;
 * bnn_set_net clears the pattern.  When the pattern's block cover is not thin enough (or
 * the network has no hidden layer, more than 8 outputs, or a program too large for shared memory) the call succeeds and
 * prediction stays dense.  Option "predict_tf32" does not apply to the block-sparse kernels: with a pattern in use,
 * prediction runs them in FP64 whatever the option. */
int bnn_set_predict_mask(bnn_ctx* ctx, const double* mask_host);

/* Number of kernel launches issued by this context so far (bench.py's gpu_launches). */
int64_t bnn_launch_count(const bnn_ctx* ctx);
/* With option "time_forward" = 1 every forward launch is bracketed by CUDA events on its stream; this
 * returns the accumulated device time and launch count (and optionally resets them). */
int bnn_forward_time(bnn_ctx* ctx, double* total_ms, int64_t* n_launches, int32_t reset);
/* Measured FP64 tensor-pipe peak of this GPU in TFLOP/s (back-to-back DMMA): roofline denominator. */
int bnn_measure_fp64_peak(bnn_ctx* ctx, double* tflops);
/* Name of the forward kernel variant used by the last call ("k_fwd3<...>" or "k_fwd_generic"). */
const char* bnn_last_kernel(const bnn_ctx* ctx);

/* ---- Row sharding (few chains, many rows; SURVEY.md 8e-2) ------------------------------------------------------
 * Every rank stages ITS rows with bnn_set_data, calls bnn_rowshard_config(n_train_global) and then drives the same
 * chains (same seeds / injected draws) on every rank.  One MH iteration is
 *     bnn_rowshard_update(accept_mode = 0, propose = 1, inj)   proposal + forward pass over the local rows
 *     bnn_rowshard_local(red)                                  per-chain sums of the local partials, [C, n_values]
 *     all-reduce(red, SUM) over the ranks                      (NCCL / gloo: the one exchange step of this mode)
 *     bnn_rowshard_commit(red)                                 the accept step will see the global sums
 *     bnn_rowshard_update(accept_mode = 1, propose = 0, NULL)  accept / reject: identical on every rank
 * After bnn_chains_init the same local / all-reduce / commit sequence is followed by accept_mode = 2 (initial state).
 * The reductions are fixed-order, so every rank holds bit-identical chain states.  Every likelihood kind is served.
 * The count kinds exchange the same 1 + 3K slots as the Gaussian one (log-likelihood, then sum r, sum r^2 and the
 * test sum r^2 per modelled column); lgamma(k + 1) is staged by bnn_set_data from the rank's own targets, and the
 * companion MSE is the exchanged sum over the global row count, which the caller divides by. */
int bnn_rowshard_config(bnn_ctx* ctx, int64_t n_train_global);
int bnn_rowshard_n_values(const bnn_ctx* ctx);                 /* doubles per chain in the exchanged vector */
int bnn_rowshard_local(bnn_ctx* ctx, double* red_dev, void* stream);
int bnn_rowshard_commit(bnn_ctx* ctx, const double* red_global_dev, void* stream);
int bnn_rowshard_update(bnn_ctx* ctx, int32_t accept_mode, int32_t propose, const bnn_injection* inj, void* stream);

/* Posterior-predictive resampling: sample_from_categorical (BNN_lib.py:682-713), i.e. get_posterior_cat_prob with
 * post_summary_mode = 2, fused into the prediction pass.  u_dev [n, n_sets] holds the uniforms of the reference
 * (np.random.random(n_sets) per instance, instance-major); for every (row, set) the class is the first one whose
 * cumulative softmax probability reaches u (class 0 when none does, as argmin over the clipped differences gives).
 *   est_dev          [n, K]       share of the n_sets draws per class   ('predictions')
 *   class_counts_dev [n_sets, K]  int32, instances per class and set     ('class_counts'), may be NULL
 *   post_pred_dev    [n, n_sets]  the drawn class as f64                 ('post_predictions'), may be NULL */
int bnn_predict_sample(bnn_ctx* ctx, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                       const double* alpha_dev, const double* u_dev, double* est_dev, int32_t* class_counts_dev,
                       double* post_pred_dev, void* stream);

/* The same resampling with the uniforms generated inside the kernel (Philox4x32-10, counter = (row, set), key = seed):
 * nothing of size n x n_sets is ever stored, so get_posterior_cat_prob(post_summary_mode=2) runs at BASELINE config 5
 * scale (10,000 samples x 1,000,000 rows) in O(n K) memory, on the shape-specialised kernel where one exists.
 * bnn_predict_sample (injected uniforms) reproduces the reference's draws; this one agrees with it statistically. */
int bnn_predict_sample_philox(bnn_ctx* ctx, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                              const double* alpha_dev, uint64_t seed, double* est_dev, int32_t* class_counts_dev,
                              double* post_pred_dev, void* stream);

/* bnn_predict_sample_philox over a block of a larger prediction: x_dev holds rows row0 ... row0 + n - 1 and w_dev the
 * weight sets set0 ... set0 + n_sets - 1 of it, and the uniforms are keyed on the global (row0 + row, set0 + set).  The
 * block's outputs are then that block of the larger call's: post_pred_dev bit for bit where both run the same kernel,
 * est_dev and class_counts_dev as the block's share and counts.  Ranks that split a prediction into row x sample blocks
 * draw the single-process run's uniforms.  bnn_predict_sample_philox is this call with row0 = set0 = 0. */
int bnn_predict_sample_philox_at(bnn_ctx* ctx, const double* x_dev, int64_t n, const double* w_dev, int32_t n_sets,
                                 const double* alpha_dev, uint64_t seed, int64_t row0, int32_t set0, double* est_dev,
                                 int32_t* class_counts_dev, double* post_pred_dev, void* stream);

/* Debugging aid (no reference counterpart).
 * bnn_debug_read_part: per-warp-tile partial sums of the last forward pass, [sets in pass][slots][n_tiles16]. */
int bnn_debug_read_part(bnn_ctx* ctx, double* out_host, int64_t n_doubles);
/* Options: "force_generic" = 1 disables the shape-specialised forward kernels (cross-check in tests);
 * "time_forward" = 1 enables bnn_forward_time; "sparse" = 0 evaluates masked chains with the dense kernels;
 * "graphs" = 0 launches the free-running bnn_mh_steps loop eagerly instead of replaying a CUDA graph;
 * "chain_loop" = 1 (default) steps small data sets inside one persistent launch per bnn_mh_steps call (k_chain_loop: a
 * thread-block cluster per chain) where that beats one launch pair per iteration, 2 = wherever the problem fits, 0 = never
 * (results are bit-identical either way);
 * "chain_loop_cluster" = 1 | 2 | 4 | 8 | 16 caps the cluster size of that kernel (default 16);
 * "predict_tf32" = 1 (default 0) evaluates the prediction calls of every dense network -- bnn_predict summaries (mean /
 * votes, every likelihood) and the resampling of bnn_predict_sample / bnn_predict_sample_philox(_at) -- on the TF32 tensor
 * cores in error-compensated 3xTF32 form, with FP32 activations, softmax and softplus and FP64 sums over the sets in set
 * order (bnn_last_kernel: "k_pred_tf32x3<act>" for the 64-64-32-16 categorical family, "k_pred_tf32x3_generic<act>" for
 * every other network).  Stated tolerances against the FP64 kernels: class probabilities 5e-6 absolute; regression,
 * sigma-head and count means 1e-5 * max(1, |y|); vote flips at most 1e-4 * n * n_sets; a drawn class differs from the FP64
 * draw only where the FP64 running sum lies within 1e-5 of u at a class boundary.  2 = plain TF32 (one product,
 * "k_pred_tf32x1...": 5e-3 in the same forms).  A call that asks for dense_dev, a call on the block-sparse kernels, and
 * bnn_mh_steps and the likelihood calls always run in FP64; so do, under option 1 only, Gaussian and count outputs of
 * networks padded to the 32-32-16 width family (measured slower in 3xTF32 than the FP64 kernel there).  Any other name is refused. */
int bnn_set_option(bnn_ctx* ctx, const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* NPBNN_B200_H */
