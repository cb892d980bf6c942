"""Host-side mirror of the reference's Python interface for the MCMC hot path.

Same names, argument meaning and attribute surface as `np_bnn` (reference np_bnn/__init__.py:6-25), so
the reference's scripts and the parity tests read the same; the arithmetic of every call runs in the
CUDA library behind the C ABI (include/npbnn_b200.h).  There is no CPU fallback.

What is on the device path            reference
  npBNN.calc_prior                    BNN_env.py:180-194
  MCMC.__init__ / MCMC.mh_step        BNN_env.py:274-532   (update_function = UpdateNormal)
  count likelihoods (custom mode)     BNN_lik.py:5-66      (poi_likelihood, negbin_likelihood, negbin_likelihood2d,
                                                          negbin_likelihood_base10 and their accuracy functions)
  run_mcmc                            BNN_mcmc.py:153-170
  MC3.run_mcmc                        BNN_mc3.py:87-126
  RunPredict / RunPredictInd / predict  BNN_lib.py:245-272, BNN_env.py:662-670
  get_posterior_cat_prob (modes 0, 1) BNN_lib.py:352-397
  get_posterior_est                   BNN_lib.py:715-748
  get_pdp / pdp                       BNN_pdp.py:48-108

Random numbers.  `rng="host"` (default of MCMC) draws every proposal from `self._rs`
(np.random.default_rng(1234), BNN_env.py:362) with exactly the reference's call sequence and replays
the draws on the device: the chain is then the reference's chain (same accept/reject decisions; the
log-likelihood differs in the last bits because of the summation order).  `rng="philox"` generates the
proposals on the device and never leaves it between logging points.

Trainable activation parameters (ActFun(trainable=True)), init_additional_prob, mh_step(additional_prob=), weight
indicators (freq_indicator > 0) and feature indicators (feature_indicators=True) run on the device with either source of
random numbers; hyper-prior scales (hyper_p) are drawn on the host and evaluated on the device.  With rng="philox",
mh_step(additional_prob=a) copies a into the chain's device value when it changes (bnn_chains_set_additional_prob).
MC3 runs trainable activation parameters in every chain, on every rank layout.  Chains start from the model's
indicators, all ones or not.

Resuming.  The [bnn, mcmc, logger] pickle that postLogger.log_weights writes carries the chain's device state as of
the logging point (state rows, indicators, additional_prob, the host generator _rs); load_obj it, raise
mcmc._n_iterations and run_mcmc(bnn, mcmc, logger) continues the chain bit for bit.  A pickled MC3 continues all its
chains on the next run_mcmc; the caller restores np.random's state where the run draws from it (swaps of a single-process
MC3, host-drawn indicator flips).  Not resumable: pickles written before samplers carried their state (RuntimeError: use
npBNN(pickle_file=)), the cold-chain mcmc that MC3's logger pickles (RuntimeError: resume the MC3 object), and samplers
run over torch.distributed ranks -- MCMC(row_shard=True) and MC3 with world > 1 (NotImplementedError).

Several GPUs.  Under an initialised torch.distributed process group of more than one rank, MC3 shards its chains
(mc3.chain_grid) and MCMC(row_shard=True) one chain's rows.  The posterior-prediction callers (get_posterior_cat_prob,
sample_from_categorical, get_posterior_est, get_pdp / pdp, feature_importance, hostlib's predictBNN and
get_posterior_threshold) all go through one routine, predshard.predict_ranks, in one process and on many ranks alike.
They are collective: every rank calls them with the same arguments (ValueError on every rank otherwise), scores its
rows x samples block on its current device and returns the result of one process.  Rank 0 alone draws from numpy's
global stream and writes files.  A single process is a group of one rank: it scores the whole problem on GPU 0 and
makes no torch.distributed call.

estimation_mode="custom" runs with output_act_fun=RegressTransform and one of the count likelihoods of BNN_lik.py as
MCMC / MC3(likelihood_f=), recognised by identity (SURVEY.md, item 9 on pluggable callables); accuracy_f=None means the likelihood's
companion MSE.  Options of the reference that are not on the device path raise
NotImplementedError: other user-supplied likelihood / proposal / output functions (gamma_likelihood among them),
MCMC(row_shard=True) with a count likelihood outside an initialised torch.distributed process group, MC3 with
more ranks than chains (row-sharded chain blocks) together with host-drawn weight or feature indicators (rng="host" and
freq_indicator > 0 or feature_indicators=True), init_additional_prob inside an MC3 group (the reference's MC3 never
passes it, BNN_mc3.py:61-75), and the regression error-parameter proposal (estimate_error with
empirical_error=False once the iteration passes `_estimate_error` -- a branch on which the reference itself raises
AttributeError as soon as one proposal has been accepted before that iteration, BNN_mcmc.py:105).
"""
import csv
import os
import pickle
from copy import deepcopy
from types import SimpleNamespace

import numpy as np

from . import _lib as L
from . import mc3 as _mc3
from . import predshard
from .engine import ChainState, Engine, NetShape, flatten_weights, unflatten_weights

small_number = 1e-10


# names the reference exports and user code passes around (SoftMax, calc_likelihood, UpdateNormal ...): inside the
# sampler they are identity tokens that select device code; hostlib holds their host-table forms and the file / summary
# callers around the path
from .hostlib import (CalcAccuracy, CalcAccuracyRegression, CalcLabelAccuracy, CalcLabelAccuracyRegression,  # noqa: E402,F401
                      CalcLabelFreq, RegressTransform, RegressTransformError, SoftMax, UpdateNormal, calc_likelihood,
                      calc_likelihood_regression, calc_likelihood_regression_error, gamma_likelihood, load_obj, log_header,
                      negbin2d_acc, negbin_acc, negbin_acc_base10, negbin_likelihood, negbin_likelihood2d,
                      negbin_likelihood_base10, poi_acc, poi_likelihood)


class ActFun:
    """Activation selector (BNN_lib.py:68-94).  Later `if`s override earlier ones exactly as in the reference:
    fun="ReLU" with trainable=True still evaluates as plain ReLU (eval passes prm 0 unless fun=="genReLU")."""

    def __init__(self, fun="ReLU", prm=np.zeros(1), trainable=False):
        if fun not in ("ReLU", "genReLU", "swish", "tanh"):
            raise ValueError("unknown activation %r" % (fun,))
        self._prm = prm
        self._acc_prm = prm
        self._trainable = trainable
        self._function = fun

    def reset_prm(self, prm):
        self._prm = prm

    def reset_accepted_prm(self):
        self._acc_prm = self._prm + 0

    def alphas(self, n_layers):
        """Per-layer slopes for the device state: the parameters matter for the forward pass only with
        fun == "genReLU" (eval, BNN_lib.py:83-87), but trainable ones are proposed and enter the prior whatever the
        function is (BNN_env.py:416-421), so they are carried in the chain state in that case too."""
        if self._function != "genReLU" and not self._trainable:
            return None
        a = np.zeros(n_layers)
        p = np.atleast_1d(np.asarray(self._acc_prm if self._trainable else self._prm, dtype=np.float64))
        a[:min(len(p), n_layers)] = p[:n_layers]
        return a

    def n_trainable(self):
        return len(np.atleast_1d(self._acc_prm)) if self._trainable else 0


def init_weight_prm(n_nodes, n_features, size_output, init_std=0.1, bias_node=0):
    """N(0, init_std) weights from the global numpy state; bias columns per `bias_node`
    (>=1 first layer, >=2 hidden layers, 3 or -1 last layer), as BNN_mcmc.py:9-25."""
    b_first = 1 if bias_node >= 1 else 0
    b_hidden = 1 if bias_node >= 2 else 0
    b_last = 1 if bias_node in (3, -1) else 0
    widths = [n_features] + list(n_nodes)
    layers = []
    for i, out in enumerate(n_nodes):
        layers.append(np.random.normal(0, init_std, (out, widths[i] + (b_first if i == 0 else b_hidden))))
    layers.append(np.random.normal(0, init_std, (size_output, n_nodes[-1] + b_last)))
    return layers


def create_mask(w_layers, indx_input_list, nodes_per_feature_list):
    """Block masks (BNN_lib.py:16-47): in layer l, input column i belongs to group indx_input_list[l][i];
    consecutive columns of one group share a block of nodes_per_feature_list[l][group] rows; blocks stack
    downwards; an empty list means fully connected."""
    masks = []
    for l, w in enumerate(w_layers):
        groups, rows = indx_input_list[l], nodes_per_feature_list[l]
        if len(groups) == 0:
            masks.append(np.ones(w.shape))
            continue
        m = np.zeros(w.shape)
        g, row0 = 0, 0
        for col in range(len(groups)):
            if col > 0 and groups[col] != groups[col - 1]:
                row0 += rows[g]
                g += 1
            m[row0:row0 + rows[g], col] = 1
        masks.append(m)
    return masks


# device likelihood of each estimation mode.  A custom model's own engine (prior, identity prediction) is the Gaussian
# one; its sampler's kind is the count likelihood that MCMC(likelihood_f=) selects (_count_likelihood).
_LIK = {"classification": L.LIK_CATEGORICAL, "regression": L.LIK_GAUSSIAN, "regression-error": L.LIK_GAUSSIAN_HEAD,
        "custom": L.LIK_GAUSSIAN}

# custom likelihoods on the device (BNN_lik.py), selected by function identity: likelihood_f -> (device kind, companion
# accuracy_f)
_COUNT_LIK = {poi_likelihood: (L.LIK_POISSON, poi_acc), negbin_likelihood: (L.LIK_NEGBIN, negbin_acc),
              negbin_likelihood2d: (L.LIK_NEGBIN, negbin2d_acc),
              negbin_likelihood_base10: (L.LIK_NEGBIN10, negbin_acc_base10)}


def _count_likelihood(bnn, likelihood_f, accuracy_f, accuracy_lab_f):
    """The device likelihood kind and accuracy function of a sampler: None for a built-in estimation mode (which takes
    no user functions), the count kind of likelihood_f for estimation_mode="custom"."""
    if bnn._estimation_mode != "custom":
        if likelihood_f is not None or accuracy_f is not None or accuracy_lab_f is not None:
            raise NotImplementedError("user-supplied likelihood / accuracy functions are not on the device path")
        return None, None
    if likelihood_f is gamma_likelihood:
        raise NotImplementedError("gamma_likelihood is not on the device path: it passes its second parameter as scipy's "
                                  "location (BNN_lik.py:83) and broadcasts [N, 1] labels against [N] parameters into an "
                                  "N x N table")
    if likelihood_f not in _COUNT_LIK:
        raise NotImplementedError("estimation_mode='custom' runs on the device with likelihood_f = poi_likelihood, "
                                  "negbin_likelihood, negbin_likelihood2d or negbin_likelihood_base10")
    kind, companion = _COUNT_LIK[likelihood_f]
    if accuracy_f is not None and accuracy_f is not companion:
        raise NotImplementedError("accuracy_f of %s must be %s (or None)" % (likelihood_f.__name__, companion.__name__))
    if accuracy_lab_f is not None:
        raise NotImplementedError("user-supplied accuracy_lab_f is not on the device path")
    o, n_lab = bnn._size_output, bnn._labels.shape[1]
    if likelihood_f is negbin_likelihood2d and o != 2 * n_lab:
        raise ValueError("negbin_likelihood2d needs size_output = 2 x the label columns (%d), not %d" % (2 * n_lab, o))
    if kind != L.LIK_POISSON and likelihood_f is not negbin_likelihood2d and o != 2:
        raise NotImplementedError("%s on the device needs size_output=2 (mean, dispersion)" % likelihood_f.__name__)
    return kind, companion


def _net_of(weights, n_features, act_fun, estimation_mode, lik=None):
    return NetShape.from_weights(weights, n_features, act=act_fun._function, lik=_LIK[estimation_mode] if lik is None else lik)


class npBNN:
    """Model state (BNN_env.py:19-270).  Same constructor signature and attributes as the reference."""

    def __init__(self, dat, n_nodes=[50, 5], use_bias_node=1, init_std=0.1, p_scale=1, prior_ind1=0.5, prior_f=1,
                 hyper_p=0, freq_indicator=0, w_bound=np.inf, pickle_file="", seed=1234, use_class_weights=0,
                 actFun=None, init_weights=None, estimation_mode="classification", instance_weights=None,
                 empirical_error=False, size_output=None, output_act_fun=None, feature_indicators=None):
        if actFun is None:
            actFun = ActFun()
        if hyper_p not in (0, 1, 2, 3):
            raise ValueError("hyper_p must be 0, 1, 2 or 3")
        if estimation_mode not in _LIK:
            raise NotImplementedError("estimation_mode=%r (custom likelihoods) is not on the device path" % (estimation_mode,))
        if output_act_fun is not None and not (estimation_mode == "regression-error" and output_act_fun is RegressTransformError) \
                and not (estimation_mode in ("regression", "custom") and output_act_fun is RegressTransform):
            raise NotImplementedError("user-supplied output_act_fun is not on the device path")
        if estimation_mode == "custom":
            # the count likelihoods read identity outputs; the reference crashes on None (RunPredict calls it)
            if output_act_fun is not RegressTransform:
                raise NotImplementedError("estimation_mode='custom' runs on the device with output_act_fun=RegressTransform")
            if size_output is None:
                raise ValueError("estimation_mode='custom' needs size_output")
        data, labels = dat["data"], dat["labels"]
        self._seed = seed
        self._data = np.ascontiguousarray(data, dtype=np.float64)
        self._labels = labels.astype(int) if estimation_mode == "classification" else np.asarray(labels, dtype=np.float64)
        self._test_data = dat["test_data"]
        tl = dat["test_labels"]
        if len(tl) > 0:
            self._test_labels = tl.astype(int) if estimation_mode == "classification" else np.asarray(tl, dtype=np.float64)
        else:
            self._test_labels = []
        self._error_prm = []
        if estimation_mode == "classification":
            self._size_output = len(np.unique(self._labels))
            self._n_output_prm = self._size_output
            self._output_act_fun = SoftMax
        elif estimation_mode == "regression":
            self._output_act_fun = RegressTransform
            self._size_output = self._labels.shape[1]
            self._n_output_prm = self._labels.shape[1]
            self._error_prm = np.ones(self._size_output)
        elif estimation_mode == "custom":
            self._output_act_fun = RegressTransform
            self._size_output = int(size_output)
            self._n_output_prm = self._labels.shape[1]
        else:
            self._output_act_fun = RegressTransformError
            self._size_output = self._labels.shape[1] * 2
            self._n_output_prm = self._labels.shape[1]
        self._empirical_error = empirical_error
        self._init_std = init_std
        try:
            n_nodes = list(n_nodes)
        except TypeError:
            n_nodes = [n_nodes]
        self._n_layers = len(n_nodes) + 1
        self._n_nodes = n_nodes
        self._use_bias_node = use_bias_node
        self._n_samples, self._n_features = self._data.shape
        self._w_bound = w_bound
        self._freq_indicator = freq_indicator
        self._hyper_p = hyper_p
        self._sample_id = np.arange(self._n_samples)
        self._prior = prior_f
        self._p_scale = p_scale
        self._prior_ind1 = prior_ind1
        self._estimation_mode = estimation_mode
        self._mask = None
        # feature indicators (BNN_env.py:169-172): all ones, means of the training features
        if feature_indicators:
            self._feature_indicators = np.ones(self._data.shape[1]).astype(int)
            self._feature_means = np.mean(self._data, axis=0)
        else:
            self._feature_indicators = None
            self._feature_means = None
        if use_class_weights:
            counts = np.unique(self._labels, return_counts=True)[1]
            cw = 1 / (counts / np.max(counts))
            self._class_w = cw / np.mean(cw)
        else:
            self._class_w = []
        self._instance_weights = instance_weights
        if init_weights is None:
            if pickle_file == "":
                # the reference passes the literal 0.1 here, ignoring its init_std argument (BNN_env.py:111-115)
                w_layers = init_weight_prm(self._n_nodes, self._n_features, self._size_output, init_std=0.1,
                                           bias_node=use_bias_node)
            else:
                _, _, logger_obj = load_obj(pickle_file)
                w_layers = logger_obj._post_weight_samples[-1]["weights"]
        else:
            w_layers = init_weights
        self._w_layers = w_layers
        self._indicators = np.ones(self._w_layers[0].shape)
        self._act_fun = actFun
        if self._prior == 0:
            self._w_bound = self._p_scale            # uniform prior: bounds = p_scale (BNN_env.py:135-137)
        self._prior_scale = np.ones(self._n_layers) * self._p_scale
        self._n_params = int(np.sum([np.size(w) for w in self._w_layers]))
        self._eng = None

    # prior_f: 0 uniform, 2 Cauchy, 3 Laplace, anything else Normal (selection quirk of BNN_env.py:139-150)
    def _prior_kind(self):
        return self._prior if self._prior in (0, 2, 3) else 1

    def _net(self):
        return _net_of(self._w_layers, self._n_features, self._act_fun, self._estimation_mode)

    def _engine(self):
        if self._eng is None:
            self._eng = Engine(self._net())
        return self._eng

    def _scales_per_layer(self):
        """True while _prior_scale holds one scalar per layer (no hyper-prior sample yet)."""
        return all(np.ndim(s) == 0 for s in self._prior_scale)

    def _entry_scales(self):
        """_prior_scale broadcast to one scale per weight entry, flattened in the canonical order: a scalar per layer
        (hyper_p 1), a vector per input node = per weight-matrix column (2), a matrix per weight (3) -- the broadcasting
        scipy's logpdf(w, 0, scale=...) applies in calc_prior (BNN_env.py:184-189)."""
        return np.concatenate([np.broadcast_to(np.asarray(s, dtype=np.float64), w.shape).ravel()
                               for s, w in zip(self._prior_scale, self._w_layers)])

    def calc_prior(self, w=0, ind=[]):
        if isinstance(w, int) and w == 0:
            w = self._w_layers
        lp = 0
        if self._prior != 0:
            ps = self._prior_scale if self._scales_per_layer() else self._entry_scales()
            lp = float(self._engine().log_prior([w], self._prior_kind(), ps)[0])
        if self._freq_indicator:                 # BNN_env.py:191-193 (two scalars; the sums over w are on the device)
            if len(ind) == 0:
                ind = self._indicators
            lp += np.sum(ind) * np.log(self._prior_ind1) + (self._indicators.size - np.sum(ind)) * np.log(1 - self._prior_ind1)
        return lp

    def sample_prior_scale(self):
        """Gibbs draw of the prior standard deviations from their conjugate Gamma posteriors on the precision
        (BNN_env.py:196-219; GibbsSampleNormStdGammaVector / 2D / ONE, BNN_mcmc.py:124-141).  O(n_params) host
        arithmetic on the host copy of the weights with the reference's global-generator call sequence (one
        np.random.gamma call per layer), so a seeded run draws the reference's scales."""
        if self._prior != 1:
            print("Hyper-priors available only for Normal priors.")
            quit()
        if self._hyper_p not in (1, 2, 3):
            return
        scales = []
        for w in self._w_layers:
            w = np.asarray(w, dtype=np.float64)
            if self._hyper_p == 1:                                  # one scale per layer: Gamma(2 + n/2, 0.1 + SS/2)
                tau = np.random.gamma(2 + w.size / 2.0, scale=1.0 / (0.1 + np.sum(w.flatten() ** 2) / 2.0))
            elif self._hyper_p == 2:                                # per input node (column): Gamma(1 + rows/2, .)
                tau = np.random.gamma(1 + w.shape[0] / 2.0, scale=1.0 / (0.1 + np.sum(w ** 2, axis=0) / 2.0))
            else:                                                   # per weight: Gamma(1.5 + 1/2, 0.1 + w^2/2)
                tau = np.random.gamma(1.5 + 0.5, scale=1.0 / (0.1 + (w ** 2) / 2.0))
            scales.append(1 / np.sqrt(tau))
        self._prior_scale = scales

    def reset_weights(self, w):
        self._data_version = self.__dict__.get("_data_version", 0) + 1     # staged chain state no longer matches
        self._w_layers = w

    def reset_indicators(self, ind):
        self._indicators = ind

    def reset_error_prm(self, p):
        self._error_prm = p

    def update_data(self, data_dict):
        # samplers built before this call hold the previous data on the device: MCMC.run refuses to continue on them
        self._data_version = self.__dict__.get("_data_version", 0) + 1
        self._data = np.ascontiguousarray(data_dict["data"], dtype=np.float64)
        self._labels = data_dict["labels"]
        self._test_data = data_dict["test_data"]
        self._test_labels = data_dict["test_labels"]

    def apply_mask(self, m=None):
        if m is not None:
            self._mask = m
        self._w_layers = [self._w_layers[i] * self._mask[i] for i in range(self._n_layers)]

    def reset_seed(self, seed):
        self._seed = seed

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_eng"] = None          # device handles never enter a pickle (postLogger pickles the live objects)
        return d


def _has_test(bnn):
    return len(bnn._test_data) > 0


class _ChainGroup:
    """C chains of one model on one GPU: engine + the host bookkeeping that turns numpy draws into the
    injection arrays of bnn_mh_steps.  row_shard = (R, r): this GPU holds row shard r of R of the training and test rows,
    and the R ranks of process group `row_group` (None: the default group) run the same chains (rowshard.py)."""

    def __init__(self, bnn, weights_per_chain, temperatures, update_f, update_ws, lik_temp, adapt_f, adapt_fM,
                 adapt_freq, adapt_stop, sample_from_prior, seed, device=0, init_additional_prob=0.0, row_shard=(1, 0),
                 row_group=None, chain_offset=0, lik=None, saved=None):
        """saved: one MCMC._chain_state per chain (an unpickled sampler): the chains continue from it instead of
        starting from the weights as MCMC.__init__ does."""
        self.bnn = bnn
        net = _net_of(weights_per_chain[0], bnn._n_features, bnn._act_fun, bnn._estimation_mode, lik)
        self.net = net
        self.eng = Engine(net, device=device)
        cw = bnn._class_w if len(bnn._class_w) else None
        R, r = row_shard
        if R > 1:
            # rows split over the R ranks of the group, same chains on each, one all-reduce per MH iteration (rowshard.py)
            from . import rowshard
            a, b = rowshard.row_partition(len(bnn._data), R, r)
            iw = None if bnn._instance_weights is None else bnn._instance_weights[a:b]
            if _has_test(bnn):
                ta, tb = rowshard.row_partition(len(bnn._test_data), R, r)
                self.eng.set_data(bnn._data[a:b], bnn._labels[a:b], bnn._test_data[ta:tb], bnn._test_labels[ta:tb],
                                  inst_w=iw, class_w=cw)
            else:
                self.eng.set_data(bnn._data[a:b], bnn._labels[a:b], inst_w=iw, class_w=cw)
            self.eng.enable_rowshard(len(bnn._data), lambda t: rowshard.dist_all_reduce_sum(t, row_group))
        else:
            self.eng.set_data(bnn._data, bnn._labels, bnn._test_data if _has_test(bnn) else None,
                              bnn._test_labels if _has_test(bnn) else None, inst_w=bnn._instance_weights, class_w=cw)
        self.n = len(weights_per_chain)
        sigma0 = None
        if bnn._estimation_mode == "regression":
            sigma0 = np.ones(bnn._size_output) * np.asarray(bnn._error_prm, dtype=np.float64)
        per_layer = bnn._scales_per_layer()
        self.eng.chains_init(weights_per_chain, temperature=temperatures, update_f=update_f, update_ws=update_ws,
                             prior=bnn._prior_kind(),
                             prior_scale=bnn._prior_scale if per_layer else np.ones(net.n_layers) * bnn._p_scale,
                             w_bound=bnn._w_bound,
                             mask=bnn._mask, alphas=bnn._act_fun.alphas(net.n_layers), sigma0=sigma0,
                             sigma_mode=L.SIGMA_EMPIRICAL if (bnn._estimation_mode == "regression" and bnn._empirical_error)
                             else L.SIGMA_FIXED,
                             lik_temp=lik_temp, adapt_f=adapt_f, adapt_fM=adapt_fM, adapt_freq=adapt_freq,
                             adapt_stop=adapt_stop, sample_from_prior=sample_from_prior, seed=seed,
                             n_act_prm=bnn._act_fun.n_trainable(), init_additional_prob=init_additional_prob,
                             prior_ind1=bnn._prior_ind1 if bnn._freq_indicator else None,
                             feature_means=bnn._feature_means if bnn._feature_indicators is not None else None,
                             chain_offset=chain_offset, freq_indicator=float(bnn._freq_indicator))
        self.freq_indicator = float(bnn._freq_indicator)
        self.use_fi = bnn._feature_indicators is not None
        if not per_layer:        # a model that already carries sampled hyper-prior scales
            self.eng.set_prior_scales(np.tile(bnn._entry_scales(), (self.n, 1)))
        # bnn_chains_init starts every chain from all-one indicators (as npBNN.__init__ leaves them); other values are
        # written and the weights scored again under them
        ind = fi = None
        if saved is not None:
            ind = np.stack([s["ind"] for s in saved]) if self.freq_indicator else None
            fi = np.stack([s["fi"] for s in saved]) if self.use_fi else None
        else:
            if self.freq_indicator and np.any(np.asarray(bnn._indicators) != 1):
                ind = np.broadcast_to(np.asarray(bnn._indicators, dtype=np.float64), (self.n,) + tuple(net.shapes[0]))
            if self.use_fi and np.any(np.asarray(bnn._feature_indicators) != 1):
                fi = np.broadcast_to(np.asarray(bnn._feature_indicators, dtype=np.float64), (self.n, net.n_features))
        if ind is not None or fi is not None:
            self.eng.write_indicators(ind, fi)
        if saved is not None:
            add_prob = [s["add_prob"] for s in saved]
            if any(add_prob):
                self.eng.set_additional_prob(add_prob)
            # last: set_prior_scales and write_indicators recompute logPrior without the additional_prob / Exp(10) term
            # of the last proposal, and the saved values must win
            self.eng.write_state(ChainState(np.stack([s["f64"] for s in saved]), np.stack([s["i32"] for s in saved]),
                                            None, net, self.eng.K))
        self.n_act_prm = bnn._act_fun.n_trainable()
        if self.n_act_prm > net.n_layers:
            raise ValueError("more trainable activation parameters than layers")
        self.labels_count = None
        if bnn._estimation_mode == "classification":
            self.labels_count = np.bincount(bnn._labels, minlength=bnn._size_output)

    def draw_steps(self, rngs, state, chain_ids, n_steps, reseed=None, additional_prob=0, adapt_stop=0, step0=0):
        """Consume each chain's generator exactly as mh_step + UpdateNormal do (BNN_env.py:446-453,493;
        BNN_mcmc.py:62-65) for n_steps iterations during which no adaptation fires.
        reseed(chain, iteration) -> Generator implements randomize_seed (BNN_env.py:383-384).
        step0: the draws are those of iterations state.iteration + step0 ... + step0 + n_steps - 1 (a later slice of
        the same adaptation-free stretch; only meaningful with reseed, whose generators do not depend on the slicing)."""
        assert step0 == 0 or reseed is not None
        nl = self.net.n_layers
        shapes = self.net.shapes
        cap = max(1, int(np.max(np.sum(state.update_n, axis=1))))
        inj = {"proposed": np.zeros((n_steps, self.n, nl), np.int32), "count": np.zeros((n_steps, self.n, nl), np.int32),
               "ix": np.zeros((n_steps, self.n, cap), np.int32), "iy": np.zeros((n_steps, self.n, cap), np.int32),
               "dz": np.zeros((n_steps, self.n, cap)), "log_u": np.zeros((n_steps, self.n))}
        if self.n_act_prm:
            inj["alpha_ix"] = np.zeros((n_steps, self.n), np.int32)
            inj["alpha_dz"] = np.zeros((n_steps, self.n))
        if additional_prob:
            inj["add_prob"] = np.full((n_steps, self.n), float(additional_prob))
        p0 = int(np.prod(shapes[0]))
        if self.freq_indicator:
            inj["ind_move"] = np.zeros((n_steps, self.n), np.int32)
            inj["ind_flip"] = np.zeros((n_steps, self.n, p0), np.uint8)
        if self.use_fi:
            inj["fi_move"] = np.zeros((n_steps, self.n), np.int32)
            inj["fi_flip"] = np.zeros((n_steps, self.n, self.net.n_features), np.uint8)
        for c in range(self.n):
            flu, un, uws = state.freq_layer_update[c], state.update_n[c], state.update_ws[c]
            for s in range(n_steps):
                rs = rngs[c] if reseed is None else reseed(chain_ids[c], int(state.iteration[c]) + step0 + s)
                if self.n_act_prm:        # UpdateNormal1D(_acc_prm, d=0.05, n=1, ...) comes first (BNN_env.py:416-417)
                    inj["alpha_ix"][s, c] = rs.integers(0, self.n_act_prm, 1)[0]
                    inj["alpha_dz"][s, c] = rs.normal(0, 0.05, 1)[0]
                # feature indicators (BNN_env.py:423-431): once past adapt_stop, with probability 0.2 the indicators are
                # flipped by UpdateBinomial(ind, 0.5, shape) -- numpy's GLOBAL generator (BNN_mcmc.py:98-99)
                if self.use_fi and int(state.iteration[c]) + step0 + s > adapt_stop and rs.random() < 0.2:
                    inj["fi_move"][s, c] = 1
                    inj["fi_flip"][s, c] = np.random.binomial(1, np.random.random() * 0.5, self.net.n_features)
                rr = rs.random(nl)
                rr[np.argmin(rr)] = 0
                o = 0
                for l in range(nl):
                    if l == 0 and rr[0] < self.freq_indicator:
                        # the first layer keeps its weights, its indicators move instead (BNN_env.py:449-460)
                        inj["ind_move"][s, c] = 1
                        # update_f[3]: the reference indexes its per-layer list here (BNN_env.py:460), so the branch exists
                        # for networks of at least four layers and raises IndexError otherwise -- as it does here
                        inj["ind_flip"][s, c] = np.random.binomial(1, np.random.random() * state.update_f[c][3],
                                                                   shapes[0]).ravel()
                        continue
                    if rr[l] < flu[l]:
                        n = int(un[l])
                        ix = rs.integers(0, shapes[l][0], n)
                        iy = rs.integers(0, shapes[l][1], n)
                        dz = rs.normal(0, np.full(n, uws[l]), n)
                        inj["proposed"][s, c, l] = 1
                        inj["count"][s, c, l] = n
                        inj["ix"][s, c, o:o + n], inj["iy"][s, c, o:o + n], inj["dz"][s, c, o:o + n] = ix, iy, dz
                        o += n
                with np.errstate(divide="ignore"):
                    inj["log_u"][s, c] = np.log(rs.random())
        return inj


def _steps_to_adaptation(it, adapt_freq, adapt_stop):
    """How many iterations can run from `it` (inclusive) before the adaptation block (BNN_env.py:392) can
    fire again.  The iteration `it` itself may adapt (the device does it); the host only needs the state
    AFTER that adaptation to draw, so a batch never crosses a firing iteration except at its start."""
    if it >= adapt_stop:
        return 1 << 30
    nxt = (it // adapt_freq + 1) * adapt_freq
    return max(1, nxt - it) if nxt < adapt_stop else 1 << 30


class MCMC:
    """Sampler state + step (BNN_env.py:273-550) for one chain, resident on the GPU."""

    def __init__(self, bnn_obj, update_f=None, update_ws=None, temperature=1, n_iteration=100000, sampling_f=100,
                 print_f=1000, n_post_samples=1000, update_function=UpdateNormal, sample_from_prior=0, run_ID="",
                 init_additional_prob=0, likelihood_tempering=1, mcmc_id=0, randomize_seed=False, adapt_f=0,
                 estimate_error=True, adapt_fM=1, adapt_freq=1000, adapt_stop=None, likelihood_f=None,
                 adapt_verbose=False, accuracy_f=None, accuracy_lab_f=None, rng="host", device=0, row_shard=False,
                 _group=None, _slot=0):
        if update_function is not UpdateNormal:
            raise NotImplementedError("only update_function=UpdateNormal runs on the device")
        count_kind, count_acc = _count_likelihood(bnn_obj, likelihood_f, accuracy_f, accuracy_lab_f)
        import torch.distributed as dist
        if count_kind is not None and row_shard and not (dist.is_available() and dist.is_initialized()):
            # a count model is row-sharded over the ranks of a process group; without one there are no ranks to shard
            # over, and the request stays refused rather than silently running unsharded
            raise NotImplementedError("row_shard=True with a count likelihood shards the rows over the ranks of "
                                      "torch.distributed: initialise the process group first")
        if rng not in ("host", "philox"):
            raise ValueError("rng must be 'host' or 'philox'")
        if rng == "philox" and bnn_obj._freq_indicator and bnn_obj._n_layers < 4:
            # the reference reads update_f[3] in this branch (BNN_env.py:460): IndexError below four layers
            raise IndexError("freq_indicator > 0 needs a network of at least four layers (the reference indexes update_f[3])")
        nl = bnn_obj._n_layers
        if update_ws is None:
            update_ws = [0.075] * nl
        if update_f is None:
            update_f = [0.05] * nl
        self._runID = bnn_obj._seed if run_ID == "" else run_ID
        self._n_iterations = n_iteration
        self._sampling_f = sampling_f
        self._print_f = print_f
        self._n_post_samples = n_post_samples
        self._sample_from_prior = sample_from_prior
        self._lik_temp = likelihood_tempering
        self._mcmc_id = mcmc_id
        self._randomize_seed = randomize_seed
        self._rs = np.random.default_rng(1234)        # BNN_env.py:362
        self._adapt_f, self._adapt_fM, self._adapt_freq = adapt_f, adapt_fM, adapt_freq
        self._adapt_stop = int(n_iteration * 0.05) if adapt_stop is None else adapt_stop
        self._adapt_verbose = adapt_verbose
        self._max_n = np.array([w.size for w in bnn_obj._w_layers]).astype(int)
        self._estimate_error = np.min([20000, 0.1 * n_iteration]) if estimate_error else n_iteration
        self._rng_mode = rng
        self._regression_error_proposal = (bnn_obj._estimation_mode == "regression" and not bnn_obj._empirical_error)
        self.update_function = update_function
        self._dev_add_prob = 0.0          # additional_prob the device holds for rng="philox" (set_additional_prob)
        self._own_group = _group is None
        self._device = device
        self._row_sharded = False
        if _group is None:
            shard = (1, 0)
            if row_shard and dist.is_available() and dist.is_initialized():
                shard = (dist.get_world_size(), dist.get_rank())
            self._row_sharded = shard[0] > 1
            _group = _ChainGroup(bnn_obj, [bnn_obj._w_layers], [temperature], list(update_f)[:nl], list(update_ws)[:nl],
                                 likelihood_tempering, adapt_f, adapt_fM, adapt_freq, self._adapt_stop, sample_from_prior,
                                 seed=int(bnn_obj._seed) + 7919 * int(mcmc_id), device=device,
                                 init_additional_prob=init_additional_prob, row_shard=shard, lik=count_kind)
        elif init_additional_prob:
            # the reference's MC3 builds its chains without it (BNN_mc3.py:61-75)
            raise NotImplementedError("init_additional_prob inside an MC3 group")
        self._group, self._slot = _group, _slot
        self._seen_version = bnn_obj.__dict__.get("_data_version", 0)
        self._bnn_shapes = [w.shape for w in bnn_obj._w_layers]
        # the function attributes user scripts call on host tables (bnn_regress.py:55: mcmc._accuracy_lab_f(mcmc._y, ...))
        cls = bnn_obj._estimation_mode == "classification"
        if count_kind is not None:
            self._likelihood_f, self._accuracy_f, self._accuracy_lab_f = likelihood_f, count_acc, None
        else:
            self._likelihood_f = {"classification": calc_likelihood, "regression": calc_likelihood_regression,
                                  "regression-error": calc_likelihood_regression_error}[bnn_obj._estimation_mode]
            self._accuracy_f = CalcAccuracy if cls else CalcAccuracyRegression
            self._accuracy_lab_f = CalcLabelAccuracy if cls else CalcLabelAccuracyRegression
        self._bnn_view = bnn_obj
        self._sync(bnn_obj, self._group.eng.read_state())

    # ---------------------------------------------------------------- state export
    def _sync(self, bnn_obj, st, indicators=None):
        """indicators: (weight, feature) indicators of the same export as st (a snapshot); None reads the live ones."""
        c = self._slot
        g = self._group
        self._logLik = float(st.logLik[c])
        self._logPrior = float(st.logPrior[c])
        self._logPost = float(st.logPost[c])
        self._temperature = float(st.temperature[c])
        self._acceptance_rate = float(st.acceptance_rate[c])
        self._last_accepted = int(st.last_accepted[c])
        self._current_iteration = int(st.iteration[c])
        self._update_f = np.array(st.update_f[c])
        self._update_n = np.array(st.update_n[c])
        self._update_ws = [np.ones(s) * st.update_ws[c][i] for i, s in enumerate(self._bnn_shapes)]
        self._freq_layer_update = np.array(st.freq_layer_update[c])
        n = bnn_obj._n_samples
        nt = len(bnn_obj._test_data) if _has_test(bnn_obj) else 0
        if bnn_obj._estimation_mode == "classification":
            self._accuracy = st.n_correct[c] / n
            present = g.labels_count > 0
            self._label_acc = st.class_correct[c][present] / g.labels_count[present]
            self._label_freq = st.pred_hist[c] / n
            self._test_accuracy = st.n_correct_test[c] / nt if nt else 0
        elif bnn_obj._estimation_mode == "custom":
            # the companion MSE of the count likelihood (poi_acc, negbin_acc, ...): mean of (mean - k)^2 over the K
            # modelled columns; no per-output accuracies
            o = g.eng.K
            self._accuracy = float(np.sum(st.sum_r2[c]) / (n * o))
            self._label_acc = []
            self._label_freq = None
            self._test_accuracy = float(np.sum(st.sum_r2_test[c]) / (nt * o)) if nt else 0
        else:
            o = bnn_obj._n_output_prm
            self._accuracy = float(np.sum(st.sum_r2[c]) / (n * o))
            self._label_acc = np.array(st.sum_r2[c]) / n
            self._label_freq = None
            self._test_accuracy = float(np.sum(st.sum_r2_test[c]) / (nt * o)) if nt else 0
            if bnn_obj._estimation_mode == "regression":
                bnn_obj._error_prm = np.array(st.sigma[c])
        if bnn_obj._act_fun._trainable:
            na = bnn_obj._act_fun.n_trainable()
            bnn_obj._act_fun._acc_prm = np.array(st.alpha[c][:na])          # reset_accepted_prm
            bnn_obj._act_fun._prm = np.array(st.alpha_prop[c][:na])         # the last proposal (BNN_env.py:421)
        if st.w is not None:
            bnn_obj._w_layers = st.weights(c)        # fresh arrays: logged samples keep their own copies
        ind = fi = None
        if g.freq_indicator or g.use_fi:
            ind, fi = indicators if indicators is not None else \
                g.eng.read_indicators(weight=bool(g.freq_indicator), feature=g.use_fi)
            if ind is not None:
                bnn_obj._indicators = ind[c]
            if fi is not None:
                bnn_obj._feature_indicators = fi[c].astype(int)
        # what a pickle of this sampler needs to continue the chain (_restage): the raw state rows (accept ring,
        # counters, update sizes, temperature, slopes, sigma, iteration), the indicators and the device additional_prob.
        # Fresh arrays and a fresh dict at every sync: the background pickle writer holds shallow copies of earlier ones.
        self._chain_state = {"f64": np.array(st.f64[c]), "i32": np.array(st.i32[c]),
                             "ind": None if ind is None else ind[c], "fi": None if fi is None else fi[c],
                             "add_prob": self._dev_add_prob}
        # the host generator as of this point: the next slice's draws advance _rs in place before the writer pickles
        self._rs_state = self._rs.bit_generator.state
        self._bnn_view = bnn_obj
        self._y_cache = {}

    # mcmc._y / mcmc._y_test (BNN_env.py:299,343,507,513): the prediction tables of the current state.  The sampler never
    # needs them on the host (likelihood and accuracies are reduced inside the forward kernel); they are produced by one
    # prediction pass when a script reads the attribute and cached until the state changes.
    @property
    def _y(self):
        if "y" not in self._y_cache:
            self._y_cache["y"] = self._materialise_y(self._bnn_view, False)
        return self._y_cache["y"]

    @property
    def _y_test(self):
        if "y_test" not in self._y_cache:
            self._y_cache["y_test"] = self.y_test(self._bnn_view)
        return self._y_cache["y_test"]

    def _materialise_y(self, bnn_obj, test=False):
        x = bnn_obj._test_data if test else bnn_obj._data
        al = bnn_obj._act_fun.alphas(bnn_obj._n_layers)
        w = bnn_obj._w_layers
        if bnn_obj._freq_indicator:
            w = [w[0] * bnn_obj._indicators] + list(w[1:])
        ov = None
        if bnn_obj._feature_indicators is not None:
            cols, vals = data_transform_obj(bnn_obj._feature_indicators, bnn_obj._feature_means).override()
            ov = (cols, vals) if len(cols) else None
        out = self._group.eng.predict(x, [w], alphas=None if al is None else al[None, :], override=ov, mean=False, dense=True)
        return out["dense"][0]

    # `_y` / `_y_test` (N x K predictions of the current state, BNN_env.py:299,507) are materialised on demand
    def y(self, bnn_obj):
        return self._materialise_y(bnn_obj, False)

    def y_test(self, bnn_obj):
        return self._materialise_y(bnn_obj, True) if _has_test(bnn_obj) else []

    def _check_supported(self, n_steps):
        if self._regression_error_proposal and self._current_iteration + n_steps - 1 > self._estimate_error:
            # the reference itself cannot take this branch once any proposal has been accepted: accepts before
            # _estimate_error reset error_prm to the scalar 1 and multiplier_proposal_vector(1, ...) raises
            # AttributeError (BNN_mcmc.py:105) -- measured, tests/golden/make_golden.py
            raise NotImplementedError("the regression error-parameter proposal (BNN_env.py:435-442) is not on the device path; "
                                      "use empirical_error=True or estimate_error=False")

    # ---------------------------------------------------------------- stepping
    def run(self, bnn_obj, n_steps, additional_prob=0):
        """n_steps MH iterations (BNN_env.py:381-532 each) with as few host round trips as the rng mode allows."""
        if self._group is None:
            self._restage(bnn_obj)
        self._check_supported(n_steps)
        if bnn_obj.__dict__.get("_data_version", 0) != self._seen_version:
            raise RuntimeError("npBNN.update_data / reset_weights was called after this MCMC staged the model on the device; "
                               "construct a new MCMC (the device state would silently ignore the change)")
        g = self._group
        if not self._own_group:
            raise RuntimeError("this MCMC belongs to an MC3 group; step the group instead")
        if self._rng_mode == "philox":
            self._set_device_additional_prob(additional_prob)
        done = 0
        while done < n_steps:
            if self._rng_mode == "philox":
                g.eng.mh_steps(n_steps - done)
                done = n_steps
            else:
                st = g.eng.read_state(weights=False)
                it = int(st.iteration[0])
                # the adaptation of iteration `it` happens on the device before the draw is used; mirror it on
                # the host copy of the state so that the draw uses the post-adaptation sizes
                _mirror_adaptation(st, 0, it, self._adapt_freq, self._adapt_stop, self._adapt_f, self._adapt_fM,
                                   self._max_n, int(np.sum(self._max_n)))
                k = min(n_steps - done, _steps_to_adaptation(it, self._adapt_freq, self._adapt_stop))
                reseed = (lambda cid, i: np.random.default_rng(i + self._mcmc_id)) if self._randomize_seed else None
                inj = g.draw_steps([self._rs], st, [self._mcmc_id], k, reseed, additional_prob, adapt_stop=self._adapt_stop)
                g.eng.mh_steps(k, inj)
                done += k
        self._sync(bnn_obj, g.eng.read_state())

    def _set_device_additional_prob(self, a):
        """Device-drawn proposals read additional_prob from the chain's device value: copy it there when it changes."""
        a = float(a)
        if a != self._dev_add_prob:
            self._group.eng.set_additional_prob([a])
            self._dev_add_prob = a

    def mh_step(self, bnn_obj, additional_prob=0, return_bnn=False):
        self.run(bnn_obj, 1, additional_prob)
        if return_bnn:
            return bnn_obj, self

    def gibbs_step(self, bnn_obj):
        """BNN_env.py:534-538: new prior scales from their conditional posterior (host draw, sample_prior_scale), then
        logPrior / logPost of the current weights under them (device) and one iteration counted."""
        if not self._own_group:
            raise RuntimeError("this MCMC belongs to an MC3 group")
        if self._group is None:
            self._restage(bnn_obj)
        bnn_obj.sample_prior_scale()
        eng = self._group.eng
        eng.set_prior_scales(bnn_obj._entry_scales()[None, :])
        st = eng.read_state(weights=False)
        st.i32[:, L.I_ITERATION] += 1
        eng.write_state(st)
        self._sync(bnn_obj, eng.read_state())

    def _edit_state(self, edit):
        if not self._own_group:
            raise RuntimeError("this MCMC belongs to an MC3 group")
        if self._group is None and "_chain_state" in self.__dict__:
            # unpickled and not restaged yet: edit the saved rows, which the restaging writes to the device
            cs = dict(self._chain_state)
            st = SimpleNamespace(f64=cs["f64"][None].copy(), i32=cs["i32"][None].copy())
            edit(st)
            cs["f64"], cs["i32"] = st.f64[0], st.i32[0]
            self._chain_state = cs
            return
        eng = self._group.eng
        st = eng.read_state(weights=False)
        edit(st)
        eng.write_state(st)

    # BNN_env.py:540-547.  The reference only rebinds the attribute; here the value also goes to the device state.
    def reset_update_n(self, n):
        n = np.asarray(n).astype(int)
        self._update_n = n
        self._edit_state(lambda st: st.i32.__setitem__((slice(None), slice(L.I_UPDATE_N, L.I_UPDATE_N + len(n))), n))

    def reset_update_f(self, f):
        f = np.asarray(f, dtype=np.float64)
        self._update_f = f
        self._edit_state(lambda st: st.f64.__setitem__((slice(None), slice(L.F_UPDATE_F, L.F_UPDATE_F + len(f))), f))

    def reset_update_ws(self, w):
        ws = []
        for m in w:
            m = np.asarray(m, dtype=np.float64)
            if m.size > 1 and not np.all(m == m.flat[0]):
                raise NotImplementedError("per-weight proposal widths are not on the device path (one width per layer)")
            ws.append(float(m.flat[0]))
        self._update_ws = [np.ones(s) * ws[i] for i, s in enumerate(self._bnn_shapes)]
        ws = np.asarray(ws)
        self._edit_state(lambda st: st.f64.__setitem__((slice(None), slice(L.F_UPDATE_WS, L.F_UPDATE_WS + len(ws))), ws))

    def reset_temperature(self, temp):
        self._temperature = temp
        if self._own_group and self._group is None:
            self._edit_state(lambda st: st.f64.__setitem__((slice(None), L.F_TEMPERATURE), temp))
        elif self._own_group:
            self._group.eng.set_temperature([temp])

    # ---------------------------------------------------------------- pickling and resuming
    # postLogger pickles the live [bnn, mcmc, logger] at every sample (BNN_env.py:658); as in the reference,
    # load_obj(pkl) -> raise mcmc._n_iterations -> run_mcmc(bnn, mcmc, logger) continues the chain.  The pickle holds no
    # device handle: the first step of an unpickled sampler stages the model again (_restage) and writes the state saved
    # at the last sync, so the chain continues bit for bit (device generators are keyed on seed, chain and iteration).
    def __getstate__(self):
        d = dict(self.__dict__)
        d["_group"] = None
        d["update_function"] = None
        d["_bnn_view"] = None
        d["_y_cache"] = {}
        if "_rs_state" in d:
            # the host generator travels as its state as of the last sync (the live one may have advanced since) and is
            # rebuilt on first use (__getattr__): a logging point's shallow copy builds no generator
            d.pop("_rs", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self.update_function = UpdateNormal

    def __getattr__(self, name):
        # only reached for attributes the instance lacks: _rs of an unpickled sampler
        if name == "_rs" and "_rs_state" in self.__dict__:
            rs = np.random.default_rng(0)
            rs.bit_generator.state = self.__dict__["_rs_state"]
            self.__dict__["_rs"] = rs
            return rs
        raise AttributeError(name)

    def _restage(self, bnn_obj):
        """Rebuild the device chain of an unpickled sampler from the pickled model (data, weights, mask, prior scales,
        feature means) and this sampler's settings, then write its saved state (_ChainGroup(saved=))."""
        if "_chain_state" not in self.__dict__:
            raise RuntimeError("this MCMC was pickled without its chain state (by a version that could not resume "
                               "samplers): rebuild it from npBNN(pickle_file=...), which restores the last weights")
        if not self._own_group:
            raise RuntimeError("this MCMC is a chain of an MC3 group (the cold chain its logger pickles): unpickle and "
                               "run the MC3 object to resume the chains")
        if self._row_sharded:
            raise NotImplementedError("resuming a row-sharded MCMC is not built: only rank 0 writes the pickle, and it "
                                      "holds rank 0's own chains alone")
        cs = self._chain_state
        nl = bnn_obj._n_layers
        count_kind = _COUNT_LIK[self._likelihood_f][0] if self._likelihood_f in _COUNT_LIK else None
        self._group = _ChainGroup(bnn_obj, [bnn_obj._w_layers], [float(cs["f64"][L.F_TEMPERATURE])],
                                  list(cs["f64"][L.F_UPDATE_F:L.F_UPDATE_F + nl]),
                                  list(cs["f64"][L.F_UPDATE_WS:L.F_UPDATE_WS + nl]), self._lik_temp, self._adapt_f,
                                  self._adapt_fM, self._adapt_freq, self._adapt_stop, self._sample_from_prior,
                                  seed=int(bnn_obj._seed) + 7919 * int(self._mcmc_id), device=self._device,
                                  lik=count_kind, saved=[cs])
        self._bnn_view = bnn_obj


def _mirror_adaptation(st, c, it, adapt_freq, adapt_stop, adapt_f, adapt_fM, max_n, n_params):
    """Host copy of the adaptation block (BNN_env.py:392-413) applied to the exported state of chain c, so that
    host-drawn proposals use the sizes the device will use in iteration `it`."""
    if it % adapt_freq == 0 and it < adapt_stop:
        ar = st.acceptance_rate[c]
        if ar < adapt_f:
            st.freq_layer_update[c] *= 0.8
            st.update_f[c] *= 0.85
            n = (max_n * st.update_f[c]).astype(int)
            n[n < 1] = 1
            st.update_n[c] = n
            st.update_ws[c] *= 0.9
        if ar > adapt_fM and np.sum(st.update_n[c]) < n_params:
            st.update_f[c] = np.exp(np.log(st.update_f[c]) * 0.85)
            n = (max_n * st.update_f[c]).astype(int)
            n[n < 1] = 1
            st.update_n[c] = n
            st.update_ws[c] *= 1.2


def _report(bnn, mcmc, logger):
    """Print / log decisions of the reference's loop for the state just synchronised (BNN_mcmc.py:156-167)."""
    if (mcmc._current_iteration % mcmc._print_f == 0 or mcmc._current_iteration == 1) and _is_rank0():
        print(mcmc._current_iteration, np.round([mcmc._logLik, mcmc._accuracy, mcmc._test_accuracy,
                                                  mcmc._acceptance_rate], 3), flush=True)
        if bnn._estimation_mode == "regression":
            print(bnn._error_prm)
    if mcmc._current_iteration % mcmc._sampling_f == 0:
        logger.log_sample(bnn, mcmc)
        logger.log_weights(bnn, mcmc)


def _next_stop(mcmc, it):
    nxt = [mcmc._n_iterations]
    if it == 0:
        nxt.append(1)                                  # the reference prints at iteration 1
    nxt.append((it // mcmc._print_f + 1) * mcmc._print_f)
    nxt.append((it // mcmc._sampling_f + 1) * mcmc._sampling_f)
    return max(1, min(nxt) - it)


def _run_mcmc_pipelined(bnn, mcmc, logger, depth):
    """Free-running chains (rng="philox"): the host queues the MH launches up to `depth` logging points ahead and
    exports each logging point through the asynchronous snapshot ring (bnn_chains_snapshot), so printing, csv rows
    and pickles are written while the device keeps stepping (SURVEY.md 8f-4).  Same decisions, same samples and
    the same files as the synchronous loop."""
    from collections import deque
    eng = mcmc._group.eng
    mcmc._set_device_additional_prob(0)      # the loop's mh_step passes none (BNN_mcmc.py:153-170)
    it = mcmc._current_iteration
    pending, free = deque(), list(range(depth))
    if hasattr(logger, "begin_async"):
        logger.begin_async()

    g = mcmc._group

    def retire():
        slot = pending.popleft()
        # the indicators of the snapshot's iteration: the live ones already belong to the steps queued behind it
        ind = eng.snapshot_read_indicators(slot, weight=bool(g.freq_indicator), feature=g.use_fi) \
            if g.freq_indicator or g.use_fi else None
        mcmc._sync(bnn, eng.snapshot_read(slot), ind)
        free.append(slot)
        _report(bnn, mcmc, logger)

    while it < mcmc._n_iterations:
        k = _next_stop(mcmc, it)
        mcmc._check_supported(k)
        eng.mh_steps(k)
        it += k
        if not free:
            retire()
        slot = free.pop()
        eng.snapshot(slot)
        pending.append(slot)
    try:
        while pending:
            retire()
    finally:
        if hasattr(logger, "end_async"):
            logger.end_async()


def run_mcmc(bnn, mcmc, logger, pipeline_depth=4):
    """The driver loop of BNN_mcmc.py:153-170, batched: the device runs up to the next print / sampling /
    final iteration without returning to the host; with device-generated proposals (rng="philox") the logging
    points are exported asynchronously and the loop never waits for the device (pipeline_depth=0: synchronous).
    An unpickled mcmc continues its chain (MCMC._restage)."""
    if mcmc._group is None:
        mcmc._restage(bnn)
    if mcmc._rng_mode == "philox" and mcmc._own_group and pipeline_depth > 0 and mcmc._current_iteration < mcmc._n_iterations:
        return _run_mcmc_pipelined(bnn, mcmc, logger, int(pipeline_depth))
    # host-drawn proposals: the loop returns to the host at every logging point anyway, but the pickle of
    # [bnn, mcmc, logger] (X included, rewritten at every sample) still goes to the background writer
    if pipeline_depth > 0 and hasattr(logger, "begin_async"):
        logger.begin_async()
    try:
        while True:
            it = mcmc._current_iteration
            mcmc.run(bnn, _next_stop(mcmc, it))
            _report(bnn, mcmc, logger)
            if mcmc._current_iteration >= mcmc._n_iterations:
                break
    finally:
        if pipeline_depth > 0 and hasattr(logger, "end_async"):
            logger.end_async()


def _chain_view(bnn):
    """A per-chain copy of the model object that SHARES the row-sized read-only arrays (features, labels, sample ids,
    instance weights) with the original: the reference deep-copies / pickles the whole object per chain
    (BNN_mc3.py:42-47), which at BASELINE config 4 is 32 x 512 MB of host memory and 4 s for views whose data nobody
    writes (update_data rebinds the attributes).  Weights, indicators, prior scales ... stay private copies."""
    memo = {}
    for k in ("_data", "_labels", "_test_data", "_test_labels", "_sample_id", "_instance_weights", "_instance_id"):
        v = bnn.__dict__.get(k)
        if isinstance(v, np.ndarray):
            memo[id(v)] = v
    return deepcopy(bnn, memo)


class MC3:
    """Metropolis-coupled chains (BNN_mc3.py:8-126).  All chains live on the GPU(s); there is no fork pool
    and nothing is pickled between swap periods.  With torch.distributed initialised the ranks form Q chain blocks x
    R row shards (mc3.chain_grid): the chains are sharded over the blocks, the R ranks of a block split its rows
    (rowshard.py), and the swap step all-gathers the log-posteriors (npbnn_b200/mc3.py)."""

    R = 1          # row shards per chain block

    def __init__(self, data, logger, n_post_samples=100, sampling_f=100, n_chains=4, swap_frequency=100, verbose=1,
                 print_f=100, temperatures=None, min_temperature=0.8, likelihood_f=None, accuracy_f=None, adapt_freq=50,
                 adapt_f=0.1, adapt_fM=0.6, adapt_stop=1000, n_iteration=100000, rng="host", device=0, swap_seed=None):
        count_kind, _ = _count_likelihood(data, likelihood_f, accuracy_f, None)
        import torch.distributed as dist
        self.n_chains = n_chains
        self.swap_frequency = swap_frequency
        self.verbose = verbose
        self.print_f = print_f / swap_frequency
        self.n_post_samples = n_post_samples
        self.sampling_f = sampling_f
        self.adapt_freq, self.adapt_f, self.adapt_fM, self.adapt_stop = adapt_freq, adapt_f, adapt_fM, adapt_stop
        self.n_mc3_iteration = np.round(n_iteration / swap_frequency).astype(int)
        self.rseeds = np.random.choice(range(1000, 9999), n_chains, replace=False)     # BNN_mc3.py:44
        if data._estimation_mode == "regression" and not data._empirical_error:
            # MC3 builds its chains with estimate_error=True and n_iteration=swap_frequency (BNN_mc3.py:61-74), so the
            # error-parameter proposal starts after 0.1 * swap_frequency iterations -- the branch that is not on the device
            # path (and on which the reference raises AttributeError after the first accept, BNN_mcmc.py:105)
            raise NotImplementedError("MC3 on a regression model needs empirical_error=True (the error-parameter proposal "
                                      "of BNN_env.py:435-442 is not on the device path)")
        if temperatures is None:
            temperatures = _mc3.default_temperatures(n_chains, min_temperature)
        self.temperatures = np.array(temperatures, dtype=np.float64)
        self.logger = logger
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank() if self.world > 1 else 0
        self.Q, self.R = _mc3.chain_grid(n_chains, self.world)
        q, r = divmod(self.rank, self.R)
        if self.R > 1 and rng == "host" and (data._freq_indicator or data._feature_indicators is not None):
            # the indicator flips come from numpy's global generator (_ChainGroup.draw_steps), whose state differs
            # between the ranks of a block
            raise NotImplementedError("MC3 with more ranks (%d) than chains (%d) and rng='host' does not run weight or "
                                      "feature indicators; use rng='philox'" % (self.world, n_chains))
        if self.world > 1:
            # every rank must hold the same chain seeds and swap generator whatever its own numpy state is
            self.rseeds = np.asarray(_mc3.broadcast_from_rank0(self.rseeds))
        self.start, self.n_local = _mc3.chain_partition(n_chains, self.Q, q)
        row_group = None
        if 1 < self.R < self.world:
            from .predshard import block_group
            row_group = block_group(self.world, self.R, q)
        self._rng_mode = rng
        if swap_seed is None and self.world == 1:
            self._swap_rng = _mc3.GlobalSwapRNG()      # the reference's own stream (np.random, BNN_mc3.py:99,109)
        else:
            self._swap_rng = _mc3.SwapRNG(int(self.rseeds[0]) if swap_seed is None else int(swap_seed))
        nl = data._n_layers
        self._bnn = data
        self._device = device
        self._group = _ChainGroup(data, [data._w_layers] * self.n_local,
                                  self.temperatures[self.start:self.start + self.n_local], [0.05] * nl, [0.075] * nl,
                                  1, adapt_f, adapt_fM, adapt_freq, adapt_stop, 0, seed=int(self.rseeds[0]), device=device,
                                  row_shard=(self.R, r), row_group=row_group, chain_offset=self.start, lik=count_kind)
        # per-chain views with the reference's attribute surface (singleChainArgs[i] = [bnn, mcmc])
        self.singleChainArgs = []
        for i in range(self.n_local):
            b = _chain_view(data)
            b.reset_seed(self.rseeds[self.start + i])
            m = MCMC(b, temperature=self.temperatures[self.start + i], n_iteration=swap_frequency, sampling_f=sampling_f,
                     print_f=swap_frequency * 10, n_post_samples=n_post_samples, mcmc_id=self.start + i, randomize_seed=True,
                     adapt_freq=adapt_freq, adapt_f=adapt_f, adapt_fM=adapt_fM, adapt_stop=adapt_stop, rng=rng,
                     likelihood_f=likelihood_f, accuracy_f=accuracy_f, _group=self._group, _slot=i)
            self.singleChainArgs.append([b, m])
        self.current_temperatures = self.temperatures.copy()

    def _run_period(self):
        g = self._group
        n = self.swap_frequency
        if self._rng_mode == "philox":
            g.eng.mh_steps(n)
            return
        mc0 = self.singleChainArgs[0][1]
        max_n = mc0._max_n
        done = 0
        while done < n:
            st = g.eng.read_state(weights=False)
            it = int(st.iteration[0])
            for c in range(self.n_local):
                _mirror_adaptation(st, c, it, self.adapt_freq, self.adapt_stop, self.adapt_f, self.adapt_fM, max_n,
                                   int(np.sum(max_n)))
            k = min(n - done, _steps_to_adaptation(it, self.adapt_freq, self.adapt_stop))
            # randomize_seed=True: every step reseeds default_rng(iteration + mcmc_id) (BNN_env.py:383-384), so the
            # draws of an iteration depend on nothing but (iteration, chain) and the adaptation state read above
            def draw(s0, m):
                return g.draw_steps([None] * self.n_local, st, [self.start + c for c in range(self.n_local)], m,
                                    reseed=lambda cid, i: np.random.default_rng(i + cid), adapt_stop=self.adapt_stop,
                                    step0=s0)
            # slices: many on large data (the first slice's draw is the only one the device waits for), few on small
            # data, where every bnn_mh_steps call costs about as much as several device iterations
            sub = max(4, k // (16 if self._bnn._n_samples >= 20000 else 4))
            if k <= sub or g.freq_indicator or g.use_fi:      # (the indicator moves consume numpy's GLOBAL generator
                g.eng.mh_steps(k, draw(0, k))                  #  chain by chain: keep that order)
            else:
                # The host needs ~80 us per (chain, iteration) for the reference's generator calls -- 0.26 s per 100
                # iterations of 32 chains, 15 % of the device time at BASELINE config 4: a worker thread draws slice
                # j + 1 while this thread waits inside bnn_mh_steps for slice j (ctypes releases the GIL).
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(max_workers=1) as pool:
                    s0 = 0
                    fut = pool.submit(draw, 0, min(sub, k))
                    while s0 < k:
                        m = min(sub, k - s0)
                        inj = fut.result()
                        s0 += m
                        if s0 < k:
                            fut = pool.submit(draw, s0, min(sub, k - s0))
                        g.eng.mh_steps(m, inj)
            done += k

    def run_mcmc(self):
        # The reference rewrites the [bnn, mcmc, logger] pickle -- the feature matrix included, 512 MB at BASELINE config 4
        # -- after every swap period (BNN_mc3.py:118-122 -> BNN_env.py:658).  As in run_mcmc above the writes go to the
        # logger's background writer (newest snapshot wins, the last one is on disk when this returns) so that the
        # device does not idle while the host pickles: tools/mc3_api_c4.py.
        if self._group is None:
            self._restage()
        lg = self.logger if hasattr(self.logger, "begin_async") and self.__dict__.get("async_pickle", True) else None
        if lg is not None:
            lg.begin_async()
        try:
            self._run_mcmc()
        finally:
            if lg is not None:
                lg.end_async()

    def _run_mcmc(self):
        g = self._group
        for mc3_it in range(self.n_mc3_iteration):
            self._run_period()
            if self.n_chains > 1:
                temps, swapped, (j, k), lp = _mc3.exchange(g.eng.gather(L.F_LOGPOST), self.current_temperatures,
                                                           self._swap_rng, None, self.world, self.R)
                if swapped:
                    if self.verbose > 0 and self.rank == 0:
                        print(mc3_it, "SWAPPED", lp[j], lp[k], self.current_temperatures[j], self.current_temperatures[k])
                    self.current_temperatures = temps
                    g.eng.set_temperature(temps[self.start:self.start + self.n_local])
            st = g.eng.read_state()
            cold = None
            for i, (b, m) in enumerate(self.singleChainArgs):
                m._sync(b, st)
                if m._temperature == 1:                     # the logger follows the cold chain (BNN_mc3.py:118-122)
                    cold = (b, m)
            self._log_on_rank0(cold)
            if mc3_it % self.print_f == 0 and self.rank == 0 and self.n_local:
                b0, m0 = self.singleChainArgs[0]
                print(mc3_it, m0._logPost, b0._w_layers[0][0][0:5])


    # A pickled MC3 holds its chain views (each [bnn, mcmc] with its saved state, MCMC._chain_state), the temperatures,
    # the logger and the swap generator (a seeded SwapRNG pickles its state); the next run_mcmc continues every chain.
    # A single-process MC3 without swap_seed draws its swaps from numpy's global generator, as the reference does
    # (GlobalSwapRNG), and so do host-drawn indicator flips: to continue those streams the caller restores np.random's
    # state (np.random.set_state) before run_mcmc; unpickling neither saves nor touches it.
    def __getstate__(self):
        d = dict(self.__dict__)
        d["_group"] = None
        d.pop("_cold_view", None)
        return d

    def _restage(self):
        """One chain group from the chain views of an unpickled MC3: each view's weights and saved state."""
        import torch.distributed as dist
        if self.world > 1 or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            raise NotImplementedError("resuming MC3 over torch.distributed ranks is not built: only rank 0 writes the "
                                      "pickle, and it holds rank 0's own chains alone")
        views = self.singleChainArgs
        m0 = views[0][1]
        count_kind = _COUNT_LIK[m0._likelihood_f][0] if m0._likelihood_f in _COUNT_LIK else None
        nl = self._bnn._n_layers
        self._group = _ChainGroup(self._bnn, [b._w_layers for b, _ in views], [m._temperature for _, m in views],
                                  [0.05] * nl, [0.075] * nl, 1, self.adapt_f, self.adapt_fM, self.adapt_freq,
                                  self.adapt_stop, 0, seed=int(self.rseeds[0]), device=self._device,
                                  chain_offset=self.start, lik=count_kind, saved=[m._chain_state for _, m in views])
        for b, m in views:
            m._group, m._bnn_view = self._group, b

    def _log_on_rank0(self, cold):
        """The logger follows the cold chain (`cold`: this rank's (bnn, mcmc) at temperature 1, or None), and the files
        belong to rank 0.  In a single process, and whenever rank 0 holds the cold chain, rank 0 logs its own chain.
        Chains sharded over ranks: the cold temperature migrates between ranks with the swaps, and the r = 0 rank of the
        block holding the cold chain sends its exported state (statistics + weights, a few kB) to rank 0, which is the
        only rank that writes the .log / .pkl and keeps the posterior sample list."""
        import torch.distributed as dist
        cold_chain = int(np.flatnonzero(self.current_temperatures == 1)[0]) if np.any(self.current_temperatures == 1) else -1
        if cold_chain < 0:
            return
        owner = _mc3.owner_of(cold_chain, self.n_chains, self.world, self.R)
        box = [None]
        if owner != 0 and self.rank == owner:          # only a state that travels is exported
            b, m = cold
            box[0] = {"bnn": {k: getattr(b, k) for k in ("_w_layers", "_indicators", "_error_prm", "_feature_indicators",
                                                          "_prior_scale", "_seed")},
                      "act_prm": (b._act_fun._prm, b._act_fun._acc_prm),
                      "mcmc": {k: v for k, v in m.__getstate__().items() if k not in ("_likelihood_f", "_accuracy_f",
                                                                                      "_accuracy_lab_f")}}
        if owner != 0:
            dist.broadcast_object_list(box, src=owner)
        if self.rank != 0:
            return
        if owner == 0:
            b, m = cold
        else:
            if getattr(self, "_cold_view", None) is None:
                b = _chain_view(self._bnn)
                m = object.__new__(MCMC)
                self._cold_view = (b, m)
            b, m = self._cold_view
            for k, v in box[0]["bnn"].items():
                setattr(b, k, v)
            b._act_fun._prm, b._act_fun._acc_prm = box[0]["act_prm"]
            m.__dict__.update(box[0]["mcmc"])
        self.logger.log_sample(b, m)
        self.logger.log_weights(b, m)


# ------------------------------------------------------------------------------------------------------
# prediction callers
# ------------------------------------------------------------------------------------------------------
def _lik_of_output(output_act_fun):
    if output_act_fun is RegressTransformError:
        return L.LIK_GAUSSIAN_HEAD
    if output_act_fun is RegressTransform:
        return L.LIK_GAUSSIAN
    if output_act_fun is SoftMax or output_act_fun is None:
        return L.LIK_CATEGORICAL
    raise NotImplementedError("user-supplied output_act_fun is not on the device path")


_ENGINE_CACHE = {}


def _predict_engine(weights, n_features, actFun, output_act_fun):
    """The cached prediction engine of a network shape: on GPU 0 in a single process, on the rank's current device
    (torch.cuda.set_device of a torchrun script) under a process group of several ranks."""
    import torch
    device = torch.cuda.current_device() if predshard.ranks()[0] > 1 else 0
    key = (tuple(tuple(w.shape) for w in weights), n_features, actFun._function, _lik_of_output(output_act_fun), device)
    if key not in _ENGINE_CACHE:
        _ENGINE_CACHE[key] = Engine(NetShape.from_weights(weights, n_features, act=actFun._function,
                                                          lik=_lik_of_output(output_act_fun)), device=device)
    return _ENGINE_CACHE[key]


def _alpha_rows(post_alphas, actFun, n_layers):
    if actFun._function != "genReLU":
        return None
    rows = []
    for a in post_alphas:
        r = np.zeros(n_layers)
        a = np.atleast_1d(np.asarray(a, dtype=np.float64))
        r[:min(len(a), n_layers)] = a[:n_layers]
        rows.append(r)
    return np.stack(rows)


class data_transform_obj:
    """BNN_env.py:9-17: features whose indicator is 0 are replaced by their training mean.  On the device the
    replacement is a column override applied while X is packed (k_pack_x), the same mechanism as the PDP grid."""

    def __init__(self, feature_indicators, feature_means):
        self.feature_indicators = feature_indicators
        self.feature_means = feature_means

    def transform(self, x):
        """Host form (BNN_env.py:14-17) for callers that hand the object to RunHiddenLayer."""
        cols, vals = self.override()
        x = np.array(x, dtype=np.float64, copy=True)
        x[:, cols] = vals
        return x

    def override(self):
        cols = np.flatnonzero(np.asarray(self.feature_indicators) == 0).astype(np.int32)
        return cols, np.asarray(self.feature_means, dtype=np.float64)[cols]


def RunPredict(data, weights, actFun, output_act_fun, data_transform=None):
    """Forward pass of one weight set (BNN_lib.py:245-256) -> [N, O]."""
    data = np.ascontiguousarray(data, dtype=np.float64)
    eng = _predict_engine(weights, data.shape[1], actFun, output_act_fun)
    al = _alpha_rows([actFun._prm], actFun, len(weights))
    ov = None
    if data_transform is not None:
        cols, vals = data_transform.override()
        ov = (cols, vals) if len(cols) else None
    return eng.predict(data, [weights], alphas=al, override=ov, mean=False, dense=True)["dense"][0]


def RunPredictInd(data, weights, ind, actFun, output_act_fun, data_transform=None):
    """BNN_lib.py:258-272: layer-0 weights multiplied by the indicator matrix."""
    w = [weights[0] * ind] + list(weights[1:])
    return RunPredict(data, w, actFun, output_act_fun, data_transform)


def predict(bnn_obj, data):
    """BNN_env.py:662-670."""
    return RunPredict(data, bnn_obj._w_layers, actFun=bnn_obj._act_fun, output_act_fun=bnn_obj._output_act_fun)


_HOST_UNIFORM_LIMIT = 1 << 26       # n x S above which mode 2 draws its uniforms inside the kernel (512 MB of float64)


def _sampling_kind(n, s, rng):
    """rng=None picks "host" while the (N, S) array of uniforms stays below 512 MB and "philox" beyond (BASELINE config
    5: 80 GB)."""
    if rng is None:
        return "host" if n * s <= _HOST_UNIFORM_LIMIT else "philox"
    if rng not in ("host", "philox"):
        raise ValueError("rng must be None, 'host' or 'philox'")
    return rng


def _sampling_uniforms(n, s, rng):
    """(u, seed) of the posterior-predictive resampling.  rng="host": the reference's draw -- np.random.random(S) per
    instance in instance order = one (N, S) draw from the global stream (reproduces the reference for a seeded run).
    rng="philox": uniforms generated inside the kernel, seeded from the global stream, O(1) extra memory.  rng=None:
    _sampling_kind."""
    if _sampling_kind(n, s, rng) == "host":
        return np.random.random((n, s)), None
    return None, int(np.random.randint(0, 2 ** 31 - 1)) * 2654435761 + 1


def get_posterior_cat_prob(pred_features, post_samples=None, feature_index_to_shuffle=None, post_summary_mode=0,
                           unlink_features_within_block=False, actFun=None, output_act_fun=None, return_dense=True,
                           rng=None):
    """BNN_lib.py:352-397 with all posterior samples scored in ONE pass over the features.
    return_dense=False skips the [S, N, K] tensor (it is 800 GB at BASELINE config 5) and returns None for it.  Mode 2
    resamples as sample_from_categorical (BNN_lib.py:682-713), inside the prediction kernel."""
    if len(pred_features) == 0:
        print("Data not found.")
        return 0
    if post_summary_mode not in (0, 1, 2):
        raise ValueError("post_summary_mode must be 0 (argmax votes), 1 (mean softmax) or 2 (categorical resampling)")
    x = np.ascontiguousarray(pred_features, dtype=np.float64)
    weights = [s["weights"] for s in post_samples]
    eng = _predict_engine(weights[0], x.shape[1], actFun, output_act_fun)
    al = _alpha_rows([s["alphas"] for s in post_samples], actFun, len(weights[0]))
    n, S = x.shape[0], len(weights)
    shuffle = []
    if feature_index_to_shuffle:
        if unlink_features_within_block and type(feature_index_to_shuffle) == list:
            shuffle = list(feature_index_to_shuffle)
        else:
            shuffle = [feature_index_to_shuffle]
    sample = _sampling_kind(n, S, rng) if post_summary_mode == 2 else None

    def draw():
        # the reference's order: the permutations of the shuffled blocks, then the uniforms (np.random.permutation(N)
        # makes the draws np.random.permutation(x[:, fi]) makes)
        perms = [np.random.permutation(n) for _ in shuffle]
        u, seed = _sampling_uniforms(n, S, sample) if sample else (None, None)
        return perms, u, seed

    out = predshard.predict_ranks(eng, x, weights, al, mean=post_summary_mode == 1, votes=post_summary_mode == 0,
                                  dense=return_dense, sample=sample, shuffle=shuffle, draw=draw)
    summary = {0: "votes", 1: "mean", 2: "predictions"}[post_summary_mode]
    return out.get("dense"), out[summary]


def sample_from_categorical(pred_features, post_samples, actFun=None, output_act_fun=None, rng=None,
                            post_predictions=True):
    """Posterior-predictive resampling with the outputs of the reference's sample_from_categorical
    (BNN_lib.py:682-713: 'predictions', 'class_counts', 'post_predictions'), computed from the features and the
    posterior samples in one device pass instead of from a materialised [S, N, K] probability tensor."""
    x = np.ascontiguousarray(pred_features, dtype=np.float64)
    weights = [s["weights"] for s in post_samples]
    eng = _predict_engine(weights[0], x.shape[1], actFun, output_act_fun)
    al = _alpha_rows([s["alphas"] for s in post_samples], actFun, len(weights[0]))
    n, S = x.shape[0], len(weights)
    sample = _sampling_kind(n, S, rng)
    return predshard.predict_ranks(eng, x, weights, al, sample=sample, post_predictions=post_predictions,
                                   draw=lambda: ([],) + _sampling_uniforms(n, S, sample))


def feature_importance(input_features, weights_pkl=None, weights_posterior=None, true_labels=[], fname_stem="",
                       feature_names=[], verbose=False, post_summary_mode=0, n_permutations=100, feature_blocks=dict(),
                       write_to_file=True, predictions_outdir="", unlink_features_within_block=True, actFun=None,
                       output_act_fun=None):
    """Permutation feature importance (BNN_lib.py:503-598): accuracy drop when a feature block is shuffled between
    instances, n_permutations times per block.  Every evaluation is ONE device pass over all posterior samples
    (get_posterior_cat_prob without the dense tensor); shuffling uses np.random.permutation like the reference, so
    the permutations are the reference's for the same global seed."""
    import pandas as pd
    feature_indices = np.arange(np.asarray(input_features).shape[1])
    if len(feature_names) == 0:
        feature_names = feature_indices.astype(str)
    if type(feature_blocks) is dict:
        if len(feature_blocks.keys()) > 0:
            selected_features, feature_block_names = list(feature_blocks.values()), list(feature_blocks.keys())
        else:
            selected_features = [[i] for i in feature_indices]
            feature_block_names = [i for i in feature_names]
    else:
        selected_features = feature_blocks
        feature_block_names = ["block_" + str(i) for i in range(len(feature_blocks))]
    if weights_pkl:
        bnn_obj, mcmc_obj, logger_obj = load_obj(weights_pkl)
        weights_posterior = logger_obj._post_weight_samples
        actFun, output_act_fun = bnn_obj._act_fun, bnn_obj._output_act_fun
    kw = dict(post_summary_mode=post_summary_mode, actFun=actFun, output_act_fun=output_act_fun, return_dense=False)
    _, pred = get_posterior_cat_prob(input_features, weights_posterior, **kw)
    ref_accuracy = CalcAccuracy(pred, true_labels)
    if verbose:
        print("Reference accuracy (mean):", np.mean(ref_accuracy))
    accuracies_wo_feature = []
    for block_id, feature_block in enumerate(selected_features):
        if verbose:
            print("Processing feature block %i", block_id + 1)
        accs = []
        for _ in np.arange(n_permutations):
            _, pred = get_posterior_cat_prob(input_features, weights_posterior, feature_index_to_shuffle=feature_block,
                                             unlink_features_within_block=unlink_features_within_block, **kw)
            accs.append(CalcAccuracy(pred, true_labels))
        accuracies_wo_feature.append(accs)
    accuracies_wo_feature = np.array(accuracies_wo_feature)
    delta_accs = ref_accuracy - accuracies_wo_feature
    df = pd.DataFrame({"feature_block_index": np.arange(len(selected_features)), "feature_name": list(feature_block_names),
                       "delta_acc_mean": np.mean(delta_accs, axis=1), "delta_acc_std": np.std(delta_accs, axis=1),
                       "acc_with_feature_randomized_mean": np.mean(accuracies_wo_feature, axis=1),
                       "acc_with_feature_randomized_std": np.std(accuracies_wo_feature, axis=1)})
    df = df.sort_values("delta_acc_mean", ascending=False)
    if write_to_file and _is_rank0():
        if predictions_outdir == "":
            predictions_outdir = os.path.dirname(weights_pkl) if weights_pkl else "."
        if not os.path.exists(predictions_outdir) and predictions_outdir != "":
            os.makedirs(predictions_outdir)
        stem = fname_stem + "_" if fname_stem != "" else ""
        path = os.path.join(predictions_outdir, stem + "feature_importance.txt")
        df.to_csv(path, sep="\t", index=False, header=True, float_format="%.6f")
        print("Output saved in: %s" % path)
    return df


def get_posterior_est(pkl_file):
    """BNN_lib.py:715-748."""
    bnn_obj, mcmc_obj, logger_obj = load_obj(pkl_file)
    ps = logger_obj._post_weight_samples
    weights = [s["weights"] for s in ps]
    res = {"error_prm": [s["error_prm"] for s in ps] if "error_prm" in ps[0] else []}
    for key, x in (("", bnn_obj._data), ("_test", bnn_obj._test_data)):
        if len(x) == 0:
            res["post_est" + key], res["prm_mean" + key] = np.array([]), np.nan
            continue
        x = np.ascontiguousarray(x, dtype=np.float64)
        eng = _predict_engine(weights[0], x.shape[1], bnn_obj._act_fun, bnn_obj._output_act_fun)
        al = _alpha_rows([s["alphas"] for s in ps], bnn_obj._act_fun, len(weights[0]))
        out = predshard.predict_ranks(eng, x, weights, al, mean=True, dense=True)
        res["post_est" + key], res["prm_mean" + key] = out["dense"], out["mean"]
    return res


def make_pdp_features(data, focal_features, steps_continuous=100):
    """The feature grid of a partial-dependence curve (BNN_pdp.py:14-45): ordinal / binary features step
    through their integer range, a single continuous feature through 100 equally spaced values, several
    focal features are treated as one-hot."""
    lo = np.array([np.nanmin(data[:, f]) for f in focal_features])
    hi = np.array([np.nanmax(data[:, f]) for f in focal_features])
    integer_like = [bool(np.all(np.isin(np.unique(data[:, f]), np.arange(l, h + 1)))) for f, l, h in zip(focal_features, lo, hi)]
    if len(focal_features) == 1 and not integer_like[0]:
        return np.linspace(lo[0], hi[0], num=steps_continuous).reshape(steps_continuous, 1)
    if len(focal_features) == 1:
        m = int(hi[0])
        return np.linspace(lo[0], m, num=m + 1).reshape((m + 1, 1))
    return np.eye(len(focal_features))


def get_pdp(data, focal_features, estimation_mode, size_output, actFun, output_act_fun, weights, alphas, data_transform):
    """Partial dependence (BNN_pdp.py:48-84).  Per grid step the focal columns are overwritten while X is
    staged (no host copy of the data), all posterior samples run in one pass and only the per-row mean over
    samples comes back: cumsum over classes, mean over rows and the 2.5 / 97.5 % row quantiles commute with it."""
    data = np.ascontiguousarray(data, dtype=np.float64)
    grid = make_pdp_features(data, focal_features)
    dt_cols, dt_vals = data_transform.override() if data_transform is not None else ([], [])
    out = np.zeros((grid.shape[0], size_output, 3))
    eng = _predict_engine(weights[0], data.shape[1], actFun, output_act_fun)
    al = _alpha_rows(alphas, actFun, len(weights[0]))
    for n in range(grid.shape[0]):
        # the grid value is written first, the feature-indicator transform inside RunPredict then replaces masked
        # features by their mean (BNN_pdp.py:65-73, BNN_lib.py:248-249): the transform wins on a shared column
        ov = dict(zip([int(f) for f in focal_features], [float(v) for v in grid[n, :]]))
        ov.update(zip([int(cc) for cc in dt_cols], [float(v) for v in dt_vals]))
        # every rank gets the full [N, K] mean: the row quantiles below need all rows
        smean = predshard.predict_ranks(eng, data, weights, al, override=(list(ov.keys()), list(ov.values())),
                                        mean=True)["mean"]
        if estimation_mode == "classification":
            smean = np.cumsum(smean, axis=1)
        out[n, :, 0] = np.mean(smean, axis=0)
        q = np.quantile(smean, q=(0.025, 0.975), axis=0)
        out[n, :, 1], out[n, :, 2] = q[0, :], q[1, :]
    return {"feature": grid, "pdp": out}


def pdp(pickle_file, pdp_features):
    """BNN_pdp.py:87-108."""
    bnn_obj, mcmc_obj, logger_obj = load_obj(pickle_file)
    ps = logger_obj._post_weight_samples
    weights, alphas = [s["weights"] for s in ps], [s["alphas"] for s in ps]
    dt = None
    if bnn_obj._feature_indicators is not None:
        dt = data_transform_obj(bnn_obj._feature_indicators, bnn_obj._feature_means)
    return [get_pdp(bnn_obj._data, f, bnn_obj._estimation_mode, bnn_obj._size_output, bnn_obj._act_fun,
                    bnn_obj._output_act_fun, weights, alphas, dt) for f in pdp_features]


# ------------------------------------------------------------------------------------------------------
# logger / pickle helpers the drivers need (I/O, host side; same file formats as BNN_env.py:553-658)
# ------------------------------------------------------------------------------------------------------
def SaveObject(obj, filename):
    with open(filename, "wb") as output:
        pickle.dump(obj, output, pickle.HIGHEST_PROTOCOL)


def _is_rank0():
    import torch.distributed as dist
    return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0


class postLogger:
    """Tab-separated .log of the chain statistics and a .pkl with [bnn, mcmc, logger] holding the last
    n_post_samples weight sets -- the formats predictBNN / pdp / npBNN(pickle_file=) consume."""

    def __init__(self, bnn_obj, filename="BNN", wdir="", sample_from_prior=0, add_prms=None, continue_logfile=False,
                 log_all_weights=0):
        self._writer = _is_rank0()        # under torch.distributed only rank 0 touches the files
        outdir = os.path.dirname(filename)
        if outdir and not os.path.exists(outdir) and self._writer:
            os.makedirs(outdir)
        stem = "%s_l%s" % (filename, "_".join(map(str, bnn_obj._n_nodes)))          # BNN_files.py:127
        self._logfile = os.path.join(wdir, stem + ".log")
        self._w_file = os.path.join(wdir, stem + "_W.log") if log_all_weights else None
        self._pklfile = os.path.join(wdir, stem + ".pkl")
        self._log_all_weights = log_all_weights
        self._post_weight_samples = []
        self._estimation_mode = bnn_obj._estimation_mode
        head = log_header(bnn_obj, add_prms)
        if not continue_logfile and self._writer:
            with open(self._logfile, "w", newline="") as f:
                csv.writer(f, delimiter="\t").writerow(head)
        if log_all_weights and self._writer:
            with open(self._w_file, "w", newline="") as f:
                csv.writer(f, delimiter="\t").writerow(
                    ["it"] + ["w_%s_%s" % (i, j) for i in range(bnn_obj._n_layers) for j in range(bnn_obj._w_layers[i].size)])

    def update_post_weight_samples(self, row):
        self._post_weight_samples += [row]

    def replace_post_weight_samples(self, post_weight_samples):
        self._post_weight_samples = post_weight_samples

    def control_weight_sample_length(self, maxlength):
        if len(self._post_weight_samples) > maxlength:
            self._post_weight_samples = self._post_weight_samples[-maxlength:]

    def log_sample(self, bnn_obj, mcmc_obj, add_prms=None):
        row = [mcmc_obj._current_iteration, mcmc_obj._logPost, mcmc_obj._logLik, mcmc_obj._logPrior, mcmc_obj._accuracy,
               mcmc_obj._test_accuracy] + list(mcmc_obj._label_acc)
        for i, w in enumerate(bnn_obj._w_layers):                                  # BNN_env.py:594-612
            row += [np.mean(w), np.std(w)]
            if bnn_obj._hyper_p:
                row.append(bnn_obj._prior_scale[i] if bnn_obj._hyper_p == 1 else np.mean(bnn_obj._prior_scale[i]))
        if bnn_obj._freq_indicator > 0:
            row.append(np.mean(bnn_obj._indicators))
        if add_prms:
            row += add_prms
        if bnn_obj._act_fun._trainable:
            row += list(np.atleast_1d(bnn_obj._act_fun._acc_prm))
        if self._estimation_mode == "regression":
            row += list(bnn_obj._error_prm)
        if bnn_obj._feature_indicators is not None:
            row += list(bnn_obj._feature_indicators)
        row += [mcmc_obj._acceptance_rate, mcmc_obj._mcmc_id]
        if not self.__dict__.get("_writer", True):
            return
        with open(self._logfile, "a", newline="") as f:
            csv.writer(f, delimiter="\t").writerow(row)

    def log_weights(self, bnn_obj, mcmc_obj, add_prms=None, add_obj=None):
        if not self.__dict__.get("_writer", True):
            return
        if self._log_all_weights:
            row = [mcmc_obj._current_iteration] + [v for w in bnn_obj._w_layers for v in w.flatten()]
            with open(self._w_file, "a", newline="") as f:
                csv.writer(f, delimiter="\t").writerow(row)
        else:
            w = bnn_obj._w_layers
            if bnn_obj._freq_indicator:                                            # BNN_env.py:635-641
                w = [w[0] * bnn_obj._indicators] + list(w[1:])
            post = {"weights": w, "alphas": list(np.atleast_1d(bnn_obj._act_fun._acc_prm)),
                    "mcmc_it": mcmc_obj._current_iteration}
            if len(bnn_obj._error_prm):
                post["error_prm"] = list(bnn_obj._error_prm)
            if add_prms:
                post["additional_prm"] = list(add_prms)
            self.update_post_weight_samples(post)
            self.control_weight_sample_length(mcmc_obj._n_post_samples)
        self._save([bnn_obj, mcmc_obj, self] + ([add_obj] if add_obj else []))

    # ---- non-blocking pickle (SURVEY.md 8f-4).  The reference rewrites the whole [bnn, mcmc, logger] pickle -- X
    # included -- at every logged sample (BNN_env.py:658); every write replaces the previous one, so only the newest
    # matters.  Between begin_async() and end_async() the writes go to a worker thread that always pickles the newest
    # snapshot and skips the ones it was too slow for; end_async() writes the last one and returns when it is on
    # disk.  Snapshots are shallow copies taken at call time: the drivers rebind attributes (fresh weight arrays per
    # logging point), they never mutate logged arrays in place.
    def _save(self, objs):
        st = self.__dict__.get("_async")
        if st is None:
            SaveObject(objs, self._pklfile)
            return
        from copy import copy
        snap = [copy(o) for o in objs]
        for o in snap:
            if isinstance(o, postLogger):
                o.__dict__["_post_weight_samples"] = list(self._post_weight_samples)
        with st["cv"]:
            st["job"] = snap
            st["cv"].notify()

    def begin_async(self):
        import threading
        if self.__dict__.get("_async") is not None:
            return
        st = {"cv": threading.Condition(), "job": None, "stop": False, "written": 0, "error": None}

        def work():
            while True:
                with st["cv"]:
                    while st["job"] is None and not st["stop"]:
                        st["cv"].wait()
                    job, st["job"] = st["job"], None
                    if job is None and st["stop"]:
                        return
                try:
                    SaveObject(job, self._pklfile)
                    st["written"] += 1
                except Exception as e:          # surfaced by end_async
                    st["error"] = e
        st["thread"] = threading.Thread(target=work, name="postLogger-pickle", daemon=True)
        self.__dict__["_async"] = st
        st["thread"].start()

    def end_async(self):
        st = self.__dict__.get("_async")
        if st is None:
            return 0
        with st["cv"]:
            st["stop"] = True
            st["cv"].notify()
        st["thread"].join()
        self.__dict__["_async"] = None
        if st["error"] is not None:
            raise st["error"]
        return st["written"]

    def __getstate__(self):
        d = dict(self.__dict__)
        d.pop("_async", None)
        return d
