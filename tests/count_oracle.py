"""numpy restatement of the count likelihoods of estimation_mode="custom" (BNN_lik.py:5-66; written down in
npbnn_b200/hostlib.py:712-760) and of MCMC.mh_step with them, built on the building blocks of oracle/npbnn_oracle.py
(forward pass, prior, proposal draws, adaptation).  Test infrastructure only.

z = identity outputs (RegressTransform), k = the label table; none of the functions applies lik_temp.
  poisson  : K = 1,     rate = exp(z0)
  negbin   : K = O / 2, mean_j = exp(z_j), p_j = 1 / (1 + exp(-z_{K+j}))  (negbin_likelihood is K = 1, 2d is K = O_lab)
  negbin10 : negbin with 10** in place of exp (negbin_likelihood_base10)
"""
from dataclasses import dataclass

import numpy as np

from oracle import npbnn_oracle as orc

COUNT_MODES = ("poisson", "negbin", "negbin10")


def count_k(y: np.ndarray, mode: str) -> int:
    return 1 if mode == "poisson" else y.shape[1] // 2


def count_mean(y: np.ndarray, mode: str) -> np.ndarray:
    """[N, K] predicted means: exp(z_j), or 10**z_j for negbin10."""
    z = y[:, :count_k(y, mode)]
    with np.errstate(all="ignore"):
        return 10 ** z if mode == "negbin10" else np.exp(z)


def nbinom_logpmf(k, n, p):
    """scipy.stats.nbinom.logpmf as _nbinom_logpmf writes it."""
    from scipy.special import gammaln, xlog1py, xlogy
    return gammaln(k + n) - gammaln(k + 1) - gammaln(n) + xlogy(n, p) + xlog1py(k, -p)


def loglik_count(y: np.ndarray, labels: np.ndarray, mode: str) -> float:
    """Sum over the training rows and the K modelled columns (labels: the first K columns are the counts)."""
    from scipy.special import gammaln, xlogy
    K = count_k(y, mode)
    k = labels[:, :K]
    mean = count_mean(y, mode)
    with np.errstate(all="ignore"):
        if mode == "poisson":
            return float(np.sum(xlogy(k, mean) - gammaln(k + 1) - mean))
        d = y[:, K:2 * K]
        p = 1 / (1 + (10 ** (-d) if mode == "negbin10" else np.exp(-d)))
        return float(np.sum(nbinom_logpmf(k, p * mean / (1 - p), p)))


def count_sums(y: np.ndarray, labels: np.ndarray, mode: str):
    """sum r_j and sum r_j^2 with r = mean - k; the companion MSE (poi_acc, negbin_acc, negbin2d_acc,
    negbin_acc_base10) is sum r^2 / (N K)."""
    r = count_mean(y, mode) - labels[:, :count_k(y, mode)]
    with np.errstate(all="ignore"):
        return np.sum(r, axis=0), np.sum(r * r, axis=0)


@dataclass
class CountModel(orc.Model):
    """orc.Model with mode = poisson | negbin | negbin10: identity outputs, no error parameter."""

    @property
    def out_kind(self):
        return "identity"


def _mse(y, labels, mode):
    _, sr2 = count_sums(y, labels, mode)
    return float(np.sum(sr2) / sr2.size / y.shape[0])


def refresh_accuracy(m: CountModel, s: orc.Sampler, y: np.ndarray, weights) -> None:
    """The companion MSE on the training / test rows; custom mode logs no per-output accuracies."""
    s.accuracy = _mse(y, m.labels, m.mode)
    s.label_acc = np.array([])
    s.label_freq = None
    if m.x_test is not None and len(m.x_test) > 0:
        s.test_accuracy = _mse(orc.forward(m.x_test, weights, m.act, m.alphas, "identity"), m.labels_test, m.mode)
    else:
        s.test_accuracy = 0


def make_sampler(m: CountModel, update_f=None, update_ws=None, temperature=1.0, n_iteration=100000, lik_temp=1.0,
                 adapt_f=0.0, adapt_fM=1.0, adapt_freq=1000, adapt_stop=None) -> orc.Sampler:
    """MCMC.__init__ (BNN_env.py:274-379) of a count model, as orc.make_sampler does it for the built-in modes."""
    nl = len(m.weights)
    update_ws = [0.075] * nl if update_ws is None else update_ws
    update_f = np.array(([0.05] * nl if update_f is None else update_f)[:nl], dtype=np.float64)
    sizes = np.array([w.size for w in m.weights])
    update_n = np.array([max(1, int(np.round(sizes[i] * update_f[i]))) for i in range(nl)])
    s = orc.Sampler(update_f=update_f, update_ws=np.array(update_ws[:nl], dtype=np.float64), update_n=update_n,
                    max_n=sizes.astype(int), temperature=temperature, lik_temp=lik_temp, adapt_f=adapt_f,
                    adapt_fM=adapt_fM, adapt_freq=adapt_freq,
                    adapt_stop=int(n_iteration * 0.05) if adapt_stop is None else adapt_stop,
                    freq_layer_update=np.ones(nl), estimate_error=float(n_iteration))
    y = orc.forward(m.x, m.weights, m.act, m.alphas, "identity")
    s.logLik = loglik_count(y, m.labels, m.mode)
    s.logPrior = orc.log_prior(m.weights, m.prior, m.prior_scale)
    s.logPost = s.logLik + s.logPrior
    refresh_accuracy(m, s, y, m.weights)
    return s


def mh_step(m: CountModel, s: orc.Sampler, inj=None, rs=None) -> dict:
    """One MH iteration (BNN_env.py:381-532) of a count model: adaptation, the injected (or drawn) UpdateNormal
    proposal, prior + count likelihood, accept rule, acceptance window.  Mutates m.weights (on accept) and s."""
    orc.adapt(m, s)
    if inj is None:
        inj = orc.draw_injection(m, s, rs)
    w_prime = []
    for i, w in enumerate(m.weights):
        upd = inj.layers[i]
        z = w + 0 if upd is None else orc.apply_update_normal(w, upd[0], upd[1], upd[2], m.w_bound, -m.w_bound)
        if m.mask is not None:
            z = z * m.mask[i]
        w_prime.append(z)
    y = orc.forward(m.x, w_prime, m.act, m.alphas, "identity")
    lp = orc.log_prior(w_prime, m.prior, m.prior_scale) + inj.add_prob
    ll = loglik_count(y, m.labels, m.mode)
    post = ll + lp
    accept = bool((post - s.logPost) * s.temperature >= inj.log_u)
    if accept:
        m.weights = w_prime
        s.logPost, s.logLik, s.logPrior = post, ll, lp
        refresh_accuracy(m, s, y, w_prime)
    s.last_accepted = int(accept)
    s.acc_mem.append(s.last_accepted)
    s.acceptance_rate = float(np.mean(s.acc_mem))
    if len(s.acc_mem) > 100:
        s.acc_mem = s.acc_mem[-100:]
    s.it += 1
    return {"logLik_prime": ll, "logPrior_prime": lp, "accepted": int(accept)}
