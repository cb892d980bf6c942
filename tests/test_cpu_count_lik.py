"""CPU: the count likelihoods of tests/count_oracle.py (estimation_mode="custom", BNN_lik.py:5-66) restate the host
functions of npbnn_b200.hostlib -- values, companion MSEs and the kind of non-finite value at overflow / underflow --, its
MH step keeps the chain's statistics equal to them, and the public surface refuses what is not on the device path before
any device call."""
import numpy as np
import pytest

from npbnn_b200 import hostlib as H
from tests import count_oracle as corc

# mode -> (likelihood, accuracy, output width per label column set)
CASES = {"poisson": (H.poi_likelihood, H.poi_acc), "negbin": (H.negbin_likelihood, H.negbin_acc),
         "negbin10": (H.negbin_likelihood_base10, H.negbin_acc_base10)}


def _table(rng, n, width, scale):
    z = rng.normal(0, scale, (n, width))
    k = rng.poisson(3.0, (n, max(1, width // 2))).astype(np.float64)
    k[::7] = 0.0                                              # k = 0 rows
    k[3::11] = rng.integers(200, 5000, k[3::11].shape)        # large counts
    return z, k


def _same(a, b):
    """Equal within 1e-12 relative, or the same non-finite value."""
    if not np.isfinite(a) or not np.isfinite(b):
        return (np.isnan(a) and np.isnan(b)) or a == b
    return abs(a - b) <= 1e-12 * max(1.0, abs(b))


@pytest.mark.parametrize("mode", ["poisson", "negbin", "negbin10"])
def test_oracle_matches_hostlib_on_random_tables(mode):
    rng = np.random.default_rng(3)
    lik, acc = CASES[mode]
    z, k = _table(rng, 500, 2, 1.0)
    with np.errstate(all="ignore"):
        ref = lik(z, k)
    assert _same(corc.loglik_count(z, k, mode), ref)
    _, sr2 = corc.count_sums(z, k, mode)
    assert abs(np.sum(sr2) / z.shape[0] - acc(z, k)) <= 1e-12 * acc(z, k)


def test_oracle_matches_hostlib_negbin2d():
    rng = np.random.default_rng(4)
    z = rng.normal(0, 1.0, (300, 6))
    k = rng.poisson(2.0, (300, 3)).astype(np.float64)
    k[::5, 1] = 0.0
    assert _same(corc.loglik_count(z, k, "negbin"), H.negbin_likelihood2d(z, k))
    _, sr2 = corc.count_sums(z, k, "negbin")
    assert abs(np.sum(sr2) / k.size - H.negbin2d_acc(z, k)) <= 1e-12 * H.negbin2d_acc(z, k)


@pytest.mark.parametrize("mode", ["poisson", "negbin", "negbin10"])
def test_extreme_outputs_give_the_host_formulas_non_finite_kind(mode):
    """Row by row, with outputs that overflow exp / 10** to inf and push n to 0 or p to 0 / 1."""
    lik, acc = CASES[mode]
    extremes = [-800.0, -400.0, -40.0, 0.0, 40.0, 400.0, 800.0]
    kinds = set()
    for z0 in extremes:
        for z1 in extremes:
            for kk in (0.0, 1.0, 37.0, 1e6):
                z, k = np.array([[z0, z1]]), np.array([[kk]])
                with np.errstate(all="ignore"):
                    ref, ref_acc = lik(z, k), acc(z, k)
                got = corc.loglik_count(z, k, mode)
                assert _same(got, ref), (z0, z1, kk, got, ref)
                assert _same(float(corc.count_sums(z, k, mode)[1][0]), ref_acc)
                kinds.add("nan" if np.isnan(ref) else ("-inf" if ref == -np.inf else "finite"))
    assert {"nan", "-inf", "finite"} <= kinds


def test_oracle_chain_statistics_follow_the_host_functions():
    """make_sampler / mh_step of the count oracle: after every step the chain's logLik and MSE are the host functions'
    values on its current weights, and the lik_temp argument changes nothing."""
    from oracle import npbnn_oracle as orc
    rng = np.random.default_rng(6)
    x = rng.standard_normal((200, 3))
    k = rng.poisson(2.0, (200, 1)).astype(np.float64)
    w0 = [rng.normal(0, 0.3, (4, 4)), rng.normal(0, 0.3, (2, 4))]
    m = corc.CountModel(x=x, labels=k, weights=[w.copy() for w in w0], act="tanh", mode="negbin")
    s = corc.make_sampler(m, update_f=[0.3, 0.3], lik_temp=0.25)
    rs = np.random.default_rng(1)
    n_acc = 0
    for _ in range(30):
        n_acc += corc.mh_step(m, s, rs=rs)["accepted"]
        y = orc.forward(x, m.weights, "tanh", None, "identity")
        assert _same(s.logLik, H.negbin_likelihood(y, k)) and _same(s.accuracy, H.negbin_acc(y, k))
        assert _same(s.logPost, s.logLik + s.logPrior)
    assert 0 < n_acc < 30


def _count_dat(rng, n=60, cols=1):
    x = rng.standard_normal((n, 3))
    y = rng.poisson(2.0, (n, cols)).astype(np.float64)
    return {"data": x, "labels": y, "test_data": [], "test_labels": []}


def test_api_refusals_before_any_device_call():
    import npbnn_b200 as bn
    rng = np.random.default_rng(0)
    dat = _count_dat(rng)
    # custom mode needs the identity output transform (the reference crashes on None too)
    with pytest.raises(NotImplementedError):
        bn.npBNN(dat, n_nodes=[4], estimation_mode="custom", size_output=2)
    with pytest.raises(NotImplementedError):
        bn.npBNN(dat, n_nodes=[4], estimation_mode="custom", size_output=2, output_act_fun=bn.SoftMax)
    bnn = bn.npBNN(dat, n_nodes=[4], estimation_mode="custom", size_output=2, output_act_fun=bn.RegressTransform)
    assert bnn._error_prm == [] and bnn._n_output_prm == 1 and bnn._labels.dtype == np.float64
    assert bnn._w_layers[-1].shape[0] == 2
    # a custom model needs one of the four count likelihoods; anything else raises
    for f in (None, lambda *a, **k: 0.0, bn.calc_likelihood_regression):
        with pytest.raises(NotImplementedError):
            bn.MCMC(bnn, likelihood_f=f)
    with pytest.raises(NotImplementedError, match="location"):
        bn.MCMC(bnn, likelihood_f=bn.gamma_likelihood)
    # the accuracy function is the likelihood's companion (or None)
    with pytest.raises(NotImplementedError):
        bn.MCMC(bnn, likelihood_f=bn.negbin_likelihood, accuracy_f=bn.negbin2d_acc)
    with pytest.raises(NotImplementedError):
        bn.MCMC(bnn, likelihood_f=bn.negbin_likelihood, accuracy_lab_f=bn.CalcLabelAccuracyRegression)
    with pytest.raises(NotImplementedError):
        bn.MCMC(bnn, likelihood_f=bn.negbin_likelihood, row_shard=True)
    with pytest.raises(NotImplementedError):
        bn.MC3(bnn, None, likelihood_f=lambda *a, **k: 0.0)
    # output widths the likelihood cannot read
    b3 = bn.npBNN(dat, n_nodes=[4], estimation_mode="custom", size_output=3, output_act_fun=bn.RegressTransform)
    with pytest.raises(NotImplementedError):
        bn.MCMC(b3, likelihood_f=bn.negbin_likelihood)
    with pytest.raises(ValueError):
        bn.MCMC(b3, likelihood_f=bn.negbin_likelihood2d)
    # count likelihoods on a built-in estimation mode stay refused
    reg = bn.npBNN(dat, n_nodes=[4], estimation_mode="regression")
    with pytest.raises(NotImplementedError):
        bn.MCMC(reg, likelihood_f=bn.poi_likelihood)


def test_custom_log_header_has_no_per_output_columns():
    import npbnn_b200 as bn
    bnn = bn.npBNN(_count_dat(np.random.default_rng(1), cols=2), n_nodes=[4, 3], estimation_mode="custom", size_output=4,
                   output_act_fun=bn.RegressTransform)
    head = bn.log_header(bnn)
    assert head[:6] == ["it", "posterior", "likelihood", "prior", "MSE", "test_MSE"]
    assert not any(h.startswith("sig_") or h.startswith("MSE_prm") for h in head)
