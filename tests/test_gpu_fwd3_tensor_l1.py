"""GPU: the 64 -> 64 -> 32 family's likelihood kernel with layer 1 on the int8 tensor cores (k_fwd3i, base-256 digits
of X and W1, six diagonal accumulators in tensor memory, exact integer recombination).  Against the FP64 generic
kernel: data sets made of one kind of row each (zero rows, features in different units, huge and tiny values,
subnormal entries, a timestamp feature) at row counts that are not multiples of 16 or 128, a large feature with a
compensating weight, the data sets that run the FP64 first layer instead, and repeated launches at the config-4 shape
for 4 to 32 chains, each with its own sets."""
import zlib

import numpy as np
import pytest

from oracle import npbnn_oracle as orc

pytestmark = pytest.mark.gpu

SHAPES = [(64, 64), (32, 64), (10, 33)]          # config 4: 64 -> 64 -> 32 -> 10, bias on the last layer


def _engine(x, labels, sets, act="swish", lik=0, targets=None):
    from npbnn_b200.engine import Engine, NetShape
    net = NetShape.from_weights(sets[0], 64, act=act, lik=lik)
    eng = Engine(net)
    if lik == 0:
        eng.set_data(x, labels)
    else:
        eng.set_data(x, targets)
    return eng


def _both(eng, sets, **kw):
    res = eng.forward_lik(sets, **kw)
    kernel = eng.last_kernel
    eng.set_option("force_generic", 1)
    ref = eng.forward_lik(sets, **kw)
    assert eng.last_kernel == "k_fwd_generic"
    eng.set_option("force_generic", 0)
    return res, ref, kernel


I8 = {"swish": "k_fwd3<swish,64,64,32,16,i8l1>", "ReLU": "k_fwd3<relu,64,64,32,i8l1>"}
F64 = {"swish": "k_fwd3<swish,64,64,32,16>", "ReLU": "k_fwd3<relu,64,64,32>"}


def _kind(kind, n, rng):
    """n rows of one kind, so that the log-likelihood of a data set is made of that kind of row only."""
    x = rng.standard_normal((n, 64))
    if kind == "zero rows":
        x[:] = 0.0
    elif kind == "zero rows among ordinary ones":
        x[::3] = 0.0
        x[:, 5] = 0.0
    elif kind == "features in different units":           # ragged magnitudes across every row, 1e-120 .. 1e120
        x *= np.logspace(-120, 120, 64)
    elif kind == "huge values":
        x *= 1e100
    elif kind == "tiny values":
        x *= 1e-120
    elif kind == "subnormal and normal entries in each row":
        x[(np.arange(n)[:, None] + np.arange(64)[None, :]) % 4 == 0] *= 1e-310
    elif kind == "timestamp feature":                      # one feature ~1.7e9 with a small spread
        x[:, 0] = 1.7e9 + rng.uniform(0, 1e6, n)
    return x


def _sets(rng, shapes, n_sets, x):
    """Weight sets whose first-layer column k is scaled by 1 / (typical |x_k|): every feature contributes alike (the
    weights MH drives to for features in large units), so that the products, not one feature, set the result."""
    col = np.sqrt(np.mean(x * x, axis=0))
    col[col == 0] = 1.0
    sets = [[rng.normal(0, 0.3, s) for s in shapes] for _ in range(n_sets)]
    for w in sets:
        w[0][:, w[0].shape[1] - 64:] /= col
    return sets


KINDS = ["zero rows", "zero rows among ordinary ones", "features in different units", "huge values", "tiny values",
         "subnormal and normal entries in each row", "timestamp feature"]


@pytest.mark.parametrize("n", [16 * 7 + 3, 128 * 5 + 77, 2 * 18944 + 131])
@pytest.mark.parametrize("kind", KINDS)
def test_rows_of_one_kind_categorical_against_fp64(kind, n):
    """The config-4 network on a data set made of one kind of row (row counts not multiples of 16 or 128): the
    int8 first layer runs, log-likelihoods within 1e-12 of the FP64 generic kernel, identical counters."""
    rng = np.random.default_rng(zlib.crc32(kind.encode()) + n)
    x = _kind(kind, n, rng)
    labels = rng.integers(0, 10, n)
    sets = _sets(rng, SHAPES, 4, x)
    eng = _engine(x, labels, sets)
    res, ref, kernel = _both(eng, sets)
    assert kernel == I8["swish"], kernel
    for i in range(len(sets)):
        assert np.isclose(res["loglik"][i], ref["loglik"][i], rtol=1e-12, atol=0), (i, res["loglik"][i], ref["loglik"][i])
        assert np.array_equal(res["counts"][i], ref["counts"][i])
    eng.close()


@pytest.mark.parametrize("kind", ["features in different units", "timestamp feature", "zero rows among ordinary ones"])
def test_rows_of_one_kind_regression_against_fp64(kind):
    """Gaussian likelihood of a ReLU network (pre-activations reach the outputs almost linearly): every per-output sum
    of residuals and squared residuals within 1e-12 of the FP64 generic kernel, each against its own magnitude."""
    from npbnn_b200 import _lib as L
    rng = np.random.default_rng(len(kind))
    n = 1000 + 5
    x = _kind(kind, n, rng)
    shapes = [(64, 65), (32, 65), (8, 33)]
    sets = _sets(rng, shapes, 3, x)
    sets[1][0][4, :] = 0.0                                 # an all-zero unit
    targets = rng.standard_normal((n, 8))
    eng = _engine(x, None, sets, act="ReLU", lik=L.LIK_GAUSSIAN, targets=targets)
    res, ref, kernel = _both(eng, sets, sigma_mode=L.SIGMA_EMPIRICAL)
    assert kernel == I8["ReLU"], kernel
    for i in range(len(sets)):
        a, b = np.asarray(res["sums"][i]), np.asarray(ref["sums"][i])
        sq = b[1:]                                          # sums of squares: positive, compared relatively
        assert np.allclose(a[1:], sq, rtol=1e-12, atol=0), (i, a, b)
        # sum r cancels: against the sum of |r| it is made of (sqrt(n * sum r^2) bounds it)
        assert np.all(np.abs(a[0] - b[0]) <= 1e-12 * np.sqrt(n * b[1])), (i, a[0], b[0])
        assert np.isclose(res["loglik"][i], ref["loglik"][i], rtol=1e-12, atol=0)
    eng.close()


def test_large_feature_with_compensating_weight_against_fp64():
    """A feature of ~1.7e9 (a timestamp) whose first-layer weights are ~1e-9, beside standardised features: the
    per-feature power-of-two scaling keeps its products as precise as the others'.  Within 1e-12 of FP64."""
    rng = np.random.default_rng(3)
    n = 4099
    x = rng.standard_normal((n, 64))
    x[:, 0] = 1.7e9 + rng.uniform(0, 3e7, n)
    labels = rng.integers(0, 10, n)
    sets = [[rng.normal(0, 0.3, s) for s in SHAPES] for _ in range(4)]
    for w in sets:
        w[0][:, 0] = rng.normal(0, 1e-9, 64)
    eng = _engine(x, labels, sets)
    res, ref, kernel = _both(eng, sets)
    assert kernel == I8["swish"], kernel
    assert np.allclose(res["loglik"], ref["loglik"], rtol=1e-12, atol=0), (res["loglik"], ref["loglik"])
    assert np.array_equal(res["counts"], ref["counts"])
    eng.close()


@pytest.mark.parametrize("kind", ["rare outliers in a feature", "one row with a huge entry", "infinite entry", "nan entry",
                                  "all-subnormal feature"])
def test_data_outside_the_int8_range_runs_the_fp64_first_layer(kind):
    """Data sets the int8 first layer would not represent to its bound (a feature with more than half of its nonzero
    entries below 2^-6 of its largest magnitude, a non-finite entry, a feature below 2^-500) run k_fwd3 with the FP64 first layer: the
    same results as the generic kernel (non-finite ones included)."""
    rng = np.random.default_rng(9)
    n = 2000
    x = rng.standard_normal((n, 64))
    if kind == "rare outliers in a feature":
        x[::500, 3] *= 1e6
    elif kind == "one row with a huge entry":
        x[7, 0] = 2.0 ** 100
    elif kind == "infinite entry":
        x[11, 2] = np.inf
    elif kind == "nan entry":
        x[13, 4] = np.nan
    else:
        x[:, 9] *= 1e-310
    labels = rng.integers(0, 10, n)
    sets = [[rng.normal(0, 0.3, s) for s in SHAPES] for _ in range(3)]
    eng = _engine(x, labels, sets)
    res, ref, kernel = _both(eng, sets)
    assert kernel == F64["swish"], kernel
    assert np.array_equal(np.isnan(res["loglik"]), np.isnan(ref["loglik"]))
    fin = np.isfinite(ref["loglik"])
    assert np.array_equal(res["loglik"][~fin & ~np.isnan(ref["loglik"])], ref["loglik"][~fin & ~np.isnan(ref["loglik"])])
    assert np.allclose(res["loglik"][fin], ref["loglik"][fin], rtol=1e-12, atol=0)
    eng.close()


def test_c4_shape_launches_the_int8_kernel_many_times_against_fp64():
    """64 launches at the config-4 network shape, 16 each with 4, 8, 31 and 32 chains, every launch with weight sets of
    its own: log-likelihoods within 1e-12 of the FP64 generic kernel and identical counters.  Each launch reuses the
    tensor-memory accumulators, the two W1 digit slots and the two X digit tiles many times per CTA, so a buffer
    overwritten before the tensor core has read it shows up as a mismatch."""
    rng = np.random.default_rng(21)
    n = 300_007
    x = rng.standard_normal((n, 64))
    teacher = [rng.normal(0, 0.5, s) for s in SHAPES]
    labels = np.argmax(orc.forward(x, teacher, "swish", None, "softmax"), axis=1)
    eng = _engine(x, labels, [teacher])
    for n_sets in (4, 8, 31, 32):
        for _ in range(16):
            sets = [[rng.normal(0, 0.3, s) for s in SHAPES] for _ in range(n_sets)]
            res, ref, kernel = _both(eng, sets)
            assert kernel == "k_fwd3<swish,64,64,32,16,i8l1>", kernel
            ll, rl = np.asarray(res["loglik"]), np.asarray(ref["loglik"])
            assert np.allclose(ll, rl, rtol=1e-12, atol=0), (n_sets, np.max(np.abs(ll - rl) / np.abs(rl)))
            assert np.array_equal(np.asarray(res["counts"]), np.asarray(ref["counts"])), n_sets
    eng.close()
