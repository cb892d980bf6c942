"""CPU: the zero pattern the prediction callers hand to the engine (predshard.zero_pattern) and its way through
predict_ranks."""
import numpy as np

from npbnn_b200 import predshard
from npbnn_b200.engine import NetShape, flatten_weights


def block_net(rng, f=12, k=3):
    shapes = [(2 * f, f), (f, 2 * f), (k, f + 1)]
    mask = [np.zeros(s) for s in shapes]
    for g in range(f):
        mask[0][2 * g:2 * g + 2, g] = 1
        mask[1][g, 2 * g:2 * g + 2] = 1
    mask[2][:] = 1
    return shapes, mask


class FirstOnly:
    """A sample list that fails when anything but sample 0 is read."""

    def __init__(self, first, n):
        self.first, self.n = first, n

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if i == 0:
            return self.first
        raise AssertionError("looked past sample 0")


def test_pattern_is_the_exact_union_of_nonzeros():
    rng = np.random.default_rng(1)
    shapes, mask = block_net(rng)
    net = NetShape(12, shapes, act="tanh", lik=0)
    samples = []
    for s in range(5):
        # each sample keeps a random part of the mask, so only the union covers all of it
        samples.append([rng.normal(0, 1, sh) * m * (rng.random(sh) < 0.7) for sh, m in zip(shapes, mask)])
    want = np.zeros(net.n_params)
    for ws in samples:
        want[flatten_weights(ws) != 0] = 1.0
    got = predshard.zero_pattern(samples, net)
    assert got.dtype == np.float64 and np.array_equal(got, want)
    flat = np.stack([flatten_weights(ws) for ws in samples])
    assert np.array_equal(predshard.zero_pattern(flat, net), want)
    samples[2][1][0, 5] = np.nan                          # outside the mask, and NaN is not zero
    assert predshard.zero_pattern(samples, net)[shapes[0][0] * shapes[0][1] + 5] == 1.0


def test_dense_network_is_decided_from_sample_zero_alone():
    rng = np.random.default_rng(2)
    shapes = [(16, 6), (8, 16), (3, 9)]
    net = NetShape(6, shapes, act="tanh", lik=0)
    first = [rng.normal(0, 1, s) for s in shapes]
    assert predshard.zero_pattern(FirstOnly(first, 1000), net) is None
    # and a block network's pattern needs every sample
    shapes, mask = block_net(rng)
    first = [rng.normal(0, 1, s) * m for s, m in zip(shapes, mask)]
    try:
        predshard.zero_pattern(FirstOnly(first, 3), NetShape(12, shapes, act="tanh", lik=0))
        assert False, "the union must read every sample"
    except AssertionError as e:
        assert "past sample 0" in str(e)


def test_no_hidden_layer_has_no_pattern():
    net = NetShape(4, [(3, 5)], act="tanh", lik=0)
    assert predshard.zero_pattern([[np.zeros((3, 5))]], net) is None


class RecordingEngine:
    def __init__(self, net, K):
        self.net, self.K, self.O = net, K, K
        self.patterns = []

    def predict(self, x, w, alphas=None, override=None, mean=True, votes=False, dense=False, device_out=False,
                pattern=None):
        self.patterns.append(pattern)
        return {"mean": np.full((len(x), self.K), 1.0 / self.K)}


def test_predict_ranks_hands_the_pattern_of_all_samples_to_the_engine():
    rng = np.random.default_rng(3)
    shapes, mask = block_net(rng)
    net = NetShape(12, shapes, act="tanh", lik=0)
    samples = [[rng.normal(0, 1, s) * m for s, m in zip(shapes, mask)] for _ in range(4)]
    eng = RecordingEngine(net, 3)
    predshard.predict_ranks(eng, rng.standard_normal((10, 12)), samples, mean=True)
    assert np.array_equal(eng.patterns[-1], np.concatenate([m.ravel() for m in mask]))
    dense = [[rng.normal(0, 1, s) for s in shapes] for _ in range(2)]
    predshard.predict_ranks(eng, rng.standard_normal((10, 12)), dense, mean=True)
    assert eng.patterns[-1] is None


def test_a_given_pattern_is_used_as_it_is():
    """Callers that score the same samples many times (pdp, feature_importance) compute the pattern once and pass it."""
    rng = np.random.default_rng(4)
    shapes, mask = block_net(rng)
    net = NetShape(12, shapes, act="tanh", lik=0)
    samples = [[rng.normal(0, 1, s) * m for s, m in zip(shapes, mask)] for _ in range(3)]
    eng = RecordingEngine(net, 3)
    given = np.concatenate([m.ravel() for m in mask])
    given[-1] = 1.0
    predshard.predict_ranks(eng, rng.standard_normal((10, 12)), samples, mean=True, pattern=given)
    assert eng.patterns[-1] is given
    predshard.predict_ranks(eng, rng.standard_normal((10, 12)), samples, mean=True, pattern=None)
    assert eng.patterns[-1] is None


def test_tensor_samples():
    import torch
    rng = np.random.default_rng(5)
    shapes, mask = block_net(rng)
    net = NetShape(12, shapes, act="tanh", lik=0)
    flat = np.stack([flatten_weights([rng.normal(0, 1, s) * m for s, m in zip(shapes, mask)]) for _ in range(4)])
    assert np.array_equal(predshard.zero_pattern(torch.from_numpy(flat), net), np.concatenate([m.ravel() for m in mask]))
    dense = torch.from_numpy(rng.normal(0, 1, (4, net.n_params)))
    assert predshard.zero_pattern(dense, net) is None
