"""GPU: the life cycle of a context and engines on two devices in one process.

Contexts are created and destroyed repeatedly with every kind of resource in use (sparse program, graph, snapshot ring)
and must hand all their device memory back.  Kernel attributes (the dynamic shared-memory opt-in, non-portable cluster
sizes) belong to one device's context, so engines on two devices must both be able to launch every kernel family and
reach the same chain state."""
import gc

import numpy as np
import pytest
import torch

from npbnn_b200 import _lib as L
from npbnn_b200 import workloads as wl
from npbnn_b200.engine import Engine, NetShape
from tests.test_gpu_parity import _random_block_net

pytestmark = pytest.mark.gpu


def _masked_problem(n=3000, seed=7):
    """create_mask-style block network (uniform 3 -> 2 node pairs: k_fwd_sparse<pairs>) and two chains inside the mask."""
    rng = np.random.default_rng(seed)
    f, k = 12, 4
    shapes, mask, w = _random_block_net(rng, f, 3, 2, k)
    x = rng.standard_normal((n, f))
    labels = rng.integers(0, k, n)
    sets = [w, [a + rng.normal(0, 0.2, a.shape) * m for a, m in zip(w, mask)]]
    return NetShape(f, shapes, act="tanh", lik=L.LIK_CATEGORICAL), x, labels, sets, dict(mask=mask)


def _device_free(dev=0):
    gc.collect()
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info(dev)[0]


def _lifecycle(net, x, labels, sets, kw):
    eng = Engine(net, device=0)
    eng.set_data(x, labels)
    eng.chains_init(sets, seed=5, **kw)
    assert eng.last_kernel == "k_fwd_sparse<pairs>", eng.last_kernel
    eng.mh_steps(4)          # the first free-running call after chains_init runs eagerly ...
    eng.mh_steps(4)          # ... the next one is captured into a CUDA graph and replayed
    eng.snapshot(0)
    st = eng.snapshot_read(0)
    eng.close()
    return st


def test_context_lifecycle_returns_device_memory():
    """20 create / set_data / masked chains_init / eager and graph-replayed mh_steps / snapshot / close cycles: the free
    device memory returns to where it was after the first cycle (which loads the kernels), and every cycle computes the
    same chains."""
    net, x, labels, sets, kw = _masked_problem()
    first = _lifecycle(net, x, labels, sets, kw)
    free0 = _device_free()
    for _ in range(20):
        st = _lifecycle(net, x, labels, sets, kw)
        assert np.array_equal(st.f64, first.f64, equal_nan=True) and np.array_equal(st.i32, first.i32)
        assert np.array_equal(st.w, first.w)
    lost = free0 - _device_free()
    assert lost <= 2 << 20, "device memory not returned: %d bytes over 20 contexts" % lost


def _c4_case():
    """64 -> 64 -> 32 -> 10 swish classifier on >= 28,416 rows: the chains' forward pass is k_fwd3."""
    x, labels = wl.c4_data(30_000, seed=1)
    return NetShape(64, list(wl.C4_SHAPES), act="swish", lik=L.LIK_CATEGORICAL), x, labels, wl.c4_init_weights(3), {}


def _small_case():
    """[5, 5] tanh classifier on 400 rows: every step runs inside k_chain_loop (a thread-block cluster per chain)."""
    rs = np.random.default_rng(4)
    x = rs.standard_normal((400, 24))
    labels = rs.integers(0, 3, 400)
    sets = [[rs.normal(0, 0.3, s) for s in ((5, 25), (5, 6), (3, 5))] for _ in range(2)]
    return NetShape(24, [(5, 25), (5, 6), (3, 5)], act="tanh", lik=L.LIK_CATEGORICAL), x, labels, sets, {}


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("case,kernel", [("fwd3", "k_fwd3"), ("pairs", "k_fwd_sparse<pairs>"),
                                         ("chain_loop", "k_chain_loop")])
def test_engines_on_two_devices_match(case, kernel):
    """The same net, data and seeds on device 0 and device 1 of one process: each device runs the kernel family under
    test and the chain state is bit-identical."""
    net, x, labels, sets, kw = {"fwd3": _c4_case, "pairs": _masked_problem, "chain_loop": _small_case}[case]()
    states = []
    for dev in (0, 1):
        eng = Engine(net, device=dev)
        eng.set_data(x, labels)
        eng.chains_init(sets, seed=9, **kw)
        eng.mh_steps(6)
        assert eng.last_kernel.startswith(kernel), (dev, eng.last_kernel)
        states.append(eng.read_state())
        eng.close()
    a, b = states
    assert np.array_equal(a.f64, b.f64, equal_nan=True) and np.array_equal(a.i32, b.i32) and np.array_equal(a.w, b.w)
