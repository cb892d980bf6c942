"""Device engine: a thin object over the C ABI (include/npbnn_b200.h).

PyTorch is used for device buffers and streams only; every computation on the path is a
hand-written sm_100a kernel behind the C ABI.  There is no CPU fallback: constructing an
Engine without a CUDA device (or without the shared library) raises.
"""
import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L
from . import rowshard


@dataclass
class NetShape:
    """Shapes of the weight matrices [(out, in + bias), ...] as init_weight_prm builds them
    (reference BNN_mcmc.py:9-25); bias presence is inferred like MatrixMultiplicationD does
    (BNN_lib.py:154-162): a matrix with one more column than its input width has a bias column 0."""
    n_features: int
    shapes: List[tuple]
    act: str = "ReLU"
    lik: int = L.LIK_CATEGORICAL

    @property
    def n_layers(self):
        return len(self.shapes)

    @property
    def sizes(self):
        return [int(r * c) for r, c in self.shapes]

    @property
    def n_params(self):
        return int(sum(self.sizes))

    def has_bias(self):
        out, width = [], self.n_features
        for r, c in self.shapes:
            if c == width:
                out.append(0)
            elif c == width + 1:
                out.append(1)
            else:
                raise ValueError("weight matrix %s does not match its input width %d" % ((r, c), width))
            width = r
        return out

    @staticmethod
    def from_weights(weights: Sequence[np.ndarray], n_features: int, act="ReLU", lik=L.LIK_CATEGORICAL):
        return NetShape(n_features, [tuple(w.shape) for w in weights], act, lik)


def flatten_weights(weights: Sequence[np.ndarray]) -> np.ndarray:
    """Canonical weight-set layout: row-major layers concatenated."""
    return np.concatenate([np.ascontiguousarray(w, dtype=np.float64).ravel() for w in weights])


def unflatten_weights(flat: np.ndarray, shapes: Sequence[tuple]) -> List[np.ndarray]:
    out, o = [], 0
    for r, c in shapes:
        out.append(np.array(flat[o:o + r * c], dtype=np.float64).reshape(r, c))
        o += r * c
    return out


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class ChainState:
    """Host copy of the per-chain device state (slot layout: enum in include/npbnn_b200.h)."""

    def __init__(self, f64, i32, w, net: NetShape, K: int):
        self.f64, self.i32, self.w, self.net, self.K = f64, i32, w, net, K
        nl = net.n_layers
        self.logLik = f64[:, L.F_LOGLIK]
        self.logPrior = f64[:, L.F_LOGPRIOR]
        self.logPost = f64[:, L.F_LOGPOST]
        self.temperature = f64[:, L.F_TEMPERATURE]
        self.acceptance_rate = f64[:, L.F_ACC_RATE]
        self.logLik_prop = f64[:, L.F_LOGLIK_PROP]
        self.logPrior_prop = f64[:, L.F_LOGPRIOR_PROP]
        self.alpha = f64[:, L.F_ALPHA:L.F_ALPHA + nl]              # accepted activation parameters per layer
        self.alpha_prop = f64[:, L.F_ALPHA_PROP:L.F_ALPHA_PROP + nl]
        self.update_f = f64[:, L.F_UPDATE_F:L.F_UPDATE_F + nl]
        self.update_ws = f64[:, L.F_UPDATE_WS:L.F_UPDATE_WS + nl]
        self.freq_layer_update = f64[:, L.F_FREQ_LAYER:L.F_FREQ_LAYER + nl]
        self.sigma = f64[:, L.F_SIGMA:L.F_SIGMA + K]
        self.sum_r = f64[:, L.F_SUM_R:L.F_SUM_R + K]
        self.sum_r2 = f64[:, L.F_SUM_R2:L.F_SUM_R2 + K]
        self.sum_r2_test = f64[:, L.F_SUM_R2_TEST:L.F_SUM_R2_TEST + K]
        self.iteration = i32[:, L.I_ITERATION]
        self.last_accepted = i32[:, L.I_LAST_ACCEPTED]
        self.n_accepted = i32[:, L.I_N_ACCEPTED]
        self.update_n = i32[:, L.I_UPDATE_N:L.I_UPDATE_N + nl]
        self.proposed = i32[:, L.I_PROPOSED:L.I_PROPOSED + nl]
        self.n_correct = i32[:, L.I_N_CORRECT]
        self.n_correct_test = i32[:, L.I_N_CORRECT_TEST]
        self.class_correct = i32[:, L.I_CLASS_CORRECT:L.I_CLASS_CORRECT + K]
        self.pred_hist = i32[:, L.I_PRED_HIST:L.I_PRED_HIST + K]

    def weights(self, chain: int) -> List[np.ndarray]:
        return unflatten_weights(self.w[chain], self.net.shapes)


class Engine:
    def __init__(self, net: NetShape, device: int = 0):
        if not torch.cuda.is_available():
            raise L.NpbnnError("npbnn_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = L.load()
        self.net = net
        self.device = torch.device("cuda", device)
        h = C.c_void_p()
        L.check(self.lib.bnn_ctx_create(C.byref(h), device))
        self._h = h
        spec = L.NetSpec()
        spec.n_layers, spec.n_features = net.n_layers, net.n_features
        hb = net.has_bias()
        for i, (r, c) in enumerate(net.shapes[:L.MAX_LAYERS]):      # (deeper networks: bnn_set_net refuses n_layers)
            spec.out_dim[i], spec.has_bias[i] = int(r), int(hb[i])
        spec.act, spec.lik = L.ACT[net.act], net.lik
        L.check(self.lib.bnn_set_net(h, C.byref(spec)))
        assert self.lib.bnn_n_params(h) == net.n_params
        out = net.shapes[-1][0]
        # modelled output columns: sigma head / negative binomial = (value | parameter) halves, Poisson = column 0
        self.K = out // 2 if net.lik in (L.LIK_GAUSSIAN_HEAD, L.LIK_NEGBIN, L.LIK_NEGBIN10) else \
            (1 if net.lik == L.LIK_POISSON else out)
        self.O = out
        self.n_train = self.n_test = 0
        self.n_chains = 0
        self._keep = []
        self._rowshard = None          # callable(tensor) summing a device tensor over the ranks, or None

    def close(self):
        if getattr(self, "_h", None):
            self.lib.bnn_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, a, dtype):
        if a is None:
            return None
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(self.device)

    def set_option(self, name: str, value: int):
        L.check(self.lib.bnn_set_option(self._h, name.encode(), int(value)))

    @property
    def last_kernel(self) -> str:
        return self.lib.bnn_last_kernel(self._h).decode()

    @property
    def launch_count(self) -> int:
        return int(self.lib.bnn_launch_count(self._h))

    # ---------------------------------------------------------------- data
    def set_data(self, x, y, x_test=None, y_test=None, inst_w=None, class_w=None):
        """Stage training (+ optional test) rows once (npBNN._data/_labels..., reference BNN_env.py:35-49).  The count
        likelihoods model the first K label columns (the ones BNN_lik.py reads)."""
        with torch.cuda.device(self.device):
            xs = [self._dev(x, torch.float64)]
            n_train, n_test = xs[0].shape[0], 0
            cat = self.net.lik == L.LIK_CATEGORICAL
            ydt = torch.int32 if cat else torch.float64
            ys = [self._dev(y, ydt)]
            if x_test is not None and len(x_test) > 0:
                xs.append(self._dev(x_test, torch.float64))
                ys.append(self._dev(y_test, ydt))
                n_test = xs[1].shape[0]
            xd = torch.cat(xs, 0).contiguous() if n_test else xs[0]
            yd = torch.cat(ys, 0).contiguous() if n_test else ys[0]
            assert xd.shape[1] == self.net.n_features
            if not cat:
                yd = yd.reshape(n_train + n_test, -1)
                if self.net.lik in L.LIK_COUNT:
                    assert yd.shape[1] >= self.K
                    yd = yd[:, :self.K].contiguous()
                assert yd.shape[1] == self.K
            iw, cw = self._dev(inst_w, torch.float64), self._dev(class_w, torch.float64)
            L.check(self.lib.bnn_set_data(self._h, _ptr(xd), n_train, n_test, _ptr(yd) if cat else None,
                                          None if cat else _ptr(yd), _ptr(iw), _ptr(cw), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
        self.n_train, self.n_test = n_train, n_test

    # ---------------------------------------------------------------- stateless scoring
    def forward_lik(self, weight_sets, alphas=None, sigma=None, sigma_mode=L.SIGMA_FIXED, lik_temp=1.0, host=False):
        """Score weight sets against the staged data.  weight_sets: [C, P] array/tensor or a list of
        per-layer weight lists.  Returns dict(loglik, counts | sums) as numpy arrays."""
        w = self._as_sets(weight_sets)
        n = w.shape[0]
        NC = 2 + 2 * self.K
        cat = self.net.lik == L.LIK_CATEGORICAL
        if host:
            wh = np.ascontiguousarray(w if isinstance(w, np.ndarray) else w.cpu().numpy(), dtype=np.float64)
            ah = None if alphas is None else np.ascontiguousarray(alphas, dtype=np.float64)
            sh = None if sigma is None else np.ascontiguousarray(sigma, dtype=np.float64)
            ll = np.empty(n)
            sums = np.zeros((n, 3, self.K))
            counts = np.zeros((n, NC), dtype=np.int32)
            L.check(self.lib.bnn_forward_lik_host(self._h, _np_ptr(wh), n, _np_ptr(ah), _np_ptr(sh), sigma_mode,
                                                  float(lik_temp), _np_ptr(ll), _np_ptr(sums), _np_ptr(counts),
                                                  self._stream()))
            return {"loglik": ll, "sums": sums, "counts": counts}
        with torch.cuda.device(self.device):
            wd = self._dev(w, torch.float64)
            ad, sd = self._dev(alphas, torch.float64), self._dev(sigma, torch.float64)
            ll = torch.empty(n, dtype=torch.float64, device=self.device)
            sums = torch.zeros((n, 3, self.K), dtype=torch.float64, device=self.device)
            counts = torch.zeros((n, NC), dtype=torch.int32, device=self.device)
            L.check(self.lib.bnn_forward_lik(self._h, _ptr(wd), n, _ptr(ad), _ptr(sd), sigma_mode, float(lik_temp),
                                             _ptr(ll), None if cat else _ptr(sums), _ptr(counts) if cat else None,
                                             self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
            return {"loglik": ll.cpu().numpy(), "sums": sums.cpu().numpy(), "counts": counts.cpu().numpy()}

    def log_prior(self, weight_sets, prior: int, prior_scale):
        w = self._as_sets(weight_sets)
        with torch.cuda.device(self.device):
            wd = self._dev(w, torch.float64)
            out = torch.empty(wd.shape[0], dtype=torch.float64, device=self.device)
            if isinstance(prior_scale, np.ndarray) and prior_scale.shape == (self.net.n_params,) \
                    and self.net.n_params != self.net.n_layers:
                # one scale per weight entry (hyper-priors)
                ps = np.ascontiguousarray(prior_scale, dtype=np.float64)
                L.check(self.lib.bnn_log_prior_entries(self._h, _ptr(wd), wd.shape[0], int(prior), _np_ptr(ps), _ptr(out),
                                                       self._stream()))
            else:
                ps = np.ascontiguousarray(np.broadcast_to(np.asarray(prior_scale, dtype=np.float64), (self.net.n_layers,)))
                L.check(self.lib.bnn_log_prior(self._h, _ptr(wd), wd.shape[0], int(prior), _np_ptr(ps), _ptr(out),
                                               self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
            return out.cpu().numpy()

    def _as_sets(self, weight_sets):
        if isinstance(weight_sets, (np.ndarray, torch.Tensor)):
            w = weight_sets
        else:
            w = np.stack([flatten_weights(ws) for ws in weight_sets])
        assert w.ndim == 2 and w.shape[1] == self.net.n_params, (tuple(w.shape), self.net.n_params)
        return w

    # ---------------------------------------------------------------- chains
    def chains_init(self, w0, temperature=None, update_f=None, update_ws=None, prior=L.PRIOR_NORMAL, prior_scale=1.0,
                    w_bound=np.inf, mask=None, alphas=None, sigma0=None, sigma_mode=L.SIGMA_FIXED, lik_temp=1.0,
                    adapt_f=0.0, adapt_fM=1.0, adapt_freq=1000, adapt_stop=0, sample_from_prior=0, seed=1234,
                    n_act_prm=0, init_additional_prob=0.0, prior_ind1=None, feature_means=None, chain_offset=0,
                    freq_indicator=0.0):
        w = np.ascontiguousarray(self._as_sets(w0), dtype=np.float64)
        n, nl = w.shape[0], self.net.n_layers

        def per_chain(v, default, width):
            if v is None:
                v = default
            return np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (n, width)))

        temp = np.ascontiguousarray(np.broadcast_to(np.asarray(1.0 if temperature is None else temperature,
                                                               dtype=np.float64), (n,)))
        uf = per_chain(update_f, 0.05, nl)
        uws = per_chain(update_ws, 0.075, nl)
        al = None if alphas is None else per_chain(alphas, 0.0, nl)
        sg = None if sigma0 is None else per_chain(sigma0, 1.0, self.K)
        cfg = L.SamplerConfig()
        cfg.prior, cfg.sigma_mode, cfg.sample_from_prior = int(prior), int(sigma_mode), int(sample_from_prior)
        cfg.adapt_freq, cfg.adapt_stop = int(adapt_freq), int(adapt_stop)
        cfg.adapt_f, cfg.adapt_fM, cfg.lik_temp, cfg.w_bound = float(adapt_f), float(adapt_fM), float(lik_temp), float(w_bound)
        ps = np.broadcast_to(np.asarray(prior_scale, dtype=np.float64), (nl,))
        for i in range(nl):
            cfg.prior_scale[i] = float(ps[i])
        cfg.seed = int(seed)
        cfg.chain_offset = int(chain_offset)        # device generators are keyed on the GLOBAL chain index
        cfg.n_act_prm, cfg.init_additional_prob = int(n_act_prm), float(init_additional_prob)
        mk = None
        if mask is not None:
            mk = np.ascontiguousarray(flatten_weights(mask) if not isinstance(mask, np.ndarray) else mask, dtype=np.float64)
            assert mk.shape == (self.net.n_params,)
        cfg.use_mask = int(mk is not None)
        # weight indicators (npBNN(freq_indicator > 0)) / feature indicators (npBNN(feature_indicators=True))
        cfg.use_indicators = int(prior_ind1 is not None)
        cfg.prior_ind1 = float(prior_ind1) if prior_ind1 is not None else 0.5
        cfg.use_feature_indicators = int(feature_means is not None)
        cfg.freq_indicator = float(freq_indicator) if prior_ind1 is not None else 0.0
        if feature_means is not None:
            fm = np.ascontiguousarray(feature_means, dtype=np.float64)
            assert fm.shape == (self.net.n_features,)
            L.check(self.lib.bnn_set_feature_means(self._h, _np_ptr(fm), self._stream()))
        self._p0 = int(np.prod(self.net.shapes[0]))
        L.check(self.lib.bnn_chains_init(self._h, n, C.byref(cfg), _np_ptr(w), _np_ptr(mk), _np_ptr(temp), _np_ptr(uf),
                                         _np_ptr(uws), _np_ptr(al), _np_ptr(sg), self._stream()))
        self.n_chains = n
        if callable(self._rowshard):
            rowshard.exchange([self], self._all_reduce_own, 2)

    def _pack_injection(self, injection, n_steps):
        arrs = {k: np.ascontiguousarray(injection[k], dtype=(np.float64 if k in ("dz", "log_u") else np.int32))
                for k in ("proposed", "count", "ix", "iy", "dz", "log_u")}
        for k, dt in (("alpha_ix", np.int32), ("alpha_dz", np.float64), ("add_prob", np.float64),
                      ("ind_move", np.int32), ("ind_flip", np.uint8), ("fi_move", np.int32), ("fi_flip", np.uint8)):   # optional branches
            if injection.get(k) is not None:
                arrs[k] = np.ascontiguousarray(injection[k], dtype=dt)
                assert arrs[k].shape[:2] == arrs["log_u"].shape
        T, Cn, cap = arrs["ix"].shape
        assert Cn == self.n_chains and T >= n_steps
        inj = L.Injection()
        inj.n_steps, inj.cap = T, cap
        for k, a in arrs.items():
            setattr(inj, k, a.ctypes.data)
        return inj, arrs

    def mh_steps(self, n_steps: int, injection: Optional[dict] = None):
        """Run n_steps MH iterations for all chains on the device.  injection: dict of arrays
        proposed/count [T,C,L] int32, ix/iy [T,C,cap] int32, dz [T,C,cap] f64, log_u [T,C] f64."""
        if self._rowshard is not None:
            return self._mh_steps_rowshard(int(n_steps), injection)
        if injection is None:
            L.check(self.lib.bnn_mh_steps(self._h, int(n_steps), None, self._stream()))
            return
        inj, keep = self._pack_injection(injection, n_steps)
        L.check(self.lib.bnn_mh_steps(self._h, int(n_steps), C.byref(inj), self._stream()))

    # ---------------------------------------------------------------- row sharding (SURVEY.md 8e-2)
    def enable_rowshard(self, n_train_global: int, all_reduce_sum="manual"):
        """Rows of X are split over the ranks (set_data was given this rank's rows); all_reduce_sum(t) sums the device
        tensor t in place over the ranks (rowshard.dist_all_reduce_sum on NCCL / gloo).  "manual": the caller drives
        rowshard_update / rowshard_local / rowshard_commit itself (chains_init then stops before the initial accept).
        Call before chains_init.  Every rank must use the same seeds / injected draws."""
        L.check(self.lib.bnn_rowshard_config(self._h, int(n_train_global)))
        self._rowshard = all_reduce_sum

    def rowshard_update(self, accept_mode: int, propose: bool, injection: Optional[dict] = None):
        """accept_mode 0 none / 1 MH accept / 2 initial state; propose: draw (or take the injected) proposal and run the
        forward pass over the local rows."""
        if propose and injection is not None:
            inj, keep = self._pack_injection(injection, 1)
            L.check(self.lib.bnn_rowshard_update(self._h, int(accept_mode), 1, C.byref(inj), self._stream()))
            return
        L.check(self.lib.bnn_rowshard_update(self._h, int(accept_mode), int(bool(propose)), None, self._stream()))

    def rowshard_local(self) -> torch.Tensor:
        """Per-chain sums of this rank's partials: device tensor [C, n_values], the operand of the all-reduce."""
        red = torch.empty((self.n_chains, int(self.lib.bnn_rowshard_n_values(self._h))), dtype=torch.float64, device=self.device)
        L.check(self.lib.bnn_rowshard_local(self._h, _ptr(red), self._stream()))
        return red

    def rowshard_commit(self, red: torch.Tensor):
        L.check(self.lib.bnn_rowshard_commit(self._h, _ptr(red), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()      # red may be released by the caller

    def _all_reduce_own(self, reds):
        self._rowshard(reds[0])                   # the exchange step: C * n_values doubles

    def _mh_steps_rowshard(self, n_steps, injection):
        if not callable(self._rowshard):
            raise L.NpbnnError("manual row sharding: drive rowshard_update / rowshard_local / rowshard_commit yourself")
        rowshard.mh_steps([self], n_steps, injection, self._all_reduce_own)

    def read_state(self, weights=True) -> ChainState:
        n = self.n_chains
        f64 = np.empty((n, L.F_STRIDE))
        i32 = np.empty((n, L.I_STRIDE), dtype=np.int32)
        w = np.empty((n, self.net.n_params)) if weights else None
        L.check(self.lib.bnn_chains_read(self._h, _np_ptr(f64), _np_ptr(i32), _np_ptr(w), self._stream()))
        return ChainState(f64, i32, w, self.net, self.K)

    def snapshot(self, slot: int):
        """Queue an asynchronous export of the chain state into ring slot `slot` (bnn_chains_snapshot); no wait."""
        L.check(self.lib.bnn_chains_snapshot(self._h, int(slot), self._stream()))

    def snapshot_ready(self, slot: int) -> bool:
        return self.lib.bnn_snapshot_ready(self._h, int(slot)) == 1

    def snapshot_read(self, slot: int, weights=True) -> ChainState:
        """Wait for ring slot `slot`, return it as a ChainState and free the slot."""
        n = self.n_chains
        f64 = np.empty((n, L.F_STRIDE))
        i32 = np.empty((n, L.I_STRIDE), dtype=np.int32)
        w = np.empty((n, self.net.n_params)) if weights else None
        L.check(self.lib.bnn_snapshot_read(self._h, int(slot), _np_ptr(f64), _np_ptr(i32), _np_ptr(w)))
        return ChainState(f64, i32, w, self.net, self.K)

    def snapshot_read_indicators(self, slot: int, weight=True, feature=True):
        """The indicators ring slot `slot` holds (read_indicators' layouts); call before snapshot_read frees the slot."""
        ind = np.empty((self.n_chains, self._p0)) if weight else None
        fi = np.empty((self.n_chains, self.net.n_features)) if feature else None
        L.check(self.lib.bnn_snapshot_read_indicators(self._h, int(slot), _np_ptr(ind), _np_ptr(fi)))
        if ind is not None:
            ind = ind.reshape((self.n_chains,) + tuple(self.net.shapes[0]))
        return ind, fi

    def read_indicators(self, weight=True, feature=True):
        """(weight indicators [C, out0, in0+b0] or None, feature indicators [C, F] or None) of the chains' current state."""
        ind = np.empty((self.n_chains, self._p0)) if weight else None
        fi = np.empty((self.n_chains, self.net.n_features)) if feature else None
        L.check(self.lib.bnn_chains_read_indicators(self._h, _np_ptr(ind), _np_ptr(fi), self._stream()))
        if ind is not None:
            ind = ind.reshape((self.n_chains,) + tuple(self.net.shapes[0]))
        return ind, fi

    def write_indicators(self, ind=None, fi=None):
        """Set the chains' current indicators (weight [C, out0, in0+b0], feature [C, F], 0/1; None: unchanged) and score
        their current weights under them as chains_init scores w0 (bnn_chains_write_indicators)."""
        ind = None if ind is None else np.ascontiguousarray(np.reshape(ind, (self.n_chains, self._p0)), dtype=np.float64)
        fi = None if fi is None else np.ascontiguousarray(np.reshape(fi, (self.n_chains, self.net.n_features)), dtype=np.float64)
        L.check(self.lib.bnn_chains_write_indicators(self._h, _np_ptr(ind), _np_ptr(fi), self._stream()))
        if callable(self._rowshard) and (ind is not None or fi is not None):
            rowshard.exchange([self], self._all_reduce_own, 2)

    def write_state(self, st: ChainState):
        """Write an edited host copy of the state arrays back (bnn_chains_write)."""
        f64 = np.ascontiguousarray(st.f64, dtype=np.float64)
        i32 = np.ascontiguousarray(st.i32, dtype=np.int32)
        assert f64.shape == (self.n_chains, L.F_STRIDE) and i32.shape == (self.n_chains, L.I_STRIDE)
        L.check(self.lib.bnn_chains_write(self._h, _np_ptr(f64), _np_ptr(i32), self._stream()))

    def set_prior_scales(self, entry_scales):
        """Per-entry prior scales [C, n_params] of the chains (None: back to per-layer scalars) and the refresh of
        logPrior / logPost that MCMC.gibbs_step does (BNN_env.py:534-538)."""
        e = None
        if entry_scales is not None:
            e = np.ascontiguousarray(entry_scales, dtype=np.float64)
            assert e.shape == (self.n_chains, self.net.n_params), e.shape
        L.check(self.lib.bnn_chains_set_prior_scales(self._h, _np_ptr(e), self._stream()))

    def set_additional_prob(self, values):
        """additional_prob [C] of the chains' device-drawn proposals (bnn_chains_set_additional_prob); None: 0."""
        a = None
        if values is not None:
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(values, dtype=np.float64), (self.n_chains,)))
        L.check(self.lib.bnn_chains_set_additional_prob(self._h, _np_ptr(a), self._stream()))

    def set_temperature(self, temps):
        t = np.ascontiguousarray(temps, dtype=np.float64)
        assert t.shape == (self.n_chains,)
        L.check(self.lib.bnn_chains_set_temperature(self._h, _np_ptr(t), self._stream()))

    def gather(self, slot: int = L.F_LOGPOST) -> torch.Tensor:
        """One f64 state slot of every local chain as a device tensor [C] (send buffer of the MC3 all-gather)."""
        out = torch.empty(self.n_chains, dtype=torch.float64, device=self.device)
        L.check(self.lib.bnn_chains_gather(self._h, int(slot), _ptr(out), self._stream()))
        return out

    def forward_time(self, reset=True):
        """(total device ms, launches) of the forward kernel since the last reset (option time_forward=1)."""
        ms, n = C.c_double(), C.c_int64()
        L.check(self.lib.bnn_forward_time(self._h, C.byref(ms), C.byref(n), int(reset)))
        return ms.value, n.value

    def measure_fp64_peak(self) -> float:
        tf = C.c_double()
        L.check(self.lib.bnn_measure_fp64_peak(self._h, C.byref(tf)))
        return tf.value

    def synchronize(self):
        torch.cuda.current_stream(self.device).synchronize()

    # ---------------------------------------------------------------- prediction
    def _set_pattern(self, pattern):
        """Zero pattern [n_params] (0/1) of the weight sets of this call (predshard.zero_pattern), or None: dense kernels.
        Set on every call, so a cached engine never carries one network's pattern into the next network's call."""
        pt = None
        if pattern is not None:
            pt = np.ascontiguousarray(pattern, dtype=np.float64)
            assert pt.shape == (self.net.n_params,), pt.shape
        L.check(self.lib.bnn_set_predict_mask(self._h, _np_ptr(pt)))

    def predict(self, x, weight_sets, alphas=None, override=None, mean=True, votes=False, dense=False, device_out=False,
                pattern=None):
        """Posterior prediction over rows of x for every weight set (reference BNN_lib.py:376-392).
        override: (cols, vals) PDP column overwrite (BNN_pdp.py:65).  pattern: zero pattern of the weight sets (a
        block-masked network then runs the block-sparse kernels; None: dense kernels).  Returns dict of numpy arrays
        (device_out: of tensors on this engine's device)."""
        w = self._as_sets(weight_sets)
        self._set_pattern(pattern)
        with torch.cuda.device(self.device):
            xd = self._dev(x, torch.float64)
            wd = self._dev(w, torch.float64)
            ad = self._dev(alphas, torch.float64)
            n, S = xd.shape[0], wd.shape[0]
            W = self.K if self.net.lik == L.LIK_CATEGORICAL else self.O
            md = torch.empty((n, W), dtype=torch.float64, device=self.device) if mean else None
            vd = torch.empty((n, W), dtype=torch.float64, device=self.device) if votes else None
            dd = torch.empty((S, n, W), dtype=torch.float64, device=self.device) if dense else None
            oc = ov = None
            n_ov = 0
            if override is not None:
                oc = np.ascontiguousarray(override[0], dtype=np.int32)
                ov = np.ascontiguousarray(override[1], dtype=np.float64)
                n_ov = len(oc)
            L.check(self.lib.bnn_predict(self._h, _ptr(xd), n, _ptr(wd), S, _ptr(ad), _np_ptr(oc), _np_ptr(ov), n_ov,
                                         _ptr(md), _ptr(vd), _ptr(dd), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
            out = {}
            if mean:
                out["mean"] = md
            if votes:
                out["votes"] = vd
            if dense:
                out["dense"] = dd
            return out if device_out else {k: v.cpu().numpy() for k, v in out.items()}

    def predict_sample(self, x, weight_sets, u=None, alphas=None, post_predictions=True, seed=None, row0=0, set0=0,
                       device_out=False, pattern=None):
        """sample_from_categorical (BNN_lib.py:682-713) fused into the prediction pass.  u [n, S]: the reference's
        uniforms (np.random.random(S) per instance); u=None: uniforms generated in the kernel from `seed` (Philox,
        nothing of size n x S is stored), keyed on (row0 + row, set0 + set): rows row0... and sets set0... of a larger
        call draw that call's uniforms.  Returns dict(predictions [n,K], class_counts [S,K], post_predictions [n,S]
        or None) of numpy arrays (device_out: of float64 tensors on this engine's device).  pattern: as in predict."""
        w = self._as_sets(weight_sets)
        self._set_pattern(pattern)
        with torch.cuda.device(self.device):
            xd, wd, ad = self._dev(x, torch.float64), self._dev(w, torch.float64), self._dev(alphas, torch.float64)
            n, S = xd.shape[0], wd.shape[0]
            est = torch.empty((n, self.K), dtype=torch.float64, device=self.device)
            cc = torch.empty((S, self.K), dtype=torch.int32, device=self.device)
            pp = torch.empty((n, S), dtype=torch.float64, device=self.device) if post_predictions else None
            if u is None:
                L.check(self.lib.bnn_predict_sample_philox_at(self._h, _ptr(xd), n, _ptr(wd), S, _ptr(ad),
                                                              int(0 if seed is None else seed) & (2 ** 64 - 1), int(row0),
                                                              int(set0), _ptr(est), _ptr(cc), _ptr(pp), self._stream()))
            else:
                ud = self._dev(u, torch.float64)
                assert tuple(ud.shape) == (n, S)
                L.check(self.lib.bnn_predict_sample(self._h, _ptr(xd), n, _ptr(wd), S, _ptr(ad), _ptr(ud), _ptr(est), _ptr(cc),
                                                    _ptr(pp), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()
            if device_out:
                return {"predictions": est, "class_counts": cc.to(torch.float64), "post_predictions": pp}
            return {"predictions": est.cpu().numpy(), "class_counts": cc.cpu().numpy().astype(np.float64),
                    "post_predictions": None if pp is None else pp.cpu().numpy()}
