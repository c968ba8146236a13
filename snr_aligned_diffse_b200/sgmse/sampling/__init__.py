"""Sampler factories (mirror of sgmse-bbed/sgmse/sampling/__init__.py:28-171)."""
import numpy as np
import torch
from scipy import integrate

from .correctors import Corrector, CorrectorRegistry
from .predictors import Predictor, PredictorRegistry, ReverseDiffusionPredictor

__all__ = ['PredictorRegistry', 'CorrectorRegistry', 'Predictor', 'Corrector', 'get_pc_sampler', 'get_ode_sampler']


def to_flattened_numpy(x):
    return x.detach().cpu().numpy().reshape((-1,))


def from_flattened_numpy(x, shape):
    return torch.from_numpy(x.reshape(shape))


def timesteps_space(sdeT, sdeN, eps, device, type='linear'):
    return torch.linspace(sdeT, eps, sdeN, device=device)


def _time_vector(B, t, device):
    """[B] float32 device tensor filled with t, tagged with its host value (SDE helpers that need host-side special
    functions, BBED._std, read the tag instead of copying the tensor back)."""
    v = torch.full((B,), float(t), dtype=torch.float32, device=device)
    v._host_value = float(t)
    return v


class GraphedPCLoop:
    """The whole reverse loop of `pc_sampler` (sampling/__init__.py:54-75) as ONE CUDA graph.

    Step i = corrector update(s) + predictor update at t_i: 1 + n_steps network evaluations, the complex noise draws
    and the fused state updates; all N steps are recorded back to back into a single graph (N x ~720 kernel nodes).
    The per-step scalars (t_i, step size, SDE coefficients) are host constants baked into the nodes of step i; the state
    lives in static buffers.  Noise comes from torch's CUDA generator, which advances its Philox offset on every replay."""

    def __init__(self, predictor, corrector, timesteps, Y):
        dev = Y.device
        self.Y = Y.clone()
        self.x = torch.empty_like(self.Y)
        self.mean = torch.empty_like(self.Y)
        self.stream = torch.cuda.Stream(device=dev)
        self.graphs = []
        B = Y.shape[0]
        n = len(timesteps)
        steps = []
        for i in range(n):
            t = timesteps[i]
            stepsize = t - timesteps[i + 1] if i != n - 1 else timesteps[-1]
            steps.append((_time_vector(B, t, dev), stepsize))
        self._steps = steps                          # the captured kernels read these time vectors: keep them alive

        def one(i):
            vec_t, stepsize = steps[i]
            xt, _ = corrector.update_fn(self.x, vec_t, self.Y)
            xt, xm = predictor.update_fn(xt, vec_t, self.Y, stepsize)
            self.x.copy_(xt)
            self.mean.copy_(xm)

        rng = torch.cuda.get_rng_state(dev)          # warm-up draws must not shift the caller's noise sequence
        self.stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(self.stream):
            self.x.copy_(self.Y)
            one(0)                                   # eager warm-up: plans, workspaces, function attributes
            self.stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                for i in range(n):
                    one(i)
            self.graphs.append(g)
        torch.cuda.current_stream(dev).wait_stream(self.stream)
        torch.cuda.set_rng_state(rng, dev)

    def run(self, x0, Y):
        cur = torch.cuda.current_stream(Y.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            self.Y.copy_(Y)
            self.x.copy_(x0)
            for g in self.graphs:
                g.replay()
        cur.wait_stream(self.stream)
        return self.x, self.mean


def get_pc_sampler(predictor_name, corrector_name, sde, score_fn, Y, Y_prior=None, denoise=True, eps=3e-2, snr=0.1,
                   corrector_steps=1, probability_flow: bool = False, intermediate=False, timestep_type=None, graph=None,
                   graph_cache=None, **kwargs):
    """Predictor-corrector sampler; returns a zero-argument callable -> (sample, nfe).

    `graph` (extension): True = the whole reverse loop (every corrector + predictor step: network evaluations, noise
    draws, state updates) is replayed from ONE CUDA graph captured on first use (`GraphedPCLoop`); False = host loop
    with eager launches; None (default) = eager the first time a (shape, settings) combination is seen through
    `graph_cache`, captured and replayed from the second time on, i.e. whenever shapes repeat.  `graph_cache` (a dict,
    e.g. one per model: `ScoreModel.get_pc_sampler` supplies it) keeps the captured loops across sampler objects."""
    predictor_cls = PredictorRegistry.get_by_name(predictor_name)
    corrector_cls = CorrectorRegistry.get_by_name(corrector_name)
    predictor = predictor_cls(sde, score_fn, probability_flow=probability_flow)
    corrector = corrector_cls(sde, score_fn, snr=snr, n_steps=corrector_steps)
    if intermediate:
        raise NotImplementedError("intermediate=True returns an undefined name in the reference "
                                  "(sampling/__init__.py:77-78) and is not supported")
    if not Y.is_cuda:
        Y = Y.cuda()

    def pc_sampler(Y_prior=Y_prior, timestep_type=timestep_type):
        with torch.no_grad():
            if Y_prior is None:
                Y_prior = Y
            xt, _ = sde.prior_sampling(Y_prior.shape, Y_prior if Y_prior.is_cuda else Y_prior.cuda())
            # time grid on the host: every step's scalars are known before the first launch
            timesteps = torch.linspace(sde.T, eps, sde.N)
            ns = len(timesteps) * (corrector.n_steps + 1)
            use_graph = graph
            cache = graph_cache if graph_cache is not None else _local_graphs
            key = (predictor_name, corrector_name, tuple(Y.shape), int(sde.N), float(sde.T), float(eps), float(snr),
                   int(corrector_steps), bool(probability_flow), type(sde).__name__)
            if use_graph is None:
                # shapes repeat -> capture: the first call of a combination runs the host loop, later calls replay.
                # Only with a caller-supplied cache, i.e. through ScoreModel.get_pc_sampler, whose score function is known
                # to be capturable (no host synchronisation); an arbitrary `score_fn` handed to this module-level factory
                # keeps the reference's eager loop unless graph=True is asked for.
                seen = cache.get(("seen",) + key, 0)
                cache[("seen",) + key] = seen + 1
                use_graph = graph_cache is not None and seen >= 1
            if use_graph:
                loop = cache.get(key)
                if loop is None:
                    # the entry holds score_fn alive, so a cache shared between models cannot hand a loop captured for a
                    # collected model to a new object that reuses its id()
                    loop = GraphedPCLoop(predictor, corrector, timesteps, Y)
                    cache[key] = loop
                    loop.score_fn = score_fn
                if getattr(loop, "score_fn", score_fn) is not score_fn:
                    raise RuntimeError("graph_cache holds a loop captured for another score function; use one cache per model")
                xt, xt_mean = loop.run(xt, Y)
                return (xt_mean if denoise else xt), ns
            xt_mean = xt
            B = Y.shape[0]
            for i in range(len(timesteps)):
                t = timesteps[i]
                stepsize = t - timesteps[i + 1] if i != len(timesteps) - 1 else timesteps[-1]
                vec_t = _time_vector(B, t, Y.device)
                xt, xt_mean = corrector.update_fn(xt, vec_t, Y)
                xt, xt_mean = predictor.update_fn(xt, vec_t, Y, stepsize)
            x_result = xt_mean if denoise else xt
            return x_result, ns

    _local_graphs = {}

    return pc_sampler


def get_ode_sampler(sde, score_fn, y, Y_prior=None, inverse_scaler=None, denoise=True, rtol=1e-5, atol=1e-5,
                    timestep_type=None, method='RK45', eps=3e-2, device='cuda', on_device=False, **kwargs):
    """Probability-flow ODE sampler (sampling/__init__.py:95-171).  Default: scipy's RK45 with a host round trip per
    RHS evaluation, as in the reference.  `on_device=True` (extension, RK45 only): the same Dormand-Prince scheme and
    step control with the state and all stage arithmetic resident on the GPU (`sampling/ode.py`)."""
    if not y.is_cuda:
        y = y.cuda()
    predictor = ReverseDiffusionPredictor(sde, score_fn, probability_flow=False)
    rsde = sde.reverse(score_fn, probability_flow=True)

    def denoise_update_fn(x):
        vec_eps = torch.ones(x.shape[0], device=x.device) * eps
        _, x = predictor.update_fn(x, vec_eps, y, 0.03)
        return x

    def ode_sampler(z=None, Y_prior=Y_prior, **kw):
        with torch.no_grad():
            if Y_prior is None:
                Y_prior = y
            xt, _ = sde.prior_sampling(Y_prior.shape, Y_prior if Y_prior.is_cuda else Y_prior.cuda())

            def ode_func(t, x):
                x = from_flattened_numpy(x, y.shape).to(device).type(torch.complex64)
                vec_t = torch.ones(y.shape[0], device=x.device) * t
                return to_flattened_numpy(rsde.sde(x, vec_t, y)[0])

            if on_device:
                if method != 'RK45':
                    raise NotImplementedError("on_device=True implements RK45 only")
                from .ode import rk45_integrate

                def ode_func_dev(t, x):
                    vec_t = torch.full((y.shape[0],), float(t), dtype=torch.float32, device=x.device)
                    return rsde.sde(x, vec_t, y)[0]

                res = rk45_integrate(ode_func_dev, float(sde.T), xt.to(torch.complex64), float(eps), rtol=rtol, atol=atol)
                if res.status != 0:
                    raise RuntimeError("on-device RK45: required step size below the spacing between numbers")
                nfe, x = res.nfev, res.y
            else:
                solution = integrate.solve_ivp(ode_func, (sde.T, eps), to_flattened_numpy(xt), rtol=rtol, atol=atol,
                                               method=method, **kw)
                nfe = solution.nfev
                x = torch.tensor(solution.y[:, -1]).reshape(y.shape).to(device).type(torch.complex64)
            if denoise:
                x = denoise_update_fn(x)
            if inverse_scaler is not None:
                x = inverse_scaler(x)
            return x, nfe

    return ode_sampler
