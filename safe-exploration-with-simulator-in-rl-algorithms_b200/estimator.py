"""Parameter estimation with the reference's interface (ars/estimator.py:16-120).

`Estimator.I(x)` -- the one-step-prediction error of a candidate (m_i, l_i, k) against recorded
real trajectories -- is H-1 *independent* single steps per trajectory, so it maps onto one
batched policy product + one batched step (swm_policy_actions, swm_step_batched) per trajectory
instead of H-1 Python iterations.  `I_population` evaluates a whole population of candidates over all
recorded transitions in one fused launch (swm_prediction_error).  `estimate_on_device` runs CMA-ES on the
device (swm_cmaes_generation: sampling, objective and update, replayed as a CUDA graph); the reference's
third-party host optimiser (`cma`) is still what `estimate_real_env_param` calls when it can be imported.
"""
import dataclasses

import numpy as np
import torch

from . import _lib, ops
from .parameters import EnvParam


class Estimator:
    def __init__(self, database, guess_param, capacity, unknowns=("m_i", "l_i", "k"), device=None):
        assert database.size > 0, "Database is empty"
        assert len(database.trajectories[0]) == guess_param.H, "Rollouts are not the same"
        self.guess_param = guess_param
        self.unknowns = unknowns
        self.database = database
        self.subset = np.random.randint(0, self.database.size, capacity)
        self.iter = 0
        _lib.require_cuda()
        self.device = torch.device(device) if device is not None else torch.device(
            "cuda", torch.cuda.current_device())
        self._cache = {}
        self._data = None

    def _device_data(self, max_candidates):
        """The subset's trajectories and policies, uploaded once, with objective scratch for max_candidates."""
        if self._data is None or self._data.max_candidates < max_candidates:
            traj = torch.stack([self._traj(int(k))[0] for k in self.subset])
            pol = torch.stack([self._traj(int(k))[1].reshape(-1) for k in self.subset])
            self._data = ops.EstimateData(traj, pol, self.unknowns, max_candidates)
        return self._data

    def _base_params(self):
        p = self.guess_param
        return _lib.make_params(n=p.n, l_i=p.l_i, m_i=p.m_i, k=p.k, h=p.h)

    def _traj(self, k):
        if k not in self._cache:
            t = torch.as_tensor(np.asarray(self.database.trajectories[k], dtype=np.float64))
            p = torch.as_tensor(np.asarray(self.database.policies[k], dtype=np.float64))
            self._cache[k] = (t.to(self.device).contiguous(), p.to(self.device).contiguous())
        return self._cache[k]

    def convert_to_env_param(self, x):
        d = dataclasses.asdict(self.guess_param)
        for i, name in enumerate(self.unknowns):
            d[name] = x[i]
        return EnvParam(**d)

    def I(self, x):
        """sum_k sum_t || step_x(s_t, W_k s_t) - s_{t+1} ||_2 (ars/estimator.py:36-62)."""
        p = self.convert_to_env_param(x)
        params = _lib.make_params(n=p.n, l_i=p.l_i, m_i=p.m_i, k=p.k, h=p.h)
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        for k in self.subset:
            traj, policy = self._traj(int(k))
            s = traj[:-1].contiguous()
            act = ops.policy_actions(params, s, policy.reshape(1, -1), rollouts_per_policy=s.shape[0])
            nxt, _ = ops.step_batched(params, s, act, want_reward=False)
            total = total + torch.linalg.norm(nxt - traj[1:], dim=1).sum()
        return float(total.cpu())

    def I_population(self, xs):
        """Objective for a whole CMA-ES generation (list of candidates) -> list of floats: one fused launch
        (swm_prediction_error) steps every candidate's model from every recorded state; the states' sines and
        cosines and the actions W_k s_t do not depend on the candidate and are formed once."""
        cand = torch.as_tensor(np.asarray(xs, dtype=np.float64).reshape(len(xs), -1)).to(self.device)
        data = self._device_data(min(len(xs), _lib.MAX_CANDIDATES))
        base = self._base_params()
        err = torch.cat([ops.prediction_error(base, data, cand[lo:lo + _lib.MAX_CANDIDATES])
                         for lo in range(0, len(xs), _lib.MAX_CANDIDATES)])
        return err.cpu().tolist()

    def estimate_on_device(self, seed=0, sigma0=1.0, popsize=None, max_generations=None, tolfun=1e-11,
                           tolx=1e-11, generations_per_poll=16):
        """CMA-ES over I on the device, from the reference's start (x0 = the guess, sigma0 = 1,
        ars/estimator.py:103).  The recorded subset is uploaded once; a CUDA graph of `generations_per_poll`
        generations is replayed until the status word the update kernel writes says stop, and that read is the
        only host synchronisation.  -> (EnvParam of the best candidate ever evaluated, info) with info = dict(x,
        f, generations, evaluations, stop, popsize)."""
        d = len(self.unknowns)
        lam = ops.cmaes_default_popsize(d) if popsize is None else int(popsize)
        g = dataclasses.asdict(self.guess_param)
        x0 = [float(g[u]) for u in self.unknowns]
        with torch.cuda.device(self.device):
            data = self._device_data(lam)
            base = self._base_params()
            f64 = dict(dtype=torch.float64, device=self.device)
            state = torch.empty(ops.cmaes_state_doubles(d, lam), **f64)
            cand, fit = torch.empty(lam, d, **f64), torch.empty(lam, **f64)
            ops.cmaes_init(state, x0, lam, sigma0=sigma0, tolfun=tolfun, tolx=tolx,
                           max_generations=max_generations or 0)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(int(generations_per_poll)):
                    ops.cmaes_generation(state, lam, seed, base, data, cand, fit)
            while True:
                graph.replay()
                if state[1].item() != 0.0:
                    break
            v = {k: t.cpu().numpy() for k, t in ops.cmaes_view(state, d, lam).items()}
        self.cmaes_state = state
        info = dict(x=v["best_x"].copy(), f=float(v["best_f"]), generations=int(v["generation"]),
                    evaluations=int(v["generation"]) * lam, stop=_lib.CMAES_STOP[int(v["status"])], popsize=lam)
        return self.convert_to_env_param([float(x) for x in v["best_x"]]), info

    def estimate_real_env_param(self, seed=0):
        """CMA-ES over I (ars/estimator.py:89-110): the third-party `cma` package exactly as the reference calls it
        when it can be imported, else `estimate_on_device(seed=seed)`."""
        try:
            import cma
        except ImportError:
            return self.estimate_on_device(seed=seed)[0]
        d = dataclasses.asdict(self.guess_param)
        x0 = np.array([d[u] for u in self.unknowns], dtype=np.float64)
        es = cma.CMAEvolutionStrategy(x0, 1).optimize(self.I)
        est_x, _, _ = es.best.get()
        return self.convert_to_env_param(est_x)
