"""ARSAgent with the reference's constructor, fields and train/update interface
(ars/ars_agent.py:15-220), running on the batched engine.

What is kept: `ARSAgent(real_env_param, agent_param, data_path, seed, guess_param, approx_error,
sim_thresh)`, `.policy .mean .covariance .database .sim_threshold .estimated_param`,
`sort_directions / update_policy / runOneIteration / runTraining`, the quirks that define its
numbers (all N sorted directions are used, b is only a divisor; population std; uniform
perturbations; no action clipping; V2 statistics cumulative over every real state since
iteration 0 and applied from the next iteration on).

What changes underneath: the 2N rollouts of an iteration are one kernel launch instead of a
sequential Python loop; perturbations come either from numpy's global stream exactly like the
reference (`delta_source="numpy"`, default: same seed => same learning curve as the reference) or
from in-kernel Philox (`delta_source="philox"`: nothing is uploaded).  Under Ray the reference
wraps the class with @ray.remote; here `ARSAgent.remote(...)` is available when ray is installed.

Documented deviations (SURVEY appendix D): safe mode with N > 1 compacts the surviving
(delta, r+, r-) triples instead of raising IndexError (D-2); `estimated_param` is a copy, the
caller's dataclass is not mutated (D-5); `.covariance` is the diagonal matrix of the tracked
variances (only the diagonal is ever used, ars/environment.py:32); `.saved_states` stays empty
unless `keep_states=True` (D-6: the reference keeps every state ever seen).
"""
import dataclasses

import os

import numpy as np
import torch

from . import _lib, ops
from ._lib import ARS_AGENT
from .database import Database
from .engine import ArsEngine
from .environment import Environment


def _env_params(p, variant_direction=(1.0, 0.0)):
    return _lib.make_params(n=p.n, l_i=p.l_i, m_i=p.m_i, k=p.k, h=p.h, direction=variant_direction)


class ARSAgent:
    def __init__(self, real_env_param, agent_param, data_path=None, seed=None, guess_param=None,
                 approx_error=None, sim_thresh=None, *, delta_source="numpy", keep_states=False,
                 record_trajectories=None, device=None, group=None, distributed=None):
        assert delta_source in ("numpy", "philox")
        self.real_env_param = real_env_param
        self.real_world = Environment(real_env_param, device=device)
        self.agent_param = agent_param
        self.delta_source = delta_source
        self.keep_states = keep_states

        self.database = Database()
        self.estimated_param = None
        self.sim_threshold = None
        if agent_param.safe:
            self.database.load(data_path)
            if guess_param is not None and data_path is not None:
                from .estimator import Estimator
                print("Using computed estimation...")
                self.estimator = Estimator(self.database, guess_param, capacity=1)
                self.estimated_param = self.estimator.estimate_real_env_param(seed=0 if seed is None else seed)
            elif approx_error is not None:
                print("Using approximated estimation...")
                # drawn BEFORE np.random.seed, like ars_agent.py:52 vs :95
                delta = np.random.rand(3)
                delta = delta / np.linalg.norm(delta, ord=2) * approx_error
                self.estimated_param = dataclasses.replace(
                    real_env_param, name="LeonSwimmer-Simulator",
                    m_i=real_env_param.m_i + delta[0], l_i=real_env_param.l_i + delta[1],
                    k=real_env_param.k + delta[2])
            else:
                print("Using exact estimation...")
                self.estimated_param = dataclasses.replace(real_env_param)
            print(f"Used estimation: {self.estimated_param}")
            if sim_thresh is not None:
                alpha = sim_thresh.compute_alpha(agent_param.H)
                self.sim_threshold = agent_param.threshold + alpha * real_env_param.epsilon
                print(f"Simulator threshold is {self.sim_threshold}")
            else:
                raise NotImplementedError(
                    "safe exploration needs sim_thresh (the reference leaves this case as a TODO, "
                    "ars_agent.py:70-71)")

        n_act = self.real_world.env.action_space.shape[0]
        n_obs = self.real_world.env.observation_space.shape[0]
        if agent_param.initial_w == "Zero":
            W0 = np.zeros((n_act, n_obs))
        else:
            W0 = np.load(agent_param.initial_w)
            assert W0.shape == (n_act, n_obs)

        self.engine = ArsEngine(
            _env_params(real_env_param), N=agent_param.N, b=agent_param.b, alpha=agent_param.alpha,
            nu=agent_param.nu, H=agent_param.H, v2=not agent_param.V1, semantics=ARS_AGENT,
            seed=seed, initial_policy=W0, device=device, group=group, distributed=distributed,
            sim_params=_env_params(self.estimated_param) if agent_param.safe else None,
            sim_threshold=self.sim_threshold)
        self.record_trajectories = record_trajectories
        self.saved_states = []
        self.screened_fraction = []  # per iteration, safe mode

        self.n_seed = seed
        np.random.seed(self.n_seed)

    # ---- host views of device state ----
    @property
    def policy(self):
        return self.engine.policy_numpy()

    @policy.setter
    def policy(self, W):
        self.engine.set_policy(np.asarray(W, dtype=np.float64))

    @property
    def mean(self):
        return None if self.agent_param.V1 else self.engine.mean.cpu().numpy()

    @property
    def covariance(self):
        if self.agent_param.V1:
            return None
        return np.diag(self.engine.inv_sigma.cpu().numpy() ** -2.0)

    # ---- reference methods ----
    def sort_directions(self, deltas, rewards):
        """argsort(max(r+, r-))[::-1] as a list (ars_agent.py:97-108), computed by swm_ars_topb."""
        r = torch.as_tensor(np.asarray(rewards, dtype=np.float64)[:2 * len(deltas)]).to(self.engine.device)
        return ops.ars_topb(r).cpu().tolist()

    def update_policy(self, deltas, rewards, order):
        """policy += alpha/(b sigma_R) sum_{i in order} (r+_i - r-_i) delta_i (ars_agent.py:110-130)."""
        dev = self.engine.device
        N = len(deltas)
        d = torch.as_tensor(np.asarray(deltas, dtype=np.float64).reshape(N, -1)).to(dev)
        r = torch.as_tensor(np.asarray(rewards, dtype=np.float64)[:2 * N]).to(dev)
        o = torch.as_tensor(np.asarray(order, dtype=np.int32)).to(dev)
        ops.ars_update(self.engine.W, r, N, order=o, n_order=len(order), divisor=self.agent_param.b,
                       ddof=0, alpha=self.agent_param.alpha, deltas=d)

    def runOneIteration(self):
        """One ARS iteration; returns the list of real-world returns like ars_agent.py:132-185
        (2 per direction that was rolled out, in direction order)."""
        eng, ap = self.engine, self.agent_param
        deltas = None
        host_deltas = None
        if self.delta_source == "numpy":
            host_deltas = [2 * np.random.rand(*self.policy_shape) - 1 for _ in range(ap.N)]
            deltas = torch.as_tensor(np.stack(host_deltas).reshape(ap.N, -1)).to(eng.device)
        record = self.record_trajectories or self.keep_states
        pre_W = eng.policy_numpy() if record else None
        returns = eng.run_iteration(deltas=deltas, want_trajectory=bool(record))
        rewards = returns.cpu().numpy()
        if ap.safe:
            ok = ~np.isnan(rewards.reshape(-1, 2)[:, 0])
            self.screened_fraction.append(1.0 - ok.mean())
            for r in rewards.reshape(-1, 2)[ok].ravel():
                if r < ap.threshold:
                    print(f"Obtained in real world rollout a return of {r}, below the "
                          f"threshold {ap.threshold}")
            kept = rewards.reshape(-1, 2)[ok].ravel().tolist()
        else:
            ok = np.ones(ap.N, dtype=bool)
            kept = rewards.tolist()
        if record:
            traj = eng.last.trajectory.cpu().numpy()  # [H, 2N, no]
            if host_deltas is None:
                host_deltas = ops.philox_deltas(eng.seed, eng.iteration - 1, 0, ap.N, eng.ws,
                                                eng.delta_dist, eng.device).cpu().numpy()
            kept_dirs = np.nonzero(ok)[0]
            if len(kept_dirs):
                d = np.stack([np.asarray(host_deltas[i]).reshape(pre_W.shape) for i in kept_dirs])
                pols = np.stack([pre_W + ap.nu * d, pre_W - ap.nu * d], axis=1).reshape((-1,) + pre_W.shape)
                cols = np.stack([2 * kept_dirs, 2 * kept_dirs + 1], axis=1).reshape(-1)  # [+0, -0, +1, -1, ...]
                self.database.extend_from_rollout(traj[:, cols, :], pols)
                if self.keep_states and not ap.V1:
                    for c in cols:
                        self.saved_states += traj[:, c, :].tolist()
        return kept

    @property
    def policy_shape(self):
        n = self.real_env_param.n
        return (n - 1, 2 * n + 2)

    def runTraining(self, save_data_path=None, save_policy_path=None):
        """n_iter + 1 iterations; curve[j] = mean of iteration j's returns (previous value if every
        direction was screened out) -- ars_agent.py:187-220."""
        if save_data_path is not None and self.record_trajectories is None:
            self.record_trajectories = True
        ap = self.agent_param
        rewards = [np.mean(self.runOneIteration())]
        for j in range(1, ap.n_iter + 1):
            all_rewards = self.runOneIteration()
            r = np.mean(all_rewards) if len(all_rewards) > 0 else rewards[-1]
            rewards.append(r)
            if j % 10 == 0:
                print(f"Seed {self.n_seed} ------ V1 = {ap.V1}; n={self.real_env_param.n}; "
                      f"h={self.real_env_param.h}; alpha={ap.alpha}; nu={ap.nu}; N={ap.N}; b={ap.b}; "
                      f"m_i={self.real_env_param.m_i}; l_i={self.real_env_param.l_i} "
                      f"------ Iteration {j}/{ap.n_iter}: {r}")
                if save_data_path is not None:
                    self.database.save(save_data_path)
        self.real_world.close()
        if save_policy_path is not None:
            np.save(save_policy_path, self.policy)
        return np.array(rewards)


try:  # optional: the reference decorates the class with @ray.remote (ars_agent.py:15)
    import ray as _ray

    # an actor without a GPU share would see CUDA_VISIBLE_DEVICES='' and fail in require_cuda(): by default
    # eight agents share one GPU (ars/experiment.py runs one actor per seed)
    ARSAgent.remote = staticmethod(lambda *a, **k: _ray.remote(
        num_gpus=float(os.environ.get("SWM_RAY_NUM_GPUS", "0.125")))(ARSAgent).remote(*a, **k))
except Exception:  # ray is not installed in this image
    pass
