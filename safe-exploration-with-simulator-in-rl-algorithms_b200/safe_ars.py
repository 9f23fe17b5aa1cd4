"""Basic_ARS / Safe_ARS with the reference's interface (safe_ars/ars.py:9-153) on the batched
engine: true top-b truncation (`order[:b]`), ARS V1 only, and -- for Safe_ARS -- per-step
state-constraint screening through a simulator environment, fused into the rollout kernel
(each step evaluates the simulator model and the real model from the same state in the same
thread).

The `cost` callable of the reference is arbitrary Python; the kernels implement the one the
reference uses (safe_ars/experiment.py:44, cost(obs) = max_i |obs[3+2i]|) and any maximum of affine
forms of the observation (MaxAffineCost).  A different callable is rejected loudly rather than
silently evaluated on the host.
"""
import numpy as np
import torch

from . import _lib, ops
from ._lib import ARS_TOPB
from .engine import ArsEngine
from .swimmer_env import SwimmerEnv


def builtin_cost(x):
    """cost(obs) = max_i |theta_dot_i| (safe_ars/experiment.py:44)."""
    x = np.asarray(x)
    return np.max(np.abs(x[3::2]))


class MaxAffineCost:
    """cost(obs) = max_j (A[j] . obs + b[j]) over J = 1..32 affine forms of the observation
    obs = [Gdot_x, Gdot_y, th_1, thd_1, ..., th_n, thd_n]; NaN if any form is NaN (like np.max).

    Covers bounds |obs_k| <= c (rows +-e_k), bending limits |th_i - th_{i+1}|, signed velocity bounds
    and the built-in cost (rows +-e_{3+2i}).  A, b must be finite.  Safe_ARS screens with it on the GPU
    (one thread per environment)."""

    def __init__(self, A, b=None):
        A = np.array(A, dtype=np.float64, copy=True)
        if A.ndim != 2 or A.shape[1] % 2 or not _lib.MIN_SEGMENTS <= A.shape[1] // 2 - 1 <= _lib.MAX_SEGMENTS:
            raise ValueError("A must be [J, 2n+2] with %d <= n <= %d, got shape %s"
                             % (_lib.MIN_SEGMENTS, _lib.MAX_SEGMENTS, A.shape))
        J = A.shape[0]
        if not 1 <= J <= _lib.MAX_COST_FORMS:
            raise ValueError("a cost has 1 to %d forms, got %d" % (_lib.MAX_COST_FORMS, J))
        b = np.zeros(J) if b is None else np.array(b, dtype=np.float64, copy=True)
        if b.shape != (J,):
            raise ValueError("b must have shape (%d,), got %s" % (J, b.shape))
        if not (np.isfinite(A).all() and np.isfinite(b).all()):
            raise ValueError("the coefficients of a cost must be finite")
        self.A, self.b = A, b
        self.n = A.shape[1] // 2 - 1
        self.forms = np.ascontiguousarray(np.hstack([A, b[:, None]]))  # [J, 2n+3]: the layout of swm_rollout_costed

    def __call__(self, obs):
        return float(np.max(self.A @ np.asarray(obs, dtype=np.float64) + self.b))


def _check_cost(cost, n):
    if cost is builtin_cost:
        return
    rng = np.random.RandomState(1234)
    for _ in range(8):
        x = rng.normal(size=2 * n + 2) * 3
        if not np.isclose(float(cost(x)), float(builtin_cost(x)), rtol=0, atol=0):
            raise NotImplementedError(
                "Safe_ARS on the GPU supports the reference's cost max_i|obs[3+2i]| only; the "
                "given callable computes something else")


class Basic_ARS:
    """ARS V1 without safe exploration (safe_ars/ars.py:9-100)."""

    delta_source = "numpy"  # "numpy": consume np.random like the reference; "philox": in-kernel

    def _screen(self, real_env):
        return None

    def _t(self, a, dev):
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)

    def _device(self):
        """Device of the environment this agent last trained on, else the current CUDA device."""
        eng = getattr(self, "engine", None)
        return eng.device if eng is not None else torch.device("cuda", torch.cuda.current_device())

    def rollout(self, real_env, policy, H, render=False):
        """-> (R, states[H][2n+2]) like safe_ars/ars.py:13-35 (post-step observations)."""
        res = real_env.rollout_batched(H, policies=np.asarray(policy, dtype=np.float64)[None],
                                       want_trajectory=True, screen=self._screen(real_env))
        self.last_rollout = res
        return float(res.returns.cpu()[0]), res.trajectory[:, 0, :].cpu().numpy().tolist()

    def sort_directions(self, deltas, rewards):
        r = self._t(np.asarray(rewards, dtype=np.float64)[:2 * len(deltas)], self._device())
        return ops.ars_topb(r).cpu().tolist()

    def update_policy(self, deltas, returns, order, alpha):
        """policy += alpha/(len(order) sigma_R) sum_{i in order} (r+ - r-) delta_i
        (safe_ars/ars.py:48-65); self.policy is a host array as in the reference."""
        N = len(deltas)
        dev = self._device()
        W = self._t(self.policy, dev).reshape(-1)
        ops.ars_update(W, self._t(np.asarray(returns)[:2 * N], dev), N,
                       order=torch.as_tensor(np.asarray(order, dtype=np.int32)).to(dev),
                       n_order=len(order), divisor=0.0, ddof=0, alpha=alpha,
                       deltas=self._t(np.asarray(deltas).reshape(N, -1), dev))
        self.policy = W.cpu().numpy().reshape(np.asarray(self.policy).shape)

    def train(self, n_iter, real_env, N, b, alpha, nu, H, return_states=True, seed=0):
        """-> (mean return per iteration [n_iter], states [2N n_iter, H, 2n+2]) like
        safe_ars/ars.py:67-100.  `return_states=False` skips the trajectory download."""
        assert isinstance(real_env, SwimmerEnv)
        n = real_env.n
        eng = ArsEngine(real_env.params(), N=N, b=b, alpha=alpha, nu=nu, H=H, v2=False,
                        semantics=ARS_TOPB, seed=seed, variant=real_env.variant,
                        device=real_env._dev(), step_screen=self._screen(real_env))
        self.engine = eng
        self.policy = np.zeros((n - 1, 2 * n + 2))
        all_returns, states = [], []
        for it in range(n_iter):
            deltas = None
            if self.delta_source == "numpy":
                d = np.stack([2 * np.random.rand(n - 1, 2 * n + 2) - 1 for _ in range(N)])
                deltas = self._t(d.reshape(N, -1), eng.device)
            ret = eng.run_iteration(deltas=deltas, want_trajectory=return_states)
            all_returns.append(float(ret.mean().cpu()))
            if return_states:
                states.append(eng.last.trajectory.permute(1, 0, 2).cpu().numpy())
            if it % 10 == 0:
                print(f"Iteration {it}/{n_iter}: return = {all_returns[-1]}")
        self.policy = eng.policy_numpy()
        st = np.concatenate(states, axis=0) if states else np.zeros((0, H, 2 * n + 2))
        return np.array(all_returns), st


class Safe_ARS(Basic_ARS):
    """ARS V1 with per-step safe exploration through a simulator (safe_ars/ars.py:103-153).

    `sim_env` may also be a sequence of 1..16 SwimmerEnv (an ensemble of simulator models, e.g. points of the set
    the real parameters are known to lie in): a step is then taken only if every model judges it safe.

    `backup_policy` W_b [n-1, 2n+2] and / or `backup_action` u_0 [n-1] (declared extension; default: none) add a
    shield: a step whose action the simulator(s) reject is taken with the backup action W_b obs + u_0 if the same
    simulator(s) judge that safe (zero torque, a damping controller, a known hand controller), and the rollout freezes
    only if the backup is unsafe too.  Without them the agent behaves as the reference.

    `lookahead` K > 0 (declared extension; needs a backup) makes that shield look ahead: an action, the policy's or
    the backup's, is safe only if after it the backup keeps every simulator's cost within sim_threshold for K more
    steps.  That is what lets the shield act on costs of the angles, such as bending limits, which no action changes
    within one explicit-Euler step.  K = 0 is the one-step shield."""

    def __init__(self, cost, real_threshold, sim_threshold, sim_env, backup_policy=None, backup_action=None,
                 lookahead=0):
        if isinstance(sim_env, SwimmerEnv):
            n = sim_env.n
        else:
            envs = list(sim_env)
            if not 1 <= len(envs) <= _lib.MAX_SIM_MODELS:
                raise ValueError("an ensemble has 1 to %d simulator models, got %d" % (_lib.MAX_SIM_MODELS, len(envs)))
            assert all(isinstance(e, SwimmerEnv) for e in envs)
            n = envs[0].n
            if any(e.n != n for e in envs):
                raise ValueError("the simulator models of an ensemble must have the same n, got %s"
                                 % [e.n for e in envs])
            sim_env = envs
        if isinstance(cost, MaxAffineCost):
            if cost.n != n:
                raise ValueError("the cost is for n=%d segments, the environment has n=%d" % (cost.n, n))
        else:
            _check_cost(cost, n)
        self.cost = cost
        self.real_thresh = real_threshold
        self.sim_thresh = sim_threshold
        self.sim_env = sim_env
        self.backup = None
        if backup_policy is not None or backup_action is not None:
            b = ops.backup_array(n, backup_policy, backup_action)  # ValueError for a wrong shape or non-finite value
            ws = (n - 1) * (2 * n + 2)
            self.backup = dict(policy=b[:ws].reshape(n - 1, 2 * n + 2), action=b[ws:])
        self.lookahead = ops.check_lookahead(lookahead, self.backup is not None)  # ValueError without a backup

    def _screen(self, real_env):
        if isinstance(self.sim_env, SwimmerEnv):
            assert self.sim_env.n == real_env.n
            sim = self.sim_env.params()
        else:
            if self.sim_env[0].n != real_env.n:
                raise ValueError("the simulator models have n=%d segments, the real environment has n=%d"
                                 % (self.sim_env[0].n, real_env.n))
            sim = [e.params() for e in self.sim_env]
        screen = dict(sim_params=sim, sim_thresh=self.sim_thresh, real_thresh=self.real_thresh)
        if isinstance(self.cost, MaxAffineCost):
            screen["cost"] = self.cost
        if self.backup is not None:
            screen["backup"] = self.backup
        if self.lookahead > 0:
            screen["lookahead"] = self.lookahead
        return screen

    def isSafe(self, cost, thresh, env, state, action):
        """Simulate `action` from `state` on `env` and compare the cost with the threshold
        (safe_ars/ars.py:111-122).  Leaves env in the simulated state, like the reference.  With a sequence of
        environments: True only if every one of them is safe; each is left in its simulated state."""
        if not isinstance(env, SwimmerEnv):
            return all([self.isSafe(cost, thresh, e, state, action) for e in env])
        env.set_state(state)
        obs, _, _, _ = env.step(action)
        return cost(obs) <= thresh

    def isRecoverable(self, cost, thresh, env, state, action):
        """isSafe with the lookahead K: simulate `action` from `state`, then K steps of the backup action, and True only
        if every one of the K+1 costs is within the threshold (for a sequence of environments: in every one of them).
        With K = 0 this is isSafe."""
        if self.lookahead == 0:
            return self.isSafe(cost, thresh, env, state, action)
        if not isinstance(env, SwimmerEnv):
            return all([self.isRecoverable(cost, thresh, e, state, action) for e in env])
        env.set_state(state)
        obs, _, _, _ = env.step(action)
        if not cost(obs) <= thresh:
            return False
        for _ in range(self.lookahead):
            obs, _, _, _ = env.step(self._backup_action(obs))
            if not cost(obs) <= thresh:
                return False
        return True

    def _backup_action(self, obs):
        return self.backup["policy"] @ np.asarray(obs, dtype=np.float64) + self.backup["action"]

    def shielded_action(self, cost, thresh, env, state, action):
        """The action the shielded rollout takes from `state` (host counterpart of the kernel's decision): `action` if
        isRecoverable judges it safe, else the backup action W_b state + u_0 if isRecoverable judges that safe, else
        None (the rollout freezes).  Without a backup an unsafe action gives None.  Leaves env in its last simulated
        state."""
        if self.isRecoverable(cost, thresh, env, state, action):
            return action
        if self.backup is None:
            return None
        b = self._backup_action(state)
        return b if self.isRecoverable(cost, thresh, env, state, b) else None
