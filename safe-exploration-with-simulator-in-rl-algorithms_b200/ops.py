"""Tensor-level wrappers over the C ABI (include/swimmer_ars.h).

Every function takes/returns CUDA float64 tensors, enqueues on torch's current stream and does
not synchronise.  These are the batched entry points the reference lacks
(`step_batched(actions[B])`, fused rollouts, the ARS update); the reference-shaped classes in
swimmer_env.py / environment.py / ars_agent.py / safe_ars.py are thin layers over them.
"""
import ctypes
import math
import numbers

import numpy as np
import torch

from . import _lib
from ._lib import (ARS_AGENT, ARS_RLGLUE, ARS_TOPB, DELTA_01, DELTA_PM1, GYM, POLICY_DELTAS,
                   POLICY_EXPLICIT, POLICY_FIXED_ACTION, POLICY_PHILOX, RLGLUE)

__all__ = ["step_batched", "step_batched_models", "accelerations_batched", "rollout", "rollout_models", "backup_array", "check_lookahead", "RolloutResult", "ChunkedRollout", "plan_chunks", "philox_deltas",
           "ars_topb", "ars_update", "pack_exchange", "counter_add", "record_nanmean", "stats_finalize", "stats_merge", "reduce_returns", "screen_mask", "policy_actions", "update_args",
           "EstimateData", "prediction_error", "cmaes_default_popsize", "cmaes_state_doubles", "cmaes_view", "cmaes_init",
           "cmaes_sample", "cmaes_update", "cmaes_generation",
           "fp64_probe", "obs_dim", "act_dim", "policy_size", "reset_state", "lane_split_envs_per_warp", "rollout_kernel_choice"]


def obs_dim(n):
    return 2 * n + 2


def act_dim(n):
    return n - 1


def policy_size(n):
    return (n - 1) * (2 * n + 2)


def lane_split_envs_per_warp(n):
    """Environments per warp (= per stats_partial row) of the lane-split rollout kernel: 32 / L with
    L = 4, 8 or 16 lanes per environment (csrc/lane_rollout.cuh LaneSplit)."""
    return 32 // (4 if n + 1 <= 4 else 8 if n + 1 <= 8 else 16)


def rollout_kernel_choice(params, B, *, fixed_actions=False, rollouts_per_policy=1, kernel=0):
    """Name of the rollout kernel swm_rollout picks for a gym-dynamics batch of B environments on the current
    device: 'thread' (one thread per environment), 'lanes' (one environment over 4/8/16 lanes) or 'lanes2'
    (lanes + a second, operator warp per lane group)."""
    cfg = _lib.SwmRollout()
    cfg.policy_mode = POLICY_FIXED_ACTION if fixed_actions else POLICY_PHILOX
    cfg.H, cfg.B, cfg.rollouts_per_policy, cfg.kernel = 1, int(B), int(rollouts_per_policy), int(kernel)
    k = _lib.lib().swm_rollout_kernel_choice(ctypes.byref(params), ctypes.byref(cfg))
    _lib.check(min(k, 0))
    return {_lib.KERNEL_THREAD: "thread", _lib.KERNEL_LANES: "lanes", _lib.KERNEL_LANES2: "lanes2",
            _lib.KERNEL_LANES3: "lanes3"}[k]


def reset_state(n, variant=GYM, device="cuda"):
    """reset() of remy_swimmer_env.py:58-67 (gym) or env_start of SwimmerEnvironment.cpp:39-42."""
    s = torch.zeros(2 * n + 2, dtype=torch.float64, device=device)
    if variant == GYM:
        s[2::2] = 1.5707963267948966
    else:
        s[:] = 0.001
    return s


def _dev(t):
    return t.device if t is not None else torch.device("cuda", torch.cuda.current_device())


def step_batched(params, states, actions, variant=GYM, out=None, want_reward=True):
    """states[B, 2n+2], actions[B, n-1] -> (next_states[B, 2n+2], rewards[B])."""
    _lib.require_cuda()
    n = params.n
    B = states.shape[0]
    _lib.f64(states, (B, obs_dim(n)))
    _lib.f64(actions, (B, act_dim(n)))
    states, actions = states.contiguous(), actions.contiguous()
    out = torch.empty_like(states) if out is None else out
    rew = torch.empty(B, dtype=torch.float64, device=states.device) if want_reward else None
    if B == 0:
        return out, rew
    with torch.cuda.device(states.device):
        _lib.check(_lib.lib().swm_step_batched(ctypes.byref(params), variant, _lib.ptr(states),
                                               _lib.ptr(actions), _lib.ptr(out), _lib.ptr(rew), B,
                                               _lib.stream_ptr()))
    return out, rew


def step_batched_models(params_list, states, actions, out=None, want_reward=False):
    """states[M, T, 2n+2], actions[M, T, n-1]: model m (params_list[m]) steps its T environments, all
    in one launch (swm_step_batched_models; at most MAX_MODELS_PER_STEP models per launch, more are
    chunked).  -> (next_states[M, T, 2n+2], rewards[M, T] or None)."""
    _lib.require_cuda()
    M = len(params_list)
    n = params_list[0].n
    T = states.shape[1]
    _lib.f64(states, (M, T, obs_dim(n)))
    _lib.f64(actions, (M, T, act_dim(n)))
    states, actions = states.contiguous(), actions.contiguous()
    out = torch.empty_like(states) if out is None else out
    rew = torch.empty(M, T, dtype=torch.float64, device=states.device) if want_reward else None
    with torch.cuda.device(states.device):
        for lo in range(0, M, _lib.MAX_MODELS_PER_STEP):
            hi = min(M, lo + _lib.MAX_MODELS_PER_STEP)
            arr = (_lib.SwmParams * (hi - lo))(*params_list[lo:hi])
            _lib.check(_lib.lib().swm_step_batched_models(
                arr, hi - lo, T, _lib.ptr(states[lo:hi]), _lib.ptr(actions[lo:hi]), _lib.ptr(out[lo:hi]),
                _lib.ptr(rew[lo:hi]) if rew is not None else None, _lib.stream_ptr()))
    return out, rew


def accelerations_batched(params, states, actions, variant=GYM):
    """-> acc[B, n+2] = [Gdd_x, Gdd_y, thdd_1..n] (compute_accelerations)."""
    _lib.require_cuda()
    n = params.n
    B = states.shape[0]
    _lib.f64(states, (B, obs_dim(n)))
    _lib.f64(actions, (B, act_dim(n)))
    states, actions = states.contiguous(), actions.contiguous()
    acc = torch.empty(B, n + 2, dtype=torch.float64, device=states.device)
    with torch.cuda.device(states.device):
        _lib.check(_lib.lib().swm_accelerations_batched(ctypes.byref(params), variant,
                                                        _lib.ptr(states), _lib.ptr(actions),
                                                        _lib.ptr(acc), B, _lib.stream_ptr()))
    return acc


class RolloutResult:
    __slots__ = ("returns", "final_state", "trajectory", "stats_partial", "stats_blocks",
                 "violations", "frozen_at", "overrides", "samples")

    def __init__(self):
        for s in self.__slots__:
            setattr(self, s, None)


def rollout(params, H, *, B=None, variant=GYM, actions=None, policies=None, base_policy=None, nu=0.0,
            deltas=None, dir_mask=None, init_perturb=0.0,
            seed=0, iteration=0, iteration_dev=None, dir0=0, delta_dist=DELTA_PM1, rollouts_per_policy=1, mean=None,
            inv_sigma=None, clip_actions=False, init_state=None, want_final=False,
            want_trajectory=False, stats_pivot=None, screen=None, out=None, device=None,
            accumulate_returns=False, kernel=0, schedule=None, _models=None):
    """One fused H-step rollout of B environments (swm_rollout).

    Exactly one of
      actions[B, n-1]                  fixed actions (BASELINE config 2),
      policies[P, n-1, 2n+2]           explicit policies, env e uses policy e // rollouts_per_policy,
      base_policy[n-1, 2n+2] (+ nu, seed, iteration, dir0): W +- nu*delta_k from in-kernel Philox,
                                       B = 2 * n_directions * rollouts_per_policy
                                       (+ deltas[D, n-1, 2n+2]: read delta_k from memory instead)
    dir_mask[D] int32 (base_policy modes): directions with 0 are not rolled out (returns NaN).
    screen = dict(sim_params=..., sim_thresh=..., real_thresh=...) enables Safe_ARS screening with the built-in
    cost max_i |thd_i|; screen["cost"] = a max-of-affine cost (safe_ars.MaxAffineCost: `.n`, `.forms` [J, 2n+3])
    screens with that cost instead (swm_rollout_costed; one thread per environment, one plain launch).
    screen["sim_params"] = a list or tuple of 1..16 params (the real model's n) screens by the whole ensemble, with
    either cost: a step is taken only if every model judges it safe (swm_rollout_ensemble; same kernel and launch).
    screen["backup"] = dict(policy=W_b [n-1, 2n+2] or None, action=u_0 [n-1] or None) adds a shield: a step whose
    action the model(s) reject is taken with the backup action W_b obs + u_0 instead if the same model(s) judge that
    safe, and freezes only otherwise (swm_rollout_shielded; a single simulator is the ensemble of one).  The result
    then has `overrides` [B] int32, the number of steps each environment took with the backup.
    screen["lookahead"] = K (an int in 0..MAX_LOOKAHEAD; K > 0 needs the backup) makes the shield judge every action by
    K more simulator steps: an action is safe only if, after it, the backup keeps every model's cost within sim_thresh
    for K more steps (swm_rollout_lookahead; up to M (K+1) simulator steps per judgement).  K = 0 is the shield above.
    stats_pivot[2n+2] enables the V2 moment accumulation.  `out` may carry preallocated
    tensors (returns, final_state, trajectory, stats_partial) to stay allocation-free in loops.
    kernel: _lib.KERNEL_AUTO (chosen from B, n and the SM count) / KERNEL_THREAD (one thread per
    environment) / KERNEL_LANES (one environment over 4/8/16 lanes; small batches).
    schedule: None = the library decides between one plain launch and a chunked schedule (needs want_final;
    swm_rollout_t.schedule_sub); "plain" = always one launch; (n_sub, chunk) = forced.
    _models: see rollout_models.
    """
    lookahead = check_lookahead(screen.get("lookahead", 0) if screen is not None else 0,
                                screen is not None and screen.get("backup") is not None)
    _lib.require_cuda()
    n = params.n
    no, na, ws = obs_dim(n), act_dim(n), policy_size(n)
    cfg = _lib.SwmRollout()
    keep = []  # keep contiguous temporaries alive until the launch is enqueued
    if actions is not None:
        actions = _lib.f64(actions).contiguous()
        B = actions.shape[0] if B is None else B
        assert tuple(actions.shape) == (B, na)
        cfg.policy_mode, cfg.actions = POLICY_FIXED_ACTION, actions.data_ptr()
        dev = actions.device
        keep.append(actions)
    elif policies is not None:
        policies = _lib.f64(policies).contiguous().reshape(-1, ws)
        P = policies.shape[0]
        B = P * rollouts_per_policy if B is None else B
        assert B == P * rollouts_per_policy
        cfg.policy_mode, cfg.policies = POLICY_EXPLICIT, policies.data_ptr()
        dev = policies.device
        keep.append(policies)
    elif base_policy is not None:
        base_policy = _lib.f64(base_policy).contiguous().reshape(-1)
        assert base_policy.numel() == ws and B is not None
        cfg.policy_mode, cfg.policies = POLICY_PHILOX, base_policy.data_ptr()
        dev = base_policy.device
        keep.append(base_policy)
        if deltas is not None:
            deltas = _lib.f64(deltas).contiguous().reshape(-1, ws)
            assert deltas.shape[0] * 2 * rollouts_per_policy == B
            cfg.policy_mode, cfg.deltas = POLICY_DELTAS, deltas.data_ptr()
            keep.append(deltas)
        if dir_mask is not None:
            assert dir_mask.dtype == torch.int32 and dir_mask.is_contiguous()
            assert dir_mask.numel() * 2 * rollouts_per_policy == B
            cfg.dir_mask = dir_mask.data_ptr()
    else:
        raise ValueError("one of actions / policies / base_policy is required")
    if device is not None:
        dev = torch.device(device)
    cfg.variant, cfg.H, cfg.B = variant, int(H), int(B)
    cfg.rollouts_per_policy = int(rollouts_per_policy)
    cfg.clip_actions = int(bool(clip_actions))
    cfg.accumulate_returns = int(bool(accumulate_returns))
    cfg.kernel = int(kernel)
    if schedule == "plain":
        cfg.schedule_sub = -1
    elif schedule is not None:
        cfg.schedule_sub, cfg.schedule_chunk = int(schedule[0]), int(schedule[1])
    cfg.screen.enabled = int(screen is not None)  # before swm_rollout_stats_blocks: it decides the kernel
    cfg.nu = float(nu)
    cfg.init_perturb = float(init_perturb)
    cfg.philox.seed, cfg.philox.iteration = int(seed) & (2 ** 64 - 1), int(iteration)
    cfg.philox.dir0, cfg.philox.dist = int(dir0), int(delta_dist)
    cfg.philox.iteration_dev = _counter_ptr(iteration_dev)
    if (mean is None) != (inv_sigma is None):
        raise ValueError("mean and inv_sigma go together")
    if mean is not None:
        mean = _lib.f64(mean, (no,)).contiguous()
        inv_sigma = _lib.f64(inv_sigma, (no,)).contiguous()
        cfg.normalize, cfg.mean, cfg.inv_sigma = 1, mean.data_ptr(), inv_sigma.data_ptr()
        keep += [mean, inv_sigma]
    if init_state is not None:
        init_state = _lib.f64(init_state).contiguous().reshape(-1, no)
        cfg.init_state, cfg.init_state_count = init_state.data_ptr(), init_state.shape[0]
        keep.append(init_state)
    res = RolloutResult()
    out = out or {}
    lead = () if _models is None else (len(_models),)  # model-set mode: one row of outputs per model

    def buf(name, shape, dtype=torch.float64):
        t = out.get(name)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=dev)
        assert tuple(t.shape) == tuple(shape) and t.is_contiguous()
        return t

    res.returns = buf("returns", lead + (B,))
    cfg.returns = res.returns.data_ptr()
    if want_final:
        res.final_state = buf("final_state", lead + (B, no))
        cfg.final_state = res.final_state.data_ptr()
    if want_trajectory:
        res.trajectory = buf("trajectory", (H, B, no))
        cfg.trajectory = res.trajectory.data_ptr()
    if stats_pivot is not None:
        stats_pivot = _lib.f64(stats_pivot, (no,)).contiguous()
        with torch.cuda.device(dev):
            nb = _lib.lib().swm_rollout_stats_blocks(ctypes.byref(params), ctypes.byref(cfg), _lib.stream_ptr())
        res.stats_partial = buf("stats_partial", (nb, 2, no))
        res.stats_blocks = nb
        res.samples = float(B) * float(H)
        cfg.stats_partial, cfg.stats_pivot = res.stats_partial.data_ptr(), stats_pivot.data_ptr()
        keep.append(stats_pivot)
    sim_models = None
    if screen is not None:
        cfg.screen.enabled = 1
        if isinstance(screen["sim_params"], (list, tuple)):
            sim_models = screen["sim_params"]  # an ensemble: cfg.screen.sim is not read
        else:
            cfg.screen.sim = screen["sim_params"]
        cfg.screen.sim_thresh = float(screen["sim_thresh"])
        cfg.screen.real_thresh = float(screen["real_thresh"])
        res.violations = buf("violations", (B,), torch.int32)
        res.frozen_at = buf("frozen_at", (B,), torch.int32)
        cfg.screen.violations = res.violations.data_ptr()
        cfg.screen.frozen_at = res.frozen_at.data_ptr()
    cost = screen.get("cost") if screen is not None else None
    if cost is not None and cost.n != n:
        raise ValueError("the cost is for n=%d segments, the model has n=%d" % (cost.n, n))
    forms = cost.forms if cost is not None else None  # host [J, 2n+3], copied into the launch's arguments
    backup = screen.get("backup") if screen is not None else None
    if backup is not None:
        backup = backup_array(n, backup.get("policy"), backup.get("action"))  # host, copied into the launch's arguments
        res.overrides = buf("overrides", (B,), torch.int32)
        if sim_models is None:
            sim_models = [cfg.screen.sim]
    model_list = _models if _models is not None else sim_models  # the list of the call made below
    if model_list is not None:
        models = (_lib.SwmParams * len(model_list))(*model_list)  # host copies, copied into the launch's arguments
    with torch.cuda.device(dev):
        if _models is not None:
            _lib.check(_lib.lib().swm_rollout_models(models, len(model_list), ctypes.byref(cfg), _lib.stream_ptr()))
        elif backup is not None and lookahead > 0:
            _lib.check(_lib.lib().swm_rollout_lookahead(
                ctypes.byref(params), ctypes.byref(cfg), models, len(model_list),
                None if forms is None else forms.ctypes.data_as(ctypes.c_void_p),
                0 if forms is None else forms.shape[0], backup.ctypes.data_as(ctypes.c_void_p), lookahead,
                res.overrides.data_ptr(), _lib.stream_ptr()))
        elif backup is not None:
            _lib.check(_lib.lib().swm_rollout_shielded(
                ctypes.byref(params), ctypes.byref(cfg), models, len(model_list),
                None if forms is None else forms.ctypes.data_as(ctypes.c_void_p),
                0 if forms is None else forms.shape[0], backup.ctypes.data_as(ctypes.c_void_p),
                res.overrides.data_ptr(), _lib.stream_ptr()))
        elif model_list is not None:
            _lib.check(_lib.lib().swm_rollout_ensemble(
                ctypes.byref(params), ctypes.byref(cfg), models, len(model_list),
                None if forms is None else forms.ctypes.data_as(ctypes.c_void_p),
                0 if forms is None else forms.shape[0], _lib.stream_ptr()))
        elif cost is None:
            _lib.check(_lib.lib().swm_rollout(ctypes.byref(params), ctypes.byref(cfg), _lib.stream_ptr()))
        else:
            _lib.check(_lib.lib().swm_rollout_costed(ctypes.byref(params), ctypes.byref(cfg),
                                                     forms.ctypes.data_as(ctypes.c_void_p), forms.shape[0],
                                                     _lib.stream_ptr()))
    return res


def backup_array(n, policy=None, action=None):
    """The backup action W_b obs + u_0 of a shield as swm_rollout_shielded takes it: a host float64 array of W_b
    [n-1, 2n+2] row-major followed by u_0 [n-1] (None: zero).  Raises ValueError for another shape or a non-finite
    entry."""
    def host(x, shape, name):
        if x is None:
            return np.zeros(shape)
        x = np.array(x.cpu() if torch.is_tensor(x) else x, dtype=np.float64)
        if x.shape != shape:
            raise ValueError("the backup %s must have shape %s for n=%d, got %s" % (name, shape, n, x.shape))
        if not np.isfinite(x).all():
            raise ValueError("the backup %s must be finite" % name)
        return x
    W = host(policy, (act_dim(n), obs_dim(n)), "policy")
    u0 = host(action, (act_dim(n),), "action")
    return np.ascontiguousarray(np.concatenate([W.reshape(-1), u0]))


def check_lookahead(lookahead, has_backup):
    """The lookahead K of a shield as swm_rollout_lookahead takes it: an int in 0..MAX_LOOKAHEAD, and K > 0 only with
    a backup.  Raises ValueError otherwise."""
    if isinstance(lookahead, bool) or not isinstance(lookahead, numbers.Integral):
        raise ValueError("the lookahead must be an integer, got %r" % (lookahead,))
    lookahead = int(lookahead)
    if not 0 <= lookahead <= _lib.MAX_LOOKAHEAD:
        raise ValueError("the lookahead must be in 0..%d, got %d" % (_lib.MAX_LOOKAHEAD, lookahead))
    if lookahead > 0 and not has_backup:
        raise ValueError("a lookahead needs a backup (a zero-torque backup is backup=dict(policy=None, action=None))")
    return lookahead


def rollout_models(params_list, H, **kw):
    """The rollout of `rollout(params, H, **kw)` under each of 1..MAX_SIM_MODELS models with the same n, in one launch
    (swm_rollout_models): env e of model m runs exactly what env e of rollout(params_list[m], ...) runs, with
    model m's physics.  B counts the environments per model; returns is [M, B], final_state [M, B, 2n+2].  For the
    simulator rollouts of ARS screening: linear policies, V1 or V2 without statistics, no screening, trajectory
    or clipping (the library refuses them).  kernel: as for rollout, AUTO chosen for M * B environments."""
    params_list = list(params_list)
    if not 1 <= len(params_list) <= _lib.MAX_SIM_MODELS:
        raise ValueError("need 1 to %d models, got %d" % (_lib.MAX_SIM_MODELS, len(params_list)))
    if any(p.n != params_list[0].n for p in params_list):
        raise ValueError("every model must have the same number of segments")
    return rollout(params_list[0], H, _models=params_list, **kw)


def plan_chunks(B, unit, n_sub, H, chunk):
    """Host-side partition behind ChunkedRollout: B environments in whole groups of `unit` (the envs that
    share a direction) are cut into at most `n_sub` contiguous sub-batches, H steps into chunks of `chunk`
    (a multiple of 64; the last one may be shorter).  -> ([(lo, hi), ...], [len, ...])."""
    if chunk % 64 != 0 or chunk < 64:
        raise ValueError("chunk must be a positive multiple of 64")
    if B % unit != 0:
        raise ValueError("B=%d is not a whole number of groups of %d environments" % (B, unit))
    groups = B // unit
    n_sub = max(1, min(int(n_sub), groups))
    cuts = [unit * ((groups * i) // n_sub) for i in range(n_sub + 1)]
    subs = [(cuts[i], cuts[i + 1]) for i in range(n_sub) if cuts[i + 1] > cuts[i]]
    lens = [min(chunk, H - t) for t in range(0, H, chunk)]
    return subs, lens


class ChunkedRollout:
    """One rollout call scheduled as `n_sub` sub-batches x time-chunks of `chunk` steps on `n_sub` CUDA
    streams (swm_rollout launches chained through final_state -> init_state, returns accumulated on the
    device).  Why: one thread owns one environment for all H steps, so a mid-size batch is quantised over
    SM sub-partitions (65,536 three-segment envs = 3.46 warps each, the busiest holds 4) or over waves of
    resident CTAs; short launches from several streams let the hardware refill whatever finishes first
    (+17 % on BASELINE config[1]).  `chunk` must be a multiple of 64: the kernel re-evaluates its tracked
    sines/cosines exactly every 64th step, so every visited state is bit-identical to the single launch
    (returns differ by the rounding of K partial sums).  Not available with screening or trajectory
    output.  All tensors handed in are captured by reference: call `run()` repeatedly (also inside a CUDA
    graph capture) after updating them in place."""

    def __init__(self, params, H, *, B, n_sub=8, chunk=128, variant=GYM, actions=None, base_policy=None,
                 policies=None, rollouts_per_policy=1, stats_pivot=None, want_final=True, device=None, **kw):
        _lib.require_cuda()
        if kw.get("screen") is not None or kw.get("want_trajectory"):
            raise ValueError("chunked rollouts do not support screening or trajectory output")
        n = params.n
        self.params, self.H, self.B, self.variant, self.kw = params, int(H), int(B), variant, kw
        self.R = int(rollouts_per_policy)
        self.actions, self.base_policy, self.policies = actions, base_policy, policies
        src = actions if actions is not None else (base_policy if base_policy is not None else policies)
        self.device = torch.device(device) if device is not None else src.device
        # sub-batches are whole policy groups (2R envs per direction for perturbed policies)
        unit = self.R * (2 if base_policy is not None else 1)
        self.subs, self.lens = plan_chunks(self.B, unit, n_sub, self.H, chunk)
        f64 = dict(dtype=torch.float64, device=self.device)
        self.returns = torch.zeros(self.B, **f64)
        self.state = torch.empty(self.B, obs_dim(n), **f64)
        self.want_final = want_final
        self.stats_pivot = stats_pivot
        self.stats_partial, self._rows = None, None
        if stats_pivot is not None:
            blocks = [(hi - lo + 63) // 64 for lo, hi in self.subs]  # kRolloutBlock
            self._rows, r = [], 0
            for _ in self.lens:
                row = []
                for b in blocks:
                    row.append((r, r + b))
                    r += b
                self._rows.append(row)
            self.stats_partial = torch.zeros(r, 2, obs_dim(n), **f64)
        self.streams = [torch.cuda.Stream(device=self.device) for _ in self.subs]
        self.launches = len(self.subs) * len(self.lens)

    def run(self, dir0=0, **overrides):
        """Enqueues all launches (current stream forks into the sub-batch streams and joins again) and
        returns a RolloutResult with returns[B], final_state[B, 2n+2], stats_partial / samples."""
        kw = dict(self.kw)
        kw.update(overrides)
        init_perturb = kw.pop("init_perturb", 0.0)
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(cur)
        unit = self.R * (2 if self.base_policy is not None else 1)
        for c, L in enumerate(self.lens):
            for i, ((lo, hi), st) in enumerate(zip(self.subs, self.streams)):
                out = {"returns": self.returns[lo:hi], "final_state": self.state[lo:hi]}
                if self.stats_partial is not None:
                    r0, r1 = self._rows[c][i]
                    out["stats_partial"] = self.stats_partial[r0:r1]
                src = {}
                if self.actions is not None:
                    src["actions"] = self.actions[lo:hi]
                elif self.base_policy is not None:
                    src.update(base_policy=self.base_policy, B=hi - lo, dir0=dir0 + lo // unit)
                    if kw.get("deltas") is not None:
                        src["deltas"] = kw["deltas"][lo // unit:hi // unit]
                    if kw.get("dir_mask") is not None:
                        src["dir_mask"] = kw["dir_mask"][lo // unit:hi // unit]
                else:
                    src["policies"] = self.policies.reshape(self.B // self.R, -1)[lo // self.R:hi // self.R]
                call = {k: v for k, v in kw.items() if k not in ("deltas", "dir_mask")}
                with torch.cuda.stream(st):
                    rollout(self.params, L, variant=self.variant, rollouts_per_policy=self.R,
                            init_state=None if c == 0 else self.state[lo:hi],
                            init_perturb=init_perturb if c == 0 else 0.0, want_final=True,
                            stats_pivot=self.stats_pivot, accumulate_returns=c > 0, out=out,
                            kernel=_lib.KERNEL_THREAD, schedule="plain", **src, **call)
        for st in self.streams:
            cur.wait_stream(st)
        res = RolloutResult()
        res.returns, res.final_state = self.returns, self.state
        res.stats_partial = self.stats_partial
        if self.stats_partial is not None:
            res.stats_blocks = self.stats_partial.shape[0]
            res.samples = float(self.B) * float(self.H)
        return res


def _counter_ptr(t):
    """Device iteration counter: one int32 CUDA element (read as uint32 by the kernels)."""
    if t is None:
        return None
    if not (t.is_cuda and t.dtype == torch.int32 and t.numel() == 1):
        raise ValueError("iteration_dev must be a CUDA int32 tensor with one element")
    return t.data_ptr()


def _philox(seed, iteration, dir0, dist, iteration_dev=None):
    p = _lib.SwmPhilox()
    p.seed, p.iteration, p.dir0, p.dist = int(seed) & (2 ** 64 - 1), int(iteration), int(dir0), int(dist)
    p.iteration_dev = _counter_ptr(iteration_dev)
    return p


def counter_add(counter, inc=1):
    """counter[0] += inc on the current stream (the device iteration counter of a captured graph)."""
    with torch.cuda.device(counter.device):
        _lib.check(_lib.lib().swm_counter_add(_counter_ptr(counter), int(inc), _lib.stream_ptr()))
    return counter


def record_nanmean(x, curve, index=None):
    """curve[min(index[0], len-1)] = mean of the non-NaN entries of x (learning-curve entry)."""
    x = _lib.f64(x).contiguous()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().swm_record_nanmean(_lib.ptr(x), x.numel(), _lib.ptr(curve),
                                                 _counter_ptr(index), curve.numel(), _lib.stream_ptr()))
    return curve


def philox_deltas(seed, iteration, dir0, count, wsize, dist=DELTA_PM1, device="cuda", iteration_dev=None):
    """delta_k for k = dir0..dir0+count-1 as [count, wsize] -- what the kernels regenerate."""
    _lib.require_cuda()
    out = torch.empty(count, wsize, dtype=torch.float64, device=device)
    ph = _philox(seed, iteration, dir0, dist, iteration_dev)
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().swm_philox_deltas(ctypes.byref(ph), count, wsize, _lib.ptr(out),
                                                _lib.stream_ptr()))
    return out


def ars_topb(returns, mask=None, out=None):
    """returns[2N] -> order[N] int32 (sort_directions; ties: higher index first, NaN first)."""
    _lib.require_cuda()
    returns = _lib.f64(returns).contiguous()
    N = returns.numel() // 2
    order = torch.empty(N, dtype=torch.int32, device=returns.device) if out is None else out
    with torch.cuda.device(returns.device):
        _lib.check(_lib.lib().swm_ars_topb(_lib.ptr(returns), _lib.ptr(mask), N, _lib.ptr(order),
                                           _lib.stream_ptr()))
    return order


def update_args(semantics, N, b):
    """(use_order, n_order, divisor, ddof) of the three reference update rules (SURVEY app. C)."""
    if semantics == ARS_AGENT:   # ars/ars_agent.py:110-130: every sorted direction, divisor b
        return True, N, float(b), 0
    if semantics == ARS_TOPB:    # safe_ars/ars.py:96 + :48-65: order[:b], divisor len(order)
        return True, min(b, N), 0.0, 0
    if semantics == ARS_RLGLUE:  # rlglue/agent/SwimmerAgent.py:223-241: first b, sample std
        return False, min(b, N), float(b), 1
    raise ValueError("unknown ARS semantics %r" % (semantics,))


def ars_update(W, returns, N, *, order=None, n_order=None, divisor=0.0, ddof=0, alpha=1.0, seed=0,
               iteration=0, iteration_dev=None, dir0=0, delta_dist=DELTA_PM1, deltas=None, mask=None,
               sigma_out=None):
    """In-place W += alpha * sum_{k in order[:n_order]} (r+ - r-) delta_k / (divisor * sigma_R)."""
    _lib.require_cuda()
    assert W.is_contiguous() and W.dtype == torch.float64
    ph = _philox(seed, iteration, dir0, delta_dist, iteration_dev)
    if deltas is not None:
        deltas = _lib.f64(deltas).contiguous().reshape(N, W.numel())
    n_order = N if n_order is None else int(n_order)
    with torch.cuda.device(W.device):
        _lib.check(_lib.lib().swm_ars_update(_lib.ptr(W), W.numel(), _lib.ptr(returns), N,
                                             _lib.ptr(order), n_order, _lib.ptr(mask),
                                             float(divisor), int(ddof), float(alpha),
                                             ctypes.byref(ph), _lib.ptr(deltas), _lib.ptr(sigma_out),
                                             _lib.stream_ptr()))
    return W


def screen_mask(sim_returns, threshold, mask_out=None, n_pass_out=None, n_pass_total=None):
    """mask[k] = r_sim+_k > threshold and r_sim-_k > threshold (ars_agent.py:150-157).  n_pass_total: optional
    int64 device tensor accumulating the number of survivors over calls.  A 2-D sim_returns [M, 2N] holds the
    returns under M models (swm_screen_mask_models): a direction passes only if it passes under every model."""
    dev = sim_returns.device
    M = sim_returns.shape[0] if sim_returns.dim() == 2 else None
    N = sim_returns.numel() // 2 if M is None else sim_returns.shape[1] // 2
    mask = torch.empty(N, dtype=torch.int32, device=dev) if mask_out is None else mask_out
    n_pass = torch.empty(1, dtype=torch.int32, device=dev) if n_pass_out is None else n_pass_out
    with torch.cuda.device(dev):
        if M is None:
            _lib.check(_lib.lib().swm_screen_mask(_lib.ptr(sim_returns), N, float(threshold),
                                                  _lib.ptr(mask), _lib.ptr(n_pass), _lib.ptr(n_pass_total),
                                                  _lib.stream_ptr()))
        else:
            _lib.check(_lib.lib().swm_screen_mask_models(_lib.ptr(sim_returns), M, N, float(threshold),
                                                         _lib.ptr(mask), _lib.ptr(n_pass), _lib.ptr(n_pass_total),
                                                         _lib.stream_ptr()))
    return mask, n_pass


def policy_actions(params, obs, policies, rollouts_per_policy=1, mean=None, inv_sigma=None,
                   clip=False):
    """Batched select_action (ars/environment.py:19-35): -> actions[B, n-1]."""
    _lib.require_cuda()
    n = params.n
    B = obs.shape[0]
    obs = _lib.f64(obs, (B, obs_dim(n))).contiguous()
    policies = _lib.f64(policies).contiguous().reshape(-1, policy_size(n))
    assert policies.shape[0] * rollouts_per_policy == B
    out = torch.empty(B, act_dim(n), dtype=torch.float64, device=obs.device)
    with torch.cuda.device(obs.device):
        _lib.check(_lib.lib().swm_policy_actions(ctypes.byref(params), _lib.ptr(obs),
                                                 _lib.ptr(policies), rollouts_per_policy,
                                                 _lib.ptr(mean), _lib.ptr(inv_sigma), int(clip),
                                                 _lib.ptr(out), B, _lib.stream_ptr()))
    return out


def stats_finalize(partial, samples, pivot, out=None, units=None):
    """Per-block moment sums [nb, 2, F] -> record [1 + 2F] = (count, mean, M2).
    count = samples (* units[0] if the device int32 `units` is given)."""
    nb, _, F = partial.shape
    rec = torch.empty(1 + 2 * F, dtype=torch.float64, device=partial.device) if out is None else out
    with torch.cuda.device(partial.device):
        _lib.check(_lib.lib().swm_stats_finalize(_lib.ptr(partial), nb, F, float(samples),
                                                 _lib.ptr(units), _lib.ptr(pivot), _lib.ptr(rec),
                                                 _lib.stream_ptr()))
    return rec


def stats_merge(running, records, mean_out=None, inv_sigma_out=None):
    """running <- merge(running, records[0], ..) in index order; optional mean / inv_sigma."""
    F = (running.numel() - 1) // 2
    records = records.reshape(-1, 1 + 2 * F)
    with torch.cuda.device(running.device):
        _lib.check(_lib.lib().swm_stats_merge(_lib.ptr(running), _lib.ptr(records), records.shape[0],
                                              F, _lib.ptr(mean_out), _lib.ptr(inv_sigma_out),
                                              _lib.stream_ptr()))
    return running


def pack_exchange(handle, *, returns_local=None, n_local, R=1, mask_local=None, stats_partial=None, samples=0.0,
                  units=None, pivot=None, n_features=0, returns_all=None, mask_all=None, records=None,
                  record_out=None, gathered_in=None, gathered_world=0):
    """One launch of swm_ars_pack_exchange (include/swimmer_ars.h): packs this rank's record from the rollout
    outputs, exchanges it over NVLink peer memory when `handle` (swm_exchange_t*) spans several ranks, and
    unpacks returns_all / mask_all / records.  handle None + gathered_in: unpack a collective's result;
    handle None + record_out + gathered_world > 1: pack only."""
    p = _lib.SwmPack()
    ref = returns_all if returns_all is not None else record_out
    p.returns_local, p.n_local, p.rollouts_per_policy = _lib.ptr(returns_local), int(n_local), int(R)
    p.mask_local = _lib.ptr(mask_local)
    if stats_partial is not None:
        p.stats_partial, p.n_blocks = _lib.ptr(stats_partial), stats_partial.shape[0]
    p.n_features, p.gathered_world, p.samples = int(n_features), int(gathered_world), float(samples)
    p.units, p.pivot = _lib.ptr(units), _lib.ptr(pivot)
    p.returns_all, p.mask_all, p.records = _lib.ptr(returns_all), _lib.ptr(mask_all), _lib.ptr(records)
    p.record_out, p.gathered_in = _lib.ptr(record_out), _lib.ptr(gathered_in)
    with torch.cuda.device(ref.device):
        _lib.check(_lib.lib().swm_ars_pack_exchange(handle, ctypes.byref(p), _lib.stream_ptr()))


def reduce_returns(returns, R, out=None):
    G = returns.numel() // R
    o = torch.empty(G, dtype=torch.float64, device=returns.device) if out is None else out
    with torch.cuda.device(returns.device):
        _lib.check(_lib.lib().swm_reduce_returns(_lib.ptr(returns), G, R, _lib.ptr(o),
                                                 _lib.stream_ptr()))
    return o


class EstimateData:
    """Recorded data of the simulator-model estimation objective, resident on the device: trajectories[K, H, 2n+2]
    recorded under policies[K, n-1, 2n+2], the unknowns (names of the EnvParam fields x replaces, any subset of
    m_i, l_i, k in any order) and the scratch of the objective's fixed-order sum for up to `max_candidates`
    candidates (swm_estimate_data_t)."""

    def __init__(self, trajectories, policies, unknowns=("m_i", "l_i", "k"), max_candidates=_lib.MAX_CANDIDATES):
        self.trajectories = _lib.f64(trajectories).contiguous()
        K, H, no = self.trajectories.shape
        self.n = (no - 2) // 2
        self.policies = _lib.f64(policies).contiguous().reshape(K, policy_size(self.n))
        if not 1 <= len(unknowns) <= 3 or len(set(unknowns)) != len(unknowns):
            raise ValueError("unknowns must be 1 to 3 distinct names of m_i, l_i, k, got %r" % (unknowns,))
        self.unknowns = tuple(unknowns)
        self.max_candidates = int(max_candidates)
        nws = _lib.lib().swm_prediction_error_workspace_doubles(K, H, self.max_candidates)
        if nws <= 0:
            raise ValueError("need K >= 1 trajectories of H >= 2 observations and max_candidates >= 1")
        self.workspace = torch.empty(nws, dtype=torch.float64, device=self.trajectories.device)
        c = _lib.SwmEstimateData()
        c.trajectories, c.policies = self.trajectories.data_ptr(), self.policies.data_ptr()
        c.K, c.H, c.d = K, H, len(self.unknowns)
        for i, name in enumerate(self.unknowns):
            c.fields[i] = _lib.FIELDS[name]
        c.workspace = self.workspace.data_ptr()
        self.c = c

    @property
    def d(self):
        return len(self.unknowns)


def _est_tensors(device, *checks):
    """Host-side checks of the tensors an estimation kernel reads or writes, before anything is enqueued.  checks:
    (name, tensor, shape) with shape a tuple, or an int for "at least that many elements".  First the format of
    each (float64, shape, contiguous), then that each is a CUDA tensor, on `device` if given."""
    for name, t, shape in checks:
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float64:
            raise ValueError("%s must be a float64 tensor, got %s" % (name, getattr(t, "dtype", type(t).__name__)))
        if isinstance(shape, int):
            if t.numel() < shape:
                raise ValueError("%s must hold at least %d doubles, got %d" % (name, shape, t.numel()))
        elif tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
        if not t.is_contiguous():
            raise ValueError("%s must be contiguous" % name)
    for name, t, _ in checks:
        if not t.is_cuda:
            raise ValueError("%s must be a CUDA tensor, got one on %s" % (name, t.device))
        if device is not None and t.device != device:
            raise ValueError("%s must be on %s, got %s" % (name, device, t.device))


def _est_model(base_params, data):
    """The objective indexes the recorded data with the strides of base_params.n: they must agree."""
    if base_params.n != data.n:
        raise ValueError("the base model has n=%d segments, the recorded data n=%d" % (base_params.n, data.n))


def prediction_error(base_params, data, candidates, out=None):
    """err[M] = sum_k sum_t || step_x(s_kt, W_k s_kt) - s_k,t+1 || for candidates[M, d] (Estimator.I of a whole
    population in one launch; +inf for m_i or l_i not positive and finite and for non-finite sums).
    `data`: EstimateData for base_params.n segments."""
    _est_model(base_params, data)
    candidates = _lib.f64(candidates).contiguous()
    M = candidates.shape[0]
    if tuple(candidates.shape) != (M, data.d) or M > data.max_candidates:
        raise ValueError("candidates must be [M <= %d, %d]" % (data.max_candidates, data.d))
    checks = [("candidates", candidates, (M, data.d))] + ([("out", out, (M,))] if out is not None else [])
    _est_tensors(data.trajectories.device, *checks)
    _lib.require_cuda()
    err = torch.empty(M, dtype=torch.float64, device=candidates.device) if out is None else out
    with torch.cuda.device(candidates.device):
        _lib.check(_lib.lib().swm_prediction_error(ctypes.byref(base_params), ctypes.byref(data.c),
                                                   _lib.ptr(candidates), M, _lib.ptr(err), _lib.stream_ptr()))
    return err


def cmaes_default_popsize(d):
    """lambda = 4 + floor(3 ln d) (Hansen's tutorial, the cma package's default)."""
    return 4 + int(math.floor(3.0 * math.log(d)))


def cmaes_state_doubles(d, popsize):
    n = _lib.lib().swm_cmaes_state_doubles(int(d), int(popsize))
    if n <= 0:
        raise ValueError("CMA-ES needs 1 <= d <= 3 and %d <= popsize <= %d" % (_lib.CMAES_MIN_POPSIZE,
                                                                             _lib.MAX_CANDIDATES))
    return n


def cmaes_view(state, d, popsize):
    """Named views into a CMA-ES state buffer (layout of include/swimmer_ars.h)."""
    L = 10 + -(-30 * d // popsize)
    o = 7
    v = {"generation": state[0], "status": state[1], "sigma": state[2], "best_f": state[3],
         "max_generations": state[4], "tolfun": state[5], "tolx": state[6]}
    for name, size, shape in (("mean", d, (d,)), ("best_x", d, (d,)), ("p_sigma", d, (d,)), ("p_c", d, (d,)),
                              ("D", d, (d,)), ("C", d * d, (d, d)), ("B", d * d, (d, d)), ("history", L, (L,)),
                              ("z", popsize * d, (popsize, d))):
        v[name] = state[o:o + size].view(shape)
        o += size
    return v


def cmaes_init(state, x0, popsize, sigma0=1.0, tolfun=1e-11, tolx=1e-11, max_generations=0):
    """Fresh CMA-ES state around x0 (host sequence of d floats); max_generations <= 0: the cma default."""
    d = len(x0)
    _est_tensors(None, ("state", state, cmaes_state_doubles(d, popsize)))
    x = (ctypes.c_double * d)(*[float(v) for v in x0])
    with torch.cuda.device(state.device):
        _lib.check(_lib.lib().swm_cmaes_init(_lib.ptr(state), d, int(popsize), x, float(sigma0), float(tolfun),
                                             float(tolx), int(max_generations), _lib.stream_ptr()))
    return state


def cmaes_sample(state, d, popsize, seed, candidates):
    """candidates[popsize, d] = mean + sigma B D z of the current generation (z is kept in the state)."""
    _est_tensors(state.device, ("state", state, cmaes_state_doubles(d, popsize)),
                 ("candidates", candidates, (popsize, d)))
    with torch.cuda.device(state.device):
        _lib.check(_lib.lib().swm_cmaes_sample(_lib.ptr(state), int(d), int(popsize), int(seed) & (2 ** 64 - 1),
                                               _lib.ptr(candidates), _lib.stream_ptr()))
    return candidates


def cmaes_update(state, d, popsize, candidates, fitness):
    """One CMA-ES update from the sampled candidates and their fitness[popsize]."""
    _est_tensors(state.device, ("state", state, cmaes_state_doubles(d, popsize)),
                 ("candidates", candidates, (popsize, d)), ("fitness", fitness, (popsize,)))
    with torch.cuda.device(state.device):
        _lib.check(_lib.lib().swm_cmaes_update(_lib.ptr(state), int(d), int(popsize), _lib.ptr(candidates),
                                               _lib.ptr(fitness), _lib.stream_ptr()))
    return state


def cmaes_generation(state, popsize, seed, base_params, data, candidates, fitness):
    """sample + prediction_error + update of one generation, enqueued without a host round trip (capturable).
    The objective runs for M = popsize candidates in data's workspace: data.max_candidates must cover it."""
    _est_model(base_params, data)
    if int(popsize) > data.max_candidates:
        raise ValueError("popsize %d exceeds the %d candidates data's workspace holds" % (popsize, data.max_candidates))
    _est_tensors(data.trajectories.device, ("state", state, cmaes_state_doubles(data.d, popsize)),
                 ("candidates", candidates, (popsize, data.d)), ("fitness", fitness, (popsize,)))
    with torch.cuda.device(state.device):
        _lib.check(_lib.lib().swm_cmaes_generation(_lib.ptr(state), data.d, int(popsize), int(seed) & (2 ** 64 - 1),
                                                   ctypes.byref(base_params), ctypes.byref(data.c),
                                                   _lib.ptr(candidates), _lib.ptr(fitness), _lib.stream_ptr()))
    return state


def fp64_probe(blocks, threads, iters, sink):
    flops = ctypes.c_double(0.0)
    with torch.cuda.device(sink.device):
        _lib.check(_lib.lib().swm_fp64_probe(blocks, threads, iters, _lib.ptr(sink),
                                             ctypes.byref(flops), _lib.stream_ptr()))
    return flops.value
