"""Device-resident ARS iteration: the batched replacement of the sequential loop in
ARSAgent.runOneIteration (ars/ars_agent.py:132-185) and Basic_ARS.train (safe_ars/ars.py:82-97).

One iteration =
  1. [reward-constraint safe mode] 2N simulator rollouts -> screening mask        (swm_rollout, swm_screen_mask)
     (an ensemble of M simulator models: M x 2N rollouts in one launch, a direction survives only if it
     clears the threshold under every model                                        (swm_rollout_models, swm_screen_mask_models))
  2. 2N (x R) real rollouts, all in one fused kernel launch                        (swm_rollout)
     (V1 safe mode: 1 and 2 run side by side on two streams, the mask is applied to the returns in step 3 --
     `speculate`; otherwise 2 rolls out the survivors of 1 only)
  3. ONE launch that packs this rank's record (per-direction mean returns, screening mask, V2 moment
     record), exchanges it with every other rank over NVLink peer memory and unpacks all ranks'
     records                                                                       (swm_ars_pack_exchange)
  4. redundantly on every rank, bit-identically: top-b ranking, delta-weighted
     update with deltas regenerated from Philox, Welford merge in rank order       (swm_ars_topb, swm_ars_update, swm_stats_merge)

Directions are sharded contiguously across ranks (rank r owns [r N/world, (r+1) N/world)); the
delta tensors never move.  Nothing in an iteration synchronises with the host.

The iteration number that keys Philox lives in device memory (`iter_dev`, advanced by
swm_counter_add at the end of the update), so the whole iteration is a fixed sequence of launches
with fixed arguments: `use_graph=True` captures it once into a CUDA graph and replays it (one
launch per iteration instead of 5-7).  Sharded engines are captured too: their exchange is a kernel
(distributed.RecordExchange, transport "p2p"), not a collective; only the collective fallback
(no peer access between the GPUs) enqueues eagerly.
"""
import torch
import torch.distributed as dist

from . import _lib, ops
from ._lib import ARS_AGENT, DELTA_PM1, GYM
from .distributed import RecordExchange, RecordLayout


class ArsEngine:
    def __init__(self, params, *, N, b, alpha, nu, H, v2=False, semantics=ARS_AGENT,
                 rollouts_per_direction=1, seed=0, variant=GYM, delta_dist=DELTA_PM1,
                 clip_actions=False, init_perturb=0.0, initial_policy=None, group=None,
                 distributed=None, device=None, sim_params=None, sim_threshold=None,
                 step_screen=None, use_graph=False, curve_capacity=0, rollout_chunks=None, transport="auto",
                 rollout_kernel=0, speculate=True, shard="auto"):
        _lib.require_cuda()
        self.params, self.N, self.b, self.alpha, self.nu, self.H = params, int(N), int(b), alpha, nu, int(H)
        self.v2, self.semantics, self.R = bool(v2), semantics, int(rollouts_per_direction)
        self.seed = 0 if seed is None else int(seed)
        self.variant, self.delta_dist, self.clip = variant, delta_dist, clip_actions
        self.init_perturb = float(init_perturb)
        self.device = torch.device(device) if device is not None else torch.device(
            "cuda", torch.cuda.current_device())
        self.group = group
        use_dist = dist.is_available() and dist.is_initialized() if distributed is None else distributed
        # shard="auto": a problem whose WHOLE batch already runs on the latency-optimised kernels (two / three warps
        # per lane group, every warp alone on an SM sub-partition) does not get faster on fewer environments per GPU
        # -- the rollout is one dependent chain of H steps either way -- and sharding it only adds the exchange.
        # Such engines run replicated: every rank computes all N directions, bit-identically, with no exchange.
        # shard=True always shards over the process group.
        self.replicated, self.shard_replicas = False, 1
        if use_dist and shard == "auto" and dist.get_world_size(group) > 1:
            with torch.cuda.device(self.device):
                whole = ops.rollout_kernel_choice(params, 2 * self.N * self.R, rollouts_per_policy=self.R,
                                                  kernel=int(rollout_kernel))
            if variant == GYM and not clip_actions and step_screen is None and whole in ("lanes2", "lanes3"):
                use_dist, self.replicated = False, True
            elif group is None and variant == GYM and not clip_actions and step_screen is None:
                # ... and it is sharded only as far as that helps: over the smallest number of ranks S whose share runs
                # on those kernels with at most one lane group per SM; the world/S blocks of S consecutive ranks then
                # each run the whole problem (config[2] on 8 GPUs: 2 blocks of 4, the exchange has 4 peers not 8)
                W = dist.get_world_size()
                S = self._useful_shards(params, W, rollout_kernel)
                if S < W:
                    me = dist.get_rank()
                    for blk in range(W // S):
                        g = dist.new_group(list(range(blk * S, (blk + 1) * S)))
                        if me // S == blk:
                            group = g
                    self.group, self.shard_replicas = group, W // S
        self.world = dist.get_world_size(group) if use_dist else 1
        self.rank = dist.get_rank(group) if use_dist else 0
        if self.N % self.world != 0:
            raise ValueError("N=%d directions do not shard over %d ranks" % (self.N, self.world))
        self.N_local = self.N // self.world
        self.dir0 = self.rank * self.N_local
        n = params.n
        self.no, self.ws = ops.obs_dim(n), ops.policy_size(n)
        f64 = dict(dtype=torch.float64, device=self.device)
        self.W = torch.zeros(self.ws, **f64)
        if initial_policy is not None:
            self.W.copy_(torch.as_tensor(initial_policy, dtype=torch.float64).reshape(-1))
        self.iteration = 0  # host mirror of iter_dev
        self.iter_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        # optional device-side learning curve: curve[j] = nanmean(returns of iteration j)
        self.curve = torch.full((int(curve_capacity),), float("nan"), **f64) if curve_capacity > 0 else None
        self.rollout_kernel = int(rollout_kernel)  # _lib.KERNEL_AUTO / KERNEL_THREAD / KERNEL_LANES
        self._graph = None
        self._warm = False
        # V2 running statistics: record = [count, mean[F], M2[F]]; mean=0 / sigma=1 until the first
        # update (ars_agent.py:87-90)
        self.stats = torch.zeros(1 + 2 * self.no, **f64)
        self.mean = torch.zeros(self.no, **f64)
        self.inv_sigma = torch.ones(self.no, **f64)
        self.pivot = ops.reset_state(n, variant, self.device)
        # reward-constraint screening through a simulator model (ars_agent.py:144-157), or through every model of a
        # list: a direction reaches the real world only if both its returns clear sim_threshold under each of them
        self.sim_params, self.sim_threshold = sim_params, sim_threshold
        n_sim = None
        if isinstance(sim_params, (list, tuple)):
            n_sim = len(sim_params)
            if not 1 <= n_sim <= _lib.MAX_SIM_MODELS or any(p.n != params.n for p in sim_params):
                raise ValueError("sim_params must be 1 to %d models with the real model's n=%d"
                                 % (_lib.MAX_SIM_MODELS, params.n))
            if variant != GYM or clip_actions:
                raise ValueError("screening by several simulator models needs gym dynamics without action clipping")
        # speculate: the real-world rollouts of ALL directions run beside the simulator rollouts that screen them
        # (second stream; both are small batches that leave most of the chip idle) and the screening mask is
        # applied to their returns afterwards (swm_ars_pack_exchange writes NaN for screened-out directions).
        # Results are bit-identical to screening first: a rollout never depends on the mask.  Only where nothing
        # else of a screened-out rollout is kept: not with V2 statistics, not when trajectories are requested.
        self.speculate = bool(speculate) and sim_params is not None and not self.v2
        self._side = torch.cuda.Stream(device=self.device) if self.speculate else None
        # per-step state-constraint screening (safe_ars/ars.py:124-153)
        self.step_screen = step_screen
        # persistent buffers: the iteration loop allocates nothing
        Bl = 2 * self.N_local * self.R
        self.B_local = Bl
        self._out = {"returns": torch.empty(Bl, **f64)}
        lead = () if n_sim is None else (n_sim,)  # model lists: one row per model
        self._sim_out = {"returns": torch.empty(lead + (Bl,), **f64)} if sim_params is not None else None
        self.returns = torch.zeros(2 * self.N, **f64)        # last iteration, all ranks
        self._records = torch.zeros(self.world, 1 + 2 * self.no, **f64)
        self.order = torch.zeros(self.N, dtype=torch.int32, device=self.device)
        self.sigma = torch.zeros(1, **f64)
        self.mask = None
        if sim_params is not None:
            self.mask_local = torch.ones(self.N_local, dtype=torch.int32, device=self.device)
            self.n_pass_local = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.n_pass_total = torch.zeros(1, dtype=torch.int64, device=self.device)  # survivors so far (this rank)
            self.mask = torch.ones(self.N, dtype=torch.int32, device=self.device)
            self.sim_returns = torch.zeros(lead + (2 * self.N_local,), **f64)
        self.last = None
        # per-iteration record exchange (one packed record per rank): peer-memory kernel or collective
        self.layout = RecordLayout(self.N_local, self.no if self.v2 else 0, has_mask=sim_params is not None)
        self.exchange = RecordExchange(self.layout, group=group, device=self.device, transport=transport,
                                       distributed=use_dist)
        # a captured NCCL all-gather next to eager collectives on the same communicator hung (round 1):
        # only the kernel transports are captured
        self.use_graph = bool(use_graph) and self.exchange.capturable
        # optional (n_sub, chunk): schedule the real rollouts as sub-batches x time-chunks on several streams
        # (ops.ChunkedRollout) -- pays off when 2 N R / world environments are a mid-size batch
        self._chunked = None
        if rollout_chunks is not None and step_screen is None:
            n_sub, chunk = rollout_chunks
            kw = dict(nu=self.nu, seed=self.seed, iteration=0, iteration_dev=self.iter_dev,
                      delta_dist=self.delta_dist, clip_actions=self.clip, init_perturb=self.init_perturb)
            if self.v2:
                kw.update(mean=self.mean, inv_sigma=self.inv_sigma)
            self._chunked = ops.ChunkedRollout(
                params, self.H, B=Bl, n_sub=n_sub, chunk=chunk, variant=self.variant, base_policy=self.W,
                rollouts_per_policy=self.R, stats_pivot=self.pivot if self.v2 else None, device=self.device, **kw)

    def _useful_shards(self, params, world, rollout_kernel):
        sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        per_warp = ops.lane_split_envs_per_warp(params.n)
        with torch.cuda.device(self.device):
            for cand in range(2, world):
                if world % cand or self.N % cand:
                    continue
                share = 2 * self.N * self.R // cand
                name = ops.rollout_kernel_choice(params, share, rollouts_per_policy=self.R, kernel=int(rollout_kernel))
                if name in ("lanes2", "lanes3") and (share + per_warp - 1) // per_warp <= sms:
                    return cand
        return world

    # -------------------------------------------------------------------------------------------
    def _rollouts(self, params, out, deltas_local, dir_mask, want_stats, want_trajectory, screen):
        if (self._chunked is not None and params is self.params and not want_trajectory and screen is None
                and want_stats == self.v2):
            return self._chunked.run(dir0=self.dir0, deltas=deltas_local, dir_mask=dir_mask)
        fn = ops.rollout_models if isinstance(params, (list, tuple)) else ops.rollout
        return fn(
            params, self.H, B=self.B_local, variant=self.variant, base_policy=self.W, nu=self.nu,
            deltas=deltas_local, dir_mask=dir_mask, init_perturb=self.init_perturb, seed=self.seed,
            iteration=0, iteration_dev=self.iter_dev, dir0=self.dir0, delta_dist=self.delta_dist,
            rollouts_per_policy=self.R, mean=self.mean if self.v2 else None,
            inv_sigma=self.inv_sigma if self.v2 else None, clip_actions=self.clip,
            stats_pivot=self.pivot if want_stats else None, want_trajectory=want_trajectory,
            screen=screen, out=out, kernel=self.rollout_kernel)

    def run_iteration(self, deltas=None, want_trajectory=False, update=True):
        """One ARS iteration.  `deltas` ([N, ws] device tensor): use these perturbations instead of
        Philox (replaying the reference's numpy draws).  Returns the device tensor of all 2N
        per-policy returns (NaN for screened-out directions); never synchronises."""
        plain = deltas is None and not want_trajectory and update
        if self.use_graph and plain:
            if not self._warm:
                # first iteration eagerly: sizes the scratch buffers and sets kernel attributes
                self._warm = True
            elif self._graph is None:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue(None, False, True)
                self._graph = g
            if self._graph is not None:
                self._graph.replay()
                self.iteration += 1
                return self.returns
        out = self._enqueue(deltas, want_trajectory, update)
        if update:
            self.iteration += 1
        return out

    def _enqueue(self, deltas, want_trajectory, update):
        Nl, R = self.N_local, self.R
        deltas_local = None if deltas is None else deltas.reshape(self.N, self.ws)[self.dir0:self.dir0 + Nl]
        dir_mask = None
        def screen():
            sim = self._rollouts(self.sim_params, self._sim_out, deltas_local, None, False, False, None)
            sim_ret = sim.returns if R == 1 else ops.reduce_returns(sim.returns, R, out=self.sim_returns)
            self.sim_returns = sim_ret
            ops.screen_mask(sim_ret, self.sim_threshold, self.mask_local, self.n_pass_local, self.n_pass_total)

        if self.sim_params is not None and self.speculate and not want_trajectory:
            main = torch.cuda.current_stream(self.device)
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):
                screen()
            res = self._rollouts(self.params, self._out, deltas_local, None, False, False, self.step_screen)
            main.wait_stream(self._side)
            dir_mask = self.mask_local
        else:
            if self.sim_params is not None:
                screen()
                dir_mask = self.mask_local
            res = self._rollouts(self.params, self._out, deltas_local, dir_mask, self.v2, want_trajectory,
                                 self.step_screen)
        self.last = res
        if res.stats_partial is not None and res.stats_partial is not getattr(self._chunked, "stats_partial", None):
            self._out["stats_partial"] = res.stats_partial  # reuse: iterations allocate nothing
        # statistics count: every state of every rolled-out environment; in safe mode only the directions
        # that survived screening were rolled out (device-side count)
        units = self.n_pass_local if (self.v2 and dir_mask is not None) else None
        samples = (float(2 * R * self.H) if units is not None else res.samples) if self.v2 else 0.0
        pack = dict(returns_local=res.returns, n_local=Nl, R=R, mask_local=dir_mask,
                    stats_partial=res.stats_partial if self.v2 else None, samples=samples, units=units,
                    pivot=self.pivot if self.v2 else None, n_features=self.layout.n_features)
        out = dict(returns_all=self.returns, mask_all=self.mask, records=self._records if self.v2 else None)
        ex = self.exchange
        if ex.transport in ("local", "p2p"):
            ops.pack_exchange(ex.handle, **pack, **out)           # one launch: pack, peer stores + flags, unpack
        else:
            # collective fallback: pack kernel, torch.distributed all-gather, torch unpack (eager only)
            ops.pack_exchange(None, **pack, record_out=ex.record, gathered_world=self.world)
            returns, mask, records = ex.gather_split(ex.record)
            self.returns.copy_(returns)
            if mask is not None:
                self.mask.copy_(mask)
            if records is not None:
                self._records.copy_(records)
        if update:
            self._enqueue_update(deltas)
        return self.returns

    def apply_update(self, deltas=None):
        """Ranking + update + statistics merge for the returns of the last `run_iteration(update=False)`."""
        self._enqueue_update(deltas)
        self.iteration += 1

    def _enqueue_update(self, deltas=None):
        use_order, n_order, divisor, ddof = ops.update_args(self.semantics, self.N, self.b)
        order = None
        if use_order:
            order = ops.ars_topb(self.returns, self.mask, out=self.order)
        ops.ars_update(self.W, self.returns, self.N, order=order, n_order=n_order, divisor=divisor,
                       ddof=ddof, alpha=self.alpha, seed=self.seed, iteration=0, iteration_dev=self.iter_dev, dir0=0,
                       delta_dist=self.delta_dist, deltas=deltas, mask=self.mask if use_order else None,
                       sigma_out=self.sigma)
        if self.v2:
            ops.stats_merge(self.stats, self._records, self.mean, self.inv_sigma)
        if self.curve is not None:
            ops.record_nanmean(self.returns, self.curve, self.iter_dev)
        ops.counter_add(self.iter_dev, 1)

    def check_exchange(self):
        """Raises if a peer failed to deliver its record in time (sticky device status); synchronises."""
        epoch, status = self.exchange.status()
        if status:
            raise _lib.SwimmerLibError("record exchange timed out waiting for rank %d (epoch %d)" % (status - 1, epoch))
        return epoch

    # ---- host views ----
    def policy_numpy(self):
        n = self.params.n
        return self.W.cpu().numpy().reshape(n - 1, 2 * n + 2).copy()

    def set_policy(self, W):
        self.W.copy_(torch.as_tensor(W, dtype=torch.float64).reshape(-1))

    def state_dict(self):
        """Everything needed to resume bit-exactly: policy, Philox position, V2 statistics."""
        sd = {"W": self.W.cpu().numpy(), "iteration": self.iteration, "seed": self.seed,
              "stats": self.stats.cpu().numpy(), "mean": self.mean.cpu().numpy(),
              "inv_sigma": self.inv_sigma.cpu().numpy()}
        if self.curve is not None:
            sd["curve"] = self.curve.cpu().numpy()
        return sd

    def load_state_dict(self, sd):
        self.W.copy_(torch.as_tensor(sd["W"]))
        if int(sd["seed"]) != self.seed:
            self._graph = None  # the seed is a frozen kernel argument of the captured graph ...
            if self._chunked is not None:
                self._chunked.kw["seed"] = int(sd["seed"])  # ... and of the chunked rollout schedule
        self.iteration, self.seed = int(sd["iteration"]), int(sd["seed"])
        if self.curve is not None and "curve" in sd:
            self.curve.copy_(torch.as_tensor(sd["curve"]))
        self.iter_dev.fill_(self.iteration)
        self.stats.copy_(torch.as_tensor(sd["stats"]))
        self.mean.copy_(torch.as_tensor(sd["mean"]))
        self.inv_sigma.copy_(torch.as_tensor(sd["inv_sigma"]))
