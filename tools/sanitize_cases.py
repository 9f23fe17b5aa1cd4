"""Small invocations of every kernel family (all policy-storage modes, V2 moments in registers and in
shared memory, screening, trajectories, ragged last block, ARS epilogue, every rollout kernel: per-thread,
lane-split, lane-split with operator warp; the RL-Glue protocol kernel; the estimation objective at n = 2, 8, 10
and CMA-ES at lambda = 2, 33, 1024) for
`compute-sanitizer --tool memcheck|racecheck|synccheck python tools/sanitize_cases.py [n ...]`."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import swimmer_ars_b200 as S


def main(ns=(2, 3, 4, 5, 6, 7, 8, 9, 10)):
    rng = np.random.default_rng(0)
    H = 70  # crosses the step-63 re-evaluation
    for n in ns:
        p = S.make_params(n=n)
        no, na, ws = 2 * n + 2, n - 1, (n - 1) * (2 * n + 2)
        B = 70  # ragged second block
        ac = torch.as_tensor(rng.uniform(-5, 5, (B, na))).cuda()
        st = torch.as_tensor(rng.normal(size=(B, no))).cuda()
        for variant in (S.GYM, S.RLGLUE):
            S.ops.step_batched(p, st, ac, variant)
            S.ops.accelerations_batched(p, st, ac, variant)
            S.ops.rollout(p, H, variant=variant, actions=ac, want_final=True, want_trajectory=True)
        W = torch.as_tensor(rng.uniform(-1, 1, ws) * 0.1).cuda()
        mean = torch.zeros(no, dtype=torch.float64, device="cuda")
        inv = torch.ones_like(mean)
        piv = S.ops.reset_state(n)
        for R, Bp in ((1, 70), (3, 2 * 7 * 3), (32, 2 * 2 * 32), (64, 2 * 1 * 64)):
            r = S.ops.rollout(p, H, B=Bp, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=R,
                              init_perturb=1e-2 if R > 1 else 0.0, mean=mean, inv_sigma=inv, stats_pivot=piv)
            rec = S.ops.stats_finalize(r.stats_partial, r.samples, piv)
            assert bool(torch.isfinite(r.returns).all()) and bool(torch.isfinite(rec).all())
            assert float(rec[0]) == Bp * H
            S.ops.rollout(p, H, B=Bp, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=R, want_final=True)
            S.ops.rollout(p, H, B=Bp, variant=S.RLGLUE, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=R,
                          clip_actions=True, delta_dist=S.DELTA_01)
        # the three rollout kernels forced (AUTO picks by batch size): fixed actions, V1, V2 + moments, trajectories
        for kern in (S._lib.KERNEL_THREAD, S._lib.KERNEL_LANES, S._lib.KERNEL_LANES2, S._lib.KERNEL_LANES3):
            S.ops.rollout(p, H, actions=ac, want_final=True, want_trajectory=True, kernel=kern)
            S.ops.rollout(p, H, B=2 * 9, base_policy=W, nu=0.05, seed=3, want_final=True, kernel=kern)
            r = S.ops.rollout(p, H, B=2 * 5 * 3, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=3, init_perturb=1e-2,
                              mean=mean, inv_sigma=inv, stats_pivot=piv, kernel=kern, schedule="plain")
            assert bool(torch.isfinite(r.returns).all())
        ex = S.RlglueArsExperiment(n_seg=n, N=2, b=1, H=9, protocol="reference", replicas=3)
        assert np.isfinite(ex.run_training(2)).all()
        sim = S.make_params(n=n, l_i=1.01, m_i=0.99, k=10.1)
        S.ops.rollout(p, H, B=70, base_policy=W, nu=0.05, seed=3,
                      screen=dict(sim_params=sim, sim_thresh=0.5, real_thresh=0.6), want_trajectory=True)
        eng = S.ArsEngine(p, N=6, b=4, alpha=0.02, nu=0.05, H=H, v2=True, semantics=S.ARS_TOPB, seed=1,
                          distributed=False, sim_params=sim, sim_threshold=-1.0, curve_capacity=4)
        eng.run_iteration()
        eng.run_iteration()
        if n in (2, 8, 10):
            estimation(n, rng)
        torch.cuda.synchronize()
        print("n=%d ok" % n, flush=True)
    print("sanitize cases done")


def estimation(n, rng):
    """The prediction-error objective at a ragged transition count (T = 3 * 43 = 129: a second CTA with one
    transition, CTAs across trajectory boundaries) and M = 129 (a second block of the reduce grid), then CMA-ES
    generations at lambda = 2, 33 and 1024 (one, two and 32 warps of ranking; 1, 1 and 8 sampling blocks)."""
    no, K, H = 2 * n + 2, 3, 44
    trajs = torch.as_tensor(rng.normal(size=(K, H, no)) * 0.5).cuda()
    pols = torch.as_tensor(rng.uniform(-0.3, 0.3, (K, n - 1, no))).cuda()
    base = S.make_params(n=n)
    cand = torch.as_tensor(np.array([1.0, 1.0, 10.0]) * rng.uniform(0.9, 1.1, (129, 3))).cuda()
    data = S.ops.EstimateData(trajs, pols, ("m_i", "l_i", "k"), max_candidates=1024)
    assert bool(torch.isfinite(S.ops.prediction_error(base, data, cand)).all())
    for lam in (2, 33, 1024):
        state = torch.empty(S.ops.cmaes_state_doubles(3, lam), dtype=torch.float64, device="cuda")
        S.ops.cmaes_init(state, [1.0, 1.0, 10.0], lam, sigma0=0.05)
        x = torch.empty(lam, 3, dtype=torch.float64, device="cuda")
        f = torch.empty(lam, dtype=torch.float64, device="cuda")
        S.ops.cmaes_sample(state, 3, lam, 1, x)
        S.ops.prediction_error(base, data, x, out=f)
        S.ops.cmaes_update(state, 3, lam, x, f)
        for _ in range(2):
            S.ops.cmaes_generation(state, lam, 1, base, data, x, f)


if __name__ == "__main__":
    main(tuple(int(a) for a in sys.argv[1:]) or (2, 3, 4, 5, 6, 7, 8, 9, 10))
