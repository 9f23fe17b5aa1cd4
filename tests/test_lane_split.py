"""Lane-split rollout kernel (csrc/lane_rollout.cuh: one environment over 4/8/16 lanes, lane = segment):
same parity bar as the one-thread-per-environment kernel -- H-step returns within 1e-6 relative of the
oracle (observed ~1e-12), visited states 1e-8, V2 moments 1e-9 -- plus its own size-independent
properties (determinism, batch-order invariance, chunk chaining)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import golden, rand_states, rel_err

pytestmark = pytest.mark.gpu
RET_TOL = 1e-6


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _ret_err(got, want):
    got, want = np.asarray(got), np.asarray(want)
    return float(np.max(np.abs(got - want) / np.maximum(1e-3, np.abs(want))))


LANE_KERNELS = ["LANES", "LANES2", "LANES3"]


def _k(S, name):
    return getattr(S, "KERNEL_" + name)


@pytest.mark.parametrize("kern", LANE_KERNELS)
@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 10])
def test_lane_fixed_action_rollout_matches_oracle(S, O, n, kern):
    rng = np.random.default_rng(n)
    B, H = 37, 300  # ragged: the last warp holds idle lane groups
    ps, po = S.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, direction=(.6, .8)), \
        O.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, direction=(.6, .8))
    ac = rng.uniform(-5, 5, (B, n - 1))
    init = rand_states(rng, n, B, scale=1.0)
    res = S.ops.rollout(ps, H, actions=_cuda(ac), init_state=_cuda(init), want_final=True, want_trajectory=True,
                        kernel=_k(S, kern))
    traj = res.trajectory.cpu().numpy()
    got_r, got_f = res.returns.cpu().numpy(), res.final_state.cpu().numpy()
    for e in range(B):
        want_r, want_f, want_t = O.rollout(po, O.GYM, H, action=ac[e], init_state=init[e], want_traj=True)
        assert abs(got_r[e] - want_r) < RET_TOL * max(1e-3, abs(want_r))
        assert rel_err(got_f[e], want_f) < 1e-8
        assert rel_err(traj[:, e, :], want_t) < 1e-8
    # reset start (no init_state) and the thread kernel agree too
    r0 = S.ops.rollout(ps, H, actions=_cuda(ac), want_final=True, kernel=_k(S, kern))
    r1 = S.ops.rollout(ps, H, actions=_cuda(ac), want_final=True, kernel=S.KERNEL_THREAD)
    assert rel_err(r0.final_state.cpu().numpy(), r1.final_state.cpu().numpy()) < 1e-10
    np.testing.assert_allclose(r0.returns.cpu().numpy(), r1.returns.cpu().numpy(), rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("kern", ["LANES2", "LANES3"])
@pytest.mark.parametrize("n", [3, 5, 7])
def test_lane_per_step_screening_matches_thread_kernel(S, n, kern):
    """Safe_ARS per-step screening (safe_ars/ars.py:124-153) in the warp-specialised kernels: the simulator's
    accelerations are a second right-hand side on the same solution rows.  Against the one-thread-per-environment
    kernel: the step an environment freezes at and its violation count are identical, returns / final states /
    trajectories (frozen tail repeated) agree to rounding; thresholds are set so that some environments freeze
    early, some late and some never."""
    B, H = 40, 200
    rng = np.random.default_rng(10 * n)
    real = S.make_params(n=n, l_i=.9, m_i=1.1, k=9.5)
    sim = S.make_params(n=n, l_i=.93, m_i=1.05, k=9.9)
    W = _cuda(rng.uniform(-1, 1, (B, (n - 1) * (2 * n + 2))) * 1.5)
    init = _cuda(rand_states(rng, n, B, scale=0.3))
    probe = S.ops.rollout(real, H, policies=W, init_state=init, want_trajectory=True, kernel=S.KERNEL_THREAD)
    peak = probe.trajectory[:, :, 3::2].abs().amax(dim=(0, 2)).cpu().numpy()      # max |thd| per environment
    thr = float(np.median(peak)) * 0.6
    kw = dict(policies=W, init_state=init, want_final=True, want_trajectory=True,
              screen=dict(sim_params=sim, sim_thresh=thr, real_thresh=0.9 * thr))
    a, b = S.ops.rollout(real, H, kernel=_k(S, kern), **kw), S.ops.rollout(real, H, kernel=S.KERNEL_THREAD, **kw)
    fa, fb = a.frozen_at.cpu().numpy(), b.frozen_at.cpu().numpy()
    assert np.array_equal(fa, fb) and np.array_equal(a.violations.cpu().numpy(), b.violations.cpu().numpy())
    assert (fb < H).sum() >= 5 and (fb == H).sum() >= 5 and len(set(fb.tolist())) >= 5
    np.testing.assert_allclose(a.returns.cpu().numpy(), b.returns.cpu().numpy(), rtol=1e-9, atol=1e-12)
    assert rel_err(a.final_state.cpu().numpy(), b.final_state.cpu().numpy()) < 1e-9
    assert rel_err(a.trajectory.cpu().numpy(), b.trajectory.cpu().numpy()) < 1e-9
    # a NaN state is unsafe at once (np.max semantics of the cost), its neighbours in the warp are untouched
    init2 = init.clone()
    init2[3, 3] = float("nan")
    c = S.ops.rollout(real, H, kernel=_k(S, kern), **dict(kw, init_state=init2))
    fc = c.frozen_at.cpu().numpy()
    assert fc[3] == 0 and np.array_equal(np.delete(fc, 3), np.delete(fa, 3))
    keep = np.arange(B) != 3
    assert torch.equal(c.returns[torch.as_tensor(keep)], a.returns[torch.as_tensor(keep)])


@pytest.mark.parametrize("kern", LANE_KERNELS)
@pytest.mark.parametrize("H", [1, 2, 3, 63, 64, 65, 129])
def test_lane_short_and_odd_horizons(S, kern, H):
    """Horizons around the unroll-by-two of the step loop, the alternate-step hand-over of the operator warps and the
    re-evaluation of the sines/cosines at step 63: every lane-split kernel follows the one-thread-per-environment
    kernel (V2 policies + moments, and fixed actions)."""
    n, B = 5, 22
    p = S.make_params(n=n, l_i=.9, m_i=1.1, k=9.5)
    rng = np.random.default_rng(H)
    W = _cuda(rng.uniform(-1, 1, (n - 1) * (2 * n + 2)) * 0.2)
    mean, inv = _cuda(rng.normal(size=2 * n + 2) * 0.1), _cuda(rng.uniform(0.5, 2.0, 2 * n + 2))
    piv = S.ops.reset_state(n)
    kw = dict(B=B, base_policy=W, nu=0.05, seed=H, mean=mean, inv_sigma=inv, stats_pivot=piv, want_final=True)
    a, b = S.ops.rollout(p, H, kernel=_k(S, kern), **kw), S.ops.rollout(p, H, kernel=S.KERNEL_THREAD, **kw)
    np.testing.assert_allclose(a.returns.cpu().numpy(), b.returns.cpu().numpy(), rtol=1e-9, atol=1e-13)
    assert rel_err(a.final_state.cpu().numpy(), b.final_state.cpu().numpy()) < 1e-10
    ra, rb = S.ops.stats_finalize(a.stats_partial, a.samples, piv), S.ops.stats_finalize(b.stats_partial, b.samples, piv)
    assert float(ra[0]) == B * H == float(rb[0]) and rel_err(ra.cpu().numpy(), rb.cpu().numpy()) < 1e-9
    ac = _cuda(rng.uniform(-5, 5, (B, n - 1)))
    a, b = (S.ops.rollout(p, H, actions=ac, want_final=True, kernel=k) for k in (_k(S, kern), S.KERNEL_THREAD))
    np.testing.assert_allclose(a.returns.cpu().numpy(), b.returns.cpu().numpy(), rtol=1e-9, atol=1e-13)
    assert rel_err(a.final_state.cpu().numpy(), b.final_state.cpu().numpy()) < 1e-10


@pytest.mark.parametrize("kern", LANE_KERNELS)
@pytest.mark.parametrize("n", [3, 5, 10])
def test_lane_policy_rollouts_match_reference_fixture(S, n, kern):
    """Fixtures generated by the unmodified Python reference (oracle/make_golden.py)."""
    g = golden("gym_rollout.npz")
    H = int(g[f"n{n}_H"])
    p = S.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    res = S.ops.rollout(p, H, policies=_cuda(g[f"n{n}_W"]), want_final=True, want_trajectory=True,
                        kernel=_k(S, kern))
    assert _ret_err(res.returns.cpu().numpy(), g[f"n{n}_v1_return"]) < RET_TOL
    assert rel_err(res.final_state.cpu().numpy(), g[f"n{n}_v1_final"]) < 1e-8
    traj = res.trajectory.cpu().numpy()
    assert rel_err(traj[49::50].transpose(1, 0, 2), g[f"n{n}_v1_traj50"]) < 1e-8
    res = S.ops.rollout(p, H, policies=_cuda(g[f"n{n}_W"]), mean=_cuda(g[f"n{n}_mean"]),
                        inv_sigma=_cuda(g[f"n{n}_var"] ** -0.5), want_final=True, kernel=_k(S, kern))
    assert _ret_err(res.returns.cpu().numpy(), g[f"n{n}_v2_return"]) < RET_TOL
    assert rel_err(res.final_state.cpu().numpy(), g[f"n{n}_v2_final"]) < 1e-8


@pytest.mark.parametrize("kern", LANE_KERNELS)
@pytest.mark.parametrize("n,R", [(3, 1), (5, 1), (5, 3), (7, 1), (10, 2)])
def test_lane_v2_philox_rollouts_and_moments_match_oracle(S, O, n, R, kern):
    H, D = 90, 5
    ps, po = S.make_params(n=n), O.make_params(n=n)
    no, ws = 2 * n + 2, (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(200 + n + R)
    W = rng.uniform(-1, 1, ws) * 0.1
    mean, var = rng.normal(size=no) * 0.05, rng.uniform(.5, 2, no)
    pivot = S.ops.reset_state(n)
    init = rand_states(rng, n, R, scale=0.3) if R > 1 else None
    B = 2 * D * R
    kw = dict(B=B, base_policy=_cuda(W), nu=0.05, seed=12, iteration=1, dir0=2, rollouts_per_policy=R,
              mean=_cuda(mean), inv_sigma=_cuda(var ** -0.5), stats_pivot=pivot,
              init_state=None if init is None else _cuda(init))
    res = S.ops.rollout(ps, H, kernel=_k(S, kern), **kw)
    got = res.returns.cpu().numpy().reshape(D, 2, R)
    rec = S.ops.stats_finalize(res.stats_partial, res.samples, pivot).cpu().numpy()
    trajs = []
    for k in range(D):
        d = O.philox_delta(12, 1, 2 + k, ws)
        for j, sign in enumerate((+1, -1)):
            for r in range(R):
                ret, _, tr = O.rollout(po, O.GYM, H, policy=W + sign * 0.05 * d, mean=mean, inv_sigma=var ** -0.5,
                                       init_state=None if init is None else init[r], want_traj=True)
                assert abs(got[k, j, r] - ret) < RET_TOL * max(1e-3, abs(ret))
                trajs.append(tr)
    m, v = O.mean_var(np.concatenate(trajs))
    assert rec[0] == B * H
    np.testing.assert_allclose(rec[1:1 + no], m, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rec[1 + no:] / (rec[0] - 1), v, rtol=1e-8)
    # the thread kernel sees the same perturbations: returns and moments agree to rounding
    ref = S.ops.rollout(ps, H, kernel=S.KERNEL_THREAD, **kw)
    np.testing.assert_allclose(res.returns.cpu().numpy(), ref.returns.cpu().numpy(), rtol=1e-9, atol=1e-12)
    rec2 = S.ops.stats_finalize(ref.stats_partial, ref.samples, pivot).cpu().numpy()
    np.testing.assert_allclose(rec, rec2, rtol=1e-9, atol=1e-11)
    # perturbations read from memory instead of Philox: bit-identical
    d_gpu = S.ops.philox_deltas(12, 1, 2, D, ws)
    kw2 = dict(kw)
    kw2.update(deltas=d_gpu)
    mem = S.ops.rollout(ps, H, kernel=_k(S, kern), **kw2)
    assert torch.equal(mem.returns, res.returns)


@pytest.mark.parametrize("kern", LANE_KERNELS)
def test_lane_dir_mask_and_init_perturb(S, kern):
    n, H, D, R = 5, 70, 9, 2
    p = S.make_params(n=n)
    ws = (n - 1) * (2 * n + 2)
    W = _cuda(np.random.default_rng(5).uniform(-1, 1, ws) * 0.1)
    mask = torch.tensor([1, 0, 1, 1, 0, 0, 1, 1, 0], dtype=torch.int32, device="cuda")
    kw = dict(B=2 * D * R, base_policy=W, nu=0.03, seed=3, iteration=7, rollouts_per_policy=R, init_perturb=1e-2,
              dir_mask=mask, want_final=True)
    a = S.ops.rollout(p, H, kernel=_k(S, kern), **kw)
    b = S.ops.rollout(p, H, kernel=S.KERNEL_THREAD, **kw)
    ra, rb = a.returns.cpu().numpy().reshape(D, 2 * R), b.returns.cpu().numpy().reshape(D, 2 * R)
    m = mask.cpu().numpy().astype(bool)
    assert np.isnan(ra[~m]).all() and np.isfinite(ra[m]).all()
    np.testing.assert_allclose(ra[m], rb[m], rtol=1e-9, atol=1e-12)
    fa, fb = a.final_state.cpu().numpy().reshape(D, 2 * R, -1), b.final_state.cpu().numpy().reshape(D, 2 * R, -1)
    assert rel_err(fa, fb) < 1e-10  # screened-out directions keep their (perturbed) start state in both


@pytest.mark.parametrize("kern", LANE_KERNELS)
def test_lane_rollout_deterministic_batch_order_invariant_and_nan_isolated(S, kern):
    """BASELINE config[2] shape (n = 5, 2,048 envs, H = 1000): two runs are bit-identical, an environment's
    result does not depend on where it sits in the batch (which warp, which lane group), and a NaN
    environment does not disturb the environments that share its warp."""
    n, B, H = 5, 2048, 1000
    p = S.make_params(n=n)
    no = 2 * n + 2
    rng = np.random.default_rng(0)
    Ws = _cuda(rng.uniform(-1, 1, (B, n - 1, no)) * 0.05)
    mean, inv = _cuda(rng.normal(size=no) * 0.05), _cuda(rng.uniform(.7, 1.4, no))
    kw = dict(mean=mean, inv_sigma=inv, want_final=True, kernel=_k(S, kern))
    a = S.ops.rollout(p, H, policies=Ws, **kw)
    b = S.ops.rollout(p, H, policies=Ws, **kw)
    assert torch.equal(a.returns, b.returns) and torch.equal(a.final_state, b.final_state)
    assert bool(torch.isfinite(a.returns).all())
    perm = torch.randperm(B, device="cuda")
    c = S.ops.rollout(p, H, policies=Ws[perm].contiguous(), **kw)
    assert torch.equal(c.returns, a.returns[perm]) and torch.equal(c.final_state, a.final_state[perm])
    # a sub-batch gives the same numbers as the full batch
    d = S.ops.rollout(p, H, policies=Ws[100:163].contiguous(), **kw)
    assert torch.equal(d.returns, a.returns[100:163])
    init = np.zeros((B, no))
    init[:, 2::2] = np.pi / 2
    init[77, 5] = np.nan
    e = S.ops.rollout(p, 200, policies=Ws, init_state=_cuda(init), **kw)
    f = S.ops.rollout(p, 200, policies=Ws, **kw)
    keep = torch.arange(B, device="cuda") != 77
    assert bool(torch.isnan(e.returns[77])) and torch.equal(e.returns[keep], f.returns[keep])


@pytest.mark.parametrize("kern", LANE_KERNELS)
def test_lane_chunk_chaining_is_bit_identical(S, kern):
    """final_state -> init_state chaining in chunks that are multiples of 64 steps (the exact re-evaluation
    of the tracked sines/cosines) reproduces the single launch bit for bit; returns accumulate.  Inputs: explicit
    policies from the reset state, and fixed actions on calm and spun environments sharing warps (one segment at
    20-300 rad/s, test_trig_tiers population (b)), whose steps run in the tail and exact tiers."""
    from test_trig_tiers import _spun
    n, H = 5, 192
    rng = np.random.default_rng(8)
    Ws = _cuda(rng.uniform(-1, 1, (50, n - 1, 2 * n + 2)) * 0.1)
    init, ac, _ = _spun(n)
    for p, src, start in ((S.make_params(n=n), dict(policies=Ws), None),
                          (S.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, direction=(.6, .8)), dict(actions=_cuda(ac)),
                           _cuda(init))):
        B = len(next(iter(src.values())))
        one = S.ops.rollout(p, H, want_final=True, kernel=_k(S, kern), init_state=start, **src)
        out = {"returns": torch.zeros(B, dtype=torch.float64, device="cuda"),
               "final_state": torch.empty(B, 2 * n + 2, dtype=torch.float64, device="cuda")}
        for c in range(3):
            S.ops.rollout(p, 64, want_final=True, kernel=_k(S, kern), out=out,
                          init_state=start if c == 0 else out["final_state"], accumulate_returns=c > 0, **src)
        assert np.array_equal(out["final_state"].cpu().numpy().view(np.int64), one.final_state.cpu().numpy().view(np.int64))
        np.testing.assert_allclose(out["returns"].cpu().numpy(), one.returns.cpu().numpy(), rtol=1e-12, atol=1e-14)


def test_kernel_choice(S):
    """AUTO picks the lane-split kernel for small batches of short chains, the thread kernel otherwise;
    asking for LANES where it has no kernel (per-step screening, clipping, rlglue dynamics) fails loudly."""
    L = S._lib.lib()

    def choice(n, B, **f):
        cfg = S._lib.SwmRollout()
        cfg.variant, cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = f.get("variant", 0), 1, 10, B, 1
        cfg.kernel, cfg.clip_actions = f.get("kernel", 0), f.get("clip", 0)
        cfg.screen.enabled = f.get("screen", 0)
        if cfg.screen.enabled:
            cfg.screen.sim = S.make_params(n=n)
        return L.swm_rollout_kernel_choice(ctypes.byref(S.make_params(n=n)), ctypes.byref(cfg))

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert choice(5, 4 * (2 * sms + 1)) == S.KERNEL_LANES           # more than two lane groups per SM: one warp per group
    assert choice(5, 4 * 2 * sms) == S.KERNEL_LANES2                # up to two per SM: main + operator warp
    assert choice(3, 512) == S.KERNEL_LANES2 and choice(5, 256) == S.KERNEL_LANES2
    # from 6 segments on and at most one lane group per SM: two operator warps taking alternate steps
    assert choice(7, 4 * sms) == S.KERNEL_LANES3 and choice(7, 4 * sms + 4) == S.KERNEL_LANES2 and choice(6, 256) == S.KERNEL_LANES3
    assert choice(5, 64, kernel=S.KERNEL_LANES3) == S.KERNEL_LANES3 and choice(5, 64, clip=1, kernel=S.KERNEL_LANES3) == -2
    assert choice(3, 65536) == S.KERNEL_THREAD and choice(5, 131072) == S.KERNEL_THREAD
    assert choice(10, 2048) == S.KERNEL_THREAD  # tuned for chains of up to 7 segments
    assert choice(10, 2048, kernel=S.KERNEL_LANES) == S.KERNEL_LANES
    assert choice(5, 64, kernel=S.KERNEL_THREAD) == S.KERNEL_THREAD and choice(5, 64, kernel=S.KERNEL_LANES) == S.KERNEL_LANES
    assert choice(5, 2048, screen=1) == S.KERNEL_THREAD and choice(5, 2048, clip=1) == S.KERNEL_THREAD
    assert choice(5, 2048, variant=1) == S.KERNEL_THREAD
    assert choice(5, 2048, screen=1, kernel=S.KERNEL_LANES) == -2  # SWM_ERR_UNSUPPORTED
    assert choice(3, 64, screen=1) == S.KERNEL_LANES2                # per-step screening: warp-specialised kernels only
    assert choice(5, 2048, kernel=S.KERNEL_LANES2) == S.KERNEL_LANES2 and choice(5, 64, clip=1, kernel=S.KERNEL_LANES2) == -2
    with pytest.raises(S.SwimmerLibError):
        S.ops.rollout(S.make_params(n=3), 10, variant=S.RLGLUE, kernel=S.KERNEL_LANES,
                      actions=torch.zeros(4, 2, dtype=torch.float64, device="cuda"))
