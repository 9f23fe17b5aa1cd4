"""Fused H-step rollout parity.  Tolerance (BASELINE.json north_star): H=1000 returns within 1e-6
relative; in practice the kernels agree with the oracle to ~1e-12."""
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


@pytest.mark.parametrize("n,variant,H", [(3, 0, 1000), (5, 0, 400), (10, 0, 200), (2, 0, 300),
                                         (3, 1, 500), (5, 1, 200), (7, 0, 200)])
def test_fixed_action_rollout_matches_oracle(S, O, n, variant, H):
    rng = np.random.default_rng(n * 7 + variant)
    B = 130
    h = 0.001 if variant == 0 else 0.01
    ps, po = S.make_params(n=n, h=h), O.make_params(n=n, h=h)
    ac = rng.uniform(-5, 5, (B, n - 1))
    res = S.ops.rollout(ps, H, variant=variant, actions=_cuda(ac), want_final=True)
    want_r, want_f = O.rollout_fixed_batch(po, variant, ac, H)
    assert _ret_err(res.returns.cpu().numpy(), want_r) < RET_TOL
    assert rel_err(res.final_state.cpu().numpy(), want_f) < 1e-8


@pytest.mark.parametrize("n", [3, 5, 10])
def test_policy_rollouts_match_reference_fixture(S, n):
    g = golden("gym_rollout.npz")
    H = int(g[f"n{n}_H"])
    p = S.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    res = S.ops.rollout(p, H, policies=_cuda(g[f"n{n}_W"]), want_final=True, want_trajectory=True)
    assert _ret_err(res.returns.cpu().numpy(), g[f"n{n}_v1_return"]) < RET_TOL
    assert rel_err(res.final_state.cpu().numpy(), g[f"n{n}_v1_final"]) < 1e-8
    traj = res.trajectory.cpu().numpy()  # [H, B, no]
    assert rel_err(traj[49::50].transpose(1, 0, 2), g[f"n{n}_v1_traj50"]) < 1e-8
    res = S.ops.rollout(p, H, policies=_cuda(g[f"n{n}_W"]), mean=_cuda(g[f"n{n}_mean"]),
                        inv_sigma=_cuda(g[f"n{n}_var"] ** -0.5), want_final=True)
    assert _ret_err(res.returns.cpu().numpy(), g[f"n{n}_v2_return"]) < RET_TOL
    assert rel_err(res.final_state.cpu().numpy(), g[f"n{n}_v2_final"]) < 1e-8


def test_environment_rollout_api(S):
    g = golden("gym_rollout.npz")
    ep = S.EnvParam("x", n=3, H=1000, l_i=.8, m_i=1.2, h=1e-3, k=10.2, epsilon=0)
    E = S.Environment(ep)
    total, states = E.rollout(g["n3_W"][1])
    assert isinstance(total, float) and isinstance(states, list) and len(states) == 1000 and len(states[0]) == 8
    assert abs(total - g["n3_v1_return"][1]) < RET_TOL * abs(g["n3_v1_return"][1])
    total, _ = E.rollout(g["n3_W"][1], covariance=np.diag(g["n3_var"]), mean=g["n3_mean"])
    assert abs(total - g["n3_v2_return"][1]) < RET_TOL * abs(g["n3_v2_return"][1])
    a = E.select_action(g["n3_W"][0], states[10])
    np.testing.assert_allclose(a, g["n3_W"][0] @ np.array(states[10]), rtol=1e-13, atol=1e-15)
    a = E.select_action(g["n3_W"][0], states[10], covariance=np.diag(g["n3_var"]), mean=g["n3_mean"])
    want = (g["n3_W"][0] @ np.diag(g["n3_var"] ** -0.5)) @ (np.array(states[10]) - g["n3_mean"])
    np.testing.assert_allclose(a, want, rtol=1e-13, atol=1e-15)
    E.close()


@pytest.mark.parametrize("n", [3, 5, 10])
def test_philox_rollouts_match_oracle_with_injected_deltas(S, O, n):
    """The kernel's in-register W +- nu*delta_k (Philox) equals the oracle run on the oracle's own
    Philox restatement: pins generator, addressing, sign convention and ordering [r+_0, r-_0, ...]."""
    H, N, nu, seed, it, dir0 = 150, 6, 0.05, 0xDEADBEEFCAFE, 4, 3
    ps, po = S.make_params(n=n), O.make_params(n=n)
    ws = (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(n)
    W = rng.uniform(-1, 1, ws) * 0.3
    res = S.ops.rollout(ps, H, B=2 * N, base_policy=_cuda(W), nu=nu, seed=seed, iteration=it, dir0=dir0)
    d_gpu = S.ops.philox_deltas(seed, it, dir0, N, ws).cpu().numpy()
    want = []
    for k in range(N):
        d = O.philox_delta(seed, it, dir0 + k, ws)
        np.testing.assert_array_equal(d, d_gpu[k])  # bit-exact generator
        for sign in (+1, -1):
            want.append(O.rollout(po, 0, H, policy=W + sign * nu * d)[0])
    assert _ret_err(res.returns.cpu().numpy(), want) < RET_TOL
    # same thing through the "deltas from memory" path
    res2 = S.ops.rollout(ps, H, B=2 * N, base_policy=_cuda(W), nu=nu, deltas=_cuda(d_gpu))
    np.testing.assert_array_equal(res2.returns.cpu().numpy(), res.returns.cpu().numpy())


@pytest.mark.parametrize("n,R", [(3, 4), (10, 32), (10, 3), (6, 64)])
def test_shared_policy_groups_and_init_states(S, O, n, R):
    """R rollouts per policy from R different initial states (registers / per-thread smem / per-warp
    smem policy storage all give the oracle's numbers)."""
    H, P = 120, 4
    ps, po = S.make_params(n=n), O.make_params(n=n)
    rng = np.random.default_rng(n + R)
    Ws = rng.uniform(-1, 1, (P, n - 1, 2 * n + 2)) * 0.2
    init = rand_states(rng, n, R, scale=0.5)
    res = S.ops.rollout(ps, H, policies=_cuda(Ws), rollouts_per_policy=R, init_state=_cuda(init))
    got = res.returns.cpu().numpy().reshape(P, R)
    for q in range(P):
        for r in range(0, R, max(1, R // 4)):
            want = O.rollout(po, 0, H, policy=Ws[q], init_state=init[r])[0]
            assert abs(got[q, r] - want) < RET_TOL * max(1e-3, abs(want))
    red = S.ops.reduce_returns(res.returns, R).cpu().numpy()
    np.testing.assert_allclose(red, got.mean(1), rtol=1e-14)


def test_v2_moments_match_oracle(S, O):
    n, H, P = 3, 200, 70  # 70 envs -> two blocks, second one ragged
    ps, po = S.make_params(n=n), O.make_params(n=n)
    rng = np.random.default_rng(9)
    Ws = rng.uniform(-1, 1, (P, 2, 8)) * 0.3
    mean, var = rng.normal(size=8) * 0.1, rng.uniform(.5, 2, 8)
    pivot = S.ops.reset_state(n)
    res = S.ops.rollout(ps, H, policies=_cuda(Ws), mean=_cuda(mean), inv_sigma=_cuda(var ** -0.5),
                        stats_pivot=pivot)
    rec = S.ops.stats_finalize(res.stats_partial, res.samples, pivot).cpu().numpy()
    trajs = [O.rollout(po, 0, H, policy=W, mean=mean, inv_sigma=var ** -0.5, want_traj=True)[2] for W in Ws]
    allst = np.concatenate(trajs)
    m, v = O.mean_var(allst)
    assert rec[0] == P * H
    np.testing.assert_allclose(rec[1:9], m, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(rec[9:] / (rec[0] - 1), v, rtol=1e-9)
    # merging two halves in order reproduces the whole (Chan), and yields mean / inv_sigma
    running = torch.zeros(17, dtype=torch.float64, device="cuda")
    recs = []
    for half in (Ws[:32], Ws[32:]):
        r = S.ops.rollout(ps, H, policies=_cuda(half), mean=_cuda(mean), inv_sigma=_cuda(var ** -0.5),
                          stats_pivot=pivot)
        recs.append(S.ops.stats_finalize(r.stats_partial, r.samples, pivot))
    mo, so = torch.zeros(8, dtype=torch.float64, device="cuda"), torch.zeros(8, dtype=torch.float64, device="cuda")
    S.ops.stats_merge(running, torch.stack(recs), mo, so)
    np.testing.assert_allclose(mo.cpu().numpy(), m, rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(so.cpu().numpy(), v ** -0.5, rtol=1e-9)


def test_safe_step_screening_matches_reference_fixture(S, O):
    g = golden("safe_ars.npz")
    m, l, k = g["sim_mlk"]
    real = S.SwimmerEnv("RealWorld", n=3)
    sim = S.SwimmerEnv("Simulator", n=3, m_i=m, l_i=l, k=k)
    for i in range(6):
        ag = S.Safe_ARS(S.builtin_cost, g["safe_real_thresh"][i], g["safe_sim_thresh"][i], sim)
        R, states = ag.rollout(real, g["safe_W"][i], 400)
        assert abs(R - g["safe_returns"][i]) < RET_TOL * max(1e-3, abs(g["safe_returns"][i]))
        assert len(states) == 400
        assert rel_err(states[-1], g["safe_finals"][i]) < 1e-8
        fr = int(ag.last_rollout.frozen_at.cpu()[0])
        # fixture: index from which saved states repeat; kernel: first step judged unsafe
        assert fr == g["safe_frozen_from"][i] or (fr == 400 and g["safe_frozen_from"][i] == 400)
        if fr < 400:
            assert states[fr] == states[-1] and states[fr - 1] == states[fr]
    # a cost the kernel does not implement is rejected loudly
    with pytest.raises(NotImplementedError):
        S.Safe_ARS(lambda x: float(np.sum(np.abs(x))), 1.0, 0.5, sim)
    # isSafe keeps the reference's semantics
    ag = S.Safe_ARS(S.builtin_cost, 6.0, 5.8, sim)
    st = rand_states(np.random.default_rng(1), 3, 1)[0]
    simp = O.make_params(n=3, m_i=m, l_i=l, k=k)
    nxt, _ = O.step(simp, 0, st, [1., 2.])
    assert ag.isSafe(S.builtin_cost, 5.8, sim, st.tolist(), [1., 2.]) == (np.max(np.abs(nxt[3::2])) <= 5.8)


def test_rlglue_rollout_fixture_and_clip(S, O):
    g = golden("rlglue_step.npz")
    p = S.make_params(n=3, h=0.01)
    res = S.ops.rollout(p, 500, variant=1, actions=_cuda(g["roll_action"][None]), want_final=True)
    assert rel_err(res.final_state.cpu().numpy()[0], g["roll_final"]) < 1e-8
    assert abs(float(res.returns.cpu()[0]) - g["roll_return"]) < RET_TOL * abs(g["roll_return"])
    # clipped linear policy (RL-Glue agent semantics) vs oracle
    po = O.make_params(n=3, h=0.01)
    W = np.random.default_rng(2).uniform(-1, 1, (2, 8)) * 40
    want = O.rollout(po, 1, 200, policy=W, clip=True)[0]
    got = S.ops.rollout(p, 200, variant=1, policies=_cuda(W[None]), clip_actions=True)
    assert abs(float(got.returns.cpu()[0]) - want) < RET_TOL * max(1e-3, abs(want))


def test_rollout_is_deterministic_and_batch_order_invariant(S):
    """Size-independent properties at BASELINE config-2 scale (65,536 envs, 1,000 steps): two runs
    are bit-identical, and an environment's result does not depend on where it sits in the batch."""
    p = S.make_params(n=3)
    rng = np.random.default_rng(0)
    ac = torch.as_tensor(rng.uniform(-5, 5, (65536, 2))).cuda()
    a = S.ops.rollout(p, 1000, actions=ac, want_final=True)
    b = S.ops.rollout(p, 1000, actions=ac, want_final=True)
    assert torch.equal(a.returns, b.returns) and torch.equal(a.final_state, b.final_state)
    perm = torch.randperm(65536, device="cuda")
    c = S.ops.rollout(p, 1000, actions=ac[perm].contiguous(), want_final=True)
    assert torch.equal(c.returns, a.returns[perm]) and torch.equal(c.final_state, a.final_state[perm])
    assert bool(torch.isfinite(a.returns).all())
    # zero torque from reset is a fixed point of the dynamics: state and return stay exactly 0
    z = S.ops.rollout(p, 1000, actions=torch.zeros(64, 2, dtype=torch.float64, device="cuda"), want_final=True)
    assert float(z.returns.abs().max()) < 1e-12


@pytest.mark.parametrize("n,R", [(5, 1), (7, 1), (8, 1), (10, 1), (7, 32), (10, 64)])
def test_v2_rollouts_and_moments_every_storage_mode(S, O, n, R):
    """V2 rollouts + moments for every combination of policy storage (per-thread / per-warp shared
    memory) and moment storage (registers up to n = 7, shared memory above), including the
    shared-memory sizes right at the 48 KB opt-in limit (n = 7)."""
    H, D = 80, 3
    ps, po = S.make_params(n=n), O.make_params(n=n)
    no, ws = 2 * n + 2, (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(100 + n + R)
    W = rng.uniform(-1, 1, ws) * 0.1
    mean, var = rng.normal(size=no) * 0.05, rng.uniform(.5, 2, no)
    pivot = S.ops.reset_state(n)
    init = rand_states(rng, n, R, scale=0.3) if R > 1 else None
    B = 2 * D * R
    res = S.ops.rollout(ps, H, B=B, base_policy=_cuda(W), nu=0.05, seed=12, iteration=1, rollouts_per_policy=R,
                        mean=_cuda(mean), inv_sigma=_cuda(var ** -0.5), stats_pivot=pivot,
                        init_state=None if init is None else _cuda(init))
    got = res.returns.cpu().numpy().reshape(D, 2, R)
    rec = S.ops.stats_finalize(res.stats_partial, res.samples, pivot).cpu().numpy()
    trajs = []
    for k in range(D):
        d = O.philox_delta(12, 1, k, ws)
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


@pytest.mark.parametrize("n", [3, 5, 10])
def test_one_step_rollout_equals_batched_step(S, O, n):
    """H = 1: the fused kernel's step (tracked trig, folded constants) and the batched single-step kernel
    (fresh sincos) agree to round-off, and both with the oracle within the single-step tolerance 1e-12."""
    ps, po = S.make_params(n=n), O.make_params(n=n)
    rng = np.random.default_rng(70 + n)
    B = 200
    st = rand_states(rng, n, B)
    ac = rng.uniform(-5, 5, (B, n - 1))
    roll = S.ops.rollout(ps, 1, actions=_cuda(ac), init_state=_cuda(st), want_final=True)
    nxt, rew = S.ops.step_batched(ps, _cuda(st), _cuda(ac))
    want, want_r = O.step_batch(po, O.GYM, st, ac)
    assert rel_err(roll.final_state.cpu().numpy(), want) < 1e-12
    assert rel_err(nxt.cpu().numpy(), want) < 1e-12
    assert rel_err(roll.final_state.cpu().numpy(), nxt.cpu().numpy()) < 1e-13
    np.testing.assert_allclose(roll.returns.cpu().numpy(), want_r, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(rew.cpu().numpy(), want_r, rtol=1e-11, atol=1e-13)


@pytest.mark.parametrize("case", ["fixed_n3", "philox_v2_n5", "grouped_n10", "explicit_n7"])
def test_chunked_rollout_equals_single_launch(S, case):
    """ops.ChunkedRollout (sub-batches x 64-step-aligned time chunks on several streams, state chained through
    final_state -> init_state, returns accumulated on the device): every final state bit-identical to the
    single launch, returns equal up to the rounding of the partial sums, V2 moments equal to 1e-12."""
    rng = np.random.default_rng(31)
    if case == "fixed_n3":
        n, B, H = 3, 5000, 300
        p = S.make_params(n=n)
        kw = dict(actions=_cuda(rng.uniform(-5, 5, (B, n - 1))))
        extra = {}
    elif case == "philox_v2_n5":
        n, B, H = 5, 2 * 150, 200
        p = S.make_params(n=n)
        no = 2 * n + 2
        kw = dict(base_policy=_cuda(rng.uniform(-1, 1, (n - 1) * no) * 0.1), stats_pivot=S.ops.reset_state(n))
        extra = dict(nu=0.05, seed=4, iteration=3, mean=_cuda(rng.normal(size=no) * 0.05),
                     inv_sigma=_cuda(rng.uniform(.5, 2, no)))
    elif case == "grouped_n10":
        n, R, D, H = 10, 32, 6, 150
        B = 2 * D * R
        p = S.make_params(n=n)
        no = 2 * n + 2
        kw = dict(base_policy=_cuda(rng.uniform(-1, 1, (n - 1) * no) * 0.05), rollouts_per_policy=R,
                  stats_pivot=S.ops.reset_state(n))
        extra = dict(nu=0.05, seed=9, iteration=1, init_perturb=1e-2, mean=_cuda(np.zeros(no)),
                     inv_sigma=_cuda(np.ones(no)))
    else:
        n, B, H = 7, 96, 130
        p = S.make_params(n=n)
        kw = dict(policies=_cuda(rng.uniform(-1, 1, (B, n - 1, 2 * n + 2)) * 0.1))
        extra = {}
    single_kw = dict(kw)
    single_kw.update(extra)
    if "actions" not in kw and "policies" not in kw:
        single_kw["B"] = B
    # the chunked schedule launches the one-thread-per-environment kernel (bit-identical chaining)
    ref = S.ops.rollout(p, H, want_final=True, dir0=5 if "base_policy" in kw else 0, kernel=S.KERNEL_THREAD,
                        **single_kw)
    for n_sub, chunk in ((1, 64), (3, 64), (4, 128)):
        plan = S.ops.ChunkedRollout(p, H, B=B, n_sub=n_sub, chunk=chunk, **kw, **extra)
        for _ in range(2):  # re-running reuses the buffers
            got = plan.run(dir0=5 if "base_policy" in kw else 0)
            torch.cuda.synchronize()
            assert torch.equal(got.final_state, ref.final_state), (case, n_sub, chunk)
            np.testing.assert_allclose(got.returns.cpu().numpy(), ref.returns.cpu().numpy(), rtol=1e-12, atol=1e-13)
            if ref.stats_partial is not None:
                piv = kw["stats_pivot"]
                a = S.ops.stats_finalize(got.stats_partial, got.samples, piv).cpu().numpy()
                b = S.ops.stats_finalize(ref.stats_partial, ref.samples, piv).cpu().numpy()
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-13)
    with pytest.raises(ValueError):
        S.ops.ChunkedRollout(p, H, B=B, chunk=100, **kw, **extra)


def test_native_schedule_equals_plain_launch(S):
    """swm_rollout's own chunked schedule (sub-batches x 64-step chunks on internal streams, chosen by the
    library for batches that leave 3-4 warps per SM sub-partition, or forced through schedule_sub / _chunk):
    final states bit-identical to one plain launch, returns equal to the rounding of the partial sums, V2
    moments to 1e-12; unschedulable requests fail loudly; the query entry point reports the choice."""
    import ctypes
    rng = np.random.default_rng(5)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    # auto: fixed actions, n = 3, 3.46 warps per sub-partition on a 148-SM part
    B = int(3.46 * 4 * sms * 32) // 64 * 64
    p = S.make_params(n=3)
    ac = _cuda(rng.uniform(-5, 5, (B, 2)))
    auto = S.ops.rollout(p, 300, actions=ac, want_final=True)
    plain = S.ops.rollout(p, 300, actions=ac, want_final=True, schedule="plain")
    assert torch.equal(auto.final_state, plain.final_state)
    np.testing.assert_allclose(auto.returns.cpu().numpy(), plain.returns.cpu().numpy(), rtol=1e-12, atol=1e-13)
    cfg = S._lib.SwmRollout()
    cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = 0, 300, B, 1
    cfg.actions, cfg.returns, cfg.final_state = ac.data_ptr(), auto.returns.data_ptr(), auto.final_state.data_ptr()
    ns, ch = ctypes.c_int(-1), ctypes.c_int(-1)
    assert S._lib.lib().swm_rollout_schedule(ctypes.byref(p), ctypes.byref(cfg), None, ctypes.byref(ns), ctypes.byref(ch)) == 0
    assert (ns.value, ch.value) == (8, 256)    # enqueued eagerly: few launches; 16 x 64 while capturing a graph
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = S.ops.rollout(p, 300, actions=ac, want_final=True)
        assert S._lib.lib().swm_rollout_schedule(ctypes.byref(p), ctypes.byref(cfg), S._lib.stream_ptr(), ctypes.byref(ns),
                                                 ctypes.byref(ch)) == 0
    assert (ns.value, ch.value) == (16, 64)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured.final_state, plain.final_state)
    cfg.final_state = None   # no chaining buffer: plain
    assert S._lib.lib().swm_rollout_schedule(ctypes.byref(p), ctypes.byref(cfg), None, ctypes.byref(ns), ctypes.byref(ch)) == 0
    assert ns.value == 0
    # forced: V2 Philox policies with moments, R rollouts per policy from R start states, dir_mask, n = 5
    n, R, D, H = 5, 4, 24, 200
    p = S.make_params(n=n)
    no = 2 * n + 2
    kw = dict(B=2 * D * R, base_policy=_cuda(rng.uniform(-1, 1, (n - 1) * no) * 0.1), nu=0.05, seed=4, iteration=2, dir0=3,
              rollouts_per_policy=R, init_state=_cuda(rand_states(rng, n, R, scale=0.3)), init_perturb=1e-2,
              mean=_cuda(rng.normal(size=no) * 0.05), inv_sigma=_cuda(rng.uniform(.5, 2, no)),
              stats_pivot=S.ops.reset_state(n), want_final=True, kernel=S.KERNEL_THREAD,
              dir_mask=torch.tensor([1, 1, 0, 1] * 6, dtype=torch.int32, device="cuda"))
    plain = S.ops.rollout(p, H, schedule="plain", **kw)
    for sched in ((3, 64), (5, 128), (16, 64)):
        got = S.ops.rollout(p, H, schedule=sched, **kw)
        torch.cuda.synchronize()
        assert torch.equal(torch.nan_to_num(got.final_state), torch.nan_to_num(plain.final_state)), sched
        np.testing.assert_allclose(got.returns.cpu().numpy(), plain.returns.cpu().numpy(), rtol=1e-12, atol=1e-13)
        a = S.ops.stats_finalize(got.stats_partial, got.samples, kw["stats_pivot"]).cpu().numpy()
        b = S.ops.stats_finalize(plain.stats_partial, plain.samples, kw["stats_pivot"]).cpu().numpy()
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-13)
    with pytest.raises(S.SwimmerLibError):   # trajectories cannot be chunked
        S.ops.rollout(p, H, schedule=(4, 64), want_trajectory=True, **kw)
    with pytest.raises(S.SwimmerLibError):   # chunk must be a multiple of 64
        S.ops.rollout(p, H, schedule=(4, 100), **kw)
