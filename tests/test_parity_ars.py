"""ARS update / agent parity against the reference fixtures and the oracle.
north_star: top-b selection bit-exact given identical rewards; weight updates within 1e-6."""
import io
import contextlib
import os
import tempfile

import numpy as np
import pytest
import torch

from conftest import golden, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-6


def _cuda(a, dtype=np.float64):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=dtype)).cuda()


def test_topb_bit_exact(S):
    g = golden("topb.npz")
    for N in (1, 2, 8, 33, 256, 1024):
        order = S.ops.ars_topb(_cuda(g[f"returns_{N}"])).cpu().numpy()
        np.testing.assert_array_equal(order, g[f"order_{N}"])
    np.testing.assert_array_equal(S.ops.ars_topb(_cuda(g["returns_ties"])).cpu().numpy(), g["order_ties"])


def test_topb_large_random_vs_numpy(S):
    rng = np.random.default_rng(4)
    for N in (4096, 5000):
        r = rng.normal(size=2 * N)
        want = np.argsort(np.maximum(r[0::2], r[1::2]), kind="stable")[::-1]
        np.testing.assert_array_equal(S.ops.ars_topb(_cuda(r)).cpu().numpy(), want)
    # all-equal keys: stable rule = higher index first
    np.testing.assert_array_equal(S.ops.ars_topb(_cuda(np.zeros(64))).cpu().numpy(), np.arange(32)[::-1])
    # screened-out directions sort last
    r = rng.normal(size=16); mask = np.array([1, 0, 1, 1, 0, 1, 1, 1], dtype=np.int32)
    order = S.ops.ars_topb(_cuda(r), _cuda(mask, np.int32)).cpu().numpy()
    assert set(order[-2:]) == {1, 4} and sorted(order) == list(range(8))


@pytest.mark.parametrize("semantics", [0, 1, 2])
@pytest.mark.parametrize("n,N,b", [(3, 8, 8), (5, 64, 16), (10, 33, 7)])
def test_update_matches_oracle(S, O, semantics, n, N, b):
    ws = (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(n * N + semantics)
    W0, rets = rng.normal(size=ws), rng.normal(size=2 * N) * 30
    seed, it = 99, 7
    dist = 1 if semantics == 2 else 0
    deltas = np.stack([O.philox_delta(seed, it, k, ws, dist=dist) for k in range(N)])
    want, want_sigma = O.update_policy(W0, deltas, rets, b=b, alpha=0.02, semantics=semantics)
    use_order, n_order, divisor, ddof = S.ops.update_args(semantics, N, b)
    for explicit in (False, True):
        W = _cuda(W0)
        r = _cuda(rets)
        order = S.ops.ars_topb(r) if use_order else None
        sig = torch.zeros(1, dtype=torch.float64, device="cuda")
        S.ops.ars_update(W, r, N, order=order, n_order=n_order, divisor=divisor, ddof=ddof, alpha=0.02,
                         seed=seed, iteration=it, delta_dist=dist,
                         deltas=_cuda(deltas) if explicit else None, sigma_out=sig)
        assert rel_err(W.cpu().numpy(), want) < 1e-12
        assert abs(float(sig.cpu()[0]) - want_sigma) < 1e-12 * want_sigma


def test_ars_agent_config1_matches_reference_run(S):
    """BASELINE config 1 (n=3, V1, N=8, b=8, H=1000, seed 0): same numpy seed => the reference's own
    iteration returns and policies (fixture recorded from the unmodified reference)."""
    g = golden("ars_agent.npz")
    ep = S.EnvParam("LeonSwimmer-RealWorld", n=3, H=1000, l_i=1., m_i=1., h=1e-3, k=10., epsilon=0)
    ap = S.ARSParam("RLControl", V1=True, n_iter=2, H=1000, N=8, b=8, alpha=0.0075, nu=0.01,
                    safe=False, threshold=0, initial_w="Zero")
    ag = S.ARSAgent(ep, ap, seed=0)
    for it in range(3):
        rets = ag.runOneIteration()
        assert isinstance(rets, list) and len(rets) == 16
        np.testing.assert_allclose(rets, g["c1_returns"][it], rtol=TOL, atol=1e-9)
        assert rel_err(ag.policy, g["c1_policies"][it]) < TOL
    # the reference-shaped helper methods
    d = 2 * g["c1_rand"][0] - 1
    order = ag.sort_directions(list(d), g["c1_returns"][0].tolist())
    mx = np.maximum(g["c1_returns"][0][0::2], g["c1_returns"][0][1::2])
    assert order == np.argsort(mx)[::-1].tolist()
    ag.policy = np.zeros((2, 8))
    ag.update_policy(list(d), g["c1_returns"][0].tolist(), order)
    assert rel_err(ag.policy, g["c1_policies"][0]) < 1e-10


def test_ars_agent_v2_matches_reference_run(S):
    g = golden("ars_agent.npz")
    ep = S.EnvParam("x", n=3, H=250, l_i=.8, m_i=1.2, h=1e-3, k=10.2, epsilon=0)
    ap = S.ARSParam("x", V1=False, n_iter=2, H=250, N=4, b=4, alpha=0.0075, nu=0.01,
                    safe=False, threshold=0, initial_w="Zero")
    ag = S.ARSAgent(ep, ap, seed=3)
    assert np.all(ag.mean == 0) and np.all(ag.covariance == np.eye(8))
    for it in range(3):
        rets = ag.runOneIteration()
        np.testing.assert_allclose(rets, g["v2_returns"][it], rtol=TOL, atol=1e-9)
        assert rel_err(ag.policy, g["v2_policies"][it]) < TOL
        np.testing.assert_allclose(ag.mean, g["v2_means"][it], rtol=TOL, atol=1e-9)
        np.testing.assert_allclose(np.diag(ag.covariance), g["v2_vars"][it], rtol=TOL)


def test_ars_agent_run_training_curve(S):
    g = golden("ars_agent.npz")
    ep = S.EnvParam("x", n=3, H=200, l_i=1., m_i=1., h=1e-3, k=10., epsilon=0)
    ap = S.ARSParam("x", V1=True, n_iter=4, H=200, N=2, b=2, alpha=0.02, nu=0.05,
                    safe=False, threshold=0, initial_w="Zero")
    with tempfile.TemporaryDirectory() as td:
        ag = S.ARSAgent(ep, ap, seed=11)
        curve = ag.runTraining(save_data_path=os.path.join(td, "db.npz"),
                               save_policy_path=os.path.join(td, "pol"))
        assert isinstance(curve, np.ndarray) and curve.shape == (5,)
        np.testing.assert_allclose(curve, g["rt_curve"], rtol=TOL, atol=1e-9)
        assert rel_err(ag.policy, g["rt_policy"]) < TOL
        assert rel_err(np.load(os.path.join(td, "pol.npy")), g["rt_policy"]) < TOL
        assert ag.database.size == 5 * 4 and len(ag.database.trajectories[0]) == 200


def test_ars_agent_safe_mode_matches_reference_run(S):
    """Reward-constraint safe exploration, N=1 (the reference's own use): screened iterations do no
    real rollout and no update; surviving ones reproduce the reference's returns and policies."""
    g = golden("ars_agent_safe.npz")
    l, m, k = g["sim_params"]
    with tempfile.TemporaryDirectory() as td:
        wpath = os.path.join(td, "w0.npy"); np.save(wpath, g["W0"])
        dpath = os.path.join(td, "db.npz")
        np.savez(dpath, policies=[g["W0"]], trajectories=[np.zeros((50, 8))])
        ep = S.EnvParam("real", n=3, H=300, l_i=.8, m_i=1.2, h=1e-3, k=10.2, epsilon=0.001)
        ap = S.ARSParam("x", V1=True, n_iter=7, H=300, N=1, b=1, alpha=0.0075, nu=0.01, safe=True,
                        threshold=float(g["threshold"]), initial_w=wpath)
        np.random.seed(99)
        with contextlib.redirect_stdout(io.StringIO()):
            ag = S.ARSAgent(ep, ap, data_path=dpath, seed=4, approx_error=0.001,
                            sim_thresh=S.Threshold(K=1, A=0.1, B=0.001))
        assert abs(ag.sim_threshold - float(g["sim_threshold"])) < 1e-12
        np.testing.assert_allclose([ag.estimated_param.l_i, ag.estimated_param.m_i, ag.estimated_param.k],
                                   [l, m, k], rtol=1e-14)
        assert (ep.l_i, ep.m_i, ep.k) == (.8, 1.2, 10.2)  # caller's dataclass is not mutated (D-5)
        for it in range(8):
            with contextlib.redirect_stdout(io.StringIO()):
                rets = ag.runOneIteration()
            want = g["returns"][it]
            if np.isnan(want[0]):
                assert rets == []
            else:
                np.testing.assert_allclose(rets, want, rtol=TOL)
            assert rel_err(ag.policy, g["policies"][it]) < TOL


def test_basic_and_safe_ars_train_match_reference_run(S):
    g = golden("safe_ars.npz")
    real = S.SwimmerEnv("RealWorld", n=3)
    ag = S.Basic_ARS()
    np.random.seed(1)
    with contextlib.redirect_stdout(io.StringIO()):
        curve, states = ag.train(3, real, 4, 2, 0.02, 0.05, 200)
    np.testing.assert_allclose(curve, g["basic_curve"], rtol=TOL, atol=1e-10)
    assert rel_err(ag.policy, g["basic_policy"]) < TOL
    assert states.shape == (3 * 8, 200, 8)
    assert rel_err(states[-1][-1], g["basic_states_last"]) < 1e-8
    m, l, k = g["sim_mlk"]
    sim = S.SwimmerEnv("Simulator", n=3, m_i=m, l_i=l, k=k)
    sag = S.Safe_ARS(S.builtin_cost, 3.0, 2.0, sim)
    np.random.seed(2)
    with contextlib.redirect_stdout(io.StringIO()):
        curve, _ = sag.train(2, real, 3, 2, 0.02, 0.3, 150)
    np.testing.assert_allclose(curve, g["safetrain_curve"], rtol=TOL, atol=1e-10)
    assert rel_err(sag.policy, g["safetrain_policy"]) < TOL


def test_philox_agent_matches_oracle_loop(S, O):
    """delta_source='philox' (nothing uploaded): an oracle loop fed the same Philox deltas gives the
    same returns, policy and V2 statistics after 3 iterations (n=5, V2, true top-b)."""
    n, N, b, H, nu, alpha, seed = 5, 6, 3, 120, 0.03, 0.02, 1234
    ps, po = S.make_params(n=n), O.make_params(n=n)
    ws = (n - 1) * (2 * n + 2)
    eng = S.ArsEngine(ps, N=N, b=b, alpha=alpha, nu=nu, H=H, v2=True, semantics=S.ARS_TOPB, seed=seed,
                      distributed=False)
    W = np.zeros(ws); mean, inv_sigma = np.zeros(2 * n + 2), np.ones(2 * n + 2); states = []
    for it in range(3):
        got = eng.run_iteration().cpu().numpy()
        deltas = np.stack([O.philox_delta(seed, it, k, ws) for k in range(N)])
        rets = []
        for kdir in range(N):
            for sign in (+1, -1):
                r, _, traj = O.rollout(po, 0, H, policy=W + sign * nu * deltas[kdir], mean=mean,
                                       inv_sigma=inv_sigma, want_traj=True)
                rets.append(r); states.append(traj)
        np.testing.assert_allclose(got, rets, rtol=TOL, atol=1e-9)
        W, _ = O.update_policy(W, deltas, np.array(rets), b=b, alpha=alpha, semantics=1)
        mean, var = O.mean_var(np.concatenate(states)); inv_sigma = var ** -0.5
        assert rel_err(eng.W.cpu().numpy(), W) < TOL
        np.testing.assert_allclose(eng.mean.cpu().numpy(), mean, rtol=TOL, atol=1e-9)
        np.testing.assert_allclose(eng.inv_sigma.cpu().numpy(), inv_sigma, rtol=TOL)


def test_engine_masked_update_and_resume(S, O):
    """Reward-constraint screening with N > 1 (the case the reference cannot run, SURVEY D-2):
    survivors are compacted; the update equals the oracle's over the surviving triples.  Also
    state_dict round trip => bit-identical continuation."""
    n, N, H, nu = 3, 8, 100, 0.05
    real = S.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    sim = S.make_params(n=n, l_i=.81, m_i=1.21, k=10.25)
    W0 = np.random.default_rng(0).uniform(-1, 1, 16) * 0.3
    probe = S.ArsEngine(sim, N=N, b=N, alpha=0.01, nu=nu, H=H, seed=5, initial_policy=W0, distributed=False)
    sim_ret = probe.run_iteration(update=False).cpu().numpy()
    thr = float(np.median(np.minimum(sim_ret[0::2], sim_ret[1::2])))
    eng = S.ArsEngine(real, N=N, b=N, alpha=0.01, nu=nu, H=H, seed=5, initial_policy=W0,
                      sim_params=sim, sim_threshold=thr, distributed=False)
    rets = eng.run_iteration().cpu().numpy()
    ok = (sim_ret[0::2] > thr) & (sim_ret[1::2] > thr)
    assert 0 < ok.sum() < N
    assert np.array_equal(np.isnan(rets[0::2]), ~ok) and np.array_equal(eng.mask.cpu().numpy() != 0, ok)
    deltas = np.stack([O.philox_delta(5, 0, k, 16) for k in range(N)])
    keep = np.nonzero(ok)[0]
    r_keep = rets.reshape(N, 2)[keep].ravel()
    want, _ = O.update_policy(W0, deltas[keep], r_keep, b=N, alpha=0.01, semantics=0)
    assert rel_err(eng.W.cpu().numpy(), want) < 1e-12
    sd = eng.state_dict()
    a = eng.run_iteration().clone()
    eng2 = S.ArsEngine(real, N=N, b=N, alpha=0.01, nu=nu, H=H, seed=0, sim_params=sim, sim_threshold=thr,
                       distributed=False)
    eng2.load_state_dict(sd)
    b = eng2.run_iteration()
    assert torch.equal(torch.nan_to_num(a), torch.nan_to_num(b)) and torch.equal(eng.W, eng2.W)


@pytest.mark.parametrize("use_graph", [False, True])
def test_speculative_real_rollouts_equal_screen_first(S, use_graph):
    """Reward-constraint safe mode, V1: rolling out ALL directions in the real world beside the simulator
    rollouts and masking afterwards (engine default) is bit-identical to screening first and rolling out the
    survivors only -- returns (NaN pattern included), mask, survivor count and policy, over several
    iterations, eagerly and as a replayed graph.  V2 engines and trajectory requests never speculate."""
    n, N, H, nu = 3, 16, 130, 0.05
    real = S.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    sim = S.make_params(n=n, l_i=.81, m_i=1.21, k=10.25)
    W0 = np.random.default_rng(2).uniform(-1, 1, 16) * 0.3
    probe = S.ArsEngine(sim, N=N, b=N, alpha=0.01, nu=nu, H=H, seed=5, initial_policy=W0, distributed=False)
    sim_ret = probe.run_iteration(update=False).cpu().numpy()
    thr = float(np.median(np.minimum(sim_ret[0::2], sim_ret[1::2])))
    kw = dict(N=N, b=5, alpha=0.01, nu=nu, H=H, seed=5, initial_policy=W0, sim_params=sim, sim_threshold=thr,
              distributed=False, semantics=S.ARS_TOPB, use_graph=use_graph)
    spec, first = S.ArsEngine(real, **kw), S.ArsEngine(real, speculate=False, **kw)
    assert spec.speculate and not first.speculate
    screened = []
    for it in range(5):
        a, b = spec.run_iteration().clone(), first.run_iteration().clone()
        assert torch.equal(torch.isnan(a), torch.isnan(b)), it
        screened.append(int(torch.isnan(a).sum()))
        assert torch.equal(torch.nan_to_num(a), torch.nan_to_num(b)), it
        assert torch.equal(spec.mask, first.mask) and torch.equal(spec.W, first.W)
        assert torch.equal(spec.n_pass_total, first.n_pass_total)
    assert 0 < screened[0] < 2 * N and (spec._graph is not None) == use_graph
    # not where a screened-out rollout would leave something behind
    assert not S.ArsEngine(real, v2=True, **kw).speculate
    t = spec.run_iteration(want_trajectory=True, update=False)
    assert torch.equal(torch.isnan(t), torch.isnan(spec.last.returns))  # screened first: the rollout kernel wrote the NaNs


def test_estimator_objective(S, O):
    """Estimator.I (ars/estimator.py:36-62): zero at the true parameters (the reference's own
    self-check, estimator.py:136), and equal to the oracle's value elsewhere."""
    n, H = 3, 80
    po = O.make_params(n=n, l_i=1., m_i=1., k=10.)
    rng = np.random.default_rng(8)
    W = rng.uniform(-1, 1, (2, 8)) * 0.5
    _, _, traj = O.rollout(po, 0, H, policy=W, want_traj=True)
    db = S.Database(); db.add_trajectory(traj.tolist(), W)
    guess = S.EnvParam("sim", n=n, H=H, m_i=1.01, l_i=1.01, h=0.001, k=10.01, epsilon=0.01)
    est = S.Estimator(db, guess, capacity=1)
    assert est.I([1.0, 1.0, 10.0]) < 1e-12
    x = [1.05, 0.97, 10.4]
    p2 = O.make_params(n=n, m_i=x[0], l_i=x[1], k=x[2])
    want = 0.0
    for t in range(H - 1):
        nxt, _ = O.step(p2, 0, traj[t], W @ traj[t])
        want += np.linalg.norm(nxt - traj[t + 1])
    assert abs(est.I(x) - want) < 1e-9 * want
    # a whole CMA-ES generation in one launch per trajectory (swm_step_batched_models): same numbers as
    # one candidate at a time, also beyond the 24 models one launch carries
    xs = [[1.0, 1.0, 10.0], x] + [list(np.array(x) * (1 + 0.01 * i)) for i in range(1, 28)]
    pop = est.I_population(xs)
    assert len(pop) == 29 and pop[0] < 1e-12 and abs(pop[1] - want) < 1e-9 * want
    for i in (2, 17, 23, 24, 28):
        assert abs(pop[i] - est.I(xs[i])) <= 1e-12 * max(1.0, pop[i])


def test_seed_fanout_equals_sequential_agents(S, tmp_path):
    """Seed fan-out (ars/experiment.py:64-72): S engines on S streams give, bit for bit, the curves
    and policies of S agents trained one after the other; Experiment.plot keeps the call shape."""
    p = S.make_params(n=3)
    kw = dict(N=8, b=8, alpha=0.0075, nu=0.05, H=120, v2=True, semantics=S.ARS_AGENT)
    fan = S.SeedFanout(p, range(5), **kw)
    curves = fan.run(3)
    assert curves.shape == (5, 4) and np.isfinite(curves).all()
    for i, seed in enumerate(range(5)):
        eng = S.ArsEngine(p, seed=seed, distributed=False, curve_capacity=8, **kw)  # eager, no graph
        want = [float(torch.nanmean(eng.run_iteration()).cpu()) for _ in range(4)]
        np.testing.assert_array_equal(curves[i], eng.curve[:4].cpu().numpy())
        np.testing.assert_allclose(curves[i], want, rtol=1e-13)
        np.testing.assert_array_equal(fan.policies()[i], eng.policy_numpy())
    assert len({tuple(c) for c in curves}) == 5  # different seeds, different curves
    ep = S.EnvParam("LeonSwimmer", n=3, H=120, l_i=1., m_i=1., h=1e-3, k=10., epsilon=0)
    ap = S.ARSParam("agent", V1=False, n_iter=3, H=120, N=8, b=8, alpha=0.0075, nu=0.05, safe=False,
                    threshold=0, initial_w="Zero")
    r_graphs = S.Experiment(ep, results_path=str(tmp_path) + "/").plot(5, ap)
    np.testing.assert_array_equal(r_graphs, curves)
    saved = list((tmp_path / "array").glob("*.npy"))
    assert len(saved) == 1 and np.array_equal(np.load(saved[0]), r_graphs)


@pytest.mark.parametrize("mode", ["v1", "v2", "safe", "grouped", "step_screen"])
def test_graph_replay_equals_eager_iterations(S, mode):
    """The captured CUDA graph of one iteration (device-side Philox iteration counter) replays to
    exactly the eager sequence: returns, policy, statistics and curve bit for bit, including a
    state_dict resume in the middle."""
    n = 10 if mode == "grouped" else 3
    p = S.make_params(n=n, l_i=.8, m_i=1.2, k=10.2)
    kw = dict(N=6, b=4, alpha=0.02, nu=0.05, H=60, semantics=S.ARS_TOPB, seed=9, distributed=False, curve_capacity=16)
    if mode == "v2":
        kw.update(v2=True, semantics=S.ARS_AGENT)
    if mode == "grouped":
        kw.update(v2=True, rollouts_per_direction=32, init_perturb=1e-2)
    if mode == "safe":
        kw.update(sim_params=S.make_params(n=n, l_i=.81, m_i=1.21, k=10.25), sim_threshold=-0.002)
    if mode == "step_screen":  # per-step screening: thresholds inside the spread of the directions' peak |thd|
        kw.update(step_screen=dict(sim_params=S.make_params(n=n, l_i=.81, m_i=1.21, k=10.25, h=0.0012),
                                   sim_thresh=0.1, real_thresh=0.08))
    eager, graph = S.ArsEngine(p, **kw), S.ArsEngine(p, use_graph=True, **kw)
    frozen = []
    for it in range(6):
        a, b = eager.run_iteration().clone(), graph.run_iteration().clone()
        assert torch.equal(torch.nan_to_num(a, nan=-7.0), torch.nan_to_num(b, nan=-7.0)), it
        assert torch.equal(eager.W, graph.W) and torch.equal(eager.stats, graph.stats)
        if mode == "step_screen":
            assert torch.equal(eager.last.frozen_at, graph.last.frozen_at), it
            assert torch.equal(eager.last.violations, graph.last.violations), it
            frozen.append(eager.last.frozen_at.cpu().numpy())
        if it == 3:  # resume both from the eager engine's checkpoint
            sd = eager.state_dict()
            eager.load_state_dict(sd)
            graph.load_state_dict(sd)
    assert graph._graph is not None and eager._graph is None
    assert eager.iteration == graph.iteration == 6 == int(graph.iter_dev.cpu()[0])
    ce, cg = eager.curve.cpu().numpy(), graph.curve.cpu().numpy()
    np.testing.assert_array_equal(np.nan_to_num(ce, nan=-7.0), np.nan_to_num(cg, nan=-7.0))
    assert np.isfinite(cg[:6]).any()
    if mode == "step_screen":
        frozen = np.concatenate(frozen)
        assert (frozen < kw["H"]).any() and (frozen == kw["H"]).any()


def test_rlglue_agent_experiment_matches_oracle_loop(S, O, tmp_path):
    """RL-Glue agent semantics end to end (SwimmerAgent.py:181-241 + SwimmerExperiment.cpp:65-84):
    clipped actions, delta ~ U[0,1), index order, first b directions, sample std, semi-implicit C++
    dynamics from the 0.001 start state, one frozen evaluation rollout per iteration."""
    (tmp_path / "parameters.txt").write_text(
        "n_seg 3\ndirection 1.0 0.\nh_global 0.01\nN 4\nb 3\nH 150\nalpha 0.02\nnu 0.02\nmax_u 5.\nl_i 1.\nk 10.\nm_i 1.\n")
    exp = S.RlglueArsExperiment.from_parameters_file(str(tmp_path / "parameters.txt"), seed=77)
    assert (exp.N, exp.b, exp.H, exp.params.n, exp.params.h) == (4, 3, 150, 3, 0.01)
    got = exp.run_training(4)
    po = O.make_params(n=3, h=0.01)
    W = np.zeros(16)
    want = []
    for it in range(4):
        deltas = np.stack([O.philox_delta(77, it, k, 16, dist=1) for k in range(4)])
        assert deltas.min() >= 0.0 and deltas.max() < 1.0
        rets = [O.rollout(po, O.RLGLUE, 150, policy=W + s * 0.02 * deltas[k], clip=True)[0]
                for k in range(4) for s in (+1, -1)]
        W, _ = O.update_policy(W, deltas, np.array(rets), b=3, alpha=0.02, semantics=2)
        want.append(O.rollout(po, O.RLGLUE, 150, policy=W, clip=True)[0])
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(exp.policy.reshape(-1), W, rtol=1e-6, atol=1e-12)
    exp.write_results(str(tmp_path / "results.txt"))
    lines = (tmp_path / "results.txt").read_text().splitlines()
    assert len(lines) == 4 and lines[0].startswith("Reward for one rollout with policy at iteration 0: ")


def test_reference_scripts_run_with_changed_imports(tmp_path):
    """examples/plot_graph.py and examples/safe_exploration.py are the reference's ars/plot_graph.py and
    ars/safe_exploration.py with only the imports changed; a miniature run of both must complete and
    respect the reward constraint semantics (a real rollout is only made when both simulated returns of
    its direction exceed the simulator threshold)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "plot_graph.py"), "--n_seed", "3",
                          "--n_iter", "4", "--results_path", str(tmp_path) + "/"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    saved = list((tmp_path / "array").glob("*.npy"))
    assert len(saved) == 1 and np.load(saved[0]).shape == (3, 5)
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "safe_exploration.py"), "--quick",
                          "--data_dir", str(tmp_path / "data")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "Safety threshold" in out.stdout and "Using approximated estimation" in out.stdout
    res = np.load(next((tmp_path / "data").glob("epsilon_sim_threshold_*.npz")))
    assert res["min_return"].shape == (2,) and np.isfinite(res["safety_threshold"])
    db = np.load(tmp_path / "data" / "real_world_2.npz")
    assert db["trajectories"].shape[1:] == (200, 8) and db["policies"].shape[1:] == (2, 8)
    # safe_ars/experiment.py: per-step state-constraint screening keeps every real step under the threshold
    out = subprocess.run([sys.executable, os.path.join(root, "examples", "safe_ars_experiment.py"), "--n_iter", "6",
                          "--n_rollout", "150", "--n_seeds", "2", "--thresh", "1.5", "--nu", "0.3",
                          "--path", str(tmp_path / "safe_ars")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    res = np.load(next((tmp_path / "safe_ars").glob("*.npz")))
    assert res["safe_returns"].shape == (2, 6) and res["safe_costs"].shape == (2, 2 * 6 * 150)
    # the simulator screens every step at thresh - 1 = 0.5: the real cost never reaches the threshold 1.5,
    # while the unconstrained agent is free to exceed it
    assert 0.0 < res["safe_costs"].max() <= 1.5


@pytest.mark.parametrize("mode", ["v2", "grouped", "safe"])
def test_engine_with_chunked_rollouts_matches_plain_engine(S, mode):
    """ArsEngine(rollout_chunks=(n_sub, chunk)) schedules the real rollouts as sub-batches x time-chunks on
    several streams: same returns (rounding of the partial sums), same policy and statistics within 1e-10
    after three iterations, also under graph replay and with a screening mask."""
    n = 10 if mode == "grouped" else 5
    p = S.make_params(n=n)
    kw = dict(N=12, b=6, alpha=0.02, nu=0.05, H=200, v2=True, semantics=S.ARS_TOPB, seed=2, distributed=False)
    if mode == "grouped":
        kw.update(rollouts_per_direction=32, init_perturb=1e-2)
    if mode == "safe":
        kw.update(sim_params=S.make_params(n=n, l_i=1.01, m_i=0.99, k=10.1), sim_threshold=-0.001)
    plain = S.ArsEngine(p, **kw)
    chunked = S.ArsEngine(p, rollout_chunks=(3, 64), **kw)
    graphed = S.ArsEngine(p, rollout_chunks=(3, 64), use_graph=True, **kw)
    for it in range(3):
        a, b, c = plain.run_iteration().clone(), chunked.run_iteration().clone(), graphed.run_iteration().clone()
        assert torch.equal(torch.isnan(a), torch.isnan(b))
        np.testing.assert_allclose(torch.nan_to_num(b).cpu().numpy(), torch.nan_to_num(a).cpu().numpy(),
                                   rtol=1e-9, atol=1e-12)
        assert torch.equal(torch.nan_to_num(b), torch.nan_to_num(c))  # graph replay = eager, bit for bit
        np.testing.assert_allclose(chunked.W.cpu().numpy(), plain.W.cpu().numpy(), rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(chunked.inv_sigma.cpu().numpy(), plain.inv_sigma.cpu().numpy(), rtol=1e-9)
        assert torch.equal(chunked.W, graphed.W) and torch.equal(chunked.stats, graphed.stats)
    assert graphed._graph is not None


@pytest.mark.parametrize("R,with_mask,v2", [(1, False, True), (3, True, True), (2, False, False)])
def test_pack_exchange_kernel_matches_separate_kernels(S, R, with_mask, v2):
    """swm_ars_pack_exchange (one launch: per-direction mean returns, screening mask, V2 moment record, unpack)
    against the separate kernels it replaces (swm_reduce_returns + swm_stats_finalize), and its collective
    fallback (record_out -> all-gather -> gathered_in) against distributed.RecordLayout.split."""
    from swimmer_ars_b200 import distributed as D
    n, Nl, H = 5, 7, 60
    no = 2 * n + 2
    p = S.make_params(n=n)
    rng = np.random.default_rng(R)
    W = torch.as_tensor(rng.uniform(-1, 1, (n - 1) * no) * 0.1).cuda()
    mask = torch.tensor([1, 0, 1, 1, 1, 0, 1], dtype=torch.int32, device="cuda") if with_mask else None
    piv = S.ops.reset_state(n)
    mean, inv = torch.zeros(no, dtype=torch.float64, device="cuda"), torch.ones(no, dtype=torch.float64, device="cuda")
    res = S.ops.rollout(p, H, B=2 * Nl * R, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=R, dir_mask=mask,
                        mean=mean if v2 else None, inv_sigma=inv if v2 else None, stats_pivot=piv if v2 else None)
    F = no if v2 else 0
    f64 = dict(dtype=torch.float64, device="cuda")
    returns_all, records = torch.zeros(2 * Nl, **f64), torch.zeros(1, 1 + 2 * no, **f64)
    mask_all = torch.zeros(Nl, dtype=torch.int32, device="cuda") if with_mask else None
    units = torch.tensor([int(mask.sum())], dtype=torch.int32, device="cuda") if with_mask else None
    samples = float(2 * R * H) if with_mask else (res.samples if v2 else 0.0)
    pack = dict(returns_local=res.returns, n_local=Nl, R=R, mask_local=mask, stats_partial=res.stats_partial,
                samples=samples, units=units, pivot=piv if v2 else None, n_features=F)
    S.ops.pack_exchange(None, **pack, returns_all=returns_all, mask_all=mask_all, records=records if v2 else None)
    want_r = S.ops.reduce_returns(res.returns, R) if R > 1 else res.returns
    assert torch.equal(torch.nan_to_num(returns_all), torch.nan_to_num(want_r))
    assert torch.equal(torch.isnan(returns_all), torch.isnan(want_r))
    if with_mask:
        assert torch.equal(mask_all, mask)
        # returns of a screened-out direction are NaN in the record even when its rollouts did run (the engine's
        # speculative real-world rollouts): same result from unmasked rollouts + the mask
        full = S.ops.rollout(p, H, B=2 * Nl * R, base_policy=W, nu=0.05, seed=3, rollouts_per_policy=R,
                             mean=mean if v2 else None, inv_sigma=inv if v2 else None)
        assert not bool(torch.isnan(full.returns).any())
        r2 = torch.zeros(2 * Nl, **f64)
        S.ops.pack_exchange(None, returns_local=full.returns, n_local=Nl, R=R, mask_local=mask, n_features=0,
                            returns_all=r2, mask_all=torch.zeros(Nl, dtype=torch.int32, device="cuda"))
        assert torch.equal(torch.isnan(r2), torch.isnan(returns_all))
        assert torch.equal(torch.nan_to_num(r2), torch.nan_to_num(returns_all))
    if v2:
        want_rec = S.ops.stats_finalize(res.stats_partial, samples, piv, units=units)
        np.testing.assert_allclose(records[0].cpu().numpy(), want_rec.cpu().numpy(), rtol=1e-12, atol=1e-13)
    # collective fallback: pack only, a pretend all-gather over 3 ranks, unpack by the kernel and by torch
    lay = D.RecordLayout(Nl, F, with_mask)
    rec = torch.zeros(lay.length, **f64)
    S.ops.pack_exchange(None, **pack, record_out=rec, gathered_world=3)
    gathered = torch.cat([rec, rec * 2.0, rec * 3.0])
    ra, rc = torch.zeros(3 * 2 * Nl, **f64), torch.zeros(3, 1 + 2 * no, **f64)
    ma = torch.zeros(3 * Nl, dtype=torch.int32, device="cuda") if with_mask else None
    S.ops.pack_exchange(None, n_local=Nl, n_features=F, mask_local=mask, gathered_in=gathered, gathered_world=3,
                        returns_all=ra, mask_all=ma, records=rc if v2 else None)
    t_r, t_m, t_rec = lay.split(gathered, 3)
    assert torch.equal(torch.nan_to_num(ra), torch.nan_to_num(t_r))
    if with_mask:
        assert torch.equal(ma, t_m)
    if v2:
        assert torch.equal(rc[:, :1 + 2 * F], t_rec)


def test_v2_safe_engine_with_everything_screened_out_keeps_identity_normalisation(S):
    """ars_agent.py:179-182 recomputes mean / cov only `if len(rewards) > 0`: an iteration whose directions
    are all screened out (threshold above every simulated return) must leave W, mean = 0 and sigma = 1
    untouched instead of dividing by a zero count."""
    n = 3
    p, sim = S.make_params(n=n), S.make_params(n=n, l_i=1.001)
    eng = S.ArsEngine(p, N=6, b=6, alpha=0.02, nu=0.03, H=50, v2=True, seed=1, distributed=False,
                      sim_params=sim, sim_threshold=1e9)
    for _ in range(2):
        r = eng.run_iteration()
        assert bool(torch.isnan(r).all())
    assert float(eng.W.abs().max()) == 0.0
    assert torch.equal(eng.mean, torch.zeros_like(eng.mean)) and torch.equal(eng.inv_sigma, torch.ones_like(eng.inv_sigma))
    assert float(eng.stats[0]) == 0.0
    eng.sim_threshold = -1e9   # now everything passes: statistics start from this iteration
    r = eng.run_iteration()
    assert bool(torch.isfinite(r).all()) and float(eng.stats[0]) == 12 * 50
    assert bool(torch.isfinite(eng.inv_sigma).all()) and float(eng.W.abs().max()) > 0.0
    # a NaN simulator return is screened out (declared deviation from the reference's `<=`)
    m, cnt = S.ops.screen_mask(torch.tensor([1.0, float("nan"), 1.0, 2.0], dtype=torch.float64, device="cuda"), 0.0)
    assert m.tolist() == [0, 1] and int(cnt) == 1


@pytest.mark.parametrize("tag", ["a", "b"])
def test_rlglue_reference_protocol_kernel_matches_unmodified_agent(S, O, tag):
    """RlglueArsExperiment(protocol='reference') = the reference's literal step-level loop (csrc/rlglue_protocol.cu)
    against the fixture produced by the unmodified agent + compiled C++ swimmer (tests/golden/rlglue_agent.npz),
    replaying the agent's own U[0,1) draws: evaluation returns, reward tables and policies to 1e-9."""
    g = golden("rlglue_agent.npz")
    n, N, b, H, alpha, nu, max_u, l_i, k, m_i, h = g[tag + "_par"]
    kw = dict(n_seg=int(n), N=int(N), b=int(b), H=int(H), alpha=alpha, nu=nu, max_u=max_u, l_i=l_i, k=k, m_i=m_i,
              h_global=h)
    n_it = len(g[tag + "_results"])
    ex = S.RlglueArsExperiment(protocol="reference", **kw)
    # in two calls: the experiment continues where it stopped
    r1, t1 = ex.run_reference_protocol(2, deltas=g[tag + "_deltas"])
    r2, t2 = ex.run_reference_protocol(n_it - 2, deltas=g[tag + "_deltas"])
    res = torch.cat([r1, r2], dim=1)[0].cpu().numpy()
    tab = torch.cat([t1, t2], dim=1)[0].cpu().numpy()
    np.testing.assert_allclose(res, g[tag + "_results"], rtol=1e-9)
    np.testing.assert_allclose(tab, g[tag + "_rewards"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(ex.policy, g[tag + "_policies"][-1], rtol=1e-8, atol=1e-12)
    # Philox perturbations, several replicas: against the restated loop fed with the same Philox draws
    from oracle import rlglue_protocol as RP
    par = dict(kw, direction=(1.0, 0.0))
    ws = (int(n) - 1) * (2 * int(n) + 2)
    ex2 = S.RlglueArsExperiment(protocol="reference", seed=77, replicas=3, **kw)
    got = ex2.run_reference_protocol(2)[0].cpu().numpy()
    for rep in (0, 2):
        d = np.stack([[O.philox_delta(77 + rep, it, kdir, ws, dist=1).reshape(int(n) - 1, -1) for kdir in range(int(N))]
                      for it in range(3)])
        want, _ = RP.restated_protocol(par, 2, d)
        np.testing.assert_allclose(got[rep], want, rtol=1e-9)
    # the drop-in class front end
    ex3 = S.RlglueArsExperiment(protocol="reference", seed=77, **kw)
    np.testing.assert_allclose(ex3.run_training(2), got[0], rtol=0, atol=0)
