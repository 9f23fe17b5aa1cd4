"""The RL-Glue path (semi-implicit C++ dynamics, clipped linear policies, U[0,1) perturbations, the batched and the
step-level experiment protocols, the environment plugin) against the CPU oracle for every segment count.

The oracle solves the full (5n+2)^2 system of SwimmerEnvironment.cpp with a column-pivoted QR; the kernels solve a
reduced (n+2)-unknown system with a partially pivoted LU, in registers up to n = 7 and in local memory above.  The
project's RL-Glue tolerance is 1e-11 per step (DESIGN.md section 6), so the main check is per step: every state a
rollout visited is stepped once by the oracle, with the action clip(W_e . x, +-max_u) recomputed from the kernel's own
state, and compared with the kernel's next state.  Whole trajectories and returns are compared only up to the step
where an oracle twin started 1e-14 away still agrees with the oracle to 1e-10 (test_trig_tiers.py)."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from conftest import rand_states, rel_err
import test_step_screening as scr
import test_trig_tiers as tt

pytestmark = pytest.mark.gpu
NS = [2, 3, 4, 5, 6, 7, 8, 9, 10]
MAX_U, H_STEP = 5.0, 0.01
STEP_TOL = 1e-11       # per-step check against the oracle (norm-relative, floor 1)
EXACT_TOL = 1e-12      # returns against the kernel's own trajectory
RET_TOL, STATE_TOL = 1e-6, 1e-8
PROTO_TOL = 1e-9       # experiment protocols: returns, reward tables, policies
CLIP_FRAC = 0.05       # each clipped launch: >= 5 % of action components at +max_u, at -max_u and in between
H = 100


def _cuda(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _params(mod, n, h=H_STEP):
    return mod.make_params(n=n, l_i=.9, m_i=1.1, k=9.5, h=h, max_u=MAX_U, direction=(.6, .8))


def _kernel_choice(S, p, variant, mode, B, R=1, clip=False, kernel=0):
    cfg = S._lib.SwmRollout()
    cfg.variant, cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = variant, mode, 10, B, R
    cfg.clip_actions, cfg.kernel = int(clip), kernel
    return S._lib.lib().swm_rollout_kernel_choice(ctypes.byref(p), ctypes.byref(cfg))


# ---- (a) per-step rollout conformance ---------------------------------------------------------------------------
# case: (policy source, B, R, clip).  R = 32 keeps one policy per warp in shared memory (W_SMEM_GROUP, n >= 5); R = 1
# policies live in registers (n <= 4) or one column per thread in shared memory (W_SMEM_THREAD).  B = 1, 63, 65 and
# 130 leave idle lanes in the last warp / CTA.
CASES = {
    "fixed": ("fixed", 65, 1, False),
    "explicit": ("explicit", 63, 1, True),
    "explicit_unclipped": ("explicit", 130, 1, False),
    "single": ("explicit", 1, 1, False),
    "group": ("explicit", 64, 32, True),
    "init_count": ("explicit", 65, 1, True),
    "philox01": ("philox01", 130, 1, True),
    "philoxpm1": ("philoxpm1", 64, 1, True),
    "masked": ("philox01", 40, 1, True),
    "perturb": ("philox01", 64, 4, True),
}
SCALES = 2.0 ** np.arange(-3, 7)


def _setup(S, O, n, case, scale):
    """-> (rollout kwargs, per-environment policies [B, n-1, 2n+2] or None, fixed actions [B, n-1] or None,
    start states [B, 2n+2] as the kernel sees them, live mask [B], Philox (seed, it, dir0, D, dist) or None)."""
    src, B, R, clip = CASES[case]
    no, na, ws = 2 * n + 2, n - 1, (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(100 * n + list(CASES).index(case))
    count = 7 if case == "init_count" else (R if R > 1 else B)
    init = rand_states(rng, n, count, scale=0.5)
    starts = init[np.arange(B) % count]
    kw = dict(B=B, variant=S.RLGLUE, clip_actions=clip, rollouts_per_policy=R, init_state=_cuda(init))
    live = np.ones(B, dtype=bool)
    pols = acts = philox = None
    if src == "fixed":
        acts = rng.uniform(-MAX_U, MAX_U, (B, na))
        kw["actions"] = _cuda(acts)
    elif src == "explicit":
        W = rng.uniform(-1, 1, (B // R, na, no)) * scale
        kw["policies"] = _cuda(W)
        pols = W[np.arange(B) // R]
    else:
        D = B // (2 * R)
        dist = S.DELTA_01 if src == "philox01" else S.DELTA_PM1
        seed, it, dir0 = 40 + n, 3, 2
        Wb = rng.uniform(-1, 1, ws) * scale
        nu = 0.5 * scale
        kw.update(base_policy=_cuda(Wb), nu=nu, seed=seed, iteration=it, dir0=dir0, delta_dist=dist)
        pols = np.array([(Wb + (-nu if (e // R) & 1 else nu) * O.philox_delta(seed, it, dir0 + e // (2 * R), ws,
                                                                               dist=dist)).reshape(na, no)
                         for e in range(B)])
        philox = (seed, it, dir0, D, dist)
        if case == "masked":
            mask = (rng.uniform(size=D) < 0.7).astype(np.int32)
            mask[:2] = (0, 1)
            kw["dir_mask"] = torch.as_tensor(mask).cuda()
            live = np.repeat(mask.astype(bool), 2 * R)
        if case == "perturb":  # start = init + init_perturb * U[0,1), Philox stream 1, rollout index e % R
            p = 0.5
            kw["init_perturb"] = p
            starts = np.array([starts[e] + p * O.philox_delta(seed, it, e % R, no, dist=1, stream=1)
                               for e in range(B)])
    return kw, pols, acts, starts, live, philox


def _actions(pols, acts, e, x, clip):
    if pols is None:
        return acts[e]
    a = pols[e] @ x
    return np.clip(a, -MAX_U, MAX_U) if clip else a


def _clip_coverage(pols, seen, live):
    """Fractions of the policy's action components at +max_u, at -max_u and strictly inside, over every state the
    kernel visited (x_0 .. x_{H-1} of every live environment)."""
    raw = np.concatenate([x[:-1] @ pols[e].T for e, x in enumerate(seen) if live[e]])
    return np.mean(raw >= MAX_U), np.mean(raw <= -MAX_U), np.mean(np.abs(raw) < MAX_U), raw.size


def _visited(starts, traj, live):
    return [tt._visited(starts, traj, e) if live[e] else None for e in range(len(starts))]


def _per_step(O, po, seen, pols, acts, clip):
    """Oracle step from every visited state with the recomputed action against the kernel's next state."""
    worst = 0.0
    for e, x in enumerate(seen):
        if x is None or len(x) < 2:
            continue
        want = np.array([O.step(po, O.RLGLUE, x[t], _actions(pols, acts, e, x[t], clip))[0]
                         for t in range(len(x) - 1)])
        err = np.max(np.abs(x[1:] - want), axis=1) / np.maximum(1.0, np.max(np.abs(want), axis=1))
        assert err.max() <= STEP_TOL, (e, int(np.argmax(err)), float(err.max()))
        worst = max(worst, float(err.max()))
    return worst


def _returns_consistent(ret, traj, live, direction):
    """RL-Glue reward = Gdot_{t+1} . direction: the return is the sum over the kernel's own trajectory."""
    (dx, dy), gx, gy = direction, traj[:, live, 0], traj[:, live, 1]
    want = (dx * gx + dy * gy).sum(axis=0)
    scale = (np.abs(dx * gx) + np.abs(dy * gy)).sum(axis=0)
    assert (np.abs(ret[live] - want) <= EXACT_TOL * np.maximum(1.0, scale)).all()


def _within_horizon(O, po, ret, traj, starts, pols, acts, clip, live, Hh):
    """Whole trajectories and returns (partial sums where the twin horizon stops short of H) against the oracle up to
    each live environment's twin horizon; at least half of them must carry the comparison past step 63."""
    rng = np.random.default_rng(11)
    er = es = 0.0
    hz_all = []
    dx, dy = po.direction
    for e in np.flatnonzero(live):
        kw = dict(clip=clip, want_traj=True)
        if pols is None:
            kw["action"] = acts[e]
        else:
            kw["policy"] = pols[e]
        want_r, _, want_t = O.rollout(po, O.RLGLUE, Hh, init_state=starts[e], **kw)
        _, _, twin = O.rollout(po, O.RLGLUE, Hh, init_state=tt._twin(starts[e], rng), **kw)
        hz = tt._horizon(want_t, twin)
        hz_all.append(hz)
        if not hz:
            continue
        es = max(es, rel_err(traj[:hz, e], want_t[:hz]))
        if hz == Hh:
            er = max(er, scr._ret_err(ret[e], want_r))
        else:
            part = lambda t: dx * t[:hz, 0].sum() + dy * t[:hz, 1].sum()
            er = max(er, scr._ret_err(part(traj[:, e]), part(want_t)))
    hz_all = np.array(hz_all)
    assert np.sum(hz_all >= 64) * 2 >= len(hz_all), hz_all
    assert er < RET_TOL and es < STATE_TOL, (er, es)
    return er, es


def _launch(S, p, kw):
    res = S.ops.rollout(p, H, want_final=True, want_trajectory=True, **kw)
    torch.cuda.synchronize()
    return res


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("n", NS)
def test_rlglue_rollout_per_step_matches_oracle(S, O, n, case):
    """rollout_kernel<N, RLGLUE>: every visited state stepped by the oracle (1e-11), returns equal to the sum over
    the kernel's own trajectory (1e-12), whole trajectories within the twin horizon.  Clipped launches scale the
    policies until the clip coverage holds; Philox perturbations equal the same perturbations read from memory bit
    for bit; masked directions return NaN and keep their start state."""
    src, B, R, clip = CASES[case]
    ps, po = _params(S, n), _params(O, n)
    mode = {"fixed": S.ops.POLICY_FIXED_ACTION, "explicit": S.ops.POLICY_EXPLICIT}.get(src, S.ops.POLICY_PHILOX)
    assert _kernel_choice(S, ps, S.RLGLUE, mode, B, R, clip) == S.KERNEL_THREAD
    for scale in (SCALES if clip else [0.3]):
        kw, pols, acts, starts, live, philox = _setup(S, O, n, case, scale)
        res = _launch(S, ps, kw)
        traj = res.trajectory.cpu().numpy()
        seen = _visited(starts, traj, live)
        cov = _clip_coverage(pols, seen, live) if clip else None
        if not clip or min(cov[:3]) >= CLIP_FRAC:
            break
    if clip:
        assert min(cov[:3]) >= CLIP_FRAC, cov
    ret, fin = res.returns.cpu().numpy(), res.final_state.cpu().numpy()
    if not live.all():
        assert (~live).any() and live.any()
        assert np.isnan(ret[~live]).all()
        assert np.array_equal(tt._bits(fin[~live]), tt._bits(starts[~live]))
    worst = _per_step(O, po, seen, pols, acts, clip)
    # the RL-Glue model itself blows up from a few states under strong clipped control: returns of the rollouts
    # that stayed finite
    _returns_consistent(ret, traj, live & np.isfinite(traj).all(axis=(0, 2)), ps.direction)
    er, es = _within_horizon(O, po, ret, traj, starts, pols, acts, clip, live, H)
    if philox is not None:
        seed, it, dir0, D, dist = philox
        ws = (n - 1) * (2 * n + 2)
        mem = _launch(S, ps, dict(kw, deltas=S.ops.philox_deltas(seed, it, dir0, D, ws, dist=dist)))
        for name in ("returns", "final_state"):
            assert np.array_equal(tt._bits(getattr(mem, name).cpu().numpy()), tt._bits(getattr(res, name).cpu().numpy()))
        assert np.array_equal(tt._bits(mem.trajectory.cpu().numpy()[:, live]), tt._bits(traj[:, live]))
    extra = ", clip +/-/inside %.2f/%.2f/%.2f of %d" % cov if clip else ""
    print("\n[rlglue] n=%d %s: max per-step err %.2e, whole trajectory: return %.2e, state %.2e%s"
          % (n, case, worst, er, es, extra))


@pytest.mark.parametrize("n", [3, 6])
def test_gym_clipped_rollout_runs_on_thread_kernel(S, O, n):
    """clip_actions with gym dynamics: the thread kernel honours it (per-step check at the gym bar 1e-12), the lane
    kernels have no clip, so AUTO picks THREAD for a batch that would otherwise go to them and forcing one fails."""
    B, Hg = 37, 150
    ps, po = S.make_params(n=n, max_u=MAX_U), O.make_params(n=n, max_u=MAX_U)
    assert _kernel_choice(S, ps, S.GYM, S.ops.POLICY_EXPLICIT, B, clip=False) != S.KERNEL_THREAD
    assert _kernel_choice(S, ps, S.GYM, S.ops.POLICY_EXPLICIT, B, clip=True) == S.KERNEL_THREAD
    rng = np.random.default_rng(60 + n)
    init = rand_states(rng, n, B, scale=0.5)
    W0 = rng.uniform(-1, 1, (B, n - 1, 2 * n + 2))
    for kern in (S.KERNEL_LANES, S.KERNEL_LANES2, S.KERNEL_LANES3):
        assert _kernel_choice(S, ps, S.GYM, S.ops.POLICY_EXPLICIT, B, clip=True, kernel=kern) < 0
        with pytest.raises(S.SwimmerLibError):
            S.ops.rollout(ps, Hg, policies=_cuda(W0), clip_actions=True, init_state=_cuda(init), kernel=kern)
    live = np.ones(B, dtype=bool)
    for scale in SCALES:
        W = W0 * scale
        res = S.ops.rollout(ps, Hg, policies=_cuda(W), clip_actions=True, init_state=_cuda(init),
                            want_trajectory=True)
        traj = res.trajectory.cpu().numpy()
        seen = [tt._visited(init, traj, e) for e in range(B)]
        cov = _clip_coverage(W, seen, live)
        if min(cov[:3]) >= CLIP_FRAC:
            break
    assert min(cov[:3]) >= CLIP_FRAC, cov
    assert all(len(x) == Hg + 1 for x in seen)
    worst = 0.0
    for e, x in enumerate(seen):
        want = np.array([O.step(po, O.GYM, x[t], np.clip(W[e] @ x[t], -MAX_U, MAX_U))[0] for t in range(Hg)])
        err = np.max(np.abs(x[1:] - want), axis=1) / np.maximum(1.0, np.max(np.abs(want), axis=1))
        assert err.max() <= tt.STEP_TOL, (e, int(np.argmax(err)), float(err.max()))
        worst = max(worst, float(err.max()))
    print("\n[rlglue] gym clipped n=%d: max per-step err %.2e, clip +/-/inside %.2f/%.2f/%.2f of %d"
          % ((n, worst) + cov))


# ---- (b) chunked schedules ---------------------------------------------------------------------------------------
def _schedule(S, p, Hh, kw, buf, stream=None):
    """(n_sub, chunk) swm_rollout takes for the RL-Glue rollout ops.rollout(p, Hh, want_final=True, **kw) (0, 0: one
    plain launch); buf: any device pointer (the query reads no memory)."""
    cfg = S._lib.SwmRollout()
    mode = S.ops.POLICY_FIXED_ACTION if "actions" in kw else S.ops.POLICY_PHILOX
    cfg.variant, cfg.policy_mode, cfg.H, cfg.B, cfg.rollouts_per_policy = S.RLGLUE, mode, Hh, kw["B"], 1
    cfg.clip_actions = int(kw.get("clip_actions", False))
    sched = kw.get("schedule")
    cfg.returns = cfg.final_state = cfg.actions = cfg.policies = buf
    if sched is not None:
        cfg.schedule_sub, cfg.schedule_chunk = sched
    ns, ch = ctypes.c_int(-1), ctypes.c_int(-1)
    assert S._lib.lib().swm_rollout_schedule(ctypes.byref(p), ctypes.byref(cfg), stream, ctypes.byref(ns),
                                             ctypes.byref(ch)) == 0
    return ns.value, ch.value


def _same(got, plain):
    torch.cuda.synchronize()
    assert torch.equal(torch.nan_to_num(got.final_state), torch.nan_to_num(plain.final_state))
    assert torch.equal(torch.isnan(got.returns), torch.isnan(plain.returns))
    np.testing.assert_allclose(torch.nan_to_num(got.returns).cpu().numpy(),
                               torch.nan_to_num(plain.returns).cpu().numpy(), rtol=EXACT_TOL, atol=1e-13)


@pytest.mark.parametrize("graph", [False, True])
def test_rlglue_chunked_schedules_equal_plain_launch(S, graph):
    """RL-Glue rollouts under the library's chunked schedule (sub-batches x 64-step-aligned chunks on internal
    streams, state chained through final_state -> init_state): final states bit-identical to one plain launch,
    returns to the rounding of the partial sums; eagerly and under CUDA-graph capture."""
    rng = np.random.default_rng(8)
    sms = torch.cuda.get_device_properties(0).multi_processor_count

    def run(p, Hh, want, **kw):
        """The rollout, eagerly or captured and replayed; `want`: the schedule it must take."""
        if not graph:
            out = S.ops.rollout(p, Hh, want_final=True, **kw)
            assert _schedule(S, p, Hh, kw, out.returns.data_ptr()) == want
            return out
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = S.ops.rollout(p, Hh, want_final=True, **kw)
            assert _schedule(S, p, Hh, kw, out.returns.data_ptr(), S._lib.stream_ptr()) == want
        g.replay()
        return out

    # the library's own choice: fixed actions, n = 3, 3.46 warps per SM sub-partition
    B, Hh = int(3.46 * 4 * sms * 32) // 64 * 64, 300
    p = _params(S, 3)
    ac = _cuda(rng.uniform(-MAX_U, MAX_U, (B, 2)))
    plain = S.ops.rollout(p, Hh, variant=S.RLGLUE, actions=ac, want_final=True, schedule="plain")
    # enqueued eagerly: 8 x 256; while capturing a graph: 16 x 64
    _same(run(p, Hh, want=(16, 64) if graph else (8, 256), variant=S.RLGLUE, B=B, actions=ac),
          plain)
    # forced: Philox U[0,1) policies, dir_mask, clip, one start state per environment, n = 5
    n, D, Hh = 5, 48, 300
    p = _params(S, n)
    ws = (n - 1) * (2 * n + 2)
    mask = (rng.uniform(size=D) < 0.75).astype(np.int32)
    mask[0] = 0
    kw = dict(variant=S.RLGLUE, B=2 * D, base_policy=_cuda(rng.uniform(-1, 1, ws) * 2.0), nu=1.0, seed=6,
              iteration=1, dir0=4, delta_dist=S.DELTA_01, clip_actions=True, dir_mask=torch.as_tensor(mask).cuda(),
              init_state=_cuda(rand_states(rng, n, 2 * D, scale=0.5)))
    plain = S.ops.rollout(p, Hh, want_final=True, schedule="plain", **kw)
    assert torch.isnan(plain.returns).any() and torch.isfinite(plain.returns).any()
    for sched in ((3, 64), (8, 256), (16, 64)):
        _same(run(p, Hh, want=sched, schedule=sched, **kw), plain)


# ---- (c) batched experiment ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,b", [(1, 1), (4, 3), (5, 5)])
@pytest.mark.parametrize("n", NS)
def test_batched_experiment_matches_oracle_loop(S, O, n, N, b):
    """RlglueArsExperiment(protocol='batched'): every iteration against an oracle loop started from the engine's
    own previous policy -- 2N clipped rollouts of W +- nu delta_k (delta ~ U[0,1)), the first-b / sample-std update
    (update_policy semantics 2), the evaluation rollout of the updated policy."""
    Hh, nu, alpha, seed = 80, 0.3, 0.1, 70 + n
    exp = S.RlglueArsExperiment(n_seg=n, direction=(.6, .8), h_global=H_STEP, N=N, b=b, H=Hh, alpha=alpha, nu=nu,
                                max_u=MAX_U, l_i=.9, k=9.5, m_i=1.1, seed=seed)
    po = _params(O, n)
    ws = (n - 1) * (2 * n + 2)
    worst = [0.0, 0.0, 0.0]
    for it in range(3):
        W = exp.engine.W.cpu().numpy().reshape(-1).copy()
        ev = float(exp.run_one_training_iteration().cpu()[0])
        got = exp.engine.returns.cpu().numpy()
        deltas = np.stack([O.philox_delta(seed, it, k, ws, dist=1) for k in range(N)])
        rets = np.array([O.rollout(po, O.RLGLUE, Hh, policy=W + s * nu * deltas[k], clip=True)[0]
                         for k in range(N) for s in (1.0, -1.0)])
        W_new, _ = O.update_policy(W, deltas, rets, b=b, alpha=alpha, semantics=2)
        W_got = exp.engine.W.cpu().numpy().reshape(-1)
        ev_want = O.rollout(po, O.RLGLUE, Hh, policy=W_got, clip=True)[0]
        errs = (scr._ret_err(got, rets), rel_err(W_got, W_new), scr._ret_err(ev, ev_want))
        assert max(errs) < PROTO_TOL, (it, errs)
        worst = [max(a, c) for a, c in zip(worst, errs)]
    assert np.abs(exp.policy).max() > 0
    print("\n[rlglue] batched experiment n=%d N=%d b=%d: training returns %.2e, policy %.2e, evaluation %.2e"
          % ((n, N, b) + tuple(worst)))


# ---- (d) reference protocol --------------------------------------------------------------------------------------
# (N, b, H): b < N, H = 1, N = b = 1, and b = N, whose update reads the reward slot filled one iteration late.
# With H = 1 every rollout is one step from the reloaded start state, and a torque does not move the centre of mass
# in its first step: all returns are equal up to rounding, sigma is rounding noise and so is the updated policy (0 / 0 =
# NaN where the returns agree exactly).  That case runs one iteration and compares returns and reward tables only.
PROTO = {"base": (3, 2, 16), "h1": (3, 2, 1), "single": (1, 1, 12), "b_eq_n": (3, 3, 12)}
REPLICAS = 40


def _proto_par(n, case):
    N, b, Hh = PROTO[case]
    return dict(n_seg=n, N=N, b=b, H=Hh, alpha=0.05, nu=0.5, max_u=MAX_U, l_i=.9, k=9.5, m_i=1.1, h_global=H_STEP,
                direction=(.6, .8))


@pytest.mark.parametrize("n,case", [(n, "base") for n in NS] + [(n, c) for n in (2, 6, 10)
                                                                 for c in ("h1", "single", "b_eq_n")])
def test_reference_protocol_matches_restated_loop(S, O, n, case):
    """rlglue_protocol_kernel: 40 replicas (two full CTAs of 32 threads and a partial one) against the restated
    step-level loop fed the same Philox U[0,1) draws -- evaluation totals, reward tables and final policies to 1e-9.
    1 + 2 iterations equal one call of 3 bit for bit; explicit deltas reproduce replica 0 bit for bit."""
    from oracle import rlglue_protocol as RP
    par = _proto_par(n, case)
    seed, ws = 900 + n, (n - 1) * (2 * n + 2)
    N_IT = 1 if case == "h1" else 3
    ex = S.RlglueArsExperiment(protocol="reference", seed=seed, replicas=REPLICAS, **par)
    r1, t1 = ex.run_reference_protocol(N_IT)
    res, tab = r1.cpu().numpy(), t1.cpu().numpy()
    if N_IT > 1:  # in two calls: the experiment continues where it stopped
        split = S.RlglueArsExperiment(protocol="reference", seed=seed, replicas=REPLICAS, **par)
        r2, t2 = zip(split.run_reference_protocol(1), split.run_reference_protocol(N_IT - 1))
        assert np.array_equal(tt._bits(torch.cat(r2, dim=1).cpu().numpy()), tt._bits(res))
        assert np.array_equal(tt._bits(torch.cat(t2, dim=1).cpu().numpy()), tt._bits(tab))
        assert np.array_equal(tt._bits(split._state.cpu().numpy()), tt._bits(ex._state.cpu().numpy()))
    reps = range(REPLICAS) if n <= 3 else (0, 31, 32, 39)
    worst = [0.0, 0.0, 0.0]
    state = ex._state.cpu().numpy()
    for rep in reps:
        d = np.stack([[O.philox_delta(seed + rep, it, k, ws, dist=1).reshape(n - 1, -1) for k in range(par["N"])]
                      for it in range(N_IT + 1)])
        tables = []
        want, pols = RP.restated_protocol(par, N_IT, d, tables)
        errs = (scr._ret_err(res[rep], want), rel_err(tab[rep], np.array(tables)),
                0.0 if case == "h1" else rel_err(state[rep, :ws], pols[-1].reshape(-1)))
        assert max(errs) < PROTO_TOL, (rep, errs)
        worst = [max(a, c) for a, c in zip(worst, errs)]
    # explicit deltas, one per iteration, reproduce replica 0's Philox run
    dl = torch.stack([S.ops.philox_deltas(seed, it, 0, par["N"], ws, dist=S.DELTA_01) for it in range(N_IT + 1)])
    ex0 = S.RlglueArsExperiment(protocol="reference", seed=seed, **par)
    r0, t0 = ex0.run_reference_protocol(N_IT, deltas=dl.cpu().numpy())
    assert np.array_equal(tt._bits(r0.cpu().numpy()[0]), tt._bits(res[0]))
    assert np.array_equal(tt._bits(t0.cpu().numpy()[0]), tt._bits(tab[0]))
    assert np.array_equal(tt._bits(ex0._state[0].cpu().numpy()), tt._bits(ex._state[0].cpu().numpy()))
    print("\n[rlglue] reference protocol n=%d %s (%d replicas checked): evaluation %.2e, reward table %.2e, "
          "policy %.2e" % ((n, case, len(reps)) + tuple(worst)))


# ---- (e) environment plugin --------------------------------------------------------------------------------------
class _RL(ctypes.Structure):
    _fields_ = [("numInts", ctypes.c_uint), ("numDoubles", ctypes.c_uint), ("numChars", ctypes.c_uint),
                ("intArray", ctypes.POINTER(ctypes.c_int)), ("doubleArray", ctypes.POINTER(ctypes.c_double)),
                ("charArray", ctypes.c_char_p)]


class _ROT(ctypes.Structure):
    _fields_ = [("reward", ctypes.c_double), ("observation", ctypes.POINTER(_RL)), ("terminal", ctypes.c_int)]


DEFAULT_FILE = "n_seg 3\ndirection 1.0 0.\nh_global 0.01\nmax_u 5.\nl_i 1.\nk 10.\nm_i 1.\n"


@functools.lru_cache(maxsize=None)
def _shim(S):
    L = S._lib.lib()
    L.env_init.restype = ctypes.c_char_p
    L.env_start.restype = ctypes.POINTER(_RL)
    L.env_step.restype = ctypes.POINTER(_ROT)
    L.env_step.argtypes = [ctypes.POINTER(_RL)]
    L.env_message.restype = ctypes.c_char_p
    L.env_message.argtypes = [ctypes.c_char_p]
    return L


def _set(L, path, text):
    path.write_text(text)
    return L.env_message(("set parameters " + str(path)).encode()).decode()


def _action(vals):
    arr = (ctypes.c_double * max(1, len(vals)))(*vals)
    return _RL(0, len(vals), 0, None, arr, None), arr


def _obs(r, n):
    return np.array([r.observation.contents.doubleArray[i] for i in range(2 * n + 2)])


@pytest.fixture
def shim(S, tmp_path):
    """The plugin's process-global state, released and reset to the default parameters afterwards."""
    L = _shim(S)
    L.env_cleanup()
    yield L
    L.env_cleanup()
    assert "n_seg=3" in _set(L, tmp_path / "default.txt", DEFAULT_FILE)


def _param_file(n, h=H_STEP, max_u=MAX_U):
    return "n_seg %s\ndirection 0.6 0.8\nh_global %r\nmax_u %r\nl_i 0.9\nk 9.5\nm_i 1.1\n" % (n, h, max_u)


@pytest.mark.parametrize("n", [2, 5, 10])
def test_env_plugin_matches_oracle(S, O, shim, tmp_path, monkeypatch, n):
    """env_* symbols for n_seg = 2, 5, 10: task-spec dimensions, start state, steps against the oracle (1e-11),
    save / load state; an invalid action (out of range, wrong count) gives terminal = 1 and leaves the state."""
    L = shim
    msg = _set(L, tmp_path / "parameters.txt", _param_file(n))
    assert "n_seg=%d;" % n in msg and "Refused" not in msg
    spec = L.env_init().decode()
    assert "OBSERVATIONS DOUBLES (%d UNSPEC UNSPEC)" % (2 * n + 2) in spec
    assert "ACTIONS DOUBLES (%d -5.000000 5.000000)" % (n - 1) in spec
    obs = L.env_start().contents
    assert obs.numDoubles == 2 * n + 2 and [obs.doubleArray[i] for i in range(2 * n + 2)] == [0.001] * (2 * n + 2)
    po = _params(O, n)
    rng = np.random.default_rng(n)
    st, saved, acts = np.full(2 * n + 2, 0.001), None, rng.uniform(-MAX_U, MAX_U, (25, n - 1))
    for t in range(20):
        act, _keep = _action(acts[t])
        r = L.env_step(ctypes.byref(act)).contents
        st, want_rew = O.step(po, O.RLGLUE, st, acts[t])
        assert rel_err(_obs(r, n), st) < STEP_TOL and abs(r.reward - want_rew) < STEP_TOL * max(1.0, abs(want_rew))
        assert r.terminal == 0
        if t == 6:
            assert L.env_message(b"save state").decode().startswith("saved_observation")
            saved = st.copy()
    assert L.env_message(b"load state").decode().startswith("this_observation")
    act, _keep = _action(acts[20])
    r = L.env_step(ctypes.byref(act)).contents
    st, _ = O.step(po, O.RLGLUE, saved, acts[20])
    assert rel_err(_obs(r, n), st) < STEP_TOL
    # invalid actions, only with SWM_RLGLUE_NO_ABORT set (without it the shim aborts like the reference)
    monkeypatch.setenv("SWM_RLGLUE_NO_ABORT", "1")
    prev = _obs(r, n)
    for bad in ([MAX_U * 1.1] + [0.0] * (n - 2), [0.0] * n):
        act, _keep = _action(bad)
        r = L.env_step(ctypes.byref(act)).contents
        assert r.terminal == 1 and np.array_equal(_obs(r, n), prev)
    act, _keep = _action(acts[21])
    r = L.env_step(ctypes.byref(act)).contents
    st, _ = O.step(po, O.RLGLUE, st, acts[21])
    assert r.terminal == 0 and rel_err(_obs(r, n), st) < STEP_TOL


def test_env_plugin_refuses_unusable_segment_counts(S, O, shim, tmp_path):
    """"set parameters" keeps the previous n_seg -- and says so -- for an n_seg outside 2..10 or not an integer,
    and for a changed n_seg between env_init and env_cleanup (the buffers are sized for the old chain); the file's
    other parameters still apply.  swm_rlglue_set_params refuses the same changes."""
    L = shim
    f = tmp_path / "parameters.txt"
    for bad in ("11", "1", "2.5", "nan"):
        msg = _set(L, f, _param_file(bad, h=0.02))
        assert msg.startswith("Refused") and "n_seg=3;" in msg and "h_global=0.020000" in msg, msg
    msg = _set(L, f, _param_file(3, h=0.005, max_u=4.0))
    assert "Refused" not in msg
    L.env_init()
    msg = _set(L, f, _param_file(5, h=0.004, max_u=4.0))
    assert msg.startswith("Refused") and "n_seg=3;" in msg and "h_global=0.004000" in msg, msg
    assert "Refused" not in _set(L, f, _param_file(3, h=0.004, max_u=4.0))
    assert L.swm_rlglue_set_params(ctypes.byref(S.make_params(n=5))) == -1  # SWM_ERR_BAD_ARG
    # the environment still steps the chain it was sized for, with the parameters that did apply
    L.env_start()
    po = O.make_params(n=3, l_i=.9, m_i=1.1, k=9.5, h=0.004, max_u=4.0, direction=(.6, .8))
    st = np.full(8, 0.001)
    for a in ([3.5, -2.0], [-1.0, 4.0]):
        act, _keep = _action(a)
        r = L.env_step(ctypes.byref(act)).contents
        st, want = O.step(po, O.RLGLUE, st, a)
        assert r.terminal == 0 and rel_err(_obs(r, 3), st) < STEP_TOL and abs(r.reward - want) < STEP_TOL
    good = S.make_params(n=3, l_i=.9, m_i=1.1, k=9.5, h=0.004, max_u=4.0, direction=(.6, .8))
    assert L.swm_rlglue_set_params(ctypes.byref(good)) == 0
    L.env_cleanup()
    assert "n_seg=5;" in _set(L, f, _param_file(5))
    assert L.swm_rlglue_set_params(ctypes.byref(good)) == 0
