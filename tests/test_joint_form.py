"""The joint-angle form of the gym accelerations (gym_accelerations_joint in csrc/dynamics.cuh, used for chains of up to
kJointFormMaxN segments) against the CPU oracle.

The CPU test restates the formulation in numpy and checks it against the oracle's dense pivoted solve for n = 2..7,
together with the bound the unpivoted LDL^T relies on (every pivot of 1 + 12 K o C is >= 1).  The GPU tests check the
CUDA code of every n that uses the joint form: the accelerations, one step, and 1000-step rollouts stepped state by
state by the oracle, on random states, fast spins (|thd| ~ 300) and increments on the edges of the rotation tiers; and
bench.py's own outputs against a build with the block-tridiagonal form everywhere."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import rand_states, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "safe-exploration-with-simulator-in-rl-algorithms_b200", "csrc")


def joint_max_n():
    src = open(os.path.join(CSRC, "dynamics.cuh")).read()
    return int(re.search(r"#define SWM_JOINT_FORM_MAX_N (\d+)", src).group(1))


JOINT_NS = list(range(2, joint_max_n() + 1))


def tables(n):
    """A[i, q] = [q < i] + 1/2 [q = i] - (n - q - 1/2)/n (segment centres about G), K = A^T A."""
    q = np.arange(n)
    A = (q[None, :] < q[:, None]) + 0.5 * (q[None, :] == q[:, None]) - ((n - q - 0.5) / n)[None, :]
    return A, A.T @ A


def joint_accelerations(p, state, u):
    """The non-dimensional joint-angle form exactly as the kernel evaluates it, with a dense solve."""
    n, l, m, k = p.n, p.l_i, p.m_i, p.k
    A, K = tables(n)
    kappa, m2kappa = k * l / m, -2 * k * l / m
    v, th, thd = np.asarray(state[:2]) / l, state[2::2], state[3::2]
    s, c = np.sin(th), np.cos(th)
    C = np.cos(th[None, :] - th[:, None])                         # C[r, q] = cos(th_q - th_r)
    S = np.sin(th[None, :] - th[:, None])                         # S[r, q] = sin(th_q - th_r)
    vn = -v[0] * s + v[1] * c + (A * C.T * thd[None, :]).sum(1)   # centre velocity along n_i
    F = (6 * A * C.T * vn[:, None]).sum(0)                        # F_r = sum_i 6 A_ir C_ir vn_i
    ut = np.asarray(u) * 12 / (m * l * l)
    tau = kappa * thd
    tau[1:] += ut
    tau[:-1] -= ut
    M = np.eye(n) + 12 * K * C
    thdd = np.linalg.solve(M, tau + m2kappa * F + (12 * K * S * thd[None, :] ** 2).sum(1))
    gdd = m2kappa * l / (2 * n) * np.array([-(vn * s).sum(), (vn * c).sum()])
    return np.concatenate([gdd, thdd]), M


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7])
def test_joint_form_restatement_matches_oracle(O, n):
    rng = np.random.default_rng(n)
    p = O.make_params(n=n, l_i=0.8, m_i=1.2, k=10.2)
    worst = 0.0
    for scale in (3.0, 10.0, 300.0):   # thd ~ N(0, scale^2), angles in [-4, 4]
        for st in rand_states(rng, n, 50, scale):
            u = rng.uniform(-5, 5, n - 1)
            want = np.concatenate(O.accelerations(p, O.GYM, st, u))
            got, M = joint_accelerations(p, st, u)
            worst = max(worst, rel_err(got, want))
            # K o C is PSD (Schur product), so M >= I and every LDL^T pivot is >= 1
            L = np.linalg.cholesky(M)
            assert np.diag(L).min() ** 2 >= 1 - 1e-12
    print("n=%d: largest relative difference %.2e" % (n, worst))
    assert worst < 5e-14, worst


# ---- the CUDA code --------------------------------------------------------------------------------------------------
H_STEP = 1e-3
STEP_TOL = 1e-12


def _states(rng, n, B):
    """Random states, fast spins, and increments h*thd exactly on and beside the 1/32 and 1/8 tier edges."""
    st = rand_states(rng, n, B)
    st[B // 4: B // 2, 3::2] = rng.choice([-1, 1], (B // 2 - B // 4, n)) * rng.uniform(250, 350, (B // 2 - B // 4, n))
    edges = np.array([1 / 32, 1 / 8]) / H_STEP
    k = B // 2
    for j, fac in enumerate((1.0, 1 - 1e-12, 1 + 1e-12, 1 - 1e-6, 1 + 1e-6)):
        for e, edge in enumerate(edges):
            row = k + 2 * j + e
            st[row, 3::2] = rng.uniform(-edge, edge, n)
            st[row, 3 + 2 * rng.integers(n)] = rng.choice([-1, 1]) * edge * fac
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("n", JOINT_NS)
def test_joint_form_step_matches_oracle(S, O, n):
    import torch
    rng = np.random.default_rng(100 + n)
    B = 256
    st = _states(rng, n, B)
    act = rng.uniform(-5, 5, (B, n - 1))
    ps, po = (m.make_params(n=n, l_i=0.9, m_i=1.1, k=9.5, h=H_STEP) for m in (S, O))
    acc = S.ops.accelerations_batched(ps, torch.as_tensor(st).cuda(), torch.as_tensor(act).cuda()).cpu().numpy()
    nxt, rew = S.ops.step_batched(ps, torch.as_tensor(st).cuda(), torch.as_tensor(act).cuda())
    want_nxt, want_rew = O.step_batch(po, O.GYM, st, act)
    for e in range(B):
        want = np.concatenate(O.accelerations(po, O.GYM, st[e], act[e]))
        assert rel_err(acc[e], want) < STEP_TOL, (e, rel_err(acc[e], want))
    assert rel_err(nxt.cpu().numpy(), want_nxt) < STEP_TOL
    assert rel_err(rew.cpu().numpy(), want_rew) < STEP_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("n", JOINT_NS)
def test_joint_form_rollout_matches_oracle_step_by_step(S, O, n):
    """1000-step rollouts of the thread kernel from the same starts: every visited state stepped once by the oracle."""
    import torch
    import test_trig_tiers as tt
    rng = np.random.default_rng(200 + n)
    B, H = 64, 1000
    st = _states(rng, n, B)
    act = rng.uniform(-5, 5, (B, n - 1))
    ps, po = (m.make_params(n=n, l_i=0.9, m_i=1.1, k=9.5, h=H_STEP) for m in (S, O))
    res = S.ops.rollout(ps, H, actions=torch.as_tensor(act).cuda(), init_state=torch.as_tensor(st).cuda(),
                        want_final=True, want_trajectory=True, kernel=S.KERNEL_THREAD)
    traj = res.trajectory.cpu().numpy()
    worst, seen = tt._per_step(st, traj, lambda e, x: O.step(po, O.GYM, x, act[e])[0])
    assert sum(len(x) for x in seen) > B * H // 2
    print("n=%d: largest per-step error %.2e over %d states" % (n, worst, sum(len(x) for x in seen)))


@pytest.mark.gpu
def test_bench_outputs_match_block_tridiagonal_build(O, tmp_path):
    """bench.py --dump-outputs (config[1], n = 3) from this build and from one whose thread kernel uses the
    block-tridiagonal form for every n: the same rollouts to the rollout tolerances."""
    import swimmer_ars_b200 as pkg
    objdir = os.path.join(CSRC, "build")
    alt = tmp_path / "obj"
    shutil.copytree(objdir, alt)
    os.remove(alt / "rollout_n3.o")   # the only object bench.py's config[1] depends on
    lib = tmp_path / "libswimmer_ars_block.so"
    subprocess.run(["make", "-C", CSRC, "OBJDIR=%s" % alt, "OUT=%s" % lib, "EXTRA_NVFLAGS=-DSWM_JOINT_FORM_MAX_N=1"],
                   check=True, stdout=subprocess.DEVNULL)
    outs = {}
    for tag, path in (("joint", pkg._lib.LIB_PATH), ("block", str(lib))):
        d = tmp_path / tag
        env = dict(os.environ, SWM_LIB_PATH=path)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0",
                            "--no-ars", "--no-cpu", "--no-sustained", "--dump-outputs", str(d)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=env)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[tag] = np.load(d / "returns.npy"), np.load(d / "final_state.npy")
    (rj, fj), (rb, fb) = outs["joint"], outs["block"]
    dr = np.abs(rj - rb) / np.maximum(1e-3, np.abs(rb))
    df = np.abs(fj - fb).max(axis=1) / np.maximum(1.0, np.abs(fb).max(axis=1))
    print("joint vs block: returns %.2e, final state %.2e (largest relative differences over %d envs)"
          % (dr.max(), df.max(), len(rb)))
    assert dr.max() < 1e-6
    # A few of the 65,536 rollouts amplify rounding enough to move the final state by more than 1e-8 (the tolerance
    # of the sampled oracle comparison in test_bench_dump.py).  For those, the oracle's own sensitivity bounds the
    # difference: the oracle rollout with the actions scaled by 1 + 1e-14 must move at least 1/100 as far (an error
    # in the algebra moves a rollout by far more than that, and every other rollout is held to 1e-8).
    far = np.flatnonzero(df >= 1e-8)
    assert len(far) <= len(rb) // 1000, len(far)
    if len(far):
        n, H = 3, 1000
        actions = np.random.default_rng(0).uniform(-5, 5, (len(rb), n - 1))[far]   # bench.py's inputs on rank 0
        p = O.make_params(n=n)
        _, f0 = O.rollout_fixed_batch(p, O.GYM, actions, H)
        _, f1 = O.rollout_fixed_batch(p, O.GYM, actions * (1 + 1e-14), H)
        twin = np.abs(f1 - f0).max(axis=1) / np.maximum(1.0, np.abs(f0).max(axis=1))
        print("%d envs beyond 1e-8; their oracle twins differ by %s" % (len(far), np.array2string(twin, precision=2)))
        assert (df[far] <= 100 * twin).all(), (df[far], twin)
