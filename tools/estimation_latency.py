"""Latency of simulator-model estimation on the device; prints one JSON line.

  objective: time per CMA-ES generation of the prediction-error objective for lambda candidates over K recorded
             trajectories of H = 1000 observations (n = 3 and 5): the fused kernel (swm_prediction_error) against
             the per-trajectory loop it replaces (swm_policy_actions + swm_step_batched_models in chunks of 24
             models + torch norms and sums, the former Estimator.I_population).  CUDA events around `reps`
             back-to-back evaluations after warm-up; both arms include their host enqueue, which is what a
             generation costs.  max_rel_diff compares the two arms' values (different summation orders).
  estimate:  wall time (host clock, ending in the status read that synchronises) and generation count of whole
             Estimator.estimate_on_device runs at the reference settings (K = 1, lambda = 7, n = 3), graph
             capture included.

The card's name and power limit are read in the same run."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import swimmer_ars_b200 as S

REAL = dict(m_i=1.2, l_i=0.8, k=10.2)
H = 1000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, check=True)
        name, power = [s.strip() for s in out.stdout.strip().splitlines()[0].split(",")]
        return name, float(power)
    except (OSError, subprocess.CalledProcessError, ValueError):
        return torch.cuda.get_device_name(), None


def record(n, K, seed):
    """K trajectories [K, H, 2n+2] of the real model under random V1 policies (rollout kernel output)."""
    rng = np.random.default_rng(seed)
    pols = torch.as_tensor(rng.uniform(-1, 1, (K, n - 1, 2 * n + 2)) * 0.5).cuda()
    res = S.ops.rollout(S.make_params(n=n, **REAL), H, policies=pols, want_trajectory=True)
    return res.trajectory.transpose(0, 1).contiguous(), pols.reshape(K, -1).contiguous()


def old_objective(plist, trajs, pols):
    M = len(plist)
    total = torch.zeros(M, dtype=torch.float64, device=trajs.device)
    for k in range(trajs.shape[0]):
        s = trajs[k, :-1]
        act = S.ops.policy_actions(plist[0], s, pols[k].reshape(1, -1), rollouts_per_policy=s.shape[0])
        nxt, _ = S.ops.step_batched_models(plist, s.unsqueeze(0).expand(M, -1, -1).contiguous(),
                                           act.unsqueeze(0).expand(M, -1, -1).contiguous())
        total = total + torch.linalg.norm(nxt - trajs[k, 1:].unsqueeze(0), dim=2).sum(dim=1)
    return total


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def objective_rows():
    rows = []
    for n in (3, 5):
        for K in (1, 16, 256):
            trajs, pols = record(n, K, seed=100 * n + K)
            for lam in (7, 64, 256):
                rng = np.random.default_rng(lam)
                x = np.array([REAL["m_i"], REAL["l_i"], REAL["k"]]) * (1 + rng.uniform(-0.1, 0.1, (lam, 3)))
                cand = torch.as_tensor(x).cuda()
                data = S.ops.EstimateData(trajs, pols, ("m_i", "l_i", "k"), max_candidates=lam)
                base = S.make_params(n=n)
                err = torch.empty(lam, dtype=torch.float64, device="cuda")
                plist = [S.make_params(n=n, m_i=a, l_i=b, k=c) for a, b, c in x]
                new_ms, new = timed(lambda: S.ops.prediction_error(base, data, cand, out=err), 3, 50)
                reps = 20 if K * lam <= 1024 else 5
                old_ms, old = timed(lambda: old_objective(plist, trajs, pols), 2, reps)
                diff = float(torch.max(torch.abs(new - old) / torch.abs(old)))
                rows.append(dict(n=n, K=K, H=H, lam=lam, new_ms=round(new_ms, 4), old_ms=round(old_ms, 4),
                                 speedup=round(old_ms / new_ms, 1), max_rel_diff=diff))
    return rows


def estimate_rows():
    n = 3
    trajs, pols = record(n, 1, seed=7)
    db = S.Database()
    db.add_trajectory(trajs[0].cpu().numpy(), pols[0].reshape(n - 1, -1).cpu().numpy())
    guess = S.EnvParam("sim", n=n, H=H, m_i=1.0, l_i=1.0, h=0.001, k=10.0, epsilon=0.01)
    est = S.Estimator(db, guess, capacity=1)
    est.estimate_on_device(seed=0)  # warm-up: module load, first capture
    rows = []
    for seed in (0, 1, 2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p, info = est.estimate_on_device(seed=seed)
        wall = time.perf_counter() - t0
        rel = max(abs(getattr(p, k) - REAL[k]) / REAL[k] for k in REAL)
        rows.append(dict(seed=seed, wall_ms=round(1e3 * wall, 2), generations=info["generations"],
                         evaluations=info["evaluations"], stop=info["stop"], f=info["f"], max_rel_param_err=rel))
    return rows


def main():
    if not torch.cuda.is_available():
        raise SystemExit("estimation_latency.py measures the GPU: no CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    print(json.dumps(dict(card=name, power_limit_w=power, objective=objective_rows(), estimate=estimate_rows())))


if __name__ == "__main__":
    main()
