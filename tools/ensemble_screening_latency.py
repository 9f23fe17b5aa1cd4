"""Latency of one graph-replayed Safe_ARS iteration with per-step screening by an ensemble of M simulator models.

The engine is built like bench.py's "safe_ars per-step screening" entry (and tools/costed_screening_latency.py):
256 directions (512 rollouts), H = 1000, the config[3] real model, sim_thresh 50, real_thresh 51, true top-b,
use_graph=True, kernel THREAD.  The ensemble's models are the config[3] simulator and models spread around it by up
to +-0.1 % in l, m, k (ensemble of M = its first M).  Cases, at n = 3 and n = 5:
  single model, built-in cost (swm_rollout, THREAD)           -- the reference for M = 1
  single model, bending limits |th_i - th_{i+1}| <= 50 (swm_rollout_costed)
  ensemble, built-in cost, M = 1, 2, 4, 7, 16 (swm_rollout_ensemble)
  ensemble, bending limits, M = 1, 2, 4, 7, 16
Each case: 5 warm-up iterations (the first eager, the second captures the graph), then CUDA events around `iters`
replays, repeated `reps` times, cases interleaved; the median of the per-rep means is reported, with its ratio to the
single-model case of the same cost.

usage: python tools/ensemble_screening_latency.py [--iters 20] [--reps 5] [--out profiles/r05_ensemble_screening.txt]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import swimmer_ars_b200 as S  # noqa: E402

MS = (1, 2, 4, 7, 16)


def bending_rows(n):
    A = np.zeros((2 * (n - 1), 2 * n + 2))
    for i in range(n - 1):
        A[2 * i, 2 + 2 * i], A[2 * i, 4 + 2 * i] = 1.0, -1.0
        A[2 * i + 1] = -A[2 * i]
    return S.MaxAffineCost(A)


def models(n):
    rng = np.random.default_rng(5)
    out = [S.make_params(n=n, l_i=0.8006, m_i=1.2006, k=10.2006)]
    for _ in range(max(MS) - 1):
        f = 1.0 + rng.uniform(-1e-3, 1e-3, 3)
        out.append(S.make_params(n=n, l_i=0.8006 * f[0], m_i=1.2006 * f[1], k=10.2006 * f[2]))
    return out


def engine(n, sim, cost):
    real = S.make_params(n=n, l_i=0.8, m_i=1.2, k=10.2)
    screen = dict(sim_params=sim, sim_thresh=50.0, real_thresh=51.0)
    if cost is not None:
        screen["cost"] = cost
    eng = S.ArsEngine(real, N=256, b=256, alpha=0.0075, nu=0.01, H=1000, semantics=S.ARS_TOPB, seed=3,
                      distributed=False, use_graph=True, step_screen=screen, rollout_kernel=S.KERNEL_THREAD)
    for _ in range(5):
        eng.run_iteration()
    torch.cuda.synchronize()
    assert eng._graph is not None
    return eng


def time_ms(eng, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        eng.run_iteration()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_ensemble_screening.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# tools/ensemble_screening_latency.py --iters %d --reps %d" % (args.iters, args.reps),
             "# GPU: %s (name, power limit, max SM clock; nvidia-smi, same run)" % (q[0] if q else "unknown"),
             "# one graph-replayed ArsEngine iteration: 256 directions (512 rollouts), H = 1000, per-step screening,",
             "# one thread per environment; CUDA events around %d replays, median over %d interleaved reps;" % (
                 args.iters, args.reps),
             "# ratio = this case / the single-model case of the same cost",
             "%-3s %-40s %10s %10s %10s %7s" % ("n", "case", "ms/iter", "min", "max", "ratio")]
    for n in (3, 5):
        sims = models(n)
        cases = [("single model, built-in cost", sims[0], None, "b"),
                 ("single model, bending limits", sims[0], bending_rows(n), "a")]
        cases += [("ensemble M=%d, built-in cost" % M, sims[:M], None, "b") for M in MS]
        cases += [("ensemble M=%d, bending limits" % M, sims[:M], bending_rows(n), "a") for M in MS]
        engs = [engine(n, sim, cost) for _, sim, cost, _ in cases]
        times = [[] for _ in cases]
        for _ in range(args.reps):
            for i, eng in enumerate(engs):
                times[i].append(time_ms(eng, args.iters))
        med = [float(np.median(t)) for t in times]
        base = {"b": med[0], "a": med[1]}
        for (name, _, _, c), t, m in zip(cases, times, med):
            lines.append("%-3d %-40s %10.4f %10.4f %10.4f %7.2f" % (n, name, m, min(t), max(t), m / base[c]))
        del engs
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
