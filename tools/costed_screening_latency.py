"""Latency of one graph-replayed Safe_ARS iteration with per-step screening, by cost and kernel.

The engine is built like bench.py's "safe_ars per-step screening" entry: 256 directions (512 rollouts), H = 1000,
the config[3] real and simulator models, sim_thresh 50, real_thresh 51, true top-b, use_graph=True.  Cases, at n = 3
and n = 5:
  (a) built-in cost max_i |thd_i|, kernel AUTO (the two-warp lane kernel at this size)
  (b) built-in cost, one thread per environment (KERNEL_THREAD)
  (c) MaxAffineCost with the built-in rows +-e_{3+2i} (2n forms; swm_rollout_costed, one thread per environment)
  (d) MaxAffineCost bending limits |th_i - th_{i+1}| <= 50 (2(n-1) forms)
Each case: 5 warm-up iterations (the first eager, the second captures the graph), then CUDA events around `iters`
replays, repeated `reps` times, cases interleaved; the median of the per-rep means is reported.

usage: python tools/costed_screening_latency.py [--iters 20] [--reps 5] [--out profiles/r04_costed_screening.txt]
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


def builtin_rows(n):
    A = np.zeros((2 * n, 2 * n + 2))
    for i in range(n):
        A[2 * i, 3 + 2 * i], A[2 * i + 1, 3 + 2 * i] = 1.0, -1.0
    return S.MaxAffineCost(A)


def bending_rows(n):
    A = np.zeros((2 * (n - 1), 2 * n + 2))
    for i in range(n - 1):
        A[2 * i, 2 + 2 * i], A[2 * i, 4 + 2 * i] = 1.0, -1.0
        A[2 * i + 1] = -A[2 * i]
    return S.MaxAffineCost(A)


def engine(n, kernel, cost):
    real = S.make_params(n=n, l_i=0.8, m_i=1.2, k=10.2)
    sim = S.make_params(n=n, l_i=0.8006, m_i=1.2006, k=10.2006)
    screen = dict(sim_params=sim, sim_thresh=50.0, real_thresh=51.0)
    if cost is not None:
        screen["cost"] = cost
    eng = S.ArsEngine(real, N=256, b=256, alpha=0.0075, nu=0.01, H=1000, semantics=S.ARS_TOPB, seed=3,
                      distributed=False, use_graph=True, step_screen=screen, rollout_kernel=kernel)
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_costed_screening.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# tools/costed_screening_latency.py --iters %d --reps %d" % (args.iters, args.reps),
             "# GPU: %s (name, power limit, max SM clock; nvidia-smi, same run)" % (q[0] if q else "unknown"),
             "# one graph-replayed ArsEngine iteration: 256 directions (512 rollouts), H = 1000, per-step screening;",
             "# CUDA events around %d replays, median over %d interleaved reps" % (args.iters, args.reps),
             "%-3s %-46s %-8s %10s %10s %10s" % ("n", "case", "kernel", "ms/iter", "min", "max")]
    for n in (3, 5):
        cases = [("(a) built-in cost, AUTO", S.KERNEL_AUTO, None),
                 ("(b) built-in cost, THREAD", S.KERNEL_THREAD, None),
                 ("(c) MaxAffineCost, built-in rows (%d forms)" % (2 * n), S.KERNEL_AUTO, builtin_rows(n)),
                 ("(d) MaxAffineCost, bending limits (%d forms)" % (2 * (n - 1)), S.KERNEL_AUTO, bending_rows(n))]
        engs = [engine(n, k, c) for _, k, c in cases]
        kernels = []
        for (_, k, c), eng in zip(cases, engs):
            kernels.append("thread" if c is not None else
                           S.ops.rollout_kernel_choice(eng.params, 512, rollouts_per_policy=1, kernel=k))
        times = [[] for _ in cases]
        for _ in range(args.reps):
            for i, eng in enumerate(engs):
                times[i].append(time_ms(eng, args.iters))
        for (name, _, _), kern, t in zip(cases, kernels, times):
            lines.append("%-3d %-46s %-8s %10.4f %10.4f %10.4f" % (n, name, kern, np.median(t), min(t), max(t)))
        del engs
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
