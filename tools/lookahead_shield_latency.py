"""Latency of one graph-replayed Safe_ARS iteration with a lookahead shield (swm_rollout_lookahead).

The engine is tools/shield_screening_latency.py's: 256 directions (512 rollouts), H = 1000, the config[3] real model,
true top-b, use_graph=True, kernel THREAD, thresholds at which screening rejects steps (built-in cost: sim_thresh 1.0,
real_thresh 1.2; bending limits |th_i - th_{i+1}|: 0.6 / 0.7), the first M of tools/ensemble_screening_latency.py's
models.  Cases, at n = 3 and 5, M = 1 and 4, both costs, the zero and the damping backup, and lookaheads
K = 0 (swm_rollout_shielded, the reference), 1, 4, 16 and 64.
Reported per case: ms per iteration (CUDA events around `iters` replays, median over `reps` interleaved reps), its
ratio to K = 0 with the same n, M, cost and backup, the fraction of real steps that took the backup and the fraction
of rollouts that froze (from the last replay).  A rollout that used to freeze now runs on, so an iteration can get
slower because its rollouts get longer as well as because each judgement costs more.

usage: python tools/lookahead_shield_latency.py [--iters 10] [--reps 5] [--lookaheads 0,1,4,16,64]
                                                [--out profiles/r08_lookahead_shield.txt]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import swimmer_ars_b200 as S  # noqa: E402
from ensemble_screening_latency import bending_rows, models  # noqa: E402

H = 1000


def backup(kind, n):
    W = np.zeros((n - 1, 2 * n + 2))
    if kind == "damping":
        for k in range(n - 1):
            W[k, 3 + 2 * k], W[k, 5 + 2 * k] = -0.5, 0.5
    return dict(policy=W, action=None)


def engine(n, sims, cost, bk, K):
    real = S.make_params(n=n, l_i=0.8, m_i=1.2, k=10.2)
    thr = (1.0, 1.2) if cost is None else (0.6, 0.7)
    screen = dict(sim_params=sims, sim_thresh=thr[0], real_thresh=thr[1])
    if cost is not None:
        screen["cost"] = cost
    screen["backup"] = bk
    if K > 0:
        screen["lookahead"] = K
    eng = S.ArsEngine(real, N=256, b=256, alpha=0.0075, nu=0.01, H=H, semantics=S.ARS_TOPB, seed=3,
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
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lookaheads", default="0,1,4,16,64")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_lookahead_shield.txt"))
    args = ap.parse_args()
    ks = [int(k) for k in args.lookaheads.split(",")]
    assert ks[0] == 0, "the first lookahead is the reference, K = 0"
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# tools/lookahead_shield_latency.py --iters %d --reps %d --lookaheads %s" % (args.iters, args.reps,
                                                                                         args.lookaheads),
             "# library: %s" % S._lib.LIB_PATH.replace(ROOT + os.sep, ""),
             "# GPU: %s (name, power limit, max SM clock; nvidia-smi, same run)" % (q[0] if q else "unknown"),
             "# one graph-replayed ArsEngine iteration: 256 directions (512 rollouts), H = 1000, per-step screening,",
             "# one thread per environment; CUDA events around %d replays, median over %d interleaved reps;" % (
                 args.iters, args.reps),
             "# ratio = this case / K = 0 with the same n, M, cost and backup; backup = fraction of real steps that took",
             "# the backup; frozen = fraction of rollouts that froze (last replay)",
             "%-3s %-3s %-15s %-8s %4s %10s %7s %8s %8s" % ("n", "M", "cost", "backup", "K", "ms/iter", "ratio",
                                                            "backup", "frozen")]
    for n in (3, 5):
        sims = models(n)
        cases = [(M, cname, cost, bname, K) for M in (1, 4) for cname, cost in (("built-in", None),
                                                                               ("bending limits", bending_rows(n)))
                 for bname in ("zero", "damping") for K in ks]
        engs = [engine(n, sims[:M], cost, backup(b, n), K) for M, _, cost, b, K in cases]
        times = [[] for _ in cases]
        for _ in range(args.reps):
            for i, eng in enumerate(engs):
                times[i].append(time_ms(eng, args.iters))
        med = [float(np.median(t)) for t in times]
        for i, ((M, cname, _, bname, K), eng) in enumerate(zip(cases, engs)):
            last = eng.last
            over = float(last.overrides.sum()) / (last.overrides.numel() * H)
            frozen = float((last.frozen_at < H).float().mean())
            base = med[i - ks.index(K)]
            lines.append("%-3d %-3d %-15s %-8s %4d %10.4f %7.2f %8.4f %8.4f" % (n, M, cname, bname, K, med[i],
                                                                              med[i] / base, over, frozen))
        del engs
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
