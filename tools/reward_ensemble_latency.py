"""Latency of one graph-replayed reward-constraint safe-exploration ARS iteration whose directions are screened by an
ensemble of M simulator models (ArsEngine(sim_params=[...]): M x 512 simulator rollouts in one launch, then the mask
over all models).

The engine is built like bench.py's config[3]: V1, 256 directions, H = 1000, ARSAgent semantics, real (l, m, k) =
(0.8, 1.2, 10.2), W0 pre-trained by 40 plain iterations from zero, and a threshold taken from a probe iteration (median
of min(r+_sim, r-_sim) under bench's simulator).  Model 0 is bench's simulator, real + 1e-3 u/|u|; every other model
is real + 1e-3 u_m/|u_m| with its own u_m.  Cases, at n = 3 and n = 5:
  single model (sim_params=p: swm_rollout + swm_screen_mask)  -- the reference
  M = 1, 2, 4, 8, 16 (sim_params=[p_0 .. p_{M-1}])
each with `speculate` (real rollouts beside the screening on a second stream, the engine default) and screen-first.
The simulator kernel is the one AUTO picks for M x 512 environments.  Each case: 5 warm-up iterations (the first
eager, the second captures the graph), then CUDA events around `iters` replays, repeated `reps` times, cases
interleaved; the median of the per-rep means is reported, with its ratio to the single-model case of the same
schedule.

usage: python tools/reward_ensemble_latency.py [--iters 20] [--reps 5] [--out profiles/r06_reward_ensemble_screening.txt]
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

MS = (1, 2, 4, 8, 16)
EPS = 1e-3


def models(n):
    """bench.py's simulator, then models at the same distance EPS from the real model in independent directions."""
    out = []
    for m in range(max(MS)):
        u = np.random.default_rng(7 if m == 0 else 1000 + m).normal(size=3)
        u /= np.linalg.norm(u)
        out.append(S.make_params(n=n, m_i=1.2 + EPS * u[0], l_i=0.8 + EPS * u[1], k=10.2 + EPS * u[2]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_reward_ensemble_screening.txt"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    lines = ["# tools/reward_ensemble_latency.py --iters %d --reps %d" % (args.iters, args.reps),
             "# GPU: %s (name, power limit, max SM clock; nvidia-smi, same run)" % (q[0] if q else "unknown"),
             "# one graph-replayed ArsEngine iteration of bench.py's config[3] (V1, 256 directions, H = 1000) screened by",
             "# M simulator models; CUDA events around %d replays, median over %d interleaved reps;" % (args.iters,
                                                                                                     args.reps),
             "# ratio = this case / the single-model case of the same schedule; kernel = AUTO's choice for M x 512 envs",
             "%-3s %-14s %-12s %-7s %10s %10s %10s %7s %9s" % ("n", "case", "schedule", "kernel", "ms/iter", "min", "max",
                                                           "ratio", "screened")]
    for n in (3, 5):
        real = S.make_params(n=n, l_i=0.8, m_i=1.2, k=10.2)
        sims = models(n)
        base = dict(N=256, b=256, alpha=0.0075, nu=0.01, H=1000, v2=False, semantics=S.ARS_AGENT)
        pre = S.ArsEngine(real, seed=11, distributed=False, use_graph=True, **base)
        for _ in range(40):
            pre.run_iteration()
        W0 = pre.W.clone()
        probe = S.ArsEngine(real, seed=12, distributed=False, sim_params=sims[0], sim_threshold=-1e300,
                            initial_policy=W0, **base)
        probe.run_iteration(update=False)
        thr = float(torch.quantile(probe.sim_returns.view(256, 2).min(dim=1).values, 0.5).cpu())
        del pre, probe
        cases = [("single", sims[0], "-")] + [("M=%d" % M, sims[:M], S.ops.rollout_kernel_choice(sims[0], 512 * M))
                                              for M in MS]
        engs, meta = [], []
        for name, sim, kern in cases:
            for spec in (True, False):
                eng = S.ArsEngine(real, seed=12, distributed=False, sim_params=sim, sim_threshold=thr, initial_policy=W0,
                                  use_graph=True, speculate=spec, **base)
                for _ in range(5):
                    eng.run_iteration()
                torch.cuda.synchronize()
                assert eng._graph is not None
                engs.append(eng)
                meta.append((name, "speculative" if spec else "screen-first", kern))
        times = [[] for _ in engs]
        passed = [0 for _ in engs]
        for _ in range(args.reps):
            for i, eng in enumerate(engs):
                p0 = int(eng.n_pass_total.item())
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.iters):
                    eng.run_iteration()
                b.record()
                b.synchronize()
                times[i].append(a.elapsed_time(b) / args.iters)
                passed[i] += int(eng.n_pass_total.item()) - p0
        med = [float(np.median(t)) for t in times]
        ref = {"speculative": med[0], "screen-first": med[1]}
        for (name, sched, kern), t, m, p in zip(meta, times, med, passed):
            screened = 1.0 - p / (256.0 * args.iters * args.reps)
            lines.append("%-3d %-14s %-12s %-7s %10.4f %10.4f %10.4f %7.2f %9.3f" % (
                n, name, sched, kern, m, min(t), max(t), m / ref[sched], screened))
        del engs
    text = "\n".join(lines) + "\n"
    print(text)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)


if __name__ == "__main__":
    main()
