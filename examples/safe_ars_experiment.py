"""safe_ars/experiment.py of the reference with only the imports changed (no matplotlib): unsafe ARS vs ARS
with per-step state-constraint safe exploration on the 3-segment swimmer, several random seeds; the
per-step costs are computed on the device from the returned states instead of a Python double loop.

    python examples/safe_ars_experiment.py --epsilon 0.01 --thresh 6 --n_iter 20 --n_rollout 500 \
        --N 1 --b 1 --alpha 0.0075 --nu 0.01 --n_seeds 2 --path results/safe_ars/
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from swimmer_ars_b200 import Basic_ARS, Safe_ARS, SwimmerEnv  # reference: safe_ars.ars, envs.gym_swimmer...

parser = argparse.ArgumentParser()
parser.add_argument("--epsilon", help="precision of parameter estimation", type=float, default=0.01)
parser.add_argument("--thresh", help="safety threshold: the state cost should never be higher than this threshold",
                    type=float, default=6.0)
parser.add_argument("--n_iter", help="number of ARS training iterations", type=int, default=20)
parser.add_argument("--n_rollout", help="length of one rollout for ARS training", type=int, default=500)
parser.add_argument("--N", help="number of policy perturbations sampled", type=int, default=1)
parser.add_argument("--b", help="number of pertubations used for policy update", type=int, default=1)
parser.add_argument("--alpha", help="step size", type=float, default=0.0075)
parser.add_argument("--nu", help="perturbations standard deviation", type=float, default=0.01)
parser.add_argument("--path", help="directory for saving the results", type=str, default="results/safe_ars/")
parser.add_argument("--n_seeds", help="number of random seeds", type=int, default=2)
parser.add_argument("--backup", help="shield: the action tried when the simulator rejects a step (none: freeze, as the "
                    "reference; zero: zero torque; damping: torque damping the joint velocities)",
                    choices=["none", "zero", "damping"], default="none")
args = parser.parse_args()

n = 3
theta_real = [1., 1., 10.]
real_env = SwimmerEnv("RealWorld", n=3, m_i=theta_real[0], l_i=theta_real[1], k=theta_real[2])
delta = np.random.rand(len(theta_real))
theta_sim = theta_real + delta / np.linalg.norm(delta, ord=2) * args.epsilon
print(f"Real world parameter: {theta_real}\nEstimated parameter: {theta_sim}")
sim_env = SwimmerEnv("Simulator", n=3, m_i=theta_sim[0], l_i=theta_sim[1], k=theta_sim[2])

# cost of safe_ars/experiment.py:44 (the kernel's built-in cost; any callable computing the same is accepted)
cost = lambda x: np.max([abs(x[3 + 2 * i]) for i in range(n)])  # noqa: E731


backup = {}
if args.backup != "none":
    W_b = np.zeros((n - 1, 2 * n + 2))
    if args.backup == "damping":  # torque_k = -0.5 (theta_dot_k - theta_dot_{k+1})
        for k in range(n - 1):
            W_b[k, 3 + 2 * k], W_b[k, 5 + 2 * k] = -0.5, 0.5
    backup = dict(backup_policy=W_b)


def experience(seed):
    unsafe_agent = Basic_ARS()
    sim_thresh = args.thresh - 1
    safe_agent = Safe_ARS(cost, args.thresh, sim_thresh, sim_env, **backup)
    np.random.seed(seed)
    unsafe_returns, unsafe_states = unsafe_agent.train(args.n_iter, real_env, args.N, args.b, args.alpha, args.nu,
                                                       args.n_rollout)
    np.random.seed(seed)
    safe_returns, safe_states = safe_agent.train(args.n_iter, real_env, args.N, args.b, args.alpha, args.nu,
                                                 args.n_rollout)
    return unsafe_returns, unsafe_states, safe_returns, safe_states


all_unsafe_returns, all_unsafe_costs, all_safe_returns, all_safe_costs = [], [], [], []
for i in range(args.n_seeds):
    seed = np.random.randint(2 ** 32 - 1)
    print(f"\n------------Experience {i}/{args.n_seeds} with random seed {seed}------------\n")
    unsafe_returns, unsafe_states, safe_returns, safe_states = experience(seed)
    # states[2N n_iter, H, 2n+2] -> per-step cost max_i |theta_dot_i|
    unsafe_costs = np.abs(unsafe_states[:, :, 3::2]).max(axis=2).reshape(-1)
    safe_costs = np.abs(safe_states[:, :, 3::2]).max(axis=2).reshape(-1)
    all_unsafe_returns.append(unsafe_returns)
    all_safe_returns.append(safe_returns)
    all_unsafe_costs.append(unsafe_costs)
    all_safe_costs.append(safe_costs)

os.makedirs(args.path, exist_ok=True)
out = os.path.join(args.path, f"safe_ars_eps={args.epsilon}_thresh={args.thresh}.npz")
np.savez(out, unsafe_returns=np.array(all_unsafe_returns), safe_returns=np.array(all_safe_returns),
         unsafe_costs=np.array(all_unsafe_costs), safe_costs=np.array(all_safe_costs))
print(f"max per-step cost: unsafe {np.max(all_unsafe_costs):.4g}, safe {np.max(all_safe_costs):.4g} "
      f"(threshold {args.thresh}); saved {out}")
