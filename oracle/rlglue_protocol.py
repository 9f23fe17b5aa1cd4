"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

In-process emulation of the four-process RL-Glue experiment of the reference, so that the UNMODIFIED
agent (rlglue/agent/SwimmerAgent.py, loaded from the reference tree) can be driven against the UNMODIFIED
C++ swimmer (rlglue/environment/SwimmerEnvironment.cpp compiled in place -> oracle/_ref) exactly the way
rlglue/experiment/SwimmerExperiment.cpp:65-100 drives them through the RL-Glue runtime:

  RL_init   = env_init (task-spec string, cpp:30) -> agent_init(task_spec)
  RL_start  = env_start (all entries 0.001 + save_state, cpp:39-44) -> agent_start(obs) -> action
  RL_step   = env_step(last action) (updateState + reward = Gdot . direction, cpp:52-68)
              -> agent_step(reward, obs) -> next action
  messages  = "set parameters", "(un)freeze training", "load state", "get total_reward"

RL-Glue 3.04 and its Python codec are not installed (SURVEY 8c); they are transport only (no
arithmetic), so tiny stand-ins for the four modules the agent imports are injected:
  rlglue.agent.Agent.Agent            base class
  rlglue.agent.AgentLoader            loadAgent (only used under __main__)
  rlglue.types.Action / Observation   numDoubles + doubleArray containers
  rlglue.utils.TaskSpecVRLGLUE3       TaskSpecParser: .valid, getDoubleActions(), getDoubleObservations()
Also provides `restated_protocol`, the same step-level loop over the C restatement (oracle_lib),
which the tests pin against the fixture this module generates (tests/golden/rlglue_agent.npz).
"""
import contextlib
import importlib.util
import io
import os
import re
import sys
import tempfile
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("SWIMMER_REFERENCE_ROOT", "/root/reference")


def _install_rlglue_stubs():
    if "rlglue" in sys.modules and getattr(sys.modules["rlglue"], "_swimmer_stub", False):
        return
    rlglue = types.ModuleType("rlglue"); rlglue._swimmer_stub = True; rlglue.__path__ = []
    agent_pkg = types.ModuleType("rlglue.agent"); agent_pkg.__path__ = []
    agent_mod = types.ModuleType("rlglue.agent.Agent")

    class Agent:
        pass
    agent_mod.Agent = Agent
    loader = types.ModuleType("rlglue.agent.AgentLoader")
    loader.loadAgent = lambda agent: None
    types_mod = types.ModuleType("rlglue.types")

    class _Abstract:
        def __init__(self, numInts=None, numDoubles=None, numChars=None):
            self.intArray = [0] * (numInts or 0)
            self.doubleArray = [0.0] * (numDoubles or 0)
            self.charArray = [""] * (numChars or 0)

    class Action(_Abstract):
        pass

    class Observation(_Abstract):
        pass
    types_mod.Action, types_mod.Observation = Action, Observation
    utils = types.ModuleType("rlglue.utils"); utils.__path__ = []
    ts = types.ModuleType("rlglue.utils.TaskSpecVRLGLUE3")

    class TaskSpecParser:
        """The subset of the RL-Glue 3 task-spec grammar SwimmerEnvironment.cpp:30 emits:
        `OBSERVATIONS DOUBLES (n lo hi) ACTIONS DOUBLES (n lo hi)`; a leading count repeats the range."""

        def __init__(self, spec):
            s = spec.decode() if isinstance(spec, bytes) else spec
            self.valid = s.startswith("VERSION RL-Glue-3.0")
            self._obs = self._ranges(re.search(r"OBSERVATIONS DOUBLES \(([^)]*)\)", s))
            self._act = self._ranges(re.search(r"ACTIONS DOUBLES \(([^)]*)\)", s))

        @staticmethod
        def _ranges(m):
            tok = m.group(1).split()
            n = int(tok[0]) if len(tok) == 3 else 1
            lo, hi = tok[-2], tok[-1]
            conv = lambda x: x if x == "UNSPEC" else float(x)
            return [[conv(lo), conv(hi)] for _ in range(n)]

        def getDoubleActions(self):
            return self._act

        def getDoubleObservations(self):
            return self._obs
    ts.TaskSpecParser = TaskSpecParser
    rlglue.agent, rlglue.types, rlglue.utils = agent_pkg, types_mod, utils
    agent_pkg.Agent, agent_pkg.AgentLoader = agent_mod, loader
    utils.TaskSpecVRLGLUE3 = ts
    sys.modules.update({"rlglue": rlglue, "rlglue.agent": agent_pkg, "rlglue.agent.Agent": agent_mod,
                        "rlglue.agent.AgentLoader": loader, "rlglue.types": types_mod, "rlglue.utils": utils,
                        "rlglue.utils.TaskSpecVRLGLUE3": ts})


def load_agent_class():
    """The reference's SwimmerARSAgent class, loaded unmodified."""
    _install_rlglue_stubs()
    path = os.path.join(REFERENCE_ROOT, "rlglue", "agent", "SwimmerAgent.py")
    spec = importlib.util.spec_from_file_location("reference_rlglue_swimmer_agent", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.SwimmerARSAgent


def task_spec(n, max_u):
    """SwimmerEnvironment.cpp:30 (std::to_string prints six decimals)."""
    return ("VERSION RL-Glue-3.0 PROBLEMTYPE continuing DISCOUNTFACTOR 0.9 OBSERVATIONS DOUBLES (%d UNSPEC UNSPEC) "
            "ACTIONS DOUBLES (%d %f %f) REWARDS (UNSPEC UNSPEC) EXTRA SwimmerEnvironment(C++) by Leon Zheng"
            % (2 * n + 2, n - 1, -max_u, max_u))


def run_reference_protocol(par, n_it, seed):
    """Runs SwimmerExperiment.cpp's run_training for n_it iterations with the unmodified agent and the
    compiled reference environment.  par: dict with the keys of rlglue/parameters.txt.
    -> dict(results[n_it] = evaluation returns, policies[n_it+1], deltas[n_it+1, N, n-1, 2n+2] (the U[0,1)
    draws the agent made), rewards[n_it, 2N] (the agent's reward table at each update))."""
    from oracle import oracle_lib as O
    Agent = load_agent_class()               # installs the rlglue stand-ins
    from rlglue.types import Observation
    assert O.ref_cpp() is not None, "oracle/_ref/libref_swimmer.so missing: make -C oracle ref"
    n, N, H = int(par["n_seg"]), int(par["N"]), int(par["H"])
    p = O.make_params(n=n, l_i=par["l_i"], m_i=par["m_i"], k=par["k"], h=par["h_global"], max_u=par["max_u"],
                      direction=tuple(par["direction"]))
    O.ref_cpp_set_params(p)
    direction = np.array(par["direction"], dtype=np.float64)
    agent = Agent()
    cwd = os.getcwd()
    out = {"results": [], "policies": [], "deltas": [], "rewards": []}
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "run"))
        with open(os.path.join(td, "parameters.txt"), "w") as f:      # agent reads ../parameters.txt (:243-257)
            for key in ("n_seg", "h_global", "N", "b", "H", "alpha", "nu", "max_u", "l_i", "k", "m_i"):
                f.write("%s %s\n" % (key, par[key]))
            f.write("direction %s %s\n" % tuple(par["direction"]))
        os.chdir(os.path.join(td, "run"))
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                np.random.seed(seed)
                agent.agent_message(b"set parameters")                  # setParameters(), cpp:40-46
                agent.agent_init(task_spec(n, par["max_u"]).encode())    # RL_init
                state = np.full(2 * n + 2, 0.001)                        # env_start, cpp:39-44
                saved = state.copy()

                def obs_of(s):
                    o = Observation(numDoubles=s.size)
                    o.doubleArray = s.tolist()
                    return o

                def rl_step(state, action):
                    a = np.asarray(action.doubleArray, dtype=np.float64)
                    assert np.all(np.abs(a) <= par["max_u"])             # env_step asserts, cpp:56-58
                    state = O.ref_cpp_step(state, a)                     # unmodified updateState
                    reward = float(state[0] * direction[0] + state[1] * direction[1])
                    return state, agent.agent_step(reward, obs_of(state))
                action = agent.agent_start(obs_of(state))                # RL_start
                out["policies"].append(np.array(agent.agentPolicy, copy=True))
                for it in range(n_it):                                   # runOneTrainingIteration, cpp:65-84
                    out["deltas"].append(np.array(agent.deltas, copy=True))
                    agent.agent_message(b"unfreeze training")
                    table = None
                    for i in range(2 * H * N):
                        if i % H == 0:
                            state = saved.copy()                         # RL_env_message("load state")
                        if i == 2 * H * N - 1:
                            # the update happens inside this agent_step; capture the reward table it will use
                            table = list(agent.rewards)
                        state, action = rl_step(state, action)
                    out["rewards"].append(np.array(table))
                    agent.agent_message(b"freeze training")
                    state = saved.copy()
                    for i in range(H):
                        state, action = rl_step(state, action)
                    out["results"].append(float(agent.agent_message(b"get total_reward")))
                    out["policies"].append(np.array(agent.agentPolicy, copy=True))
                out["deltas"].append(np.array(agent.deltas, copy=True))
        finally:
            os.chdir(cwd)
    return {k: np.array(v) for k, v in out.items()}


def restated_protocol(par, n_it, deltas, tables=None):
    """The same step-level loop restated over the C port (oracle_lib.step, rlglue variant): one agent state
    machine (SwimmerAgent.py:79-130), clip (:181-201), index order + sample stdev update (:214-241), and the
    experiment's load-state / freeze schedule (SwimmerExperiment.cpp:65-84).  deltas[n_it+1, N, n-1, 2n+2]
    replaces the agent's np.random.rand draws.  Literal behaviours kept (they are what the reference does):
      * the first env step after every "load state" applies the action the agent chose from the LAST
        observation of the previous rollout with the PREVIOUS rollout's policy;
      * at the first agent step of a rollout the agent acts on the stored initial observation, not on the
        observation it was just given;
      * rollout k's return therefore sums the rewards of env steps kH+1 .. (k+1)H, and the last slot of the
        reward table (r- of the last direction) is filled at the first step of the NEXT iteration: it holds
        the first reward (iteration 0) or the previous evaluation total plus that reward.
    `tables` (a list): the reward table [2N] each update uses is appended to it."""
    from oracle import oracle_lib as O
    n, N, b, H = int(par["n_seg"]), int(par["N"]), int(par["b"]), int(par["H"])
    alpha, nu, max_u = par["alpha"], par["nu"], par["max_u"]
    p = O.make_params(n=n, l_i=par["l_i"], m_i=par["m_i"], k=par["k"], h=par["h_global"], max_u=max_u,
                      direction=tuple(par["direction"]))
    no = 2 * n + 2
    W = np.zeros((n - 1, no))
    o0 = np.full(no, 0.001)
    rewards = [0.0] * (2 * N)
    total, count, ev_count, freeze = 0.0, 0, 0, False
    results, policies = [], [W.copy()]

    def pols(it):
        return [W + s * nu * deltas[it][k] for k in range(N) for s in (1.0, -1.0)]
    dp = pols(0)
    act = np.clip(dp[0] @ o0, -max_u, max_u)                     # agent_start
    state = o0.copy()
    it_deltas = 0
    for it in range(n_it):
        freeze = False
        for i in range(2 * H * N + H):
            training = i < 2 * H * N
            if training and i % H == 0:
                state = o0.copy()
            if i == 2 * H * N:
                freeze, ev_count = True, 0
                state = o0.copy()
            state, r = O.step(p, O.RLGLUE, state, act)
            total += r
            obs = state
            if not freeze:
                if count % H == 0:
                    rewards[(count // H - 1) % (2 * N)] = total
                    total = 0.0
                    obs = o0
                pol = dp[(count % (2 * N * H)) // H]
            else:
                if ev_count == 0:
                    total = 0.0
                    obs = o0
                pol = W
            act = np.clip(pol @ obs, -max_u, max_u)
            if not freeze:
                count += 1
                if count % (2 * N * H) == 0:
                    if tables is not None:
                        tables.append(np.array(rewards))
                    used = [rewards[2 * k + s] for k in range(b) for s in (0, 1)]
                    sigma = float(np.std(used, ddof=1))
                    grad = sum((rewards[2 * k] - rewards[2 * k + 1]) * deltas[it_deltas][k] for k in range(b))
                    W = W + alpha * grad / (b * sigma)
                    it_deltas += 1
                    dp = pols(it_deltas)
                    rewards = [0.0] * (2 * N)
            else:
                ev_count += 1
        results.append(total)
        policies.append(W.copy())
    return np.array(results), np.array(policies)
