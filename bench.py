"""bench.py -- the metric of BASELINE.json: swimmer env-steps/s and ARS iterations/s on 1/2/4/8 B200, % FP64 peak.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-ars] [--no-cpu]
                  [--dump-outputs DIR]

The driver-parsed headline (`metric`, `value`, `e2e`, `roofline`) is BASELINE config[1] (isolated batched
physics: 3-segment swimmer, 65,536 envs per GPU, fixed random actions, 1,000 explicit-Euler steps; a "step"
is one pass of the fused rollout over one batch = 65.5 M env-steps per GPU).  The same JSON line carries, as
first-class keys under `ars`, the ARS iterations/s of BASELINE config[2] (V2, n = 5, 1,024 directions),
config[3] (safe exploration, n = 3, 256 directions, simulator screening then real rollouts) and config[4]
(n = 10, 4,096 directions x 2 x 128 rollouts), each sharded over the N GPUs, with their parity against an
unsharded engine, plus a >= 2 s sustained run and the CPU legs.  Prints ONE JSON line (rank 0).
See DESIGN.md section "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SEG, B_PER_GPU, H = 3, 65536, 1000
W_REF = {3: 822, 5: 1751, 10: 5701}        # algorithmic flops per env-step (SURVEY 8d / app. F)
W_REF_V2 = {3: 838, 5: 1775, 10: 5745}
# Measured once per kernel change with ncu (profiles/r02_summary.md, final-build captures r02z_*):
NCU_DRAM_BYTES_PER_LAUNCH = 1.073e6         # config[1] kernel: dram__bytes_read.sum + dram__bytes_write.sum
# FP64 flops one environment step costs in the one-thread-per-environment kernels (2 per DFMA, 1 per DADD/DMUL,
# ncu source-page instruction counts / 32 lanes): the non-redundant work of a step
EXEC_FLOPS = {"n3_fixed": 312.0, "n3_v1": 344.0, "n5_v2": 735.0, "n10_v2": 1800.0}
METRIC, UNIT = "swimmer env-steps/sec", "env-steps/s"
WORKLOAD = "config[1]: 3-segment swimmer, 65,536 envs per GPU, fixed random actions U(-5,5), 1,000 explicit-Euler steps"
CONFIG = {"workload": WORKLOAD, "n_segments": N_SEG, "envs_per_gpu": B_PER_GPU, "H": H}  # identical on both arms


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-ars", action="store_true", help="skip the ARS-iteration measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s sustained run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (returns, final_state) as "
                         "DIR/<name>.npy, float64, to compare two builds output for output (the inputs are seeded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    return args


# ----------------------------------------------------------------------------------------------
# CPU legs.  The only place bench.py executes oracle/ (the C port of the reference, all host threads) and
# baseline/_ref (the unmodified Python reference, staged by oracle/stage_reference.py).
# ----------------------------------------------------------------------------------------------
def _threads_run(work, threads):
    t0 = time.perf_counter()
    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    return time.perf_counter() - t0


def cpu_fixed_action_rate(n_envs, steps, threads):
    """env-steps/s of the C port of the reference dynamics on `threads` host threads."""
    from oracle import oracle_lib as O
    p = O.make_params(n=N_SEG)
    actions = np.random.default_rng(0).uniform(-5, 5, (n_envs, N_SEG - 1))
    O.lib()
    bounds = np.linspace(0, n_envs, threads + 1).astype(int)

    def work(i):
        O.rollout_fixed_batch(p, O.GYM, actions, steps, int(bounds[i]), int(bounds[i + 1]), want_final=False)
    dt = _threads_run(work, threads)
    return n_envs * steps / dt, dt


def cpu_sample_size(threads, target_s):
    rate1, _ = cpu_fixed_action_rate(64, 200, 1)   # calibration: ~12.8k steps on one thread
    envs = int(max(threads, min(B_PER_GPU, rate1 * threads * target_s / H)))
    return max(threads, (envs // threads) * threads)


def cpu_ars_iteration(n, N_dirs, v2, threads, target_s=6.0, safe=False):
    """One ARS iteration of the C port (linear-policy rollouts on all host threads + numpy ranking / update) on
    a bounded sample of the N directions; the iteration rate is extrapolated from the sample's rollout rate
    (the update is < 1 % of an iteration).  safe: every direction also costs two simulator rollouts."""
    from oracle import oracle_lib as O
    p = O.make_params(n=n)
    no, ws = 2 * n + 2, (n - 1) * (2 * n + 2)
    rng = np.random.default_rng(1)
    W = rng.uniform(-1, 1, ws) * 0.05
    mean, inv = (np.zeros(no), np.ones(no)) if v2 else (None, None)
    O.lib()

    def run(dirs):
        d = 2 * rng.random((dirs, ws)) - 1
        pol = np.stack([W + s * 0.01 * d[k] for k in range(dirs) for s in (1, -1)])
        bounds = np.linspace(0, 2 * dirs, threads + 1).astype(int)
        out = [None] * threads

        def work(i):
            out[i] = O.rollout_policy_batch(p, O.GYM, pol, H, mean, inv, int(bounds[i]), int(bounds[i + 1]))
        dt = _threads_run(work, threads)
        rets = np.sum(out, axis=0)
        O.update_policy(W, d, rets, b=dirs, alpha=0.0075, semantics=0)
        return dt
    t_probe = run(threads)                                   # 2 rollouts per thread
    per_dir = t_probe / threads
    dirs = int(max(threads, min(N_dirs, target_s / per_dir)))
    t = run(dirs)
    rollouts_per_dir = 4 if safe else 2
    iter_s = t / dirs * N_dirs * (rollouts_per_dir / 2)
    return {"iters_per_s": 1.0 / iter_s, "env_steps_per_s": N_dirs * rollouts_per_dir * H / iter_s, "cores": threads,
            "kind": "port", "sample": "%d of %d directions (x2 rollouts x %d steps) in %.1f s, extrapolated" % (dirs, N_dirs, H, t)}


def python_reference_legs(threads, procs_iters=1):
    """The UNMODIFIED Python reference (baseline/_ref, staged from the reference tree): BASELINE config[0] =
    ARSAgent(seed=0).runOneIteration() with n = 3, V1, N = 8, H = 1000 on one core, and one such agent per
    host core (the reference's own parallelism: one Ray actor per seed, ars/experiment.py:64-72)."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref_root, "ars", "ars_agent.py")):
        return {"unavailable": "baseline/_ref not staged (run __graft_entry__.build() where /root/reference exists)"}
    code = (
        "import sys, time, os\n"
        "os.environ['SWIMMER_REFERENCE_ROOT'] = %r\n"
        "sys.path.insert(0, %r)\n"
        "from oracle import ref_harness as R\n"
        "ns = R.load()\n"
        "ep = ns.EnvParam('x', n=3, H=1000, l_i=1., m_i=1., h=1e-3, k=10., epsilon=0)\n"
        "ap = ns.ARSParam('a', V1=True, n_iter=1, H=1000, N=8, b=8, alpha=0.0075, nu=0.01, safe=False, threshold=0, initial_w='Zero')\n"
        "ag = ns.ARSAgent(ep, ap, seed=int(sys.argv[1]))\n"
        "t = time.perf_counter(); r = ag.runOneIteration(); dt = time.perf_counter() - t\n"
        "print('RESULT', dt, float(r[0]), float(r[1]))\n" % (ref_root, ROOT))
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1")

    def launch(seed):
        return subprocess.Popen([sys.executable, "-c", code, str(seed)], stdout=subprocess.PIPE,
                                stderr=subprocess.DEVNULL, text=True, env=env)

    def result(pr):
        out = pr.communicate(timeout=300)[0]
        for ln in out.splitlines():
            if ln.startswith("RESULT"):
                _, dt, r0, r1 = ln.split()
                return float(dt), float(r0), float(r1)
        raise RuntimeError("python reference leg failed: " + out[-500:])
    dt1, r0, r1 = result(launch(0))
    # survey-recorded returns of config[0], seed 0, iteration 0 (SURVEY 8c): proves it is the reference that ran
    ok = abs(r0 - (-0.11878042019245531)) < 1e-12 and abs(r1 - 0.46055543070364563) < 1e-12
    t0 = time.perf_counter()
    prs = [launch(s) for s in range(threads)]
    dts = [result(pr)[0] for pr in prs]
    wall = time.perf_counter() - t0
    return {"kind": "reference", "workload": "config[0]: ARS V1, 3-segment swimmer, 8 directions, H=1000 (ars/ars_agent.py runOneIteration, numpy)",
            "one_core": {"iters_per_s": 1.0 / dt1, "env_steps_per_s": 16 * H / dt1, "cores": 1},
            "all_cores": {"agent_iters_per_s": threads / wall, "env_steps_per_s": threads * 16 * H / wall, "cores": threads,
                          "note": "one agent (seed) per core, one iteration each, process start-up included in the wall time; "
                                  "mean in-process iteration time %.2f s" % float(np.mean(dts))},
            "returns_match_survey": bool(ok)}


def ref_cpp_rate(steps=20000):
    """Secondary: the unmodified reference C++ swimmer (oracle/_ref, RL-Glue variant, Eigen QR +
    redundant inverse), one core, no printing.  Different dynamics variant: reported, not compared."""
    from oracle import oracle_lib as O
    if O.ref_cpp() is None:
        return None
    p = O.make_params(n=N_SEG, h=0.01)
    O.ref_cpp_set_params(p)
    st = np.full(2 * N_SEG + 2, 0.001)
    a = np.array([1.5, -2.0])
    t0 = time.perf_counter()
    O.ref_cpp().ref_rollout_fixed(st.ctypes.data_as(O._dp), a.ctypes.data_as(O._dp), steps)
    return steps / (time.perf_counter() - t0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # bounded sample per step: the whole run (K timed + W warm-up steps) stays near two minutes
    per_step_s = min(4.0, max(0.25, 100.0 / max(1, args.steps + args.warmup)))
    envs = cpu_sample_size(threads, per_step_s)
    for _ in range(args.warmup):
        cpu_fixed_action_rate(max(threads, envs // 8), H, threads)
    t_tot, done = 0.0, 0
    for _ in range(args.steps):
        rate, dt = cpu_fixed_action_rate(envs, H, threads)
        t_tot += dt
        done += envs * H
    value = done / t_tot
    sample = "%d envs x %d steps per step (of %d), %d host threads" % (envs, H, B_PER_GPU, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": dict(CONFIG),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "value = C port of the reference gym swimmer (oracle/swimmer_oracle.c, the dense (n+2) formulation of "
                "remy_swimmer_env.py) on all host threads: ~270x faster per core than the reference's own numpy code, "
                "i.e. the conservative baseline; the unmodified Python reference is timed beside it (python_reference)",
    }
    if not args.no_cpu:
        line["python_reference"] = python_reference_legs(threads)
        line["ars_cpu"] = {"config[2]": cpu_ars_iteration(5, 1024, True, threads),
                           "config[3]": cpu_ars_iteration(3, 256, False, threads, target_s=3.0, safe=True)}
    cpp = ref_cpp_rate()
    if cpp:
        line["ref_cpp_rlglue_1core"] = {"value": cpp, "unit": UNIT, "kind": "reference",
                                        "note": "unmodified rlglue/environment/SwimmerEnvironment.cpp updateState, n=3"}
    emit(line)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.rows = None, []
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def window(self, t0, t1):
        """Samples taken in [t0, t1] (perf_counter): median SM clock, median / max power, throttle reasons."""
        sm, pw, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in list(self.rows):
            if t < t0 or t > t1:
                continue
            c = [x.strip() for x in r.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); pw.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz_median": float(np.median(sm)) if sm else None, "power_w_median": float(np.median(pw)) if pw else None,
                "power_w_max": float(np.max(pw)) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for _, r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx = float(c[1])
            except ValueError:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # idle samples (before the first launch) sit at the idle clock: take the median of the upper half
        hot = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(hot)) if hot else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm),
                "note": "nvidia-smi -lms 100 from before warm-up to the end of the sustained run; median of the "
                        "upper half of samples (the lower half contains idle gaps between the measured regions)"}


def run_b200(args):
    import torch
    import torch.distributed as dist
    import swimmer_ars_b200 as S
    from swimmer_ars_b200 import distributed as D

    rank, world, device = D.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    if world != args.gpus and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE=%d" % (args.gpus, world), file=sys.stderr)
    params = S.make_params(n=N_SEG)
    rng = np.random.default_rng(rank)
    host_actions = torch.as_tensor(rng.uniform(-5, 5, (B_PER_GPU, N_SEG - 1))).pin_memory()
    actions = host_actions.to(device)
    out = {"returns": torch.empty(B_PER_GPU, dtype=torch.float64, device=device),
           "final_state": torch.empty(B_PER_GPU, 2 * N_SEG + 2, dtype=torch.float64, device=device)}
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=device)
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.cpu()[0])

    def single_launch():
        return S.ops.rollout(params, H, actions=actions, want_final=True, out=out, schedule="plain")

    # The timed step: ONE call of the public batched entry point with no tuning argument --
    # SwimmerEnv.rollout_batched(H, actions) -> swm_rollout -- captured once in a CUDA graph and replayed.  For this
    # batch (3.46 warps per SM sub-partition) the library itself schedules the rollout as sub-batches x 64-step
    # chunks on internal streams (swm_rollout_t.schedule_sub = 0: decided from B, n and the SM count; 16 x 64 while
    # capturing, 8 x 256 when enqueued eagerly); every final state is bit-identical to one plain launch.
    env0 = S.SwimmerEnv(n=N_SEG, device=device)
    out_def = {"returns": torch.empty_like(out["returns"]), "final_state": torch.empty_like(out["final_state"])}

    def default_call():
        return env0.rollout_batched(H, actions=actions, want_final=True, out=out_def)
    default_call()
    torch.cuda.synchronize()
    step_graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(step_graph):
        default_call()
        import ctypes as _ct
        _cfg = S._lib.SwmRollout()
        _cfg.policy_mode, _cfg.H, _cfg.B, _cfg.rollouts_per_policy = 0, H, B_PER_GPU, 1
        _cfg.actions, _cfg.returns, _cfg.final_state = actions.data_ptr(), out_def["returns"].data_ptr(), out_def["final_state"].data_ptr()
        _ns, _ch = _ct.c_int(0), _ct.c_int(0)
        S._lib.lib().swm_rollout_schedule(_ct.byref(params), _ct.byref(_cfg), S._lib.stream_ptr(), _ct.byref(_ns), _ct.byref(_ch))
    launches_per_step = max(1, _ns.value) * (-(-H // _ch.value) if _ns.value else 1)
    ref_res = single_launch()
    step_graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out_def["final_state"], ref_res.final_state), "library schedule must reproduce the single launch"

    def one_step():
        step_graph.replay()

    # ---- FP64 roofline denominator: DFMA probe measured live on this GPU ----
    sink = torch.zeros(8, dtype=torch.float64, device=device)
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    S.ops.fp64_probe(sms * 8, 256, 200, sink)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        flops = S.ops.fp64_probe(sms * 8, 256, 4000, sink)
        e1.record(stream)
        e1.synchronize()
        best = max(best, flops / (e0.elapsed_time(e1) * 1e-3))
    fp64_peak_tflops = best / 1e12

    sampler = ClockSampler(device.index) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    # ---- device-resident timing: K steps, each its own event pair, L2 flushed in between ----
    evs = []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        one_step()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - t_wall0
    if args.dump_outputs:
        # out_def holds the last timed step's results; the supplementary runs below overwrite it
        dump_outputs(args.dump_outputs, out_def, rank, world)
    t_dev_s = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs)) * 1e-3
    # ---- supplementary: one plain swm_rollout launch per step (no chunking), and the default call enqueued
    # eagerly (no graph), same timing method ----
    def timed_steps(fn):
        ev = []
        for _ in range(args.steps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            ev.append((e0, e1))
        barrier()
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in ev)) * 1e-3
    t_single_s = timed_steps(single_launch)
    t_eager_s = timed_steps(default_call)

    # ---- supplementary: the same K launches with TWO in flight (two streams, device-resident inputs, no
    # flush).  One config[1] batch is only 3.46 warps per SM sub-partition; two batches fill the FP64 pipe. ----
    side = [torch.cuda.Stream(device=device) for _ in range(2)]
    outs2 = [{"returns": torch.empty_like(out["returns"]), "final_state": torch.empty_like(out["final_state"])}
             for _ in range(2)]
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(stream)
    for st in side:
        st.wait_stream(stream)
    for k in range(args.steps):
        with torch.cuda.stream(side[k & 1]):
            S.ops.rollout(params, H, actions=actions, want_final=True, out=outs2[k & 1], schedule="plain")
    for st in side:
        stream.wait_stream(st)
    c1.record(stream)
    barrier()
    t_conc_s = max_over_ranks(c0.elapsed_time(c1)) * 1e-3

    # ---- end-to-end through the host-buffer entry point: every step uploads its actions from pinned host
    # memory and downloads returns + final states into pinned host memory (SwimmerEnv.rollout_batched_host,
    # double-buffered on two streams: the copies of one step overlap the kernel of its neighbour).  No L2
    # flush here: the inputs are re-uploaded from the host on every step. ----
    host_ret = [torch.empty(B_PER_GPU, dtype=torch.float64).pin_memory() for _ in range(2)]
    host_fin = [torch.empty(B_PER_GPU, 2 * N_SEG + 2, dtype=torch.float64).pin_memory() for _ in range(2)]
    env = S.SwimmerEnv(n=N_SEG, device=device)

    def e2e_step(k):
        return env.rollout_batched_host(H, host_actions, host_ret[k & 1], host_fin[k & 1])
    for k in range(3):
        e2e_step(k)
    env.synchronize_host()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        e2e_step(k)
    env.synchronize_host()
    e1.record(stream)
    barrier()
    t_e2e_s = max_over_ranks(e0.elapsed_time(e1)) * 1e-3
    e2e_check = float(host_ret[(args.steps - 1) & 1].sum())  # the host really holds the results
    assert np.isfinite(e2e_check)

    total_steps = float(world) * B_PER_GPU * H * args.steps
    value = total_steps / t_dev_s
    e2e_value = total_steps / t_e2e_s
    conc_value = total_steps / t_conc_s
    single_value = total_steps / t_single_s
    eager_value = total_steps / t_eager_s

    # ---- sustained run: the timed step replayed back to back for >= 2 s (no flush, no host gaps) with the
    # clock / power samples of exactly that window: the 18 ms headline survives thermals and the power cap ----
    sustained = None
    if not args.no_sustained:
        reps = max(50, int(2.2 / (t_dev_s / args.steps)))
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        s0.record(stream)
        for _ in range(reps):
            one_step()
        s1.record(stream)
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        t_sus = max_over_ranks(s0.elapsed_time(s1)) * 1e-3
        sustained = {"value": float(world) * B_PER_GPU * H * reps / t_sus, "unit": UNIT, "seconds": t_sus, "steps": reps,
                     "note": "the same CUDA-graph step replayed back to back (device-resident inputs, no L2 flush between steps)"}
        if sampler:
            sustained["clocks"] = sampler.window(w0 + 0.15, w1)
    clocks = sampler.stop() if sampler else None

    ars = None
    if not args.no_ars:
        ars = measure_ars(S, D, dist, device, rank, world, barrier, max_over_ranks, fp64_peak_tflops)

    if rank == 0:
        cpu = None
        extra_cpu = {}
        if not args.no_cpu:
            threads = os.cpu_count() or 1
            envs = cpu_sample_size(threads, 10.0)
            rate, dt = cpu_fixed_action_rate(envs, H, threads)
            cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": "%d envs x %d steps of the same workload in %.1f s (oracle C port of the "
                             "reference gym swimmer)" % (envs, H, dt)}
            if world == 1:
                extra_cpu["ars_cpu"] = {"config[2]": cpu_ars_iteration(5, 1024, True, threads),
                                        "config[3]": cpu_ars_iteration(3, 256, False, threads, target_s=3.0, safe=True)}
                extra_cpu["python_reference"] = python_reference_legs(threads)
        ms_per_step = 1e3 * t_dev_s / args.steps
        per_gpu = value / world
        exec_tf = per_gpu * EXEC_FLOPS["n3_fixed"] / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(CONFIG),
            "run": {"l2": "flushed between steps (256 MiB write outside the timed events); inputs 1 MiB",
                    "schedule": "each step = SwimmerEnv.rollout_batched(H, actions) with NO schedule argument, captured in a "
                                "CUDA graph: the library picked %d sub-batches x %d-step chunks (%d kernel launches per "
                                "step, state chained through final_state, final states bit-identical to one plain "
                                "launch)" % (_ns.value, _ch.value, launches_per_step),
                    "timing": "CUDA events per step on the launch stream, summed; max over ranks"},
            "roofline": {"bound": "fp64", "achieved": exec_tf, "peak": fp64_peak_tflops, "unit": "TFLOP/s",
                         "frac": exec_tf / fp64_peak_tflops, "flops_per_env_step": EXEC_FLOPS["n3_fixed"],
                         "traffic": NCU_DRAM_BYTES_PER_LAUNCH,
                         "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, "
                                         "profiles/r02z_n3_fixed_plain_ncu.csv): ~0 B per env-step, not HBM-bound",
                         "peak_source": "DFMA probe kernel measured in this run (MEASURED_PEAKS.json has no FP64 "
                                        "entry; nominal 37.2 TFLOP/s)",
                         "note": "achieved = per-GPU env-steps/s x 312 FP64 flops the O(n) kernel EXECUTES per env-step "
                                 "(ncu instruction counts, profiles/r02_summary.md); a DFMA with three register sources "
                                 "issues every 3.1 cycles on B200, so the pipe saturates below 1.0",
                         "algorithmic": {"flops_per_env_step": W_REF[N_SEG], "achieved": per_gpu * W_REF[N_SEG] / 1e12,
                                         "frac": per_gpu * W_REF[N_SEG] / 1e12 / fp64_peak_tflops,
                                         "note": "SURVEY 8d accounting: the reference's dense O(n^3) formulation costs "
                                                 "822 flops per env-step; > 1 because the kernel solves the same "
                                                 "equations in O(n)"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B_PER_GPU * (N_SEG - 1) * 8,
                    "d2h_bytes_per_step": B_PER_GPU * (2 * N_SEG + 3) * 8,
                    "api": "SwimmerEnv.rollout_batched_host: pinned host actions in, pinned host returns + final states "
                           "out every step, double-buffered on two streams; CUDA events around all K steps"},
            "single_launch": {"value": single_value, "unit": UNIT,
                              "note": "one plain swm_rollout launch per step (schedule forced to 'plain': the whole batch in "
                                      "one kernel), same events / flush as `value`"},
            "default_api_eager": {"value": eager_value, "unit": UNIT,
                                  "note": "the same default call enqueued eagerly every step (no CUDA graph): the library "
                                          "then uses 8 sub-batches x 256-step chunks (32 launches)"},
            "two_in_flight": {"value": conc_value, "unit": UNIT, "streams": 2,
                              "roofline_frac_executed": (conc_value / world) * EXEC_FLOPS["n3_fixed"] / 1e12 / fp64_peak_tflops,
                              "note": "same kernel, same inputs resident in HBM, K launches alternating on two streams "
                                      "(no L2 flush): one 65,536-env batch is 3.46 warps per SM sub-partition (the busiest "
                                      "holds 4), two batches in flight balance and fill the FP64 pipe; this is also why "
                                      "the double-buffered e2e number exceeds the one-launch-at-a-time `value`"},
            "sustained": sustained,
            "gpu_launches": args.steps * launches_per_step, "clocks": clocks, "cpu_baseline": cpu,
            "wall_s_timed_region": wall,
        }
        line.update(extra_cpu)
        if ars:
            line["ars"] = ars
            line["ars_iters_per_s"] = {k: v["iters_per_s"] for k, v in ars.items() if "iters_per_s" in v}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_ars(S, D, dist, device, rank, world, barrier, max_over_ranks, fp64_peak_tflops):
    """ARS iterations/s of BASELINE config[2], config[3], config[4]: rollouts + record exchange + ranking +
    update, directions sharded over the `world` GPUs (strong scaling), one CUDA-graph launch per iteration."""
    import torch
    stream = torch.cuda.current_stream()
    res = {}

    def rel(x, y):
        x, y = torch.nan_to_num(x), torch.nan_to_num(y)
        return float(((x - y).abs().max() / y.abs().max().clamp_min(1e-300)).cpu())

    def timed(eng, iters, warm):
        for _ in range(warm):   # eager warm-up, graph capture, replay
            eng.run_iteration()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            eng.run_iteration()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) * 1e-3

    def parity(make, iters=3):
        """Sharded engine vs an unsharded engine run by rank 0 alone, same seed, `iters` iterations: relative
        difference of the policy and of the last returns (north-star tolerance 1e-6)."""
        if world == 1:
            return None
        sh = make(True)
        for _ in range(iters):
            sh.run_iteration()
        out = None
        if rank == 0:
            single = make(False)
            for _ in range(iters):
                single.run_iteration()
            out = {"iterations": iters, "policy_rel_diff": rel(sh.W, single.W), "returns_rel_diff": rel(sh.returns, single.returns),
                   "tolerance": 1e-6}
            out["ok"] = bool(out["policy_rel_diff"] < 1e-6 and out["returns_rel_diff"] < 1e-6)
            del single
        sh.exchange.close()
        barrier()
        return out

    KERNEL_TEXT = {"thread": "one thread per environment", "lanes": "lane-split: one environment over %d lanes, one warp per lane group",
                   "lanes2": "lane-split over %d lanes, two warps per lane group (main + operator warp)",
                   "lanes3": "lane-split over %d lanes, three warps per lane group (main + two operator warps)"}

    def describe(eng, note=""):
        name = S.ops.rollout_kernel_choice(eng.params, eng.B_local, rollouts_per_policy=eng.R)
        lanes = 32 // S.ops.lane_split_envs_per_warp(eng.params.n)
        text = KERNEL_TEXT[name] % lanes if "%d" in KERNEL_TEXT[name] else KERNEL_TEXT[name]
        out = {"launch": "CUDA graph replay" if eng._graph is not None else "eager",
               "exchange": eng.exchange.transport, "rollout_kernel": text + note, "envs_per_gpu": eng.B_local}
        if eng.shard_replicas > 1:
            out["sharding"] = ("sharded over blocks of %d GPUs, %d blocks each running the whole problem (ArsEngine shard='auto': "
                               "a share smaller than one lane group per SM is not faster, more peers only lengthen the exchange)"
                               % (eng.world, eng.shard_replicas))
        if eng.replicated:
            out["sharding"] = ("replicated on every rank, no exchange (ArsEngine shard='auto': the whole batch already runs on "
                               "the latency-optimised kernel, a smaller share per GPU would not be faster)")
        return out

    # ---------------- config[2]: ARS V2, n = 5, 1,024 directions ----------------
    if 1024 % world == 0:
        def make2(sharded):
            return S.ArsEngine(S.make_params(n=5), N=1024, b=1024, alpha=0.0075, nu=0.01, H=1000, v2=True,
                               semantics=S.ARS_AGENT, seed=0, device=device, use_graph=True,
                               distributed=None if sharded else False)
        par = parity(make2)
        eng = make2(True)
        K = 20
        t = timed(eng, K, 5)
        steps = 2.0 * 1024 * 1000
        ee = eng.check_exchange()
        res["config[2]"] = dict(
            workload="config[2]: ARS V2 (obs normalisation), 5-segment swimmer, 1,024 directions (2,048 rollouts), H=1000; "
                     "directions sharded over %d GPU(s)%s (strong scaling)"
                     % (eng.world, " in each of %d blocks of the %d" % (eng.shard_replicas, world) if eng.shard_replicas > 1 else ""),
            iters_per_s=K / t, ms_per_iter=1e3 * t / K, env_steps_per_s=K * steps / t, iters_timed=K,
            mean_return_last=float(eng.returns.mean().cpu()), exchange_epochs=ee, parity_vs_single=par,
            roofline={"bound": "latency (2,048 envs in all: at most one lane-split warp per SM sub-partition)",
                      "executed": {"flops_per_env_step": EXEC_FLOPS["n5_v2"],
                                   "frac": (K * steps / t / eng.world) * EXEC_FLOPS["n5_v2"] / 1e12 / fp64_peak_tflops},
                      "algorithmic_frac": (K * steps / t / eng.world) * W_REF_V2[5] / 1e12 / fp64_peak_tflops},
            **describe(eng))
        eng.exchange.close()
        del eng

    # ---------------- config[3]: safe-exploration ARS, n = 3, 256 directions ----------------
    if 256 % world == 0:
        n3 = 3
        real = S.make_params(n=n3, l_i=0.8, m_i=1.2, k=10.2)
        u = np.random.default_rng(7).normal(size=3)
        u /= np.linalg.norm(u)
        eps = 1e-3                                  # ars/safe_exploration.py:22-24, 65-80
        sim = S.make_params(n=n3, m_i=1.2 + eps * u[0], l_i=0.8 + eps * u[1], k=10.2 + eps * u[2])
        base = dict(N=256, b=256, alpha=0.0075, nu=0.01, H=1000, v2=False, semantics=S.ARS_AGENT, device=device)
        # pre-trained policy (every rank trains the same one alone: 40 plain iterations from zero) and a fixed
        # threshold taken from a probe of the simulator returns, so that a realistic share is screened out
        pre = S.ArsEngine(real, seed=11, distributed=False, use_graph=True, **base)
        for _ in range(40):
            pre.run_iteration()
        W0 = pre.W.clone()
        probe = S.ArsEngine(real, seed=12, distributed=False, sim_params=sim, sim_threshold=-1e300, initial_policy=W0, **base)
        probe.run_iteration(update=False)
        worst = probe.sim_returns.view(256, 2).min(dim=1).values
        thr = float(torch.quantile(worst, 0.5).cpu())
        alpha_h = S.Threshold(K=1., A=0.1, B=0.001).compute_alpha(1000)
        del pre, probe

        def make3(sharded, speculate=True):
            return S.ArsEngine(real, seed=12, sim_params=sim, sim_threshold=thr, initial_policy=W0, use_graph=True,
                               distributed=None if sharded else False, speculate=speculate, **base)

        def run3(eng, K):
            for _ in range(5):
                eng.run_iteration()
            barrier()
            pass0 = int(eng.n_pass_total.cpu()[0])  # device-side running count of surviving directions (this rank)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(K):
                eng.run_iteration()
            e1.record(stream)
            barrier()
            t = max_over_ranks(e0.elapsed_time(e1)) * 1e-3
            npass = torch.tensor([float(int(eng.n_pass_total.cpu()[0]) - pass0)], dtype=torch.float64, device=device)
            if world > 1 and not eng.replicated:
                dist.all_reduce(npass)
            return t, float(npass.cpu()[0]) / (K * 256.0), eng.check_exchange()

        par = parity(make3)
        K = 20
        # the same iterations with the real-world rollouts started only after the screening mask exists
        eng = make3(True, speculate=False)
        t_first, frac_first, _ = run3(eng, K)
        eng.exchange.close()
        del eng
        eng = make3(True)
        t, frac_pass, ee = run3(eng, K)
        steps = (2.0 * 256 + 2.0 * 256 * frac_pass) * 1000
        res["config[3]"] = dict(
            workload="config[3]: safe-exploration ARS V1 (reward constraint), 3-segment swimmer, 256 directions: 512 simulator "
                     "rollouts screen every +-delta pair, surviving pairs are rolled out in the real world; real (l,m,k) = "
                     "(0.8,1.2,10.2), simulator = real + 1e-3 u/|u|, pre-trained W0; %s %d GPU(s)"
                     % ("replicated on each of" if eng.replicated else "sharded over", world),
            iters_per_s=K / t, ms_per_iter=1e3 * t / K, env_steps_per_s=K * steps / t, iters_timed=K,
            screened_fraction=1.0 - frac_pass, sim_threshold=thr,
            schedule="speculative (engine default for V1 safe mode): the real-world rollouts of all 256 directions run beside "
                     "the simulator rollouts on a second stream, the screening mask is applied to their returns afterwards; "
                     "bit-identical to screening first (tests/test_parity_ars.py); env_steps_per_s counts the simulator "
                     "rollouts and the SURVIVING real rollouts only",
            screen_first={"iters_per_s": K / t_first, "ms_per_iter": 1e3 * t_first / K, "screened_fraction": 1.0 - frac_first,
                          "note": "speculate=False: simulator rollouts, mask, then the surviving real rollouts (two dependent "
                                  "1000-step rollouts per iteration)"},
            threshold_note="threshold = median of min(r+_sim, r-_sim) of a probe iteration; the reference adds "
                           "alpha(H) * eps = %.3g to its threshold (ars_agent.py:64-69), constant, already inside" % (alpha_h * eps),
            exchange_epochs=ee, parity_vs_single=par,
            roofline={"bound": "latency (512 + 512 envs side by side)",
                      "executed": {"flops_per_env_step": EXEC_FLOPS["n3_v1"],
                                   "frac": (K * steps / t / (1 if eng.replicated else world)) * EXEC_FLOPS["n3_v1"] / 1e12
                                   / fp64_peak_tflops}},
            **describe(eng))
        eng.exchange.close()
        del eng

    # ---------------- config[4]: n = 10, 4,096 directions x 2 x 128 rollouts ----------------
    if 4096 % world == 0:
        def make4(sharded):
            return S.ArsEngine(S.make_params(n=10), N=4096, b=4096, alpha=0.0075, nu=0.01, H=1000, v2=True,
                               semantics=S.ARS_AGENT, seed=0, device=device, rollouts_per_direction=128,
                               init_perturb=1e-2, use_graph=True, distributed=None if sharded else False)
        par = parity(make4, iters=2)
        eng = make4(True)
        K = 3 if world == 1 else 6
        t = timed(eng, K, 2)
        steps = 2.0 * 4096 * 128 * 1000
        ee = eng.check_exchange()
        res["config[4]"] = dict(
            workload="config[4]: ARS V2, 10-segment swimmer, 4,096 directions x 2 x 128 rollouts (1,048,576 envs, reset + "
                     "1e-2*U[0,1) starts), H=1000; directions sharded over %d GPU(s) (strong scaling)" % world,
            iters_per_s=K / t, ms_per_iter=1e3 * t / K, env_steps_per_s=K * steps / t, iters_timed=K,
            mean_return_last=float(eng.returns.mean().cpu()), exchange_epochs=ee, parity_vs_single=par,
            roofline={"bound": "fp64",
                      "executed": {"flops_per_env_step": EXEC_FLOPS["n10_v2"],
                                   "frac": (K * steps / t / world) * EXEC_FLOPS["n10_v2"] / 1e12 / fp64_peak_tflops},
                      "algorithmic_frac": (K * steps / t / world) * W_REF_V2[10] / 1e12 / fp64_peak_tflops},
            **describe(eng, ", one policy copy per warp"))
        eng.exchange.close()
        del eng

    if world == 1:
        # seed fan-out (ars/experiment.py:64-72: one agent per seed): 32 agents of config[0]
        # (n=3, V1, 8 directions, H=1000), one CUDA stream + one graph launch per agent-iteration
        seeds, K3 = 32, 20
        fan = S.SeedFanout(S.make_params(n=3), range(seeds), N=8, b=8, alpha=0.0075, nu=0.01, H=1000, device=device)
        fan.run(2)
        barrier()
        t0 = time.perf_counter()
        fan.run(K3, include_initial=False)
        dt = time.perf_counter() - t0
        res["config[0] x 32 seeds"] = {
            "workload": "config[0] x %d seeds: ARS V1, 3-segment swimmer, 8 directions, H=1000, one agent per "
                        "seed on one GPU (seed fan-out)" % seeds,
            "agent_iters_per_s": seeds * K3 / dt, "env_steps_per_s": seeds * K3 * 16 * 1000 / dt,
            "ms_per_round": 1e3 * dt / K3, "timing": "host wall clock around %d rounds incl. final sync" % K3}
        del fan

        # Safe_ARS (safe_ars/ars.py: per-step state-constraint screening through a simulator model, V1), 256
        # directions of the config[3] models: every step of every rollout is first tried on the simulator
        real = S.make_params(n=3, l_i=0.8, m_i=1.2, k=10.2)
        sim = S.make_params(n=3, l_i=0.8006, m_i=1.2006, k=10.2006)
        eng = S.ArsEngine(real, N=256, b=256, alpha=0.0075, nu=0.01, H=1000, semantics=S.ARS_TOPB, seed=3, device=device,
                          distributed=False, use_graph=True, step_screen=dict(sim_params=sim, sim_thresh=50.0, real_thresh=51.0))
        K4 = 20
        t = timed(eng, K4, 5)
        res["safe_ars per-step screening"] = dict(
            workload="Safe_ARS (per-step screening: one simulator step before every real step, max|thd| <= threshold), V1, "
                     "3-segment swimmer, 256 directions (512 rollouts), H=1000, one GPU",
            iters_per_s=K4 / t, ms_per_iter=1e3 * t / K4, env_steps_per_s=K4 * 512e3 / t, iters_timed=K4,
            mean_return_last=float(torch.nan_to_num(eng.returns).mean().cpu()),
            **describe(eng, ", per-step screening as a second right-hand side on the same solution rows"))
        del eng
    return res


def dump_outputs(path, outputs, rank, world):
    """Writes the arrays a caller of the timed step receives (SwimmerEnv.rollout_batched: returns [B], final_state
    [B, 2n+2]) as <path>/<name>.npy in float64, 4.7 MB per rank.  The actions are drawn from a generator seeded
    with the rank, so the same arguments give the same inputs on every run.  With several ranks each writes its
    own batch as <name>_rank<r>.npy."""
    os.makedirs(path, exist_ok=True)
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, t in outputs.items():
        np.save(os.path.join(path, name + suffix + ".npy"), t.cpu().numpy().astype(np.float64, copy=False))


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints there while the run
    is in progress (e.g. NCCL's version banner) has been redirected to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
