"""A/B of the joint-angle form (csrc/dynamics.cuh, n <= SWM_JOINT_FORM_MAX_N) against the block-tridiagonal form it
replaces, in one process tree on one GPU:

  python tools/ab_joint_form.py [--rounds 3] [--out DIR]

Builds the package library as it stands and a second one with -DSWM_JOINT_FORM_MAX_N=1 (every n on the
block-tridiagonal form, i.e. the previous code) from copies of the package's objects, then alternates the two builds
`--rounds` times over
  * tools/ab_thread_kernel.py: config[1] under graph replay with the default and the plain schedule, and the
    n = 5 / n = 10 V2 thread kernel at 131,072 environments (CUDA events, L2 flushed before every timed replay), and
  * bench.py --no-ars --no-cpu (its JSON line, sustained clocks and throttle reasons included).
The card name and power limit are printed first.  Run after __graft_entry__.build()."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "safe-exploration-with-simulator-in-rl-algorithms_b200", "csrc")
LIB = os.path.join(ROOT, "safe-exploration-with-simulator-in-rl-algorithms_b200", "libswimmer_ars.so")


def build_block(tmp):
    """The library with the block-tridiagonal form for every n: only the thread-kernel objects are recompiled."""
    obj = os.path.join(tmp, "obj")
    shutil.copytree(os.path.join(CSRC, "build"), obj)
    for f in os.listdir(obj):
        if f.startswith("rollout_n") or f in ("capi.o", "estimate.o"):
            os.remove(os.path.join(obj, f))
    out = os.path.join(tmp, "libswimmer_ars_block.so")
    subprocess.run(["make", "-C", CSRC, "-j", str(os.cpu_count() or 4), "OBJDIR=" + obj, "OUT=" + out,
                    "EXTRA_NVFLAGS=-DSWM_JOINT_FORM_MAX_N=1"], check=True, stdout=subprocess.DEVNULL)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for the bench.py JSON lines (default: none kept)")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", smi, flush=True)
    tmp = tempfile.mkdtemp(prefix="ab_joint_")
    try:
        libs = {"joint": LIB, "block": build_block(tmp)}
        rows = {k: [] for k in libs}
        for r in range(args.rounds):
            for tag, lib in libs.items():
                env = dict(os.environ, SWM_LIB_PATH=lib)
                ab = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ab_thread_kernel.py")], env=env,
                                    capture_output=True, text=True)
                print("[round %d %s]\n%s%s" % (r, tag, ab.stdout, ab.stderr[-1000:] if ab.returncode else ""),
                      flush=True)
                b = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-ars",
                                    "--no-cpu"], env=env, capture_output=True, text=True)
                line = [ln for ln in b.stdout.splitlines() if ln.startswith("{")]
                if b.returncode or not line:
                    print("bench.py failed:", b.stderr[-2000:], flush=True)
                    continue
                res = json.loads(line[-1])
                rows[tag].append(res)
                if args.out:
                    os.makedirs(args.out, exist_ok=True)
                    with open(os.path.join(args.out, "bench_%s_%d.json" % (tag, r)), "w") as f:
                        f.write(line[-1] + "\n")
                sus = res.get("sustained") or {}
                print("bench %-5s value %.4e  single_launch %s  two_in_flight %s  sustained %.4e clocks %s"
                      % (tag, res["value"], json.dumps(res.get("single_launch", {}).get("value")),
                         json.dumps(res.get("two_in_flight", {}).get("value")), sus.get("value", float("nan")),
                         json.dumps(sus.get("clocks"))), flush=True)
        for tag in libs:
            v = [x["value"] for x in rows[tag]]
            if v:
                print("%-5s value: %s  median %.4e  spread %.2f %%" % (tag, " ".join("%.4e" % x for x in v),
                      sorted(v)[len(v) // 2], 100 * (max(v) - min(v)) / min(v)))
        if rows["joint"] and rows["block"]:
            mj = sorted(x["value"] for x in rows["joint"])[len(rows["joint"]) // 2]
            mb = sorted(x["value"] for x in rows["block"])[len(rows["block"]) // 2]
            print("joint / block median value: %.3f" % (mj / mb))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
