"""Serial env: same-call, alternated timing of two or more builds of the library (the first is the baseline).

usage: python tools/ab_serial.py --lib parent=PATH.so --lib new=PATH.so [--lib ...] [--workloads invmgmt,invmgmt_backlog]
                                 [--pairs 3] [--steps 10] [--warmup 2] [--launches 100] [--out DIR]

Per round (at least 3) and per build, in an order that rotates from round to round: one child process times the rollout
kernel alone for every workload (the rollout without the summary, i.e. one launch per call, CUDA events around
--launches calls), then `bench.py --no-extras` runs once per workload.  In the first round every bench run also writes
its outputs (--dump-outputs) into a temporary directory, and each build's files are compared with the baseline's
(np.array_equal).  Prints the card's name, power limit and maximum SM clock, one line per measurement and a median
table; --out DIR also writes the lines to DIR/ab_serial.txt.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(workloads, launches):
    """Kernel-alone time per workload for the library ORGYM_B200_LIB points at: {workload: ms per launch}."""
    sys.path.insert(0, ROOT)
    import torch
    import bench
    import or_gym_inventory_b200  # noqa: F401
    res = {}
    for wname in workloads:
        wl = bench.Rollout(wname, torch.device("cuda", 0), bench.WORKLOADS[wname]["envs"], 0)
        want = ("ep_return", "stats")

        def call(ep):
            return wl.env.rollout(wl.policy, seed=wl.W["seed"], episode=ep, want=want, **wl.kw)
        for ep in range(5):
            call(ep)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for ep in range(launches):
            call(100 + ep)
        e1.record()
        torch.cuda.synchronize()
        res[wname] = {"kernel_ms": e0.elapsed_time(e1) / launches, "kernel": wl.kernel_name()}
        wl.close()
    print(json.dumps(res))


def run(cmd, lib, cache):
    env = dict(os.environ, ORGYM_B200_LIB=os.path.abspath(lib), ORGYM_JIT_CACHE=cache, ORGYM_INV_JIT="2")
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
    if p.returncode != 0:
        raise SystemExit(f"{' '.join(cmd)} with {lib} failed:\n{p.stderr[-3000:]}")
    return json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a liborgym_b200.so; the first is the baseline")
    ap.add_argument("--workloads", default="invmgmt,invmgmt_backlog")
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    wls = a.workloads.split(",")
    if a.child:
        return child(wls, a.launches)
    if len(a.lib) < 2 or a.pairs < 3:
        ap.error("needs at least two --lib and --pairs >= 3")
    libs = [tuple(s.split("=", 1)) for s in a.lib]
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    say(f"# card: {card}")
    say(f"# kernel alone: CUDA events over {a.launches} rollouts (ep_return + stats, no summary), 2^24 instances x 30 periods; "
        f"bench: bench.py --gpus 1 --steps {a.steps} --warmup {a.warmup} --no-extras")
    tmp = tempfile.mkdtemp(prefix="ab_serial_")
    cache = os.path.join(tmp, "jit_cache")
    os.makedirs(cache, mode=0o700)
    kern = {(n, w): [] for n, _ in libs for w in wls}
    val = {(n, w): [] for n, _ in libs for w in wls}
    for r in range(a.pairs):
        order = libs[r % len(libs):] + libs[:r % len(libs)]
        for name, lib in order:
            k = run([sys.executable, os.path.abspath(__file__), "--child", "--workloads", a.workloads,
                     "--launches", str(a.launches)], lib, cache)
            for w in wls:
                kern[(name, w)].append(k[w]["kernel_ms"])
                say(f"round {r + 1} {name:8s} {w:16s} kernel {k[w]['kernel_ms'] * 1e3:9.2f} us  ({k[w]['kernel']})")
            for w in wls:
                cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup", str(a.warmup),
                       "--no-extras", "--workload", w]
                if r == 0:
                    cmd += ["--dump-outputs", os.path.join(tmp, name, w)]
                d = run(cmd, lib, cache)
                val[(name, w)].append(d["value"])
                say(f"round {r + 1} {name:8s} {w:16s} bench value {d['value']:.6e}  ms_per_step {d['ms_per_step']:.4f}  "
                    f"sm_mhz {(d.get('clocks') or {}).get('sm_mhz')}")
    import numpy as np
    base = libs[0][0]
    for name, _ in libs[1:]:
        for w in wls:
            d0, d1 = os.path.join(tmp, base, w), os.path.join(tmp, name, w)
            files = sorted(os.listdir(d0))
            same = files == sorted(os.listdir(d1)) and all(
                np.array_equal(np.load(os.path.join(d0, f)), np.load(os.path.join(d1, f))) for f in files)
            say(f"outputs {name} vs {base} {w}: {'identical' if same else 'DIFFERENT'} ({', '.join(files)})")
    say("# medians (change vs the baseline; spread = (max - min) / median over the rounds)")
    for w in wls:
        k0, v0 = statistics.median(kern[(base, w)]), statistics.median(val[(base, w)])
        for name, _ in libs:
            k, v = statistics.median(kern[(name, w)]), statistics.median(val[(name, w)])
            ks = (max(kern[(name, w)]) - min(kern[(name, w)])) / k
            vs = (max(val[(name, w)]) - min(val[(name, w)])) / v
            say(f"{w:16s} {name:8s} kernel {k * 1e3:9.2f} us ({(k0 / k - 1) * 100:+6.2f} % rate, spread {ks * 100:.2f} %)  "
                f"bench {v:.4e} ({(v / v0 - 1) * 100:+6.2f} %, spread {vs * 100:.2f} %)")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "ab_serial.txt"), "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
