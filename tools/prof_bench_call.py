"""Where the time of one bench.py call of a serial-env workload goes: rollout kernel, partial-sum reduction, accumulate,
gaps.  The bench call (rollout with ep_return + stats + summary, then acc.add_(summary)) runs --reps times under
torch.profiler (CUDA activities); a separate unprofiled run gives the call's CUDA-event time.

usage: python tools/prof_bench_call.py [--workload invmgmt] [--reps 50] [--out DIR]"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="invmgmt")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    dev = torch.device("cuda", 0)
    wl = bench.Rollout(a.workload, dev, bench.WORKLOADS[a.workload]["envs"], 0)
    acc = torch.zeros(8, dtype=torch.float64, device=dev)

    def call(ep):
        acc.add_(wl.call(ep)["summary"])
    call_ms = bench.time_calls(call, a.reps)
    alone_ms = bench.time_calls(lambda ep: wl.env.rollout(wl.policy, seed=wl.W["seed"], episode=ep,
                                                          want=("ep_return", "stats"), **wl.kw), a.reps)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(a.reps):
            call(1000 + k)
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                 key=lambda e: e.time_range.start)
    per = {}
    for e in evs:
        per.setdefault(e.name, []).append(e.time_range.elapsed_us())
    span = (evs[-1].time_range.end - evs[0].time_range.start) / a.reps
    busy = sum(sum(v) for v in per.values()) / a.reps
    lines = [f"# {torch.cuda.get_device_name(0)}; workload {a.workload}; {a.reps} bench calls",
             f"bench call (CUDA events, unprofiled): {call_ms * 1e3:.1f} us; rollout alone without summary: {alone_ms * 1e3:.1f} us",
             f"profiled: first kernel start -> last kernel end per call {span:.1f} us, kernels busy {busy:.1f} us, "
             f"gaps {span - busy:.1f} us"]
    for name, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
        lines.append(f"  {sum(v) / a.reps:9.1f} us per call  {len(v) / a.reps:.0f} launches  {name[:110]}")
    print("\n".join(lines))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prof_bench_call.txt"), "a") as f:
            f.write("\n".join(lines) + "\n")
    wl.close()


if __name__ == "__main__":
    main()
