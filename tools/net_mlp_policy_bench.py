"""Fused MLP-policy rollout vs the step-API loop a user would write today, on NetInvMgmtBacklogEnv() (the default 9-node
graph, 30 periods) with an SB3-default (64, 64) tanh actor (68 -> 64 -> 64 -> 11).  Prints one JSON object (also
written to --out):
  (a) env.rollout(net)                                               -- net_mlp_rollout_kernel, policy evaluated on chip
  (b) reset + T x (obs -> net -> clip to [0, action_space.high] -> env.step)          -- torch forward per period
timed with CUDA events, warmed up, alternated; env-steps/s for both, the fused kernel's FP32 FLOP/s against the
CUDA-core peak of the card it ran on (SMs x 128 lanes x 2 x max SM clock; 2 (68*64 + 64*64 + 64*11) = 18 304 FLOP per
env-step), the card's power limit and max SM clock (read, never set), and the fraction of episodes on which (a) and (b)
give a bitwise-equal ep_return (the rest differ through an action that moved by an ulp: torch sums the dot products in
another order).
usage: python tools/net_mlp_policy_bench.py [--sizes 20,22] [--reps 3] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
FLOP_PER_STEP = 2 * (68 * 64 + 64 * 64 + 64 * 11)    # 18 304 at (64, 64) on the default graph


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, pl, clk = [x.strip() for x in q.split(",")]
    return dict(name=name, power_limit_w=float(pl), clocks_max_sm_mhz=float(clk))


def sb3_default_actor(torch, od, high, seed=0):
    """(64, 64) tanh actor whose orders spread over [0, high] on the env's observations (an untrained net saturates):
    the first layer is scaled down, the last one is scaled and shifted so that every output has mean high / 2 and
    standard deviation high / 3 over observations drawn uniformly from [0, 400]."""
    torch.manual_seed(seed)
    nn = torch.nn
    E = len(high)
    net = nn.Sequential(nn.Linear(od, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh(), nn.Linear(64, E)).double()
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((4096, od), generator=g, dtype=torch.float64) * 400
    hi = torch.as_tensor(high, dtype=torch.float64)
    with torch.no_grad():
        net[0].weight.mul_(0.005)
        y = net(x)
        s = hi / 3 / y.std(0).clamp_min(1e-6)
        net[4].weight.mul_(s[:, None])
        net[4].bias.copy_(hi / 2 + (net[4].bias - y.mean(0)) * s)
    return net.float().cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20,22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_net_mlp_policy_bench.json"))
    args = ap.parse_args()
    import torch
    import or_gym_inventory_b200 as pkg
    if not torch.cuda.is_available():
        sys.exit("net_mlp_policy_bench.py needs a CUDA device")
    info = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    peak = sms * 128 * 2 * info["clocks_max_sm_mhz"] * 1e6
    res = dict(card=info, sms=sms, fp32_cuda_core_peak_flops=peak, flop_per_env_step=FLOP_PER_STEP, sizes=[])
    net = None
    for lg in [int(x) for x in args.sizes.split(",")]:
        N = 1 << lg
        env = pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled", info_level=0)
        T = int(env.num_periods)
        high = env.single_action_space.high
        if net is None:
            net = sb3_default_actor(torch, env.obs_dim, high)
        high_t = torch.as_tensor(high, device="cuda")

        def fused(ep):
            return env.rollout(net, seed=5000, episode=ep, want=("ep_return", "summary"))

        def step_loop():
            obs, _ = env.reset(seed=5000)
            ret = torch.zeros(N, dtype=torch.float64, device="cuda")
            with torch.no_grad():
                for _ in range(T):
                    a = torch.minimum(net(obs).clamp_min(0.0), high_t)    # SB3 predict: clip to [low, high]
                    obs, r, _, _, _ = env.step(a)
                    ret += r
            return ret

        # agreement on the same seed and episode (the step loop always plays episode 0 of seed 5000)
        ra = fused(0)["ep_return"].clone()
        rb = step_loop()
        torch.cuda.synchronize()
        agree = float((ra == rb).double().mean())
        for f in (fused, step_loop):      # warm-up
            f(0) if f is fused else f()
        torch.cuda.synchronize()
        times = {"fused": [], "step_api": []}
        for _ in range(args.reps):
            for name in ("fused", "step_api"):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                inner = 3 if name == "fused" else 1
                s.record()
                for k in range(inner):
                    fused(k) if name == "fused" else step_loop()
                e.record()
                e.synchronize()
                times[name].append(s.elapsed_time(e) / 1e3 / inner)
        best = {k: min(v) for k, v in times.items()}
        row = dict(log2_envs=lg, envs=N, periods=T, seconds_per_rollout=best, all_seconds=times,
                   env_steps_per_s={k: N * T / v for k, v in best.items()},
                   speedup_fused_over_step_api=best["step_api"] / best["fused"],
                   fused_fp32_flops=N * T * FLOP_PER_STEP / best["fused"],
                   fused_fraction_of_fp32_peak=N * T * FLOP_PER_STEP / best["fused"] / peak,
                   ep_return_bitwise_equal_fraction=agree)
        res["sizes"].append(row)
        env.close()
        del env
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
