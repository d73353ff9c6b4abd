"""GPU parity tests of the serial multi-echelon env (csrc/invmgmt.cu) through the C ABI:
CUDA step / fused rollout vs the golden vectors of the reference and vs the C oracle."""
import os

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from helpers import ROOT, golden_files, ids, load_golden, seq_sum

pytestmark = pytest.mark.gpu
INV = golden_files("invmgmt_")


def _torch():
    import torch
    return torch


def _mk(meta, n, **kw):
    cls = pkg.InvManagementBacklogEnv if meta["backlog"] else pkg.InvManagementLostSalesEnv
    return cls(num_envs=n, device="cuda:0", **meta["cfg"], **kw)


@pytest.mark.parametrize("wide", [False, True], ids=["int32state", "int64state"])
@pytest.mark.parametrize("path", INV, ids=ids(INV))
def test_step_matches_reference(path, wide):
    torch = _torch()
    g, meta = load_golden(path)
    E = len(g["seeds"])
    env = _mk(meta, E, wide_state=wide, autoreset_mode="disabled")
    T = env.num_periods
    obs, _ = env.reset(seed=0)
    assert np.array_equal(obs.cpu().numpy(), g["obs"][:, 0])
    float_actions = meta["policy"] == "wild"
    for t in range(T):
        a = g["actions"][:, t]
        a = torch.from_numpy(a if float_actions else a.astype(np.int64)).cuda()
        obs, r, term, trunc, info = env.step(a, demand=torch.from_numpy(g["D"][:, t]).cuda())
        assert np.array_equal(obs.cpu().numpy(), g["obs"][:, t + 1]), t
        assert np.array_equal(r.cpu().numpy(), g["reward"][:, t]), t      # bit-exact float64
        assert np.array_equal(trunc.cpu().numpy(), g["truncated"][:, t])
        assert not term.any()
        assert np.array_equal(info["sales"].cpu().numpy(), g["S"][:, t])
        unf = g["B"][:, t + 1] if meta["backlog"] else g["LS"][:, t]
        assert np.array_equal(info["unfulfilled"].cpu().numpy(), unf)
        assert np.array_equal(info["period_profit"].cpu().numpy(), g["profit"][:, t])
        assert np.array_equal(info["demand_realized"].cpu().numpy(), g["D"][:, t])
        I, B, per = env.export_state()
        assert np.array_equal(I.cpu().numpy(), g["I"][:, t + 1])
        assert np.array_equal(B.cpu().numpy(), g["B"][:, t + 1])
        assert (per.cpu().numpy() == t + 1).all()
    assert env.errors() == 0
    env.close()


@pytest.mark.parametrize("path", INV, ids=ids(INV))
def test_rollout_replay_matches_reference(path):
    g, meta = load_golden(path)
    E = len(g["seeds"])
    env = _mk(meta, E)
    acts = np.trunc(np.maximum(g["actions"], 0)).astype(np.int64)  # rollout takes int64 actions
    out = env.rollout("actions", actions=acts, demand=g["D"],
                      want=("ep_return", "stats", "reward_traj", "final_I", "final_B", "summary"))
    _torch().cuda.synchronize()
    assert np.array_equal(out["reward_traj"].cpu().numpy(), g["reward"])
    ret = out["ep_return"].cpu().numpy()
    for e in range(E):
        assert ret[e] == seq_sum(g["reward"][e])
    assert np.array_equal(out["final_I"].cpu().numpy(), g["I"][:, -1])
    assert np.array_equal(out["final_B"].cpu().numpy(), g["B"][:, -1])
    st = out["stats"].cpu().numpy()
    assert np.array_equal(st[:, 0], g["S"][:, :, 0].sum(axis=1))
    assert np.array_equal(st[:, 1], g["D"].sum(axis=1))
    unf0 = (g["B"][:, 1:, 0] if meta["backlog"] else g["LS"][:, :, 0]).sum(axis=1)
    assert np.array_equal(st[:, 2], unf0)
    assert np.array_equal(st[:, 3], np.maximum(g["I"][:, 1:], 0).sum(axis=(1, 2)))
    summ = out["summary"].cpu().numpy()
    assert summ[0] == E and np.isclose(summ[1], ret.sum(), rtol=1e-12)
    # time-major layouts give the same result
    out2 = env.rollout("actions", actions=np.ascontiguousarray(acts.transpose(1, 0, 2)),
                       demand=np.ascontiguousarray(g["D"].T), time_major=True, want=("ep_return",))
    assert np.array_equal(out2["ep_return"].cpu().numpy(), ret)
    if meta["policy"] == "base_stock":
        out3 = env.rollout("base_stock", demand=g["D"], want=("ep_return", "reward_traj", "final_I"))
        assert np.array_equal(out3["reward_traj"].cpu().numpy(), g["reward"])
        assert np.array_equal(out3["final_I"].cpu().numpy(), g["I"][:, -1])
    env.close()


@pytest.mark.parametrize("backlog", [True, False])
def test_large_batch_vs_oracle(backlog):
    """Default config, 20k instances (tail tile included), random actions / demand: step API and fused rollout
    against the C oracle on a sample of instances, and against each other on all of them."""
    from oracle import oracle
    torch = _torch()
    N = 20011
    cls = pkg.InvManagementBacklogEnv if backlog else pkg.InvManagementLostSalesEnv
    env = cls(num_envs=N, device="cuda:0")
    T, n = env.num_periods, env.num_stages - 1
    rng = np.random.default_rng(3)
    acts = rng.integers(0, env.supply_capacity + 1, size=(N, T, n)).astype(np.int64)
    dem = rng.poisson(20, size=(N, T)).astype(np.int64)
    a_d, d_d = torch.from_numpy(acts).cuda(), torch.from_numpy(dem).cuda()
    obs, _ = env.reset(seed=3)
    rew = torch.zeros((N, T), dtype=torch.float64, device="cuda")
    obs_hist = []
    for t in range(T):
        obs, r, term, trunc, info = env.step(a_d[:, t], demand=d_d[:, t])
        rew[:, t] = r
        if t in (0, 9, T - 1):
            obs_hist.append((t, obs.clone()))
    out = env.rollout("actions", actions=a_d, demand=d_d, want=("ep_return", "reward_traj", "final_I", "final_B"))
    assert torch.equal(out["reward_traj"], rew)
    I, B, per = env.export_state()
    assert torch.equal(I, out["final_I"]) and torch.equal(B, out["final_B"])
    rew = rew.cpu().numpy()
    for e in list(range(0, N, 997)) + [N - 1]:
        o = oracle.invmgmt_episode(env.params, actions=acts[e], demand=dem[e])
        assert np.array_equal(o["reward"], rew[e])
        for t, ob in obs_hist:
            assert np.array_equal(o["obs"][t + 1], ob[e].cpu().numpy())
    env.close()


def test_sampled_demand_consistent_between_step_and_rollout():
    """On-device Philox demand: the step API and the fused rollout draw the same stream for (seed, env, period),
    and the stream does not depend on batch size or env_offset sharding."""
    torch = _torch()
    N = 3000
    env = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0")
    T, n = env.num_periods, env.num_stages - 1
    acts = torch.zeros((N, n), dtype=torch.int64, device="cuda") + 20
    env.reset(seed=5000)
    dem = torch.zeros((N, T), dtype=torch.int64, device="cuda")
    rew = torch.zeros((N, T), dtype=torch.float64, device="cuda")
    for t in range(T):
        _, r, _, _, info = env.step(acts)
        dem[:, t] = info["demand_realized"]
        rew[:, t] = r
    out = env.rollout("actions", actions=acts[:, None, :].expand(N, T, n).contiguous(), seed=5000,
                      want=("ep_return", "stats", "reward_traj"))
    assert torch.equal(out["stats"][:, 1], dem.sum(dim=1))
    assert torch.equal(out["reward_traj"], rew)
    # sharding invariance: instances [1000, 1500) simulated alone reproduce the same numbers
    sub = pkg.InvManagementLostSalesEnv(num_envs=500, device="cuda:0", env_offset=1000)
    o2 = sub.rollout("actions", actions=acts[:500, None, :].expand(500, T, n).contiguous(), seed=5000,
                     want=("ep_return", "stats"))
    assert torch.equal(o2["ep_return"], out["ep_return"][1000:1500])
    assert torch.equal(o2["stats"], out["stats"][1000:1500])
    # a different episode index gives a different demand path
    o3 = env.rollout("actions", actions=acts[:, None, :].expand(N, T, n).contiguous(), seed=5000, episode=1,
                     want=("stats",))
    assert not torch.equal(o3["stats"][:, 1], dem.sum(dim=1))
    env.close(); sub.close()


def test_on_device_policies():
    """base-stock and random-action rollouts: sane statistics and agreement with the oracle's base-stock driver
    when it is fed the demand the device sampled."""
    from oracle import oracle
    torch = _torch()
    N = 4096
    env = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled")
    T, n = env.num_periods, env.num_stages - 1
    # recover the device's demand stream through the step API (actions are irrelevant to the demand draw)
    env.reset(seed=4000)
    dem = torch.zeros((N, T), dtype=torch.int64, device="cuda")
    for t in range(T):
        _, _, _, _, info = env.step(torch.zeros((N, n), dtype=torch.int64, device="cuda"))
        dem[:, t] = info["demand_realized"]
    out = env.rollout("base_stock", seed=4000, want=("ep_return", "stats", "final_I", "final_B", "summary"))
    dem_h = dem.cpu().numpy()
    ret = out["ep_return"].cpu().numpy()
    for e in range(0, N, 211):
        o = oracle.invmgmt_episode(env.params, policy="base_stock", demand=dem_h[e])
        assert ret[e] == seq_sum(o["reward"])
        assert np.array_equal(out["final_I"][e].cpu().numpy(), o["I"][-1])
        assert np.array_equal(out["final_B"][e].cpu().numpy(), o["B"][-1])
    summ = out["summary"].cpu().numpy()
    assert summ[0] == N and np.isclose(summ[1], ret.sum(), rtol=1e-12) and summ[4] == dem_h.sum()
    assert 15 < dem_h.mean() < 25
    r = env.rollout("random", seed=1, want=("ep_return", "stats", "summary"))
    assert np.isfinite(r["ep_return"].cpu().numpy()).all()
    env.close()


def test_autoreset_modes():
    torch = _torch()
    N, cfg = 300, dict(periods=4, I0=[10, 10], p=5, r=[3, 2, 1], k=[1, 1, 1], h=[0.5, 0.2], c=[15, 20], L=[1, 2],
                       dist_param={"mu": 8})
    a = torch.full((N, 2), 7, dtype=torch.int64, device="cuda")
    # next_step: the call after truncation returns the reset observation, reward 0, flags False
    env = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="next_step", **cfg)
    obs0 = env.reset(seed=9)[0].clone()
    for t in range(4):
        obs, r, term, trunc, _ = env.step(a)
    assert trunc.all()
    last = obs.clone()
    obs, r, term, trunc, _ = env.step(a)
    assert torch.equal(obs, obs0) and (r == 0).all() and not trunc.any()
    assert not torch.equal(last, obs0)
    obs, r, term, trunc, _ = env.step(a)
    assert (env.period == 1).all()
    # same_step: reset inside the truncating step, terminal observation in info['final_obs']
    env2 = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="same_step", **cfg)
    env2.reset(seed=9)
    for t in range(4):
        obs2, r2, term2, trunc2, info2 = env2.step(a)
    assert trunc2.all() and torch.equal(obs2, obs0) and torch.equal(info2["final_obs"], last)
    assert (env2.period == 0).all()
    # disabled: stepping past the end raises like the reference
    env3 = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled", **cfg)
    env3.reset(seed=9)
    for t in range(5):
        env3.step(a)
    with pytest.raises(IndexError):
        env3.check_errors()
    # partial reset through a mask
    env3.reset(options={"reset_mask": (torch.arange(N) % 2 == 0)})
    per = env3.period.cpu().numpy()
    assert (per[::2] == 0).all() and (per[1::2] == 4).all()
    for e in (env, env2, env3):
        e.close()


def test_int32_range_guard():
    torch = _torch()
    env = pkg.InvManagementBacklogEnv(num_envs=64, device="cuda:0")
    env.reset(seed=0)
    env.step(torch.full((64, 3), 2**40, dtype=torch.int64, device="cuda"))
    with pytest.raises(OverflowError):
        env.check_errors()
    env.close()


def test_no_bulk_path_matches(monkeypatch):
    """The cooperative (non-TMA) tile path is used for tail tiles; make sure a ragged batch is exact."""
    torch = _torch()
    g, meta = load_golden(INV[1])
    env = _mk(meta, 131)  # one full 128-tile + a 3-env tail
    T = env.num_periods
    reps = 131 // len(g["seeds"]) + 1
    acts = np.tile(g["actions"], (reps, 1, 1))[:131].astype(np.int64)
    dem = np.tile(g["D"], (reps, 1))[:131]
    ref_obs = np.tile(g["obs"], (reps, 1, 1))[:131]
    env.reset(seed=0)
    for t in range(T):
        obs, *_ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
        assert np.array_equal(obs.cpu().numpy(), ref_obs[:, t + 1])
    env.close()


def test_evaluate_pipelined_host_results():
    """env.evaluate(): double-buffered rollouts with results in pinned host memory == plain rollouts, episode by
    episode; int32 statistics equal the int64 ones."""
    torch = _torch()
    N = 5000
    env = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0")
    ref = []
    for ep in range(5):
        o = env.rollout("base_stock", seed=5000, episode=ep, want=("ep_return", "stats", "summary"))
        ref.append({k: v.cpu().clone() for k, v in o.items()})
    got = []
    for res in env.evaluate("base_stock", episodes=5, seed=5000, want=("ep_return", "stats32", "summary")):
        assert res["ep_return"].is_pinned() and res["ep_return"].device.type == "cpu"
        got.append({k: v.clone() for k, v in res.items()})
    assert len(got) == 5
    for a, b in zip(ref, got):
        assert torch.equal(a["ep_return"], b["ep_return"]) and torch.equal(a["summary"], b["summary"])
        assert torch.equal(a["stats"], b["stats32"].long())
    assert not torch.equal(got[0]["ep_return"], got[1]["ep_return"])     # different episodes, different demand
    env.close()


@pytest.mark.parametrize("path", [p for p in INV if "default_lost_random" in p or "zerolt_backlog_wild" in p],
                         ids=lambda p: p.split("/")[-1][:-4])
def test_history_buffers_match_reference_arrays(path):
    """record_history=True: the batched I/B/R/S/LS/D/P/action_log arrays equal the reference's per-episode arrays."""
    torch = _torch()
    g, meta = load_golden(path)
    env = _mk(meta, len(g["seeds"]), autoreset_mode="disabled", record_history=True)
    env.reset(seed=0)
    floats = meta["policy"] == "wild"
    for t in range(env.num_periods):
        a = g["actions"][:, t]
        env.step(torch.from_numpy(a if floats else a.astype(np.int64)).cuda(), demand=torch.from_numpy(g["D"][:, t]).cuda())
    for name in ("I", "B", "R", "S", "LS", "D", "action_log"):
        assert np.array_equal(getattr(env, name).cpu().numpy(), g[name]), name
    assert np.array_equal(env.P.cpu().numpy(), g["reward"])
    env.close()


@pytest.mark.parametrize("case", [-1] + list(range(8 * max(1, int(__import__("os").environ.get("ORGYM_STRESS", "1"))))))
def test_specialised_rollout_matches_ahead_of_time_kernel(case, monkeypatch):
    """The rollout kernels generated per configuration at run time (invmgmt_jit.cu: rings in registers, straight-line
    periods) must reproduce the ahead-of-time kernel bit for bit: returns, statistics, summary, both policies."""
    torch = _torch()
    rng = np.random.default_rng(500 + case)
    if case == -1:
        cfg = dict(alpha=1e-10)  # exact profit, but alpha**29 * 2^-29 is too small to scale: the fused multiply-add form
    elif case == 0:
        cfg = {}
    elif case == 1:
        cfg = dict(dist=2, dist_param={"n": 40, "p": 0.45})
    else:
        n = int(rng.integers(1, 7))
        L = rng.integers(0, 7, n)
        # every other case uses coefficients on a 1/8 grid: coarse enough for the generator's proof that the profit
        # arithmetic never rounds, which switches it to integer arithmetic on coefficient / quantum (the rest keeps the
        # reference order)
        grid = (lambda a: (np.round(np.asarray(a) * 8) / 8)) if case % 4 >= 2 else (lambda a: np.asarray(a).round(3))
        cfg = dict(periods=int(rng.integers(2, 65)), I0=rng.integers(0, 200, n).tolist(), p=float(grid(rng.uniform(5, 40))),
                   r=grid(np.sort(rng.uniform(0.5, 30, n + 1))[::-1]).tolist(), k=grid(rng.uniform(0, 1, n + 1)).tolist(),
                   h=grid(rng.uniform(0, 0.5, n)).tolist(), c=rng.integers(1, 300, n).tolist(), L=L.tolist(),
                   dist_param={"mu": float(rng.integers(1, 50))}, alpha=float(rng.uniform(0.8, 1.0)))
    cls = pkg.InvManagementBacklogEnv if case % 2 else pkg.InvManagementLostSalesEnv
    N = 1000 + case
    want = ("ep_return", "stats", "stats32", "summary")
    outs = {}
    for mode in ("jit", "aot"):
        monkeypatch.setenv("ORGYM_INV_JIT", "1" if mode == "jit" else "0")
        env = cls(num_envs=N, device="cuda:0", env_offset=17, **cfg)
        res = []
        for pol, kw in (("base_stock", dict(safety_factor=1.0)), ("base_stock", dict(safety_factor=2.0)), ("random", {})):
            o = env.rollout(pol, seed=99, episode=3, want=want, **kw)
            res.append({k: v.cpu().numpy().copy() for k, v in o.items()})
        assert env.rollout_specialised == (mode == "jit")
        # outputs the specialised kernels do not produce fall back to the ahead-of-time kernel transparently
        o = env.rollout("base_stock", seed=99, episode=3, safety_factor=1.0, want=("ep_return", "reward_traj"))
        assert np.array_equal(o["ep_return"].cpu().numpy(), res[0]["ep_return"])
        outs[mode] = res
        env.close()
    for a, b in zip(outs["jit"], outs["aot"]):
        for k in want:
            assert np.array_equal(a[k], b[k]), (case, k)


@pytest.mark.parametrize("cls_name", ["InvManagementLostSalesEnv", "InvManagementBacklogEnv"])
def test_specialised_rollout_kernels_vs_oracle_at_bench_config(cls_name, monkeypatch):
    """The kernels bench.py times (inv_jit_rollout_bs / inv_jit_rollout_rnd at the env defaults, seed 5000) checked
    DIRECTLY against the oracle: the device's demand is recovered through the step API, the random policy's actions
    from an independent numpy restatement of its Philox stream, and the oracle replays both.  Only outputs the
    specialised kernels produce are requested, and ORGYM_INV_JIT=2 makes a failed specialisation an error."""
    from oracle import oracle
    from helpers import device_random_actions
    torch = _torch()
    monkeypatch.setenv("ORGYM_INV_JIT", "2")
    N, seed, off, ep = 8192, 5000, 3 << 20, 0
    env = getattr(pkg, cls_name)(num_envs=N, device="cuda:0", env_offset=off, autoreset_mode="disabled")
    T, n = env.num_periods, env.num_stages - 1
    env.reset(seed=seed)
    dem = torch.zeros((N, T), dtype=torch.int64, device="cuda")
    zero = torch.zeros((N, n), dtype=torch.int64, device="cuda")
    for t in range(T):
        dem[:, t] = env.step(zero)[4]["demand_realized"]
    dem = dem.cpu().numpy()
    pick = np.r_[0:16, np.random.default_rng(1).choice(N, 80, replace=False), N - 16:N]
    want = ("ep_return", "stats", "stats32", "summary")

    def check(out, episodes):
        ret, st = out["ep_return"].cpu().numpy(), out["stats"].cpu().numpy()
        assert np.array_equal(st, out["stats32"].cpu().numpy().astype(np.int64))
        for e, o in zip(pick, episodes):
            assert ret[e] == seq_sum(o["reward"]), e
            unf0 = (o["B"][1:, 0] if env.params.backlog else o["LS"][:, 0]).sum()
            assert st[e].tolist() == [o["S"][:, 0].sum(), dem[e].sum(), unf0, np.maximum(o["I"][1:], 0).sum()], e
        summ = out["summary"].cpu().numpy()
        assert summ[0] == N and np.isclose(summ[1], ret.sum(), rtol=1e-12) and summ[4] == dem.sum()

    out = env.rollout("base_stock", seed=seed, episode=ep, safety_factor=1.0, want=want)
    assert env.rollout_specialised
    check(out, [oracle.invmgmt_episode(env.params, policy="base_stock", demand=dem[e]) for e in pick])
    out = env.rollout("random", seed=seed, episode=ep, want=want)
    acts = device_random_actions(seed, off + pick, ep, T, env.params.supply_capacity)
    assert acts.min() >= 0 and (acts.max(axis=(0, 1)) <= np.asarray(env.params.supply_capacity)).all()
    check(out, [oracle.invmgmt_episode(env.params, actions=acts[i].astype(np.float64), demand=dem[e])
                for i, e in enumerate(pick)])
    env.close()


def test_evaluation_report_reproduces_the_reference_summary_row():
    """The reference's per-agent summary (mean / median / std / min / max of TotalReward, mean service level, stock-out
    quantity and ending inventory -- benchmark_InvManagementBacklogEnv.py:493-504) from one fused rollout, on device."""
    import pandas as pd
    N = 20001
    env = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0")
    out = env.rollout("base_stock", seed=4000, safety_factor=1.0, want=("ep_return", "stats", "summary"))
    rep = pkg.evaluation_report(out, env.num_periods)
    ret, st = out["ep_return"].cpu().numpy(), out["stats"].cpu().numpy().astype(np.float64)
    sl = np.where(st[:, 1] > 1e-6, st[:, 0] / np.maximum(1e-6, st[:, 1]), 1.0)
    df = pd.DataFrame(dict(TotalReward=ret, AvgServiceLevel=sl, TotalStockoutQty=st[:, 2], AvgEndingInv=st[:, 3] / env.num_periods))
    assert rep["SuccessfulEpisodes"] == N
    assert rep["MedianReward"] == df.TotalReward.median() and rep["MinReward"] == ret.min() and rep["MaxReward"] == ret.max()
    assert np.isclose(rep["AvgReward"], ret.mean(), rtol=1e-12) and np.isclose(rep["StdReward"], df.TotalReward.std(), rtol=1e-10)
    assert np.isclose(rep["AvgServiceLevel"], sl.mean(), rtol=1e-12)
    assert np.isclose(rep["AvgStockoutQty"], st[:, 2].mean(), rtol=1e-12)
    assert np.isclose(rep["AvgEndInv"], df.AvgEndingInv.mean(), rtol=1e-12)
    # the in-kernel summary agrees on what it carries (means, population std)
    d = pkg.describe_summary(out["summary"].cpu().numpy(), env.num_periods)
    assert d["episodes"] == N and np.isclose(d["TotalReward_mean"], rep["AvgReward"], rtol=1e-12)
    assert np.isclose(d["TotalStockoutQty_mean"], rep["AvgStockoutQty"], rtol=1e-12)
    # order statistic by bisection == sort
    assert pkg.kth_smallest(out["ep_return"], 1234) == np.sort(ret)[1234]
    env.close()


def _report_reference(ret, st, periods):
    """pandas restatement of process_and_report_results (benchmark_InvManagementBacklogEnv.py:493-504)."""
    import pandas as pd
    st = st.astype(np.float64)
    sl = np.where(st[:, 1] > 1e-6, st[:, 0] / np.maximum(1e-6, st[:, 1]), 1.0)
    df = pd.DataFrame(dict(TotalReward=ret, AvgServiceLevel=sl, TotalStockoutQty=st[:, 2], AvgEndingInv=st[:, 3] / periods))
    return dict(SuccessfulEpisodes=len(ret), AvgReward=df.TotalReward.mean(), MedianReward=df.TotalReward.median(),
                StdReward=df.TotalReward.std(), MinReward=df.TotalReward.min(), MaxReward=df.TotalReward.max(),
                AvgServiceLevel=df.AvgServiceLevel.mean(), AvgStockoutQty=df.TotalStockoutQty.mean(),
                AvgEndInv=df.AvgEndingInv.mean())


@pytest.mark.parametrize("case", ["rollout_odd", "rollout_even", "mixed_sign", "constant", "two_values", "n1", "n2", "n3",
                                  "ties", "wide_range", "float_stats", "big"])
def test_device_report_kernels_match_pandas(case):
    """csrc/report.cu (radix-select median, two-pass std, min / max, service-level means) against pandas on rollout
    outputs and on adversarial synthetic inputs: mixed signs and many binades (first-digit histogram path), all-equal
    returns, central order statistics in different histogram bins, tiny batches, heavy ties, every stats dtype."""
    torch = _torch()
    rng = np.random.default_rng(11)
    T = 30
    if case.startswith("rollout"):
        N = 20001 if case == "rollout_odd" else 65536
        env = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0")
        out = env.rollout("base_stock", seed=4000, safety_factor=1.0, want=("ep_return", "stats32"))
        ret, st = out["ep_return"], out["stats32"]
    else:
        n = dict(mixed_sign=50001, constant=4097, two_values=2, n1=1, n2=2, n3=3, ties=30000, wide_range=77777,
                 float_stats=12345, big=3_000_001)[case]
        if case == "mixed_sign":
            r = rng.normal(0.0, 500.0, n)
        elif case == "constant":
            r = np.full(n, 1234.5)
        elif case == "two_values":
            r = np.array([1.0, 1e10])
        elif case == "ties":
            r = rng.integers(0, 7, n).astype(np.float64) * 0.25 - 0.5
        elif case == "wide_range":
            r = np.exp(rng.uniform(-30, 30, n)) * rng.choice([-1.0, 1.0], n)
        else:
            r = rng.normal(3900.0, 300.0, n)
        s = rng.integers(0, 900, size=(n, 4))
        s[rng.random(n) < 0.01, 1] = 0                              # episodes without demand: service level 1.0
        ret = torch.from_numpy(r).cuda()
        if case == "float_stats":
            st = torch.from_numpy(s.astype(np.float64)).cuda()
        elif case in ("ties", "big"):
            st = torch.from_numpy(s.astype(np.int32)).cuda()
        else:
            st = torch.from_numpy(s.astype(np.int64)).cuda()
    rep, scratch = pkg.evaluation_report_device({"ep_return": ret, "stats": st}, T)
    got = pkg.report_to_dict(rep)
    rep2, _ = pkg.evaluation_report_device({"ep_return": ret, "stats": st}, T, report=torch.zeros_like(rep), scratch=scratch)
    assert torch.equal(rep.view(torch.int64), rep2.view(torch.int64))   # bitwise reproducible, buffers reusable
    want = _report_reference(ret.cpu().numpy(), st.cpu().numpy(), T)
    assert got["SuccessfulEpisodes"] == want["SuccessfulEpisodes"]
    for k in ("MedianReward", "MinReward", "MaxReward"):
        assert got[k] == want[k], (k, got[k], want[k])
    for k in ("AvgReward", "AvgServiceLevel", "AvgStockoutQty", "AvgEndInv"):
        assert np.isclose(got[k], want[k], rtol=1e-11, atol=1e-9), (k, got[k], want[k])
    if want["SuccessfulEpisodes"] > 1:
        assert np.isclose(got["StdReward"], want["StdReward"], rtol=1e-9, atol=1e-12), (got["StdReward"], want["StdReward"])
    else:
        assert np.isnan(got["StdReward"])


def test_evaluate_default_product_is_the_device_report():
    """env.evaluate() default: per episode index the reference's summary row, computed on the device; only 16 numbers
    cross PCIe.  Same numbers as the torch / pandas path on the per-episode tensors; dicts stay valid while the next
    one is being consumed (three buffer sets)."""
    torch = _torch()
    N = 10000
    env = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0")
    held = []
    for k, res in enumerate(env.evaluate("base_stock", episodes=5, seed=5000, safety_factor=1.0)):
        assert set(res) == {"report"} and not res["report"].is_cuda
        held.append((res, res["report"].clone()))
        if k >= 1:                                   # the previous result has not been overwritten yet
            assert torch.equal(held[k - 1][0]["report"], held[k - 1][1])
        o = env.rollout("base_stock", seed=5000, episode=k, safety_factor=1.0, want=("ep_return", "stats"))
        want = pkg.evaluation_report(o, env.num_periods)
        got = pkg.report_to_dict(res["report"])
        assert got["MedianReward"] == want["MedianReward"] and got["MinReward"] == want["MinReward"]
        assert np.isclose(got["AvgReward"], want["AvgReward"], rtol=1e-12)
        assert np.isclose(got["StdReward"], want["StdReward"], rtol=1e-10)
        assert np.isclose(got["AvgServiceLevel"], want["AvgServiceLevel"], rtol=1e-12)
    env.close()


def test_explicit_specialisation_and_strict_mode(monkeypatch):
    """orgym_invmgmt_specialise builds the kernel for a policy ahead of time and says why when it cannot;
    ORGYM_INV_JIT=2 turns a rollout that cannot get its specialised kernel into an error instead of a silent fall-back
    to the 2-3x slower ahead-of-time kernel; ORGYM_INV_JIT=0 never specialises."""
    from or_gym_inventory_b200._capi import OrgymError, E_UNSUPPORTED
    env = pkg.InvManagementLostSalesEnv(num_envs=500, device="cuda:0")
    assert env.specialise("base_stock", safety_factor=1.0) and env.rollout_specialised
    assert env.specialise("random")
    a = env.rollout("base_stock", seed=3, safety_factor=1.0, want=("ep_return",))["ep_return"].clone()
    assert env.rollout_specialised
    # a second safety factor is a second kernel variant (levels are literals); results differ, both specialised
    b = env.rollout("base_stock", seed=3, safety_factor=1.5, want=("ep_return",))["ep_return"].clone()
    assert env.rollout_specialised and not _torch().equal(a, b)
    # non-integer levels cannot be specialised: the ahead-of-time kernel evaluates them in float64
    with pytest.raises(OrgymError) as ei:
        env.specialise("base_stock", safety_factor=1.013)
    assert ei.value.code == E_UNSUPPORTED
    env.rollout("base_stock", seed=3, safety_factor=1.013, want=("ep_return",))
    assert not env.rollout_specialised
    env.close()
    # seven stages are outside the specialiser's range
    big = dict(I0=[10] * 7, r=[9, 8, 7, 6, 5, 4, 3, 2], k=[0.1] * 8, h=[0.1] * 7, c=[10] * 7, L=[1] * 7)
    env = pkg.InvManagementBacklogEnv(num_envs=100, device="cuda:0", **big)
    with pytest.raises(OrgymError) as ei:
        env.specialise("base_stock", safety_factor=1.0, mu=10)
    assert ei.value.code == E_UNSUPPORTED and "specialiser" in str(ei.value)
    ref = env.rollout("base_stock", seed=1, safety_factor=1.0, mu=10, want=("ep_return",))["ep_return"].clone()
    assert not env.rollout_specialised
    monkeypatch.setenv("ORGYM_INV_JIT", "2")
    with pytest.raises(OrgymError):
        env.rollout("base_stock", seed=1, safety_factor=1.0, mu=10, want=("ep_return",))
    monkeypatch.setenv("ORGYM_INV_JIT", "0")
    assert _torch().equal(env.rollout("base_stock", seed=1, safety_factor=1.0, mu=10, want=("ep_return",))["ep_return"], ref)
    env.close()
    env = pkg.InvManagementLostSalesEnv(num_envs=500, device="cuda:0")
    c = env.rollout("base_stock", seed=3, safety_factor=1.0, want=("ep_return",))["ep_return"]
    assert not env.rollout_specialised and _torch().equal(a, c)      # ahead-of-time kernel: the same numbers
    env.close()


def test_bench_dump_outputs_are_the_last_timed_rollout(tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last rollout of the last timed step returned (bench step k runs
    episodes k * inner + r, timed steps are k = 100 .. 100 + K - 1), the same arrays from run to run."""
    import json
    import subprocess
    import sys
    N, K = 4096, 2
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", "1", "--inner", "1",
                            "--envs-per-gpu", str(N), "--no-extras", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout)["steps"] == K
        dumps.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    assert sorted(dumps[0]) == ["ep_return", "stats", "summary"]
    for name, a in dumps[0].items():
        assert a.dtype == np.float64 and np.array_equal(a, dumps[1][name]), name
    env = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0")
    out = env.rollout("base_stock", seed=5000, episode=100 + K - 1, safety_factor=1.0, want=("ep_return", "stats", "summary"))
    for name, t in out.items():
        assert np.array_equal(dumps[0][name], t.cpu().numpy().astype(np.float64)), name
    env.close()
