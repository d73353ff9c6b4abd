"""GPU suite for the MLP actor policy of the serial env's fused rollout (inv_mlp_rollout_kernel): the dynamics it drives
are the env's own (replay through the 'actions' rollout and the CPU oracle), the orders it places are the network's
(float64 forward pass on the observations the step API returns), results do not depend on batching or sharding, and
evaluate() reports on it like on the on-device heuristics."""
import ctypes as C

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from or_gym_inventory_b200 import _capi
from helpers import seq_sum

pytestmark = pytest.mark.gpu
# float32 network vs float64 recomputation: an output is a near-tie when |y - nearest integer| <= REL_TOL * max(1, mag),
# mag = |b_L| + sum_k |W_L,k h_k| of the last layer in float64 -- float32 dot-product error scales with the magnitude of
# the summands, not of the (possibly cancelled) result; 1e-4 is ~100x the last layer's own worst case (K u <= 128 * 2^-24)
# and leaves room for the error the hidden layers pass on (tanh / ReLU are 1-Lipschitz)
REL_TOL = 1e-4
ALL_OUT = ("ep_return", "stats", "stats32", "summary", "reward_traj", "final_I", "final_B", "action_traj")

CONFIGS = {
    "lost": (pkg.InvManagementLostSalesEnv, {}),
    "backlog_wide": (pkg.InvManagementBacklogEnv, dict(wide_state=True)),
    "zero_lead": (pkg.InvManagementBacklogEnv, dict(I0=[50, 60], r=[1.5, 1.0, 0.5], k=[0.1, 0.05, 0.02], h=[0.1, 0.05],
                                                    c=[80, 70], L=[0, 3], periods=12, alpha=0.9)),
    "lt_max0": (pkg.InvManagementLostSalesEnv, dict(L=[0, 0, 0])),
    "one_stage": (pkg.InvManagementBacklogEnv, dict(I0=[40], r=[3.0, 1.0], k=[0.2, 0.1], h=[0.1], c=[60], L=[2],
                                                    periods=20)),
    "seven_stages": (pkg.InvManagementLostSalesEnv, dict(I0=[30] * 7, r=[9, 8, 7, 6, 5, 4, 3, 2], k=[0.1] * 8, h=[0.05] * 7,
                                                         c=[60] * 7, L=[1, 0, 2, 1, 3, 1, 2], periods=15)),
}


def _torch():
    import torch
    return torch


def _seq(widths, act):
    nn = _torch().nn
    mods = []
    for i in range(len(widths) - 1):
        mods.append(nn.Linear(widths[i], widths[i + 1]))
        if i < len(widths) - 2:
            mods.append(act())
    return nn.Sequential(*mods)


def _sample_obs(env_cls, kw, N=256, seed=7):
    """Observations of random-order episodes (the range a network meets), float64 [N*T, obs_dim]."""
    torch = _torch()
    env = env_cls(num_envs=N, device="cuda:0", autoreset_mode="disabled", **kw)
    obs, _ = env.reset(seed=seed)
    c = torch.as_tensor(np.asarray(env.params.supply_capacity), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    rows = [obs.double().clone()]
    for _ in range(env.num_periods - 1):
        a = (torch.rand((N, len(c)), device="cuda", generator=g, dtype=torch.float64) * (c + 1)).long()
        rows.append(env.step(a)[0].double().clone())
    env.close()
    return torch.cat(rows)


def _net(env_cls, kw, widths, act="tanh", seed=0):
    """A network whose outputs span below 0, the interior and above c_i on the env's observations."""
    torch = _torch()
    torch.manual_seed(seed)
    P = pkg.InvManagementParams(**{k: v for k, v in kw.items() if k != "wide_state"})
    widths = (P.pipeline_length,) + tuple(widths) + (P.num_stages - 1,)
    net = _seq(widths, torch.nn.Tanh if act == "tanh" else torch.nn.ReLU).cuda()
    x = _sample_obs(env_cls, kw)
    with torch.no_grad():
        net[0].weight.mul_(0.02)
        h = net[:-1].double()(x) if len(net) > 1 else x
        net.float()
        last = net[-1]
        y = h @ last.weight.double().t()
        c = torch.as_tensor(np.asarray(P.supply_capacity, np.float64), device="cuda")
        s = (0.8 * c / y.std(0).clamp(min=1e-6)).float()
        last.weight.mul_(s[:, None])
        last.bias.copy_((0.5 * c - (y * s.double()).mean(0)).float())
    return net


def _order_up_to_net(P, width=64):
    """A (width, width) ReLU network that orders max(0, (L_i + 1) * 20 - I_i - sum of stage i's window) for every stage,
    exactly (integer inputs and weights): varied interior orders whatever the configuration."""
    torch = _torch()
    n, od = P.num_stages - 1, P.pipeline_length
    net = _seq((od, width, width, n), torch.nn.ReLU)
    with torch.no_grad():
        for lin in net[::2]:
            lin.weight.zero_()
            lin.bias.zero_()
        for i in range(n):
            net[0].weight[i, i::n] = -1.0
            net[0].bias[i] = 20.0 * (float(P.lead_time[i]) + 1.0)
            net[2].weight[i, i] = 1.0
            net[4].weight[i, i] = 1.0
    return net.cuda()


def _device_demand_and_obs(env_cls, kw, N, seed, actions):
    """Reset with `seed` and replay `actions` through the step API: per period the observation the policy saw (before
    the step) and the demand the device drew."""
    torch = _torch()
    env = env_cls(num_envs=N, device="cuda:0", autoreset_mode="disabled", **kw)
    T = env.num_periods
    obs, _ = env.reset(seed=seed)
    O = torch.zeros((N, T, obs.shape[1]), dtype=torch.int64, device="cuda")
    D = torch.zeros((N, T), dtype=torch.int64, device="cuda")
    for t in range(T):
        O[:, t] = obs
        obs, _, _, _, info = env.step(actions[:, t])
        D[:, t] = info["demand_realized"]
    env.close()
    return O, D


def _f64_actions(net, O, cap):
    """The contract's quantisation of a float64 forward pass: trunc(clip(y, 0, c)), NaN -> 0; plus the tie mask."""
    torch = _torch()
    import copy
    net64 = copy.deepcopy(net).double()
    with torch.no_grad():
        x = O.double().reshape(-1, O.shape[-1])
        h = net64[:-1](x) if len(net64) > 1 else x
        last = net64[-1]
        y = last(h)
        mag = h.abs() @ last.weight.abs().t() + (last.bias.abs() if last.bias is not None else 0.0)
        y, mag = (t.reshape(O.shape[0], O.shape[1], -1) for t in (y, mag))
    c = torch.as_tensor(np.asarray(cap, np.float64), device=y.device)
    q = torch.nan_to_num(torch.minimum(torch.clamp(y, min=0.0), c), nan=0.0).trunc().long()
    q = torch.where(torch.isnan(y), torch.zeros_like(q), q)
    near = (y - y.round()).abs() <= REL_TOL * torch.clamp(mag, min=1.0)
    tie = near & (y > -1.0) & (y < c + 1.0)
    return q, tie, y


@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_dynamics_are_the_envs_own(cfg):
    """An MLP rollout's state and rewards are exactly what the 'actions' rollout and the CPU oracle compute for the
    orders it placed (action_traj) under the device's demand."""
    from oracle import oracle
    torch = _torch()
    cls, kw = CONFIGS[cfg]
    N, seed = 777, 31
    env = cls(num_envs=N, device="cuda:0", **kw)
    net = _order_up_to_net(env.params)
    out = {k: v.clone() for k, v in env.rollout(net, seed=seed, want=ALL_OUT).items()}
    acts = out["action_traj"]
    c = np.asarray(env.params.supply_capacity)
    a = acts.cpu().numpy()
    assert a.min() >= 0 and (a.max(axis=(0, 1)) <= c).all() and ((a > 0) & (a < c)).any()
    rep = env.rollout("actions", actions=acts, seed=seed, want=ALL_OUT)
    for k in ALL_OUT:
        assert torch.equal(out[k], rep[k]), k
    P = env.params
    env.close()
    _, D = _device_demand_and_obs(cls, kw, N, seed, acts)
    dem = D.cpu().numpy()
    rt, ret = out["reward_traj"].cpu().numpy(), out["ep_return"].cpu().numpy()
    fI, fB = out["final_I"].cpu().numpy(), out["final_B"].cpu().numpy()
    for e in list(range(0, N, 97)) + [N - 1]:
        o = oracle.invmgmt_episode(P, actions=a[e].astype(np.float64), demand=dem[e])
        assert np.array_equal(o["reward"], rt[e]) and ret[e] == seq_sum(o["reward"]), e
        assert np.array_equal(o["I"][-1], fI[e]) and np.array_equal(o["B"][-1], fB[e]), e


NETS = [("tanh", (64, 64)), ("relu", (128,)), ("tanh", ()), ("relu", (17, 1, 128)), ("tanh", (128, 128)),
        ("tanh", (176, 176))]


@pytest.mark.parametrize("act, hidden", NETS, ids=[f"{a}-{'x'.join(map(str, h)) or 'linear'}" for a, h in NETS])
def test_policy_is_the_network(act, hidden):
    """Every order equals trunc(clip(y, 0, c)) of a float64 forward pass on the observation step() returns, except where
    y is a near-tie (REL_TOL: float32 rounding may fall either side of the integer); such exemptions stay below 0.5 %.
    The observations come from the device's own orders, so one flipped order does not cascade."""
    cls, kw = CONFIGS["lost"]
    N, seed = 2048, 5
    net = _net(cls, kw, hidden, act=act, seed=3)
    env = cls(num_envs=N, device="cuda:0")
    acts = env.rollout(net, seed=seed, want=("action_traj",))["action_traj"].clone()
    env.close()
    O, _ = _device_demand_and_obs(cls, kw, N, seed, acts)
    q, tie, y = _f64_actions(net, O, pkg.InvManagementParams().supply_capacity)
    diff = q != acts
    bad = diff & ~tie
    assert not bool(bad.any()), (int(bad.sum()), y[bad][:5].tolist(), acts[bad][:5].tolist())
    assert float(diff.double().mean()) < 0.005
    yc = y.cpu().numpy()
    assert (yc < 0).any() and (yc > np.asarray(pkg.InvManagementParams().supply_capacity)).any()


def test_nan_outputs_order_nothing():
    torch = _torch()
    net = _seq((33, 8, 3), torch.nn.Tanh).cuda()
    with torch.no_grad():
        net[-1].bias[1] = float("nan")
    env = pkg.InvManagementLostSalesEnv(num_envs=300, device="cuda:0")
    a = env.rollout(net, seed=2, want=("action_traj", "ep_return"))
    assert bool((a["action_traj"][:, :, 1] == 0).all()) and bool(torch.isfinite(a["ep_return"]).all())
    env.close()


@pytest.mark.parametrize("hidden", [(64, 64), (176, 176)])   # 64-env and 32-env sub-tiles
def test_results_do_not_depend_on_batching_or_sharding(hidden):
    torch = _torch()
    cls, kw = CONFIGS["lost"]
    net = _net(cls, kw, hidden, seed=4)
    full_n = 1000 + 7
    want = ("ep_return", "action_traj")
    env = cls(num_envs=full_n, device="cuda:0")
    ref = {k: v.clone() for k, v in env.rollout(net, seed=9, episode=2, want=want).items()}
    env.close()
    for N in (1, 31, 129):
        e = cls(num_envs=N, device="cuda:0")
        o = e.rollout(net, seed=9, episode=2, want=want)
        for k in want:
            assert torch.equal(o[k], ref[k][:N]), (N, k)
        e.close()
    a = cls(num_envs=500, device="cuda:0", env_offset=0)
    b = cls(num_envs=full_n - 500, device="cuda:0", env_offset=500)
    oa, ob = a.rollout(net, seed=9, episode=2, want=want), b.rollout(net, seed=9, episode=2, want=want)
    for k in want:
        assert torch.equal(torch.cat([oa[k], ob[k]]), ref[k]), k
    a.close(), b.close()


def test_evaluate_reports_on_the_network(monkeypatch):
    torch = _torch()
    monkeypatch.setenv("ORGYM_INV_JIT", "2")       # an MLP rollout is not a specialisable one: it must simply run
    cls, kw = CONFIGS["lost"]
    net = _net(cls, kw, (64, 64), seed=6)
    env = cls(num_envs=5000, device="cuda:0")
    res = [{k: v.clone() for k, v in r.items()}
           for r in env.evaluate(net, episodes=3, seed=77, want=("report", "ep_return", "stats32"))]
    assert not env.rollout_specialised and len(res) == 3
    for k, r in enumerate(res):
        o = env.rollout(net, seed=77, episode=k, want=("ep_return", "stats32"))
        assert torch.equal(r["ep_return"], o["ep_return"].cpu()) and torch.equal(r["stats32"], o["stats32"].cpu())
        want = pkg.evaluation_report(o, env.num_periods)
        got = pkg.report_to_dict(r["report"])
        assert got["SuccessfulEpisodes"] == 5000
        for f in ("MedianReward", "MinReward", "MaxReward"):
            assert got[f] == want[f], f
        for f in ("AvgReward", "AvgServiceLevel", "AvgStockoutQty", "AvgEndInv"):
            assert np.isclose(got[f], want[f], rtol=1e-12), f
        assert np.isclose(got["StdReward"], want["StdReward"], rtol=1e-10)
    assert not torch.equal(res[0]["ep_return"], res[1]["ep_return"])
    env.close()


@pytest.mark.parametrize("policy", ["base_stock", "random"])
def test_action_traj_of_the_on_device_policies(policy):
    """action_traj records the orders the heuristics placed: replayed through the step API (record_history) they give
    the same action_log and rewards; the random policy's equal an independent restatement of its Philox stream, the
    base-stock policy's the oracle's driver under the device's demand.  Requesting it runs the ahead-of-time kernel."""
    from oracle import oracle
    from helpers import device_random_actions
    torch = _torch()
    N, seed = 600, 5000
    env = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0")
    out = env.rollout(policy, seed=seed, want=("action_traj", "reward_traj"))
    assert not env.rollout_specialised
    acts, rt = out["action_traj"].clone(), out["reward_traj"].clone()
    env.close()
    rec = pkg.InvManagementLostSalesEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled", record_history=True)
    rec.reset(seed=seed)
    for t in range(rec.num_periods):
        rec.step(acts[:, t])
    assert torch.equal(rec.action_log, acts) and torch.equal(rec.P, rt)
    a, dem = acts.cpu().numpy(), rec.D.cpu().numpy()
    pick = np.r_[0:5, N - 5:N]
    if policy == "random":
        assert np.array_equal(device_random_actions(seed, pick, 0, rec.num_periods, rec.params.supply_capacity), a[pick])
    else:
        for e in pick:
            o = oracle.invmgmt_episode(rec.params, policy="base_stock", demand=dem[e])
            assert np.array_equal(o["action_log"], a[e]), e
    rec.close()


# ---- canaries: no write outside the requested outputs (compute-sanitizer is not available on the GPU pool) -----------
PAD = 4096


@pytest.fixture
def guard():
    torch = _torch()
    items = []

    def wrap(t):
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * PAD,), 0xA5, dtype=torch.uint8, device=t.device)
        inner = big[PAD:PAD + nbytes].view(t.dtype).view(t.shape)
        inner.copy_(t)
        items.append((big, nbytes))
        return inner
    yield wrap
    torch.cuda.synchronize()
    for big, nbytes in items:
        assert bool((big[:PAD] == 0xA5).all()) and bool((big[PAD + nbytes:] == 0xA5).all()), "canary overwritten"


@pytest.mark.parametrize("N", [1, 127, 129, 1000])
@pytest.mark.parametrize("hidden", [(64, 64), (176, 176)])
def test_mlp_rollout_writes_stay_in_bounds(N, hidden, guard):
    torch = _torch()
    cls, kw = CONFIGS["lost"]
    net = _net(cls, kw, hidden, seed=8)
    env = cls(num_envs=N, device="cuda:0", periods=7)
    T, n = 7, 3
    shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.int64), stats32=((N, 4), torch.int32),
                  reward_traj=((N, T), torch.float64), action_traj=((N, T, n), torch.int64))
    cache = env.__dict__.setdefault("_rollout_buf", {}).setdefault(0, {})
    for name, (shp, dt) in shapes.items():
        cache[name] = guard(torch.zeros(shp, dtype=dt, device="cuda"))
    env.rollout(net, seed=3, want=tuple(shapes))
    torch.cuda.synchronize()
    env.close()


# ---- errors on the device path -----------------------------------------------------------------------------------
def _raw_rollout(env, widths, num_layers=None, act=_capi.MLP_TANH):
    """orgym_invmgmt_rollout with a hand-built orgym_mlp_t (zero weights of the declared shapes)."""
    torch = _torch()
    m = _capi.Mlp()
    L = len(widths) - 1 if num_layers is None else num_layers
    m.num_layers, m.activation = L, act
    keep = []
    for l in range(min(len(widths), _capi.MLP_MAX_LAYERS + 1)):
        m.width[l] = widths[l]
    for l in range(min(L, _capi.MLP_MAX_LAYERS)):
        w = torch.zeros((max(widths[min(l + 1, len(widths) - 1)], 1), max(widths[l], 1)), device="cuda")
        keep.append(w)
        m.weight[l] = w.data_ptr()
    rin = _capi.InvRolloutIn()
    rin.policy = 3
    rin.mlp = C.pointer(m)
    ret = torch.zeros(env.num_envs, dtype=torch.float64, device="cuda")
    rout = _capi.InvRolloutOut()
    rout.ep_return = ret.data_ptr()
    rc = _capi.lib().orgym_invmgmt_rollout(env._h, 1, 0, 0, C.byref(rin), C.byref(rout), env._stream())
    torch.cuda.synchronize()
    return rc, _capi.lib().orgym_last_error().decode()


def test_device_path_errors():
    torch = _torch()
    from or_gym_inventory_b200._capi import OrgymError
    env = pkg.InvManagementLostSalesEnv(num_envs=64, device="cuda:0")
    assert _raw_rollout(env, (33, 64, 3))[0] == 0
    rc, msg = _raw_rollout(env, (32, 64, 3))
    assert rc == _capi.E_INVALID and "obs_dim" in msg
    rc, msg = _raw_rollout(env, (33, 64, 4))
    assert rc == _capi.E_INVALID and "m-1" in msg
    rc, msg = _raw_rollout(env, (33, 8, 8, 8, 8, 3), num_layers=5)
    assert rc == _capi.E_INVALID and "num_layers" in msg
    rc, msg = _raw_rollout(env, (33, 8, 3), act=7)
    assert rc == _capi.E_INVALID and "activation" in msg
    with pytest.raises(OrgymError, match="outside 1..256") as ei:
        env.rollout(_seq((33, 300, 3), torch.nn.Tanh).cuda(), seed=1)
    assert ei.value.code == _capi.E_INVALID
    with pytest.raises(OrgymError, match="bytes of shared memory") as ei:
        env.rollout(_seq((33, 256, 256, 256, 3), torch.nn.Tanh).cuda(), seed=1)
    assert ei.value.code == _capi.E_UNSUPPORTED
    with pytest.raises(OrgymError):
        env.specialise(_seq((33, 8, 3), torch.nn.Tanh))
    with pytest.raises(ValueError, match="at most 4"):
        env.rollout(_seq((33, 8, 8, 8, 8, 3), torch.nn.Tanh).cuda(), seed=1)
    # weights on the host and in float64 are converted, not refused: same orders as the float32 CUDA copy
    net = _seq((33, 16, 3), torch.nn.ReLU)
    with torch.no_grad():
        net[-1].bias.fill_(60.0)
    a = env.rollout(net.double(), seed=4, want=("action_traj",))["action_traj"].clone()
    b = env.rollout(net.float().cuda(), seed=4, want=("action_traj",))["action_traj"]
    assert torch.equal(a, b)
    env.close()
