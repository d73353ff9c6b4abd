"""GPU suite for the MLP actor policy of the newsvendor's fused rollout (nv_mlp_rollout_kernel): the dynamics it drives
are the env's own (replay through the 'actions' rollout), an exactly representable network reproduces the on-device
order-up-to heuristic bit for bit, the actions are the network's (float64 forward pass on the observations the step API
returns), NaN outputs follow the env's own rule, results do not depend on batching or sharding, evaluate() reports on
it, writes stay in bounds and malformed requests are refused."""
import ctypes as C

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from or_gym_inventory_b200 import _capi

pytestmark = pytest.mark.gpu
ALL_OUT = ("ep_return", "stats", "summary", "reward_traj", "action_traj", "final_obs")
MAXQ = 2000.0
U = 2.0 ** -24       # float32 unit roundoff


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


def _random_obs(od, n=4096, seed=0):
    """float64 observations over the env's ranges: price, cost, h, k, mu, then orders in [0, 2000]."""
    torch = _torch()
    g = torch.Generator().manual_seed(seed)
    hi = torch.tensor([100.0, 100.0, 5.0, 10.0, 200.0] + [MAXQ] * (od - 5), dtype=torch.float64)
    return torch.rand((n, od), generator=g, dtype=torch.float64) * hi


def _net(lead_time, hidden, act="tanh", seed=0, first_obs=None):
    """A network whose outputs spread over [0, 2000] with some below 0 and some above 2000 on the env's observations.
    The pipeline columns get 1 % of the first layer's weight: the network still reads them, but the spread comes from
    the per-env parameters, so it survives the feedback of the orders into the pipeline over an episode.
    With first_obs (float64 [N, obs_dim], the episode's first observations) the last layer maps those observations'
    outputs affinely onto [-500, 2500] exactly, so the first period alone is certain to contain actions below 0, above
    2000 and between; otherwise it gives random observations a mean of 1000 and a standard deviation of 900."""
    torch = _torch()
    torch.manual_seed(seed)
    od = lead_time + 5
    net = _seq((od,) + tuple(hidden) + (1,), torch.nn.Tanh if act == "tanh" else torch.nn.ReLU).double()
    x = _random_obs(od, seed=seed) if first_obs is None else first_obs.double().cpu()
    with torch.no_grad():
        net[0].weight.mul_(0.01)
        net[0].weight[:, 5:] *= 0.01
        h = net[:-1](x) if len(net) > 1 else x
        y = h @ net[-1].weight.t()
        if first_obs is None:
            s = 900.0 / float(y.std().clamp(min=1e-9))
            off = 1000.0 - float((y * s).mean())
        else:
            lo, hi = float(y.min()), float(y.max())
            assert hi > lo, "the network's output does not depend on the first observations"
            s = 3000.0 / (hi - lo)
            off = -500.0 - lo * s
        net[-1].weight.mul_(s)
        net[-1].bias.fill_(off)
    return net.float().cuda()


def _fixed(N, integer=False, seed=0):
    torch = _torch()
    g = torch.Generator().manual_seed(seed)
    r = lambda: torch.rand(N, generator=g, dtype=torch.float64)   # noqa: E731
    price = 1.0 + 99.0 * r()
    cost = 1.0 + (price - 1.0) * r()
    f = torch.stack([price, cost, 5.0 * r(), 10.0 * r(), 200.0 * r()], 1)
    if integer:
        f = f.floor()
    return f.cuda()


def _demand(N, T, seed=0):
    torch = _torch()
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 400, (N, T), generator=g, dtype=torch.int64).cuda()


def _same(a, b):
    """bitwise equality with NaN equal to NaN"""
    torch = _torch()
    if a.dtype.is_floating_point:
        return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
    return torch.equal(a, b)


def _replay(env, out, seed, **inputs):
    """The 'actions' rollout fed the MLP rollout's own actions, everything else equal."""
    acts = out["action_traj"].clone()
    got = {k: v.clone() for k, v in out.items()}
    ref = env.rollout("actions", actions=acts, seed=seed, want=ALL_OUT, buffer_set=1, **inputs)
    return got, ref


@pytest.mark.parametrize("lead_time", [0, 1, 5, 7, 8, 17])
@pytest.mark.parametrize("inputs", ["sampled", "demand", "fixed_params"])
def test_dynamics_are_the_envs_own(lead_time, inputs):
    torch = _torch()
    N = 3000
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=lead_time)
    kw = {}
    if inputs == "demand":
        kw["demand"] = _demand(N, env.step_limit, seed=lead_time)
    elif inputs == "fixed_params":
        kw["fixed_params"] = _fixed(N, seed=lead_time)
    net = _net(lead_time, (64, 64), seed=lead_time)
    out = env.rollout(net, seed=11, want=ALL_OUT, **kw)
    got, ref = _replay(env, out, 11, **kw)
    a = got["action_traj"]
    assert bool(((a > 0) & (a < MAXQ)).any())
    assert bool(torch.isfinite(got["ep_return"]).all())
    for k in ALL_OUT:
        assert torch.equal(got[k], ref[k]), k
    env.close()


def _order_up_to_net(lead_time, width=8):
    """relu((L+1) mu - sum of the pipeline), then the identity: with integer mu every float32 operation is exact."""
    torch = _torch()
    od = lead_time + 5
    net = _seq((od, width, 1), torch.nn.ReLU)
    with torch.no_grad():
        for lin in (net[0], net[2]):
            lin.weight.zero_()
            lin.bias.zero_()
        net[0].weight[0, 4] = float(lead_time + 1)
        net[0].weight[0, 5:] = -1.0
        net[2].weight[0, 0] = 1.0
    return net.cuda()


@pytest.mark.parametrize("lead_time", [0, 3, 5, 8, 17])
def test_exact_network_is_the_order_up_to_heuristic(lead_time):
    torch = _torch()
    N = 2000
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=lead_time)
    fp = _fixed(N, integer=True, seed=3)
    got = {k: v.clone() for k, v in env.rollout(_order_up_to_net(lead_time), seed=5, fixed_params=fp,
                                                   want=ALL_OUT).items()}
    ref = env.rollout("order_up_to", safety_factor=1.0, seed=5, fixed_params=fp, want=ALL_OUT, buffer_set=1)
    a = got["action_traj"]
    assert bool(((a > 0) & (a < MAXQ)).any())
    for k in ALL_OUT:
        assert torch.equal(got[k], ref[k]), k
    env.close()


def _f64_forward_with_bound(net, x):
    """float64 forward pass and a bound on the float32 evaluation's error, per row.  Each output of a layer is a chain
    of K fmaf from the bias: its rounding error is at most (K + 1) u (|b| + sum |w||h|) (u = 2^-24); tanhf adds 2 ulp
    of its result, ReLU nothing; both are 1-Lipschitz, so an input error e reaches the output as at most |W| e."""
    torch = _torch()
    lins = [m for m in net if isinstance(m, torch.nn.Linear)]
    tanh = any(isinstance(m, torch.nn.Tanh) for m in net)
    h, err = x, torch.zeros_like(x)
    for i, lin in enumerate(lins):
        W, b = lin.weight.double(), lin.bias.double()
        y = h @ W.t() + b
        mag = h.abs() @ W.abs().t() + b.abs()
        err = err @ W.abs().t() + (W.shape[1] + 1) * U * mag
        if i + 1 < len(lins):
            if tanh:
                y = torch.tanh(y)
                err = err + 2 * U * y.abs()
            else:
                y = y.clamp(min=0)
        h = y
    return h[:, 0], err[:, 0]


NETS = [("tanh", (64, 64)), ("relu", (64, 64)), ("tanh", (176, 176)), ("relu", ()), ("tanh", (32, 48, 32)),
        ("relu", (7,))]


@pytest.mark.parametrize("act, hidden", NETS, ids=[f"{a}-{'x'.join(map(str, h)) or 'linear'}" for a, h in NETS])
@pytest.mark.parametrize("lead_time", [0, 5, 9])
def test_policy_is_the_network(act, hidden, lead_time):
    """Each device action is clip(y64, 0, 2000) of a float64 forward pass on the observation the step API returns, to
    within the float32 evaluation's error bound (4x the bound of _f64_forward_with_bound, at least 1 float32 ulp)."""
    torch = _torch()
    N = 1500
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=lead_time)
    T = env.step_limit
    fp, dem = _fixed(N, seed=7), _demand(N, T, seed=7)
    first = torch.cat([fp.float().double(), torch.zeros((N, lead_time), dtype=torch.float64, device=fp.device)], 1)
    net = _net(lead_time, hidden, act, seed=1, first_obs=first)
    acts = env.rollout(net, seed=2, fixed_params=fp, demand=dem, want=("action_traj",))["action_traj"].clone()
    env.close()
    rec = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=lead_time, autoreset_mode="disabled")
    obs, _ = rec.reset(seed=2, options={"fixed_params": fp})
    rows = []
    for t in range(T):
        rows.append(obs.double().clone())
        obs = rec.step(acts[:, t], demand=dem[:, t])[0]
    rec.close()
    X = torch.stack(rows, 1).reshape(N * T, -1)
    y64, err = _f64_forward_with_bound(net, X)
    want = y64.clamp(0.0, MAXQ)
    got = acts.reshape(-1).double()
    tol = torch.maximum(4 * err, want.abs() * 2 * U)
    assert bool((y64 < 0).any()) and bool((y64 > MAXQ).any()) and bool(((y64 > 0) & (y64 < MAXQ)).any())
    bad = (got - want).abs() > tol
    assert not bool(bad.any()), (int(bad.sum()), float((got - want).abs().max()))


@pytest.mark.parametrize("lead_time", [0, 4, 9])
def test_nan_outputs_follow_the_envs_rule(lead_time):
    """A NaN last-layer bias gives NaN actions.  Every output equals the 'actions' rollout fed those NaN actions.  With
    lead_time > 0 the env's rule places no order and the returns stay finite; with lead_time = 0 the action is also the
    stock on hand (newsvendor.py:136-139), so the reward is NaN, as in the reference."""
    torch = _torch()
    N = 300
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=lead_time)
    net = _net(lead_time, (16,), "relu", seed=2)
    with torch.no_grad():
        net[-1].bias.fill_(float("nan"))
    out = env.rollout(net, seed=4, want=ALL_OUT)
    got, ref = _replay(env, out, 4)
    assert bool(torch.isnan(got["action_traj"]).all())
    for k in ALL_OUT:
        assert _same(got[k], ref[k]), k
    if lead_time > 0:
        assert bool(torch.isfinite(got["ep_return"]).all()) and bool((got["final_obs"][:, 5:] == 0).all())
    else:
        assert bool(torch.isnan(got["ep_return"]).all())
    env.close()


@pytest.mark.parametrize("hidden", [(64, 64), (176, 176)])   # 64-env and 32-env sub-tiles
def test_results_do_not_depend_on_batching_or_sharding(hidden):
    torch = _torch()
    net = _net(5, hidden, seed=4)
    full_n = 1000
    want = ("ep_return", "stats", "action_traj", "final_obs", "reward_traj")
    env = pkg.NewsvendorEnv(num_envs=full_n, device="cuda:0")
    ref = {k: v.clone() for k, v in env.rollout(net, seed=9, episode=2, want=want).items()}
    env.close()
    for N in (1, 127, 129):
        e = pkg.NewsvendorEnv(num_envs=N, device="cuda:0")
        o = e.rollout(net, seed=9, episode=2, want=want)
        for k in want:
            assert torch.equal(o[k], ref[k][:N]), (N, k)
        e.close()
    a = pkg.NewsvendorEnv(num_envs=500, device="cuda:0", env_offset=0)
    b = pkg.NewsvendorEnv(num_envs=full_n - 500, device="cuda:0", env_offset=500)
    oa, ob = a.rollout(net, seed=9, episode=2, want=want), b.rollout(net, seed=9, episode=2, want=want)
    for k in want:
        assert torch.equal(torch.cat([oa[k], ob[k]]), ref[k]), k
    a.close(), b.close()


def test_evaluate_reports_on_the_network():
    torch = _torch()
    net = _net(5, (64, 64), seed=6)
    env = pkg.NewsvendorEnv(num_envs=5000, device="cuda:0")
    res = [{k: v.clone() for k, v in r.items()}
           for r in env.evaluate(net, episodes=3, seed=77, want=("report", "ep_return", "stats"))]
    assert len(res) == 3
    for k, r in enumerate(res):
        o = env.rollout(net, seed=77, episode=k, want=("ep_return", "stats"))
        assert r["stats"].dtype == torch.float64
        assert torch.equal(r["ep_return"], o["ep_return"].cpu()) and torch.equal(r["stats"], o["stats"].cpu())
        want = pkg.evaluation_report(o, env.step_limit)
        got = pkg.report_to_dict(r["report"])
        assert got["SuccessfulEpisodes"] == 5000
        for f in ("MedianReward", "MinReward", "MaxReward"):
            assert got[f] == want[f], f
        for f in ("AvgReward", "AvgServiceLevel", "AvgStockoutQty", "AvgEndInv"):
            assert np.isclose(got[f], want[f], rtol=1e-12), f
        assert np.isclose(got["StdReward"], want["StdReward"], rtol=1e-10)
    assert not torch.equal(res[0]["ep_return"], res[1]["ep_return"])
    env.close()


# ---- canaries: no write outside the requested outputs -------------------------------------------------------------
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
    T, L = 6, 7
    net = _net(L, hidden, seed=8)
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", step_limit=T, lead_time=L)
    shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.float64), reward_traj=((N, T), torch.float64),
                  action_traj=((N, T), torch.float32), final_obs=((N, env.obs_dim), torch.float32),
                  summary=((8,), torch.float64))
    cache = env.__dict__.setdefault("_rollout_buf", {}).setdefault(0, {})
    for name, (shp, dt) in shapes.items():
        cache[name] = guard(torch.zeros(shp, dtype=dt, device="cuda"))
    env.rollout(net, seed=3, want=tuple(shapes))
    torch.cuda.synchronize()
    env.close()


# ---- errors on the device path -----------------------------------------------------------------------------------
def _raw_rollout(env, widths, num_layers=None, null_weight=None, no_mlp=False):
    """orgym_newsvendor_rollout with a hand-built orgym_mlp_t (zero weights of the declared shapes)."""
    torch = _torch()
    m = _capi.Mlp()
    L = len(widths) - 1 if num_layers is None else num_layers
    m.num_layers, m.activation = L, _capi.MLP_TANH
    keep = []
    for l in range(min(len(widths), _capi.MLP_MAX_LAYERS + 1)):
        m.width[l] = widths[l]
    for l in range(min(L, _capi.MLP_MAX_LAYERS)):
        w = torch.zeros((max(widths[min(l + 1, len(widths) - 1)], 1), max(widths[l], 1)), device="cuda")
        keep.append(w)
        m.weight[l] = None if l == null_weight else w.data_ptr()
    rin = _capi.NvRolloutIn()
    rin.policy = 4
    rin.mlp = None if no_mlp else C.pointer(m)
    ret = torch.zeros(env.num_envs, dtype=torch.float64, device="cuda")
    rout = _capi.NvRolloutOut()
    rout.ep_return = ret.data_ptr()
    rc = _capi.lib().orgym_newsvendor_rollout(env._h, 1, 0, 0, C.byref(rin), C.byref(rout), env._stream())
    torch.cuda.synchronize()
    return rc, _capi.lib().orgym_last_error().decode()


def test_device_path_errors():
    torch = _torch()
    from or_gym_inventory_b200._capi import OrgymError
    env = pkg.NewsvendorEnv(num_envs=64, device="cuda:0")
    assert _raw_rollout(env, (10, 64, 1))[0] == 0
    rc, msg = _raw_rollout(env, (10, 64, 1), no_mlp=True)
    assert rc == _capi.E_INVALID and "in->mlp" in msg
    rc, msg = _raw_rollout(env, (11, 64, 1))
    assert rc == _capi.E_INVALID and "obs_dim = 10" in msg
    rc, msg = _raw_rollout(env, (10, 64, 2))
    assert rc == _capi.E_INVALID and "width[2] = 2" in msg and "action dimension = 1" in msg
    rc, msg = _raw_rollout(env, (10, 64, 1), null_weight=1)
    assert rc == _capi.E_INVALID and "weight_dev[1] is NULL" in msg
    rc, msg = _raw_rollout(env, (10, 8, 8, 8, 8, 1), num_layers=5)
    assert rc == _capi.E_INVALID and "num_layers" in msg
    rc, msg = _raw_rollout(env, (10, 256, 256, 256, 1))
    assert rc == _capi.E_UNSUPPORTED and "bytes of shared memory" in msg and "this build's limit is" in msg
    rin = _capi.NvRolloutIn()
    rin.policy = 5
    rout = _capi.NvRolloutOut()
    assert _capi.lib().orgym_newsvendor_rollout(env._h, 1, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    with pytest.raises(OrgymError, match="bytes of shared memory") as ei:
        env.rollout(_seq((10, 256, 256, 256, 1), torch.nn.Tanh).cuda(), seed=1)
    assert ei.value.code == _capi.E_UNSUPPORTED
    with pytest.raises(ValueError, match="at most 4"):
        env.rollout(_seq((10, 8, 8, 8, 8, 1), torch.nn.Tanh).cuda(), seed=1)
    with pytest.raises(ValueError, match="the observation has 10"):
        env.rollout(_seq((9, 8, 1), torch.nn.Tanh).cuda(), seed=1)
    # weights on the host and in float64 are converted, not refused: same actions as the float32 CUDA copy
    net = _net(5, (16,), "relu", seed=3)
    a = env.rollout(net.cpu().double(), seed=4, want=("action_traj",))["action_traj"].clone()
    b = env.rollout(net.float().cuda(), seed=4, want=("action_traj",))["action_traj"]
    assert torch.equal(a, b)
    env.close()
