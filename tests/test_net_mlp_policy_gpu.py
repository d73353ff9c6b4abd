"""GPU suite for the MLP actor policy of the network env's fused rollout (net_mlp_rollout_kernel): the dynamics it drives
are the env's own (replay through the 'actions' rollout under every kernel mode), an exactly representable network
reproduces the constant-order rollout and a float64 step-API loop bit for bit, the actions are the network's (float64
forward pass on the observations the step API returns), NaN outputs follow the env's own rule, results do not depend on
batching or sharding, weights are read at every call, evaluate() reports on it, writes stay in bounds and requests the
kernel cannot serve are refused."""
import ctypes as C

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from or_gym_inventory_b200 import _capi
from helpers import golden_files, load_golden, net_kwargs, set_net_kernel_mode

pytestmark = pytest.mark.gpu
ALL_OUT = ("ep_return", "stats", "summary", "reward_traj", "final_X", "final_Y", "final_U", "action_traj")
CMP = ("ep_return", "stats", "summary", "reward_traj", "final_X", "final_Y", "final_U")
NET_MODES = ["specialised", "stream_jit", "stream_jit_twopass", "stream_jit_fused_obs", "generic"]
U = 2.0 ** -24       # float32 unit roundoff


def _torch():
    import torch
    return torch


def _random_graph(seed):
    from test_random_configs_gpu import _random_graph as rg
    return rg(np.random.default_rng(seed), ordered=bool(seed % 2))


def _graph_kwargs(kind):
    """Constructor keywords: the reference's default and custom graphs, a yield < 1 multi-market graph, a user_D
    trace, random graphs."""
    if kind in ("default", "custom"):
        return dict(default_graph_kind=kind)
    if kind in ("yield", "userD"):
        g, meta = load_golden(golden_files(f"net_{kind}_backlog")[0])
        return net_kwargs(meta)
    return dict(graph=_random_graph(int(kind[6:])), num_periods=12)


def _net(od, E, high, hidden=(64, 64), act="tanh", seed=0):
    """A network whose outputs fall below 0, above `high` and in between on the env's observations: first layer scaled
    down so that tanh does not saturate, last layer mapped so that its outputs on random observations in [0, 400] have
    mean high / 2 and standard deviation high."""
    torch = _torch()
    torch.manual_seed(seed)
    mods, widths = [], (od,) + tuple(hidden) + (E,)
    for i in range(len(widths) - 1):
        mods.append(torch.nn.Linear(widths[i], widths[i + 1]))
        if i < len(widths) - 2:
            mods.append(torch.nn.Tanh() if act == "tanh" else torch.nn.ReLU())
    net = torch.nn.Sequential(*mods).double()
    x = torch.rand((2048, od), dtype=torch.float64) * 400
    hi = torch.as_tensor(np.asarray(high, dtype=np.float64))
    with torch.no_grad():
        net[0].weight.mul_(0.005)
        y = net(x)
        mu, sd = y.mean(0), y.std(0).clamp_min(1e-6)
        net[-1].weight.mul_((hi / sd)[:, None])
        net[-1].bias.copy_(0.5 * hi + (net[-1].bias - mu) * hi / sd)
    return net.float()


def _env(kind, n, backlog=True, **kw):
    return pkg.NetInvMgmtMasterEnv(**dict(_graph_kwargs(kind), backlog=backlog), num_envs=n, device="cuda:0", **kw)


def _equal(a, b):
    torch = _torch()
    return a.shape == b.shape and bool(torch.equal(torch.isnan(a), torch.isnan(b))) and \
        bool(torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0)))


# ---- 1) the dynamics are the env's own -------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["default", "custom", "yield", "userD", "random1", "random2", "random5"])
@pytest.mark.parametrize("backlog", [True, False])
@pytest.mark.parametrize("inputs", ["sampled", "replayed"])
def test_dynamics_are_the_envs_own(kind, backlog, inputs):
    torch = _torch()
    N = 300
    env = _env(kind, N, backlog=backlog)
    E, M, T = len(env.reorder_links), len(env.retail_links), int(env.num_periods)
    net = _net(env.obs_dim, E, env.single_action_space.high, seed=1)
    dem = None
    if inputs == "replayed":
        dem = torch.as_tensor(np.random.default_rng(1).poisson(15, size=(N, T, M)).astype(np.float64), device="cuda")
    a = env.rollout(net, seed=5, demand=dem, want=ALL_OUT)
    a = {k: v.clone() for k, v in a.items()}
    acts = a["action_traj"]
    b = env.rollout("actions", seed=5, actions=acts, demand=dem, want=CMP)
    for k in CMP:
        assert _equal(a[k], b[k]), k
    env.close()


@pytest.mark.parametrize("mode", NET_MODES)
def test_replay_matches_under_every_kernel_mode(mode, monkeypatch):
    torch = _torch()
    set_net_kernel_mode(monkeypatch, mode)
    N = 257
    env = _env("default", N)
    E, M, T = len(env.reorder_links), len(env.retail_links), int(env.num_periods)
    net = _net(env.obs_dim, E, env.single_action_space.high, seed=2)
    dem = torch.as_tensor(np.random.default_rng(2).poisson(20, size=(N, T, M)).astype(np.float64), device="cuda")
    a = {k: v.clone() for k, v in env.rollout(net, seed=1, demand=dem, want=ALL_OUT).items()}
    b = env.rollout("actions", seed=1, actions=a["action_traj"], demand=dem, want=CMP)
    for k in CMP:
        assert _equal(a[k], b[k]), (mode, k)
    env.close()


# ---- 2) exact cross-kernel checks ----------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["default", "custom"])
def test_constant_network_is_the_constant_rollout(kind, monkeypatch):
    torch = _torch()
    set_net_kernel_mode(monkeypatch, "specialised")
    env = _env(kind, 1000)
    assert env.specialised
    E = len(env.reorder_links)
    c = (env.single_action_space.high * 0.1).astype(np.float32)
    net = torch.nn.Sequential(torch.nn.Linear(env.obs_dim, 64), torch.nn.Tanh(), torch.nn.Linear(64, E))
    with torch.no_grad():
        for m in (net[0], net[2]):
            m.weight.zero_()
            m.bias.zero_()
        net[2].bias.copy_(torch.from_numpy(c))
    a = {k: v.clone() for k, v in env.rollout(net, seed=9, want=ALL_OUT).items()}
    b = env.rollout("constant", seed=9, actions=c, want=CMP)
    for k in CMP:
        assert _equal(a[k], b[k]), k
    assert bool((a["action_traj"] == torch.from_numpy(c).cuda()).all())
    env.close()


def test_dyadic_network_is_the_float64_step_loop():
    """Dyadic weights on integer-valued observations (yield 1): every float32 operation of the device is exact, so a
    float64 torch forward pass driving reset / step gives the same actions, returns and final state."""
    torch = _torch()
    N = 200
    env = _env("default", N, autoreset_mode="disabled")
    E, T = len(env.reorder_links), int(env.num_periods)
    g = torch.Generator().manual_seed(3)
    net = torch.nn.Sequential(torch.nn.Linear(env.obs_dim, 8), torch.nn.ReLU(), torch.nn.Linear(8, E))
    with torch.no_grad():
        net[0].weight.copy_(torch.randint(-1, 2, (8, env.obs_dim), generator=g) / 8.0)
        net[0].bias.copy_(torch.randint(-64, 65, (8,), generator=g) / 8.0)
        net[2].weight.copy_(torch.randint(-2, 3, (E, 8), generator=g) / 8.0)
        net[2].bias.copy_(torch.randint(0, 800, (E,), generator=g) / 4.0)
    net64 = net.double().cuda()
    high = torch.as_tensor(env.single_action_space.high, dtype=torch.float64, device="cuda")
    obs, _ = env.reset(seed=4)
    ret = torch.zeros(N, dtype=torch.float64, device="cuda")
    acts = []
    with torch.no_grad():
        for t in range(T):
            x = obs.double()
            assert bool((x == x.round()).all())
            a = torch.minimum(net64(x).clamp_min(0.0), high).float()
            acts.append(a)
            obs, r, _, _, _ = env.step(a)
            ret += r
    X, Y, U_, _ = env.export_state()
    out = env.rollout(net.float(), seed=4, want=("ep_return", "final_X", "final_Y", "final_U", "action_traj"))
    assert torch.equal(out["action_traj"], torch.stack(acts, 1))
    assert torch.equal(out["ep_return"], ret)
    assert torch.equal(out["final_X"], X) and torch.equal(out["final_Y"], Y) and torch.equal(out["final_U"], U_)
    env.close()


# ---- 3) the actions are the network's --------------------------------------------------------------------------------
def _forward_with_bound(net, x):
    """float64 forward pass and a bound on the float32 evaluation's absolute error (fmaf chains in ascending k, accurate
    tanhf), propagated layer by layer."""
    torch = _torch()
    lin = [m for m in net if isinstance(m, torch.nn.Linear)]
    h, err = x, torch.zeros_like(x)
    for i, m in enumerate(lin):
        W, b = m.weight.double(), m.bias.double()
        K = W.shape[1]
        y = h @ W.t() + b
        mag = h.abs() @ W.abs().t() + b.abs()
        err = err @ W.abs().t() + (K + 2) * U * mag
        if i < len(lin) - 1:
            h, err = torch.tanh(y), err + 4 * U
        else:
            h = y
    return h, err


@pytest.mark.parametrize("kind", ["default", "custom"])
def test_actions_are_the_networks(kind):
    torch = _torch()
    N = 256
    env = _env(kind, N, autoreset_mode="disabled")
    E, T = len(env.reorder_links), int(env.num_periods)
    net = _net(env.obs_dim, E, env.single_action_space.high, seed=4)
    out = env.rollout(net, seed=7, want=("action_traj", "ep_return"))
    acts = out["action_traj"].clone()
    high = torch.as_tensor(env.single_action_space.high, dtype=torch.float64, device="cuda")
    a64 = acts.double()
    assert bool((a64 == 0).any()) and bool((a64 == high).any()) and bool(((a64 > 0) & (a64 < high)).any())
    netc = net.cuda()
    obs, _ = env.reset(seed=7)
    ret = torch.zeros(N, dtype=torch.float64, device="cuda")
    with torch.no_grad():
        for t in range(T):
            y, err = _forward_with_bound(netc, obs.double())
            lo = torch.minimum((y - err).clamp_min(0.0), high)
            hi = torch.minimum((y + err).clamp_min(0.0), high)
            a = acts[:, t].double()
            assert bool(((a >= lo * (1 - 2 * U)) & (a <= hi * (1 + 2 * U))).all()), t
            obs, r, _, _, _ = env.step(acts[:, t])
            ret += r
    assert torch.equal(ret, out["ep_return"])
    env.close()


# ---- 4) NaN outputs --------------------------------------------------------------------------------------------------
def test_nan_outputs_order_nothing_and_replay():
    torch = _torch()
    env = _env("default", 200)
    E = len(env.reorder_links)
    net = _net(env.obs_dim, E, env.single_action_space.high, seed=5)
    with torch.no_grad():
        net[-1].bias[[1, 4, 7]] = float("nan")
    a = {k: v.clone() for k, v in env.rollout(net, seed=2, want=ALL_OUT).items()}
    acts = a["action_traj"]
    assert bool(torch.isnan(acts[:, :, [1, 4, 7]]).all()) and not bool(torch.isnan(acts[:, :, [0, 2, 3]]).any())
    zero = acts.clone()
    zero[:, :, [1, 4, 7]] = 0.0
    for replay in (acts, zero):
        b = env.rollout("actions", seed=2, actions=replay, want=CMP)
        for k in CMP:
            assert _equal(a[k], b[k]), k
    env.close()


# ---- 5) invariance ---------------------------------------------------------------------------------------------------
def test_results_do_not_depend_on_batching_or_sharding():
    torch = _torch()
    full = _env("default", 1000)
    E = len(full.reorder_links)
    net = _net(full.obs_dim, E, full.single_action_space.high, seed=6)
    ref = {k: v.clone() for k, v in full.rollout(net, seed=11, episode=2, want=ALL_OUT).items() if k != "summary"}
    full.close()
    for n, off in ((300, 0), (129, 0), (400, 300), (1, 999), (571, 429)):
        env = _env("default", n, env_offset=off)
        got = env.rollout(net, seed=11, episode=2, want=tuple(ref))
        for k in ref:
            assert _equal(got[k], ref[k][off:off + n]), (n, off, k)
        env.close()


# ---- 6) weights are read at every call -------------------------------------------------------------------------------
def test_weights_are_read_at_every_call():
    torch = _torch()
    env = _env("default", 256)
    net = _net(env.obs_dim, len(env.reorder_links), env.single_action_space.high, seed=7).cuda()
    a = env.rollout(net, seed=1, want=("ep_return",))["ep_return"].clone()
    with torch.no_grad():
        net[-1].bias.add_(100.0)
    b = env.rollout(net, seed=1, want=("ep_return",))["ep_return"].clone()
    assert not torch.equal(a, b)
    with torch.no_grad():
        net[-1].bias.sub_(100.0)
    assert torch.equal(env.rollout(net, seed=1, want=("ep_return",))["ep_return"], a)
    env.close()


# ---- 7) evaluate() ---------------------------------------------------------------------------------------------------
def test_evaluate_reports_on_the_network():
    torch = _torch()
    env = _env("default", 5000)
    net = _net(env.obs_dim, len(env.reorder_links), env.single_action_space.high, seed=8)
    res = [{k: v.clone() for k, v in r.items()}
           for r in env.evaluate(net, episodes=3, seed=77, want=("report", "ep_return", "stats"))]
    assert len(res) == 3
    for k, r in enumerate(res):
        o = env.rollout(net, seed=77, episode=k, want=("ep_return", "stats"))
        assert torch.equal(r["ep_return"], o["ep_return"].cpu()) and torch.equal(r["stats"], o["stats"].cpu())
        want = pkg.evaluation_report(o, int(env.num_periods))
        got = pkg.report_to_dict(r["report"])
        assert got["SuccessfulEpisodes"] == 5000
        for f in ("MedianReward", "MinReward", "MaxReward"):
            assert got[f] == want[f], f
        for f in ("AvgReward", "AvgServiceLevel", "AvgStockoutQty", "AvgEndInv"):
            assert np.isclose(got[f], want[f], rtol=1e-12), f
        assert np.isclose(got["StdReward"], want["StdReward"], rtol=1e-10)
    assert not torch.equal(res[0]["ep_return"], res[1]["ep_return"])
    env.close()


# ---- 8) canaries: no write outside the requested outputs -------------------------------------------------------------
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


@pytest.mark.parametrize("N", [1, 127, 129, 300])
@pytest.mark.parametrize("hidden", [(64, 64), (256,)])
def test_mlp_rollout_writes_stay_in_bounds(N, hidden, guard):
    torch = _torch()
    env = _env("default", N)
    J, E, M, T = len(env.main_nodes), len(env.reorder_links), len(env.retail_links), int(env.num_periods)
    net = _net(env.obs_dim, E, env.single_action_space.high, hidden=hidden, seed=9)
    f64, f32 = torch.float64, torch.float32
    shapes = dict(ep_return=((N,), f64), stats=((N, 4), f64), reward_traj=((N, T), f64), final_X=((N, J), f64),
                  final_Y=((N, E), f64), final_U=((N, M), f64), summary=((8,), f64), action_traj=((N, T, E), f32))
    cache = env.__dict__.setdefault("_rollout_buf", {}).setdefault(0, {})
    for name, (shp, dt) in shapes.items():
        cache[name] = guard(torch.zeros(shp, dtype=dt, device="cuda"))
    env._scratch = guard(torch.zeros_like(env._state))
    env.rollout(net, seed=3, want=tuple(shapes))
    torch.cuda.synchronize()
    env.close()


# ---- 9) refusals and dispatch ----------------------------------------------------------------------------------------
def test_large_graph_is_refused_with_the_sizes():
    from or_gym_inventory_b200._capi import OrgymError
    from or_gym_inventory_b200.network_management import synthetic_graph
    env = pkg.NetInvMgmtMasterEnv(graph=synthetic_graph(64), num_envs=64, device="cuda:0", specialise=False)
    net = _net(env.obs_dim, len(env.reorder_links), env.single_action_space.high, seed=1)
    with pytest.raises(OrgymError, match="bytes of shared memory") as ei:
        env.rollout(net, seed=1)
    assert ei.value.code == _capi.E_UNSUPPORTED
    assert str(env.obs_dim) in str(ei.value)
    env.close()


def test_malformed_network_is_refused_on_a_handle():
    torch = _torch()
    env = _env("default", 64)
    E = len(env.reorder_links)
    high = np.ascontiguousarray(env.single_action_space.high, dtype=np.float32)
    w = torch.zeros((E, env.obs_dim), device="cuda")
    m = _capi.Mlp()
    m.num_layers, m.activation = 1, _capi.MLP_TANH
    m.width[0], m.width[1] = env.obs_dim, E
    m.weight[0] = w.data_ptr()
    rin = _capi.NetRolloutIn()
    rin.policy = 2
    rin.mlp = C.pointer(m)
    rin.action_high = high.ctypes.data
    ret = torch.zeros(64, dtype=torch.float64, device="cuda")
    rout = _capi.NetRolloutOut()
    rout.ep_return = ret.data_ptr()
    scratch = torch.zeros_like(env._state)
    call = lambda: _capi.lib().orgym_netinv_rollout(env._h, scratch.data_ptr(), 1, 0, 0, C.byref(rin),  # noqa: E731
                                                   C.byref(rout), env._stream())
    assert call() == _capi.OK
    for bad in ("width", "layers", "weight", "high", "traj"):
        m.width[1], m.num_layers, m.weight[0], rin.action_high = E, 1, w.data_ptr(), high.ctypes.data
        rin.policy, rout.action_traj = 2, None
        if bad == "width":
            m.width[1] = E + 1
        elif bad == "layers":
            m.num_layers = 0
        elif bad == "weight":
            m.weight[0] = None
        elif bad == "high":
            rin.action_high = None
        else:   # action_traj with another policy
            rin.policy, rin.actions, rout.action_traj = 1, torch.zeros(E, device="cuda").data_ptr(), ret.data_ptr()
        assert call() == _capi.E_INVALID, bad
    torch.cuda.synchronize()
    env.close()


@pytest.mark.parametrize("jit", ["0", "2"])
def test_mlp_runs_whatever_the_jit_setting(jit, monkeypatch):
    torch = _torch()
    env = _env("default", 300)
    net = _net(env.obs_dim, len(env.reorder_links), env.single_action_space.high, seed=10)
    ref = {k: v.clone() for k, v in env.rollout(net, seed=3, want=ALL_OUT).items()}
    env.close()
    monkeypatch.setenv("ORGYM_NET_JIT", jit)
    env = _env("default", 300)
    assert env.specialised == (jit == "2")
    got = env.rollout(net, seed=3, want=ALL_OUT)
    for k in ALL_OUT:
        assert _equal(got[k], ref[k]), k
    env.close()
