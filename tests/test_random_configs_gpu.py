"""Property-style parity: randomly generated configurations / topologies (fixed seeds), CUDA step + fused rollout vs the
C oracle (which is pinned to the reference by the golden vectors).  Covers what the goldens cannot enumerate: stage
counts 1..12, lead times including 0, lost sales / backlog, float / negative / over-capacity actions, random graphs
with yields < 1, multi-market retailers, L = 0 links, both network kernels."""
import os

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from helpers import seq_sum, set_net_kernel_mode

pytestmark = pytest.mark.gpu
# ORGYM_STRESS=k multiplies the number of random cases (one-off soak runs; the default suite stays short)
STRESS = max(1, int(os.environ.get("ORGYM_STRESS", "1")))


def _torch():
    import torch
    return torch


@pytest.mark.parametrize("case", range(12 * STRESS))
def test_invmgmt_random_config(case):
    from oracle import oracle
    torch = _torch()
    rng = np.random.default_rng(1000 + case)
    n = int(rng.integers(1, 13))
    T = int(rng.integers(3, 41))
    cfg = dict(periods=T, I0=rng.integers(0, 200, n).tolist(), p=float(rng.uniform(5, 40)),
               r=np.sort(rng.uniform(0.5, 30, n + 1))[::-1].round(3).tolist(), k=rng.uniform(0, 1, n + 1).round(3).tolist(),
               h=rng.uniform(0, 0.5, n).round(3).tolist(), c=rng.integers(1, 300, n).tolist(),
               L=rng.integers(0, 13, n).tolist(), dist_param={"mu": float(rng.uniform(0.5, 60))},
               alpha=float(rng.uniform(0.8, 1.0)))
    backlog = bool(case % 2)
    N = 257
    cls = pkg.InvManagementBacklogEnv if backlog else pkg.InvManagementLostSalesEnv
    env = cls(num_envs=N, device="cuda:0", wide_state=bool(case % 3 == 0), autoreset_mode="disabled", **cfg)
    cap = np.asarray(cfg["c"])
    acts = rng.uniform(-0.3, 1.5, size=(N, T, n)) * cap          # float actions: negative and above capacity
    dem = rng.poisson(cfg["dist_param"]["mu"], size=(N, T)).astype(np.int64)
    obs, _ = env.reset(seed=case)
    rew = np.zeros((N, T))
    for t in range(T):
        obs, r, _, trunc, _ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
        rew[:, t] = r.cpu().numpy()
    assert trunc.all()
    last = obs.cpu().numpy()
    I, B, _ = env.export_state()
    ai = np.trunc(np.maximum(acts, 0)).astype(np.int64)
    out = env.rollout("actions", actions=ai, demand=dem, want=("reward_traj", "ep_return", "final_I", "final_B"))
    assert np.array_equal(out["reward_traj"].cpu().numpy(), rew)
    assert torch.equal(out["final_I"], I) and torch.equal(out["final_B"], B)
    for e in range(0, N, 32):
        o = oracle.invmgmt_episode(env.params, actions=acts[e], demand=dem[e])
        assert np.array_equal(o["reward"], rew[e]), (case, e)
        assert np.array_equal(o["obs"][-1], last[e])
        assert np.array_equal(o["I"][-1], I[e].cpu().numpy()) and np.array_equal(o["B"][-1], B[e].cpu().numpy())
    # base-stock with a fractional safety factor (float64 policy path) vs the oracle's driver
    sf = float(rng.uniform(0.6, 1.6))
    ob = env.rollout("base_stock", demand=dem, safety_factor=sf, want=("ep_return", "final_I"))
    for e in range(0, N, 64):
        o = oracle.invmgmt_episode(env.params, policy="base_stock", demand=dem[e], safety_factor=sf)
        assert ob["ep_return"][e].item() == seq_sum(o["reward"])
        assert np.array_equal(o["I"][-1], ob["final_I"][e].cpu().numpy())
    assert env.errors() == 0
    env.close()


@pytest.mark.parametrize("case", range(8 * STRESS))
def test_newsvendor_random_config(case):
    from oracle import oracle
    torch = _torch()
    rng = np.random.default_rng(2000 + case)
    L = int(rng.integers(0, 21))
    cfg = dict(lead_time=L, step_limit=int(rng.integers(5, 50)), max_inventory=int(rng.integers(200, 5000)),
               max_order_quantity=int(rng.integers(50, 2500)), p_max=float(rng.uniform(10, 200)),
               h_max=float(rng.uniform(0.5, 10)), k_max=float(rng.uniform(1, 20)), mu_max=float(rng.uniform(5, 300)))
    N = 300
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", **cfg)
    T = env.step_limit
    env.reset(seed=case)
    par = env.export_params().cpu().numpy()
    acts = (rng.uniform(-0.2, 1.3, size=(N, T)) * cfg["max_order_quantity"]).astype(np.float32)
    acts[rng.random((N, T)) < 0.25] = 0.0
    dem = rng.poisson(par[:, 4:5], size=(N, T)).astype(np.int64)
    out = env.rollout("actions", actions=acts, demand=dem, fixed_params=par, want=("reward_traj", "final_obs"))
    rew, fin = out["reward_traj"].cpu().numpy(), out["final_obs"].cpu().numpy()
    for e in range(0, N, 25):
        o = oracle.newsvendor_episode(env.params, actions=acts[e], demand=dem[e], fixed=par[e])
        assert np.array_equal(o["reward"], rew[e]), (case, e)
        assert np.array_equal(o["obs"][-1], fin[e])
    for pol, pp, kw in (("classic", 0.9, dict(safety_factor=0.9)), ("sS", 1.3, dict(S_factor=1.3)),
                        ("order_up_to", 1.2, dict(safety_factor=1.2))):
        o2 = env.rollout(pol, demand=dem, fixed_params=par, want=("action_traj", "ep_return"), **kw)
        a2 = o2["action_traj"].cpu().numpy()
        for e in range(0, N, 50):
            o = oracle.newsvendor_episode(env.params, policy=pol, pparam=pp, demand=dem[e], fixed=par[e])
            assert np.array_equal(o["actions"], a2[e]), (case, pol, e)
            assert o2["ep_return"][e].item() == seq_sum(o["reward"])
    env.close()


def _random_graph(rng, ordered=False):
    import networkx as nx
    g = nx.DiGraph()
    n_mk, n_rt, n_ds, n_fc, n_raw = 2, int(rng.integers(1, 4)), int(rng.integers(1, 3)), int(rng.integers(1, 4)), 2
    ids = list(rng.permutation(n_mk + n_rt + n_ds + n_fc + n_raw) + 10)   # shuffled node ids: sorted order != insertion order
    if ordered:   # ids ascending market -> raw material, as in the reference's graphs (single-pass streaming kernel)
        ids = sorted(ids, reverse=True)
    take = lambda k: [int(ids.pop()) for _ in range(k)]  # noqa: E731
    mk, rt, ds, fc, raw = take(n_mk), take(n_rt), take(n_ds), take(n_fc), take(n_raw)
    g.add_nodes_from(mk)
    for j in rt + ds:
        g.add_node(j, I0=float(rng.choice([rng.integers(20, 300), rng.uniform(20, 300)])), h=float(rng.uniform(0, 0.1)))
    for j in fc:
        g.add_node(j, I0=float(rng.integers(50, 400)), h=float(rng.uniform(0, 0.05)), C=float(rng.integers(20, 120)),
                   o=float(rng.uniform(0, 0.05)), v=float(rng.choice([1.0, rng.uniform(0.5, 1.0)])))
    g.add_nodes_from(raw)
    edges = []
    for r in rt:
        for m in rng.choice(mk, size=int(rng.integers(1, 3)), replace=False):
            edges.append((r, int(m), dict(p=float(rng.uniform(2, 9)), b=float(rng.uniform(0, 0.5)),
                                          dist_param={"lam": float(rng.integers(1, 30))})))
    for lower, upper in ((rt, ds), (ds, fc), (fc, raw)):
        for j in lower:
            for s in rng.choice(upper, size=int(rng.integers(1, len(upper) + 1)), replace=False):
                edges.append((int(s), j, dict(L=int(rng.integers(0, 9)), p=float(rng.uniform(0.1, 2)),
                                              g=float(rng.uniform(0, 0.02)))))
    for i in rng.permutation(len(edges)):                                  # random insertion order
        u, v, a = edges[i]
        if "dist_param" in a:
            a = dict(a, demand_dist_func=lambda **p: 0)
        g.add_edge(u, v, **a)
    return g


@pytest.mark.parametrize("mode", ["specialised", "stream_jit", "stream_jit_twopass", "generic"])
@pytest.mark.parametrize("case", range(6 * STRESS))
def test_netinv_random_graph(case, mode, monkeypatch):
    from oracle import oracle
    torch = _torch()
    set_net_kernel_mode(monkeypatch, mode)
    rng = np.random.default_rng(3000 + case)
    g = _random_graph(rng, ordered=bool(case % 2))
    T = int(rng.integers(4, 26))
    N = 130
    env = pkg.NetInvMgmtMasterEnv(graph=g, num_periods=T, backlog=bool(case % 2), alpha=float(rng.uniform(0.9, 1.0)),
                                  num_envs=N, device="cuda:0")
    P = env.params
    E, M = len(P.reorder_links), len(P.retail_links)
    acts = (rng.uniform(-0.05, 0.3, size=(N, T, E)) * 300).astype(np.float32)
    acts[rng.random((N, T, E)) < 0.2] = np.float32(rng.integers(0, 40)) + np.float32(0.5)
    lam = np.array([g.edges[e]["dist_param"]["lam"] for e in P.retail_links])
    dem = rng.poisson(lam, size=(N, T, M)).astype(np.float64)
    obs, _ = env.reset(seed=case)
    rew = np.zeros((N, T))
    for t in range(T):
        obs, r, _, _, _ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
        rew[:, t] = r.cpu().numpy()
    last = obs.cpu().numpy()
    X, Y, U, _ = env.export_state()
    out = env.rollout("actions", actions=acts, demand=dem, want=("reward_traj", "final_X", "final_Y", "final_U"))
    assert np.array_equal(out["reward_traj"].cpu().numpy(), rew)
    assert torch.equal(out["final_X"], X) and torch.equal(out["final_Y"], Y) and torch.equal(out["final_U"], U)
    for e in range(0, N, 16):
        o = oracle.netinv_episode(P, actions=acts[e], demand=dem[e])
        assert np.array_equal(o["reward"], rew[e]), (case, mode, e)
        assert np.array_equal(o["obs"][-1], last[e])
        assert np.array_equal(o["X"][-1], X[e].cpu().numpy()) and np.array_equal(o["Y"][-1], Y[e].cpu().numpy())
    env.close()


def test_invmgmt_maximum_sizes():
    """The build limits of include/orgym_b200.h: 16 stages, lead times up to 64 (and 0), a horizon longer than the
    longest lead time; observation rows of 16*65 int64 do not fit a shared-memory tile."""
    from oracle import oracle
    torch = _torch()
    rng = np.random.default_rng(77)
    n, T, N = 16, 70, 130
    L = rng.integers(0, 65, n)
    L[0], L[1], L[2] = 64, 0, 63
    cfg = dict(periods=T, I0=rng.integers(0, 200, n).tolist(), p=31.5,
               r=np.sort(rng.uniform(0.5, 30, n + 1))[::-1].round(3).tolist(), k=rng.uniform(0, 1, n + 1).round(3).tolist(),
               h=rng.uniform(0, 0.5, n).round(3).tolist(), c=rng.integers(1, 300, n).tolist(), L=L.tolist(),
               dist_param={"mu": 33.0}, alpha=0.97)
    for backlog, wide in ((True, False), (False, True)):
        cls = pkg.InvManagementBacklogEnv if backlog else pkg.InvManagementLostSalesEnv
        env = cls(num_envs=N, device="cuda:0", wide_state=wide, autoreset_mode="disabled", **cfg)
        assert env.observation_space.shape[-1] == n * 65
        acts = rng.integers(0, 320, size=(N, T, n))
        dem = rng.poisson(33.0, size=(N, T)).astype(np.int64)
        obs, _ = env.reset(seed=1)
        rew = np.zeros((N, T))
        mid = None
        for t in range(T):
            obs, r, _, trunc, _ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
            rew[:, t] = r.cpu().numpy()
            if t == 40:
                mid = obs.cpu().numpy().copy()
        last = obs.cpu().numpy()
        out = env.rollout("actions", actions=acts, demand=dem, want=("reward_traj",))
        assert np.array_equal(out["reward_traj"].cpu().numpy(), rew)
        for e in (0, 1, 64, 127, 128, 129):
            o = oracle.invmgmt_episode(env.params, actions=acts[e], demand=dem[e])
            assert np.array_equal(o["reward"], rew[e])
            assert np.array_equal(o["obs"][41], mid[e]) and np.array_equal(o["obs"][-1], last[e])
        # on-device base-stock: both ring sets (fulfilled orders, requested orders) exceed shared memory here
        ob = env.rollout("base_stock", demand=dem, safety_factor=1.25, want=("ep_return", "final_I"))
        for e in (0, 64, 129):
            o = oracle.invmgmt_episode(env.params, policy="base_stock", demand=dem[e], safety_factor=1.25)
            assert ob["ep_return"][e].item() == seq_sum(o["reward"])
            assert np.array_equal(o["I"][-1], ob["final_I"][e].cpu().numpy())
        sampled = env.rollout("base_stock", seed=3, want=("ep_return", "summary"))
        assert np.isfinite(sampled["ep_return"].cpu().numpy()).all() and sampled["summary"][0].item() == N
        assert env.errors() == 0
        env.close()
    with pytest.raises(Exception):
        pkg.InvManagementBacklogEnv(num_envs=4, device="cuda:0", I0=[10] * 17, r=[1.0] * 18, k=[0.1] * 18, h=[0.1] * 17,
                                    c=[10] * 17, L=[1] * 17)
    with pytest.raises(Exception):
        pkg.InvManagementBacklogEnv(num_envs=4, device="cuda:0", L=[65, 5, 10])


def test_newsvendor_maximum_lead_time():
    from oracle import oracle
    torch = _torch()
    rng = np.random.default_rng(78)
    N, Lmax = 200, 64
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", lead_time=Lmax, step_limit=80, autoreset_mode="disabled")
    env.reset(seed=4)
    par = env.export_params().cpu().numpy()
    T = env.step_limit
    acts = (rng.random((N, T)) * 60).astype(np.float32)
    dem = rng.poisson(30.0, size=(N, T)).astype(np.int64)
    rew = np.zeros((N, T))
    for t in range(T):
        obs, r, _, _, _ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
        rew[:, t] = r.cpu().numpy()
    last = obs.cpu().numpy()
    out = env.rollout("actions", actions=acts, demand=dem, fixed_params=par, want=("reward_traj", "final_obs"))
    assert np.array_equal(out["reward_traj"].cpu().numpy(), rew)
    assert np.array_equal(out["final_obs"].cpu().numpy(), last)
    for e in (0, 99, 199):
        o = oracle.newsvendor_episode(env.params, actions=acts[e], demand=dem[e], fixed=par[e])
        assert np.array_equal(o["reward"], rew[e]) and np.array_equal(o["obs"][-1], last[e])
    env.close()
    with pytest.raises(Exception):
        pkg.NewsvendorEnv(num_envs=4, device="cuda:0", lead_time=65)


def test_netinv_maximum_sizes(monkeypatch):
    """Network env at the build limits: 64 main nodes, 128 reorder links, 30 retail links, lead times 0..64, 70 periods
    (observation rows of ~1000 float32) -- through the generic kernel (the specialised kernels are covered by the
    64-node test of test_netinv_gpu.py)."""
    from oracle import oracle
    torch = _torch()
    monkeypatch.setenv("ORGYM_NET_JIT", "0")
    g = pkg.synthetic_graph(1, layers=(16, 20, 22, 22, 20))
    links = [e for e in g.edges() if "L" in g.edges[e]]
    for k, e in enumerate(links[:6]):
        g.edges[e]["L"] = [64, 63, 0, 1, 64, 33][k]
    T, N = 70, 70
    rng = np.random.default_rng(9)
    for backlog in (True, False):
        env = pkg.NetInvMgmtMasterEnv(graph=g, num_periods=T, backlog=backlog, num_envs=N, device="cuda:0",
                                      autoreset_mode="disabled")
        P = env.params
        J, E, M = len(P.main_nodes), len(P.reorder_links), len(P.retail_links)
        assert (J, E) == (64, 128) and 16 <= M <= 32 and not env.specialised
        acts = (rng.random((N, T, E)) * 90).astype(np.float32)
        dem = rng.poisson(20, size=(N, T, M)).astype(np.float64)
        obs, _ = env.reset(seed=2)
        rew = np.zeros((N, T))
        for t in range(T):
            obs, r, _, _, _ = env.step(torch.from_numpy(acts[:, t]).cuda(), demand=torch.from_numpy(dem[:, t]).cuda())
            rew[:, t] = r.cpu().numpy()
        last = obs.cpu().numpy()
        out = env.rollout("actions", actions=acts, demand=dem, want=("reward_traj",))
        assert np.array_equal(out["reward_traj"].cpu().numpy(), rew)
        for e in (0, 33, 69):
            o = oracle.netinv_episode(P, actions=acts[e], demand=dem[e])
            assert np.array_equal(o["reward"], rew[e]) and np.array_equal(o["obs"][-1], last[e])
        env.close()
