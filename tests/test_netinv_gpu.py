"""GPU parity tests of the network env (csrc/netinv.cu) through the C ABI."""
import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from helpers import golden_files, ids, load_golden, net_kwargs, net_S_columns, seq_sum, set_net_kernel_mode

pytestmark = pytest.mark.gpu
NET = golden_files("net_")


def _torch():
    import torch
    return torch


@pytest.fixture(params=["specialised", "stream_jit", "stream_jit_twopass", "stream_jit_fused_obs", "generic"])
def kernel_mode(request, monkeypatch):
    """Run the parity tests through all network kernels: the NVRTC-specialised register-resident one; the streaming
    STEP path meant for large graphs, forced here, in its forms -- generated streaming kernel (single pass over the
    nodes: the default for large graphs; or two passes with scratch rows, the form for graphs whose suppliers do not
    follow their purchasers in node order) + observation kernel, generated kernel with its own fused observation
    pass --; and the generic constant-bank interpreter."""
    set_net_kernel_mode(monkeypatch, request.param)
    return request.param


def _mk(meta, n, **kw):
    return pkg.NetInvMgmtMasterEnv(**net_kwargs(meta), num_envs=n, device="cuda:0", **kw)


@pytest.mark.parametrize("path", NET, ids=ids(NET))
def test_step_matches_reference(path, kernel_mode):
    torch = _torch()
    g, meta = load_golden(path)
    E = len(g["seeds"])
    env = _mk(meta, E, autoreset_mode="disabled")
    cols = net_S_columns(meta)
    obs, _ = env.reset(seed=0)
    assert np.array_equal(obs.cpu().numpy(), g["obs"][:, 0])
    for t in range(env.num_periods):
        obs, r, term, trunc, info = env.step(torch.from_numpy(g["actions"][:, t]).cuda(),
                                             demand=torch.from_numpy(g["D"][:, t]).cuda())
        assert np.array_equal(obs.cpu().numpy(), g["obs"][:, t + 1]), t
        assert np.array_equal(r.cpu().numpy(), g["reward"][:, t]), t   # bit-exact float64
        assert np.array_equal(trunc.cpu().numpy(), g["truncated"][:, t])
        assert not term.any()
        X, Y, U, per = env.export_state()
        assert np.array_equal(X.cpu().numpy(), g["X"][:, t + 1])
        assert np.array_equal(Y.cpu().numpy(), g["Y"][:, t + 1])
        assert np.array_equal(U.cpu().numpy(), g["U"][:, t + 1])
        assert np.array_equal(info["sales"].cpu().numpy(), g["S"][:, t][:, cols])
        assert np.array_equal(info["profit_node"].cpu().numpy(), g["P"][:, t])
        assert np.array_equal(info["profit_period_undiscounted"].cpu().numpy(), g["profit"][:, t])
        assert np.array_equal(info["demand"].cpu().numpy(), g["D"][:, t])
    assert env.errors() == 0
    env.close()


@pytest.mark.parametrize("path", NET, ids=ids(NET))
def test_rollout_replay_matches_reference(path, kernel_mode):
    g, meta = load_golden(path)
    E = len(g["seeds"])
    env = _mk(meta, E)
    out = env.rollout("actions", actions=g["actions"], demand=g["D"],
                      want=("ep_return", "stats", "reward_traj", "final_X", "final_Y", "final_U", "summary"))
    assert np.array_equal(out["reward_traj"].cpu().numpy(), g["reward"])
    assert np.array_equal(out["final_X"].cpu().numpy(), g["X"][:, -1])
    assert np.array_equal(out["final_Y"].cpu().numpy(), g["Y"][:, -1])
    assert np.array_equal(out["final_U"].cpu().numpy(), g["U"][:, -1])
    ret = out["ep_return"].cpu().numpy()
    for e in range(E):
        assert ret[e] == seq_sum(g["reward"][e])
    st = out["stats"].cpu().numpy()
    assert np.array_equal(st[:, 1], g["D"].sum(axis=(1, 2)))
    assert np.allclose(st[:, 3], np.maximum(g["X"][:, 1:], 0).sum(axis=(1, 2)), rtol=1e-12)
    out2 = env.rollout("actions", actions=np.ascontiguousarray(g["actions"].transpose(1, 0, 2)),
                       demand=np.ascontiguousarray(g["D"].transpose(1, 0, 2)), time_major=True, want=("ep_return",))
    assert np.array_equal(out2["ep_return"].cpu().numpy(), ret)
    env.close()


USER_D = [p for p in NET if "userD" in p]


@pytest.mark.parametrize("path", USER_D, ids=ids(USER_D))
def test_user_D_trace_drives_the_market_link(path, kernel_mode):
    """network_management.py:250-255: a retail link with a user_D trace (sum > 0) and sample_path False replays the
    trace (rounded, clamped at 0, last entry repeated); with sample_path True it samples from its distribution.  No
    `demand=` override here: the trace lives in the handle.  Sampled links get the recorded demand replayed through
    the override only where the trace does not apply, so the whole episode can be compared with the reference."""
    torch = _torch()
    g, meta = load_golden(path)
    n = len(g["seeds"])
    rt = [tuple(x) for x in meta["retail_links"]]
    sp = {(u, v): bool(f) for u, v, f in meta["sample_path"]}
    traced = [i for i, e in enumerate(rt) if e in sp and not sp[e]]
    sampled = [i for i in range(len(rt)) if i not in traced]
    assert traced or "samplepath" in path
    env = _mk(meta, n, autoreset_mode="disabled")
    T = env.num_periods
    # (1) device-side demand: traced links equal the reference's D column, sampled links do not replay the trace
    env.reset(seed=77)
    D = np.zeros((n, T, len(rt)))
    for t in range(T):
        _, _, _, _, info = env.step(torch.from_numpy(g["actions"][:, t]).cuda())
        D[:, t] = info["demand"].cpu().numpy()
    assert np.array_equal(D[:, :, traced], g["D"][:, :, traced])
    for i in sampled:
        assert (D[:, :, i] >= 0).all() and D[:, :, i].std() > 0
        tr = dict(((u, v), t_) for u, v, t_ in meta["user_D"]).get(rt[i])
        if tr is not None:
            assert not np.array_equal(D[0, :, i], np.maximum(0, np.round(np.asarray(tr[:T]))))
    # (2) the fused rollout reads the same trace
    out = env.rollout("actions", actions=g["actions"], seed=77, want=("stats", "reward_traj"))
    assert np.array_equal(out["stats"].cpu().numpy()[:, 1], D.sum(axis=(1, 2)))
    if not sampled:      # every market link traced: the whole episode is the reference's, without any override
        assert np.array_equal(out["reward_traj"].cpu().numpy(), g["reward"])
    env.close()


def test_synthetic_64_generator_matches_golden_topology(kernel_mode):
    """The product's synthetic_graph(64) is the graph the reference ran for the net_synth64 goldens; stepping an env
    built from the generator directly (not from the recorded spec) reproduces the reference."""
    torch = _torch()
    path = [p for p in NET if "synth64_lost_random" in p][0]
    g, meta = load_golden(path)
    G = pkg.synthetic_graph(meta["synthetic_graph_seed"])
    env = pkg.NetInvMgmtMasterEnv(graph=G, backlog=meta["backlog"], num_periods=meta["num_periods"],
                                  num_envs=len(g["seeds"]), device="cuda:0", autoreset_mode="disabled")
    assert [int(j) for j in env.main_nodes] == meta["main_nodes"]
    assert [list(e) for e in env.reorder_links] == meta["reorder_links"]
    assert [list(e) for e in env.retail_links] == meta["retail_links"]
    env.reset(seed=0)
    for t in range(env.num_periods):
        obs, r, *_ = env.step(torch.from_numpy(g["actions"][:, t]).cuda(), demand=torch.from_numpy(g["D"][:, t]).cuda())
        assert np.array_equal(obs.cpu().numpy(), g["obs"][:, t + 1]), t
        assert np.array_equal(r.cpu().numpy(), g["reward"][:, t]), t
    env.close()


def test_class_surface_and_constant_policy(kernel_mode):
    """Class names / defaults of the reference, ConstantOrderAgent rollout vs oracle with device-sampled demand."""
    from oracle import oracle
    torch = _torch()
    N = 3001
    env = pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled")
    assert env.obs_dim == 68 and env.single_action_space.shape == (11,) and env.single_action_space.high[0] == 1700
    assert pkg.NetInvMgmtLostSalesEnv(num_envs=2, device="cuda:0").backlog is True      # reference quirk
    assert pkg.NetInvMgmtLostSalesEnv(num_envs=2, device="cuda:0", backlog=False).backlog is False
    ec = pkg.network_management_custom.NetInvMgmtLostSalesEnv(num_envs=2, device="cuda:0", num_periods=40)
    assert ec.obs_dim == 12 and ec.single_action_space.high[0] == 3200
    a = (env.single_action_space.high * 0.1).astype(np.float32)
    T = env.num_periods
    env.reset(seed=6000)
    dem = torch.zeros((N, T, 1), dtype=torch.float64, device="cuda")
    rew = torch.zeros((N, T), dtype=torch.float64, device="cuda")
    a_d = torch.from_numpy(np.tile(a, (N, 1))).cuda()
    for t in range(T):
        obs, r, _, trunc, info = env.step(a_d)
        dem[:, t] = info["demand"]
        rew[:, t] = r
    last = obs.clone()
    out = env.rollout("constant", order_fraction=0.1, seed=6000, want=("ep_return", "reward_traj", "final_X", "stats", "summary"))
    assert torch.equal(out["reward_traj"], rew)                 # same Philox stream in step and rollout
    assert torch.equal(out["stats"][:, 1], dem.sum(dim=(1, 2)))
    dem_h, rew_h = dem.cpu().numpy(), rew.cpu().numpy()
    assert 15 < dem_h.mean() < 25
    for e in range(0, N, 250):
        o = oracle.netinv_episode(env.params, actions=a, demand=dem_h[e], constant=True)
        assert np.array_equal(o["reward"], rew_h[e])
        assert np.array_equal(o["obs"][-1], last[e].cpu().numpy())
        assert np.array_equal(o["X"][-1], out["final_X"][e].cpu().numpy())
    s = out["summary"].cpu().numpy()
    assert s[0] == N and np.isclose(s[1], out["ep_return"].sum().item(), rtol=1e-12)
    # sharding invariance
    sub = pkg.NetInvMgmtBacklogEnv(num_envs=100, device="cuda:0", env_offset=500)
    o2 = sub.rollout("constant", order_fraction=0.1, seed=6000, want=("ep_return",))
    assert torch.equal(o2["ep_return"], out["ep_return"][500:600])
    env.close()


@pytest.mark.parametrize("spec", [True, False], ids=["specialised-streaming", "generic"])
def test_synthetic_64_node_network_vs_oracle(spec):
    """Config 5's synthetic 64-node network (lost sales): random actions, device demand, vs the oracle -- through the
    specialised kernels (streaming STEP kernel for large graphs) and the generic one."""
    from oracle import oracle
    torch = _torch()
    G = pkg.synthetic_graph(64)
    N = 300
    env = pkg.NetInvMgmtMasterEnv(graph=G, backlog=False, num_envs=N, device="cuda:0", specialise=spec)
    assert env.specialised == spec
    P = env.params
    E, M, T = len(P.reorder_links), len(P.retail_links), env.num_periods
    assert len(G.nodes) == 64
    rng = np.random.default_rng(5)
    acts = (rng.uniform(0, 0.08, size=(N, T, E)) * env.single_action_space.high).astype(np.float32)
    env.reset(seed=12000)
    dem = torch.zeros((N, T, M), dtype=torch.float64, device="cuda")
    rew = torch.zeros((N, T), dtype=torch.float64, device="cuda")
    a_d = torch.from_numpy(acts).cuda()
    for t in range(T):
        obs, r, _, _, info = env.step(a_d[:, t])
        dem[:, t] = info["demand"]
        rew[:, t] = r
    out = env.rollout("actions", actions=a_d, seed=12000, want=("reward_traj", "final_X"))
    assert torch.equal(out["reward_traj"], rew)
    dem_h, rew_h = dem.cpu().numpy(), rew.cpu().numpy()
    for e in range(0, N, 37):
        o = oracle.netinv_episode(P, actions=acts[e], demand=dem_h[e])
        assert np.array_equal(o["reward"], rew_h[e])
        assert np.array_equal(o["obs"][-1], obs[e].cpu().numpy())
    env.close()


def test_masked_reset_puts_instances_of_one_tile_in_different_periods(kernel_mode):
    """After reset(options={'reset_mask': ...}) the instances of a 128-instance state tile are in different periods; the
    observation window of every instance must still be rotated by ITS period (the TMA-staged observation kernel takes
    its per-instance path for such tiles).  Checked against a second env that is stepped from a fresh reset."""
    torch = _torch()
    N, E = 300, 11
    rng = np.random.default_rng(3)
    acts = torch.from_numpy((rng.uniform(0, 0.1, size=(12, N, E)) * 1700).astype(np.float32)).cuda()
    dem = torch.from_numpy(rng.poisson(20, size=(12, N, 1)).astype(np.float64)).cuda()
    a = pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled")
    b = pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled")
    a.reset(seed=5)
    for t in range(5):
        a.step(acts[t], demand=dem[t])
    mask = torch.zeros(N, dtype=torch.bool, device="cuda")
    mask[::3] = True
    a.reset(options={"reset_mask": mask})
    b.reset(seed=5)
    for t in range(5, 12):                       # masked instances of `a` restart at period 0, the others continue
        oa, ra, *_ = a.step(acts[t], demand=dem[t])
        ob, rb, *_ = b.step(acts[t], demand=dem[t])
        assert torch.equal(oa[mask], ob[mask]) and torch.equal(ra[mask], rb[mask])
    per = a.export_state()[3]
    assert (per[mask] == 7).all() and (per[~mask] == 12).all()
    # the instances that were not reset continue their own episode: compare with an uninterrupted run
    c = pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="disabled")
    c.reset(seed=5)
    for t in range(12):
        oc, rc, *_ = c.step(acts[t], demand=dem[t])
    assert torch.equal(oa[~mask], oc[~mask]) and torch.equal(ra[~mask], rc[~mask])
    for e in (a, b, c):
        e.close()


def test_autoreset_next_step(kernel_mode):
    torch = _torch()
    env = pkg.NetInvMgmtBacklogEnv(num_envs=130, device="cuda:0", num_periods=3)
    obs0 = env.reset(seed=1)[0].clone()
    a = torch.full((130, 11), 50.0, device="cuda")
    for _ in range(3):
        obs, r, term, trunc, _ = env.step(a)
    assert trunc.all() and not torch.equal(obs, obs0)
    obs, r, term, trunc, _ = env.step(a)
    assert torch.equal(obs, obs0) and (r == 0).all() and not trunc.any()
    env.close()


def test_mlp_policy_drives_step_api_zero_copy():
    """BASELINE config 5 in miniature: a torch MLP (obs -> 64 -> 64 -> actions, tanh, scaled to the action bound)
    drives the 64-node lost-sales network through the step API; observations and actions never leave the GPU.
    The recorded trajectory is replayed through the oracle."""
    from oracle import oracle
    torch = _torch()
    G = pkg.synthetic_graph(64)
    N = 96
    env = pkg.NetInvMgmtMasterEnv(graph=G, backlog=False, num_envs=N, device="cuda:0", autoreset_mode="disabled")
    E, M, T = len(env.reorder_links), len(env.retail_links), env.num_periods
    torch.manual_seed(0)
    mlp = torch.nn.Sequential(torch.nn.Linear(env.obs_dim, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh(),
                              torch.nn.Linear(64, E), torch.nn.Sigmoid()).cuda()
    high = torch.from_numpy(env.single_action_space.high).cuda()
    obs, _ = env.reset(seed=12000)
    acts = torch.zeros((N, T, E), dtype=torch.float32, device="cuda")
    dem = torch.zeros((N, T, M), dtype=torch.float64, device="cuda")
    rew = torch.zeros((N, T), dtype=torch.float64, device="cuda")
    with torch.no_grad():
        for t in range(T):
            assert obs.data_ptr() == env._obs.data_ptr()           # zero-copy: the env's own buffer
            a = mlp(obs / 1000.0) * high * 0.05
            obs, r, term, trunc, info = env.step(a)
            acts[:, t], dem[:, t], rew[:, t] = a, info["demand"], r
    assert trunc.all()
    a_h, d_h, r_h = acts.cpu().numpy(), dem.cpu().numpy(), rew.cpu().numpy()
    for e in range(0, N, 19):
        o = oracle.netinv_episode(env.params, actions=a_h[e], demand=d_h[e])
        assert np.array_equal(o["reward"], r_h[e])
        assert np.array_equal(o["obs"][-1], obs[e].cpu().numpy())
    env.close()


def test_history_buffers_match_reference_frames():
    """record_history=True: X/Y/U/R/S/D/P history tensors equal the reference's DataFrames."""
    torch = _torch()
    path = [p for p in NET if "yield_backlog_random" in p][0]
    g, meta = load_golden(path)
    env = _mk(meta, len(g["seeds"]), autoreset_mode="disabled", record_history=True)
    cols = net_S_columns(meta)
    env.reset(seed=0)
    for t in range(env.num_periods):
        env.step(torch.from_numpy(g["actions"][:, t]).cuda(), demand=torch.from_numpy(g["D"][:, t]).cuda())
    for name in ("X", "Y", "U", "R", "D", "P"):
        assert np.array_equal(getattr(env, name).cpu().numpy(), g[name]), name
    assert np.array_equal(env.S.cpu().numpy(), g["S"][:, :, cols])
    env.close()
