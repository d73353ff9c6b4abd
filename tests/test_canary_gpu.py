"""Out-of-bounds write detection without compute-sanitizer (it is closed on this GPU pool): every device buffer the
kernels write (state, obs, reward, flags, info, rollout outputs) is re-seated inside a larger allocation filled with a
canary pattern; after reset / step / rollout with ragged batch sizes the canaries must be intact."""
import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from helpers import set_net_kernel_mode

pytestmark = pytest.mark.gpu
PAD = 4096  # bytes on each side


def _torch():
    import torch
    return torch


class Guard:
    def __init__(self):
        self.items = []

    def wrap(self, t):
        """Return a tensor like `t` (same shape/dtype/content) living inside a canary-padded allocation."""
        torch = _torch()
        nbytes = t.numel() * t.element_size()
        big = torch.full((nbytes + 2 * PAD,), 0xA5, dtype=torch.uint8, device=t.device)
        inner = big[PAD:PAD + nbytes].view(t.dtype).view(t.shape)
        inner.copy_(t)
        self.items.append((big, nbytes))
        return inner

    def check(self):
        torch = _torch()
        torch.cuda.synchronize()
        for big, nbytes in self.items:
            assert bool((big[:PAD] == 0xA5).all()) and bool((big[PAD + nbytes:] == 0xA5).all()), "canary overwritten"


def _guard_env(env, g, rollout_names, shapes):
    torch = _torch()
    for name in ("_state", "_obs", "_reward", "_terminated", "_truncated", "_final_obs"):
        if hasattr(env, name) and getattr(env, name) is not None:
            setattr(env, name, g.wrap(getattr(env, name)))
    for k in list(env._info_t):
        env._info_t[k] = g.wrap(env._info_t[k])
    # re-point the info struct at the guarded tensors
    info = env._info
    mapping = {"invmgmt": dict(demand="demand_realized", sales="sales", unfulfilled="unfulfilled", profit="period_profit"),
               "newsvendor": dict(demand="demand", parts="parts"),
               "netinv": dict(demand="demand", sales="sales", profit="profit_node", profit_total="profit_period_undiscounted")}
    for field, key in mapping[env._family].items():
        if key in env._info_t:
            setattr(info, field, env._info_t[key].data_ptr())
    if hasattr(env, "_final_obs"):
        info.final_obs = env._final_obs.data_ptr()
    cache = env.__dict__.setdefault("_rollout_buf", {}).setdefault(0, {})
    for name in rollout_names:
        shp, dt = shapes[name]
        cache[name] = g.wrap(torch.zeros(shp, dtype=dt, device=env.device))


@pytest.mark.parametrize("N", [1, 127, 129, 1000])
@pytest.mark.parametrize("wide", [False, True])
def test_invmgmt_no_oob_writes(N, wide):
    torch = _torch()
    env = pkg.InvManagementBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="same_step", wide_state=wide, periods=7)
    g = Guard()
    T, n, m = 7, 3, 4
    shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.int64), reward_traj=((N, T), torch.float64),
                  final_I=((N, n), torch.int64), final_B=((N, m), torch.int64), summary=((8,), torch.float64),
                  stats32=((N, 4), torch.int32))
    _guard_env(env, g, list(shapes), shapes)
    env.reset(seed=1)
    a = torch.randint(0, 200, (N, n), dtype=torch.int64, device="cuda")
    for _ in range(9):      # crosses an episode boundary (same-step autoreset writes final_obs)
        env.step(a)
    for pol in ("base_stock", "random"):
        env.rollout(pol, want=tuple(shapes))
    g.check()
    env.close()


@pytest.mark.parametrize("N", [1, 127, 129, 1000])
def test_newsvendor_no_oob_writes(N):
    torch = _torch()
    env = pkg.NewsvendorEnv(num_envs=N, device="cuda:0", autoreset_mode="same_step", step_limit=6, lead_time=7)
    g = Guard()
    T = 6
    shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.float64), reward_traj=((N, T), torch.float64),
                  action_traj=((N, T), torch.float32), final_obs=((N, env.obs_dim), torch.float32),
                  summary=((8,), torch.float64))
    _guard_env(env, g, list(shapes), shapes)
    env.reset(seed=1)
    a = torch.rand((N, 1), device="cuda") * 300
    for _ in range(8):
        env.step(a)
    for pol in ("classic", "sS", "order_up_to"):
        env.rollout(pol, want=tuple(shapes))
    g.check()
    env.close()


@pytest.mark.parametrize("mode", ["specialised", "stream_jit", "stream_jit_twopass", "generic"])
@pytest.mark.parametrize("N", [1, 127, 129, 600])
def test_netinv_no_oob_writes(N, mode, monkeypatch):
    torch = _torch()
    set_net_kernel_mode(monkeypatch, mode)
    env =pkg.NetInvMgmtBacklogEnv(num_envs=N, device="cuda:0", autoreset_mode="same_step", num_periods=5)
    g = Guard()
    T, J, E, M = 5, 6, 11, 1
    shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.float64), reward_traj=((N, T), torch.float64),
                  final_X=((N, J), torch.float64), final_Y=((N, E), torch.float64), final_U=((N, M), torch.float64),
                  summary=((8,), torch.float64))
    _guard_env(env, g, list(shapes), shapes)
    env._scratch = g.wrap(torch.zeros_like(env._state))
    env.reset(seed=1)
    a = torch.rand((N, E), device="cuda") * 200
    for _ in range(7):
        env.step(a)
    env.rollout("constant", want=tuple(shapes))
    g.check()
    env.close()
