"""Batched multi-period newsvendor -- drop-in for the reference's `newsvendor.py` (NewsvendorEnv).

Same constructor keywords (newsvendor.py:52-61), spaces (:76-88), reset/step semantics (:100-204) for
`num_envs` independent instances on one GPU (csrc/newsvendor.cu behind the C ABI).
"""
import ctypes as C
from typing import Dict, Optional

import numpy as np

from . import _capi
from .mlp import pack_mlp
from .spaces import Box
from .vector import BatchedEnv, _AUTORESET, _torch

POLICIES = {"actions": 0, "order_up_to": 1, "classic": 2, "sS": 3}
POLICY_MLP = 4


class NewsvendorParams:
    """Host mirror of NewsvendorEnv.__init__ (newsvendor.py:52-98)."""

    def __init__(self, lead_time: int = 5, max_inventory: int = 4000, max_order_quantity: int = 2000,
                 step_limit: int = 40, p_max: float = 100.0, h_max: float = 5.0, k_max: float = 10.0,
                 mu_max: float = 200.0, gamma: float = 1.0, env_config: Optional[Dict] = None):
        if env_config:  # convenience: the same keys in a dict (RLlib-style env_creator(env_config))
            locals_ = dict(lead_time=lead_time, max_inventory=max_inventory, max_order_quantity=max_order_quantity,
                           step_limit=step_limit, p_max=p_max, h_max=h_max, k_max=k_max, mu_max=mu_max, gamma=gamma)
            locals_.update(env_config)
            lead_time, max_inventory, max_order_quantity = locals_["lead_time"], locals_["max_inventory"], locals_["max_order_quantity"]
            step_limit, p_max, h_max, k_max = locals_["step_limit"], locals_["p_max"], locals_["h_max"], locals_["k_max"]
            mu_max, gamma = locals_["mu_max"], locals_["gamma"]
        self.lead_time = max(0, lead_time)  # :65
        self.max_inventory = max_inventory
        self.max_order_quantity = max_order_quantity
        self.step_limit = step_limit
        self.p_max, self.h_max, self.k_max, self.mu_max = p_max, h_max, k_max, mu_max
        self.gamma = gamma
        self.obs_dim = self.lead_time + 5  # :76

    def spaces(self):
        obs_low = np.zeros(self.obs_dim, dtype=np.float32)
        obs_high = np.array([self.p_max, self.p_max, self.h_max, self.k_max, self.mu_max] +
                            [self.max_order_quantity] * self.lead_time, dtype=np.float32)
        observation_space = Box(low=obs_low, high=obs_high, dtype=np.float32)
        action_space = Box(low=np.array([0], dtype=np.float32),
                           high=np.array([self.max_order_quantity], dtype=np.float32), dtype=np.float32)
        return observation_space, action_space

    def to_c(self, keep=None):
        c = _capi.NvConfig()
        c.lead_time = int(self.lead_time)
        c.step_limit = int(self.step_limit)
        c.max_inventory = float(self.max_inventory)
        c.max_order_quantity = float(self.max_order_quantity)
        c.p_max, c.h_max, c.k_max, c.mu_max = float(self.p_max), float(self.h_max), float(self.k_max), float(self.mu_max)
        return c


class NewsvendorEnv(BatchedEnv):
    """`num_envs` newsvendor instances in lock-step on one GPU.  Extra keywords: `num_envs`, `device`,
    `env_offset`, `autoreset_mode`, `info_level` (see InvManagementMasterEnv)."""

    _family = "newsvendor"
    metadata = {"render_modes": [], "render_fps": 4}

    def __init__(self, *args, num_envs: int = 1, device="cuda", env_offset: int = 0,
                 autoreset_mode: str = "next_step", info_level: int = 1, **kwargs):
        torch = _torch()
        self.params = NewsvendorParams(*args, **kwargs)
        P = self.params
        for name in ("lead_time", "max_inventory", "max_order_quantity", "step_limit", "p_max", "h_max", "k_max",
                     "mu_max", "gamma", "obs_dim"):
            setattr(self, name, getattr(P, name))
        self.observation_space_single, self.action_space_single = P.spaces()
        self._setup_batch(num_envs, device, env_offset, autoreset_mode)
        self.info_level = int(info_level)
        lib = _capi.lib()
        cfg = P.to_c()
        _capi.check(lib.orgym_newsvendor_create(C.byref(cfg), self.num_envs, self.device.index, C.byref(self._h)))
        N, od, dev = self.num_envs, P.obs_dim, self.device
        self._alloc_state(lib.orgym_newsvendor_state_bytes(self._h))
        self._obs = torch.zeros((N, od), dtype=torch.float32, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float64, device=dev)
        self._terminated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._info = _capi.NvInfo()
        self._info_views = None
        self._info_t = {}
        if self.info_level >= 1:
            self._info_t = dict(demand=torch.zeros(N, dtype=torch.int64, device=dev),
                                parts=torch.zeros((4, N), dtype=torch.float64, device=dev).t())  # column-major storage
            self._info.info_ld = N
            self._info.demand = self._info_t["demand"].data_ptr()
            self._info.parts = self._info_t["parts"].data_ptr()
        if autoreset_mode == "same_step":
            self._final_obs = torch.zeros((N, od), dtype=torch.float32, device=dev)
            self._info.final_obs = self._final_obs.data_ptr()
        self._has_reset = False

    def reset(self, *, seed=None, options: Optional[Dict] = None):
        """reset (newsvendor.py:100-123).  options={'fixed_params': {...}} pins (price, cost, h, k, mu) like
        CustomizableNewsvendorEnv (benchmark_newsvendor_sb3_rllib.py:276-291); each value may be a scalar or a
        length-N array.  options={'reset_mask': bool[N]} resets a subset."""
        torch = _torch()
        reseed, base = self._resolve_seed(seed)
        mask = fixed = None
        if options and options.get("reset_mask") is not None:
            mask = self._to_dev(options["reset_mask"], torch.uint8, (self.num_envs,))
        if options and options.get("fixed_params") is not None:
            fp = options["fixed_params"]
            if isinstance(fp, dict):
                cols = [np.broadcast_to(np.asarray(fp[k], np.float64), (self.num_envs,)) for k in
                        ("price", "cost", "h", "k", "mu")]
                fp = np.stack(cols, axis=1)
            fixed = self._to_dev(fp, torch.float64, (self.num_envs, 5))
        _capi.check(_capi.lib().orgym_newsvendor_reset(self._h, self._ptr(self._state), reseed, C.c_uint64(base),
                                                       self.env_offset, self._ptr(mask), self._ptr(fixed),
                                                       self._ptr(self._obs), self._stream()))
        self._has_reset = True
        return self._obs, {}

    def step(self, actions, demand=None):
        """step (newsvendor.py:125-204): actions float32 [N,1] (or [N]); optional replayed demand int64[N]."""
        torch = _torch()
        if not self._has_reset:
            raise RuntimeError("call reset() before step()")
        a = self._to_dev(actions, torch.float32, (self.num_envs,))
        d = self._to_dev(demand, torch.int64, (self.num_envs,)) if demand is not None else None
        _capi.check(_capi.lib().orgym_newsvendor_step(
            self._h, self._ptr(self._state), self._ptr(a), self._ptr(d), _AUTORESET[self.autoreset_mode],
            self._ptr(self._obs), self._ptr(self._reward), self._ptr(self._terminated), self._ptr(self._truncated),
            C.byref(self._info), self._stream()))
        if self._info_views is None:      # views of the (fixed) output buffers, built once: slicing costs microseconds
            v = {}
            if self._info_t:
                p = self._info_t["parts"]
                v = dict(demand=self._info_t["demand"], revenue=p[:, 0], purchase_cost=p[:, 1], holding_cost=p[:, 2],
                         lost_sales_penalty=p[:, 3])
            if self.autoreset_mode == "same_step":
                v["final_obs"] = self._final_obs
            self._info_views = (v, self._terminated.view(torch.bool), self._truncated.view(torch.bool))
        v, term, trunc = self._info_views
        return self._obs, self._reward, term, trunc, dict(v)

    def export_params(self):
        """float64[N,5]: price, cost, h, k, mu as the reference's Python floats (newsvendor.py:105-111)."""
        torch = _torch()
        out = torch.empty((self.num_envs, 5), dtype=torch.float64, device=self.device)
        _capi.check(_capi.lib().orgym_newsvendor_export_params(self._h, self._ptr(self._state), self._ptr(out),
                                                               self._stream()))
        return out

    def rollout(self, policy="classic", *, seed=None, episode=0, safety_factor=1.0, S_factor=1.2, actions=None,
                demand=None, fixed_params=None, time_major=False, want=("ep_return", "stats", "summary"), buffer_set=0):
        """Fused reset + step_limit periods (K1/K2).  policy: 'order_up_to' | 'classic' | 'sS' | 'actions'
        (float32 [N,T] or [T,N]) | an actor network -- a torch.nn.Sequential (Linear, Tanh|ReLU, ..., Linear) or an
        SB3 ActorCriticPolicy (e.g. `model.policy` of a trained PPO) -- evaluated on the device every period on the
        observation step() would return, its output clipped to [0, max_order_quantity] like SB3's deterministic
        predict.  Returns device tensors: ep_return f64[N], stats f64[N,4] (sum sales units, demand, lost units,
        excess units), summary f64[8]; on request reward_traj, action_traj, final_obs."""
        torch = _torch()
        P = self.params
        N, T = self.num_envs, int(P.step_limit)
        rin = _capi.NvRolloutIn()
        keep = []
        if isinstance(policy, str):
            rin.policy = POLICIES[policy]
            rin.param[0] = float(S_factor if policy == "sS" else safety_factor)
        else:
            mlp, tensors = pack_mlp(policy, P.obs_dim, 1, self.device)
            keep += [mlp, tensors]
            rin.policy = POLICY_MLP
            rin.mlp = C.pointer(mlp)
        if policy == "actions":
            a = self._to_dev(actions, torch.float32, (T, N) if time_major else (N, T))
            keep.append(a)
            rin.actions = a.data_ptr()
            rin.act_stride_env, rin.act_stride_t = (1, N) if time_major else (T, 1)
        if demand is not None:
            d = self._to_dev(demand, torch.int64, (T, N) if time_major else (N, T))
            keep.append(d)
            rin.demand = d.data_ptr()
            rin.dem_stride_env, rin.dem_stride_t = (1, N) if time_major else (T, 1)
        if fixed_params is not None:
            f = self._to_dev(fixed_params, torch.float64, (N, 5))
            keep.append(f)
            rin.fixed_params = f.data_ptr()
        shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.float64),
                      reward_traj=((N, T), torch.float64), action_traj=((N, T), torch.float32),
                      final_obs=((N, P.obs_dim), torch.float32), summary=((8,), torch.float64))
        out = {}
        rout = _capi.NvRolloutOut()
        cache = self.__dict__.setdefault("_rollout_buf", {}).setdefault(int(buffer_set), {})
        for name in want:
            shp, dt = shapes[name]
            if name not in cache:
                cache[name] = torch.zeros(shp, dtype=dt, device=self.device)
            out[name] = cache[name]
            setattr(rout, name, out[name].data_ptr())
        if seed is not None:
            self._resolve_seed(seed)
        elif not self._seeded:
            self._resolve_seed(None)
        _capi.check(_capi.lib().orgym_newsvendor_rollout(self._h, C.c_uint64(self._seed), self.env_offset,
                                                         C.c_uint32(int(episode)), C.byref(rin), C.byref(rout),
                                                         self._stream()))
        return out
