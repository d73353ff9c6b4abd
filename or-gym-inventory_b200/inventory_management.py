"""Batched serial multi-echelon inventory env -- drop-in for the reference's
`inventory_management.py` (InvManagementMasterEnv / InvManagementBacklogEnv / InvManagementLostSalesEnv).

Same constructor keywords and `env_config` keys (inventory_management.py:48-63), same spaces
(:111-128, :442-451), same step semantics (:224-352) -- for `num_envs` independent instances at once, on
one GPU.  The dynamics run in the CUDA library (csrc/invmgmt.cu) behind the C ABI.
"""
import ctypes as C
from typing import Any, Dict, List, Optional

import numpy as np

from . import _capi
from .mlp import mlp_layers, pack_mlp  # noqa: F401  (re-exported: part of this module's interface)
from .spaces import Box
from .vector import BatchedEnv, _AUTORESET, _torch


class InvManagementParams:
    """Host mirror of InvManagementMasterEnv.__init__ (inventory_management.py:48-141): defaults,
    `env_config` overrides applied with setattr (:83-84), derived arrays (:87-100) and the reference's
    input validation (:144-167, AssertionError with the same messages)."""

    def __init__(self, periods: int = 30, I0: List[int] = (100, 150, 200), p: float = 20,
                 r: List[float] = (15, 10, 7, 5), k: List[float] = (0.10, 0.075, 0.05, 0.025),
                 h: List[float] = (0.15, 0.10, 0.05), c: List[int] = (100, 200, 230), L: List[int] = (1, 5, 10),
                 backlog: bool = True, dist: int = 1, dist_param: Optional[Dict] = None, alpha: float = 0.97,
                 seed_int: int = 0, user_D: Optional[List[int]] = None, env_config: Optional[Dict] = None):
        self.periods = periods
        self.I0 = list(I0)
        self.p = p
        self.r = list(r)
        self.k = list(k)
        self.h = list(h)
        self.c = list(c)
        self.L = list(L)
        self.backlog = backlog
        self.dist = dist
        self.dist_param = dict(dist_param) if dist_param is not None else {"mu": 20}
        self.alpha = alpha
        self.seed_int = seed_int
        self.user_D = user_D if user_D is not None else []
        if env_config:
            for key, value in env_config.items():  # assign_env_config (:15-17)
                setattr(self, key, value)
        self.init_inv = np.array(list(self.I0), dtype=np.int32)
        self.num_periods = self.periods
        self.unit_price = np.append(self.p, self.r[:-1]).astype(np.float32)
        self.unit_cost = np.array(self.r, dtype=np.float32)
        self.demand_cost = np.array(self.k, dtype=np.float32)
        self.holding_cost = np.append(self.h, 0).astype(np.float32)
        self.supply_capacity = np.array(list(self.c), dtype=np.int64)
        self.lead_time = np.array(list(self.L), dtype=np.int64)
        self.discount = self.alpha
        self.user_D = np.array(list(self.user_D), dtype=np.int64)
        self.num_stages = len(self.init_inv) + 1
        m = self.num_stages
        self.lt_max = 0 if m <= 1 else int(self.lead_time.max())
        self._validate_inputs()
        self.pipeline_length = (m - 1) * (self.lt_max + 1)

    def _validate_inputs(self):
        m = self.num_stages
        assert np.all(self.init_inv >= 0), "Initial inventory cannot be negative"
        assert self.num_periods > 0, "Number of periods must be positive"
        assert np.all(self.unit_price >= 0), "Sales prices cannot be negative"
        assert np.all(self.unit_cost >= 0), "Procurement costs cannot be negative"
        assert np.all(self.demand_cost >= 0), "Unfulfilled demand costs cannot be negative"
        assert np.all(self.holding_cost >= 0), "Holding costs cannot be negative"
        assert np.all(self.supply_capacity > 0), "Supply capacities must be positive"
        assert np.all(self.lead_time >= 0), "Lead times cannot be negative"
        assert isinstance(self.backlog, bool), "Backlog parameter must be boolean"
        assert m >= 2, "Minimum number of stages is 2"
        assert len(self.unit_cost) == m, f"Length of r ({len(self.unit_cost)}) != num stages ({m})"
        assert len(self.demand_cost) == m, f"Length of k ({len(self.demand_cost)}) != num stages ({m})"
        assert len(self.holding_cost) == m, f"Length of h ({len(self.holding_cost)}) != num stages ({m})"
        assert len(self.supply_capacity) == m - 1, f"Length of c ({len(self.supply_capacity)}) != num stages - 1 ({m-1})"
        assert len(self.lead_time) == m - 1, f"Length of L ({len(self.lead_time)}) != num stages - 1 ({m-1})"
        assert self.dist in [1, 2, 3, 4, 5], "dist must be one of 1, 2, 3, 4, 5"
        if self.dist == 5:
            assert len(self.user_D) == self.num_periods, "User specified demand length != num periods"
        assert 0 < self.alpha <= 1, "alpha must be in the range (0, 1]"

    # -- spaces (inventory_management.py:111-128; lost-sales lower bound :442-451) ----------------------------
    def spaces(self):
        m = self.num_stages
        action_space = Box(low=np.zeros(m - 1, dtype=np.int64), high=self.supply_capacity.astype(np.int64),
                           shape=(m - 1,), dtype=np.int64)
        cap = self.supply_capacity.sum() * self.num_periods * 2
        low = -np.ones(self.pipeline_length, dtype=np.int64) * cap if self.backlog \
            else np.zeros(self.pipeline_length, dtype=np.int64)
        high = np.ones(self.pipeline_length, dtype=np.int64) * cap
        observation_space = Box(low=low, high=high, shape=(self.pipeline_length,), dtype=np.int64)
        return observation_space, action_space

    # -- flattening for the C ABI ---------------------------------------------------------------------------------
    def dist_struct(self, keep):
        dp = self.dist_param
        if self.dist == 1:
            return _capi.make_dist(_capi.DIST_POISSON, dp["mu"])
        if self.dist == 2:
            return _capi.make_dist(_capi.DIST_BINOMIAL, dp["n"], dp["p"])
        if self.dist == 3:
            return _capi.make_dist(_capi.DIST_RANDINT, dp["low"], dp["high"])
        if self.dist == 4:
            return _capi.make_dist(_capi.DIST_GEOMETRIC, dp["p"])
        return _capi.make_dist(_capi.DIST_USER, user_D=self.user_D, keep=keep)

    def to_c(self, keep, wide_state=False):
        """orgym_invmgmt_config_t; `keep` receives the numpy buffers the struct points into."""
        def arr(a, dt):
            a = np.ascontiguousarray(np.asarray(a, dtype=dt))
            keep.append(a)
            return a
        cfg = _capi.InvConfig()
        cfg.num_stages = self.num_stages
        cfg.periods = int(self.num_periods)
        cfg.backlog = int(bool(self.backlog))
        cfg.wide_state = int(bool(wide_state))
        cfg.init_inv = arr(self.init_inv, np.int64).ctypes.data_as(_capi.c_i64p)
        cfg.capacity = arr(self.supply_capacity, np.int64).ctypes.data_as(_capi.c_i64p)
        cfg.lead_time = arr(self.lead_time, np.int64).ctypes.data_as(_capi.c_i64p)
        # coefficients are float32-rounded in the reference (:89-92) and widened to float64 when they meet int64
        cfg.unit_price = arr(self.unit_price, np.float64).ctypes.data_as(_capi.c_f64p)
        cfg.unit_cost = arr(self.unit_cost, np.float64).ctypes.data_as(_capi.c_f64p)
        cfg.demand_cost = arr(self.demand_cost, np.float64).ctypes.data_as(_capi.c_f64p)
        cfg.holding_cost = arr(self.holding_cost, np.float64).ctypes.data_as(_capi.c_f64p)
        cfg.alpha = float(self.alpha)
        cfg.dist = self.dist_struct(keep)
        return cfg


POLICY_ACTIONS, POLICY_BASE_STOCK, POLICY_RANDOM, POLICY_MLP = 0, 1, 2, 3


class InvManagementMasterEnv(BatchedEnv):
    """`num_envs` instances of the reference env stepped in lock-step on one B200.

    Extra keyword arguments (not in the reference): `num_envs`, `device`, `env_offset` (global id of
    instance 0 -- Philox streams are keyed by global id so results are independent of how instances are
    sharded over GPUs), `autoreset_mode` ('next_step' | 'same_step' | 'disabled'), `wide_state` (int64 state;
    default is a compact int32 state with an on-device range check), `info_level` (0: no per-step info tensors,
    1: demand/sales/unfulfilled/profit tensors).
    """

    _family = "invmgmt"
    metadata = {"render_modes": [], "render_fps": 4}

    def __init__(self, *args, num_envs: int = 1, device="cuda", env_offset: int = 0,
                 autoreset_mode: str = "next_step", wide_state: bool = False, info_level: int = 1,
                 record_history: bool = False, **kwargs):
        torch = _torch()
        self.record_history = bool(record_history)
        if self.record_history:
            if autoreset_mode != "disabled":
                raise ValueError("record_history=True needs autoreset_mode='disabled' (episodes are reset explicitly, "
                                 "like the reference's evaluators do)")
            info_level = max(int(info_level), 1)
        self.params = InvManagementParams(*args, **kwargs)
        P = self.params
        # attributes the reference agents read (benchmark_InvManagementLostSalesEnv.py:142-153)
        for name in ("periods", "num_periods", "I0", "p", "r", "k", "h", "c", "L", "backlog", "dist", "dist_param",
                     "alpha", "num_stages", "lt_max", "lead_time", "supply_capacity", "unit_price", "unit_cost",
                     "demand_cost", "holding_cost", "pipeline_length", "init_inv", "user_D", "discount"):
            setattr(self, name, getattr(P, name))
        self.observation_space_single, self.action_space_single = P.spaces()
        self._setup_batch(num_envs, device, env_offset, autoreset_mode)
        self.wide_state = bool(wide_state)
        self.info_level = int(info_level)
        lib = _capi.lib()
        cfg = P.to_c(self._keep, wide_state)
        _capi.check(lib.orgym_invmgmt_create(C.byref(cfg), self.num_envs, self.device.index, C.byref(self._h)))
        assert lib.orgym_invmgmt_obs_dim(self._h) == P.pipeline_length
        N, m, od = self.num_envs, P.num_stages, P.pipeline_length
        self._alloc_state(lib.orgym_invmgmt_state_bytes(self._h))
        dev = self.device
        self._obs = torch.zeros((N, od), dtype=torch.int64, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float64, device=dev)
        self._terminated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._term_b, self._trunc_b = self._terminated.view(torch.bool), self._truncated.view(torch.bool)  # cached views
        self._info = _capi.InvInfo()
        self._info_t = {}
        if self.info_level >= 1:
            self._info_t = dict(demand_realized=torch.zeros(N, dtype=torch.int64, device=dev),
                                # [N, m] tensors over column-major storage: coalesced stores in the step kernel
                                sales=torch.zeros((m, N), dtype=torch.int64, device=dev).t(),
                                unfulfilled=torch.zeros((m, N), dtype=torch.int64, device=dev).t(),
                                period_profit=torch.zeros(N, dtype=torch.float64, device=dev))
            self._info.info_ld = N
            self._info.demand = self._info_t["demand_realized"].data_ptr()
            self._info.sales = self._info_t["sales"].data_ptr()
            self._info.unfulfilled = self._info_t["unfulfilled"].data_ptr()
            self._info.profit = self._info_t["period_profit"].data_ptr()
        if autoreset_mode == "same_step":
            self._final_obs = torch.zeros((N, od), dtype=torch.int64, device=dev)
            self._info.final_obs = self._final_obs.data_ptr()
        self._has_reset = False

    # -- gymnasium API --------------------------------------------------------------------------------------------
    def reset(self, *, seed=None, options: Optional[Dict] = None):
        """reset (inventory_management.py:186-222).  options={'reset_mask': bool[N]} resets a subset."""
        reseed, base = self._resolve_seed(seed)
        mask = None
        if options and options.get("reset_mask") is not None:
            mask = self._to_dev(options["reset_mask"], _torch().uint8, (self.num_envs,))
        _capi.check(_capi.lib().orgym_invmgmt_reset(self._h, self._ptr(self._state), reseed, C.c_uint64(base),
                                                    self.env_offset, self._ptr(mask), self._ptr(self._obs),
                                                    self._stream()))
        self._has_reset = True
        if self.record_history:
            if mask is not None:
                raise NotImplementedError("record_history keeps all instances in lock-step: reset without a mask")
            self._alloc_history()
        return self._obs, {}

    # -- full-history buffers (SURVEY §8f rank 4): the arrays the reference keeps per episode (:203-211), batched ----
    def _alloc_history(self):
        torch = _torch()
        P = self.params
        N, T, n, m, dev = self.num_envs, int(P.num_periods), P.num_stages - 1, P.num_stages, self.device
        z = lambda *shape, dt=torch.int64: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.I, self.B = z(N, T + 1, n), z(N, T + 1, m)
        self.R, self.S, self.LS = z(N, T, n), z(N, T, m), z(N, T, m)
        self.D, self.action_log = z(N, T), z(N, T, n)
        self.P = z(N, T, dt=torch.float64)   # discounted profit (the reference stores it as float32, :210/:323)
        self.I[:, 0] = torch.as_tensor(np.asarray(P.init_inv, np.int64), device=dev)
        self._t_host = 0

    def _record(self, a_req, reward, info):
        t = self._t_host
        if t >= int(self.params.num_periods):
            return
        I, B, _ = self.export_state()
        self.I[:, t + 1], self.B[:, t + 1] = I, B
        self.D[:, t], self.S[:, t], self.P[:, t] = info["demand_realized"], info["sales"], reward
        self.R[:, t] = info["sales"][:, 1:]
        if not self.params.backlog:
            self.LS[:, t] = info["unfulfilled"]
        self.action_log[:, t] = a_req
        self._t_host = t + 1

    def step(self, actions, demand=None):
        """step (inventory_management.py:224-352) for all instances.

        actions: [N, m-1] int64 (or float64: truncated toward zero after max(a, 0) like the reference, :250).
        demand:  optional int64[N] replayed demand for this period (parity / trace-driven runs).
        Returns (obs int64[N,obs_dim], reward float64[N], terminated bool[N], truncated bool[N], info);
        the tensors alias the env's buffers and are overwritten by the next call.
        """
        torch = _torch()
        if not self._has_reset:
            raise RuntimeError("call reset() before step()")
        n = self.params.num_stages - 1
        if isinstance(actions, torch.Tensor) and actions.dtype in (torch.float64, torch.float32, torch.float16,
                                                                    torch.bfloat16):
            a = self._to_dev(actions, torch.float64, (self.num_envs, n))
            is_f64 = 1
        elif not isinstance(actions, torch.Tensor) and np.asarray(actions).dtype.kind == "f":
            a = self._to_dev(actions, torch.float64, (self.num_envs, n))
            is_f64 = 1
        else:
            a = self._to_dev(actions, torch.int64, (self.num_envs, n))
            is_f64 = 0
        d = self._to_dev(demand, torch.int64, (self.num_envs,)) if demand is not None else None
        _capi.check(_capi.lib().orgym_invmgmt_step(
            self._h, self._ptr(self._state), self._ptr(a), is_f64, self._ptr(d), _AUTORESET[self.autoreset_mode],
            self._ptr(self._obs), self._ptr(self._reward), self._ptr(self._terminated), self._ptr(self._truncated),
            C.byref(self._info), self._stream()))
        info = dict(self._info_t)
        if self.autoreset_mode == "same_step":
            info["final_obs"] = self._final_obs
        if self.record_history:
            self._record(torch.clamp(a, min=0).to(torch.int64), self._reward, info)  # requested order (:250)
        return self._obs, self._reward, self._term_b, self._trunc_b, info

    @property
    def rollout_specialised(self):
        """True when the most recent `rollout` ran a kernel generated for this configuration and policy (on-device
        base-stock with integer levels or random policy, sampled demand, no trajectory outputs)."""
        return bool(_capi.lib().orgym_invmgmt_is_specialised(self._h))

    def _policy_struct(self, policy, safety_factor=1.0, mu=None, keep=None):
        rin = _capi.InvRolloutIn()
        if not isinstance(policy, str):
            P = self.params
            mlp, tensors = pack_mlp(policy, P.pipeline_length, P.num_stages - 1, self.device)
            if keep is not None:
                keep += [mlp, tensors]
            rin.policy = POLICY_MLP
            rin.mlp = C.pointer(mlp)
        elif policy == "base_stock":
            rin.policy = POLICY_BASE_STOCK
            rin.param[0] = float(safety_factor)
            rin.param[1] = float(self.params.dist_param.get("mu", 10) if mu is None else mu)
        elif policy == "random":
            rin.policy = POLICY_RANDOM
        elif policy == "actions":
            rin.policy = POLICY_ACTIONS
        else:
            raise ValueError(f"unknown policy {policy!r}")
        return rin

    def specialise(self, policy="base_stock", *, safety_factor=1.0, mu=None):
        """Build the rollout kernel specialised for this configuration and policy now (NVRTC, about a second; cached on
        disk) instead of inside the first rollout.  Raises OrgymError with the reason (NVRTC log included) when the
        configuration or policy is outside the specialiser's range or the compile fails."""
        keep = []
        rin = self._policy_struct(policy, safety_factor, mu, keep)
        _capi.check(_capi.lib().orgym_invmgmt_specialise(self._h, C.byref(rin)))
        return True

    # -- batched views of the attributes the reference agents read ---------------------------------------------------
    def export_state(self):
        """(I int64[N,m-1], B int64[N,m], period int32[N]) -- current on-hand inventory, backlog, period."""
        torch = _torch()
        N, m = self.num_envs, self.params.num_stages
        I = torch.empty((N, m - 1), dtype=torch.int64, device=self.device)
        B = torch.empty((N, m), dtype=torch.int64, device=self.device)
        t = torch.empty(N, dtype=torch.int32, device=self.device)
        _capi.check(_capi.lib().orgym_invmgmt_export_state(self._h, self._ptr(self._state), self._ptr(I),
                                                           self._ptr(B), self._ptr(t), self._stream()))
        return I, B, t

    @property
    def period(self):
        return self.export_state()[2]

    # -- fused rollout ------------------------------------------------------------------------------------------------
    def rollout(self, policy="base_stock", *, seed=None, episode=0, safety_factor=1.0, mu=None, actions=None,
                demand=None, time_major=False, want=("ep_return", "stats", "summary"), buffer_set=0):
        """Fused reset + `periods` steps with state held on chip (K4).

        policy: 'base_stock' (benchmark_InvManagementBacklogEnv.py:142-198), 'random' (a_i ~ U{0..c_i}),
                'actions' with `actions` int64 [N,T,m-1] ([T,N,m-1] if time_major), or a trained actor network -- a
                torch.nn.Sequential (Linear, Tanh|ReLU, ..., Linear) or an SB3 ActorCriticPolicy -- evaluated on the
                device every period on the observation step() would return (float32, SB3's deterministic predict:
                mean clipped to [0, c], then truncated like a float action; include/orgym_b200.h states the numerics).
                Its weights are read at every call.
        demand: optional int64 [N,T] ([T,N] if time_major) replayed demand; default = on-device Philox sampling.
        Returns a dict of device tensors: ep_return f64[N], stats i64[N,4] (sum sales[0], sum demand,
        sum unfulfilled[0], sum_t sum_i max(0,I_i)), summary f64[8], and on request reward_traj f64[N,T],
        final_I, final_B, stats32 (the statistics as int32), action_traj i64[N,T,m-1] (the requested orders, the
        reference's action_log).  The result tensors are owned by the env and reused by
        the next rollout that uses the same `buffer_set`.
        """
        torch = _torch()
        P = self.params
        N, T, n, m = self.num_envs, int(P.num_periods), P.num_stages - 1, P.num_stages
        keep = []
        rin = self._policy_struct(policy, safety_factor, mu, keep)
        if "_ring_scratch" not in self.__dict__:      # caller-owned scratch for very long lead-time rings (rare)
            nb = int(_capi.lib().orgym_invmgmt_rollout_scratch_bytes(self._h))
            self._ring_scratch = torch.empty(nb, dtype=torch.uint8, device=self.device) if nb > 0 else None
        if self._ring_scratch is not None:
            rin.scratch = self._ring_scratch.data_ptr()
        if policy == "actions":
            shape = (T, N, n) if time_major else (N, T, n)
            a = self._to_dev(actions, torch.int64, shape)
            keep.append(a)
            rin.actions = a.data_ptr()
            rin.act_stride_env, rin.act_stride_t = (n, N * n) if time_major else (T * n, n)
        if demand is not None:
            d = self._to_dev(demand, torch.int64, (T, N) if time_major else (N, T))
            keep.append(d)
            rin.demand = d.data_ptr()
            rin.dem_stride_env, rin.dem_stride_t = (1, N) if time_major else (T, 1)
        out = {}
        rout = _capi.InvRolloutOut()
        dev = self.device
        shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.int64),
                      reward_traj=((N, T), torch.float64), final_I=((N, n), torch.int64),
                      final_B=((N, m), torch.int64), summary=((8,), torch.float64), stats32=((N, 4), torch.int32),
                      action_traj=((N, T, n), torch.int64))
        cache = self.__dict__.setdefault("_rollout_buf", {}).setdefault(int(buffer_set), {})
        for name in want:
            shp, dt = shapes[name]
            if name not in cache:
                cache[name] = torch.zeros(shp, dtype=dt, device=dev)
            out[name] = cache[name]
            setattr(rout, name, out[name].data_ptr())
        if seed is not None:
            self._resolve_seed(seed)
        elif not self._seeded:
            self._resolve_seed(None)
        _capi.check(_capi.lib().orgym_invmgmt_rollout(self._h, C.c_uint64(self._seed), self.env_offset,
                                                      C.c_uint32(int(episode)), C.byref(rin), C.byref(rout),
                                                      self._stream()))
        return out


class InvManagementBacklogEnv(InvManagementMasterEnv):
    """Backlogging variant: the `backlog` kwarg is forced True (inventory_management.py:429-434)."""

    def __init__(self, *args, **kwargs):
        kwargs["backlog"] = True
        super().__init__(*args, **kwargs)


class InvManagementLostSalesEnv(InvManagementMasterEnv):
    """Lost-sales variant: `backlog` kwarg forced False and observation lower bound 0 (:436-451)."""

    def __init__(self, *args, **kwargs):
        kwargs["backlog"] = False
        super().__init__(*args, **kwargs)
        P = self.params
        cap = P.supply_capacity.sum() * P.num_periods * 2
        self.observation_space_single = Box(low=np.zeros(P.pipeline_length, dtype=np.int64),
                                            high=np.ones(P.pipeline_length, dtype=np.int64) * cap,
                                            shape=(P.pipeline_length,), dtype=np.int64)
        self.single_observation_space = self.observation_space_single
