"""GPU tests of the step API across episode boundaries, in all three env families and every kernel path.

Results are a pure function of (seed, global env id, episode, period), whether they come from the step API or from the
fused rollout (DESIGN §3).  Episode 0 is covered by the parity tests; here every instance is stepped through several
episodes -- reached by `next_step` / `same_step` autoreset, by reset() without a seed and by a masked reset in the middle
of an episode -- and its episode k is compared bit for bit with `rollout(episode=k)` on the same action schedule, and on a
sample of instances (first, last, both sides of a 128-instance tile boundary) with the CPU oracle fed the demand the
device drew.  Every action is non-zero, so at each boundary the lead-time rings and observation windows hold orders that
an in-kernel reset has to clear; the tests assert that precondition on the terminal observations."""
import os

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from helpers import set_net_kernel_mode

pytestmark = pytest.mark.gpu
STRESS = max(1, int(os.environ.get("ORGYM_STRESS", "1")))
EPISODES = 2 + STRESS
REACH = ["next_step", "same_step", "reset", "masked"]
NET_MODES = ["specialised", "stream_jit", "stream_jit_twopass", "stream_jit_fused_obs", "generic"]


def _torch():
    import torch
    return torch


def _oracle():
    from oracle import oracle
    return oracle


# ---- the three families behind one interface ------------------------------------------------------------------------
class _Serial:
    """Serial multi-echelon env; actions int64 [N, T, n] with every order in [1, c_i]."""
    dem_key = "demand_realized"
    want = ("reward_traj", "stats", "final_I", "final_B")

    def __init__(self, N, backlog=True, wide=False, seed=0, **cfg):
        self.N, self.seed = N, seed
        self.cls = pkg.InvManagementBacklogEnv if backlog else pkg.InvManagementLostSalesEnv
        self.kw = dict(wide_state=wide, **cfg)

    def make(self, mode):
        env = self.cls(num_envs=self.N, device="cuda:0", autoreset_mode=mode, **self.kw)
        if not hasattr(self, "sched"):
            self.T, self.n, self.od = env.num_periods, env.num_stages - 1, env.pipeline_length
            self.obs_dtype, self.dem_dtype, self.dem_shape = np.int64, np.int64, ()
            self.rings = [[c] for c in range(self.n, self.od)]     # the window of the last lt_max requests
            rng = np.random.default_rng(self.seed)
            self.sched = rng.integers(1, env.supply_capacity + 1, size=(self.N, self.T, self.n)).astype(np.int64)
        return env

    def action(self, per):
        return _torch().from_numpy(self.sched[np.arange(self.N), per]).cuda()

    def reset_options(self):
        return None

    def export(self, env):
        I, B, per = env.export_state()
        return dict(final_I=I.cpu().numpy(), final_B=B.cpu().numpy()), per.cpu().numpy()

    def params(self, env):
        return None

    def check_reset_obs(self, env, obs, rows, ref):
        assert np.array_equal(obs[rows], np.broadcast_to(ref, obs[rows].shape))

    def rollout(self, env, seed, k):
        out = env.rollout("actions", actions=self.sched, seed=seed, episode=k, want=self.want)
        return {name: t.cpu().numpy() for name, t in out.items()}

    def check_terminal(self, out, b, rows):
        assert np.array_equal(out["final_I"][rows], b["term"][rows][:, :self.n])    # observation = [I, window]

    def oracle(self, env, e, b):
        o = _oracle().invmgmt_episode(env.params, actions=self.sched[e].astype(np.float64), demand=b["dem"][e])
        return o["reward"], o["obs"]


class _Newsvendor:
    """Newsvendor; actions float32 [N, T] in [1, 300); optionally every instance pinned to its own parameters."""
    dem_key = "demand"
    want = ("reward_traj", "stats", "final_obs")

    def __init__(self, N, lead_time, pinned, T=12, seed=0):
        self.N, self.L, self.T, self.pinned, self.seed = N, lead_time, T, pinned, seed

    def make(self, mode):
        env = pkg.NewsvendorEnv(num_envs=self.N, device="cuda:0", autoreset_mode=mode, lead_time=self.L,
                                step_limit=self.T)
        if not hasattr(self, "sched"):
            self.od, self.obs_dtype, self.dem_dtype, self.dem_shape = env.obs_dim, np.float32, np.int64, ()
            self.rings = [[c] for c in range(5, self.od)]           # the order pipeline
            rng = np.random.default_rng(self.seed)
            self.sched = rng.uniform(1, 300, size=(self.N, self.T)).astype(np.float32)
            price = rng.uniform(20, 100, self.N)
            self.fixed = np.stack([price, rng.uniform(0.2, 0.9, self.N) * price, rng.uniform(0.1, 5, self.N),
                                   rng.uniform(0.1, 10, self.N), rng.uniform(10, 200, self.N)], axis=1)
        return env

    def action(self, per):
        return _torch().from_numpy(self.sched[np.arange(self.N), per]).cuda()

    def reset_options(self):
        return {"fixed_params": self.fixed} if self.pinned else None

    def export(self, env):
        return {}, None                                             # no period / state export in this family

    def params(self, env):
        return env.export_params().cpu().numpy()

    def check_reset_obs(self, env, obs, rows, ref):
        par = self.params(env)
        assert np.array_equal(obs[rows, :5], par[rows].astype(np.float32))
        assert (obs[rows, 5:] == 0).all()

    def rollout(self, env, seed, k):
        out = env.rollout("actions", actions=self.sched, seed=seed, episode=k, want=self.want,
                          fixed_params=self.fixed if self.pinned else None)
        return {name: t.cpu().numpy() for name, t in out.items()}

    def check_terminal(self, out, b, rows):
        assert np.array_equal(out["final_obs"][rows], b["term"][rows])
        # the parameters the step API used in episode k are the ones the rollout draws (or pins) for episode k
        assert np.array_equal(out["final_obs"][rows, :5], b["params"][rows].astype(np.float32))
        if self.pinned:
            assert np.array_equal(b["params"][rows], self.fixed[rows])

    def oracle(self, env, e, b):
        o = _oracle().newsvendor_episode(env.params, actions=self.sched[e], demand=b["dem"][e], fixed=b["params"][e])
        return o["reward"], o["obs"]


class _Network:
    """Network env; actions float32 [N, T, E] = U(lo, hi) * action bound."""
    dem_key = "demand"
    want = ("reward_traj", "stats", "final_X", "final_Y", "final_U")

    def __init__(self, N, graph=None, backlog=True, T=None, order=(0.02, 0.1), seed=0):
        self.N, self.graph, self.backlog, self.T, self.order, self.seed = N, graph, backlog, T, order, seed

    def make(self, mode):
        kw = dict(num_envs=self.N, device="cuda:0", autoreset_mode=mode, backlog=self.backlog)
        if self.graph is not None:
            kw["graph"] = self.graph
        if self.T is None:     # one period more than the longest lead time: every ring slot holds an order at the end
            self.T = pkg.NetInvMgmtParams(**{k: v for k, v in kw.items() if k in ("graph", "backlog")}).lt_max + 1
        env = pkg.NetInvMgmtMasterEnv(num_periods=self.T, **kw)
        if not hasattr(self, "sched"):
            self.E, self.M, self.J = len(env.reorder_links), len(env.retail_links), len(env.main_nodes)
            self.od, self.obs_dtype, self.dem_dtype, self.dem_shape = env.obs_dim, np.float32, np.float64, (self.M,)
            # the pipeline window of every lead-time link; some of its slots can be empty in every instance (an upstream
            # node whose replenishment has not arrived yet ships nothing), so the precondition is one order per window
            self.rings, c = [], self.M + self.J
            for link in env.reorder_links:
                L = env.lead_times[link]
                if L > 0:
                    self.rings.append(list(range(c, c + L)))
                    c += L
            assert c == self.od
            rng = np.random.default_rng(self.seed)
            self.sched = (rng.uniform(*self.order, size=(self.N, self.T, self.E)) *
                          env.single_action_space.high).astype(np.float32)
        return env

    def action(self, per):
        return _torch().from_numpy(self.sched[np.arange(self.N), per]).cuda()

    def reset_options(self):
        return None

    def export(self, env):
        X, Y, U, per = env.export_state()
        return dict(final_X=X.cpu().numpy(), final_Y=Y.cpu().numpy(), final_U=U.cpu().numpy()), per.cpu().numpy()

    def params(self, env):
        return None

    def check_reset_obs(self, env, obs, rows, ref):
        assert np.array_equal(obs[rows], np.broadcast_to(ref, obs[rows].shape))

    def rollout(self, env, seed, k):
        out = env.rollout("actions", actions=self.sched, seed=seed, episode=k, want=self.want)
        return {name: t.cpu().numpy() for name, t in out.items()}

    def check_terminal(self, out, b, rows):
        pass                                                        # the state comparison covers X / Y / U

    def oracle(self, env, e, b):
        o = _oracle().netinv_episode(env.params, actions=self.sched[e], demand=b["dem"][e])
        return o["reward"], o["obs"]


# ---- per-instance bookkeeping of a stepped batch ---------------------------------------------------------------------
def _picks(N):
    """First, last, and both sides of the first 128-instance tile boundary."""
    return sorted({e for e in (0, 1, 2, 126, 127, 128, 129, N - 2, N - 1) if 0 <= e < N})


class _Run:
    """Steps an env and mirrors, per instance, the episode and period the kernels are expected to be in; records per
    episode the rewards, the demand the device drew, the terminal observation and state, the newsvendor parameters and
    the whole observation sequence of the sampled instances."""

    def __init__(self, fam, env, mode, seed):
        self.f, self.env, self.mode, self.seed = fam, env, mode, seed
        N = fam.N
        self.ep = np.zeros(N, np.int64)
        self.per = np.zeros(N, np.int64)
        self.picks = _picks(N)
        self.rec = {}
        self.obs = None
        self.ref0 = None     # reset observation of the serial / network envs (the same in every episode)

    def _book(self, k):
        f = self.f
        if k not in self.rec:
            self.rec[k] = dict(rew=np.full((f.N, f.T), np.nan), dem=np.zeros((f.N, f.T) + f.dem_shape, f.dem_dtype),
                               term=np.zeros((f.N, f.od), f.obs_dtype), done=np.zeros(f.N, bool), state={},
                               params=np.full((f.N, 5), np.nan), hist=np.zeros((len(self.picks), f.T + 1, f.od), f.obs_dtype))
        return self.rec[k]

    def _after(self, rows_started, obs):
        par = self.f.params(self.env)
        if par is not None:
            for k in np.unique(self.ep):
                self._book(k)["params"][self.ep == k] = par[self.ep == k]
        if rows_started is not None and rows_started.any():
            self.f.check_reset_obs(self.env, obs, rows_started, self.ref0)
            for i, e in enumerate(self.picks):
                if rows_started[e]:
                    self._book(self.ep[e])["hist"][i, 0] = obs[e]
        state, per = self.f.export(self.env)
        if per is not None:
            assert np.array_equal(per, self.per)
        self.obs = obs
        return state

    def reset(self, seed=None, mask=None):
        opts = dict(self.f.reset_options() or {})
        if mask is not None:
            opts["reset_mask"] = mask
        prev = self.obs
        obs = self.env.reset(seed=seed, options=opts or None)[0].cpu().numpy()
        if self.ref0 is None:
            self.ref0 = obs[0].copy()
        rows = np.ones(self.f.N, bool) if mask is None else np.asarray(mask, bool)
        if mask is not None:
            assert np.array_equal(obs[~rows], prev[~rows])        # the other instances keep their observation
        self.ep[rows] = 0 if seed is not None else self.ep[rows] + 1
        self.per[rows] = 0
        self._after(rows, obs)

    def step(self):
        f, T = self.f, self.f.T
        obs, r, term, trunc, info = self.env.step(f.action(np.minimum(self.per, T - 1)))
        obs, r, term, trunc = (x.cpu().numpy() for x in (obs, r, term, trunc))
        dem = info[f.dem_key].cpu().numpy()
        fin = info["final_obs"].cpu().numpy() if self.mode == "same_step" else None
        assert not term.any()
        again = self.per >= T                     # the extra step of next_step autoreset
        if again.any():
            assert self.mode == "next_step"
            assert (r[again] == 0).all() and not trunc[again].any()
            self.ep[again] += 1
            self.per[again] = 0
        run = ~again
        last = run & (self.per == T - 1)
        assert np.array_equal(trunc[run], last[run])
        for k in np.unique(self.ep[run]):
            rows = run & (self.ep == k)
            b = self._book(k)
            b["rew"][rows, self.per[rows]] = r[rows]
            b["dem"][rows, self.per[rows]] = dem[rows]
        term_obs = fin if fin is not None else obs
        for i, e in enumerate(self.picks):
            if run[e]:
                self._book(self.ep[e])["hist"][i, self.per[e] + 1] = term_obs[e] if last[e] else obs[e]
        finished = {k: last & (self.ep == k) for k in np.unique(self.ep[last])}
        for k, rows in finished.items():
            b = self._book(k)
            b["term"][rows] = term_obs[rows]
            b["done"][rows] = True
        self.per[run] += 1
        started = again.copy()
        if self.mode == "same_step":              # the truncating step returned episode k+1's first observation
            self.ep[last] += 1
            self.per[last] = 0
            started |= last
        state = self._after(started, obs)
        if fin is None:                           # terminal state of the instances that just finished
            for k, rows in finished.items():
                for name, v in state.items():
                    self._book(k)["state"].setdefault(name, np.zeros_like(v))[rows] = v[rows]
        return obs, r, trunc

    def verify(self):
        """Episode k of every instance that completed it == rollout(episode=k) on its subset == the oracle on the
        sampled instances.  Returns {episode: number of instances compared}."""
        f, counts = self.f, {}
        for k in sorted(self.rec):
            b = self.rec[k]
            rows = b["done"]
            if not rows.any():
                continue
            counts[k] = int(rows.sum())
            # precondition: every ring / window holds an order in some instance at the boundary
            nz = (b["term"][rows] != 0).any(axis=0)
            assert all(nz[g].any() for g in f.rings), f"episode {k}: a ring is empty at the boundary"
            out = f.rollout(self.env, self.seed, k)
            assert not np.isnan(b["rew"][rows]).any()
            assert np.array_equal(out["reward_traj"][rows], b["rew"][rows]), f"episode {k}: rewards"
            dsum = b["dem"][rows].reshape(counts[k], -1).sum(axis=1)
            assert np.array_equal(out["stats"][rows, 1], dsum), f"episode {k}: demand"
            for name, v in b["state"].items():
                assert np.array_equal(out[name][rows], v[rows]), f"episode {k}: {name}"
            f.check_terminal(out, b, rows)
            for i, e in enumerate(self.picks):
                if rows[e]:
                    rew, obs = f.oracle(self.env, e, b)
                    assert np.array_equal(rew, b["rew"][e]), f"episode {k}, instance {e}: rewards vs oracle"
                    assert np.array_equal(obs, b["hist"][i]), f"episode {k}, instance {e}: observations vs oracle"
        return counts


def _drive(fam, reach, seed):
    """Reach episodes 1, 2, ... in one of four ways and compare every completed episode."""
    K, N = EPISODES, fam.N
    mode = {"next_step": "next_step", "same_step": "same_step", "reset": "disabled", "masked": "next_step"}[reach]
    env = fam.make(mode)
    T = fam.T
    run = _Run(fam, env, mode, seed)
    run.reset(seed=seed)
    if reach == "next_step":
        for _ in range(K * (T + 1)):
            run.step()
    elif reach == "same_step":
        for _ in range(K * T):
            run.step()
    elif reach == "reset":
        for k in range(K):
            for _ in range(T):
                run.step()
            if k + 1 < K:
                run.reset()                       # no seed: the next episode of every instance
    else:
        mask = np.arange(N) % 3 == 0
        for _ in range(max(1, T // 2)):
            run.step()
        run.reset(mask=mask)                      # one tile now holds instances of two episodes and two periods
        for _ in range(2 * (T + 1) + T - max(1, T // 2)):     # ends on the last period of episode 2 of the others
            run.step()
    counts = run.verify()
    env.close()
    if reach == "masked":
        assert counts == {0: int((~mask).sum()), 1: N, 2: N}, counts
    else:
        assert counts == {k: N for k in range(K)}, counts


# ---- 1/2. the episode identity, per family and kernel form -----------------------------------------------------------
SERIAL_CFG = dict(periods=12)      # longer than the largest lead time (10) of the default chain


def _serial_max(N=130):
    """test_invmgmt_maximum_sizes' 16-stage chain with lead times up to 64: its 1040-entry observation rows do not fit a
    shared-memory tile, so the step kernel writes them directly into the caller's rows."""
    rng = np.random.default_rng(77)
    n = 16
    L = rng.integers(0, 65, n)
    L[0], L[1], L[2] = 64, 0, 63
    return dict(periods=66, I0=rng.integers(0, 200, n).tolist(), p=31.5,
                r=np.sort(rng.uniform(0.5, 30, n + 1))[::-1].round(3).tolist(), k=rng.uniform(0, 1, n + 1).round(3).tolist(),
                h=rng.uniform(0, 0.5, n).round(3).tolist(), c=rng.integers(1, 300, n).tolist(), L=L.tolist(),
                dist_param={"mu": 33.0}, alpha=0.97)


@pytest.mark.parametrize("reach", REACH)
@pytest.mark.parametrize("wide", [False, True], ids=["int32state", "int64state"])
@pytest.mark.parametrize("backlog", [True, False], ids=["backlog", "lost"])
def test_serial_episodes_match_rollout_and_oracle(backlog, wide, reach):
    _drive(_Serial(300, backlog=backlog, wide=wide, seed=11, **SERIAL_CFG), reach, seed=700)


@pytest.mark.parametrize("reach", REACH)
@pytest.mark.parametrize("backlog,wide", [(True, False), (False, True)], ids=["backlog-int32state", "lost-int64state"])
def test_serial_direct_observation_rows_episodes(backlog, wide, reach):
    _drive(_Serial(130, backlog=backlog, wide=wide, seed=12, **_serial_max()), reach, seed=710)


@pytest.mark.parametrize("reach", REACH)
@pytest.mark.parametrize("pinned", [False, True], ids=["drawn", "pinned"])
@pytest.mark.parametrize("lead_time", [0, 5])
def test_newsvendor_episodes_match_rollout_and_oracle(lead_time, pinned, reach):
    _drive(_Newsvendor(300, lead_time, pinned, seed=13), reach, seed=720)


@pytest.mark.parametrize("reach", REACH)
@pytest.mark.parametrize("kernel", NET_MODES)
def test_network_episodes_match_rollout_and_oracle(kernel, reach, monkeypatch):
    set_net_kernel_mode(monkeypatch, kernel)
    _drive(_Network(300, seed=14), reach, seed=730)


def _net64():
    """Lost sales on synthetic_graph(64) (longest lead time 12).  Small orders and 16 periods: with larger orders some
    distributors run dry for longer than the lead time of the links they supply, and those rings stay empty."""
    return _Network(200, graph=pkg.synthetic_graph(64), backlog=False, T=16, order=(0.002, 0.02), seed=15)


def _default_plan(monkeypatch):
    for var in ("ORGYM_NET_JIT", "ORGYM_NET_JIT_STREAM", "ORGYM_NET_OBS_TMA", "ORGYM_NET_JIT_ONEPASS"):
        monkeypatch.delenv(var, raising=False)


@pytest.mark.parametrize("reach", REACH)
@pytest.mark.parametrize("kernel", ["default_plan", "generic"])
def test_network_64_node_episodes_match_rollout_and_oracle(kernel, reach, monkeypatch):
    """Config 5's graph: its default plan is the single-pass streaming step kernel + net_obs_kernel reading the float32
    ring copy, which every in-kernel reset has to clear too.  The masked case makes net_obs_kernel take its
    per-instance path."""
    if kernel == "generic":
        set_net_kernel_mode(monkeypatch, "generic")
    else:
        _default_plan(monkeypatch)
    _drive(_net64(), reach, seed=740)


# ---- speculative and non-speculative serial step paths ---------------------------------------------------------------
@pytest.mark.parametrize("mode", ["next_step", "same_step", "disabled"])
@pytest.mark.parametrize("cfg", ["default", "direct_rows"])
def test_serial_speculative_step_equals_reloading_step(cfg, mode):
    """The serial step kernel loads the rings at the period the host expects the whole batch to be in, and reloads for
    an instance whose period differs.  A reset whose mask selects no instance keeps every state but makes the period
    unknown to the host: that env takes the non-speculative path and must return exactly what its untouched twin
    returns, through two boundaries (past the end, for `disabled`)."""
    torch = _torch()
    N, kw = (131, dict(SERIAL_CFG)) if cfg == "default" else (130, _serial_max())
    fam = _Serial(N, seed=16, **kw)
    a, b = fam.make(mode), fam.make(mode)
    T = fam.T
    for env in (a, b):
        env.reset(seed=750)
    per = np.zeros(N, np.int64)

    def step_both():
        act = fam.action(np.minimum(per, T - 1))
        ra, rb = a.step(act), b.step(act)
        for x, y in zip(ra[:4], rb[:4]):
            assert torch.equal(x, y)
        assert ra[4].keys() == rb[4].keys()
        for name in ra[4]:
            assert torch.equal(ra[4][name], rb[4][name]), name
        return ra

    for _ in range(3):
        step_both()
        per += 1
    b.reset(options={"reset_mask": np.zeros(N, bool)})
    assert torch.equal(a.export_state()[2], b.export_state()[2])
    steps = {"next_step": 2 * (T + 1) + 1, "same_step": 2 * T + 1, "disabled": T - 3 + 1}[mode]
    for _ in range(steps):
        step_both()
        per = (per + 1) % (T + 1) if mode == "next_step" else ((per + 1) % T if mode == "same_step" else per + 1)
    for x, y in zip(a.export_state(), b.export_state()):
        assert torch.equal(x, y)
    if mode == "disabled":
        for env in (a, b):
            with pytest.raises(IndexError):
                env.check_errors()
    assert a.errors() == 0 and b.errors() == 0
    a.close()
    b.close()


# ---- disabled autoreset: one step past the end ---------------------------------------------------------------------------
def _past_end(fam, seed):
    """Step T periods, then once more: ORGYM_ERR_STEP_PAST_END (IndexError), previous observation, reward 0, truncated.
    A masked reset of every third instance restarts those in episode 1 while the others stay past the end; a full
    reset with the seed reproduces episode 0."""
    torch = _torch()
    from or_gym_inventory_b200 import _capi
    N = fam.N
    env = fam.make("disabled")
    T = fam.T
    env.reset(seed=seed)
    for t in range(T):
        obs, r, term, trunc, _ = env.step(fam.action(np.full(N, t)))
    assert trunc.all()
    assert env.errors() == 0
    prev = obs.clone()
    obs, r, term, trunc, _ = env.step(fam.action(np.zeros(N, np.int64)))
    assert torch.equal(obs, prev) and (r == 0).all() and trunc.all() and not term.any()
    assert env.errors(clear=False) & _capi.ERR_STEP_PAST_END
    with pytest.raises(IndexError):
        env.check_errors()
    assert env.errors() == 0
    # masked reset after the end: the reset instances start episode 1, the others are still past the end
    mask = np.arange(N) % 3 == 0
    env.reset(options=dict(fam.reset_options() or {}, reset_mask=mask))
    obs, r, term, trunc, _ = env.step(fam.action(np.zeros(N, np.int64)))
    r1 = fam.rollout(env, seed, 1)["reward_traj"][:, 0]
    obs_h, r_h, trunc_h = obs.cpu().numpy(), r.cpu().numpy(), trunc.cpu().numpy()
    assert np.array_equal(r_h[mask], r1[mask]) and not trunc_h[mask].any()
    assert np.array_equal(obs_h[~mask], prev.cpu().numpy()[~mask]) and (r_h[~mask] == 0).all() and trunc_h[~mask].all()
    with pytest.raises(IndexError):
        env.check_errors()
    # a full reset recovers: episode 0 again, without errors
    env.reset(seed=seed, options=fam.reset_options())
    rew = np.zeros((N, T))
    for t in range(T):
        rew[:, t] = env.step(fam.action(np.full(N, t)))[1].cpu().numpy()
    assert np.array_equal(rew, fam.rollout(env, seed, 0)["reward_traj"])
    assert env.errors() == 0
    env.close()


@pytest.mark.parametrize("cfg", ["default", "direct_rows"])
def test_serial_disabled_step_past_end(cfg):
    fam = _Serial(131, seed=17, **SERIAL_CFG) if cfg == "default" else _Serial(130, seed=17, **_serial_max())
    _past_end(fam, seed=760)


@pytest.mark.parametrize("pinned", [False, True], ids=["drawn", "pinned"])
@pytest.mark.parametrize("lead_time", [0, 5])
def test_newsvendor_disabled_step_past_end(lead_time, pinned):
    _past_end(_Newsvendor(300, lead_time, pinned, seed=18), seed=770)


@pytest.mark.parametrize("kernel", NET_MODES)
def test_network_disabled_step_past_end(kernel, monkeypatch):
    set_net_kernel_mode(monkeypatch, kernel)
    _past_end(_Network(300, seed=19), seed=780)


def test_network_64_node_disabled_step_past_end(monkeypatch):
    _default_plan(monkeypatch)
    _past_end(_net64(), seed=790)
