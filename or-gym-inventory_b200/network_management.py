"""Batched network inventory env -- drop-in for the reference's `network_management.py`
(NetInvMgmtMasterEnv / NetInvMgmtBacklogEnv / NetInvMgmtLostSalesEnv) and, through
`default_graph="custom"`, for `network_management_custom.py`.

Same constructor keywords (network_management.py:55-63), graph attribute conventions (:108-144), node/link
classification (:146-195), validation (:197-238) and spaces (:270-298).  The networkx graph is flattened here
into the CSR arrays of `orgym_netinv_config_t`; the dynamics run in csrc/netinv.cu.
"""
import ctypes as C
from typing import Any, Dict, List, Optional, Tuple

import numpy as np

from . import _capi
from .mlp import pack_mlp
from .spaces import Box
from .vector import BatchedEnv, _AUTORESET, _torch

try:
    import networkx as nx
except Exception:  # noqa: BLE001  pragma: no cover
    nx = None


POLICY_MLP = 2


def _np_poisson_marker(**p):  # stands in for `lambda **p: self.np_random.poisson(**p)` of the default graph
    raise RuntimeError("demand is sampled on the device; this callable only marks the link as Poisson")


def default_graph(kind="default"):
    """The reference's default topologies: network_management.py:110-139 ('default') and
    network_management_custom.py:113-139 ('custom')."""
    g = nx.DiGraph()
    mk = dict(demand_dist_func=_np_poisson_marker, dist_param={"lam": 20})
    if kind == "default":
        g.add_nodes_from([0])
        g.add_nodes_from([1], I0=100, h=0.030)
        g.add_nodes_from([2], I0=110, h=0.020)
        g.add_nodes_from([3], I0=80, h=0.015)
        g.add_nodes_from([4], I0=400, C=90, o=0.010, v=1.000, h=0.012)
        g.add_nodes_from([5], I0=350, C=90, o=0.015, v=1.000, h=0.013)
        g.add_nodes_from([6], I0=380, C=80, o=0.012, v=1.000, h=0.011)
        g.add_nodes_from([7, 8])
        g.add_edges_from([
            (1, 0, dict(p=2.000, b=0.100, **mk)),
            (2, 1, {"L": 5, "p": 1.500, "g": 0.010}), (3, 1, {"L": 3, "p": 1.600, "g": 0.015}),
            (4, 2, {"L": 8, "p": 1.000, "g": 0.008}), (4, 3, {"L": 10, "p": 0.800, "g": 0.006}),
            (5, 2, {"L": 9, "p": 0.700, "g": 0.005}), (6, 2, {"L": 11, "p": 0.750, "g": 0.007}),
            (6, 3, {"L": 12, "p": 0.800, "g": 0.004}), (7, 4, {"L": 0, "p": 0.150, "g": 0.000}),
            (7, 5, {"L": 1, "p": 0.050, "g": 0.005}), (8, 5, {"L": 2, "p": 0.070, "g": 0.002}),
            (8, 6, {"L": 0, "p": 0.200, "g": 0.000})])
    elif kind == "custom":
        g.add_nodes_from([0])
        g.add_nodes_from([1, 2, 3], I0=120, h=0.200)
        g.add_nodes_from([4], I0=900, h=0.200)
        g.add_nodes_from([5], I0=1200, C=80, o=0.012, v=1.000, h=0.100)
        g.add_nodes_from([6])
        g.add_edges_from([
            (1, 0, dict(p=25.000, b=0.200, **mk)), (2, 0, dict(p=25.000, b=0.200, **mk)),
            (3, 0, dict(p=25.000, b=0.200, **mk)),
            (4, 1, {"L": 1, "p": 5.500, "g": 0.010}), (4, 2, {"L": 1, "p": 5.500, "g": 0.010}),
            (4, 3, {"L": 1, "p": 5.500, "g": 0.010}), (5, 4, {"L": 1, "p": 1.2, "g": 0.015}),
            (6, 5, {"L": 0, "p": 0.500, "g": 0.000})])
    else:
        raise ValueError(kind)
    return g


def graph_from_spec(spec):
    """Build a DiGraph from a JSON-able {'nodes': [[id, attrs]...], 'edges': [[u, v, attrs]...]} description."""
    g = nx.DiGraph()
    for j, a in spec["nodes"]:
        g.add_node(j, **a)
    for u, v, a in spec["edges"]:
        a = dict(a)
        if "L" in a:
            a["L"] = int(a["L"])
        if "dist_param" in a and "demand_dist_func" not in a:
            a["demand_dist_func"] = _np_poisson_marker
        g.add_edge(u, v, **a)
    return g


def synthetic_graph(seed=64, layers=(4, 12, 12, 20, 16)):
    """Layered synthetic network (SURVEY.md §8d, config 5): markets / retailers / distributors / factories / raw
    materials; every non-raw, non-market node buys from 2 nodes of the layer above, every retailer serves 1-2
    markets.  Passes the reference's validation (network_management.py:197-238)."""
    rng = np.random.default_rng(seed)
    n_mk, n_rt, n_ds, n_fc, n_raw = layers
    g = nx.DiGraph()
    ids = iter(range(sum(layers)))
    markets = [next(ids) for _ in range(n_mk)]
    retailers = [next(ids) for _ in range(n_rt)]
    distribs = [next(ids) for _ in range(n_ds)]
    factories = [next(ids) for _ in range(n_fc)]
    raws = [next(ids) for _ in range(n_raw)]
    g.add_nodes_from(markets)
    for j in retailers + distribs:
        g.add_node(j, I0=int(rng.integers(50, 501)), h=float(rng.uniform(0.01, 0.05)))
    for j in factories:
        g.add_node(j, I0=int(rng.integers(50, 501)), h=float(rng.uniform(0.01, 0.05)),
                   C=int(rng.integers(50, 151)), o=float(rng.uniform(0.005, 0.02)), v=1.0)
    g.add_nodes_from(raws)
    for r in retailers:
        for mk in rng.choice(markets, size=int(rng.integers(1, 3)), replace=False):
            g.add_edge(r, int(mk), p=float(rng.uniform(2, 30)), b=float(rng.uniform(0.05, 0.5)),
                       demand_dist_func=_np_poisson_marker, dist_param={"lam": int(rng.integers(5, 41))})
    for lower, upper in ((retailers, distribs), (distribs, factories), (factories, raws)):
        for j in lower:
            for s in rng.choice(upper, size=2, replace=False):
                g.add_edge(int(s), j, L=int(rng.integers(0, 13)), p=float(rng.uniform(0.5, 2.0)),
                           g=float(rng.uniform(0.0, 0.02)))
    return g


class NetInvMgmtParams:
    """Host mirror of NetInvMgmtMasterEnv.__init__ (network_management.py:55-106)."""

    _default_kind = "default"

    def __init__(self, graph=None, num_periods: int = 30, backlog: bool = True, alpha: float = 1.00,
                 seed_int: int = 0, user_D: Optional[Dict[Tuple[int, int], List[int]]] = None,
                 sample_path: Optional[Dict[Tuple[int, int], bool]] = None, env_config: Optional[Dict] = None,
                 default_graph_kind: Optional[str] = None):
        if nx is None:
            raise ImportError("networkx is required for the network env (the reference's graph container)")
        self.num_periods = num_periods
        self.backlog = backlog
        self.alpha = alpha
        self.seed_int = seed_int
        self.user_D = user_D if user_D is not None else {}
        self.sample_path = sample_path if sample_path is not None else {}
        if graph is not None:
            self.graph = graph_from_spec(graph) if isinstance(graph, dict) else graph.copy()  # :77
        else:
            self.graph = default_graph(default_graph_kind or self._default_kind)  # :79
            for e in list(self.graph.edges()):  # default user_D / sample_path of the market links (:141-144)
                if "L" not in self.graph.edges[e]:
                    self.user_D.setdefault(e, np.zeros(self.num_periods))
                    self.sample_path.setdefault(e, False)
        # the ctor's `backlog` argument overrides whatever env_config says (:83-85) -- which is why the reference's
        # NetInvMgmtLostSalesEnv() actually runs with backlog=True unless backlog=False is passed explicitly
        _env_config = dict(env_config) if env_config else {}
        _env_config["backlog"] = self.backlog
        for key, value in _env_config.items():
            if key == "graph" and isinstance(value, nx.DiGraph):
                self.graph = value.copy()
            else:
                setattr(self, key, value)
        self._initialize_graph_dependent_attributes()
        self._validate_inputs()

    # network_management.py:146-195
    def _initialize_graph_dependent_attributes(self):
        g = self.graph
        for link, d in self.user_D.items():
            if link in g.edges:
                g.edges[link]["user_D"] = list(d) if not isinstance(d, (list, np.ndarray)) else d
                g.edges[link]["sample_path"] = self.sample_path.get(link, False)
        self.retail_links = [e for e in g.edges() if "L" not in g.edges[e]]
        for link in self.retail_links:
            g.edges[link].setdefault("user_D", np.zeros(self.num_periods))
            g.edges[link].setdefault("sample_path", False)
        self.num_nodes = g.number_of_nodes()
        self.market = [j for j in g.nodes() if not list(g.successors(j))]
        self.rawmat = [j for j in g.nodes() if not list(g.predecessors(j))]
        self.factory = [j for j in g.nodes() if "C" in g.nodes[j]]
        self.distrib = [j for j in g.nodes() if "I0" in g.nodes[j] and "C" not in g.nodes[j] and j not in self.rawmat]
        self.retail = [j for j in self.distrib if any(s in self.market for s in g.successors(j))]
        self.main_nodes = sorted(list(set(self.distrib + self.factory)))
        self.reorder_links = sorted([e for e in g.edges() if "L" in g.edges[e]])
        self.network_links = sorted([e for e in g.edges()])
        self.lead_times = {e: g.edges[e]["L"] for e in self.reorder_links}
        self.lt_max = max(self.lead_times.values()) if self.lead_times else 0
        self.pipeline_obs_length = sum(self.lead_times.values())
        self.obs_dim = len(self.retail_links) + len(self.main_nodes) + self.pipeline_obs_length
        self.init_inv_max = max((g.nodes[j].get("I0", 0) for j in self.main_nodes), default=100)
        self.capacity_max = max((g.nodes[j].get("C", 0) for j in self.factory), default=100)
        self.order_cap_heuristic = self.init_inv_max + self.capacity_max * 5

    # network_management.py:197-238 (same messages)
    def _validate_inputs(self):
        g = self.graph
        for j in g.nodes():
            attrs = g.nodes[j]
            if j in self.main_nodes:
                assert "I0" in attrs and attrs["I0"] >= 0, f"Node {j}: Invalid or missing I0>=0"
                assert "h" in attrs and attrs["h"] >= 0, f"Node {j}: Invalid or missing h>=0"
            if j in self.factory:
                assert "C" in attrs and attrs["C"] > 0, f"Node {j}: Invalid or missing C>0"
                assert "o" in attrs and attrs["o"] >= 0, f"Node {j}: Invalid or missing o>=0"
                assert "v" in attrs and 0 < attrs["v"] <= 1, f"Node {j}: Invalid or missing v in (0, 1]"
        for u, v, attrs in g.edges(data=True):
            edge = (u, v)
            if edge in self.reorder_links:
                assert "L" in attrs and attrs["L"] >= 0, f"Edge {edge}: Invalid or missing L>=0"
                assert "p" in attrs and attrs["p"] >= 0, f"Edge {edge}: Invalid or missing p>=0"
                assert "g" in attrs and attrs["g"] >= 0, f"Edge {edge}: Invalid or missing g>=0"
            if edge in self.retail_links:
                assert "p" in attrs and attrs["p"] >= 0, f"Edge {edge}: Invalid or missing p>=0 (price)"
                assert "b" in attrs and attrs["b"] >= 0, f"Edge {edge}: Invalid or missing b>=0 (backlog cost)"
                assert "demand_dist_func" in attrs or "user_D" in attrs, \
                    f"Edge {edge}: Missing demand source ('demand_dist_func' or 'user_D')"
                if "demand_dist_func" in attrs:
                    assert "dist_param" in attrs, f"Edge {edge}: Missing 'dist_param' for 'demand_dist_func'"
                if "user_D" in attrs and np.sum(attrs["user_D"]) > 0 and not attrs.get("sample_path", False):
                    assert len(attrs["user_D"]) == self.num_periods, \
                        f"Edge {edge}: user_D length {len(attrs['user_D'])} != num_periods {self.num_periods}"
        assert isinstance(self.backlog, bool), "backlog must be boolean"
        assert 0 < self.alpha <= 1, "alpha must be in (0, 1]"
        assert self.num_periods > 0, "num_periods must be positive"

    # network_management.py:270-298
    def spaces(self, lost_sales_class=False):
        n_re = len(self.reorder_links)
        action_high = np.ones(n_re, dtype=np.float32) * self.order_cap_heuristic * 2
        action_space = Box(low=np.zeros(n_re, dtype=np.float32), high=action_high, shape=(n_re,), dtype=np.float32)
        hi = self.order_cap_heuristic * self.num_periods * 2
        lo = 0.0 if not self.backlog else -hi
        obs_low = np.full(self.obs_dim, lo, dtype=np.float32)
        obs_high = np.full(self.obs_dim, hi, dtype=np.float32)
        obs_low[0:len(self.retail_links)] = 0.0
        observation_space = Box(low=obs_low, high=obs_high, shape=(self.obs_dim,), dtype=np.float32)
        return observation_space, action_space

    # demand source of a retail link (network_management.py:240-267)
    def _link_dist(self, edge, keep):
        data = self.graph.edges[edge]
        use_user_d = ("user_D" in data and np.sum(data["user_D"]) > 0 and not data.get("sample_path", False))
        if use_user_d:  # :250-255; values pass through max(0, int(round(.))) in step (:540)
            tr = [max(0, int(round(float(x)))) for x in data["user_D"]]
            return _capi.make_dist(_capi.DIST_USER, user_D=tr, keep=keep)
        if "demand_dist_func" in data and "dist_param" in data:
            dp = data["dist_param"]
            kind = data.get("dist")
            keys = set(dp)
            if kind is None and data["demand_dist_func"] is not _np_poisson_marker:
                # an arbitrary Python callable cannot run on the GPU: the law is inferred from the parameter names, which
                # is only a guess (a negative-binomial sampler also takes n and p) -- say so instead of guessing silently
                guess = ("poisson" if keys and keys <= {"lam", "mu"} else "binomial" if keys == {"n", "p"} else
                         "randint" if keys == {"low", "high"} else "geometric" if keys == {"p"} else None)
                if guess is not None:
                    import warnings
                    warnings.warn(f"Edge {edge}: demand_dist_func is a Python callable; assuming a {guess} distribution "
                                  f"from dist_param keys {sorted(keys)} (set edge attribute dist='{guess}' to confirm, or "
                                  "another supported name to override)", stacklevel=3)
            if kind == "poisson" or (kind is None and keys <= {"lam", "mu"} and keys):
                return _capi.make_dist(_capi.DIST_POISSON, dp.get("lam", dp.get("mu")))
            if kind == "binomial" or (kind is None and keys == {"n", "p"}):
                return _capi.make_dist(_capi.DIST_BINOMIAL, dp["n"], dp["p"])
            if kind == "randint" or (kind is None and keys == {"low", "high"}):
                return _capi.make_dist(_capi.DIST_RANDINT, dp["low"], dp["high"] - 1)  # numpy integers(): high exclusive
            if kind == "geometric" or (kind is None and keys == {"p"}):
                return _capi.make_dist(_capi.DIST_GEOMETRIC, dp["p"])
            raise NotImplementedError(
                f"Edge {edge}: cannot run an arbitrary Python demand_dist_func on the GPU; dist_param keys {sorted(keys)} "
                "do not identify a supported distribution (set edge attribute dist='poisson'|'binomial'|'randint'|'geometric', "
                "or pass user_D)")
        return _capi.make_dist(_capi.DIST_USER, user_D=[0] * int(self.num_periods), keep=keep)  # :264-267

    def to_c(self, keep):
        """orgym_netinv_config_t; `keep` receives every buffer the struct points into."""
        g = self.graph
        main = self.main_nodes
        idx = {j: i for i, j in enumerate(main)}
        J, E, M = len(main), len(self.reorder_links), len(self.retail_links)

        def arr(a, dt):
            a = np.ascontiguousarray(np.asarray(a, dtype=dt))
            keep.append(a)
            return a

        c = _capi.NetConfig()
        c.num_periods = int(self.num_periods)
        c.backlog = int(bool(self.backlog))
        c.alpha = float(self.alpha)
        c.num_main = J
        c.node_I0 = arr([g.nodes[j].get("I0", 0) for j in main], np.float64).ctypes.data_as(_capi.c_f64p)
        c.node_h = arr([g.nodes[j]["h"] for j in main], np.float64).ctypes.data_as(_capi.c_f64p)
        c.node_is_factory = arr([j in self.factory for j in main], np.uint8).ctypes.data_as(_capi.c_u8p)
        c.node_is_retail = arr([j in self.retail for j in main], np.uint8).ctypes.data_as(_capi.c_u8p)
        c.node_C = arr([g.nodes[j].get("C", 0) for j in main], np.float64).ctypes.data_as(_capi.c_f64p)
        c.node_v = arr([g.nodes[j].get("v", 1.0) for j in main], np.float64).ctypes.data_as(_capi.c_f64p)
        c.node_o = arr([g.nodes[j].get("o", 0) for j in main], np.float64).ctypes.data_as(_capi.c_f64p)
        c.num_reorder = E
        sup = []
        for (s, p) in self.reorder_links:
            if s in self.rawmat:  # checked first in the reference (:453)
                sup.append(-1)
            elif s in idx:
                sup.append(idx[s])
            else:
                sup.append(-2)
        c.re_supplier = arr(sup, np.int32).ctypes.data_as(_capi.c_i32p)
        c.re_purchaser = arr([idx.get(p, -1) for (s, p) in self.reorder_links], np.int32).ctypes.data_as(_capi.c_i32p)
        c.re_lead = arr([g.edges[e]["L"] for e in self.reorder_links], np.int32).ctypes.data_as(_capi.c_i32p)
        c.re_p = arr([g.edges[e]["p"] for e in self.reorder_links], np.float64).ctypes.data_as(_capi.c_f64p)
        c.re_g = arr([g.edges[e]["g"] for e in self.reorder_links], np.float64).ctypes.data_as(_capi.c_f64p)
        c.num_retail = M
        for (r, mk) in self.retail_links:
            if r not in idx:
                raise KeyError(f"retail link {(r, mk)}: node {r} holds no inventory (the reference fails at :547)")
        c.rt_retailer = arr([idx[r] for (r, mk) in self.retail_links], np.int32).ctypes.data_as(_capi.c_i32p)
        c.rt_p = arr([g.edges[e]["p"] for e in self.retail_links], np.float64).ctypes.data_as(_capi.c_f64p)
        c.rt_b = arr([g.edges[e]["b"] for e in self.retail_links], np.float64).ctypes.data_as(_capi.c_f64p)
        dists = (_capi.Dist * max(M, 1))()
        for i, e in enumerate(self.retail_links):
            dists[i] = self._link_dist(e, keep)
        keep.append(dists)
        c.rt_dist = C.cast(dists, C.POINTER(_capi.Dist))
        re_id = {e: i for i, e in enumerate(self.reorder_links)}
        rt_id = {e: i for i, e in enumerate(self.retail_links)}
        sp, si, pp, pi = [0], [], [0], []
        for j in main:
            for k in g.successors(j):  # adjacency (insertion) order = Python sum order (:582)
                e = (j, k)
                si.append(re_id[e] if e in re_id else E + rt_id[e])
            sp.append(len(si))
            for k in g.predecessors(j):  # (:586)
                e = (k, j)
                if e in re_id:
                    pi.append(re_id[e])
            pp.append(len(pi))
        c.succ_ptr = arr(sp, np.int32).ctypes.data_as(_capi.c_i32p)
        c.succ_idx = arr(si or [0], np.int32).ctypes.data_as(_capi.c_i32p)
        c.pred_ptr = arr(pp, np.int32).ctypes.data_as(_capi.c_i32p)
        c.pred_idx = arr(pi or [0], np.int32).ctypes.data_as(_capi.c_i32p)
        return c


class NetInvMgmtMasterEnv(BatchedEnv):
    """`num_envs` instances of the network env in lock-step on one GPU.  Extra keywords: `num_envs`, `device`,
    `env_offset`, `autoreset_mode`, `info_level`."""

    _family = "netinv"
    _default_kind = "default"
    metadata = {"render_modes": ["human"], "render_fps": 4}

    def __init__(self, *args, num_envs: int = 1, device="cuda", env_offset: int = 0,
                 autoreset_mode: str = "next_step", info_level: int = 1, specialise: Optional[bool] = None,
                 record_history: bool = False, **kwargs):
        """specialise: True = compile kernels for this topology with NVRTC at construction (1-2 s for small graphs,
        10-15 s for the 64-node one, then cached on disk; 3-5x faster stepping), False = generic kernel, None =
        automatic (graphs with up to 128 reorder links).  The environment variable ORGYM_NET_JIT (0/1/2) takes
        precedence when set."""
        torch = _torch()
        self.record_history = bool(record_history)
        if self.record_history:
            if autoreset_mode != "disabled":
                raise ValueError("record_history=True needs autoreset_mode='disabled'")
            info_level = max(int(info_level), 1)
        kwargs.setdefault("default_graph_kind", self._default_kind)
        self.params = NetInvMgmtParams(*args, **kwargs)
        P = self.params
        for name in ("graph", "num_periods", "backlog", "alpha", "user_D", "sample_path", "retail_links", "market",
                     "rawmat", "factory", "distrib", "retail", "main_nodes", "reorder_links", "network_links",
                     "lead_times", "lt_max", "pipeline_obs_length", "obs_dim", "order_cap_heuristic", "num_nodes"):
            setattr(self, name, getattr(P, name))
        self.observation_space_single, self.action_space_single = P.spaces()
        self._setup_batch(num_envs, device, env_offset, autoreset_mode)
        self.info_level = int(info_level)
        lib = _capi.lib()
        cfg = P.to_c(self._keep)
        import os
        had = os.environ.get("ORGYM_NET_JIT")
        if specialise is not None and had is None:
            os.environ["ORGYM_NET_JIT"] = "1" if specialise else "0"
        try:
            _capi.check(lib.orgym_netinv_create(C.byref(cfg), self.num_envs, self.device.index, C.byref(self._h)))
        finally:
            if specialise is not None and had is None:
                os.environ.pop("ORGYM_NET_JIT", None)
        assert lib.orgym_netinv_obs_dim(self._h) == P.obs_dim
        self.specialised = bool(lib.orgym_netinv_is_specialised(self._h))
        N, od, dev = self.num_envs, P.obs_dim, self.device
        J, E, M = len(P.main_nodes), len(P.reorder_links), len(P.retail_links)
        self._alloc_state(lib.orgym_netinv_state_bytes(self._h))
        self._obs = torch.zeros((N, od), dtype=torch.float32, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float64, device=dev)
        self._terminated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._truncated = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._term_b, self._trunc_b = self._terminated.view(torch.bool), self._truncated.view(torch.bool)  # cached views
        self._info = _capi.NetInfo()
        self._info_t = {}
        if self.info_level >= 1:
            # [N, dim] tensors backed by column-major storage (a transposed view): the kernels then write every info
            # value with coalesced stores; indexing / .cpu() / .numpy() behave as for any [N, dim] tensor
            self._info_t = dict(demand=torch.zeros((M, N), dtype=torch.float64, device=dev).t(),
                                sales=torch.zeros((E + M, N), dtype=torch.float64, device=dev).t(),
                                profit_node=torch.zeros((J, N), dtype=torch.float64, device=dev).t(),
                                profit_period_undiscounted=torch.zeros(N, dtype=torch.float64, device=dev))
            self._info.info_ld = N
            self._info.demand = self._info_t["demand"].data_ptr()
            self._info.sales = self._info_t["sales"].data_ptr()
            self._info.profit = self._info_t["profit_node"].data_ptr()
            self._info.profit_total = self._info_t["profit_period_undiscounted"].data_ptr()
        if autoreset_mode == "same_step":
            self._final_obs = torch.zeros((N, od), dtype=torch.float32, device=dev)
            self._info.final_obs = self._final_obs.data_ptr()
        self._has_reset = False
        self._scratch = None

    def _out_tensor(self, t, shape, dtype, what):
        """A caller-provided output buffer (e.g. slot t of a trajectory tensor): must be a contiguous CUDA tensor of
        the right shape / dtype on this env's device -- the kernels write into it directly (zero-copy)."""
        torch = _torch()
        if not (isinstance(t, torch.Tensor) and t.device == self.device and t.dtype == dtype and
                tuple(t.shape) == tuple(shape) and t.is_contiguous()):
            raise ValueError(f"{what} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {self.device}")
        return t

    def reset(self, *, seed=None, options: Optional[Dict] = None, obs_out=None):
        """reset (network_management.py:301-332).  obs_out: optional float32 [N, obs_dim] tensor that receives the
        first observation instead of the env's own buffer."""
        reseed, base = self._resolve_seed(seed)
        mask = None
        if options and options.get("reset_mask") is not None:
            mask = self._to_dev(options["reset_mask"], _torch().uint8, (self.num_envs,))
        obs = self._obs if obs_out is None else self._out_tensor(obs_out, self._obs.shape, self._obs.dtype, "obs_out")
        _capi.check(_capi.lib().orgym_netinv_reset(self._h, self._ptr(self._state), reseed, C.c_uint64(base),
                                                   self.env_offset, self._ptr(mask), self._ptr(obs),
                                                   self._stream()))
        self._has_reset = True
        if self.record_history:
            if mask is not None:
                raise NotImplementedError("record_history keeps all instances in lock-step: reset without a mask")
            self._alloc_history()
        return obs, {}

    # -- full-history buffers: the DataFrames the reference keeps (:315-321) as [N, T(+1), columns] tensors; columns in
    # main_nodes / reorder_links / retail_links order, S = reorder links then retail links -----------------------------
    def _alloc_history(self):
        torch = _torch()
        N, T, dev = self.num_envs, int(self.num_periods), self.device
        J, E, M = len(self.main_nodes), len(self.reorder_links), len(self.retail_links)
        z = lambda *shape: torch.zeros(shape, dtype=torch.float64, device=dev)  # noqa: E731
        self.X, self.Y, self.U = z(N, T + 1, J), z(N, T + 1, E), z(N, T + 1, M)
        self.R, self.S, self.D, self.P = z(N, T, E), z(N, T, E + M), z(N, T, M), z(N, T, J)
        self.X[:, 0] = torch.as_tensor([float(self.graph.nodes[j].get("I0", 0)) for j in self.main_nodes],
                                       dtype=torch.float64, device=dev)
        self._t_host = 0

    def _record(self, info):
        t = self._t_host
        if t >= int(self.num_periods):
            return
        E = len(self.reorder_links)
        X, Y, U, _ = self.export_state()
        self.X[:, t + 1], self.Y[:, t + 1], self.U[:, t + 1] = X, Y, U
        self.S[:, t], self.R[:, t] = info["sales"], info["sales"][:, :E]
        self.D[:, t], self.P[:, t] = info["demand"], info["profit_node"]
        self._t_host = t + 1

    def step(self, actions, demand=None, *, obs_out=None, reward_out=None):
        """step (network_management.py:436-635): actions float32 [N, len(reorder_links)] in sorted link order;
        optional replayed demand float64 [N, len(retail_links)] in retail_links order.  obs_out / reward_out: optional
        float32 [N, obs_dim] / float64 [N] tensors the kernels write into instead of the env's own buffers (e.g. slot
        t of a rollout-collection buffer: no copy between the env and the learner's storage)."""
        torch = _torch()
        if not self._has_reset:
            raise RuntimeError("call reset() before step()")
        E, M = len(self.reorder_links), len(self.retail_links)
        a = self._to_dev(actions, torch.float32, (self.num_envs, E))
        d = self._to_dev(demand, torch.float64, (self.num_envs, M)) if demand is not None else None
        obs = self._obs if obs_out is None else self._out_tensor(obs_out, self._obs.shape, self._obs.dtype, "obs_out")
        rew = self._reward if reward_out is None else self._out_tensor(reward_out, self._reward.shape, self._reward.dtype,
                                                                       "reward_out")
        _capi.check(_capi.lib().orgym_netinv_step(
            self._h, self._ptr(self._state), self._ptr(a), self._ptr(d), _AUTORESET[self.autoreset_mode],
            self._ptr(obs), self._ptr(rew), self._ptr(self._terminated), self._ptr(self._truncated),
            C.byref(self._info), self._stream()))
        info = dict(self._info_t)
        if self.autoreset_mode == "same_step":
            info["final_obs"] = self._final_obs
        if self.record_history:
            self._record(info)
        return obs, rew, self._term_b, self._trunc_b, info

    def export_state(self):
        """(X f64[N,J], Y f64[N,E], U f64[N,M], period i32[N]) in main_nodes / reorder_links / retail_links order."""
        torch = _torch()
        N = self.num_envs
        J, E, M = len(self.main_nodes), len(self.reorder_links), len(self.retail_links)
        X = torch.empty((N, J), dtype=torch.float64, device=self.device)
        Y = torch.empty((N, E), dtype=torch.float64, device=self.device)
        U = torch.empty((N, M), dtype=torch.float64, device=self.device)
        t = torch.empty(N, dtype=torch.int32, device=self.device)
        _capi.check(_capi.lib().orgym_netinv_export_state(self._h, self._ptr(self._state), self._ptr(X), self._ptr(Y),
                                                          self._ptr(U), self._ptr(t), self._stream()))
        return X, Y, U, t

    @property
    def period(self):
        return self.export_state()[3]

    def rollout(self, policy="constant", *, seed=None, episode=0, order_fraction=0.1, actions=None, demand=None,
                time_major=False, want=("ep_return", "stats", "summary"), buffer_set=0):
        """Fused reset + num_periods steps (K5).  policy 'constant': the ConstantOrderAgent action
        (high * order_fraction as float32, benchmark_NetInvMgmtBacklogEnv.py:119-136) or an explicit float32[E]
        `actions` vector; policy 'actions': float32 [N,T,E] ([T,N,E] if time_major); or an actor network -- a
        torch.nn.Sequential (Linear, Tanh|ReLU, ..., Linear) or an SB3 ActorCriticPolicy (e.g. `model.policy` of a
        trained PPO) -- evaluated on the device every period on the observation step() would return, its output
        clipped to [0, single_action_space.high] like SB3's deterministic predict.  demand: optional float64
        [N,T,M].  Returns device tensors ep_return, stats [N,4] (sum retail sales, demand, backlog, on-hand),
        summary [8]; on request reward_traj, final_X, final_Y, final_U and, for a network, action_traj
        (float32 [N,T,E], the actions it took)."""
        torch = _torch()
        N, T = self.num_envs, int(self.num_periods)
        J, E, M = len(self.main_nodes), len(self.reorder_links), len(self.retail_links)
        rin = _capi.NetRolloutIn()
        keep = []
        if not isinstance(policy, str):
            mlp, tensors = pack_mlp(policy, self.obs_dim, E, self.device)
            high = np.ascontiguousarray(self.single_action_space.high, dtype=np.float32)
            keep += [mlp, tensors, high]
            rin.policy = POLICY_MLP
            rin.mlp = C.pointer(mlp)
            rin.action_high = high.ctypes.data
        elif "action_traj" in want:
            raise ValueError("action_traj is recorded only for an actor network policy")
        elif policy == "constant":
            rin.policy = 1
            if actions is None:
                actions = (self.single_action_space.high * order_fraction).astype(np.float32)
            a = self._to_dev(actions, torch.float32, (E,))
        elif policy == "actions":
            rin.policy = 0
            a = self._to_dev(actions, torch.float32, (T, N, E) if time_major else (N, T, E))
            rin.act_stride_env, rin.act_stride_t = (E, N * E) if time_major else (T * E, E)
        else:
            raise ValueError(policy)
        if rin.policy != POLICY_MLP:
            keep.append(a)
            rin.actions = a.data_ptr()
        if demand is not None:
            d = self._to_dev(demand, torch.float64, (T, N, M) if time_major else (N, T, M))
            keep.append(d)
            rin.demand = d.data_ptr()
            rin.dem_stride_env, rin.dem_stride_t = (M, N * M) if time_major else (T * M, M)
        shapes = dict(ep_return=((N,), torch.float64), stats=((N, 4), torch.float64),
                      reward_traj=((N, T), torch.float64), final_X=((N, J), torch.float64),
                      final_Y=((N, E), torch.float64), final_U=((N, M), torch.float64), summary=((8,), torch.float64),
                      action_traj=((N, T, E), torch.float32))
        out = {}
        rout = _capi.NetRolloutOut()
        cache = self.__dict__.setdefault("_rollout_buf", {}).setdefault(int(buffer_set), {})
        for name in want:
            shp, dt = shapes[name]
            if name not in cache:
                cache[name] = torch.zeros(shp, dtype=dt, device=self.device)
            out[name] = cache[name]
            setattr(rout, name, out[name].data_ptr())
        if self._scratch is None:
            self._scratch = torch.zeros_like(self._state)
        if seed is not None:
            self._resolve_seed(seed)
        elif not self._seeded:
            self._resolve_seed(None)
        _capi.check(_capi.lib().orgym_netinv_rollout(self._h, self._ptr(self._scratch), C.c_uint64(self._seed),
                                                     self.env_offset, C.c_uint32(int(episode)), C.byref(rin),
                                                     C.byref(rout), self._stream()))
        return out


class NetInvMgmtBacklogEnv(NetInvMgmtMasterEnv):
    """network_management.py:747-753.  env_config['backlog']=True is set, then overridden by the ctor's `backlog`
    argument (default True) exactly as in the reference."""

    def __init__(self, *args, **kwargs):
        env_config = dict(kwargs.pop("env_config", None) or {})
        env_config["backlog"] = True
        super().__init__(*args, env_config=env_config, **kwargs)


class NetInvMgmtLostSalesEnv(NetInvMgmtMasterEnv):
    """network_management.py:755-770.  Reference-faithful: the subclass only sets env_config['backlog']=False,
    which the master ctor overwrites with its own `backlog` argument (default True), so
    `NetInvMgmtLostSalesEnv()` simulates BACKLOG dynamics -- pass `backlog=False` for real lost sales."""

    def __init__(self, *args, **kwargs):
        env_config = dict(kwargs.pop("env_config", None) or {})
        env_config["backlog"] = False
        super().__init__(*args, env_config=env_config, **kwargs)
        low = self.observation_space_single.low.copy()
        low[0:len(self.retail_links)] = 0.0
        self.observation_space_single = Box(low=low, high=self.observation_space_single.high, shape=(self.obs_dim,),
                                            dtype=np.float32)
        self.single_observation_space = self.observation_space_single
