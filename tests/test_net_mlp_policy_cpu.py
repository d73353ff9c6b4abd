"""CPU suite for the MLP actor policy of the network env's fused rollout: the ctypes mirrors of
orgym_netinv_rollout_in_t / _out_t with their new fields, and the refusals that fire before any device work."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn as nn

from or_gym_inventory_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_capi.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _capi.lib()


def _offsets(tmp_path, ctype, cls, cnames, extra=()):
    fields = [f[0] for f in cls._fields_]
    assert fields == list(cnames)
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "orgym_b200.h"', 'int main(void) {',
           f'  printf("size %zu\\n", sizeof({ctype}));'] + list(extra)
    for f in fields:
        src.append(f'  printf("{f} %zu\\n", offsetof({ctype}, {cnames[f]}));')
    src.append('  return 0; }')
    c = tmp_path / f"{ctype}.c"
    c.write_text("\n".join(src))
    exe = tmp_path / ctype
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(c),
                           "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(cls)
    for f in fields:
        assert int(got[f]) == getattr(cls, f).offset, f
    return got


def test_net_rollout_in_matches_the_header(tmp_path):
    """orgym_netinv_rollout_in_t: size and every field offset as gcc lays out the header; the policy constant."""
    cnames = dict(policy="policy", actions="actions_dev", act_stride_env="act_stride_env", act_stride_t="act_stride_t",
                  demand="demand_dev", dem_stride_env="dem_stride_env", dem_stride_t="dem_stride_t", mlp="mlp",
                  action_high="action_high")
    got = _offsets(tmp_path, "orgym_netinv_rollout_in_t", _capi.NetRolloutIn, cnames,
                   ['  printf("policy_mlp %d\\n", ORGYM_NET_POLICY_MLP);'])
    from or_gym_inventory_b200.network_management import POLICY_MLP
    assert int(got["policy_mlp"]) == POLICY_MLP


def test_net_rollout_out_matches_the_header(tmp_path):
    cnames = dict(ep_return="ep_return_dev", stats="stats_dev", reward_traj="reward_traj_dev", final_X="final_X_dev",
                  final_Y="final_Y_dev", final_U="final_U_dev", summary="summary_dev", action_traj="action_traj_dev")
    _offsets(tmp_path, "orgym_netinv_rollout_out_t", _capi.NetRolloutOut, cnames)


class _NoDeviceEnv:
    """Just enough of NetInvMgmtMasterEnv for rollout() to reach the packing: any device call would raise."""

    def __init__(self):
        from or_gym_inventory_b200.network_management import NetInvMgmtParams
        P = NetInvMgmtParams()
        self.params = P
        for name in ("num_periods", "main_nodes", "reorder_links", "retail_links", "obs_dim"):
            setattr(self, name, getattr(P, name))
        self.num_envs = 4
        self.device = torch.device("cpu")

    def __getattr__(self, name):
        raise AssertionError(f"device work reached ({name}) before the network was checked")


@pytest.mark.parametrize("case, msg", [
    ("in_features", "the observation has"), ("out_features", "the action has 11"), ("five", "at most 4"),
    ("act_last", "end with a Linear"), ("sigmoid", "Sigmoid"), ("other", "neither"),
])
def test_network_env_refuses_wrong_networks_before_device_work(case, msg):
    from or_gym_inventory_b200.network_management import NetInvMgmtMasterEnv
    od, E = 68, 11   # the default graph
    nets = {
        "in_features": lambda: nn.Sequential(nn.Linear(od + 1, 8), nn.Tanh(), nn.Linear(8, E)),
        "out_features": lambda: nn.Sequential(nn.Linear(od, 8), nn.Tanh(), nn.Linear(8, 1)),
        "five": lambda: nn.Sequential(*[m for _ in range(4) for m in (nn.Linear(od if _ == 0 else 8, 8), nn.Tanh())],
                                      nn.Linear(8, E)),
        "act_last": lambda: nn.Sequential(nn.Linear(od, E), nn.Tanh()),
        "sigmoid": lambda: nn.Sequential(nn.Linear(od, 8), nn.Sigmoid(), nn.Linear(8, E)),
        "other": lambda: nn.Linear(od, E),
    }
    with pytest.raises(ValueError, match=msg):
        NetInvMgmtMasterEnv.rollout(_NoDeviceEnv(), nets[case]())


@pytest.mark.parametrize("policy", ["constant", "actions"])
def test_action_traj_needs_a_network(policy):
    from or_gym_inventory_b200.network_management import NetInvMgmtMasterEnv
    with pytest.raises(ValueError, match="action_traj"):
        NetInvMgmtMasterEnv.rollout(_NoDeviceEnv(), policy, want=("ep_return", "action_traj"))


def test_abi_refuses_mlp_requests_without_a_gpu(lib):
    """Without a handle (no GPU here) the network rollout refuses an MLP request with ORGYM_E_INVALID: a malformed
    network, no network, no action bound."""
    m = _capi.Mlp()
    m.num_layers = 9                                   # malformed on purpose
    high = np.full(11, 100.0, dtype=np.float32)
    rin = _capi.NetRolloutIn()
    rin.policy = 2
    rin.mlp = C.pointer(m)
    rin.action_high = high.ctypes.data
    rout = _capi.NetRolloutOut()
    assert lib.orgym_netinv_rollout(None, None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    rin.mlp = None
    assert lib.orgym_netinv_rollout(None, None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    rin.mlp = C.pointer(m)
    rin.action_high = None
    assert lib.orgym_netinv_rollout(None, None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
