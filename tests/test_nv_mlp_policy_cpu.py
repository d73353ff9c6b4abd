"""CPU suite for the MLP actor policy of the newsvendor's fused rollout: the ctypes mirror of
orgym_newsvendor_rollout_in_t with its `mlp` field, and the network-shape refusals that fire before any device work."""
import ctypes as C
import os
import subprocess

import pytest
import torch
import torch.nn as nn

from or_gym_inventory_b200 import _capi
from or_gym_inventory_b200.mlp import pack_mlp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_capi.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _capi.lib()


def test_nv_rollout_in_matches_the_header(tmp_path):
    """orgym_newsvendor_rollout_in_t: size and every field offset as gcc lays out the header."""
    cnames = dict(policy="policy", param="param", actions="actions_dev", act_stride_env="act_stride_env",
                  act_stride_t="act_stride_t", demand="demand_dev", dem_stride_env="dem_stride_env",
                  dem_stride_t="dem_stride_t", fixed_params="fixed_params_dev", mlp="mlp")
    fields = [f[0] for f in _capi.NvRolloutIn._fields_]
    assert fields == list(cnames) and fields[-1] == "mlp"
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "orgym_b200.h"', 'int main(void) {',
           '  printf("size %zu\\n", sizeof(orgym_newsvendor_rollout_in_t));',
           '  printf("policy_mlp %d\\n", ORGYM_NV_POLICY_MLP);']
    for f in fields:
        src.append(f'  printf("{f} %zu\\n", offsetof(orgym_newsvendor_rollout_in_t, {cnames[f]}));')
    src.append('  return 0; }')
    c = tmp_path / "nv_mlp_abi.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "nv_mlp_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(c),
                           "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(_capi.NvRolloutIn)
    for f in fields:
        assert int(got[f]) == getattr(_capi.NvRolloutIn, f).offset, f
    from or_gym_inventory_b200.newsvendor import POLICY_MLP
    assert int(got["policy_mlp"]) == POLICY_MLP


def test_serial_module_still_exports_the_packing():
    from or_gym_inventory_b200 import inventory_management, mlp
    assert inventory_management.pack_mlp is mlp.pack_mlp and inventory_management.mlp_layers is mlp.mlp_layers


class _NoDeviceEnv:
    """Just enough of NewsvendorEnv for rollout() to reach the packing: any device call would raise."""

    def __init__(self, lead_time):
        from or_gym_inventory_b200.newsvendor import NewsvendorParams
        self.params = NewsvendorParams(lead_time=lead_time)
        self.num_envs = 4
        self.device = torch.device("cpu")

    def __getattr__(self, name):
        raise AssertionError(f"device work reached ({name}) before the network was checked")


@pytest.mark.parametrize("lead_time", [0, 5])
@pytest.mark.parametrize("case, msg", [
    ("in_features", "the observation has"), ("out_features", "the action has 1"), ("five", "at most 4"),
    ("act_last", "end with a Linear"), ("sigmoid", "Sigmoid"), ("other", "neither"),
])
def test_newsvendor_refuses_wrong_networks_before_device_work(lead_time, case, msg):
    from or_gym_inventory_b200.newsvendor import NewsvendorEnv
    od = lead_time + 5
    nets = {
        "in_features": lambda: nn.Sequential(nn.Linear(od + 1, 8), nn.Tanh(), nn.Linear(8, 1)),
        "out_features": lambda: nn.Sequential(nn.Linear(od, 8), nn.Tanh(), nn.Linear(8, 2)),
        "five": lambda: nn.Sequential(*[m for _ in range(4) for m in (nn.Linear(od if _ == 0 else 8, 8), nn.Tanh())],
                                      nn.Linear(8, 1)),
        "act_last": lambda: nn.Sequential(nn.Linear(od, 1), nn.Tanh()),
        "sigmoid": lambda: nn.Sequential(nn.Linear(od, 8), nn.Sigmoid(), nn.Linear(8, 1)),
        "other": lambda: nn.Linear(od, 1),
    }
    with pytest.raises(ValueError, match=msg):
        NewsvendorEnv.rollout(_NoDeviceEnv(lead_time), nets[case]())


def test_packing_for_the_newsvendor():
    net = nn.Sequential(nn.Linear(10, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh(), nn.Linear(64, 1))
    m, keep = pack_mlp(net, 10, 1, torch.device("cpu"))
    assert m.num_layers == 3 and list(m.width)[:4] == [10, 64, 64, 1] and m.activation == _capi.MLP_TANH


def test_abi_refuses_mlp_requests_without_a_gpu(lib):
    """Without a handle (no GPU here) the newsvendor rollout refuses an MLP request with ORGYM_E_INVALID."""
    m = _capi.Mlp()
    m.num_layers = 9                                   # malformed on purpose
    rin = _capi.NvRolloutIn()
    rin.policy = 4
    rin.mlp = C.pointer(m)
    rout = _capi.NvRolloutOut()
    assert lib.orgym_newsvendor_rollout(None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    rin.mlp = None
    assert lib.orgym_newsvendor_rollout(None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
