"""CPU suite for the MLP actor policy of the serial env's fused rollout: the ctypes mirror of orgym_mlp_t, the packing of
torch modules (plain Sequential and SB3 ActorCriticPolicy-shaped actors) and the ABI refusals reachable without a GPU."""
import ctypes as C
import os
import subprocess

import pytest
import torch
import torch.nn as nn

from or_gym_inventory_b200 import _capi
from or_gym_inventory_b200.inventory_management import mlp_layers, pack_mlp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_capi.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _capi.lib()


class _Stub:
    """An object shaped like stable-baselines3's ActorCriticPolicy (MlpPolicy): features extractor, mlp_extractor with
    a policy_net ending in its activation, action_net."""

    class FlattenExtractor(nn.Module):
        def forward(self, x):
            return x.flatten(1)

    def __init__(self, obs=33, act=3, hidden=(64, 64), squash=False, fe=None, act_fn=nn.Tanh):
        layers, w = [], obs
        for h in hidden:
            layers += [nn.Linear(w, h), act_fn()]
            w = h
        self.mlp_extractor = type("MlpExtractor", (), {})()
        self.mlp_extractor.policy_net = nn.Sequential(*layers)
        self.action_net = nn.Linear(w, act)
        self.squash_output = squash
        self.features_extractor = fe if fe is not None else _Stub.FlattenExtractor()


def test_mlp_struct_matches_the_header(tmp_path):
    """orgym_mlp_t: size and every field offset as gcc lays out the header."""
    fields = [f[0] for f in _capi.Mlp._fields_]
    cnames = dict(num_layers="num_layers", activation="activation", width="width", weight="weight_dev", bias="bias_dev")
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "orgym_b200.h"', 'int main(void) {',
           '  printf("size %zu\\n", sizeof(orgym_mlp_t));']
    for f in fields:
        src.append(f'  printf("{f} %zu\\n", offsetof(orgym_mlp_t, {cnames[f]}));')
    src.append('  printf("in_mlp %zu\\n", offsetof(orgym_invmgmt_rollout_in_t, mlp));')
    src.append('  printf("out_action_traj %zu\\n", offsetof(orgym_invmgmt_rollout_out_t, action_traj_dev));')
    src.append('  return 0; }')
    c = tmp_path / "mlp_abi.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "mlp_abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(c),
                           "-o", str(exe)])
    got = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(got["size"]) == C.sizeof(_capi.Mlp)
    for f in fields:
        assert int(got[f]) == getattr(_capi.Mlp, f).offset, f
    assert int(got["in_mlp"]) == _capi.InvRolloutIn.mlp.offset
    assert int(got["out_action_traj"]) == _capi.InvRolloutOut.action_traj.offset


def _seq(widths, act=nn.Tanh, bias=True):
    mods = []
    for i in range(len(widths) - 1):
        mods.append(nn.Linear(widths[i], widths[i + 1], bias=bias))
        if i < len(widths) - 2:
            mods.append(act())
    return nn.Sequential(*mods)


@pytest.mark.parametrize("widths", [(33, 3), (33, 64, 3), (33, 64, 64, 3), (33, 17, 1, 128, 3)])
@pytest.mark.parametrize("act, code", [(nn.Tanh, _capi.MLP_TANH), (nn.ReLU, _capi.MLP_RELU)])
@pytest.mark.parametrize("bias", [True, False])
def test_packing_accepts_sequential_actors(widths, act, code, bias):
    net = _seq(widths, act, bias).double()              # any dtype: packed as float32
    m, keep = pack_mlp(net, 33, 3, torch.device("cpu"))
    L = len(widths) - 1
    assert m.num_layers == L and list(m.width)[:L + 1] == list(widths)
    assert m.activation == (code if L > 1 else _capi.MLP_TANH)
    ws = [t for t in keep if t.dim() == 2]
    assert len(ws) == L and all(t.dtype == torch.float32 and t.is_contiguous() for t in ws)
    for l in range(L):
        assert m.weight[l] == ws[l].data_ptr()
        assert bool(m.bias[l]) == bias
    assert torch.equal(ws[0], net[0].weight.float())


def test_packing_accepts_an_sb3_shaped_actor():
    pol = _Stub(hidden=(64, 64))
    lin, act = mlp_layers(pol)
    assert [l.out_features for l in lin] == [64, 64, 3] and act == _capi.MLP_TANH
    assert lin[-1] is pol.action_net
    m, _ = pack_mlp(pol, 33, 3, torch.device("cpu"))
    assert m.num_layers == 3 and list(m.width)[:4] == [33, 64, 64, 3]
    assert mlp_layers(_Stub(hidden=(), act=3))[0][0] is not None       # net_arch=[]: action_net alone
    assert mlp_layers(_Stub(act_fn=nn.ReLU))[1] == _capi.MLP_RELU
    assert mlp_layers(_Stub(fe=nn.Flatten()))[0]


@pytest.mark.parametrize("case, msg", [
    ("mixed", "one activation type"), ("act_last", "end with a Linear"), ("sigmoid", "Sigmoid"), ("dropout", "Dropout"),
    ("in_features", "in_features"), ("out_features", "out_features"), ("inner_mismatch", "in_features 32"),
    ("five", "at most 4"), ("squash", "squash_output"), ("cnn", "features_extractor"), ("other", "neither"),
])
def test_packing_refuses_what_the_device_cannot_evaluate(case, msg):
    nets = {
        "mixed": lambda: nn.Sequential(nn.Linear(33, 8), nn.Tanh(), nn.Linear(8, 8), nn.ReLU(), nn.Linear(8, 3)),
        "act_last": lambda: nn.Sequential(nn.Linear(33, 3), nn.Tanh()),
        "sigmoid": lambda: nn.Sequential(nn.Linear(33, 8), nn.Sigmoid(), nn.Linear(8, 3)),
        "dropout": lambda: nn.Sequential(nn.Linear(33, 8), nn.Tanh(), nn.Dropout(0.1), nn.Linear(8, 3)),
        "in_features": lambda: _seq((32, 8, 3)),
        "out_features": lambda: _seq((33, 8, 4)),
        "inner_mismatch": lambda: nn.Sequential(nn.Linear(33, 8), nn.Tanh(), nn.Linear(32, 3)),
        "five": lambda: _seq((33, 8, 8, 8, 8, 3)),
        "squash": lambda: _Stub(squash=True),
        "cnn": lambda: _Stub(fe=nn.Conv1d(1, 1, 1)),
        "other": lambda: nn.Linear(33, 3),
    }
    with pytest.raises(ValueError, match=msg):
        pack_mlp(nets[case](), 33, 3, torch.device("cpu"))


def test_abi_refuses_mlp_requests_without_a_gpu(lib):
    """Without a handle (no GPU here) the rollout and the specialiser refuse with ORGYM_E_INVALID; the code generator
    says the MLP policy is not specialised (ORGYM_E_UNSUPPORTED) -- neither needs a device."""
    import or_gym_inventory_b200 as pkg
    m = _capi.Mlp()
    m.num_layers = 9                                   # malformed on purpose
    rin = _capi.InvRolloutIn()
    rin.policy = 3
    rin.mlp = C.pointer(m)
    rout = _capi.InvRolloutOut()
    assert lib.orgym_invmgmt_rollout(None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    rin.mlp = None
    assert lib.orgym_invmgmt_rollout(None, 0, 0, 0, C.byref(rin), C.byref(rout), None) == _capi.E_INVALID
    assert lib.orgym_invmgmt_specialise(None, C.byref(rin)) == _capi.E_INVALID
    keep = []
    cfg = pkg.InvManagementParams().to_c(keep)
    need = C.c_int64(0)
    assert lib.orgym_invmgmt_codegen(C.byref(cfg), C.byref(rin), 0, None, 0, C.byref(need)) == _capi.E_UNSUPPORTED
    assert b"MLP" in lib.orgym_last_error()
