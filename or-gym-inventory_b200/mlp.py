"""Actor networks evaluated inside the fused rollouts (orgym_mlp_t): which torch modules qualify and how they are packed.

Shared by the serial env (InvManagement*Env.rollout / evaluate), the newsvendor (NewsvendorEnv.rollout / evaluate) and
the network env (NetInvMgmt*Env.rollout / evaluate)."""
from . import _capi
from ._capi import MLP_RELU, MLP_TANH


def mlp_layers(policy):
    """The Linear layers and the activation of an actor network, in evaluation order: (linears, activation code).

    Accepted: a `torch.nn.Sequential` of the form Linear, act, Linear, act, ..., Linear with one activation type (Tanh or
    ReLU) throughout, or a stable-baselines3 `ActorCriticPolicy`-shaped object (duck-typed: `.mlp_extractor.policy_net`, a
    Sequential ending in its activation, followed by `.action_net`, a Linear) without output squashing and with a flatten
    features extractor -- SB3's deterministic `predict` for a Box action space.  Anything else raises ValueError naming
    the offending layer or attribute."""
    import torch.nn as nn
    if isinstance(policy, nn.Sequential):
        mods, where = list(policy), "Sequential"
    elif hasattr(policy, "mlp_extractor") and hasattr(policy, "action_net"):
        if getattr(policy, "squash_output", False):
            raise ValueError("policy.squash_output is True: a tanh-squashed action is not the clipped Gaussian mean "
                             "the device evaluates")
        fe = getattr(policy, "features_extractor", None)
        if fe is not None and not (isinstance(fe, nn.Flatten) or type(fe).__name__ == "FlattenExtractor"):
            raise ValueError(f"policy.features_extractor is {type(fe).__name__}, only a flatten is supported")
        pn = getattr(policy.mlp_extractor, "policy_net", None)
        if not isinstance(pn, nn.Sequential):
            raise ValueError("policy.mlp_extractor.policy_net is not a torch.nn.Sequential")
        if not isinstance(policy.action_net, nn.Linear):
            raise ValueError(f"policy.action_net is {type(policy.action_net).__name__}, not a Linear")
        mods, where = list(pn) + [policy.action_net], "policy_net + action_net"
    else:
        raise ValueError(f"policy {type(policy).__name__!r} is neither a policy name, a torch.nn.Sequential nor an "
                         "SB3 ActorCriticPolicy")
    acts = {nn.Tanh: MLP_TANH, nn.ReLU: MLP_RELU}
    linears, act = [], None
    for i, mod in enumerate(mods):
        want_linear = i % 2 == 0
        if want_linear and not isinstance(mod, nn.Linear):
            raise ValueError(f"{where}[{i}] is {type(mod).__name__}, expected Linear")
        if not want_linear:
            if type(mod) not in acts:
                raise ValueError(f"{where}[{i}] is {type(mod).__name__}, expected Tanh or ReLU")
            if act is not None and acts[type(mod)] != act:
                raise ValueError(f"{where}[{i}] is {type(mod).__name__}: one activation type throughout")
            act = acts[type(mod)]
        if want_linear:
            linears.append(mod)
    if not mods or not isinstance(mods[-1], nn.Linear):
        raise ValueError(f"{where} must end with a Linear (no activation after the last layer)")
    if len(linears) > _capi.MLP_MAX_LAYERS:
        raise ValueError(f"{where} has {len(linears)} Linear layers, at most {_capi.MLP_MAX_LAYERS} are supported")
    for i in range(1, len(linears)):
        if linears[i].in_features != linears[i - 1].out_features:
            raise ValueError(f"{where}: Linear {i} has in_features {linears[i].in_features}, the layer before has "
                             f"out_features {linears[i - 1].out_features}")
    return linears, (act if act is not None else MLP_TANH)


def pack_mlp(policy, obs_dim, act_dim, device):
    """orgym_mlp_t for `policy` (see mlp_layers) with the current weights, plus the tensors it points into (keep them
    alive until the rollout is enqueued).  Weights are detached, cast to float32, moved to `device` and made contiguous
    with device-side torch ops: no host synchronisation, so a network being trained is evaluated as it is now."""
    linears, act = mlp_layers(policy)
    if linears[0].in_features != obs_dim:
        raise ValueError(f"first Linear has in_features {linears[0].in_features}, the observation has {obs_dim}")
    if linears[-1].out_features != act_dim:
        raise ValueError(f"last Linear has out_features {linears[-1].out_features}, the action has {act_dim}")
    import torch
    m = _capi.Mlp()
    m.num_layers, m.activation = len(linears), act
    m.width[0] = obs_dim
    keep = []
    for l, lin in enumerate(linears):
        m.width[l + 1] = lin.out_features
        w = lin.weight.detach().to(device=device, dtype=torch.float32).contiguous()
        keep.append(w)
        m.weight[l] = w.data_ptr()
        if lin.bias is not None:
            b = lin.bias.detach().to(device=device, dtype=torch.float32).contiguous()
            keep.append(b)
            m.bias[l] = b.data_ptr()
    return m, keep
