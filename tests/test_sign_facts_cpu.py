"""CPU suite: the sign facts behind the serial-env specialiser's dropped clamps.  Where inv_value_bounds proves that a
stage's on-hand inventory is never negative after a period, the generated kernel uses the value itself instead of
max(value, 0) in the holding cost and the inventory statistic.  Each such fact is checked here against brute-force
simulation with the oracle, and the stages whose on-hand does go negative must keep the clamp."""
import ctypes as C
import re

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from or_gym_inventory_b200 import _capi
from oracle import oracle


def _source(P, policy=None):
    keep = []
    cfg = P.to_c(keep)
    rin = None
    if policy is not None:
        r = _capi.InvRolloutIn()
        r.policy = policy
        rin = C.byref(r)
    need = C.c_int64(0)
    buf = C.create_string_buffer(4 << 20)
    lib = _capi.lib()
    assert lib.orgym_invmgmt_codegen(C.byref(cfg), rin, 0, buf, len(buf), C.byref(need)) == 0, lib.orgym_last_error()
    return buf.value.decode()


def _unclamped(src, n):
    """stages whose on-hand enters the inventory statistic without the clamp"""
    got = dict(re.findall(r"I_(\d+) = Ic_\d+; s_inv \+= (.*?);", src))
    assert sorted(int(j) for j in got) == list(range(n))
    return {int(j) for j, x in got.items() if x == f"Ic_{j}"}


def test_base_stock_defaults_drop_only_the_retailers_clamp():
    """Defaults (lead times 3, 5, 10): upstream on-hand can go negative (a stage subtracts its own inbound order), the
    retailer's cannot (it keeps max(on-hand - demand - backlog, 0)).  Under base-stock the retailer's terms and the
    upstream stages' terms are merged separately, and discount factors come from the constant table."""
    for backlog in (False, True):
        src = _source(pkg.InvManagementParams(backlog=backlog))
        assert _unclamped(src, 3) == {0}
        assert "pa -= 80530640LL * (long long)(Ic_0);" in src                        # 0.15 / 2^-29, no clamp
        assert "pa -= 53687092LL * (long long)(U_0);" in src                         # not merged with stage 1's holding
        assert "pa -= 53687092LL * (long long)((Ic_1 > 0 ? Ic_1 : 0));" in src
        assert "ret += c_disc[29] * (" in src and "0x1.b7abfc78b016bp-30 *" not in src


@pytest.mark.parametrize("case", range(24))
def test_sign_facts_hold_under_brute_force(case):
    rng = np.random.default_rng(9100 + case)
    n = int(rng.integers(1, 7))
    T = int(rng.integers(3, 41))
    c = rng.integers(1, 60, n)
    L = rng.integers(0, 7, n)
    while L.sum() > 40:
        L[int(np.argmax(L))] -= 1
    I0 = np.where(rng.random(n) < 0.5, rng.integers(0, 100, n), L * c + rng.integers(0, 20, n))   # half with a proof
    cfg = dict(periods=T, I0=I0.tolist(), p=30.0, r=np.sort(rng.uniform(0.5, 25, n + 1))[::-1].round(2).tolist(),
               k=rng.uniform(0, 1, n + 1).round(2).tolist(), h=rng.uniform(0, 0.5, n).round(2).tolist(), c=c.tolist(),
               L=L.tolist(), dist_param={"mu": float(rng.integers(1, 80))})
    P = pkg.InvManagementParams(backlog=bool(case % 2), **cfg)
    facts = _unclamped(_source(P, policy=2), n)                                    # random-policy kernel
    assert 0 in facts
    patterns = [rng.integers(0, c + 1, size=(T, n)) for _ in range(6)]
    patterns += [np.tile(c, (T, 1)), np.zeros((T, n), np.int64),
                 np.where((np.arange(T)[:, None] // 3) % 2 == 0, c, 0),
                 np.where(np.arange(n)[None, :] % 2 == 0, c, 0) * np.ones((T, 1), np.int64)]
    lowest = np.full(n, np.inf)
    for a in patterns:
        dem = rng.poisson(cfg["dist_param"]["mu"], size=T).astype(np.int64)
        if rng.random() < 0.3:
            dem[:] = 0
        o = oracle.invmgmt_episode(P, actions=a.astype(np.float64), demand=dem)
        lowest = np.minimum(lowest, o["I"][1:].min(axis=0))
    for j in facts:
        assert lowest[j] >= 0, (j, lowest, cfg)
    # upstream: the fact is the telescoping bound I0_j - min(L_j, T) * c_j >= 0, whatever the backlog mode
    assert facts == {0} | {j for j in range(1, n) if I0[j] - min(L[j], T) * c[j] >= 0}
