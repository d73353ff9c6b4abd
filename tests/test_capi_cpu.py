"""CPU suite: the C-ABI library loads and exports every symbol the header declares; host-side config logic
mirrors the reference's constructors; no compute call is made without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import or_gym_inventory_b200 as pkg
from or_gym_inventory_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_capi.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    return _capi.lib()


def test_header_symbols_are_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "orgym_b200.h")).read()
    names = set(re.findall(r"\b(orgym_[a-z0-9_]+)\s*\(", hdr))
    assert names, "no prototypes found"
    assert names == set(_capi.SYMBOLS), names ^ set(_capi.SYMBOLS)
    for n in names:
        assert hasattr(lib, n)
    assert lib.orgym_version() == 100


def test_no_gpu_fails_loudly(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert lib.orgym_device_count() == 0
    keep = []
    cfg = pkg.InvManagementParams().to_c(keep)
    h = C.c_void_p()
    rc = lib.orgym_invmgmt_create(C.byref(cfg), 16, 0, C.byref(h))
    assert rc == _capi.E_CUDA and b"no CUDA device" in lib.orgym_last_error()
    with pytest.raises(RuntimeError):
        pkg.InvManagementBacklogEnv(num_envs=4, device="cpu")


def test_invmgmt_params_mirror_reference_defaults():
    P = pkg.InvManagementParams()
    assert P.num_stages == 4 and P.lt_max == 10 and P.pipeline_length == 33
    assert P.unit_price.dtype == np.float32 and P.unit_price.tolist() == [20, 15, 10, 7]
    assert P.holding_cost.tolist() == [np.float32(0.15), np.float32(0.10), np.float32(0.05), 0]
    obs_space, act_space = P.spaces()
    assert obs_space.shape == (33,) and obs_space.dtype == np.int64
    assert act_space.high.tolist() == [100, 200, 230] and act_space.low.tolist() == [0, 0, 0]
    cap = (100 + 200 + 230) * 30 * 2
    assert obs_space.high[0] == cap and obs_space.low[0] == -cap
    # env_config overrides are applied after the keyword arguments (inventory_management.py:83-84)
    P2 = pkg.InvManagementParams(periods=10, env_config={"periods": 12, "L": [0, 0, 0]})
    assert P2.num_periods == 12 and P2.lt_max == 0 and P2.pipeline_length == 3


@pytest.mark.parametrize("bad, msg", [
    (dict(I0=[-1, 5, 5]), "Initial inventory"), (dict(periods=0), "periods"), (dict(c=[0, 1, 1]), "capacities"),
    (dict(L=[1, -2, 3]), "Lead times"), (dict(backlog=1), "boolean"), (dict(r=[1, 2, 3]), "Length of r"),
    (dict(dist=7), "dist must be"), (dict(alpha=0.0), "alpha"), (dict(dist=5, user_D=[1, 2]), "User specified"),
])
def test_invmgmt_validation_matches_reference(bad, msg):
    with pytest.raises(AssertionError, match=msg):
        pkg.InvManagementParams(**bad)


@pytest.mark.parametrize("kind", ["default", "custom", "yield"])
def test_network_kernel_specialiser_compiles_without_gpu(lib, kind):
    """The topology -> CUDA source generator (netinv_jit.cu) and NVRTC: compile check for sm_100a on the CPU box."""
    import json
    if kind == "yield":
        g = np.load(os.path.join(ROOT, "tests", "golden", "net_yield_backlog_random.npz"))
        meta = json.loads(str(g["meta"]))
        P = pkg.NetInvMgmtParams(graph=meta["graph"], num_periods=meta["num_periods"], backlog=True, alpha=meta["alpha"])
    else:
        P = pkg.NetInvMgmtParams(default_graph_kind=kind)
    keep = []
    cfg = P.to_c(keep)
    need = C.c_int64(0)
    buf = C.create_string_buffer(1 << 20)
    rc = lib.orgym_netinv_codegen(C.byref(cfg), 1, buf, len(buf), C.byref(need))
    assert rc == 0, lib.orgym_last_error()
    src = buf.value.decode()
    assert len(src) == need.value and "net_jit_step" in src and "net_jit_rollout" in src and f"#define NE {len(P.reorder_links)}" in src


def test_streaming_step_kernel_form_follows_node_order(lib, monkeypatch):
    """netinv_jit.cu: the streaming STEP kernel is generated as one pass over the nodes (no scratch rows) when every
    inventory-holding supplier has a larger node id than its purchasers -- the reference's numbering, market -> raw
    material -- and as two passes otherwise (the same network with the ids mirrored)."""
    import networkx as nx
    monkeypatch.setenv("ORGYM_NET_JIT_STREAM", "1")

    def form(P, compile_check=0):
        keep = []
        cfg = P.to_c(keep)
        need = C.c_int64(0)
        buf = C.create_string_buffer(8 << 20)
        rc = lib.orgym_netinv_codegen(C.byref(cfg), compile_check, buf, len(buf), C.byref(need))
        assert rc == 0, lib.orgym_last_error()
        src = buf.value.decode()
        assert "step_kernel_kind=stream" in src
        return "onepass" if "stream_form=onepass" in src else "twopass", src

    P = pkg.NetInvMgmtParams(default_graph_kind="default")
    f, src = form(P, 1)
    assert f == "onepass" and "sc_R[" not in src.split("net_jit_step(")[1].split("net_jit_rollout")[0].split("stream_form")[1].split("const int tn")[0]
    from or_gym_inventory_b200.network_management import default_graph
    g = default_graph()
    n = max(g.nodes)
    g2 = nx.relabel_nodes(g, {k: n - k for k in g.nodes}, copy=True)
    P2 = pkg.NetInvMgmtParams(graph=g2)
    f2, src2 = form(P2, 1)
    assert f2 == "twopass" and "sc_R[" in src2
    monkeypatch.setenv("ORGYM_NET_JIT_ONEPASS", "0")
    assert form(P)[0] == "twopass"


def test_large_graph_kernels_compile_without_gpu(lib):
    """BASELINE config 5's synthetic 64-node network: the generator picks the streaming STEP form on its own (graph
    size), in its single-pass variant, with the float32 ring copy for the observation kernel; NVRTC accepts the ~5600
    generated lines for sm_100a."""
    P = pkg.NetInvMgmtParams(graph=pkg.synthetic_graph(64), num_periods=30, backlog=False)
    keep = []
    cfg = P.to_c(keep)
    need = C.c_int64(0)
    buf = C.create_string_buffer(8 << 20)
    rc = lib.orgym_netinv_codegen(C.byref(cfg), 1, buf, len(buf), C.byref(need))
    assert rc == 0, lib.orgym_last_error()
    src = buf.value.decode()
    assert len(src) == need.value and f"#define NE {len(P.reorder_links)}" in src and len(P.reorder_links) == 88
    assert "step_kernel_kind=stream" in src and "stream_form=onepass" in src
    assert "float* const r32" in src and "__syncthreads();" in src.split("stream_form=onepass")[1].split("net_jit_rollout")[0]


@pytest.mark.parametrize("kind", ["default_lost", "default_backlog", "zero_lead", "binomial"])
def test_serial_rollout_specialiser_compiles_without_gpu(lib, kind):
    """invmgmt_jit.cu: configuration -> straight-line CUDA for the fused rollout -> NVRTC compile check for sm_100a."""
    cfgs = {"default_lost": dict(backlog=False), "default_backlog": dict(backlog=True),
            "zero_lead": dict(backlog=True, I0=[50, 60], r=[1.5, 1.0, 0.5], k=[0.1, 0.05, 0.02], h=[0.1, 0.05], c=[80, 70],
                              L=[0, 3], periods=12, alpha=0.9),
            "binomial": dict(backlog=False, dist=2, dist_param={"n": 30, "p": 0.4})}
    P = pkg.InvManagementParams(**cfgs[kind])
    keep = []
    cfg = P.to_c(keep)
    rnd = _capi.InvRolloutIn()
    rnd.policy = 2
    for rin, name in ((None, "inv_jit_rollout_bs"), (C.byref(rnd), "inv_jit_rollout_rnd")):
        need = C.c_int64(0)
        buf = C.create_string_buffer(1 << 20)
        rc = lib.orgym_invmgmt_codegen(C.byref(cfg), rin, 1, buf, len(buf), C.byref(need))
        assert rc == 0, lib.orgym_last_error()
        src = buf.value.decode()
        assert len(src) == need.value and name in src
        if name.endswith("_bs"):       # straight-line periods (the compiler folds the demand-independent stages)
            assert src.count("// ---- period") == P.num_periods
        else:                          # random policy: a loop over blocks of periods + a straight-line tail
            import re as _re
            m = _re.search(r"for \(int tb = 0; tb < (\d+); tb \+= (\d+)\)", src)
            assert m, "the random-policy kernel should loop over blocks of periods"
            tloop, unr = int(m.group(1)), int(m.group(2))
            assert tloop == P.num_periods - P.num_periods % unr and unr == (8 if P.num_periods >= 16 else 4)
            assert src.count("// ---- period") == unr + P.num_periods - tloop


def test_serial_rollout_specialiser_reports_unsupported_configs(lib):
    P = pkg.InvManagementParams(backlog=True, I0=[10] * 7, r=[9, 8, 7, 6, 5, 4, 3, 2], k=[0.1] * 8, h=[0.1] * 7, c=[10] * 7,
                                L=[1] * 7)
    keep = []
    cfg = P.to_c(keep)
    need = C.c_int64(0)
    rc = lib.orgym_invmgmt_codegen(C.byref(cfg), None, 0, None, 0, C.byref(need))
    assert rc == -3 and b"specialiser" in lib.orgym_last_error()


def test_header_is_plain_c_and_matches_the_ctypes_mirror(tmp_path):
    """include/orgym_b200.h must compile as C99 (it is the drop-in boundary for any host language), and every struct of
    the Python host's ctypes mirror must have the size and field offsets the C compiler gives the header's struct."""
    import subprocess
    from or_gym_inventory_b200 import _capi
    pairs = [("orgym_dist_t", _capi.Dist), ("orgym_invmgmt_config_t", _capi.InvConfig), ("orgym_invmgmt_info_t", _capi.InvInfo),
             ("orgym_invmgmt_rollout_in_t", _capi.InvRolloutIn), ("orgym_invmgmt_rollout_out_t", _capi.InvRolloutOut),
             ("orgym_newsvendor_config_t", _capi.NvConfig), ("orgym_newsvendor_info_t", _capi.NvInfo),
             ("orgym_newsvendor_rollout_in_t", _capi.NvRolloutIn), ("orgym_newsvendor_rollout_out_t", _capi.NvRolloutOut),
             ("orgym_netinv_config_t", _capi.NetConfig), ("orgym_netinv_info_t", _capi.NetInfo),
             ("orgym_netinv_rollout_in_t", _capi.NetRolloutIn), ("orgym_netinv_rollout_out_t", _capi.NetRolloutOut)]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "orgym_b200.h"', 'int main(void) {']
    for cname, _ in pairs:
        src.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
    src.append('  return 0; }')
    c = tmp_path / "abi.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)])
    sizes = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for cname, cls in pairs:
        assert int(sizes[cname]) == C.sizeof(cls), (cname, sizes[cname], C.sizeof(cls))
    # field order / count: the last field of every mirror sits where the C struct ends (modulo tail padding <= 8)
    for cname, cls in pairs:
        last = cls._fields_[-1][0]
        end = getattr(cls, last).offset + getattr(cls, last).size
        assert 0 <= int(sizes[cname]) - end < 8, cname


def _build_c_host(tmp_path):
    import subprocess
    exe = tmp_path / "c_host"
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", f"{cuda}/include",
                           os.path.join(ROOT, "examples", "c_host.c"), "-L", os.path.join(ROOT, "or-gym-inventory_b200", "csrc"),
                           "-lorgym_b200", "-L", f"{cuda}/lib64", "-lcudart", "-lm", "-o", str(exe)])
    env = dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join(
        [os.path.join(ROOT, "or-gym-inventory_b200", "csrc"), f"{cuda}/lib64", os.environ.get("LD_LIBRARY_PATH", "")]))
    return exe, env


def test_c_host_example_builds_and_fails_loudly_without_a_gpu(lib, tmp_path):
    """examples/c_host.c drives the library from plain C (no Python, no torch); without a device it must say so."""
    import subprocess
    import torch
    exe, env = _build_c_host(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked run of the example")
    p = subprocess.run([str(exe)], env=env, capture_output=True, text=True)
    assert p.returncode == 2 and "no CUDA device" in p.stderr


@pytest.mark.gpu
def test_c_host_example_matches_the_python_host(lib, tmp_path):
    import re
    import subprocess
    exe, env = _build_c_host(tmp_path)
    p = subprocess.run([str(exe)], env=env, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    m = re.search(r"rollout,\s+base-stock SF=1.0:\s+mean episode return ([-0-9.]+) over 4096", p.stdout)
    s = re.search(r"step API,\s+constant order 20: mean episode return ([-0-9.]+) over 4096", p.stdout)
    assert m and s, p.stdout
    e = pkg.InvManagementBacklogEnv(num_envs=4096, device="cuda:0")
    out = e.rollout("base_stock", seed=4000, safety_factor=1.0, want=("ep_return", "summary"))
    assert abs(out["ep_return"].mean().item() - float(m.group(1))) < 1e-3
    import torch
    e.reset(seed=4000)
    a = torch.full((4096, 3), 20, dtype=torch.int64, device="cuda")
    tot = 0.0
    for _ in range(e.num_periods):
        tot += e.step(a)[1].sum().item()
    assert abs(tot / 4096 - float(s.group(1))) < 1e-3
    e.close()


def test_serial_rollout_specialiser_uses_integer_profit_only_when_provably_exact_and_scalable(lib):
    """Defaults: float32 coefficients on a 2^-29 grid and small integers -> no float64 operation of the reference's profit
    can round -> the generator emits integer multiply-adds on coefficient / 2^-29 (and, the rewards being undiscounted
    and the 30-period running sum exact as well, converts once per episode).  With discounting: one conversion per
    period.  A discount so small that alpha**29 * 2^-29 is below the generator's 1e-290 guard keeps the exact profit
    but not the integer scaling: one fused multiply-add chain.  Capacities of a million push the bound past
    2^52 * quantum -> it must keep the reference's operation order (4 products + 3 subtractions per stage, sequential
    sum)."""
    rin = None

    def source(backlog=True, **kw):
        P = pkg.InvManagementParams(backlog=backlog, **kw)
        keep = []
        cfg = P.to_c(keep)
        need = C.c_int64(0)
        buf = C.create_string_buffer(4 << 20)
        assert lib.orgym_invmgmt_codegen(C.byref(cfg), rin, 0, buf, len(buf), C.byref(need)) == 0, lib.orgym_last_error()
        return buf.value.decode()
    exact = source(backlog=False, alpha=1.0)
    assert "long long acc = 0;" in exact and "pa -= 13421773LL * (long long)(U_3);" in exact      # 0.025f = 13421773 * 2^-29
    assert "pa += 536870912LL * (long long)(5 * (s0 + r_0));" in exact                             # (20 - 15) * 2^29 in two steps
    assert "fma(" not in exact and "tm_0" not in exact and "ret = (double)acc * 0x1p-29;" in exact
    disc = source()                                                                                # default alpha = 0.97
    assert "long long acc" not in disc and "(__longlong_as_double(pa + 0x4338000000000000LL) - 0x1.8p52);" in disc
    assert "tm_0" not in disc
    fused = source(alpha=1e-10)
    assert "fma(" in fused and "tm_0" not in fused and "long long pa" not in fused
    big = source(c=[1_000_000, 2_000_000, 2_300_000])
    assert "fma(" not in big and "long long pa" not in big and "tm_0" in big and "pr = pr + tm_3;" in big


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` runs without a GPU (it times the C port of the reference loop on the host cores) and
    prints exactly one JSON line with the keys the driver reads."""
    import json
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 1e5 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_product_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: on a box without a CUDA device the product arm must stop with a clear message, not time the CPU."""
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "CUDA device" in (p.stderr + p.stdout) and not p.stdout.strip().startswith("{")


def test_geometric_demand_with_a_long_tail_is_refused_not_truncated(lib):
    """numpy's geometric has unbounded support; the 4096-entry alias table covers it only for p >= ~0.0107.  Below
    that the library must return ORGYM_E_UNSUPPORTED instead of cutting the tail and renormalising (which would bias
    the mean well below 1/p)."""
    def bounds(p):
        P = pkg.InvManagementParams(dist=4, dist_param={"p": p})
        keep = []
        cfg = P.to_c(keep)
        xv, xs = C.c_double(0), C.c_double(0)
        return lib.orgym_invmgmt_value_bounds(C.byref(cfg), C.byref(xv), C.byref(xs), None)
    assert bounds(0.12) == 0 and bounds(0.011) == 0
    assert bounds(0.01) == _capi.E_UNSUPPORTED and b"geometric" in lib.orgym_last_error()
    assert bounds(0.001) == _capi.E_UNSUPPORTED


def test_new_entry_points_reject_bad_handles_without_a_gpu(lib):
    """specialise / scratch-size / report entry points: argument checking works on a box without a GPU."""
    rin = _capi.InvRolloutIn()
    assert lib.orgym_invmgmt_specialise(None, C.byref(rin)) == _capi.E_INVALID
    assert lib.orgym_invmgmt_rollout_scratch_bytes(None) == -1
    assert lib.orgym_report_scratch_bytes(1 << 24) > (1 << 20) and lib.orgym_report_scratch_bytes(-1) == -1
    assert lib.orgym_evaluation_report(0, None, None, 0, 10, 30, None, None, None) == _capi.E_INVALID
