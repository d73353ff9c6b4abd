"""Shared helpers for the parity tests."""
import glob
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def golden_files(prefix):
    return sorted(glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def load_golden(path):
    g = np.load(path)
    meta = json.loads(str(g["meta"]))
    return g, meta


def ids(paths):
    return [os.path.basename(p)[:-4] for p in paths]


def seq_sum(x):
    """Python's `total += reward` accumulation order."""
    s = 0.0
    for v in np.asarray(x).tolist():
        s += v
    return s


def net_kwargs(meta):
    """Constructor keywords of a golden network case (graph spec + flags recorded by make_golden.py; user_D /
    sample_path are stored as [u, v, value] triples because JSON has no tuple keys)."""
    kw = dict(graph=meta["graph"], num_periods=meta["num_periods"], backlog=meta["backlog"], alpha=meta["alpha"])
    if "user_D" in meta:
        kw["user_D"] = {(u, v): list(tr) for u, v, tr in meta["user_D"]}
        kw["sample_path"] = {(u, v): bool(sp) for u, v, sp in meta.get("sample_path", [])}
    return kw


def net_params(meta, pkg):
    """NetInvMgmtParams for a golden network case."""
    return pkg.NetInvMgmtParams(**net_kwargs(meta))


def set_net_kernel_mode(monkeypatch, mode):
    """Route the network envs created next through one kernel path: "generic" (constant-bank interpreter),
    "specialised" (NVRTC, register-resident), or the streaming STEP form forced on a small graph -- "stream_jit"
    (single pass + observation kernel), "stream_jit_twopass" (two passes with scratch rows), "stream_jit_fused_obs"
    (the kernel's own observation pass)."""
    monkeypatch.setenv("ORGYM_NET_JIT", "0" if mode == "generic" else "2")
    monkeypatch.setenv("ORGYM_NET_JIT_STREAM", "1" if mode.startswith("stream") else "0")
    monkeypatch.setenv("ORGYM_NET_OBS_TMA", "0" if mode == "stream_jit_fused_obs" else "1")
    monkeypatch.setenv("ORGYM_NET_JIT_ONEPASS", "0" if mode == "stream_jit_twopass" else "1")


def net_S_columns(meta):
    """The reference's S frame is ordered by sorted network_links; ours is reorder links then retail links."""
    nl = [tuple(x) for x in meta["network_links"]]
    re = [tuple(x) for x in meta["reorder_links"]]
    rt = [tuple(x) for x in meta["retail_links"]]
    return [nl.index(e) for e in re] + [nl.index(e) for e in rt]


# ---- independent numpy restatement of the device's counter-based streams (csrc/device_rng.cuh) ----------------------
def philox4x32_10(c, k0, k1):
    """Philox4x32-10 over arrays: c = (c0, c1, c2, c3) uint32 arrays, key words k0, k1 uint32 arrays."""
    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
    c0, c1, c2, c3 = (np.asarray(x, np.uint32).copy() for x in c)
    k0, k1 = np.asarray(k0, np.uint32).copy(), np.asarray(k1, np.uint32).copy()
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = M0 * c0.astype(np.uint64)
        p1 = M1 * c2.astype(np.uint64)
        hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & m32).astype(np.uint32)
        hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & m32).astype(np.uint32)
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0.astype(np.uint64) + np.uint64(W0)).astype(np.uint32)
        k1 = (k1.astype(np.uint64) + np.uint64(W1)).astype(np.uint32)
    return c0, c1, c2, c3


def device_random_actions(seed, env_ids, episode, T, capacity):
    """The on-device random-action policy of the serial env (STREAM_ACTION = 1): action of (env, period t, stage i) =
    mulhi(word i%4 of Philox(key=seed+env, counter=(t, episode, 1, i//4)), c_i + 1), i.e. uniform on {0..c_i}."""
    env_ids = np.asarray(env_ids, np.uint64)
    key = np.uint64(seed) + env_ids
    n = len(capacity)
    out = np.zeros((len(env_ids), T, n), np.int64)
    for t in range(T):
        for grp in range((n + 3) // 4):
            z = np.zeros(len(env_ids), np.uint32)
            w = philox4x32_10((z + np.uint32(t), z + np.uint32(episode), z + np.uint32(1), z + np.uint32(grp)),
                              (key & np.uint64(0xFFFFFFFF)).astype(np.uint32), (key >> np.uint64(32)).astype(np.uint32))
            for i in range(4 * grp, min(n, 4 * grp + 4)):
                out[:, t, i] = ((w[i & 3].astype(np.uint64) * np.uint64(int(capacity[i]) + 1)) >> np.uint64(32)).astype(np.int64)
    return out
