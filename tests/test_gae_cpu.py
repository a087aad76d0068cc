"""GAE advantages and value targets of a rollout (include/ppg.h ppg_gae) on the CPU: a numpy float32 reference of the
kernel's link rule and recursion, fed the C oracle's outputs, checked against an independent float64 formulation (textbook
backward GAE per agent life), against the edge cases lambda = 0 and gamma = lambda = 1 with V = 0 (cross-checked with the
episode-returns tracker), and for the count identity of the links; and the SASS of the kernel.  tests/test_gpu_gae.py
compares the device with this reference bit for bit."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from predpreygrass_b200.config import BASE_CONFIG, STAG_CONFIG, VARIANT_STAG, make_config
from tests.test_returns_cpu import CONSERVATION_CASES, REUSE_CONFIG, Tracker

TERM, TRUNC, NEWBORN, FOUNDER = 0x01, 0x02, 0x04, 0x08
ENV_TERM, ENV_TRUNC, ENV_RESET, ENV_IDLE = 0x01, 0x02, 0x04, 0x08
COLS = ("row_env", "row_agent", "flags", "reward", "old_off", "new_off", "new_cnt")


def snapshot(out):
    """the columns of one output the rollout keeps (copies: the oracle's views change with the next call)"""
    snap = {k: out[k] for k in ("n", "n_old")}
    for s in range(2):
        for c in COLS:
            snap[f"{c}{s}"] = np.array(out[f"{c}{s}"])
    snap["env_flags"] = np.array(out["env_flags"])
    return snap


def synth_values(out, t):
    """a fixed hash of (env, id, t) mapped to fp32 values in [-2, 2): identical on both backends"""
    vals = []
    for s in range(2):
        n = out["n"][s]
        h = (out[f"row_env{s}"][:n].astype(np.uint64) * np.uint64(0x9E3779B1) + out[f"row_agent{s}"][:n].astype(np.uint64)
             * np.uint64(0x85EBCA6B) + np.uint64(t) * np.uint64(0xC2B2AE35) + np.uint64(s)) & np.uint64(0xFFFFFFFF)
        h ^= h >> np.uint64(15)
        h = (h * np.uint64(0x2C1B3C6D)) & np.uint64(0xFFFFFFFF)
        h ^= h >> np.uint64(12)
        vals.append(((h >> np.uint64(8)).astype(np.float64) / 2.0 ** 24 * 4.0 - 2.0).astype(np.float32))
    return vals


def oracle_rollout(cfg, n_envs, T, *, preroll=0, mask_at=None, action_seed=7, track=False):
    """T+1 outputs of the oracle stepped with its Philox random actions after `preroll` steps from the reset; every third env's
    reset scheduled before step `mask_at` of the rollout.  With track, also the tracker's row_return of every output."""
    from oracle.oracle import Oracle

    ora = Oracle(cfg, n_envs, threads=4)
    tr = Tracker(n_envs, cfg.n_possible) if track else None
    outs, rets = [], []
    try:
        out = ora.reset()
        if track:
            tr.update(out)
        for t in range(-preroll, T + 1):
            if t >= 0:
                outs.append(snapshot(out))
                if track:
                    rets.append([tr.row_return[s].copy() for s in range(2)])
            if t == T:
                break
            if t == mask_at:
                ora.reset(mask=(np.arange(n_envs) % 3 == 0).astype(np.uint8))
            a0, a1 = ora.random_actions(action_seed)
            A0 = np.zeros(max(1, len(a0)), np.int32); A0[: len(a0)] = a0
            A1 = np.zeros(max(1, len(a1)), np.int32); A1[: len(a1)] = a1
            out = ora.step(A0, A1)
            if track:
                tr.update(out)
        return (outs, rets) if track else outs
    finally:
        ora.close()


def _end_of_life(f1, ef1):
    """terminal / truncated of successor rows with row flags f1 and env flags ef1 (include/ppg.h)"""
    term = ((f1 & TERM) != 0) | (((ef1 & ENV_TERM) != 0) & ((f1 & TRUNC) == 0))
    trunc = ~term & (((f1 & TRUNC) != 0) | ((ef1 & ENV_TRUNC) != 0))
    return term, trunc


def gae_reference(outputs, values, gamma, lam):
    """numpy float32 model of ppg_gae_kernel: per species lists over t < T of adv, value_target (float32 [n_t]) and next_row
    (int32 [n_t]).  The links come from a map keyed by (env, id) of the old, non-FOUNDER rows of output t+1; the recursion
    repeats the kernel's expressions one fp32 operation at a time."""
    T = len(outputs) - 1
    g = np.float32(gamma)
    gl = np.float32(g * np.float32(lam))
    res = []
    for s in range(2):
        adv, vt, nxt = [None] * T, [None] * T, [None] * T
        for t in range(T - 1, -1, -1):
            o, o1 = outputs[t], outputs[t + 1]
            n, n1, n1_old = o["n"][s], o1["n"][s], o1["n_old"][s]
            env1, id1, f1 = o1[f"row_env{s}"][:n1], o1[f"row_agent{s}"][:n1], o1[f"flags{s}"][:n1]
            succ = {(int(env1[r]), int(id1[r])): r for r in range(n1_old) if not f1[r] & (FOUNDER | NEWBORN)}
            env0, id0, f0 = o[f"row_env{s}"][:n], o[f"row_agent{s}"][:n], o[f"flags{s}"][:n]
            ef1 = o1["env_flags"]
            rn = np.array([succ.get((int(e), int(i)), -1) for e, i in zip(env0, id0)], np.int32).reshape(-1)
            rn[((f0 & (TERM | TRUNC)) != 0) | ((ef1[env0] & (ENV_RESET | ENV_IDLE)) != 0)] = -1
            a, v = np.full(n, np.nan, np.float32), np.full(n, np.nan, np.float32)
            k = rn >= 0
            r1 = rn[k]
            term, trunc = _end_of_life(f1[r1], ef1[env0[k]])
            vn = np.where(term, np.float32(0), values[t + 1][s][r1]).astype(np.float32)
            cont = ~term & ~trunc
            if t + 1 < T:
                cont &= nxt[t + 1][r1] >= 0
                an = np.where(cont, adv[t + 1][r1], np.float32(0)).astype(np.float32)
            else:
                an = np.zeros(len(r1), np.float32)
            v0 = values[t][s][:n][k]
            delta = (o1[f"reward{s}"][r1] + g * vn) - v0
            a[k] = delta + gl * an
            v[k] = a[k] + v0
            adv[t], vt[t], nxt[t] = a, v, rn
        res.append({"adv": adv, "value_target": vt, "next_row": nxt})
    return res


def life_sequences(outputs, s):
    """the rows of species s split into per-(env, id, life) sequences of (t, row), from the row flags alone (no links): a
    FOUNDER or NEWBORN row (and every row of output 0) starts a life, an old row continues the life of the live row of the same (env, id) in the output
    before, a TERMINATED or TRUNCATED row ends it, and a life whose next output has no row of it (a reset env, an idle env,
    the end of the rollout) ends at its last row"""
    live, seqs = {}, []
    for t, o in enumerate(outputs):
        n, n_old = o["n"][s], o["n_old"][s]
        env, ids, f = o[f"row_env{s}"][:n], o[f"row_agent{s}"][:n], o[f"flags{s}"][:n]
        nxt = {}
        for r in range(n):
            key = (int(env[r]), int(ids[r]))
            if t == 0 or r >= n_old or f[r] & (FOUNDER | NEWBORN):  # output 0 may be mid-episode
                seq = [(t, r)]
                seqs.append(seq)
            else:
                assert key in live, (t, s, key)  # an old row has its predecessor
                seq = live.pop(key)
                seq.append((t, r))
            if not f[r] & (TERM | TRUNC):
                nxt[key] = seq
        live = nxt
    return [q for q in seqs if len(q) > 1]


def textbook_gae(outputs, values, s, gamma, lam):
    """float64 backward GAE per life sequence: A_k = delta_k + gamma * lambda * A_{k+1} inside a sequence, the last
    transition bootstraps from V unless its successor is terminal.  -> {(t, r): (adv, value_target)}"""
    out = {}
    for seq in life_sequences(outputs, s):
        A = 0.0
        for k in range(len(seq) - 2, -1, -1):
            (t, r), (t1, r1) = seq[k], seq[k + 1]
            o1 = outputs[t1]
            term, trunc = _end_of_life(o1[f"flags{s}"][r1:r1 + 1], o1["env_flags"][o1[f"row_env{s}"][r1:r1 + 1]])
            last = k == len(seq) - 2
            vn = 0.0 if term[0] else float(values[t1][s][r1])
            delta = float(o1[f"reward{s}"][r1]) + gamma * vn - float(values[t][s][r])
            A = delta + (0.0 if last else gamma * lam * A)
            out[(t, r)] = (A, A + float(values[t][s][r]))
    return out


def _case(name):
    base = lambda **kw: make_config(dict(BASE_CONFIG, **kw), cap_live=(64, 192), seed=3)  # noqa: E731
    stag = lambda strict: make_config(dict(STAG_CONFIG, max_steps=70, n_initial_active_type_1_predator=2,  # noqa: E731
                                           strict_rllib_output=strict), variant=VARIANT_STAG, cap_live=(64, 192), seed=6)
    return {
        "base_truncation": lambda: (base(max_steps=25), 48, 60, {}),
        "base_extinction": lambda: (base(max_steps=100, n_initial_active_predator=2, n_initial_active_prey=3), 48, 80, {}),
        "eco_crowded": lambda: (CONSERVATION_CASES["eco_crowded"](), 48, 70, {}),
        "eco_pool_exhausted": lambda: (REUSE_CONFIG(), 64, 90, {}),
        "stag_strict": lambda: (stag(True), 48, 100, {}),
        "stag_not_strict": lambda: (stag(False), 48, 100, {}),
        "base_masked_reset": lambda: (base(max_steps=40), 48, 40, {"preroll": 5, "mask_at": 12}),
        "base_autoreset_off": lambda: (make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=3, autoreset=False),
                                       48, 40, {}),
    }[name]()


CASES = ["base_truncation", "base_extinction", "eco_crowded", "eco_pool_exhausted", "stag_strict", "stag_not_strict",
         "base_masked_reset", "base_autoreset_off"]


def ends_seen(outputs, ref):
    """(terminal, truncated, extinction survivors unflagged, extinction survivors flagged TRUNCATED) among the transitions"""
    seen = np.zeros(4, np.int64)
    for s in range(2):
        for t in range(len(outputs) - 1):
            rn = ref[s]["next_row"][t]
            r1 = rn[rn >= 0]
            o1 = outputs[t + 1]
            f1, ef1 = o1[f"flags{s}"][r1], o1["env_flags"][o1[f"row_env{s}"][r1]]
            term, trunc = _end_of_life(f1, ef1)
            ext = (ef1 & ENV_TERM) != 0
            seen += [term.sum(), trunc.sum(), (ext & ((f1 & (TERM | TRUNC)) == 0)).sum(), (ext & ((f1 & TRUNC) != 0)).sum()]
    return seen


@pytest.mark.parametrize("case", CASES)
def test_reference_matches_textbook_gae_per_life(case):
    cfg, B, T, kw = _case(case)
    outputs = oracle_rollout(cfg, B, T, **kw)
    values = [synth_values(o, t) for t, o in enumerate(outputs)]
    gamma, lam = 0.99, 0.95
    ref = gae_reference(outputs, values, gamma, lam)
    n_tr = 0
    for s in range(2):
        want = textbook_gae(outputs, values, s, gamma, lam)
        linked = [(t, int(r)) for t in range(T) for r in np.nonzero(ref[s]["next_row"][t] >= 0)[0]]
        assert sorted(want) == sorted(linked), (case, s)  # the reference's links are exactly the lives' transitions
        succ = {seq[k]: seq[k + 1][1] for seq in life_sequences(outputs, s) for k in range(len(seq) - 1)}
        assert all(int(ref[s]["next_row"][t][r]) == succ[(t, r)] for t, r in linked), (case, s)
        got = np.array([[ref[s]["adv"][t][r], ref[s]["value_target"][t][r]] for t, r in linked], np.float64).reshape(-1, 2)
        exp = np.array([want[k] for k in linked], np.float64).reshape(-1, 2)
        assert np.allclose(got, exp, rtol=1e-5, atol=1e-5), (case, s, np.abs(got - exp).max())
        for t in range(T):  # rows without a successor: NaN
            k = ref[s]["next_row"][t] < 0
            assert np.isnan(ref[s]["adv"][t][k]).all() and np.isnan(ref[s]["value_target"][t][k]).all()
        n_tr += len(linked)
    assert n_tr > 1000, n_tr
    term, trunc, unflagged, flagged_trunc = ends_seen(outputs, ref)
    assert term > 0, case
    flags = np.bitwise_or.reduce([int(np.bitwise_or.reduce(o["env_flags"])) for o in outputs])
    if case == "base_extinction":
        assert flags & ENV_TERM and unflagged > 0  # survivors of an extinction, unflagged: terminal transitions
    if case.startswith("stag"):
        assert flags & ENV_TERM and flagged_trunc > 0 and trunc > 0  # STAG flags them TRUNCATED: they bootstrap
    if case in ("base_truncation", "eco_pool_exhausted"):
        assert flags & ENV_TRUNC and trunc > 0
    if case == "base_masked_reset":
        assert any(o["env_flags"][0] & ENV_RESET for o in outputs[1:])
    if case == "base_autoreset_off":
        assert flags & ENV_IDLE


@pytest.mark.parametrize("case", ["base_truncation", "eco_crowded", "stag_strict", "base_masked_reset", "base_autoreset_off"])
def test_count_identity(case):
    """in every output t+1, the rows of output t with a successor are as many as the old, non-FOUNDER rows of t+1"""
    cfg, B, T, kw = _case(case)
    outputs = oracle_rollout(cfg, B, T, **kw)
    ref = gae_reference(outputs, [synth_values(o, t) for t, o in enumerate(outputs)], 0.9, 0.8)
    for s in range(2):
        for t in range(T):
            o1 = outputs[t + 1]
            old = o1[f"flags{s}"][: o1["n_old"][s]]
            assert int((ref[s]["next_row"][t] >= 0).sum()) == int(((old & FOUNDER) == 0).sum()), (case, s, t)


def test_lambda_zero_is_the_one_step_td_error():
    cfg, B, T, kw = _case("base_truncation")
    outputs = oracle_rollout(cfg, B, T, **kw)
    values = [synth_values(o, t) for t, o in enumerate(outputs)]
    g = np.float32(0.97)
    ref = gae_reference(outputs, values, g, 0.0)
    for s in range(2):
        for t in range(T):
            rn = ref[s]["next_row"][t]
            k = rn >= 0
            o1 = outputs[t + 1]
            term, _ = _end_of_life(o1[f"flags{s}"][rn[k]], o1["env_flags"][o1[f"row_env{s}"][rn[k]]])
            vn = np.where(term, np.float32(0), values[t + 1][s][rn[k]]).astype(np.float32)
            delta = (o1[f"reward{s}"][rn[k]] + g * vn) - values[t][s][k]
            assert np.array_equal(ref[s]["adv"][t][k], delta), (s, t)


@pytest.mark.parametrize("case", ["base_truncation", "base_extinction", "eco_crowded", "stag_strict", "base_masked_reset"])
def test_undiscounted_value_targets_are_the_future_rewards(case):
    """gamma = lambda = 1, V = 0: value_target is the sum of the rewards of the agent's future rows in the rollout, which the
    episode-returns tracker gives as the row_return of the life's last row minus the row's own"""
    cfg, B, T, kw = _case(case)
    outputs, rets = oracle_rollout(cfg, B, T, track=True, **kw)
    zeros = [[np.zeros(o["n"][s], np.float32) for s in range(2)] for o in outputs]
    ref = gae_reference(outputs, zeros, 1.0, 1.0)
    checked = 0
    for s in range(2):
        for seq in life_sequences(outputs, s):
            rewards = [float(outputs[t][f"reward{s}"][r]) for t, r in seq]
            t_end, r_end = seq[-1]
            for k, (t, r) in enumerate(seq[:-1]):
                vt = float(ref[s]["value_target"][t][r])
                assert vt == pytest.approx(sum(rewards[k + 1:]), rel=1e-5, abs=1e-4), (case, s, t, r)
                assert vt == pytest.approx(rets[t_end][s][r_end] - rets[t][s][r], rel=1e-5, abs=1e-4), (case, s, t, r)
                checked += 1
    assert checked > 1000


CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_gae_kernel_never_triggers_dependent_launches():
    """ppg_gae is a plain launch: it must not execute griddepcontrol.launch_dependents (PREEXIT) or wait on one (ACQBULK)"""
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    sass = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {m.group(1): body for m, body in zip(re.finditer(r"Function : (\S+)", sass), re.split(r"Function : \S+", sass)[1:])}
    mine = {f: b for f, b in funcs.items() if "ppg_gae_kernel" in f}
    assert len(mine) == 1, sorted(mine)
    for f, body in mine.items():
        assert "PREEXIT" not in body and "ACQBULK" not in body, f
