"""Episode returns and agent lifetimes (include/ppg.h ppg_track_returns) on the CPU: a numpy reference tracker of the
semantics, with the device's fixed summation order, checked on the oracle's outputs for the conservation identity and
against the agents' ages; the conversion of the statistics vector to RLlib's metric names; the all-reduce of that vector in
a world-size-2 gloo job; and the SASS of the kernels.  tests/test_gpu_returns.py compares the device with this tracker."""
import os
import re
import shutil
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from predpreygrass_b200.config import (BASE_CONFIG, N_EP_STATS, STAG_CONFIG, VARIANT_ECO, VARIANT_STAG,
                                       make_config)

TERM, TRUNC, NEWBORN, FOUNDER = 0x01, 0x02, 0x04, 0x08
ENV_END, ENV_RESET, ENV_IDLE = 0x03, 0x04, 0x08


def _butterfly(p):
    """the kernel's xor-butterfly over the 32 lane partials of every env (p: [B, 32]); every lane ends with the same bits"""
    lanes = np.arange(32)
    for k in (16, 8, 4, 2, 1):
        p = p + p[:, lanes ^ k]
    return p[:, 0]


class Tracker:
    """numpy model of ppg_returns_kernel, fed the outputs (Oracle.outputs() / outputs_numpy()) one by one"""

    def __init__(self, n_envs, n_possible):
        self.B, self.n_possible = n_envs, (int(n_possible[0]), int(n_possible[1]))
        self.tab_ret = [np.zeros(n_envs * self.n_possible[s]) for s in range(2)]
        self.tab_life = [np.zeros(n_envs * self.n_possible[s], np.int32) for s in range(2)]
        self.env_valid = np.zeros(n_envs, np.uint8)
        self.env_return = np.full((n_envs, 2), np.nan)
        self.env_acc = np.zeros((n_envs, N_EP_STATS))
        self.env_acc[:, 6:8] = -np.inf
        self.row_return, self.row_life = [None, None], [None, None]
        self.ended_sum = np.zeros((n_envs, 2))  # this output's sum of the lifetime returns of the lives that ended
        self.reused = 0  # outputs where an old TERMINATED row and a NEWBORN row share (env, id)

    def invalidate(self):
        """switch-on and restore"""
        self.env_valid[:] = 0
        self.env_return[:] = np.nan

    def update(self, out):
        ef = out["env_flags"].astype(np.int64)
        idle = (ef & ENV_IDLE) != 0
        valid = ((ef & ENV_RESET) != 0) | (self.env_valid != 0)
        upd = valid & ~idle
        step, ended = np.zeros((self.B, 2)), np.zeros((self.B, 2))
        counts = np.zeros((self.B, 2, 3), np.int64)  # lives, deaths, rows
        for s in range(2):
            n_old, n = out["n_old"][s], out["n"][s]
            env = out[f"row_env{s}"][:n].astype(np.int64)
            ids = out[f"row_agent{s}"][:n].astype(np.int64)
            fl = out[f"flags{s}"][:n].astype(np.int64)
            rw = out[f"reward{s}"][:n].astype(np.float64)
            rows = np.arange(n)
            first = np.where(rows < n_old, out[f"old_off{s}"][env], out[f"new_off{s}"][env])
            j = rows - first
            lane, k = j % 32, j // 32
            v = valid[env]
            key = env * self.n_possible[s] + ids
            ret, life = np.full(n, np.nan), np.zeros(n, np.int32)
            for phase in (rows < n_old, rows >= n_old):  # old rows, then newborn rows
                sel = phase & v
                start = (fl[sel] & (FOUNDER | NEWBORN)) != 0
                ret[sel] = np.where(start, rw[sel], self.tab_ret[s][key[sel]] + rw[sel])
                life[sel] = np.where(start, 1, self.tab_life[s][key[sel]] + 1)
                self.tab_ret[s][key[sel]] = ret[sel]
                self.tab_life[s][key[sel]] = life[sel]
            self.row_return[s], self.row_life[s] = ret, life
            end = ((fl & (TERM | TRUNC)) != 0) & v
            term_old = set(zip(env[(rows < n_old) & ((fl & TERM) != 0)].tolist(), ids[(rows < n_old) & ((fl & TERM) != 0)].tolist()))
            if term_old and term_old & set(zip(env[rows >= n_old].tolist(), ids[rows >= n_old].tolist())):
                self.reused += 1
            ps, pe = np.zeros((self.B, 32)), np.zeros((self.B, 32))
            for phase in (rows < n_old, rows >= n_old):
                for kk in range(int(k[phase].max()) + 1 if phase.any() else 0):
                    sel = phase & v & (k == kk)
                    ps[env[sel], lane[sel]] += rw[sel]
                    sel = sel & end
                    pe[env[sel], lane[sel]] += ret[sel]
            step[:, s], ended[:, s] = _butterfly(ps), _butterfly(pe)
            counts[:, s, 0] = np.bincount(env[end], minlength=self.B)
            counts[:, s, 1] = np.bincount(env[end & ((fl & TERM) != 0)], minlength=self.B)
            counts[:, s, 2] = np.bincount(env[end], weights=life[end], minlength=self.B).astype(np.int64)
        self.ended_sum = np.where(upd[:, None], ended, 0.0)
        er = np.where((ef & ENV_RESET)[:, None] != 0, 0.0, self.env_return)
        er = er + step
        self.env_return[upd] = er[upd]
        a = self.env_acc
        for s in range(2):
            q = 8 + 4 * s
            a[upd, q] += counts[upd, s, 0].astype(np.float64)
            a[upd, q + 1] += counts[upd, s, 1].astype(np.float64)
            a[upd, q + 2] += ended[upd, s]
            a[upd, q + 3] += counts[upd, s, 2].astype(np.float64)
        fin = upd & ((ef & ENV_END) != 0)
        total = er[:, 0] + er[:, 1]
        a[fin, 0] += 1.0
        a[fin, 1] += out["env_step"][fin].astype(np.float64)
        a[fin, 2] += total[fin]
        a[fin, 3] += total[fin] * total[fin]
        a[fin, 4] += er[fin, 0]
        a[fin, 5] += er[fin, 1]
        a[fin, 6] = np.fmax(a[fin, 6], total[fin])
        a[fin, 7] = np.fmax(a[fin, 7], -total[fin])
        self.env_valid[upd] = 1

    def stats(self):
        """the aggregate vector over the valid envs, summed in numpy's order"""
        a = self.env_acc[self.env_valid != 0]
        v = a.sum(axis=0) if len(a) else np.zeros(N_EP_STATS)
        v[6:8] = a[:, 6:8].max(axis=0) if len(a) else -np.inf
        return v


def run_oracle(cfg, n_envs, steps, action_seed=7, check=None):
    """the oracle stepped with its Philox random actions, the tracker (switched on before the reset) fed every output;
    check(tracker, out, t) after every output"""
    from oracle.oracle import Oracle

    ora = Oracle(cfg, n_envs, threads=4)
    tr = Tracker(n_envs, cfg.n_possible)
    try:
        out = ora.reset()
        tr.update(out)
        if check:
            check(tr, out, -1, ora)
        for t in range(steps):
            a0, a1 = ora.random_actions(action_seed)
            A0 = np.zeros(max(1, len(a0)), np.int32); A0[: len(a0)] = a0
            A1 = np.zeros(max(1, len(a1)), np.int32); A1[: len(a1)] = a1
            out = ora.step(A0, A1)
            tr.update(out)
            if check:
                check(tr, out, t, ora)
        return tr
    finally:
        ora.close()


def _eco_crowded():
    from tests.test_gpu_parity_eco import CROWDED

    return CROWDED


CONSERVATION_CASES = {
    "base": lambda: make_config(dict(BASE_CONFIG, max_steps=25), cap_live=(64, 192), seed=3),
    "eco_crowded": lambda: make_config(dict(_eco_crowded(), max_steps=60), variant=VARIANT_ECO, cap_live=(64, 64), seed=5),
    "stag": lambda: make_config(dict(STAG_CONFIG, max_steps=40), variant=VARIANT_STAG, cap_live=(64, 192), seed=6),
    "stag_not_strict": lambda: make_config(dict(STAG_CONFIG, max_steps=40, strict_rllib_output=False), variant=VARIANT_STAG,
                                           cap_live=(64, 192), seed=6),
}


@pytest.mark.parametrize("case", sorted(CONSERVATION_CASES))
def test_conservation_identity_on_the_oracle(case):
    """at every output, per valid env and species: the lifetime returns of the lives ended in this episode plus the running
    returns of the live agents equal the env's episode return, exactly"""
    cfg = CONSERVATION_CASES[case]()
    B = 48
    ended_ep = np.zeros((B, 2))
    seen = {"episodes": 0, "lives": 0}

    def check(tr, out, t, ora):
        ef = out["env_flags"]
        ended_ep[(ef & ENV_RESET) != 0] = 0.0
        ended_ep[:] += tr.ended_sum
        for s in range(2):
            n = out["n"][s]
            env = out[f"row_env{s}"][:n]
            live = (out[f"flags{s}"][:n] & (TERM | TRUNC)) == 0
            running = np.bincount(env[live], weights=tr.row_return[s][live], minlength=B)
            ok = tr.env_valid != 0
            assert np.array_equal(ended_ep[ok, s] + running[ok], tr.env_return[ok, s]), (case, t, s)
        seen["episodes"] = int(tr.env_acc[:, 0].sum())
        seen["lives"] = int(tr.env_acc[:, 8].sum() + tr.env_acc[:, 12].sum())

    tr = run_oracle(cfg, B, 90, check=check)
    assert seen["episodes"] >= B and seen["lives"] > 0, seen
    assert (tr.env_valid == 1).all()


def _age_relation(cfg, read, steps=60):
    """pairs (row_life, age) of every live agent of a few envs after every step"""
    pairs = set()

    def check(tr, out, t, ora):
        for e in (0, 3, 7):
            if out["env_flags"][e] & ENV_END:  # the state of a finished episode is not kept
                continue
            st = read(ora, e)
            for s in range(2):
                n = out["n"][s]
                mine = (out[f"row_env{s}"][:n] == e) & ((out[f"flags{s}"][:n] & (TERM | TRUNC)) == 0)
                life = dict(zip(out[f"row_agent{s}"][:n][mine].tolist(), tr.row_life[s][mine].tolist()))
                assert sorted(life) == sorted(st["ids"][s].tolist()), (t, e, s)
                pairs.update((life[i], int(a)) for i, a in zip(st["ids"][s].tolist(), st["age"][s].tolist()))

    run_oracle(cfg, 8, steps, check=check)
    return pairs


def test_row_life_relates_to_eco_ages():
    """ECO: an agent's age after a step is its number of rows in this life minus one (a founder or newborn row has age 0)"""
    cfg = make_config(dict(_eco_crowded(), max_steps=60), variant=VARIANT_ECO, cap_live=(64, 64), seed=5)
    pairs = _age_relation(cfg, lambda ora, e: ora.read_env_eco(e))
    assert pairs and all(age == life - 1 for life, age in pairs), sorted(pairs)[:10]
    assert max(life for life, _ in pairs) > 20


def test_row_life_relates_to_stag_ages():
    cfg = make_config(dict(STAG_CONFIG, max_steps=60), variant=VARIANT_STAG, cap_live=(64, 192), seed=6)
    pairs = _age_relation(cfg, lambda ora, e: ora.read_env_stag(e))
    assert pairs and all(age == life - 1 for life, age in pairs), sorted(pairs)[:10]
    assert max(life for life, _ in pairs) > 20


# ECO with an id pool small enough to run dry within an episode (PPG_STATUS_ID_POOL_EMPTY)
REUSE_CONFIG = lambda: make_config(dict(_eco_crowded(), max_steps=80, n_possible_predators=12, n_possible_prey=24),  # noqa: E731
                                   variant=VARIANT_ECO, cap_live=(32, 32), seed=5)


def test_ids_are_never_reused_within_an_episode():
    """Every variant hands a newborn the smallest never-used id, and a dry pool suppresses the birth: no output holds an old
    TERMINATED row and a NEWBORN row of the same (env, id), even with the pool exhausted.  (The kernel still finishes the
    old rows before it starts the newborn rows, so the tables stay right should an id ever be reused in the step that
    freed it.)"""
    status = []
    tr = run_oracle(REUSE_CONFIG(), 64, 80, check=lambda tr, out, t, ora: status.append(int(np.bitwise_or.reduce(out["env_status"]))))
    assert any(st & 0x10 for st in status)  # PPG_STATUS_ID_POOL_EMPTY
    assert tr.reused == 0 and tr.env_acc[:, 0].sum() > 0


# ------------------------------------------------------------------------------------------------ vector -> RLlib dict
def test_episode_metrics_from_stats():
    from predpreygrass_b200.batched import episode_metrics_from_stats

    v = np.zeros(N_EP_STATS)
    v[6:8] = -np.inf
    m = episode_metrics_from_stats(v)
    assert m["num_episodes"] == 0 and np.isnan(m["episode_return_mean"]) and np.isnan(m["episode_len_mean"])
    assert m["episode_return_max"] == -np.inf and m["episode_return_min"] == np.inf
    assert all(np.isnan(x) for x in m["module_episode_returns_mean"].values())
    assert all(np.isnan(x) for d in ("agent_lifetime_return_mean", "agent_lifetime_rows_mean") for x in m[d].values())
    assert m["agent_deaths"] == {"predator": 0, "prey": 0}
    # two episodes of total returns 3 and -1 (lengths 10, 30), predator 1.5 + prey 0.5 per episode on average;
    # predators: 4 lives ended (3 deaths), lifetime returns 8, 20 rows; prey: none ended
    v = np.array([2, 40, 2, 10, 3, -1, 3, 1, 4, 3, 8, 20, 0, 0, 0, 0], np.float64)
    m = episode_metrics_from_stats(v)
    assert m["num_episodes"] == 2 and m["episode_return_mean"] == 1.0 and m["episode_len_mean"] == 20.0
    assert m["episode_return_max"] == 3.0 and m["episode_return_min"] == -1.0
    assert m["module_episode_returns_mean"] == {"predator": 1.5, "prey": -0.5}
    assert m["agent_lifetime_return_mean"]["predator"] == 2.0 and m["agent_lifetime_rows_mean"]["predator"] == 5.0
    assert np.isnan(m["agent_lifetime_return_mean"]["prey"]) and np.isnan(m["agent_lifetime_rows_mean"]["prey"])
    assert m["agent_deaths"] == {"predator": 3, "prey": 0} and m["agent_lives_ended"] == {"predator": 4, "prey": 0}
    with pytest.raises(ValueError):
        episode_metrics_from_stats(np.zeros(15))


# ------------------------------------------------------------------------------------------------ all-reduce over ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_vector(rank):
    v = np.array([3 + rank, 10, 1.5 * (rank + 1), 4.0, 1.0, 0.5, 7.0 - 5 * rank, -2.0 + 4 * rank] + [rank + k for k in range(8)], np.float64)
    return v


def _worker(rank, world, port, q):
    from predpreygrass_b200.sharding import allreduce_episode_stats

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    v = torch.from_numpy(_rank_vector(rank))
    out = allreduce_episode_stats(v)
    q.put((rank, out.numpy().copy(), out is v))
    dist.barrier()
    dist.destroy_process_group()


def test_allreduce_episode_stats_two_rank_gloo():
    from predpreygrass_b200.sharding import allreduce_episode_stats

    port = _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    a, b = _rank_vector(0), _rank_vector(1)
    want = a + b
    want[6:8] = np.maximum(a[6:8], b[6:8])
    for rank, got, inplace in res:
        assert inplace and np.array_equal(got, want), (rank, got, want)
    # without an initialised process group the vector is returned as it is
    v = torch.from_numpy(a.copy())
    assert allreduce_episode_stats(v) is v and np.array_equal(v.numpy(), a)
    with pytest.raises(ValueError):
        allreduce_episode_stats(torch.zeros(16, dtype=torch.float32))


# ------------------------------------------------------------------------------------------------ SASS
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_returns_kernels_never_trigger_or_wait_on_dependent_launches():
    """with the launch chain on, the next step's kernels start only after ppg_returns_kernel has read the rows: it must not
    execute griddepcontrol.launch_dependents (PREEXIT), and it is never launched as a dependent (no griddepcontrol.wait, ACQBULK)"""
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    sass = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {m.group(1): body for m, body in zip(re.finditer(r"Function : (\S+)", sass), re.split(r"Function : \S+", sass)[1:])}
    mine = {f: b for f, b in funcs.items() if "ppg_returns_kernel" in f or "ppg_episode_stats" in f}
    assert any("ppg_returns_kernel" in f for f in mine) and len(mine) >= 3, sorted(mine)
    for f, body in mine.items():
        assert "PREEXIT" not in body and "ACQBULK" not in body, f
