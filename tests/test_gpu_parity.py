"""CUDA path vs the CPU oracle through the C-ABI, on a real GPU (`-m gpu`)."""
import numpy as np
import pytest

from predpreygrass_b200.config import BASE_CONFIG, make_config
from tests.helpers import GOLDEN_DIR, config_from_golden, dict_order_rows, golden_cases, load_golden
from tests.parity import compare_outputs, lockstep_parity

pytestmark = pytest.mark.gpu

CROWDED = dict(BASE_CONFIG, grid_size=6, initial_num_grass=14, n_initial_active_predator=5, n_initial_active_prey=12,
               predator_creation_energy_threshold=6.0, prey_creation_energy_threshold=3.5, initial_energy_predator=3.0,
               initial_energy_prey=2.0, energy_gain_per_step_grass=0.5, energy_loss_per_step_prey=0.02,
               energy_loss_per_step_predator=0.1, predator_obs_range=5, prey_obs_range=7, n_possible_predators=300,
               n_possible_prey=300, max_steps=60)


def _reset_tape(n):
    z = np.load(f"{GOLDEN_DIR}/base_reset_cells_4096.npz")
    return [z["cells"][i].astype(np.int32) for i in range(n)]


def test_small_philox():
    st = lockstep_parity(make_config(BASE_CONFIG, cap_live=(64, 192), seed=7), 64, 120, state_envs=(0, 5, 63))
    assert st["status_envs"] == 0 and st["episodes"] > 0


def test_replay_4096_envs_300_steps():
    """BASELINE configs[1]: 4096 envs, reset placements replayed from the reference's numpy RNG tape,
    every output array of every step compared with the oracle."""
    cfg = make_config(BASE_CONFIG, cap_live=(64, 192), seed=11)
    st = lockstep_parity(cfg, 4096, 300, tape=_reset_tape(4096), state_envs=(0, 1000, 4095), check_every=1)
    assert st["status_or"] & ~4 == 0  # only TAPE_EXHAUSTED (second episodes run on the Philox stream)
    assert st["env_steps"] > 4096 * 250


@pytest.mark.parametrize("mode,switches", [pytest.param(m, {}, id=m) for m in ("sparse", "dense", "additive", "kickback")] + [
    # the one-kernel step's CTA-ganged warps and rows through the bulk-copy engine (DESIGN.md §4 experiment switches)
    pytest.param("kickback", {"PPG_WARPS_PER_CTA": "4"}, id="kickback-warps4"),
    pytest.param("dense", {"PPG_WARPS_PER_CTA": "8"}, id="dense-warps8"),
    pytest.param("sparse", {"PPG_OBS_BULK": "1"}, id="sparse-bulk"),
    pytest.param("additive", {"PPG_OBS_BULK": "1", "PPG_WARPS_PER_CTA": "4"}, id="additive-bulk-warps4"),
])
def test_reward_modes_crowded(mode, switches, monkeypatch):
    """crowded 6x6 world: births every step, blocked moves, co-located agents, spawn fallback draws"""
    for k, v in switches.items():
        monkeypatch.setenv(k, v)  # read when the handle is created
    cfg = make_config(CROWDED, reward_mode=mode, cap_live=(64, 64), seed=3)
    st = lockstep_parity(cfg, 256, 150, state_envs=(0, 17, 255))
    assert st["spawn_fallback"] > 0 and st["births_prey"] > 0 and st["truncated"] >= 0


def test_eating_constants_and_founders_over_10():
    cfg = dict(BASE_CONFIG, reward_predator_catch_prey=1.0, reward_prey_eat_grass=0.1, penalty_prey_caught=-2.0,
               n_initial_active_predator=12, n_initial_active_prey=14, max_steps=80)
    st = lockstep_parity(make_config(cfg, cap_live=(64, 192), seed=5), 128, 200, state_envs=(0, 127))
    assert st["truncated"] > 0


def test_slot_overflow_and_id_pool_exhaustion_match_oracle():
    cfg = dict(CROWDED, n_possible_prey=40, n_possible_predators=12, max_steps=50)
    st = lockstep_parity(make_config(cfg, cap_live=(32, 32), seed=9), 64, 120)
    assert st["births_prey"] > 0


def test_no_autoreset_goes_idle():
    cfg = make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=2, autoreset=False)
    lockstep_parity(cfg, 32, 40)


@pytest.mark.parametrize("name", golden_cases())
def test_golden_trajectories_on_gpu(name):
    """Golden trajectories of the unmodified reference replayed on the GPU (one env, tape-driven):
    ids, dict order, rewards, terminations bit-exact; float64 energies bit-exact.  The `shuffle`
    cases pass their action dicts in a random key order (ppg_step_ordered)."""
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    z, cfg = load_golden(name)
    c = config_from_golden(cfg, autoreset=False)
    c.cap_live[0] = min(c.cap_live[0], 320)
    c.cap_live[1] = min(c.cap_live[1], 320)
    g = BatchedPredPreyGrass(c, 1)
    g.load_tape([np.concatenate([z["init_cells"], z["fallback_cells"]])])
    g.reset()
    out = g.outputs_numpy()
    rows = dict_order_rows(out)
    assert [int(out[f"row_agent{s}"][r]) for s, r in rows] == list(z["reset_row_id"])
    T = len(z["steps"])
    for t in range(T):
        if z["all_trunc"][t] and t == T - 1 and int(z["steps"][t]) == int(z["steps"][t - 1]):
            break  # BASE's extra truncation call: folded into the previous step on the device
        a0, a1 = z["act_off"][t], z["act_off"][t + 1]
        act, rank, seen = {}, {}, [0, 0]
        for s, i, v in zip(z["act_s"][a0:a1], z["act_id"][a0:a1], z["act_v"][a0:a1]):
            act[(int(s), int(i))] = int(v)
            rank[(int(s), int(i))] = seen[int(s)]  # position among the species' keys of the action dict
            seen[int(s)] += 1
        import torch
        orders = []
        for s in range(2):
            n = out["n"][s]
            a = np.full(max(n, 1), 4, np.int32)
            o = np.zeros(max(n, 1), np.int32)
            for r in range(n):
                if not (out[f"flags{s}"][r] & 1):
                    a[r] = act[(s, int(out[f"row_agent{s}"][r]))]
                    o[r] = rank[(s, int(out[f"row_agent{s}"][r]))]
            g.actions[s][: len(a)].copy_(torch.from_numpy(a))
            orders.append(torch.from_numpy(o).cuda())
        if str(z["order"]) == "shuffle":
            g.step_ordered(g.actions[0], g.actions[1], orders[0], orders[1])
        else:
            g.step()
        out = g.outputs_numpy()
        rows = dict_order_rows(out)
        r0, r1 = z["row_off"][t], z["row_off"][t + 1]
        assert [s for s, _ in rows] == list(z["row_s"][r0:r1]), (name, t)
        assert [int(out[f"row_agent{s}"][r]) for s, r in rows] == list(z["row_id"][r0:r1]), (name, t)
        rew = np.array([out[f"reward{s}"][r] for s, r in rows], np.float32)
        assert np.array_equal(rew, z["row_rew"][r0:r1].astype(np.float32)), (name, t)
        fl = np.array([out[f"flags{s}"][r] for s, r in rows], np.uint8)
        assert np.array_equal(fl & 1, z["row_term"][r0:r1]), (name, t)
        assert bool(out["env_flags"][0] & 1) == bool(z["all_term"][t]), (name, t)
        if out["env_flags"][0] & 3:
            break
        st = g.read_env(0)
        s0, s1 = z["st_off"][t], z["st_off"][t + 1]
        for s in range(2):
            m = z["st_s"][s0:s1] == s
            assert np.array_equal(st["ids"][s], z["st_id"][s0:s1][m]), (name, t, s)
            assert np.array_equal(st["xy"][s][:, 0], z["st_x"][s0:s1][m]) and np.array_equal(st["xy"][s][:, 1], z["st_y"][s0:s1][m])
            assert np.array_equal(st["energy"][s], z["st_e"][s0:s1][m]), (name, t, s)
        assert np.array_equal(st["grass_energy"], z["grass_e"][t]), (name, t)
    g.close()


def test_step_host_matches_step_and_snapshot_restore():
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(BASE_CONFIG, cap_live=(64, 192), seed=21)
    a, b = BatchedPredPreyGrass(cfg, 96), BatchedPredPreyGrass(cfg, 96)
    a.reset(); b.reset()
    host = b.make_host_buffers()
    snap = None
    for t in range(60):
        a0, a1 = a.random_actions(5)
        n0, n1 = a.out.counts()
        host["actions0"][:n0].copy_(a0[:n0].cpu()); host["actions1"][:n1].copy_(a1[:n1].cpu())
        a.step(a0, a1)
        m0, m1 = b.step_host(host)
        ga = a.outputs_numpy()
        assert (m0, m1) == ga["n"]
        for s in range(2):
            k = ga["n"][s]
            assert np.array_equal(host[f"obs{s}"][:k].numpy(), ga[f"obs{s}"])
            assert np.array_equal(host[f"row_agent{s}"][:k].numpy(), ga[f"row_agent{s}"])
            assert np.array_equal(host[f"reward{s}"][:k].numpy(), ga[f"reward{s}"])
            assert np.array_equal(host[f"flags{s}"][:k].numpy(), ga[f"flags{s}"])
        assert np.array_equal(host["env_flags"].numpy(), ga["env_flags"])
        if t == 29:
            snap = a.snapshot()
            ref_later = []
        if t >= 30:
            ref_later.append({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in ga.items()})
    # restore the step-30 state into a fresh handle and replay: per-env results identical
    c = BatchedPredPreyGrass(cfg, 96)
    c.reset()
    c.restore(snap)
    a.restore(snap)
    for t in range(30, 60):
        for h in (a, c):
            x0, x1 = h.random_actions(5)
            h.step(x0, x1)
        ga, gc = a.outputs_numpy(), c.outputs_numpy()
        compare_outputs(ga, gc, f"restored step {t}")
    torch.cuda.synchronize()
    a.close(); b.close(); c.close()


def test_full_size_properties_16384_envs():
    """Size-independent properties at BASELINE configs[2] size (no oracle): determinism (two
    handles, same seed -> identical row batches), row-count bookkeeping, own-cell observation."""
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(BASE_CONFIG, reward_mode="additive", cap_live=(64, 192), seed=77)
    B = 16384
    a, b = BatchedPredPreyGrass(cfg, B), BatchedPredPreyGrass(cfg, B)
    a.reset(); b.reset()
    for t in range(80):
        for h in (a, b):
            x0, x1 = h.random_actions(99)
            h.step(x0, x1)
        if t % 20 == 19:
            n = a.out.n_rows.tolist()
            assert n == b.out.n_rows.tolist()
            for s in range(2):
                k = n[s] + n[2 + s]
                assert torch.equal(a.out.obs[s][:k], b.out.obs[s][:k])
                assert torch.equal(a.out.reward[s][:k], b.out.reward[s][:k])
                assert torch.equal(a.out.row_agent[s][:k], b.out.row_agent[s][:k])
                # rows are grouped by env in ascending order
                re = a.out.row_env[s][: n[s]]
                assert bool((re[1:] >= re[:-1]).all())
                # centre cell of the own-species channel holds the agent's (positive) energy for live rows,
                # wall channel is 0 at the centre
                R = cfg.obs_range[s]
                live = (a.out.flags[s][:k] & 1) == 0
                centre = a.out.obs[s][:k, 1 + s, R // 2, R // 2]
                assert bool((a.out.obs[s][:k, 0, R // 2, R // 2] == 0).all())
                assert float((centre[live] > 0).float().mean()) > 0.999  # hidden co-located agents are the rare exception
            # live counts = rows that are not terminated, per env
            cnt = a.out.env_count.long()
            for s in range(2):
                k = n[s] + n[2 + s]
                live = ((a.out.flags[s][:k] & 1) == 0).long()
                per_env = torch.zeros(B, dtype=torch.long, device=live.device).index_add_(0, a.out.row_env[s][:k].long(), live)
                running = (a.out.env_flags & 4) == 0
                assert torch.equal(per_env[running], cnt[running, s])
    st = a.stats()
    assert st["status_envs"] == 0
    a.close(); b.close()


@pytest.mark.parametrize("name", ["base_default_s1", "base_default_s7_shuffle", "base_trunc_s2", "additive_default_s1", "kickback_default_s6",
                                  "seasonal_default_s1", "seasonal_trunc_s3", "seasonal_default_s5",
                                  "base_crowded_s1", "base_crowded_s2_shuffle", "additive_crowded_s2", "kickback_crowded_s1", "base_rewards_s8",
                                  "dense_crowded_s3", "seasonal_crowded_s2_shuffle"])
def test_dict_adapter_replays_reference_episode(name):
    """`PredPreyGrass` (the MultiAgentEnv-shaped adapter) against an episode recorded from the reference
    through the same dict API: reset(seed) placement, observation-dict key order, rewards,
    terminations, truncations (incl. BASE's extra truncation call, BASE:228-238), `agents`, state."""
    from predpreygrass_b200.env import PredPreyGrass

    z, cfg = load_golden(name)
    variant = cfg.pop("variant")
    cfg = dict(cfg, reward_variant=variant, cap_live=(min(cfg["n_possible_predators"], 320), min(cfg["n_possible_prey"], 320)))
    env = PredPreyGrass(cfg)
    # spawn-fallback cells (BASE:764, global numpy generator) are the reference's recorded ones
    obs, infos = env.reset(seed=int(z["seed"]), options={"ppg_tape": z["fallback_cells"]})
    assert infos == {}
    G = env.grid_size
    names = ("predator", "prey")
    assert list(obs) == [f"{names[s]}_{i}" for s, i in zip(z["reset_row_s"], z["reset_row_id"])]
    pos = env.agent_positions
    cells = [pos[a][0] * G + pos[a][1] for a in env.agents] + [p[0] * G + p[1] for p in env.grass_positions.values()]
    assert cells == list(z["init_cells"])  # numpy PCG64 + set order reproduced on the host (BASE:156-187)
    for a, o in obs.items():
        assert o.dtype == np.float64 and o.shape == env.observation_spaces[a].shape
    T = len(z["steps"])
    for t in range(T):
        a0, a1 = z["act_off"][t], z["act_off"][t + 1]
        acts = {f"{names[s]}_{i}": int(v) for s, i, v in zip(z["act_s"][a0:a1], z["act_id"][a0:a1], z["act_v"][a0:a1])}
        obs, rew, term, trunc, infos = env.step(acts)
        r0, r1 = z["row_off"][t], z["row_off"][t + 1]
        keys = [f"{names[s]}_{i}" for s, i in zip(z["row_s"][r0:r1], z["row_id"][r0:r1])]
        assert list(obs) == keys, (name, t)
        assert list(rew) == keys and [k for k in term if k != "__all__"] == keys
        assert np.array_equal(np.array([rew[k] for k in keys], np.float32), z["row_rew"][r0:r1].astype(np.float32)), (name, t)
        assert [int(term[k]) for k in keys] == list(z["row_term"][r0:r1]), (name, t)
        assert [int(trunc[k]) for k in keys] == list(z["row_trunc"][r0:r1]), (name, t)
        assert term["__all__"] == bool(z["all_term"][t]) and trunc["__all__"] == bool(z["all_trunc"][t]), (name, t)
        assert env.current_step == int(z["steps"][t])
        g0, g1 = z["ag_off"][t], z["ag_off"][t + 1]
        assert env.agents == [f"{names[s]}_{i}" for s, i in zip(z["ag_s"][g0:g1], z["ag_id"][g0:g1])], (name, t)
        if not (term["__all__"] or trunc["__all__"]):
            s0, s1 = z["st_off"][t], z["st_off"][t + 1]
            want = {f"{names[s]}_{i}": ((int(x), int(y)), float(e)) for s, i, x, y, e in
                    zip(z["st_s"][s0:s1], z["st_id"][s0:s1], z["st_x"][s0:s1], z["st_y"][s0:s1], z["st_e"][s0:s1])}
            got_p, got_e = env.agent_positions, env.agent_energies
            assert sorted(got_p) == sorted(want), (name, t)
            assert all(got_p[k] == want[k][0] and got_e[k] == want[k][1] for k in want), (name, t)
    with pytest.raises(KeyError):
        e2 = PredPreyGrass(cfg)
        e2.reset(seed=1)
        e2.step({"predator_1999": 0})
    env.close()
