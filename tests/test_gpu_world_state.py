"""`BatchedPredPreyGrass.world_state()` (include/ppg.h ppg_world_state) and the dict adapters' `grid_world_state` on the GPU
(`-m gpu`): against the unmodified reference's recordings (sha1 of its float32 grid; BASE through the oracle, which
tests/test_oracle_golden.py pins to the reference's float64 grid), against the oracle at scale, queued without host
synchronisation with the launch chain off and on, and its error states."""
import numpy as np
import pytest

from predpreygrass_b200.config import BASE_CONFIG, ECO_CONFIG, SEASONAL_CONFIG, STAG_CONFIG, VARIANT_ECO, VARIANT_STAG, make_config
from tests.helpers import config_from_golden, golden_cases, load_golden, sha_f32

pytestmark = pytest.mark.gpu

BASE_FAMILY = ("base", "eating", "dense", "additive", "kickback", "seasonal")
TRAITS = ("mr", "inv", "coop", "cad")


def _oracle_world(ora, envs):
    return np.stack([ora.read_grid(e).astype(np.float32) for e in envs])


def _assert_world(got, want, where):
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)[:5]
        raise AssertionError(f"{where}: world differs at [env, c, x, y] {bad.tolist()}: gpu={got[tuple(bad.T)]} oracle={want[tuple(bad.T)]}")


# ------------------------------------------------------------------------------------------------ reference recordings
@pytest.mark.parametrize("name", golden_cases(BASE_FAMILY + ("eco", "stag") + TRAITS))
def test_world_state_replays_reference_grid(name):
    """Every recording replayed on one env, tape-driven (the pattern of the golden GPU tests): the world after every step
    where the oracle golden tests compare the grid."""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    z, cfg = load_golden(name)
    fam = name.split("_")[0]
    base, stag = fam in BASE_FAMILY, fam == "stag"
    c = config_from_golden(dict(cfg, include_visibility_channel=False) if stag else cfg, autoreset=False)
    lim = (320, 320) if base else (224, 416)
    c.cap_live[0], c.cap_live[1] = min(c.cap_live[0], lim[0]), min(c.cap_live[1], lim[1])
    g = BatchedPredPreyGrass(c, 1)
    ora = None
    if base:
        g.load_tape([np.concatenate([z["init_cells"], z["fallback_cells"]])])
        ora = Oracle(c, 1)
        ora.load_tape([z["fallback_cells"]])
        ora.env_reset_cells(0, z["init_cells"])
    elif fam == "eco":
        g.load_tape([np.concatenate([z["init_cells"], z["fallback_cells"]])], [np.concatenate([z["founder_speed"], z["step_reals"]])])
    elif stag:
        reals = np.concatenate([z["founder_trait_raw"] if c.coop_trait_enabled else np.zeros(0), z["step_reals"]])
        g.load_tape([np.concatenate([z["init_cells"], z["founder_facing"], z["step_ints"]])], [reals])
    elif fam == "cad":
        g.load_tape([np.concatenate([z["init_cells"], z["fallback_cells"]])],
                    [np.concatenate([z["founder_trait"], z["founder_acc"], z["step_reals"]])])
    else:
        g.load_tape([np.concatenate([z["n_found"], z["init_cells"], z["fallback_cells"]])],
                    [np.concatenate([z["founder_trait"], z["step_reals"]])])
    g.reset()
    out = g.outputs_numpy()
    if base:
        _assert_world(g.world_state().cpu().numpy(), _oracle_world(ora, [0]), f"{name} reset")
    stay = g.n_actions() // 2
    T, compared = len(z["steps"]), 0
    for t in range(T):
        if base and z["all_trunc"][t] and t == T - 1 and int(z["steps"][t]) == int(z["steps"][t - 1]):
            break  # BASE's extra truncation call: folded into the previous step on the device
        a0, a1 = z["act_off"][t], z["act_off"][t + 1]
        alive = {(s, int(out[f"row_agent{s}"][r])) for s in range(2) for r in range(out["n"][s]) if not (out[f"flags{s}"][r] & 1)}
        values = (z["act_move"][a0:a1].astype(np.int32) | (np.maximum(z["act_join"][a0:a1], 0).astype(np.int32) << 8)) if stag \
            else z["act_v"][a0:a1]
        act, rank, seen = {}, {}, [0, 0]
        for s, i, v in zip(z["act_s"][a0:a1], z["act_id"][a0:a1], values):
            if (int(s), int(i)) not in alive:  # STAG's recordings act for agents that ended in the step before (STAG:806-807)
                continue
            act[(int(s), int(i))] = int(v)
            rank[(int(s), int(i))] = seen[int(s)]
            seen[int(s)] += 1
        orders = []
        for s in range(2):
            n = out["n"][s]
            a = np.full(max(n, 1), stay, np.int32)
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
        ended = bool(out["env_flags"][0] & 3)
        world = g.world_state().cpu().numpy()
        assert world.shape == (1, c.num_obs_channels, c.grid_size, c.grid_size) and world.dtype == np.float32
        if base:
            ora.env_step_ordered(0, z["act_s"][a0:a1], z["act_id"][a0:a1], z["act_v"][a0:a1])
            _assert_world(world, _oracle_world(ora, [0]), f"{name} step {t}")
            compared += 1
        elif stag or not ended:  # ECO family: the reference clears its agents at the end; the recordings stop comparing there
            assert np.array_equal(sha_f32([world[0]]), z["grid_sha"][t]), (name, t)
            compared += 1
        if ended:
            break
    assert compared > 0
    g.close()
    if ora is not None:
        ora.close()


# ------------------------------------------------------------------------------------------------ lockstep at scale
def _lockstep_world(cfg, n_envs, steps, every=1, mask_at=None, action_seed=77):
    """GPU and oracle stepped with the same Philox actions; every `every` steps (and the last) all envs' worlds compared.
    mask_at: step before which every third env's reset is scheduled with a masked reset on both sides."""
    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    gpu, ora = BatchedPredPreyGrass(cfg, n_envs), Oracle(cfg, n_envs, threads=8)
    envs = range(n_envs)
    try:
        gpu.reset(); ora.reset()
        _assert_world(gpu.world_state().cpu().numpy(), _oracle_world(ora, envs), "reset")
        flags_seen = 0
        for t in range(steps):
            if t == mask_at:  # only schedules the resets: the world stays that of the last output
                before = gpu.world_state().clone()
                mask = (np.arange(n_envs) % 3 == 0).astype(np.uint8)
                gpu.reset(mask=mask); ora.reset(mask=mask)
                assert gpu.world_state().equal(before)
            a0, a1 = gpu.random_actions(action_seed)
            o0, o1 = ora.random_actions(action_seed)
            gpu.step(a0, a1)
            A0 = np.zeros(max(1, len(o0)), np.int32); A0[: len(o0)] = o0
            A1 = np.zeros(max(1, len(o1)), np.int32); A1[: len(o1)] = o1
            ora.step(A0, A1)
            if t % every == 0 or t == steps - 1:
                _assert_world(gpu.world_state().cpu().numpy(), _oracle_world(ora, envs), f"step {t}")
                flags_seen |= int(np.bitwise_or.reduce(ora.outputs()["env_flags"]))
        return flags_seen
    finally:
        gpu.close(); ora.close()


def test_world_state_base_4096_envs():
    flags = _lockstep_world(make_config(BASE_CONFIG, cap_live=(64, 192), seed=11), 4096, 60, every=5)
    assert flags & 1  # episodes end (and the envs reset) inside the window


@pytest.mark.parametrize("kind", ["additive", "seasonal"])
def test_world_state_add_and_seasonal(kind):
    cfg = make_config(BASE_CONFIG, reward_mode="additive", cap_live=(64, 192), seed=3) if kind == "additive" \
        else make_config(SEASONAL_CONFIG, cap_live=(64, 192), seed=4)
    _lockstep_world(cfg, 256, 100, every=3)


def _eco_crowded():
    from tests.test_gpu_parity_eco import CROWDED

    return CROWDED


def test_world_state_eco_ghost_cells():
    """ECO's ghost cells (stale prey values on the reference's grid, ECO:826-832) are part of the world"""
    cfg = dict(_eco_crowded(), max_agent_age={"predator": None, "prey": 9}, max_energy_gain_per_prey=0.4, max_steps=80,
               energy_gain_per_step_grass=0.8, prey_creation_energy_threshold=3.0)
    _lockstep_world(make_config(cfg, variant=VARIANT_ECO, cap_live=(96, 192), seed=17), 256, 100)


def test_world_state_eco_carcasses_and_no_genome():
    cfg = dict(_eco_crowded(), max_energy_gain_per_prey=0.8, max_energy_gain_per_grass=1.0)
    _lockstep_world(make_config(cfg, variant=VARIANT_ECO, cap_live=(64, 64), seed=9), 256, 120, every=2)
    from tests.test_gpu_parity_eco import RICH

    cfg = dict(RICH, genome_enabled=False, include_speed_in_obs=False, max_steps=50)
    _lockstep_world(make_config(cfg, variant=VARIANT_ECO, cap_live=(128, 320), seed=13), 64, 120, every=2)


@pytest.mark.parametrize("trait", ["metabolic", "investment", "cooperation", "cadence"])
def test_world_state_trait_variants(trait):
    from predpreygrass_b200.config import TRAIT_CONFIGS

    _lockstep_world(make_config(TRAIT_CONFIGS[trait], variant=VARIANT_ECO, cap_live=(64, 160), seed=7), 256, 120, every=3)


def test_world_state_stag_16bit_maps_and_walls():
    """STAG with caps 160+640 (16-bit owner maps), and STAG with walls and line of sight (walls are channel 0)"""
    _lockstep_world(make_config(STAG_CONFIG, variant=VARIANT_STAG, cap_live=(160, 640), seed=21), 512, 80, every=4)
    from tests.test_gpu_parity_stag import CROWDED

    walls = [(3, y) for y in range(2, 8)] + [(6, 1), (6, 2), (7, 7), (8, 7), (1, 8), (9, 9)]
    cfg = dict(CROWDED, grid_size=10, manual_wall_positions=walls, respect_los_for_movement=True, type_2_action_range=5)
    _lockstep_world(make_config(cfg, variant=VARIANT_STAG, cap_live=(96, 224), seed=31), 256, 120, every=3)


def test_world_state_idle_envs_keep_their_final_world():
    """autoreset off: an env whose episode is over produces no rows and keeps the world of its final step"""
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=2, autoreset=False)
    flags = _lockstep_world(cfg, 64, 40)
    assert flags & 8  # PPG_ENV_IDLE
    cfg = make_config(dict(_eco_crowded(), max_steps=30), variant=VARIANT_ECO, cap_live=(64, 64), seed=2, autoreset=False)
    assert _lockstep_world(cfg, 64, 50) & 8
    # the world of an idle env does not change from one step to the next
    g = BatchedPredPreyGrass(make_config(dict(STAG_CONFIG, max_steps=10), variant=VARIANT_STAG, cap_live=(64, 160), seed=5,
                                         autoreset=False), 32)
    g.reset()
    for _ in range(10):
        g.step(*g.random_actions(3))
    final = g.world_state().clone()  # every episode has ended by max_steps
    for _ in range(3):
        g.step(*g.random_actions(3))
        assert bool((g.out.env_flags == 8).all()) and g.world_state().equal(final)
    g.close()


def test_world_state_masked_reset():
    _lockstep_world(make_config(BASE_CONFIG, cap_live=(64, 192), seed=5), 256, 30, mask_at=10)
    _lockstep_world(make_config(ECO_CONFIG, variant=VARIANT_ECO, cap_live=(64, 128), seed=5), 128, 30, mask_at=12)


# ------------------------------------------------------------------------------------------------ ranges, queueing, isolation
def test_world_state_ranges_match_the_full_call():
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g = BatchedPredPreyGrass(make_config(ECO_CONFIG, variant=VARIANT_ECO, cap_live=(64, 128), seed=3), 300)
    g.reset()
    for _ in range(15):
        g.step(*g.random_actions(1))
    full = g.world_state().clone()
    for b, n in ((0, 300), (0, 1), (7, 93), (150, 150), (299, 1)):
        assert g.world_state(b, n).equal(full[b: b + n]), (b, n)
        out = torch.full((n,) + tuple(full.shape[1:]), -1.0, device=g.device)
        assert g.world_state(b, n, out=out) is out and out.equal(full[b: b + n]), (b, n)
    assert g.world_state(250).shape[0] == 50
    # G = 7, C = 3: an env's slab is 588 bytes, not a multiple of 16 (scalar stores)
    h = BatchedPredPreyGrass(make_config(dict(_eco_crowded(), grid_size=7, initial_num_grass=14, predator_obs_range=5, prey_obs_range=5),
                                         variant=VARIANT_ECO, cap_live=(64, 64), seed=4), 33)
    h.reset()
    for _ in range(5):
        h.step(*h.random_actions(2))
    w = h.world_state().clone()
    assert w.shape == (33, 3, 7, 7)
    for b in range(0, 33, 4):
        assert h.world_state(b, 1).equal(w[b: b + 1])
    g.close(); h.close()


@pytest.mark.parametrize("chain", [0, 1])
def test_world_state_queued_without_host_synchronisation(chain):
    """20 x {random actions, step, world_state into a per-step buffer} on one stream, nothing synchronised in between; with
    the launch chain on, the next step kernel must not overwrite the images while world_state still reads them"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(BASE_CONFIG, cap_live=(64, 192), seed=13)
    B, T = 768, 20
    before = _lib.load().ppg_set_pdl_chain(chain)
    try:
        g = BatchedPredPreyGrass(cfg, B)
        worlds = [torch.empty((B, 4, cfg.grid_size, cfg.grid_size), device=g.device) for _ in range(T)]
        acts = []
        g.reset()
        torch.cuda.synchronize()
        for t in range(T):
            a0, a1 = g.random_actions(555)
            acts.append((a0.clone(), a1.clone()))
            g.step(a0, a1)
            g.world_state(out=worlds[t])
        torch.cuda.synchronize()
    finally:
        _lib.load().ppg_set_pdl_chain(before)
    ora = Oracle(cfg, B, threads=8)
    ora.reset()
    for t in range(T):
        n = ora.outputs()["n"]
        A0 = np.zeros(max(1, n[0]), np.int32); A0[: n[0]] = acts[t][0][: n[0]].cpu().numpy()
        A1 = np.zeros(max(1, n[1]), np.int32); A1[: n[1]] = acts[t][1][: n[1]].cpu().numpy()
        ora.step(A0, A1)
        _assert_world(worlds[t].cpu().numpy(), _oracle_world(ora, range(B)), f"queued step {t} (chain {chain})")
    g.close(); ora.close()


def test_world_state_does_not_change_the_outputs():
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from tests.parity import compare_outputs

    cfg = make_config(STAG_CONFIG, variant=VARIANT_STAG, cap_live=(64, 160), seed=8)
    a, b = BatchedPredPreyGrass(cfg, 256), BatchedPredPreyGrass(cfg, 256)
    a.reset(); b.reset()
    for t in range(40):
        a.step(*a.random_actions(9))
        a.world_state()
        b.step(*b.random_actions(9))
        compare_outputs(a.outputs_numpy(), b.outputs_numpy(), f"step {t}")
    a.close(); b.close()


def test_world_state_errors():
    import torch

    from predpreygrass_b200._lib import PpgError
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g = BatchedPredPreyGrass(make_config(BASE_CONFIG, cap_live=(64, 192), seed=1), 16)
    with pytest.raises(PpgError, match="no output since ppg_create"):
        g.world_state()
    g.reset()
    g.step(*g.random_actions(1))
    blob = g.snapshot()
    g.world_state()
    for b, n in ((-1, 2), (0, 0), (0, 17), (16, 1), (10, 7)):
        with pytest.raises(PpgError, match="env range"):
            g.world_state(b, n)
    G = g.cfg.grid_size
    with pytest.raises(ValueError):
        g.world_state(0, 2, out=torch.empty((2, 4, G, G), device=g.device, dtype=torch.float64))
    with pytest.raises(ValueError):
        g.world_state(0, 2, out=torch.empty((2, 4, G, G - 1), device=g.device))
    with pytest.raises(ValueError):
        g.world_state(0, 2, out=torch.empty((2, 4, G, 2 * G), device=g.device)[..., ::2])
    g.restore(blob)
    with pytest.raises(PpgError, match="ppg_restore"):
        g.world_state()
    g.step(*g.random_actions(1))
    g.world_state()
    g.close()
    # a snapshot holding idle envs: their image is never rewritten by a step, only a full reset makes the world valid again
    g = BatchedPredPreyGrass(make_config(dict(BASE_CONFIG, max_steps=3), cap_live=(64, 192), seed=1, autoreset=False), 8)
    g.reset()
    for _ in range(4):
        g.step(*g.random_actions(1))
    blob = g.snapshot()
    g.restore(blob)
    g.step(*g.random_actions(1))
    with pytest.raises(PpgError, match="idle"):
        g.world_state()
    g.reset()
    g.world_state()
    g.close()


# ------------------------------------------------------------------------------------------------ dict adapters
def replay_adapter_grid(name):
    """`grid_world_state` of the dict adapters through a recorded episode (reset(seed) + the recorded draws after it, as
    tests/test_gpu_dict_adapters.py replays them) against the reference's float32 grid"""
    from predpreygrass_b200 import env_evolutionary as E

    z, cfg = load_golden(name)
    fam = cfg.pop("variant")
    stag = fam == "stag"
    if stag:
        caps = (cfg.get("n_possible_type_1_predators", 0) + cfg.get("n_possible_type_2_predators", 0),
                cfg.get("n_possible_type_1_prey", 0) + cfg.get("n_possible_type_2_prey", 0))
    else:
        caps = (cfg["n_possible_predators"], cfg["n_possible_prey"])
    cfg["cap_live"] = (min(caps[0], 224), min(caps[1], 416))
    cls = {"eco": E.PredPreyGrassEco, "stag": E.PredPreyGrassStag, "mr": E.PredPreyGrassMetabolicRate, "inv": E.PredPreyGrassInvestment,
           "coop": E.PredPreyGrassCooperation, "cad": E.PredPreyGrassCadence}[fam]
    env = cls(cfg)
    if stag:
        n1 = (cfg.get("n_possible_type_1_predators", 0), cfg.get("n_possible_type_1_prey", 0))
        sp = ("predator", "prey")
        key = lambda s, i: f"type_1_{sp[s]}_{i}" if i < n1[s] else f"type_2_{sp[s]}_{i - n1[s]}"  # noqa: E731
        env.reset(seed=int(z["seed"]), options={"ppg_tape": (z["step_ints"], z["step_reals"])})
    else:
        key = lambda s, i: f"{('predator', 'prey')[s]}_{i}"  # noqa: E731
        env.reset(seed=int(z["seed"]), options={"ppg_tape": (z["fallback_cells"], z["step_reals"])})
    compared = 0
    for t in range(len(z["steps"])):
        a0, a1 = z["act_off"][t], z["act_off"][t + 1]
        if stag:
            acts = {key(s, i): (int(mv) if s == 1 else (int(mv), int(jn)))
                    for s, i, mv, jn in zip(z["act_s"][a0:a1], z["act_id"][a0:a1], z["act_move"][a0:a1], z["act_join"][a0:a1])}
        else:
            acts = {key(s, i): int(v) for s, i, v in zip(z["act_s"][a0:a1], z["act_id"][a0:a1], z["act_v"][a0:a1])}
        _, _, term, trunc, _ = env.step(acts)
        ended = term["__all__"] or trunc["__all__"]
        if stag or not ended:
            grid = env.grid_world_state
            assert grid.dtype == np.float32 and grid.shape == (env.num_obs_channels, env.grid_size, env.grid_size)
            assert np.array_equal(sha_f32([grid]), z["grid_sha"][t]), (name, t)
            compared += 1
        if ended:
            break
    assert compared > 0
    env.close()


@pytest.mark.parametrize("name", golden_cases(("eco", "stag") + TRAITS))
def test_adapter_grid_world_state_replays_reference(name):
    replay_adapter_grid(name)
