"""ppg_snapshot / ppg_restore of the optional state arrays on the GPU (`-m gpu`): BASE kickback (ag_par), ECO lineage rewards
(lin_*), the cadence variant (ag_acc) and ECO episode sums (ep_sums).  After a restore the handle replays the steps that
followed the snapshot bit for bit: every output and every per-env reader."""
import numpy as np
import pytest

from predpreygrass_b200.config import BASE_CONFIG, CADENCE_CONFIG, ECO_CONFIG, VARIANT_ECO, make_config

pytestmark = pytest.mark.gpu

ECO_RICH = dict(ECO_CONFIG, energy_gain_per_step_grass=0.3, prey_creation_energy_threshold=5.0, predator_creation_energy_threshold=8.0,
                energy_loss_per_step_predator=0.1)
CASES = {
    "base_kickback": lambda: make_config(BASE_CONFIG, reward_mode="kickback", cap_live=(64, 192), seed=3),
    "eco_lineage": lambda: make_config(dict(ECO_RICH, lineage_reward_coeff={"predator": 0.5, "prey": 0.25}), variant=VARIANT_ECO,
                                       cap_live=(128, 320), seed=5),
    "cadence": lambda: make_config(CADENCE_CONFIG, variant=VARIANT_ECO, cap_live=(64, 160), seed=7),
    "eco_episode_sums": lambda: make_config(ECO_RICH, variant=VARIANT_ECO, cap_live=(128, 320), seed=11, track_episode_sums=True),
}
N_ENVS, WARMUP, K = 128, 40, 12
READ_ENVS = (0, 1, N_ENVS // 2, N_ENVS - 1)


def _readers(g, name):
    res = []
    for env in READ_ENVS:
        if name == "base_kickback":
            res.append(g.read_env(env))
            continue
        res.append(g.read_env_eco(env))
        if name == "cadence":
            res.append(g.read_env_acc(env))
        if name == "eco_episode_sums":
            res.append(g.read_episode_eco(env))
            res.append(g.read_episode_events_eco(env))
    return res


def _assert_bit_identical(a, b, where):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), where
        for k in a:
            _assert_bit_identical(a[k], b[k], f"{where} {k}")
    elif isinstance(a, (tuple, list)):
        assert len(a) == len(b), where
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_bit_identical(x, y, f"{where}[{i}]")
    else:
        x, y = np.asarray(a), np.asarray(b)
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), where


@pytest.mark.parametrize("name", list(CASES))
def test_snapshot_restore_replays_bit_identically(name):
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g = BatchedPredPreyGrass(CASES[name](), N_ENVS)
    g.reset()
    for t in range(WARMUP):
        g.step(*g.random_actions(99))
    blob = g.snapshot()
    ref = []
    for t in range(K):
        g.step(*g.random_actions(5))
        ref.append((g.outputs_numpy(), _readers(g, name)))
    g.restore(blob)
    for t in range(K):
        g.step(*g.random_actions(5))
        _assert_bit_identical((g.outputs_numpy(), _readers(g, name)), ref[t], f"{name} step {t}")
    g.close()
