"""`config_env` dict  <->  the POD `ppg_config` of include/ppg.h.

The reference envs read a plain dict with per-key defaults (BASE:22-61,
base_environment/config_env.py:1-38).  The same dict, unchanged, configures this package; it is
flattened once into the C struct the kernels read.
"""
import ctypes as C

import numpy as np

VARIANT_BASE, VARIANT_ECO, VARIANT_STAG = 0, 1, 2
REWARD_SPARSE, REWARD_DENSE, REWARD_DENSE_ADDITIVE, REWARD_SPARSE_KICKBACK = 0, 1, 2, 3

REWARD_MODES = {
    "sparse": REWARD_SPARSE,
    "eating": REWARD_SPARSE,  # sparse_rewards_plus_eating: same code as BASE, constants differ
    "dense": REWARD_DENSE,
    "additive": REWARD_DENSE_ADDITIVE,
    "kickback": REWARD_SPARSE_KICKBACK,
    "seasonal": REWARD_SPARSE,  # base_environment_seasonal: BASE rewards; the season keys of the config select the regrowth cycle
}

ROW_TERMINATED, ROW_TRUNCATED, ROW_NEWBORN, ROW_FOUNDER, ROW_ATE = 0x01, 0x02, 0x04, 0x08, 0x10
ENV_TERMINATED, ENV_TRUNCATED, ENV_RESET, ENV_IDLE = 0x01, 0x02, 0x04, 0x08
STATUS_SLOT_OVERFLOW, STATUS_NO_SPAWN_CELL, STATUS_TAPE_EXHAUSTED, STATUS_BAD_ACTION = 0x01, 0x02, 0x04, 0x08
STATUS_ID_POOL_EMPTY, STATUS_GHOST_CELL = 0x10, 0x20
ROW_CARCASS = 0x20
ROW_REPRODUCED = 0x40
ROW_FROZEN = 0x80  # CAD: the agent's next action mask allows only "stay"
N_STATS = 16
STAT_NAMES = [
    "env_steps", "agent_steps", "episodes", "episode_steps", "births_pred", "births_prey", "starved_pred",
    "starved_prey", "eaten_prey", "grass_eaten", "truncated", "rows_pred", "rows_prey", "spawn_fallback",
    "status_envs", "capture_attempts",
]
# include/ppg.h PPG_EP_*: the episode-returns vector (ppg_episode_stats_device); slots 6 and 7 reduce with MAX, the others with SUM
N_EP_STATS = 16
EP_STAT_NAMES = [
    "episodes", "length_sum", "return_sum", "return_sq_sum", "return_pred", "return_prey", "return_max", "return_neg_min",
    "lives_pred", "deaths_pred", "life_return_pred", "life_rows_pred", "lives_prey", "deaths_prey", "life_return_prey", "life_rows_prey",
]
EP_MAX_SLOTS = (6, 7)


class PpgConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("variant", C.c_int32),
        ("reward_mode", C.c_int32),
        ("grid_size", C.c_int32),
        ("max_steps", C.c_int32),
        ("num_obs_channels", C.c_int32),
        ("obs_range", C.c_int32 * 2),
        ("n_possible", C.c_int32 * 2),
        ("n_initial", C.c_int32 * 2),
        ("n_grass", C.c_int32),
        ("cap_live", C.c_int32 * 2),
        ("autoreset", C.c_int32),
        ("energy_loss", C.c_double * 2),
        ("creation_threshold", C.c_double * 2),
        ("initial_energy", C.c_double * 2),
        ("initial_energy_grass", C.c_double),
        ("energy_gain_grass", C.c_double),
        ("reward_predator_catch_prey", C.c_double),
        ("reward_prey_eat_grass", C.c_double),
        ("reward_predator_step", C.c_double),
        ("reward_prey_step", C.c_double),
        ("penalty_prey_caught", C.c_double),
        ("reproduction_reward", C.c_double * 2),
        ("kickback_reward", C.c_double * 2),
        ("seed", C.c_uint64),
        ("env_index_base", C.c_int32),
        ("reserved0", C.c_int32),
        # ---- ECO ----
        ("action_range", C.c_int32),
        ("genome_enabled", C.c_int32),
        ("include_speed_in_obs", C.c_int32),
        ("max_agent_age", C.c_int32 * 2),
        ("carcass_only_predator_age", C.c_int32),
        ("slow_max_move_distance", C.c_int32),
        ("fast_max_move_distance", C.c_int32),
        ("track_episode_sums", C.c_int32),
        ("reserved1", C.c_int32),
        ("move_cost_per_cell", C.c_double * 2),
        ("move_speed_cost_exponent", C.c_double),
        ("max_energy_grass", C.c_double),
        ("max_energy_gain_per_grass", C.c_double),
        ("max_energy_gain_per_prey", C.c_double),
        ("founder_speed_mean", C.c_double * 2),
        ("founder_speed_std", C.c_double * 2),
        ("mutation_rate", C.c_double),
        ("mutation_std", C.c_double),
        ("speed_bounds", C.c_double * 2),
        ("speed_distance_threshold", C.c_double),
        # ---- STAG ----
        ("n_possible_t", (C.c_int32 * 2) * 2),
        ("n_initial_t", (C.c_int32 * 2) * 2),
        ("type_action_range", C.c_int32 * 2),
        ("team_capture_equal_split", C.c_int32),
        ("coop_trait_enabled", C.c_int32),
        ("team_capture_success_model", C.c_int32),
        ("strict_rllib_output", C.c_int32),
        ("energy_loss_prey_t", C.c_double * 2),
        ("creation_threshold_prey_t", C.c_double * 2),
        ("initial_energy_prey_t", C.c_double * 2),
        ("bite_size_prey_t", C.c_double * 2),
        ("reproduction_reward_t", (C.c_double * 2) * 2),
        ("death_penalty", C.c_double * 3),
        ("team_capture_margin", C.c_double),
        ("team_capture_join_cost", C.c_double),
        ("team_capture_scavenger_fraction", C.c_double),
        ("team_capture_nature_weight", C.c_double),
        ("team_capture_base_success_p0", C.c_double),
        ("team_capture_force_success_ratio", C.c_double),
        ("team_capture_min_success_prob", C.c_double),
        ("coop_trait_init_mean", C.c_double),
        ("coop_trait_init_std", C.c_double),
        ("coop_trait_mutation_std", C.c_double),
        ("coop_trait_mutation_rate", C.c_double),
        ("season_multiplier", C.c_double * 2),
        ("season_length_steps", C.c_int32),
        ("reserved2", C.c_int32),
        # ---- trait variants of eco_evolutionary ----
        ("trait_mode", C.c_int32),
        ("n_initial_min", C.c_int32 * 2),
        ("satiation_cooldown", C.c_int32),
        ("cooperation_range", C.c_int32),
        ("max_cooldown", C.c_int32),
        ("trait_alpha", C.c_double),
        ("repro_max_ratio", C.c_double),
        ("metabolic_speed_coeff", C.c_double),
        ("lineage_reward_coeff", C.c_double * 2),
        ("wall_cells", C.c_void_p),
        ("n_walls", C.c_int32),
        ("respect_los_for_movement", C.c_int32),
        ("include_visibility_channel", C.c_int32),
        ("reserved3", C.c_int32),
    ]


class PpgTape(C.Structure):
    _fields_ = [
        ("cells", C.POINTER(C.c_int32)),
        ("cell_off", C.POINTER(C.c_int64)),
        ("reals", C.POINTER(C.c_double)),
        ("real_off", C.POINTER(C.c_int64)),
    ]


class PpgBuffers(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p * 2),
        ("row_env", C.c_void_p * 2),
        ("row_agent", C.c_void_p * 2),
        ("reward", C.c_void_p * 2),
        ("flags", C.c_void_p * 2),
        ("old_off", C.c_void_p * 2),
        ("new_off", C.c_void_p * 2),
        ("new_cnt", C.c_void_p * 2),
        ("n_rows", C.c_void_p),
        ("env_flags", C.c_void_p),
        ("env_status", C.c_void_p),
        ("env_step", C.c_void_p),
        ("env_count", C.c_void_p),
        ("row_capacity", C.c_int64 * 2),
        ("obs_row_elems", C.c_int32 * 2),
        ("n_envs", C.c_int32),
    ]


class PpgReturns(C.Structure):
    _fields_ = [
        ("row_return", C.c_void_p * 2),
        ("row_life", C.c_void_p * 2),
        ("env_return", C.c_void_p),
        ("env_valid", C.c_void_p),
        ("env_acc", C.c_void_p),
    ]


def _round32(n):
    return max(32, (int(n) + 31) // 32 * 32)


TRAITS = {"speed": 0, "metabolic_rate": 1, "offspring_investment_fraction": 2, "cooperation_rate": 3, "cadence": 4}
TRAIT_SPEED, TRAIT_METABOLIC, TRAIT_INVESTMENT, TRAIT_COOPERATION, TRAIT_CADENCE = 0, 1, 2, 3, 4
# founder mean and bounds each variant's genome.py falls back to (GENOME_FIELD_DEFAULTS / DEFAULT_TRAIT_BOUNDS)
TRAIT_DEFAULTS = {"metabolic_rate": (1.0, (0.5, 2.0)), "offspring_investment_fraction": (0.35, (0.10, 0.80)),
                  "cooperation_rate": (0.0, (0.0, 1.0))}


def make_config(config=None, *, reward_mode="sparse", variant=VARIANT_BASE, cap_live=None, autoreset=True, seed=0,
                env_index_base=0, track_episode_sums=False, trait=None):
    """Flatten a reference `config_env` dict (missing keys take the reference's own defaults,
    BASE:22-61) into a PpgConfig."""
    cfg = dict(config or {})
    g = cfg.get
    if variant == VARIANT_STAG:  # per-type dict values are read by _fill_stag
        g = {k: v for k, v in cfg.items() if not isinstance(v, dict)}.get
    c = PpgConfig()
    c.struct_size = C.sizeof(PpgConfig)
    c.variant = variant
    c.reward_mode = REWARD_MODES[reward_mode] if isinstance(reward_mode, str) else int(reward_mode)
    c.grid_size = g("grid_size", 10)
    c.max_steps = g("max_steps", 10000)
    c.num_obs_channels = g("num_obs_channels", 4)
    c.obs_range[0] = g("predator_obs_range", 7)
    c.obs_range[1] = g("prey_obs_range", 5)
    c.n_possible[0] = g("n_possible_predators", 50)
    c.n_possible[1] = g("n_possible_prey", 50)
    c.n_initial[0] = g("n_initial_active_predator", g("n_initial_active_predators", 6))
    c.n_initial[1] = g("n_initial_active_prey", 8)
    c.n_grass = g("initial_num_grass", 25)
    cap_live_given = cap_live is not None
    if cap_live is None:
        # enough for every cell of the grid to hold one agent of the species (the reference cannot
        # place a newborn without a free cell, BASE:754-766), bounded by the id pool
        cells = c.grid_size * c.grid_size
        cap_live = (min(_round32(cells), _round32(c.n_possible[0])), min(_round32(cells), _round32(c.n_possible[1])))
    c.cap_live[0], c.cap_live[1] = _round32(cap_live[0]), _round32(cap_live[1])
    c.autoreset = 1 if autoreset else 0
    c.energy_loss[0] = g("energy_loss_per_step_predator", 0.15)
    c.energy_loss[1] = g("energy_loss_per_step_prey", 0.05)
    c.creation_threshold[0] = g("predator_creation_energy_threshold", 12.0)
    c.creation_threshold[1] = g("prey_creation_energy_threshold", 8.0)
    c.initial_energy[0] = g("initial_energy_predator", 5.0)
    c.initial_energy[1] = g("initial_energy_prey", 3.0)
    c.initial_energy_grass = g("initial_energy_grass", 2.0)
    c.energy_gain_grass = g("energy_gain_per_step_grass", 0.2)
    c.reward_predator_catch_prey = g("reward_predator_catch_prey", 0.0)
    c.reward_prey_eat_grass = g("reward_prey_eat_grass", 0.0)
    c.reward_predator_step = g("reward_predator_step", 0.0)
    c.reward_prey_step = g("reward_prey_step", 0.0)
    c.penalty_prey_caught = g("penalty_prey_caught", 0.0)
    if variant != VARIANT_ECO:
        c.reproduction_reward[0] = g("reproduction_reward_predator", 10.0)
        c.reproduction_reward[1] = g("reproduction_reward_prey", 10.0)
    c.kickback_reward[0] = g("kickback_reward_predator", 10.0)
    c.kickback_reward[1] = g("kickback_reward_prey", 10.0)
    c.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    c.env_index_base = int(env_index_base)
    c.action_range = 3
    c.max_agent_age[0] = c.max_agent_age[1] = -1
    c.carcass_only_predator_age = -1
    c.slow_max_move_distance = c.fast_max_move_distance = 1
    c.move_speed_cost_exponent = 2.0
    c.max_energy_grass = c.initial_energy_grass  # BASE caps regrowth at the initial energy (BASE:253-255)
    c.max_energy_gain_per_grass = c.max_energy_gain_per_prey = float("inf")
    c.speed_bounds[0], c.speed_bounds[1] = 0.5, 2.0
    c.speed_distance_threshold = 1.5
    # base_environment_seasonal (SEASON:63-67): present only in that variant's config_env; 0 = no seasons
    c.season_multiplier[0] = c.season_multiplier[1] = 1.0
    if variant == VARIANT_BASE and "season_length_steps" in cfg:
        c.season_length_steps = int(g("season_length_steps", 40))
        if c.season_length_steps <= 0:
            raise ValueError("season_length_steps must be positive (SEASON:232 divides by it)")
        c.season_multiplier[0] = float(g("season_high_multiplier", 1.5))
        c.season_multiplier[1] = float(g("season_low_multiplier", 0.5))
    c.n_initial_min[0], c.n_initial_min[1] = c.n_initial[0], c.n_initial[1]
    c.repro_max_ratio = -1.0
    c.trait_alpha = 1.0
    if variant == VARIANT_ECO:
        trait = cfg.get("ppg_trait", "speed") if trait is None else trait
        if trait not in TRAITS:
            raise ValueError(f"unknown trait variant {trait!r}")
        if TRAITS[trait] == TRAIT_SPEED:
            _fill_eco(c, cfg)
        else:
            _fill_trait(c, cfg, trait)
        c.track_episode_sums = 1 if track_episode_sums else 0
    if variant == VARIANT_STAG:
        _fill_stag(c, cfg, cap_live_given)
    return c


def _role(value, role, default=None):
    """ECO `_get_role_specific` (ECO:1723-1731): a scalar, or a dict keyed by an agent-id prefix."""
    if isinstance(value, dict):
        for k, v in value.items():
            if role.startswith(k):
                return v
        return default
    return default if value is None else value


def _age(value):
    return -1 if value is None or not isinstance(value, (int, float)) or value < 0 else int(value)


def _fill_eco(c, cfg):
    """ECO `_initialize_from_config` (ECO:36-120) — same keys, same defaults."""
    g = cfg.get
    c.n_initial[0] = cfg["n_initial_active_predators"]
    c.n_initial[1] = cfg["n_initial_active_prey"]
    c.num_obs_channels = cfg["num_obs_channels"]
    c.action_range = cfg["action_range"]
    c.genome_enabled = 1 if g("genome_enabled", True) else 0
    c.include_speed_in_obs = 1 if g("include_speed_in_obs", False) else 0
    caps = {"predator": 120, "prey": 100}  # ECO:51-54 defaults for roles omitted from the dict
    if isinstance(g("max_agent_age"), dict):
        caps.update(g("max_agent_age"))
    c.max_agent_age[0], c.max_agent_age[1] = _age(caps.get("predator")), _age(caps.get("prey"))
    carc = g("carcass_only_predator_age")
    c.carcass_only_predator_age = _age(carc.get("predator")) if isinstance(carc, dict) else -1
    c.slow_max_move_distance = int(g("slow_max_move_distance", 1))
    c.fast_max_move_distance = int(g("fast_max_move_distance", 2))
    c.move_cost_per_cell[0] = float(g("movement_energy_cost_per_cell_predator", 0.0))
    c.move_cost_per_cell[1] = float(g("movement_energy_cost_per_cell_prey", 0.0))
    c.move_speed_cost_exponent = float(g("movement_speed_cost_exponent", 2.0))
    c.max_energy_grass = float(cfg["max_energy_grass"])
    c.max_energy_gain_per_grass = float(g("max_energy_gain_per_grass", float("inf")))
    c.max_energy_gain_per_prey = float(g("max_energy_gain_per_prey", float("inf")))
    for s, role in enumerate(("predator", "prey")):
        f = g("founder_genome", {}).get(role, {})
        c.founder_speed_mean[s] = float(f.get("speed_mean", 1.0))
        c.founder_speed_std[s] = float(f.get("speed_std", 0.0))
    m = g("genome_mutation", {})
    c.mutation_rate, c.mutation_std = float(m.get("rate", 0.0)), float(m.get("std", 0.0))
    b = g("trait_bounds", {}).get("speed", (0.5, 2.0))
    c.speed_bounds[0], c.speed_bounds[1] = float(b[0]), float(b[1])
    c.speed_distance_threshold = float(g("speed_distance_threshold", 1.5))
    # ECO reads only the reproduction rewards and the lineage coefficient from the config (ECO:47-50);
    # `_get_role_specific` finds no `*_config` attribute for the other reward keys and returns 0.0 (ECO:1724)
    c.reward_predator_catch_prey = c.reward_prey_eat_grass = c.reward_predator_step = c.reward_prey_step = 0.0
    c.penalty_prey_caught = 0.0
    c.reproduction_reward[0] = float(_role(cfg["reproduction_reward_predator"], "predator", 0.0))
    c.reproduction_reward[1] = float(_role(cfg["reproduction_reward_prey"], "prey", 0.0))
    lin = cfg["lineage_reward_coeff"]  # ECO:52 (mandatory key)
    for s, role in enumerate(("predator", "prey")):
        c.lineage_reward_coeff[s] = float(_role(lin, role, 0.0) or 0.0)  # `_get_role_specific` (ECO:1723-1731)


def _fill_cadence(c, cfg):
    """`_initialize_from_config` of eco_evolutionary_cadence (CAD:44-124): ECO's keys and defaults without the carcass /
    lineage / distance-gating ones, plus `max_cooldown` and `metabolic_speed_coeff`."""
    g = cfg.get
    _fill_eco(c, dict(cfg, lineage_reward_coeff=0.0))
    c.trait_mode = TRAIT_CADENCE
    c.carcass_only_predator_age = -1
    d = (int(c.action_range) - 1) // 2
    c.slow_max_move_distance = c.fast_max_move_distance = max(d, 0)  # `_get_move` does not clip the move vector (CAD:708-731)
    c.speed_distance_threshold = float("inf")
    c.max_energy_gain_per_prey = float("inf")   # CAD:857: the whole prey
    c.max_cooldown = int(g("max_cooldown", 10))
    if c.max_cooldown < 1:
        raise ValueError("max_cooldown must be >= 1")
    c.metabolic_speed_coeff = float(g("metabolic_speed_coeff", 1.0))
    c.n_initial_min[0], c.n_initial_min[1] = c.n_initial[0], c.n_initial[1]


def _fill_trait(c, cfg, trait):
    """`_initialize_from_config` of the other trait variants (MR:38-114, INV:38-114, COOP:38-98; mandatory keys are read
    with `cfg[...]` exactly where the reference does, so a missing one raises KeyError here as well)."""
    g = cfg.get
    mode = TRAITS[trait]
    if mode == TRAIT_CADENCE:
        return _fill_cadence(c, cfg)
    c.trait_mode = mode
    c.max_steps = cfg["max_steps"]
    c.n_initial[0] = cfg["n_initial_active_predators"]
    c.n_initial[1] = cfg["n_initial_active_prey"]
    # MR:74-81: ~33 % of the maximum unless configured; MR:189-190 clamps to the maximum
    c.n_initial_min[0] = min(int(g("n_initial_active_predators_min", max(1, c.n_initial[0] // 3))), c.n_initial[0])
    c.n_initial_min[1] = min(int(g("n_initial_active_prey_min", max(1, c.n_initial[1] // 3))), c.n_initial[1])
    if c.n_initial_min[0] < 0 or c.n_initial_min[1] < 0:
        raise ValueError("n_initial_active_*_min must be >= 0")
    c.n_possible[0], c.n_possible[1] = cfg["n_possible_predators"], cfg["n_possible_prey"]
    c.grid_size = cfg["grid_size"]
    c.num_obs_channels = cfg["num_obs_channels"]
    c.obs_range[0], c.obs_range[1] = cfg["predator_obs_range"], cfg["prey_obs_range"]
    c.n_grass = cfg["initial_num_grass"]
    c.initial_energy_grass = cfg["initial_energy_grass"]
    c.energy_gain_grass = cfg["energy_gain_per_step_grass"]
    c.max_energy_grass = float(cfg["max_energy_grass"])
    c.action_range = cfg["action_range"]
    c.genome_enabled = 1 if g("genome_enabled", True) else 0
    c.include_speed_in_obs = 0
    c.max_agent_age[0] = c.max_agent_age[1] = -1   # ages are counted (MR:570) but nothing expires
    c.carcass_only_predator_age = -1
    d = (int(c.action_range) - 1) // 2
    c.slow_max_move_distance = c.fast_max_move_distance = max(d, 0)  # no distance gating: `_get_move` (MR:590-614) has none
    c.move_cost_per_cell[0] = float(g("movement_energy_cost_per_cell_predator", 0.0))
    c.move_cost_per_cell[1] = float(g("movement_energy_cost_per_cell_prey", 0.0))
    c.move_speed_cost_exponent = 1.0
    c.max_energy_gain_per_grass = float("inf")
    if mode == TRAIT_INVESTMENT:
        c.energy_loss[0], c.energy_loss[1] = cfg["energy_loss_per_step_predator"], cfg["energy_loss_per_step_prey"]
        c.initial_energy[0], c.initial_energy[1] = cfg["initial_energy_predator_at_reset"], cfg["initial_energy_prey_at_reset"]
    else:
        c.energy_loss[0], c.energy_loss[1] = cfg["basal_energy_cost_predator"], cfg["basal_energy_cost_prey"]
        c.initial_energy[0], c.initial_energy[1] = cfg["initial_energy_predator"], cfg["initial_energy_prey"]
    c.creation_threshold[0] = cfg["predator_creation_energy_threshold"]
    c.creation_threshold[1] = cfg["prey_creation_energy_threshold"]
    if mode in (TRAIT_METABOLIC, TRAIT_INVESTMENT):
        c.satiation_cooldown = int(g("predator_satiation_cooldown", 0))
        c.max_energy_gain_per_prey = float(g("max_energy_gain_per_prey", float("inf")))
        if not 0 <= c.satiation_cooldown <= 250:
            raise ValueError("predator_satiation_cooldown must be in [0, 250]")
    else:
        c.satiation_cooldown = 0
        c.max_energy_gain_per_prey = float("inf")   # COOP:777: the whole prey
    if mode == TRAIT_METABOLIC:
        c.trait_alpha = float(g("metabolic_rate_alpha", 0.7))
        r = g("predator_reproduction_max_ratio", None)
        c.repro_max_ratio = -1.0 if r is None else float(r)
        if r is not None and float(r) < 0:
            raise ValueError("predator_reproduction_max_ratio must be >= 0 or None")
    if mode == TRAIT_COOPERATION:
        c.cooperation_range = int(g("cooperation_range", 2))
    if g("genome_neutral_drift_control", False):
        raise ValueError("genome_neutral_drift_control (the neutral-drift null model, MR:108-114) is not supported")
    default_mean, default_bounds = TRAIT_DEFAULTS[trait]
    for s, role in enumerate(("predator", "prey")):
        f = g("founder_genome", {}).get(role, {})
        c.founder_speed_mean[s] = float(f.get(f"{trait}_mean", default_mean))
        c.founder_speed_std[s] = float(f.get(f"{trait}_std", 0.0))
    m = g("genome_mutation", {})
    c.mutation_rate, c.mutation_std = float(m.get("rate", 0.0)), float(m.get("std", 0.0))
    b = g("trait_bounds", {}).get(trait, default_bounds)
    c.speed_bounds[0], c.speed_bounds[1] = float(b[0]), float(b[1])
    c.speed_distance_threshold = float("inf")
    c.reward_predator_catch_prey = c.reward_prey_eat_grass = c.reward_predator_step = c.reward_prey_step = 0.0
    c.penalty_prey_caught = 0.0
    c.reproduction_reward[0] = float(_role(cfg["reproduction_reward_predator"], "predator", 0.0))
    c.reproduction_reward[1] = float(_role(cfg["reproduction_reward_prey"], "prey", 0.0))


CAPTURE_MODELS = {"deterministic": 0, "probabilistic": 1, "hybrid": 2}


def _by_type(value, kind, default, fallback_key="type_1"):
    """STAG per-type config values: a scalar applies to both types, a dict is keyed `type_1_<kind>` / `type_2_<kind>`
    with the reference's own fallbacks (STAG:38-97)."""
    if isinstance(value, dict):
        return [float(value.get(f"type_{t}_{kind}", default)) for t in (1, 2)]
    v = default if value is None else float(value)
    return [v, v]


def _fill_stag(c, cfg, cap_live_given):
    """STAG `__init__` (STAG:19-266) — same keys, same defaults, same clamps."""
    g = cfg.get
    c.grid_size = g("grid_size", 0)
    # `_create_wall_positions` (STAG:2107-2127): the in-bounds manual positions, duplicates dropped; `num_walls` and
    # `wall_placement_mode` are read by the reference (STAG:172-173) but never used
    walls = []
    for x, y in (g("manual_wall_positions") or []):
        if 0 <= x < c.grid_size and 0 <= y < c.grid_size and int(x) * c.grid_size + int(y) not in walls:
            walls.append(int(x) * c.grid_size + int(y))
    c._walls = np.asarray(sorted(walls), np.int32)  # kept alive with the config object
    c.n_walls = len(walls)
    c.wall_cells = c._walls.ctypes.data if walls else None
    c.respect_los_for_movement = 1 if g("respect_los_for_movement", False) else 0
    c.include_visibility_channel = 1 if g("include_visibility_channel", False) else 0
    # mask_observation_with_visibility multiplies by the reference's masks, which are all ones (computed before any wall
    # exists, STAG:408-412): accepted, no effect
    c.max_steps = g("max_steps", 0)
    c.num_obs_channels = max(int(g("num_obs_channels", 0)), 5)  # STAG:118-119
    c.obs_range[0], c.obs_range[1] = g("predator_obs_range", 0), g("prey_obs_range", 0)
    for s, (poss, init) in enumerate((("n_possible_type_{}_predators", "n_initial_active_type_{}_predator"),
                                      ("n_possible_type_{}_prey", "n_initial_active_type_{}_prey"))):
        for t in (1, 2):
            c.n_possible_t[s][t - 1] = int(g(poss.format(t), 0))
            c.n_initial_t[s][t - 1] = int(g(init.format(t), 0))
        c.n_possible[s] = c.n_possible_t[s][0] + c.n_possible_t[s][1]
        c.n_initial[s] = c.n_initial_t[s][0] + c.n_initial_t[s][1]
        if c.n_possible[s] > 65535:
            raise ValueError("more than 65535 possible agents of one species")
    if not cap_live_given:
        cells = c.grid_size * c.grid_size
        c.cap_live[0] = min(_round32(cells), _round32(c.n_possible[0]))
        c.cap_live[1] = min(_round32(cells), _round32(c.n_possible[1]))
    c.n_grass = g("initial_num_grass", 0)
    c.type_action_range[0], c.type_action_range[1] = int(g("type_1_action_range", 0)), int(g("type_2_action_range", 0))
    c.action_range = max(c.type_action_range[0], c.type_action_range[1])
    c.energy_loss[0] = float(g("energy_loss_per_step_predator", 0.0))
    loss = g("energy_loss_per_step_prey", 0.0)
    c.energy_loss_prey_t[0], c.energy_loss_prey_t[1] = _by_type(loss, "prey", 0.0)
    c.energy_loss[1] = c.energy_loss_prey_t[0]
    c.creation_threshold[0] = float(g("energy_treshold_creation_predator", g("predator_creation_energy_threshold", 0.0)))
    thr = g("energy_treshold_creation_prey", None)
    if thr is None:
        thr = g("prey_creation_energy_threshold", 0.0)
    c.creation_threshold_prey_t[0], c.creation_threshold_prey_t[1] = _by_type(thr, "prey", 0.0)
    c.creation_threshold[1] = c.creation_threshold_prey_t[0]
    c.initial_energy[0] = float(g("initial_energy_predator", 0.0))
    c.initial_energy_prey_t[0], c.initial_energy_prey_t[1] = _by_type(g("initial_energy_prey", 0.0), "prey", 0.0)
    c.initial_energy[1] = c.initial_energy_prey_t[0]
    c.bite_size_prey_t[0], c.bite_size_prey_t[1] = _by_type(g("bite_size_prey", float("inf")), "prey", float("inf"))
    c.death_penalty[0] = float(g("death_penalty_predator", 0.0))
    c.death_penalty[1] = float(g("death_penalty_type_1_prey", 0.0))
    c.death_penalty[2] = float(g("death_penalty_type_2_prey", 0.0))
    for s, (key, kind) in enumerate((("reproduction_reward_predator", "predator"), ("reproduction_reward_prey", "prey"))):
        v = g(key, 0.0)
        if isinstance(v, dict):  # `_get_type_specific` (STAG:2052-2059): first key the agent id starts with, else KeyError
            for t in (1, 2):
                hit = [val for k, val in v.items() if f"type_{t}_{kind}_0".startswith(k)]
                if not hit and c.n_possible_t[s][t - 1] > 0:
                    raise KeyError(f"Type-specific key 'type_{t}_{kind}' not found under '{key}'")
                c.reproduction_reward_t[s][t - 1] = float(hit[0]) if hit else 0.0
        else:
            c.reproduction_reward_t[s][0] = c.reproduction_reward_t[s][1] = float(v)
        c.reproduction_reward[s] = c.reproduction_reward_t[s][0]
    clamp = lambda v, lo, hi: min(max(float(v), lo), hi)  # noqa: E731
    c.team_capture_margin = float(g("team_capture_margin", 0.0))
    c.team_capture_equal_split = 1 if g("team_capture_equal_split", False) else 0
    c.team_capture_join_cost = max(0.0, float(g("team_capture_join_cost", 0.0)))
    c.team_capture_scavenger_fraction = clamp(g("team_capture_scavenger_fraction", 0.0), 0.0, 1.0)
    c.coop_trait_enabled = 1 if g("coop_trait_enabled", True) else 0
    c.coop_trait_init_mean = float(g("coop_trait_init_mean", 0.6))
    c.coop_trait_init_std = max(0.0, float(g("coop_trait_init_std", 0.12)))
    c.coop_trait_mutation_std = max(0.0, float(g("coop_trait_mutation_std", 0.04)))
    c.coop_trait_mutation_rate = clamp(g("coop_trait_mutation_rate", 1.0), 0.0, 1.0)
    c.team_capture_nature_weight = clamp(g("team_capture_nature_weight", 0.75), 0.0, 1.0)
    c.team_capture_success_model = CAPTURE_MODELS.get(str(g("team_capture_success_model", "hybrid")).lower(), 2)
    c.team_capture_base_success_p0 = clamp(g("team_capture_base_success_p0", 0.6), 1e-6, 1.0 - 1e-6)
    c.team_capture_force_success_ratio = max(float(g("team_capture_force_success_ratio", 1.05)), 0.0)
    c.team_capture_min_success_prob = clamp(g("team_capture_min_success_prob", 0.0), 0.0, 1.0)
    c.strict_rllib_output = 1 if g("strict_rllib_output", False) else 0
    c.max_energy_grass = float(g("max_energy_grass", float("inf")))
    c.initial_energy_grass = float(g("initial_energy_grass", 0.0))
    c.energy_gain_grass = float(g("energy_gain_per_step_grass", 0.0))
    c.reward_predator_catch_prey = c.reward_prey_eat_grass = c.reward_predator_step = c.reward_prey_step = 0.0
    c.penalty_prey_caught = 0.0


# base_environment/config_env.py:1-38 — the BASELINE configs 1 and 2
BASE_CONFIG = {
    "max_steps": 1000,
    "grid_size": 25,
    "num_obs_channels": 4,
    "predator_obs_range": 7,
    "prey_obs_range": 9,
    "reward_predator_catch_prey": 0.0,
    "reward_prey_eat_grass": 0.0,
    "reward_predator_step": 0.0,
    "reward_prey_step": 0.0,
    "penalty_prey_caught": 0.0,
    "reproduction_reward_predator": 10.0,
    "reproduction_reward_prey": 10.0,
    "energy_loss_per_step_predator": 0.15,
    "energy_loss_per_step_prey": 0.05,
    "predator_creation_energy_threshold": 12.0,
    "prey_creation_energy_threshold": 8.0,
    "n_possible_predators": 2000,
    "n_possible_prey": 2000,
    "n_initial_active_predator": 6,
    "n_initial_active_prey": 8,
    "initial_energy_predator": 5.0,
    "initial_energy_prey": 3.0,
    "initial_num_grass": 100,
    "initial_energy_grass": 2.0,
    "energy_gain_per_step_grass": 0.04,
}


# base_environment_seasonal/config_env.py:1-44 — BASE plus the square-wave regrowth cycle
SEASONAL_CONFIG = dict(BASE_CONFIG, season_length_steps=40, season_high_multiplier=1.5, season_low_multiplier=0.5)


def season_multiplier(config, current_step):
    """`_current_season_multiplier` (SEASON:224-234) for a config dict"""
    phase = (current_step // config.get("season_length_steps", 40)) % 2
    return config.get("season_high_multiplier", 1.5) if phase == 0 else config.get("season_low_multiplier", 0.5)


# eco_evolutionary/config/config_env_eco_evolutionary.py:1-88 — BASELINE config 4
ECO_CONFIG = {
    "seed": 41,
    "max_steps": 1000,
    "grid_size": 25,
    "num_obs_channels": 3,
    "predator_obs_range": 7,
    "prey_obs_range": 9,
    "action_range": 5,
    "reproduction_reward_predator": {"predator": 10.0},
    "reproduction_reward_prey": {"prey": 10.0},
    "lineage_reward_coeff": {"predator": 0.0, "prey": 0.0},
    "max_agent_age": {"predator": None, "prey": 400},
    "carcass_only_predator_age": {"predator": None},
    "energy_loss_per_step_predator": 0.20,
    "energy_loss_per_step_prey": 0.05,
    "movement_energy_cost_per_cell_predator": 0.05,
    "movement_energy_cost_per_cell_prey": 0.02,
    "predator_creation_energy_threshold": 12.0,
    "prey_creation_energy_threshold": 8.0,
    "initial_energy_predator": 5.0,
    "initial_energy_prey": 3.0,
    "genome_enabled": True,
    "include_speed_in_obs": True,
    "founder_genome": {"predator": {"speed_mean": 1.0, "speed_std": 0.2}, "prey": {"speed_mean": 1.0, "speed_std": 0.2}},
    "genome_mutation": {"rate": 0.05, "std": 0.1},
    "trait_bounds": {"speed": (0.5, 2.0)},
    "speed_distance_threshold": 1.5,
    "slow_max_move_distance": 1,
    "fast_max_move_distance": 2,
    "movement_speed_cost_exponent": 2.0,
    "max_energy_gain_per_grass": float("inf"),
    "max_energy_gain_per_prey": float("inf"),
    "max_energy_grass": 2.0,
    "n_possible_predators": 400,
    "n_possible_prey": 1200,
    "n_initial_active_predators": 10,
    "n_initial_active_prey": 10,
    "initial_num_grass": 100,
    "initial_energy_grass": 2.0,
    "energy_gain_per_step_grass": 0.04,
    "verbose_engagement": False,
    "verbose_movement": False,
    "verbose_decay": False,
    "verbose_reproduction": False,
    "debug_mode": False,
}


# stag_hunt_forward_view_nature_nurture/config/config_env_stag_hunt_forward_view.py:1-105 — BASELINE config 5
STAG_CONFIG = {
    "seed": 41,
    "max_steps": 1000,
    "strict_rllib_output": True,
    "grid_size": 30,
    "num_obs_channels": 5,
    "predator_obs_range": 9,
    "prey_obs_range": 9,
    "type_1_action_range": 3,
    "type_2_action_range": 3,
    "reproduction_reward_predator": {"type_1_predator": 10.0, "type_2_predator": 0.0},
    "reproduction_reward_prey": {"type_1_prey": 10.0, "type_2_prey": 10.0},
    "death_penalty_predator": 0.0,
    "death_penalty_type_1_prey": 0.0,
    "death_penalty_type_2_prey": 0.0,
    "energy_loss_per_step_predator": 0.08,
    "energy_loss_per_step_prey": {"type_1_prey": 0.1, "type_2_prey": 0.01},
    "energy_treshold_creation_predator": 10.0,
    "energy_treshold_creation_prey": {"type_1_prey": 18.0, "type_2_prey": 2.7},
    "initial_energy_predator": 4.0,
    "initial_energy_prey": {"type_1_prey": 10.0, "type_2_prey": 1.5},
    "bite_size_prey": {"type_1_prey": 3.0, "type_2_prey": 0.3},
    "team_capture_margin": 0.0,
    "team_capture_equal_split": True,
    "team_capture_join_cost": 0.01,
    "team_capture_scavenger_fraction": 0.2,
    "coop_trait_enabled": True,
    "coop_trait_init_mean": 0.6,
    "coop_trait_init_std": 0.12,
    "coop_trait_mutation_std": 0.04,
    "coop_trait_mutation_rate": 1.0,
    "team_capture_nature_weight": 0.75,
    "team_capture_success_model": "hybrid",
    "team_capture_base_success_p0": 0.6,
    "team_capture_force_success_ratio": 1.05,
    "team_capture_min_success_prob": 0.0,
    "max_energy_grass": 3.0,
    "n_possible_type_1_predators": 2000,
    "n_possible_type_2_predators": 0,
    "n_possible_type_1_prey": 1000,
    "n_possible_type_2_prey": 2000,
    "n_initial_active_type_1_predator": 10,
    "n_initial_active_type_2_predator": 0,
    "n_initial_active_type_1_prey": 10,
    "n_initial_active_type_2_prey": 10,
    "initial_num_grass": 100,
    "initial_energy_grass": 3.0,
    "energy_gain_per_step_grass": 0.08,
    "mask_observation_with_visibility": False,
    "include_visibility_channel": False,
    "respect_los_for_movement": False,
    "wall_placement_mode": "manual",
    "num_walls": 0,
    "manual_wall_positions": (),
}


# default config_env of the other heritable-trait variants (the reference's config/config_env_eco_evolutionary.py of each)
_TRAIT_COMMON = {
    "seed": 41, "max_steps": 1000, "grid_size": 25, "num_obs_channels": 3, "predator_obs_range": 7, "prey_obs_range": 9,
    "action_range": 3, "reproduction_reward_predator": {"predator": 10.0}, "reproduction_reward_prey": {"prey": 10.0},
    "movement_energy_cost_per_cell_predator": 0.0, "movement_energy_cost_per_cell_prey": 0.0,
    "predator_creation_energy_threshold": 12.0, "prey_creation_energy_threshold": 8.0, "genome_enabled": True,
    "genome_mutation": {"rate": 0.05, "std": 0.04}, "max_energy_grass": 2.0, "n_possible_prey": 1000,
    "n_initial_active_predators": 6, "n_initial_active_prey": 8, "initial_num_grass": 100, "initial_energy_grass": 2.0,
    "energy_gain_per_step_grass": 0.04, "debug_mode": False,
}
METABOLIC_CONFIG = dict(  # eco_evolutionary_metabolic_rate/config/config_env_eco_evolutionary.py
    _TRAIT_COMMON, ppg_trait="metabolic_rate", basal_energy_cost_predator=0.15, basal_energy_cost_prey=0.05,
    predator_reproduction_max_ratio=None, predator_satiation_cooldown=8, max_energy_gain_per_prey=8.0,
    initial_energy_predator=5.0, initial_energy_prey=3.0, genome_neutral_drift_control=False,
    founder_genome={"predator": {"metabolic_rate_mean": 1.0, "metabolic_rate_std": 0.10},
                    "prey": {"metabolic_rate_mean": 1.0, "metabolic_rate_std": 0.10}},
    trait_bounds={"metabolic_rate": (0.5, 2.0)}, metabolic_rate_alpha=0.4, n_possible_predators=500)
INVESTMENT_CONFIG = dict(  # eco_evolutionary_investment/config/config_env_eco_evolutionary.py
    _TRAIT_COMMON, ppg_trait="offspring_investment_fraction", energy_loss_per_step_predator=0.15, energy_loss_per_step_prey=0.05,
    initial_energy_predator_at_reset=5.0, initial_energy_prey_at_reset=3.0, predator_satiation_cooldown=8,
    max_energy_gain_per_prey=8.0,
    founder_genome={"predator": {"offspring_investment_fraction_mean": 0.35, "offspring_investment_fraction_std": 0.08},
                    "prey": {"offspring_investment_fraction_mean": 0.35, "offspring_investment_fraction_std": 0.08}},
    trait_bounds={"offspring_investment_fraction": (0.10, 0.80)}, n_possible_predators=200,
    verbose_engagement=False, verbose_movement=False, verbose_decay=False, verbose_reproduction=False)
COOPERATION_CONFIG = dict(  # eco_evolutionary_cooperation/config/config_env_eco_evolutionary.py
    _TRAIT_COMMON, ppg_trait="cooperation_rate", basal_energy_cost_predator=0.15, basal_energy_cost_prey=0.05,
    initial_energy_predator=5.0, initial_energy_prey=3.0,
    founder_genome={"predator": {"cooperation_rate_mean": 0.0, "cooperation_rate_std": 0.05},
                    "prey": {"cooperation_rate_mean": 0.0, "cooperation_rate_std": 0.05}},
    trait_bounds={"cooperation_rate": (0.0, 1.0)}, cooperation_range=2, n_possible_predators=500)
CADENCE_CONFIG = {  # eco_evolutionary_cadence/config/config_env_eco_evolutionary.py
    "ppg_trait": "cadence", "seed": 41, "max_steps": 1000, "grid_size": 25, "num_obs_channels": 3, "predator_obs_range": 7,
    "prey_obs_range": 9, "action_range": 3, "reproduction_reward_predator": {"predator": 10.0},
    "reproduction_reward_prey": {"prey": 10.0}, "max_agent_age": {"predator": None, "prey": 400},
    "energy_loss_per_step_predator": 0.20, "energy_loss_per_step_prey": 0.05, "movement_energy_cost_per_cell_predator": 0.05,
    "movement_energy_cost_per_cell_prey": 0.02, "predator_creation_energy_threshold": 12.0, "prey_creation_energy_threshold": 8.0,
    "initial_energy_predator": 5.0, "initial_energy_prey": 3.0, "genome_enabled": True, "include_speed_in_obs": True,
    "founder_genome": {"predator": {"speed_mean": 0.75, "speed_std": 0.1}, "prey": {"speed_mean": 0.5, "speed_std": 0.1}},
    "genome_mutation": {"rate": 0.05, "std": 0.05}, "trait_bounds": {"speed": (0.0, 1.0)}, "max_cooldown": 10,
    "movement_speed_cost_exponent": 2.0, "metabolic_speed_coeff": 0.3, "max_energy_gain_per_grass": float("inf"),
    "max_energy_grass": 2.0, "n_possible_predators": 400, "n_possible_prey": 1200, "n_initial_active_predators": 10,
    "n_initial_active_prey": 10, "initial_num_grass": 100, "initial_energy_grass": 2.0, "energy_gain_per_step_grass": 0.04,
    "verbose_engagement": False, "verbose_movement": False, "verbose_decay": False, "verbose_reproduction": False,
    "debug_mode": False, "record_step_data": False,
}
TRAIT_CONFIGS = {"metabolic": METABOLIC_CONFIG, "investment": INVESTMENT_CONFIG, "cooperation": COOPERATION_CONFIG,
                 "cadence": CADENCE_CONFIG}
