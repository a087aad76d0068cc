/*
 * ppg.h — C-ABI of the B200-native batched PredPreyGrass environment step.
 *
 * This is the drop-in boundary for the one hot path of doesburg11/PredPreyGrass:
 * `PredPreyGrass.reset()/step()` of the RLlib MultiAgentEnv classes.  The reference is pure
 * Python and has no FFI of its own; each entry point below names the reference interface it
 * replaces (paths relative to the reference checkout):
 *
 *   BASE = predpreygrass/non_evolutionary/base_environment/predpreygrass_rllib_env.py
 *   ADD  = predpreygrass/non_evolutionary/project_reward_shaping/
 *            base_environment_dense_rewards_additive/predpreygrass_rllib_env.py
 *   ECO  = predpreygrass/evolutionary/eco_evolutionary/predpreygrass_rllib_env.py
 *   STAG = predpreygrass/evolutionary/stag_hunt_forward_view_nature_nurture/predpreygrass_rllib_env.py
 *
 * Plain pointers and sizes only; no torch types.  A handle owns the state of `n_envs`
 * independent environment instances on one CUDA device (structure-of-arrays in HBM) and the
 * output buffers of the last step.  A handle is not thread-safe; all work is stream-ordered
 * on the stream passed to the call and no call synchronises the host unless it says so.
 *
 * Row model (replaces the reference's per-agent dicts, BASE:451-463): every step produces,
 * per species, a compact batch of ROWS, one per agent that appears in that step's
 * observation dict.  Rows [0, n_old) are agents that were alive when the step started, grouped
 * by environment (ascending env index) and, inside an environment, in the reference's
 * observation-dict order (BASE: lexicographic agent-id string order, BASE:459,468).  Rows
 * [n_old, n_old+n_new) are this step's newborns, grouped by environment (ascending env index), in
 * birth order (BASE:398,427 append them after the sorted survivors).  An agent's action for the next
 * step is read from `actions[species][row]` of the row it occupied in THIS step's output,
 * so `actions = policy(obs)` needs no gather.
 */
#ifndef PPG_H_
#define PPG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPG_ABI_VERSION 10

/* species index used throughout */
#define PPG_PREDATOR 0
#define PPG_PREY 1

/* which reference env class the handle reproduces */
enum {
  PPG_VARIANT_BASE = 0, /* BASE / project_reward_shaping family (one kernel, reward_mode flag) */
  PPG_VARIANT_ECO = 1,  /* ECO: heritable speed trait, 25 actions, ageing, carcasses */
  PPG_VARIANT_STAG = 2  /* STAG: two prey types, join_hunt team capture, forward view */
};

/* reward_mode (BASE family): which project_reward_shaping variant */
enum {
  PPG_REWARD_SPARSE = 0,         /* BASE:288,322,328,341,365,375,409,438 (also plus_eating: constants only) */
  PPG_REWARD_DENSE = 1,          /* base_environment_dense_rewards/...:244,291,329,446-449 */
  PPG_REWARD_DENSE_ADDITIVE = 2, /* ADD:256,308,346,419,450,468-471 */
  PPG_REWARD_SPARSE_KICKBACK = 3 /* base_environment_sparse_rewards_plus_kickback/...:434-449 */
};

/* per-row flag bits (ppg_buffers.flags) */
#define PPG_ROW_TERMINATED 0x01u /* terminations[agent] == True (BASE:289,332) */
#define PPG_ROW_TRUNCATED 0x02u  /* truncations[agent] == True (BASE:232; ECO:452-472) */
#define PPG_ROW_NEWBORN 0x04u    /* born this step (BASE:396-414) */
#define PPG_ROW_FOUNDER 0x08u    /* row produced by reset(), not by step() (BASE:215) */
#define PPG_ROW_ATE 0x10u        /* member of agents_just_ate (BASE:319,362) */
#define PPG_ROW_CARCASS 0x20u    /* ECO: member of dead_prey after the step (bitten, not fully eaten; ECO:826-845) */
#define PPG_ROW_REPRODUCED 0x40u /* the agent had an offspring this step (BASE:396-409; ECO:1161 `agent_offspring_counts[agent] += 1`) */
#define PPG_ROW_FROZEN 0x80u     /* CAD: the agent's action mask allows only "stay" in its next step (move accumulator + rate < 1; CAD:577-585,746-753) */

/* per-env flag bits (ppg_buffers.env_flags), describe the step that just ran */
#define PPG_ENV_TERMINATED 0x01u /* terminations["__all__"] (BASE:466) */
#define PPG_ENV_TRUNCATED 0x02u  /* truncations["__all__"]: step counter reached max_steps (BASE:228-238) */
#define PPG_ENV_RESET 0x04u      /* this call performed reset() for the env instead of step() */
#define PPG_ENV_IDLE 0x08u       /* episode over, autoreset off: env produced no rows */

/* sticky per-env status bits (ppg_buffers.env_status) — in-kernel conditions the reference
 * would raise on (SURVEY §5 "failure detection") */
#define PPG_STATUS_SLOT_OVERFLOW 0x01u  /* live agents of a species exceeded cap_live: birth suppressed */
#define PPG_STATUS_NO_SPAWN_CELL 0x02u  /* no free cell for a newborn (reference: TypeError, BASE:766) */
#define PPG_STATUS_TAPE_EXHAUSTED 0x04u /* replay tape ran out; Philox stream used instead */
#define PPG_STATUS_BAD_ACTION 0x08u     /* action outside the action space (reference: KeyError, BASE:502) */
#define PPG_STATUS_ID_POOL_EMPTY 0x10u  /* ECO: id pool exhausted, birth suppressed (reference: SystemExit, ECO:1104-1111) */
#define PPG_STATUS_GHOST_CELL 0x20u     /* ECO: more than 16 stale prey-channel cells at once in one env (a prey that aged out and was
                                         * bitten under a finite intake cap in the same step leaves its grid value behind, ECO:826-832
                                         * after :1060-1090; the device carries up to 16 such ghost cells per env, ppg_eco.cu) */

/* error codes */
#define PPG_OK 0
#define PPG_ERR_INVALID 1  /* bad argument / config (reference: ValueError, BASE:167-168) */
#define PPG_ERR_CUDA 2     /* CUDA runtime error, see ppg_last_error */
#define PPG_ERR_NO_DEVICE 3
#define PPG_ERR_STATE 4    /* call not valid in the handle's current state */

/*
 * Flattened `config_env` dict (BASE:22-61; base_environment/config_env.py:1-38).  Index [0] is
 * the predator value, [1] the prey value of the corresponding `*_predator` / `*_prey` key.
 */
typedef struct ppg_config {
  uint32_t struct_size; /* sizeof(ppg_config), ABI check */
  int32_t variant;      /* PPG_VARIANT_* */
  int32_t reward_mode;  /* PPG_REWARD_* */
  int32_t grid_size;    /* "grid_size" */
  int32_t max_steps;    /* "max_steps" */
  int32_t num_obs_channels; /* "num_obs_channels" (4 for BASE: wall, predator, prey, grass) */
  int32_t obs_range[2];     /* "predator_obs_range", "prey_obs_range" (odd) */
  int32_t n_possible[2];    /* "n_possible_predators", "n_possible_prey" (agent-id pool) */
  int32_t n_initial[2];     /* "n_initial_active_predator", "n_initial_active_prey" */
  int32_t n_grass;          /* "initial_num_grass" */
  int32_t cap_live[2];      /* device slot capacity per env and species (multiple of 32) */
  int32_t autoreset;        /* 1: an env whose episode ended resets itself on the next ppg_step */
  double energy_loss[2];        /* "energy_loss_per_step_*" */
  double creation_threshold[2]; /* "*_creation_energy_threshold" */
  double initial_energy[2];     /* "initial_energy_*" */
  double initial_energy_grass;  /* "initial_energy_grass" (also the regrowth cap, BASE:253-255) */
  double energy_gain_grass;     /* "energy_gain_per_step_grass" */
  double reward_predator_catch_prey;
  double reward_prey_eat_grass;
  double reward_predator_step;
  double reward_prey_step;
  double penalty_prey_caught;
  double reproduction_reward[2]; /* "reproduction_reward_*" */
  double kickback_reward[2];     /* "kickback_reward_*" (plus_kickback variant only) */
  uint64_t seed;                 /* Philox key for normal (non-replay) runs */
  int32_t env_index_base;        /* global index of this handle's env 0: the Philox streams are keyed by
                                  * env_index_base + env, so a job sharded over several handles / GPUs
                                  * produces the same trajectories as one handle owning all envs */
  int32_t reserved0;
  /* ---- ECO (eco_evolutionary/config/config_env_eco_evolutionary.py:1-88; ECO:36-120).  Ignored by the BASE family. ---- */
  int32_t action_range;           /* "action_range" (ECO:102, 5 -> 25 actions `a -> (a // R - d, a % R - d)`, ECO:225-232); BASE: 3 */
  int32_t genome_enabled;         /* "genome_enabled" (ECO:103) */
  int32_t include_speed_in_obs;   /* "include_speed_in_obs" (ECO:112): one extra constant plane after the grid channels (ECO:707-711) */
  int32_t max_agent_age[2];       /* "max_agent_age" per role, -1 = None = unlimited (ECO:51-63,1042-1058) */
  int32_t carcass_only_predator_age; /* "carcass_only_predator_age"["predator"], -1 = None (ECO:65-72,1060-1090) */
  int32_t slow_max_move_distance; /* ECO:110 */
  int32_t fast_max_move_distance; /* ECO:111 */
  int32_t track_episode_sums;     /* 1: keep per-episode totals of distance moved / locomotion energy per species on the device
                                   * (the inputs of `_build_episode_training_metrics`, ECO:1613-1661; read by ppg_read_episode_eco) */
  int32_t reserved1;
  double move_cost_per_cell[2];   /* "movement_energy_cost_per_cell_*" (ECO:78-79,565-573) */
  double move_speed_cost_exponent;/* "movement_speed_cost_exponent" (ECO:80,559-563) */
  double max_energy_grass;        /* "max_energy_grass": regrowth cap (ECO:83,618-626) */
  double max_energy_gain_per_grass; /* intake caps, +inf = none (ECO:909-911, ECO:812-814) */
  double max_energy_gain_per_prey;
  double founder_speed_mean[2];   /* "founder_genome"[role]["speed_mean"/"speed_std"] (genome.py:42-46) */
  double founder_speed_std[2];
  double mutation_rate;           /* "genome_mutation"["rate"/"std"] (genome.py:49-59) */
  double mutation_std;
  double speed_bounds[2];         /* "trait_bounds"["speed"] (genome.py:37-39); also the observation normalisation (ECO:113-115) */
  double speed_distance_threshold;/* ECO:109,551-557 */
  /* ---- STAG (stag_hunt_forward_view_nature_nurture/config/config_env_stag_hunt_forward_view.py:1-105; STAG:19-266).
   * Ignored by the other variants.  Index [t] = agent type t+1 (`type_1_*`, `type_2_*`); for STAG n_possible[s] /
   * n_initial[s] above hold the sums over both types and a numeric agent id is FLAT: `type_1_<species>_k` -> k,
   * `type_2_<species>_k` -> n_possible_t[s][0] + k (STAG:1768-1782 lists possible_agents in exactly this order).
   * Species 1 holds both prey types (type 1 = mammoth, type 2 = rabbit: STAG:112-117 channels 2 and 3). ---- */
  int32_t n_possible_t[2][2];      /* "n_possible_type_{t}_predators", "n_possible_type_{t}_prey" (STAG:26-29) */
  int32_t n_initial_t[2][2];       /* "n_initial_active_type_{t}_predator", "..._prey" (STAG:31-34,373-380) */
  int32_t type_action_range[2];    /* "type_1_action_range", "type_2_action_range" (STAG:178-193): moves a -> (a / R - d, a % R - d) */
  int32_t team_capture_equal_split;/* STAG:132 */
  int32_t coop_trait_enabled;      /* STAG:139 */
  int32_t team_capture_success_model; /* PPG_CAPTURE_* (STAG:153-155) */
  int32_t strict_rllib_output;     /* STAG:126; output assembly (STAG:562-580): when 0 the rewards of agents that ended
                                    * this step (their death penalty) are dropped (STAG:577,609) */
  double energy_loss_prey_t[2];        /* "energy_loss_per_step_prey"[type] (STAG:75-83) */
  double creation_threshold_prey_t[2]; /* "energy_treshold_creation_prey"[type] (STAG:58-73) */
  double initial_energy_prey_t[2];     /* "initial_energy_prey"[type] (STAG:38-53) */
  double bite_size_prey_t[2];          /* "bite_size_prey"[type] (STAG:84-97,1459-1465) */
  double reproduction_reward_t[2][2];  /* "reproduction_reward_predator"/"_prey" by type (STAG:103-104,2052-2059) */
  double death_penalty[3];             /* predator, type_1_prey, type_2_prey (STAG:98-100,1999-2006) */
  double team_capture_margin;          /* STAG:131,1118 */
  double team_capture_join_cost;       /* STAG:133 */
  double team_capture_scavenger_fraction; /* STAG:134-135 */
  double team_capture_nature_weight;   /* STAG:147-148,1133 */
  double team_capture_base_success_p0; /* STAG:156-157,1137 */
  double team_capture_force_success_ratio; /* STAG:158-159,1139 */
  double team_capture_min_success_prob;    /* STAG:160-161,1138 */
  double coop_trait_init_mean;         /* STAG:140,1087 */
  double coop_trait_init_std;          /* STAG:141 */
  double coop_trait_mutation_std;      /* STAG:142,1095-1096 */
  double coop_trait_mutation_rate;     /* STAG:143-144 */
  /* ---- seasonal grass regrowth of the BASE family (SEASON = predpreygrass/non_evolutionary/base_environment_seasonal/
   * predpreygrass_rllib_env.py:63-67,224-234,268-271): `energy_gain_per_step_grass` is multiplied by season_multiplier[0]
   * ("season_high_multiplier") while (current_step / season_length_steps) is even and by season_multiplier[1]
   * ("season_low_multiplier") while it is odd.  season_length_steps = 0: no seasons (BASE). ---- */
  double season_multiplier[2];
  int32_t season_length_steps;         /* "season_length_steps" (SEASON:64) */
  int32_t reserved2;
  /* ---- the other heritable-trait variants of eco_evolutionary (variant == PPG_VARIANT_ECO, trait_mode != PPG_TRAIT_SPEED).
   * MR   = predpreygrass/evolutionary/eco_evolutionary_metabolic_rate/predpreygrass_rllib_env.py
   * INV  = .../eco_evolutionary_investment/predpreygrass_rllib_env.py
   * COOP = .../eco_evolutionary_cooperation/predpreygrass_rllib_env.py
   * CAD  = .../eco_evolutionary_cadence/predpreygrass_rllib_env.py
   * They share ECO's skeleton (same step order, id allocation, spawn rule, mutation law, output assembly) and re-use
   * the ECO fields above for what they have in common: the ONE heritable trait lives where the speed does
   * (founder_speed_mean/std = "<trait>_mean"/"<trait>_std", speed_bounds = "trait_bounds"[<trait>], mutation_rate/std),
   * energy_loss = "basal_energy_cost_*" (MR, COOP) / "energy_loss_per_step_*" (INV, CAD), initial_energy =
   * "initial_energy_*" (MR, COOP, CAD) / "initial_energy_*_at_reset" (INV), max_energy_gain_per_prey (MR:64, INV). ---- */
  int32_t trait_mode;            /* PPG_TRAIT_* */
  int32_t n_initial_min[2];      /* MR:74-81 "n_initial_active_predators_min" / "_prey_min": founders of an episode ~ U{min..n_initial}
                                  * (MR:189-192, two `rng.integers` draws per reset, predators first) */
  int32_t satiation_cooldown;    /* "predator_satiation_cooldown" (MR:63,734-740,756-757; INV), 0 = off */
  int32_t cooperation_range;     /* "cooperation_range" (COOP:93,556-565): Chebyshev radius of meal sharing */
  int32_t max_cooldown;          /* "max_cooldown" (CAD:116,556-571): slowest agents move every max_cooldown-th step */
  double trait_alpha;            /* "metabolic_rate_alpha" (MR:102,751,807): gain = food * rate ** alpha */
  double repro_max_ratio;        /* "predator_reproduction_max_ratio" (MR:60,843-854), < 0 = None */
  double metabolic_speed_coeff;  /* "metabolic_speed_coeff" (CAD:79,626-633): decay *= 1 + coeff * speed */
  /* ---- ECO lineage survival rewards (ECO:943-984,1422-1470): every living agent is paid coeff * (change of its number of
   * living descendants since the last step), on top of its other reward.  0 / 0 (the shipped config): off. ---- */
  double lineage_reward_coeff[2]; /* "lineage_reward_coeff" per role (ECO:52) */
  /* ---- STAG walls and line of sight (STAG:112-124,172-175,860-925,977-994,1026-1037,2107-2160).  Walls are static cells of
   * channel 0: nobody moves or is born onto them and the reset placement avoids them.  respect_los_for_movement: a move
   * that is neither blocked by a wall nor by an occupied cell is cancelled if it cuts a wall corner diagonally or if a wall
   * lies strictly between its end points (integer Bresenham, STAG:892-925).  include_visibility_channel appends one
   * observation channel holding the reference's line-of-sight mask — all ones: the reference computes its masks once in
   * __init__, before any wall exists (STAG:408-412), which also makes mask_observation_with_visibility a no-op. ---- */
  const int32_t* wall_cells;            /* [n_walls] cells x * grid_size + y ("manual_wall_positions", in bounds, distinct); copied by ppg_create */
  int32_t n_walls;
  int32_t respect_los_for_movement;     /* STAG:123 */
  int32_t include_visibility_channel;   /* STAG:122 */
  int32_t reserved3;
} ppg_config;

/* ppg_config.trait_mode: which heritable trait the ECO-family handle carries */
enum {
  PPG_TRAIT_SPEED = 0,       /* ECO: speed gates the move distance (ECO:551-557) */
  PPG_TRAIT_METABOLIC = 1,   /* MR: metabolic_rate scales the basal cost linearly and every energy gain by rate ** alpha */
  PPG_TRAIT_INVESTMENT = 2,  /* INV: offspring_investment_fraction of the parent's energy goes to each child (INV:546-557,890,977) */
  PPG_TRAIT_COOPERATION = 3, /* COOP: cooperation_rate of every meal is shared with same-species neighbours (COOP:537-589) */
  PPG_TRAIT_CADENCE = 4      /* CAD: speed sets the move RATE through an accumulator; action mask in the observation */
};

/* ppg_config.team_capture_success_model (STAG:1141-1148) */
enum { PPG_CAPTURE_DETERMINISTIC = 0, PPG_CAPTURE_PROBABILISTIC = 1, PPG_CAPTURE_HYBRID = 2 };

/* STAG predator action = MultiDiscrete([n_moves, 2]) (STAG:1813-1816) packed into one int32:
 * move | join_hunt << 8  (`_split_action`, STAG:771-799).  Prey: move only. */
#define PPG_STAG_JOIN_SHIFT 8
#define PPG_STAG_ACTION(move, join) ((int32_t)(move) | ((int32_t)((join) != 0) << PPG_STAG_JOIN_SHIFT))

/*
 * Replay tape: the random draws of the reference, captured from its numpy RNG, consumed by the
 * device in the reference's consumption order (SURVEY §8c "Tape contents").  Per env two
 * streams; env e owns cells[cell_off[e] .. cell_off[e+1]) and reals[real_off[e] .. real_off[e+1]).
 *   cells: reset — n_initial[0]+n_initial[1]+n_grass cells `x*grid_size+y` in the order
 *          predators, prey, grass (BASE:185-187; ECO:1752-1762); then one cell per spawn fallback
 *          draw (BASE:764; ECO:759-762).
 *   reals: unused by BASE.  ECO: per reset the founders' speeds in `self.agents` order (predators,
 *          prey; genome.py:42-46, only if genome_enabled), then per birth `u = rng.random()` and,
 *          iff u < mutation_rate, `delta = rng.normal(0, std)` (genome.py:56-58).
 *   STAG cells: reset — the cells (predators, prey, grass; STAG:2140-2148), then one facing index 0..7 per founder
 *          predator (`_predator_facing_options`, STAG:197-206,941,2168); then in consumption order the cell of each
 *          spawn-fallback draw (STAG:1039-1042) and the facing index of each newborn predator (STAG:1559).
 *   STAG reals: reset — the founders' cooperation traits BEFORE clipping (`rng.normal(mean, std)`, STAG:1087; only if
 *          coop_trait_enabled); then per predator birth `u = rng.random()` (iff mutation_std > 0) and, iff
 *          u < mutation_rate, `delta = rng.normal(0, std)` (STAG:1095-1096); per capture attempt `u = rng.random()`
 *          iff the success model draws (STAG:1146,1148: probabilistic always, hybrid unless force-success).
 * All pointers are HOST pointers; the call copies.  When a stream is exhausted the env sets
 * PPG_STATUS_TAPE_EXHAUSTED and continues on the Philox stream.
 */
typedef struct ppg_tape {
  const int32_t* cells;
  const int64_t* cell_off; /* [n_envs+1] */
  const double* reals;
  const int64_t* real_off; /* [n_envs+1] */
} ppg_tape;

/* Device pointers to the outputs of the last ppg_step/ppg_reset; owned by the handle and valid
 * until the next call on it.  [s] = species. */
typedef struct ppg_buffers {
  float* obs[2];         /* [row_capacity[s]][C][R_s][R_s] fp32, index order [c][x][y] (BASE:518-524) */
  int32_t* row_env[2];   /* env index of each row */
  int32_t* row_agent[2]; /* numeric agent id: row is f"predator_{id}" / f"prey_{id}" (BASE:70-72) */
  float* reward[2];      /* rewards[agent] (BASE:460) */
  uint8_t* flags[2];     /* PPG_ROW_* */
  int32_t* old_off[2];   /* [n_envs+1] row range of each env inside [0, n_old) */
  int32_t* new_off[2];   /* [n_envs] first newborn row of the env (absolute row, >= n_old); defined where new_cnt > 0 */
  int32_t* new_cnt[2];   /* [n_envs] newborn rows of the env: rows [new_off, new_off + new_cnt) */
  int32_t* n_rows;       /* [4] = n_old[0], n_old[1], n_new[0], n_new[1] */
  uint8_t* env_flags;    /* [n_envs] PPG_ENV_* */
  uint8_t* env_status;   /* [n_envs] PPG_STATUS_* (sticky until reset of the env) */
  int32_t* env_step;     /* [n_envs] current_step after the call (BASE:471) */
  int32_t* env_count;    /* [n_envs][2] live predators, prey after the call (BASE:210-211) */
  int64_t row_capacity[2];
  int32_t obs_row_elems[2]; /* C*R_s*R_s */
  int32_t n_envs;
} ppg_buffers;

/* Aggregate statistics since ppg_create / last ppg_stats_clear, reduced over the handle's envs on
 * the device (one block-reduce kernel); fixed-size so ranks can all-reduce it (SURVEY §8e). */
#define PPG_N_STATS 16
enum {
  PPG_STAT_ENV_STEPS = 0,     /* real env steps executed (reset calls excluded) */
  PPG_STAT_AGENT_STEPS = 1,   /* agents that acted (alive at step start) summed over env steps */
  PPG_STAT_EPISODES = 2,      /* episodes finished (terminated or truncated) */
  PPG_STAT_EPISODE_STEPS = 3, /* sum of lengths of finished episodes */
  PPG_STAT_BIRTHS_PRED = 4,
  PPG_STAT_BIRTHS_PREY = 5,
  PPG_STAT_STARVED_PRED = 6,
  PPG_STAT_STARVED_PREY = 7,
  PPG_STAT_EATEN_PREY = 8,
  PPG_STAT_GRASS_EATEN = 9,
  PPG_STAT_TRUNCATED = 10,  /* episodes that ended by max_steps */
  PPG_STAT_ROWS_PRED = 11,  /* observation rows written */
  PPG_STAT_ROWS_PREY = 12,
  PPG_STAT_SPAWN_FALLBACK = 13,
  PPG_STAT_STATUS_ENVS = 14, /* envs with a non-zero status word right now */
  PPG_STAT_CAPTURE_ATTEMPTS = 15 /* STAG team_capture_attempts (STAG:1178); 0 for the other variants */
};

typedef struct ppg_handle_s* ppg_handle;

/* PredPreyGrass.__init__(config) (BASE:18-127) for n_envs instances on CUDA device `device`.
 * Validates the config (PPG_ERR_INVALID ~ ValueError BASE:167-168). */
int ppg_create(const ppg_config* cfg, int32_t n_envs, int32_t device, ppg_handle* out);
int ppg_destroy(ppg_handle h);

/* Fills a config with base_environment/config_env.py:1-38 defaults. */
void ppg_default_config(ppg_config* cfg);

/* Loads a replay tape (host pointers), resets the cursors. NULL tape clears it. */
int ppg_load_tape(ppg_handle h, const ppg_tape* tape);

/* PredPreyGrass.reset(seed=...) (BASE:129-217).
 * mask == NULL: resets every env now and writes the founders' observation rows (PPG_ROW_FOUNDER): the output of this
 * call is the reset output of all envs.
 * mask != NULL (host, [n_envs]): SCHEDULES the reset of every env with mask[e] != 0 and returns without producing an
 * output; the next ppg_step performs it — for a masked env that call is reset() instead of step() (PPG_ENV_RESET, its
 * actions are ignored, its rows are the founders' rows), for the others an ordinary step.  This is the lockstep form of
 * "reset the envs whose episode the caller wants to end early"; an env whose episode ended does the same by itself when
 * autoreset is on.
 * seeds (host, [n_envs], may be NULL) re-key the Philox stream of the envs being reset (BASE:135,170). */
int ppg_reset(ppg_handle h, const uint64_t* seeds, const uint8_t* mask, void* cuda_stream);

/* PredPreyGrass.step(action_dict) (BASE:219-473) for all envs in lockstep.
 * actions_pred / actions_prey: DEVICE int32 arrays indexed by the rows of the previous call's
 * output (rows of terminated agents are ignored).  Each live agent must have an action — the
 * contract RLlib's env runner fulfils (an agent missing from action_dict would neither decay nor
 * move, BASE:244,259; that case is not supported).  Movement order inside an env = row order of
 * the previous output (= the observation-dict order a caller iterates, BASE:259). */
int ppg_step(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey, void* cuda_stream);

/* ppg_step with an explicit action-dict iteration order (BASE:244,259 iterate `action_dict.items()`):
 * order_pred / order_prey are DEVICE int32 arrays indexed like the actions; order[row] = position of
 * that agent among its env's acting agents of the same species (a permutation of 0..n-1 per env and
 * species; only the relative order inside a species can change an outcome, BASE:506).  An env whose
 * order is not a permutation falls back to row order and raises PPG_STATUS_BAD_ACTION.  NULL = row order. */
int ppg_step_ordered(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey, const int32_t* order_pred,
                     const int32_t* order_prey, void* cuda_stream);

/* Same step with HOST buffers end to end: copies actions host->device, steps, copies the row
 * batch (obs, ids, rewards, flags, offsets) device->host into `out` (host pointers, pinned
 * recommended, capacities in out->row_capacity) and synchronises the stream.  n_rows_out[4]. */
int ppg_step_host(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey,
                  ppg_buffers* out, int32_t* n_rows_out, void* cuda_stream);

/* Uniform random actions for the rows of the last output (synthetic rollouts: bench, tests).
 * Philox keyed (seed, env, agent id, step) so the choice does not depend on row layout. */
int ppg_random_actions(ppg_handle h, uint64_t seed, int32_t* actions_pred, int32_t* actions_prey,
                       void* cuda_stream);

/* Random-policy rollout driver (the reference's `random_policy.py` loop: `env.step({a: env.action_spaces[a].sample()})`,
 * base_environment/random_policy.py:24-40) for SEVERAL handles at once: n_steps times, for every handle in turn,
 * ppg_random_actions into the handle's own action staging buffers followed by ppg_step, each handle on its own stream
 * (cuda_streams[g], NULL array = the default stream for all).  Handles on different streams overlap on the device:
 * the latency-bound step kernel of one group of envs runs under the bandwidth-bound observation kernel of another
 * (DESIGN.md §3.6).  No host synchronisation; results are exactly those of the same calls made one by one. */
int ppg_rollout_random(ppg_handle* handles, int32_t n_handles, void** cuda_streams, int32_t n_steps, uint64_t seed);

/* Launch chain of a step (process-wide switch, returns the previous setting).  off (default): plain stream order between the
 * steps.  on (PPG_PDL_CHAIN=1): the action kernel and the step kernel are launched with programmatic stream serialization
 * behind the observation kernel of the step before, i.e. their CTAs become resident in the slots that kernel's tail leaves
 * free and wait there (griddepcontrol.wait) until it has completed, which hides the launch ramp (+1 % on the BASE configuration).
 * Results are identical (tests/test_gpu_rollout.py: 55 queued steps against the oracle, chain on and off); the switch is off by
 * default because the last fix to this path (a load the compiler had hoisted above griddepcontrol.wait in the action kernels)
 * landed after the round's measurements.  ppg_rollout_random with n_handles > 1 always runs with the chain off: a parked grid
 * holds SM slots the other streams could use.  No counterpart in the reference (there is no device). */
int ppg_set_pdl_chain(int32_t on);

int ppg_get_buffers(ppg_handle h, ppg_buffers* out);

/* get_state_snapshot()/restore_state_snapshot() (BASE:768-804): the whole SoA slab incl. RNG
 * counters and tape cursors as an opaque host blob.  ppg_snapshot_size gives the byte count.  The blob's header
 * records the byte count and a hash of the shape-defining config fields (n_envs, variant, reward mode, grid, slot
 * capacities, grass patches); ppg_restore refuses (PPG_ERR_INVALID) a blob taken from a handle of another shape. */
size_t ppg_snapshot_size(ppg_handle h);
int ppg_snapshot(ppg_handle h, void* host_blob, size_t bytes, void* cuda_stream);
int ppg_restore(ppg_handle h, const void* host_blob, size_t bytes, void* cuda_stream);

/* Readable state of one env for renderers / tests (BASE attributes agent_positions,
 * agent_energies, grass_positions, grass_energies; random_policy.py:32-39).  Host arrays sized
 * cap_live[s] / n_grass; counts returned in n_live[2]. Synchronises. */
int ppg_read_env(ppg_handle h, int32_t env, int32_t* n_live, int32_t* ids_pred, int32_t* xy_pred,
                 double* energy_pred, int32_t* ids_prey, int32_t* xy_prey, double* energy_prey,
                 int32_t* xy_grass, double* energy_grass);

/* `grid_world_state` (BASE:311; ECO, STAG and the trait variants alike) of the envs [env_begin, env_begin + n_envs):
 * out (DEVICE, [n_envs][num_obs_channels][grid_size][grid_size] fp32, index order [c][x][y] like the rows) receives the
 * grid as the reference holds it after step(), rounded to fp32 the way the observation rows round it (BASE keeps its
 * grid in float64: this is its fp32 rounding).  Channels as in the rows: BASE wall, predator, prey, grass; ECO
 * family predator, prey, grass; STAG walls, predators, mammoths, rabbits, grass.  ECO's own-speed plane is row-only.
 * The result is the world of the handle's last output (ppg_step / full ppg_reset): for an env reset by that call
 * (autoreset, scheduled masked reset, full reset) the world after the reset; for an env whose episode ended in it the
 * world after the final step; an idle env (autoreset off) keeps the world of its final step.  A masked ppg_reset only
 * schedules resets and changes nothing here.  Stream-ordered, no synchronisation; one kernel launch.
 * PPG_ERR_INVALID: NULL handle or out, n_envs < 1 or the range not inside [0, n_envs of the handle).
 * PPG_ERR_STATE: no output since ppg_create; no output since ppg_restore (a snapshot does not carry the world image),
 * or no full ppg_reset since a ppg_restore that left envs idle (their image is never rewritten by a step); the one-kernel
 * step (PPG_OBS_SPLIT=0) keeps no image. */
int ppg_world_state(ppg_handle h, int32_t env_begin, int32_t n_envs, float* out, void* cuda_stream);

/*
 * Agent state aligned with the rows: for every row of the handle's last output (the rows of ppg_get_buffers after the last
 * ppg_step, ppg_step_ordered, ppg_step_host, full ppg_reset or step of ppg_rollout_random), the state of the agent behind it,
 * as ppg_read_env / ppg_read_env_eco / ppg_read_env_stag / ppg_read_env_acc report it after the same output.
 *
 *   Present: row r of species s, with e = row_env[s][r] and id = row_agent[s][r] (STAG: the flat id, which the rows and the
 *     lists both carry), is present when env_flags[e] has neither PPG_ENV_TERMINATED nor PPG_ENV_TRUNCATED and env e's agent
 *     list of species s holds an entry with that id.  Its columns are that entry's:
 *       pos (x, y); energy (f64); age (ECO family, STAG); trait (f64: the ECO family's genome `speed` as ppg_read_env_eco
 *       reports it, which holds the trait of the trait variants; STAG predators' cooperation trait); facing (STAG predators,
 *       index into `_predator_facing_options`); acc (cadence variant: the move accumulator).
 *   Absent rows get present = 0, pos = (-1, -1), energy = trait = acc = NaN, age = facing = -1.  That covers every row of an
 *     env whose episode ended in this output (survivors and ECO newborn rows kept at birth included: an auto-resetting env
 *     does not write its lists back on the step that ends its episode, so they are not its final state), and every row whose
 *     agent left the list (BASE and STAG deaths, eaten ECO prey).  ECO carcasses stay in the list: their TERMINATED row is
 *     present and flagged PPG_ROW_CARCASS.  Rows at or beyond the output's row count are not written.
 *   Grass, per env: grass_pos and grass_energy as ppg_read_env reports them; -1 / NaN for an env whose episode ended in this
 *     output.  An idle env (autoreset off) has no rows; its grass is that of its final step.
 *
 * The state of an ended env's final step is not reported (out of reach for auto-resetting envs, see above; one rule for
 * every ended env).  The call describes the last output until the next one: a masked ppg_reset only schedules resets and
 * changes nothing here.  It works with the two-kernel and the one-kernel step (PPG_OBS_SPLIT=0).
 *
 * Kernel: one warp per env.  Per species it writes the sentinels into the env's rows, then (after __syncwarp) each lane takes
 * list entries k and writes entry k's columns into row ag_prow[k] when that row lies in the env's row ranges and carries the
 * entry's id.  The ids of one env's rows are distinct, so every present row is written by exactly one entry; a list entry
 * without a row in this output (an ECO carcass of an earlier output, whose recorded row is stale) writes nothing.  No atomics:
 * the result does not depend on scheduling.  Launched after the observation kernel with plain stream order, it never triggers
 * dependent launches, so with the launch chain on the next step's kernels do not start while it still reads the lists and rows.
 */
typedef struct ppg_agent_state_args {
  uint8_t* present[2];   /* [row_capacity[s]] required: 1 = present */
  int32_t* pos[2];       /* [row_capacity[s]][2] x, y */
  double* energy[2];     /* [row_capacity[s]] */
  double* trait[2];      /* [row_capacity[s]] ECO family both species, STAG predators */
  double* acc[2];        /* [row_capacity[s]] cadence variant */
  int32_t* age[2];       /* [row_capacity[s]] ECO family, STAG */
  int8_t* facing[2];     /* [row_capacity[s]] STAG predators */
  int32_t* grass_pos;    /* [n_envs][n_grass][2] x, y */
  double* grass_energy;  /* [n_envs][n_grass] */
} ppg_agent_state_args;

/* Writes the columns above into the caller's DEVICE arrays: one kernel launch on cuda_stream, no synchronisation.  A NULL
 * column pointer (other than present) is not written.
 * PPG_ERR_INVALID: NULL handle or args, a NULL present[s], or a non-NULL column the variant or species does not have (age on
 * BASE, trait on BASE or STAG prey, facing other than on STAG predators, acc other than on the cadence variant).
 * PPG_ERR_STATE: no output since ppg_create, or no output since ppg_restore. */
int ppg_agent_state(ppg_handle h, const ppg_agent_state_args* a, void* cuda_stream);

/*
 * Episode returns and agent lifetimes on the device (RLlib's episode_return_mean, episode_len_mean,
 * module_episode_returns_mean; the per-life records the evolutionary analyses read).  Off by default: while off nothing is
 * launched, allocated or changed.  While on, every output (ppg_reset without a mask, ppg_step, ppg_step_ordered,
 * ppg_step_host, every step of ppg_rollout_random) is followed by one more kernel on the same stream that updates:
 *
 *   Row columns, per species, indexed like the rows of the output they belong to:
 *     row_return[s][r] (f64): the agent's return so far in this life: the sum, in f64, of the fp32 reward[s] of every row
 *       the agent has had in the current episode, this one included (the rewards the rows hand out, not the reference's
 *       internal float64 ones);
 *     row_life[s][r] (int32): the number of rows the agent has had in this episode, this one included.
 *     A row flagged PPG_ROW_FOUNDER or PPG_ROW_NEWBORN starts a new life (row_return = reward, row_life = 1); any other row
 *     continues the life of the same (env, numeric id) of the previous output.  On a row flagged TERMINATED or TRUNCATED
 *     they are the agent's lifetime return and lifetime rows.
 *   Per env:
 *     env_return[e][2] (f64): the running episode return per species after this output.  An output with PPG_ENV_RESET
 *       starts it from 0 before adding its own rows.  An output with PPG_ENV_TERMINATED | PPG_ENV_TRUNCATED ends the
 *       episode, which is folded into the env's accumulators env_acc[e][PPG_EP_*]: one episode, its length env_step[e],
 *       its return per species and in total, the square of the total, the max and -min of the total.  A masked reset
 *       abandons a running episode: it is not counted.  Idle envs (PPG_ENV_IDLE) change nothing.
 *     For every row flagged TERMINATED or TRUNCATED the env's per-species accumulators add one life ended, one death
 *       (TERMINATED only), its row_return and its row_life.
 *   Validity: env_valid[e] is cleared when tracking is switched on and by ppg_restore (the tracking state is not part of
 *     the snapshot blob), and set again by the env's next output with PPG_ENV_RESET.  An invalid env writes NaN / 0 into
 *     its rows' columns, keeps env_return at NaN and accumulates nothing.  Switched on before the first full reset,
 *     tracking sees every episode; envs part-way through an episode are counted from their next episode on.
 *
 * Kernel: one warp per env.  Per species it first updates the env's old rows (lanes in parallel, the old rows of an env
 * have distinct ids), then, after __syncwarp, its newborn rows, so an old TERMINATED row finishes its id's life before a
 * newborn row could restart that id (every variant hands newborns never-used ids today, so no id is reused within an
 * episode; the order keeps the tables right should one ever be reused in the step that freed it).  The per-step
 * sums (the step reward per species, the returns of the lives ended) are formed in one fixed order: lane l adds, in f64 and
 * in row order, old rows l, l+32, ... and then newborn rows l, l+32, ... to a partial starting at 0.0; the 32 partials are
 * combined by an xor-butterfly (v += shfl_xor(v, k), k = 16, 8, 4, 2, 1).  Per-agent state lives in tables indexed by
 * (env, numeric id; STAG: the flat id): 12 bytes x n_envs x (n_possible[0] + n_possible[1]), allocated with the row
 * columns and the per-env state when tracking is first switched on.  The kernel is launched after the observation kernel
 * with plain stream order and never triggers dependent launches, so with the launch chain on the next step's kernels do
 * not start while it still reads reward, flags and row_agent.
 */
#define PPG_N_EP_STATS 16
enum {
  PPG_EP_EPISODES = 0,       /* episodes finished */
  PPG_EP_LENGTH_SUM = 1,     /* sum of their lengths (env_step at the end) */
  PPG_EP_RETURN_SUM = 2,     /* sum of their total returns (predator + prey) */
  PPG_EP_RETURN_SQ_SUM = 3,  /* sum of the squares of their total returns */
  PPG_EP_RETURN_PRED = 4,    /* sum of their predator returns */
  PPG_EP_RETURN_PREY = 5,    /* sum of their prey returns */
  PPG_EP_RETURN_MAX = 6,     /* max total return (-inf: no episode); reduces with MAX */
  PPG_EP_RETURN_NEG_MIN = 7, /* -(min total return) (-inf: no episode); reduces with MAX */
  PPG_EP_LIVES = 8,          /* per species, slot + 4 * s: lives ended (rows flagged TERMINATED or TRUNCATED) */
  PPG_EP_DEATHS = 9,         /* ... of them TERMINATED */
  PPG_EP_LIFE_RETURN = 10,   /* ... sum of their lifetime returns (row_return) */
  PPG_EP_LIFE_ROWS = 11      /* ... sum of their lifetime rows (row_life) */
};
#define PPG_EP_SPECIES_STRIDE 4

/* Device pointers of the tracking state; valid while tracking is on, until ppg_destroy. */
typedef struct ppg_returns {
  double* row_return[2]; /* [row_capacity[s]] */
  int32_t* row_life[2];  /* [row_capacity[s]] */
  double* env_return;    /* [n_envs][2] */
  uint8_t* env_valid;    /* [n_envs] */
  double* env_acc;       /* [n_envs][PPG_N_EP_STATS]: each env's share of the aggregate vector */
} ppg_returns;

/* Switches tracking on (on != 0) or off.  The first switch-on allocates the state and clears the accumulators; every
 * switch-on marks all envs invalid until their next reset (stream-ordered on cuda_stream).  Switching off keeps the state
 * and the accumulators.  PPG_ERR_CUDA if the allocation fails. */
int ppg_track_returns(ppg_handle h, int32_t on, void* cuda_stream);
/* The device pointers of the tracking state.  PPG_ERR_STATE while tracking is off. */
int ppg_get_returns(ppg_handle h, ppg_returns* out);
/* The aggregate vector: env_acc summed over the envs whose env_valid is set (slots 6 and 7: max), PPG_N_EP_STATS doubles
 * left in a device buffer of the handle (valid until the next call).  Reduced in a fixed order, so it is bit-identical from
 * run to run.  Stream-ordered, no synchronisation; two kernel launches.  PPG_ERR_STATE before tracking was first on. */
int ppg_episode_stats_device(ppg_handle h, double** dev_out, void* cuda_stream);
/* Clears every env's accumulators (stream-ordered, one kernel launch).  PPG_ERR_STATE before tracking was first on. */
int ppg_episode_stats_clear(ppg_handle h, void* cuda_stream);

/*
 * Advantages and value targets of a rollout (RLlib PPO's GAE: `advantages` are the lambda-returns minus `vf_preds`).
 * A rollout is T+1 consecutive outputs 0..T of one handle, copied by the caller into slabs (slot t = output t).  For every
 * output the caller supplies value[s][t][r] (fp32), the value estimate of row r of output t, for every row, including rows
 * flagged TERMINATED or TRUNCATED.
 *
 *   Successor link: row r of output t < T has a successor when output t+1 holds a row of the same (env, row_agent) (STAG: the
 *     flat id) that is flagged neither FOUNDER nor NEWBORN; next_row[s][t][r] is its row, else -1.  Rows flagged TERMINATED
 *     or TRUNCATED, rows of an env whose output t+1 has PPG_ENV_RESET (a masked or automatic reset: the step did not happen
 *     for them) and the rows of output T have none.  A row with a successor is exactly a transition: the rows of output t
 *     with a successor are as many as the rows of output t+1 that are old and not FOUNDER.
 *   End of a life: a successor row r' of output t+1, with row flags f and env flags ef of output t+1, is
 *     terminal  when (f & TERMINATED) or ((ef & PPG_ENV_TERMINATED) and not (f & TRUNCATED));
 *     truncated when it is not terminal and (f & TRUNCATED) or (ef & PPG_ENV_TRUNCATED).
 *     So each variant's own flags decide: BASE leaves the survivors of an extinction unflagged and ECO flags them
 *     TERMINATED, both are terminal (RLlib's `__all__` ends every agent); STAG flags them TRUNCATED (STAG:587-591), they
 *     bootstrap.
 *   Recursion, in fp32, each expression evaluated exactly as written (no fused multiply-add), gl = fp32(gamma) * fp32(lambda)
 *   computed once; for every transition (t, r) -> (t+1, r'):
 *     vn    = terminal(r') ? 0 : value[t+1][r']
 *     cont  = t+1 < T && !terminal(r') && !truncated(r') && next_row[t+1][r'] >= 0
 *     An    = cont ? adv[t+1][r'] : 0
 *     delta = (reward[t+1][r'] + gamma * vn) - value[t][r]
 *     adv[t][r]          = delta + gl * An
 *     value_target[t][r] = adv[t][r] + value[t][r]
 *   A live agent at the end of the rollout bootstraps from V(output T); so does an agent whose next output is a masked reset
 *   (its last row has no successor) and a truncated life (from the value of its final row).  Rows of output t without a
 *   successor get adv = value_target = NaN; rows at or beyond the output's row count are not written.
 *
 * Slabs, [s] = species, C = row_capacity[s] of the handle, B = n_envs; slot t of a slab starts at element t * C (rows) or
 * t * B, t * (B + 1) (per-env columns), every slab is a DEVICE array.  The env's rows of output t are
 * [old_off[t][e], old_off[t][e+1]) and [new_off[t][e], new_off[t][e] + new_cnt[t][e]) as in ppg_buffers.
 */
#define PPG_GAE_ERR_ID 0x1u    /* a row's id is outside [0, n_possible[s]) */
#define PPG_GAE_ERR_LINK 0x2u  /* an old, non-FOUNDER row of output t+1 has no live row of the same id in output t */
#define PPG_GAE_ERR_RANGE 0x4u /* an env's row range lies outside [0, C), or it holds more old rows than fit the link table */
typedef struct ppg_gae_args {
  int32_t T;                  /* steps of the rollout (>= 1): outputs 0..T */
  float gamma, lam;            /* discount and GAE lambda, each in [0, 1] */
  const int32_t* row_agent[2]; /* [T+1][C] */
  const uint8_t* flags[2];     /* [T+1][C] PPG_ROW_* */
  const float* reward[2];      /* [T+1][C] */
  const float* value[2];       /* [T+1][C] */
  const int32_t* old_off[2];   /* [T+1][B+1] */
  const int32_t* new_off[2];   /* [T+1][B] */
  const int32_t* new_cnt[2];   /* [T+1][B] */
  const uint8_t* env_flags;    /* [T+1][B] PPG_ENV_* */
  float* adv[2];               /* [T][C] out */
  float* value_target[2];      /* [T][C] out */
  int32_t* next_row[2];        /* [T][C] out */
  uint32_t* error;             /* [1] out: cleared by the call, then PPG_GAE_ERR_* bits ORed in by the kernel */
} ppg_gae_args;

/* Links the rows of the rollout and runs the recursion above: one kernel launch on cuda_stream (after a 4-byte memset of
 * a->error), one warp per env and species walking backward from t = T-1 to 0.  The links are matched per env in a hash table
 * of the env's old rows in shared memory (2 x 4 bytes x the next power of two >= 2 * max(cap_live) per warp): the memory
 * does not grow with n_possible.  It reads only the caller's slabs, never the handle's live outputs, keeps no state in the
 * handle, does not synchronise and never triggers dependent launches.  The result is deterministic: every value is one chain
 * of fp32 operations.  Malformed slabs do not fault: the kernel sets PPG_GAE_ERR_* in *a->error (a device word the caller
 * reads when it synchronises, as it reads the step kernels' status words) and leaves the affected rows unlinked.
 * PPG_ERR_INVALID: NULL handle, args or pointer, T < 1, gamma or lambda outside [0, 1], max(cap_live) > 8192 (the two tables
 * of one warp would not fit in shared memory). */
int ppg_gae(ppg_handle h, const ppg_gae_args* a, void* cuda_stream);

/* ECO extras of one env (ECO attributes agent_ages, agent_genomes[..].speed, dead_prey,
 * active_num_predators/prey), in the list order of ppg_read_env.  Any pointer may be NULL. Synchronises. */
int ppg_read_env_eco(ppg_handle h, int32_t env, int32_t* age_pred, double* speed_pred, int32_t* age_prey,
                     double* speed_prey, uint8_t* dead_prey, int32_t* active_num);

/* CAD: `agent_move_accumulator` (CAD:183-186) of the live agents of one env, in the order of ppg_read_env (cadence handles
 * only; either pointer may be NULL).  Synchronises the device. */
int ppg_read_env_acc(ppg_handle h, int32_t env, double* acc_pred, double* acc_prey);

/* ECO per-episode totals of one env for `_build_episode_training_metrics` (ECO:1613-1661), valid with
 * ppg_config.track_episode_sums: sums[4] = distance moved by all predators / all prey of the running episode (the sum of
 * record["distance_traveled"] over the species' agent records, ECO:659), locomotion energy spent likewise
 * (record["movement_energy_spent"], ECO:660); spawned[2] = agents born so far per species (= the sum of
 * record["offspring_count"], ECO:1168,1262; the species' record count is founders + spawned).  Synchronises. */
int ppg_read_episode_eco(ppg_handle h, int32_t env, double* sums, int32_t* spawned);

/* Trait variants (MR / INV / COOP), valid with ppg_config.track_episode_sums: the event counters of the running episode that
 * `_build_episode_training_metrics` reports — events[6] = {reproduction_blocked_due_to_capacity_predator, _prey (id pool
 * exhausted: MR:857,943 -> "predator_reproduction_blocked", "prey_reproduction_blocked", MR:1347-1348),
 * reproduction_blocked_due_to_density_predator (MR:852 -> "predator_reproduction_blocked_density", MR:1349),
 * satiation_blocked_catches_predator (MR:739 -> "predator_satiation_blocked_catches", MR:1350),
 * total_energy_donated["predator"], ["prey"] (= total_energy_received; COOP:585-586 -> "*_energy_donated_total",
 * "*_energy_received_total", COOP:1365-1368), accumulated in the reference's order}.  Synchronises. */
int ppg_read_episode_events_eco(ppg_handle h, int32_t env, double* events);

/* STAG extras of one env (STAG attributes agent_ages, predator_facing as an index into `_predator_facing_options`
 * STAG:197-206, predator_cooperation_trait), in the list order of ppg_read_env, plus the team-capture counters
 * capture[12] = {successes, failures, coop_successes, coop_failures, mammoth_successes, mammoth_failures,
 * rabbit_successes, rabbit_failures, attempts, helper_total, spawned_predators, spawned_prey} (STAG:237-254) and
 * capture_real[3] = {last_success_prob, last_effort_ratio, success_prob_sum} (STAG:249-251).  Any pointer may be NULL.
 * Synchronises. */
int ppg_read_env_stag(ppg_handle h, int32_t env, int32_t* age_pred, int32_t* facing_pred, double* trait_pred,
                      int32_t* age_prey, int64_t* capture, double* capture_real);

/* Device-side reduction of the per-env counters into PPG_N_STATS int64 values (host out).
 * Synchronises the stream. ppg_stats_device leaves them on the device for an NCCL all-reduce. */
int ppg_stats(ppg_handle h, int64_t* out, void* cuda_stream);
int ppg_stats_device(ppg_handle h, int64_t** dev_out, void* cuda_stream);
int ppg_stats_clear(ppg_handle h, void* cuda_stream);

/* Kernel launches issued by this handle since creation (bench `gpu_launches`). */
int64_t ppg_launch_count(ppg_handle h);

/* Per-kernel timing of the steps between the two calls (bench.py `roofline`): CUDA events are recorded on the
 * step's own stream before the step kernel, between it and the observation kernel, and after the latter.
 * ppg_profile_end synchronises and returns the summed durations in milliseconds and the number of steps timed
 * (ms_obs_kernel = 0 when the handle runs the one-kernel step, PPG_OBS_SPLIT=0). */
int ppg_profile_begin(ppg_handle h);
/* SM cycles the step kernel spent on every env in the last launch (host out [n_envs]); info = mode (0 idle, 1 reset,
 * 2 step) | births << 8 | agents << 16; start_ns = low 32 bits of the GPU's nanosecond timer when the env was taken;
 * sm = the SM it ran on (info, start_ns, sm may be NULL).  One warp owns an env for a whole step, so this is the
 * per-env step latency and the kernel's schedule. */
int ppg_profile_env_cycles(ppg_handle h, uint32_t* cycles, uint32_t* info, uint32_t* start_ns, uint32_t* sm, void* cuda_stream);
int ppg_profile_end(ppg_handle h, double* ms_step_kernel, double* ms_obs_kernel, int32_t* n_steps);

/* Diagnostic: out[i] = the device's pow(x[i], y[i]) (include/ppg_pow.h: glibc's pow repeated bit for bit — what the
 * kernels use for `speed ** exponent`, ECO:559-563, and `(1 - p0) ** ratio`, STAG:1137).  Host pointers; synchronises.
 * tests/test_gpu_pow.py compares it with the host libm on millions of arguments. */
int ppg_selftest_pow(const double* x, const double* y, double* out, int64_t n, int32_t device);

const char* ppg_last_error(ppg_handle h);
int ppg_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PPG_H_ */
